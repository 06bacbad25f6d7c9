// G1 instantiation of the MSM / table entry points (include/zkp_b200.h).
#include "msm_api.cuh"

namespace zkp {
static MsmOptions g_msm_options;
MsmOptions& msm_options() { return g_msm_options; }
}  // namespace zkp
namespace zkp {
int g2_msm_enqueue(Context& c, uint64_t table, uint64_t scalars, uint64_t n, int slot, char* dev_out);  // msm_g2.cu
}
using namespace zkp;
using Api = GroupApi<Fp>;

extern "C" {

int zkp_msm_set_window_bits(int c) {
  if (c != 0 && (c < 2 || c > MSM_MAX_C)) {
    set_last_error("zkp_msm_set_window_bits: c must be 0 or in [2,20]");
    return ZKP_ERR_INVALID_ARGUMENT;
  }
  msm_options().window_bits = c;
  return ZKP_OK;
}

int zkp_msm_set_option(const char* name, int value) {
  std::string n = name ? name : "";
  if (n == "window_bits") return zkp_msm_set_window_bits(value);
  if (n == "accumulate" && value >= 0 && value <= 2) {  // 0 automatic, 1 XYZZ chains, 2 affine tree
    msm_options().accumulate = value;
    return ZKP_OK;
  }
  if (n == "tree_items" && value >= 0 && value <= 256) {  // additions per thread under one shared inversion
    msm_options().tree_items = value;
    return ZKP_OK;
  }
  if (n == "parts" && value >= 0 && value <= 8) {  // point ranges of a part-streamed MSM (0 = automatic)
    msm_options().parts = value;
    return ZKP_OK;
  }
  if (n == "tree_rounds" && value >= 0 && value <= 9) {  // affine rounds before the XYZZ chains take over
    msm_options().tree_rounds = value;
    return ZKP_OK;
  }
  if (n == "reduce_radix" && (value == 0 || value == 2 || value == 4 || value == 8 || value == 16 || value == 32)) {
    msm_options().reduce_radix = value;  // items per thread of a wide level of the weighted-sum recursion
    return ZKP_OK;
  }
  if (n == "wide_log2" && value >= 0 && value <= 31) {  // item count from which a level is a wide one
    msm_options().wide_log2 = value;
    return ZKP_OK;
  }
  if (n == "quad_log2" && value >= 0 && value <= 31) {  // radix-2 output count up to which levels are fused on quads
    msm_options().quad_log2 = value;
    return ZKP_OK;
  }
  set_last_error("zkp_msm_set_option: unknown option or value (window_bits, accumulate 0..2, tree_items 0..256, tree_rounds 0..9, parts 0..8, reduce_radix 0/2/4/8/16/32, wide_log2, quad_log2)");
  return ZKP_ERR_INVALID_ARGUMENT;
}

int zkp_g1_msm_multi(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                     uint8_t out_xy[64], int* out_is_inf) {
  return Api::msm_multi(table, offset, scalars, sc_offset, n, out_xy, out_is_inf);
}
int zkp_g1_msm_dev_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n) {
  return Api::msm_begin(table, offset, scalars, sc_offset, n, false);
}
int zkp_g1_msm_dev_end(uint8_t out_xy[64], int* out_is_inf) { return Api::msm_multi_end(out_xy, out_is_inf); }
int zkp_g1_msm_multi_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n) {
  return Api::msm_multi_begin(table, offset, scalars, sc_offset, n);
}
int zkp_g1_msm_multi_end(uint8_t out_xy[64], int* out_is_inf) { return Api::msm_multi_end(out_xy, out_is_inf); }
int zkp_g1_msm_multi_table(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t out_xy[64],
                           int* out_is_inf) {
  return Api::msm_multi_host(table, offset, scalars, n, out_xy, out_is_inf);
}

int zkp_g1_msm(const uint8_t* pts, const uint8_t* scalars, uint64_t n, uint8_t out_xy[64], int* out_is_inf) {
  return Api::msm_host(pts, scalars, n, out_xy, out_is_inf);
}
int zkp_g1_table_load(const uint8_t* pts, uint64_t n, uint64_t* handle) { return Api::table_load(pts, n, handle); }
int zkp_g1_msm_table(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t out_xy[64],
                     int* out_is_inf) {
  return Api::msm_table(table, offset, scalars, n, out_xy, out_is_inf);
}
int zkp_g1_msm_dev(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                   uint8_t out_xy[64], int* out_is_inf) {
  return Api::msm_dev(table, offset, scalars, sc_offset, n, out_xy, out_is_inf, false);
}
int zkp_g1_msm_dev_partial(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                           uint8_t out_xyzz[128]) {
  return Api::msm_dev(table, offset, scalars, sc_offset, n, out_xyzz, nullptr, true);
}
int zkp_g1_combine_partials(const uint8_t* partials, uint32_t count, uint8_t out_xy[64], int* out_is_inf) {
  return Api::combine(partials, count, out_xy, out_is_inf);
}
int zkp_g1_fixed_base_mul(const uint8_t base_xy[64], const uint8_t* scalars, uint64_t n, uint64_t* out_table) {
  return Api::fixed_base_host(base_xy, scalars, n, out_table);
}
int zkp_g1_fixed_base_mul_dev(const uint8_t base_xy[64], uint64_t scalars, uint64_t n, uint64_t* out_table) {
  return Api::fixed_base_dev(base_xy, scalars, n, out_table);
}

int zkp_g1_table_scale(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                       uint64_t* out_table) {
  return Api::table_scale(table, offset, scalars, sc_offset, n, out_table);
}
int zkp_g1_table_validate(uint64_t table, uint64_t offset, uint64_t n, uint64_t* first_bad) {
  return Api::table_validate(table, offset, n, 0, first_bad);
}

int zkp_g1_msm_dev_batch(uint64_t table, uint32_t count, const uint64_t* scalars, const uint64_t* sc_offsets,
                         const uint64_t* offsets, const uint64_t* lens, uint8_t* out_xy, int* out_is_inf) {
  return Api::msm_batch(table, count, scalars, sc_offsets, offsets, lens, out_xy, out_is_inf);
}
int zkp_g1_table_precompute(uint64_t table, int window_bits) { return Api::table_precompute(table, window_bits); }
int zkp_g1_msm_dev_many(uint64_t table, uint64_t offset, uint64_t n, uint32_t count, uint64_t scalars, uint64_t sc_offset,
                        uint8_t* out_xy, int* out_is_inf) {
  return Api::msm_dev_many(table, offset, n, count, scalars, sc_offset, out_xy, out_is_inf);
}

// G1 or G2 table -> canonical affine points on the host
int zkp_table_download(uint64_t table, uint64_t offset, uint64_t n, uint8_t* out_pts) {
  return guarded([&](Context& c) {
    if (n && !out_pts) throw InvalidArgument("zkp_table_download: null output");
    if (Resource* t = registry().get(table, HandleKind::G1Table)) {
      GroupApi<Fp>::download(c, t, offset, n, out_pts);
    } else if (Resource* t2 = registry().get(table, HandleKind::G2Table)) {
      GroupApi<Fp2>::download(c, t2, offset, n, out_pts);
    } else {
      throw BadHandle("zkp_table_download: not a point table");
    }
  });
}

int zkp_g1_table_load_compressed(const uint8_t* enc, uint64_t n, uint64_t* handle, uint64_t* first_bad) {
  return Api::table_load_compressed(enc, n, false, handle, first_bad);
}

// G1 or G2 table -> compressed encodings on the host (32 / 64 B per point)
int zkp_table_download_compressed(uint64_t table, uint64_t offset, uint64_t n, uint8_t* out) {
  return guarded([&](Context& c) {
    if (n && !out) throw InvalidArgument("zkp_table_download_compressed: null output");
    if (Resource* t = registry().get(table, HandleKind::G1Table)) {
      GroupApi<Fp>::download_compressed(c, t, offset, n, out);
    } else if (Resource* t2 = registry().get(table, HandleKind::G2Table)) {
      GroupApi<Fp2>::download_compressed(c, t2, offset, n, out);
    } else {
      throw BadHandle("zkp_table_download_compressed: not a point table");
    }
  });
}

// The three multi-scalar multiplications of one Groth16 proof (proving.py:23-75 reduced to one MSM per
// element, device_prover.py): B (G2) runs on the second stream beside A and C (G1) on the first.  The G2
// accumulation keeps only 8 warps per SM busy (228 registers per thread), so blocks of the G1 kernels
// co-reside with it and fill the integer pipe, and each lane's latency-bound tail hides behind the other.
int zkp_groth16_msms_dev(uint64_t ta, uint64_t sa, uint64_t na, uint64_t tb2, uint64_t sb, uint64_t nb, uint64_t tc,
                         uint64_t sc, uint64_t nc, uint8_t out_a[64], uint8_t out_b[128], uint8_t out_c[64],
                         int out_is_inf[3]) {
  return guarded([&](Context& c) {
    if (!out_a || !out_b || !out_c) throw InvalidArgument("zkp_groth16_msms_dev: null output");
    Resource* rta = need(ta, HandleKind::G1Table, "zkp_groth16_msms_dev");
    Resource* rtc = need(tc, HandleKind::G1Table, "zkp_groth16_msms_dev");
    Resource* rsa = need(sa, HandleKind::Scalars, "zkp_groth16_msms_dev");
    Resource* rsc = need(sc, HandleKind::Scalars, "zkp_groth16_msms_dev");
    if (na > rta->n || na > rsa->n || nc > rtc->n || nc > rsc->n) throw InvalidArgument("zkp_groth16_msms_dev: range out of bounds");
    static DevBuf res;  // A: [0,64) flag [64,68) | C: [128,192) flag [192,196) | B: [256,384) flag [384,388)
    res.reserve(512);
    char* r = res.as<char>();
    CUDA_CHECK(cudaEventRecord(c.ev_fork, c.stream));
    CUDA_CHECK(cudaStreamWaitEvent(c.stream2, c.ev_fork, 0));
    c.launches += g2_msm_enqueue(c, tb2, sb, nb, 1, r + 256);
    MsmEngine<Fp>& e = Api::engine(0);
    c.launches += Api::run_on_table(c, rta, 0, rsa->buf.as<uint32_t>(), na, false, 0);
    CUDA_CHECK(cudaMemcpyAsync(r, e.result.p, 64, cudaMemcpyDeviceToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(r + 64, e.flag.p, sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
    c.launches += Api::run_on_table(c, rtc, 0, rsc->buf.as<uint32_t>(), nc, false, 0);
    CUDA_CHECK(cudaMemcpyAsync(r + 128, e.result.p, 64, cudaMemcpyDeviceToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(r + 192, e.flag.p, sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
    CUDA_CHECK(cudaEventRecord(c.ev_join, c.stream2));
    CUDA_CHECK(cudaStreamWaitEvent(c.stream, c.ev_join, 0));
    uint8_t host[512];
    CUDA_CHECK(cudaMemcpyAsync(host, r, 512, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    int fa, fc, fb;
    memcpy(&fa, host + 64, 4);
    memcpy(&fc, host + 192, 4);
    memcpy(&fb, host + 384, 4);
    if (fa) memset(out_a, 0, 64); else memcpy(out_a, host, 64);
    if (fc) memset(out_c, 0, 64); else memcpy(out_c, host + 128, 64);
    if (fb) memset(out_b, 0, 128); else memcpy(out_b, host + 256, 128);
    if (out_is_inf) { out_is_inf[0] = fa; out_is_inf[1] = fb; out_is_inf[2] = fc; }
  });
}

// window width of a precomputed table (0 = plain layout)
int zkp_table_window_bits(uint64_t table, int* window_bits) {
  return guarded([&](Context&) {
    if (!window_bits) throw InvalidArgument("zkp_table_window_bits: null output");
    Resource* t = registry().get(table, HandleKind::G1Table);
    if (!t) t = registry().get(table, HandleKind::G2Table);
    if (!t) throw BadHandle("zkp_table_window_bits: not a point table");
    *window_bits = t->pre_c;
  });
}

}  // extern "C"
