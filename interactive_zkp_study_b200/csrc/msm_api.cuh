// Group-generic implementation of the MSM / table entry points; instantiated for G1 (msm_g1.cu)
// and G2 (msm_g2.cu).  See include/zkp_b200.h for the contract of each function.
#pragma once
#include <type_traits>
#include "comm.cuh"
#include "curve_check.cuh"
#include "msm.cuh"
#include "point_codec.cuh"
#include "registry.cuh"

namespace zkp {

// s = scalars[i] mod r: any 256-bit value, 32 B canonical little-endian (2^256 < 6 r: at most five subtractions)
ZKP_DEVINL void load_scalar_mod_r(const uint32_t* __restrict__ scalars, uint64_t i, uint32_t s[8]) {
  const uint4* sp = reinterpret_cast<const uint4*>(scalars + 8 * i);
  uint4 lo = sp[0], hi = sp[1];
  s[0] = lo.x; s[1] = lo.y; s[2] = lo.z; s[3] = lo.w;
  s[4] = hi.x; s[5] = hi.y; s[6] = hi.z; s[7] = hi.w;
  for (int it = 0; it < 6; it++) {
    uint32_t t[8], borrow = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      uint64_t d = (uint64_t)s[k] - FrParams::MOD_(k) - borrow;
      t[k] = (uint32_t)d;
      borrow = (uint32_t)(d >> 63);
    }
    if (borrow) break;
#pragma unroll
    for (int k = 0; k < 8; k++) s[k] = t[k];
  }
}

// out[i] = scalars[i] * base: MSB-first double-and-add in XYZZ with mixed additions, one thread per
// scalar, then one inversion per point.  Replaces the n sequential Python scalar-muls of
// SRS.generate (/root/reference/zkp/plonk/srs.py:78-82) and sigma12/15/22 (setup.py:18-23,56-69).
template <class F>
__global__ void __launch_bounds__(128) fixed_base_mul_kernel(Affine<F> base_canon, const uint32_t* __restrict__ scalars,
                                                              uint64_t n, Affine<F>* __restrict__ out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Affine<F> base = {base_canon.x.to_mont(), base_canon.y.to_mont()};
  uint32_t s[8];
  load_scalar_mod_r(scalars, i, s);
  XYZZ<F> acc = XYZZ<F>::inf();
  for (int w = 7; w >= 0; w--) {
    uint32_t word = s[w];
    for (int b = 31; b >= 0; b--) {
      acc = acc.dbl();
      if ((word >> b) & 1) acc.madd(base);
    }
  }
  out[i] = acc.to_affine();  // Montgomery affine, (0,0) for infinity
}

// Windowed fixed-base multiplication for large batches: tab[j*256 + d] = d * 2^(8j) * base (affine
// Montgomery, j < 32, d < 256; built once per call with the kernel above on 8192 small scalars), then
// out[i] = sum_j tab[j][byte_j(s_i)]: at most 32 mixed additions per scalar instead of 254 doublings
// + ~127 additions (11x less work), one inversion per point.
static __global__ void fixed_base_table_scalars_kernel(uint32_t* __restrict__ out) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;  // t = j*256 + d
  if (t >= 8192) return;
  uint32_t j = t >> 8, d = t & 255;
  uint32_t v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  v[j >> 2] = d << ((j & 3) * 8);
#pragma unroll
  for (int k = 0; k < 8; k++) out[8 * t + k] = v[k];
}

template <class F>
__global__ void __launch_bounds__(128) fixed_base_windowed_kernel(const Affine<F>* __restrict__ tab,
                                                                   const uint32_t* __restrict__ scalars, uint64_t n,
                                                                   Affine<F>* __restrict__ out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t s[8];
  load_scalar_mod_r(scalars, i, s);
  XYZZ<F> acc = XYZZ<F>::inf();
#pragma unroll 1
  for (int j = 0; j < 32; j++) {
    uint32_t d = (s[j >> 2] >> ((j & 3) * 8)) & 255u;
    if (d) acc.madd(tab[j * 256 + d]);
  }
  out[i] = acc.to_affine();
}

// out[i] = scalars[i] * pts[i], a different base per thread (zkp_g1/g2_table_scale; the powers-of-tau update
// [tau^i]_1 -> [(s tau)^i]_1 = s^i [tau^i]_1).  Table and result are Montgomery affine, (0,0) for infinity.
//   - tab[d - 1] = d P for d = 1..15, built in XYZZ (one doubling, 13 mixed additions) and made affine with one
//     inversion shared by the 15 entries (Montgomery's trick: 1/(ZZ ZZZ) gives 1/ZZ and 1/ZZZ).
//   - k mod r in 4-bit windows from the top: 4 doublings and at most one mixed addition of tab[d - 1] per window
//     (~252 doublings + <= 64 additions, against 254 doublings + ~127 additions bit by bit), one inversion at the end.
// The table is indexed by a data-dependent digit and so lives in local memory (L1-resident: 15 x 64 B in G1).
template <class F>
__global__ void __launch_bounds__(128) table_scale_kernel(const Affine<F>* __restrict__ pts,
                                                          const uint32_t* __restrict__ scalars, uint64_t n,
                                                          Affine<F>* __restrict__ out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Affine<F> p = pts[i];
  if (p.is_inf()) {
    out[i] = Affine<F>::inf();
    return;
  }
  uint32_t s[8];
  load_scalar_mod_r(scalars, i, s);
  constexpr int TAB = 15;
  Affine<F> tab[TAB];
  F zz[TAB], zzz[TAB], pre[TAB];  // pre[j] = prod_{m <= j} zz[m] zzz[m]
  XYZZ<F> acc = XYZZ<F>::from_affine(p);
  F prod = F::one();
#pragma unroll 1
  for (int j = 0; j < TAB; j++) {
    if (j) acc.madd(p);  // (j + 1) P; an entry at infinity (P of small order off G2) stays (0,0) below
    const bool inf = acc.is_inf();
    tab[j] = {acc.x, acc.y};
    zz[j] = inf ? F::one() : acc.zz;
    zzz[j] = inf ? F::one() : acc.zzz;
    prod = prod * (zz[j] * zzz[j]);
    pre[j] = prod;
  }
  F inv = prod.inv();  // 1 / prod_{m <= j} for the current j, walking down
#pragma unroll 1
  for (int j = TAB - 1; j >= 0; j--) {
    const F im = j ? inv * pre[j - 1] : inv;  // 1 / (zz[j] zzz[j])
    inv = inv * (zz[j] * zzz[j]);
    tab[j] = {tab[j].x * (im * zzz[j]), tab[j].y * (im * zz[j])};
  }
  XYZZ<F> r = XYZZ<F>::inf();
#pragma unroll 1
  for (int w = 63; w >= 0; w--) {
    if (!r.is_inf()) r = r.dbl().dbl().dbl().dbl();
    const uint32_t d = (s[w >> 3] >> ((w & 7) * 4)) & 15u;
    if (d) r.madd(tab[d - 1]);
  }
  out[i] = r.to_affine();
}

// *first_bad = min(first_bad, base + i) for every pts[i], i < n, that is not on its curve (Montgomery coordinates as
// stored in a table) or, with `subgroup` (G2 only), not in the order-r subgroup.  Infinity (0,0) is valid.
template <class F>
__global__ void __launch_bounds__(64) table_validate_kernel(const Affine<F>* __restrict__ pts, uint64_t n, uint64_t base,
                                                            bool subgroup, unsigned long long* __restrict__ first_bad) {
  using FC = typename CompactOf<F>::type;  // same layout, out-of-line products: this is not a hot loop
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Affine<FC> a = reinterpret_cast<const Affine<FC>*>(pts)[i];
  if (a.is_inf()) return;
  bool ok = on_curve_mont(a);
  if constexpr (std::is_same<FC, Fp2>::value) {
    if (ok && subgroup) ok = g2_in_subgroup(a);
  }
  if (!ok) atomicMin(first_bad, (unsigned long long)(base + i));
}

template <class F>
__global__ void combine_partials_kernel(const XYZZ<F>* __restrict__ parts, uint32_t count, Affine<F>* __restrict__ out,
                                        int* __restrict__ inf_flag) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  XYZZ<F> r = XYZZ<F>::inf();
  for (uint32_t k = 0; k < count; k++) r.add(parts[k]);
  Affine<F> a = r.to_affine();
  *inf_flag = r.is_inf() ? 1 : 0;
  a.x = a.x.from_mont();
  a.y = a.y.from_mont();
  *out = a;
}

template <class F>
struct GroupApi {
  static constexpr size_t PT = sizeof(Affine<F>);  // 64 (G1) / 128 (G2)
  static constexpr uint64_t FE_PER_PT = PT / 32;
  static constexpr HandleKind KIND = sizeof(F) == 32 ? HandleKind::G1Table : HandleKind::G2Table;

  // slot 0: the library stream; slot 1: the second lane used by the batched pipeline
  static MsmEngine<F>& engine(int slot = 0) {
    static MsmEngine<F> e[2];
    return e[slot];
  }
  static DevBuf& scratch_pts() {
    static DevBuf b;
    return b;
  }
  static DevBuf& scratch_scalars() {
    static DevBuf b;
    return b;
  }

  static void upload_points(Context& c, const uint8_t* pts, uint64_t n, void* dst) {
    CUDA_CHECK(cudaMemcpyAsync(dst, pts, n * PT, cudaMemcpyHostToDevice, c.stream));
    fe_to_mont_kernel<Fp><<<ceil_div(n * FE_PER_PT, 256), 256, 0, c.stream>>>(reinterpret_cast<Fp*>(dst), n * FE_PER_PT);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  }

  static void fetch_result(Context& c, uint8_t* out_xy, int* out_is_inf) {
    MsmEngine<F>& e = engine();
    int flag = 0;
    CUDA_CHECK(cudaMemcpyAsync(out_xy, e.result.p, PT, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(&flag, e.flag.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    if (flag) memset(out_xy, 0, PT);
    if (out_is_inf) *out_is_inf = flag;
  }

  // plain table: the sub-range is just a pointer offset; precomputed table: stride/offset indexing
  // host_scalars: the scalars are still in host memory and `dscalars` is where they go (uploaded in chunks on
  // the second stream, recoded chunk by chunk on the first: slot 0 only)
  static int run_on_table(Context& c, Resource* t, uint64_t offset, const uint32_t* dscalars, uint64_t n, bool partial,
                          int slot = 0, const uint8_t* host_scalars = nullptr) {
    cudaStream_t st = slot ? c.stream2 : c.stream;
    cudaStream_t lane = slot ? nullptr : c.stream_hi;  // the part-streamed form belongs to the first lane
    if (t->pre_c)
      return engine(slot).run(t->buf.as<Affine<F>>(), dscalars, n, st, partial, t->pre_c, (uint32_t)t->n,
                              (uint32_t)offset, host_scalars, c.stream2, lane);
    return engine(slot).run(t->buf.as<Affine<F>>() + offset, dscalars, n, st, partial, msm_options().window_bits, 0, 0,
                            host_scalars, c.stream2, lane);
  }

  // `count` independent MSMs on one table, alternating between two streams (each with its own
  // workspace): the latency-bound tail of MSM k (bucket fold, reduction levels, inversion: a handful of
  // warps) runs while the integer-bound accumulation of MSM k+1 fills the machine.  A prover issues its
  // commitments in groups (PLONK rounds 1, 3, 5; Groth16 A and C), so this is its natural call shape.
  static int msm_batch(uint64_t table, uint32_t count, const uint64_t* scalars, const uint64_t* sc_off,
                       const uint64_t* offsets, const uint64_t* lens, uint8_t* out_xy, int* out_is_inf) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "msm_batch");
      if (count && (!scalars || !sc_off || !offsets || !lens || !out_xy)) throw InvalidArgument("msm_batch: null argument");
      std::vector<Resource*> sv(count);
      for (uint32_t k = 0; k < count; k++) {
        sv[k] = need(scalars[k], HandleKind::Scalars, "msm_batch");
        if (!range_ok(offsets[k], lens[k], t->n) || !range_ok(sc_off[k], lens[k], sv[k]->n)) throw InvalidArgument("msm_batch: range out of bounds");
      }
      if (!count) return;
      static DevBuf res;
      const size_t stride = PT + 16;
      res.reserve((size_t)count * stride);
      CUDA_CHECK(cudaEventRecord(c.ev_fork, c.stream));
      CUDA_CHECK(cudaStreamWaitEvent(c.stream2, c.ev_fork, 0));
      for (uint32_t k = 0; k < count; k++) {
        int slot = k & 1;
        cudaStream_t st = slot ? c.stream2 : c.stream;
        c.launches += run_on_table(c, t, offsets[k], sv[k]->buf.template as<uint32_t>() + 8 * sc_off[k], lens[k], false, slot);
        MsmEngine<F>& e = engine(slot);
        CUDA_CHECK(cudaMemcpyAsync(res.as<char>() + k * stride, e.result.p, PT, cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(res.as<char>() + k * stride + PT, e.flag.p, sizeof(int), cudaMemcpyDeviceToDevice, st));
      }
      CUDA_CHECK(cudaEventRecord(c.ev_join, c.stream2));
      CUDA_CHECK(cudaStreamWaitEvent(c.stream, c.ev_join, 0));
      std::vector<uint8_t> host((size_t)count * stride);
      CUDA_CHECK(cudaMemcpyAsync(host.data(), res.p, host.size(), cudaMemcpyDeviceToHost, c.stream));
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
      for (uint32_t k = 0; k < count; k++) {
        int flag;
        memcpy(&flag, host.data() + k * stride + PT, sizeof(int));
        if (flag) memset(out_xy + (size_t)k * PT, 0, PT);
        else memcpy(out_xy + (size_t)k * PT, host.data() + k * stride, PT);
        if (out_is_inf) out_is_inf[k] = flag;
      }
    });
  }

  // `count` MSMs over the same points [offset, offset + n), scalar vector j at sc_offset + j * n: one Pippenger pass
  // (MsmEngine::run_many).  The limits are checked on the host before anything is launched.
  static int msm_dev_many(uint64_t table, uint64_t offset, uint64_t n, uint32_t count, uint64_t scalars, uint64_t sc_offset,
                          uint8_t* out_xy, int* out_is_inf) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "msm_dev_many");
      Resource* s = need(scalars, HandleKind::Scalars, "msm_dev_many");
      if (count && !out_xy) throw InvalidArgument("msm_dev_many: null output");
      if (!range_ok(offset, n, t->n)) throw InvalidArgument("msm_dev_many: point range exceeds the table");
      if (!count) return;
      const int force_c = t->pre_c ? t->pre_c : msm_options().window_bits;
      const MsmPlan pl = msm_plan(n ? n : 1, force_c);
      if ((uint64_t)count * pl.W * n >= (1ull << 32)) throw InvalidArgument("msm_dev_many: count * W * n must be < 2^32");
      const uint64_t per_msm = t->pre_c ? pl.B : (uint64_t)pl.W * pl.B;
      if (n && (uint64_t)count * per_msm >= (1ull << 31))
        throw InvalidArgument("msm_dev_many: count * buckets per MSM must be < 2^31");
      if (!range_ok(sc_offset, (uint64_t)count * n, s->n)) throw InvalidArgument("msm_dev_many: scalar range exceeds the handle");
      MsmEngine<F>& e = engine();
      const uint32_t* sc = s->buf.as<uint32_t>() + 8 * sc_offset;
      if (t->pre_c)
        c.launches += e.run_many(t->buf.as<Affine<F>>(), sc, n, count, c.stream, t->pre_c, (uint32_t)t->n, (uint32_t)offset);
      else
        c.launches += e.run_many(t->buf.as<Affine<F>>() + offset, sc, n, count, c.stream, force_c, 0, 0);
      std::vector<uint8_t> host((size_t)count * (PT + sizeof(int)));
      int* flags = reinterpret_cast<int*>(host.data() + (size_t)count * PT);
      CUDA_CHECK(cudaMemcpyAsync(host.data(), e.many_out.p, (size_t)count * PT, cudaMemcpyDeviceToHost, c.stream));
      CUDA_CHECK(cudaMemcpyAsync(flags, e.many_flag.p, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
      for (uint32_t j = 0; j < count; j++) {
        if (flags[j]) memset(out_xy + (size_t)j * PT, 0, PT);
        else memcpy(out_xy + (size_t)j * PT, host.data() + (size_t)j * PT, PT);
        if (out_is_inf) out_is_inf[j] = flags[j];
      }
    });
  }

  static int table_precompute(uint64_t table, int window_bits) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "table_precompute");
      if (t->pre_c) throw InvalidArgument("table_precompute: table is already precomputed");
      if (window_bits == 0) window_bits = msm_auto_precomputed_c(t->n);
      if (window_bits < 2 || window_bits > MSM_MAX_C) throw InvalidArgument("table_precompute: window_bits must be 0 (automatic) or in [2,20]");
      if (t->n == 0) return;
      MsmPlan pl = msm_plan(t->n, window_bits);
      if ((uint64_t)pl.W * t->n >= (1ull << 31)) throw InvalidArgument("table_precompute: W*n must be < 2^31");
      ScopedDevBuf big;  // several GiB: must not leak if the precomputation runs out of memory half way
      big.reserve((size_t)pl.W * t->n * PT);
      c.launches += engine().precompute(t->buf.as<Affine<F>>(), t->n, window_bits, big.as<Affine<F>>(), c.stream);
      t->buf.release();
      t->buf = big.detach();
      t->pre_c = window_bits;
    });
  }

  static int table_load(const uint8_t* pts, uint64_t n, uint64_t* handle) {
    return guarded([&](Context& c) {
      if (!handle || (n && !pts)) throw InvalidArgument("table_load: null argument");
      auto r = std::make_unique<Resource>();
      r->kind = KIND;
      r->n = n;
      r->buf.reserve_pooled(n ? n * PT : PT);
      if (n) upload_points(c, pts, n, r->buf.p);
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
      *handle = registry().put(std::move(r));
    });
  }

  static int msm_host(const uint8_t* pts, const uint8_t* scalars, uint64_t n, uint8_t* out_xy, int* out_is_inf) {
    return guarded([&](Context& c) {
      if (!out_xy || (n && (!pts || !scalars))) throw InvalidArgument("msm: null argument");
      DevBuf& dp = scratch_pts();
      DevBuf& ds = scratch_scalars();
      if (n) {
        dp.reserve(n * PT);
        ds.reserve(n * 32);
        upload_points(c, pts, n, dp.p);
        CUDA_CHECK(cudaMemcpyAsync(ds.p, scalars, n * 32, cudaMemcpyHostToDevice, c.stream));
      }
      c.launches += engine().run(dp.as<Affine<F>>(), ds.as<uint32_t>(), n, c.stream, false, msm_options().window_bits);
      fetch_result(c, out_xy, out_is_inf);
    });
  }

  static int msm_table(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t* out_xy,
                       int* out_is_inf) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "msm_table");
      if (!out_xy || (n && !scalars)) throw InvalidArgument("msm_table: null argument");
      if (!range_ok(offset, n, t->n)) throw InvalidArgument("msm_table: point range exceeds the table");
      DevBuf& ds = scratch_scalars();
      if (n) ds.reserve(n * 32);
      c.launches += run_on_table(c, t, offset, ds.as<uint32_t>(), n, false, 0, scalars);
      fetch_result(c, out_xy, out_is_inf);
    });
  }

  static int msm_dev(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n, uint8_t* out,
                     int* out_is_inf, bool partial) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "msm_dev");
      Resource* s = need(scalars, HandleKind::Scalars, "msm_dev");
      if (!out) throw InvalidArgument("msm_dev: null output");
      if (!range_ok(offset, n, t->n) || !range_ok(sc_offset, n, s->n)) throw InvalidArgument("msm_dev: range out of bounds");
      MsmEngine<F>& e = engine();
      c.launches += run_on_table(c, t, offset, s->buf.as<uint32_t>() + 8 * sc_offset, n, partial);
      if (partial) {
        // cudaMemcpyDefault: `out` may be host memory or a device buffer of this GPU (e.g. the send
        // buffer of the NCCL gather), resolved by unified addressing
        CUDA_CHECK(cudaMemcpyAsync(out, e.result.template as<char>() + PT, sizeof(XYZZ<F>), cudaMemcpyDefault,
                                   c.stream));
        CUDA_CHECK(cudaStreamSynchronize(c.stream));
      } else {
        fetch_result(c, out, out_is_inf);
      }
    });
  }

  // Sharded MSM, one rank's call (SURVEY 8e): local Pippenger over this rank's point range -> XYZZ partial
  // -> all-gather of one partial per rank -> fold + affine, all enqueued on the library stream back to
  // back; the host only waits for the final 64 / 128 bytes.  Every rank returns the full result.
  static void multi_enqueue_tail(Context& c, int slot) {
    MsmEngine<F>& e = engine(slot);
    cudaStream_t st = slot ? c.stream2 : c.stream;
    CommState& cs = comm_state();
    const size_t PB = sizeof(XYZZ<F>);
    DevBuf& gathered = cs.gathered[slot];
    gathered.reserve((size_t)cs.world * PB);
    comm_all_gather(e.result.template as<char>() + PT, gathered.p, PB, st);
    using FC = typename CompactOf<F>::type;
    combine_partials_kernel<FC><<<1, 32, 0, st>>>(gathered.template as<XYZZ<FC>>(), (uint32_t)cs.world,
                                                 e.result.template as<Affine<FC>>(), e.flag.template as<int>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
  }
  static void multi_tail(Context& c, uint8_t* out_xy, int* out_is_inf) {
    multi_enqueue_tail(c, 0);
    fetch_result(c, out_xy, out_is_inf);
  }

  // The same collective on the second lane without waiting for it: begin enqueues local MSM -> all-gather -> fold
  // on the second stream (behind everything already queued on the first) and returns; end fetches the point.
  // What the caller enqueues on the first stream in between -- the quotient of a Groth16 proof, which the A and
  // B elements do not depend on -- runs beside it.  One pending call per group.
  static int msm_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n, bool multi) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "msm_begin");
      Resource* s = need(scalars, HandleKind::Scalars, "msm_begin");
      if (!range_ok(offset, n, t->n) || !range_ok(sc_offset, n, s->n)) throw InvalidArgument("msm_begin: range out of bounds");
      if (multi && !comm_state().ready) throw InvalidArgument("msm_multi_begin: zkp_comm_init has not been called on this rank");
      CUDA_CHECK(cudaEventRecord(c.ev_fork, c.stream));
      CUDA_CHECK(cudaStreamWaitEvent(c.stream2, c.ev_fork, 0));
      c.launches += run_on_table(c, t, offset, s->buf.as<uint32_t>() + 8 * sc_offset, n, multi, 1);
      if (multi) multi_enqueue_tail(c, 1);
    });
  }
  static int msm_multi_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n) {
    return msm_begin(table, offset, scalars, sc_offset, n, true);
  }
  static int msm_multi_end(uint8_t* out_xy, int* out_is_inf) {
    return guarded([&](Context& c) {
      if (!out_xy) throw InvalidArgument("msm_multi_end: null output");
      MsmEngine<F>& e = engine(1);
      if (!e.result.p) throw InvalidArgument("msm_end: no begin call is pending");
      int flag = 0;
      CUDA_CHECK(cudaMemcpyAsync(out_xy, e.result.p, PT, cudaMemcpyDeviceToHost, c.stream2));
      CUDA_CHECK(cudaMemcpyAsync(&flag, e.flag.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream2));
      CUDA_CHECK(cudaStreamSynchronize(c.stream2));
      if (flag) memset(out_xy, 0, PT);
      if (out_is_inf) *out_is_inf = flag;
    });
  }

  static int msm_multi(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n, uint8_t* out_xy,
                       int* out_is_inf) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "msm_multi");
      Resource* s = need(scalars, HandleKind::Scalars, "msm_multi");
      if (!out_xy) throw InvalidArgument("msm_multi: null output");
      if (!range_ok(offset, n, t->n) || !range_ok(sc_offset, n, s->n)) throw InvalidArgument("msm_multi: range out of bounds");
      if (!comm_state().ready) throw InvalidArgument("msm_multi: zkp_comm_init has not been called on this rank");
      c.launches += run_on_table(c, t, offset, s->buf.as<uint32_t>() + 8 * sc_offset, n, true);
      multi_tail(c, out_xy, out_is_inf);
    });
  }

  // the same with this rank's scalars in host memory (the end-to-end form of the sharded commit)
  static int msm_multi_host(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t* out_xy,
                            int* out_is_inf) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "msm_multi_table");
      if (!out_xy || (n && !scalars)) throw InvalidArgument("msm_multi_table: null argument");
      if (!range_ok(offset, n, t->n)) throw InvalidArgument("msm_multi_table: point range exceeds the table");
      if (!comm_state().ready) throw InvalidArgument("msm_multi_table: zkp_comm_init has not been called on this rank");
      DevBuf& ds = scratch_scalars();
      if (n) ds.reserve(n * 32);
      c.launches += run_on_table(c, t, offset, ds.as<uint32_t>(), n, true, 0, scalars);
      multi_tail(c, out_xy, out_is_inf);
    });
  }

  static int combine(const uint8_t* partials, uint32_t count, uint8_t* out_xy, int* out_is_inf) {
    return guarded([&](Context& c) {
      if (!out_xy || (count && !partials)) throw InvalidArgument("combine_partials: null argument");
      MsmEngine<F>& e = engine();
      e.result.reserve(sizeof(XYZZ<F>) + sizeof(Affine<F>));
      e.flag.reserve(sizeof(int));
      DevBuf& dp = scratch_pts();
      dp.reserve((size_t)(count ? count : 1) * sizeof(XYZZ<F>));
      if (count)
        CUDA_CHECK(cudaMemcpyAsync(dp.p, partials, (size_t)count * sizeof(XYZZ<F>), cudaMemcpyDefault, c.stream));
      using FC = typename CompactOf<F>::type;
      combine_partials_kernel<FC><<<1, 32, 0, c.stream>>>(dp.as<XYZZ<FC>>(), count, e.result.template as<Affine<FC>>(),
                                                        e.flag.template as<int>());
      CUDA_CHECK_LAUNCH();
      c.launches++;
      fetch_result(c, out_xy, out_is_inf);
    });
  }

  static void fixed_base_run(Context& c, const uint8_t* base_xy, const uint32_t* dscalars, uint64_t n,
                             uint64_t* out_table) {
    Affine<F> base;
    memcpy(&base, base_xy, PT);
    auto r = std::make_unique<Resource>();
    r->kind = KIND;
    r->n = n;
    r->buf.reserve_pooled(n ? n * PT : PT);
    if (n >= 4096) {
      PooledDevBuf tsc, tab;
      tsc.reserve_pooled(8192 * 32);
      tab.reserve_pooled(8192 * PT);
      fixed_base_table_scalars_kernel<<<32, 256, 0, c.stream>>>(tsc.as<uint32_t>());
      CUDA_CHECK_LAUNCH();
      fixed_base_mul_kernel<F><<<64, 128, 0, c.stream>>>(base, tsc.as<uint32_t>(), 8192, tab.as<Affine<F>>());
      CUDA_CHECK_LAUNCH();
      fixed_base_windowed_kernel<F><<<ceil_div(n, 128), 128, 0, c.stream>>>(tab.as<Affine<F>>(), dscalars, n,
                                                                           r->buf.as<Affine<F>>());
      CUDA_CHECK_LAUNCH();
      c.launches += 3;
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
    } else if (n) {
      fixed_base_mul_kernel<F><<<ceil_div(n, 128), 128, 0, c.stream>>>(base, dscalars, n, r->buf.as<Affine<F>>());
      CUDA_CHECK_LAUNCH();
      c.launches++;
    }
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *out_table = registry().put(std::move(r));
  }

  static int fixed_base_host(const uint8_t* base_xy, const uint8_t* scalars, uint64_t n, uint64_t* out_table) {
    return guarded([&](Context& c) {
      if (!base_xy || !out_table || (n && !scalars)) throw InvalidArgument("fixed_base_mul: null argument");
      DevBuf& ds = scratch_scalars();
      if (n) {
        ds.reserve(n * 32);
        CUDA_CHECK(cudaMemcpyAsync(ds.p, scalars, n * 32, cudaMemcpyHostToDevice, c.stream));
      }
      fixed_base_run(c, base_xy, ds.as<uint32_t>(), n, out_table);
    });
  }

  static int fixed_base_dev(const uint8_t* base_xy, uint64_t scalars, uint64_t n, uint64_t* out_table) {
    return guarded([&](Context& c) {
      Resource* s = need(scalars, HandleKind::Scalars, "fixed_base_mul_dev");
      if (!base_xy || !out_table) throw InvalidArgument("fixed_base_mul_dev: null argument");
      if (n > s->n) throw InvalidArgument("fixed_base_mul_dev: n exceeds the scalar vector");
      fixed_base_run(c, base_xy, s->buf.as<uint32_t>(), n, out_table);
    });
  }

  // Points [offset, offset + n) of either layout: a precomputed table keeps the points themselves in row 0.
  static const Affine<F>* table_points(Resource* t, uint64_t offset) { return t->buf.as<Affine<F>>() + offset; }

  static int table_scale(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                         uint64_t* out_table) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "table_scale");
      Resource* s = need(scalars, HandleKind::Scalars, "table_scale");
      if (!out_table) throw InvalidArgument("table_scale: null output");
      if (!range_ok(offset, n, t->n) || !range_ok(sc_offset, n, s->n)) throw InvalidArgument("table_scale: range out of bounds");
      auto r = std::make_unique<Resource>();
      r->kind = KIND;
      r->n = n;
      r->buf.reserve_pooled(n ? n * PT : PT);
      if (n) {
        table_scale_kernel<F><<<ceil_div(n, 128), 128, 0, c.stream>>>(table_points(t, offset),
                                                                     s->buf.as<uint32_t>() + 8 * sc_offset, n,
                                                                     r->buf.as<Affine<F>>());
        CUDA_CHECK_LAUNCH();
        c.launches++;
      }
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
      *out_table = registry().put(std::move(r));
    });
  }

  static int table_validate(uint64_t table, uint64_t offset, uint64_t n, int subgroup, uint64_t* first_bad) {
    return guarded([&](Context& c) {
      Resource* t = need(table, KIND, "table_validate");
      if (!first_bad) throw InvalidArgument("table_validate: null output");
      if (!range_ok(offset, n, t->n)) throw InvalidArgument("table_validate: range out of bounds");
      unsigned long long bad = ~0ull;
      if (n) {
        ScopedDevBuf flag;
        flag.reserve(sizeof bad);
        CUDA_CHECK(cudaMemsetAsync(flag.p, 0xff, sizeof bad, c.stream));
        table_validate_kernel<F><<<ceil_div(n, 64), 64, 0, c.stream>>>(table_points(t, offset), n, offset, subgroup != 0,
                                                                       flag.as<unsigned long long>());
        CUDA_CHECK_LAUNCH();
        c.launches++;
        CUDA_CHECK(cudaMemcpyAsync(&bad, flag.p, sizeof bad, cudaMemcpyDeviceToHost, c.stream));
        CUDA_CHECK(cudaStreamSynchronize(c.stream));
      }
      *first_bad = bad;
    });
  }

  // n compressed encodings (PT / 2 bytes each, point_codec.cuh) -> a new plain table, decoded and checked in one
  // launch.  *first_bad = lowest rejected index or UINT64_MAX; on a rejection no handle is made (*handle = 0).
  static int table_load_compressed(const uint8_t* enc, uint64_t n, bool subgroup, uint64_t* handle, uint64_t* first_bad) {
    return guarded([&](Context& c) {
      if (!handle || !first_bad || (n && !enc)) throw InvalidArgument("table_load_compressed: null argument");
      *handle = 0;
      auto r = std::make_unique<Resource>();
      r->kind = KIND;
      r->n = n;
      r->buf.reserve_pooled(n ? n * PT : PT);
      unsigned long long bad = ~0ull;
      if (n) {
        DevBuf& de = scratch_pts();
        de.reserve(n * PT / 2);
        ScopedDevBuf flag;
        flag.reserve(sizeof bad);
        CUDA_CHECK(cudaMemcpyAsync(de.p, enc, n * PT / 2, cudaMemcpyHostToDevice, c.stream));
        CUDA_CHECK(cudaMemsetAsync(flag.p, 0xff, sizeof bad, c.stream));
        constexpr unsigned BLK = std::is_same<F, Fp2>::value ? 64 : 128;
        decompress_kernel<F><<<ceil_div(n, BLK), BLK, 0, c.stream>>>(de.as<uint4>(), n, subgroup, r->buf.as<Affine<F>>(),
                                                                     flag.as<unsigned long long>());
        CUDA_CHECK_LAUNCH();
        c.launches++;
        CUDA_CHECK(cudaMemcpyAsync(&bad, flag.p, sizeof bad, cudaMemcpyDeviceToHost, c.stream));
      }
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
      *first_bad = bad;
      if (bad == ~0ull) *handle = registry().put(std::move(r));
    });
  }

  static void download_compressed(Context& c, Resource* t, uint64_t offset, uint64_t n, uint8_t* out) {
    if (!range_ok(offset, n, t->n)) throw InvalidArgument("table_download_compressed: range out of bounds");
    if (!n) return;
    DevBuf& dp = scratch_pts();
    dp.reserve(n * PT / 2);
    compress_kernel<F><<<ceil_div(n, 128), 128, 0, c.stream>>>(table_points(t, offset), n, dp.as<uint4>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out, dp.p, n * PT / 2, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  }

  static void download(Context& c, Resource* t, uint64_t offset, uint64_t n, uint8_t* out_pts) {
    if (!range_ok(offset, n, t->n)) throw InvalidArgument("table_download: range out of bounds");
    if (!n) return;
    DevBuf& dp = scratch_pts();
    dp.reserve(n * PT);
    CUDA_CHECK(cudaMemcpyAsync(dp.p, t->buf.as<uint8_t>() + offset * PT, n * PT, cudaMemcpyDeviceToDevice, c.stream));
    fe_from_mont_kernel<Fp><<<ceil_div(n * FE_PER_PT, 256), 256, 0, c.stream>>>(dp.as<Fp>(), n * FE_PER_PT);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out_pts, dp.p, n * PT, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  }
};

}  // namespace zkp
