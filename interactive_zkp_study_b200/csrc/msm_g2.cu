// G2 instantiation of the MSM / table entry points (include/zkp_b200.h).
#include "msm_api.cuh"

using namespace zkp;
using Api = GroupApi<Fp2>;

// zkp_table_download (msm_g1.cu) needs the G2 download path
template struct zkp::GroupApi<Fp2>;

namespace zkp {
// G2 MSM enqueued on lane `slot` (1 = the second stream); result (128 B) and infinity flag (4 B) are
// copied to dev_out on that lane.  Used by zkp_groth16_msms_dev (msm_g1.cu) to run the G2 element of a
// Groth16 proof beside the two G1 elements.
int g2_msm_enqueue(Context& c, uint64_t table, uint64_t scalars, uint64_t n, int slot, char* dev_out) {
  Resource* t = need(table, HandleKind::G2Table, "zkp_groth16_msms_dev");
  Resource* s = need(scalars, HandleKind::Scalars, "zkp_groth16_msms_dev");
  if (n > t->n || n > s->n) throw InvalidArgument("zkp_groth16_msms_dev: G2 range out of bounds");
  cudaStream_t st = slot ? c.stream2 : c.stream;
  int launches = Api::run_on_table(c, t, 0, s->buf.as<uint32_t>(), n, false, slot);
  MsmEngine<Fp2>& e = Api::engine(slot);
  CUDA_CHECK(cudaMemcpyAsync(dev_out, e.result.p, 128, cudaMemcpyDeviceToDevice, st));
  CUDA_CHECK(cudaMemcpyAsync(dev_out + 128, e.flag.p, sizeof(int), cudaMemcpyDeviceToDevice, st));
  return launches;
}
}  // namespace zkp

extern "C" {

int zkp_g2_msm(const uint8_t* pts, const uint8_t* scalars, uint64_t n, uint8_t out_xy[128], int* out_is_inf) {
  return Api::msm_host(pts, scalars, n, out_xy, out_is_inf);
}
int zkp_g2_table_load(const uint8_t* pts, uint64_t n, uint64_t* handle) { return Api::table_load(pts, n, handle); }
int zkp_g2_msm_table(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t out_xy[128],
                     int* out_is_inf) {
  return Api::msm_table(table, offset, scalars, n, out_xy, out_is_inf);
}
int zkp_g2_msm_dev(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                   uint8_t out_xy[128], int* out_is_inf) {
  return Api::msm_dev(table, offset, scalars, sc_offset, n, out_xy, out_is_inf, false);
}
int zkp_g2_msm_multi(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                     uint8_t out_xy[128], int* out_is_inf) {
  return Api::msm_multi(table, offset, scalars, sc_offset, n, out_xy, out_is_inf);
}
int zkp_g2_msm_dev_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n) {
  return Api::msm_begin(table, offset, scalars, sc_offset, n, false);
}
int zkp_g2_msm_dev_end(uint8_t out_xy[128], int* out_is_inf) { return Api::msm_multi_end(out_xy, out_is_inf); }
int zkp_g2_msm_multi_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n) {
  return Api::msm_multi_begin(table, offset, scalars, sc_offset, n);
}
int zkp_g2_msm_multi_end(uint8_t out_xy[128], int* out_is_inf) { return Api::msm_multi_end(out_xy, out_is_inf); }
int zkp_g2_fixed_base_mul_dev(const uint8_t base_xy[128], uint64_t scalars, uint64_t n, uint64_t* out_table) {
  return Api::fixed_base_dev(base_xy, scalars, n, out_table);
}
int zkp_g2_table_scale(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                       uint64_t* out_table) {
  return Api::table_scale(table, offset, scalars, sc_offset, n, out_table);
}
int zkp_g2_table_validate(uint64_t table, uint64_t offset, uint64_t n, int subgroup_check, uint64_t* first_bad) {
  return Api::table_validate(table, offset, n, subgroup_check, first_bad);
}
int zkp_g2_table_load_compressed(const uint8_t* enc, uint64_t n, int subgroup_check, uint64_t* handle,
                                 uint64_t* first_bad) {
  return Api::table_load_compressed(enc, n, subgroup_check != 0, handle, first_bad);
}
int zkp_g2_table_precompute(uint64_t table, int window_bits) { return Api::table_precompute(table, window_bits); }
int zkp_g2_msm_dev_many(uint64_t table, uint64_t offset, uint64_t n, uint32_t count, uint64_t scalars, uint64_t sc_offset,
                        uint8_t* out_xy, int* out_is_inf) {
  return Api::msm_dev_many(table, offset, n, count, scalars, sc_offset, out_xy, out_is_inf);
}
int zkp_g2_fixed_base_mul(const uint8_t base_xy[128], const uint8_t* scalars, uint64_t n, uint64_t* out_table) {
  return Api::fixed_base_host(base_xy, scalars, n, out_table);
}

}  // extern "C"
