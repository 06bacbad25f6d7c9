// Internal interface of the Fr NTT engine (ntt.cu), shared with the polynomial layer (poly.cu).
#pragma once
#include "common.cuh"
#include "ff.cuh"

namespace zkp {

// Canonical little-endian Fr element on the host.
struct FrBytes {
  uint8_t b[32];
  bool operator==(const FrBytes& o) const { return memcmp(b, o.b, 32) == 0; }
};

// In-place transform of a device vector of n = 2^log_n elements, natural order in and out.
// The data may be in canonical or Montgomery form (the transform is linear and the twiddles are
// Montgomery constants, so the form is preserved).
//   forward:  out[k] = sum_j in[j] * omega^(jk), optionally pre-scaled in[j] *= shift^j
//   inverse:  same with omega^-1, scaled by n^-1, optionally post-scaled out[j] *= shift^-j
// `scratch` must hold as many elements as `data`.  Returns the number of kernels launched.
// log_batch: transform 2^log_batch contiguous vectors of n elements each in the same launches.
int ntt_device(Context& c, Fr* data, Fr* scratch, uint32_t log_n, const FrBytes& omega, bool inverse,
               const FrBytes* coset_shift, uint32_t log_batch = 0);
// The same for any number `count` of contiguous transforms (count * 2^log_n < 2^32).
int ntt_device_count(Context& c, Fr* data, Fr* scratch, uint32_t log_n, const FrBytes& omega, bool inverse,
                     const FrBytes* coset_shift, uint64_t count);

// x^(2^k), k < 32, in Montgomery form on the device (cached per x); `inverted`: of x^-1 instead.
const Fr* pow2_table(Context& c, const FrBytes& x, bool inverted, int* launches);

// Two-level power table of x (or x^-1) covering exponents below 2^log_n: 1024 low powers x^j followed by
// the high powers x^(1024 k); x^e = lo[e & 1023] * hi[e >> 10], two products instead of a
// square-and-multiply walk over the bits of e.  Montgomery form, cached per (x, inverted, log_n).
const Fr* power_table(Context& c, const FrBytes& x, bool inverted, uint32_t log_n, int* launches);
__device__ __forceinline__ Fr power_at(const Fr* __restrict__ tab, uint32_t e) {
  Fr lo = tab[e & 1023u];
  uint32_t h = e >> 10;
  return h ? lo * tab[1024 + h] : lo;
}


}  // namespace zkp
