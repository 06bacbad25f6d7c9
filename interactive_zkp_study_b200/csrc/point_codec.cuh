// Compressed point encodings (include/zkp_b200.h zkp_g1/g2_table_load_compressed, zkp_table_download_compressed):
// a point is its x coordinate plus two flag bits in the top of the last field element, which p < 2^254 leaves free.
//   G1, 32 B:  x little-endian; byte 31 bit 7 = y-sign, bit 6 = infinity.
//   G2, 64 B:  x.c0 | x.c1 little-endian; the flags in byte 63.
//   y-sign:    G1 y > (p - 1) / 2;  G2 (y1 != 0 ? y1 : y0) > (p - 1) / 2  (y = y0 + y1 u, c1 compared first).
//   infinity:  every bit zero except the infinity flag.
// Decoding takes one square root per point (x^3 + b must be a square), so a decoded point lies on its curve by
// construction; G2 points can also be put through the subgroup test of curve_check.cuh in the same pass.
#pragma once
#include <type_traits>
#include "curve_check.cuh"

namespace zkp {

// Exponents derived from p at compile time.  p = 3 mod 4, so (p + 1) / 4 = (p >> 2) + 1, (p - 3) / 4 = p >> 2 and
// (p - 1) / 2 = p >> 1.  Word i of (p >> SHIFT) + ADD, little-endian.
template <int SHIFT, uint32_t ADD>
struct FpExp {
  static __host__ __device__ constexpr uint32_t W(int i) {
    return ((FpParams::MOD_(i) >> SHIFT) | (FpParams::MOD_(i + 1) << (32 - SHIFT))) + (i == 0 ? ADD : 0u);
  }
  static constexpr int TOP = 253 - SHIFT;  // highest set bit (p has 254 bits)
};
static_assert((FpParams::MOD_(0) & 3u) == 3u, "the square roots below need p = 3 mod 4");
static_assert(((FpParams::MOD_(0) >> 2) | (FpParams::MOD_(1) << 30)) != 0xffffffffu, "(p >> 2) + 1 must not carry");
using ExpSqrtFp = FpExp<2, 1>;   // (p + 1) / 4
using ExpP3Over4 = FpExp<2, 0>;  // (p - 3) / 4
using ExpHalf = FpExp<1, 0>;     // (p - 1) / 2

// a^E for a compile-time exponent E (its top bit at E::TOP): plain square-and-multiply from the top, 251-252
// squarings and 108-109 products for the exponents above.  One loop body, not unrolled: a product is large and the
// loop runs once per point.
template <class F, class E>
ZKP_DEVINL F pow_fixed(const F& a) {
  F acc = a;
#pragma unroll 1
  for (int bit = E::TOP - 1; bit >= 0; bit--) {
    acc = acc.sqr();
    if ((E::W(bit >> 5) >> (bit & 31)) & 1u) acc = acc * a;
  }
  return acc;
}

// Square root in Fp (Montgomery form, Fp or FpC): y = a^((p+1)/4); false when y^2 != a (a is not a square).
template <class F>
ZKP_DEVINL bool fp_sqrt(const F& a, F& y) {
  y = pow_fixed<F, ExpSqrtFp>(a);
  return y.sqr() == a;
}

// Square root in Fp2 = Fp[u]/(u^2 + 1), p = 3 mod 4: Algorithm 9 of Adj and Rodriguez-Henriquez, "Square root
// computation over even extension fields" (2012).
//   a1 = a^((p-3)/4), alpha = a1^2 a, x0 = a1 a;  norm(alpha) = conj(alpha) alpha = -1: no root;
//   alpha = -1: y = u x0;  otherwise y = (1 + alpha)^((p-1)/2) x0.
// The root is squared back before it is accepted, as in fp_sqrt.
ZKP_DEVINL bool fp2_sqrt(const Fp2& a, Fp2& y) {
  const Fp2 a1 = pow_fixed<Fp2, ExpP3Over4>(a);
  const Fp2 alpha = a1.sqr() * a;
  const Fp2 x0 = a1 * a;
  const FpC minus_one = FpC::one().neg();
  if (alpha.c0.sqr() + alpha.c1.sqr() == minus_one) return false;
  if (alpha.c1.is_zero() && alpha.c0 == minus_one) {
    y = {x0.c1.neg(), x0.c0};  // u (x0.c0 + x0.c1 u) = -x0.c1 + x0.c0 u
  } else {
    y = pow_fixed<Fp2, ExpHalf>(alpha + Fp2::one()) * x0;
  }
  return y.sqr() == a;
}

ZKP_DEVINL bool field_sqrt(const Fp& a, Fp& y) { return fp_sqrt(a, y); }
ZKP_DEVINL bool field_sqrt(const Fp2& a, Fp2& y) { return fp2_sqrt(a, y); }

// canonical v (8 little-endian limbs, v < p) > (p - 1) / 2
ZKP_DEVINL bool fp_gt_half(const uint32_t (&v)[8]) {
  uint32_t borrow = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    uint64_t d = (uint64_t)ExpHalf::W(k) - v[k] - borrow;
    borrow = (uint32_t)(d >> 63);
  }
  return borrow != 0;
}
ZKP_DEVINL bool words_below_p(const uint32_t* v) {
  uint32_t borrow = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    uint64_t d = (uint64_t)v[k] - FpParams::MOD_(k) - borrow;
    borrow = (uint32_t)(d >> 63);
  }
  return borrow != 0;
}

// The y-sign flag of a Montgomery-form coordinate
ZKP_DEVINL bool y_sign(const Fp& y) { return fp_gt_half(y.from_mont().v); }
ZKP_DEVINL bool y_sign(const Fp2& y) {
  const FpC y1 = y.c1.from_mont();
  return y1.is_zero() ? fp_gt_half(y.c0.from_mont().v) : fp_gt_half(y1.v);
}

ZKP_DEVINL Fp curve_b(const Fp&) {
  Fp b;
#pragma unroll
  for (int k = 0; k < 8; k++) b.v[k] = FpParams::B3_(k);
  return b;
}
ZKP_DEVINL Fp2 curve_b(const Fp2&) { return twist_b(); }

// One thread per point: encoding i -> out[i], Montgomery affine as in every table ((0,0) for infinity).  A rejected
// encoding (flags, x >= p, no square root, or with `subgroup` a G2 point outside the order-r subgroup) lowers
// *first_bad to i; its row of `out` is left unwritten.
template <class F>
__global__ void __launch_bounds__(std::is_same<F, Fp2>::value ? 64 : 128)
    decompress_kernel(const uint4* __restrict__ enc, uint64_t n, bool subgroup, Affine<F>* __restrict__ out,
                      unsigned long long* __restrict__ first_bad) {
  constexpr int NW = sizeof(F) / 4;  // 32-bit words of one encoding: 8 (G1) / 16 (G2)
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t w[NW];
#pragma unroll
  for (int q = 0; q < NW / 4; q++) {
    const uint4 v = enc[i * (NW / 4) + q];
    w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
  }
  const bool sign = w[NW - 1] >> 31, infinity = (w[NW - 1] >> 30) & 1u;
  w[NW - 1] &= 0x3fffffffu;
  Affine<F> p = Affine<F>::inf();
  bool ok;
  if (infinity) {
    uint32_t o = sign;
#pragma unroll
    for (int k = 0; k < NW; k++) o |= w[k];
    ok = o == 0;
  } else {
    ok = words_below_p(w);
    if constexpr (NW == 16) ok = ok && words_below_p(w + 8);
    if (ok) {
      F x;
      uint32_t* xw = reinterpret_cast<uint32_t*>(&x);
#pragma unroll
      for (int k = 0; k < NW; k++) xw[k] = w[k];
      x = x.to_mont();
      F y;
      ok = field_sqrt(x.sqr() * x + curve_b(x), y);
      if (ok) {
        if (y_sign(y) != sign) y = y.neg();
        p = {x, y};
        if constexpr (NW == 16) {
          if (subgroup) ok = g2_in_subgroup(p);
        }
      }
    }
  }
  if (!ok) {
    atomicMin(first_bad, (unsigned long long)i);
    return;
  }
  out[i] = p;
}

// One thread per point of a table (plain, or row 0 of a precomputed one): canonical x plus the flags.
template <class F>
__global__ void __launch_bounds__(128) compress_kernel(const Affine<F>* __restrict__ pts, uint64_t n,
                                                       uint4* __restrict__ enc) {
  constexpr int NW = sizeof(F) / 4;  // 32-bit words of one encoding: 8 (G1) / 16 (G2)
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Affine<F> p = pts[i];
  uint32_t w[NW];
  if (p.is_inf()) {
#pragma unroll
    for (int k = 0; k < NW; k++) w[k] = 0;
    w[NW - 1] = 1u << 30;
  } else {
    const F x = p.x.from_mont();
    const uint32_t* xw = reinterpret_cast<const uint32_t*>(&x);
#pragma unroll
    for (int k = 0; k < NW; k++) w[k] = xw[k];
    if (y_sign(p.y)) w[NW - 1] |= 1u << 31;
  }
#pragma unroll
  for (int q = 0; q < NW / 4; q++) enc[i * (NW / 4) + q] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
}

}  // namespace zkp
