// Curve-membership tests shared by the pairing (pairing.cu: its inputs) and the table validator (msm_api.cuh:
// zkp_g1/g2_table_validate).  G1: y^2 = x^3 + 3 over Fp, cofactor 1, so on-curve is membership.  G2: the D-type
// twist y^2 = x^3 + 3/(9+u) over Fp2, whose order is r (2p - r): an on-curve point can lie outside G2, which
// [r] Q == infinity decides.
#pragma once
#include "ec.cuh"

namespace zkp {

using G1A = Affine<FpC>;  // same layout as G1Affine: x || y, 8 limbs each
using G2A = Affine<Fp2>;

ZKP_DEVINL bool fp_canonical(const FpC& a) {
  uint32_t borrow = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    uint64_t d = (uint64_t)a.v[k] - FpParams::MOD_(k) - borrow;
    borrow = (uint32_t)(d >> 63);
  }
  return borrow != 0;
}

ZKP_DEVINL Fp2 twist_b() {
  Fp2 b;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    b.c0.v[k] = FpParams::B2_C0_(k);
    b.c1.v[k] = FpParams::B2_C1_(k);
  }
  return b;
}

// y^2 == x^3 + b on Montgomery coordinates (the point must not be the (0,0) encoding of infinity)
ZKP_DEVINL bool on_curve_mont(const G1A& a) {
  FpC b;
#pragma unroll
  for (int k = 0; k < 8; k++) b.v[k] = FpParams::B3_(k);
  return a.y.sqr() == a.x.sqr() * a.x + b;
}
ZKP_DEVINL bool on_curve_mont(const G2A& a) { return a.y.sqr() == a.x.sqr() * a.x + twist_b(); }

// canonical input -> Montgomery form; false when a coordinate is not below p or the point is not on its curve
// (infinity, all zeros, is valid)
ZKP_DEVINL bool load_g1(const G1A& in, G1A& out) {
  out = in;
  if (in.is_inf()) return true;
  if (!fp_canonical(in.x) || !fp_canonical(in.y)) return false;
  out = {in.x.to_mont(), in.y.to_mont()};
  return on_curve_mont(out);
}
ZKP_DEVINL bool load_g2(const G2A& in, G2A& out) {
  out = in;
  if (in.is_inf()) return true;
  if (!fp_canonical(in.x.c0) || !fp_canonical(in.x.c1) || !fp_canonical(in.y.c0) || !fp_canonical(in.y.c1)) return false;
  out = {in.x.to_mont(), in.y.to_mont()};
  return on_curve_mont(out);
}

// [r] a == infinity for an on-curve twist point a (Montgomery form, not infinity)
ZKP_DEVINL bool g2_in_subgroup(const G2A& a) {
  XYZZ<Fp2> acc = XYZZ<Fp2>::from_affine(a);
#pragma unroll 1
  for (int bit = 252; bit >= 0; bit--) {  // r < 2^254, bit 253 is set: acc starts there
    acc = acc.dbl();
    if ((FrParams::MOD_(bit >> 5) >> (bit & 31)) & 1) acc.madd(a);
  }
  return acc.is_inf();
}

}  // namespace zkp
