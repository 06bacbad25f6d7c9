// The group-law step of the MSM's bucket-accumulation loop (msm.cuh msm_accumulate_kernel): the mixed addition
// XYZZ += affine with the field products split between inlined and shared out-of-line bodies.  Its own header so
// that the self-test hooks (diag.cu, zkp_dbg_point_add groups 4 / 5) run exactly the body the MSM runs.
#pragma once
#include "ec.cuh"

namespace zkp {

// The mixed addition of the accumulation loop with a chosen subset of its ten field products routed through the
// shared out-of-line bodies (bit i of OUTLINE: product i; 2 and 5 are the squarings).  Ten inlined products are
// 68 KB of loop body, more than the instruction cache keeps near the schedulers (ncu: no_instruction 1.1 stalls per
// issue); a call costs a few register moves.  Same formulas and edge cases as XYZZ::madd (ec.cuh).
template <int OUTLINE>
struct AccMul {
  template <int I>
  static ZKP_DEVINL Fp mul(const Fp& a, const Fp& b) {
    if constexpr ((OUTLINE >> I) & 1) return mont_mul_outlined<FpParams>(a, b);
    else return Fp::mul_inline(a, b);
  }
  template <int I>
  static ZKP_DEVINL Fp sqr(const Fp& a) {
    if constexpr ((OUTLINE >> I) & 1) return mont_sqr_outlined<FpParams>(a);
    else return Fp::sqr_inline(a);
  }
  static ZKP_DEVINL void madd(XYZZ<Fp>& a, const Affine<Fp>& p) {
    if (p.is_inf()) return;
    if (a.is_inf()) {
      a.x = p.x; a.y = p.y; a.zz = Fp::one(); a.zzz = Fp::one();
      return;
    }
    Fp u2 = mul<0>(p.x, a.zz);
    Fp s2 = mul<1>(p.y, a.zzz);
    Fp pp_ = u2 - a.x;
    Fp r = s2 - a.y;
    if (pp_.is_zero()) {
      if (r.is_zero()) a = XYZZ<Fp>::dbl_affine(p);
      else a = XYZZ<Fp>::inf();
      return;
    }
    Fp pp = sqr<2>(pp_);
    Fp ppp = mul<3>(pp_, pp);
    Fp q = mul<4>(a.x, pp);
    Fp x3 = sqr<5>(r) - ppp - q.dbl();
    if constexpr ((OUTLINE >> 10) & 1) a.y = fp_mulsub_outlined(r, q - x3, a.y, ppp);  // one reduction for both products
    else a.y = mul<6>(r, q - x3) - mul<7>(a.y, ppp);
    a.x = x3;
    a.zz = mul<8>(a.zz, pp);
    a.zzz = mul<9>(a.zzz, ppp);
  }
};
static constexpr int MSM_ACC_OUTLINE = 0x71B;  // products 0, 1, 3, 4, 8, 9 out of line; the squarings (2, 5) inlined; bit 10: Y3 = R (Q - X3) - Y1 PPP as one lazily reduced pair
// The G2 flavour of the same loop body: XYZZ::madd with the two squarings through inlined Fp products
// (Fp2::sqr_inline_products); the eight Fp2 products stay calls of the shared lazily reduced body.
struct AccMul2 {
  // XYZZ::dbl_affine with the same squarings (the rare P + P case; kept in the same style so that the whole loop
  // body is compiled under one pipe balance)
  static ZKP_DEVINL XYZZ<Fp2> dbl_affine(const Affine<Fp2>& p) {
    Fp2 u = p.y.dbl();
    Fp2 v = u.sqr_inline_products();
    Fp2 w = fp2_mul_inline(u, v);
    Fp2 s = fp2_mul_inline(p.x, v);
    Fp2 xx = p.x.sqr_inline_products();
    Fp2 m = xx.dbl() + xx;
    XYZZ<Fp2> r;
    r.x = m.sqr_inline_products() - s.dbl();
    r.y = fp2_mul_inline(m, s - r.x) - fp2_mul_inline(w, p.y);
    r.zz = v;
    r.zzz = w;
    return r;
  }
  static ZKP_DEVINL void madd(XYZZ<Fp2>& a, const Affine<Fp2>& p) {
    if (p.is_inf()) return;
    if (a.is_inf()) {
      a.x = p.x; a.y = p.y; a.zz = Fp2::one(); a.zzz = Fp2::one();
      return;
    }
    Fp2 u2 = p.x * a.zz;
    Fp2 s2 = p.y * a.zzz;
    Fp2 pp_ = u2 - a.x;
    Fp2 r = s2 - a.y;
    if (pp_.is_zero()) {
      if (r.is_zero()) a = dbl_affine(p);
      else a = XYZZ<Fp2>::inf();
      return;
    }
    Fp2 pp = pp_.sqr_inline_products();
    Fp2 ppp = pp_ * pp;
    Fp2 q = a.x * pp;
    Fp2 x3 = r.sqr_inline_products() - ppp - q.dbl();
    a.y = r * (q - x3) - a.y * ppp;
    a.x = x3;
    a.zz = a.zz * pp;
    a.zzz = a.zzz * ppp;
  }
};
template <class F, int OUTLINE>
ZKP_DEVINL void acc_madd(XYZZ<F>& a, const Affine<F>& p) {
  if constexpr (sizeof(F) == 32 && OUTLINE != 0) AccMul<OUTLINE>::madd(a, p);
  else if constexpr (sizeof(F) == 64 && OUTLINE != 0) AccMul2::madd(a, p);
  else a.madd(p);
}

}  // namespace zkp
