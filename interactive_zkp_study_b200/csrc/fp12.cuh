// Fp6 = Fp2[v]/(v^3 - xi), xi = 9 + u, and Fp12 = Fp6[w]/(w^2 - v): the target group of the BN254 pairing.
// Device-side replacement for py_ecc's FQ12 as the verifiers reach it through bn128.pairing
// (zkp/groth16/verifying.py:29-40, zkp/plonk/verifier.py:42-208, zkp/plonk/kzg.py:117-160).
//
// Basis.  With w^6 = xi an element is sum_i g_i w^i, g_i in Fp2, where (g_0 .. g_5) = (c0.c0, c1.c0, c0.c1,
// c1.c1, c0.c2, c1.c2).  py_ecc's FQ12 is Fp[w]/(w^12 - 18 w^6 + 82), where w^6 = 9 + u as well, so
// g_i = a_i + b_i u has the py_ecc coefficients coeff[i] = a_i - 9 b_i and coeff[i + 6] = b_i
// (to_pyecc / from_pyecc below; tests/tower_model.py states the same on integers).
//
// Every operation takes its operands by reference and is out of line: an Fp12 value is 96 registers, so the
// kernels keep their values in local memory and share one body per operation (compact code, fast to compile).
// The Fp2 products underneath are the lazily reduced Karatsuba of fp2.cuh.
#pragma once
#include "fp2.cuh"

namespace zkp {

ZKP_DEVINL Fp2 fp2_mul_fp(const Fp2& a, const FpC& s) { return {a.c0 * s, a.c1 * s}; }
ZKP_DEVINL Fp2 fp2_conj(const Fp2& a) { return {a.c0, a.c1.neg()}; }
// (a0 + a1 u)(9 + u) = (9 a0 - a1) + (a0 + 9 a1) u
ZKP_DEVINL Fp2 fp2_mul_xi(const Fp2& a) {
  FpC n0 = a.c0.dbl().dbl().dbl() + a.c0, n1 = a.c1.dbl().dbl().dbl() + a.c1;
  return {n0 - a.c1, a.c0 + n1};
}
ZKP_DEVINL Fp2 fp2_triple(const Fp2& a) { return a.dbl() + a; }
ZKP_DEVINL Fp2 fp2_frob_coeff(int idx) {
  Fp2 r;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    r.c0.v[j] = FP12_FROB[idx][j];
    r.c1.v[j] = FP12_FROB[idx][8 + j];
  }
  return r;
}

struct Fp6 {
  Fp2 c0, c1, c2;
  static ZKP_DEVINL Fp6 zero() { return {Fp2::zero(), Fp2::zero(), Fp2::zero()}; }
  static ZKP_DEVINL Fp6 one() { return {Fp2::one(), Fp2::zero(), Fp2::zero()}; }
  ZKP_DEVINL bool operator==(const Fp6& b) const { return c0 == b.c0 && c1 == b.c1 && c2 == b.c2; }
  friend ZKP_DEVINL Fp6 operator+(const Fp6& a, const Fp6& b) { return {a.c0 + b.c0, a.c1 + b.c1, a.c2 + b.c2}; }
  friend ZKP_DEVINL Fp6 operator-(const Fp6& a, const Fp6& b) { return {a.c0 - b.c0, a.c1 - b.c1, a.c2 - b.c2}; }
  ZKP_DEVINL Fp6 neg() const { return {c0.neg(), c1.neg(), c2.neg()}; }
  ZKP_DEVINL Fp6 mul_v() const { return {fp2_mul_xi(c2), c0, c1}; }   // times v: v^3 = xi
};

// Karatsuba over Fp2 (6 Fp2 products)
__device__ __noinline__ inline Fp6 fp6_mul(const Fp6& a, const Fp6& b) {
  Fp2 t0 = a.c0 * b.c0, t1 = a.c1 * b.c1, t2 = a.c2 * b.c2;
  Fp6 r;
  r.c0 = fp2_mul_xi((a.c1 + a.c2) * (b.c1 + b.c2) - t1 - t2) + t0;
  r.c1 = (a.c0 + a.c1) * (b.c0 + b.c1) - t0 - t1 + fp2_mul_xi(t2);
  r.c2 = (a.c0 + a.c2) * (b.c0 + b.c2) - t0 - t2 + t1;
  return r;
}

// a (b0 + b1 v): the line half with two non-zero coefficients (5 Fp2 products)
__device__ __noinline__ inline Fp6 fp6_mul_01(const Fp6& a, const Fp2& b0, const Fp2& b1) {
  Fp2 t0 = a.c0 * b0, t1 = a.c1 * b1;
  Fp6 r;
  r.c0 = fp2_mul_xi((a.c1 + a.c2) * b1 - t1) + t0;
  r.c1 = (a.c0 + a.c1) * (b0 + b1) - t0 - t1;
  r.c2 = (a.c0 + a.c2) * b0 - t0 + t1;
  return r;
}

// 1 / a through the norm to Fp2 (and Fp2::inv through its norm to Fp, Mont256::inv)
__device__ __noinline__ inline Fp6 fp6_inv(const Fp6& a) {
  Fp2 c0 = a.c0.sqr() - fp2_mul_xi(a.c1 * a.c2);
  Fp2 c1 = fp2_mul_xi(a.c2.sqr()) - a.c0 * a.c1;
  Fp2 c2 = a.c1.sqr() - a.c0 * a.c2;
  Fp2 t = (a.c0 * c0 + fp2_mul_xi(a.c2 * c1 + a.c1 * c2)).inv();
  return {c0 * t, c1 * t, c2 * t};
}

struct Fp12 {
  Fp6 c0, c1;
  static ZKP_DEVINL Fp12 one() { return {Fp6::one(), Fp6::zero()}; }
  ZKP_DEVINL bool operator==(const Fp12& b) const { return c0 == b.c0 && c1 == b.c1; }
  ZKP_DEVINL bool is_one() const { return *this == one(); }
  ZKP_DEVINL Fp12 conj() const { return {c0, c1.neg()}; }   // pi^6: the inverse on the cyclotomic subgroup
  // Fp2 coefficient of w^i (i = 0..5) and back
  ZKP_DEVINL Fp2& g(int i) {
    Fp6& h = (i & 1) ? c1 : c0;
    return i < 2 ? h.c0 : (i < 4 ? h.c1 : h.c2);
  }
};

__device__ __noinline__ inline Fp12 fp12_mul(const Fp12& a, const Fp12& b) {
  Fp6 t0 = fp6_mul(a.c0, b.c0), t1 = fp6_mul(a.c1, b.c1);
  Fp12 r;
  r.c1 = fp6_mul(a.c0 + a.c1, b.c0 + b.c1) - t0 - t1;
  r.c0 = t0 + t1.mul_v();
  return r;
}

// (a0 + a1 w)^2 = (a0 + a1)(a0 + v a1) - m - v m + 2 m w,  m = a0 a1
__device__ __noinline__ inline Fp12 fp12_sqr(const Fp12& a) {
  Fp6 m = fp6_mul(a.c0, a.c1);
  Fp12 r;
  r.c0 = fp6_mul(a.c0 + a.c1, a.c0 + a.c1.mul_v()) - m - m.mul_v();
  r.c1 = m + m;
  return r;
}

// f (l00 + l10 w + l11 w^3): a Miller-loop line (coefficients at w^0, w^1, w^3 = c0.c0, c1.c0, c1.c1)
__device__ __noinline__ inline Fp12 fp12_mul_line(const Fp12& f, const Fp2& l00, const Fp2& l10, const Fp2& l11) {
  Fp6 t0 = {f.c0.c0 * l00, f.c0.c1 * l00, f.c0.c2 * l00};
  Fp6 t1 = fp6_mul_01(f.c1, l10, l11);
  Fp12 r;
  r.c1 = fp6_mul_01(f.c0 + f.c1, l00 + l10, l11) - t0 - t1;
  r.c0 = t0 + t1.mul_v();
  return r;
}

__device__ __noinline__ inline Fp12 fp12_inv(const Fp12& a) {
  Fp6 t = fp6_inv(fp6_mul(a.c0, a.c0) - fp6_mul(a.c1, a.c1).mul_v());
  return {fp6_mul(a.c0, t), fp6_mul(a.c1, t).neg()};
}

// pi^k, k = 1..3: g_i -> g_i^(p^k) xi^(i (p^k - 1) / 6)
__device__ __noinline__ inline Fp12 fp12_frobenius(const Fp12& a, int k) {
  Fp12 r = a;
#pragma unroll 1
  for (int i = 0; i < 6; i++) {
    Fp2 x = r.g(i);
    if (k & 1) x = fp2_conj(x);
    r.g(i) = i == 0 ? x : x * fp2_frob_coeff(6 * (k - 1) + i);
  }
  return r;
}

// Granger-Scott squaring: valid on the cyclotomic subgroup (every value after the easy part of the final
// exponentiation), 9 Fp2 squarings instead of 12 Fp2 products.
__device__ __noinline__ inline Fp12 fp12_cyclotomic_sqr(const Fp12& a) {
  Fp2 z0 = a.c0.c0, z4 = a.c0.c1, z3 = a.c0.c2, z2 = a.c1.c0, z1 = a.c1.c1, z5 = a.c1.c2;
  auto fp4_sqr = [](const Fp2& x, const Fp2& y, Fp2& s0, Fp2& s1) {
    Fp2 t0 = x.sqr(), t1 = y.sqr();
    s0 = fp2_mul_xi(t1) + t0;
    s1 = (x + y).sqr() - t0 - t1;
  };
  Fp2 t0, t1, t2, t3;
  fp4_sqr(z0, z1, t0, t1);
  z0 = (t0 - z0).dbl() + t0;
  z1 = (t1 + z1).dbl() + t1;
  fp4_sqr(z2, z3, t0, t1);
  fp4_sqr(z4, z5, t2, t3);
  z4 = (t0 - z4).dbl() + t0;
  z5 = (t1 + z5).dbl() + t1;
  t0 = fp2_mul_xi(t3);
  z2 = (t0 + z2).dbl() + t0;
  z3 = (t2 - z3).dbl() + t2;
  return {{z0, z4, z3}, {z2, z1, z5}};
}

// a^x, x = 4965661367192848881 (the BN parameter, 63 bits), a in the cyclotomic subgroup
__device__ __noinline__ inline Fp12 fp12_exp_by_x(const Fp12& a) {
  constexpr uint64_t BN_X = 4965661367192848881ull;
  Fp12 r = a;
#pragma unroll 1
  for (int i = 61; i >= 0; i--) {
    r = fp12_cyclotomic_sqr(r);
    if ((BN_X >> i) & 1) r = fp12_mul(r, a);
  }
  return r;
}

// f^((p^12 - 1) / r), the exact exponent of py_ecc's final_exponentiate.
//   easy part: f^((p^6 - 1)(p^2 + 1))
//   hard part: (p^4 - p^2 + 1) / r = l3 p^3 + l2 p^2 + l1 p + l0 with l3 = 1, l2 = 6x^2 + 1,
//   l1 = -36x^3 - 18x^2 - 12x + 1, l0 = -36x^3 - 30x^2 - 18x - 2, by the addition chain of Scott, Benger,
//   Charlemagne, Dominguez Perez, Kachisa (Pairing 2009, section 6): three exponentiations by x, exactly
//   that power (not a multiple of it).
__device__ __noinline__ inline Fp12 fp12_final_exponentiation(const Fp12& f_in) {
  Fp12 f = fp12_mul(f_in.conj(), fp12_inv(f_in));
  f = fp12_mul(fp12_frobenius(f, 2), f);
  Fp12 fx = fp12_exp_by_x(f);
  Fp12 fx2 = fp12_exp_by_x(fx);
  Fp12 fx3 = fp12_exp_by_x(fx2);
  Fp12 y0 = fp12_mul(fp12_mul(fp12_frobenius(f, 1), fp12_frobenius(f, 2)), fp12_frobenius(f, 3));
  Fp12 y1 = f.conj();
  Fp12 y2 = fp12_frobenius(fx2, 2);
  Fp12 y3 = fp12_frobenius(fx, 1).conj();
  Fp12 y4 = fp12_mul(fx, fp12_frobenius(fx2, 1)).conj();
  Fp12 y5 = fx2.conj();
  Fp12 y6 = fp12_mul(fx3, fp12_frobenius(fx3, 1)).conj();
  Fp12 t0 = fp12_mul(fp12_mul(fp12_cyclotomic_sqr(y6), y4), y5);
  Fp12 t1 = fp12_mul(fp12_mul(y3, y5), t0);
  t0 = fp12_mul(t0, y2);
  t1 = fp12_cyclotomic_sqr(fp12_mul(fp12_cyclotomic_sqr(t1), t0));
  t0 = fp12_mul(t1, y1);
  t1 = fp12_mul(t1, y0);
  t0 = fp12_cyclotomic_sqr(t0);
  return fp12_mul(t0, t1);
}

// py_ecc's 12 canonical coefficients (w^0..w^11 mod w^12 - 18 w^6 + 82) <-> tower element in Montgomery form
ZKP_DEVINL Fp12 fp12_from_pyecc(const FpC (&c)[12]) {
  Fp12 r;
#pragma unroll 1
  for (int i = 0; i < 6; i++) {
    FpC a = c[i].to_mont(), b = c[i + 6].to_mont();
    r.g(i) = {a + b.dbl().dbl().dbl() + b, b};
  }
  return r;
}
ZKP_DEVINL void fp12_to_pyecc(Fp12 a, FpC (&c)[12]) {
#pragma unroll 1
  for (int i = 0; i < 6; i++) {
    const Fp2& x = a.g(i);
    c[i] = (x.c0 - (x.c1.dbl().dbl().dbl() + x.c1)).from_mont();
    c[i + 6] = x.c1.from_mont();
  }
}

}  // namespace zkp
