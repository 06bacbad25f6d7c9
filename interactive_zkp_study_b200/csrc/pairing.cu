// The BN254 optimal-Ate pairing on the device (include/zkp_b200.h zkp_pairing / zkp_pairing_check).
// Replaces py_ecc's bn128.pairing as the verifiers call it: zkp/groth16/verifying.py:29-40 (four pairings),
// zkp/plonk/verifier.py:42-208 (two), zkp/plonk/kzg.py:117-160 (two).
//
// One thread per (Q in G2, P in G1) pair runs the whole Miller loop (optionally after k P on the same thread),
// a tree of Fp12 products folds the values, and one thread applies the final exponentiation.
//   - Miller loop over 6x + 2 (65 bits, the top bit implicit in T = Q), in py_ecc's binary walk, then the two
//     Frobenius steps T + pi(Q) and T - pi^2(Q).  Homogeneous projective steps on the D-type twist
//     y^2 = x^3 + 3/xi (Costello-Lange-Naehrig 2010; Aranha et al. 2010), each giving the line through the
//     step's points evaluated at P as l00 + l10 w + l11 w^3 scaled by an element of Fp2: that factor and the
//     dropped denominators die in the final exponentiation, whose exponent is a multiple of p^6 - 1, so
//     the result equals py_ecc's FQ12 bit for bit.
//   - Final exponentiation with the exact exponent (p^12 - 1)/r (fp12.cuh).
// tests/tower_model.py states every formula on integers; the CPU suite checks it against py_ecc.
#include <cstring>
#include "../../include/zkp_b200_diag.h"
#include "curve_check.cuh"
#include "fp12.cuh"
#include "registry.cuh"

namespace zkp {

constexpr uint64_t ATE_LOW = 11347224129447541672ull;  // 6x + 2 - 2^64: the 64 bits below the implicit top bit
constexpr uint64_t NONE = ~0ull;

// first_bad[0] / [1]: lowest index of a G1 / G2 input that fails load_g1 / load_g2
__global__ void pairing_validate_kernel(const G2A* q, const G1A* p, uint64_t n, unsigned long long* first_bad) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G1A a;
  G2A b;
  if (!load_g1(p[i], a)) atomicMin(first_bad + 0, (unsigned long long)i);
  if (!load_g2(q[i], b)) atomicMin(first_bad + 1, (unsigned long long)i);
}

// [r] Q == infinity, one thread per point: the twist has order r (2p - r), so an on-curve point can miss G2.
// first_bad[2]: lowest index outside G2.  Inputs are validated first (pairing_validate_kernel).
__global__ void g2_subgroup_kernel(const G2A* q, uint64_t n, unsigned long long* first_bad) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G2A a;
  if (!load_g2(q[i], a) || a.is_inf()) return;
  if (!g2_in_subgroup(a)) atomicMin(first_bad + 2, (unsigned long long)i);
}

struct G2Proj {
  Fp2 x, y, z;
};

// T <- 2T; line l00 + l10 w + l11 w^3 = -2YZ yP + 3X^2 xP w + (3b'Z^2 - Y^2) w^3.  The new point is scaled by 4
// (X3 = 2XY(B - F), Y3 = (B + F)^2 - 12E^2, Z3 = 4BH) so no halving is needed.
__device__ __noinline__ void miller_dbl_step(G2Proj& t, const FpC& xp3, const FpC& nyp, Fp2& l00, Fp2& l10, Fp2& l11) {
  Fp2 a = t.x * t.y, b = t.y.sqr(), c = t.z.sqr();
  Fp2 e = fp2_triple(twist_b() * c);   // 3 b' Z^2
  Fp2 f = fp2_triple(e);
  Fp2 h = (t.y + t.z).sqr() - (b + c);  // 2 Y Z
  Fp2 j = t.x.sqr();
  l00 = fp2_mul_fp(h, nyp);
  l10 = fp2_mul_fp(j, xp3);
  l11 = e - b;
  Fp2 bf = b + f, e2 = e.sqr().dbl().dbl();
  t.x = (a * (b - f)).dbl();
  t.y = bf.sqr() - fp2_triple(e2);
  t.z = (b * h).dbl().dbl();
}

// T <- T + Q (Q affine); line -lambda yP + theta xP w + (lambda yQ - theta xQ) w^3 with theta = Y - yQ Z,
// lambda = X - xQ Z
__device__ __noinline__ void miller_add_step(G2Proj& t, const G2A& q, const FpC& xp, const FpC& nyp, Fp2& l00, Fp2& l10,
                                             Fp2& l11) {
  Fp2 theta = t.y - q.y * t.z, lam = t.x - q.x * t.z;
  Fp2 c = theta.sqr(), d = lam.sqr();
  Fp2 e = lam * d, f = t.z * c, g = t.x * d;
  Fp2 h = e + f - g.dbl();
  l00 = fp2_mul_fp(lam, nyp);
  l10 = fp2_mul_fp(theta, xp);
  l11 = lam * q.y - theta * q.x;
  t.x = lam * h;
  t.y = theta * (g - h) - t.y * e;
  t.z = t.z * e;
}

// Miller value of (Q, P), both affine in Montgomery form and not at infinity
__device__ __noinline__ Fp12 miller_loop(const G2A& q, const G1A& p) {
  const FpC xp = p.x, nyp = p.y.neg(), xp3 = p.x.dbl() + p.x;
  G2Proj t = {q.x, q.y, Fp2::one()};
  Fp12 f = Fp12::one();
  Fp2 l00, l10, l11;
#pragma unroll 1
  for (int i = 63; i >= 0; i--) {
    miller_dbl_step(t, xp3, nyp, l00, l10, l11);
    f = fp12_mul_line(fp12_sqr(f), l00, l10, l11);
    if ((ATE_LOW >> i) & 1) {
      miller_add_step(t, q, xp, nyp, l00, l10, l11);
      f = fp12_mul_line(f, l00, l10, l11);
    }
  }
  // pi(Q) = (conj(x) g_{1,2}, conj(y) g_{1,3});  -pi^2(Q) = (x g_{2,2}, -y g_{2,3})
  G2A q1 = {fp2_conj(q.x) * fp2_frob_coeff(2), fp2_conj(q.y) * fp2_frob_coeff(3)};
  G2A nq2 = {q.x * fp2_frob_coeff(8), (q.y * fp2_frob_coeff(9)).neg()};
  miller_add_step(t, q1, xp, nyp, l00, l10, l11);
  f = fp12_mul_line(f, l00, l10, l11);
  miller_add_step(t, nq2, xp, nyp, l00, l10, l11);
  return fp12_mul_line(f, l00, l10, l11);
}

// out[i] = Miller value of (q[i], k_i p[i]) (Montgomery form); k_i = scalars[i] mod r, or 1 without scalars.
// A pair with infinity on either side (also k_i p[i] = infinity) contributes 1.  Inputs are validated first.
__global__ void __launch_bounds__(64) miller_loop_kernel(const G2A* q, const G1A* p, const uint32_t* scalars, uint64_t n,
                                                          Fp12* out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G1A a;
  G2A b;
  load_g1(p[i], a);
  load_g2(q[i], b);
  if (scalars && !a.is_inf()) {
    uint32_t k[8];
#pragma unroll
    for (int j = 0; j < 8; j++) k[j] = scalars[8 * i + j];
#pragma unroll 1
    for (int rep = 0; rep < 6; rep++) {  // 2^256 < 6 r: at most five subtractions
      uint32_t s[8], borrow = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) {
        uint64_t d = (uint64_t)k[j] - FrParams::MOD_(j) - borrow;
        s[j] = (uint32_t)d;
        borrow = (uint32_t)(d >> 63);
      }
      if (borrow) break;
#pragma unroll
      for (int j = 0; j < 8; j++) k[j] = s[j];
    }
    XYZZ<FpC> acc = XYZZ<FpC>::inf();
#pragma unroll 1
    for (int bit = 253; bit >= 0; bit--) {
      acc = acc.dbl();
      if ((k[bit >> 5] >> (bit & 31)) & 1) acc.madd(a);
    }
    a = acc.to_affine();
  }
  out[i] = (a.is_inf() || b.is_inf()) ? Fp12::one() : miller_loop(b, a);
}

// out[t] = product of in[t chunk .. min(n, (t + 1) chunk))
__global__ void __launch_bounds__(64) fp12_product_kernel(const Fp12* in, uint64_t n, uint32_t chunk, Fp12* out) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t lo = t * chunk;
  if (lo >= n) return;
  uint64_t hi = lo + chunk < n ? lo + chunk : n;
  Fp12 acc = in[lo];
#pragma unroll 1
  for (uint64_t j = lo + 1; j < hi; j++) acc = fp12_mul(acc, in[j]);
  out[t] = acc;
}

// final exponentiation of in[0]: *ok = [result == 1] and / or the result in py_ecc's basis (12 canonical values)
__global__ void final_exp_kernel(const Fp12* in, int* ok, FpC* out_pyecc) {
  if (blockIdx.x || threadIdx.x) return;
  Fp12 r = fp12_final_exponentiation(in[0]);
  if (ok) *ok = r.is_one() ? 1 : 0;
  if (out_pyecc) {
    FpC c[12];
    fp12_to_pyecc(r, c);
#pragma unroll 1
    for (int j = 0; j < 12; j++) out_pyecc[j] = c[j];
  }
}

// self-test hook (zkp_dbg_fp12_op): elements in py_ecc's basis
__global__ void dbg_fp12_op_kernel(int op, const FpC* a, const FpC* b, uint64_t n, FpC* out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  FpC ca[12], cb[12];
#pragma unroll 1
  for (int j = 0; j < 12; j++) {
    ca[j] = a[12 * i + j];
    cb[j] = b ? b[12 * i + j] : FpC::zero();
  }
  Fp12 x = fp12_from_pyecc(ca), y = fp12_from_pyecc(cb), r;
  switch (op) {
    case 0: r = fp12_mul(x, y); break;
    case 1: r = fp12_sqr(x); break;
    case 2: r = fp12_cyclotomic_sqr(x); break;
    case 3: r = fp12_inv(x); break;
    case 4: case 5: case 6: r = fp12_frobenius(x, op - 3); break;
    default: r = fp12_final_exponentiation(x); break;
  }
  fp12_to_pyecc(r, ca);
#pragma unroll 1
  for (int j = 0; j < 12; j++) out[12 * i + j] = ca[j];
}

// Uploads n pairs (and scalars), validates them and leaves the product of their Miller values in f[0].
// Throws InvalidArgument for an input that is not on its curve; with `subgroup` returns false (and computes
// nothing) when a G2 input lies outside G2.
static bool pairing_product(Context& c, const char* what, const uint8_t* g2s, const uint8_t* g1s, const uint8_t* scalars,
                            uint64_t n, bool subgroup, ScopedDevBuf& f) {
  ScopedDevBuf dq, dp, ds, dflags, tmp;
  dq.reserve(n * 128);
  dp.reserve(n * 64);
  dflags.reserve(3 * sizeof(unsigned long long));
  CUDA_CHECK(cudaMemcpyAsync(dq.p, g2s, n * 128, cudaMemcpyHostToDevice, c.stream));
  CUDA_CHECK(cudaMemcpyAsync(dp.p, g1s, n * 64, cudaMemcpyHostToDevice, c.stream));
  if (scalars) {
    ds.reserve(n * 32);
    CUDA_CHECK(cudaMemcpyAsync(ds.p, scalars, n * 32, cudaMemcpyHostToDevice, c.stream));
  }
  CUDA_CHECK(cudaMemsetAsync(dflags.p, 0xff, 3 * sizeof(unsigned long long), c.stream));
  pairing_validate_kernel<<<ceil_div(n, 128), 128, 0, c.stream>>>(dq.as<G2A>(), dp.as<G1A>(), n,
                                                                  dflags.as<unsigned long long>());
  CUDA_CHECK_LAUNCH();
  c.launches++;
  if (subgroup) {
    g2_subgroup_kernel<<<ceil_div(n, 64), 64, 0, c.stream>>>(dq.as<G2A>(), n, dflags.as<unsigned long long>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
  }
  unsigned long long flags[3];
  CUDA_CHECK(cudaMemcpyAsync(flags, dflags.p, sizeof flags, cudaMemcpyDeviceToHost, c.stream));
  CUDA_CHECK(cudaStreamSynchronize(c.stream));
  for (int g = 0; g < 2; g++)
    if (flags[g] != NONE)
      throw InvalidArgument(std::string(what) + ": " + (g ? "G2" : "G1") + " point " + std::to_string(flags[g]) +
                            " is not on its curve (or has a coordinate not below p)");
  if (subgroup && flags[2] != NONE) return false;
  constexpr uint32_t CHUNK = 8;
  f.reserve(n * sizeof(Fp12));
  tmp.reserve(((n + CHUNK - 1) / CHUNK) * sizeof(Fp12));
  miller_loop_kernel<<<ceil_div(n, 64), 64, 0, c.stream>>>(dq.as<G2A>(), dp.as<G1A>(), scalars ? ds.as<uint32_t>() : nullptr,
                                                           n, f.as<Fp12>());
  CUDA_CHECK_LAUNCH();
  c.launches++;
  // fold: f -> tmp -> f ... until one value is left, which ends up in f[0]
  Fp12 *src = f.as<Fp12>(), *dst = tmp.as<Fp12>();
  for (uint64_t m = n; m > 1; m = (m + CHUNK - 1) / CHUNK) {
    uint64_t outs = (m + CHUNK - 1) / CHUNK;
    fp12_product_kernel<<<ceil_div(outs, 64), 64, 0, c.stream>>>(src, m, CHUNK, dst);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    Fp12* t = src;
    src = dst;
    dst = t;
  }
  if (src != f.as<Fp12>()) CUDA_CHECK(cudaMemcpyAsync(f.p, src, sizeof(Fp12), cudaMemcpyDeviceToDevice, c.stream));
  CUDA_CHECK(cudaStreamSynchronize(c.stream));  // tmp is released at scope end
  return true;
}

}  // namespace zkp

using namespace zkp;

extern "C" {

int zkp_pairing(const uint8_t g2_xy[128], const uint8_t g1_xy[64], uint8_t out_fq12[384]) {
  return guarded([&](Context& c) {
    if (!g2_xy || !g1_xy || !out_fq12) throw InvalidArgument("zkp_pairing: null argument");
    ScopedDevBuf f, dout;
    pairing_product(c, "zkp_pairing", g2_xy, g1_xy, nullptr, 1, false, f);
    dout.reserve(384);
    final_exp_kernel<<<1, 1, 0, c.stream>>>(f.as<Fp12>(), nullptr, dout.as<FpC>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out_fq12, dout.p, 384, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_pairing_check(const uint8_t* g2s, const uint8_t* g1s, const uint8_t* scalars, uint64_t count,
                      int g2_subgroup_check, int* out_ok) {
  return guarded([&](Context& c) {
    if (!out_ok || (count && (!g2s || !g1s))) throw InvalidArgument("zkp_pairing_check: null argument");
    *out_ok = 1;
    if (count == 0) return;
    ScopedDevBuf f, dok;
    if (!pairing_product(c, "zkp_pairing_check", g2s, g1s, scalars, count, g2_subgroup_check != 0, f)) {
      *out_ok = 0;
      return;
    }
    dok.reserve(sizeof(int));
    final_exp_kernel<<<1, 1, 0, c.stream>>>(f.as<Fp12>(), dok.as<int>(), nullptr);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out_ok, dok.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_dbg_fp12_op(int op, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out) {
  return guarded([&](Context& c) {
    if (!a || !out || op < 0 || op > 7 || (op == 0 && !b)) throw InvalidArgument("zkp_dbg_fp12_op: bad argument");
    if (n == 0) return;
    ScopedDevBuf da, db, dout;
    da.reserve(n * 384);
    dout.reserve(n * 384);
    CUDA_CHECK(cudaMemcpyAsync(da.p, a, n * 384, cudaMemcpyHostToDevice, c.stream));
    if (b) {
      db.reserve(n * 384);
      CUDA_CHECK(cudaMemcpyAsync(db.p, b, n * 384, cudaMemcpyHostToDevice, c.stream));
    }
    dbg_fp12_op_kernel<<<ceil_div(n, 64), 64, 0, c.stream>>>(op, da.as<FpC>(), b ? db.as<FpC>() : nullptr, n,
                                                            dout.as<FpC>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out, dout.p, n * 384, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

}  // extern "C"
