// libzkp_b200 diagnostics: integer-pipe and latency microbenchmarks (bench.py's roofline denominator) and
// the field / group-law self-test hooks the parity tests call.  Declared in include/zkp_b200_diag.h --
// not part of the product ABI (include/zkp_b200.h); nothing on a prover path calls into this file.
#include <cstdlib>
#include <cstring>
#include "../../include/zkp_b200_diag.h"
#include "ec.cuh"
#include "ec_quad.cuh"
#include "point_codec.cuh"
#include "registry.cuh"

namespace zkp {

static cudaEvent_t d_ev0 = nullptr, d_ev1 = nullptr;
static void diag_events() {
  if (!d_ev0) {
    CUDA_CHECK(cudaEventCreate(&d_ev0));
    CUDA_CHECK(cudaEventCreate(&d_ev1));
  }
}

// ------------------------------------------------------------------ integer-MAD microbenchmark
// Independent accumulator chains per thread, 256 threads x 4-8 blocks per SM: the issue rate of the
// integer-multiply pipe is the only limit (asm volatile keeps every instruction; see the variants below).
static constexpr int PEAK_UNROLL = 16;

// One thread, dependent chains: the latency a lone thread pays per operation (what bounds the MSM's
// reduction tail).  mode 0/1/2: 1/2/4 independent Fp product chains per iteration (time per iteration);
// 3: XYZZ add, inlined products; 4: XYZZ add, out-of-line products; 5: XYZZ mixed add; 6: XYZZ double.
template <class F>
__device__ __noinline__ uint32_t quad_probe(int mode, int iters) {
  const int ql = threadIdx.x & 3;
  XYZZ<F> acc, q;
  for (int k = 0; k < 8; k++) {
    uint32_t m = k == 7 ? 0x0fffffffu : 0xffffffffu;
    acc.x.v[k] = (0x9e3779b9u * (k + 1)) & m; acc.y.v[k] = (0x9e3779b9u * (k + 9)) & m;
    acc.zz.v[k] = (0x9e3779b9u * (k + 17)) & m; acc.zzz.v[k] = (0x9e3779b9u * (k + 25)) & m;
    q.x.v[k] = (0x85ebca6bu * (k + 3)) & m; q.y.v[k] = (0x85ebca6bu * (k + 11)) & m;
    q.zz.v[k] = (0x85ebca6bu * (k + 19)) & m; q.zzz.v[k] = (0x85ebca6bu * (k + 27)) & m;
  }
  for (int it = 0; it < iters; it++) {
    if (mode == 0) acc = Quad<F>::add(acc, q, ql);
    else acc = Quad<F>::dbl(acc, ql);
  }
  return acc.x.v[0] ^ acc.zzz.v[0];
}

// Where the time of a quad addition goes (modes 12-15, one warp): 12 = the addition without its edge-case tail,
// 13 = only its four dependent select / product / broadcast levels, 14 = four dependent products on a lone
// thread, 15 = four dependent products each followed by one broadcast.
template <class F>
__device__ __noinline__ uint32_t quad_bisect(int mode, int iters) {
  using Q = Quad<F>;
  const int ql = threadIdx.x & 3;
  XYZZ<F> a, b;
  for (int k = 0; k < 8; k++) {
    uint32_t m = k == 7 ? 0x0fffffffu : 0xffffffffu;
    a.x.v[k] = (0x9e3779b9u * (k + 1)) & m; a.y.v[k] = (0x9e3779b9u * (k + 9)) & m;
    a.zz.v[k] = (0x9e3779b9u * (k + 17)) & m; a.zzz.v[k] = (0x9e3779b9u * (k + 25)) & m;
    b.x.v[k] = (0x85ebca6bu * (k + 3)) & m; b.y.v[k] = (0x85ebca6bu * (k + 11)) & m;
    b.zz.v[k] = (0x85ebca6bu * (k + 19)) & m; b.zzz.v[k] = (0x85ebca6bu * (k + 27)) & m;
  }
  for (int it = 0; it < iters; it++) {
    if (mode == 12) {
      F m1 = Q::sel(ql, a.x, b.x, a.y, b.y) * Q::sel(ql, b.zz, a.zz, b.zzz, a.zzz);
      F u1 = Q::from(m1, 0), u2 = Q::from(m1, 1), s1 = Q::from(m1, 2), s2 = Q::from(m1, 3);
      F p = u2 - u1, rr = s2 - s1;
      F m2 = Q::sel(ql, p, a.zz, rr, a.zzz) * Q::sel(ql, p, b.zz, rr, b.zzz);
      F pp = Q::from(m2, 0), r2 = Q::from(m2, 2);
      F m3 = Q::sel(ql, p, m2, u1, p) * pp;
      F ppp = Q::from(m3, 0), q = Q::from(m3, 2);
      XYZZ<F> r;
      r.x = r2 - ppp - q.dbl();
      r.zz = Q::from(m3, 1);
      F m4 = Q::sel(ql, s1, s1, rr, m2) * Q::sel(ql, ppp, ppp, q - r.x, ppp);
      r.y = Q::from(m4, 2) - Q::from(m4, 0);
      r.zzz = Q::from(m4, 3);
      a = r;
    } else if (mode == 13) {
      F m1 = Q::sel(ql, a.x, b.x, a.y, b.y) * Q::sel(ql, b.zz, a.zz, b.zzz, a.zzz);
      F u1 = Q::from(m1, 0), u2 = Q::from(m1, 1), s1 = Q::from(m1, 2), s2 = Q::from(m1, 3);
      F m2 = Q::sel(ql, u1, a.zz, s1, a.zzz) * Q::sel(ql, u2, b.zz, s2, b.zzz);
      F pp = Q::from(m2, 0), r2 = Q::from(m2, 2);
      F m3 = Q::sel(ql, u1, m2, r2, s2) * pp;
      F ppp = Q::from(m3, 0), q = Q::from(m3, 2);
      a.zz = Q::from(m3, 1);
      F m4 = Q::sel(ql, s1, s1, r2, m2) * Q::sel(ql, ppp, ppp, q, ppp);
      a.x = Q::from(m4, 2);
      a.y = Q::from(m4, 0);
      a.zzz = Q::from(m4, 3);
    } else if (mode == 14) {
      a.x = a.x * b.x;
      a.x = a.x * b.y;
      a.x = a.x * b.zz;
      a.x = a.x * b.zzz;
    } else {
      a.x = Q::from(a.x * b.x, 0);
      a.x = Q::from(a.x * b.y, 1);
      a.x = Q::from(a.x * b.zz, 2);
      a.x = Q::from(a.x * b.zzz, 3);
    }
  }
  return a.x.v[0] ^ a.zzz.v[0] ^ a.y.v[1] ^ a.zz.v[2];
}

__global__ void latency_probe_kernel(int mode, int iters, uint32_t* out) {
  if (mode >= 12) {
    uint32_t s = quad_bisect<FpC>(mode, iters);
    if (threadIdx.x == 0) out[0] = s;
    return;
  }
  if (mode >= 7 && mode <= 9) {  // one warp, quad operations: 7 add (inlined products), 8 add (out-of-line), 9 double (out-of-line)
    uint32_t s = mode == 7 ? quad_probe<Fp>(0, iters) : quad_probe<FpC>(mode == 8 ? 0 : 1, iters);
    if (threadIdx.x == 0) out[0] = s;
    return;
  }
  if (threadIdx.x != 0) return;
  Fp x[4], y;
  for (int j = 0; j < 4; j++)
#pragma unroll
    for (int k = 0; k < 8; k++) x[j].v[k] = (0x9e3779b9u * (k + 1 + 8 * j)) & (k == 7 ? 0x0fffffffu : 0xffffffffu);
#pragma unroll
  for (int k = 0; k < 8; k++) y.v[k] = (0x85ebca6bu * (k + 3)) & (k == 7 ? 0x0fffffffu : 0xffffffffu);
  uint32_t s = 0;
  if (mode >= 10 && mode <= 11) {  // 10: inversion by batched division steps (Mont256::inv), 11: binary extended Euclid
    for (int it = 0; it < iters; it++) x[0] = mode == 10 ? (x[0] + y).inv() : (x[0] + y).inv_euclid();
    out[0] = x[0].v[0];
    return;
  }
  if (mode <= 2) {
    for (int it = 0; it < iters; it++) {
      x[0] = x[0] * y;
      if (mode >= 1) x[1] = x[1] * y;
      if (mode >= 2) { x[2] = x[2] * y; x[3] = x[3] * y; }
    }
    for (int j = 0; j < 4; j++) s ^= x[j].v[0];
  } else if (mode == 3 || mode == 5 || mode == 6) {
    XYZZ<Fp> acc, q;
    acc.x = x[0]; acc.y = x[1]; acc.zz = x[2]; acc.zzz = x[3];
    q.x = y; q.y = x[1] * y; q.zz = x[2] * y; q.zzz = x[3] * y;
    Affine<Fp> qa;
    qa.x = q.x; qa.y = q.y;
    for (int it = 0; it < iters; it++) {
      if (mode == 3) acc.add(q);
      else if (mode == 5) acc.madd(qa);
      else acc = acc.dbl();
    }
    s = acc.x.v[0] ^ acc.zzz.v[0];
  } else {
    XYZZ<FpC> acc, q;
    for (int k = 0; k < 8; k++) {
      acc.x.v[k] = x[0].v[k]; acc.y.v[k] = x[1].v[k]; acc.zz.v[k] = x[2].v[k]; acc.zzz.v[k] = x[3].v[k];
      q.x.v[k] = y.v[k]; q.y.v[k] = x[1].v[k] ^ 5; q.zz.v[k] = x[2].v[k] ^ 9; q.zzz.v[k] = x[3].v[k] ^ 3;
    }
    for (int it = 0; it < iters; it++) acc.add(q);
    s = acc.x.v[0] ^ acc.zzz.v[0];
  }
  out[0] = s;
}
// Variants of zkp_imad_peak (G limb-MAC/s over the chip; every kernel checked in SASS for the instruction named):
//   0: IMAD.WIDE.U32 peak in the form the field arithmetic issues it -- mad.lo.cc / madc.hi.cc pairs, four
//      64-bit lanes deep (ptxas: 1 IMAD.WIDE.U32 + 3 IMAD.WIDE.U32.X + 1 IADD3.X per 4 limb-MACs), 4
//      independent chains per thread per step, multiplicands taken from another chain's limbs so nothing is
//      loop invariant (a loop-invariant product is strength-reduced to additions by ptxas).  This is the
//      roofline denominator: 9.14 T limb-MAC/s measured = 31.4 lanes/clk/SM, the rate of IMAD.HI.
//   1: mad.lo.u32 (IMAD), 2: mad.hi.u32 (IMAD.HI): 8 dependent chains per thread
//   3: chains of whole Fp Montgomery products (136 limb-MACs each): the practical ceiling of a product loop
//   4: plain mad.wide.u32 with both factors in registers, 12 accumulators (ptxas splits the 64-bit accumulate
//      into IMAD.WIDE.U32 ..., RZ + IADD3 / IADD3.X: reads BELOW variant 0, it is bound by the extra additions)
//   5: variant 4 interleaved one-to-one with 64-bit shift-and-add steps on the integer ALU
template <int VARIANT>
__global__ void __launch_bounds__(256) imad_peak_kernel(uint32_t* out, int iters, uint32_t m0) {
  uint32_t seed = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u + 12345u;
  uint32_t b = m0 | 1u;
  if (VARIANT == 3) {
    Fp x, y;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      x.v[k] = seed + k * 0x9e3779b9u;
      y.v[k] = (seed ^ 0x5bd1e995u) + k * 0x85ebca6bu;
    }
    x.v[7] &= 0x0fffffffu;
    y.v[7] &= 0x0fffffffu;
    for (int it = 0; it < iters; it++) {
      x = x * y;
      y = y * x;
    }
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= x.v[k] ^ y.v[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    return;
  }
  if (VARIANT == 0) {
    // the multiplier is a per-thread register, as the limb b_i of a CIOS row is (with a kernel-uniform multiplier
    // ptxas feeds it from a uniform register and the same loop reads 10 % lower)
    const uint32_t y = (seed * 3u) | b;
    uint32_t a[4][8];
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
      for (int j = 0; j < 8; j++) a[k][j] = seed + 17 * k + j;
    uint32_t cs = 0;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < PEAK_UNROLL; u++) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
          uint32_t c;
          asm volatile("mad.lo.cc.u32   %0, %9,  %13, %0;\n\t"
                       "madc.hi.cc.u32  %1, %9,  %13, %1;\n\t"
                       "madc.lo.cc.u32  %2, %10, %13, %2;\n\t"
                       "madc.hi.cc.u32  %3, %10, %13, %3;\n\t"
                       "madc.lo.cc.u32  %4, %11, %13, %4;\n\t"
                       "madc.hi.cc.u32  %5, %11, %13, %5;\n\t"
                       "madc.lo.cc.u32  %6, %12, %13, %6;\n\t"
                       "madc.hi.cc.u32  %7, %12, %13, %7;\n\t"
                       "addc.u32        %8, 0, 0;"
                       : "+r"(a[k][0]), "+r"(a[k][1]), "+r"(a[k][2]), "+r"(a[k][3]), "+r"(a[k][4]), "+r"(a[k][5]),
                         "+r"(a[k][6]), "+r"(a[k][7]), "=r"(c)
                       : "r"(a[(k + 1) & 3][0]), "r"(a[(k + 1) & 3][2]), "r"(a[(k + 1) & 3][4]), "r"(a[(k + 1) & 3][6]), "r"(y));
          cs += c;
        }
      }
    }
    uint32_t s = cs;
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
      for (int j = 0; j < 8; j++) s ^= a[k][j];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    return;
  }
  if (VARIANT == 1 || VARIANT == 2) {
    uint32_t acc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = seed * (k + 3);
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < PEAK_UNROLL; u++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
          if (VARIANT == 1) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(acc[k]) : "r"(b), "r"(seed));
          else asm volatile("mad.hi.u32 %0, %0, %1, %2;" : "+r"(acc[k]) : "r"(b), "r"(seed));
        }
      }
    }
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= acc[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    return;
  }
  // 4 / 5
  const uint32_t x = seed | 1u;
  unsigned long long acc[12];
#pragma unroll
  for (int k = 0; k < 12; k++) acc[k] = ((unsigned long long)(seed + k) << 32) | (seed * (k + 3));
  unsigned long long carry[4] = {seed, seed + 1, seed + 2, seed + 3};
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < PEAK_UNROLL; u++) {
#pragma unroll
      for (int k = 0; k < 12; k++) {
        asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[k]) : "r"((uint32_t)acc[(k + 7) % 12] ^ x), "r"(b));
        if (VARIANT == 5)
          asm volatile("{\n\t.reg .u64 t;\n\tshr.u64 t, %0, 29;\n\tadd.u64 %0, t, %1;\n\t}" : "+l"(carry[k & 3]) : "l"(acc[(k + 3) % 12]));
      }
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < 12; k++) s ^= (uint32_t)acc[k] ^ (uint32_t)(acc[k] >> 32);
#pragma unroll
  for (int k = 0; k < 4; k++) s ^= (uint32_t)carry[k] ^ (uint32_t)(carry[k] >> 32);
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ------------------------------------------------------------------ debug kernels (tests only)
template <class FE>
__global__ void dbg_field_op_kernel(int op, const FE* a, const FE* b, uint64_t n, FE* out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  FE x = a[i].to_mont(), y = b ? b[i].to_mont() : FE::zero(), r;
  if constexpr (FE::Params::MOD_(0) == FpParams::MOD_(0)) {
    if (op == 9) {
      if (!fp_sqrt(x, r)) r.v[0] = r.v[1] = r.v[2] = r.v[3] = r.v[4] = r.v[5] = r.v[6] = r.v[7] = ~0u;
      else r = r.from_mont();
      out[i] = r;
      return;
    }
  }
  switch (op) {
    case 0: r = x + y; break;
    case 1: r = x - y; break;
    case 2: r = x * y; break;
    case 3: r = x.inv(); break;
    case 5: r = x.inv_fermat(); break;
    case 7: r = x.inv_euclid(); break;
    case 6: {  // the two-step product of the lazily reduced Fp2 arithmetic: 512-bit product, then one reduction
      uint32_t t[16];
      FE::mul_wide(x, y, t);
      r = FE::redc_wide(t);
      break;
    }
    case 8:  // x y - (x + y)(x - y) through the lazily reduced product pair (Fp; any other field: two products)
      if constexpr (FE::Params::MOD_(0) == FpParams::MOD_(0))
        r = fp_mulsub_outlined(x, y, x + y, x - y);
      else
        r = x * y - (x + y) * (x - y);
      break;
    default: r = x.sqr(); break;
  }
  out[i] = r.from_mont();
}

// Fp2 products / squarings / inverses of n pairs (64-byte elements c0 || c1, canonical)
__global__ void dbg_fp2_op_kernel(int op, const Fp2* a, const Fp2* b, uint64_t n, Fp2* out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp2 x = a[i].to_mont(), y = b ? b[i].to_mont() : Fp2::zero(), r;
  switch (op) {
    case 2: r = x * y; break;
    case 3: r = x.inv(); break;
    case 9:
      if (!fp2_sqrt(x, r)) {
        for (int k = 0; k < 8; k++) r.c0.v[k] = r.c1.v[k] = ~0u;
        out[i] = r;
        return;
      }
      break;
    default: r = x.sqr(); break;
  }
  out[i] = r.from_mont();
}

template <class F>
__global__ void dbg_point_add_kernel(const Affine<F>* a, const Affine<F>* b, uint64_t n, Affine<F>* out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Affine<F> p = {a[i].x.to_mont(), a[i].y.to_mont()};
  Affine<F> q = {b[i].x.to_mont(), b[i].y.to_mont()};
  // exercise both the mixed and the full addition: (p as XYZZ) + q, then + infinity via add()
  XYZZ<F> acc = XYZZ<F>::from_affine(p);
  acc.madd(q);
  XYZZ<F> z = XYZZ<F>::inf();
  z.add(acc);
  Affine<F> r = z.to_affine();
  out[i] = {r.x.from_mont(), r.y.from_mont()};
}

// The same sum through the quad-lane operations of ec_quad.cuh (four lanes per pair): a + b by Quad::add,
// and 2*(a + b) - (a + b) folded in through Quad::dbl and a second Quad::add so the doubling path and the
// P + (-P) path of the combination are exercised too:  r = (2s) + (-s) with s = a + b.
template <class F>
__global__ void dbg_point_add_quad_kernel(const Affine<F>* a, const Affine<F>* b, uint64_t n, Affine<F>* out) {
  const uint64_t gt = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t i = gt >> 2;
  const int ql = threadIdx.x & 3;
  const bool live = i < n;
  if (!live) i = n - 1;  // whole warps take part in the shuffles
  Affine<F> p = {a[i].x.to_mont(), a[i].y.to_mont()};
  Affine<F> q = {b[i].x.to_mont(), b[i].y.to_mont()};
  XYZZ<F> s = Quad<F>::add(XYZZ<F>::from_affine(p), XYZZ<F>::from_affine(q), ql);
  XYZZ<F> r = Quad<F>::add(Quad<F>::dbl(s, ql), s.neg(), ql);
  if (live && ql == 0) {
    Affine<F> o = r.to_affine();
    out[i] = {o.x.from_mont(), o.y.from_mont()};
  }
}

}  // namespace zkp

using namespace zkp;

extern "C" {

int zkp_latency_probe(int mode, double* ns_per_op) {
  return guarded([&](Context& c) {
    diag_events();
    if (mode < 0 || mode > 15 || !ns_per_op) throw InvalidArgument("zkp_latency_probe: bad mode");
    ScopedDevBuf out;
    out.reserve(64);
    const int iters = (mode == 10 || mode == 11) ? 100 : 2000;
    latency_probe_kernel<<<1, 32, 0, c.stream>>>(mode, iters / 10, out.as<uint32_t>());
    CUDA_CHECK_LAUNCH();
    float best = 1e30f;
    for (int rep = 0; rep < 3; rep++) {
      CUDA_CHECK(cudaEventRecord(d_ev0, c.stream));
      latency_probe_kernel<<<1, 32, 0, c.stream>>>(mode, iters, out.as<uint32_t>());
      CUDA_CHECK_LAUNCH();
      CUDA_CHECK(cudaEventRecord(d_ev1, c.stream));
      CUDA_CHECK(cudaEventSynchronize(d_ev1));
      float ms;
      CUDA_CHECK(cudaEventElapsedTime(&ms, d_ev0, d_ev1));
      if (ms < best) best = ms;
    }
    c.launches += 4;
    *ns_per_op = (double)best * 1e6 / iters;
  });
}

int zkp_imad_peak(int variant, double* gmacs_per_s, double* sm_clock_mhz_effective) {
  return guarded([&](Context& c) {
    diag_events();
    if (variant < 0 || variant > 5 || !gmacs_per_s) throw InvalidArgument("zkp_imad_peak: bad variant");
    const int blocks = c.sm_count * ((variant == 1 || variant == 2) ? 8 : 4), threads = 256;
    const int iters = variant == 3 ? 2000 : 4000;
    ScopedDevBuf out;
    out.reserve((size_t)blocks * threads * 4);
    auto launch = [&](int it) {
      switch (variant) {
        case 0: imad_peak_kernel<0><<<blocks, threads, 0, c.stream>>>(out.as<uint32_t>(), it, 0x12345677u); break;
        case 1: imad_peak_kernel<1><<<blocks, threads, 0, c.stream>>>(out.as<uint32_t>(), it, 0x12345677u); break;
        case 2: imad_peak_kernel<2><<<blocks, threads, 0, c.stream>>>(out.as<uint32_t>(), it, 0x12345677u); break;
        case 3: imad_peak_kernel<3><<<blocks, threads, 0, c.stream>>>(out.as<uint32_t>(), it, 0x12345677u); break;
        case 4: imad_peak_kernel<4><<<blocks, threads, 0, c.stream>>>(out.as<uint32_t>(), it, 0x12345677u); break;
        default: imad_peak_kernel<5><<<blocks, threads, 0, c.stream>>>(out.as<uint32_t>(), it, 0x12345677u); break;
      }
      CUDA_CHECK_LAUNCH();
      c.launches++;
    };
    launch(iters / 10);  // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
      CUDA_CHECK(cudaEventRecord(d_ev0, c.stream));
      launch(iters);
      CUDA_CHECK(cudaEventRecord(d_ev1, c.stream));
      CUDA_CHECK(cudaEventSynchronize(d_ev1));
      float ms;
      CUDA_CHECK(cudaEventElapsedTime(&ms, d_ev0, d_ev1));
      if (ms < best) best = ms;
    }
    double per_iter = variant == 3 ? 2.0 * 136 : variant == 0 ? PEAK_UNROLL * 16.0 : variant >= 4 ? PEAK_UNROLL * 12.0 : PEAK_UNROLL * 8.0;
    double macs = per_iter * iters * blocks * threads;
    *gmacs_per_s = macs / (best * 1e-3) / 1e9;
    if (sm_clock_mhz_effective) *sm_clock_mhz_effective = 0.0;  // clocks are sampled by bench.py via nvidia-smi
  });
}

int zkp_dbg_field_op(int field, int op, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out) {
  return guarded([&](Context& c) {
    if (!a || !out || op < 0 || op > 9) throw InvalidArgument("zkp_dbg_field_op: bad argument");
    if (n == 0) return;
    if (field < 0 || field > 2) throw InvalidArgument("zkp_dbg_field_op: field must be 0 (Fp), 1 (Fr) or 2 (Fp2)");
    if (op == 9 && field == 1) throw InvalidArgument("zkp_dbg_field_op: the square root is for Fp and Fp2 (p = 3 mod 4)");
    const size_t sz = field == 2 ? 64 : 32;
    ScopedDevBuf da, db, dout;
    da.reserve(n * sz);
    dout.reserve(n * sz);
    CUDA_CHECK(cudaMemcpyAsync(da.p, a, n * sz, cudaMemcpyHostToDevice, c.stream));
    if (b) {
      db.reserve(n * sz);
      CUDA_CHECK(cudaMemcpyAsync(db.p, b, n * sz, cudaMemcpyHostToDevice, c.stream));
    }
    if (field == 2)
      dbg_fp2_op_kernel<<<ceil_div(n, 128), 128, 0, c.stream>>>(op, da.as<Fp2>(), b ? db.as<Fp2>() : nullptr, n, dout.as<Fp2>());
    else if (field == 0)
      dbg_field_op_kernel<Fp><<<ceil_div(n, 128), 128, 0, c.stream>>>(op, da.as<Fp>(), b ? db.as<Fp>() : nullptr, n,
                                                                     dout.as<Fp>());
    else
      dbg_field_op_kernel<Fr><<<ceil_div(n, 128), 128, 0, c.stream>>>(op, da.as<Fr>(), b ? db.as<Fr>() : nullptr, n,
                                                                     dout.as<Fr>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out, dout.p, n * sz, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_dbg_point_add(int group, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out) {
  return guarded([&](Context& c) {
    if (!a || !b || !out) throw InvalidArgument("zkp_dbg_point_add: null argument");
    if (n == 0) return;
    if (group < 0 || group > 3) throw InvalidArgument("zkp_dbg_point_add: group must be 0 (G1), 1 (G2), 2 / 3 (the same on quads of lanes)");
    size_t sz = (group & 1) == 0 ? 64 : 128;
    ScopedDevBuf da, db, dout;
    da.reserve(n * sz);
    db.reserve(n * sz);
    dout.reserve(n * sz);
    CUDA_CHECK(cudaMemcpyAsync(da.p, a, n * sz, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(db.p, b, n * sz, cudaMemcpyHostToDevice, c.stream));
    if (group == 2)
      dbg_point_add_quad_kernel<Fp><<<ceil_div(4 * n, 64), 64, 0, c.stream>>>(da.as<G1Affine>(), db.as<G1Affine>(), n,
                                                                             dout.as<G1Affine>());
    else if (group == 3)
      dbg_point_add_quad_kernel<Fp2><<<ceil_div(4 * n, 64), 64, 0, c.stream>>>(da.as<G2Affine>(), db.as<G2Affine>(), n,
                                                                              dout.as<G2Affine>());
    else if (group == 0)
      dbg_point_add_kernel<Fp><<<ceil_div(n, 64), 64, 0, c.stream>>>(da.as<G1Affine>(), db.as<G1Affine>(), n,
                                                                    dout.as<G1Affine>());
    else
      dbg_point_add_kernel<Fp2><<<ceil_div(n, 64), 64, 0, c.stream>>>(da.as<G2Affine>(), db.as<G2Affine>(), n,
                                                                     dout.as<G2Affine>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out, dout.p, n * sz, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

}  // extern "C"
