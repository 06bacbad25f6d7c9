// Fr vector / polynomial layer of libzkp_b200 (include/zkp_b200.h): pointwise ops, batch inversion,
// Horner evaluation, NTT-based products, division with remainder, the Groth16 quotient.
//
// Replaces the coefficient-form Python loops of the reference:
//   Polynomial.__add__/__sub__/__mul__/evaluate   /root/reference/zkp/plonk/polynomial.py:85-159
//   poly_div (long division)                      /root/reference/zkp/plonk/polynomial.py:385-435
//   _multiply_polys/_subtract_polys/_div_polys/hxr /root/reference/zkp/groth16/poly_utils.py:17-45,116-125
//   _multiply_vec_matrix                          /root/reference/zkp/groth16/poly_utils.py:52-59
//   compute_accumulator's n-1 divisions           /root/reference/zkp/plonk/permutation.py:120-135
// The reference's schoolbook product is O(n^2) and its long division O(n^2)..O(n^3); here a product
// is three NTTs and a division is a Newton power-series inversion of the reversed divisor
// (quotient) followed by one cyclic product (remainder).  The quotient and remainder of a division
// are unique, so the results are bit-identical with the reference's.
#include <cstring>
#include <vector>
#include "ntt.cuh"
#include "registry.cuh"

namespace zkp {

// ------------------------------------------------------------------ arena of reusable device chunks
struct Arena {
  struct Chunk {
    DevBuf buf;
    bool used = false;
  };
  std::vector<std::unique_ptr<Chunk>> chunks;
  Fr* alloc(uint64_t n_elems) {
    size_t bytes = (size_t)(n_elems ? n_elems : 1) * sizeof(Fr);
    Chunk* best = nullptr;
    for (auto& ch : chunks)
      if (!ch->used && ch->buf.cap >= bytes && (!best || ch->buf.cap < best->buf.cap)) best = ch.get();
    if (!best) {
      for (auto& ch : chunks)
        if (!ch->used && (!best || ch->buf.cap > best->buf.cap)) best = ch.get();
      if (!best) {
        chunks.emplace_back(new Chunk());
        best = chunks.back().get();
      }
      best->buf.reserve(bytes);
    }
    best->used = true;
    return best->buf.as<Fr>();
  }
  // stream-ordered reuse: a freed chunk may be handed out again to work enqueued later on the same stream
  void free(Fr* p) {
    for (auto& ch : chunks)
      if (ch->buf.p == p) ch->used = false;
  }
  void reset() {
    for (auto& ch : chunks) ch->used = false;
  }
};
static Arena g_arena;
struct ArenaScope {
  ~ArenaScope() { g_arena.reset(); }
};

static FrBytes omega_for(uint32_t log_n) {
  FrBytes w;
  memcpy(w.b, FrParams::OMEGA[log_n], 32);
  return w;
}
static uint32_t log2_ceil(uint64_t n) {
  uint32_t l = 0;
  while ((uint64_t(1) << l) < n) l++;
  return l;
}

// ------------------------------------------------------------------ elementwise kernels
#define GRID_1D(n) ceil_div((n), 256), 256, 0, c.stream
#define IDX64 ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x)

// canonical in, canonical out.  op: 0 add, 1 sub, 2 mul, 3 scale by b[0]
__global__ void fr_vec_op_kernel(int op, const Fr* __restrict__ a, const Fr* __restrict__ b, uint64_t n,
                                 Fr* __restrict__ out) {
  uint64_t i = IDX64;
  if (i >= n) return;
  Fr x = a[i], y = b[op == 3 ? 0 : i], r;
  if (op == 0) r = x + y;
  else if (op == 1) r = x - y;
  else r = (x * y) * Fr::r2();  // (xy R^-1)(R^2) R^-1 = xy
  out[i] = r;
}
__global__ void fr_to_mont_kernel(const Fr* __restrict__ in, uint64_t n, Fr* __restrict__ out) {
  uint64_t i = IDX64;
  if (i < n) out[i] = in[i].to_mont();
}
__global__ void fr_from_mont_kernel(const Fr* __restrict__ in, uint64_t n, Fr* __restrict__ out) {
  uint64_t i = IDX64;
  if (i < n) out[i] = in[i].from_mont();
}
__global__ void fr_mul_inplace_kernel(Fr* __restrict__ a, const Fr* __restrict__ b, uint64_t n) {
  uint64_t i = IDX64;
  if (i < n) a[i] = a[i] * b[i];
}
__global__ void fr_sub_inplace_kernel(Fr* __restrict__ a, const Fr* __restrict__ b, uint64_t n) {
  uint64_t i = IDX64;
  if (i < n) a[i] = a[i] - b[i];
}
// out[i] = in[len-1-i] for i < m (zero where the index runs off the front)
__global__ void fr_reverse_kernel(const Fr* __restrict__ in, uint64_t len, uint64_t m, Fr* __restrict__ out) {
  uint64_t i = IDX64;
  if (i < m) out[i] = i < len ? in[len - 1 - i] : Fr::zero();
}
// out[i] = sum_k in[i + k*N], i < N   (reduction modulo x^N - 1)
__global__ void fr_fold_kernel(const Fr* __restrict__ in, uint64_t len, uint64_t N, Fr* __restrict__ out) {
  uint64_t i = IDX64;
  if (i >= N) return;
  Fr acc = Fr::zero();
  for (uint64_t k = i; k < len; k += N) acc = acc + in[k];
  out[i] = acc;
}
// t[i] = (i == 0 ? 2 : 0) - t[i]   (Montgomery)
__global__ void fr_two_minus_kernel(Fr* __restrict__ t, uint64_t n) {
  uint64_t i = IDX64;
  if (i >= n) return;
  Fr two = Fr::one() + Fr::one();
  t[i] = (i == 0 ? two : Fr::zero()) - t[i];
}
__global__ void fr_inv_single_kernel(const Fr* __restrict__ in, Fr* __restrict__ out) {
  if (IDX64 == 0) *out = in->inv();
}
// out[i] = a[i] * (*s)
__global__ void fr_scale_by_dev_kernel(const Fr* __restrict__ a, const Fr* __restrict__ s, uint64_t n,
                                       Fr* __restrict__ out) {
  uint64_t i = IDX64;
  if (i < n) out[i] = a[i] * (*s);
}

// Batch inversion, Montgomery's trick on strided chunks: thread t owns elements t, t+T, t+2T, ...
// (coalesced), one Fermat inversion per BATCH_INV_CHUNK elements.  Zeros map to zero (py_ecc inv(0)=0).
// Input and output in the same form F: canonical (mont == 0) or Montgomery (mont == 1).
// sum_i a[i] * b[i] over canonical vectors: every product is a Montgomery product of two canonical values
// (= a*b/R); the partial sums stay in that form and the last step multiplies by R^2 (mont: * R) once.
static constexpr int DOT_THREADS = 256;
__device__ __forceinline__ Fr dot_block_reduce(Fr acc, Fr* sm) {
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = DOT_THREADS / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sm[threadIdx.x] = sm[threadIdx.x] + sm[threadIdx.x + s];
    __syncthreads();
  }
  return sm[0];
}
__global__ void __launch_bounds__(DOT_THREADS) fr_dot_partial_kernel(const Fr* __restrict__ a, const Fr* __restrict__ b,
                                                                      uint64_t n, Fr* __restrict__ partial) {
  __shared__ Fr sm[DOT_THREADS];
  Fr acc = Fr::zero();
  for (uint64_t i = (uint64_t)blockIdx.x * DOT_THREADS + threadIdx.x; i < n; i += (uint64_t)gridDim.x * DOT_THREADS)
    acc = acc + a[i] * b[i];
  Fr tot = dot_block_reduce(acc, sm);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(DOT_THREADS) fr_dot_final_kernel(const Fr* __restrict__ partial, uint32_t count,
                                                                    Fr* __restrict__ out) {
  __shared__ Fr sm[DOT_THREADS];
  Fr acc = Fr::zero();
  for (uint32_t i = threadIdx.x; i < count; i += DOT_THREADS) acc = acc + partial[i];
  Fr tot = dot_block_reduce(acc, sm);
  if (threadIdx.x == 0) *out = tot * Fr::r2();
}

static constexpr int BATCH_INV_CHUNK = 32;
__global__ void __launch_bounds__(128) fr_batch_inverse_kernel(const Fr* __restrict__ in, uint64_t n, uint64_t T, int mont,
                                                                Fr* __restrict__ out) {
  uint64_t t = IDX64;
  if (t >= T) return;
  Fr pre[BATCH_INV_CHUNK];
  Fr acc = Fr::one();
  int cnt = 0;
  for (uint64_t i = t; i < n && cnt < BATCH_INV_CHUNK; i += T, cnt++) {
    Fr x = in[i];
    if (!mont) x = x.to_mont();
    pre[cnt] = acc;
    if (!x.is_zero()) acc = acc * x;
  }
  Fr inv = acc.inv();
  for (int k = cnt - 1; k >= 0; k--) {
    uint64_t i = t + (uint64_t)k * T;
    Fr x = in[i];
    if (!mont) x = x.to_mont();
    Fr r = Fr::zero();
    if (!x.is_zero()) {
      r = inv * pre[k];
      inv = inv * x;
    }
    out[i] = mont ? r : r.from_mont();
  }
}

// Horner evaluation in levels of HORNER_CHUNK: thread j evaluates its chunk of 64 coefficients at x
// (level 0), the n/64 partial values are the coefficients of a polynomial in x^64 (level 1), and so
// on until one value is left: log_64(n) launches, each 64 sequential multiply-adds deep.
// coeffs canonical, powers Montgomery (xs[l] = x^(64^l)), results canonical.
static constexpr int HORNER_CHUNK = 64;
__global__ void horner_powers_kernel(const Fr* __restrict__ x_canon, Fr* __restrict__ xs, int levels) {
  if (IDX64 != 0) return;
  Fr x = x_canon->to_mont();
  for (int l = 0; l < levels; l++) {
    xs[l] = x;
    for (int k = 1; k < HORNER_CHUNK; k <<= 1) x = x.sqr();
  }
}
__global__ void horner_partial_kernel(const Fr* __restrict__ coeffs, uint64_t n, const Fr* __restrict__ xp,
                                      Fr* __restrict__ partial) {
  uint64_t j = IDX64;
  uint64_t beg = j * HORNER_CHUNK;
  if (beg >= n) return;
  uint64_t end = beg + HORNER_CHUNK < n ? beg + HORNER_CHUNK : n;
  Fr x = *xp;
  Fr acc = Fr::zero();
  for (uint64_t i = end; i > beg; i--) acc = acc * x + coeffs[i - 1];  // canonical coeffs: acc stays canonical
  partial[j] = acc;
}

// p(x) for n device coefficients (canonical); x: 32 canonical bytes on the host; result left in *out_dev
static int poly_eval_dev_impl(Context& c, const Fr* coeffs, uint64_t n, const uint8_t* x, Fr* out_dev) {
  int levels = 0;
  for (uint64_t m = n; m > 1; m = (m + HORNER_CHUNK - 1) / HORNER_CHUNK) levels++;
  if (levels == 0) levels = 1;
  Fr* xs = g_arena.alloc(levels + 1);
  Fr* xc = xs + levels;
  CUDA_CHECK(cudaMemcpyAsync(xc, x, 32, cudaMemcpyHostToDevice, c.stream));
  horner_powers_kernel<<<1, 32, 0, c.stream>>>(xc, xs, levels);
  CUDA_CHECK_LAUNCH();
  int launches = 1;
  const Fr* cur = coeffs;
  uint64_t m = n;
  for (int l = 0; l < levels; l++) {
    uint64_t np = (m + HORNER_CHUNK - 1) / HORNER_CHUNK;
    Fr* part = np == 1 ? out_dev : g_arena.alloc(np);
    horner_partial_kernel<<<GRID_1D(np)>>>(cur, m, xs + l, part);
    CUDA_CHECK_LAUNCH();
    launches++;
    cur = part;
    m = np;
  }
  return launches;
}

// Several polynomials evaluated in the same launches (blockIdx.y = item): PLONK round 4 needs six
// evaluations of ~n coefficients (round4.py:39-81), each only a few latency-bound Horner levels deep.
static constexpr int MULTI_MAX = 16;
struct MultiEvalArgs {
  const Fr* coeffs[MULTI_MAX];
  uint64_t n[MULTI_MAX];
  int point[MULTI_MAX];  // which of the evaluation points
};
__global__ void horner_powers_multi_kernel(const Fr* __restrict__ x_canon, int points, Fr* __restrict__ xs, int levels) {
  int p = (int)IDX64;
  if (p >= points) return;
  Fr x = x_canon[p].to_mont();
  for (int l = 0; l < levels; l++) {
    xs[p * levels + l] = x;
    for (int k = 1; k < HORNER_CHUNK; k <<= 1) x = x.sqr();
  }
}
__global__ void horner_multi_kernel(MultiEvalArgs a, int level, int levels, const Fr* __restrict__ xs,
                                    const Fr* __restrict__ prev, uint64_t stride_prev, Fr* __restrict__ cur,
                                    uint64_t stride_cur) {
  const int k = blockIdx.y;
  uint64_t m = a.n[k];
  for (int l = 0; l < level; l++) m = (m + HORNER_CHUNK - 1) / HORNER_CHUNK;
  const Fr* in = level == 0 ? a.coeffs[k] : prev + (uint64_t)k * stride_prev;
  uint64_t j = IDX64;
  uint64_t beg = j * HORNER_CHUNK;
  if (beg >= m) return;
  uint64_t end = beg + HORNER_CHUNK < m ? beg + HORNER_CHUNK : m;
  Fr x = xs[a.point[k] * levels + level];
  Fr acc = Fr::zero();
  for (uint64_t i = end; i > beg; i--) acc = acc * x + in[i - 1];
  cur[(uint64_t)k * stride_cur + j] = acc;
}

// dst[i] = sum_k coeff_k * src_k[i] over the items long enough to have an i-th element (canonical in/out)
struct LinCombArgs {
  const Fr* src[MULTI_MAX];
  uint64_t len[MULTI_MAX];
  Fr coeff[MULTI_MAX];  // Montgomery
  int count;
};
__global__ void fr_lincomb_kernel(LinCombArgs a, uint64_t n, Fr* __restrict__ dst) {
  uint64_t i = IDX64;
  if (i >= n) return;
  Fr acc = Fr::zero();
  for (int k = 0; k < a.count; k++)
    if (i < a.len[k]) acc = acc + a.src[k][i] * a.coeff[k];
  dst[i] = acc;
}

// out[j] = sum_i vec[i] * mat[i*cols + j]   (canonical in/out)
__global__ void fr_vec_matrix_kernel(const Fr* __restrict__ vec, const Fr* __restrict__ mat, uint64_t rows, uint64_t cols,
                                     Fr* __restrict__ out) {
  uint64_t j = IDX64;
  if (j >= cols) return;
  Fr acc = Fr::zero();
  for (uint64_t i = 0; i < rows; i++) acc = acc + vec[i].to_mont() * mat[i * cols + j];  // (vR)(m)R^-1 = vm
  out[j] = acc;
}

// Division by x^n - 1: q_i = sum_{k>=1} a[i + k n], r_i = a_i + q_i (i < n).  One thread per residue.
__global__ void fr_div_vanishing_kernel(const Fr* __restrict__ a, uint64_t la, uint64_t n, Fr* __restrict__ q,
                                        uint64_t lq, Fr* __restrict__ r) {
  uint64_t i = IDX64;
  if (i >= n) return;
  // walk the residue class from the top down
  uint64_t top = i + ((la - 1 - i) / n) * n;  // largest index == i mod n below la (la > i guaranteed by caller)
  Fr run = Fr::zero();
  for (uint64_t k = top; k >= n + i; k -= n) {
    run = run + a[k];
    q[k - n] = run;
  }
  r[i] = a[i] + run;
  (void)lq;
}


// ------------------------------------------------------------------ exclusive prefix product
// out[0] = 1, out[i] = in[0] * ... * in[i-1]  (canonical in and out).  Tiles of 1024 elements:
// tile products -> single-block scan of the tile products -> per-tile scan.  Replaces running
// products such as tau^i (srs.py:78-82) and the accumulator z (permutation.py:120-135).
static constexpr int PP_THREADS = 256, PP_ITEMS = 4, PP_TILE = PP_THREADS * PP_ITEMS;

// The scans are generic over the monoid: SUM == false -> products (canonical in/out, Montgomery
// inside), SUM == true -> sums (form-agnostic).
template <bool SUM>
__device__ __forceinline__ Fr scan_op(const Fr& a, const Fr& b) {
  if (SUM) return a + b;
  return a * b;
}
template <bool SUM>
__device__ __forceinline__ Fr scan_id() {
  return SUM ? Fr::zero() : Fr::one();
}
template <bool SUM>
__device__ __forceinline__ Fr scan_in(const Fr& a) {
  return SUM ? a : a.to_mont();
}
template <bool SUM>
__device__ __forceinline__ Fr scan_out(const Fr& a) {
  return SUM ? a : a.from_mont();
}

// inclusive block scan (Hillis-Steele in shared memory) of one value per thread
template <bool SUM>
__device__ __forceinline__ Fr block_inclusive_scan(Fr v, Fr* sm) {
  sm[threadIdx.x] = v;
  __syncthreads();
  for (int o = 1; o < PP_THREADS; o <<= 1) {
    Fr t = v;
    if ((int)threadIdx.x >= o) t = scan_op<SUM>(sm[threadIdx.x - o], v);
    __syncthreads();
    v = t;
    sm[threadIdx.x] = v;
    __syncthreads();
  }
  return v;
}

template <bool SUM>
__global__ void __launch_bounds__(PP_THREADS) pp_tile_products_kernel(const Fr* __restrict__ in, uint64_t n,
                                                                       Fr* __restrict__ tile_prod) {
  __shared__ Fr sm[PP_THREADS];
  uint64_t base = (uint64_t)blockIdx.x * PP_TILE + (uint64_t)threadIdx.x * PP_ITEMS;
  Fr p = scan_id<SUM>();
#pragma unroll
  for (int k = 0; k < PP_ITEMS; k++)
    if (base + k < n) p = scan_op<SUM>(p, scan_in<SUM>(in[base + k]));
  Fr inc = block_inclusive_scan<SUM>(p, sm);
  if (threadIdx.x == PP_THREADS - 1) tile_prod[blockIdx.x] = inc;
}

// single block: tile_prod[i] <- exclusive prefix; *total (optional) <- the grand total
template <bool SUM>
__global__ void __launch_bounds__(PP_THREADS) pp_tile_scan_kernel(Fr* __restrict__ tile_prod, uint64_t ntiles,
                                                                   Fr* __restrict__ total) {
  __shared__ Fr sm[PP_THREADS];
  __shared__ Fr carry;
  if (threadIdx.x == 0) carry = scan_id<SUM>();
  __syncthreads();
  for (uint64_t base = 0; base < ntiles; base += PP_THREADS) {
    uint64_t i = base + threadIdx.x;
    Fr v = i < ntiles ? tile_prod[i] : scan_id<SUM>();
    Fr inc = block_inclusive_scan<SUM>(v, sm);
    Fr c = carry;
    Fr prev = threadIdx.x ? sm[threadIdx.x - 1] : scan_id<SUM>();
    __syncthreads();
    if (i < ntiles) tile_prod[i] = scan_op<SUM>(c, prev);
    if (threadIdx.x == PP_THREADS - 1) carry = scan_op<SUM>(c, inc);
    __syncthreads();
  }
  if (total && threadIdx.x == 0) *total = scan_out<SUM>(carry);
}

template <bool SUM>
__global__ void __launch_bounds__(PP_THREADS) pp_apply_kernel(const Fr* __restrict__ in, uint64_t n,
                                                               const Fr* __restrict__ tile_off, Fr* __restrict__ out) {
  __shared__ Fr sm[PP_THREADS];
  uint64_t base = (uint64_t)blockIdx.x * PP_TILE + (uint64_t)threadIdx.x * PP_ITEMS;
  Fr x[PP_ITEMS];
  Fr p = scan_id<SUM>();
#pragma unroll
  for (int k = 0; k < PP_ITEMS; k++) {
    x[k] = (base + k < n) ? scan_in<SUM>(in[base + k]) : scan_id<SUM>();
    p = scan_op<SUM>(p, x[k]);
  }
  block_inclusive_scan<SUM>(p, sm);
  Fr run = tile_off[blockIdx.x];
  if (threadIdx.x) run = scan_op<SUM>(run, sm[threadIdx.x - 1]);
#pragma unroll
  for (int k = 0; k < PP_ITEMS; k++) {
    if (base + k < n) out[base + k] = scan_out<SUM>(run);
    run = scan_op<SUM>(run, x[k]);
  }
}

// exclusive scan of n device elements: out[i] = op(in[0..i)); optional grand total.  in != out.
template <bool SUM>
static int scan_dev(Context& c, const Fr* in, uint64_t n, Fr* out, Fr* total) {
  uint64_t ntiles = (n + PP_TILE - 1) / PP_TILE;
  Fr* tiles = g_arena.alloc(ntiles);
  pp_tile_products_kernel<SUM><<<(unsigned)ntiles, PP_THREADS, 0, c.stream>>>(in, n, tiles);
  CUDA_CHECK_LAUNCH();
  pp_tile_scan_kernel<SUM><<<1, PP_THREADS, 0, c.stream>>>(tiles, ntiles, total);
  CUDA_CHECK_LAUNCH();
  pp_apply_kernel<SUM><<<(unsigned)ntiles, PP_THREADS, 0, c.stream>>>(in, n, tiles, out);
  CUDA_CHECK_LAUNCH();
  return 3;
}


// ------------------------------------------------------------------ device-handle vector kernels
__global__ void fr_axpy_kernel(Fr* __restrict__ dst, Fr k_mont, const Fr* __restrict__ src, uint64_t n) {
  uint64_t i = IDX64;
  if (i < n) dst[i] = dst[i] + src[i] * k_mont;  // canonical * Montgomery constant -> canonical
}
__global__ void fr_add_const_kernel(Fr* __restrict__ v, Fr k, uint64_t n) {
  uint64_t i = IDX64;
  if (i < n) v[i] = v[i] + k;
}
// v[i] = first * base^i (canonical out); ptab: two-level power table of base (ntt.cuh)
__global__ void fr_fill_powers_kernel(Fr* __restrict__ v, uint64_t n, Fr first, const Fr* __restrict__ ptab) {
  uint64_t i = IDX64;
  if (i >= n) return;
  v[i] = i ? first * power_at(ptab, (uint32_t)i) : first;
}
// v[i] *= x^i
__global__ void fr_scale_powers_kernel(Fr* __restrict__ v, uint64_t n, const Fr* __restrict__ ptab) {
  uint64_t i = IDX64;
  if (i < n && i) v[i] = v[i] * power_at(ptab, (uint32_t)i);
}
__global__ void fr_is_zero_kernel(const Fr* __restrict__ v, uint64_t n, int* __restrict__ flag) {
  uint64_t i = IDX64;
  if (i < n && !v[i].is_zero()) *flag = 0;
}
// q_k = zeta^-(k+1) * (T - P_k - d_k), d_j = c_j zeta^j, P = exclusive prefix sums of d, T = sum d.
// zinv_tab: two-level power table of zeta^-1 (ntt.cuh).  All values canonical.
__global__ void fr_div_linear_finish_kernel(const Fr* __restrict__ d, const Fr* __restrict__ P, const Fr* __restrict__ T,
                                            const Fr* __restrict__ zinv_tab, uint64_t n_out, Fr* __restrict__ q) {
  uint64_t k = IDX64;
  if (k >= n_out) return;
  q[k] = (*T - P[k] - d[k]) * power_at(zinv_tab, (uint32_t)(k + 1));
}

// PLONK grand-product factors (permutation.py:120-135), canonical in/out:
//   num_i = (a_i + beta w^i + gamma)(b_i + beta K1 w^i + gamma)(c_i + beta K2 w^i + gamma)
//   den_i = (a_i + beta s1_i + gamma)(b_i + beta s2_i + gamma)(c_i + beta s3_i + gamma)
__global__ void plonk_perm_terms_kernel(const Fr* __restrict__ a, const Fr* __restrict__ b, const Fr* __restrict__ c,
                                        const Fr* __restrict__ s1, const Fr* __restrict__ s2, const Fr* __restrict__ s3,
                                        uint64_t n, const Fr* __restrict__ omega_tab, Fr beta_c, Fr gamma_c,
                                        Fr* __restrict__ num, Fr* __restrict__ den) {
  uint64_t i = IDX64;
  if (i >= n) return;
  Fr beta = beta_c.to_mont(), gamma = gamma_c.to_mont();
  Fr w = power_at(omega_tab, (uint32_t)i);  // two-level power table (ntt.cuh); entry 0 is one
  Fr bw = beta * w;
  Fr am = a[i].to_mont() + gamma, bm = b[i].to_mont() + gamma, cm = c[i].to_mont() + gamma;
  Fr nu = (am + bw) * (bm + bw.dbl()) * (cm + bw.dbl() + bw);
  Fr de = (am + beta * s1[i].to_mont()) * (bm + beta * s2[i].to_mont()) * (cm + beta * s3[i].to_mont());
  num[i] = nu.from_mont();
  den[i] = de.from_mont();
}

// zh_inv[j] = 1 / (g^n * (w8^n)^j - 1), j < 8 (Montgomery): Z_H on the 8n coset takes 8 values.
__global__ void plonk_zh_inv_kernel(Fr g_n_canon, Fr w8n_canon, uint32_t ext, Fr* __restrict__ out) {
  uint32_t j = threadIdx.x;
  if (j >= ext) return;
  Fr v = g_n_canon.to_mont(), w = w8n_canon.to_mont();
  for (uint32_t k = 0; k < j; k++) v = v * w;
  out[j] = (v - Fr::one()).inv();
}

struct PlonkQuotArgs {
  const Fr *a, *b, *c, *z, *ql, *qr, *qo, *qm, *qc, *s1, *s2, *s3;  // 8n coset evaluations, Montgomery
  const Fr *x;        // coset points x_i = g w8^i, Montgomery
  const Fr *l1f;      // 1 / (n (x_i - 1)), Montgomery
  const Fr *zh_inv;   // 8 values
  Fr beta, gamma, alpha;  // canonical
  uint64_t N;         // ext * n
  uint32_t ext;       // coset size / n: 4 (n >= 8), 8 (n = 2, 4), 16 (n = 1); N >= 3n + 6
  Fr* t;              // out: quotient evaluations, Montgomery
};
// t(x) = [gate + alpha*(perm_num - perm_den)] / Z_H(x) + alpha^2 (z(x) - 1) / (n (x - 1))
// (round3.py:114-147 evaluated pointwise on a coset where Z_H != 0; the L1 term's Z_H cancels).
__global__ void __launch_bounds__(128) plonk_quotient_kernel(PlonkQuotArgs q) {
  uint64_t i = IDX64;
  if (i >= q.N) return;
  Fr beta = q.beta.to_mont(), gamma = q.gamma.to_mont(), alpha = q.alpha.to_mont();
  Fr a = q.a[i], b = q.b[i], c = q.c[i], z = q.z[i];
  Fr zw = q.z[(i + q.ext) & (q.N - 1)];  // z(w x): w = w_N^ext
  Fr gate = q.ql[i] * a + q.qr[i] * b + q.qo[i] * c + q.qm[i] * (a * b) + q.qc[i];
  Fr bx = beta * q.x[i];
  Fr ag = a + gamma, bg = b + gamma, cg = c + gamma;
  Fr num = (ag + bx) * (bg + bx.dbl()) * (cg + bx.dbl() + bx) * z;
  Fr den = (ag + beta * q.s1[i]) * (bg + beta * q.s2[i]) * (cg + beta * q.s3[i]) * zw;
  Fr main = (gate + alpha * (num - den)) * q.zh_inv[i & (q.ext - 1)];
  Fr l1 = alpha * alpha * ((z - Fr::one()) * q.l1f[i]);
  q.t[i] = main + l1;
}
// x_i = g * w8^i and l1f_i = 1/(n (x_i - 1)) before inversion: writes x (Montgomery) and n(x_i-1) (Montgomery)
__global__ void plonk_coset_points_kernel(uint64_t N, Fr g_canon, const Fr* __restrict__ w8_pow2, Fr n_canon,
                                          Fr* __restrict__ x, Fr* __restrict__ l1den) {
  uint64_t i = IDX64;
  if (i >= N) return;
  Fr r = g_canon.to_mont();
  uint64_t e = i;
  for (int k = 0; e; k++, e >>= 1)
    if (e & 1) r = r * w8_pow2[k];
  x[i] = r;
  l1den[i] = n_canon.to_mont() * (r - Fr::one());
}

// ------------------------------------------------------------------ device-level polynomial ops (Montgomery)
// out[0..out_len) = (a * b)[0..out_len); a, b, out device Montgomery; out must not alias a or b.
static int poly_mul_dev(Context& c, const Fr* a, uint64_t la, const Fr* b, uint64_t lb, Fr* out, uint64_t out_len) {
  int launches = 0;
  uint64_t full = la + lb - 1;
  uint32_t lg = log2_ceil(full);
  uint64_t N = uint64_t(1) << lg;
  Fr* fa = g_arena.alloc(N);
  Fr* fb = (a == b && la == lb) ? fa : g_arena.alloc(N);
  Fr* scratch = g_arena.alloc(N);
  CUDA_CHECK(cudaMemcpyAsync(fa, a, la * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
  CUDA_CHECK(cudaMemsetAsync(fa + la, 0, (N - la) * sizeof(Fr), c.stream));
  FrBytes w = omega_for(lg);
  launches += ntt_device(c, fa, scratch, lg, w, false, nullptr);
  if (fb != fa) {
    CUDA_CHECK(cudaMemcpyAsync(fb, b, lb * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
    CUDA_CHECK(cudaMemsetAsync(fb + lb, 0, (N - lb) * sizeof(Fr), c.stream));
    launches += ntt_device(c, fb, scratch, lg, w, false, nullptr);
  }
  fr_mul_inplace_kernel<<<GRID_1D(N)>>>(fa, fb, N);
  CUDA_CHECK_LAUNCH();
  launches++;
  launches += ntt_device(c, fa, scratch, lg, w, true, nullptr);
  uint64_t take = out_len < full ? out_len : full;
  CUDA_CHECK(cudaMemcpyAsync(out, fa, take * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
  if (out_len > full) CUDA_CHECK(cudaMemsetAsync(out + full, 0, (out_len - full) * sizeof(Fr), c.stream));
  if (fb != fa) g_arena.free(fb);
  g_arena.free(fa);
  g_arena.free(scratch);
  return launches;
}

// out[0..out_len) = (a * b)[0..out_len) where b (lb coefficients) is given by its forward transform `bhat` of
// size 2^lg >= la + lb - 1 (a fixed operand: the transform is computed once and kept by the caller).
static int poly_mul_cached_dev(Context& c, const Fr* a, uint64_t la, const Fr* bhat, uint64_t lb, uint32_t lg, Fr* out,
                               uint64_t out_len) {
  int launches = 0;
  uint64_t full = la + lb - 1;
  uint64_t N = uint64_t(1) << lg;
  Fr* fa = g_arena.alloc(N);
  Fr* scratch = g_arena.alloc(N);
  CUDA_CHECK(cudaMemcpyAsync(fa, a, la * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
  CUDA_CHECK(cudaMemsetAsync(fa + la, 0, (N - la) * sizeof(Fr), c.stream));
  FrBytes w = omega_for(lg);
  launches += ntt_device(c, fa, scratch, lg, w, false, nullptr);
  fr_mul_inplace_kernel<<<GRID_1D(N)>>>(fa, bhat, N);
  CUDA_CHECK_LAUNCH();
  launches++;
  launches += ntt_device(c, fa, scratch, lg, w, true, nullptr);
  uint64_t take = out_len < full ? out_len : full;
  CUDA_CHECK(cudaMemcpyAsync(out, fa, take * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
  if (out_len > full) CUDA_CHECK(cudaMemsetAsync(out + full, 0, (out_len - full) * sizeof(Fr), c.stream));
  g_arena.free(fa);
  g_arena.free(scratch);
  return launches;
}

// g = f^-1 mod x^m by Newton iteration (f[0] != 0); f has lf coefficients.  g: m elements.
static int series_inverse_dev(Context& c, const Fr* f, uint64_t lf, uint64_t m, Fr* g) {
  int launches = 0;
  fr_inv_single_kernel<<<1, 32, 0, c.stream>>>(f, g);
  CUDA_CHECK_LAUNCH();
  launches++;
  uint64_t k = 1;
  Fr* t = g_arena.alloc(2 * m + 2);
  Fr* g2 = g_arena.alloc(2 * m + 2);
  while (k < m) {
    uint64_t k2 = 2 * k < m ? 2 * k : m;
    uint64_t fl = lf < k2 ? lf : k2;
    launches += poly_mul_dev(c, f, fl, g, k, t, k2);  // t = f*g mod x^k2
    fr_two_minus_kernel<<<GRID_1D(k2)>>>(t, k2);
    CUDA_CHECK_LAUNCH();
    launches++;
    launches += poly_mul_dev(c, g, k, t, k2, g2, k2);  // g2 = g*(2 - f g) mod x^k2
    CUDA_CHECK(cudaMemcpyAsync(g, g2, k2 * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
    k = k2;
  }
  return launches;
}

// a = b*q + r.  a (la), b (lb >= 1, b[lb-1] != 0), la >= lb.  q: la-lb+1 elements, r: lb-1 elements.
// All device Montgomery.  vanishing: b is x^(lb-1) - 1 (fast path).
// inv_cache: optional persistent buffer holding rev(b)^-1 mod x^m from an earlier call with the same
// divisor (the Groth16 Z(x) is fixed per circuit); *inv_cached tells whether it is already filled.
// inv_hat: optional buffer of 2^log2_ceil(2m - 1) elements next to inv_cache that keeps the forward
// transform of the cached inverse (one transform less per division by the same divisor).
static int poly_divmod_dev(Context& c, const Fr* a, uint64_t la, const Fr* b, uint64_t lb, Fr* q, Fr* r, bool vanishing,
                           Fr* inv_cache = nullptr, bool* inv_cached = nullptr, Fr* inv_hat = nullptr) {
  int launches = 0;
  uint64_t m = la - lb + 1;
  if (vanishing && lb >= 2) {
    uint64_t n = lb - 1;
    fr_div_vanishing_kernel<<<GRID_1D(n)>>>(a, la, n, q, m, r);
    CUDA_CHECK_LAUNCH();
    return 1;
  }
  Fr* ra = g_arena.alloc(m);
  uint64_t lrb = lb < m ? lb : m;
  Fr* rb = g_arena.alloc(lrb);
  Fr* g = inv_cache ? inv_cache : g_arena.alloc(m);
  Fr* qr = g_arena.alloc(m);
  fr_reverse_kernel<<<GRID_1D(m)>>>(a, la, m, ra);
  CUDA_CHECK_LAUNCH();
  fr_reverse_kernel<<<GRID_1D(lrb)>>>(b, lb, lrb, rb);
  CUDA_CHECK_LAUNCH();
  launches += 2;
  const uint32_t lg_q = log2_ceil(2 * m - 1);
  if (!(inv_cached && *inv_cached)) {
    launches += series_inverse_dev(c, rb, lrb, m, g);
    if (inv_cached) *inv_cached = true;
    if (inv_hat) {
      uint64_t N = uint64_t(1) << lg_q;
      Fr* scratch = g_arena.alloc(N);
      CUDA_CHECK(cudaMemcpyAsync(inv_hat, g, m * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
      CUDA_CHECK(cudaMemsetAsync(inv_hat + m, 0, (N - m) * sizeof(Fr), c.stream));
      launches += ntt_device(c, inv_hat, scratch, lg_q, omega_for(lg_q), false, nullptr);
      g_arena.free(scratch);
    }
  }
  if (inv_hat) launches += poly_mul_cached_dev(c, ra, m, inv_hat, m, lg_q, qr, m);
  else launches += poly_mul_dev(c, ra, m, g, m, qr, m);
  fr_reverse_kernel<<<GRID_1D(m)>>>(qr, m, m, q);
  CUDA_CHECK_LAUNCH();
  launches++;
  if (lb >= 2 && r) {  // r == nullptr: the caller only wants the quotient
    // r = (a - b q) mod (x^N - 1), N >= lb-1: exact because deg r < lb-1 <= N
    uint64_t lr = lb - 1;
    uint32_t lg = log2_ceil(lr);
    uint64_t N = uint64_t(1) << lg;
    Fr* fa = g_arena.alloc(N);
    Fr* fb = g_arena.alloc(N);
    Fr* fq = g_arena.alloc(N);
    Fr* scratch = g_arena.alloc(N);
    fr_fold_kernel<<<GRID_1D(N)>>>(a, la, N, fa);
    CUDA_CHECK_LAUNCH();
    fr_fold_kernel<<<GRID_1D(N)>>>(b, lb, N, fb);
    CUDA_CHECK_LAUNCH();
    fr_fold_kernel<<<GRID_1D(N)>>>(q, m, N, fq);
    CUDA_CHECK_LAUNCH();
    launches += 3;
    FrBytes w = omega_for(lg);
    launches += ntt_device(c, fb, scratch, lg, w, false, nullptr);
    launches += ntt_device(c, fq, scratch, lg, w, false, nullptr);
    fr_mul_inplace_kernel<<<GRID_1D(N)>>>(fb, fq, N);
    CUDA_CHECK_LAUNCH();
    launches += ntt_device(c, fb, scratch, lg, w, true, nullptr);
    fr_sub_inplace_kernel<<<GRID_1D(N)>>>(fa, fb, N);
    CUDA_CHECK_LAUNCH();
    launches += 2;
    CUDA_CHECK(cudaMemcpyAsync(r, fa, lr * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
  }
  return launches;
}

// upload canonical host bytes -> device Montgomery
static Fr* upload_mont(Context& c, const uint8_t* host, uint64_t n, int* launches) {
  Fr* d = g_arena.alloc(n);
  if (n) {
    CUDA_CHECK(cudaMemcpyAsync(d, host, n * 32, cudaMemcpyHostToDevice, c.stream));
    fr_to_mont_kernel<<<GRID_1D(n)>>>(d, n, d);
    CUDA_CHECK_LAUNCH();
    (*launches)++;
  }
  return d;
}
static void download_canon(Context& c, Fr* d, uint64_t n, uint8_t* host, int* launches) {
  if (!n) return;
  fr_from_mont_kernel<<<GRID_1D(n)>>>(d, n, d);
  CUDA_CHECK_LAUNCH();
  (*launches)++;
  CUDA_CHECK(cudaMemcpyAsync(host, d, n * 32, cudaMemcpyDeviceToHost, c.stream));
}

static bool host_is_vanishing(const uint8_t* b, uint64_t lb) {
  if (lb < 2) return false;
  uint8_t minus_one[32], one[32] = {1};
  memcpy(minus_one, FrParams::MOD, 32);
  minus_one[0] -= 1;  // r - 1: low byte of r is 0x01
  if (memcmp(b, minus_one, 32) != 0 || memcmp(b + (lb - 1) * 32, one, 32) != 0) return false;
  for (uint64_t i = 1; i + 1 < lb; i++) {
    const uint64_t* p = reinterpret_cast<const uint64_t*>(b + i * 32);
    if (p[0] | p[1] | p[2] | p[3]) return false;
  }
  return true;
}
static bool host_is_zero32(const uint8_t* p) {
  for (int i = 0; i < 32; i++)
    if (p[i]) return false;
  return true;
}

}  // namespace zkp

using namespace zkp;

extern "C" {

int zkp_fr_vec_op(int op, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out) {
  return guarded([&](Context& c) {
    if (op < 0 || op > 3 || (n && (!a || !b || !out))) throw InvalidArgument("zkp_fr_vec_op: bad argument");
    if (!n) return;
    ArenaScope scope;
    Fr* da = g_arena.alloc(n);
    uint64_t nb = op == 3 ? 1 : n;
    Fr* db = g_arena.alloc(nb);
    CUDA_CHECK(cudaMemcpyAsync(da, a, n * 32, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(db, b, nb * 32, cudaMemcpyHostToDevice, c.stream));
    fr_vec_op_kernel<<<GRID_1D(n)>>>(op, da, db, n, da);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out, da, n * 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_batch_inverse(const uint8_t* a, uint64_t n, uint8_t* out) {
  return guarded([&](Context& c) {
    if (n && (!a || !out)) throw InvalidArgument("zkp_fr_batch_inverse: null argument");
    if (!n) return;
    ArenaScope scope;
    Fr* da = g_arena.alloc(n);
    Fr* dout = g_arena.alloc(n);
    CUDA_CHECK(cudaMemcpyAsync(da, a, n * 32, cudaMemcpyHostToDevice, c.stream));
    uint64_t T = (n + BATCH_INV_CHUNK - 1) / BATCH_INV_CHUNK;
    fr_batch_inverse_kernel<<<ceil_div(T, 128), 128, 0, c.stream>>>(da, n, T, 0, dout);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out, dout, n * 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_prefix_product(const uint8_t* a, uint64_t n, uint8_t* out) {
  return guarded([&](Context& c) {
    if (n && (!a || !out)) throw InvalidArgument("zkp_fr_prefix_product: null argument");
    if (!n) return;
    ArenaScope scope;
    Fr* da = g_arena.alloc(n);
    Fr* dout = g_arena.alloc(n);
    CUDA_CHECK(cudaMemcpyAsync(da, a, n * 32, cudaMemcpyHostToDevice, c.stream));
    c.launches += scan_dev<false>(c, da, n, dout, nullptr);
    CUDA_CHECK(cudaMemcpyAsync(out, dout, n * 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_poly_eval(const uint8_t* coeffs, uint64_t n, const uint8_t x[32], uint8_t out[32]) {
  return guarded([&](Context& c) {
    if (!x || !out || (n && !coeffs)) throw InvalidArgument("zkp_fr_poly_eval: null argument");
    if (!n) {
      memset(out, 0, 32);
      return;
    }
    ArenaScope scope;
    Fr* dc = g_arena.alloc(n);
    Fr* res = g_arena.alloc(1);
    CUDA_CHECK(cudaMemcpyAsync(dc, coeffs, n * 32, cudaMemcpyHostToDevice, c.stream));
    c.launches += poly_eval_dev_impl(c, dc, n, x, res);
    CUDA_CHECK(cudaMemcpyAsync(out, res, 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_vec_matrix(const uint8_t* vec, const uint8_t* mat, uint64_t rows, uint64_t cols, uint8_t* out) {
  return guarded([&](Context& c) {
    if (!rows || !cols) return;
    if (!vec || !mat || !out) throw InvalidArgument("zkp_fr_vec_matrix: null argument");
    ArenaScope scope;
    Fr* dv = g_arena.alloc(rows);
    Fr* dm = g_arena.alloc(rows * cols);
    Fr* dout = g_arena.alloc(cols);
    CUDA_CHECK(cudaMemcpyAsync(dv, vec, rows * 32, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(dm, mat, rows * cols * 32, cudaMemcpyHostToDevice, c.stream));
    fr_vec_matrix_kernel<<<GRID_1D(cols)>>>(dv, dm, rows, cols, dout);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out, dout, cols * 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_poly_mul(const uint8_t* a, uint64_t a_len, const uint8_t* b, uint64_t b_len, uint8_t* out) {
  return guarded([&](Context& c) {
    if (!a_len || !b_len || !a || !b || !out) throw InvalidArgument("zkp_fr_poly_mul: empty or null operand");
    ArenaScope scope;
    int launches = 0;
    Fr* da = upload_mont(c, a, a_len, &launches);
    Fr* db = upload_mont(c, b, b_len, &launches);
    uint64_t lo = a_len + b_len - 1;
    Fr* dout = g_arena.alloc(lo);
    launches += poly_mul_dev(c, da, a_len, db, b_len, dout, lo);
    download_canon(c, dout, lo, out, &launches);
    c.launches += launches;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_poly_divmod(const uint8_t* a, uint64_t a_len, const uint8_t* b, uint64_t b_len, uint8_t* q_out,
                       uint8_t* r_out) {
  return guarded([&](Context& c) {
    if (!a || !b || !q_out || !b_len || a_len < b_len) throw InvalidArgument("zkp_fr_poly_divmod: need a_len >= b_len >= 1");
    if (b_len > 1 && !r_out) throw InvalidArgument("zkp_fr_poly_divmod: null remainder buffer");
    if (host_is_zero32(b + (b_len - 1) * 32)) throw InvalidArgument("zkp_fr_poly_divmod: leading coefficient of the divisor is zero");
    ArenaScope scope;
    int launches = 0;
    bool van = host_is_vanishing(b, b_len);
    Fr* da = upload_mont(c, a, a_len, &launches);
    Fr* db = upload_mont(c, b, b_len, &launches);
    uint64_t m = a_len - b_len + 1;
    Fr* dq = g_arena.alloc(m);
    Fr* dr = g_arena.alloc(b_len);
    launches += poly_divmod_dev(c, da, a_len, db, b_len, dq, dr, van);
    download_canon(c, dq, m, q_out, &launches);
    download_canon(c, dr, b_len - 1, r_out, &launches);
    c.launches += launches;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

// ------------------------------------------------------------------ device-resident Fr vectors (handles)
struct DivisorCache {
  uint64_t z_handle = 0, z_len = 0, m = 0;
  DevBuf inv, inv_hat;  // rev(Z)^-1 mod x^m and its forward transform
  bool filled = false;
};
static DivisorCache g_div_cache;

int zkp_scalars_alloc(uint64_t n, uint64_t* handle) {
  return guarded([&](Context& c) {
    if (!handle) throw InvalidArgument("zkp_scalars_alloc: null handle");
    auto r = std::make_unique<Resource>();
    r->kind = HandleKind::Scalars;
    r->n = n;
    r->buf.reserve_pooled(n ? n * 32 : 32);
    CUDA_CHECK(cudaMemsetAsync(r->buf.p, 0, n ? n * 32 : 32, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *handle = registry().put(std::move(r));
  });
}

int zkp_scalars_copy(uint64_t dst, uint64_t dst_off, uint64_t src, uint64_t src_off, uint64_t n) {
  return guarded([&](Context& c) {
    Resource* d = need(dst, HandleKind::Scalars, "zkp_scalars_copy");
    Resource* s = need(src, HandleKind::Scalars, "zkp_scalars_copy");
    if (!range_ok(dst_off, n, d->n) || !range_ok(src_off, n, s->n)) throw InvalidArgument("zkp_scalars_copy: range out of bounds");
    if (n) CUDA_CHECK(cudaMemcpyAsync(d->buf.as<Fr>() + dst_off, s->buf.as<Fr>() + src_off, n * 32,
                                     cudaMemcpyDeviceToDevice, c.stream));
  });
}

int zkp_scalars_upload(uint64_t dst, uint64_t dst_off, const uint8_t* host, uint64_t n) {
  return guarded([&](Context& c) {
    Resource* d = need(dst, HandleKind::Scalars, "zkp_scalars_upload");
    if (!range_ok(dst_off, n, d->n) || (n && !host)) throw InvalidArgument("zkp_scalars_upload: bad range or null source");
    if (n) CUDA_CHECK(cudaMemcpyAsync(d->buf.as<Fr>() + dst_off, host, n * 32, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_scalars_scale(uint64_t h, uint64_t off, uint64_t n, const uint8_t k[32]) {
  return guarded([&](Context& c) {
    Resource* d = need(h, HandleKind::Scalars, "zkp_scalars_scale");
    if (!range_ok(off, n, d->n) || !k) throw InvalidArgument("zkp_scalars_scale: bad range or null factor");
    if (!n) return;
    ArenaScope scope;
    Fr* dk = g_arena.alloc(1);
    CUDA_CHECK(cudaMemcpyAsync(dk, k, 32, cudaMemcpyHostToDevice, c.stream));
    fr_vec_op_kernel<<<GRID_1D(n)>>>(3, d->buf.as<Fr>() + off, dk, n, d->buf.as<Fr>() + off);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_fr_poly_eval_dev(uint64_t h, uint64_t off, uint64_t n, const uint8_t x[32], uint8_t out[32]) {
  return guarded([&](Context& c) {
    Resource* d = need(h, HandleKind::Scalars, "zkp_fr_poly_eval_dev");
    if (!range_ok(off, n, d->n) || !x || !out) throw InvalidArgument("zkp_fr_poly_eval_dev: bad argument");
    if (!n) {
      memset(out, 0, 32);
      return;
    }
    ArenaScope scope;
    Fr* res = g_arena.alloc(1);
    c.launches += poly_eval_dev_impl(c, d->buf.as<Fr>() + off, n, x, res);
    CUDA_CHECK(cudaMemcpyAsync(out, res, 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

// hxr on device-resident coefficient vectors (SURVEY F12: the 2^20 configuration needs
// coefficient-level entry points).  a, b, c: `len` canonical coefficients each; z: z_len coefficients of
// the (fixed) divisor.  Creates two new scalar handles: the quotient (2*len - z_len coefficients) and
// the remainder (z_len - 1).  The power-series inverse of the reversed divisor is cached per z handle.
int zkp_groth16_quotient_dev(uint64_t a, uint64_t b, uint64_t cc, uint64_t len, uint64_t z, uint64_t z_len,
                             uint64_t* h_out, uint64_t* rem_out) {
  return guarded([&](Context& c) {
    Resource* ra = need(a, HandleKind::Scalars, "zkp_groth16_quotient_dev");
    Resource* rb = need(b, HandleKind::Scalars, "zkp_groth16_quotient_dev");
    Resource* rc = need(cc, HandleKind::Scalars, "zkp_groth16_quotient_dev");
    Resource* rz = need(z, HandleKind::Scalars, "zkp_groth16_quotient_dev");
    if (!h_out || !len || z_len < 2) throw InvalidArgument("zkp_groth16_quotient_dev: bad argument");
    if (len > ra->n || len > rb->n || len > rc->n || z_len > rz->n) throw InvalidArgument("zkp_groth16_quotient_dev: length exceeds a vector");
    uint64_t lp = 2 * len - 1;
    if (lp < z_len) throw InvalidArgument("zkp_groth16_quotient_dev: divisor longer than the product");
    ArenaScope scope;
    int launches = 0;
    auto to_mont_copy = [&](Resource* r, uint64_t n) {
      Fr* d = g_arena.alloc(n);
      fr_to_mont_kernel<<<GRID_1D(n)>>>(r->buf.as<Fr>(), n, d);
      CUDA_CHECK_LAUNCH();
      launches++;
      return d;
    };
    Fr* da = to_mont_copy(ra, len);
    Fr* db = to_mont_copy(rb, len);
    Fr* dc = to_mont_copy(rc, len);
    Fr* dz = to_mont_copy(rz, z_len);
    Fr* dp = g_arena.alloc(lp);
    launches += poly_mul_dev(c, da, len, db, len, dp, lp);
    fr_sub_inplace_kernel<<<GRID_1D(len)>>>(dp, dc, len);
    CUDA_CHECK_LAUNCH();
    launches++;
    uint64_t m = lp - z_len + 1;
    if (g_div_cache.z_handle != z || g_div_cache.z_len != z_len || g_div_cache.m != m) {
      g_div_cache.z_handle = z;
      g_div_cache.z_len = z_len;
      g_div_cache.m = m;
      g_div_cache.filled = false;
      g_div_cache.inv.reserve(m * sizeof(Fr));
      g_div_cache.inv_hat.reserve((size_t(1) << log2_ceil(2 * m - 1)) * sizeof(Fr));
    }
    auto hq = std::make_unique<Resource>();
    hq->kind = HandleKind::Scalars;
    hq->n = m;
    hq->buf.reserve_pooled(m * 32);
    // rem_out == NULL: the prover only needs H (the remainder of a satisfied instance is zero and costs
    // three more transforms to compute)
    std::unique_ptr<Resource> hr;
    if (rem_out) {
      hr = std::make_unique<Resource>();
      hr->kind = HandleKind::Scalars;
      hr->n = z_len - 1;
      hr->buf.reserve_pooled(z_len * 32);
    }
    launches += poly_divmod_dev(c, dp, lp, dz, z_len, hq->buf.as<Fr>(), hr ? hr->buf.as<Fr>() : nullptr, false,
                                g_div_cache.inv.as<Fr>(), &g_div_cache.filled, g_div_cache.inv_hat.as<Fr>());
    fr_from_mont_kernel<<<GRID_1D(m)>>>(hq->buf.as<Fr>(), m, hq->buf.as<Fr>());
    CUDA_CHECK_LAUNCH();
    launches++;
    if (hr) {
      fr_from_mont_kernel<<<GRID_1D(z_len - 1)>>>(hr->buf.as<Fr>(), z_len - 1, hr->buf.as<Fr>());
      CUDA_CHECK_LAUNCH();
      launches++;
    }
    c.launches += launches;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *h_out = registry().put(std::move(hq));
    if (hr) *rem_out = registry().put(std::move(hr));
  });
}

// ------------------------------------------------------------------ handle-based vector API (PLONK at scale)
static Fr fr_from_bytes(const uint8_t* b) {
  Fr x;
  memcpy(x.v, b, 32);
  return x;
}
static Fr* hptr(uint64_t h, uint64_t off, uint64_t n, const char* what) {
  Resource* r = need(h, HandleKind::Scalars, what);
  if (!range_ok(off, n, r->n)) throw InvalidArgument(std::string(what) + ": range out of bounds");
  return r->buf.as<Fr>() + off;
}
// canonical constant -> Montgomery on the device (one tiny kernel + 32-byte read back)
static Fr host_to_mont(Context& c, const uint8_t* k) {
  Fr* d = g_arena.alloc(1);
  CUDA_CHECK(cudaMemcpyAsync(d, k, 32, cudaMemcpyHostToDevice, c.stream));
  fr_to_mont_kernel<<<1, 32, 0, c.stream>>>(d, 1, d);
  CUDA_CHECK_LAUNCH();
  Fr out;
  CUDA_CHECK(cudaMemcpyAsync(&out, d, 32, cudaMemcpyDeviceToHost, c.stream));
  CUDA_CHECK(cudaStreamSynchronize(c.stream));
  c.launches++;
  return out;
}

int zkp_fr_vec_op_dev(int op, uint64_t dst, uint64_t dst_off, uint64_t a, uint64_t a_off, uint64_t b, uint64_t b_off,
                      uint64_t n) {
  return guarded([&](Context& c) {
    if (op < 0 || op > 2) throw InvalidArgument("zkp_fr_vec_op_dev: op must be 0 (add), 1 (sub) or 2 (mul)");
    if (!n) return;
    Fr* d = hptr(dst, dst_off, n, "zkp_fr_vec_op_dev");
    Fr* pa = hptr(a, a_off, n, "zkp_fr_vec_op_dev");
    Fr* pb = hptr(b, b_off, n, "zkp_fr_vec_op_dev");
    fr_vec_op_kernel<<<GRID_1D(n)>>>(op, pa, pb, n, d);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_fr_axpy_dev(uint64_t dst, uint64_t dst_off, const uint8_t k[32], uint64_t src, uint64_t src_off, uint64_t n) {
  return guarded([&](Context& c) {
    if (!k) throw InvalidArgument("zkp_fr_axpy_dev: null factor");
    if (!n) return;
    ArenaScope scope;
    Fr* d = hptr(dst, dst_off, n, "zkp_fr_axpy_dev");
    Fr* s = hptr(src, src_off, n, "zkp_fr_axpy_dev");
    Fr km = host_to_mont(c, k);
    fr_axpy_kernel<<<GRID_1D(n)>>>(d, km, s, n);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_scalars_add_const(uint64_t h, uint64_t off, uint64_t n, const uint8_t k[32]) {
  return guarded([&](Context& c) {
    if (!k) throw InvalidArgument("zkp_scalars_add_const: null constant");
    if (!n) return;
    Fr* d = hptr(h, off, n, "zkp_scalars_add_const");
    fr_add_const_kernel<<<GRID_1D(n)>>>(d, fr_from_bytes(k), n);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_scalars_fill_powers(uint64_t h, uint64_t off, uint64_t n, const uint8_t first[32], const uint8_t base[32]) {
  return guarded([&](Context& c) {
    if (!first || !base) throw InvalidArgument("zkp_scalars_fill_powers: null argument");
    if (!n) return;
    Fr* d = hptr(h, off, n, "zkp_scalars_fill_powers");
    FrBytes bb;
    memcpy(bb.b, base, 32);
    int launches = 0;
    if (n > (uint64_t(1) << 28)) throw InvalidArgument("zkp_scalars_fill_powers: n must be <= 2^28");
    const Fr* tab = power_table(c, bb, false, log2_ceil(n), &launches);
    fr_fill_powers_kernel<<<GRID_1D(n)>>>(d, n, fr_from_bytes(first), tab);
    CUDA_CHECK_LAUNCH();
    c.launches += launches + 1;
  });
}

int zkp_scalars_convert(uint64_t h, uint64_t off, uint64_t n, int to_montgomery) {
  return guarded([&](Context& c) {
    if (!n) return;
    Fr* d = hptr(h, off, n, "zkp_scalars_convert");
    if (to_montgomery) fr_to_mont_kernel<<<GRID_1D(n)>>>(d, n, d);
    else fr_from_mont_kernel<<<GRID_1D(n)>>>(d, n, d);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_scalars_is_zero(uint64_t h, uint64_t off, uint64_t n, int* out_all_zero) {
  return guarded([&](Context& c) {
    if (!out_all_zero) throw InvalidArgument("zkp_scalars_is_zero: null output");
    *out_all_zero = 1;
    if (!n) return;
    ArenaScope scope;
    Fr* d = hptr(h, off, n, "zkp_scalars_is_zero");
    int* flag = reinterpret_cast<int*>(g_arena.alloc(1));
    int one = 1;
    CUDA_CHECK(cudaMemcpyAsync(flag, &one, 4, cudaMemcpyHostToDevice, c.stream));
    fr_is_zero_kernel<<<GRID_1D(n)>>>(d, n, flag);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaMemcpyAsync(out_all_zero, flag, 4, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_batch_inverse_dev(uint64_t h, uint64_t off, uint64_t n, int montgomery) {
  return guarded([&](Context& c) {
    if (!n) return;
    ArenaScope scope;
    Fr* d = hptr(h, off, n, "zkp_fr_batch_inverse_dev");
    Fr* tmp = g_arena.alloc(n);
    uint64_t T = (n + BATCH_INV_CHUNK - 1) / BATCH_INV_CHUNK;
    fr_batch_inverse_kernel<<<ceil_div(T, 128), 128, 0, c.stream>>>(d, n, T, montgomery ? 1 : 0, tmp);
    CUDA_CHECK_LAUNCH();
    CUDA_CHECK(cudaMemcpyAsync(d, tmp, n * 32, cudaMemcpyDeviceToDevice, c.stream));
    c.launches++;
  });
}

int zkp_fr_poly_eval_multi_dev(uint32_t count, const uint64_t* handles, const uint64_t* offs, const uint64_t* lens,
                               const uint8_t* xs, uint8_t* out) {
  return guarded([&](Context& c) {
    if (count == 0) return;
    if (count > (uint32_t)MULTI_MAX || !handles || !offs || !lens || !xs || !out)
      throw InvalidArgument("zkp_fr_poly_eval_multi_dev: 1..16 items, no null arguments");
    ArenaScope scope;
    MultiEvalArgs a;
    std::vector<FrBytes> points;
    uint64_t max_n = 1;
    for (uint32_t k = 0; k < count; k++) {
      if (!lens[k]) throw InvalidArgument("zkp_fr_poly_eval_multi_dev: empty polynomial");
      a.coeffs[k] = hptr(handles[k], offs[k], lens[k], "zkp_fr_poly_eval_multi_dev");
      a.n[k] = lens[k];
      if (lens[k] > max_n) max_n = lens[k];
      FrBytes x;
      memcpy(x.b, xs + 32 * k, 32);
      size_t p = 0;
      while (p < points.size() && !(points[p] == x)) p++;
      if (p == points.size()) points.push_back(x);
      a.point[k] = (int)p;
    }
    int levels = 0;
    for (uint64_t m = max_n; m > 1; m = (m + HORNER_CHUNK - 1) / HORNER_CHUNK) levels++;
    if (levels == 0) levels = 1;
    Fr* xc = g_arena.alloc(points.size());
    Fr* xp = g_arena.alloc(points.size() * levels);
    CUDA_CHECK(cudaMemcpyAsync(xc, points.data(), points.size() * 32, cudaMemcpyHostToDevice, c.stream));
    horner_powers_multi_kernel<<<1, 32, 0, c.stream>>>(xc, (int)points.size(), xp, levels);
    CUDA_CHECK_LAUNCH();
    int launches = 1;
    const Fr* prev = nullptr;
    uint64_t stride_prev = 0, m = max_n;
    Fr* cur = nullptr;
    for (int l = 0; l < levels; l++) {
      uint64_t np = (m + HORNER_CHUNK - 1) / HORNER_CHUNK;
      cur = g_arena.alloc(np * count);
      dim3 grid((unsigned)ceil_div(np, (uint64_t)256), count);
      horner_multi_kernel<<<grid, 256, 0, c.stream>>>(a, l, levels, xp, prev, stride_prev, cur, np);
      CUDA_CHECK_LAUNCH();
      launches++;
      prev = cur;
      stride_prev = np;
      m = np;
    }
    // m == 1: the results are contiguous
    CUDA_CHECK(cudaMemcpyAsync(out, cur, (size_t)count * 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    c.launches += launches;
  });
}

int zkp_fr_lincomb_dev(uint64_t dst, uint64_t dst_off, uint64_t n, uint32_t count, const uint64_t* handles,
                       const uint64_t* offs, const uint64_t* lens, const uint8_t* coeffs) {
  return guarded([&](Context& c) {
    if (!n) return;
    if (count > (uint32_t)MULTI_MAX || (count && (!handles || !offs || !lens || !coeffs)))
      throw InvalidArgument("zkp_fr_lincomb_dev: at most 16 items, no null arguments");
    ArenaScope scope;
    Fr* d = hptr(dst, dst_off, n, "zkp_fr_lincomb_dev");
    LinCombArgs a;
    a.count = (int)count;
    if (count) {
      // coefficients -> Montgomery on the device in one go
      Fr* dk = g_arena.alloc(count);
      CUDA_CHECK(cudaMemcpyAsync(dk, coeffs, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
      fr_to_mont_kernel<<<1, 32, 0, c.stream>>>(dk, count, dk);
      CUDA_CHECK_LAUNCH();
      CUDA_CHECK(cudaMemcpyAsync(a.coeff, dk, (size_t)count * 32, cudaMemcpyDeviceToHost, c.stream));
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
      c.launches++;
    }
    for (uint32_t k = 0; k < count; k++) {
      if (lens[k] > n) throw InvalidArgument("zkp_fr_lincomb_dev: an item is longer than the destination");
      a.src[k] = hptr(handles[k], offs[k], lens[k], "zkp_fr_lincomb_dev");
      if (a.src[k] < d + n && d < a.src[k] + lens[k]) throw InvalidArgument("zkp_fr_lincomb_dev: destination overlaps a source");
      a.len[k] = lens[k];
    }
    fr_lincomb_kernel<<<GRID_1D(n)>>>(a, n, d);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

// <a, b> = sum_i a[i] * b[i] mod r of two device-resident canonical vectors.  The O(1)-host verification
// of an MSM over points with known discrete logs, sum_i k_i (s_i G) == (<k, s>) G (SURVEY 8d), at any size;
// also sum_i c_i x^i style evaluations against a powers vector.
int zkp_fr_dot_dev(uint64_t a, uint64_t a_off, uint64_t b, uint64_t b_off, uint64_t n, uint8_t out[32]) {
  return guarded([&](Context& c) {
    if (!out) throw InvalidArgument("zkp_fr_dot_dev: null output");
    if (!n) {
      memset(out, 0, 32);
      return;
    }
    ArenaScope scope;
    Fr* pa = hptr(a, a_off, n, "zkp_fr_dot_dev");
    Fr* pb = hptr(b, b_off, n, "zkp_fr_dot_dev");
    uint32_t blocks = ceil_div(n, DOT_THREADS);
    uint32_t cap = (uint32_t)c.sm_count * 8;
    if (blocks > cap) blocks = cap;
    Fr* partial = g_arena.alloc(blocks + 1);
    fr_dot_partial_kernel<<<blocks, DOT_THREADS, 0, c.stream>>>(pa, pb, n, partial);
    CUDA_CHECK_LAUNCH();
    fr_dot_final_kernel<<<1, DOT_THREADS, 0, c.stream>>>(partial, blocks, partial + blocks);
    CUDA_CHECK_LAUNCH();
    c.launches += 2;
    CUDA_CHECK(cudaMemcpyAsync(out, partial + blocks, 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

// exclusive scan: op 0 product (dst[0] = 1), 1 sum (dst[0] = 0); canonical values; dst must not overlap src
int zkp_fr_scan_dev(int op, uint64_t dst, uint64_t dst_off, uint64_t src, uint64_t src_off, uint64_t n) {
  return guarded([&](Context& c) {
    if (op != 0 && op != 1) throw InvalidArgument("zkp_fr_scan_dev: op must be 0 (product) or 1 (sum)");
    if (!n) return;
    ArenaScope scope;
    Fr* d = hptr(dst, dst_off, n, "zkp_fr_scan_dev");
    Fr* s = hptr(src, src_off, n, "zkp_fr_scan_dev");
    c.launches += op == 0 ? scan_dev<false>(c, s, n, d, nullptr) : scan_dev<true>(c, s, n, d, nullptr);
  });
}

// dst[0..n-1) = coefficients of (p(x) - p(zeta)) / (x - zeta) for p = src[0..n)   (poly_div by a linear
// factor, round5.py:165-171 / kzg.py:95-104), as scale-by-powers + one sum scan.  zeta != 0.
int zkp_fr_div_linear_dev(uint64_t src, uint64_t src_off, uint64_t n, const uint8_t zeta[32], uint64_t dst,
                          uint64_t dst_off) {
  return guarded([&](Context& c) {
    if (!zeta) throw InvalidArgument("zkp_fr_div_linear_dev: null zeta");
    if (n < 2) return;
    ArenaScope scope;
    Fr* p = hptr(src, src_off, n, "zkp_fr_div_linear_dev");
    Fr* q = hptr(dst, dst_off, n - 1, "zkp_fr_div_linear_dev");
    if (host_is_zero32(zeta)) {
      CUDA_CHECK(cudaMemcpyAsync(q, p + 1, (n - 1) * 32, cudaMemcpyDeviceToDevice, c.stream));
      return;
    }
    FrBytes zb;
    memcpy(zb.b, zeta, 32);
    int launches = 0;
    if (n > (uint64_t(1) << 28)) throw InvalidArgument("zkp_fr_div_linear_dev: n must be <= 2^28");
    const Fr* zp = power_table(c, zb, false, log2_ceil(n + 1), &launches);
    const Fr* zip = power_table(c, zb, true, log2_ceil(n + 1), &launches);
    Fr* d = g_arena.alloc(n);
    Fr* P = g_arena.alloc(n);
    Fr* T = g_arena.alloc(1);
    CUDA_CHECK(cudaMemcpyAsync(d, p, n * 32, cudaMemcpyDeviceToDevice, c.stream));
    fr_scale_powers_kernel<<<GRID_1D(n)>>>(d, n, zp);
    CUDA_CHECK_LAUNCH();
    launches += 1 + scan_dev<true>(c, d, n, P, T);
    fr_div_linear_finish_kernel<<<GRID_1D(n - 1)>>>(d, P, T, zip, n - 1, q);
    CUDA_CHECK_LAUNCH();
    c.launches += launches + 1;
  });
}

int zkp_plonk_perm_terms_dev(uint64_t a, uint64_t b, uint64_t cc, uint64_t s1, uint64_t s2, uint64_t s3, uint64_t n,
                             const uint8_t omega[32], const uint8_t beta[32], const uint8_t gamma[32], uint64_t num,
                             uint64_t den) {
  return guarded([&](Context& c) {
    if (!omega || !beta || !gamma) throw InvalidArgument("zkp_plonk_perm_terms_dev: null scalar");
    if (!n) return;
    const char* w = "zkp_plonk_perm_terms_dev";
    FrBytes ob;
    memcpy(ob.b, omega, 32);
    int launches = 0;
    const Fr* tab = power_table(c, ob, false, log2_ceil(n), &launches);
    plonk_perm_terms_kernel<<<GRID_1D(n)>>>(hptr(a, 0, n, w), hptr(b, 0, n, w), hptr(cc, 0, n, w), hptr(s1, 0, n, w),
                                            hptr(s2, 0, n, w), hptr(s3, 0, n, w), n, tab, fr_from_bytes(beta),
                                            fr_from_bytes(gamma), hptr(num, 0, n, w), hptr(den, 0, n, w));
    CUDA_CHECK_LAUNCH();
    c.launches += launches + 1;
  });
}

// Static per-domain data of the quotient kernel: x (N = 8n coset points, Montgomery), l1f = 1/(n (x_i-1))
// (Montgomery), zh_inv (8 values at zh8[0..8)).  g = coset shift, w8 = primitive 8n-th root.
int zkp_plonk_coset_setup_dev(uint64_t n, uint32_t ext, const uint8_t g[32], const uint8_t w8[32],
                              const uint8_t g_pow_n[32], const uint8_t w8_pow_n[32], uint64_t x_out, uint64_t l1f_out,
                              uint64_t zh8_out) {
  return guarded([&](Context& c) {
    if (!g || !w8 || !g_pow_n || !w8_pow_n) throw InvalidArgument("zkp_plonk_coset_setup_dev: null scalar");
    const char* w = "zkp_plonk_coset_setup_dev";
    if (ext != 4 && ext != 8 && ext != 16) throw InvalidArgument("zkp_plonk_coset_setup_dev: ext must be 4, 8 or 16");
    uint64_t N = (uint64_t)ext * n;
    ArenaScope scope;
    Fr* x = hptr(x_out, 0, N, w);
    Fr* l1 = hptr(l1f_out, 0, N, w);
    Fr* zh = hptr(zh8_out, 0, ext, w);
    FrBytes wb;
    memcpy(wb.b, w8, 32);
    int launches = 0;
    const Fr* tab = pow2_table(c, wb, false, &launches);
    uint8_t nb[32] = {0};
    for (int i = 0; i < 8; i++) nb[i] = (uint8_t)(n >> (8 * i));
    plonk_coset_points_kernel<<<GRID_1D(N)>>>(N, fr_from_bytes(g), tab, fr_from_bytes(nb), x, l1);
    CUDA_CHECK_LAUNCH();
    Fr* tmp = g_arena.alloc(N);
    uint64_t T = (N + BATCH_INV_CHUNK - 1) / BATCH_INV_CHUNK;
    fr_batch_inverse_kernel<<<ceil_div(T, 128), 128, 0, c.stream>>>(l1, N, T, 1, tmp);
    CUDA_CHECK_LAUNCH();
    CUDA_CHECK(cudaMemcpyAsync(l1, tmp, N * 32, cudaMemcpyDeviceToDevice, c.stream));
    plonk_zh_inv_kernel<<<1, 32, 0, c.stream>>>(fr_from_bytes(g_pow_n), fr_from_bytes(w8_pow_n), ext, zh);
    CUDA_CHECK_LAUNCH();
    c.launches += launches + 3;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

// evals: 12 handles in the order a, b, c, z, q_l, q_r, q_o, q_m, q_c, s_sigma1, s_sigma2, s_sigma3 (8n
// Montgomery coset evaluations each); writes the quotient's coset evaluations (Montgomery) to t_out.
int zkp_plonk_quotient_dev(const uint64_t evals[12], uint64_t n, uint32_t ext, uint64_t x, uint64_t l1f, uint64_t zh8,
                           const uint8_t beta[32], const uint8_t gamma[32], const uint8_t alpha[32], uint64_t t_out) {
  return guarded([&](Context& c) {
    if (!evals || !beta || !gamma || !alpha) throw InvalidArgument("zkp_plonk_quotient_dev: null argument");
    const char* w = "zkp_plonk_quotient_dev";
    if (ext != 4 && ext != 8 && ext != 16) throw InvalidArgument("zkp_plonk_quotient_dev: ext must be 4, 8 or 16");
    uint64_t N = (uint64_t)ext * n;
    if (N & (N - 1)) throw InvalidArgument("zkp_plonk_quotient_dev: n must be a power of two");
    if (N < 3 * n + 6) throw InvalidArgument("zkp_plonk_quotient_dev: coset too small for the quotient degree");
    PlonkQuotArgs q;
    const Fr** slots[12] = {&q.a, &q.b, &q.c, &q.z, &q.ql, &q.qr, &q.qo, &q.qm, &q.qc, &q.s1, &q.s2, &q.s3};
    for (int k = 0; k < 12; k++) *slots[k] = hptr(evals[k], 0, N, w);
    q.x = hptr(x, 0, N, w);
    q.l1f = hptr(l1f, 0, N, w);
    q.zh_inv = hptr(zh8, 0, ext, w);
    q.ext = ext;
    q.beta = fr_from_bytes(beta);
    q.gamma = fr_from_bytes(gamma);
    q.alpha = fr_from_bytes(alpha);
    q.N = N;
    q.t = hptr(t_out, 0, N, w);
    plonk_quotient_kernel<<<ceil_div(N, 128), 128, 0, c.stream>>>(q);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_groth16_quotient(const uint8_t* a, const uint8_t* b, const uint8_t* cc, uint64_t len, const uint8_t* z,
                         uint64_t z_len, uint8_t* h_out, uint8_t* rem_out) {
  return guarded([&](Context& c) {
    if (!a || !b || !cc || !z || !h_out || !len || !z_len) throw InvalidArgument("zkp_groth16_quotient: null/empty argument");
    uint64_t lp = 2 * len - 1;
    if (lp < z_len) throw InvalidArgument("zkp_groth16_quotient: divisor longer than the product");
    if (z_len > 1 && !rem_out) throw InvalidArgument("zkp_groth16_quotient: null remainder buffer");
    if (host_is_zero32(z + (z_len - 1) * 32)) throw InvalidArgument("zkp_groth16_quotient: leading coefficient of Z is zero");
    ArenaScope scope;
    int launches = 0;
    Fr* da = upload_mont(c, a, len, &launches);
    Fr* db = upload_mont(c, b, len, &launches);
    Fr* dc = upload_mont(c, cc, len, &launches);
    Fr* dz = upload_mont(c, z, z_len, &launches);
    Fr* dp = g_arena.alloc(lp);
    launches += poly_mul_dev(c, da, len, db, len, dp, lp);
    fr_sub_inplace_kernel<<<GRID_1D(len)>>>(dp, dc, len);  // P = a*b - c
    CUDA_CHECK_LAUNCH();
    launches++;
    uint64_t m = lp - z_len + 1;
    Fr* dq = g_arena.alloc(m);
    Fr* dr = g_arena.alloc(z_len);
    launches += poly_divmod_dev(c, dp, lp, dz, z_len, dq, dr, host_is_vanishing(z, z_len));
    download_canon(c, dq, m, h_out, &launches);
    download_canon(c, dr, z_len - 1, rem_out, &launches);
    c.launches += launches;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

}  // extern "C"

#include "qap.cuh"
#include "groth16_batch.cuh"
#include "plonk_batch.cuh"
#include "witness.cuh"
