// Batch PLONK proving: the vector work of `count` proofs of one circuit in the same launches
// (zkp/plonk/device_prover.py prove_batch).  Included once, by poly.cu, after groth16_batch.cuh: shares the arena,
// the scans, the Horner levels and the power tables.  Every proof has its own Fiat-Shamir challenges, so the per-round
// kernels read a count-long canonical array of each challenge instead of one scalar; segmented scans keep the proofs
// apart.  Every entry computes, per proof, exactly what its single-proof counterpart computes (exact field
// arithmetic: same values, whatever the launch shape).
#pragma once

namespace zkp {

// ------------------------------------------------------------------ blinding and restriding
// out[v * out_stride + i] = (i < n ? in[v * in_stride + i] : 0) - (i < k ? b_v[i] : 0) + (n <= i < n + k ? b_v[i - n] : 0):
// vector v's coefficients plus (b_v0 + b_v1 x + ...)(x^n - 1), the _blind of device_prover (round1.py:38-108,
// round2.py), written at the stride of its commitment.  b_v = blinds[v * k ..].  Canonical in and out.
__global__ void plonk_blind_many_kernel(const Fr* __restrict__ in, uint64_t in_stride, uint64_t n, uint32_t k,
                                        const Fr* __restrict__ blinds, uint64_t out_stride, uint64_t total,
                                        Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t v = idx / out_stride, i = idx % out_stride;
  Fr x = i < n ? in[v * in_stride + i] : Fr::zero();
  if (i < k) x = x - blinds[v * k + i];
  if (i >= n && i < n + k) x = x + blinds[v * k + (i - n)];
  out[idx] = x;
}

// The round-3 transform inputs of every proof: vector v < 3 count is wire v (n + 2 coefficients at stride n + 2),
// vector 3 count + j is z_j (n + 3 at stride n + 3), vector 4 count + j (when total covers it) is PI_j (n at stride
// n); each lands zero-padded and in Montgomery form in its own block of 2^log_N elements.
__global__ void plonk_coset_inputs_many_kernel(const Fr* __restrict__ wires, const Fr* __restrict__ z,
                                               const Fr* __restrict__ pi, uint64_t n, uint64_t count, uint32_t log_N,
                                               uint64_t total, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t v = idx >> log_N, i = idx & ((uint64_t(1) << log_N) - 1);
  Fr x = Fr::zero();
  if (v < 3 * count) {
    if (i < n + 2) x = wires[v * (n + 2) + i].to_mont();
  } else if (v < 4 * count) {
    if (i < n + 3) x = z[(v - 3 * count) * (n + 3) + i].to_mont();
  } else if (i < n) {
    x = pi[(v - 4 * count) * n + i].to_mont();
  }
  out[idx] = x;
}

// ------------------------------------------------------------------ public inputs
// out[j * n + i] = i < ell ? pub[j * stride + i] : 0: the evaluations of PI_j on H (utils.py:84-116), canonical
__global__ void plonk_pi_scatter_many_kernel(const Fr* __restrict__ pub, uint64_t stride, uint64_t ell, uint32_t log_n,
                                             uint64_t total, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx >> log_n, i = idx & ((uint64_t(1) << log_n) - 1);
  out[idx] = i < ell ? pub[j * stride + i] : Fr::zero();
}

// gap[j * ell + i] = n (zeta_j - w^i), Montgomery: the denominator of L_i(zeta_j), zero when zeta_j = w^i
__global__ void plonk_pi_gap_many_kernel(const Fr* __restrict__ zetas, const Fr* __restrict__ omega_tab, uint64_t ell,
                                         uint64_t n, uint64_t total, Fr* __restrict__ gap) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / ell, i = idx % ell;
  Fr nc = Fr::zero();
  nc.v[0] = (uint32_t)n;  // n <= 2^28
  gap[idx] = (zetas[j].to_mont() - power_at(omega_tab, (uint32_t)i)) * nc.to_mont();
}

// one block per proof: out_j = sum_{i < ell} x_j,i w^i (zeta_j^n - 1) / (n (zeta_j - w^i)) from the inverted gaps;
// a zero inverse marks zeta_j = w^i (at most one i per proof), and then out_j = x_j,i (utils.py lagrange_basis_eval)
__global__ void __launch_bounds__(DOT_THREADS) plonk_pi_eval_many_kernel(const Fr* __restrict__ pub, uint64_t stride,
                                                                          uint64_t ell, uint32_t log_n,
                                                                          const Fr* __restrict__ zetas,
                                                                          const Fr* __restrict__ omega_tab,
                                                                          const Fr* __restrict__ inv, Fr* __restrict__ out) {
  __shared__ Fr sm[DOT_THREADS];
  __shared__ uint64_t hit;
  const uint64_t j = blockIdx.x;
  if (threadIdx.x == 0) hit = ~uint64_t(0);
  __syncthreads();
  const Fr* x = pub + j * stride;
  const Fr* iv = inv + j * ell;
  Fr acc = Fr::zero();
  for (uint64_t i = threadIdx.x; i < ell; i += DOT_THREADS) {
    const Fr d = iv[i];
    if (d.is_zero()) hit = i;
    else acc = acc + x[i] * (power_at(omega_tab, (uint32_t)i) * d);  // canonical * Montgomery -> canonical
  }
  const Fr tot = dot_block_reduce(acc, sm);  // ends with a barrier: `hit` is visible
  if (threadIdx.x == 0) {
    if (hit != ~uint64_t(0)) {
      out[j] = x[hit];
    } else {
      Fr zn = zetas[j].to_mont();
      for (uint32_t k = 0; k < log_n; k++) zn = zn.sqr();
      out[j] = tot * (zn - Fr::one());
    }
  }
}

// plonk_perm_terms_kernel for proof j = idx >> log_n with its own beta_j, gamma_j (canonical arrays); the witness of
// proof j at a/b/c[j * n], sigma shared
__global__ void plonk_perm_terms_many_kernel(const Fr* __restrict__ a, const Fr* __restrict__ b, const Fr* __restrict__ c,
                                             const Fr* __restrict__ s1, const Fr* __restrict__ s2, const Fr* __restrict__ s3,
                                             uint32_t log_n, const Fr* __restrict__ omega_tab, const Fr* __restrict__ betas,
                                             const Fr* __restrict__ gammas, uint64_t total, Fr* __restrict__ num,
                                             Fr* __restrict__ den) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx >> log_n, i = idx & ((uint64_t(1) << log_n) - 1);
  Fr beta = betas[j].to_mont(), gamma = gammas[j].to_mont();
  Fr w = power_at(omega_tab, (uint32_t)i);
  Fr bw = beta * w;
  Fr am = a[idx].to_mont() + gamma, bm = b[idx].to_mont() + gamma, cm = c[idx].to_mont() + gamma;
  Fr nu = (am + bw) * (bm + bw.dbl()) * (cm + bw.dbl() + bw);
  Fr de = (am + beta * s1[i].to_mont()) * (bm + beta * s2[i].to_mont()) * (cm + beta * s3[i].to_mont());
  num[idx] = nu.from_mont();
  den[idx] = de.from_mont();
}

// ------------------------------------------------------------------ segmented exclusive scan
// The 3-kernel tile scan of poly.cu (pp_*) over count segments of `seg` elements back to back: out[e] = op(in[s..e))
// with s the start of e's segment (out[s] = identity).  The block scans carry (value, flag) pairs: the flag says
// that a segment starts inside the covered range, the value is the op over the range from the last such start
// (the whole range without one).  (l, fl) then (r, fr) = (fr ? r : l op r, fl | fr), which is associative.
template <bool SUM>
__device__ __forceinline__ void seg_pair_after(Fr& v, int& f, const Fr& lv, int lf) {
  if (!f) v = scan_op<SUM>(lv, v);
  f |= lf;
}
template <bool SUM>
__device__ __forceinline__ Fr seg_block_inclusive_scan(Fr v, int& f, Fr* sm, int* smf) {
  sm[threadIdx.x] = v;
  smf[threadIdx.x] = f;
  __syncthreads();
  for (int o = 1; o < PP_THREADS; o <<= 1) {
    Fr tv = v;
    int tf = f;
    if ((int)threadIdx.x >= o) seg_pair_after<SUM>(tv, tf, sm[threadIdx.x - o], smf[threadIdx.x - o]);
    __syncthreads();
    v = tv;
    f = tf;
    sm[threadIdx.x] = v;
    smf[threadIdx.x] = f;
    __syncthreads();
  }
  return v;
}

template <bool SUM>
__global__ void __launch_bounds__(PP_THREADS) pp_seg_tile_kernel(const Fr* __restrict__ in, uint64_t total, uint64_t seg,
                                                                  Fr* __restrict__ tile_v, int* __restrict__ tile_f) {
  __shared__ Fr sm[PP_THREADS];
  __shared__ int smf[PP_THREADS];
  uint64_t base = (uint64_t)blockIdx.x * PP_TILE + (uint64_t)threadIdx.x * PP_ITEMS;
  Fr p = scan_id<SUM>();
  int f = 0;
#pragma unroll
  for (int k = 0; k < PP_ITEMS; k++) {
    const uint64_t e = base + k;
    if (e < total) {
      if (e % seg == 0) {
        p = scan_id<SUM>();
        f = 1;
      }
      p = scan_op<SUM>(p, scan_in<SUM>(in[e]));
    }
  }
  Fr inc = seg_block_inclusive_scan<SUM>(p, f, sm, smf);
  if (threadIdx.x == PP_THREADS - 1) {
    tile_v[blockIdx.x] = inc;
    tile_f[blockIdx.x] = f;
  }
}

// single block: tile_v[i] <- the exclusive prefix pair's value over tiles 0..i-1
template <bool SUM>
__global__ void __launch_bounds__(PP_THREADS) pp_seg_tile_scan_kernel(Fr* __restrict__ tile_v, const int* __restrict__ tile_f,
                                                                       uint64_t ntiles) {
  __shared__ Fr sm[PP_THREADS];
  __shared__ int smf[PP_THREADS];
  __shared__ Fr carry;
  __shared__ int carry_f;
  if (threadIdx.x == 0) {
    carry = scan_id<SUM>();
    carry_f = 0;
  }
  __syncthreads();
  for (uint64_t base = 0; base < ntiles; base += PP_THREADS) {
    uint64_t i = base + threadIdx.x;
    Fr v = i < ntiles ? tile_v[i] : scan_id<SUM>();
    int f = i < ntiles ? tile_f[i] : 0;
    Fr inc = seg_block_inclusive_scan<SUM>(v, f, sm, smf);
    Fr ev = threadIdx.x ? sm[threadIdx.x - 1] : scan_id<SUM>();
    int ef = threadIdx.x ? smf[threadIdx.x - 1] : 0;
    Fr cv = carry;
    int cf = carry_f;
    __syncthreads();
    Fr out = ev;
    int of = ef;
    seg_pair_after<SUM>(out, of, cv, cf);
    if (i < ntiles) tile_v[i] = out;
    if (threadIdx.x == PP_THREADS - 1) {
      seg_pair_after<SUM>(inc, f, cv, cf);
      carry = inc;
      carry_f = f;
    }
    __syncthreads();
  }
}

template <bool SUM>
__global__ void __launch_bounds__(PP_THREADS) pp_seg_apply_kernel(const Fr* __restrict__ in, uint64_t total, uint64_t seg,
                                                                   const Fr* __restrict__ tile_off, Fr* __restrict__ out) {
  __shared__ Fr sm[PP_THREADS];
  __shared__ int smf[PP_THREADS];
  uint64_t base = (uint64_t)blockIdx.x * PP_TILE + (uint64_t)threadIdx.x * PP_ITEMS;
  Fr x[PP_ITEMS];
  Fr p = scan_id<SUM>();
  int f = 0;
#pragma unroll
  for (int k = 0; k < PP_ITEMS; k++) {
    const uint64_t e = base + k;
    x[k] = e < total ? scan_in<SUM>(in[e]) : scan_id<SUM>();
    if (e < total && e % seg == 0) {
      p = scan_id<SUM>();
      f = 1;
    }
    p = scan_op<SUM>(p, x[k]);
  }
  seg_block_inclusive_scan<SUM>(p, f, sm, smf);
  Fr run = threadIdx.x ? sm[threadIdx.x - 1] : scan_id<SUM>();
  int rf = threadIdx.x ? smf[threadIdx.x - 1] : 0;
  seg_pair_after<SUM>(run, rf, tile_off[blockIdx.x], 0);
#pragma unroll
  for (int k = 0; k < PP_ITEMS; k++) {
    const uint64_t e = base + k;
    if (e < total) {
      if (e % seg == 0) run = scan_id<SUM>();
      out[e] = scan_out<SUM>(run);
    }
    run = scan_op<SUM>(run, x[k]);
  }
}

// exclusive segmented scan of `total` device elements in segments of `seg`; in != out
template <bool SUM>
static int seg_scan_dev(Context& c, const Fr* in, uint64_t total, uint64_t seg, Fr* out) {
  uint64_t ntiles = (total + PP_TILE - 1) / PP_TILE;
  Fr* tiles = g_arena.alloc(ntiles);
  int* flags = reinterpret_cast<int*>(g_arena.alloc(ntiles / 8 + 1));
  pp_seg_tile_kernel<SUM><<<(unsigned)ntiles, PP_THREADS, 0, c.stream>>>(in, total, seg, tiles, flags);
  CUDA_CHECK_LAUNCH();
  pp_seg_tile_scan_kernel<SUM><<<1, PP_THREADS, 0, c.stream>>>(tiles, flags, ntiles);
  CUDA_CHECK_LAUNCH();
  pp_seg_apply_kernel<SUM><<<(unsigned)ntiles, PP_THREADS, 0, c.stream>>>(in, total, seg, tiles, out);
  CUDA_CHECK_LAUNCH();
  g_arena.free(reinterpret_cast<Fr*>(flags));
  g_arena.free(tiles);
  return 3;
}

// ------------------------------------------------------------------ round 3: quotient, divisibility, split
struct PlonkQuotManyArgs {
  const Fr* ev;  // 4 count blocks of N: a_0..a_{count-1}, b_*, c_*, z_* (Montgomery coset evaluations)
  const Fr *ql, *qr, *qo, *qm, *qc, *s1, *s2, *s3;  // shared circuit coset evaluations, Montgomery
  const Fr *x, *l1f, *zh_inv;                       // static coset data of the device key
  const Fr *betas, *gammas, *alphas;                // count canonical challenges each
  const Fr* pi;  // with public inputs: count blocks of N, the Montgomery coset evaluations of PI_j (round3.py:33)
  uint64_t count;
  uint32_t log_N, ext;
  Fr* t;  // out: count blocks of N quotient evaluations, Montgomery
};
// plonk_quotient_kernel for proof j = idx >> log_N with its own challenges; z(w x) wraps inside proof j's block.
// PI: q_c + PI_j in the gate term (a separate instantiation, so the kernel without public inputs is unchanged)
template <bool PI>
__global__ void __launch_bounds__(128) plonk_quotient_many_kernel(PlonkQuotManyArgs q) {
  uint64_t idx = IDX64;
  const uint64_t N = uint64_t(1) << q.log_N;
  if (idx >= q.count * N) return;
  const uint64_t j = idx >> q.log_N, i = idx & (N - 1);
  const uint64_t blk = q.count * N;
  Fr beta = q.betas[j].to_mont(), gamma = q.gammas[j].to_mont(), alpha = q.alphas[j].to_mont();
  Fr a = q.ev[idx], b = q.ev[blk + idx], c = q.ev[2 * blk + idx];
  const Fr* zj = q.ev + 3 * blk + (j << q.log_N);
  Fr z = zj[i];
  Fr zw = zj[(i + q.ext) & (N - 1)];
  Fr qc = q.qc[i];
  if (PI) qc = qc + q.pi[idx];
  Fr gate = q.ql[i] * a + q.qr[i] * b + q.qo[i] * c + q.qm[i] * (a * b) + qc;
  Fr bx = beta * q.x[i];
  Fr ag = a + gamma, bg = b + gamma, cg = c + gamma;
  Fr num = (ag + bx) * (bg + bx.dbl()) * (cg + bx.dbl() + bx) * z;
  Fr den = (ag + beta * q.s1[i]) * (bg + beta * q.s2[i]) * (cg + beta * q.s3[i]) * zw;
  Fr main = (gate + alpha * (num - den)) * q.zh_inv[i & (q.ext - 1)];
  Fr l1 = alpha * alpha * ((z - Fr::one()) * q.l1f[i]);
  q.t[idx] = main + l1;
}

// *first = lowest j with a non-zero coefficient t_j[i], from <= i < N (t_j = t[j * N ..]; zero is zero in either form)
__global__ void plonk_divisible_many_kernel(const Fr* __restrict__ t, uint32_t log_N, uint64_t from, uint64_t total,
                                            unsigned int* __restrict__ first) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t width = (uint64_t(1) << log_N) - from;
  const uint64_t j = idx / width, i = from + idx % width;
  if (!t[(j << log_N) + i].is_zero()) atomicMin(first, (unsigned int)j);
}

// t_lo | t_mid | t_hi of every proof (round3.py:169-171), canonical, each at stride n + 6:
// out[(part * count + j) * (n + 6) + i] = t_j[part * n + i] for i < (part < 2 ? n : n + 6), zero above.
// t: count blocks of 2^log_N Montgomery coefficients.
__global__ void plonk_split_t_many_kernel(const Fr* __restrict__ t, uint32_t log_N, uint64_t n, uint64_t count,
                                          uint64_t total, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t v = idx / (n + 6), i = idx % (n + 6);
  const uint64_t part = v / count, j = v % count;
  const uint64_t len = part < 2 ? n : n + 6;
  out[idx] = i < len ? t[(j << log_N) + part * n + i].from_mont() : Fr::zero();
}

// ------------------------------------------------------------------ round 4: batched Horner
static constexpr int MANY_GROUPS = 16;
struct HornerManyArgs {
  const Fr* src[MANY_GROUPS];
  uint64_t stride[MANY_GROUPS];  // 0: one vector shared by every proof
  uint64_t len[MANY_GROUPS];
  uint32_t sel[MANY_GROUPS];     // which of the point sets
  uint32_t groups;
  uint64_t count;
};
// item = g * count + j evaluates group g's vector of proof j at point (sel[g], j); level as in horner_multi_kernel
__global__ void horner_many_kernel(HornerManyArgs a, int level, int levels, const Fr* __restrict__ xs,
                                   const Fr* __restrict__ prev, uint64_t np_prev, Fr* __restrict__ cur, uint64_t np,
                                   uint64_t total) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t item = idx / np, jj = idx % np;
  const uint64_t g = item / a.count, j = item % a.count;
  uint64_t m = a.len[g];
  for (int l = 0; l < level; l++) m = (m + HORNER_CHUNK - 1) / HORNER_CHUNK;
  const uint64_t beg = jj * HORNER_CHUNK;
  Fr acc = Fr::zero();
  if (beg < m) {
    const Fr* in = level == 0 ? a.src[g] + j * a.stride[g] : prev + item * np_prev;
    const uint64_t end = beg + HORNER_CHUNK < m ? beg + HORNER_CHUNK : m;
    Fr x = xs[((uint64_t)a.sel[g] * a.count + j) * levels + level];
    for (uint64_t i = end; i > beg; i--) acc = acc * x + in[i - 1];
  }
  cur[idx] = acc;
}

// ------------------------------------------------------------------ round 5: lincomb and division by (x - zeta)
struct LinCombManyArgs {
  const Fr* src[MANY_GROUPS];
  uint64_t stride[MANY_GROUPS];  // 0: shared
  uint64_t len[MANY_GROUPS];
  uint32_t K;
};
// dst[j * dst_stride + i] = sum_k coef[j][k] * src_k,j[i] (+ coef[j][K] at i = 0), i < n.  coef: count x (K + 1)
// Montgomery (the constant column too); sources canonical, so every product comes out canonical.
__global__ void fr_lincomb_many_kernel(LinCombManyArgs a, const Fr* __restrict__ coef, uint64_t n, uint64_t dst_stride,
                                       uint64_t total, Fr* __restrict__ dst) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / n, i = idx % n;
  const Fr* cj = coef + j * (a.K + 1);
  Fr acc = Fr::zero();
  for (uint32_t k = 0; k < a.K; k++)
    if (i < a.len[k]) acc = acc + a.src[k][j * a.stride[k] + i] * cj[k];
  if (i == 0) acc = acc + cj[a.K].from_mont();
  dst[j * dst_stride + i] = acc;
}

// tabs[j * 2L + k] = zeta_j^(2^k), tabs[j * 2L + L + k] = zeta_j^-(2^k), k < L (Montgomery; zeta_j = 0 gives zeros,
// the caller shifts instead)
__global__ void dl_pow2_many_kernel(const Fr* __restrict__ zetas, uint64_t count, uint32_t L, Fr* __restrict__ tabs) {
  uint64_t j = IDX64;
  if (j >= count) return;
  Fr z = zetas[j].to_mont();
  Fr zi = z.inv();
  Fr* t = tabs + j * 2 * L;
  for (uint32_t k = 0; k < L; k++) {
    t[k] = z;
    t[L + k] = zi;
    z = z.sqr();
    zi = zi.sqr();
  }
}
__device__ __forceinline__ Fr dl_pow(const Fr* __restrict__ tab, uint64_t e) {
  Fr r = Fr::one();
  for (int k = 0; e; k++, e >>= 1)
    if (e & 1) r = r * tab[k];
  return r;
}
// d[j * len + i] = src_j[i] * zeta_j^i
__global__ void dl_scale_many_kernel(const Fr* __restrict__ src, uint64_t src_stride, uint64_t len, uint32_t L,
                                     const Fr* __restrict__ tabs, uint64_t total, Fr* __restrict__ d) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / len, i = idx % len;
  d[idx] = src[j * src_stride + i] * dl_pow(tabs + j * 2 * L, i);  // canonical * Montgomery -> canonical
}
// q_j[k] = zeta_j^-(k+1) (T_j - P_j[k] - d_j[k]), T_j = P_j[len-1] + d_j[len-1] (fr_div_linear_finish_kernel per
// segment); zeta_j = 0: q_j[k] = src_j[k + 1] (the shift of the single path)
__global__ void dl_finish_many_kernel(const Fr* __restrict__ src, uint64_t src_stride, const Fr* __restrict__ d,
                                      const Fr* __restrict__ P, uint64_t len, uint32_t L, const Fr* __restrict__ tabs,
                                      const Fr* __restrict__ zetas, uint64_t dst_stride, uint64_t total, Fr* __restrict__ q) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / (len - 1), k = idx % (len - 1);
  Fr r;
  if (zetas[j].is_zero()) {
    r = src[j * src_stride + k + 1];
  } else {
    const uint64_t s = j * len;
    Fr T = P[s + len - 1] + d[s + len - 1];
    r = (T - P[s + k] - d[s + k]) * dl_pow(tabs + j * 2 * L + L, k + 1);
  }
  q[j * dst_stride + k] = r;
}

static Fr* upload_canon(Context& c, const uint8_t* host, uint64_t n) {
  Fr* d = g_arena.alloc(n);
  if (n) CUDA_CHECK(cudaMemcpyAsync(d, host, n * 32, cudaMemcpyHostToDevice, c.stream));
  return d;
}

static void pi_check_shape(const char* what, uint64_t n, uint64_t ell, uint64_t stride, uint32_t count) {
  if (!n || (n & (n - 1)) || n > (uint64_t(1) << 28)) throw InvalidArgument(std::string(what) + ": n must be a power of two <= 2^28");
  if (ell > n) throw InvalidArgument(std::string(what) + ": more public inputs than gates");
  if (count > 1 && stride < ell) throw InvalidArgument(std::string(what) + ": stride shorter than the public inputs");
}

// nblk = 4: a_*, b_*, c_*, z_*; nblk = 5: PI_* too, from pi (count blocks of n coefficients at pi_off)
static void coset_inputs_many(Context& c, const char* what, uint64_t wires, uint64_t z, uint64_t pi, uint64_t pi_off,
                              uint64_t n, uint32_t count, uint32_t log_N, uint64_t out, uint32_t nblk) {
  if (log_N > 28 || (uint64_t(1) << log_N) < n + 3) throw InvalidArgument(std::string(what) + ": 2^log_N must hold n + 3 coefficients");
  if (((uint64_t)nblk * count << log_N) >= (uint64_t(1) << 32))
    throw InvalidArgument(std::string(what) + ": blocks * count * 2^log_N must be < 2^32");
  Fr* pw = hptr(wires, 0, 3 * (uint64_t)count * (n + 2), what);
  Fr* pz = hptr(z, 0, (uint64_t)count * (n + 3), what);
  Fr* pp = nblk == 5 ? hptr(pi, pi_off, (uint64_t)count * n, what) : nullptr;
  const uint64_t total = (uint64_t)nblk * count << log_N;
  Fr* po = hptr(out, 0, total, what);
  if (!count) return;
  plonk_coset_inputs_many_kernel<<<GRID_1D(total)>>>(pw, pz, pp, n, count, log_N, total, po);
  CUDA_CHECK_LAUNCH();
  c.launches++;
}

// evals: 4 count blocks of N (a_*, b_*, c_*, z_*), or 5 with PI_* (with_pi)
static void quotient_many(Context& c, const char* w, uint64_t evals, const uint64_t circuit[8], uint64_t n, uint32_t ext,
                          uint32_t count, uint64_t x, uint64_t l1f, uint64_t zh8, const uint8_t* betas,
                          const uint8_t* gammas, const uint8_t* alphas, uint64_t t_out, bool with_pi) {
  if (!circuit || (count && (!betas || !gammas || !alphas))) throw InvalidArgument(std::string(w) + ": null argument");
  if (ext != 4 && ext != 8 && ext != 16) throw InvalidArgument(std::string(w) + ": ext must be 4, 8 or 16");
  const uint64_t N = (uint64_t)ext * n;
  if (!n || (N & (N - 1)) || N > (uint64_t(1) << 28)) throw InvalidArgument(std::string(w) + ": n must be a power of two");
  if (N < 3 * n + 6) throw InvalidArgument(std::string(w) + ": coset too small for the quotient degree");
  const uint64_t nblk = with_pi ? 5 : 4;
  if (nblk * count * N >= (uint64_t(1) << 32)) throw InvalidArgument(std::string(w) + ": blocks * count * N must be < 2^32");
  PlonkQuotManyArgs q;
  q.ev = hptr(evals, 0, nblk * count * N, w);
  q.pi = q.ev + 4 * (uint64_t)count * N;
  const Fr** slots[8] = {&q.ql, &q.qr, &q.qo, &q.qm, &q.qc, &q.s1, &q.s2, &q.s3};
  for (int k = 0; k < 8; k++) *slots[k] = hptr(circuit[k], 0, N, w);
  q.x = hptr(x, 0, N, w);
  q.l1f = hptr(l1f, 0, N, w);
  q.zh_inv = hptr(zh8, 0, ext, w);
  q.t = hptr(t_out, 0, (uint64_t)count * N, w);
  q.count = count;
  q.log_N = log2_ceil(N);
  q.ext = ext;
  if (!count) return;
  ArenaScope scope;
  Fr* ch = g_arena.alloc(3 * (uint64_t)count);
  CUDA_CHECK(cudaMemcpyAsync(ch, betas, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
  CUDA_CHECK(cudaMemcpyAsync(ch + count, gammas, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
  CUDA_CHECK(cudaMemcpyAsync(ch + 2 * count, alphas, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
  q.betas = ch;
  q.gammas = ch + count;
  q.alphas = ch + 2 * count;
  if (with_pi) plonk_quotient_many_kernel<true><<<ceil_div((uint64_t)count * N, 128), 128, 0, c.stream>>>(q);
  else plonk_quotient_many_kernel<false><<<ceil_div((uint64_t)count * N, 128), 128, 0, c.stream>>>(q);
  CUDA_CHECK_LAUNCH();
  c.launches++;
  CUDA_CHECK(cudaStreamSynchronize(c.stream));
}

}  // namespace zkp

using namespace zkp;

extern "C" {

int zkp_fr_ntt_many_dev(uint64_t scalars, uint64_t offset, uint32_t log_n, const uint8_t omega[32], int inverse,
                        const uint8_t* coset_shift, uint32_t count) {
  return guarded([&](Context& c) {
    const char* what = "zkp_fr_ntt_many_dev";
    if (!omega) throw InvalidArgument(std::string(what) + ": null omega");
    if (log_n > 28) throw InvalidArgument(std::string(what) + ": log_n must be <= 28");
    if (((uint64_t)count << log_n) >= (uint64_t(1) << 32)) throw InvalidArgument(std::string(what) + ": count * 2^log_n must be < 2^32");
    const uint64_t total = (uint64_t)count << log_n;
    Fr* d = hptr(scalars, offset, total, what);
    if (!count) return;
    ArenaScope scope;
    Fr* scratch = g_arena.alloc(total);
    FrBytes w, cs;
    memcpy(w.b, omega, 32);
    if (coset_shift) memcpy(cs.b, coset_shift, 32);
    c.launches += ntt_device_count(c, d, scratch, log_n, w, inverse != 0, coset_shift ? &cs : nullptr, count);
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_plonk_blind_many_dev(uint64_t src, uint64_t src_off, uint64_t src_stride, uint64_t n, uint32_t nvec,
                             const uint8_t* blinds, uint32_t k, uint64_t dst, uint64_t dst_off, uint64_t dst_stride) {
  return guarded([&](Context& c) {
    const char* what = "zkp_plonk_blind_many_dev";
    if (n > src_stride || n + k > dst_stride || (nvec && k && !blinds)) throw InvalidArgument(std::string(what) + ": bad argument");
    if (!nvec) return;
    Fr* s = hptr(src, src_off, (uint64_t)(nvec - 1) * src_stride + n, what);
    Fr* d = hptr(dst, dst_off, (uint64_t)nvec * dst_stride, what);
    if (s < d + (uint64_t)nvec * dst_stride && d < s + (uint64_t)(nvec - 1) * src_stride + n)
      throw InvalidArgument(std::string(what) + ": destination overlaps the source");
    ArenaScope scope;
    Fr* b = upload_canon(c, blinds, (uint64_t)nvec * k);
    const uint64_t total = (uint64_t)nvec * dst_stride;
    plonk_blind_many_kernel<<<GRID_1D(total)>>>(s, src_stride, n, k, b, dst_stride, total, d);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_plonk_perm_terms_many_dev(uint64_t a, uint64_t b, uint64_t cc, uint64_t off, uint64_t s1, uint64_t s2, uint64_t s3,
                                  uint64_t n, uint32_t count, const uint8_t omega[32], const uint8_t* betas,
                                  const uint8_t* gammas, uint64_t num, uint64_t den) {
  return guarded([&](Context& c) {
    const char* w = "zkp_plonk_perm_terms_many_dev";
    if (!omega || (count && (!betas || !gammas))) throw InvalidArgument(std::string(w) + ": null argument");
    if (!n || (n & (n - 1)) || n > (uint64_t(1) << 28)) throw InvalidArgument(std::string(w) + ": n must be a power of two <= 2^28");
    const uint64_t total = (uint64_t)count * n;
    Fr *pa = hptr(a, off, total, w), *pb = hptr(b, off, total, w), *pc = hptr(cc, off, total, w);
    Fr *p1 = hptr(s1, 0, n, w), *p2 = hptr(s2, 0, n, w), *p3 = hptr(s3, 0, n, w);
    Fr *pn = hptr(num, 0, total, w), *pd = hptr(den, 0, total, w);
    if (!count) return;
    ArenaScope scope;
    FrBytes ob;
    memcpy(ob.b, omega, 32);
    int launches = 0;
    const Fr* tab = power_table(c, ob, false, log2_ceil(n), &launches);
    Fr* ch = g_arena.alloc(2 * (uint64_t)count);
    CUDA_CHECK(cudaMemcpyAsync(ch, betas, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(ch + count, gammas, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
    plonk_perm_terms_many_kernel<<<GRID_1D(total)>>>(pa, pb, pc, p1, p2, p3, log2_ceil(n), tab, ch, ch + count, total, pn, pd);
    CUDA_CHECK_LAUNCH();
    c.launches += launches + 1;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

// exclusive scan per segment: op 0 product (dst_j[0] = 1), 1 sum (dst_j[0] = 0) over count segments of seg elements
int zkp_fr_scan_many_dev(int op, uint64_t dst, uint64_t dst_off, uint64_t src, uint64_t src_off, uint64_t seg,
                         uint32_t count) {
  return guarded([&](Context& c) {
    const char* what = "zkp_fr_scan_many_dev";
    if (op != 0 && op != 1) throw InvalidArgument(std::string(what) + ": op must be 0 (product) or 1 (sum)");
    if (!seg) throw InvalidArgument(std::string(what) + ": empty segments");
    const uint64_t total = (uint64_t)count * seg;
    Fr* d = hptr(dst, dst_off, total, what);
    Fr* s = hptr(src, src_off, total, what);
    if (!total) return;
    if (s < d + total && d < s + total) throw InvalidArgument(std::string(what) + ": destination overlaps the source");
    if ((total + PP_TILE - 1) / PP_TILE >= (uint64_t(1) << 31)) throw InvalidArgument(std::string(what) + ": too many tiles");
    ArenaScope scope;
    c.launches += op == 0 ? seg_scan_dev<false>(c, s, total, seg, d) : seg_scan_dev<true>(c, s, total, seg, d);
  });
}

int zkp_plonk_coset_inputs_many_dev(uint64_t wires, uint64_t z, uint64_t n, uint32_t count, uint32_t log_N, uint64_t out) {
  return guarded([&](Context& c) {
    coset_inputs_many(c, "zkp_plonk_coset_inputs_many_dev", wires, z, 0, 0, n, count, log_N, out, 4);
  });
}

int zkp_plonk_coset_inputs_pi_many_dev(uint64_t wires, uint64_t z, uint64_t pi, uint64_t pi_off, uint64_t n, uint32_t count,
                                       uint32_t log_N, uint64_t out) {
  return guarded([&](Context& c) {
    coset_inputs_many(c, "zkp_plonk_coset_inputs_pi_many_dev", wires, z, pi, pi_off, n, count, log_N, out, 5);
  });
}

int zkp_plonk_quotient_many_dev(uint64_t evals, const uint64_t circuit[8], uint64_t n, uint32_t ext, uint32_t count,
                                uint64_t x, uint64_t l1f, uint64_t zh8, const uint8_t* betas, const uint8_t* gammas,
                                const uint8_t* alphas, uint64_t t_out) {
  return guarded([&](Context& c) {
    quotient_many(c, "zkp_plonk_quotient_many_dev", evals, circuit, n, ext, count, x, l1f, zh8, betas, gammas, alphas,
                  t_out, false);
  });
}

int zkp_plonk_quotient_pi_many_dev(uint64_t evals, const uint64_t circuit[8], uint64_t n, uint32_t ext, uint32_t count,
                                   uint64_t x, uint64_t l1f, uint64_t zh8, const uint8_t* betas, const uint8_t* gammas,
                                   const uint8_t* alphas, uint64_t t_out) {
  return guarded([&](Context& c) {
    quotient_many(c, "zkp_plonk_quotient_pi_many_dev", evals, circuit, n, ext, count, x, l1f, zh8, betas, gammas, alphas,
                  t_out, true);
  });
}

int zkp_plonk_pi_scatter_many_dev(uint64_t pub, uint64_t off, uint64_t stride, uint64_t ell, uint64_t n, uint32_t count,
                                  uint64_t dst, uint64_t dst_off) {
  return guarded([&](Context& c) {
    const char* what = "zkp_plonk_pi_scatter_many_dev";
    pi_check_shape(what, n, ell, stride, count);
    const uint64_t total = (uint64_t)count * n;
    Fr* d = hptr(dst, dst_off, total, what);
    if (!count) return;
    Fr* px = nullptr;
    if (ell) {
      const uint64_t span = (uint64_t)(count - 1) * stride + ell;
      px = hptr(pub, off, span, what);
      if (px < d + total && d < px + span) throw InvalidArgument(std::string(what) + ": destination overlaps the source");
    }
    plonk_pi_scatter_many_kernel<<<GRID_1D(total)>>>(px, stride, ell, log2_ceil(n), total, d);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_plonk_pi_eval_many_dev(uint64_t pub, uint64_t off, uint64_t stride, uint64_t ell, uint64_t n, uint32_t count,
                               const uint8_t omega[32], const uint8_t* zetas, uint8_t* out) {
  return guarded([&](Context& c) {
    const char* what = "zkp_plonk_pi_eval_many_dev";
    if (!omega || (count && (!zetas || !out))) throw InvalidArgument(std::string(what) + ": null argument");
    pi_check_shape(what, n, ell, stride, count);
    if (!count) return;
    if (!ell) {
      memset(out, 0, (size_t)count * 32);
      return;
    }
    Fr* px = hptr(pub, off, (uint64_t)(count - 1) * stride + ell, what);
    ArenaScope scope;
    FrBytes ob;
    memcpy(ob.b, omega, 32);
    int launches = 0;
    const uint32_t log_n = log2_ceil(n);
    const Fr* tab = power_table(c, ob, false, log_n, &launches);
    Fr* zs = upload_canon(c, zetas, count);
    const uint64_t m = (uint64_t)count * ell;
    Fr* gap = g_arena.alloc(m);
    Fr* inv = g_arena.alloc(m);
    Fr* res = g_arena.alloc(count);
    plonk_pi_gap_many_kernel<<<GRID_1D(m)>>>(zs, tab, ell, n, m, gap);
    CUDA_CHECK_LAUNCH();
    const uint64_t T = (m + BATCH_INV_CHUNK - 1) / BATCH_INV_CHUNK;
    fr_batch_inverse_kernel<<<ceil_div(T, 128), 128, 0, c.stream>>>(gap, m, T, 1, inv);  // zeros stay zero
    CUDA_CHECK_LAUNCH();
    plonk_pi_eval_many_kernel<<<count, DOT_THREADS, 0, c.stream>>>(px, stride, ell, log_n, zs, tab, inv, res);
    CUDA_CHECK_LAUNCH();
    CUDA_CHECK(cudaMemcpyAsync(out, res, (size_t)count * 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    c.launches += launches + 3;
  });
}

// lowest proof index j whose quotient t_j (count blocks of N = ext * n) has a non-zero coefficient at 3n + 6 or
// above, UINT64_MAX if every proof's constraint polynomial is divisible by Z_H
int zkp_plonk_divisible_many_dev(uint64_t t, uint64_t n, uint32_t ext, uint32_t count, uint64_t* first_bad) {
  return guarded([&](Context& c) {
    const char* w = "zkp_plonk_divisible_many_dev";
    if (!first_bad) throw InvalidArgument(std::string(w) + ": null output");
    const uint64_t N = (uint64_t)ext * n;
    if (!n || (N & (N - 1)) || N < 3 * n + 6 || N > (uint64_t(1) << 28)) throw InvalidArgument(std::string(w) + ": bad n / ext");
    Fr* pt = hptr(t, 0, (uint64_t)count * N, w);
    *first_bad = ~uint64_t(0);
    if (!count) return;
    ArenaScope scope;
    unsigned int* flag = reinterpret_cast<unsigned int*>(g_arena.alloc(1));
    const unsigned int none = 0xffffffffu;
    CUDA_CHECK(cudaMemcpyAsync(flag, &none, 4, cudaMemcpyHostToDevice, c.stream));
    const uint64_t total = (uint64_t)count * (N - (3 * n + 6));
    plonk_divisible_many_kernel<<<GRID_1D(total)>>>(pt, log2_ceil(N), 3 * n + 6, total, flag);
    CUDA_CHECK_LAUNCH();
    c.launches++;
    unsigned int got = none;
    CUDA_CHECK(cudaMemcpyAsync(&got, flag, 4, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    if (got != none) *first_bad = got;
  });
}

int zkp_plonk_split_t_many_dev(uint64_t t, uint64_t n, uint32_t ext, uint32_t count, uint64_t out) {
  return guarded([&](Context& c) {
    const char* w = "zkp_plonk_split_t_many_dev";
    const uint64_t N = (uint64_t)ext * n;
    if (!n || (N & (N - 1)) || N < 3 * n + 6 || N > (uint64_t(1) << 28)) throw InvalidArgument(std::string(w) + ": bad n / ext");
    Fr* pt = hptr(t, 0, (uint64_t)count * N, w);
    const uint64_t total = 3 * (uint64_t)count * (n + 6);
    Fr* po = hptr(out, 0, total, w);
    if (!count) return;
    plonk_split_t_many_kernel<<<GRID_1D(total)>>>(pt, log2_ceil(N), n, count, total, po);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

// groups x count evaluations: item g * count + j = p_g,j(x[sel[g]][j]), p_g,j = handles[g] at offs[g] + j * strides[g]
// (stride 0: shared), lens[g] coefficients.  points: npsets x count canonical points; out: groups x count values.
int zkp_fr_poly_eval_many_dev(uint32_t groups, const uint64_t* handles, const uint64_t* offs, const uint64_t* strides,
                              const uint64_t* lens, const uint32_t* sel, uint32_t count, uint32_t npsets,
                              const uint8_t* points, uint8_t* out) {
  return guarded([&](Context& c) {
    const char* what = "zkp_fr_poly_eval_many_dev";
    if (groups == 0 || count == 0) return;
    if (groups > (uint32_t)MANY_GROUPS || !npsets || !handles || !offs || !strides || !lens || !sel || !points || !out)
      throw InvalidArgument(std::string(what) + ": 1..16 groups, no null arguments");
    HornerManyArgs a;
    a.groups = groups;
    a.count = count;
    uint64_t max_n = 1;
    for (uint32_t g = 0; g < groups; g++) {
      if (!lens[g]) throw InvalidArgument(std::string(what) + ": empty polynomial");
      if (sel[g] >= npsets) throw InvalidArgument(std::string(what) + ": point set out of range");
      if (strides[g] && strides[g] < lens[g]) throw InvalidArgument(std::string(what) + ": stride shorter than the polynomial");
      a.src[g] = hptr(handles[g], offs[g], (uint64_t)(count - 1) * strides[g] + lens[g], what);
      a.stride[g] = strides[g];
      a.len[g] = lens[g];
      a.sel[g] = sel[g];
      if (lens[g] > max_n) max_n = lens[g];
    }
    ArenaScope scope;
    int levels = 0;
    for (uint64_t m = max_n; m > 1; m = (m + HORNER_CHUNK - 1) / HORNER_CHUNK) levels++;
    if (levels == 0) levels = 1;
    const uint64_t npts = (uint64_t)npsets * count, items = (uint64_t)groups * count;
    Fr* xc = upload_canon(c, points, npts);
    Fr* xp = g_arena.alloc(npts * levels);
    horner_powers_multi_kernel<<<GRID_1D(npts)>>>(xc, (int)npts, xp, levels);
    CUDA_CHECK_LAUNCH();
    int launches = 1;
    const Fr* prev = nullptr;
    uint64_t np_prev = 0, m = max_n;
    Fr* cur = nullptr;
    for (int l = 0; l < levels; l++) {
      const uint64_t np = (m + HORNER_CHUNK - 1) / HORNER_CHUNK;
      const uint64_t total = items * np;
      cur = g_arena.alloc(total);
      horner_many_kernel<<<GRID_1D(total)>>>(a, l, levels, xp, prev, np_prev, cur, np, total);
      CUDA_CHECK_LAUNCH();
      launches++;
      prev = cur;
      np_prev = np;
      m = np;
    }
    CUDA_CHECK(cudaMemcpyAsync(out, cur, (size_t)items * 32, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    c.launches += launches;
  });
}

// dst_j[i] = sum_k coeffs[j][k] * src_k,j[i] + (i == 0 ? coeffs[j][K] : 0), i < n, j < count: source k at
// handles[k] + offs[k] + j * strides[k] (stride 0: shared), lens[k] <= n coefficients; coeffs: count x (K + 1) canonical
int zkp_fr_lincomb_many_dev(uint64_t dst, uint64_t dst_off, uint64_t dst_stride, uint64_t n, uint32_t count, uint32_t K,
                            const uint64_t* handles, const uint64_t* offs, const uint64_t* strides, const uint64_t* lens,
                            const uint8_t* coeffs) {
  return guarded([&](Context& c) {
    const char* what = "zkp_fr_lincomb_many_dev";
    if (K > (uint32_t)MANY_GROUPS || (K && (!handles || !offs || !strides || !lens)) || (count && n && !coeffs))
      throw InvalidArgument(std::string(what) + ": at most 16 sources, no null arguments");
    if (dst_stride < n) throw InvalidArgument(std::string(what) + ": destination stride shorter than n");
    if (!n || !count) return;
    Fr* d = hptr(dst, dst_off, (uint64_t)(count - 1) * dst_stride + n, what);
    const uint64_t dspan = (uint64_t)(count - 1) * dst_stride + n;
    LinCombManyArgs a;
    a.K = K;
    for (uint32_t k = 0; k < K; k++) {
      if (lens[k] > n) throw InvalidArgument(std::string(what) + ": a source is longer than the destination");
      if (strides[k] && strides[k] < lens[k]) throw InvalidArgument(std::string(what) + ": stride shorter than the source");
      const uint64_t span = (uint64_t)(count - 1) * strides[k] + lens[k];
      a.src[k] = hptr(handles[k], offs[k], span, what);
      if (lens[k] && a.src[k] < d + dspan && d < a.src[k] + span) throw InvalidArgument(std::string(what) + ": destination overlaps a source");
      a.stride[k] = strides[k];
      a.len[k] = lens[k];
    }
    ArenaScope scope;
    const uint64_t nc = (uint64_t)count * (K + 1);
    Fr* co = upload_canon(c, coeffs, nc);
    fr_to_mont_kernel<<<GRID_1D(nc)>>>(co, nc, co);
    CUDA_CHECK_LAUNCH();
    const uint64_t total = (uint64_t)count * n;
    fr_lincomb_many_kernel<<<GRID_1D(total)>>>(a, co, n, dst_stride, total, d);
    CUDA_CHECK_LAUNCH();
    c.launches += 2;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

// dst_j[0..len-1) = (p_j(x) - p_j(zeta_j)) / (x - zeta_j) for p_j = src[src_off + j * src_stride ..][0..len), j < count:
// zkp_fr_div_linear_dev per segment (zeta_j = 0: the shift p_j[1..len)).  zetas: count x 32 B canonical.
int zkp_fr_div_linear_many_dev(uint64_t src, uint64_t src_off, uint64_t src_stride, uint64_t len, uint32_t count,
                               const uint8_t* zetas, uint64_t dst, uint64_t dst_off, uint64_t dst_stride) {
  return guarded([&](Context& c) {
    const char* what = "zkp_fr_div_linear_many_dev";
    if (count && !zetas) throw InvalidArgument(std::string(what) + ": null zetas");
    if (len < 2 || !count) return;
    if (src_stride < len || dst_stride < len - 1) throw InvalidArgument(std::string(what) + ": stride shorter than the polynomial");
    if (len > (uint64_t(1) << 28)) throw InvalidArgument(std::string(what) + ": len must be <= 2^28");
    const uint64_t sspan = (uint64_t)(count - 1) * src_stride + len, dspan = (uint64_t)(count - 1) * dst_stride + len - 1;
    Fr* p = hptr(src, src_off, sspan, what);
    Fr* q = hptr(dst, dst_off, dspan, what);
    if (p < q + dspan && q < p + sspan) throw InvalidArgument(std::string(what) + ": destination overlaps the source");
    const uint64_t total = (uint64_t)count * len;
    if ((total + PP_TILE - 1) / PP_TILE >= (uint64_t(1) << 31)) throw InvalidArgument(std::string(what) + ": too many tiles");
    ArenaScope scope;
    const uint32_t L = log2_ceil(len + 1);
    Fr* zs = upload_canon(c, zetas, count);
    Fr* tabs = g_arena.alloc((uint64_t)count * 2 * L);
    dl_pow2_many_kernel<<<GRID_1D(count)>>>(zs, count, L, tabs);
    CUDA_CHECK_LAUNCH();
    Fr* d = g_arena.alloc(total);
    Fr* P = g_arena.alloc(total);
    dl_scale_many_kernel<<<GRID_1D(total)>>>(p, src_stride, len, L, tabs, total, d);
    CUDA_CHECK_LAUNCH();
    int launches = 2 + seg_scan_dev<true>(c, d, total, len, P);
    const uint64_t tout = (uint64_t)count * (len - 1);
    dl_finish_many_kernel<<<GRID_1D(tout)>>>(p, src_stride, d, P, len, L, tabs, zs, dst_stride, tout, q);
    CUDA_CHECK_LAUNCH();
    c.launches += launches + 1;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

}  // extern "C"
