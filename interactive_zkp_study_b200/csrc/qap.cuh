// QAP construction at scale over the reference's evaluation domain {1, 2, ..., k} (SURVEY.md 8 f2).
// Included once, by poly.cu (shares its arena, scans and batch inversion).
//
// The reference builds the QAP by Lagrange-interpolating every wire's column of the R1CS through
// the points x = 1..k in FLOATING POINT, scaled by the determinant of the k x k Vandermonde matrix
// (/root/reference/zkp/groth16/qap_creator_lcm.py:50-78 mk_singleton / lagrange_interp, :114-135
// r1cs_to_qap_times_lcm), keeps the dense numWires x numGates coefficient matrices and contracts
// them with the witness in hxr (/root/reference/zkp/groth16/poly_utils.py:52-59,116-125).  None of that
// survives 2^20 constraints.  Interpolation is linear, so what the prover needs is
//     uA = interp_{1..k}(A . w)      (A sparse, k x m;  w the witness)
// i.e. one sparse matrix-vector product and ONE interpolation per matrix, exact in Fr:
//     f(x) = sum_j c_j * Z(x) / (x - x_j),   c_j = y_j / Z'(x_j),   x_j = j + 1,
//     Z'(x_j) = (-1)^(k-1-j) * j! * (k-1-j)!
// summed bottom-up over a subproduct tree: a node holds M = prod (x - x_j) and N = sum_j c_j M / (x - x_j)
// over its leaves; parent: M = M_l M_r, N = N_l M_r + N_r M_l.  Every level is a batch of equal-size
// cyclic products -> batched NTTs (ntt_device, log_batch).  The M side depends on k only: its
// transformed children are cached per k; the N side climbs in evaluation form (ap_interpolate), two
// batched half-size transforms per level.
// Setup needs the Lagrange basis at the toxic point, l_j(x) = Z(x) w_j / (x - x_j): one batch inversion.
#pragma once

namespace zkp {

// ------------------------------------------------------------------ sparse matrices (CSR) on the device
// y[row] = sum_e val[e] * vec[col[e]]; values Montgomery, vec canonical -> y canonical.
// One thread per row: R1CS rows hold a handful of entries.
__global__ void sparse_matvec_kernel(const uint32_t* __restrict__ row_ptr, const uint32_t* __restrict__ col,
                                     const Fr* __restrict__ val, const Fr* __restrict__ vec, uint64_t rows,
                                     Fr* __restrict__ out) {
  uint64_t r = IDX64;
  if (r >= rows) return;
  Fr acc = Fr::zero();
  for (uint32_t e = row_ptr[r]; e < row_ptr[r + 1]; e++) acc = acc + val[e] * vec[col[e]];
  out[r] = acc;
}

// ------------------------------------------------------------------ arithmetic-progression domain {1..k}
__global__ void ap_iota_kernel(Fr* __restrict__ out, uint64_t n, uint64_t first) {
  uint64_t i = IDX64;
  if (i >= n) return;
  Fr x = Fr::zero();
  uint64_t v = first + i;
  x.v[0] = (uint32_t)v;
  x.v[1] = (uint32_t)(v >> 32);
  out[i] = x;  // canonical
}
// den[j] = (-1)^(k-1-j) * j! * (k-1-j)!   (fact canonical -> den Montgomery)
__global__ void ap_weight_den_kernel(const Fr* __restrict__ fact, uint64_t k, Fr* __restrict__ den) {
  uint64_t j = IDX64;
  if (j >= k) return;
  Fr d = fact[j].to_mont() * fact[k - 1 - j].to_mont();
  if ((k - 1 - j) & 1) d = Fr::zero() - d;
  den[j] = d;
}
// leaves of the M tree: -(j+1) for j < k (monic linear factor, top coefficient implicit), 1 beyond
__global__ void ap_leaf_m_kernel(Fr* __restrict__ lev, uint64_t K, uint64_t k) {
  uint64_t j = IDX64;
  if (j >= K) return;
  if (j < k) {
    Fr x = Fr::zero();
    x.v[0] = (uint32_t)(j + 1);
    x.v[1] = (uint32_t)((j + 1) >> 32);
    lev[j] = Fr::zero() - x.to_mont();
  } else {
    lev[j] = Fr::one();
  }
}
// children of size s (K/s of them) -> buffers of size 2s: coefficients, then the implicit monic top
// coefficient of a FULL node (all s leaves real) at position s (with_top), zeros elsewhere
__global__ void ap_pad_kernel(const Fr* __restrict__ lev, uint64_t K, uint32_t log_s, uint64_t k, int with_top,
                              Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= 2 * K) return;
  uint64_t s = uint64_t(1) << log_s;
  uint64_t node = idx >> (log_s + 1), t = idx & (2 * s - 1);
  Fr v = Fr::zero();
  if (t < s) v = lev[node * s + t];
  else if (with_top && t == s && (node + 1) * s <= k) v = Fr::one();
  out[idx] = v;
}
// parent p, frequency t: M^_p = M^_l * M^_r   (all Montgomery)
__global__ void ap_mul_children_kernel(const Fr* __restrict__ ch, uint64_t K, uint32_t log_s, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= K) return;
  uint64_t two_s = uint64_t(2) << log_s;
  uint64_t p = idx >> (log_s + 1), t = idx & (two_s - 1);
  out[idx] = ch[(2 * p) * two_s + t] * ch[(2 * p + 1) * two_s + t];
}
// a full parent's product has degree exactly 2s: its top coefficient (1) wrapped onto x^0
__global__ void ap_unwrap_kernel(Fr* __restrict__ lev, uint64_t K, uint32_t log_2s, uint64_t k) {
  uint64_t p = IDX64;
  uint64_t two_s = uint64_t(1) << log_2s;
  if (p >= (K >> log_2s)) return;
  if ((p + 1) * two_s <= k) lev[p * two_s] = lev[p * two_s] - Fr::one();
}
// leaves of the N tree: c_j = y_j * w_j (* scale); zero beyond k
__global__ void ap_leaf_n_kernel(const Fr* __restrict__ y, const Fr* __restrict__ w, uint64_t K, uint64_t k, int scaled,
                                 Fr scale_mont, Fr* __restrict__ lev) {
  uint64_t j = IDX64;
  if (j >= K) return;
  Fr v = Fr::zero();
  if (j < k) {
    v = y[j] * w[j];
    if (scaled) v = v * scale_mont;
  }
  lev[j] = v;
}
// d[j] = x - (j + 1)   (canonical)
__global__ void ap_x_minus_kernel(Fr x_canon, uint64_t k, Fr* __restrict__ d) {
  uint64_t j = IDX64;
  if (j >= k) return;
  Fr t = Fr::zero();
  t.v[0] = (uint32_t)(j + 1);
  t.v[1] = (uint32_t)((j + 1) >> 32);
  d[j] = x_canon - t;
}
// out[j] = zx * w[j] * inv[j]   (inv canonical, w Montgomery, zx canonical -> canonical)
__global__ void ap_lagrange_finish_kernel(const Fr* __restrict__ inv, const Fr* __restrict__ w, const Fr* __restrict__ zx,
                                          uint64_t k, Fr* __restrict__ out) {
  uint64_t j = IDX64;
  if (j >= k) return;
  out[j] = (inv[j] * w[j]) * zx->to_mont();
}

// host-side constants (the field type's own constructors are device functions)
static Fr host_fr_small(uint32_t v) {
  Fr x;
  memset(&x, 0, sizeof(x));
  x.v[0] = v;
  return x;
}
static Fr host_fr_one_mont() {
  Fr x;
  for (int i = 0; i < 8; i++) x.v[i] = FrParams::R1[i];
  return x;
}

struct ApDomain {
  uint64_t k = 0, K = 0;
  uint32_t L = 0;
  DevBuf weights;  // k, Montgomery: 1 / Z'(x_j)
  DevBuf mhat;     // L levels x 2K: transformed, padded children of the M tree (Montgomery)
  DevBuf z;        // K + 1 coefficients of Z (Montgomery)
};
static ApDomain g_ap;

static int ap_domain_build(Context& c, uint64_t k) {
  if (g_ap.k == k) return 0;
  if (k == 0 || k > (uint64_t(1) << 26)) throw InvalidArgument("arithmetic-progression domain: k must be in [1, 2^26]");
  int launches = 0;
  uint32_t L = log2_ceil(k);
  if (L == 0) L = 1;
  uint64_t K = uint64_t(1) << L;
  g_ap.k = 0;  // invalid until complete
  g_ap.weights.reserve(k * sizeof(Fr));
  g_ap.mhat.reserve((size_t)L * 2 * K * sizeof(Fr));
  g_ap.z.reserve((K + 1) * sizeof(Fr));
  // weights
  Fr* seq = g_arena.alloc(k);
  Fr* fact = g_arena.alloc(k);
  Fr* den = g_arena.alloc(k);
  ap_iota_kernel<<<GRID_1D(k)>>>(seq, k, 1);
  CUDA_CHECK_LAUNCH();
  launches += 1 + scan_dev<false>(c, seq, k, fact, nullptr);  // fact[j] = j!
  ap_weight_den_kernel<<<GRID_1D(k)>>>(fact, k, den);
  CUDA_CHECK_LAUNCH();
  uint64_t T = (k + BATCH_INV_CHUNK - 1) / BATCH_INV_CHUNK;
  fr_batch_inverse_kernel<<<ceil_div(T, 128), 128, 0, c.stream>>>(den, k, T, 1, g_ap.weights.as<Fr>());
  CUDA_CHECK_LAUNCH();
  launches += 2;
  g_arena.free(seq);
  g_arena.free(fact);
  g_arena.free(den);
  // M tree
  Fr* lev = g_arena.alloc(K);
  Fr* nxt = g_arena.alloc(K);
  Fr* scratch = g_arena.alloc(2 * K);
  ap_leaf_m_kernel<<<GRID_1D(K)>>>(lev, K, k);
  CUDA_CHECK_LAUNCH();
  launches++;
  for (uint32_t l = 0; l < L; l++) {
    Fr* ch = g_ap.mhat.as<Fr>() + (size_t)l * 2 * K;
    FrBytes w = omega_for(l + 1);
    ap_pad_kernel<<<GRID_1D(2 * K)>>>(lev, K, l, k, 1, ch);
    CUDA_CHECK_LAUNCH();
    launches += 1 + ntt_device(c, ch, scratch, l + 1, w, false, nullptr, L - l);
    ap_mul_children_kernel<<<GRID_1D(K)>>>(ch, K, l, nxt);
    CUDA_CHECK_LAUNCH();
    launches += 1 + ntt_device(c, nxt, scratch, l + 1, w, true, nullptr, L - l - 1);
    ap_unwrap_kernel<<<GRID_1D(K >> (l + 1))>>>(nxt, K, l + 1, k);
    CUDA_CHECK_LAUNCH();
    launches++;
    Fr* t = lev;
    lev = nxt;
    nxt = t;
  }
  CUDA_CHECK(cudaMemcpyAsync(g_ap.z.p, lev, K * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
  Fr top = k == K ? host_fr_one_mont() : host_fr_small(0);
  CUDA_CHECK(cudaMemcpyAsync(g_ap.z.as<Fr>() + K, &top, sizeof(Fr), cudaMemcpyHostToDevice, c.stream));
  CUDA_CHECK(cudaStreamSynchronize(c.stream));
  g_arena.free(lev);
  g_arena.free(nxt);
  g_arena.free(scratch);
  g_ap.k = k;
  g_ap.K = K;
  g_ap.L = L;
  return launches;
}

// N^_p on H_2s from the children's values: child q has its s values on H_s in `ev` (the even points of
// H_2s) and its s values on the coset w_2s * H_s in `odd` (the odd points).  N canonical, M^ Montgomery.
__global__ void ap_combine_eval_kernel(const Fr* __restrict__ ev, const Fr* __restrict__ odd, const Fr* __restrict__ mch,
                                       uint64_t K, uint32_t log_s, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= K) return;
  const uint64_t s = uint64_t(1) << log_s, two_s = s << 1;
  const uint64_t p = idx >> (log_s + 1), t = idx & (two_s - 1);
  const Fr* src = (t & 1) ? odd : ev;
  const uint64_t h = t >> 1;
  const Fr nl = src[(2 * p) * s + h], nr = src[(2 * p + 1) * s + h];
  out[idx] = nl * mch[(2 * p + 1) * two_s + t] + nr * mch[(2 * p) * two_s + t];
}

// coefficients (canonical) of the polynomial of degree < k through (j + 1, y[j]), times `scale`.
// The N side climbs the tree in EVALUATION form: a node of size s carries its s values on the s-th roots
// of unity H_s.  Its parent needs both children on H_2s = H_s (have) + w_2s H_s (the coset): one inverse
// transform and one coset transform of size s per child, then N^_p = N^_l M^_r + N^_r M^_l pointwise
// against the cached M^.  2 K l butterfly stages per level instead of the 3 K (l + 1) of
// pad -> transform(2s) -> combine -> inverse(2s), and no padding pass; one inverse transform of size K at the root.
static int ap_interpolate(Context& c, const Fr* y, uint64_t k, const Fr* scale_mont, Fr* out) {
  int launches = ap_domain_build(c, k);
  const uint64_t K = g_ap.K;
  const uint32_t L = g_ap.L;
  Fr* ev = g_arena.alloc(K);
  Fr* odd = g_arena.alloc(K);
  Fr* nxt = g_arena.alloc(K);
  Fr* scratch = g_arena.alloc(K);
  ap_leaf_n_kernel<<<GRID_1D(K)>>>(y, g_ap.weights.as<Fr>(), K, k, scale_mont ? 1 : 0, scale_mont ? *scale_mont : host_fr_one_mont(),
                                   ev);
  CUDA_CHECK_LAUNCH();
  launches++;
  for (uint32_t l = 0; l < L; l++) {
    const Fr* mch = g_ap.mhat.as<Fr>() + (size_t)l * 2 * K;
    const Fr* odd_src = ev;  // l == 0: a constant takes the same value everywhere
    if (l > 0) {
      FrBytes w = omega_for(l), shift = omega_for(l + 1);
      CUDA_CHECK(cudaMemcpyAsync(odd, ev, K * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
      launches += ntt_device(c, odd, scratch, l, w, true, nullptr, L - l);
      launches += ntt_device(c, odd, scratch, l, w, false, &shift, L - l);
      odd_src = odd;
    }
    ap_combine_eval_kernel<<<GRID_1D(K)>>>(ev, odd_src, mch, K, l, nxt);
    CUDA_CHECK_LAUNCH();
    launches++;
    Fr* t = ev;
    ev = nxt;
    nxt = t;
  }
  launches += ntt_device(c, ev, scratch, L, omega_for(L), true, nullptr, 0);
  CUDA_CHECK(cudaMemcpyAsync(out, ev, k * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
  g_arena.free(ev);
  g_arena.free(odd);
  g_arena.free(nxt);
  g_arena.free(scratch);
  return launches;
}

// Checks a host CSR matrix and uploads it into r: buf = values (Montgomery), aux[0] = row_ptr, aux[1] = columns.
static void sparse_upload(Context& c, Resource& r, const uint32_t* row_ptr, const uint32_t* col_idx, const uint8_t* values,
                          uint64_t rows, uint64_t cols, uint64_t nnz, const char* what) {
  if (!row_ptr || (nnz && (!col_idx || !values))) throw InvalidArgument(std::string(what) + ": null argument");
  if (rows >= (uint64_t(1) << 31) || cols >= (uint64_t(1) << 32) || nnz >= (uint64_t(1) << 32))
    throw InvalidArgument(std::string(what) + ": dimensions exceed 32-bit indices");
  if (row_ptr[0] != 0 || row_ptr[rows] != nnz) throw InvalidArgument(std::string(what) + ": row_ptr must run from 0 to nnz");
  for (uint64_t i = 0; i < rows; i++)
    if (row_ptr[i] > row_ptr[i + 1]) throw InvalidArgument(std::string(what) + ": row_ptr is not monotone");
  for (uint64_t e = 0; e < nnz; e++)
    if (col_idx[e] >= cols) throw InvalidArgument(std::string(what) + ": column index out of range");
  r.n = rows;
  r.cols = cols;
  r.nnz = nnz;
  r.buf.reserve_pooled((nnz ? nnz : 1) * sizeof(Fr));
  r.aux[0].reserve_pooled((rows + 1) * 4);
  r.aux[1].reserve_pooled((nnz ? nnz : 1) * 4);
  CUDA_CHECK(cudaMemcpyAsync(r.aux[0].p, row_ptr, (rows + 1) * 4, cudaMemcpyHostToDevice, c.stream));
  if (nnz) {
    CUDA_CHECK(cudaMemcpyAsync(r.aux[1].p, col_idx, nnz * 4, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(r.buf.p, values, nnz * 32, cudaMemcpyHostToDevice, c.stream));
    fr_to_mont_kernel<<<GRID_1D(nnz)>>>(r.buf.as<Fr>(), nnz, r.buf.as<Fr>());
    CUDA_CHECK_LAUNCH();
    c.launches++;
  }
}

}  // namespace zkp

using namespace zkp;

extern "C" {

int zkp_sparse_load(const uint32_t* row_ptr, const uint32_t* col_idx, const uint8_t* values, uint64_t rows, uint64_t cols,
                    uint64_t nnz, uint64_t* handle) {
  return guarded([&](Context& c) {
    if (!handle) throw InvalidArgument("zkp_sparse_load: null argument");
    auto r = std::make_unique<Resource>();
    r->kind = HandleKind::Sparse;
    sparse_upload(c, *r, row_ptr, col_idx, values, rows, cols, nnz, "zkp_sparse_load");
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *handle = registry().put(std::move(r));
  });
}

int zkp_sparse_matvec_dev(uint64_t matrix, uint64_t vec, uint64_t vec_off, uint64_t out, uint64_t out_off) {
  return guarded([&](Context& c) {
    Resource* m = need(matrix, HandleKind::Sparse, "zkp_sparse_matvec_dev");
    Fr* v = hptr(vec, vec_off, m->cols, "zkp_sparse_matvec_dev");
    Fr* o = hptr(out, out_off, m->n, "zkp_sparse_matvec_dev");
    if (!m->n) return;
    sparse_matvec_kernel<<<GRID_1D(m->n)>>>(m->aux[0].as<uint32_t>(), m->aux[1].as<uint32_t>(), m->buf.as<Fr>(), v, m->n, o);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_fr_ap_interpolate_dev(uint64_t values, uint64_t off, uint64_t k, const uint8_t* scale, uint64_t out,
                              uint64_t out_off) {
  return guarded([&](Context& c) {
    if (!k) throw InvalidArgument("zkp_fr_ap_interpolate_dev: k must be positive");
    ArenaScope scope;
    Fr* y = hptr(values, off, k, "zkp_fr_ap_interpolate_dev");
    Fr* o = hptr(out, out_off, k, "zkp_fr_ap_interpolate_dev");
    Fr sm;
    if (scale) sm = host_to_mont(c, scale);
    c.launches += ap_interpolate(c, y, k, scale ? &sm : nullptr, o);
  });
}

int zkp_fr_ap_vanishing_dev(uint64_t k, uint64_t out, uint64_t out_off) {
  return guarded([&](Context& c) {
    if (!k) throw InvalidArgument("zkp_fr_ap_vanishing_dev: k must be positive");
    ArenaScope scope;
    Fr* o = hptr(out, out_off, k + 1, "zkp_fr_ap_vanishing_dev");
    c.launches += ap_domain_build(c, k);
    fr_from_mont_kernel<<<GRID_1D(k + 1)>>>(g_ap.z.as<Fr>(), k + 1, o);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_fr_ap_lagrange_dev(uint64_t k, const uint8_t x[32], uint64_t out, uint64_t out_off) {
  return guarded([&](Context& c) {
    if (!k || !x) throw InvalidArgument("zkp_fr_ap_lagrange_dev: bad argument");
    ArenaScope scope;
    Fr* o = hptr(out, out_off, k, "zkp_fr_ap_lagrange_dev");
    // x on the domain itself: the basis is a unit vector (the general formula divides by zero there)
    bool small = true;
    for (int i = 8; i < 32; i++) small = small && x[i] == 0;
    uint64_t xv = 0;
    memcpy(&xv, x, 8);
    if (small && xv >= 1 && xv <= k) {
      CUDA_CHECK(cudaMemsetAsync(o, 0, k * sizeof(Fr), c.stream));
      Fr one_canon = host_fr_small(1);
      CUDA_CHECK(cudaMemcpyAsync(o + (xv - 1), &one_canon, sizeof(Fr), cudaMemcpyHostToDevice, c.stream));
      CUDA_CHECK(cudaStreamSynchronize(c.stream));
      return;
    }
    int launches = ap_domain_build(c, k);
    Fr* d = g_arena.alloc(k);
    Fr* pre = g_arena.alloc(k);
    Fr* inv = g_arena.alloc(k);
    Fr* zx = g_arena.alloc(1);
    ap_x_minus_kernel<<<GRID_1D(k)>>>(fr_from_bytes(x), k, d);
    CUDA_CHECK_LAUNCH();
    launches += 1 + scan_dev<false>(c, d, k, pre, zx);  // zx = prod_j (x - x_j) = Z(x)
    uint64_t T = (k + BATCH_INV_CHUNK - 1) / BATCH_INV_CHUNK;
    fr_batch_inverse_kernel<<<ceil_div(T, 128), 128, 0, c.stream>>>(d, k, T, 0, inv);
    CUDA_CHECK_LAUNCH();
    ap_lagrange_finish_kernel<<<GRID_1D(k)>>>(inv, g_ap.weights.as<Fr>(), zx, k, o);
    CUDA_CHECK_LAUNCH();
    c.launches += launches + 2;
  });
}

}  // extern "C"
