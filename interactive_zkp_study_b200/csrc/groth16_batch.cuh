// Batch Groth16 proving: the vector work of `count` proofs of one circuit in the same launches
// (zkp_groth16_quotient_batch_dev, zkp_groth16_batch_scalars_dev, zkp_sparse_matvec_many_dev,
// zkp_fr_ap_interpolate_many_dev).  Included once, by poly.cu, after qap.cuh: shares the arena, the divisor cache of
// zkp_groth16_quotient_dev and the cached M tree of the {1..k} domain.  Every entry computes, per proof, exactly
// what its single-proof counterpart computes (exact field arithmetic: same values, whatever the launch shape).
#pragma once

namespace zkp {

// out[j * 2^log_N + i] = i < len ? mont(in[j * len + i]) : 0   (canonical in, Montgomery out; total = count * 2^log_N)
__global__ void fr_pad_mont_many_kernel(const Fr* __restrict__ in, uint64_t len, uint32_t log_N, uint64_t total,
                                        Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx >> log_N, i = idx & ((uint64_t(1) << log_N) - 1);
  out[idx] = i < len ? in[j * len + i].to_mont() : Fr::zero();
}

// The reversed top of proof j's P - C, the operand of the power-series division (poly_divmod_dev's `ra`):
// out[j * 2^log_Nq + i] = P_j[lp - 1 - i] - C_j[lp - 1 - i] for i < m (C_j: len canonical coefficients, zero above),
// zero for m <= i < 2^log_Nq.  P: proof j's product at p[j * 2^log_N1], Montgomery.
__global__ void g16_rev_sub_many_kernel(const Fr* __restrict__ p, uint32_t log_N1, const Fr* __restrict__ cvec, uint64_t len,
                                        uint64_t lp, uint64_t m, uint32_t log_Nq, uint64_t total, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx >> log_Nq, i = idx & ((uint64_t(1) << log_Nq) - 1);
  Fr v = Fr::zero();
  if (i < m) {
    const uint64_t e = lp - 1 - i;
    v = p[(j << log_N1) + e];
    if (e < len) v = v - cvec[j * len + e].to_mont();
  }
  out[idx] = v;
}

// a[idx] *= b[idx mod 2^log_N]: one operand shared by every vector of the batch
__global__ void fr_mul_bcast_kernel(Fr* __restrict__ a, const Fr* __restrict__ b, uint32_t log_N, uint64_t total) {
  uint64_t idx = IDX64;
  if (idx < total) a[idx] = a[idx] * b[idx & ((uint64_t(1) << log_N) - 1)];
}

// h[j * m + i] = canonical(q_j[m - 1 - i]): un-reverse the truncated product (poly_divmod_dev's last reversal)
__global__ void g16_quot_out_many_kernel(const Fr* __restrict__ fq, uint32_t log_Nq, uint64_t m, uint64_t total,
                                         Fr* __restrict__ h) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / m, i = idx % m;
  h[idx] = fq[(j << log_Nq) + (m - 1 - i)].from_mont();
}

// The three scalar vectors of device_prover (_scalars_ab / _scalars_c) for proof j = idx / nC, row i = idx % nC:
//   A: uA | 1 | r     B: uB | 1 | s     C: r uB + s uA | r | rx_priv | H | s | s r
// All canonical; rs / ss canonical per proof.
__global__ void g16_batch_scalars_kernel(const Fr* __restrict__ uA, const Fr* __restrict__ uB, const Fr* __restrict__ H,
                                         const Fr* __restrict__ rx, const Fr* __restrict__ rs, const Fr* __restrict__ ss,
                                         uint64_t k, uint64_t mp, uint64_t nC, uint64_t total, Fr* __restrict__ scA,
                                         Fr* __restrict__ scB, Fr* __restrict__ scC) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / nC, i = idx % nC;
  const Fr r = rs[j], s = ss[j];
  if (i < k + 2) {
    Fr one = Fr::zero();
    one.v[0] = 1;
    scA[j * (k + 2) + i] = i < k ? uA[j * k + i] : i == k ? one : r;
    scB[j * (k + 2) + i] = i < k ? uB[j * k + i] : i == k ? one : s;
  }
  Fr v;
  if (i < k) v = uB[j * k + i] * r.to_mont() + uA[j * k + i] * s.to_mont();  // (x y R) R^-1 = x y, canonical
  else if (i == k) v = r;
  else if (i < k + 1 + mp) v = rx[j * mp + (i - k - 1)];
  else if (i + 2 < nC) v = H[j * (k - 1) + (i - k - 1 - mp)];
  else if (i + 2 == nC) v = s;
  else v = s * r.to_mont();
  scC[idx] = v;
}

// y[j * rows + r] = sum_e val[e] * vec[j * m + col[e]]: sparse_matvec_kernel over `count` witness vectors
__global__ void sparse_matvec_many_kernel(const uint32_t* __restrict__ row_ptr, const uint32_t* __restrict__ col,
                                          const Fr* __restrict__ val, const Fr* __restrict__ vec, uint64_t rows, uint64_t m,
                                          uint64_t total, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / rows, r = idx % rows;
  const Fr* v = vec + j * m;
  Fr acc = Fr::zero();
  for (uint32_t e = row_ptr[r]; e < row_ptr[r + 1]; e++) acc = acc + val[e] * v[col[e]];
  out[idx] = acc;
}

// ap_leaf_n_kernel for vector j = idx >> L: leaves y_j[i] * w[i] (* scale), zero beyond k
__global__ void ap_leaf_n_many_kernel(const Fr* __restrict__ y, const Fr* __restrict__ w, uint32_t L, uint64_t k,
                                      uint64_t total, int scaled, Fr scale_mont, Fr* __restrict__ lev) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx >> L, i = idx & ((uint64_t(1) << L) - 1);
  Fr v = Fr::zero();
  if (i < k) {
    v = y[j * k + i] * w[i];
    if (scaled) v = v * scale_mont;
  }
  lev[idx] = v;
}

// ap_combine_eval_kernel over `count` trees of K leaves back to back: the children's values (ev / odd) are
// per tree, the transformed M children (mch) are shared
__global__ void ap_combine_eval_many_kernel(const Fr* __restrict__ ev, const Fr* __restrict__ odd, const Fr* __restrict__ mch,
                                            uint32_t L, uint32_t log_s, uint64_t total, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t K = uint64_t(1) << L;
  const uint64_t base = idx & ~(K - 1), li = idx & (K - 1);
  const uint64_t s = uint64_t(1) << log_s, two_s = s << 1;
  const uint64_t p = li >> (log_s + 1), t = li & (two_s - 1);
  const Fr* src = ((t & 1) ? odd : ev) + base;
  const uint64_t h = t >> 1;
  const Fr nl = src[(2 * p) * s + h], nr = src[(2 * p + 1) * s + h];
  out[idx] = nl * mch[(2 * p + 1) * two_s + t] + nr * mch[(2 * p) * two_s + t];
}

// out[j * k + i] = in[j * 2^L + i], i < k
__global__ void fr_gather_rows_kernel(const Fr* __restrict__ in, uint32_t L, uint64_t k, uint64_t total, Fr* __restrict__ out) {
  uint64_t idx = IDX64;
  if (idx >= total) return;
  const uint64_t j = idx / k, i = idx % k;
  out[idx] = in[(j << L) + i];
}

// ap_interpolate for `count` value vectors (y_j at y + j * k, coefficients to out + j * k) in the same launches
static int ap_interpolate_many(Context& c, const Fr* y, uint64_t k, uint64_t count, const Fr* scale_mont, Fr* out) {
  int launches = ap_domain_build(c, k);
  const uint64_t K = g_ap.K;
  const uint32_t L = g_ap.L;
  const uint64_t total = count * K;
  Fr* ev = g_arena.alloc(total);
  Fr* odd = g_arena.alloc(total);
  Fr* nxt = g_arena.alloc(total);
  Fr* scratch = g_arena.alloc(total);
  ap_leaf_n_many_kernel<<<GRID_1D(total)>>>(y, g_ap.weights.as<Fr>(), L, k, total, scale_mont ? 1 : 0,
                                            scale_mont ? *scale_mont : host_fr_one_mont(), ev);
  CUDA_CHECK_LAUNCH();
  launches++;
  for (uint32_t l = 0; l < L; l++) {
    const Fr* mch = g_ap.mhat.as<Fr>() + (size_t)l * 2 * K;
    const Fr* odd_src = ev;
    if (l > 0) {
      FrBytes w = omega_for(l), shift = omega_for(l + 1);
      CUDA_CHECK(cudaMemcpyAsync(odd, ev, total * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
      launches += ntt_device_count(c, odd, scratch, l, w, true, nullptr, count << (L - l));
      launches += ntt_device_count(c, odd, scratch, l, w, false, &shift, count << (L - l));
      odd_src = odd;
    }
    ap_combine_eval_many_kernel<<<GRID_1D(total)>>>(ev, odd_src, mch, L, l, total, nxt);
    CUDA_CHECK_LAUNCH();
    launches++;
    Fr* t = ev;
    ev = nxt;
    nxt = t;
  }
  launches += ntt_device_count(c, ev, scratch, L, omega_for(L), true, nullptr, count);
  fr_gather_rows_kernel<<<GRID_1D(count * k)>>>(ev, L, k, count * k, out);
  CUDA_CHECK_LAUNCH();
  launches++;
  g_arena.free(ev);
  g_arena.free(odd);
  g_arena.free(nxt);
  g_arena.free(scratch);
  return launches;
}

static std::unique_ptr<Resource> new_scalars(uint64_t n) {
  auto r = std::make_unique<Resource>();
  r->kind = HandleKind::Scalars;
  r->n = n;
  r->buf.reserve_pooled(n ? n * 32 : 32);
  return r;
}

}  // namespace zkp

using namespace zkp;

extern "C" {

// count Groth16 quotients in one pass: batched product transforms, one shared cached divisor inverse (g_div_cache of
// zkp_groth16_quotient_dev) applied as a broadcast product, batched inverse transforms.  Quotient only.
int zkp_groth16_quotient_batch_dev(uint64_t a, uint64_t b, uint64_t cc, uint64_t len, uint32_t count, uint64_t z,
                                   uint64_t z_len, uint64_t* h_out) {
  return guarded([&](Context& c) {
    const char* what = "zkp_groth16_quotient_batch_dev";
    if (!h_out || !len || z_len < 2) throw InvalidArgument(std::string(what) + ": bad argument");
    const uint64_t lp = 2 * len - 1;
    if (lp < z_len) throw InvalidArgument(std::string(what) + ": divisor longer than the product");
    const uint64_t m = lp - z_len + 1;
    const uint32_t lg1 = log2_ceil(lp), lgq = log2_ceil(2 * m - 1);
    if (((uint64_t)count << lg1) >= (uint64_t(1) << 32) || ((uint64_t)count << lgq) >= (uint64_t(1) << 32))
      throw InvalidArgument(std::string(what) + ": count * transform size must be < 2^32");
    ArenaScope scope;
    Fr* da = hptr(a, 0, count * len, what);
    Fr* db = hptr(b, 0, count * len, what);
    Fr* dc = hptr(cc, 0, count * len, what);
    Fr* dzc = hptr(z, 0, z_len, what);
    auto hq = new_scalars(count * m);
    if (count && m) {
      int launches = 0;
      if (g_div_cache.z_handle != z || g_div_cache.z_len != z_len || g_div_cache.m != m) {
        g_div_cache.z_handle = z;
        g_div_cache.z_len = z_len;
        g_div_cache.m = m;
        g_div_cache.filled = false;
        g_div_cache.inv.reserve(m * sizeof(Fr));
        g_div_cache.inv_hat.reserve((size_t(1) << lgq) * sizeof(Fr));
      }
      if (!g_div_cache.filled) {  // rev(Z)^-1 mod x^m and its transform, as poly_divmod_dev fills them
        const uint64_t lrb = z_len < m ? z_len : m;
        Fr* dz = g_arena.alloc(z_len);
        Fr* rb = g_arena.alloc(lrb);
        fr_to_mont_kernel<<<GRID_1D(z_len)>>>(dzc, z_len, dz);
        CUDA_CHECK_LAUNCH();
        fr_reverse_kernel<<<GRID_1D(lrb)>>>(dz, z_len, lrb, rb);
        CUDA_CHECK_LAUNCH();
        launches += 2 + series_inverse_dev(c, rb, lrb, m, g_div_cache.inv.as<Fr>());
        const uint64_t Nq = uint64_t(1) << lgq;
        Fr* scratch = g_arena.alloc(Nq);
        CUDA_CHECK(cudaMemcpyAsync(g_div_cache.inv_hat.p, g_div_cache.inv.p, m * sizeof(Fr), cudaMemcpyDeviceToDevice, c.stream));
        CUDA_CHECK(cudaMemsetAsync(g_div_cache.inv_hat.as<Fr>() + m, 0, (Nq - m) * sizeof(Fr), c.stream));
        launches += ntt_device(c, g_div_cache.inv_hat.as<Fr>(), scratch, lgq, omega_for(lgq), false, nullptr);
        g_div_cache.filled = true;
        g_arena.free(scratch);
        g_arena.free(rb);
        g_arena.free(dz);
      }
      // P_j = uA_j * uB_j on 2^lg1 points
      const uint64_t t1 = (uint64_t)count << lg1, tq = (uint64_t)count << lgq;
      Fr* fa = g_arena.alloc(t1);
      Fr* fb = g_arena.alloc(t1);
      Fr* scratch = g_arena.alloc(t1 > tq ? t1 : tq);
      fr_pad_mont_many_kernel<<<GRID_1D(t1)>>>(da, len, lg1, t1, fa);
      CUDA_CHECK_LAUNCH();
      fr_pad_mont_many_kernel<<<GRID_1D(t1)>>>(db, len, lg1, t1, fb);
      CUDA_CHECK_LAUNCH();
      const FrBytes w1 = omega_for(lg1);
      launches += 2 + ntt_device_count(c, fa, scratch, lg1, w1, false, nullptr, count);
      launches += ntt_device_count(c, fb, scratch, lg1, w1, false, nullptr, count);
      fr_mul_inplace_kernel<<<GRID_1D(t1)>>>(fa, fb, t1);
      CUDA_CHECK_LAUNCH();
      launches += 1 + ntt_device_count(c, fa, scratch, lg1, w1, true, nullptr, count);
      // H_j = rev(rev(P_j - C_j) * rev(Z)^-1 mod x^m)
      Fr* fq = g_arena.alloc(tq);
      g16_rev_sub_many_kernel<<<GRID_1D(tq)>>>(fa, lg1, dc, len, lp, m, lgq, tq, fq);
      CUDA_CHECK_LAUNCH();
      const FrBytes wq = omega_for(lgq);
      launches += 1 + ntt_device_count(c, fq, scratch, lgq, wq, false, nullptr, count);
      fr_mul_bcast_kernel<<<GRID_1D(tq)>>>(fq, g_div_cache.inv_hat.as<Fr>(), lgq, tq);
      CUDA_CHECK_LAUNCH();
      launches += 1 + ntt_device_count(c, fq, scratch, lgq, wq, true, nullptr, count);
      g16_quot_out_many_kernel<<<GRID_1D(count * m)>>>(fq, lgq, m, count * m, hq->buf.as<Fr>());
      CUDA_CHECK_LAUNCH();
      launches++;
      c.launches += launches;
    }
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *h_out = registry().put(std::move(hq));
  });
}

// The A, B and C scalar vectors of `count` proofs (device_prover._scalars_ab / _scalars_c) in one launch.
// uA, uB: count * k coefficients; h: count * (k - 1); rx: count * m_priv; rs, ss: count canonical host scalars each.
int zkp_groth16_batch_scalars_dev(uint64_t ua, uint64_t ub, uint64_t h, uint64_t rx, uint64_t k, uint64_t m_priv,
                                  uint32_t count, const uint8_t* rs, const uint8_t* ss, uint64_t* out_a, uint64_t* out_b,
                                  uint64_t* out_c) {
  return guarded([&](Context& c) {
    const char* what = "zkp_groth16_batch_scalars_dev";
    if (!k || !out_a || !out_b || !out_c || (count && (!rs || !ss))) throw InvalidArgument(std::string(what) + ": bad argument");
    const uint64_t nC = 2 * k + 2 + m_priv;
    Fr* pa = hptr(ua, 0, (uint64_t)count * k, what);
    Fr* pb = hptr(ub, 0, (uint64_t)count * k, what);
    Fr* ph = k > 1 ? hptr(h, 0, (uint64_t)count * (k - 1), what) : nullptr;
    Fr* px = m_priv ? hptr(rx, 0, (uint64_t)count * m_priv, what) : nullptr;
    auto A = new_scalars((uint64_t)count * (k + 2));
    auto B = new_scalars((uint64_t)count * (k + 2));
    auto C = new_scalars((uint64_t)count * nC);
    if (count) {
      ArenaScope scope;
      Fr* drs = g_arena.alloc(2 * (uint64_t)count);
      CUDA_CHECK(cudaMemcpyAsync(drs, rs, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
      CUDA_CHECK(cudaMemcpyAsync(drs + count, ss, (size_t)count * 32, cudaMemcpyHostToDevice, c.stream));
      const uint64_t total = (uint64_t)count * nC;
      g16_batch_scalars_kernel<<<GRID_1D(total)>>>(pa, pb, ph, px, drs, drs + count, k, m_priv, nC, total, A->buf.as<Fr>(),
                                                  B->buf.as<Fr>(), C->buf.as<Fr>());
      CUDA_CHECK_LAUNCH();
      c.launches++;
    }
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *out_a = registry().put(std::move(A));
    *out_b = registry().put(std::move(B));
    *out_c = registry().put(std::move(C));
  });
}

int zkp_sparse_matvec_many_dev(uint64_t matrix, uint64_t vec, uint64_t vec_off, uint64_t out, uint64_t out_off,
                               uint32_t count) {
  return guarded([&](Context& c) {
    Resource* m = need(matrix, HandleKind::Sparse, "zkp_sparse_matvec_many_dev");
    Fr* v = hptr(vec, vec_off, (uint64_t)count * m->cols, "zkp_sparse_matvec_many_dev");
    Fr* o = hptr(out, out_off, (uint64_t)count * m->n, "zkp_sparse_matvec_many_dev");
    const uint64_t total = (uint64_t)count * m->n;
    if (!total) return;
    sparse_matvec_many_kernel<<<GRID_1D(total)>>>(m->aux[0].as<uint32_t>(), m->aux[1].as<uint32_t>(), m->buf.as<Fr>(), v,
                                                  m->n, m->cols, total, o);
    CUDA_CHECK_LAUNCH();
    c.launches++;
  });
}

int zkp_fr_ap_interpolate_many_dev(uint64_t values, uint64_t off, uint64_t k, uint32_t count, const uint8_t* scale,
                                   uint64_t out, uint64_t out_off) {
  return guarded([&](Context& c) {
    const char* what = "zkp_fr_ap_interpolate_many_dev";
    if (!k) throw InvalidArgument(std::string(what) + ": k must be positive");
    ArenaScope scope;
    Fr* y = hptr(values, off, (uint64_t)count * k, what);
    Fr* o = hptr(out, out_off, (uint64_t)count * k, what);
    if (!count) return;
    const uint32_t L = log2_ceil(k) ? log2_ceil(k) : 1;
    if (((uint64_t)count << L) >= (uint64_t(1) << 32)) throw InvalidArgument(std::string(what) + ": count * 2^ceil(log2 k) must be < 2^32");
    Fr sm;
    if (scale) sm = host_to_mont(c, scale);
    c.launches += ap_interpolate_many(c, y, k, count, scale ? &sm : nullptr, o);
  });
}

}  // extern "C"
