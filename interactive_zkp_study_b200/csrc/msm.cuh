// Pippenger multi-scalar multiplication, templated on the coordinate field (Fp -> G1, Fp2 -> G2).
//
// Replaces the reference's MSM-shaped Python loops: kzg.commit
// (/root/reference/zkp/plonk/kzg.py:59-67) and the inner loops of proof_a/proof_b/proof_c
// (/root/reference/zkp/groth16/proving.py:27-31,39-43,56-60,66-73), each of which is
// "sum_i scalar_i * point_i" done as one affine double-and-add per term.
//
// Stages (all on the device, one stream):
//   1. digits     : reduce each scalar mod r, cut it into W signed c-bit digits d in
//                   [-2^(c-1), 2^(c-1)], histogram the (window, |d|) buckets.
//   2. sort       : counting sort of (bucket, point index | sign) pairs: exclusive scan of the
//                   histogram + atomic-cursor scatter.  Order inside a bucket is irrelevant
//                   (the group is commutative and the final affine point is unique).
//   3. accumulate : each bucket's run of point indices is cut into tasks of <= 64 entries, the tasks
//                   are counting-sorted by length so a warp walks runs of equal length, one thread
//                   per task sums its points with XYZZ mixed additions (negating y for negative
//                   digits); buckets with several tasks are folded (block-per-bucket if very many).
//   4. reduce     : per window sum_b (b+1)*B_b by a weighted-sum recursion (V = sum_i i*A_i +
//                   sum_i E_i is preserved level to level: radix 8 while wide, radix 2 on two warps
//                   when narrow), then Horner over the windows, one binary-Euclid inversion, out of
//                   Montgomery form.
//
// Static tables (SRS / CRS) can be window-precomputed: T[w][i] = 2^(c*w) * P_i.  Then every window's
// digits weigh the same, all windows share ONE bucket set (stage 4 reduces a single window) and the
// 254-step doubling chain of the Horner disappears; the digits kernel just maps (w, i) to entry
// w*n + i of the big table.
//
// HBM layout: points AoS affine Montgomery (64 B G1 / 128 B G2, 16-byte aligned -> LDG.128),
// scalars canonical 8xu32, codes/sorted W*n u32, task records uint4, partials / buckets XYZZ.
#pragma once
#include "common.cuh"
#include "ec.cuh"
#include "ec_quad.cuh"
#include "msm_acc.cuh"

namespace zkp {

static constexpr uint32_t MSM_INVALID = 0xffffffffu;
static constexpr int MSM_MAX_C = 20;
static constexpr int MSM_SCALAR_BITS = 255;  // 254-bit scalars + 1 for the signed-digit carry

struct MsmPlan {
  int c;              // window bits
  int W;              // number of windows
  uint32_t B;         // buckets per window = 2^(c-1)
  uint32_t nbuckets;  // W * B
};

inline MsmPlan msm_plan(uint64_t n, int force_c = 0) {
  int c;
  if (force_c) c = force_c;
  else {
    int lg = 0;
    while ((1ull << (lg + 1)) <= n) lg++;
    c = lg - 4;
    if (c < 4) c = 4;
    if (c > 16) c = 16;  // automatic choice; explicit widths up to MSM_MAX_C are accepted
  }
  MsmPlan p;
  p.c = c;
  p.W = (MSM_SCALAR_BITS + c - 1) / c;
  p.B = 1u << (c - 1);
  p.nbuckets = (uint32_t)p.W * p.B;
  return p;
}

// Window width for a window-precomputed table of n points (zkp_*_table_precompute with window_bits = 0).
// Measured on B200 (tools/c_sweep.py): wider windows mean fewer additions per point (ceil(255/c)) but
// 2^(c-1) buckets to reduce, and only widths whose TOP window is well filled are good -- all windows
// share one bucket set, so a top window of t bits piles n / 2^t extra entries on each of its few
// buckets (c = 18: t = 3, 30 % slower than c = 17 at every size).  255 = 15*17 = 12*20 + 15 = 17*15 =
// 19*13 + 8 = 25*10 + 5 = 36*7 + 3.
inline int msm_auto_precomputed_c(uint64_t n) {
  if (n >= 741455) return 20;  // 2^19.5
  if (n >= (1u << 14)) return 17;
  if (n >= (1u << 12)) return 15;
  if (n >= 96) return 13;
  if (n >= 24) return 10;
  return 7;
}

// ---------------------------------------------------------------- stage 1: digits + histogram
// wstride: distance between the bucket sets of consecutive windows (B for a plain table; 0 for a
// window-precomputed table, where all windows share one bucket set).
static __global__ void msm_digits_kernel(const uint32_t* __restrict__ scalars, uint64_t n, uint64_t i0, uint64_t i1, int c,
                                         int W, uint32_t B, uint32_t wstride, uint32_t* __restrict__ codes,
                                         uint32_t* __restrict__ hist);

// ---------------------------------------------------------------- exclusive scan (u32), 3 kernels
static constexpr int SCAN_BLOCK = 1024;
static constexpr int SCAN_ITEMS = 4;
static constexpr int SCAN_TILE = SCAN_BLOCK * SCAN_ITEMS;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t val, uint32_t* total) {
  __shared__ uint32_t warp_sums[32];
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t inc = val;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_sums[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    uint32_t ws = lane < ((blockDim.x + 31) >> 5) ? warp_sums[lane] : 0u;  // blocks of fewer than 32 warps
    uint32_t winc = ws;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    warp_sums[lane] = winc - ws;  // exclusive warp offsets
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  uint32_t r = inc - val + warp_sums[wid];
  __syncthreads();
  return r;
}

static __global__ void scan_tile_sums_kernel(const uint32_t* __restrict__ in, uint32_t n, uint32_t* __restrict__ tile_sums) {
  __shared__ uint32_t total;
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++)
    if (base + k < n) s += in[base + k];
  block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// single block: exclusive scan of up to SCAN_TILE*? tile sums, sequential over chunks of 1024
static __global__ void scan_tile_offsets_kernel(uint32_t* __restrict__ tile_sums, uint32_t ntiles) {
  __shared__ uint32_t total;
  uint32_t running = 0;
  for (uint32_t base = 0; base < ntiles; base += SCAN_BLOCK) {
    uint32_t idx = base + threadIdx.x;
    uint32_t v = idx < ntiles ? tile_sums[idx] : 0;
    uint32_t ex = block_exclusive_scan(v, &total);
    if (idx < ntiles) tile_sums[idx] = ex + running;
    running += total;
    __syncthreads();
  }
}

// out[i] = exclusive prefix; out[n] = grand total
static __global__ void scan_apply_kernel(const uint32_t* __restrict__ in, uint32_t n, const uint32_t* __restrict__ tile_offsets,
                                  uint32_t* __restrict__ out) {
  __shared__ uint32_t total;
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS];
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    v[k] = (base + k < n) ? in[base + k] : 0;
    s += v[k];
  }
  uint32_t ex = block_exclusive_scan(s, &total) + tile_offsets[blockIdx.x];
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    if (base + k < n) out[base + k] = ex;
    ex += v[k];
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == SCAN_BLOCK - 1) out[n] = ex;
}

// ---------------------------------------------------------------- stage 2: scatter
// Plain table: the entry is the point index i.  Window-precomputed table (pre_stride != 0): the entry
// is the index of 2^(c*w) * P_i inside the [w][i] table, w * pre_stride + pre_offset + i.
static __global__ void msm_scatter_kernel(const uint32_t* __restrict__ codes, uint64_t total, uint64_t n,
                                   uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted,
                                   uint32_t pre_stride, uint32_t pre_offset, uint32_t idx_base) {
  uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  uint32_t code = codes[idx];
  if (code == MSM_INVALID) return;
  uint32_t i = (uint32_t)(idx % n) + idx_base;  // idx_base: first point of this part of a part-streamed MSM
  if (pre_stride) i += (uint32_t)(idx / n) * pre_stride + pre_offset;
  uint32_t pos = atomicAdd(&cursor[code >> 1], 1u);
  sorted[pos] = i | ((code & 1u) << 31);
}

// The same for the codes of msm_digits_many_kernel: entry idx = w * N + j * n + i is point i of window w, shared by
// all MSMs.
static __global__ void msm_scatter_many_kernel(const uint32_t* __restrict__ codes, uint64_t total, uint64_t N, uint64_t n,
                                               uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted,
                                               uint32_t pre_stride, uint32_t pre_offset) {
  uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  uint32_t code = codes[idx];
  if (code == MSM_INVALID) return;
  uint32_t i = (uint32_t)((idx % N) % n);
  if (pre_stride) i += (uint32_t)(idx / N) * pre_stride + pre_offset;
  uint32_t pos = atomicAdd(&cursor[code >> 1], 1u);
  sorted[pos] = i | ((code & 1u) << 31);
}

// ---------------------------------------------------------------- digit recoding helpers
// Canonical scalar i reduced mod r into s[0..8] (s[8] = 0): the group has order r, so
// k*P == (k mod r)*P (field.py:88).  2^256 / r < 6.
__device__ __forceinline__ void msm_load_scalar(const uint32_t* __restrict__ scalars, uint64_t i, uint32_t (&s)[9]) {
  const uint4* sp = reinterpret_cast<const uint4*>(scalars + 8 * i);
  uint4 lo = sp[0], hi = sp[1];
  s[0] = lo.x; s[1] = lo.y; s[2] = lo.z; s[3] = lo.w;
  s[4] = hi.x; s[5] = hi.y; s[6] = hi.z; s[7] = hi.w;
  s[8] = 0;
  for (int it = 0; it < 6; it++) {
    uint32_t t[8];
    uint32_t borrow = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      uint64_t d = (uint64_t)s[k] - FrParams::MOD_(k) - borrow;
      t[k] = (uint32_t)d;
      borrow = (uint32_t)(d >> 63);
    }
    if (borrow) break;
#pragma unroll
    for (int k = 0; k < 8; k++) s[k] = t[k];
  }
}

// Signed c-bit digit of window w given the carry of the windows below; returns the code
// (bucket << 1 | sign) or MSM_INVALID for a zero digit, and updates the carry.
__device__ __forceinline__ uint32_t msm_digit_code(const uint32_t (&s)[9], int w, int c, uint32_t B, uint32_t wstride,
                                                   uint32_t& carry) {
  int pos = w * c;
  int word = pos >> 5, sh = pos & 31;
  uint32_t v = 0;
  if (word < 8) {
    uint64_t two = (uint64_t)s[word] | ((uint64_t)s[word + 1] << 32);
    v = (uint32_t)(two >> sh) & ((1u << c) - 1);
  }
  v += carry;
  if (v > B) {  // digit = v - 2^c (negative), |digit| = 2^c - v in [1, B-1]
    uint32_t mag = (1u << c) - v;
    carry = 1;
    return mag ? ((((uint32_t)w * wstride + (mag - 1)) << 1) | 1u) : MSM_INVALID;
  }
  carry = 0;
  return v ? (((uint32_t)w * wstride + (v - 1)) << 1) : MSM_INVALID;
}

// scalars [i0, i1) of the n of this MSM (the host-scalar entry points upload and recode in chunks)
static __global__ void msm_digits_kernel(const uint32_t* __restrict__ scalars, uint64_t n, uint64_t i0, uint64_t i1, int c,
                                         int W, uint32_t B, uint32_t wstride, uint32_t* __restrict__ codes,
                                         uint32_t* __restrict__ hist) {
  uint64_t i = i0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= i1) return;
  uint32_t s[9];
  msm_load_scalar(scalars, i, s);
  uint32_t carry = 0;
  for (int w = 0; w < W; w++) {
    uint32_t code = msm_digit_code(s, w, c, B, wstride, carry);
    codes[(uint64_t)w * n + i] = code;
    if (code != MSM_INVALID) atomicAdd(&hist[code >> 1], 1u);
  }
}

// Many MSMs over one point range (MsmEngine::run_many): scalar q = j * n + i of the N = count * n back-to-back
// vectors belongs to MSM j and point i; MSM j owns buckets [j * per_msm, (j + 1) * per_msm).  codes[w * N + q].
static __global__ void msm_digits_many_kernel(const uint32_t* __restrict__ scalars, uint64_t n, uint64_t N, int c, int W,
                                              uint32_t B, uint32_t wstride, uint32_t per_msm,
                                              uint32_t* __restrict__ codes, uint32_t* __restrict__ hist) {
  uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= N) return;
  const uint32_t base = (uint32_t)(q / n) * per_msm;
  uint32_t s[9];
  msm_load_scalar(scalars, q, s);
  uint32_t carry = 0;
  for (int w = 0; w < W; w++) {
    uint32_t code = msm_digit_code(s, w, c, B, wstride, carry);
    if (code != MSM_INVALID) {
      code += base << 1;
      atomicAdd(&hist[code >> 1], 1u);
    }
    codes[(uint64_t)w * N + q] = code;
  }
}

// ---------------------------------------------------------------- stage 3: bucket accumulation
// Load balance: a bucket's run of entries is cut into tasks of at most MSM_TASK_LEN entries; tasks
// are counting-sorted by length (longest first) so the 32 lanes of a warp walk runs of equal length
// whatever the scalar distribution (uniform scalars: Poisson(32) runs; the top window and
// structured inputs: a few huge buckets).  One thread per task; buckets with several tasks are
// folded afterwards.
static constexpr uint32_t MSM_TASK_LEN = 64;
static constexpr uint32_t MSM_DIRECT = 0x80000000u;
#ifndef MSM_ACC_MIN_BLOCKS
#define MSM_ACC_MIN_BLOCKS 4  // resident 128-thread blocks per SM the G1 accumulate kernel is compiled for
#endif
#ifndef MSM_ACC_MIN_BLOCKS_G2
#define MSM_ACC_MIN_BLOCKS_G2 2
#endif
// 32-byte coordinates (G1): 122 registers, 4 blocks/SM (5 or 6 blocks, 96 / 80 registers with ~100 bytes of spills,
// measured 1-2 % slower again in round 2: the kernel is bound by the IMAD pipe and its dependent carry chains, not by
// occupancy); 64-byte coordinates (G2) need ~230 registers and stay at 2 blocks per SM.
template <class F>
struct AccMinBlocks {
  static constexpr int value = sizeof(F) == 32 ? MSM_ACC_MIN_BLOCKS : MSM_ACC_MIN_BLOCKS_G2;
};

// light_max != 0: buckets of up to light_max entries belong to the affine tree (msm_tree.cuh) and get no task
static __global__ void msm_task_count_kernel(const uint32_t* __restrict__ offsets, uint32_t nbuckets,
                                             uint32_t* __restrict__ ntasks, uint32_t light_max) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nbuckets) return;
  uint32_t cnt = offsets[b + 1] - offsets[b];
  if (cnt <= light_max) cnt = 0;
  ntasks[b] = (cnt + MSM_TASK_LEN - 1) / MSM_TASK_LEN;
}

// len_hist[MSM_TASK_LEN - len] counts tasks of each length (descending order of length)
static __global__ void msm_task_hist_kernel(const uint32_t* __restrict__ offsets, uint32_t nbuckets,
                                            uint32_t* __restrict__ len_hist, uint32_t light_max) {
  __shared__ uint32_t h[MSM_TASK_LEN + 1];
  for (uint32_t k = threadIdx.x; k <= MSM_TASK_LEN; k += blockDim.x) h[k] = 0;
  __syncthreads();
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nbuckets) {
    uint32_t cnt = offsets[b + 1] - offsets[b];
    if (cnt <= light_max) cnt = 0;
    uint32_t full = cnt / MSM_TASK_LEN, rem = cnt % MSM_TASK_LEN;
    if (full) atomicAdd(&h[0], full);
    if (rem) atomicAdd(&h[MSM_TASK_LEN - rem], 1u);
  }
  __syncthreads();
  for (uint32_t k = threadIdx.x; k <= MSM_TASK_LEN; k += blockDim.x)
    if (h[k]) atomicAdd(&len_hist[k], h[k]);
}

// single warp: exclusive scan of the MSM_TASK_LEN+1 length bins -> cursors
static __global__ void msm_task_bins_kernel(uint32_t* __restrict__ len_hist) {
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (uint32_t k = 0; k <= MSM_TASK_LEN; k++) {
      uint32_t v = len_hist[k];
      len_hist[k] = run;
      run += v;
    }
  }
}

// task record: x = bucket, y = first entry, z = length, w = slot in the partial-sum array, or
// MSM_DIRECT | bucket when the task is the bucket's only one: its sum then IS the bucket and the
// accumulate kernel stores it there (no copy through the partial array, nothing left for the fold)
static __global__ void msm_task_emit_kernel(const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ task_base,
                                            uint32_t nbuckets, uint32_t* __restrict__ len_cursor,
                                            uint4* __restrict__ tasks, uint32_t light_max) {
  __shared__ uint32_t h[MSM_TASK_LEN + 1];     // block-local count per bin
  __shared__ uint32_t base[MSM_TASK_LEN + 1];  // block's reserved start per bin
  for (uint32_t k = threadIdx.x; k <= MSM_TASK_LEN; k += blockDim.x) h[k] = 0;
  __syncthreads();
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t beg = 0, cnt = 0, full = 0, rem = 0, r_full = 0, r_rem = 0;
  if (b < nbuckets) {
    beg = offsets[b];
    cnt = offsets[b + 1] - beg;
    if (cnt <= light_max) cnt = 0;
    full = cnt / MSM_TASK_LEN;
    rem = cnt % MSM_TASK_LEN;
    if (full) r_full = atomicAdd(&h[0], full);
    if (rem) r_rem = atomicAdd(&h[MSM_TASK_LEN - rem], 1u);
  }
  __syncthreads();
  for (uint32_t k = threadIdx.x; k <= MSM_TASK_LEN; k += blockDim.x)
    base[k] = h[k] ? atomicAdd(&len_cursor[k], h[k]) : 0;
  __syncthreads();
  if (b < nbuckets) {
    uint32_t tb = task_base[b];
    const bool single = full + (rem ? 1u : 0u) == 1u;
    for (uint32_t k = 0; k < full; k++)
      tasks[base[0] + r_full + k] = make_uint4(b, beg + k * MSM_TASK_LEN, MSM_TASK_LEN, single ? (MSM_DIRECT | b) : tb + k);
    if (rem)
      tasks[base[MSM_TASK_LEN - rem] + r_rem] = make_uint4(b, beg + full * MSM_TASK_LEN, rem, single ? (MSM_DIRECT | b) : tb + full);
  }
}

template <class F, int OUTLINE = 0>
__global__ void __launch_bounds__(128, AccMinBlocks<F>::value) msm_accumulate_kernel(const Affine<F>* __restrict__ pts,
                                                              const uint32_t* __restrict__ sorted,
                                                              const uint4* __restrict__ tasks,
                                                              const uint32_t* __restrict__ ntasks_ptr,
                                                              XYZZ<F>* __restrict__ partials,
                                                              XYZZ<F>* __restrict__ buckets, bool cont) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= *ntasks_ptr) return;  // the task count is data dependent and stays on the device
  uint4 task = tasks[t];
  uint32_t beg = task.y, end = task.y + task.z;
  // cont: a later part of a part-streamed MSM (MsmEngine::run): the bucket already holds the earlier parts' sum
  // and a bucket that is one task continues from it
  XYZZ<F> acc = XYZZ<F>::inf();
  if (cont && (task.w & MSM_DIRECT)) acc = buckets[task.w & ~MSM_DIRECT];
  for (uint32_t k = beg; k < end; k++) {
    uint32_t e = sorted[k];
    Affine<F> p = pts[e & 0x7fffffffu];
    if (e >> 31) p.y = p.y.neg();
    acc_madd<F, OUTLINE>(acc, p);
  }
  if (task.w & MSM_DIRECT) buckets[task.w & ~MSM_DIRECT] = acc;
  else partials[task.w] = acc;
}

// buckets[b] = sum of its tasks' partial sums; empty buckets become infinity, single-task buckets were
// already written by the accumulate kernel.  Buckets with more than
// MSM_FOLD_SERIAL partials (skewed scalars, or a top window that only uses a few buckets) are queued
// for the block-per-bucket kernel below so that no single thread walks thousands of partials.
static constexpr uint32_t MSM_FOLD_SERIAL = 24;
template <class F>
__global__ void __launch_bounds__(128) msm_bucket_fold_kernel(const XYZZ<F>* __restrict__ partials,
                                                               const uint32_t* __restrict__ task_base, uint32_t nbuckets,
                                                               XYZZ<F>* __restrict__ buckets, uint32_t* __restrict__ heavy_count,
                                                               uint32_t* __restrict__ heavy_list, uint32_t serial_limit,
                                                               bool tree, bool cont) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nbuckets) return;
  uint32_t t0 = task_base[b], t1 = task_base[b + 1];
  if (t1 - t0 == 1) return;  // a single task: the accumulate kernel wrote the bucket itself
  if ((tree || cont) && t1 == t0) return;  // no task at all: the affine tree wrote the bucket (or its infinity) /
                                           // a later part of a part-streamed MSM adds nothing to it
  if (t1 - t0 > serial_limit) {
    heavy_list[atomicAdd(heavy_count, 1u)] = b;
    return;
  }
  XYZZ<F> acc = XYZZ<F>::inf();
  if (t1 > t0) acc = partials[t0];
  for (uint32_t t = t0 + 1; t < t1; t++) acc.add(partials[t]);
  if (cont) acc.add(buckets[b]);
  buckets[b] = acc;
}

template <class F>
__global__ void __launch_bounds__(128) msm_bucket_fold_heavy_kernel(const XYZZ<F>* __restrict__ partials,
                                                                     const uint32_t* __restrict__ task_base,
                                                                     const uint32_t* __restrict__ heavy_count,
                                                                     const uint32_t* __restrict__ heavy_list,
                                                                     XYZZ<F>* __restrict__ buckets, bool cont) {
  __shared__ XYZZ<F> sm[128];
  uint32_t count = *heavy_count;
  for (uint32_t h = blockIdx.x; h < count; h += gridDim.x) {
    uint32_t b = heavy_list[h];
    uint32_t t0 = task_base[b], t1 = task_base[b + 1];
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t t = t0 + threadIdx.x; t < t1; t += 128) acc.add(partials[t]);
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s > 0; s >>= 1) {
      if ((int)threadIdx.x < s) {
        acc.add(sm[threadIdx.x + s]);
        sm[threadIdx.x] = acc;
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      if (cont) acc.add(buckets[b]);
      buckets[b] = acc;
    }
    __syncthreads();
  }
}

}  // namespace zkp
#include "msm_tree.cuh"
namespace zkp {

// Window-precomputed tables: T[w][i] = 2^(c*w) * P_i, so every window's digits weigh the same and all
// windows share ONE bucket set (no per-window sums, no final doubling chain).
// cur[i] <- 2^c * cur[i]   (XYZZ, c doublings)
template <class F>
__global__ void __launch_bounds__(128) msm_pre_shift_kernel(XYZZ<F>* __restrict__ cur, uint64_t n, int c) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  XYZZ<F> p = cur[i];
  if (!p.is_inf())
    for (int k = 0; k < c; k++) p = p.dbl();
  cur[i] = p;
}
template <class F>
__global__ void msm_pre_lift_kernel(const Affine<F>* __restrict__ pts, uint64_t n, XYZZ<F>* __restrict__ cur) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) cur[i] = XYZZ<F>::from_affine(pts[i]);
}
// out[i] = affine(cur[i]) with one inversion per PRE_BATCH points (Montgomery's trick, strided).
static constexpr int PRE_BATCH = 16;
template <class F>
__global__ void __launch_bounds__(128) msm_pre_affine_kernel(const XYZZ<F>* __restrict__ cur, uint64_t n, uint64_t T,
                                                              Affine<F>* __restrict__ out) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  F pre[PRE_BATCH];
  F acc = F::one();
  int cnt = 0;
  for (uint64_t i = t; i < n && cnt < PRE_BATCH; i += T, cnt++) {
    pre[cnt] = acc;
    const XYZZ<F>& p = cur[i];
    if (!p.zz.is_zero()) acc = acc * (p.zz * p.zzz);
  }
  F inv = acc.inv();
  for (int k = cnt - 1; k >= 0; k--) {
    uint64_t i = t + (uint64_t)k * T;
    XYZZ<F> p = cur[i];
    Affine<F> a = Affine<F>::inf();
    if (!p.zz.is_zero()) {
      F d = inv * pre[k];         // 1 / (zz * zzz)
      inv = inv * (p.zz * p.zzz);
      a.x = p.x * (d * p.zzz);    // x / zz
      a.y = p.y * (d * p.zz);     // y / zzz
    }
    out[i] = a;
  }
}

// ---------------------------------------------------------------- stage 4: weighted-sum recursion
// Per window: items (A_i, E_i), i < n_in, value V = sum_i i*A_i + sum_i E_i.  One thread per chunk
// of L items j: A'_j = L * sum A_i, E'_j = sum E_i + sum_i (i mod L) * A_i; V is unchanged with
// n_in/L items.  E == nullptr means E_i = A_i (first level: bucket b has weight b+1).
// 64-thread blocks at 202 registers (5 resident blocks); capped at 170 registers for 6 blocks the level measured
// 0.39 ms instead of 0.36 (round 2)
template <class F>
__global__ void __launch_bounds__(64) msm_ws_level_kernel(const XYZZ<F>* __restrict__ A, const XYZZ<F>* __restrict__ E,
                                                            uint32_t n_in, uint32_t L, int logL, uint32_t n_windows,
                                                            XYZZ<F>* __restrict__ A_out, XYZZ<F>* __restrict__ E_out) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t T = n_in / L;
  if (t >= T * n_windows) return;
  uint32_t w = t / T, j = t % T;
  const XYZZ<F>* a = A + (uint64_t)w * n_in + (uint64_t)j * L;
  XYZZ<F> acc = XYZZ<F>::inf(), run = XYZZ<F>::inf();
  for (uint32_t i = L - 1; i >= 1; i--) {
    acc.add(a[i]);
    run.add(acc);
  }
  acc.add(a[0]);
  if (E) {
    const XYZZ<F>* e = E + (uint64_t)w * n_in + (uint64_t)j * L;
    for (uint32_t i = 0; i < L; i++) run.add(e[i]);
  } else {
    run.add(acc);
  }
  for (int k = 0; k < logL; k++) acc = acc.dbl();
  A_out[t] = acc;
  E_out[t] = run;
}

// Radix-2 level of the same recursion with the two outputs on two threads, so a level is two
// group operations deep: role 0: A' = 2*(A0+A1); role 1: E' = E0 + E1 + A1 (first level: A0 + 2*A1).
// Used once the item count is too small to fill the machine and latency is all that matters.
template <class F>
__global__ void __launch_bounds__(64) msm_ws2_kernel(const XYZZ<F>* __restrict__ A, const XYZZ<F>* __restrict__ E,
                                                      uint32_t n_in, uint32_t n_windows, XYZZ<F>* __restrict__ A_out,
                                                      XYZZ<F>* __restrict__ E_out) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t T = n_in / 2;
  // roles are split by warp (not by lane) so a warp never executes both formulas
  uint32_t warp = t >> 5, lane = t & 31;
  uint32_t chunk = (warp >> 1) * 32 + lane, role = warp & 1;
  if (chunk >= T * n_windows) return;
  uint32_t w = chunk / T, j = chunk % T;
  const XYZZ<F>* a = A + (uint64_t)w * n_in + 2 * (uint64_t)j;
  if (role == 0) {
    XYZZ<F> acc = a[0];
    acc.add(a[1]);
    A_out[chunk] = acc.dbl();
  } else {
    XYZZ<F> r;
    if (E) {
      const XYZZ<F>* e = E + (uint64_t)w * n_in + 2 * (uint64_t)j;
      r = e[0];
      r.add(e[1]);
      r.add(a[1]);
    } else {
      r = a[1].dbl();
      r.add(a[0]);
    }
    E_out[chunk] = r;
  }
}

// The narrow levels, fused: a block takes a segment of `seg` consecutive items (A_i, E_i) of one window
// and runs log2(seg) radix-2 levels on it out of shared memory (chunk j of a level reads items 2j, 2j+1
// and writes item j, so the recursion never leaves the segment).  Every group operation runs on a quad
// of lanes (ec_quad.cuh: ~4 product latencies per addition instead of 14); a warp of role 0
// (A' = 2(A0+A1)) and a warp of role 1 (E' = E0+E1+A1) serve 8 chunks.  65536 buckets -> 1 item in
// three launches of the old radix-2 kernel (throughput-bound levels) plus two launches of this one,
// instead of sixteen launches each two additions deep on a lone thread.
template <class F>
struct WsFused {
  static constexpr int SEG = sizeof(F) == 32 ? 128 : 64;  // items per block
  // G1: 256 threads, so that the kernel may use 168 registers -- under the 128-register cap of 512 threads it
  // spilled 800 bytes into a latency-bound loop; the first level (64 chunks x 2 roles x 4 lanes) then takes two
  // sweeps, every later level one.  G2 needs the 255-register limit either way and keeps 4 threads per item.
  static constexpr int THREADS = sizeof(F) == 32 ? SEG * 2 : SEG * 4;
  static constexpr int SMEM = 3 * SEG * (int)sizeof(XYZZ<F>);  // current level (A, E: 2 SEG items) + next level (SEG items)
};
template <class F>
__global__ void __launch_bounds__(WsFused<F>::THREADS) msm_ws2_fused_kernel(const XYZZ<F>* __restrict__ A,
                                                                            const XYZZ<F>* __restrict__ E, uint32_t seg,
                                                                            XYZZ<F>* __restrict__ A_out,
                                                                            XYZZ<F>* __restrict__ E_out) {
  extern __shared__ uint4 ws_smem[];
  constexpr int SEG = WsFused<F>::SEG;
  // a level reads (ca, ce) and writes (na, ne), half as many items: no operand is overwritten inside a level and
  // one barrier per level is enough; then the two pairs swap (SEG + SEG items in the first, SEG/2 + SEG/2 in the second)
  XYZZ<F>* ca = reinterpret_cast<XYZZ<F>*>(ws_smem);
  XYZZ<F>* ce = ca + SEG;
  XYZZ<F>* na = ce + SEG;
  XYZZ<F>* ne = na + SEG / 2;
  const uint64_t base = (uint64_t)blockIdx.x * seg;
  if (!E) E = A;  // first level of the recursion: E_i = A_i (bucket b weighs b + 1)
  for (uint32_t i = threadIdx.x; i < seg; i += blockDim.x) {
    ca[i] = A[base + i];
    ce[i] = E[base + i];
  }
  __syncthreads();
  // the warp index as a broadcast: the compiler then knows that `role` and `warp_live` are the same for the whole
  // warp, the branches on them are uniform and the shuffles of the quad operations inside need no reconvergence
  // guard (with threadIdx.x >> 5 every pair of SHFL sat between a WARPSYNC and an ENDCOLLECTIVE: 580 of them)
  const uint32_t warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const uint32_t role = warp & 1;
  const int ql = lane & 3;
  const uint32_t per_sweep = (blockDim.x >> 6) * 8;  // chunks served at once: a role-0 and a role-1 warp per 8 chunks
  for (uint32_t m = seg; m > 1; m >>= 1) {
    const uint32_t chunks = m >> 1;
    for (uint32_t first = (warp >> 1) * 8; first < chunks; first += per_sweep) {  // warp-uniform bounds
      uint32_t chunk = first + (lane >> 2);
      const bool live = chunk < chunks;
      if (!live) chunk = chunks - 1;  // partial warp: keep all lanes in the shuffles
      XYZZ<F> r;
      if (role == 0) {
        r = Quad<F>::dbl(Quad<F>::add(ca[2 * chunk], ca[2 * chunk + 1], ql), ql);
        if (live && ql == 0) na[chunk] = r;
      } else {
        r = Quad<F>::add(ce[2 * chunk], ce[2 * chunk + 1], ql);
        r = Quad<F>::add(r, ca[2 * chunk + 1], ql);
        if (live && ql == 0) ne[chunk] = r;
      }
    }
    __syncthreads();
    // swap: the level after reads what was just written and writes a quarter as many items into the old inputs' space
    XYZZ<F>* t = ca; ca = na; na = t;
    t = ce; ce = ne; ne = t;
  }
  if (threadIdx.x == 0) A_out[blockIdx.x] = ca[0];
  if (threadIdx.x == 32) E_out[blockIdx.x] = ce[0];
}

// Horner over the window sums, to affine, out of Montgomery form: one warp, every doubling / addition of the
// chain on quads of lanes (all eight quads run the same operands: the chain is 254 doublings deep on a plain
// table and nothing else is left to do, so what counts is the latency of one operation -- 1.9 us on a quad
// against 3.3 us on a lone thread).  The inversion stays a lone-thread computation (every lane runs it).
// out: canonical little-endian coordinates; flag = 1 when the result is the point at infinity.
template <class F>
__global__ void __launch_bounds__(32) msm_final_kernel(const XYZZ<F>* __restrict__ window_sums, int W, int c,
                                                       const XYZZ<F>* extra, int n_extra, Affine<F>* __restrict__ out,
                                                       int* __restrict__ inf_flag, XYZZ<F>* __restrict__ out_xyzz) {
  if (blockIdx.x != 0) return;
  const int ql = threadIdx.x & 3;
  XYZZ<F> r = window_sums[W - 1];
  for (int w = W - 2; w >= 0; w--) {
    if (!r.is_inf())  // the same value on every lane: uniform
      for (int k = 0; k < c; k++) r = Quad<F>::dbl(r, ql);
    r = Quad<F>::add(r, window_sums[w], ql);
  }
  for (int k = 0; k < n_extra; k++) r = Quad<F>::add(r, extra[k], ql);
  if (out_xyzz && threadIdx.x == 0) *out_xyzz = r;
  if (out) {
    Affine<F> a = r.to_affine();
    a.x = a.x.from_mont();
    a.y = a.y.from_mont();
    if (threadIdx.x == 0) {
      *inf_flag = r.is_inf() ? 1 : 0;
      *out = a;
    }
  }
}

// One warp per MSM of a run_many pass: block j runs the Horner chain over its W window sums (W = 1 for a
// precomputed table: only the affine conversion is left) and writes out[j] / inf_flag[j] as msm_final_kernel does.
template <class F>
__global__ void __launch_bounds__(32) msm_final_many_kernel(const XYZZ<F>* __restrict__ window_sums, int W, int c,
                                                            Affine<F>* __restrict__ out, int* __restrict__ inf_flag) {
  const int ql = threadIdx.x & 3;
  const XYZZ<F>* ws = window_sums + (uint64_t)blockIdx.x * W;
  XYZZ<F> r = ws[W - 1];
  for (int w = W - 2; w >= 0; w--) {
    if (!r.is_inf())
      for (int k = 0; k < c; k++) r = Quad<F>::dbl(r, ql);
    r = Quad<F>::add(r, ws[w], ql);
  }
  Affine<F> a = r.to_affine();
  a.x = a.x.from_mont();
  a.y = a.y.from_mont();
  if (threadIdx.x == 0) {
    inf_flag[blockIdx.x] = r.is_inf() ? 1 : 0;
    out[blockIdx.x] = a;
  }
}

// canonical <-> Montgomery conversion of coordinate arrays (n_fe field elements of the base field)
template <class FE>
__global__ void fe_to_mont_kernel(FE* __restrict__ v, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = v[i].to_mont();
}
template <class FE>
__global__ void fe_from_mont_kernel(FE* __restrict__ v, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = v[i].from_mont();
}

// ---------------------------------------------------------------- host driver
// Tunables (zkp_msm_set_option; 0 = automatic).
struct MsmOptions {
  int window_bits = 0;  // plain tables: window width override
  int accumulate = 0;   // bucket accumulation: 0 = automatic (XYZZ chains), 1 = XYZZ chains, 2 = affine tree where it applies
  int tree_items = 0;   // affine tree: most additions per thread and shared inversion (0 = default)
  int tree_rounds = 0;  // affine tree: rounds before the XYZZ chains take over (0 = default)
  int parts = 0;        // part-streamed MSM: point ranges per MSM (0 = 4 for host scalars, 1 for resident ones)
  int reduce_radix = 0;     // weighted-sum recursion: items per thread of a wide level (0 = 8)
  int wide_log2 = 0;        // log2 of the item count from which a level is a wide one (0 = 17)
  int quad_log2 = 0;        // log2 of the radix-2 output count up to which the levels are fused on quads (0 = 12)
};
MsmOptions& msm_options();  // defined in msm_g1.cu

template <class F>
struct MsmEngine {
  using FC = typename CompactOf<F>::type;  // same layout, out-of-line products (small code)
  DevBuf codes, sorted, hist, offsets, cursor, tile_sums, buckets, lvlA[2], lvlE[2], result, flag;
  DevBuf ntask, task_base, len_bins, tasks, partials, heavy;
  DevBuf thist, tplan, torder, tbuf[2], tpre;  // affine tree (msm_tree.cuh)
  // part-streamed form (run): the second set of the buffers one lane fills while the other reads
  static constexpr int MAX_PARTS = 8;
  DevBuf alt_sorted, alt_offsets, alt_ntask, alt_task_base, alt_len_bins, alt_tasks, alt_partials;
  cudaEvent_t ev_ready[MAX_PARTS] = {}, ev_done[MAX_PARTS] = {}, ev_lane = nullptr;
  void swap_part_sets() {
    std::swap(sorted, alt_sorted);
    std::swap(offsets, alt_offsets);
    std::swap(ntask, alt_ntask);
    std::swap(task_base, alt_task_base);
    std::swap(len_bins, alt_len_bins);
    std::swap(tasks, alt_tasks);
    std::swap(partials, alt_partials);
  }
  static constexpr int UPLOAD_CHUNKS = 4;
  cudaEvent_t ev_chunk[UPLOAD_CHUNKS] = {};
  int reduce_L = 16;  // measured at 2^20 (tools/reduce_sweep.py): radix 16 one wide level 3.20 ms, radix 8 3.25, radix 4 3.30
  uint32_t wide_threshold = 1u << 17;  // items (all windows) above which a level is throughput bound
  uint32_t quad_threshold = 1u << 12;  // radix-2 outputs (all windows) below which a level is latency bound

  // Builds the window-precomputed table T[w][i] = 2^(c*w) * P_i (w < W, affine Montgomery) from the n
  // plain points in `src`.  `dst` must hold W*n points; dst[0..n) may alias src.
  int precompute(const Affine<F>* src, uint64_t n, int c, Affine<F>* dst, cudaStream_t st) {
    MsmPlan pl = msm_plan(n, c);
    ScopedDevBuf cur;
    cur.reserve((size_t)n * sizeof(XYZZ<F>));
    int launches = 0;
    if (dst != src) CUDA_CHECK(cudaMemcpyAsync(dst, src, n * sizeof(Affine<F>), cudaMemcpyDeviceToDevice, st));
    msm_pre_lift_kernel<F><<<ceil_div(n, 256), 256, 0, st>>>(src, n, cur.as<XYZZ<F>>());
    CUDA_CHECK_LAUNCH();
    launches++;
    uint64_t T = (n + PRE_BATCH - 1) / PRE_BATCH;
    for (int w = 1; w < pl.W; w++) {
      msm_pre_shift_kernel<F><<<ceil_div(n, 128), 128, 0, st>>>(cur.as<XYZZ<F>>(), n, c);
      CUDA_CHECK_LAUNCH();
      msm_pre_affine_kernel<F><<<ceil_div(T, 128), 128, 0, st>>>(cur.as<XYZZ<F>>(), n, T, dst + (uint64_t)w * n);
      CUDA_CHECK_LAUNCH();
      launches += 2;
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
    return launches;
  }

  int scan_u32(const uint32_t* in, uint32_t count, uint32_t* out, cudaStream_t st) {
    uint32_t ntiles = ceil_div(count, SCAN_TILE);
    tile_sums.reserve((size_t)ntiles * 4);
    scan_tile_sums_kernel<<<ntiles, SCAN_BLOCK, 0, st>>>(in, count, tile_sums.as<uint32_t>());
    CUDA_CHECK_LAUNCH();
    scan_tile_offsets_kernel<<<1, SCAN_BLOCK, 0, st>>>(tile_sums.as<uint32_t>(), ntiles);
    CUDA_CHECK_LAUNCH();
    scan_apply_kernel<<<ntiles, SCAN_BLOCK, 0, st>>>(in, count, tile_sums.as<uint32_t>(), out);
    CUDA_CHECK_LAUNCH();
    return 3;
  }

  // ---- stages 1 + 2: `sorted` (entry | sign << 31, grouped by bucket) and `offsets` (nbuckets + 1).
  // Counting sort with one global atomic per digit in each pass.  A radix partition through shared-memory
  // histograms (block-local bins, then one block per bin) was built and measured in round 2: 417 us against
  // 289 us at 2^20 points -- it trades 27 M L2 atomics for 54 M shared-memory ones, which are no faster on
  // this part -- and was removed (DESIGN.md 7).
  // host_scalars != nullptr: the scalars still sit in host memory; they are copied to `scalars` in UPLOAD_CHUNKS
  // pieces on `copy_st` and each piece is recoded as soon as it has landed, so the recoding (and the histogram
  // atomics, the slow part of it) runs under the rest of the upload instead of after it.
  int sort_entries(const uint32_t* scalars, uint64_t n, const MsmPlan& pl, uint32_t wstride, uint32_t pre_stride,
                   uint32_t pre_offset, cudaStream_t st, StageTrace& tr, const uint8_t* host_scalars = nullptr,
                   cudaStream_t copy_st = nullptr, uint32_t idx_base = 0) {
    const uint64_t total = (uint64_t)pl.W * n;
    codes.reserve(total * 4);
    sorted.reserve(total * 4);
    hist.reserve((size_t)pl.nbuckets * 4);
    offsets.reserve(((size_t)pl.nbuckets + 1) * 4);
    cursor.reserve(((size_t)pl.nbuckets + 1) * 4);
    CUDA_CHECK(cudaMemsetAsync(hist.p, 0, (size_t)pl.nbuckets * 4, st));
    int launches = 0;
    const int chunks = (host_scalars && n >= (1u << 16)) ? UPLOAD_CHUNKS : 1;
    for (int k = 0; k < chunks; k++) {
      const uint64_t i0 = n * k / chunks, i1 = n * (k + 1) / chunks;
      if (host_scalars) {
        cudaStream_t cs = chunks > 1 ? copy_st : st;
        if (chunks > 1 && k == 0) {  // the copy lane starts behind everything already queued on the main one
          if (!ev_chunk[0])
            for (auto& e : ev_chunk) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
          CUDA_CHECK(cudaEventRecord(ev_chunk[0], st));
          CUDA_CHECK(cudaStreamWaitEvent(cs, ev_chunk[0], 0));
        }
        CUDA_CHECK(cudaMemcpyAsync(const_cast<uint32_t*>(scalars) + 8 * i0, host_scalars + 32 * i0, (i1 - i0) * 32,
                                   cudaMemcpyHostToDevice, cs));
        if (chunks > 1) {
          CUDA_CHECK(cudaEventRecord(ev_chunk[k], cs));
          CUDA_CHECK(cudaStreamWaitEvent(st, ev_chunk[k], 0));
        }
      }
      msm_digits_kernel<<<ceil_div(i1 - i0, 256), 256, 0, st>>>(scalars, n, i0, i1, pl.c, pl.W, pl.B, wstride,
                                                               codes.as<uint32_t>(), hist.as<uint32_t>());
      CUDA_CHECK_LAUNCH();
      launches++;
    }
    launches += scan_u32(hist.as<uint32_t>(), pl.nbuckets, offsets.as<uint32_t>(), st);
    tr.mark("digits+scan");
    CUDA_CHECK(cudaMemcpyAsync(cursor.p, offsets.p, ((size_t)pl.nbuckets + 1) * 4, cudaMemcpyDeviceToDevice, st));
    msm_scatter_kernel<<<ceil_div(total, 256), 256, 0, st>>>(codes.as<uint32_t>(), total, n, cursor.as<uint32_t>(),
                                                            sorted.as<uint32_t>(), pre_stride, pre_offset, idx_base);
    CUDA_CHECK_LAUNCH();
    tr.mark("scatter");
    return launches + 1;
  }

  // ---- stage 3a: tasks: count per bucket -> scan -> length histogram -> emit sorted by length
  int build_tasks(uint32_t nbuckets, uint32_t max_tasks, cudaStream_t st, uint32_t light_max = 0) {
    const uint32_t* off = offsets.as<uint32_t>();
    ntask.reserve(((size_t)nbuckets + 1) * 4);
    task_base.reserve(((size_t)nbuckets + 1) * 4);
    len_bins.reserve((MSM_TASK_LEN + 1) * 4);
    tasks.reserve((size_t)max_tasks * sizeof(uint4));
    partials.reserve((size_t)max_tasks * sizeof(XYZZ<F>));
    msm_task_count_kernel<<<ceil_div(nbuckets, 256), 256, 0, st>>>(off, nbuckets, ntask.as<uint32_t>(), light_max);
    CUDA_CHECK_LAUNCH();
    int launches = 1 + scan_u32(ntask.as<uint32_t>(), nbuckets, task_base.as<uint32_t>(), st);
    CUDA_CHECK(cudaMemsetAsync(len_bins.p, 0, (MSM_TASK_LEN + 1) * 4, st));
    msm_task_hist_kernel<<<ceil_div(nbuckets, 256), 256, 0, st>>>(off, nbuckets, len_bins.as<uint32_t>(), light_max);
    CUDA_CHECK_LAUNCH();
    msm_task_bins_kernel<<<1, 32, 0, st>>>(len_bins.as<uint32_t>());
    CUDA_CHECK_LAUNCH();
    msm_task_emit_kernel<<<ceil_div(nbuckets, 256), 256, 0, st>>>(off, task_base.as<uint32_t>(), nbuckets,
                                                                 len_bins.as<uint32_t>(), tasks.as<uint4>(), light_max);
    CUDA_CHECK_LAUNCH();
    return launches + 3;
  }

  // ---- stage 3, affine form: buckets of up to TREE_MAX entries summed as pairwise trees with shared inversions
  // (msm_tree.cuh).
  static bool use_tree(uint64_t total, uint32_t nbuckets) {
    static const char* env = getenv("ZKP_B200_MSM_ACC");  // "xyzz" / "tree": overrides the option (tests, A/B runs)
    int mode = msm_options().accumulate;
    if (env && !strcmp(env, "xyzz")) mode = 1;
    if (env && !strcmp(env, "tree")) mode = 2;
    if (mode == 1) return false;
    if (total >= (1ull << 32) - nbuckets || nbuckets > (1u << TREE_BUCKET_BITS)) return false;
    // Opt-in only (zkp_msm_set_option("accumulate", 2) / ZKP_B200_MSM_ACC=tree).  Measured on B200 at 2^20 points,
    // c = 20 (profiles/r2_affine_tree_experiment.txt): 788 instead of 1304 limb-MACs per addition did not pay -- a
    // round runs the integer pipe at 40-45 % (every operand is gathered twice, 32 more bytes per addition travel
    // through the prefix array, and each block idles through a ~60 us single-thread inversion), against 88 % for the
    // XYZZ chains: 2 rounds + chains 3.70 ms, 1 round + chains 2.98 ms, XYZZ chains alone 2.21 ms.
    return mode == 2;
  }
  int run_tree(const Affine<F>* pts, uint32_t nbuckets, uint64_t total, cudaStream_t st, StageTrace& tr) {
    constexpr int TB = TreeCfg<FC>::TB;
    int full = 1;
    while (full < TREE_ROUNDS && (1ull << full) < total) full++;  // a bucket holds at most `total` entries
    // rounds in affine form before the XYZZ chains take over (every round costs an inversion latency per block)
    static const int env_rounds = getenv("ZKP_B200_TREE_ROUNDS") ? atoi(getenv("ZKP_B200_TREE_ROUNDS")) : 0;
    int K = env_rounds > 0 ? env_rounds : msm_options().tree_rounds > 0 ? msm_options().tree_rounds : 2;
    if (K > full) K = full;
    thist.reserve(2 * (TREE_MAX + 1) * 4);
    tplan.reserve((size_t)TREE_ROUNDS * TREE_REC * 4);
    torder.reserve((size_t)nbuckets * sizeof(uint2));
    tbuf[0].reserve((size_t)(total / 2 + nbuckets + 2) * sizeof(Affine<F>));
    if (K > 1) tbuf[1].reserve((size_t)(total / 4 + nbuckets + 2) * sizeof(Affine<F>));
    uint32_t* hist_p = thist.as<uint32_t>();
    uint32_t* cursor_p = hist_p + (TREE_MAX + 1);
    CUDA_CHECK(cudaMemsetAsync(hist_p, 0, (TREE_MAX + 1) * 4, st));
    msm_tree_hist_kernel<FC><<<ceil_div(nbuckets, 256), 256, 0, st>>>(offsets.as<uint32_t>(), nbuckets, hist_p,
                                                                     buckets.as<XYZZ<FC>>());
    CUDA_CHECK_LAUNCH();
    msm_tree_plan_kernel<<<1, TREE_JMAX, 0, st>>>(hist_p, cursor_p, tplan.as<uint32_t>(), K);
    CUDA_CHECK_LAUNCH();
    msm_tree_emit_kernel<<<ceil_div(nbuckets, 256), 256, 0, st>>>(offsets.as<uint32_t>(), nbuckets, cursor_p,
                                                                 torder.as<uint2>());
    CUDA_CHECK_LAUNCH();
    tr.mark("tree plan");
    // items per thread of the largest blocks (= additions per shared inversion / TB): a multiple of 8, as many as
    // still leave every SM several waves of blocks
    static const int env_items = getenv("ZKP_B200_TREE_B") ? atoi(getenv("ZKP_B200_TREE_B")) : 0;
    const uint32_t max_items = env_items > 0 ? (uint32_t)env_items : msm_options().tree_items > 0 ? (uint32_t)msm_options().tree_items : 32u;
    const uint64_t nonempty = total < nbuckets ? total : nbuckets;
    const uint64_t slots = (uint64_t)TreeCfg<FC>::MIN_BLOCKS * (uint64_t)(ctx().sm_count > 0 ? ctx().sm_count : 148);
    uint32_t B[TREE_ROUNDS], blocks[TREE_ROUNDS];
    uint64_t pre_items = 0;
    for (int r = 0; r < K; r++) {
      const uint64_t expect = total >> (r + 1), upper = expect + nonempty + 1;
      uint64_t b = expect / ((uint64_t)TB * slots * 2);  // the average block is about half the largest
      if (b > max_items) b = max_items;
      if (b >= 8) b &= ~7ull;
      if (b < 2) b = 2;
      B[r] = (uint32_t)b;
      TreeSched sc;
      blocks[r] = tree_sched(upper, B[r], TB, sc) + 16;  // the split of the true item count never needs more
      if (upper > pre_items) pre_items = upper;
    }
    tpre.reserve((size_t)pre_items * sizeof(F));
    const Affine<FC>* p = reinterpret_cast<const Affine<FC>*>(pts);
    for (int r = 0; r < K; r++) {
      Affine<FC>* out = tbuf[r & 1].template as<Affine<FC>>();
      const uint32_t* rec = tplan.as<uint32_t>() + (size_t)r * TREE_REC;
      if (r == 0)
        msm_tree_round_kernel<FC, true><<<blocks[r], TB, 0, st>>>(p, sorted.as<uint32_t>(), nullptr, out, torder.as<uint2>(), rec,
                                                                 r, B[r], tpre.as<FC>(), buckets.as<XYZZ<FC>>());
      else
        msm_tree_round_kernel<FC, false><<<blocks[r], TB, 0, st>>>(nullptr, nullptr, tbuf[(r - 1) & 1].template as<Affine<FC>>(), out,
                                                                  torder.as<uint2>(), rec, r, B[r], tpre.as<FC>(),
                                                                  buckets.as<XYZZ<FC>>());
      CUDA_CHECK_LAUNCH();
      if (tr.print) tr.mark("tree round");
    }
    if (K < full) {
      msm_tree_finish_kernel<F, MSM_ACC_OUTLINE><<<ceil_div(nonempty, 128), 128, 0, st>>>(
          tbuf[(K - 1) & 1].template as<Affine<F>>(), torder.as<uint2>(), tplan.as<uint32_t>(), K, buckets.as<XYZZ<F>>());
      CUDA_CHECK_LAUNCH();
      if (tr.print) tr.mark("tree finish");
    }
    return 4 + K;
  }

  // ---- stage 3b: fold the buckets that were cut into several tasks (cont: onto what the bucket already holds)
  int fold_buckets(uint32_t nbuckets, uint64_t avg_entries, cudaStream_t st, bool tree, bool cont) {
    XYZZ<FC>* bk = buckets.as<XYZZ<FC>>();
    heavy.reserve(((size_t)nbuckets + 1) * 4);
    CUDA_CHECK(cudaMemsetAsync(heavy.p, 0, 4, st));
    msm_bucket_fold_kernel<FC><<<ceil_div(nbuckets, 128), 128, 0, st>>>(
        partials.as<XYZZ<FC>>(), task_base.as<uint32_t>(), nbuckets, bk, heavy.as<uint32_t>(), heavy.as<uint32_t>() + 1,
        // "heavy" is relative to the average bucket: every bucket of a dense MSM (many entries per
        // bucket) folds serially in parallel with the others; only outliers get a whole block
        MSM_FOLD_SERIAL + 3 * (uint32_t)(avg_entries / MSM_TASK_LEN), tree, cont);
    CUDA_CHECK_LAUNCH();
    msm_bucket_fold_heavy_kernel<FC><<<296, 128, 0, st>>>(partials.as<XYZZ<FC>>(), task_base.as<uint32_t>(),
                                                          heavy.as<uint32_t>(), heavy.as<uint32_t>() + 1, bk, cont);
    CUDA_CHECK_LAUNCH();
    return 2;
  }

  // ---- stage 4: the weighted-sum recursion down to one item per window.  Returns the window sums through `wsum`.
  int reduce_buckets(uint32_t nbuckets, int n_windows, cudaStream_t st, StageTrace& tr, const XYZZ<FC>** wsum) {
    int launches = 0;
    XYZZ<FC>* bk = buckets.as<XYZZ<FC>>();
    uint32_t n_in = nbuckets / n_windows;  // buckets per window
    const XYZZ<FC>* A = bk;
    const XYZZ<FC>* E = nullptr;
    int pp = 0;
    const MsmOptions& mo = msm_options();
    const int reduce_L = mo.reduce_radix ? mo.reduce_radix : this->reduce_L;
    const uint32_t wide_threshold = mo.wide_log2 ? 1u << mo.wide_log2 : this->wide_threshold;
    const uint32_t quad_threshold = mo.quad_log2 ? 1u << mo.quad_log2 : this->quad_threshold;
    while (n_in > 1) {
      // wide levels (many items): radix reduce_L running sums, fewest group operations per bucket;
      // middle levels: radix 2, one thread per output (still throughput bound);
      // narrow levels: fused segments on quads of lanes, shortest dependency chain.
      bool wide = (uint64_t)n_in * n_windows >= (uint64_t)wide_threshold && n_in >= (uint32_t)reduce_L;
      bool fused = !wide && (uint64_t)(n_in / 2) * n_windows <= (uint64_t)quad_threshold;
      uint32_t L = wide ? (uint32_t)reduce_L : 2u;
      if (fused) L = n_in < (uint32_t)WsFused<FC>::SEG ? n_in : (uint32_t)WsFused<FC>::SEG;
      int logL = 0;
      while ((1u << logL) < L) logL++;
      uint32_t T = n_in / L;
      size_t bytes = (size_t)T * n_windows * sizeof(XYZZ<F>);
      lvlA[pp].reserve(bytes);
      lvlE[pp].reserve(bytes);
      XYZZ<FC>* Ao = lvlA[pp].template as<XYZZ<FC>>();
      XYZZ<FC>* Eo = lvlE[pp].template as<XYZZ<FC>>();
      if (wide)
        msm_ws_level_kernel<FC><<<ceil_div((uint64_t)T * n_windows, 64), 64, 0, st>>>(A, E, n_in, L, logL, n_windows, Ao, Eo);
      else if (fused)
        msm_ws2_fused_kernel<FC><<<T * n_windows, WsFused<FC>::THREADS, WsFused<FC>::SMEM, st>>>(A, E, L, Ao, Eo);
      else
        msm_ws2_kernel<FC><<<ceil_div((uint64_t)ceil_div((uint64_t)T * n_windows, 32) * 64, 64), 64, 0, st>>>(A, E, n_in, n_windows, Ao, Eo);
      CUDA_CHECK_LAUNCH();
      launches++;
      A = Ao;
      E = Eo;
      n_in = T;
      pp ^= 1;
      tr.mark(wide ? "ws wide" : fused ? "ws fused" : "ws2");
    }
    // n_in == 1: V_w = E_w (for B == 1 the single bucket has weight 1 = itself)
    *wsum = E ? E : A;
    return launches;
  }

  // pts: device, affine Montgomery; scalars: device, canonical.  Leaves the affine canonical result
  // in `result` (and the infinity flag in `flag`), or the XYZZ Montgomery partial sum when
  // want_xyzz (multi-GPU shards).  Returns the number of kernels launched.
  // pre_stride != 0: `pts` is the base of a window-precomputed table [w][i] built with window width
  // force_c; the MSM covers points [pre_offset, pre_offset + n) of it.
  //
  // Measured and not kept (round 2, DESIGN.md 7): cutting the single bucket set of a precomputed-table MSM into
  // bucket-range parts so that one part's reduction overlaps the next part's accumulation.  Accumulation
  // blocks live ~0.3 ms (a 26-entry task at 1/512 of an SM's product rate), so every extra accumulate launch
  // costs most of a block lifetime in under-filled waves (+0.1 ms per part at 2^20) while the exposed
  // reduction of the last part is still log2(buckets) dependent levels long.
  int run(const Affine<F>* pts, const uint32_t* scalars, uint64_t n, cudaStream_t st, bool want_xyzz = false,
          int force_c = 0, uint32_t pre_stride = 0, uint32_t pre_offset = 0, const uint8_t* host_scalars = nullptr,
          cudaStream_t copy_st = nullptr, cudaStream_t lane = nullptr) {
    int launches = 0;
    result.reserve(sizeof(XYZZ<F>) + sizeof(Affine<F>));
    flag.reserve(sizeof(int));
    Affine<F>* out_aff = result.as<Affine<F>>();
    XYZZ<F>* out_xyzz = reinterpret_cast<XYZZ<F>*>(result.as<char>() + sizeof(Affine<F>));
    if (n == 0) {
      CUDA_CHECK(cudaMemsetAsync(result.p, 0, sizeof(XYZZ<F>) + sizeof(Affine<F>), st));
      int one = 1;
      CUDA_CHECK(cudaMemcpyAsync(flag.p, &one, sizeof(int), cudaMemcpyHostToDevice, st));
      CUDA_CHECK(cudaStreamSynchronize(st));
      return 0;
    }
    if (n >= (1ull << 31)) throw std::runtime_error("msm: n must be < 2^31");
    MsmPlan pl = msm_plan(n, force_c);
    uint64_t total = (uint64_t)pl.W * n;
    if (total >= (1ull << 32)) throw std::runtime_error("msm: W*n must be < 2^32");
    if (pre_stride && (uint64_t)pl.W * pre_stride >= (1ull << 31))
      throw std::runtime_error("msm: precomputed table too large for 31-bit entry indices");
    const uint32_t wstride = pre_stride ? 0u : pl.B;
    if (pre_stride) pl.nbuckets = pl.B;  // precomputed windows: every digit of every window lands in one bucket set
    const int n_windows = pre_stride ? 1 : pl.W;
    buckets.reserve((size_t)pl.nbuckets * sizeof(XYZZ<F>));

    StageTrace tr(st);
    const bool tree = use_tree(total, pl.nbuckets);
    // Part-streamed form (host scalars, large n): the points are cut into `parts` contiguous ranges that all add
    // into ONE bucket set.  A side lane (high-priority stream) uploads range p+1 and sorts its digits while the
    // main stream accumulates range p, so only the first range's upload and sort stay exposed; the bucket
    // reduction runs once.  Two workspace sets alternate between the lanes.
    static const int env_parts = getenv("ZKP_B200_MSM_PARTS") ? atoi(getenv("ZKP_B200_MSM_PARTS")) : 0;
    int parts = 1;
    if (lane && !tree) {
      const int asked = env_parts > 0 ? env_parts : msm_options().parts;  // explicit: any size (tests, A/B runs)
      if (asked > 0) parts = (uint64_t)asked < n ? asked : (int)n;
      else if (host_scalars && n >= (1u << 18)) parts = 4;
      if (parts > MAX_PARTS) parts = MAX_PARTS;
    }
    if (parts == 1) {
      launches += sort_entries(scalars, n, pl, wstride, pre_stride, pre_offset, st, tr, host_scalars, copy_st);
      // the task count is data dependent: launch for the upper bound, threads past
      // task_base[nbuckets] exit at once (no host round trip in the middle of the pipeline)
      const uint32_t max_tasks = tree ? (uint32_t)(total / MSM_TASK_LEN) + (uint32_t)(total / (TREE_MAX + 1)) + 1
                                      : (uint32_t)(total / MSM_TASK_LEN) + pl.nbuckets + 1;
      launches += build_tasks(pl.nbuckets, max_tasks, st, tree ? TREE_MAX : 0u);
      tr.mark("tasks");
      if (tree) launches += run_tree(pts, pl.nbuckets, total, st, tr);
      // G1: the eight products of the mixed addition through the shared out-of-line body, the two squarings inlined
      // (measured at 2^20: 2.213 ms; everything inlined 2.248, everything out of line 2.241, other splits between)
      msm_accumulate_kernel<F, MSM_ACC_OUTLINE><<<ceil_div(max_tasks, 128), 128, 0, st>>>(
          pts, sorted.as<uint32_t>(), tasks.as<uint4>(), task_base.as<uint32_t>() + pl.nbuckets, partials.as<XYZZ<F>>(),
          buckets.as<XYZZ<F>>(), false);
      CUDA_CHECK_LAUNCH();
      launches++;
      tr.mark("accumulate");
      launches += fold_buckets(pl.nbuckets, total / pl.nbuckets, st, tree, false);
      tr.mark("fold");
    } else {
      if (!ev_ready[0]) {
        for (auto& e : ev_ready) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : ev_done) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventCreateWithFlags(&ev_lane, cudaEventDisableTiming));
      }
      CUDA_CHECK(cudaEventRecord(ev_lane, st));  // the lane starts behind everything already queued on the main stream
      CUDA_CHECK(cudaStreamWaitEvent(lane, ev_lane, 0));
      StageTrace lane_tr(lane, false);
      // Ranges grow by 1.35x: the first one (whose upload and sort nothing hides) is small, and each later upload +
      // sort (0.9 ms per 2^20 points alone, 1.7 ms when eight ranks pull from host memory at once) still fits under
      // the accumulation of the range before it (2.2 ms per 2^20 points).
      uint64_t cut[MAX_PARTS + 1];
      {
        double w = 1.0, sum = 0.0, acc = 0.0;
        for (int p = 0; p < parts; p++, w *= 1.35) sum += w;
        w = 1.0;
        cut[0] = 0;
        for (int p = 0; p < parts; p++, w *= 1.35) {
          acc += w;
          cut[p + 1] = p + 1 == parts ? n : (uint64_t)((double)n * (acc / sum));
          if (cut[p + 1] <= cut[p]) cut[p + 1] = cut[p] + 1;  // tiny MSMs under an explicit part count: no empty range
          if (cut[p + 1] > n) cut[p + 1] = n;
        }
      }
      for (int p = 0; p < parts; p++) {
        const uint64_t i0 = cut[p], i1 = cut[p + 1], np = i1 - i0;
        if (np == 0) continue;
        if (p > 0) swap_part_sets();
        if (p >= 2) CUDA_CHECK(cudaStreamWaitEvent(lane, ev_done[p - 2], 0));  // this workspace set is free again
        if (host_scalars)
          CUDA_CHECK(cudaMemcpyAsync(const_cast<uint32_t*>(scalars) + 8 * i0, host_scalars + 32 * i0, np * 32,
                                     cudaMemcpyHostToDevice, lane));
        MsmPlan plp = pl;  // same window width and bucket set, fewer points
        launches += sort_entries(scalars + 8 * i0, np, plp, wstride, pre_stride, pre_offset + (uint32_t)i0, lane, lane_tr,
                                 nullptr, nullptr, pre_stride ? 0u : (uint32_t)i0);
        const uint64_t total_p = (uint64_t)pl.W * np;
        const uint32_t max_tasks = (uint32_t)(total_p / MSM_TASK_LEN) + pl.nbuckets + 1;
        launches += build_tasks(pl.nbuckets, max_tasks, lane);
        CUDA_CHECK(cudaEventRecord(ev_ready[p], lane));
        CUDA_CHECK(cudaStreamWaitEvent(st, ev_ready[p], 0));
        if (p == 0) tr.mark("tasks");
        msm_accumulate_kernel<F, MSM_ACC_OUTLINE><<<ceil_div(max_tasks, 128), 128, 0, st>>>(
            pts, sorted.as<uint32_t>(), tasks.as<uint4>(), task_base.as<uint32_t>() + pl.nbuckets, partials.as<XYZZ<F>>(),
            buckets.as<XYZZ<F>>(), p > 0);
        CUDA_CHECK_LAUNCH();
        launches++;
        launches += fold_buckets(pl.nbuckets, total_p / pl.nbuckets, st, false, p > 0);
        CUDA_CHECK(cudaEventRecord(ev_done[p], st));
      }
      tr.mark("accumulate");
      tr.mark("fold");
    }
    const XYZZ<FC>* wsum = nullptr;
    launches += reduce_buckets(pl.nbuckets, n_windows, st, tr, &wsum);
    msm_final_kernel<FC><<<1, 32, 0, st>>>(wsum, n_windows, pl.c, nullptr, 0,
                                          want_xyzz ? nullptr : reinterpret_cast<Affine<FC>*>(out_aff), flag.as<int>(),
                                          want_xyzz ? reinterpret_cast<XYZZ<FC>*>(out_xyzz) : nullptr);
    CUDA_CHECK_LAUNCH();
    launches++;
    tr.mark("horner+affine");
    return launches;
  }

  // `count` MSMs over the same n points, scalar vector j at scalars[8 * j * n ...]: ONE Pippenger pass whose bucket
  // sets are the MSMs' own (MSM j owns buckets [j * per_msm, (j + 1) * per_msm)).  Tasks, accumulation and fold run
  // unchanged over count times as many buckets; the reduction treats every (MSM, window) as a segment; one warp per
  // MSM finishes.  Leaves count canonical affine points in `many_out` and the infinity flags in `many_flag`.
  // The launch count does not depend on count.  The caller has checked count * W * n < 2^32 and
  // count * per_msm < 2^31 (GroupApi::msm_dev_many).
  int run_many(const Affine<F>* pts, const uint32_t* scalars, uint64_t n, uint32_t count, cudaStream_t st, int force_c,
               uint32_t pre_stride, uint32_t pre_offset) {
    many_out.reserve((size_t)(count ? count : 1) * sizeof(Affine<F>));
    many_flag.reserve((size_t)(count ? count : 1) * sizeof(int));
    if (!count) return 0;
    if (n == 0) {  // every MSM is empty: count points at infinity
      CUDA_CHECK(cudaMemsetAsync(many_out.p, 0, (size_t)count * sizeof(Affine<F>), st));
      std::vector<int> ones(count, 1);
      CUDA_CHECK(cudaMemcpyAsync(many_flag.p, ones.data(), (size_t)count * sizeof(int), cudaMemcpyHostToDevice, st));
      CUDA_CHECK(cudaStreamSynchronize(st));
      return 0;
    }
    const MsmPlan pl = msm_plan(n, force_c);
    const uint32_t per_msm = pre_stride ? pl.B : pl.nbuckets;
    const uint32_t wstride = pre_stride ? 0u : pl.B;
    const uint64_t N = (uint64_t)count * n;
    const uint64_t total = (uint64_t)pl.W * N;
    const uint32_t nbuckets = count * per_msm;
    const int n_windows = pre_stride ? (int)count : (int)count * pl.W;
    int launches = 0;
    StageTrace tr(st);
    buckets.reserve((size_t)nbuckets * sizeof(XYZZ<F>));
    codes.reserve(total * 4);
    sorted.reserve(total * 4);
    hist.reserve((size_t)nbuckets * 4);
    offsets.reserve(((size_t)nbuckets + 1) * 4);
    cursor.reserve(((size_t)nbuckets + 1) * 4);
    CUDA_CHECK(cudaMemsetAsync(hist.p, 0, (size_t)nbuckets * 4, st));
    msm_digits_many_kernel<<<ceil_div(N, 256), 256, 0, st>>>(scalars, n, N, pl.c, pl.W, pl.B, wstride, per_msm,
                                                            codes.as<uint32_t>(), hist.as<uint32_t>());
    CUDA_CHECK_LAUNCH();
    launches += 1 + scan_u32(hist.as<uint32_t>(), nbuckets, offsets.as<uint32_t>(), st);
    tr.mark("digits+scan");
    CUDA_CHECK(cudaMemcpyAsync(cursor.p, offsets.p, ((size_t)nbuckets + 1) * 4, cudaMemcpyDeviceToDevice, st));
    msm_scatter_many_kernel<<<ceil_div(total, 256), 256, 0, st>>>(codes.as<uint32_t>(), total, N, n, cursor.as<uint32_t>(),
                                                                 sorted.as<uint32_t>(), pre_stride, pre_offset);
    CUDA_CHECK_LAUNCH();
    launches++;
    tr.mark("scatter");
    const uint32_t max_tasks = (uint32_t)(total / MSM_TASK_LEN) + nbuckets + 1;
    launches += build_tasks(nbuckets, max_tasks, st);
    tr.mark("tasks");
    msm_accumulate_kernel<F, MSM_ACC_OUTLINE><<<ceil_div(max_tasks, 128), 128, 0, st>>>(
        pts, sorted.as<uint32_t>(), tasks.as<uint4>(), task_base.as<uint32_t>() + nbuckets, partials.as<XYZZ<F>>(),
        buckets.as<XYZZ<F>>(), false);
    CUDA_CHECK_LAUNCH();
    launches++;
    tr.mark("accumulate");
    launches += fold_buckets(nbuckets, total / nbuckets, st, false, false);
    tr.mark("fold");
    const XYZZ<FC>* wsum = nullptr;
    launches += reduce_buckets(nbuckets, n_windows, st, tr, &wsum);
    const int W = pre_stride ? 1 : pl.W;
    msm_final_many_kernel<FC><<<count, 32, 0, st>>>(wsum, W, pl.c, many_out.as<Affine<FC>>(), many_flag.as<int>());
    CUDA_CHECK_LAUNCH();
    launches++;
    tr.mark("horner+affine");
    return launches;
  }
  DevBuf many_out, many_flag;
};

}  // namespace zkp
