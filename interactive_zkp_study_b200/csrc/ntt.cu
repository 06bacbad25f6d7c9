// Fr number-theoretic transform on sm_100a.  Replaces the recursive radix-2 Python FFT of the
// reference: fft (/root/reference/zkp/plonk/polynomial.py:292-341), ifft (:344-378),
// coset_fft / coset_ifft (/root/reference/zkp/plonk/utils.py:145-205).  Natural order in and out,
// arbitrary root `omega` of order n (the reference passes get_root_of_unity(n) or its inverse).
//
// Algorithm: decimation-in-time radix-2 butterflies on the bit-reversed input, grouped into passes
// of up to 10 stages that run out of shared memory.  Pass 1 gathers the bit-reversed input
// (32-byte elements = one DRAM sector each) and writes contiguous 32 KB tiles; later passes work on
// tiles of 2^S strided rows x 2^(10-S) contiguous elements.  A 32-byte element is exactly one sector, so
// even a run of one element wastes no bandwidth: taking all 10 stages per pass (2^20 = 10 + 10, two
// passes) measured 4 % faster than insisting on 256-byte runs (10 + 7 + 3, three passes).  Shared memory holds
// the tile as swizzled 128-bit halves (conflict-free LDS.128 / STS.128).  A radix-8 variant (three stages per
// round in registers, first / last round straight from / to global memory) was built and measured in round 2:
// 0.27 - 0.32 ms at 2^20 against 0.24 ms for the radix-4 rounds below (its 8 scattered loads + 7 twiddle
// loads per thread stall on the load queue, ncu: lg_throttle 0.9, long_scoreboard 2.1, no_instruction 1.1 per
// issue) and was not kept.  Also measured and not kept (round 2, after the field product had been brought to the
// pipe's floor): smaller tiles (2^8 elements = one warp per block, no inter-warp barrier, 8 + 8 + 6 stages at
// 2^22: 0.868 ms against 0.909; 2^20 0.236 against 0.232; 2^24 3.65 against 3.69 -- a wash) and stage counts
// spread evenly over the passes (2^22 as 8 + 7 + 7: 0.924 ms; 2^24 as 8 + 8 + 8: 3.65): a stage costs the same
// wherever it runs, the pass overhead is small.  Twiddles omega^i, i < n/2, are
// precomputed on the device in Montgomery form and cached per (omega, n); because they are
// Montgomery constants, the data keeps whatever form it came in (canonical host data needs no
// conversion).  The n^-1 factor of the inverse and the coset scalings are fused into the
// first-pass load / last-pass store.
#include <cstring>
#include <map>
#include <vector>
#include "ntt.cuh"
#include "registry.cuh"

namespace zkp {

static constexpr int NTT_LOG_TILE = 10;  // elements per block tile (2^10 x 32 B = 32 KB shared)
static constexpr int NTT_Q = 0;          // log2 of the minimum contiguous run in the strided passes (see header)

// ------------------------------------------------------------------ small power tables
// out[k] = x^(2^k) (Montgomery), k < 32; x canonical on input.  invert: start from x^-1.
__global__ void pow2_table_kernel(Fr x_canon, int invert, Fr* out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  Fr x = x_canon.to_mont();
  if (invert) x = x.inv();
  for (int k = 0; k < 32; k++) {
    out[k] = x;
    x = x.sqr();
  }
}

// x^e from the pow2 table (e < 2^32)
__device__ __forceinline__ Fr pow_from_table(const Fr* __restrict__ tab, uint32_t e) {
  Fr r = Fr::one();
  bool first = true;
  for (int k = 0; e; k++, e >>= 1) {
    if (e & 1) {
      if (first) { r = tab[k]; first = false; }
      else r = r * tab[k];
    }
  }
  return r;
}

__global__ void twiddle_table_kernel(const Fr* __restrict__ pow2tab, uint32_t count, Fr* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = pow_from_table(pow2tab, i);
}

// ------------------------------------------------------------------ the pass kernel
struct NttPassArgs {
  const Fr* src;
  Fr* dst;
  const Fr* tw;       // omega^i, i < n/2
  uint32_t log_n;
  uint32_t s0;        // stages already done
  uint32_t S;         // stages in this pass
  uint32_t log_g;     // log2 of sub-transforms per tile; tile = 2^(S+log_g) elements
  int bitrev_in;      // first pass: gather src[bitrev(i)]
  // coset scalings as two-level power tables: shift^j = lo[j & 1023] * hi[j >> 10]  (2 products per element
  // instead of a square-and-multiply walk over the bits of j: ~11 products, as much as the transform itself)
  const Fr* pre_pow;    // forward coset: multiply input j (natural index) by shift^j   (first pass)
  const Fr* post_pow;   // inverse coset: multiply output j by shift^-j                 (last pass)
  int scale_n_inv;      // last pass of an inverse: multiply by n^-1
  Fr n_inv;             // Montgomery
};


// Shared-memory tile: element `slot` is kept as two 16-byte halves, half h at uint4 index (h << log_tile) +
// swz(slot): every access is a 128-bit LDS / STS (two per element instead of eight 32-bit ones).  swz XORs
// the low three slot bits with parities of the higher ones so that the eight lanes of a quarter-warp fall
// into eight different 16-byte bank groups for every index pattern of the radix-4 / radix-2 rounds and of
// the load / store phases (all (S, log_g) splits of a 1024-element tile, checked exhaustively; the
// limb-major 32-bit layout of round 1 took 3.7 M bank conflicts per pass).
__device__ __forceinline__ uint32_t ntt_swz(uint32_t slot) {
  const uint32_t hb = slot >> 3;
  const uint32_t p = __popc(hb & 23u) & 1u, q = __popc(hb & 42u) & 1u;
  return slot ^ (p * 5u) ^ (q << 1);
}
__device__ __forceinline__ Fr lds_elem(const uint4* sm, uint32_t tile, uint32_t slot) {
  const uint32_t i = ntt_swz(slot);
  uint4 lo = sm[i], hi = sm[tile + i];
  Fr r;
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}
__device__ __forceinline__ void sts_elem(uint4* sm, uint32_t tile, uint32_t slot, const Fr& x) {
  const uint32_t i = ntt_swz(slot);
  sm[i] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
  sm[tile + i] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
}

__global__ void __launch_bounds__(128, 4) ntt_pass_kernel(NttPassArgs a) {
  extern __shared__ uint4 sm[];
  const uint32_t log_tile = a.S + a.log_g;
  const uint32_t tile = 1u << log_tile;
  const uint32_t G = 1u << a.log_g;
  const uint32_t n = 1u << a.log_n;
  const bool first = a.s0 == 0;
  const uint32_t tid = threadIdx.x;
  const uint32_t nthreads = blockDim.x;  // tile / 4 (or 1 for tiles of fewer than 4 elements)

  // ---- global index of local slot l
  // first pass : contiguous tile, l = g * 2^S + mid, global = blockIdx * tile + l
  // later pass : global = hi * 2^(s0+S) + mid * 2^s0 + (lg * G + g), l = mid * G + g
  uint64_t tile_base;
  uint32_t lo_base = 0;
  if (first) {
    tile_base = (uint64_t)blockIdx.x * tile;
  } else {
    uint32_t groups = (1u << a.s0) >> a.log_g;  // lo groups per hi
    uint32_t hi = blockIdx.x / groups, lg = blockIdx.x % groups;
    lo_base = lg << a.log_g;
    tile_base = ((uint64_t)hi << (a.s0 + a.S)) + lo_base;
  }
  auto global_of = [&](uint32_t l) -> uint64_t {
    if (first) return tile_base + l;
    uint32_t mid = l >> a.log_g, g = l & (G - 1);
    return tile_base + ((uint64_t)mid << a.s0) + g;
  };

  // ---- load
  // (A load through the bulk-copy engine -- two 16-byte cp.async.bulk per element into the swizzled slots, one
  // mbarrier per tile -- was measured in round 2: UBLKCP takes uniform-register addresses, so the 2048 copies of a
  // tile are issued lane by lane: 0.294 ms against 0.248 at 2^20.  profiles/r2_ntt_bulk_experiment.txt)
  for (uint32_t l = tid; l < tile; l += nthreads) {
    uint64_t gi = global_of(l);
    Fr x;
    if (a.bitrev_in) {
      // batched transforms: the permutation acts on the index inside one transform (low log_n bits)
      uint32_t src_i = a.log_n ? (__brev((uint32_t)gi & (n - 1)) >> (32 - a.log_n)) : 0;
      x = a.src[(gi & ~(uint64_t)(n - 1)) | src_i];
      if (a.pre_pow && src_i) x = x * power_at(a.pre_pow, src_i);
    } else {
      x = a.src[gi];
    }
    sts_elem(sm, tile, l, x);
  }
  __syncthreads();

  // ---- S butterfly stages, two at a time (radix 4 in registers): a thread owns the four elements whose
  // `mid` differs in bits u-1 and u, runs stage u on the pairs (00,01),(10,11) and stage u+1 on the
  // pairs (00,10),(01,11) without going back to shared memory.  Half the barriers and half the
  // shared-memory traffic of one-stage-at-a-time, two independent butterflies per step, and the three
  // twiddles of a quad (w1; w2; w2 * omega^(n/4)) are requested together before any arithmetic.
  auto decode = [&](uint32_t t, uint32_t per_sub_log, uint32_t& idx, uint32_t& g) {
    if (first) { g = t >> per_sub_log; idx = t & ((1u << per_sub_log) - 1); }
    else { idx = t >> a.log_g; g = t & (G - 1); }
  };
  auto slot = [&](uint32_t mid, uint32_t g) -> uint32_t { return first ? ((g << a.S) + mid) : ((mid << a.log_g) + g); };
  uint32_t u = 1;
  for (; u + 1 <= a.S; u += 2) {
    const uint32_t h = 1u << (u - 1);
    const uint32_t s = a.s0 + u;  // global index of the first of the two stages
    for (uint32_t q = tid; q < tile / 4; q += nthreads) {
      uint32_t qi, g;
      decode(q, a.S - 2, qi, g);
      uint32_t mid = ((qi >> (u - 1)) << (u + 1)) | (qi & (h - 1));
      uint32_t imod = first ? (mid & (h - 1)) : (((mid & (h - 1)) << a.s0) + lo_base + g);
      uint32_t e1 = imod << (a.log_n - s);
      uint32_t e2 = imod << (a.log_n - s - 1);
      uint32_t l00 = slot(mid, g), l01 = slot(mid + h, g), l10 = slot(mid + 2 * h, g), l11 = slot(mid + 3 * h, g);
      Fr w1 = a.tw[e1], w2a = a.tw[e2], w2b = a.tw[e2 + (n >> 2)];
      Fr x00 = lds_elem(sm, tile, l00), x01 = lds_elem(sm, tile, l01);
      Fr x10 = lds_elem(sm, tile, l10), x11 = lds_elem(sm, tile, l11);
      if (e1) { x01 = x01 * w1; x11 = x11 * w1; }
      Fr a0 = x00 + x01, a1 = x00 - x01, b0 = x10 + x11, b1 = x10 - x11;
      if (e2) b0 = b0 * w2a;
      b1 = b1 * w2b;
      sts_elem(sm, tile, l00, a0 + b0);
      sts_elem(sm, tile, l10, a0 - b0);
      sts_elem(sm, tile, l01, a1 + b1);
      sts_elem(sm, tile, l11, a1 - b1);
    }
    __syncthreads();
  }
  if (u <= a.S) {  // odd stage count: one plain radix-2 stage
    const uint32_t h = 1u << (u - 1);
    const uint32_t s = a.s0 + u;
    for (uint32_t t = tid; t < tile / 2; t += nthreads) {
      uint32_t bf, g;
      decode(t, a.S - 1, bf, g);
      uint32_t mid = ((bf >> (u - 1)) << u) | (bf & (h - 1));
      uint32_t l0 = slot(mid, g), l1 = slot(mid + h, g);
      uint32_t imod = first ? (mid & (h - 1)) : (((mid & (h - 1)) << a.s0) + lo_base + g);
      uint32_t e = imod << (a.log_n - s);
      Fr x0 = lds_elem(sm, tile, l0);
      Fr x1 = lds_elem(sm, tile, l1);
      if (e) x1 = x1 * a.tw[e];
      sts_elem(sm, tile, l0, x0 + x1);
      sts_elem(sm, tile, l1, x0 - x1);
    }
    __syncthreads();
  }

  // ---- store
  const bool last = (a.s0 + a.S) == a.log_n;
  for (uint32_t l = tid; l < tile; l += nthreads) {
    uint64_t gi = global_of(l);
    Fr x = lds_elem(sm, tile, l);
    if (last) {
      if (a.scale_n_inv) x = x * a.n_inv;
      uint32_t li = (uint32_t)gi & (n - 1);
      if (a.post_pow && li) x = x * power_at(a.post_pow, li);
    }
    a.dst[gi] = x;
  }
}

// ------------------------------------------------------------------ caches
static std::map<std::vector<uint8_t>, DevBuf> g_pow2_cache;   // key: x (32) + inverted (1)
static std::map<std::vector<uint8_t>, DevBuf> g_twiddle_cache;  // key: omega (32) + inverted (1) + log_n (1)
static size_t g_twiddle_bytes = 0;

const Fr* pow2_table(Context& c, const FrBytes& x, bool inverted, int* launches) {
  std::vector<uint8_t> key(x.b, x.b + 32);
  key.push_back(inverted ? 1 : 0);
  auto it = g_pow2_cache.find(key);
  if (it != g_pow2_cache.end()) return it->second.as<Fr>();
  if (g_pow2_cache.size() >= 512) {  // per-proof challenges (zeta, ...) would otherwise accumulate
    // two generations: tables handed out earlier in the current call stay valid until the next purge
    static std::vector<DevBuf> graveyard;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    for (auto& b : graveyard) b.release();
    graveyard.clear();
    for (auto& kv : g_pow2_cache) graveyard.push_back(kv.second);
    g_pow2_cache.clear();
  }
  DevBuf& buf = g_pow2_cache[key];
  buf.reserve(32 * sizeof(Fr));
  Fr xv;
  memcpy(xv.v, x.b, 32);
  pow2_table_kernel<<<1, 32, 0, c.stream>>>(xv, inverted ? 1 : 0, buf.as<Fr>());
  CUDA_CHECK_LAUNCH();
  if (launches) (*launches)++;
  return buf.as<Fr>();
}

static const Fr* twiddle_table(Context& c, const FrBytes& omega, bool inverted, uint32_t log_n, int* launches) {
  std::vector<uint8_t> key(omega.b, omega.b + 32);
  key.push_back(inverted ? 1 : 0);
  key.push_back((uint8_t)log_n);
  auto it = g_twiddle_cache.find(key);
  if (it != g_twiddle_cache.end()) return it->second.as<Fr>();
  // bound the cache (callers use a handful of domains: n, 2n..8n and their inverses)
  if (g_twiddle_bytes > (size_t(6) << 30)) {
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    for (auto& kv : g_twiddle_cache) kv.second.release();
    g_twiddle_cache.clear();
    g_twiddle_bytes = 0;
  }
  const Fr* p2 = pow2_table(c, omega, inverted, launches);
  uint32_t count = log_n ? (1u << (log_n - 1)) : 1;
  DevBuf& buf = g_twiddle_cache[key];
  buf.reserve((size_t)count * sizeof(Fr));
  g_twiddle_bytes += (size_t)count * sizeof(Fr);
  twiddle_table_kernel<<<ceil_div(count, 256), 256, 0, c.stream>>>(p2, count, buf.as<Fr>());
  CUDA_CHECK_LAUNCH();
  if (launches) (*launches)++;
  return buf.as<Fr>();
}

// lo[j] = x^j (j < 1024) followed by hi[k] = x^(1024 k) (k < max(1, 2^log_n / 1024)), Montgomery; cached per (x, log_n)
static std::map<std::vector<uint8_t>, DevBuf> g_coset_cache;
const Fr* power_table(Context& c, const FrBytes& x, bool inverted, uint32_t log_n, int* launches) {
  std::vector<uint8_t> key(x.b, x.b + 32);
  key.push_back(inverted ? 1 : 0);
  key.push_back((uint8_t)log_n);
  auto it = g_coset_cache.find(key);
  if (it != g_coset_cache.end()) return it->second.as<Fr>();
  if (g_coset_cache.size() >= 64) {  // per-proof challenges (zeta, zeta*omega, ...) would otherwise accumulate
    // two generations: a table handed out earlier in the current call stays valid until the NEXT purge
    static std::vector<DevBuf> graveyard;
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    for (auto& b : graveyard) b.release();
    graveyard.clear();
    for (auto& kv : g_coset_cache) graveyard.push_back(kv.second);
    g_coset_cache.clear();
  }
  const Fr* p2 = pow2_table(c, x, inverted, launches);
  uint32_t hi = log_n > 10 ? (1u << (log_n - 10)) : 1u;
  DevBuf& buf = g_coset_cache[key];
  buf.reserve((size_t)(1024 + hi) * sizeof(Fr));
  twiddle_table_kernel<<<4, 256, 0, c.stream>>>(p2, 1024, buf.as<Fr>());
  CUDA_CHECK_LAUNCH();
  twiddle_table_kernel<<<ceil_div(hi, 256), 256, 0, c.stream>>>(p2 + 10, hi, buf.as<Fr>() + 1024);  // (x^1024)^k
  CUDA_CHECK_LAUNCH();
  if (launches) (*launches) += 2;
  return buf.as<Fr>();
}

// n^-1 mod r in Montgomery form, computed on the host: n = 2^k so n^-1 = ((r+1)/2)^k; the host only
// shifts/adds 256-bit integers here (no field library needed): inv2^k by repeated halving of 1.
static void host_n_inv_mont(uint32_t log_n, Fr* out) {
  // value = R1 (Montgomery one) halved log_n times mod r: (x even) ? x/2 : (x + r)/2
  uint32_t x[9];
  for (int i = 0; i < 8; i++) x[i] = FrParams::R1[i];
  x[8] = 0;
  for (uint32_t k = 0; k < log_n; k++) {
    if (x[0] & 1) {
      uint64_t carry = 0;
      for (int i = 0; i < 8; i++) {
        uint64_t t = (uint64_t)x[i] + FrParams::MOD[i] + carry;
        x[i] = (uint32_t)t;
        carry = t >> 32;
      }
      x[8] = (uint32_t)carry;
    }
    for (int i = 0; i < 8; i++) x[i] = (x[i] >> 1) | (x[i + 1] << 31);
    x[8] = 0;
  }
  for (int i = 0; i < 8; i++) out->v[i] = x[i];
}

// Elements per thread in a tile.  8 (128 threads on a 1024-element tile, two radix-4 quads per thread and
// round) lets FOUR blocks share an SM instead of two at the same 16 warps: with four independent barrier
// domains the load / store phases of one block hide behind the butterflies of the others (2^22: 1.10 ->
// 0.98 ms; 16 elements per thread or 5-6 blocks at 96 / 80 registers measured slower).
static constexpr uint32_t NTT_ELEMS_PER_THREAD = 8;

int ntt_device(Context& c, Fr* data, Fr* scratch, uint32_t log_n, const FrBytes& omega, bool inverse,
               const FrBytes* coset_shift, uint32_t log_batch) {
  if (log_n + log_batch > 31) throw InvalidArgument("ntt: batch * n must be < 2^32");
  return ntt_device_count(c, data, scratch, log_n, omega, inverse, coset_shift, uint64_t(1) << log_batch);
}

int ntt_device_count(Context& c, Fr* data, Fr* scratch, uint32_t log_n, const FrBytes& omega, bool inverse,
                     const FrBytes* coset_shift, uint64_t count) {
  if (log_n > FrParams::TWO_ADICITY) throw InvalidArgument("ntt: log_n exceeds the 2-adicity of Fr (28)");
  if (count == 0 || (count << log_n) >= (uint64_t(1) << 32)) throw InvalidArgument("ntt: batch * n must be < 2^32");
  int launches = 0;
  // `count` independent transforms of 2^log_n contiguous elements: the same passes over a longer
  // array (tile indices simply run on into the next transform; twiddles depend on the position inside one)
  const uint32_t n = (uint32_t)(count << log_n);
  const Fr* tw = twiddle_table(c, omega, inverse, log_n, &launches);
  const Fr* pre = nullptr;
  const Fr* post = nullptr;
  if (coset_shift) {
    if (inverse) post = power_table(c, *coset_shift, true, log_n, &launches);
    else pre = power_table(c, *coset_shift, false, log_n, &launches);
  }
  NttPassArgs a;
  a.tw = tw;
  a.log_n = log_n;
  a.pre_pow = pre;
  a.post_pow = post;
  a.scale_n_inv = inverse ? 1 : 0;
  host_n_inv_mont(log_n, &a.n_inv);

  // pass 1: bit-reversed gather data -> scratch, stages 1..S1 on contiguous tiles
  uint32_t S1 = log_n < (uint32_t)NTT_LOG_TILE ? log_n : (uint32_t)NTT_LOG_TILE;
  a.src = data;
  a.dst = scratch;
  a.s0 = 0;
  a.S = S1;
  // small batched transforms: several of them share one 1024-element tile
  a.log_g = 0;
  if (log_n < (uint32_t)NTT_LOG_TILE) {
    a.log_g = (uint32_t)NTT_LOG_TILE - log_n;
    // a first-pass tile holds 2^log_g whole transforms: 2^log_g must divide the batch
    while (count & ((uint64_t(1) << a.log_g) - 1)) a.log_g--;
  }
  a.bitrev_in = 1;
  // a single-pass transform lives entirely inside one tile, which is read completely before it is
  // written: the permuting gather can then run in place
  if (S1 == log_n) a.dst = data;
  {
    uint32_t tile = 1u << (a.S + a.log_g);
    uint32_t threads = tile >= NTT_ELEMS_PER_THREAD ? tile / NTT_ELEMS_PER_THREAD : 1;
    ntt_pass_kernel<<<n / tile, threads, tile * 32, c.stream>>>(a);
    CUDA_CHECK_LAUNCH();
    launches++;
  }
  uint32_t done = S1;
  a.bitrev_in = 0;
  a.pre_pow = nullptr;
  a.src = scratch;
  a.dst = scratch;  // in place: every tile reads and writes exactly its own elements
  while (done < log_n) {
    uint32_t rem = log_n - done;
    uint32_t S = rem < (uint32_t)(NTT_LOG_TILE - NTT_Q) ? rem : (uint32_t)(NTT_LOG_TILE - NTT_Q);
    a.s0 = done;
    a.S = S;
    a.log_g = NTT_LOG_TILE - S;  // >= NTT_Q and <= s0 (s0 >= 10)
    if (a.log_g > a.s0) a.log_g = a.s0;
    if (done + S == log_n) a.dst = data;  // the last pass lands in the caller's buffer (no extra copy)
    uint32_t tile = 1u << (a.S + a.log_g);
    uint32_t threads = tile >= NTT_ELEMS_PER_THREAD ? tile / NTT_ELEMS_PER_THREAD : 1;
    ntt_pass_kernel<<<n / tile, threads, tile * 32, c.stream>>>(a);
    CUDA_CHECK_LAUNCH();
    launches++;
    done += S;
  }
  return launches;
}

}  // namespace zkp

using namespace zkp;

static DevBuf g_ntt_data, g_ntt_scratch;

extern "C" {

int zkp_fr_ntt(uint8_t* data, uint32_t log_n, const uint8_t omega[32], int inverse, const uint8_t* coset_shift) {
  return guarded([&](Context& c) {
    if (!data || !omega) throw InvalidArgument("zkp_fr_ntt: null argument");
    if (log_n > 28) throw InvalidArgument("zkp_fr_ntt: log_n must be <= 28");
    size_t bytes = (size_t(1) << log_n) * 32;
    g_ntt_data.reserve(bytes);
    g_ntt_scratch.reserve(bytes);
    FrBytes w, cs;
    memcpy(w.b, omega, 32);
    if (coset_shift) memcpy(cs.b, coset_shift, 32);
    CUDA_CHECK(cudaMemcpyAsync(g_ntt_data.p, data, bytes, cudaMemcpyHostToDevice, c.stream));
    c.launches += ntt_device(c, g_ntt_data.as<Fr>(), g_ntt_scratch.as<Fr>(), log_n, w, inverse != 0,
                             coset_shift ? &cs : nullptr);
    CUDA_CHECK(cudaMemcpyAsync(data, g_ntt_data.p, bytes, cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

int zkp_fr_ntt_dev(uint64_t scalars, uint64_t offset, uint32_t log_n, const uint8_t omega[32], int inverse,
                   const uint8_t* coset_shift) {
  return guarded([&](Context& c) {
    Resource* s = need(scalars, HandleKind::Scalars, "zkp_fr_ntt_dev");
    if (!omega) throw InvalidArgument("zkp_fr_ntt_dev: null omega");
    if (log_n > 28) throw InvalidArgument("zkp_fr_ntt_dev: log_n must be <= 28");
    uint64_t n = uint64_t(1) << log_n;
    if (!range_ok(offset, n, s->n)) throw InvalidArgument("zkp_fr_ntt_dev: range out of bounds");
    g_ntt_scratch.reserve(n * 32);
    FrBytes w, cs;
    memcpy(w.b, omega, 32);
    if (coset_shift) memcpy(cs.b, coset_shift, 32);
    c.launches += ntt_device(c, s->buf.as<Fr>() + offset, g_ntt_scratch.as<Fr>(), log_n, w, inverse != 0,
                             coset_shift ? &cs : nullptr);
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
  });
}

}  // extern "C"
