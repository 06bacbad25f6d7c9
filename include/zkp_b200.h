/* libzkp_b200 -- C ABI of the B200-native prover hot path for interactive-zkp-study.
 *
 * The reference (tokamak-network/interactive-zkp-study) is pure Python and has no FFI; the seam
 * is the set of Python callables listed in SURVEY.md section 8(a).  Each entry point below names
 * the reference code it replaces (file:line under /root/reference).  INTEGRATION.md shows the
 * ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - Field elements cross the boundary as 32 bytes little-endian, canonical (in [0, modulus)),
 *     NOT in Montgomery form.  Scalars (Fr) may be any 256-bit value; they are reduced mod r on
 *     the device (zkp/plonk/field.py:88 does `scalar % CURVE_ORDER`).
 *   - G1 affine point = x || y (64 B).  G2 affine point = x.c0 || x.c1 || y.c0 || y.c1 (128 B),
 *     c0 + c1*u as in py_ecc FQ2.coeffs (plonk_serializers.py:56-57).
 *   - The point at infinity (py_ecc `None`) is encoded as all-zero coordinates on input and
 *     reported through `*out_is_inf = 1` (coordinates zeroed) on output.
 *   - Every function returns 0 on success, a negative value on error; zkp_last_error() gives the
 *     message of the last failure on the calling thread's process.  The caller owns all host
 *     buffers; nothing is retained after return except through explicit handles.
 *   - There is no CPU fallback: without an sm_100 device zkp_init fails and every other call
 *     returns ZKP_ERR_NOT_INITIALISED.
 *   - Entry points are serialised by an internal mutex (Flask's dev server is multi-threaded and
 *     ctypes releases the GIL; app.py:1444).
 */
#ifndef ZKP_B200_H
#define ZKP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZKP_OK 0
#define ZKP_ERR_CUDA (-1)
#define ZKP_ERR_NOT_INITIALISED (-2)
#define ZKP_ERR_INVALID_ARGUMENT (-3)
#define ZKP_ERR_BAD_HANDLE (-4)
#define ZKP_ERR_NOT_DIVISIBLE (-5)

/* ---- lifecycle ---------------------------------------------------------------------------- */
/* device < 0: use $LOCAL_RANK if set, else 0.  Fails unless the device is compute capability 10.x. */
int zkp_init(int device);
int zkp_shutdown(void);
const char* zkp_last_error(void);
int zkp_device_info(char* name, int name_cap, int* sm_count, int* cc_major, int* cc_minor, int* sm_clock_khz);
int zkp_device_mem_info(uint64_t* free_bytes, uint64_t* total_bytes);
/* "domain:bus:device.function" of the library's GPU (e.g. to pin the calling process to the GPU's NUMA node
 * before it allocates page-locked staging buffers: sharded.bind_to_gpu_numa_node) */
int zkp_device_pci_bus_id(char* out, int cap);
/* number of kernels this library has launched since zkp_init (bench.py "gpu_launches") */
uint64_t zkp_launch_count(void);
/* CUDA-event timer on the library's stream (the stream every kernel is launched on) */
int zkp_timer_start(void);
int zkp_timer_stop(float* elapsed_ms);
int zkp_sync(void);

/* ---- multi-scalar multiplication ------------------------------------------------------------
 * sum_i scalars[i] * pts[i].  Replaces the scalar-mul loops of
 *   kzg.commit            zkp/plonk/kzg.py:59-67            (G1)
 *   proof_a / proof_c     zkp/groth16/proving.py:27-31,56-60,66-73   (G1)
 *   proof_b               zkp/groth16/proving.py:39-43      (G2)
 * i.e. py_ecc bn128.multiply + bn128.add per term.  Zero scalars and infinity points contribute
 * nothing (kzg.py:62-63).  n == 0 yields infinity. */
int zkp_g1_msm(const uint8_t* pts, const uint8_t* scalars, uint64_t n, uint8_t out_xy[64], int* out_is_inf);
int zkp_g2_msm(const uint8_t* pts, const uint8_t* scalars, uint64_t n, uint8_t out_xy[128], int* out_is_inf);

/* Device-resident static tables (srs.g1_powers, sigma1_2, sigma1_5, sigma2_2 are re-passed on every
 * reference call; the host wrapper caches them by identity) and device-resident scalar vectors. */
int zkp_g1_table_load(const uint8_t* pts, uint64_t n, uint64_t* handle);
int zkp_g2_table_load(const uint8_t* pts, uint64_t n, uint64_t* handle);
int zkp_scalars_load(const uint8_t* scalars, uint64_t n, uint64_t* handle);
int zkp_free(uint64_t handle);
/* Window precomputation for static tables (SRS / CRS are fixed per circuit): rewrites the table in
 * place as T[w][i] = 2^(window_bits*w) * P_i for every window w.  MSMs on such a table use that window
 * width, fold all windows into ONE bucket set and need no final doubling chain (the 254 sequential
 * doublings of the plain algorithm).  Memory: ceil(255/window_bits) x the plain table.  Results are
 * unchanged (same group element, same affine point). */
int zkp_g1_table_precompute(uint64_t table, int window_bits); /* 0 = width chosen for the table size */
int zkp_g2_table_precompute(uint64_t table, int window_bits);
int zkp_table_window_bits(uint64_t table, int* window_bits);  /* 0 = plain layout */
/* points [offset, offset+n) of the table, scalars from the host (H2D inside the call) */
int zkp_g1_msm_table(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t out_xy[64],
                     int* out_is_inf);
int zkp_g2_msm_table(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t out_xy[128],
                     int* out_is_inf);
/* everything resident: scalars [sc_offset, sc_offset+n) of a scalar handle */
int zkp_g1_msm_dev(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                   uint8_t out_xy[64], int* out_is_inf);
int zkp_g2_msm_dev(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                   uint8_t out_xy[128], int* out_is_inf);
/* Split form of zkp_g1/g2_msm_dev on the library's second stream: begin enqueues the MSM behind everything already
 * queued and returns at once, end waits for it and fetches the point; the calls made in between run beside it
 * (device_prover.prove starts the G2 element B this way before the quotient, which B does not depend on:
 * proving.py:35-45 needs only R.Bx).  One pending call per group. */
int zkp_g1_msm_dev_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n);
int zkp_g1_msm_dev_end(uint8_t out_xy[64], int* out_is_inf);
int zkp_g2_msm_dev_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n);
int zkp_g2_msm_dev_end(uint8_t out_xy[128], int* out_is_inf);
/* `count` independent MSMs on one table in one call: MSM k uses points [offsets[k], +lens[k]) and scalars
 * [sc_offsets[k], +lens[k]) of handle scalars[k]; out_xy holds count x 64 bytes.  The MSMs alternate between
 * two streams so the latency-bound tail of one overlaps the accumulation of the next (a prover issues its
 * commitments in groups: kzg.commit x3 in round1.py:80-82, round3.py:178-180, x2 in round5.py:174-175). */
int zkp_g1_msm_dev_batch(uint64_t table, uint32_t count, const uint64_t* scalars, const uint64_t* sc_offsets,
                         const uint64_t* offsets, const uint64_t* lens, uint8_t* out_xy, int* out_is_inf);
/* Many MSMs over ONE point range, for batch proving (count proofs of one circuit: the per-proof MSMs of
 * zkp/groth16/proving.py:23-75 share their points).  MSM j = sum_i s[sc_offset + j*n + i] * T[offset + i], j < count:
 * the scalar vectors lie back to back in one handle.  Plain and window-precomputed tables.  One Pippenger pass over
 * all count*n scalars (MSM j owns its own buckets), so the launch count does not depend on count.  out_xy holds
 * count x 64 (G1) / 128 (G2) bytes; out_is_inf (may be NULL) count flags.  count = 0 returns at once; n = 0 gives
 * count points at infinity.  ZKP_ERR_INVALID_ARGUMENT before any launch when count*W*n >= 2^32 (W = windows of the
 * table's width), count * (buckets per MSM) >= 2^31, or a range runs past its table / handle. */
int zkp_g1_msm_dev_many(uint64_t table, uint64_t offset, uint64_t n, uint32_t count, uint64_t scalars,
                        uint64_t sc_offset, uint8_t* out_xy, int* out_is_inf);
int zkp_g2_msm_dev_many(uint64_t table, uint64_t offset, uint64_t n, uint32_t count, uint64_t scalars,
                        uint64_t sc_offset, uint8_t* out_xy, int* out_is_inf);
/* Shard form for the multi-GPU path (SURVEY 8e): the un-normalised XYZZ partial sum of this rank's
 * point range, 4 coordinates x 32 B Montgomery for G1 (128 B); combine folds `count` partials
 * (gathered from all ranks) into the affine result.  `out_xyzz` and `partials` may be host memory or
 * device memory of this GPU (unified addressing), so the partial can be written straight into the
 * send buffer of the NCCL gather and folded straight out of its receive buffer; both calls return
 * after the library stream has drained. */
int zkp_g1_msm_dev_partial(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                           uint8_t out_xyzz[128]);
int zkp_g1_combine_partials(const uint8_t* partials, uint32_t count, uint8_t out_xy[64], int* out_is_inf);
/* Window-width override for experiments (0 = automatic). */
int zkp_msm_set_window_bits(int c);
/* Engine tunables for measurements by name (0 = automatic): "window_bits" as above; "accumulate" 1 = XYZZ chains
 * (the default), 2 = affine pairwise tree with shared inversions for buckets of up to 511 entries (csrc/msm_tree.cuh;
 * same results, measured slower on B200 and therefore opt-in); "tree_rounds" 1..9 affine rounds before the XYZZ
 * chains take over, "tree_items" most additions per thread under one shared inversion; "parts" 1..8 point ranges of
 * the part-streamed form (host scalars: upload + sort of range p+1 under the accumulation of range p; 0 = 4 ranges
 * from 2^18 points); "reduce_radix" 2/4/8/16/32 items per thread of a wide level of the bucket reduction (0 = 16),
 * "wide_log2" / "quad_log2" the item counts at which the wide and the quad-fused levels take over (0 = 17 / 12). */
int zkp_msm_set_option(const char* name, int value);

/* ---- multi-GPU: points sharded by contiguous range, one process per GPU (SURVEY 8e) -----------------
 * Scales the commit loop zkp/plonk/kzg.py:59-67 (and the proof-element sums of zkp/groth16/proving.py:
 * 23-75) across the GPUs of one box.  The library owns one NCCL communicator per process (NCCL is bound
 * with dlopen when the first of these calls is made; a single-GPU process never needs it):
 *   rank 0:      zkp_comm_unique_id(id)  -> hand the 128 bytes to every rank (any host channel)
 *   every rank:  zkp_comm_init(rank, world, id)   (collective; after zkp_init on that rank's device)
 * zkp_g1_msm_multi is then a collective call: every rank passes ITS shard (table / scalar handles and the
 * local range), runs the single-GPU Pippenger on it, and the un-normalised XYZZ partial sums (128 B per
 * rank in G1, 256 B in G2) are all-gathered over NVLink and folded on the library's stream with no host
 * synchronisation in between; every rank receives the affine result.  zkp_g1_msm_multi_table takes the
 * rank's scalars from host memory (H2D inside the call).  world == 1 is allowed. */
#define ZKP_COMM_ID_BYTES 128
int zkp_comm_unique_id(uint8_t out_id[ZKP_COMM_ID_BYTES]);
int zkp_comm_init(int rank, int world, const uint8_t id[ZKP_COMM_ID_BYTES]);
int zkp_comm_info(int* rank, int* world, int* nccl_version);
int zkp_comm_barrier(void); /* all ranks: returns once every rank's library stream has reached this point */
int zkp_comm_destroy(void);
int zkp_g1_msm_multi(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                     uint8_t out_xy[64], int* out_is_inf);
int zkp_g1_msm_multi_table(uint64_t table, uint64_t offset, const uint8_t* scalars, uint64_t n, uint8_t out_xy[64],
                           int* out_is_inf);
int zkp_g2_msm_multi(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n,
                     uint8_t out_xy[128], int* out_is_inf);
/* Split form on the library's second stream: begin enqueues the same local MSM -> all-gather -> fold and returns at
 * once, end waits for it and fetches the point; whatever is called in between runs beside it.  A Groth16 prover
 * starts its A and B elements this way before the quotient they do not depend on (proving.py:23-45 need only
 * R.Ax / R.Bx; hxr, poly_utils.py:116-125, feeds proof_c alone).  One pending call per group; collective. */
int zkp_g1_msm_multi_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n);
int zkp_g1_msm_multi_end(uint8_t out_xy[64], int* out_is_inf);
int zkp_g2_msm_multi_begin(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n);
int zkp_g2_msm_multi_end(uint8_t out_xy[128], int* out_is_inf);

/* ---- fixed-base batch scalar multiplication (CRS generation; SURVEY 8f-1) -------------------
 * out[i] = scalars[i] * base.  Replaces SRS.generate (zkp/plonk/srs.py:78-82) and
 * sigma12/sigma15/sigma22 (zkp/groth16/setup.py:18-23,56-60,64-69).  Result stays on the device
 * as a table handle; zkp_table_download copies canonical affine points back. */
int zkp_g1_fixed_base_mul(const uint8_t base_xy[64], const uint8_t* scalars, uint64_t n, uint64_t* out_table);
int zkp_g2_fixed_base_mul(const uint8_t base_xy[128], const uint8_t* scalars, uint64_t n, uint64_t* out_table);
int zkp_g1_fixed_base_mul_dev(const uint8_t base_xy[64], uint64_t scalars, uint64_t n, uint64_t* out_table);
int zkp_g2_fixed_base_mul_dev(const uint8_t base_xy[128], uint64_t scalars, uint64_t n, uint64_t* out_table);
/* Variable-base form for a powers-of-tau contribution (zkp/plonk/srs.py:50-87 makes [tau^i]_1; a participant with
 * secret s turns it into [(s tau)^i]_1 = s^i [tau^i]_1):
 * out[i] = scalars[sc_offset + i] * T[offset + i], i < n, as a new plain table handle (affine, same encoding).
 * Scalars are any 256-bit values, reduced mod r; a zero scalar or an infinity point gives infinity.  T may be plain
 * or window-precomputed (the points are its first row).  One thread per point: a 4-bit fixed-window ladder over
 * a per-thread table of 1..15 P.  n == 0 gives an empty table. */
int zkp_g1_table_scale(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n, uint64_t* out_table);
int zkp_g2_table_scale(uint64_t table, uint64_t offset, uint64_t scalars, uint64_t sc_offset, uint64_t n, uint64_t* out_table);
/* *first_bad = lowest index in [offset, offset+n) whose point is not on its curve (G2: or, with subgroup_check,
 * not in the order-r subgroup), UINT64_MAX if none.  Infinity (0,0) counts as valid.  Validation judges the point
 * as stored: zkp_g1/g2_table_load reduces every coordinate mod p on upload, so a coordinate c >= p is checked as
 * c mod p. */
int zkp_g1_table_validate(uint64_t table, uint64_t offset, uint64_t n, uint64_t* first_bad);
int zkp_g2_table_validate(uint64_t table, uint64_t offset, uint64_t n, int subgroup_check, uint64_t* first_bad);
int zkp_table_download(uint64_t table, uint64_t offset, uint64_t n, uint8_t* out_pts);
/* Compressed points (csrc/point_codec.cuh): the storage form of SRSs, keys and proofs, half the size of the affine
 * encoding above (the wire format of plonk_serializers.py:23-250 writes x and y).  G1: 32 B, x little-endian; G2:
 * 64 B, x.c0 | x.c1.  The top two bits of the last byte are flags: bit 7 y-sign (G1: y > (p-1)/2; G2: y1 > (p-1)/2,
 * or y0 > (p-1)/2 when y1 = 0), bit 6 infinity (every other bit zero).  Decoding takes the square root of x^3 + b,
 * so it also checks the point: a field >= p, both flags, an infinity encoding with another bit set, or an x with no
 * point is invalid, and G2 with subgroup_check also a twist point outside the order-r subgroup.
 * load: n encodings -> a new plain table, usable by every table entry point.  *first_bad = lowest invalid index, or
 *   UINT64_MAX.  On an invalid encoding *handle = 0 and nothing stays allocated (the call itself returns ZKP_OK).
 * download: table rows [offset, offset + n) -> compressed encodings on the host (G1 or G2 by handle kind); plain
 *   or window-precomputed tables (the points are the first row). */
int zkp_g1_table_load_compressed(const uint8_t* enc, uint64_t n, uint64_t* handle, uint64_t* first_bad);
int zkp_g2_table_load_compressed(const uint8_t* enc, uint64_t n, int subgroup_check, uint64_t* handle, uint64_t* first_bad);
int zkp_table_download_compressed(uint64_t table, uint64_t offset, uint64_t n, uint8_t* out);
int zkp_scalars_download(uint64_t scalars, uint64_t offset, uint64_t n, uint8_t* out);

/* ---- synthetic inputs (bench / large parity tests; SURVEY 8d) --------------------------------
 * Element i of stream `seed` is the first of 16 draws  v_t = mix(seed, 64*i + 4*t + j), j < 4 limbs
 * (SplitMix64 finaliser), masked to 254 bits, that is < r; if none is, draw 15 minus r.
 * oracle/synthetic.py restates it. */
int zkp_scalars_generate(uint64_t seed, uint64_t n, uint64_t* handle);

/* ---- Fr vectors: NTT and pointwise ops --------------------------------------------------------
 * zkp_fr_ntt: in-place on a host buffer of n = 2^log_n elements, natural order in and out.
 *   out[k] = sum_j in[j] * omega^(jk)                  replaces fft   zkp/plonk/polynomial.py:292-341
 *   inverse != 0: uses omega^-1 and scales by n^-1      replaces ifft  zkp/plonk/polynomial.py:344-378
 *   coset_shift != NULL: forward pre-scales in[j] *= k^j (coset_fft, zkp/plonk/utils.py:145-176);
 *                        inverse post-scales out[j] *= k^-j (coset_ifft, zkp/plonk/utils.py:179-205).
 * omega must be an element of order n (the reference passes get_root_of_unity(n) or its inverse). */
int zkp_fr_ntt(uint8_t* data, uint32_t log_n, const uint8_t omega[32], int inverse, const uint8_t* coset_shift);
int zkp_fr_ntt_dev(uint64_t scalars, uint64_t offset, uint32_t log_n, const uint8_t omega[32], int inverse,
                   const uint8_t* coset_shift);

/* op: 0 add, 1 sub, 2 mul (pointwise), 3 scale (out[i] = a[i] * b[0]); out may alias a or b.
 * Polynomial.__add__/__sub__/scalar __mul__ (polynomial.py:108-151) and the evaluation-form
 * products behind the quotients. */
int zkp_fr_vec_op(int op, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out);
/* out[i] = a[i]^-1, inv(0) = 0 (py_ecc prime_field_inv) */
int zkp_fr_batch_inverse(const uint8_t* a, uint64_t n, uint8_t* out);
/* out[0] = 1, out[i] = a[0]*...*a[i-1]: the running products of SRS.generate (zkp/plonk/srs.py:78-82,
 * tau^i) and of the permutation accumulator (zkp/plonk/permutation.py:120-135) as a parallel scan. */
int zkp_fr_prefix_product(const uint8_t* a, uint64_t n, uint8_t* out);
/* Horner evaluation p(x), Polynomial.evaluate zkp/plonk/polynomial.py:85-106 */
int zkp_fr_poly_eval(const uint8_t* coeffs, uint64_t n, const uint8_t x[32], uint8_t out[32]);

/* out[j] = sum_i vec[i] * mat[i*cols + j]: _multiply_vec_matrix (zkp/groth16/poly_utils.py:52-59), the
 * R.Ax / R.Bx / R.Cx products of hxr and the u_j = sum_i Rx_i*Ax_ij scalars of proof_a/b/c. */
int zkp_fr_vec_matrix(const uint8_t* vec, const uint8_t* mat, uint64_t rows, uint64_t cols, uint8_t* out);

/* ---- quotients ----------------------------------------------------------------------------- */
/* Groth16 hxr (zkp/groth16/poly_utils.py:116-125): P = a*b - c (len(a)=len(b)=len(c)=len),
 * (H, rem) = P divmod Z with Z of z_len coefficients.  h_out: 2*len-1 - z_len + 1 elements,
 * rem_out: z_len - 1 elements. */
int zkp_groth16_quotient(const uint8_t* a, const uint8_t* b, const uint8_t* c, uint64_t len, const uint8_t* z,
                         uint64_t z_len, uint8_t* h_out, uint8_t* rem_out);
/* The same on device-resident coefficient vectors (the 2^20-constraint configuration cannot go through
 * the reference's dense numWires x numGates lists: SURVEY F12).  Returns two new scalar handles
 * (quotient: 2*len - z_len coefficients; remainder: z_len - 1).  The inverse power series of the
 * reversed divisor is cached per z handle (Z(x) is fixed per circuit).  rem_out may be NULL: the
 * remainder (zero for a satisfied instance; three more transforms) is then not computed. */
int zkp_groth16_quotient_dev(uint64_t a, uint64_t b, uint64_t c, uint64_t len, uint64_t z, uint64_t z_len,
                             uint64_t* h_out, uint64_t* rem_out);
/* count quotients at once: proof j's coefficients at offset j*len of a, b and c.  Creates one handle of
 * count x (2*len - z_len) coefficients, proof j's quotient at offset j*(2*len - z_len); equal to
 * zkp_groth16_quotient_dev per proof (quotient only; shares its divisor cache).  Launches do not grow with count. */
int zkp_groth16_quotient_batch_dev(uint64_t a, uint64_t b, uint64_t c, uint64_t len, uint32_t count, uint64_t z,
                                   uint64_t z_len, uint64_t* h_out);
/* The three scalar vectors of count proofs (zkp/groth16/device_prover.py _scalars_ab / _scalars_c), one launch:
 * A_j = uA_j | 1 | r_j, B_j = uB_j | 1 | s_j (k + 2 each), C_j = r_j uB_j + s_j uA_j | r_j | rx_j | H_j | s_j | s_j r_j
 * (2k + 2 + m_priv).  uA, uB: count*k; h: count*(k-1) (ignored for k = 1); rx: count*m_priv (ignored for m_priv = 0);
 * rs, ss: count x 32 B canonical.  Creates three handles, proof j's vector at offset j * (its length). */
int zkp_groth16_batch_scalars_dev(uint64_t ua, uint64_t ub, uint64_t h, uint64_t rx, uint64_t k, uint64_t m_priv,
                                  uint32_t count, const uint8_t* rs, const uint8_t* ss, uint64_t* out_a,
                                  uint64_t* out_b, uint64_t* out_c);
/* The three MSMs of one proof (proving.py:23-75 as one MSM per element): A = <sa, ta> and C' = <sc, tc>
 * in G1 on one stream, B = <sb, tb2> in G2 on a second one, so the G2 work overlaps the G1 work.
 * Whole tables from index 0, na / nb / nc entries; out_is_inf = {A, B, C'} flags (may be NULL). */
int zkp_groth16_msms_dev(uint64_t ta, uint64_t sa, uint64_t na, uint64_t tb2, uint64_t sb, uint64_t nb, uint64_t tc,
                         uint64_t sc, uint64_t nc, uint8_t out_a[64], uint8_t out_b[128], uint8_t out_c[64],
                         int out_is_inf[3]);
/* Device-resident Fr vector utilities used to assemble MSM scalar vectors without leaving HBM. */
int zkp_scalars_alloc(uint64_t n, uint64_t* handle);
int zkp_scalars_copy(uint64_t dst, uint64_t dst_off, uint64_t src, uint64_t src_off, uint64_t n);
int zkp_scalars_upload(uint64_t dst, uint64_t dst_off, const uint8_t* host, uint64_t n);
int zkp_scalars_scale(uint64_t h, uint64_t off, uint64_t n, const uint8_t k[32]);
int zkp_fr_poly_eval_dev(uint64_t h, uint64_t off, uint64_t n, const uint8_t x[32], uint8_t out[32]);
/* ---- device-resident vector ops and the PLONK rounds at scale -------------------------------------
 * All on scalar handles, canonical values unless stated.  They are the device form of the Polynomial
 * arithmetic of zkp/plonk/polynomial.py:108-159 used by the prover rounds (round1..5.py). */
int zkp_fr_vec_op_dev(int op, uint64_t dst, uint64_t dst_off, uint64_t a, uint64_t a_off, uint64_t b, uint64_t b_off,
                      uint64_t n);                              /* 0 add, 1 sub, 2 mul */
int zkp_fr_axpy_dev(uint64_t dst, uint64_t dst_off, const uint8_t k[32], uint64_t src, uint64_t src_off, uint64_t n);
int zkp_scalars_add_const(uint64_t h, uint64_t off, uint64_t n, const uint8_t k[32]);
int zkp_scalars_fill_powers(uint64_t h, uint64_t off, uint64_t n, const uint8_t first[32], const uint8_t base[32]);
int zkp_scalars_convert(uint64_t h, uint64_t off, uint64_t n, int to_montgomery);
int zkp_scalars_is_zero(uint64_t h, uint64_t off, uint64_t n, int* out_all_zero);
int zkp_fr_batch_inverse_dev(uint64_t h, uint64_t off, uint64_t n, int montgomery);
int zkp_fr_scan_dev(int op, uint64_t dst, uint64_t dst_off, uint64_t src, uint64_t src_off, uint64_t n); /* 0 product, 1 sum */
/* out = sum_i a[i] * b[i] mod r (canonical).  With points P_i = s_i * G it verifies an MSM of any size with
 * one scalar multiplication on the host: sum_i k_i P_i == (<k, s>) * G (SURVEY 8d). */
int zkp_fr_dot_dev(uint64_t a, uint64_t a_off, uint64_t b, uint64_t b_off, uint64_t n, uint8_t out[32]);
/* up to 16 polynomials evaluated in the same launches, item k at xs[k] (round4.py:39-81: six evaluations) */
int zkp_fr_poly_eval_multi_dev(uint32_t count, const uint64_t* handles, const uint64_t* offs, const uint64_t* lens,
                               const uint8_t* xs, uint8_t* out);
/* dst[i] = sum_k coeffs[k] * src_k[i], i < n (items shorter than n contribute to their own length): the
 * scalar-times-polynomial sums of round5.py:90-160 in one pass; dst must not overlap a source */
int zkp_fr_lincomb_dev(uint64_t dst, uint64_t dst_off, uint64_t n, uint32_t count, const uint64_t* handles,
                       const uint64_t* offs, const uint64_t* lens, const uint8_t* coeffs);
/* (p(x) - p(zeta)) / (x - zeta): poly_div by a linear factor (round5.py:165-171, kzg.py:95-104) */
int zkp_fr_div_linear_dev(uint64_t src, uint64_t src_off, uint64_t n, const uint8_t zeta[32], uint64_t dst,
                          uint64_t dst_off);
/* numerators / denominators of the grand-product accumulator (permutation.py:120-135) */
int zkp_plonk_perm_terms_dev(uint64_t a, uint64_t b, uint64_t c, uint64_t s1, uint64_t s2, uint64_t s3, uint64_t n,
                             const uint8_t omega[32], const uint8_t beta[32], const uint8_t gamma[32], uint64_t num,
                             uint64_t den);
/* round 3 on the coset g*<w_N>, N = ext*n >= 3n+6 (round3.py:114-147 evaluated pointwise; SURVEY H5):
 * ext = 4 for n >= 8, 8 for n = 2, 4 and 16 for n = 1. */
int zkp_plonk_coset_setup_dev(uint64_t n, uint32_t ext, const uint8_t g[32], const uint8_t w8[32],
                              const uint8_t g_pow_n[32], const uint8_t w8_pow_n[32], uint64_t x_out, uint64_t l1f_out,
                              uint64_t zh8_out);
int zkp_plonk_quotient_dev(const uint64_t evals[12], uint64_t n, uint32_t ext, uint64_t x, uint64_t l1f, uint64_t zh8,
                           const uint8_t beta[32], const uint8_t gamma[32], const uint8_t alpha[32], uint64_t t_out);
/* ---- batch PLONK proving: count proofs of one circuit per call (zkp/plonk/device_prover.py prove_batch) ----------
 * The rounds of zkp/plonk/prover/round1..5.py for count witnesses in launches whose number does not depend on
 * count.  Every proof has its own challenges: betas, gammas, alphas, zetas are count x 32 B canonical arrays.  Each
 * entry gives, per proof, exactly what its single-proof counterpart above gives.  Ranges are checked before any
 * launch (ZKP_ERR_INVALID_ARGUMENT).
 * zkp_fr_ntt_many_dev: count contiguous transforms of 2^log_n at offset (zkp_fr_ntt_dev each; fft / ifft /
 *   coset_fft of zkp/plonk/polynomial.py:292-378, utils.py:145-205); count * 2^log_n < 2^32.
 * zkp_plonk_blind_many_dev: dst_v = src_v + (b_v0 + .. + b_v,k-1 x^(k-1))(x^n - 1) at dst_stride >= n + k, v < nvec,
 *   src_v = n coefficients at src_off + v * src_stride, blinds nvec x k (round1.py:38-108 / round2.py:45-85 blinding).
 * zkp_plonk_perm_terms_many_dev: zkp_plonk_perm_terms_dev per proof (permutation.py:120-135), witness j at
 *   off + j * n of a, b, c; sigma shared; num / den: count * n.
 * zkp_fr_scan_many_dev: zkp_fr_scan_dev over count segments of seg elements, each starting afresh (the accumulator
 *   z_j of permutation.py:120-135 starts at 1 in every proof).
 * zkp_plonk_coset_inputs_many_dev: the round-3 transform inputs: 3 count wire blocks (stride n + 2) and count z
 *   blocks (stride n + 3) zero-padded to 2^log_N, Montgomery, in the order a_*, b_*, c_*, z_* (round3.py:56-184).
 * zkp_plonk_quotient_many_dev: zkp_plonk_quotient_dev per proof on those 4 count blocks; circuit = the 8 shared
 *   coset evaluations q_l, q_r, q_o, q_m, q_c, s_sigma1..3; t_out: count blocks of N = ext * n (round3.py:114-147).
 * zkp_plonk_divisible_many_dev: lowest j whose t_j has a non-zero coefficient at 3n + 6 or above, UINT64_MAX if
 *   none (the divisibility check of round3.py:150-155).
 * zkp_plonk_split_t_many_dev: t_lo | t_mid | t_hi of every proof from Montgomery t blocks, canonical, each at stride
 *   n + 6 with t_lo, t_mid zero-padded; vector part * count + j (round3.py:169-171).
 * zkp_fr_poly_eval_many_dev: groups x count Horner evaluations (round4.py:39-81, polynomial.py:85-106): group g's
 *   vector of proof j at offs[g] + j * strides[g] (0: one vector shared by all proofs), lens[g] coefficients, at
 *   points[sel[g] * count + j]; out[g * count + j]; at most 16 groups.
 * zkp_fr_lincomb_many_dev: dst_j[i] = sum_k coeffs[j][k] src_k,j[i] + (i == 0 ? coeffs[j][K] : 0), i < n, sources
 *   shared or per proof as above, coeffs count x (K + 1) (round5.py:90-160); dst must not overlap a source.
 * zkp_fr_div_linear_many_dev: zkp_fr_div_linear_dev per proof (round5.py:165-171, kzg.py:95-104), p_j at
 *   src_off + j * src_stride (len coefficients), quotient j at dst_off + j * dst_stride; zeta_j = 0 is a shift.
 * Public inputs: proof j has ell <= n public inputs x_j,0..ell-1 at off + j * stride of the scalar handle pub, and
 * PI_j(X) = sum_i x_j,i L_i(X) (utils.py:84-116 public_input_polynomial) enters the gate identity with a plus sign
 * (round3.py:33).  ell = 0 leaves every result as without public inputs.
 * zkp_plonk_pi_scatter_many_dev: count blocks of n evaluations at dst_off: x_j,i at row i < ell, zero elsewhere.
 * zkp_plonk_coset_inputs_pi_many_dev: zkp_plonk_coset_inputs_many_dev plus a fifth group of count blocks: the PI_j
 *   coefficients (count blocks of n at pi_off), zero-padded to 2^log_N, Montgomery; 5 * count * 2^log_N < 2^32.
 * zkp_plonk_quotient_pi_many_dev: zkp_plonk_quotient_many_dev on 5 count blocks, the fifth PI_j on the coset, added
 *   to q_c in the gate term (round3.py:33, 114-147).
 * zkp_plonk_pi_eval_many_dev: out_j = PI_j(zeta_j) = sum_{i < ell} x_j,i w^i (zeta_j^n - 1) / (n (zeta_j - w^i))
 *   (utils.py:25-81 lagrange_basis_eval, public_input_poly_eval; round5.py:20,30; verifier.py:99), x_j,i when
 *   zeta_j = w^i with i < ell, 0 when i >= ell; the inversions are one batch in which a zero gap stays zero. */
int zkp_fr_ntt_many_dev(uint64_t scalars, uint64_t offset, uint32_t log_n, const uint8_t omega[32], int inverse,
                        const uint8_t* coset_shift, uint32_t count);
int zkp_plonk_blind_many_dev(uint64_t src, uint64_t src_off, uint64_t src_stride, uint64_t n, uint32_t nvec,
                             const uint8_t* blinds, uint32_t k, uint64_t dst, uint64_t dst_off, uint64_t dst_stride);
int zkp_plonk_perm_terms_many_dev(uint64_t a, uint64_t b, uint64_t c, uint64_t off, uint64_t s1, uint64_t s2, uint64_t s3,
                                  uint64_t n, uint32_t count, const uint8_t omega[32], const uint8_t* betas,
                                  const uint8_t* gammas, uint64_t num, uint64_t den);
int zkp_fr_scan_many_dev(int op, uint64_t dst, uint64_t dst_off, uint64_t src, uint64_t src_off, uint64_t seg,
                         uint32_t count);
int zkp_plonk_coset_inputs_many_dev(uint64_t wires, uint64_t z, uint64_t n, uint32_t count, uint32_t log_N, uint64_t out);
int zkp_plonk_quotient_many_dev(uint64_t evals, const uint64_t circuit[8], uint64_t n, uint32_t ext, uint32_t count,
                                uint64_t x, uint64_t l1f, uint64_t zh8, const uint8_t* betas, const uint8_t* gammas,
                                const uint8_t* alphas, uint64_t t_out);
int zkp_plonk_divisible_many_dev(uint64_t t, uint64_t n, uint32_t ext, uint32_t count, uint64_t* first_bad);
int zkp_plonk_split_t_many_dev(uint64_t t, uint64_t n, uint32_t ext, uint32_t count, uint64_t out);
int zkp_fr_poly_eval_many_dev(uint32_t groups, const uint64_t* handles, const uint64_t* offs, const uint64_t* strides,
                              const uint64_t* lens, const uint32_t* sel, uint32_t count, uint32_t npsets,
                              const uint8_t* points, uint8_t* out);
int zkp_fr_lincomb_many_dev(uint64_t dst, uint64_t dst_off, uint64_t dst_stride, uint64_t n, uint32_t count, uint32_t K,
                            const uint64_t* handles, const uint64_t* offs, const uint64_t* strides, const uint64_t* lens,
                            const uint8_t* coeffs);
int zkp_fr_div_linear_many_dev(uint64_t src, uint64_t src_off, uint64_t src_stride, uint64_t len, uint32_t count,
                               const uint8_t* zetas, uint64_t dst, uint64_t dst_off, uint64_t dst_stride);
int zkp_plonk_pi_scatter_many_dev(uint64_t pub, uint64_t off, uint64_t stride, uint64_t ell, uint64_t n, uint32_t count,
                                  uint64_t dst, uint64_t dst_off);
int zkp_plonk_coset_inputs_pi_many_dev(uint64_t wires, uint64_t z, uint64_t pi, uint64_t pi_off, uint64_t n, uint32_t count,
                                       uint32_t log_N, uint64_t out);
int zkp_plonk_quotient_pi_many_dev(uint64_t evals, const uint64_t circuit[8], uint64_t n, uint32_t ext, uint32_t count,
                                   uint64_t x, uint64_t l1f, uint64_t zh8, const uint8_t* betas, const uint8_t* gammas,
                                   const uint8_t* alphas, uint64_t t_out);
int zkp_plonk_pi_eval_many_dev(uint64_t pub, uint64_t off, uint64_t stride, uint64_t ell, uint64_t n, uint32_t count,
                               const uint8_t omega[32], const uint8_t* zetas, uint8_t* out);
/* General product and exact/long division over Fr in coefficient form
 * (Polynomial.__mul__ polynomial.py:144-159; poly_div polynomial.py:385-435). */
int zkp_fr_poly_mul(const uint8_t* a, uint64_t a_len, const uint8_t* b, uint64_t b_len, uint8_t* out);
int zkp_fr_poly_divmod(const uint8_t* a, uint64_t a_len, const uint8_t* b, uint64_t b_len, uint8_t* q_out,
                       uint8_t* r_out);

/* ---- QAP construction at scale over the reference's domain {1..k} (SURVEY 8 f2) ------------------
 * The reference interpolates every wire's R1CS column through x = 1..k in floating point, scaled by
 * the Vandermonde determinant (qap_creator_lcm.py:50-78 mk_singleton/lagrange_interp, :114-135
 * r1cs_to_qap_times_lcm), and contracts the dense numWires x numGates result with the witness
 * (poly_utils.py:52-59 _multiply_vec_matrix inside hxr :116-125).  By linearity R.Ax = interp(A.w):
 * one sparse matrix-vector product and one exact interpolation per matrix.
 * zkp_sparse_load: CSR matrix (row_ptr[rows+1], col_idx[nnz], values nnz x 32 B canonical) -> handle
 * (release with zkp_free).  zkp_sparse_matvec_dev: out[row] = sum val * vec[col] on scalar handles.
 * zkp_fr_ap_interpolate_dev: coefficients (k, degree < k) of the polynomial with p(j+1) = values[j],
 * optionally times `scale` (the reference's determinant factor; NULL = 1).
 * zkp_fr_ap_vanishing_dev: the k+1 coefficients of Z(x) = (x-1)(x-2)...(x-k) (qap_creator_lcm.py:128-135).
 * zkp_fr_ap_lagrange_dev: the Lagrange basis of {1..k} evaluated at x (k values), for the CRS terms
 * A_i(x), B_i(x), C_i(x) of setup.py:26-57 without the coefficient matrices. */
int zkp_sparse_load(const uint32_t* row_ptr, const uint32_t* col_idx, const uint8_t* values, uint64_t rows, uint64_t cols,
                    uint64_t nnz, uint64_t* handle);
int zkp_sparse_matvec_dev(uint64_t matrix, uint64_t vec, uint64_t vec_off, uint64_t out, uint64_t out_off);
int zkp_fr_ap_interpolate_dev(uint64_t values, uint64_t off, uint64_t k, const uint8_t* scale, uint64_t out,
                              uint64_t out_off);
/* The same over count vectors in the same launches: witness j at vec_off + j*cols, output j at out_off + j*rows;
 * values j at off + j*k, coefficients j at out_off + j*k. */
int zkp_sparse_matvec_many_dev(uint64_t matrix, uint64_t vec, uint64_t vec_off, uint64_t out, uint64_t out_off,
                               uint32_t count);
int zkp_fr_ap_interpolate_many_dev(uint64_t values, uint64_t off, uint64_t k, uint32_t count, const uint8_t* scale,
                                   uint64_t out, uint64_t out_off);
int zkp_fr_ap_vanishing_dev(uint64_t k, uint64_t out, uint64_t out_off);
int zkp_fr_ap_lagrange_dev(uint64_t k, const uint8_t x[32], uint64_t out, uint64_t out_off);

/* ---- witness solving: count witnesses of one circuit per call (zkp/witness.py, csrc/witness.cuh) ---------------
 * Replaces the host witness computation of the reference (zkp/groth16/code_to_r1cs.py variable assignment,
 * zkp/plonk/circuit.py wire values).  A program has `vars` variables (v_0 = 1, in_var[n_in] from the caller) and
 * `steps` steps sorted by level (level_ptr[levels + 1]); step s has four linear forms, rows 4s..4s+3 of a CSR matrix
 * over the variables (row_ptr[4 steps + 1], col_idx[nnz], values nnz x 32 B canonical): alpha, beta, gamma, delta.
 * N = (alpha.v)(beta.v) + gamma.v, D = delta.v.  out_var[s] = 0xFFFFFFFF: a check step (N must be 0); otherwise
 * v[out_var[s]] = N / D (delta = 1 v_0: no inversion).  Load checks that every variable other than v_0 and the inputs
 * is written by exactly one step and that each step reads only variables of lower levels.
 * zkp_witness_solve_many_dev: witness j reads its n_in inputs at in_off + j*n_in and writes its `vars` canonical
 * values at out_off + j*vars.  *first_bad = lowest j*steps + s whose step failed (D = 0, or N != 0 in a check), or
 * UINT64_MAX.  One launch whatever count and depth are; count = 0 launches nothing.  Ranges are checked before any
 * launch (ZKP_ERR_INVALID_ARGUMENT). */
int zkp_witness_program_load(const uint32_t* row_ptr, const uint32_t* col_idx, const uint8_t* values, uint64_t nnz,
                             const uint32_t* out_var, uint64_t steps, const uint32_t* level_ptr, uint64_t levels,
                             const uint32_t* in_var, uint64_t n_in, uint64_t vars, uint64_t* handle);
int zkp_witness_solve_many_dev(uint64_t program, uint64_t inputs, uint64_t in_off, uint32_t count, uint64_t out,
                               uint64_t out_off, uint64_t* first_bad);

/* ---- pairings (verifier side) -------------------------------------------------------------------
 * The BN254 optimal-Ate pairing of py_ecc's bn128.pairing(Q, P), Q in G2, P in G1, in the encodings above
 * (csrc/pairing.cu).  Replaces the pairings of zkp/groth16/verifying.py:29-40 (e(A, B) == e(alpha, beta)
 * e(sum r_i sigma1_3[i], gamma) e(C, delta)), zkp/plonk/verifier.py:42-208 (e(A, [tau]_2) == e(B, [1]_2)) and
 * zkp/plonk/kzg.py:117-160 (verify_opening).  An input point that is not on its curve (or has a coordinate not
 * below p) fails with ZKP_ERR_INVALID_ARGUMENT, as py_ecc's `assert is_on_curve` does.
 * zkp_pairing: e(Q, P) as py_ecc's FQ12, 12 x 32 B canonical coefficients of w^0..w^11 (mod w^12 - 18 w^6 + 82);
 * either input at infinity -> 1.
 * zkp_pairing_check: *out_ok = [ prod_i e(Q_i, k_i P_i) == 1 ] over `count` pairs (g2s: count x 128 B, g1s:
 * count x 64 B); scalars == NULL means k_i = 1, otherwise count x 32 B, reduced mod r; a pair with infinity on
 * either side (also k_i P_i = infinity) contributes 1.  g2_subgroup_check != 0: any Q_i outside G2 ([r] Q_i !=
 * infinity) makes *out_ok = 0.  count == 0 -> *out_ok = 1.  One Miller loop per pair on the device, one final
 * exponentiation per call: the batch verifiers (verify_batch) check k proofs with one call. */
int zkp_pairing(const uint8_t g2_xy[128], const uint8_t g1_xy[64], uint8_t out_fq12[384]);
int zkp_pairing_check(const uint8_t* g2s, const uint8_t* g1s, const uint8_t* scalars, uint64_t count,
                      int g2_subgroup_check, int* out_ok);

/* ---- measurement helpers (bench.py) -----------------------------------------------------------
 * Per-stage CUDA-event profile of the most recent MSM (events recorded on the library stream).
 * zkp_msm_last_profile sums the stages whose name contains `stage` ("accumulate", "ws", "horner",
 * "digits", "scatter", "tasks", "fold"; NULL = the whole MSM), in microseconds. */
int zkp_msm_profile(int enable);
int zkp_msm_last_profile(const char* stage, float* out_us);
/* Page-locked host staging buffers for the end-to-end measurement (H2D from pinned memory). */
int zkp_pinned_alloc(uint64_t bytes, void** out);
int zkp_pinned_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* ZKP_B200_H */
