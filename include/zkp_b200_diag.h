/* libzkp_b200 -- diagnostics and self-test hooks (csrc/diag.cu).
 *
 * NOT part of the product ABI: nothing on a prover path calls these.  bench.py uses zkp_imad_peak for
 * the roofline denominator (MEASURED_PEAKS.json carries no integer peak), tools/ use zkp_latency_probe,
 * and tests/test_gpu_field.py drives the field / group-law kernels through zkp_dbg_*.
 * Same conventions as include/zkp_b200.h (return codes, zkp_last_error, 32-byte little-endian elements).
 */
#ifndef ZKP_B200_DIAG_H
#define ZKP_B200_DIAG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Integer-MAD microbenchmarks, G(limb-MAC)/s over the whole chip.  variant 0 = IMAD.WIDE.U32 peak in the
 * carry-chain form the field arithmetic issues (mad.lo.cc / madc.hi.cc pairs -> IMAD.WIDE.U32[.X]), four
 * independent 4-lane chains per thread: the roofline denominator; 1 = IMAD (32-bit lo); 2 = IMAD.HI;
 * 3 = chains of whole Fp Montgomery products (136 limb-MACs each); 4 = plain mad.wide.u32 with register
 * factors (ptxas adds separate 64-bit additions: reads below variant 0); 5 = variant 4 interleaved with
 * 64-bit shift-and-add steps on the integer ALU. */
int zkp_imad_peak(int variant, double* gmacs_per_s, double* sm_clock_mhz_effective);
/* Single-thread latency of one operation (ns): mode 0/1/2 = 1/2/4 independent Fp products per step,
 * 3 = XYZZ add (inlined products), 4 = XYZZ add (out-of-line products), 5 = mixed add, 6 = double;
 * 7 / 8 = XYZZ add on a quad of lanes (inlined / out-of-line products), 9 = double on a quad,
 * 10 = Fp inversion (batched division steps, Mont256::inv), 11 = Fp inversion by binary extended Euclid,
 * 12-15 = pieces of the quad addition (without its edge-case tail / product levels only / four dependent products
 * on a lone thread / the same with a broadcast after each).
 * The MSM's reduction tail is bounded by these, not by throughput. */
int zkp_latency_probe(int mode, double* ns_per_op);
/* Field-op self-test hooks used by tests/ (field: 0 = Fp, 1 = Fr, 2 = Fp2 with 64-byte elements c0 || c1 and
 * ops 2 / 3 / 4 / 9 only; op: 0 add, 1 sub, 2 mul, 3 inv, 4 sqr,
 * 5 Fermat inverse, 6 mul as 512-bit product + separate Montgomery reduction, 7 inverse by binary extended Euclid,
 * 8 a b - (a + b)(a - b) through the lazily reduced product pair of the group formulas' Y coordinate,
 * 9 the square root of the point decoder (csrc/point_codec.cuh; Fp and Fp2 only), all-ones bytes when a is not a
 * square) */
int zkp_dbg_field_op(int field, int op, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out);
/* out[i] = a[i] + b[i] (group: 0 = G1, 1 = G2; 2 / 3 = the same through the quad-lane operations of
 * csrc/ec_quad.cuh) via XYZZ, result affine; exercises all edge cases */
int zkp_dbg_point_add(int group, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out);
/* Fp12 self-test hook (csrc/pairing.cu): n elements of 384 B each in py_ecc's FQ12 basis (12 canonical
 * coefficients of w^0..w^11); op: 0 a * b, 1 a^2, 2 cyclotomic squaring (valid for a in the cyclotomic subgroup),
 * 3 1 / a, 4 / 5 / 6 the Frobenius maps pi, pi^2, pi^3, 7 the final exponentiation a^((p^12 - 1) / r).
 * b is read by op 0 only. */
int zkp_dbg_fp12_op(int op, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out);
/* Guarded allocation (start the process with ZKP_B200_GUARD=1): every device block of the library carries a
 * 512-byte canary zone on both sides; this checks the zones of all live blocks (blocks are also checked when
 * freed) and returns the number of live blocks and of blocks found damaged so far.  compute-sanitizer is closed
 * on the B200 pool; tests/conftest.py turns a damaged canary into a failure of the GPU suite. */
int zkp_debug_check_guards(uint64_t* live_buffers, uint64_t* violations);
#ifdef __cplusplus
}
#endif
#endif /* ZKP_B200_DIAG_H */
