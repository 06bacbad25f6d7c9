"""PLONK proving at scale: the five rounds of /root/reference/zkp/plonk/prover/round1..5.py on
device-resident vectors (BASELINE config 4).

The list-of-FR `Polynomial` objects of the reference cost O(n) Python conversions per operation and its
round 3 is O(n^2); at 2^20 gates the rounds have to stay in HBM.  Same protocol, same transcript, same
proof elements (bit-identical to the reference-minted golden proofs for equal blinding scalars):

  round 1  3 iNTT, blinding, 3 MSMs                          (round1.py:38-108)
  round 2  grand product = fused num/den kernel + batch inversion + product scan, iNTT, MSM (on the second stream,
           beside the coset transforms of round 3, which do not need alpha)                  (round2.py, permutation.py:89-137)
  round 3  quotient on the coset {g w_N^i}, N = 4n (the smallest power of two >= 3n+6): 4 coset NTTs of the witness polynomials (the 8 circuit
           polynomials' coset evaluations are part of the device key), one pointwise kernel
           t = [gate + alpha perm]/Z_H + alpha^2 (z-1)/(n(x-1)), one inverse coset NTT, divisibility =
           "coefficients above 3n+5 vanish", 3 MSMs                                   (round3.py:56-184)
  round 4  6 two-level Horner evaluations                     (round4.py:39-81)
  round 5  linearisation r(x) by axpy, the two openings as (P(x)-P(z))/(x-z) = powers + sum scan, 2 MSMs (round5.py:42-175)

Public inputs (beyond the reference, whose PI is always 0): a key preprocessed with num_public_inputs = l > 0 binds
each proof to l field elements x_0..x_{l-1}.  Row i < l is public input i's gate, PI(X) = sum_i x_i L_i(X) (the
reference's utils.public_input_polynomial) enters the gate identity as q_L a + q_R b + q_O c + q_M ab + q_C + PI = 0
on H, the transcript absorbs append_scalar(b"public_input", x_i) for i = 0..l-1 before the round-1 commitments, the
quotient's gate term gains PI on the coset and the linearisation constant gains PI(zeta).  l = 0 is exactly the
protocol above: nothing extra is hashed and every proof is unchanged.
"""
import numbers
import secrets

import numpy as np

from ... import native
from ...compat import curve_order, g1_from_ints
from .field import FR, get_root_of_unity
from .transcript import Transcript
from .prover import Proof

R = curve_order
K1, K2 = 2, 3
COSET_SHIFT = 5          # 5^(8n) != 1 (5 is a non-residue), so Z_H never vanishes on g*<w8>
CIRCUIT_POLYS = ("q_l", "q_r", "q_o", "q_m", "q_c", "s_sigma1", "s_sigma2", "s_sigma3")


class DeviceKey:
    """Preprocessed circuit on the device: coefficient forms (canonical), their 8n-coset evaluations
    (Montgomery), sigma evaluations on H, the static coset data and the SRS table."""

    def __init__(self):
        self.coeffs, self.coset, self.comm = {}, {}, {}
        self.ranks, self.srs_range = None, None     # sharded SRS: the communicator and this rank's row range
        self.num_public_inputs = 0


def _alloc_from(src, n, total):
    h = native.scalars_alloc(total)
    native.scalars_copy(h, 0, src, 0, n)
    return h


def _commit(key, h, off, length):
    """kzg.commit (kzg.py:32-67) of coefficients h[off : off + length] against SRS powers 0 .. length - 1."""
    if key.ranks is None:
        return native.g1_msm_dev(key.srs_table, 0, h, off, length)
    # sharded SRS (SURVEY 8e): this rank holds powers [start, start + count); its share of the commitment is the
    # MSM over the powers of its range that the polynomial reaches (possibly none), folded inside the library
    start, count = key.srs_range
    m = max(0, min(count, length - start))
    return native.g1_msm_multi(key.srs_table, 0, h, off + start if m else 0, m)


def _commit_begin(key, h, off, length):
    """_commit in split form: the MSM (or this rank's share and the collective) is enqueued on the library's second
    stream; _commit_end fetches the point.  What is called in between runs beside it."""
    if key.ranks is None:
        native.msm_dev_begin(key.srs_table, 0, h, off, length)
    else:
        start, count = key.srs_range
        m = max(0, min(count, length - start))
        native.msm_multi_begin(key.srs_table, 0, h, off + start if m else 0, m)


def _commit_end(key):
    return native.msm_dev_end("g1") if key.ranks is None else native.msm_multi_end("g1")


def _commit_many(key, items):
    """Several commitments against the SRS: items = [(handle, offset, length)].  On one GPU they go out as one
    pipelined call (the tail of one MSM overlaps the accumulation of the next); sharded, each is a collective."""
    if key.ranks is not None:
        return [_commit(key, h, off, length) for h, off, length in items]
    return native.g1_msm_dev_batch(key.srs_table, [(h, off, 0, length) for h, off, length in items])


def preprocess(n, selector_evals, sigma_evals, srs_table, srs_size, comm=None, srs_range=None, num_public_inputs=0):
    """selector_evals: 5 handles (q_l, q_r, q_o, q_m, q_c evaluations on H, n each); sigma_evals: 3
    handles with the evaluations of S_sigma1..3 (permutation.py:44-86).  Mirrors
    preprocessor.py:59-130: 8 iNTTs + 8 commitments, plus the static round-3 data.
    comm / srs_range: a sharded.Communicator and the (start, count) row range of the SRS that `srs_table`
    holds on this rank; every commitment of preprocess() and prove() is then a collective over the ranks,
    while the NTT / quotient work is done by every rank for itself (it stays single-GPU work, SURVEY 8e).
    num_public_inputs: l, 0 <= l <= n; the proofs of the key are bound to l public inputs (gates 0..l-1).
    ValueError for l outside that range or l > 0 with a sharded SRS."""
    num_public_inputs = int(num_public_inputs)
    if not 0 <= num_public_inputs <= n:
        raise ValueError("preprocess: num_public_inputs must be in [0, n = %d], got %d" % (n, num_public_inputs))
    if num_public_inputs and comm is not None:
        raise ValueError("preprocess: public inputs are not supported on a sharded key")
    key = DeviceKey()
    key.num_public_inputs = num_public_inputs
    key.ranks, key.srs_range = comm, srs_range
    key.n, key.log_n = n, n.bit_length() - 1
    key.omega = int(get_root_of_unity(n))
    # quotient coset: the smallest power-of-two multiple of n with at least 3n+6 points (deg t = 3n+5)
    key.ext = 4 if n >= 8 else (8 if n >= 2 else 16)
    key.log_ext = key.ext.bit_length() - 1
    key.N8 = key.ext * n
    key.omega8 = int(get_root_of_unity(key.N8))
    key.srs_table, key.srs_size = srs_table, srs_size
    key.sigma_evals = list(sigma_evals)
    for name, ev in zip(CIRCUIT_POLYS, list(selector_evals) + list(sigma_evals)):
        c = _alloc_from(ev, n, n)
        native.ntt_dev(c, 0, key.log_n, key.omega, inverse=True)
        key.coeffs[name] = c
        e = _alloc_from(c, n, key.N8)
        native.scalars_convert(e, 0, n, True)
        native.ntt_dev(e, 0, key.log_n + key.log_ext, key.omega8, coset_shift=COSET_SHIFT)
        key.coset[name] = e
    # the eight commitments as one pipelined launch group (SURVEY 8 f3)
    for name, pt in zip(CIRCUIT_POLYS, _commit_many(key, [(key.coeffs[name], 0, n) for name in CIRCUIT_POLYS])):
        key.comm[name] = pt
    key.x = native.scalars_alloc(key.N8)
    key.l1f = native.scalars_alloc(key.N8)
    key.zh8 = native.scalars_alloc(key.ext)
    native.plonk_coset_setup_dev(n, key.ext, COSET_SHIFT, key.omega8, key.x, key.l1f, key.zh8)
    return key


def public_input_values(values, ell, what):
    """The l public inputs as ints: ValueError unless there are exactly l of them, each an integer in [0, r) (not
    reduced: x and x + r would be one statement).  Decimal strings, as the reference's fixtures hold them, are read."""
    values = list(values) if values is not None else []
    if len(values) != ell:
        raise ValueError("%s: %d public inputs given, the circuit has %d" % (what, len(values), ell))
    out = []
    for x in values:
        if isinstance(x, (bool, float)):
            raise ValueError("%s: public input %r is not an integer" % (what, x))
        try:
            v = int(x)
        except (TypeError, ValueError):
            raise ValueError("%s: public input %r is not an integer" % (what, x)) from None
        if not 0 <= v < R:
            raise ValueError("%s: public input %d is outside [0, r)" % (what, v))
        out.append(v)
    return out


_R_WORDS = np.array([(R >> (64 * (3 - k))) & (2 ** 64 - 1) for k in range(4)], dtype=np.uint64)


def _absorb_public_inputs(trs, raw, ell, j0):
    """tr.append_scalar(b"public_input", x_j,i) for i < ell into trs[j], from raw = the inputs of every proof back to
    back as 32-byte little-endian values, checked to be below r (a device handle is not reduced on load).  j0: the
    batch index of trs[0], for the error."""
    be = np.frombuffer(raw, dtype=np.uint8).reshape(len(trs), ell, 32)[:, :, ::-1]
    words = np.ascontiguousarray(be).view(">u8").reshape(-1, 4).astype(np.uint64)
    lt, eq = np.zeros(len(words), dtype=bool), np.ones(len(words), dtype=bool)
    for k in range(4):
        lt |= eq & (words[:, k] < _R_WORDS[k])
        eq &= words[:, k] == _R_WORDS[k]
    if not lt.all():
        j, i = divmod(int(np.argmin(lt)), ell)
        raise ValueError("prove_batch: public input %d of proof %d is outside [0, r)" % (i, j0 + j))
    label = np.frombuffer(b"public_input", dtype=np.uint8)
    rec = np.empty((len(trs), ell, len(label) + 32), dtype=np.uint8)
    rec[:, :, :len(label)] = label
    rec[:, :, len(label):] = be
    for j, tr in enumerate(trs):
        tr.state += rec[j].tobytes()


def _blind(h, n, blinds):
    """p(x) += (b0 + b1 x + ...)(x^n - 1): subtract the b's at the bottom, add them at x^n."""
    k = len(blinds)
    up = native.scalars_load(native.fr_vec_bytes([b % R for b in blinds]), k)
    native.vec_op_dev(1, h, 0, h, 0, up, 0, k)
    native.vec_op_dev(0, h, n, h, n, up, 0, k)
    up.free()


def prove(key, a_vals, b_vals, c_vals, blinds=None, keep=False, public_inputs=None):
    """a_vals, b_vals, c_vals: device handles with the n wire values.  blinds: optional 9 scalars
    (round 1: 2 per wire polynomial, round 2: 3) to reproduce a golden proof; random otherwise.
    public_inputs: the key's num_public_inputs ints (ValueError otherwise).
    Returns a Proof whose fields are the reference's types."""
    n, log_n, w = key.n, key.log_n, key.omega
    N8 = key.N8
    ell = key.num_public_inputs
    pubs = public_input_values(public_inputs, ell, "prove")
    if blinds is None:
        blinds = [secrets.randbelow(R) for _ in range(9)]
    tr = Transcript()
    proof = Proof()
    for x in pubs:
        tr.append_scalar(b"public_input", x)
    # ---- round 1
    wires = {}
    for i, (name, vals) in enumerate((("a", a_vals), ("b", b_vals), ("c", c_vals))):
        h = _alloc_from(vals, n, n + 2)
        native.ntt_dev(h, 0, log_n, w, inverse=True)
        _blind(h, n, blinds[2 * i:2 * i + 2])
        wires[name] = h
    for name, pt in zip("abc", _commit_many(key, [(wires[k], 0, n + 2) for k in "abc"])):
        setattr(proof, name + "_comm", g1_from_ints(pt))
    for name in "abc":
        tr.append_point(name.encode() + b"_comm", getattr(proof, name + "_comm"))
    # ---- round 2
    beta, gamma = int(tr.challenge_scalar(b"beta")), int(tr.challenge_scalar(b"gamma"))
    z = native.scalars_alloc(n + 3)
    if n > 1:
        num, den = native.scalars_alloc(n), native.scalars_alloc(n)
        native.plonk_perm_terms_dev(a_vals, b_vals, c_vals, *key.sigma_evals, n, w, beta, gamma, num, den)
        native.batch_inverse_dev(den, 0, n)
        native.vec_op_dev(2, num, 0, num, 0, den, 0, n)
        native.scan_dev(0, z, 0, num, 0, n)               # z_0 = 1, z_{i+1} = z_i * num_i / den_i
        num.free()
        den.free()
    else:
        native.scalars_upload(z, 0, native.fe_bytes(1), 1)
    native.ntt_dev(z, 0, log_n, w, inverse=True)
    _blind(z, n, blinds[6:9])
    # the z commitment starts on the library's second stream; the four coset transforms of round 3 need a, b, c, z
    # but not alpha, so they run beside it and the challenge is drawn once the commitment is back
    _commit_begin(key, z, 0, n + 3)
    ext = []
    for h, length in ((wires["a"], n + 2), (wires["b"], n + 2), (wires["c"], n + 2), (z, n + 3)):
        e = _alloc_from(h, length, N8)
        native.scalars_convert(e, 0, length, True)
        native.ntt_dev(e, 0, log_n + key.log_ext, key.omega8, coset_shift=COSET_SHIFT)
        ext.append(e)
    proof.z_comm = g1_from_ints(_commit_end(key))
    tr.append_point(b"z_comm", proof.z_comm)
    # ---- round 3
    alpha = int(tr.challenge_scalar(b"alpha"))
    circuit = {k: key.coset[k] for k in CIRCUIT_POLYS}
    pub = None
    if ell:
        # PI on the coset, added into a copy of q_c's coset evaluations (Montgomery form is linear)
        pub = native.scalars_load(native.fr_vec_bytes(pubs), ell)
        pi = native.scalars_alloc(N8)
        native.plonk_pi_scatter_many_dev(pub, 0, ell, ell, n, 1, pi)
        native.ntt_dev(pi, 0, log_n, w, inverse=True)
        native.scalars_convert(pi, 0, n, True)
        native.ntt_dev(pi, 0, log_n + key.log_ext, key.omega8, coset_shift=COSET_SHIFT)
        circuit["q_c"] = _alloc_from(key.coset["q_c"], N8, N8)
        native.vec_op_dev(0, circuit["q_c"], 0, circuit["q_c"], 0, pi, 0, N8)
        pi.free()
    t = native.scalars_alloc(N8)
    native.plonk_quotient_dev(ext + [circuit[k] for k in CIRCUIT_POLYS], n, key.ext, key.x, key.l1f, key.zh8, beta,
                              gamma, alpha, t)
    for e in ext:
        e.free()
    if ell:
        circuit["q_c"].free()
    native.ntt_dev(t, 0, log_n + key.log_ext, key.omega8, inverse=True, coset_shift=COSET_SHIFT)
    native.scalars_convert(t, 0, N8, False)
    if not native.scalars_is_zero(t, 3 * n + 6, N8 - (3 * n + 6)):
        raise ValueError(
            "제약 다항식이 Z_H(x)로 나누어 떨어지지 않습니다. "
            "회로 또는 witness에 오류가 있습니다."
        )
    t_pts = _commit_many(key, [(t, 0, n), (t, n, n), (t, 2 * n, n + 6)])
    proof.t_lo_comm, proof.t_mid_comm, proof.t_hi_comm = (g1_from_ints(p) for p in t_pts)
    for part in ("t_lo", "t_mid", "t_hi"):
        tr.append_point(part.encode() + b"_comm", getattr(proof, part + "_comm"))
    # ---- round 4
    zeta = int(tr.challenge_scalar(b"zeta"))
    ev = native.fr_poly_eval_dev
    # the six openings in one batched set of Horner launches
    a_e, b_e, c_e, s1_e, s2_e, zw_e = native.fr_poly_eval_multi_dev(
        [(wires[k], 0, n + 2, zeta) for k in "abc"]
        + [(key.coeffs["s_sigma1"], 0, n, zeta), (key.coeffs["s_sigma2"], 0, n, zeta), (z, 0, n + 3, zeta * w % R)])
    for name, val in (("a_eval", a_e), ("b_eval", b_e), ("c_eval", c_e), ("s_sigma1_eval", s1_e),
                      ("s_sigma2_eval", s2_e), ("z_omega_eval", zw_e)):
        setattr(proof, name, FR(val))
        tr.append_scalar(name.encode(), val)
    # ---- round 5
    v = int(tr.challenge_scalar(b"v"))
    zh_zeta = (pow(zeta, n, R) - 1) % R
    l1_zeta = 1 if zeta == 1 else pow(n, -1, R) * zh_zeta % R * pow((zeta - 1) % R, -1, R) % R
    perm_z = alpha * (a_e + beta * zeta + gamma) % R * (b_e + beta * K1 * zeta + gamma) % R * (c_e + beta * K2 * zeta + gamma) % R
    ab = (a_e + beta * s1_e + gamma) * (b_e + beta * s2_e + gamma) % R
    perm_s3 = alpha * ab % R * beta % R * zw_e % R
    const = (-alpha * ab % R * zw_e % R * (c_e + gamma) - alpha * alpha % R * l1_zeta) % R   # pi(zeta) = 0
    if ell:
        const = (const + native.plonk_pi_eval_many_dev(pub, 0, ell, ell, n, w, [zeta])[0]) % R
        pub.free()
    # linearisation polynomial: seven scalar-times-polynomial terms in one pass
    r = native.scalars_alloc(n + 3)
    native.lincomb_dev(r, 0, n + 3,
                       [(k, key.coeffs[name], 0, n) for name, k in
                        (("q_m", a_e * b_e % R), ("q_l", a_e), ("q_r", b_e), ("q_o", c_e), ("q_c", 1),
                         ("s_sigma3", (-perm_s3) % R))]
                       + [((perm_z + alpha * alpha % R * l1_zeta) % R, z, 0, n + 3)])
    native.scalars_add_const(r, 0, 1, const)
    r_eval = ev(r, 0, n + 3, zeta)
    proof.r_eval = FR(r_eval)
    zeta_n = pow(zeta, n, R)
    P = native.scalars_alloc(n + 6)
    terms = [(1, t, 0, n), (zeta_n, t, n, n), (zeta_n * zeta_n % R, t, 2 * n, n + 6), (v, r, 0, n + 3)]
    vp = v
    for h, length in ((wires["a"], n + 2), (wires["b"], n + 2), (wires["c"], n + 2),
                      (key.coeffs["s_sigma1"], n), (key.coeffs["s_sigma2"], n)):
        vp = vp * v % R
        terms.append((vp, h, 0, length))
    native.lincomb_dev(P, 0, n + 6, terms)                # the batched opening polynomial in one pass
    W = native.scalars_alloc(n + 5)
    native.div_linear_dev(P, 0, n + 6, zeta, W, 0)
    Ww = native.scalars_alloc(n + 2)
    native.div_linear_dev(z, 0, n + 3, zeta * w % R, Ww, 0)
    w_pts = _commit_many(key, [(W, 0, n + 5), (Ww, 0, n + 2)])
    proof.W_zeta_comm, proof.W_zeta_omega_comm = (g1_from_ints(p) for p in w_pts)
    state = {"a": wires["a"], "b": wires["b"], "c": wires["c"], "z": z, "t": t, "r": r, "W": W, "Ww": Ww, "P": P,
             "challenges": {"beta": beta, "gamma": gamma, "alpha": alpha, "zeta": zeta, "v": v}}
    if keep:
        return proof, state
    for h in (wires["a"], wires["b"], wires["c"], z, t, r, W, Ww, P):
        h.free()
    return proof


# ------------------------------------------------------------------ many proofs of one circuit per pass
_NOT_DIVISIBLE = "제약 다항식이 Z_H(x)로 나누어 떨어지지 않습니다. 회로 또는 witness에 오류가 있습니다."
# the many-MSMs of one pass: (scalar vectors per proof, padded length - n) -- rounds 1, 2, 3 and 5
_PASS_MSMS = ((3, 2), (1, 3), (3, 6), (2, 5))
# the circuit coefficient vectors rounds 4 and 5 read, gathered per proof when a pass holds several circuits
_GATHERED = ("q_m", "q_l", "q_r", "q_o", "q_c", "s_sigma3", "s_sigma1", "s_sigma2")


def plan_chunk(key, count, free_bytes, multi=False):
    """Largest number of proofs per pass of prove_batch: within the 32-bit entry and 31-bit bucket numbering of the
    many-MSM (vectors * W * L < 2^32, vectors * buckets < 2^31 at the padded length L of each round's vectors), the
    32-bit batched coset transforms (4 * count * N8 < 2^32, 5 with public inputs), and half of `free_bytes` of device
    memory at the working set estimated below.  At least 1, at most count.  multi: a pass of prove_batch_circuits,
    whose proofs also hold their own copies of the 8 circuit coefficient vectors of rounds 4 and 5 (8n per proof)."""
    from ..groth16.device_prover import _many_msm_shape
    n, N = key.n, key.N8
    pi = 1 if key.num_public_inputs else 0             # one more coset block and one more n-block per proof
    limit = ((1 << 32) - 1) // ((4 + pi) * N)
    msm_ws = 0
    for vecs, pad in _PASS_MSMS:
        W, per = _many_msm_shape(key.srs_table, n + pad)
        limit = min(limit, ((1 << 32) - 1) // (vecs * W * (n + pad)), ((1 << 31) - 1) // (vecs * per))
        msm_ws = max(msm_ws, vecs * (8 * W * (n + pad) + per * (3 * 128 + 12)))   # entries; buckets and levels
    per_proof = msm_ws + 32 * ((9 + pi) * N + (20 + pi) * n + 64)  # coset blocks, transform scratch, per-round vectors
    if multi:
        per_proof += 32 * len(_GATHERED) * n
    limit = min(limit, (free_bytes // 2) // per_proof)
    return int(max(1, min(limit, count)))


def prove_batch(key, a_vals, b_vals, c_vals, count, blinds=None, chunk=None, public_inputs=None):
    """count proofs of the circuit of `key`, proof j from the wire values at offset j * n of a_vals, b_vals, c_vals
    and blinds[j] (9 scalars in the order of prove; fresh ones from `secrets` when blinds is None).  Proof j is
    bit-identical to prove(key, a_j, b_j, c_j, blinds=blinds[j]).  Per chunk of proofs every round is a fixed number of
    launches whatever the chunk size: batched transforms, per-proof challenge arrays, segmented scans and one many-MSM
    per commitment group.  The transcripts stay on the host, one per proof.  chunk=None picks the largest chunk
    plan_chunk allows; the result does not depend on it.  An unsatisfied witness raises the ValueError of prove,
    naming the first failing proof, before any round-3 commitment of its chunk.
    public_inputs: for a key with l = num_public_inputs > 0, a scalar handle of count * l values, proof j's at j * l
    (as witness.solve_batch returns them); proof j then equals prove(..., public_inputs=those l values)."""
    count = int(count)
    if key.ranks is not None:
        raise ValueError("prove_batch: a sharded key is not supported (batch over one GPU's SRS)")
    blinds = _batch_arguments("prove_batch", key, a_vals, b_vals, c_vals, count, blinds, chunk, public_inputs)
    if count == 0:
        return []
    step = min(int(chunk), count) if chunk is not None else plan_chunk(key, count, native.device_mem_info()[0])
    proofs = []
    for j0 in range(0, count, step):
        proofs.extend(_prove_chunk(key, a_vals, b_vals, c_vals, j0, min(step, count - j0), blinds, public_inputs))
    return proofs


def _batch_arguments(what, key, a_vals, b_vals, c_vals, count, blinds, chunk, public_inputs):
    """The checks of prove_batch's arguments before any device call (ValueError); returns the blinds as count rows of 9
    reduced ints, fresh from `secrets` when blinds is None."""
    n, ell = key.n, key.num_public_inputs
    if ell and (public_inputs is None or public_inputs.n < count * ell):
        raise ValueError("%s: public_inputs holds %s values, needs %d"
                         % (what, None if public_inputs is None else public_inputs.n, count * ell))
    if not ell and public_inputs is not None:
        raise ValueError("%s: the key has no public inputs (preprocess with num_public_inputs)" % what)
    if chunk is not None and int(chunk) <= 0:
        raise ValueError("%s: chunk must be positive" % what)
    if count < 0:
        raise ValueError("%s: count must be >= 0" % what)
    for name, h in (("a_vals", a_vals), ("b_vals", b_vals), ("c_vals", c_vals)):
        if h is None or h.n < count * n:
            raise ValueError("%s: %s holds %s values, needs %d" % (what, name, None if h is None else h.n, count * n))
    if blinds is not None:
        blinds = [list(b) for b in blinds]
        if len(blinds) != count or any(len(b) != 9 for b in blinds):
            raise ValueError("%s: blinds must be %d lists of 9 scalars" % (what, count))
    if blinds is None:
        blinds = [[secrets.randbelow(R) for _ in range(9)] for _ in range(count)]
    return [[int(b) % R for b in bl] for bl in blinds]


def _same_table(t, u):
    return t is u or (getattr(t, "handle", None) is not None and getattr(t, "handle", None) == getattr(u, "handle", None))


def prove_batch_circuits(keys, circuits, a_vals, b_vals, c_vals, blinds=None, chunk=None, public_inputs=None):
    """count = len(circuits) proofs of several circuits of one size in the passes of prove_batch: proof j proves the
    circuit of keys[circuits[j]] from the wire values at offset j * n of a_vals, b_vals, c_vals, with blinds[j] and
    (for keys with l public inputs) the l values at j * l of public_inputs, as in prove_batch.  Proof j is
    bit-identical to prove(keys[circuits[j]], a_j, b_j, c_j, blinds=blinds[j], public_inputs=...); a key may serve
    any number of proofs, none included.  PLONK's SRS is universal, so every commitment group of a pass stays one
    many-MSM over the one table; the circuit-dependent work reads each proof's circuit through a per-proof index (the
    permutation terms and the quotient) or per-proof copies of its 8 coefficient vectors (rounds 4 and 5).
    ValueError before any device call unless the keys are non-empty, of one n, one SRS table, one number of public
    inputs and none of them sharded, every index is in [0, len(keys)), and the other arguments pass prove_batch's
    checks.  An unsatisfied witness raises prove_batch's ValueError naming the first failing proof."""
    what = "prove_batch_circuits"
    keys = list(keys)
    if not keys:
        raise ValueError("%s: no keys" % what)
    key = keys[0]
    for k in keys:
        if k.ranks is not None:
            raise ValueError("%s: a sharded key is not supported (batch over one GPU's SRS)" % what)
        if k.n != key.n:
            raise ValueError("%s: the keys differ in n (%d and %d); group circuits by size" % (what, key.n, k.n))
        if not _same_table(k.srs_table, key.srs_table):
            raise ValueError("%s: the keys do not share one SRS table" % what)
        if k.num_public_inputs != key.num_public_inputs:
            raise ValueError("%s: the keys differ in num_public_inputs (%d and %d)"
                             % (what, key.num_public_inputs, k.num_public_inputs))
    circuits = list(circuits)
    for j, c in enumerate(circuits):
        if isinstance(c, bool) or not isinstance(c, numbers.Integral) or not 0 <= c < len(keys):
            raise ValueError("%s: circuit index %r of proof %d is outside [0, %d)" % (what, c, j, len(keys)))
    circuits = [int(c) for c in circuits]
    count = len(circuits)
    blinds = _batch_arguments(what, key, a_vals, b_vals, c_vals, count, blinds, chunk, public_inputs)
    if count == 0:
        return []
    step = min(int(chunk), count) if chunk is not None else plan_chunk(key, count, native.device_mem_info()[0], multi=True)
    proofs = []
    for j0 in range(0, count, step):
        cnt = min(step, count - j0)
        proofs.extend(_prove_chunk(key, a_vals, b_vals, c_vals, j0, cnt, blinds, public_inputs,
                                   (keys, circuits[j0:j0 + cnt])))
    return proofs


def _prove_chunk(key, a_vals, b_vals, c_vals, j0, cnt, blinds, pub, multi=None):
    """Proofs j0 .. j0 + cnt - 1 in one pass.  multi = None: every proof is of `key`'s circuit.  multi = (keys, circ):
    proof j0 + i is of keys[circ[i]] (all of key's n, SRS table and public-input count); the circuit data is then read
    through per-proof indices (rounds 2 and 3) and per-proof gathered coefficient blocks (rounds 4 and 5)."""
    n, log_n, w, N = key.n, key.log_n, key.omega, key.N8
    ell = key.num_public_inputs
    nb = 4 if ell else 3                                    # transform blocks per proof in round 1; + 1 in round 3
    bl = blinds[j0:j0 + cnt]
    trs = [Transcript() for _ in range(cnt)]
    if ell:
        _absorb_public_inputs(trs, native.scalars_download(pub, j0 * ell, cnt * ell), ell, j0)
    proofs = [Proof() for _ in range(cnt)]
    tmp = []

    def alloc(m):
        h = native.scalars_alloc(m)
        tmp.append(h)
        return h

    try:
        # ---- round 1: 3 cnt inverse transforms, blinding at stride n + 2 (vector i * cnt + j: wire i of proof j);
        # with public inputs cnt more for PI_j, from their evaluations on H at 3 cnt n
        ev = alloc(nb * cnt * n)
        for i, vals in enumerate((a_vals, b_vals, c_vals)):
            native.scalars_copy(ev, i * cnt * n, vals, j0 * n, cnt * n)
        if ell:
            native.plonk_pi_scatter_many_dev(pub, j0 * ell, ell, ell, n, cnt, ev, 3 * cnt * n)
        native.ntt_many_dev(ev, 0, log_n, nb * cnt, w, inverse=True)
        wires = alloc(3 * cnt * (n + 2))
        native.plonk_blind_many_dev(ev, 0, n, n, 3 * cnt, [b[2 * i:2 * i + 2] for i in range(3) for b in bl], wires, 0, n + 2)
        pts = native.msm_dev_many(key.srs_table, 0, n + 2, 3 * cnt, wires)
        for j, (prf, tr) in enumerate(zip(proofs, trs)):
            for i, name in enumerate("abc"):
                setattr(prf, name + "_comm", g1_from_ints(pts[i * cnt + j]))
                tr.append_point(name.encode() + b"_comm", getattr(prf, name + "_comm"))
        # ---- round 2: grand products with per-proof beta, gamma; segmented scan; blinding at stride n + 3
        betas = [int(tr.challenge_scalar(b"beta")) for tr in trs]
        gammas = [int(tr.challenge_scalar(b"gamma")) for tr in trs]
        zc = alloc(cnt * n)
        if n > 1:
            num, den = alloc(cnt * n), alloc(cnt * n)
            if multi:
                native.plonk_perm_terms_multi_dev(a_vals, b_vals, c_vals, j0 * n, [k.sigma_evals for k in multi[0]], multi[1],
                                                  n, w, betas, gammas, num, den)
            else:
                native.plonk_perm_terms_many_dev(a_vals, b_vals, c_vals, j0 * n, *key.sigma_evals, n, w, betas, gammas, num,
                                                 den)
            native.batch_inverse_dev(den, 0, cnt * n)
            native.vec_op_dev(2, num, 0, num, 0, den, 0, cnt * n)
            native.scan_many_dev(0, zc, 0, num, 0, n, cnt)  # z_j,0 = 1 in every proof
        else:                                               # n = 1: z = [1], as in prove
            native.scalars_upload(zc, 0, native.fr_vec_bytes([1] * cnt), cnt)
        native.ntt_many_dev(zc, 0, log_n, cnt, w, inverse=True)
        z = alloc(cnt * (n + 3))
        native.plonk_blind_many_dev(zc, 0, n, n, cnt, [b[6:9] for b in bl], z, 0, n + 3)
        for prf, tr, pt in zip(proofs, trs, native.msm_dev_many(key.srs_table, 0, n + 3, cnt, z)):
            prf.z_comm = g1_from_ints(pt)
            tr.append_point(b"z_comm", prf.z_comm)
        # ---- round 3: 4 cnt coset transforms, the quotient with per-proof challenges, cnt inverse transforms
        alphas = [int(tr.challenge_scalar(b"alpha")) for tr in trs]
        ext = alloc((nb + 1) * cnt * N)
        if ell:
            native.plonk_coset_inputs_pi_many_dev(wires, z, ev, 3 * cnt * n, n, cnt, key.log_n + key.log_ext, ext)
        else:
            native.plonk_coset_inputs_many_dev(wires, z, n, cnt, key.log_n + key.log_ext, ext)
        native.ntt_many_dev(ext, 0, log_n + key.log_ext, (nb + 1) * cnt, key.omega8, coset_shift=COSET_SHIFT)
        t = alloc(cnt * N)
        if multi:
            quotient = native.plonk_quotient_pi_multi_dev if ell else native.plonk_quotient_multi_dev
            quotient(ext, [[k.coset[p] for p in CIRCUIT_POLYS] for k in multi[0]], multi[1], n, key.ext, key.x, key.l1f,
                     key.zh8, betas, gammas, alphas, t)
        else:
            quotient = native.plonk_quotient_pi_many_dev if ell else native.plonk_quotient_many_dev
            quotient(ext, [key.coset[k] for k in CIRCUIT_POLYS], n, key.ext, key.x, key.l1f, key.zh8, betas, gammas, alphas, t)
        native.ntt_many_dev(t, 0, log_n + key.log_ext, cnt, key.omega8, inverse=True, coset_shift=COSET_SHIFT)
        bad = native.plonk_divisible_many_dev(t, n, key.ext, cnt)
        if bad is not None:
            raise ValueError(_NOT_DIVISIBLE + " (proof %d of the batch)" % (j0 + bad))
        ts = alloc(3 * cnt * (n + 6))                       # t_lo | t_mid | t_hi, vector part * cnt + j
        native.plonk_split_t_many_dev(t, n, key.ext, cnt, ts)
        pts = native.msm_dev_many(key.srs_table, 0, n + 6, 3 * cnt, ts)
        for j, (prf, tr) in enumerate(zip(proofs, trs)):
            for i, part in enumerate(("t_lo", "t_mid", "t_hi")):
                setattr(prf, part + "_comm", g1_from_ints(pts[i * cnt + j]))
                tr.append_point(part.encode() + b"_comm", getattr(prf, part + "_comm"))
        # ---- round 4: 6 cnt evaluations in one batched set of Horner launches
        zetas = [int(tr.challenge_scalar(b"zeta")) for tr in trs]
        if multi:                                           # the circuit coefficients of rounds 4 and 5, per proof
            gc = alloc(len(_GATHERED) * cnt * n)
            native.fr_gather_many_dev([[k.coeffs[p] for p in _GATHERED] for k in multi[0]], multi[1], n, gc)
            coef = lambda name: (gc, _GATHERED.index(name) * cnt * n, n, n)
        else:
            coef = lambda name: (key.coeffs[name], 0, 0, n)
        zws = [zeta * w % R for zeta in zetas]
        wl = cnt * (n + 2)
        evals = native.fr_poly_eval_many_dev(
            [(wires, 0, n + 2, n + 2, 0), (wires, wl, n + 2, n + 2, 0), (wires, 2 * wl, n + 2, n + 2, 0),
             coef("s_sigma1") + (0,), coef("s_sigma2") + (0,), (z, 0, n + 3, n + 3, 1)],
            cnt, [zetas, zws])
        names = ("a_eval", "b_eval", "c_eval", "s_sigma1_eval", "s_sigma2_eval", "z_omega_eval")
        for j, (prf, tr) in enumerate(zip(proofs, trs)):
            for g, name in enumerate(names):
                setattr(prf, name, FR(evals[g][j]))
                tr.append_scalar(name.encode(), evals[g][j])
        # ---- round 5: linearisation and opening polynomials as batched lincombs, segmented divisions by (x - zeta)
        vs = [int(tr.challenge_scalar(b"v")) for tr in trs]
        pis = native.plonk_pi_eval_many_dev(pub, j0 * ell, ell, ell, n, w, zetas) if ell else [0] * cnt
        r_rows, p_rows = [], []
        for j in range(cnt):
            beta, gamma, alpha, zeta, v = betas[j], gammas[j], alphas[j], zetas[j], vs[j]
            a_e, b_e, c_e, s1_e, s2_e, zw_e = (evals[g][j] for g in range(6))
            zh_zeta = (pow(zeta, n, R) - 1) % R
            l1_zeta = 1 if zeta == 1 else pow(n, -1, R) * zh_zeta % R * pow((zeta - 1) % R, -1, R) % R
            perm_z = alpha * (a_e + beta * zeta + gamma) % R * (b_e + beta * K1 * zeta + gamma) % R * (c_e + beta * K2 * zeta + gamma) % R
            ab = (a_e + beta * s1_e + gamma) * (b_e + beta * s2_e + gamma) % R
            perm_s3 = alpha * ab % R * beta % R * zw_e % R
            const = (-alpha * ab % R * zw_e % R * (c_e + gamma) - alpha * alpha % R * l1_zeta + pis[j]) % R
            r_rows.append([a_e * b_e % R, a_e, b_e, c_e, 1, (-perm_s3) % R, (perm_z + alpha * alpha % R * l1_zeta) % R, const])
            zeta_n = pow(zeta, n, R)
            p_rows.append([1, zeta_n, zeta_n * zeta_n % R, v] + [pow(v, e, R) for e in range(2, 7)] + [0])
        r = alloc(cnt * (n + 3))
        native.lincomb_many_dev(r, 0, n + 3, n + 3, cnt,
                                [coef(k) for k in ("q_m", "q_l", "q_r", "q_o", "q_c", "s_sigma3")]
                                + [(z, 0, n + 3, n + 3)], r_rows)
        r_evals = native.fr_poly_eval_many_dev([(r, 0, n + 3, n + 3, 0)], cnt, [zetas])[0]
        tl = cnt * (n + 6)
        P = alloc(cnt * (n + 6))
        native.lincomb_many_dev(P, 0, n + 6, n + 6, cnt,
                                [(ts, 0, n + 6, n), (ts, tl, n + 6, n), (ts, 2 * tl, n + 6, n + 6), (r, 0, n + 3, n + 3),
                                 (wires, 0, n + 2, n + 2), (wires, wl, n + 2, n + 2), (wires, 2 * wl, n + 2, n + 2),
                                 coef("s_sigma1"), coef("s_sigma2")], p_rows)
        # W_j (n + 5) and Ww_j (n + 2, zero-padded to n + 5: a zero scalar adds nothing) in one many-MSM
        Wb = alloc(2 * cnt * (n + 5))
        native.div_linear_many_dev(P, 0, n + 6, n + 6, zetas, Wb, 0, n + 5)
        native.div_linear_many_dev(z, 0, n + 3, n + 3, zws, Wb, cnt * (n + 5), n + 5)
        pts = native.msm_dev_many(key.srs_table, 0, n + 5, 2 * cnt, Wb)
        for j, prf in enumerate(proofs):
            prf.r_eval = FR(r_evals[j])
            prf.W_zeta_comm, prf.W_zeta_omega_comm = g1_from_ints(pts[j]), g1_from_ints(pts[cnt + j])
        return proofs
    finally:
        for h in tmp:
            h.free()
