"""Drop-in for /root/reference/zkp/plonk/verifier.py:42-208 (SURVEY.md 8f-4).

The reference rebuilds the transcript, then spends ~18 scalar multiplications forming the two G1
points of the final pairing check.  Here the same scalars are computed on the host and the two points
are two GPU MSMs (2 and 18 terms):

    A = W_zeta + u W_zeta_omega
    B = zeta W_zeta + u zeta omega W_zeta_omega + F + u [z] - E
    F = [t_lo] + zeta^n [t_mid] + zeta^2n [t_hi] + v D + v r0 G1 + v^2 [a] + v^3 [b] + v^4 [c] + v^5 [s1] + v^6 [s2]
    D = (a b)[q_m] + a [q_l] + b [q_r] + c [q_o] + [q_c] + (perm_z + alpha^2 L1) [z] - perm_s3 [s3]

and the check is e(A, [tau]_2) == e(B, [1]_2): the two pairings need py_ecc (or a `pairing=` callable;
zkp.pairing.pairing runs them on the GPU).

`verify_batch` checks k proofs against one SRS with e(sum rho_j A_j, [tau]_2) e(-sum rho_j B_j, [1]_2) == 1:
the same two MSMs (over all proofs' terms at once) and two pairings for any k.

By default both keep the reference's semantics: `public_inputs` is not read and PI(zeta) = 0.  With
bind_public_inputs=True they check the protocol of device_prover's public inputs: the transcript absorbs
append_scalar(b"public_input", x_i) for every input before the first challenge, and r0 gains PI(zeta), evaluated on
the GPU (one zkp_plonk_pi_eval_many_dev call for a whole batch).
"""
from ... import native
from ..pairing import batch_weights, pairing_check
from ...compat import HAVE_PY_ECC, g1_from_ints
from .field import FR, G1, CURVE_ORDER
from .transcript import Transcript
from .permutation import K1, K2
from .utils import vanishing_poly_eval, lagrange_basis_eval


def _msm(terms):
    pts = [p for p, _ in terms]
    sc = [int(s) % CURVE_ORDER for _, s in terms]
    return g1_from_ints(native.g1_msm(native.g1_vec_bytes(pts), native.fr_vec_bytes(sc), len(pts)))


def _public_inputs(public_inputs, pp, bind):
    """The inputs to bind as ints ([] when not binding); ValueError before any device call for a wrong count or a
    value that is not an integer in [0, r)."""
    if not bind:
        return []
    from .device_prover import public_input_values
    return public_input_values(public_inputs, int(getattr(pp, "num_public_inputs", 0)), "verify")


def _pi_evals(rows):
    """[PI_j(zeta_j)] for rows = [(inputs, pp, zeta)], one device call per (n, omega, count of inputs) group."""
    out = [FR(0)] * len(rows)
    groups = {}
    for j, (pubs, pp, zeta) in enumerate(rows):
        if pubs:
            groups.setdefault((int(pp.n), int(pp.omega), len(pubs)), []).append(j)
    for (n, omega, ell), idx in groups.items():
        h = native.scalars_load(native.fr_vec_bytes([x for j in idx for x in rows[j][0]]), len(idx) * ell)
        try:
            vals = native.plonk_pi_eval_many_dev(h, 0, ell, ell, n, omega, [int(rows[j][2]) for j in idx])
        finally:
            h.free()
        for j, v in zip(idx, vals):
            out[j] = FR(v)
    return out


def _challenges(proof, pubs):
    t = Transcript()
    for x in pubs:
        t.append_scalar(b"public_input", x)
    for name in ("a_comm", "b_comm", "c_comm"):
        t.append_point(name.encode(), getattr(proof, name))
    beta = t.challenge_scalar(b"beta")
    gamma = t.challenge_scalar(b"gamma")
    t.append_point(b"z_comm", proof.z_comm)
    alpha = t.challenge_scalar(b"alpha")
    for name in ("t_lo_comm", "t_mid_comm", "t_hi_comm"):
        t.append_point(name.encode(), getattr(proof, name))
    zeta = t.challenge_scalar(b"zeta")
    for name in ("a_eval", "b_eval", "c_eval", "s_sigma1_eval", "s_sigma2_eval", "z_omega_eval"):
        t.append_scalar(name.encode(), getattr(proof, name))
    v = t.challenge_scalar(b"v")
    u = t.challenge_scalar(b"u")
    return beta, gamma, alpha, zeta, v, u


def _pairing_terms(proof, preprocessed, challenges, pi_zeta):
    """(point, scalar) terms of the two G1 points A and B of the final check e(A, [tau]_2) == e(B, [1]_2)."""
    pp = preprocessed
    n, omega = pp.n, pp.omega
    beta, gamma, alpha, zeta, v, u = challenges
    a, b, c = proof.a_eval, proof.b_eval, proof.c_eval
    s1, s2, zw = proof.s_sigma1_eval, proof.s_sigma2_eval, proof.z_omega_eval
    zh = vanishing_poly_eval(n, zeta)
    l1 = lagrange_basis_eval(0, n, omega, zeta)
    perm_z = alpha * (a + beta * zeta + gamma) * (b + beta * K1 * zeta + gamma) * (c + beta * K2 * zeta + gamma)
    ab = (a + beta * s1 + gamma) * (b + beta * s2 + gamma)
    perm_s3 = alpha * ab * beta * zw
    r0 = pi_zeta - alpha * ab * zw * (c + gamma) - alpha * alpha * l1   # PI(zeta) = 0 in the reference (:99)
    zeta_n = zeta ** n
    e_scalar = proof.r_eval / zh + v * proof.r_eval
    vp = v
    for val in (a, b, c, s1, s2):
        vp = vp * v
        e_scalar = e_scalar + vp * val
    e_scalar = e_scalar + u * zw

    A = [(proof.W_zeta_comm, FR(1)), (proof.W_zeta_omega_comm, u)]
    v2 = v * v
    v4 = v2 * v2
    B = [
        (proof.W_zeta_comm, zeta), (proof.W_zeta_omega_comm, u * zeta * omega),
        (proof.t_lo_comm, FR(1)), (proof.t_mid_comm, zeta_n), (proof.t_hi_comm, zeta_n * zeta_n),
        (pp.q_m_comm, v * a * b), (pp.q_l_comm, v * a), (pp.q_r_comm, v * b), (pp.q_o_comm, v * c), (pp.q_c_comm, v),
        (proof.z_comm, v * (perm_z + alpha * alpha * l1) + u), (pp.s_sigma3_comm, FR(0) - v * perm_s3),
        (G1, v * r0 - e_scalar),
        (proof.a_comm, v2), (proof.b_comm, v2 * v), (proof.c_comm, v4),
        (pp.s_sigma1_comm, v4 * v), (pp.s_sigma2_comm, v4 * v2),
    ]
    return A, B


def verify(proof, public_inputs, preprocessed, srs, pairing=None, *, bind_public_inputs=False):
    """True iff the proof passes the reference's check; with bind_public_inputs=True, also bound to public_inputs
    (exactly preprocessed.num_public_inputs integers in [0, r), ValueError otherwise)."""
    pubs = _public_inputs(public_inputs, preprocessed, bind_public_inputs)
    ch = _challenges(proof, pubs)
    pi_zeta = _pi_evals([(pubs, preprocessed, ch[3])])[0]
    a_terms, b_terms = _pairing_terms(proof, preprocessed, ch, pi_zeta)
    A = _msm(a_terms)
    B = _msm(b_terms)
    if pairing is None:
        if not HAVE_PY_ECC:
            raise NotImplementedError("pairings are outside the GPU hot path; install py_ecc or pass pairing=")
        from py_ecc import bn128  # pragma: no cover
        pairing = bn128.pairing   # pragma: no cover
    return pairing(srs.g2_powers[1], A) == pairing(srs.g2_powers[0], B)


def verify_batch(items, srs, rng=None, *, bind_public_inputs=False):
    """True iff every (proof, public_inputs, preprocessed) in `items` passes `verify` against the one `srs`, up
    to a 2^-128 chance of accepting a bad batch: with random non-zero 128-bit weights rho_j (from `secrets`, or
    from rng.getrandbits for reproducible runs) it checks e(sum rho_j A_j, [tau]_2) e(-sum rho_j B_j, [1]_2) == 1,
    i.e. two GPU MSMs over the terms of all proofs and one pairing check with two pairs.  bind_public_inputs: as in
    verify; every input list is checked before any device call, and all PI_j(zeta_j) come from one device call."""
    items = list(items)
    if not items:
        return True
    pubs = [_public_inputs(public_inputs, pp, bind_public_inputs) for _, public_inputs, pp in items]
    chs = [_challenges(proof, p) for (proof, _, _), p in zip(items, pubs)]
    pis = _pi_evals([(p, pp, ch[3]) for p, (_, _, pp), ch in zip(pubs, items, chs)])
    a_all, b_all = [], []
    for rho, (proof, _, pp), ch, pi_zeta in zip(batch_weights(len(items), rng), items, chs, pis):
        a_terms, b_terms = _pairing_terms(proof, pp, ch, pi_zeta)
        a_all += [(p, int(s) * rho) for p, s in a_terms]
        b_all += [(p, int(s) * rho) for p, s in b_terms]
    return pairing_check([(srs.g2_powers[1], _msm(a_all)), (srs.g2_powers[0], _msm(b_all))], [1, CURVE_ORDER - 1])
