"""Drop-in for /root/reference/zkp/groth16/verifying.py (SURVEY.md 8f-4: verifier-side group work).

The public-wire combination sum_i r_i * sigma1_3[i] (:34-37) is one GPU MSM; the four pairings and the
GT product of `verify` come from py_ecc -- where py_ecc is not installed a caller passes `pairing=`
(zkp.pairing.pairing runs them on the GPU).

`verify_batch` checks k proofs of one circuit at once: a random linear combination turns the k equations into
one product of k + 3 pairings, decided by a single device call (zkp.pairing.pairing_check)."""
from ... import native
from ..pairing import batch_weights, pairing_check
from ...compat import FQ, FR, G1, G2, HAVE_PY_ECC, curve_order, g1_from_ints  # noqa: F401

g1 = G1
g2 = G2


def _pairing_fn(pairing):
    if pairing is not None:
        return pairing
    if HAVE_PY_ECC:  # pragma: no cover
        from py_ecc import bn128
        return bn128.pairing
    raise NotImplementedError("pairings are outside the GPU hot path; install py_ecc or pass pairing=")


def _public_term(sigma1_3, rx_pub):
    pts = [sigma1_3[i] for i, _ in rx_pub]
    sc = [int(ri) % curve_order for _, ri in rx_pub]
    if not pts:
        return None
    return g1_from_ints(native.g1_msm(native.g1_vec_bytes(pts), native.fr_vec_bytes(sc), len(pts)))


def lhs(prf_A, prf_B, pairing=None):
    return _pairing_fn(pairing)(prf_B, prf_A)


def rhs(prf_C, sigma1_1, sigma1_3, sigma2_1, rx_pub, pairing=None):
    e = _pairing_fn(pairing)
    return (e(sigma2_1[0], sigma1_1[0]) * e(sigma2_1[1], _public_term(sigma1_3, rx_pub))) * e(sigma2_1[2], prf_C)


def verify(prf_A, prf_B, prf_C, sigma1_1, sigma1_3, sigma2_1, rx_pub, pairing=None):
    """e(A, B) == e(alpha, beta) * e(sum r_i sigma1_3[i], gamma) * e(C, delta)   (reference :29-40);
    rx_pub = [(index_i, r_i), ...]."""
    return lhs(prf_A, prf_B, pairing) == rhs(prf_C, sigma1_1, sigma1_3, sigma2_1, rx_pub, pairing)


def verify_batch(proofs, sigma1_1, sigma1_3, sigma2_1, rx_pubs, rng=None):
    """True iff every proof j in `proofs` = [(A_j, B_j, C_j)] satisfies `verify` with public input rx_pubs[j]
    (a list of (index, r_i) as for `verify`), up to a 2^-128 chance of accepting a bad batch.  With random
    non-zero 128-bit weights rho_j (from `secrets`, or from rng.getrandbits for reproducible runs) it checks

        prod_j e(rho_j A_j, B_j) * e(-(sum rho_j) alpha, beta) * e(-sum_j rho_j P_j, gamma) * e(-sum_j rho_j C_j, delta) == 1

    (alpha = sigma1_1[0], (beta, gamma, delta) = sigma2_1[0..2], P_j = proof j's public-wire term): one GPU MSM
    over sigma1_3 with the weights folded into the per-index scalars, one over the C_j, and one pairing check
    with k + 3 pairs.  The B_j come from provers, so the check also tests that each lies in G2."""
    proofs = list(proofs)
    rx_pubs = list(rx_pubs)
    k = len(proofs)
    if len(rx_pubs) != k:
        raise ValueError("verify_batch: one public input list per proof")
    if k == 0:
        return True
    rho = batch_weights(k, rng)
    pub = {}
    for w, rx_pub in zip(rho, rx_pubs):
        for i, ri in rx_pub:
            pub[i] = (pub.get(i, 0) + w * int(ri)) % curve_order
    idx = sorted(pub)
    P = _public_term(sigma1_3, [(i, pub[i]) for i in idx])
    C = g1_from_ints(native.g1_msm(native.g1_vec_bytes([c for _, _, c in proofs]), native.fr_vec_bytes(rho), k))
    pairs = [(b, a) for a, b, _ in proofs] + [(sigma2_1[0], sigma1_1[0]), (sigma2_1[1], P), (sigma2_1[2], C)]
    minus_one = curve_order - 1
    scalars = rho + [(-sum(rho)) % curve_order, minus_one, minus_one]
    return pairing_check(pairs, scalars, g2_subgroup_check=True)
