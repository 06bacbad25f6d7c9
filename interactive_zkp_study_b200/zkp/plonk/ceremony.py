"""Powers-of-tau contributions for the PLONK SRS, and a check for any SRS a prover is handed.

``SRS.generate(max_degree, seed)`` (srs.py) derives tau from a seed, so whoever knows the seed can forge KZG
openings.  A powers-of-tau ceremony removes that trust: each participant multiplies the SRS by a secret s
(tau <- s tau), publishes a proof of the update and throws s away; the result is sound if any one participant
did.

    nxt, proof = contribute(srs)                 # [tau^i]_1 -> s^i [tau^i]_1 on the GPU, [tau]_2 -> s [tau]_2
    verify_contribution(srs, nxt, proof)         # srs already verified; a chain is a loop over this
    verify_srs(srs)                              # any SRS: shape, membership, consistent powers

The device work is one per-point scalar multiplication of the cached table (zkp_g1_table_scale), one table
validation (zkp_g1/g2_table_validate), two MSMs on the cached table and one pairing check.
"""
import hashlib
import secrets

from ... import native, tables
from ...compat import g1_from_ints, g2_from_ints
from ..pairing import batch_weights, pairing_check
from .field import G1, G2, CURVE_ORDER
from .srs import SRS

DOMAIN = b"zkp-b200 powers-of-tau v1"


class Contribution:
    """Public record of one update tau -> s tau: s_g1 = [s]_1 and a Schnorr proof of knowledge of s,
    R = [k]_1 and z = k + c s mod r with c = challenge(prev, s_g1, R)."""

    def __init__(self, s_g1, R, z):
        self.s_g1 = s_g1
        self.R = R
        self.z = int(z)


def challenge(prev, s_g1, R):
    """Fiat-Shamir challenge of a contribution on top of `prev`: SHA-256 over the domain tag and the ABI
    encodings of prev's [tau]_1, [tau]_2, s_g1 and R, read big-endian, mod r."""
    h = hashlib.sha256(DOMAIN + native.g1_bytes(prev.g1_powers[1]) + native.g2_bytes(prev.g2_powers[1]) +
                       native.g1_bytes(s_g1) + native.g1_bytes(R)).digest()
    return int.from_bytes(h, "big") % CURVE_ORDER


def _check_shape(srs):
    if srs.max_degree < 1:
        raise ValueError("SRS: max_degree must be at least 1")
    if len(srs.g1_powers) != srs.max_degree + 1:
        raise ValueError("SRS: %d G1 powers for max_degree %d (expected max_degree + 1)"
                         % (len(srs.g1_powers), srs.max_degree))
    if len(srs.g2_powers) != 2:
        raise ValueError("SRS: %d G2 powers (expected 2)" % len(srs.g2_powers))


def _on_g1(p):
    """Host check of one G1 point (cofactor 1: on the curve is in G1); infinity is not accepted here."""
    if p is None:
        return False
    x, y = int(p[0]), int(p[1])
    P = native.P_MOD
    return 0 <= x < P and 0 <= y < P and (y * y - x * x * x - 3) % P == 0


def _powers_check(srs, rho):
    """Steps 1-4 of verify_srs; then the pairs and scalars of step 5, or None when a step already failed."""
    _check_shape(srs)
    g1, g2 = srs.g1_powers, srs.g2_powers
    if native.g1_bytes(g1[0]) != native.g1_bytes(G1) or native.g2_bytes(g2[0]) != native.g2_bytes(G2):
        return None
    if g1[1] is None or g2[1] is None:
        return None
    n, d = len(g1), srs.max_degree
    table = tables.g1_table(g1)
    if native.g1_table_validate(table, 0, n) is not None:
        return None
    t2 = native.g2_table_load(native.g2_vec_bytes(g2), 2)
    try:
        if native.g2_table_validate(t2, 0, 2, subgroup_check=True) is not None:
            return None
    finally:
        t2.free()
    pw = native.scalars_alloc(d)
    native.scalars_fill_powers(pw, 0, d, 1, rho)
    A = native.g1_msm_dev(table, 0, pw, 0, d)    # sum_{i<d} rho^i [tau^i]_1
    B = native.g1_msm_dev(table, 1, pw, 0, d)    # sum_{i<d} rho^i [tau^(i+1)]_1
    pw.free()
    # e([tau]_2, A) = e([1]_2, B)
    return [(g2[1], g1_from_ints(A)), (g2[0], g1_from_ints(B))], [1, CURVE_ORDER - 1]


def verify_srs(srs, rng=None):
    """True iff `srs` is a consistent powers-of-tau SRS: [tau^i]_1, i <= max_degree, and [1]_2, [tau]_2 for one
    tau != 0.  It checks, in order:
      1. len(g1_powers) == max_degree + 1 and len(g2_powers) == 2 (otherwise ValueError, as for max_degree < 1);
      2. g1_powers[0] == G1 and g2_powers[0] == G2;
      3. g1_powers[1] and g2_powers[1] are not infinity (tau = 0 would pass step 5);
      4. every G1 point is on the curve and both G2 points are in G2 (on the GPU);
      5. with a random 128-bit rho (from `secrets`, or from rng.getrandbits for reproducible runs),
         A = sum_{i<d} rho^i [tau^i]_1 and B = sum_{i<d} rho^i [tau^(i+1)]_1 (two MSMs on the cached table) satisfy
         e([tau]_2, A) = e([1]_2, B).
    Step 5 accepts an SRS whose powers are not consecutive with probability at most d / 2^128 (a non-zero
    polynomial of degree < d in rho vanishes at a random rho)."""
    (rho,) = batch_weights(1, rng)
    check = _powers_check(srs, rho)
    if check is None:
        return False
    return pairing_check(*check)


def contribute(srs, secret=None, rng=None):
    """-> (nxt, Contribution): the SRS for tau' = s tau and the proof of the update.  s is drawn uniformly from
    [1, r) with `secrets` (or rng.randrange) unless `secret` is given; a secret that is 0 mod r is refused.
    [tau'^i]_1 = s^i [tau^i]_1 is one per-point scalar multiplication of the input's cached device table, and the
    result is registered with the table cache; the input SRS and its cache entry are left as they were."""
    _check_shape(srs)
    if secret is None:
        s = rng.randrange(1, CURVE_ORDER) if rng is not None else secrets.randbelow(CURVE_ORDER - 1) + 1
    else:
        s = int(secret) % CURVE_ORDER
        if s == 0:
            raise ValueError("contribute: the secret must not be 0 mod r")
    k = rng.randrange(1, CURVE_ORDER) if rng is not None else secrets.randbelow(CURVE_ORDER - 1) + 1
    n = srs.max_degree + 1
    pw = native.scalars_alloc(n)
    native.scalars_fill_powers(pw, 0, n, 1, s)                                # s^i
    handle = native.g1_table_scale(tables.g1_table(srs.g1_powers), 0, pw, 0, n)
    pw.free()
    raw = native.table_download(handle, 0, n)
    g1_powers = [g1_from_ints(native.g1_from_bytes(raw[64 * i:64 * i + 64])) for i in range(n)]
    h2 = native.g2_fixed_base_mul(native.g2_bytes(srs.g2_powers[1]), native.fe_bytes(s), 1)
    tau_g2 = g2_from_ints(native.g2_from_bytes(native.table_download(h2, 0, 1)))
    h2.free()
    tables.adopt_g1(g1_powers, handle)
    nxt = SRS(g1_powers, [srs.g2_powers[0], tau_g2], srs.max_degree)

    h1 = native.g1_fixed_base_mul(native.g1_bytes(G1), native.fr_vec_bytes([s, k]), 2)   # [s]_1, [k]_1
    sk = native.table_download(h1, 0, 2)
    h1.free()
    s_g1, R = g1_from_ints(native.g1_from_bytes(sk[:64])), g1_from_ints(native.g1_from_bytes(sk[64:]))
    z = (k + challenge(srs, s_g1, R) * s) % CURVE_ORDER
    return nxt, Contribution(s_g1, R, z)


def verify_contribution(prev, nxt, contribution, rng=None):
    """True iff `nxt` is `prev` updated by the secret behind `contribution`.  `prev` is assumed verified (a chain
    from a trusted start is a loop over this function).  Checks:
      - both SRSs have the same max_degree (and the shapes of verify_srs: ValueError otherwise);
      - s_g1 = [s]_1 is a point of G1 other than infinity;
      - the proof of knowledge: z G1 == R + c s_g1 (one two-point MSM: z G1 - c s_g1);
      - verify_srs(nxt) and the link e([1]_2, [tau']_1) = e([tau]_2, [s]_1), folded into verify_srs's pairing check
        with a second random weight sigma, so the whole check is one pairing check of four pairs (one final
        exponentiation)."""
    _check_shape(prev)
    _check_shape(nxt)
    if prev.max_degree != nxt.max_degree:
        return False
    s_g1, R = contribution.s_g1, contribution.R
    if not _on_g1(s_g1) or not _on_g1(R):
        return False
    c = challenge(prev, s_g1, R)
    lhs = native.g1_msm(native.g1_vec_bytes([G1, s_g1]),
                        native.fr_vec_bytes([contribution.z % CURVE_ORDER, (-c) % CURVE_ORDER]), 2)
    if native.g1_bytes(lhs) != native.g1_bytes(R):
        return False
    rho, sigma = batch_weights(2, rng)
    check = _powers_check(nxt, rho)
    if check is None:
        return False
    pairs, scalars = check
    pairs += [(nxt.g2_powers[0], nxt.g1_powers[1]), (prev.g2_powers[1], s_g1)]   # e([1]_2, [tau']_1) e([tau]_2, [s]_1)^-1
    scalars += [sigma, CURVE_ORDER - sigma]
    return pairing_check(pairs, scalars)
