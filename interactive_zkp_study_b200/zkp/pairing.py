"""The BN254 pairing on the GPU, with py_ecc's interface (SURVEY.md 8f-4: the verifiers' last step).

``pairing(Q, P)`` has bn128.pairing's argument order and result: a ``compat.FQ12`` bit-identical with py_ecc's,
``AssertionError`` for a point that is not on its curve.  It can be handed to the verifier mirrors as
``pairing=`` (groth16.verifying.verify, plonk.verifier.verify).

``pairing_check(pairs, scalars=None, g2_subgroup_check=False)`` decides prod_i e(Q_i, k_i P_i) == 1 in one
device call: one Miller loop per pair, in parallel, and one final exponentiation.  The batch verifiers
(groth16.verifying.verify_batch, plonk.verifier.verify_batch) are built on it.
"""
import secrets

from .. import native
from ..compat import FQ12, curve_order


def _g2(Q):
    return native.g2_bytes(Q)


def _g1(P):
    return native.g1_bytes(P)


def _call(fn, *args):
    try:
        return fn(*args)
    except native.ZkpB200Error as e:
        if "not on its curve" in str(e):    # py_ecc: assert is_on_curve(Q, b2) / (P, b)
            raise AssertionError(str(e)) from e
        raise


def pairing(Q, P):
    """e(Q, P), Q in G2 (a pair of FQ2, or None), P in G1 (a pair of FQ / ints, or None) -> FQ12."""
    return FQ12(_call(native.pairing, _g2(Q), _g1(P)))


def pairing_check(pairs, scalars=None, g2_subgroup_check=False):
    """[ prod_i e(Q_i, k_i P_i) == 1 ] for pairs = [(Q_i, P_i)], scalars = [k_i] (reduced mod r; None: all 1).
    With g2_subgroup_check a Q_i outside the order-r subgroup makes the check fail (points that come from a
    prover need it: the twist also has points of other orders).  An empty product is 1."""
    pairs = list(pairs)
    n = len(pairs)
    if scalars is not None:
        scalars = [int(k) % curve_order for k in scalars]
        if len(scalars) != n:
            raise ValueError("pairing_check: one scalar per pair")
    g2b = b"".join(_g2(q) for q, _ in pairs)
    g1b = b"".join(_g1(p) for _, p in pairs)
    sc = native.fr_vec_bytes(scalars) if scalars is not None else None
    return _call(native.pairing_check, g2b, g1b, n, sc, g2_subgroup_check)


def batch_weights(k, rng=None):
    """k non-zero 128-bit random weights for a batch check: from `secrets`, or from rng.getrandbits (a
    random.Random) for reproducible runs."""
    draw = (lambda: rng.getrandbits(128)) if rng is not None else (lambda: secrets.randbits(128))
    out = []
    while len(out) < k:
        w = draw()
        if w:
            out.append(w)
    return out
