"""-m gpu: powers-of-tau contributions (zkp/plonk/ceremony.py) and the two device entry points under them:
zkp_g1/g2_table_scale bit for bit against the oracle and, at 2^16 / 2^20, against fixed-base tables of the product
exponents; zkp_g1/g2_table_validate on planted faults; contribute against SRSs built from tau s; verify_srs and
verify_contribution on honest and tampered inputs; a PLONK proof under a contributed SRS."""
import random

import pytest

from oracle import bn254
from oracle.shim.py_ecc import bn128 as bn
from tests.util import load

pytestmark = pytest.mark.gpu
R = bn254.R
P = bn254.P
rng = random.Random(2024)
EDGE = [0, 1, R - 1, R, R + 5, (1 << 256) - 1]


def _g1_pts(native, exps):
    t = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes(exps), len(exps))
    raw = native.table_download(t, 0, len(exps))
    return [native.g1_from_bytes(raw[64 * i:64 * i + 64]) for i in range(len(exps))]


def _g2_pts(native, exps):
    t = native.g2_fixed_base_mul(native.g2_bytes(bn254.G2), native.fr_vec_bytes(exps), len(exps))
    raw = native.table_download(t, 0, len(exps))
    return [native.g2_from_bytes(raw[128 * i:128 * i + 128]) for i in range(len(exps))]


def _scaled(native, table, offset, ks, sc_offset=0, pad=0):
    """table_scale with the scalars uploaded at sc_offset (pad extra zeros after) -> list of points."""
    sc = native.scalars_load(native.fr_vec_bytes([0] * sc_offset + ks + [0] * pad), sc_offset + len(ks) + pad)
    fn = native.g1_table_scale if table.kind == "g1" else native.g2_table_scale
    out = fn(table, offset, sc, sc_offset, len(ks))
    assert out.n == len(ks) and out.kind == table.kind
    raw = native.table_download(out, 0, len(ks))
    sz = 64 if table.kind == "g1" else 128
    dec = native.g1_from_bytes if table.kind == "g1" else native.g2_from_bytes
    return [dec(raw[sz * i:sz * i + sz]) for i in range(len(ks))]


def test_g1_table_scale_matches_oracle(native):
    n = 64
    pts = _g1_pts(native, [rng.randrange(1, R) for _ in range(n)])
    pts[5] = pts[17] = None                                        # infinity in: infinity out
    ks = EDGE + [rng.randrange(1 << 256) for _ in range(n - len(EDGE))]
    want = [bn254.g1_mul(p, k) if p is not None else None for p, k in zip(pts, ks)]
    t = native.g1_table_load(native.g1_vec_bytes(pts), n)
    assert _scaled(native, t, 0, ks) == want
    # a sub-range of the points against a sub-range of the scalars
    assert _scaled(native, t, 10, ks[:40], sc_offset=3, pad=2) == [bn254.g1_mul(p, k) if p else None
                                                                   for p, k in zip(pts[10:50], ks[:40])]
    # the same points in a window-precomputed table (row 0 holds the points)
    t2 = native.g1_table_load(native.g1_vec_bytes(pts), n)
    assert native.table_precompute(t2, 4) == 4
    assert _scaled(native, t2, 0, ks) == want
    assert _scaled(native, t2, 7, ks[7:20]) == want[7:20]


def test_g2_table_scale_matches_oracle(native):
    n = 16
    pts = _g2_pts(native, [rng.randrange(1, R) for _ in range(n)])
    pts[3] = None
    ks = EDGE + [rng.randrange(1 << 256) for _ in range(n - len(EDGE))]
    want = [bn254.g2_mul(p, k) if p is not None else None for p, k in zip(pts, ks)]
    t = native.g2_table_load(native.g2_vec_bytes(pts), n)
    got = _scaled(native, t, 0, ks)
    assert [native.g2_bytes(g) for g in got] == [native.g2_bytes(w) for w in want]
    t2 = native.g2_table_load(native.g2_vec_bytes(pts), n)
    native.table_precompute(t2, 4)
    assert [native.g2_bytes(g) for g in _scaled(native, t2, 2, ks[2:9], sc_offset=1)] == \
        [native.g2_bytes(w) for w in want[2:9]]


def test_table_scale_errors(native):
    t1 = native.g1_table_load(native.g1_vec_bytes(_g1_pts(native, [1, 2, 3, 4])), 4)
    t2 = native.g2_table_load(native.g2_vec_bytes(_g2_pts(native, [1, 2])), 2)
    sc = native.scalars_load(native.fr_vec_bytes([1, 2, 3, 4]), 4)
    empty = native.g1_table_scale(t1, 4, sc, 4, 0)                  # n == 0 at the very end: an empty table
    assert empty.n == 0 and native.table_download(empty, 0, 0) == b""
    for args in ((t1, 1, sc, 0, 4), (t1, 0, sc, 1, 4), (t1, 5, sc, 0, 0), (t1, (1 << 64) - 1, sc, 0, 2)):
        with pytest.raises(native.ZkpB200Error, match="error -3"):  # ZKP_ERR_INVALID_ARGUMENT
            native.g1_table_scale(*args)
    with pytest.raises(native.ZkpB200Error, match="error -4"):      # ZKP_ERR_BAD_HANDLE: a G2 table
        native.g1_table_scale(t2, 0, sc, 0, 1)
    with pytest.raises(native.ZkpB200Error, match="error -4"):
        native.g2_table_scale(t1, 0, sc, 0, 1)
    with pytest.raises(native.ZkpB200Error, match="error -4"):      # a scalar vector where the table goes
        native.g1_table_scale(sc, 0, sc, 0, 1)
    with pytest.raises(native.ZkpB200Error, match="error -4"):      # a table where the scalars go
        native.g1_table_scale(t1, 0, t1, 0, 1)
    with pytest.raises(native.ZkpB200Error, match="error -3"):
        native.g2_table_validate(t2, 1, 2)
    with pytest.raises(native.ZkpB200Error, match="error -4"):
        native.g1_table_validate(t2, 0, 1)
    with pytest.raises(native.ZkpB200Error, match="error -4"):
        native.g2_table_validate(sc, 0, 1)


@pytest.mark.parametrize("group,log_n", [(1, 16), (1, 20), (2, 16)])
def test_table_scale_at_scale_equals_fixed_base_of_products(native, group, log_n):
    """(s_i G) scaled by k_i is byte-identical with the fixed-base table of (s_i k_i) G."""
    n = 1 << log_n
    s = native.scalars_generate(11 + log_n, n)
    k = native.scalars_generate(12 + log_n, n)
    edge = [0, R, (1 << 256) - 1]                                   # edge scalars in the mix at indices 3..5
    native.scalars_upload(k, 3, native.fr_vec_bytes(edge), 3)
    prod = native.scalars_alloc(n)
    native.vec_op_dev(2, prod, 0, s, 0, k, 0, n)
    s_edge = native.fr_vec_from_bytes(native.scalars_download(s, 3, 3))
    native.scalars_upload(prod, 3, native.fr_vec_bytes([a * b % R for a, b in zip(s_edge, edge)]), 3)
    if group == 1:
        base, fixed, scale = native.g1_bytes(bn254.G1), native.g1_fixed_base_mul_dev, native.g1_table_scale
    else:
        base, fixed, scale = native.g2_bytes(bn254.G2), native.g2_fixed_base_mul_dev, native.g2_table_scale
    pts = fixed(base, s, n)
    want = native.table_download(fixed(base, prod, n), 0, n)
    assert native.table_download(scale(pts, 0, k, 0, n), 0, n) == want
    if group == 1 and log_n == 16:                                  # precomputed source, offset range
        native.table_precompute(pts)
        h = scale(pts, 100, k, 100, n - 200)
        assert native.table_download(h, 0, n - 200) == want[64 * 100:64 * (n - 100)]


def _off_g1(p):
    return (p[0], (p[1] + 1) % P)


def _off_g2(q):
    return (q[0], (q[1][0], (q[1][1] + 1) % P))


def _twist_point_outside_g2():
    """A point of y^2 = x^3 + 3/(9+u) that is not in G2 (the twist's order is r (2p - r))."""
    def fsqrt(a):                                 # square root in Fp2 (p = 3 mod 4), or None
        n = (a[0] * a[0] + a[1] * a[1]) % P
        al = pow(n, (P + 1) // 4, P)
        if al * al % P != n:
            return None
        for d in ((a[0] + al) * pow(2, -1, P) % P, (a[0] - al) * pow(2, -1, P) % P):
            x0 = pow(d, (P + 1) // 4, P)
            if x0 * x0 % P == d and x0:
                x1 = a[1] * pow(2 * x0, -1, P) % P
                if ((x0 * x0 - x1 * x1) % P, 2 * x0 * x1 % P) == (a[0] % P, a[1] % P):
                    return (x0, x1)
        return None
    b2 = bn.b2
    for x0 in range(1, 100):
        x = bn.FQ2([x0, 1])
        rhs = x ** 3 + b2
        y = fsqrt((rhs.coeffs[0].n, rhs.coeffs[1].n))
        if y is not None:
            pt = (x, bn.FQ2(list(y)))
            assert bn.is_on_curve(pt, b2)
            if bn.multiply(pt, R) is not None:
                return pt
    raise AssertionError("no twist point found")


def _ints2(pt):
    return ((pt[0].coeffs[0].n, pt[0].coeffs[1].n), (pt[1].coeffs[0].n, pt[1].coeffs[1].n))


def test_g1_table_validate(native):
    n = 300
    pts = _g1_pts(native, [rng.randrange(1, R) for _ in range(n)])
    pts[7] = None                                                  # infinity is valid
    t = native.g1_table_load(native.g1_vec_bytes(pts), n)
    assert native.g1_table_validate(t, 0, n) is None
    assert native.g1_table_validate(t, 0, 0) is None
    for js in ([0], [n - 1], [123], [200, 45], [46, 45]):
        bad = list(pts)
        for j in js:
            bad[j] = _off_g1(bad[j])
        tb = native.g1_table_load(native.g1_vec_bytes(bad), n)
        assert native.g1_table_validate(tb, 0, n) == min(js), js
        assert native.g1_table_validate(tb, min(js) + 1, n - min(js) - 1) == (max(js) if len(js) > 1 else None)
        native.table_precompute(tb, 6)                             # the points are row 0 of the new layout
        assert native.g1_table_validate(tb, 0, n) == min(js), js
    big = 1 << 16
    s = native.scalars_generate(5, big)
    tbig = native.g1_fixed_base_mul_dev(native.g1_bytes(bn254.G1), s, big)
    assert native.g1_table_validate(tbig, 0, big) is None


def test_g2_table_validate_and_subgroup(native):
    n = 40
    pts = _g2_pts(native, [rng.randrange(1, R) for _ in range(n)])
    pts[2] = None
    t = native.g2_table_load(native.g2_vec_bytes(pts), n)
    assert native.g2_table_validate(t, 0, n) is None
    assert native.g2_table_validate(t, 0, n, subgroup_check=True) is None
    bad = list(pts)
    bad[31], bad[9] = _off_g2(bad[31]), _off_g2(bad[9])
    tb = native.g2_table_load(native.g2_vec_bytes(bad), n)
    assert native.g2_table_validate(tb, 0, n) == 9
    assert native.g2_table_validate(tb, 10, n - 10, subgroup_check=True) == 31
    outside = _twist_point_outside_g2()
    cof = bn.multiply(outside, 2 * P - R)                          # its cofactor multiple lies in G2
    assert cof is not None and bn.multiply(cof, R) is None
    mixed = list(pts)
    mixed[13] = _ints2(cof)
    mixed[21] = _ints2(outside)
    tm = native.g2_table_load(native.g2_vec_bytes(mixed), n)
    assert native.g2_table_validate(tm, 0, n) is None              # on the twist: only the subgroup test sees it
    assert native.g2_table_validate(tm, 0, n, subgroup_check=True) == 21
    assert native.g2_table_validate(tm, 0, 21, subgroup_check=True) is None


# ------------------------------------------------------------------ the ceremony
def _tau(seed):
    import hashlib
    return int.from_bytes(hashlib.sha256(str(seed).encode()).digest(), "big") % R


def _expected_g1(native, t, n):
    powers = native.fr_prefix_product(native.fr_vec_bytes([t] * n), n)
    return native.table_download(native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), powers, n), 0, n)


@pytest.mark.parametrize("d", [12, 1 << 10])
def test_contribute_is_exact_and_verifies(native, d):
    from interactive_zkp_study_b200 import tables
    from interactive_zkp_study_b200.zkp.plonk.ceremony import contribute, verify_contribution, verify_srs
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    seed = 900 + d
    srs = SRS.generate(d, seed=seed)
    before = native.g1_vec_bytes(srs.g1_powers)
    handle_before = tables.g1_table(srs.g1_powers)
    tau, chain, cur = _tau(seed), [], srs
    for s in (rng.randrange(1, R), rng.randrange(1, R), (1 << 256) - 1):
        nxt, proof = contribute(cur, secret=s)
        tau = tau * s % R
        assert nxt.max_degree == d and len(nxt.g1_powers) == d + 1
        assert native.g1_vec_bytes(nxt.g1_powers) == _expected_g1(native, tau, d + 1)
        assert native.g2_bytes(nxt.g2_powers[1]) == native.g2_bytes(bn254.g2_mul(bn254.G2, tau))
        assert native.g2_bytes(nxt.g2_powers[0]) == native.g2_bytes(bn254.G2)
        assert native.g1_bytes(proof.s_g1) == native.g1_bytes(bn254.g1_mul(bn254.G1, s % R))
        chain.append((cur, nxt, proof))
        cur = nxt
    for prev, nxt, proof in chain:
        assert verify_contribution(prev, nxt, proof, rng=random.Random(1)) is True
    assert verify_srs(cur) is True
    # the input and its cache entry are untouched
    assert native.g1_vec_bytes(srs.g1_powers) == before
    assert tables.g1_table(srs.g1_powers) is handle_before
    # the new table is registered: the first commit does not upload it again
    assert tables.g1_table(cur.g1_powers) is tables.g1_table(cur.g1_powers)


def test_contribute_draws_its_secret(native):
    from interactive_zkp_study_b200.zkp.plonk.ceremony import contribute, verify_contribution
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    srs = SRS.generate(6, seed=1)
    a, pa = contribute(srs)
    b, pb = contribute(srs, rng=random.Random(5))
    c, pc = contribute(srs, rng=random.Random(5))
    assert native.g1_bytes(pa.s_g1) != native.g1_bytes(pb.s_g1)
    assert native.g1_bytes(pb.s_g1) == native.g1_bytes(pc.s_g1) and pb.z == pc.z
    assert verify_contribution(srs, a, pa) and verify_contribution(srs, b, pb)


def _with(srs, g1=None, g2=None, d=None):
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    return SRS(list(srs.g1_powers if g1 is None else g1), list(srs.g2_powers if g2 is None else g2),
               srs.max_degree if d is None else d)


def test_verify_srs_accepts_honest_and_rejects_tampered(native):
    from interactive_zkp_study_b200.compat import g1_from_ints, g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk.ceremony import verify_srs
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    d = 12
    srs = SRS.generate(d, seed=31)
    assert verify_srs(srs) is True
    assert verify_srs(srs, rng=random.Random(3)) is True
    other = g1_from_ints(bn254.g1_mul(bn254.G1, rng.randrange(1, R)))
    for j in (1, d // 2, d):
        g1 = list(srs.g1_powers)
        g1[j] = other
        assert verify_srs(_with(srs, g1=g1)) is False, j
    g1 = list(srs.g1_powers)
    g1[3], g1[4] = g1[4], g1[3]
    assert verify_srs(_with(srs, g1=g1)) is False
    g1 = list(srs.g1_powers)
    g1[0] = g1_from_ints(bn254.g1_mul(bn254.G1, 2))
    assert verify_srs(_with(srs, g1=g1)) is False
    assert verify_srs(_with(srs, g2=[srs.g2_powers[0], g2_from_ints(bn254.g2_mul(bn254.G2, 5))])) is False
    assert verify_srs(_with(srs, g2=[g2_from_ints(bn254.g2_mul(bn254.G2, 2)), srs.g2_powers[1]])) is False
    zero = SRS([g1_from_ints(bn254.G1)] + [None] * d, [g2_from_ints(bn254.G2), None], d)     # tau = 0
    assert verify_srs(zero) is False
    g1 = list(srs.g1_powers)
    g1[5] = g1_from_ints(_off_g1((int(g1[5][0]), int(g1[5][1]))))
    assert verify_srs(_with(srs, g1=g1)) is False
    outside = _twist_point_outside_g2()
    assert verify_srs(_with(srs, g2=[srs.g2_powers[0], g2_from_ints(_ints2(outside))])) is False
    assert verify_srs(SRS.generate(1 << 16, seed=32)) is True


def test_verify_contribution_rejects(native):
    from interactive_zkp_study_b200.zkp.plonk.ceremony import Contribution, contribute, verify_contribution
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    d = 12
    srs = SRS.generate(d, seed=41)
    nxt, proof = contribute(srs, secret=rng.randrange(1, R))
    other, other_proof = contribute(srs, secret=rng.randrange(1, R))
    assert verify_contribution(srs, nxt, proof) is True
    assert verify_contribution(srs, nxt, Contribution(proof.s_g1, proof.R, (proof.z + 1) % R)) is False
    assert verify_contribution(srs, nxt, other_proof) is False                 # the proof of another update
    assert verify_contribution(srs, nxt, Contribution(None, proof.R, proof.z)) is False
    assert verify_contribution(srs, SRS.generate(d, seed=42), proof) is False   # honest, but an unrelated tau
    assert verify_contribution(srs, other, proof) is False
    bigger, big_proof = contribute(SRS.generate(d + 1, seed=41), secret=3)
    assert verify_contribution(srs, bigger, big_proof) is False                # max_degree differs


class _StubGate:
    def __init__(self, q_l, q_r, q_o, q_m, q_c):
        self.q = (q_l, q_r, q_o, q_m, q_c)


class _StubCircuit:
    """The four members preprocess() reads from a reference Circuit."""

    def __init__(self, f, FR):
        sel = f["selectors"]
        self.gates = [_StubGate(*(FR(int(sel[k][i])) for k in ("q_l", "q_r", "q_o", "q_m", "q_c")))
                      for i in range(f["n_raw"])]
        self._sigma = list(f["sigma"])
        self.num_public_inputs = f["num_public_inputs"]

    @property
    def n(self):
        return len(self.gates)

    def get_selector_polynomials(self):
        return tuple([g.q[k] for g in self.gates] for k in range(5))

    def build_copy_constraints(self):
        return list(self._sigma)


def test_plonk_proof_under_a_contributed_srs(native):
    import copy
    from interactive_zkp_study_b200.zkp.plonk import prover
    from interactive_zkp_study_b200.zkp.plonk.ceremony import contribute
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.preprocessor import preprocess
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    f = load("plonk_x3.json")
    start = SRS.generate(f["srs_max_degree"], seed=12345)
    srs, _ = contribute(start)
    srs, _ = contribute(srs)
    pp = preprocess(_StubCircuit(f, FR), srs)
    vals = [[FR(int(x)) for x in f[k]] for k in ("a_vals", "b_vals", "c_vals")]
    proof = prover.prove(None, *vals, [], pp, srs)
    assert verify_batch([(proof, [], pp)], srs, rng=random.Random(2)) is True
    bad = copy.deepcopy(proof)
    bad.a_eval = bad.a_eval + FR(1)
    assert verify_batch([(bad, [], pp)], srs, rng=random.Random(2)) is False
    # the proof is bound to the contributed tau: the seeded start SRS does not accept it
    pp0 = preprocess(_StubCircuit(f, FR), start)
    assert verify_batch([(proof, [], pp0)], start, rng=random.Random(2)) is False
