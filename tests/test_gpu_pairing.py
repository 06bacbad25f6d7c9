"""-m gpu: the BN254 pairing on the device (csrc/pairing.cu, zkp/pairing.py) and the batch verifiers built on it.
The Fp12 tower piece by piece and zkp_pairing bit for bit against the oracle's py_ecc restatement; the pairing
check on sets of pairs whose exponents cancel; the verifier mirrors with the device pairing; batch verification."""
import copy
import random

import pytest

from oracle import bn254
from oracle.shim.py_ecc import bn128 as bn
from tests.util import g1, g2, load

pytestmark = pytest.mark.gpu
R = bn254.R
P = bn254.P
rng = random.Random(1020)


def _fq12_bytes(vals):
    return b"".join(int(c).to_bytes(32, "little") for v in vals for c in v.coeffs)


def _fq12_list(b, n):
    return [bn.FQ12([int.from_bytes(b[384 * i + 32 * j:384 * i + 32 * j + 32], "little") for j in range(12)])
            for i in range(n)]


def _shim_g2(q):
    return None if q is None else (bn.FQ2(list(q[0])), bn.FQ2(list(q[1])))


def _shim_g1(p):
    return None if p is None else (bn.FQ(p[0]), bn.FQ(p[1]))


def test_fp12_ops_match_pyecc(native):
    n = 4
    a = [bn.FQ12([rng.randrange(P) for _ in range(12)]) for _ in range(n)]
    b = [bn.FQ12([rng.randrange(P) for _ in range(12)]) for _ in range(n)]
    ab, bb = _fq12_bytes(a), _fq12_bytes(b)
    assert _fq12_list(native.dbg_fp12_op(0, ab, bb, n), n) == [x * y for x, y in zip(a, b)]
    assert _fq12_list(native.dbg_fp12_op(1, ab, None, n), n) == [x * x for x in a]
    assert _fq12_list(native.dbg_fp12_op(3, ab, None, n), n) == [bn.FQ12.one() / x for x in a]
    for k in (1, 2, 3):
        assert _fq12_list(native.dbg_fp12_op(3 + k, ab, None, n), n) == [x ** (P ** k) for x in a], k
    fe = _fq12_list(native.dbg_fp12_op(7, ab[:2 * 384], None, 2), 2)
    assert fe == [bn.final_exponentiate(x) for x in a[:2]]
    # cyclotomic squaring on elements after the easy part f^((p^6 - 1)(p^2 + 1))
    easy = []
    for x in a:
        y = x ** (P ** 6) / x
        easy.append(y ** (P ** 2) * y)
    assert _fq12_list(native.dbg_fp12_op(2, _fq12_bytes(easy), None, n), n) == [y * y for y in easy]


def test_pairing_bit_identical_with_pyecc(native):
    from interactive_zkp_study_b200.compat import FQ12
    from interactive_zkp_study_b200.zkp.pairing import pairing
    cases = [(1, 1)] + [(rng.randrange(1, R), rng.randrange(1, R)) for _ in range(3)]
    for a, b in cases:
        q, p = bn254.g2_mul(bn254.G2, a), bn254.g1_mul(bn254.G1, b)
        want = bn.pairing(_shim_g2(q), _shim_g1(p))
        got = native.pairing(native.g2_bytes(q), native.g1_bytes(p))
        assert got == [c.n for c in want.coeffs], (a, b)
        e = pairing(bn254.g2_mul(bn254.G2, a), bn254.g1_mul(bn254.G1, b))
        assert isinstance(e, FQ12) and [int(c) for c in e.coeffs] == got
    assert pairing(None, bn254.G1) == FQ12.one()
    assert pairing(bn254.G2, None) == FQ12.one()


def _device_points(native, g1_scalars, g2_scalars):
    n1, n2 = len(g1_scalars), len(g2_scalars)
    t1 = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes(g1_scalars), n1)
    t2 = native.g2_fixed_base_mul(native.g2_bytes(bn254.G2), native.fr_vec_bytes(g2_scalars), n2)
    return native.table_download(t1, 0, n1), native.table_download(t2, 0, n2)


@pytest.mark.parametrize("n", [1, 2, 3, 64, 4096])
def test_pairing_check_cancelling_sets(native, n):
    """prod e(a_i G2, k_i b_i G1) with sum a_i b_i k_i = 0 mod r is 1; changing one k_i breaks it."""
    a = [rng.randrange(1, R) for _ in range(n)]
    b = [rng.randrange(1, R) for _ in range(n)]
    k = [rng.randrange(1, R) for _ in range(n - 1)]
    rest = sum(x * y * z for x, y, z in zip(a, b, k)) % R
    k.append((-rest * pow(a[-1] * b[-1], -1, R)) % R or R)   # n = 1: k = r, a value >= r that reduces to 0
    g1b, g2b = _device_points(native, b, a)
    sc = native.fr_vec_bytes(k)
    assert native.pairing_check(g2b, g1b, n, sc) is True
    bad = list(k)
    bad[n // 2] = (bad[n // 2] + 1) % (1 << 256)
    assert native.pairing_check(g2b, g1b, n, native.fr_vec_bytes(bad)) is False
    if n <= 64:                                              # the same with the scalars folded into the points
        pre, _ = _device_points(native, [x * y % R for x, y in zip(b, k)], [1])
        assert native.pairing_check(g2b, pre, n) is True
        assert native.pairing_check(g2b, pre, n, g2_subgroup_check=True) is True


def test_pairing_check_scalar_edge_values_agree_with_premultiplied_points(native):
    from interactive_zkp_study_b200.zkp.pairing import pairing_check
    k = [0, 1, R - 1, R + 5, (1 << 256) - 1, 7]
    a = [rng.randrange(1, R) for _ in k]
    b = [rng.randrange(1, R) for _ in k]
    rest = sum(x * y * z for x, y, z in zip(a[:-1], b[:-1], k[:-1])) % R
    b[-1] = (-rest * pow(a[-1] * k[-1], -1, R)) % R
    g1b, g2b = _device_points(native, b, a)
    pre, _ = _device_points(native, [x * y % R for x, y in zip(b, k)], [1])
    for tamper in (None, 2):
        kk = list(k)
        if tamper is not None:
            kk[tamper] += 1
        pre_t, _ = _device_points(native, [x * y % R for x, y in zip(b, kk)], [1])
        want = tamper is None
        assert native.pairing_check(g2b, g1b, len(k), native.fr_vec_bytes(kk)) is want
        assert native.pairing_check(g2b, pre_t, len(k)) is want
    # through zkp.pairing with py_ecc-style points; infinity on either side contributes 1
    pts1 = [native.g1_from_bytes(pre[64 * i:64 * i + 64]) for i in range(len(k))]
    pts2 = [native.g2_from_bytes(g2b[128 * i:128 * i + 128]) for i in range(len(k))]
    assert pairing_check(list(zip(pts2, pts1)) + [(None, bn254.G1), (bn254.G2, None)]) is True
    assert pairing_check([]) is True


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


def test_invalid_points_and_g2_subgroup(native):
    from interactive_zkp_study_b200.zkp.pairing import pairing, pairing_check
    q, p = bn254.g2_mul(bn254.G2, 3), bn254.g1_mul(bn254.G1, 5)
    off1 = (p[0], (p[1] + 1) % P)
    off2 = (q[0], (q[1][0], (q[1][1] + 1) % P))
    for g2p, g1p in ((q, off1), (off2, p)):
        with pytest.raises(native.ZkpB200Error, match="not on its curve"):
            native.pairing(native.g2_bytes(g2p), native.g1_bytes(g1p))
        with pytest.raises(native.ZkpB200Error, match="not on its curve"):
            native.pairing_check(native.g2_bytes(g2p) * 2, native.g1_bytes(g1p) * 2, 2)
        with pytest.raises(AssertionError):
            pairing(g2p, g1p)
    with pytest.raises(native.ZkpB200Error):
        native.pairing(native.g2_bytes(q), ((P).to_bytes(32, "little") + bytes(32)))   # coordinate not below p
    bad = _twist_point_outside_g2()
    h = 2 * P - R                                                  # the cofactor: h * bad lies in G2
    good = bn.multiply(bad, h)
    assert good is not None and bn.multiply(good, R) is None
    for pt, want in ((bad, False), (good, True)):
        qi = _ints2(pt)
        # e(Q, P) e(Q, -P) = 1 whatever Q is; only the subgroup check can tell the two apart
        pairs = [(qi, bn254.G1), (qi, bn254.g1_neg(bn254.G1))]
        assert pairing_check(pairs) is True
        assert pairing_check(pairs, g2_subgroup_check=True) is want


def test_verifier_mirrors_with_device_pairing(native):
    """The decisions of tests/test_gpu_verifiers.py, with zkp.pairing.pairing instead of the oracle's."""
    from interactive_zkp_study_b200.compat import FR, g1_from_ints, g2_from_ints
    from interactive_zkp_study_b200.zkp.groth16.proving import build_rpub_enum
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify
    from interactive_zkp_study_b200.zkp.pairing import pairing
    from interactive_zkp_study_b200.zkp.plonk.field import FR as PFR
    from interactive_zkp_study_b200.zkp.plonk.prover import Proof
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify as pverify
    g = load("groth16_toy.json")
    A, B, C = g1_from_ints(g1(g["proof_a"])), g2_from_ints(g2(g["proof_b"])), g1_from_ints(g1(g["proof_c"]))
    s11 = [g1_from_ints(g1(p)) for p in g["sigma1_1"]]
    s13 = [g1_from_ints(g1(p)) for p in g["sigma1_3"]]
    s21 = [g2_from_ints(g2(p)) for p in g["sigma2_1"]]
    rx_pub = build_rpub_enum(g["pub_r_indexs"], [FR(int(x)) for x in g["Rx"]])
    assert verify(A, B, C, s11, s13, s21, rx_pub, pairing=pairing) is True
    badC = g1_from_ints(bn254.g1_add(g1(g["proof_c"]), bn254.G1))
    assert verify(A, B, badC, s11, s13, s21, rx_pub, pairing=pairing) is False
    bad_pub = [(rx_pub[0][0], rx_pub[0][1]), (rx_pub[1][0], rx_pub[1][1] + FR(1))]
    assert verify(A, B, C, s11, s13, s21, bad_pub, pairing=pairing) is False
    with pytest.raises(NotImplementedError):
        verify(A, B, C, s11, s13, s21, rx_pub)          # the default stays: no py_ecc, no pairing given
    for name in ("plonk_n1.json", "plonk_x3.json", "plonk_chain16.json"):
        f = load(name)
        proof = Proof()
        for k, v in f["proof"].items():
            setattr(proof, k, g1_from_ints(g1(v)) if k.endswith("_comm") else PFR(int(v)))
        pp = type("PP", (), {})()
        pp.n, pp.omega = f["n"], PFR(int(f["omega"]))
        for k, v in f["pre_comm"].items():
            setattr(pp, k + "_comm", g1_from_ints(g1(v)))
        srs = SRS([], [g2_from_ints(g2(p)) for p in f["g2_powers"]], f["srs_max_degree"])
        assert pverify(proof, [], pp, srs, pairing=pairing) is True, name
        for field in ("a_eval", "r_eval", "z_omega_eval"):
            bad = copy.deepcopy(proof)
            setattr(bad, field, getattr(bad, field) + PFR(1))
            assert pverify(bad, [], pp, srs, pairing=pairing) is False, (name, field)


@pytest.fixture(scope="module")
def toy(native):
    from interactive_zkp_study_b200.compat import FQ, FQ2, FR
    g = load("groth16_toy.json")
    pt1 = lambda p: (FQ(int(p[0])), FQ(int(p[1])))
    pt2 = lambda p: (FQ2([int(p[0][0]), int(p[0][1])]), FQ2([int(p[1][0]), int(p[1][1])]))
    d = {"g": g}
    for k in ("Ax", "Bx", "Cx"):
        d[k] = [[FR(int(x)) for x in row] for row in g[k]]
    d["Rx"] = [FR(int(x)) for x in g["Rx"]]
    d["Hx"] = [FR(int(x)) for x in g["Hx"]]
    for k in ("sigma1_1", "sigma1_2", "sigma1_3", "sigma1_4", "sigma1_5"):
        d[k] = [pt1(p) for p in g[k]]
    for k in ("sigma2_1", "sigma2_2"):
        d[k] = [pt2(p) for p in g[k]]
    return d


def test_groth16_verify_batch_on_the_toy_statement(toy):
    from interactive_zkp_study_b200.compat import FR, g1_from_ints, g2_from_ints
    from interactive_zkp_study_b200.zkp.groth16.proving import proof_a, proof_b, proof_c, build_rpub_enum
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify, verify_batch
    from interactive_zkp_study_b200.zkp.pairing import pairing
    g = toy["g"]
    proofs = []
    for _ in range(64):                                   # fresh (r, s) per proof through the proving mirror
        r, s = FR(rng.randrange(R)), FR(rng.randrange(R))
        A = proof_a(toy["sigma1_1"], toy["sigma1_2"], toy["Ax"], toy["Rx"], r)
        B = proof_b(toy["sigma2_1"], toy["sigma2_2"], toy["Bx"], toy["Rx"], s)
        C = proof_c(toy["sigma1_1"], toy["sigma1_2"], toy["sigma1_4"], toy["sigma1_5"], toy["Bx"], toy["Rx"], toy["Hx"],
                    s, r, A, pub_r_indexs=g["pub_r_indexs"])
        proofs.append((A, B, C))
    rx_pub = build_rpub_enum(g["pub_r_indexs"], toy["Rx"])
    keys = (toy["sigma1_1"], toy["sigma1_3"], toy["sigma2_1"])
    assert verify_batch(proofs, *keys, [rx_pub] * 64, rng=random.Random(1)) is True
    assert verify_batch(proofs, *keys, [rx_pub] * 64) is True            # weights from `secrets`
    assert verify_batch([], *keys, []) is True
    bad = list(proofs)
    A, B, C = bad[17]
    bad[17] = (A, B, g1_from_ints(bn254.g1_add((int(C[0]), int(C[1])), bn254.G1)))
    assert verify_batch(bad, *keys, [rx_pub] * 64, rng=random.Random(2)) is False
    bad_pub = [(rx_pub[0][0], rx_pub[0][1]), (rx_pub[1][0], rx_pub[1][1] + FR(1))]
    assert verify_batch(proofs, *keys, [rx_pub] * 63 + [bad_pub], rng=random.Random(3)) is False
    outside = _twist_point_outside_g2()
    bad = list(proofs)
    bad[5] = (bad[5][0], g2_from_ints(_ints2(outside)), bad[5][2])
    assert verify_batch(bad, *keys, [rx_pub] * 64, rng=random.Random(4)) is False
    # k = 1 decides as verify does
    for (A, B, C), pub in ((proofs[0], rx_pub), (proofs[0], bad_pub)):
        assert verify_batch([(A, B, C)], *keys, [pub]) is verify(A, B, C, *keys, pub, pairing=pairing)


def _synthetic_groth16(native, k, seed):
    """k valid proofs for keys with known alpha, beta, gamma, delta and one public wire (sigma1_3 = [s0 G1]):
    A = a G1, B = b G2, C = c G1 with a b = alpha beta + x_j s0 gamma + c delta."""
    from interactive_zkp_study_b200.compat import g1_from_ints, g2_from_ints
    rr = random.Random(seed)
    al, be, ga, de, s0 = (rr.randrange(1, R) for _ in range(5))
    a = [rr.randrange(1, R) for _ in range(k)]
    b = [rr.randrange(1, R) for _ in range(k)]
    x = [rr.randrange(R) for _ in range(k)]
    dinv = pow(de, -1, R)
    c = [(ai * bi - al * be - xi * s0 * ga) * dinv % R for ai, bi, xi in zip(a, b, x)]
    g1b, g2b = _device_points(native, a + c + [al, s0], b + [be, ga, de])
    pt1 = [g1_from_ints(native.g1_from_bytes(g1b[64 * i:64 * i + 64])) for i in range(2 * k + 2)]
    pt2 = [g2_from_ints(native.g2_from_bytes(g2b[128 * i:128 * i + 128])) for i in range(k + 3)]
    proofs = [(pt1[j], pt2[j], pt1[k + j]) for j in range(k)]
    keys = ([pt1[2 * k]], [pt1[2 * k + 1]], pt2[k:k + 3])
    return proofs, keys, [[(0, xi)] for xi in x]


def test_groth16_verify_batch_synthetic_4096(native):
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify_batch
    proofs, keys, pubs = _synthetic_groth16(native, 4096, 7)
    assert verify_batch(proofs, *keys, pubs, rng=random.Random(5)) is True
    pubs[4000] = [(0, (pubs[4000][0][1] + 1) % R)]
    assert verify_batch(proofs, *keys, pubs, rng=random.Random(6)) is False


def test_plonk_verify_batch(native):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import plonk_synth
    from interactive_zkp_study_b200.compat import G2, g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    n = 1 << 6
    circ = plonk_synth.chain_circuit(n, seed=3)
    key, wit, tau = plonk_synth.device_setup(circ)
    pp = type("PP", (), {})()
    pp.n, pp.omega = n, FR(key.omega)
    for k in dp.CIRCUIT_POLYS:
        setattr(pp, k + "_comm", key.comm[k])
    srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)
    items = [(dp.prove(key, *wit), [], pp) for _ in range(4)]
    assert verify_batch(items, srs, rng=random.Random(8)) is True
    assert verify_batch(items[:1], srs) is True
    bad = copy.deepcopy(items[2][0])
    bad.c_eval = bad.c_eval + FR(1)
    assert verify_batch(items[:2] + [(bad, [], pp)] + items[3:], srs, rng=random.Random(9)) is False
