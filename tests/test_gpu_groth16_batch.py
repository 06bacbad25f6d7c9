"""-m gpu: batch Groth16 proving -- many proofs of one circuit per pass.

(1) zkp_g1/g2_msm_dev_many against one MSM per scalar vector, bit for bit (plain and precomputed tables, a non-zero
offset, edge scalars, an all-zero vector, duplicate vectors, a single hot bucket), and against the oracle at small n;
(2) at scale through known discrete logs; (3) the batched quotient against per-proof quotients and the reference's
long division; (4) device_prover.prove_batch against prove; (5) the golden proofs inside a batch; (6) a synthetic
2^12-constraint batch end to end through verify_batch; (7) launches independent of the batch size; (8) refusals."""
import random

import pytest

from oracle import bn254, ref_path
from tests.util import g1, g2, ints, load

pytestmark = pytest.mark.gpu
R = bn254.R
EDGE = [0, 1, R - 1, R, R + 5, (1 << 256) - 1]


def _pt(p):
    return None if p is None else (int(p[0]), int(p[1]))


def _pt2(p):
    return None if p is None else ((int(p[0].coeffs[0]), int(p[0].coeffs[1])), (int(p[1].coeffs[0]), int(p[1].coeffs[1])))


def _proof_ints(prf):
    A, B, C = prf
    return _pt(A), _pt2(B), _pt(C)


_TABLES = {}


def _table(native, group, n, pre):
    """n + 5 points with known discrete logs (G1 or G2), plain or window-precomputed, cached per shape."""
    key = (group, n, pre)
    if key not in _TABLES:
        rng = random.Random(hash(key) & 0xffff)
        sc = native.fr_vec_bytes([rng.randrange(1, R) for _ in range(n + 5)])
        if group == 1:
            t = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), sc, n + 5)
        else:
            t = native.g2_fixed_base_mul(native.g2_bytes(bn254.G2), sc, n + 5)
        if pre:
            native.table_precompute(t)
        _TABLES[key] = t
    return _TABLES[key]


def _vectors(count, n, seed):
    """count scalar vectors: edge values in vector 0, vector 1 all zero, vector 2 a copy of vector 0, the last
    (from count = 4) one repeated scalar -- every digit of every window in one bucket."""
    rng = random.Random(seed)
    vs = [[rng.randrange(1 << 256) for _ in range(n)] for _ in range(count)]
    for i, e in enumerate(EDGE):
        vs[0][i % n] = e
    if count >= 2:
        vs[1] = [0] * n
    if count >= 3:
        vs[2] = list(vs[0])
    if count >= 4:
        vs[-1] = [rng.randrange(R)] * n
    return vs


CASES = [(1, 1), (2, 2), (3, 31), (17, 1000), (64, 4096), (64, 1), (17, 31), (3, 4096), (2, 1000), (5, 64)]


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("pre", [False, True])
@pytest.mark.parametrize("count,n", CASES)
def test_many_msm_equals_single_msms(native, group, pre, count, n):
    t = _table(native, group, n, pre)
    vs = _vectors(count, n, 1000 * count + n)
    sc_off = 7
    flat = [0] * sc_off + [x for v in vs for x in v]
    sh = native.scalars_load(native.fr_vec_bytes(flat), len(flat))
    got = native.msm_dev_many(t, 3, n, count, sh, sc_off)
    single = native.g1_msm_dev if group == 1 else native.g2_msm_dev
    want = [single(t, 3, sh, sc_off + j * n, n) for j in range(count)]
    assert got == want
    if count >= 2:
        assert got[1] is None
    if count >= 3:
        assert got[2] == got[0]
    if n <= 64:                                   # the oracle's commit loop over the same points
        raw = native.table_download(t, 3, n)
        sz = 64 if group == 1 else 128
        dec = native.g1_from_bytes if group == 1 else native.g2_from_bytes
        pts = [dec(raw[sz * i:sz * i + sz]) for i in range(n)]
        msm = bn254.g1_msm if group == 1 else bn254.g2_msm
        conv = g1 if group == 1 else g2
        for j in range(count):
            assert got[j] == conv(msm(pts, [x % R for x in vs[j]]))


@pytest.mark.parametrize("group,count,n", [(1, 256, 1 << 14), (2, 64, 1 << 12)])
def test_many_msm_at_scale_by_discrete_logs(native, group, count, n):
    """Result j = <c_j, s> G with s the points' discrete logs (device-generated points)."""
    s_h = native.scalars_generate(0x5EED0101 + group, n)
    c_h = native.scalars_generate(0x5EED0201 + group, count * n)
    if group == 1:
        t = native.g1_fixed_base_mul_dev(native.g1_bytes(bn254.G1), s_h, n)
    else:
        t = native.g2_fixed_base_mul_dev(native.g2_bytes(bn254.G2), s_h, n)
    native.table_precompute(t)
    got = native.msm_dev_many(t, 0, n, count, c_h, 0)
    dots = [native.fr_dot_dev(c_h, j * n, s_h, 0, n) for j in range(count)]
    if group == 1:
        ref = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes(dots), count)
        raw = native.table_download(ref, 0, count)
        want = [native.g1_from_bytes(raw[64 * j:64 * j + 64]) for j in range(count)]
    else:
        ref = native.g2_fixed_base_mul(native.g2_bytes(bn254.G2), native.fr_vec_bytes(dots), count)
        raw = native.table_download(ref, 0, count)
        want = [native.g2_from_bytes(raw[128 * j:128 * j + 128]) for j in range(count)]
    assert got == want


def _monic(rng, n):
    return [rng.randrange(R) for _ in range(n - 1)] + [1]


@pytest.mark.parametrize("count", [1, 3, 16, 100])
@pytest.mark.parametrize("length", [8, 257, 4096])
def test_quotient_batch_equals_per_proof(native, count, length):
    rng = random.Random(count * 7 + length)
    a, b, c = ([rng.randrange(R) for _ in range(count * length)] for _ in range(3))
    if count >= 3:
        a[length:2 * length] = [0] * length
    z = _monic(rng, length + 1)
    ha, hb, hc = (native.scalars_load(native.fr_vec_bytes(v), count * length) for v in (a, b, c))
    hz = native.scalars_load(native.fr_vec_bytes(z), length + 1)
    hq = native.groth16_quotient_batch_dev(ha, hb, hc, length, count, hz, length + 1)
    m = length - 1
    got = native.fr_vec_from_bytes(native.scalars_download(hq, 0, count * m))
    for j in range(count):
        parts = []
        for h in (ha, hb, hc):
            p = native.scalars_alloc(length)
            native.scalars_copy(p, 0, h, j * length, length)
            parts.append(p)
        q, _ = native.groth16_quotient_dev(*parts, length, hz, length + 1, want_remainder=False)
        assert got[j * m:(j + 1) * m] == native.fr_vec_from_bytes(native.scalars_download(q, 0, m)), j
        if length <= 300 and j < 3:
            aj, bj, cj = (v[j * length:(j + 1) * length] for v in (a, b, c))
            prod = ref_path.g16_subtract_polys(ref_path.g16_multiply_polys(aj, bj), cj)
            qq, _ = ref_path.g16_div_polys(prod, z)
            assert got[j * m:(j + 1) * m] == [x % R for x in qq]


def _device_key(native, k, m_priv, precompute, seed=3):
    from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
    rng = random.Random(seed)
    alpha, beta, delta, x = (rng.randrange(1, R) for _ in range(4))
    Z = native.fr_ap_vanishing_dev(k)
    zx = native.fr_poly_eval_dev(Z, 0, k + 1, x)
    priv = [rng.randrange(R) for _ in range(m_priv)]
    return dp.setup_from_toxic(k, alpha, beta, delta, x, zx, priv, precompute=precompute), Z


def _batch_inputs(native, k, m_priv, count, seed):
    rng = random.Random(seed)
    u = [[rng.randrange(R) for _ in range(count * k)] for _ in range(3)]
    u[0][:k] = [0] * k                                   # proof 0: an all-zero uA
    rx = [rng.randrange(R) for _ in range(count * m_priv)]
    rs = [0] + [rng.randrange(R) for _ in range(count - 1)]   # proof 0: r = s = 0
    ss = [0] + [rng.randrange(R) for _ in range(count - 1)]
    hs = [native.scalars_load(native.fr_vec_bytes(v), count * k) for v in u]
    hrx = native.scalars_load(native.fr_vec_bytes(rx), count * m_priv) if m_priv else native.scalars_alloc(0)
    return hs, hrx, rs, ss


def _single_proofs(native, key, Z, hs, hrx, rs, ss):
    from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
    k, mp = key.k, key.m_priv
    out = []
    for j in range(len(rs)):
        parts = []
        for h in hs:
            p = native.scalars_alloc(k)
            native.scalars_copy(p, 0, h, j * k, k)
            parts.append(p)
        x = native.scalars_alloc(mp)
        if mp:
            native.scalars_copy(x, 0, hrx, j * mp, mp)
        out.append(_proof_ints(dp.prove(key, *parts, Z, x, rs[j], ss[j])))
    return out


@pytest.mark.parametrize("precompute", [False, True])
@pytest.mark.parametrize("count", [1, 5, 64])
def test_device_prove_batch_equals_prove(native, precompute, count):
    from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
    k, mp = 64, 5
    key, Z = _device_key(native, k, mp, precompute)
    hs, hrx, rs, ss = _batch_inputs(native, k, mp, count, count)
    got = [_proof_ints(p) for p in dp.prove_batch(key, *hs, Z, hrx, rs, ss)]
    assert got == _single_proofs(native, key, Z, hs, hrx, rs, ss)


def test_prove_batch_chunks_and_quotient(native):
    from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
    k, mp, count = 32, 3, 20
    key, Z = _device_key(native, k, mp, True, seed=9)
    hs, hrx, rs, ss = _batch_inputs(native, k, mp, count, 77)
    whole, H = dp.prove_batch(key, *hs, Z, hrx, rs, ss, keep_quotient=True)
    assert dp.prove_batch(key, *hs, Z, hrx, rs, ss, chunk=7) == whole
    assert dp.prove_batch(key, *hs, Z, hrx, rs, ss, chunk=1000) == whole
    hq = native.groth16_quotient_batch_dev(*hs, k, count, Z, k + 1)
    assert native.scalars_download(H, 0, count * (k - 1)) == native.scalars_download(hq, 0, count * (k - 1))
    assert dp.prove_batch(key, *hs, Z, hrx, [], []) == []


def _golden_setup(native, case):
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd
    c = load("groth16_qap.json")["cases"][case]
    r1cs = qd.SparseR1CS.from_dense(c["r1cs_A"], c["r1cs_B"], c["r1cs_C"])
    dev = qd.DeviceR1CS(r1cs)
    t = {key: int(v) for key, v in c["toxic"].items()}
    keys = qd.setup(dev, t["alpha"], t["beta"], t["gamma"], t["delta"], t["x_val"], pub_r_indexs=c["pub_r_indexs"],
                    precompute=False)
    return c, dev, keys


@pytest.mark.parametrize("case", [0, 1])
def test_golden_proofs_inside_a_batch(native, case):
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd
    c, dev, keys = _golden_setup(native, case)
    m = dev.m
    rng = random.Random(case)
    gold = ints(c["witness"])
    others = [[1] + [rng.randrange(R) for _ in range(m - 1)] for _ in range(4)]
    ws = [gold] + others + [gold]
    r, s = int(c["r"]), int(c["s"])
    rs = [r] + [rng.randrange(R) for _ in others] + [r]
    ss = [s] + [rng.randrange(R) for _ in others] + [s]
    W = native.scalars_load(native.fr_vec_bytes([x for w in ws for x in w]), len(ws) * m)
    got = [_proof_ints(p) for p in qd.prove_batch(keys, dev, W, rs, ss)]
    want = (g1(c["proof_a"]), g2(c["proof_b"]), g1(c["proof_c"]))
    assert got[0] == want and got[-1] == want
    for j in range(1, len(ws) - 1):
        w = native.scalars_load(native.fr_vec_bytes(ws[j]), m)
        assert got[j] == _proof_ints(qd.prove(keys, dev, w, rs[j], ss[j]))


def _synthetic_witnesses(ra, rb, count, seed):
    """count satisfying witnesses of tools/qap_large.circuit's gates (w_{g+2} = (A_g . w)(B_g . w)) for random inputs."""
    rng = random.Random(seed)
    out = []
    for _ in range(count):
        w = [1, rng.randrange(2, 1 << 20)]
        for a, b in zip(ra, rb):
            w.append(sum(v * w[i] for i, v in a.items()) * sum(v * w[i] for i, v in b.items()) % R)
        out.append(w)
    return out


def test_synthetic_batch_end_to_end(native):
    import sys
    import os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from qap_large import circuit
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify_batch
    k, count = 1 << 12, 128
    m = k + 2
    ra, rb, rc, _ = circuit(k, 99)
    dev = qd.DeviceR1CS(qd.SparseR1CS.from_rows(k, m, ra, rb, rc))
    rng = random.Random(5)
    keys = qd.setup(dev, *(rng.randrange(1, R) for _ in range(5)), lcm=True, precompute=True)
    ws = _synthetic_witnesses(ra, rb, count, 11)
    rs = [rng.randrange(R) for _ in range(count)]
    ss = [rng.randrange(R) for _ in range(count)]
    W = native.scalars_load(native.fr_vec_bytes([x for w in ws for x in w]), count * m)
    proofs = qd.prove_batch(keys, dev, W, rs, ss)
    for j in (0, 1, count - 1):
        wj = native.scalars_load(native.fr_vec_bytes(ws[j]), m)
        assert _proof_ints(proofs[j]) == _proof_ints(qd.prove(keys, dev, wj, rs[j], ss[j]))
    vk = (keys.sigma1_1, keys.sigma1_3, keys.sigma2_1)
    pubs = [[(i, w[i]) for i in keys.pub_idx] for w in ws]
    assert verify_batch(proofs, *vk, pubs, rng=random.Random(1)) is True
    # one unsatisfying witness: a wire off by one
    bad = [list(w) for w in ws]
    bad[40][m // 2] = (bad[40][m // 2] + 1) % R
    Wb = native.scalars_load(native.fr_vec_bytes([x for w in bad for x in w]), count * m)
    bproofs = qd.prove_batch(keys, dev, Wb, rs, ss)
    assert _proof_ints(bproofs[0]) == _proof_ints(proofs[0])
    assert verify_batch(bproofs, *vk, pubs, rng=random.Random(2)) is False
    keep = [j for j in range(count) if j != 40]
    assert verify_batch([bproofs[j] for j in keep], *vk, [pubs[j] for j in keep], rng=random.Random(3)) is True


def test_launches_do_not_grow_with_count(native):
    from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
    k, mp = 64, 4
    key, Z = _device_key(native, k, mp, True, seed=21)
    counts = {}
    for count in (16, 256, 16, 256):                    # the first pair warms caches and workspaces
        hs, hrx, rs, ss = _batch_inputs(native, k, mp, count, count)
        before = native.launch_count()
        dp.prove_batch(key, *hs, Z, hrx, rs, ss)
        counts[count] = native.launch_count() - before
    assert counts[256] <= 1.25 * counts[16], counts


def test_refusals_leave_the_library_usable(native):
    from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
    t = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes([3, 5]), 2)
    native.table_precompute(t, 20)                       # W = 13 windows, 2^19 buckets per MSM
    sh = native.scalars_load(native.fr_vec_bytes([1, 2, 3, 4, 5]), 5)
    with pytest.raises(native.ZkpB200Error, match="2\\^32"):
        native.msm_dev_many(t, 0, 2, 1 << 28, sh, 0)       # 2^28 * 13 * 2 >= 2^32
    with pytest.raises(native.ZkpB200Error, match="2\\^31"):
        native.msm_dev_many(t, 0, 2, 1 << 12, sh, 0)       # 2^12 * 2^19 = 2^31
    with pytest.raises(native.ZkpB200Error, match="scalar range"):
        native.msm_dev_many(t, 0, 2, 3, sh, 0)             # 6 scalars from a handle of 5
    with pytest.raises(native.ZkpB200Error, match="point range"):
        native.msm_dev_many(t, 1, 2, 1, sh, 0)
    assert native.msm_dev_many(t, 0, 2, 0, sh, 0) == []
    assert native.msm_dev_many(t, 0, 0, 3, sh, 0) == [None, None, None]
    assert native.msm_dev_many(t, 0, 2, 2, sh, 1) == [native.g1_msm_dev(t, 0, sh, 1, 2), native.g1_msm_dev(t, 0, sh, 3, 2)]
    key, Z = _device_key(native, 8, 2, False, seed=4)
    hs, hrx, rs, ss = _batch_inputs(native, 8, 2, 3, 4)
    with pytest.raises(ValueError):
        dp.prove_batch(key, *hs, Z, hrx, rs, ss[:2])
    with pytest.raises(ValueError):
        dp.prove_batch(key, *hs, Z, hrx, rs + [1], ss + [1])
    assert len(dp.prove_batch(key, *hs, Z, hrx, rs, ss)) == 3
