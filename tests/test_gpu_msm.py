"""-m gpu: G1 / G2 MSM through the C ABI, bit-exact against the oracle's commit()-style loop
(/root/reference/zkp/plonk/kzg.py:59-67) at sizes the oracle finishes in seconds, plus the edge
distributions of SURVEY.md 8(d) and the size-independent check result == (sum k_i s_i) * G at the
BASELINE sizes (points with known discrete logs generated on the device)."""
import random

import pytest

from oracle import bn254, synthetic
from tests.msm_groups import Group, auto_c, edge_cases

pytestmark = pytest.mark.gpu
R = bn254.R


def _points_g1(rng, n):
    # cheap distinct points: running sums of a few random multiples
    base = [bn254.g1_mul(bn254.G1, rng.randrange(1, R)) for _ in range(4)]
    pts, acc = [], base[0]
    for i in range(n):
        acc = bn254.g1_add(acc, base[i % 4])
        pts.append(acc)
    return pts


def _check_g1(native, pts, scalars):
    got = native.g1_msm(native.g1_vec_bytes(pts), native.fr_vec_bytes(scalars), len(pts))
    assert got == bn254.g1_msm(pts, scalars)


@pytest.mark.parametrize("n", [1, 2, 3, 4, 7, 33, 257, 1024])
def test_g1_msm_random(native, n):
    rng = random.Random(100 + n)
    pts = _points_g1(rng, n)
    scalars = [rng.randrange(R) for _ in range(n)]
    _check_g1(native, pts, scalars)


def test_g1_msm_empty_is_infinity(native):
    assert native.g1_msm(b"", b"", 0) is None


@pytest.mark.parametrize("c,group", [pytest.param(c, "g1", id=str(c)) for c in (2, 3, 5, 9, 13, 14, 16, 18, 20)]
                         + [pytest.param(c, "g2", id="g2-%d" % c) for c in (2, 3, 5, 9, 13, 16, 18, 20)])
def test_g1_msm_every_window_width(native, c, group):
    """Every window width on G1 and G2, plain and window-precomputed tables, with a repeated point and a P / -P pair
    under equal scalars in the data (P + P and P + (-P) inside a bucket at every width)."""
    rng = random.Random(200 + c)
    grp = Group(native, group)
    n = 300 if group == "g1" else 200
    # a plain table's MSM holds ceil(255 / c) windows of 2^(c-1) XYZZ buckets (twice the affine size: 256 B on G2),
    # 1.7 GB for G2 at c = 20
    free, _ = native.device_mem_info()
    assert free > 4 * ((255 + c - 1) // c) * (1 << (c - 1)) * 2 * grp.size
    try:
        native.set_window_bits(c)
        if group == "g1":
            pts = _points_g1(rng, 300)
            scalars = [rng.randrange(R) for _ in range(300)]
            _check_g1(native, pts, scalars)
        dlogs = [rng.randrange(1, R) for _ in range(n)]
        dlogs[7] = dlogs[3]
        dlogs[11] = R - dlogs[10]
        dlogs[n - 1] = dlogs[0]
        k = [rng.randrange(R) for _ in range(n)]
        k[7] = k[3]
        k[11] = k[10]
        k[n - 1] = k[0] = R - 1
        want = grp.want(dlogs, k)
        table = grp.table(dlogs)
        assert grp.msm_points(table, n, k) == want
        assert grp.msm_table(table, 0, native.fr_vec_bytes(k), n) == want
        native.set_window_bits(0)
        assert native.table_precompute(table, c) == c
        assert grp.msm_table(table, 0, native.fr_vec_bytes(k), n) == want
        sc = native.scalars_load(native.fr_vec_bytes(k), n)
        assert grp.msm_dev(table, 0, sc, 0, n) == want
    finally:
        native.set_window_bits(0)


def test_g1_msm_edge_distributions(native):
    """The edge distributions on G1 against the oracle's MSM, then at the window width the engine picks over
    known-discrete-log tables (tests/msm_groups.py edge_cases, shared with the G2 test below): P + P in the
    accumulation loop and in the fold, P + (-P), infinity entries, unreduced scalars, digits that carry in every
    window."""
    rng = random.Random(5)
    n = 200
    pts = _points_g1(rng, n)
    _check_g1(native, pts, [0] * n)                                   # all zero -> infinity
    _check_g1(native, pts, [1] * n)                                   # all one
    _check_g1(native, pts, [R - 1] * n)                               # all r-1
    _check_g1(native, pts, [rng.randrange(R) if i % 2 else 0 for i in range(n)])  # 50% zeros
    _check_g1(native, [pts[0]] * n, [rng.randrange(R) for _ in range(n)])        # all points equal
    _check_g1(native, [pts[0]] * n, [12345] * n)                      # same point, same scalar (P+P in buckets)
    pm = []
    for i in range(n // 2):
        pm += [pts[i], bn254.g1_neg(pts[i])]
    _check_g1(native, pm, [777] * n)                                  # P / -P pairs -> infinity
    _check_g1(native, pts, [(1 << 255) + 5, R, R + 1, 2 * R + 3] + [1] * (n - 4))  # unreduced scalars
    with_inf = list(pts)
    with_inf[3] = None
    with_inf[77] = None
    _check_g1(native, with_inf, [rng.randrange(R) for _ in range(n)])  # infinity points in the table
    _check_g1(native, pts, [(1 << 16) - 1] * n)                        # digit carries
    _check_g1(native, pts, [1 << 15] * n)                              # digit == B exactly
    _check_edge_cases(native, Group(native, "g1"), rng, 256)


def test_g2_msm_edge_distributions(native):
    """The edge distributions of the G1 test above on G2, whose accumulation loop (AccMul2) and fold have their own
    copies of the group law."""
    _check_edge_cases(native, Group(native, "g2"), random.Random(5), 256)


def _check_edge_cases(native, grp, rng, n):
    tables = {}
    for name, dlogs, k in edge_cases(rng, n, auto_c(n)):
        key = id(dlogs)
        if key not in tables:
            tables[key] = grp.table(dlogs)
        assert grp.msm_points(tables[key], n, k) == grp.want(dlogs, k), name


def test_g1_msm_table_and_dev_paths_agree(native):
    rng = random.Random(9)
    n = 500
    pts = _points_g1(rng, n)
    scalars = [rng.randrange(R) for _ in range(n)]
    want = bn254.g1_msm(pts[100:400], scalars[:300])
    table = native.g1_table_load(native.g1_vec_bytes(pts), n)
    assert native.g1_msm_table(table, 100, native.fr_vec_bytes(scalars[:300]), 300) == want
    sc = native.scalars_load(native.fr_vec_bytes(scalars), n)
    assert native.g1_msm_dev(table, 100, sc, 0, 300) == want
    # shard form: two partial sums combined == whole
    p0 = native.g1_msm_dev_partial(table, 100, sc, 0, 150)
    p1 = native.g1_msm_dev_partial(table, 250, sc, 150, 150)
    assert native.g1_combine_partials(p0 + p1, 2) == want
    back = native.table_download(table, 0, n)
    assert [native.g1_from_bytes(back[64 * i:64 * i + 64]) for i in range(n)] == pts


@pytest.mark.parametrize("n", [1, 5, 64, 300])
def test_g2_msm_random(native, n):
    rng = random.Random(300 + n)
    base = [bn254.g2_mul(bn254.G2, rng.randrange(1, 1 << 60)) for _ in range(3)]
    pts, acc = [], base[0]
    for i in range(n):
        acc = bn254.g2_add(acc, base[i % 3])
        pts.append(acc)
    scalars = [rng.randrange(R) for _ in range(n)]
    if n > 4:
        scalars[2] = 0
        pts[4] = None
    got = native.g2_msm(native.g2_vec_bytes(pts), native.fr_vec_bytes(scalars), n)
    assert got == bn254.g2_msm(pts, scalars)


def test_fixed_base_mul_matches_oracle(native):
    rng = random.Random(11)
    scalars = [0, 1, 2, R - 1, R, R + 5] + [rng.randrange(R) for _ in range(60)]
    t = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes(scalars), len(scalars))
    back = native.table_download(t, 0, len(scalars))
    got = [native.g1_from_bytes(back[64 * i:64 * i + 64]) for i in range(len(scalars))]
    assert got == [bn254.g1_mul(bn254.G1, s % R) for s in scalars]
    sc2 = scalars[:12]
    t2 = native.g2_fixed_base_mul(native.g2_bytes(bn254.G2), native.fr_vec_bytes(sc2), len(sc2))
    back = native.table_download(t2, 0, len(sc2))
    got = [native.g2_from_bytes(back[128 * i:128 * i + 128]) for i in range(len(sc2))]
    assert got == [bn254.g2_mul(bn254.G2, s % R) for s in sc2]


def test_synthetic_scalar_stream_matches_oracle(native):
    h = native.scalars_generate(0x5EED0001, 5000)
    got = native.fr_vec_from_bytes(native.scalars_download(h, 0, 5000))
    assert got == synthetic.scalars(0x5EED0001, 5000)


@pytest.mark.parametrize("log_n", [16, 20])
def test_g1_msm_full_size_known_dlog(native, log_n):
    """BASELINE config 2 sizes: P_i = s_i*G generated on the device, so the MSM has the O(n) check
    result == (sum k_i*s_i mod r)*G (one oracle scalar multiplication)."""
    n = 1 << log_n
    s_h = native.scalars_generate(0x5EED0002, n)
    k_h = native.scalars_generate(0x5EED0001, n)
    table = native.g1_fixed_base_mul_dev(native.g1_bytes(bn254.G1), s_h, n)
    # spot-check generated points against the oracle
    s = synthetic.scalars(0x5EED0002, n)
    k = synthetic.scalars(0x5EED0001, n)
    for i in (0, 1, n // 3, n - 1):
        assert native.g1_from_bytes(native.table_download(table, i, 1)) == bn254.g1_mul(bn254.G1, s[i])
    got = native.g1_msm_dev(table, 0, k_h, 0, n)
    total = sum(a * b for a, b in zip(k, s)) % R
    assert got == bn254.g1_mul(bn254.G1, total)


@pytest.mark.parametrize("c", [4, 7, 12, 14, 16, 19])
def test_precomputed_table_matches_plain(native, c):
    """Window-precomputed tables (zkp_g1_table_precompute) give the same affine point as the oracle,
    for whole-table and sub-range MSMs, host and device scalars, incl. infinity entries."""
    rng = random.Random(400 + c)
    n = 300
    pts = _points_g1(rng, n)
    pts[17] = None
    scalars = [rng.randrange(R) for _ in range(n)]
    scalars[3] = 0
    scalars[4] = R - 1
    table = native.g1_table_load(native.g1_vec_bytes(pts), n)
    native.table_precompute(table, c)
    assert native.g1_msm_table(table, 0, native.fr_vec_bytes(scalars), n) == bn254.g1_msm(pts, scalars)
    assert native.g1_msm_table(table, 50, native.fr_vec_bytes(scalars[:120]), 120) == bn254.g1_msm(pts[50:170], scalars[:120])
    sc = native.scalars_load(native.fr_vec_bytes(scalars), n)
    assert native.g1_msm_dev(table, 100, sc, 7, 150) == bn254.g1_msm(pts[100:250], scalars[7:157])
    p0 = native.g1_msm_dev_partial(table, 0, sc, 0, 150)
    p1 = native.g1_msm_dev_partial(table, 150, sc, 150, 150)
    assert native.g1_combine_partials(p0 + p1, 2) == bn254.g1_msm(pts, scalars)
    back = native.table_download(table, 0, n)     # window 0 is the plain table
    assert [native.g1_from_bytes(back[64 * i:64 * i + 64]) for i in range(n)] == pts
    assert native.g1_msm_table(table, 0, native.fr_vec_bytes([0] * n), n) is None


def test_precomputed_g2_table(native):
    rng = random.Random(55)
    base = [bn254.g2_mul(bn254.G2, rng.randrange(1, 1 << 60)) for _ in range(3)]
    pts, acc = [], base[0]
    for i in range(40):
        acc = bn254.g2_add(acc, base[i % 3])
        pts.append(acc)
    scalars = [rng.randrange(R) for _ in range(40)]
    table = native.g2_table_load(native.g2_vec_bytes(pts), 40)
    native.table_precompute(table, 8)
    assert native.g2_msm_table(table, 0, native.fr_vec_bytes(scalars), 40) == bn254.g2_msm(pts, scalars)


def test_precomputed_full_size_known_dlog(native):
    n = 1 << 18
    s_h = native.scalars_generate(0x5EED0002, n)
    k_h = native.scalars_generate(0x5EED0001, n)
    table = native.g1_fixed_base_mul_dev(native.g1_bytes(bn254.G1), s_h, n)
    plain = native.g1_msm_dev(table, 0, k_h, 0, n)
    native.table_precompute(table, 16)
    s = synthetic.scalars(0x5EED0002, n)
    k = synthetic.scalars(0x5EED0001, n)
    want = bn254.g1_mul(bn254.G1, sum(a * b for a, b in zip(k, s)) % R)
    assert plain == want
    assert native.g1_msm_dev(table, 0, k_h, 0, n) == want
    half = n // 2
    want_half = bn254.g1_mul(bn254.G1, sum(a * b for a, b in zip(k[:half], s[half:])) % R)
    assert native.g1_msm_dev(table, half, k_h, 0, half) == want_half


def test_batched_msm_matches_individual_calls(native):
    """zkp_g1_msm_dev_batch (two-stream pipeline) == the same MSMs issued one by one, for plain and
    window-precomputed tables, mixed sizes, offsets, an empty MSM and an all-zero scalar vector."""
    rng = random.Random(808)
    n = 700
    pts = _points_g1(rng, n)
    table = native.g1_table_load(native.g1_vec_bytes(pts), n)
    vecs = [[rng.randrange(R) for _ in range(n)] for _ in range(3)] + [[0] * n]
    hs = [native.scalars_load(native.fr_vec_bytes(v), n) for v in vecs]
    items = [(hs[0], 0, 0, n), (hs[1], 5, 100, 300), (hs[2], 0, 699, 1), (hs[3], 0, 0, n), (hs[0], 10, 20, 0),
             (hs[1], 0, 0, 650), (hs[2], 100, 0, 600)]
    want = [bn254.g1_msm(pts[off:off + m], vecs[hs.index(h)][so:so + m]) for h, so, off, m in items]
    assert native.g1_msm_dev_batch(table, items) == want
    native.table_precompute(table, 7)
    assert native.g1_msm_dev_batch(table, items) == want
    assert native.g1_msm_dev_batch(table, []) == []
    assert native.g1_msm_dev(table, 0, hs[0], 0, n) == want[0]          # single-call path still fine afterwards


@pytest.mark.parametrize("precompute", [0, 11])
def test_g2_msm_known_dlog_2_14(native, precompute):
    """G2 at 2^14 points (Q_i = s_i * G2 generated on the device): result == (sum k_i s_i) * G2."""
    n = 1 << 14
    s_h = native.scalars_generate(0x5EED0003, n)
    k_h = native.scalars_generate(0x5EED0001, n)
    table = native.g2_fixed_base_mul_dev(native.g2_bytes(bn254.G2), s_h, n)
    s = synthetic.scalars(0x5EED0003, n)
    k = synthetic.scalars(0x5EED0001, n)
    for i in (0, 4097, n - 1):
        assert native.g2_from_bytes(native.table_download(table, i, 1)) == bn254.g2_mul(bn254.G2, s[i])
    if precompute:
        native.table_precompute(table, precompute)
    want = bn254.g2_mul(bn254.G2, sum(a * b for a, b in zip(k, s)) % R)
    assert native.g2_msm_dev(table, 0, k_h, 0, n) == want
    half = n // 2
    want_half = bn254.g2_mul(bn254.G2, sum(a * b for a, b in zip(k[:half], s[half:])) % R)
    assert native.g2_msm_dev(table, half, k_h, 0, half) == want_half


def test_partial_wire_format(native):
    """The 128-byte shard partial decodes (x/zz, y/zzz out of Montgomery form) to the oracle's partial sum,
    and partials of two half ranges fold to the whole MSM."""
    rng = random.Random(77)
    n = 200
    pts = _points_g1(rng, n)
    scalars = [rng.randrange(R) for _ in range(n)]
    want = bn254.g1_msm(pts, scalars)
    table = native.g1_table_load(native.g1_vec_bytes(pts), n)
    sc = native.scalars_load(native.fr_vec_bytes(scalars), n)
    raw = native.g1_msm_dev_partial(table, 0, sc, 0, n)
    rinv = pow(1 << 256, -1, bn254.P)
    x, y, zz, zzz = (int.from_bytes(raw[32 * i:32 * i + 32], "little") * rinv % bn254.P for i in range(4))
    assert (x * pow(zz, -1, bn254.P) % bn254.P, y * pow(zzz, -1, bn254.P) % bn254.P) == want
    assert pow(zz, 3, bn254.P) == pow(zzz, 2, bn254.P)
    two = native.g1_msm_dev_partial(table, 0, sc, 0, 100) + native.g1_msm_dev_partial(table, 100, sc, 100, 100)
    assert native.g1_combine_partials(two, 2) == want


@pytest.mark.parametrize("n,want_c", [(5, 7), (40, 10), (300, 13), (5000, 15)])
def test_automatic_window_width(native, n, want_c):
    """window_bits = 0: the library picks the width for the table size (msm_auto_precomputed_c) and the MSM
    on the precomputed table still equals the oracle's sum, whole table and sub-range."""
    rng = random.Random(n)
    base = [bn254.g1_mul(bn254.G1, rng.randrange(1, R)) for _ in range(4)]
    pts, acc = [], base[0]
    for i in range(n):
        acc = bn254.g1_add(acc, base[i % 4])
        pts.append(acc)
    scalars = [rng.randrange(R) for _ in range(n)]
    table = native.g1_table_load(native.g1_vec_bytes(pts), n)
    assert native.table_precompute(table) == want_c and table.pre_c == want_c
    m = min(n, 200)                      # the oracle's double-and-add loop is slow: check a sub-range of large tables
    off = n - m
    assert native.g1_msm_table(table, off, native.fr_vec_bytes(scalars[:m]), m) == bn254.g1_msm(pts[off:], scalars[:m])
    if n <= 300:
        assert native.g1_msm_table(table, 0, native.fr_vec_bytes(scalars), n) == bn254.g1_msm(pts, scalars)


def test_groth16_three_msms_overlapped(native):
    """zkp_groth16_msms_dev: G1, G2, G1 results equal the three separate calls (and the oracle)."""
    rng = random.Random(91)
    n1, n2, n3 = 70, 33, 150
    p1, p3 = _points_g1(rng, n1), _points_g1(rng, n3)
    g2b = [bn254.g2_mul(bn254.G2, rng.randrange(1, 1 << 64)) for _ in range(3)]
    p2, acc = [], g2b[0]
    for i in range(n2):
        acc = bn254.g2_add(acc, g2b[i % 3])
        p2.append(acc)
    s1, s2, s3 = ([rng.randrange(R) for _ in range(k)] for k in (n1, n2, n3))
    ta = native.g1_table_load(native.g1_vec_bytes(p1), n1)
    tb = native.g2_table_load(native.g2_vec_bytes(p2), n2)
    tc = native.g1_table_load(native.g1_vec_bytes(p3), n3)
    native.table_precompute(tc)                                     # mixed plain / precomputed tables
    ha, hb, hc = (native.scalars_load(native.fr_vec_bytes(s), len(s)) for s in (s1, s2, s3))
    A, B, C = native.groth16_msms_dev(ta, ha, n1, tb, hb, n2, tc, hc, n3)
    assert A == bn254.g1_msm(p1, s1) and B == bn254.g2_msm(p2, s2) and C == bn254.g1_msm(p3, s3)
    zero = native.scalars_alloc(n2)
    assert native.groth16_msms_dev(ta, ha, n1, tb, zero, n2, tc, hc, n3)[1] is None     # infinity in the G2 slot


def test_latency_probes_run(native):
    """Diagnostics (include/zkp_b200_diag.h) stay callable: single-thread / quad latencies are positive."""
    for mode in (0, 3, 8, 9):
        assert native.latency_probe(mode) > 0
