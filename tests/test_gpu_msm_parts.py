"""-m gpu: the part-streamed MSM (MsmEngine::run with parts > 1: point ranges uploaded / sorted on a side lane while
the previous range accumulates, all ranges adding into one bucket set) against the oracle's commit()-style loop
(/root/reference/zkp/plonk/kzg.py:59-67): every part count, plain and window-precomputed tables, sub-ranges, host
and resident scalars, buckets that are continued / folded / left alone by a later part, G2, and the known-discrete-log
identity at 2^20 with the default part count of the host-scalar entry point."""
import random

import pytest

from oracle import bn254
from tests.msm_groups import Group, plus_minus

pytestmark = pytest.mark.gpu
R = bn254.R


@pytest.fixture()
def parts(native):
    yield native
    native.msm_set_option("parts", 0)
    native.set_window_bits(0)


def _points_g1(rng, n):
    base = [bn254.g1_mul(bn254.G1, rng.randrange(1, R)) for _ in range(4)]
    pts, acc = [], base[0]
    for i in range(n):
        acc = bn254.g1_add(acc, base[i % 4])
        pts.append(acc)
    return pts


@pytest.mark.parametrize("k", [2, 3, 5, 8])
@pytest.mark.parametrize("pre", [0, 6, 13])
def test_parts_match_oracle(parts, k, pre):
    rng = random.Random(2100 + 10 * k + pre)
    n = 400
    pts = _points_g1(rng, n)
    pts[11] = None
    scalars = [rng.randrange(R) for _ in range(n)]
    scalars[5] = 0
    scalars[399] = R - 1
    table = parts.g1_table_load(parts.g1_vec_bytes(pts), n)
    if pre:
        parts.table_precompute(table, pre)
    parts.msm_set_option("parts", k)
    want = bn254.g1_msm(pts, scalars)
    assert parts.g1_msm_table(table, 0, parts.fr_vec_bytes(scalars), n) == want          # host scalars
    sc = parts.scalars_load(parts.fr_vec_bytes(scalars), n)
    assert parts.g1_msm_dev(table, 0, sc, 0, n) == want                                  # resident scalars
    assert parts.g1_msm_dev(table, 37, sc, 11, 301) == bn254.g1_msm(pts[37:338], scalars[11:312])   # sub-range
    assert parts.g1_msm_table(table, 390, parts.fr_vec_bytes(scalars[:7]), 7) == bn254.g1_msm(pts[390:397], scalars[:7])
    p0 = parts.g1_msm_dev_partial(table, 0, sc, 0, 200)
    p1 = parts.g1_msm_dev_partial(table, 200, sc, 200, 200)
    assert parts.g1_combine_partials(p0 + p1, 2) == want


@pytest.mark.parametrize("c,group", [pytest.param(c, "g1", id=str(c)) for c in (3, 9)]
                         + [pytest.param(c, "g2", id="g2-%d" % c) for c in (3, 9)])
def test_parts_edge_distributions(parts, c, group):
    """One scalar for everything: every window has one bucket that each part cuts into several tasks (fold onto the
    earlier parts' sum); P / -P pairs that cancel across and inside parts; empty later parts (zero scalars).  G1
    against the oracle's MSM, G2 on known-discrete-log tables."""
    rng = random.Random(2200 + c)
    n = 600
    if group == "g2":
        _edge_distributions_dlog(parts, Group(parts, group), rng, c, n)
        return
    pts = _points_g1(rng, n)
    table = parts.g1_table_load(parts.g1_vec_bytes(pts), n)
    parts.set_window_bits(c)
    parts.msm_set_option("parts", 4)

    def check(tbl, p, s):
        assert parts.g1_msm_table(tbl, 0, parts.fr_vec_bytes(s), len(p)) == bn254.g1_msm(p, s)

    check(table, pts, [0x1234567] * n)
    check(table, pts, [1] * n)
    check(table, pts, [rng.randrange(R) for _ in range(150)] + [0] * 450)     # parts 1..3 add nothing
    check(table, pts, [0] * 450 + [rng.randrange(R) for _ in range(150)])     # only the last part adds
    check(table, pts, [0] * n)
    pm = []
    for i in range(n // 2):
        pm += [pts[i], bn254.g1_neg(pts[i])]
    t2 = parts.g1_table_load(parts.g1_vec_bytes(pm), n)
    check(t2, pm, [777] * n)
    half = pts[:300] + [bn254.g1_neg(p) for p in pts[:300]]                   # cancels across parts: buckets return to infinity
    t3 = parts.g1_table_load(parts.g1_vec_bytes(half), n)
    check(t3, half, [424242] * n)
    same = [pts[0]] * n                                                        # P + P when a later part continues a bucket
    t4 = parts.g1_table_load(parts.g1_vec_bytes(same), n)
    check(t4, same, [99] * n)


def _edge_distributions_dlog(native, grp, rng, c, n):
    native.set_window_bits(c)
    native.msm_set_option("parts", 4)
    base = [rng.randrange(1, R) for _ in range(n)]
    cases = [
        (base, [0x1234567] * n),
        (base, [1] * n),
        (base, [rng.randrange(R) for _ in range(150)] + [0] * 450),     # parts 1..3 add nothing
        (base, [0] * 450 + [rng.randrange(R) for _ in range(150)]),     # only the last part adds
        (base, [0] * n),
        (plus_minus(base[:n // 2]), [777] * n),
        (base[:300] + [R - s for s in base[:300]], [424242] * n),     # cancels across parts: buckets return to infinity
        ([base[0]] * n, [99] * n),                                     # P + P when a later part continues a bucket
    ]
    tables = {}
    for i, (dlogs, k) in enumerate(cases):
        if id(dlogs) not in tables:
            tables[id(dlogs)] = grp.table(dlogs)
        assert grp.msm_table(tables[id(dlogs)], 0, native.fr_vec_bytes(k), n) == grp.want(dlogs, k), i


def test_parts_g2(parts):
    rng = random.Random(2300)
    base = [bn254.g2_mul(bn254.G2, rng.randrange(1, 1 << 60)) for _ in range(3)]
    pts, acc = [], base[0]
    for i in range(90):
        acc = bn254.g2_add(acc, base[i % 3])
        pts.append(acc)
    scalars = [rng.randrange(R) for _ in range(90)]
    table = parts.g2_table_load(parts.g2_vec_bytes(pts), 90)
    want = bn254.g2_msm(pts, scalars)
    for k in (3, 8):
        parts.msm_set_option("parts", k)
        assert parts.g2_msm_table(table, 0, parts.fr_vec_bytes(scalars), 90) == want
    parts.table_precompute(table, 7)
    assert parts.g2_msm_table(table, 0, parts.fr_vec_bytes(scalars), 90) == want


@pytest.mark.parametrize("k", [0, 1, 2, 8])
def test_parts_2_20_known_dlog(parts, k):
    """BASELINE configs[1] through the end-to-end entry point (zkp_g1_msm_table: scalars in host memory), default and
    explicit part counts; result == <k, s> G with the dot product taken on the device."""
    n = 1 << 20
    s_h = parts.scalars_generate(0x5EED0002, n)
    k_h = parts.scalars_generate(0x5EED0001, n)
    table = parts.g1_fixed_base_mul_dev(parts.g1_bytes(bn254.G1), s_h, n)
    parts.table_precompute(table)
    want = bn254.g1_mul(bn254.G1, parts.fr_dot_dev(k_h, 0, s_h, 0, n))
    host = parts.scalars_download(k_h, 0, n)
    parts.msm_set_option("parts", k)
    assert parts.g1_msm_table(table, 0, host, n) == want
    assert parts.g1_msm_dev(table, 0, k_h, 0, n) == want
    third = n // 3
    want3 = bn254.g1_mul(bn254.G1, parts.fr_dot_dev(k_h, 0, s_h, third, third))
    assert parts.g1_msm_table(table, third, host[:32 * third], third) == want3
