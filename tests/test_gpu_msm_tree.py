"""-m gpu: the affine-tree bucket accumulation (csrc/msm_tree.cuh) forced on for every MSM, bit-exact against the
oracle's commit()-style loop (/root/reference/zkp/plonk/kzg.py:59-67) and against the XYZZ accumulation of the
same library: every window width (1 .. 9 tree rounds), the edge distributions (infinity entries, P + P and
P + (-P) inside a bucket, one bucket holding everything = the heavy path beside the tree), G2, window-precomputed
tables, sub-ranges, and the known-discrete-log identity at 2^16 .. 2^20."""
import random

import pytest

from oracle import bn254, synthetic
from tests.msm_groups import Group, auto_c, edge_cases

pytestmark = pytest.mark.gpu
R = bn254.R


@pytest.fixture()
def tree(native):
    native.msm_set_option("accumulate", 2)
    yield native
    native.msm_set_option("accumulate", 0)
    native.msm_set_option("tree_items", 0)
    native.msm_set_option("tree_rounds", 0)
    native.set_window_bits(0)


def _points_g1(rng, n):
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
def test_tree_g1_random(tree, n):
    rng = random.Random(1100 + n)
    pts = _points_g1(rng, n)
    _check_g1(tree, pts, [rng.randrange(R) for _ in range(n)])


@pytest.mark.parametrize("c", [2, 3, 5, 9, 13, 16, 20])
@pytest.mark.parametrize("items,rounds", [(0, 0), (2, 1), (5, 3), (16, 9), (8, 9)])
def test_tree_every_window_width_and_batch(tree, c, items, rounds):
    """c = 2 puts ~110 entries into each bucket (7 rounds when the tree runs to the end, chains of 28 after the
    default 2 rounds), c = 20 at most one (copies only); `items` varies the number of additions per thread under one
    inversion (block boundaries fall elsewhere), `rounds` where the XYZZ chains take over."""
    rng = random.Random(1200 + c)
    pts = _points_g1(rng, 300)
    scalars = [rng.randrange(R) for _ in range(300)]
    tree.set_window_bits(c)
    tree.msm_set_option("tree_items", items)
    tree.msm_set_option("tree_rounds", rounds)
    _check_g1(tree, pts, scalars)


def test_tree_edge_distributions(tree):
    """G1 against the oracle's MSM, then over known-discrete-log tables (tests/msm_groups.py edge_cases, shared with
    the G2 test below) in the default and in the late tree rounds."""
    rng = random.Random(15)
    n = 200
    pts = _points_g1(rng, n)
    _check_g1(tree, pts, [0] * n)
    _check_g1(tree, pts, [1] * n)
    _check_g1(tree, pts, [R - 1] * n)
    _check_g1(tree, pts, [rng.randrange(R) if i % 2 else 0 for i in range(n)])
    _check_g1(tree, [pts[0]] * n, [rng.randrange(R) for _ in range(n)])   # all points equal: P + P in the pairs
    _check_g1(tree, [pts[0]] * n, [12345] * n)                            # one bucket, doublings all the way up
    pm = []
    for i in range(n // 2):
        pm += [pts[i], bn254.g1_neg(pts[i])]
    _check_g1(tree, pm, [777] * n)                                        # P + (-P) pairs -> infinity inside the tree
    _check_g1(tree, pm, [777 if i % 2 == 0 else R - 777 for i in range(n)])   # signs make them equal again
    _check_g1(tree, pts, [(1 << 255) + 5, R, R + 1, 2 * R + 3] + [1] * (n - 4))
    with_inf = list(pts)
    with_inf[3] = None
    with_inf[77] = None
    with_inf[78] = None
    _check_g1(tree, with_inf, [rng.randrange(R) for _ in range(n)])
    _check_g1(tree, with_inf, [5] * n)                                    # infinity entries inside one bucket
    _check_g1(tree, pts, [(1 << 16) - 1] * n)
    _check_g1(tree, pts, [1 << 15] * n)
    tree.msm_set_option("tree_rounds", 9)                                 # the same special cases in the late rounds
    _check_g1(tree, [pts[0]] * n, [12345] * n)
    _check_g1(tree, pm, [777] * n)
    _check_g1(tree, with_inf, [5] * n)
    tree.msm_set_option("tree_rounds", 0)
    _edge_cases_dlog(tree, Group(tree, "g1"), rng)


def test_tree_g2_edge_distributions(tree):
    _edge_cases_dlog(tree, Group(tree, "g2"), random.Random(15))


def _edge_cases_dlog(native, grp, rng, n=256):
    cases = edge_cases(rng, n, auto_c(n))
    tables = {}
    for rounds in (0, 9):
        native.msm_set_option("tree_rounds", rounds)
        for name, dlogs, k in cases:
            if id(dlogs) not in tables:
                tables[id(dlogs)] = grp.table(dlogs)
            assert grp.msm_points(tables[id(dlogs)], n, k) == grp.want(dlogs, k), (name, rounds)


def test_tree_and_heavy_buckets_side_by_side(tree):
    """700 equal scalars fill one bucket per window beyond the tree's 511-entry range (XYZZ tasks + fold) while the
    other 500 points spread over light buckets; also exactly 511 and 512 entries."""
    rng = random.Random(16)
    n = 1200
    pts = _points_g1(rng, n)
    for heavy in (700, 511, 512):
        scalars = [0x1234567] * heavy + [rng.randrange(R) for _ in range(n - heavy)]
        for c in (4, 12):
            tree.set_window_bits(c)
            _check_g1(tree, pts, scalars)


@pytest.mark.parametrize("n", [1, 5, 64, 300])
def test_tree_g2_random(tree, n):
    rng = random.Random(1300 + n)
    base = [bn254.g2_mul(bn254.G2, rng.randrange(1, 1 << 60)) for _ in range(3)]
    pts, acc = [], base[0]
    for i in range(n):
        acc = bn254.g2_add(acc, base[i % 3])
        pts.append(acc)
    scalars = [rng.randrange(R) for _ in range(n)]
    if n > 4:
        scalars[2] = 0
        pts[4] = None
    if n > 6:
        pts[6] = pts[5]
        scalars[6] = scalars[5]
    want = bn254.g2_msm(pts, scalars)
    for c, rounds in ((0, 0), (3, 0), (3, 9)):
        tree.set_window_bits(c)
        tree.msm_set_option("tree_rounds", rounds)
        assert tree.g2_msm(tree.g2_vec_bytes(pts), tree.fr_vec_bytes(scalars), n) == want


@pytest.mark.parametrize("c", [4, 7, 12, 16])
def test_tree_precomputed_table(tree, c):
    rng = random.Random(1400 + c)
    n = 300
    pts = _points_g1(rng, n)
    pts[17] = None
    scalars = [rng.randrange(R) for _ in range(n)]
    scalars[3] = 0
    scalars[4] = R - 1
    table = tree.g1_table_load(tree.g1_vec_bytes(pts), n)
    tree.table_precompute(table, c)
    assert tree.g1_msm_table(table, 0, tree.fr_vec_bytes(scalars), n) == bn254.g1_msm(pts, scalars)
    assert tree.g1_msm_table(table, 50, tree.fr_vec_bytes(scalars[:120]), 120) == bn254.g1_msm(pts[50:170], scalars[:120])
    sc = tree.scalars_load(tree.fr_vec_bytes(scalars), n)
    assert tree.g1_msm_dev(table, 100, sc, 7, 150) == bn254.g1_msm(pts[100:250], scalars[7:157])
    p0 = tree.g1_msm_dev_partial(table, 0, sc, 0, 150)
    p1 = tree.g1_msm_dev_partial(table, 150, sc, 150, 150)
    assert tree.g1_combine_partials(p0 + p1, 2) == bn254.g1_msm(pts, scalars)
    assert tree.g1_msm_table(table, 0, tree.fr_vec_bytes([0] * n), n) is None


@pytest.mark.parametrize("log_n,pre", [(16, 0), (16, 13), (18, 16), (20, 0), (20, 20)])
def test_tree_full_size_known_dlog(tree, log_n, pre):
    """P_i = s_i G generated on the device: result == <k, s> G, and == the XYZZ accumulation's result; the same for
    a sub-range and for skewed scalars (all small: a few crowded buckets)."""
    n = 1 << log_n
    s_h = tree.scalars_generate(0x5EED0002, n)
    k_h = tree.scalars_generate(0x5EED0001, n)
    table = tree.g1_fixed_base_mul_dev(tree.g1_bytes(bn254.G1), s_h, n)
    if pre:
        tree.table_precompute(table, pre)
    dot = tree.fr_dot_dev(k_h, 0, s_h, 0, n)
    want = bn254.g1_mul(bn254.G1, dot)
    assert tree.g1_msm_dev(table, 0, k_h, 0, n) == want
    tree.msm_set_option("accumulate", 1)
    assert tree.g1_msm_dev(table, 0, k_h, 0, n) == want
    tree.msm_set_option("accumulate", 2)
    third = n // 3
    dot = tree.fr_dot_dev(k_h, 5, s_h, third, third)
    assert tree.g1_msm_dev(table, third, k_h, 5, third) == bn254.g1_mul(bn254.G1, dot)
    if log_n <= 16:
        small = [(i * 7919) % 1000 for i in range(n)]
        sm_h = tree.scalars_load(tree.fr_vec_bytes(small), n)
        dot = tree.fr_dot_dev(sm_h, 0, s_h, 0, n)
        assert tree.g1_msm_dev(table, 0, sm_h, 0, n) == bn254.g1_mul(bn254.G1, dot)


def test_tree_g2_known_dlog_2_14(tree):
    n = 1 << 14
    s_h = tree.scalars_generate(0x5EED0003, n)
    k_h = tree.scalars_generate(0x5EED0001, n)
    table = tree.g2_fixed_base_mul_dev(tree.g2_bytes(bn254.G2), s_h, n)
    s = synthetic.scalars(0x5EED0003, n)
    k = synthetic.scalars(0x5EED0001, n)
    want = bn254.g2_mul(bn254.G2, sum(a * b for a, b in zip(k, s)) % R)
    assert tree.g2_msm_dev(table, 0, k_h, 0, n) == want
    tree.table_precompute(table, 11)
    assert tree.g2_msm_dev(table, 0, k_h, 0, n) == want
