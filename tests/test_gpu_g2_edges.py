"""-m gpu: the MSM paths where a bucket continues from, or adds up to, a sum equal to what is added to it, on G2 (whose
accumulation loop and fold have their own copies of the group law: csrc/msm_acc.cuh AccMul2, XYZZ<Fp2>) and on G1:
continuation across the parts of a part-streamed MSM, the host-scalar path at 2^18 with its default part count, the
many-vector MSM over equal points, and the split form msm_dev_begin / msm_dev_end.  Tables hold known discrete logs
(tests/msm_groups.py): the expected point is (sum k_i s_i mod r) * G."""
import random

import pytest

from oracle import bn254
from tests.msm_groups import Group, part_cuts

pytestmark = pytest.mark.gpu
R = bn254.R
GROUPS = ["g1", "g2"]


@pytest.fixture()
def opts(native):
    yield native
    native.msm_set_option("parts", 0)
    native.set_window_bits(0)


@pytest.mark.parametrize("group", GROUPS)
@pytest.mark.parametrize("k", [2, 3, 8])
@pytest.mark.parametrize("pre", [0, 9])
def test_parts_continue_equal_buckets(opts, group, k, pre):
    """Scalar 3 puts every entry it multiplies into one bucket of the lowest window.
    - first entries: part 0 holds two entries of discrete logs a and b (the bucket ends with ZZ != 1) and each later
      part p exactly one, 2^(p-1) (a + b) G, which equals the bucket carried over: the accumulation loop continues
      from the carried bucket and its mixed addition takes the P + P branch.
    - part sums: every later part's entries add up to the carried bucket (2^(p-1) S, S the sum of part 0) over
      several 64-entry tasks, so the fold's XYZZ addition of the carried bucket takes the P + P branch (block per
      bucket for the larger parts)."""
    native, grp = opts, Group(opts, group)
    rng = random.Random(7100 + 10 * k + pre + (group == "g2"))
    n = 4000
    cut = part_cuts(n, k)
    assert all(cut[p + 1] - cut[p] > 64 for p in range(k))
    dlogs = [rng.randrange(1, R) for _ in range(n)]
    a, b = dlogs[0], dlogs[1]
    for p in range(1, k):
        dlogs[cut[p]] = (a + b) << (p - 1)
    part_sum = lambda p: sum(dlogs[cut[p]:cut[p + 1]]) % R
    S = part_sum(0)
    for p in range(1, k):
        last = cut[p + 1] - 1
        dlogs[last] = (dlogs[last] + (S << (p - 1)) - part_sum(p)) % R
        assert part_sum(p) == (S << (p - 1)) % R
    table = grp.table(dlogs, spot=(0, 1, cut[1], -1))
    if pre:
        native.table_precompute(table, pre)
    first = [0] * n
    for i in [0, 1] + cut[1:k]:
        first[i] = 3
    cases = {"first entries": first, "part sums": [3] * n}
    native.msm_set_option("parts", k)
    for name, sc in cases.items():
        want = grp.want(dlogs, sc)
        assert grp.msm_table(table, 0, native.fr_vec_bytes(sc), n) == want, (name, "host scalars")
        h = native.scalars_load(native.fr_vec_bytes(sc), n)
        assert grp.msm_dev(table, 0, h, 0, n) == want, (name, "resident scalars")


@pytest.mark.parametrize("group", GROUPS)
def test_host_scalars_2p18_default_parts(opts, group):
    """The end-to-end entry point (scalars in host memory) at 2^18, where the engine streams 4 parts by default: all
    points equal under all scalars equal (one bucket per window, thousands of tasks in every part: the block-per-bucket
    fold with the carried bucket), and random discrete logs under random scalars; plain and precomputed tables."""
    native, grp = opts, Group(opts, group)
    native.msm_set_option("parts", 0)
    n = 1 << 18
    rng = random.Random(7200)
    s0, k0 = rng.randrange(1, R), rng.randrange(1, R)
    same_h = native.scalars_load(native.fr_vec_bytes([s0] * n), n)
    same = grp.table_dev(same_h, n, {0: s0, n - 1: s0})
    s_h = native.scalars_generate(0x5EED0700, n)
    k_h = native.scalars_generate(0x5EED0701, n)
    spot = {i: native.fr_vec_from_bytes(native.scalars_download(s_h, i, 1))[0] for i in (0, n - 1)}
    table = grp.table_dev(s_h, n, spot)
    k_host = native.scalars_download(k_h, 0, n)
    want = grp.mul(native.fr_dot_dev(k_h, 0, s_h, 0, n))
    want_same = grp.mul(n * s0 * k0)
    for pre in (0, 17):
        if pre:
            native.table_precompute(table, pre)
            native.table_precompute(same, pre)
        assert grp.msm_table(same, 0, native.fr_vec_bytes([k0]) * n, n) == want_same, pre
        assert grp.msm_table(table, 0, k_host, n) == want, pre


@pytest.mark.parametrize("group", GROUPS)
@pytest.mark.parametrize("pre", [0, 10])
def test_msm_dev_many_equal_points(native, group, pre):
    """One Pippenger pass over several scalar vectors (msm_dev_many) on a table of equal points: vector j all equal
    to k_j (P + P in the accumulation loop and the fold of every vector's bucket), one all zero, one mixing k and
    r - k (cancelling to infinity), one random."""
    grp = Group(native, group)
    rng = random.Random(7300 + pre)
    n = 300
    s0 = rng.randrange(1, R)
    table = grp.table([s0] * n)
    if pre:
        native.table_precompute(table, pre)
    ks = [rng.randrange(1, R) for _ in range(3)]
    vecs = [[k] * n for k in ks] + [[0] * n, [ks[0] if i % 2 else R - ks[0] for i in range(n)],
                                    [rng.randrange(R) for _ in range(n)]]
    h = native.scalars_load(native.fr_vec_bytes([x for v in vecs for x in v]), n * len(vecs))
    got = native.msm_dev_many(table, 0, n, len(vecs), h)
    assert got == [grp.mul(s0 * sum(v)) for v in vecs]
    assert got[3] is None and got[4] is None


@pytest.mark.parametrize("group", GROUPS)
def test_split_form_matches_synchronous(native, group):
    """msm_dev_begin enqueues an MSM on the library's second stream and returns; an MSM of each group issued on the
    main stream before msm_dev_end runs beside it.  All results equal the synchronous msm_dev and the expected point,
    for a plain and a precomputed table."""
    grp, other = Group(native, group), Group(native, "g2" if group == "g1" else "g1")
    rng = random.Random(7400 + (group == "g2"))
    n = 1000
    dlogs = [rng.randrange(1, R) for _ in range(n)]
    dlogs[5] = dlogs[4]                                          # an equal and an opposite pair under equal scalars
    dlogs[9] = R - dlogs[8]
    k = [rng.randrange(R) for _ in range(n)]
    k[5], k[9] = k[4], k[8]
    table = grp.table(dlogs)
    sc = native.scalars_load(native.fr_vec_bytes(k), n)
    want = grp.want(dlogs, k)
    o_dlogs = [rng.randrange(1, R) for _ in range(300)]
    o_k = [rng.randrange(R) for _ in range(300)]
    o_table, o_sc = other.table(o_dlogs), native.scalars_load(native.fr_vec_bytes(o_k), 300)
    same_k = [rng.randrange(R) for _ in range(n)]
    same_sc = native.scalars_load(native.fr_vec_bytes(same_k), n)
    for pre in (0, 12):
        if pre:
            native.table_precompute(table, pre)
        sync = grp.msm_dev(table, 0, sc, 0, n)
        assert sync == want
        native.msm_dev_begin(table, 0, sc, 0, n)
        assert other.msm_dev(o_table, 0, o_sc, 0, 300) == other.want(o_dlogs, o_k)
        assert grp.msm_dev(table, 0, same_sc, 0, n) == grp.want(dlogs, same_k)   # the same group on the main stream
        assert native.msm_dev_end(group) == sync
        native.msm_dev_begin(table, 100, sc, 3, 500)                            # a sub-range, nothing in between
        assert native.msm_dev_end(group) == grp.want(dlogs[100:600], k[3:503])
