"""CPU: argument validation of the batch provers (refused before any device call) and the chunk planning of
device_prover.prove_batch, which is host arithmetic."""
import pytest

from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd


class _H:
    """Stands in for a device handle: only its length is read before the first device call."""

    def __init__(self, n, kind="fr", pre_c=0):
        self.n, self.kind, self.pre_c = n, kind, pre_c


def _key(k, mp, pre=0):
    n_ab, n_c = k + 2, dp.tc_rows(k, mp)
    return dp.DeviceKey(k, mp, _H(n_ab, "g1", pre), _H(n_ab, "g2", pre), _H(n_c, "g1", pre))


def _args(k, mp, count):
    return [_H(count * k), _H(count * k), _H(count * k), _H(k + 1), _H(count * mp)]


def test_prove_batch_refuses_bad_shapes_before_any_device_call():
    key = _key(16, 3)
    uA, uB, uC, Z, rx = _args(16, 3, 4)
    rs = ss = [1, 2, 3, 4]
    with pytest.raises(ValueError, match="differ"):
        dp.prove_batch(key, uA, uB, uC, Z, rx, rs, ss[:3])
    with pytest.raises(ValueError, match="uB"):
        dp.prove_batch(key, uA, _H(63), uC, Z, rx, rs, ss)
    with pytest.raises(ValueError, match="rx_priv"):
        dp.prove_batch(key, uA, uB, uC, Z, _H(11), rs, ss)
    with pytest.raises(ValueError, match="Z"):
        dp.prove_batch(key, uA, uB, uC, _H(16), rx, rs, ss)
    for bad in (0, -3):
        with pytest.raises(ValueError, match="chunk"):
            dp.prove_batch(key, uA, uB, uC, Z, rx, rs, ss, chunk=bad)
    assert dp.prove_batch(key, uA, uB, uC, Z, rx, [], []) == []


def test_qap_prove_batch_refuses_bad_shapes():
    class Dev:
        k, m = 8, 10
    with pytest.raises(ValueError, match="differ"):
        qd.prove_batch(None, Dev, _H(30), [1, 2, 3], [1, 2])
    with pytest.raises(ValueError, match="W holds"):
        qd.prove_batch(None, Dev, _H(29), [1, 2, 3], [1, 2, 3])
    with pytest.raises(ValueError, match="chunk"):
        qd.prove_batch(None, Dev, _H(30), [1, 2, 3], [1, 2, 3], chunk=0)
    assert qd.prove_batch(None, Dev, _H(0), [], []) == []


def test_chunk_plan_respects_the_32_bit_limits():
    big = 1 << 60
    # k = 2^12 on tables precomputed at width 15 (17 windows, 2^14 buckets per MSM): the bucket numbering allows
    # (2^31 - 1) // 2^14 = 131071 proofs, the entries (2^32 - 1) // (17 * tc_rows) fewer
    k, mp = 1 << 12, 100
    key = _key(k, mp, pre=15)
    n_c = dp.tc_rows(k, mp)
    want = min(((1 << 32) - 1) // (17 * n_c), ((1 << 32) - 1) >> 13)
    assert dp.plan_chunk(key, 10 ** 9, big) == want
    assert dp.plan_chunk(key, 5, big) == 5
    # width 20: 2^19 buckets per MSM
    assert dp.plan_chunk(_key(64, 2, pre=20), 10 ** 9, big) == ((1 << 31) - 1) // (1 << 19)
    # plain tables: the automatic width of msm_plan for n rows
    W, per = dp._many_msm_shape(_H(66, "g1"), 66)
    assert (W, per) == (64, 64 * 8)
    W, per = dp._many_msm_shape(_H(1 << 20, "g1"), 1 << 20)
    assert (W, per) == (16, 16 * (1 << 15))


def test_chunk_plan_follows_free_memory():
    key = _key(1 << 16, 10, pre=17)
    sizes = [dp.plan_chunk(key, 4096, free) for free in (0, 1 << 30, 8 << 30, 64 << 30, 1 << 44)]
    assert sizes[0] == 1                                 # always at least one proof per pass
    assert sizes == sorted(sizes)
    assert 1 < sizes[3] < sizes[4] == ((1 << 32) - 1) // (15 * dp.tc_rows(1 << 16, 10))   # then the entry numbering
