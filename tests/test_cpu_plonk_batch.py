"""CPU: argument validation of the batch PLONK prover (refused before any device call) and the chunk planning of
plonk.device_prover.prove_batch, which is host arithmetic."""
import pytest

from interactive_zkp_study_b200.zkp.plonk import device_prover as dp


class _H:
    """Stands in for a device handle: only its length is read before the first device call."""

    def __init__(self, n, kind="fr", pre_c=0):
        self.n, self.kind, self.pre_c = n, kind, pre_c


def _key(n, pre=0, ranks=None):
    key = dp.DeviceKey()
    key.n = n
    key.ext = 4 if n >= 8 else (8 if n >= 2 else 16)
    key.N8 = key.ext * n
    key.srs_table = _H(n + 6, "g1", pre)
    key.ranks = ranks
    return key


def _wires(n, count):
    return [_H(count * n) for _ in range(3)]


def test_prove_batch_refuses_bad_shapes_before_any_device_call():
    key = _key(16)
    a, b, c = _wires(16, 4)
    with pytest.raises(ValueError, match="b_vals"):
        dp.prove_batch(key, a, _H(63), c, 4)
    with pytest.raises(ValueError, match="c_vals"):
        dp.prove_batch(key, a, b, None, 4)
    for bad in ([[1] * 9] * 3, [[1] * 9] * 3 + [[1] * 8], [[1] * 10] * 4):
        with pytest.raises(ValueError, match="blinds"):
            dp.prove_batch(key, a, b, c, 4, blinds=bad)
    for bad in (0, -3):
        with pytest.raises(ValueError, match="chunk"):
            dp.prove_batch(key, a, b, c, 4, chunk=bad)
    assert dp.prove_batch(key, a, b, c, 0) == []
    assert dp.prove_batch(key, _H(0), _H(0), _H(0), 0, blinds=[]) == []


def test_prove_batch_refuses_a_sharded_key():
    key = _key(16, ranks=object())
    with pytest.raises(ValueError, match="sharded"):
        dp.prove_batch(key, *_wires(16, 2), 2)


def _fits(key, chunk):
    """The limits plan_chunk promises, restated: the many-MSM numbering of every round and the coset transforms."""
    from interactive_zkp_study_b200.zkp.groth16.device_prover import _many_msm_shape
    n = key.n
    if 4 * chunk * key.N8 >= 1 << 32:
        return False
    for vecs, pad in ((3, 2), (1, 3), (3, 6), (2, 5)):
        W, per = _many_msm_shape(key.srs_table, n + pad)
        if vecs * chunk * W * (n + pad) >= 1 << 32 or vecs * chunk * per >= 1 << 31:
            return False
    return True


@pytest.mark.parametrize("log_n,pre", [(0, 0), (2, 0), (10, 0), (12, 15), (16, 17), (20, 20), (24, 16)])
def test_chunk_plan_respects_the_32_bit_limits(log_n, pre):
    key = _key(1 << log_n, pre)
    chunk = dp.plan_chunk(key, 10 ** 9, 1 << 62)
    assert chunk >= 1
    if chunk > 1 or _fits(key, 1):
        assert _fits(key, chunk)
        assert not _fits(key, chunk + 1)                 # the largest chunk within the limits
    assert dp.plan_chunk(key, 5, 1 << 62) == min(5, chunk)


def test_chunk_plan_follows_free_memory():
    key = _key(1 << 16, 17)
    sizes = [dp.plan_chunk(key, 4096, free) for free in (0, 1 << 30, 8 << 30, 64 << 30, 1 << 50)]
    assert sizes[0] == 1                                 # always at least one proof per pass
    assert sizes == sorted(sizes)
    assert 1 < sizes[3] < sizes[4]
    assert _fits(key, sizes[4]) and not _fits(key, sizes[4] + 1)


def test_batch_wrappers_refuse_short_host_lists_before_any_device_call():
    from interactive_zkp_study_b200 import native
    h = _H(64)
    with pytest.raises(ValueError, match="gammas"):
        native.plonk_perm_terms_many_dev(h, h, h, 0, h, h, h, 4, 1, [1, 2, 3], [1, 2], h, h)
    with pytest.raises(ValueError, match="alphas"):
        native.plonk_quotient_many_dev(h, [h] * 8, 4, 8, h, h, h, [1, 2], [1, 2], [1], h)
    with pytest.raises(ValueError, match="8 circuit"):
        native.plonk_quotient_many_dev(h, [h] * 7, 4, 8, h, h, h, [1], [1], [1], h)
    with pytest.raises(ValueError, match="blinds"):
        native.plonk_blind_many_dev(h, 0, 4, 4, 3, [[1, 2], [3, 4], [5]], h, 0, 6)
    with pytest.raises(ValueError, match="blinds"):
        native.plonk_blind_many_dev(h, 0, 4, 4, 3, [[1, 2], [3, 4]], h, 0, 6)
    with pytest.raises(ValueError, match="point_sets"):
        native.fr_poly_eval_many_dev([(h, 0, 4, 4, 1)], 3, [[1, 2, 3], [4, 5]])
    with pytest.raises(ValueError, match="point set"):
        native.fr_poly_eval_many_dev([(h, 0, 4, 4, 2)], 3, [[1, 2, 3], [4, 5, 6]])
    with pytest.raises(ValueError, match="coeffs"):
        native.lincomb_many_dev(h, 0, 8, 8, 2, [(h, 0, 8, 8)], [[1, 2], [3]])
    with pytest.raises(ValueError, match="coeffs"):
        native.lincomb_many_dev(h, 0, 8, 8, 3, [(h, 0, 8, 8)], [[1, 2], [3, 4]])
