"""CPU: argument validation of plonk.device_prover.prove_batch_circuits (many circuits of one size per pass), refused
before any device call, the host-list checks of its native wrappers, and the chunk planning with the per-proof
circuit blocks, which is host arithmetic."""
import pytest

from interactive_zkp_study_b200 import native
from interactive_zkp_study_b200.zkp.plonk import device_prover as dp


class _H:
    """Stands in for a device handle: only its length (and table identity) is read before the first device call."""

    def __init__(self, n, kind="fr", pre_c=0):
        self.n, self.kind, self.pre_c = n, kind, pre_c


def _key(n, srs=None, pre=0, ranks=None, ell=0):
    key = dp.DeviceKey()
    key.n = n
    key.ext = 4 if n >= 8 else (8 if n >= 2 else 16)
    key.N8 = key.ext * n
    key.srs_table = srs if srs is not None else _H(n + 6, "g1", pre)
    key.ranks = ranks
    key.num_public_inputs = ell
    return key


def _wires(n, count):
    return [_H(count * n) for _ in range(3)]


def test_refuses_bad_key_sets_before_any_device_call():
    srs = _H(22, "g1")
    a, b, c = _wires(16, 4)
    with pytest.raises(ValueError, match="no keys"):
        dp.prove_batch_circuits([], [], a, b, c)
    with pytest.raises(ValueError, match="differ in n"):
        dp.prove_batch_circuits([_key(16, srs), _key(8, srs)], [0, 0, 0, 0], a, b, c)
    with pytest.raises(ValueError, match="one SRS table"):
        dp.prove_batch_circuits([_key(16, srs), _key(16)], [0, 0, 0, 0], a, b, c)
    with pytest.raises(ValueError, match="num_public_inputs"):
        dp.prove_batch_circuits([_key(16, srs), _key(16, srs, ell=2)], [0, 0, 0, 0], a, b, c)
    with pytest.raises(ValueError, match="sharded"):
        dp.prove_batch_circuits([_key(16, srs), _key(16, srs, ranks=object())], [0, 0, 0, 0], a, b, c)
    with pytest.raises(ValueError, match="sharded"):
        dp.prove_batch_circuits([_key(16, srs, ranks=object())], [0], a, b, c)


@pytest.mark.parametrize("bad", [-1, 2, 7, 1.0, True, "1", None])
def test_refuses_an_index_outside_the_keys(bad):
    srs = _H(22, "g1")
    keys = [_key(16, srs), _key(16, srs)]
    with pytest.raises(ValueError, match="circuit index .* proof 2 "):
        dp.prove_batch_circuits(keys, [0, 1, bad, 0], *_wires(16, 4))


def test_refuses_what_prove_batch_refuses():
    srs = _H(22, "g1")
    keys = [_key(16, srs), _key(16, srs)]
    circ = [1, 0, 1, 1]
    a, b, c = _wires(16, 4)
    with pytest.raises(ValueError, match="b_vals"):
        dp.prove_batch_circuits(keys, circ, a, _H(63), c)
    with pytest.raises(ValueError, match="c_vals"):
        dp.prove_batch_circuits(keys, circ, a, b, None)
    for bad in ([[1] * 9] * 3, [[1] * 9] * 3 + [[1] * 8], [[1] * 10] * 4):
        with pytest.raises(ValueError, match="blinds"):
            dp.prove_batch_circuits(keys, circ, a, b, c, blinds=bad)
    for bad in (0, -3):
        with pytest.raises(ValueError, match="chunk"):
            dp.prove_batch_circuits(keys, circ, a, b, c, chunk=bad)
    with pytest.raises(ValueError, match="no public inputs"):
        dp.prove_batch_circuits(keys, circ, a, b, c, public_inputs=_H(8))
    pkeys = [_key(16, srs, ell=2), _key(16, srs, ell=2)]
    with pytest.raises(ValueError, match="public_inputs"):
        dp.prove_batch_circuits(pkeys, circ, a, b, c, public_inputs=_H(7))
    with pytest.raises(ValueError, match="public_inputs"):
        dp.prove_batch_circuits(pkeys, circ, a, b, c)
    # an unused circuit and no proofs at all are fine
    assert dp.prove_batch_circuits(keys, [], a, b, c) == []
    assert dp.prove_batch_circuits(keys, [], _H(0), _H(0), _H(0), blinds=[]) == []


def _fits(key, chunk):
    """The limits plan_chunk promises (tests/test_cpu_plonk_batch.py), restated."""
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
def test_multi_chunk_plan_respects_the_32_bit_limits(log_n, pre):
    key = _key(1 << log_n, pre=pre)
    chunk = dp.plan_chunk(key, 10 ** 9, 1 << 62, multi=True)
    assert chunk >= 1
    if chunk > 1 or _fits(key, 1):
        assert _fits(key, chunk)
        assert not _fits(key, chunk + 1)
    assert dp.plan_chunk(key, 5, 1 << 62, multi=True) == min(5, chunk)


def test_multi_chunk_plan_counts_the_gathered_blocks():
    key = _key(1 << 16, pre=17)
    for free in (1 << 30, 8 << 30, 64 << 30):
        one, multi = dp.plan_chunk(key, 4096, free), dp.plan_chunk(key, 4096, free, multi=True)
        assert 1 <= multi <= one
    assert dp.plan_chunk(key, 4096, 64 << 30, multi=True) < dp.plan_chunk(key, 4096, 64 << 30)
    sizes = [dp.plan_chunk(key, 4096, free, multi=True) for free in (0, 1 << 30, 8 << 30, 64 << 30, 1 << 50)]
    assert sizes[0] == 1 and sizes == sorted(sizes)


def test_multi_wrappers_refuse_short_host_lists_before_any_device_call():
    h = _H(64)
    with pytest.raises(ValueError, match="gammas"):
        native.plonk_perm_terms_multi_dev(h, h, h, 0, [[h] * 3], [0, 0, 0], 4, 1, [1, 2, 3], [1, 2], h, h)
    with pytest.raises(ValueError, match="circuit_of"):
        native.plonk_perm_terms_multi_dev(h, h, h, 0, [[h] * 3], [0, 0], 4, 1, [1, 2, 3], [1, 2, 3], h, h)
    with pytest.raises(ValueError, match="3 handles"):
        native.plonk_perm_terms_multi_dev(h, h, h, 0, [[h] * 3, [h] * 2], [0], 4, 1, [1], [1], h, h)
    with pytest.raises(ValueError, match="3 handles"):
        native.plonk_perm_terms_multi_dev(h, h, h, 0, [], [0], 4, 1, [1], [1], h, h)
    for fn in (native.plonk_quotient_multi_dev, native.plonk_quotient_pi_multi_dev):
        with pytest.raises(ValueError, match="alphas"):
            fn(h, [[h] * 8], [0, 0], 4, 8, h, h, h, [1, 2], [1, 2], [1], h)
        with pytest.raises(ValueError, match="8 handles"):
            fn(h, [[h] * 8, [h] * 7], [0], 4, 8, h, h, h, [1], [1], [1], h)
        with pytest.raises(ValueError, match="circuit_of"):
            fn(h, [[h] * 8], [0, 0, 0], 4, 8, h, h, h, [1, 2], [1, 2], [1, 2], h)
    with pytest.raises(ValueError, match="handles"):
        native.fr_gather_many_dev([[h, h], [h]], [0, 1], 4, h)
    with pytest.raises(ValueError, match="handles"):
        native.fr_gather_many_dev([], [0, 1], 4, h)
