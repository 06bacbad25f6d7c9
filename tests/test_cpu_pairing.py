"""CPU: the arithmetic behind csrc/fp12.cuh and csrc/pairing.cu, on integers (tests/tower_model.py), against the
oracle's py_ecc restatement: the generated Frobenius constants, the map from the Fp2/Fp6/Fp12 tower to py_ecc's
FQ12 basis, the Miller-loop formulas, the final-exponentiation chain, and the compat.FQ12 value type."""
import os
import random
import re

import pytest

from oracle.shim.py_ecc import bn128 as bn
from tests import tower_model as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
rng = random.Random(20261020)


def _rand12():
    return tuple(tuple((rng.randrange(M.P), rng.randrange(M.P)) for _ in range(3)) for _ in range(2))


def _fq12(a):
    return bn.FQ12(M.to_pyecc(a))


def test_generated_frobenius_constants_equal_their_definitions():
    src = open(os.path.join(ROOT, "interactive_zkp_study_b200", "csrc", "bn254_params.cuh")).read()
    body = src[src.index("FP12_FROB[18][16]"):]
    rows = re.findall(r"\{(0x[0-9a-f]{8}u(?:, 0x[0-9a-f]{8}u){15})\}", body)
    assert len(rows) == 18
    rinv = pow(1 << 256, -1, M.P)
    for idx, row in enumerate(rows):
        limbs = [int(x.rstrip("u"), 16) for x in row.split(", ")]
        c0 = sum(l << (32 * j) for j, l in enumerate(limbs[:8])) * rinv % M.P      # out of Montgomery form
        c1 = sum(l << (32 * j) for j, l in enumerate(limbs[8:])) * rinv % M.P
        k, i = idx // 6 + 1, idx % 6
        want = bn.FQ2([9, 1]) ** (i * (M.P ** k - 1) // 6)
        assert (c0, c1) == (want.coeffs[0].n, want.coeffs[1].n), (k, i)
    # pi^2 coefficients lie in Fp; xi^((p^2 - 1) / 2) = -1, so -pi^2(Q) keeps y's sign
    assert all(M.GAMMA[1][i][1] == 0 for i in range(6)) and M.GAMMA[1][3] == (M.P - 1, 0)


def test_tower_basis_map_agrees_with_pyecc_fq12():
    for _ in range(4):
        a, b = _rand12(), _rand12()
        assert M.from_pyecc(M.to_pyecc(a)) == a
        assert _fq12(M.f12_mul(a, b)) == _fq12(a) * _fq12(b)
        assert _fq12(M.f12_sqr(a)) == _fq12(a) * _fq12(a)
        assert _fq12(M.f12_inv(a)) == bn.FQ12.one() / _fq12(a)
        assert _fq12(M.f12_conj(a)) == _fq12(a) ** (M.P ** 6)
        for k in (1, 2, 3):
            assert _fq12(M.f12_frobenius(a, k)) == _fq12(a) ** (M.P ** k), k
    # (Fp2 element) u maps to w^6 - 9
    assert M.to_pyecc(((M.f2(0, 1), M.F2_ZERO, M.F2_ZERO), M.F6_ZERO)) == [M.P - 9] + [0] * 5 + [1] + [0] * 5


def test_sparse_line_product_and_cyclotomic_squaring():
    a = _rand12()
    l00, l10, l11 = ((rng.randrange(M.P), rng.randrange(M.P)) for _ in range(3))
    full = ((l00, M.F2_ZERO, M.F2_ZERO), (l10, l11, M.F2_ZERO))
    assert M.f12_mul_line(a, l00, l10, l11) == M.f12_mul(a, full)
    e = M.f12_mul(M.f12_conj(a), M.f12_inv(a))
    e = M.f12_mul(M.f12_frobenius(e, 2), e)            # after the easy part: in the cyclotomic subgroup
    assert M.f12_cyclotomic_sqr(e) == M.f12_sqr(e)
    assert M.f12_cyclotomic_sqr(a) != M.f12_sqr(a)     # (and only there)


def test_final_exponentiation_chain_is_the_exact_power():
    a = _rand12()
    assert _fq12(M.final_exponentiation(a)) == bn.final_exponentiate(_fq12(a))


def test_miller_loop_formulas_give_pyecc_pairing():
    q, p = bn.multiply(bn.G2, 5), bn.multiply(bn.G1, 7)
    q_i = ((q[0].coeffs[0].n, q[0].coeffs[1].n), (q[1].coeffs[0].n, q[1].coeffs[1].n))
    assert _fq12(M.pairing(q_i, (p[0].n, p[1].n))) == bn.pairing(q, p)
    assert M.pairing(q_i, None) == M.ONE


def test_compat_fq12_multiplies_as_pyecc():
    from interactive_zkp_study_b200.compat import FQ12
    for _ in range(3):
        a, b = [rng.randrange(M.P) for _ in range(12)], [rng.randrange(M.P) for _ in range(12)]
        got = FQ12(a) * FQ12(b)
        want = bn.FQ12(a) * bn.FQ12(b)
        assert [int(c) for c in got.coeffs] == [c.n for c in want.coeffs]
    x = FQ12(a)
    assert x * FQ12.one() == x and FQ12.one() == FQ12([1] + [0] * 11) and x != FQ12.one()


@pytest.mark.skipif(os.path.exists("/dev/nvidiactl"), reason="a GPU is present")
def test_pairing_has_no_cpu_fallback():
    from interactive_zkp_study_b200 import native
    from interactive_zkp_study_b200.zkp import pairing as zp
    with pytest.raises(native.ZkpB200Error):
        zp.pairing(None, None)
    with pytest.raises(native.ZkpB200Error):
        zp.pairing_check([])
