"""CPU: the plain-integer references of tests/fr_reference.py against the oracle (oracle/ref_path.py) and naive
loops at small sizes, so the references the GPU shape tests rest on are themselves checked on any machine."""
import random

import pytest

from oracle import ref_path
from tests import fr_reference as ref

R = ref.R


def _rand(rng, n):
    return [rng.randrange(R) for _ in range(n)]


def test_random_bytes_are_canonical_and_cover_the_range():
    xs = ref.decode(ref.rand_fr_bytes(7, 20000))
    assert len(xs) == 20000 and all(0 <= x < R for x in xs)
    assert sum(x >= 1 << 253 for x in xs) > 2000          # the top third of [0, r) is not left out
    assert ref.rand_fr_bytes(7, 5) == ref.rand_fr_bytes(7, 5) != ref.rand_fr_bytes(8, 5)
    assert ref.encode(xs[:9]) == ref.rand_fr_bytes(7, 20000)[:9 * 32]


@pytest.mark.parametrize("n", [1, 2, 8, 64])
def test_ntt_fingerprint_matches_oracle_transforms(n):
    rng = random.Random(n)
    x = _rand(rng, n)
    w = ref_path.get_root_of_unity(n)
    for rho in (rng.randrange(R), rng.randrange(R)):
        assert ref.horner(ref_path.fft(x, w), rho) == ref.ntt_fingerprint(x, w, rho)
        assert ref.horner(ref_path.ifft(x, w), rho) == ref.ntt_fingerprint(x, w, rho, inverse=True)
        assert ref.horner(ref_path.coset_fft(x, w, 5), rho) == ref.ntt_fingerprint(x, w, rho, shift=5)
        assert ref.horner(ref_path.coset_ifft(x, w, 5), rho) == ref.ntt_fingerprint(x, w, rho, inverse=True, shift=5)
        # the denominators are shared by the plain and the coset forward transform
        dinv = ref.ntt_denominators(n, w, rho)
        assert ref.ntt_fingerprint(x, w, rho, shift=5, dinv=dinv) == ref.horner(ref_path.coset_fft(x, w, 5), rho)


def test_ntt_fingerprint_sees_a_single_wrong_output():
    rng = random.Random(5)
    n = 64
    x = _rand(rng, n)
    w = ref_path.get_root_of_unity(n)
    y = ref_path.fft(x, w)
    rho = rng.randrange(R)
    for k in (0, 1, n // 2, n - 1):
        bad = list(y)
        bad[k] = (bad[k] + 1) % R
        assert ref.horner(bad, rho) != ref.ntt_fingerprint(x, w, rho)
    with pytest.raises(ValueError):
        ref.ntt_denominators(n, w, w)                    # rho a root of unity: a denominator vanishes


@pytest.mark.parametrize("n", [0, 1, 2, 63, 64, 65, 1023, 1024, 1025, 3000])
def test_horner_matches_oracle(n):
    rng = random.Random(100 + n)
    c = _rand(rng, n)
    for x in (0, 1, R - 1, rng.randrange(R)):
        assert ref.horner(c, x) == ref_path.poly_eval(c, x)


def test_linear_references_match_naive_loops():
    rng = random.Random(11)
    n = 300
    x = _rand(rng, n)
    x[3] = x[200] = 0
    assert ref.exclusive_product(x) == [_prod(x[:i]) for i in range(n)]
    assert ref.exclusive_sum(x) == [sum(x[:i]) % R for i in range(n)]
    assert ref.batch_inverse(x) == [ref_path.inv(v) for v in x]
    assert ref.batch_inverse([0, 0]) == [0, 0]
    b, f = rng.randrange(R), rng.randrange(R)
    assert ref.powers(f, b, 40) == [f * pow(b, i, R) % R for i in range(40)]
    assert ref.powers(f, 0, 3) == [f, 0, 0]
    y = _rand(rng, n)
    assert ref.dot(x, y) == sum(u * v for u, v in zip(x, y)) % R


@pytest.mark.parametrize("n", [1, 2, 3, 17, 200])
def test_div_linear_matches_long_division(n):
    rng = random.Random(n)
    p = _rand(rng, n)
    for z in (0, 1, R - 1, rng.randrange(R)):
        q = ref.div_linear(p, z)
        pm = list(p)
        pm[0] = (pm[0] - ref_path.poly_eval(p, z)) % R
        if n == 1:
            assert q == []
            continue
        want, rem = ref_path.poly_div(pm, [(-z) % R, 1])
        assert rem == [0]
        assert q == want + [0] * (n - 1 - len(want))


@pytest.mark.parametrize("la,lb", [(1, 1), (5, 2), (40, 13), (129, 64), (300, 299)])
def test_product_and_division_identities(la, lb):
    rng = random.Random(la * 1000 + lb)
    a, b = _rand(rng, la), _rand(rng, lb)
    rhos = (rng.randrange(R), rng.randrange(R))
    c = [0] * (la + lb - 1)
    for i, u in enumerate(a):
        for j, v in enumerate(b):
            c[i + j] = (c[i + j] + u * v) % R
    assert ref.product_holds(a, b, c, rhos)
    bad = list(c)
    bad[len(c) // 2] = (bad[len(c) // 2] + 1) % R
    assert not ref.product_holds(a, b, bad, rhos)
    assert not ref.product_holds(a, b, c[:-1], rhos)
    q, r = ref_path.poly_div(a, b)
    q = q + [0] * (la - lb + 1 - len(q))
    r = r + [0] * (lb - 1 - len(r)) if lb > 1 else []
    assert ref.division_holds(a, b, q, r, rhos)
    if lb > 1:
        r2 = list(r)
        r2[0] = (r2[0] + 1) % R
        assert not ref.division_holds(a, b, q, r2, rhos)
    q2 = list(q)
    q2[-1] = (q2[-1] + 1) % R
    assert not ref.division_holds(a, b, q2, r, rhos)


def _prod(xs):
    acc = 1
    for v in xs:
        acc = acc * v % R
    return acc
