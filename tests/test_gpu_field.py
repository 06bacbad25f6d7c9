"""-m gpu: the Montgomery field core and the XYZZ group law of libzkp_b200 against Python ints
(field ops) and the plain-int oracle (group law, incl. every edge case py_ecc defines:
infinity operands, P+P, P+(-P); SURVEY.md H2)."""
import random

import pytest

from oracle import bn254

pytestmark = pytest.mark.gpu

P, R = bn254.P, bn254.R


def _vec(vals):
    return b"".join(int(v).to_bytes(32, "little") for v in vals)


def _unvec(b):
    return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


@pytest.mark.parametrize("field,mod", [(0, P), (1, R)])
def test_field_ops_bit_exact(native, field, mod):
    rng = random.Random(1234 + field)
    edge = [0, 1, 2, mod - 1, mod - 2, (1 << 253), (1 << 32) - 1, 1 << 32, (mod - 1) // 2, (mod + 1) // 2]
    a = edge + [rng.randrange(mod) for _ in range(4000)]
    b = list(reversed(edge)) + [rng.randrange(mod) for _ in range(4000)]
    n = len(a)
    ab, bb = _vec(a), _vec(b)
    assert _unvec(native.dbg_field_op(field, 0, ab, bb, n)) == [(x + y) % mod for x, y in zip(a, b)]
    assert _unvec(native.dbg_field_op(field, 1, ab, bb, n)) == [(x - y) % mod for x, y in zip(a, b)]
    assert _unvec(native.dbg_field_op(field, 2, ab, bb, n)) == [(x * y) % mod for x, y in zip(a, b)]
    assert _unvec(native.dbg_field_op(field, 4, ab, None, n)) == [(x * x) % mod for x in a]
    # limb patterns IN MONTGOMERY FORM (the device squares x = a R mod p; the dedicated squaring doubles the operand
    # across limb boundaries)
    rinv = pow(1 << 256, -1, mod)
    pats = _limb_patterns(mod)
    pa = [x * rinv % mod for x in pats]
    assert _unvec(native.dbg_field_op(field, 4, _vec(pa), None, len(pa))) == [(x * x) % mod for x in pa]
    assert _unvec(native.dbg_field_op(field, 2, _vec(pa), _vec(pa[::-1]), len(pa))) == [(x * y) % mod for x, y in zip(pa, pa[::-1])]
    # the two-step form (512-bit product, then one Montgomery reduction) behind the lazily reduced Fp2 product
    assert _unvec(native.dbg_field_op(field, 6, _vec(pa), _vec(pa[::-1]), len(pa))) == [(x * y) % mod for x, y in zip(pa, pa[::-1])]
    assert _unvec(native.dbg_field_op(field, 6, _vec(a[:500]), _vec(b[:500]), 500)) == [(x * y) % mod for x, y in zip(a[:500], b[:500])]
    # a b - c d with one reduction (the Y coordinate of every XYZZ formula): c = a + b, d = a - b, random and limb patterns
    want = lambda xs, ys: [(x * y - (x + y) * (x - y)) % mod for x, y in zip(xs, ys)]
    assert _unvec(native.dbg_field_op(field, 8, ab, bb, n)) == want(a, b)
    assert _unvec(native.dbg_field_op(field, 8, _vec(pa), _vec(pa[::-1]), len(pa))) == want(pa, pa[::-1])
    assert _unvec(native.dbg_field_op(field, 8, _vec(pats), _vec(pats[::-1]), len(pats))) == want(pats, pats[::-1])
    m = 300
    got = _unvec(native.dbg_field_op(field, 3, _vec(a[:m]), None, m))
    assert got == [bn254.inv(x, mod) for x in a[:m]]  # inv(0) == 0 as in py_ecc (batched division steps, modinv30.cuh)
    assert _unvec(native.dbg_field_op(field, 5, _vec(a[:m]), None, m)) == got  # Fermat chain agrees
    assert _unvec(native.dbg_field_op(field, 7, _vec(a[:m]), None, m)) == got  # binary extended Euclid agrees
    # values whose Montgomery form a R mod p is small / has long runs of zeros or ones (the division steps look at
    # the low bits of that integer), and small plain values
    mont_small = [x * rinv % mod for x in (1, 2, 3, 1 << 30, (1 << 30) - 1, 1 << 60, (1 << 255) % mod, mod - 1, mod - 2,
                                            (1 << 200) - 1, int("aaaaaaaa" * 7, 16))]
    more = mont_small + [1, 2, 3, 5, 1 << 30, 1 << 31, 1 << 32, mod - 1, mod - 2, (mod + 1) // 2] + [rng.randrange(1 << k) for k in range(1, 254, 3)]
    got = _unvec(native.dbg_field_op(field, 3, _vec(more), None, len(more)))
    assert got == [bn254.inv(x, mod) for x in more]


# limb patterns of a field element in Montgomery form (the form the device computes on): all-ones low limbs, top bits
# of every limb set, single-limb values, runs of zeros and ones
def _limb_patterns(mod):
    top = mod >> 224
    pats = [mod - 1, (1 << 224) - 1, ((top - 1) << 224) | ((1 << 224) - 1), int("80000000" * 7, 16),
            (0x20000000 << 224) | int("80000000" * 7, 16), int("ffffffff" * 7, 16) ^ int("0000ffff" * 7, 16),
            0xffffffff, 0xffffffff << 32, 0xffffffff << 192, 0x80000000, (0x80000000 << 96) | 0x80000000,
            (1 << 253) + (1 << 31), int("7fffffff" * 7, 16), int("0000000180000000" * 3, 16)]
    return [x % mod for x in pats]


def test_fp2_ops_bit_exact(native):
    """Fp2 sum, difference, product (Karatsuba on unreduced 512-bit products, one reduction per component), squaring,
    inverse, and the two forms of the G2 bucket-accumulation loop: the squaring with inlined Fp products (op 5) and
    the product with its body inlined (op 6).  Components are given in Montgomery form (canonical value m / 2^256), so
    the device operates on exactly the limb patterns listed: the largest unreduced operand sums of the Karatsuba
    (a0 = a1 = p - 1), its c0 input at both ends (a0 b0 = 0 with a1 b1 maximal: p^2 - (p - 1)^2; a0 b0 maximal with
    a1 b1 = 0: near 2 p^2), and squarings whose c0 + c1 crosses p or whose c0 - c1 borrows."""
    rng = random.Random(99)
    edge = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, (1 << 253), (1 << 32) - 1]
    xs = [(a, b) for a in edge for b in edge] + [(rng.randrange(P), rng.randrange(P)) for _ in range(3000)]
    ys = [(b, a) for a, b in reversed(xs[:81])] + [(rng.randrange(P), rng.randrange(P)) for _ in range(3000)]
    rinv = pow(1 << 256, -1, P)
    mont = lambda pair: tuple(c * rinv % P for c in pair)    # the canonical value whose Montgomery form is `pair`
    comps = [0, 1, P - 1, P - 2] + _limb_patterns(P)
    mx = [(a, b) for a in comps for b in comps]
    my = [(b, a) for a, b in reversed(mx)]
    M = P - 1
    bounds = [((M, M), (M, M)), ((0, M), (M, M)), ((0, M), (0, M)), ((M, 0), (M, M)), ((M, 0), (M, 0)),
              ((M, M), (0, M)), ((M, M), (M, 0)), ((M, 1), (1, M)), ((1, M), (M, 1)), ((P // 2 + 1, P // 2 + 1), (M, M))]
    # squarings: c0 + c1 just below / at / above p, c0 - c1 borrowing by 1 .. p - 1, c0 == c1
    sq = [(M, 1), (M, 2), (M - 5, 5), (M - 5, 6), ((P + 1) // 2, (P + 1) // 2), ((P - 1) // 2, (P + 1) // 2),
          (1, M), (0, M), (5, 6), (P // 3, 2 * (P // 3)), (7, 7), (M, M), (0, 1)]
    xs += [mont(x) for x in mx] + [mont(x) for x, _ in bounds] + [mont(x) for x in sq]
    ys += [mont(y) for y in my] + [mont(y) for _, y in bounds] + [mont((b, a)) for a, b in sq]
    enc = lambda v: b"".join(int(c).to_bytes(32, "little") for pair in v for c in pair)
    dec = lambda b: [(int.from_bytes(b[64 * i:64 * i + 32], "little"), int.from_bytes(b[64 * i + 32:64 * i + 64], "little"))
                     for i in range(len(b) // 64)]
    n = len(xs)
    ex, ey = enc(xs), enc(ys)
    assert dec(native.dbg_field_op(2, 0, ex, ey, n)) == [bn254.f2_add(x, y) for x, y in zip(xs, ys)]
    assert dec(native.dbg_field_op(2, 1, ex, ey, n)) == [bn254.f2_sub(x, y) for x, y in zip(xs, ys)]
    want_mul = [bn254.f2_mul(x, y) for x, y in zip(xs, ys)]
    assert dec(native.dbg_field_op(2, 2, ex, ey, n)) == want_mul
    assert dec(native.dbg_field_op(2, 6, ex, ey, n)) == want_mul
    want_sqr = [bn254.f2_mul(x, x) for x in xs]
    assert dec(native.dbg_field_op(2, 4, ex, None, n)) == want_sqr
    assert dec(native.dbg_field_op(2, 5, ex, None, n)) == want_sqr
    inv = dec(native.dbg_field_op(2, 3, enc(xs[81:381]), None, 300))
    assert all(bn254.f2_mul(x, y) == (1, 0) for x, y in zip(xs[81:381], inv))
    for op in (7, 8, 10, -1):                           # ops Fp2 does not implement are refused, not mapped to another
        with pytest.raises(native.ZkpB200Error):
            native.dbg_field_op(2, op, ex[:64], ey[:64], 1)


# group: 0 = XYZZ mixed + full addition, 2 = the quad-lane operations of ec_quad.cuh (add, double, and the P + P /
# P + (-P) / infinity cases inside them), 4 = the MSM accumulation loop's mixed addition (AccMul) onto an accumulator
# with ZZ != 1, 6 = XYZZ full addition of two operands with different ZZ (the bucket fold); odd numbers: the same on G2
def _cases(pts, neg):
    a, b = [], []
    for i in range(0, len(pts) - 8, 2):
        a.append(pts[i]); b.append(pts[i + 1])          # generic
    a += [None, pts[0], None] + pts[-4:] + pts[-4:]
    b += [pts[0], None, None] + pts[-4:] + [neg(p) for p in pts[-4:]]  # inf+P, P+inf, inf+inf, P+P, P+(-P)
    return a, b


@pytest.mark.parametrize("quad", [0, 2, 4, 6])
def test_g1_add_all_cases(native, quad):
    rng = random.Random(7)
    pts = [bn254.g1_mul(bn254.G1, rng.randrange(1, R)) for _ in range(40)]
    a, b = _cases(pts, bn254.g1_neg)
    n = len(a)
    out = native.dbg_point_add(quad, native.g1_vec_bytes(a), native.g1_vec_bytes(b), n)
    assert len(out) == 64 * n
    got = [native.g1_from_bytes(out[64 * i:64 * i + 64]) for i in range(n)]
    assert got == [bn254.g1_add(x, y) for x, y in zip(a, b)]


@pytest.mark.parametrize("quad", [1, 3, 5, 7])
def test_g2_add_all_cases(native, quad):
    rng = random.Random(8)
    pts = [bn254.g2_mul(bn254.G2, rng.randrange(1, 1 << 64)) for _ in range(18)]
    a, b = _cases(pts, bn254.g2_neg)
    n = len(a)
    enc = lambda v: b"".join(native.g2_bytes(p) for p in v)
    out = native.dbg_point_add(quad, enc(a), enc(b), n)
    assert len(out) == 128 * n
    got = [native.g2_from_bytes(out[128 * i:128 * i + 128]) for i in range(n)]
    assert got == [bn254.g2_add(x, y) for x, y in zip(a, b)]


def test_point_add_refuses_unknown_groups(native):
    one = native.g1_vec_bytes([bn254.G1])
    for group in (-1, 8):
        with pytest.raises(native.ZkpB200Error):
            native.dbg_point_add(group, one + one, one + one, 1)
