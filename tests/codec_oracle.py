"""TEST INFRASTRUCTURE -- plain-int restatement of the compressed point encoding (csrc/point_codec.cuh) on top of
oracle/bn254.py's field and group arithmetic.

    G1, 32 B: x little-endian, byte 31 bit 7 = y-sign (y > (p-1)/2), bit 6 = infinity.
    G2, 64 B: x.c0 | x.c1 little-endian, the flags in byte 63; y-sign compares y1 (or y0 when y1 = 0) with (p-1)/2.
    Infinity: every bit zero except the infinity flag.

Decoders return the point (None for infinity) or raise ValueError for an invalid encoding.
"""
from oracle import bn254

P, R = bn254.P, bn254.R
HALF = (P - 1) // 2
SIGN, INF = 1 << 255, 1 << 254


def fp_sqrt(a):
    """A square root of a in Fp (p = 3 mod 4: a^((p+1)/4)), or None."""
    a %= P
    y = pow(a, (P + 1) // 4, P)
    return y if y * y % P == a else None


def _f2_pow(a, e):
    r = (1, 0)
    for bit in bin(e)[2:]:
        r = bn254.f2_mul(r, r)
        if bit == "1":
            r = bn254.f2_mul(r, a)
    return r


def f2_sqrt(a):
    """A square root of a in Fp2 (Algorithm 9 of Adj and Rodriguez-Henriquez, 2012), or None."""
    a = (a[0] % P, a[1] % P)
    a1 = _f2_pow(a, (P - 3) // 4)
    alpha = bn254.f2_mul(bn254.f2_mul(a1, a1), a)
    x0 = bn254.f2_mul(a1, a)
    if bn254.f2_mul((alpha[0], -alpha[1] % P), alpha) == (P - 1, 0):
        return None
    if alpha == (P - 1, 0):
        y = bn254.f2_mul((0, 1), x0)
    else:
        y = bn254.f2_mul(_f2_pow(((1 + alpha[0]) % P, alpha[1]), (P - 1) // 2), x0)
    return y if bn254.f2_mul(y, y) == a else None


def g1_sign(y):
    return y > HALF


def g2_sign(y):
    return y[1] > HALF if y[1] else y[0] > HALF


def g1_compress(pt):
    if pt is None:
        return INF.to_bytes(32, "little")
    return (pt[0] | (SIGN if g1_sign(pt[1]) else 0)).to_bytes(32, "little")


def g2_compress(pt):
    if pt is None:
        return bytes(32) + INF.to_bytes(32, "little")
    (x0, x1), y = pt
    return x0.to_bytes(32, "little") + (x1 | (SIGN if g2_sign(y) else 0)).to_bytes(32, "little")


def _flags(last):
    sign, inf = bool(last & SIGN), bool(last & INF)
    if sign and inf:
        raise ValueError("both flags set")
    return sign, inf, last & (INF - 1)


def g1_decompress(b):
    if len(b) != 32:
        raise ValueError("a compressed G1 point is 32 bytes")
    sign, inf, x = _flags(int.from_bytes(b, "little"))
    if inf:
        if x:
            raise ValueError("infinity flag with other bits set")
        return None
    if x >= P:
        raise ValueError("x >= p")
    y = fp_sqrt(x * x * x + 3)
    if y is None:
        raise ValueError("x^3 + 3 is not a square")
    if g1_sign(y) != sign:
        y = (P - y) % P
    return (x, y)


def g2_decompress(b, subgroup_check=True):
    if len(b) != 64:
        raise ValueError("a compressed G2 point is 64 bytes")
    x0 = int.from_bytes(b[:32], "little")
    sign, inf, x1 = _flags(int.from_bytes(b[32:], "little"))
    if inf:
        if x0 or x1:
            raise ValueError("infinity flag with other bits set")
        return None
    if x0 >= P or x1 >= P:
        raise ValueError("x coordinate >= p")
    x = (x0, x1)
    y = f2_sqrt(bn254.f2_add(bn254.f2_mul(bn254.f2_mul(x, x), x), bn254.B2))
    if y is None:
        raise ValueError("x^3 + b is not a square")
    if g2_sign(y) != sign:
        y = (-y[0] % P, -y[1] % P)
    if subgroup_check and bn254.g2_mul((x, y), R) is not None:
        raise ValueError("not in the order-r subgroup")
    return (x, y)


def twist_point_outside_g2():
    """A point of the twist y^2 = x^3 + b that is not in G2 (the twist's order is r (2p - r))."""
    for x0 in range(1, 100):
        x = (x0, 1)
        y = f2_sqrt(bn254.f2_add(bn254.f2_mul(bn254.f2_mul(x, x), x), bn254.B2))
        if y is not None and bn254.g2_mul((x, y), R) is not None:
            return (x, y)
    raise AssertionError("no twist point found")


def g1_invalid_encodings():
    """(encoding, why) pairs of invalid G1 encodings."""
    x = g1_compress(bn254.g1_mul(bn254.G1, 5))
    return [
        (bytes(32), "x = 0 is not on the curve (3 is not a square)"),
        (P.to_bytes(32, "little"), "x = p"),
        (((1 << 254) - 1).to_bytes(32, "little"), "x = 2^254 - 1"),
        ((int.from_bytes(x, "little") | INF).to_bytes(32, "little"), "infinity with x bits"),
        ((INF | SIGN).to_bytes(32, "little"), "both flags"),
        ((INF | 1).to_bytes(32, "little"), "infinity with a low bit"),
        (((P + 1) | SIGN).to_bytes(32, "little"), "x = p + 1 with the sign flag"),
    ]


def g1_no_point_x():
    x = 1
    while fp_sqrt(x ** 3 + 3) is not None:
        x += 1
    return x


def g2_invalid_encodings():
    """(encoding, why) pairs of invalid G2 encodings (on the twist or not, subgroup aside)."""
    g = g2_compress(bn254.G2)
    x1 = int.from_bytes(g[32:], "little")
    return [
        (P.to_bytes(32, "little") + g[32:], "x.c0 = p"),
        (g[:32] + (P | SIGN).to_bytes(32, "little"), "x.c1 = p"),
        (g[:32] + (x1 | INF).to_bytes(32, "little"), "infinity with x bits"),
        (bytes(32) + (INF | SIGN).to_bytes(32, "little"), "both flags"),
        ((1).to_bytes(32, "little") + INF.to_bytes(32, "little"), "infinity with a bit of x.c0"),
        (g2_no_point_x(), "no point with this x"),
    ]


def g2_no_point_x():
    for x0 in range(1, 100):
        x = (x0, 0)
        if f2_sqrt(bn254.f2_add(bn254.f2_mul(bn254.f2_mul(x, x), x), bn254.B2)) is None:
            return x0.to_bytes(32, "little") + bytes(32)
    raise AssertionError("every x tried has a point")
