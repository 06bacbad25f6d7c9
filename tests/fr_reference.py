"""Plain-integer references for the device Fr vector primitives (tests/test_gpu_fr_shapes.py), checked against the
oracle in tests/test_cpu_fr_reference.py.

Everything is linear in the vector length, so the GPU tests can compare whole outputs up to about 2^20 elements.
Above that, an NTT is checked through a fingerprint: for y = NTT_w(x) of length n and a point rho with rho^n != 1,

    sum_k rho^k y_k = (rho^n - 1) * sum_j x_j g^j / (rho w^j - 1)

(g = 1, or the shift of a forward coset transform).  The right side costs one batched inversion.  A wrong output
changes the left side for all but at most n - 1 values of rho.
"""
from operator import mul

import numpy as np

from oracle import ref_path

R = ref_path.R
_R_LIMBS = [(R >> (64 * k)) & (2**64 - 1) for k in range(4)]


def rand_fr_bytes(seed, n):
    """n uniform-looking canonical Fr elements, 32 bytes little-endian each, from a numpy seed.  Values cover
    the whole range [0, r): 254 random bits, and bit 253 is cleared when the value is r or more."""
    v = np.random.default_rng(seed).integers(0, 2**64, size=(n, 4), dtype=np.uint64)
    v[:, 3] &= np.uint64(2**62 - 1)
    r0, r1, r2, r3 = (np.uint64(x) for x in _R_LIMBS)
    ge = (v[:, 3] > r3) | ((v[:, 3] == r3) & ((v[:, 2] > r2) | ((v[:, 2] == r2) & (
        (v[:, 1] > r1) | ((v[:, 1] == r1) & (v[:, 0] >= r0))))))
    v[ge, 3] &= np.uint64(2**61 - 1)
    return v.tobytes()


def decode(b):
    fb = int.from_bytes
    return [fb(b[i:i + 32], "little") for i in range(0, len(b), 32)]


def encode(xs):
    return b"".join([x.to_bytes(32, "little") for x in xs])


def exclusive_product(xs):
    out, acc = [0] * len(xs), 1
    for i, x in enumerate(xs):
        out[i] = acc
        acc = acc * x % R
    return out


def exclusive_sum(xs):
    out, acc = [0] * len(xs), 0
    for i, x in enumerate(xs):
        out[i] = acc
        acc = (acc + x) % R
    return out


def batch_inverse(xs):
    """x^-1 elementwise with inv(0) = 0 (py_ecc's convention), by one prefix product and one inversion."""
    n = len(xs)
    pre, acc = [0] * n, 1
    for i, x in enumerate(xs):
        pre[i] = acc
        if x:
            acc = acc * x % R
    inv = pow(acc, R - 2, R)
    out = [0] * n
    for i in range(n - 1, -1, -1):
        x = xs[i]
        if x:
            out[i] = inv * pre[i] % R
            inv = inv * x % R
    return out


def powers(first, base, n):
    """first * base^i, i < n (0^0 = 1)."""
    out, acc = [0] * n, first % R
    for i in range(n):
        out[i] = acc
        acc = acc * base % R
    return out


def horner(coeffs, x, block=1024):
    """p(x) for p = coeffs[0] + coeffs[1] x + ...; blocks of unreduced dot products with x^0..x^(block-1) so that
    only one reduction in `block` terms is a Python-level modular product."""
    n = len(coeffs)
    if n == 0:
        return 0
    pw = powers(1, x, min(block, n))
    step = pow(x, block, R)
    acc = 0
    for s in range(((n - 1) // block) * block, -1, -block):
        acc = (acc * step + sum(map(mul, coeffs[s:s + block], pw))) % R
    return acc


def div_linear(coeffs, z):
    """The n - 1 coefficients of (p(x) - p(z)) / (x - z) by synthetic division."""
    n = len(coeffs)
    q = [0] * max(n - 1, 0)
    acc = 0
    for k in range(n - 1, 0, -1):
        acc = (acc * z + coeffs[k]) % R
        q[k - 1] = acc
    return q


def dot(a, b):
    return sum(map(mul, a, b)) % R


def ntt_denominators(n, omega, rho):
    """1 / (rho w^j - 1), j < n: the part of the fingerprint that depends only on the domain and rho."""
    if pow(rho, n, R) == 1:
        raise ValueError("rho must not be an n-th root of unity")
    d, a = [0] * n, rho
    for j in range(n):
        d[j] = a - 1
        a = a * omega % R
    return batch_inverse(d)


def ntt_fingerprint(x, omega, rho, inverse=False, shift=None, dinv=None):
    """sum_k rho^k y_k for y the transform of x as the device computes it: forward y_k = sum_j x_j shift^j w^jk;
    inverse y_k = n^-1 shift^-k sum_j x_j w^-jk.  dinv: ntt_denominators of the same n, root and point, where
    the inverse transform uses w^-1 and the point rho / shift."""
    n = len(x)
    if inverse:
        omega = ref_path.inv(omega)
        if shift is not None:
            rho = rho * ref_path.inv(shift) % R
    if dinv is None:
        dinv = ntt_denominators(n, omega, rho)
    if shift is not None and not inverse:
        s = sum(map(mul, map(mul, x, powers(1, shift, n)), dinv)) % R
    else:
        s = sum(map(mul, x, dinv)) % R
    out = (pow(rho, n, R) - 1) * s % R
    return out * ref_path.inv(n) % R if inverse else out


def product_holds(a, b, c, rhos):
    """c = a b, by length and by evaluation at each rho."""
    return len(c) == len(a) + len(b) - 1 and all(horner(a, t) * horner(b, t) % R == horner(c, t) for t in rhos)


def division_holds(a, b, q, r, rhos):
    """a = b q + r with len(q) = la - lb + 1 and len(r) = lb - 1: the pair is unique, so a wrong one passes at a
    random rho with probability at most la / r."""
    return (len(q) == len(a) - len(b) + 1 and len(r) == len(b) - 1 and
            all(horner(a, t) == (horner(b, t) * horner(q, t) + horner(r, t)) % R for t in rhos))
