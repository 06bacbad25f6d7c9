"""-m gpu: the device Fr vector, scan, Horner, division and NTT entry points on scalar handles against plain Python
integers (tests/fr_reference.py), at the sizes where their launch shapes change:

- scans: 1024-element tiles, and the carry of the tile-scan kernel across chunks of 256 tiles (n > 262 144);
- batch inversion: strided chunks of 32 elements, T = ceil(n / 32) threads;
- two-level power tables: lo[e & 1023] * hi[e >> 10];
- Horner: one more level at n = 65, 4 097, 262 145;
- the dot product: a grid capped at 8 x SMs blocks of 256 threads, then a grid-stride loop;
- the NTT: passes of 10 / 10 + k / 10 + 10 + k stages, and batches whose count shrinks the first-pass tile.

Outputs are compared element by element up to about 2^20 + a few; NTT outputs through the fingerprint of
fr_reference.  Every vector sits at a non-zero offset of its handle between guard elements that must come back
unchanged."""
import pytest

from oracle import ref_path
from tests import fr_reference as ref

pytestmark = pytest.mark.gpu
R = ref.R
M = pow(2, 256, R)                                # Montgomery factor of the device representation
W20 = ref_path.get_root_of_unity(1 << 20)
OFF, TAIL = 3, 2                                  # guard elements before / after each vector
RHO = (0x1D2C3B4A59687766554433221100FFEEDDCCBBAA99887766554433221100AB % R,
       0x0F1E2D3C4B5A69788796A5B4C3D2E1F00112233445566778899AABBCCDDEEF1 % R)
BIG = (1 << 20) + 1


@pytest.fixture
def dev(native):
    """load(payload, off, tail, guard): a handle holding `payload` at `off`, between guard elements (random, or
    zeros with guard=b"zero"); intact(h) says whether the guards are unchanged.  Handles are freed when the case
    ends."""
    made = []

    class Dev:
        @staticmethod
        def load(payload, off=OFF, tail=TAIL, guard=None, seed=0):
            n = len(payload) // 32
            if guard == b"zero":
                lo, hi = bytes(32 * off), bytes(32 * tail)
            else:
                g = ref.rand_fr_bytes(0xC0FFEE + seed, off + tail)
                lo, hi = g[:32 * off], g[32 * off:]
            h = native.scalars_load(lo + payload + hi, off + n + tail)
            h.guard = (off, n, lo, hi)
            made.append(h)
            return h

        @staticmethod
        def zeros(n, off=OFF, tail=TAIL):
            return Dev.load(bytes(32 * n), off, tail, guard=b"zero")

        @staticmethod
        def get(h):
            return native.scalars_download(h, h.guard[0], h.guard[1])

        @staticmethod
        def intact(h):
            off, n, lo, hi = h.guard
            return (native.scalars_download(h, 0, off) == lo and
                    native.scalars_download(h, off + n, len(hi) // 32) == hi)

    yield Dev
    for h in made:
        h.free()


# ------------------------------------------------------------------ scans
def _scan_input(n, op, seed):
    x = ref.decode(ref.rand_fr_bytes(seed, n))
    if n >= 2:
        x[1] = R - 1
    if op == 0 and n >= 3:
        # a zero at the last element of the tile before the last one (inside the only tile when n <= 1024):
        # everything before it exercises the full carry chain, everything after it must come out zero
        z = ((n - 1) // 1024) * 1024 - 1 if n > 1024 else n - 2
        x[z] = 0
    return x


@pytest.mark.parametrize("op", [0, 1], ids=["product", "sum"])
@pytest.mark.parametrize("n", [1, 1023, 1024, 1025, 262144, 262145, (1 << 20) + 3])
def test_scan(native, dev, n, op):
    x = _scan_input(n, op, 10 + n)
    src = dev.load(ref.encode(x))
    dst = dev.load(bytes(32 * n), off=7, seed=1)
    native.scan_dev(op, dst, 7, src, OFF, n)
    want = ref.exclusive_product(x) if op == 0 else ref.exclusive_sum(x)
    assert dev.get(dst) == ref.encode(want)
    assert dev.intact(dst) and dev.intact(src)


# a segment starts on (262 144), just before (262 143) and just after (262 145, 524 290) a 256-tile chunk boundary
@pytest.mark.parametrize("op", [0, 1], ids=["product", "sum"])
@pytest.mark.parametrize("seg,count", [(1024, 3), (1025, 2), (262143, 2), (262144, 2), (262145, 3), (3, 1 << 17)])
def test_scan_many(native, dev, seg, count, op):
    x = ref.decode(ref.rand_fr_bytes(20 + seg, seg * count))
    if op == 0 and seg > 2:
        x[seg - 2] = 0                     # inside segment 0: the next segment starts afresh
    src = dev.load(ref.encode(x))
    dst = dev.load(bytes(32 * seg * count), off=5, seed=1)
    native.scan_many_dev(op, dst, 5, src, OFF, seg, count)
    scan = ref.exclusive_product if op == 0 else ref.exclusive_sum
    want = []
    for j in range(count):
        want += scan(x[j * seg:(j + 1) * seg])
    assert dev.get(dst) == ref.encode(want)
    assert dev.intact(dst)


# ------------------------------------------------------------------ batch inversion
@pytest.mark.parametrize("n", [1, 31, 32, 33, 4095, 4096, 4097, BIG])
def test_batch_inverse(native, dev, n):
    """Canonical and Montgomery modes of the device entry, and the host entry, on the same values: zeros near
    both ends and one whole strided chunk of zeros (every i = t mod T for the last thread t = T - 1).  The last
    element stays non-zero: with n mod 32 != 0 it is the one a thread count rounded down would leave out."""
    x = ref.decode(ref.rand_fr_bytes(30 + n, n))
    if n > 3:
        x[0] = 0
        x[n - 2] = 0
        x[1] = 1
        x[2] = R - 1
    T = (n + 31) // 32
    if T >= 2:
        for i in range(T - 1, n, T):
            x[i] = 0
    want = ref.batch_inverse(x)
    xb, wb = ref.encode(x), ref.encode(want)
    h = dev.load(xb)
    native.batch_inverse_dev(h, OFF, n)
    assert dev.get(h) == wb
    assert dev.intact(h)
    hm = dev.load(ref.encode([v * M % R for v in x]), seed=1)
    native.batch_inverse_dev(hm, OFF, n, montgomery=True)
    assert dev.get(hm) == ref.encode([v * M % R for v in want])
    assert dev.intact(hm)
    assert native.fr_batch_inverse(xb, n) == wb


# ------------------------------------------------------------------ power tables
@pytest.mark.parametrize("n", [1, 2, 1024, 1025, BIG])
def test_fill_powers(native, dev, n):
    h = dev.zeros(n, off=5)
    for base in (0, 1, R - 1, W20, 0x2B61D3F0E4A59C8877665544332211 % R):
        pw = ref.powers(1, base, n)
        first = 0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF % R
        for f, want in ((0, bytes(32 * n)), (1, ref.encode(pw)), (first, ref.encode([first * p % R for p in pw]))):
            native.scalars_fill_powers(h, 5, n, f, base)
            assert dev.get(h) == want, (base, f)
    assert dev.intact(h)


# ------------------------------------------------------------------ elementwise ops (n = 2^20 + 7)
NV = (1 << 20) + 7
FACTORS = (0, 1, R - 1, 0x3C2F1E0D4B5A69788796A5B4C3D2E1F00112233 % R)


@pytest.fixture(scope="module")
def vecs():
    xb, yb = ref.rand_fr_bytes(41, NV), ref.rand_fr_bytes(42, NV)
    return xb, yb, ref.decode(xb), ref.decode(yb)


@pytest.mark.parametrize("k", FACTORS, ids=["0", "1", "r-1", "rand"])
def test_axpy(native, dev, vecs, k):
    xb, yb, x, y = vecs
    d = dev.load(xb, off=6)
    s = dev.load(yb, off=1, seed=1)
    native.axpy_dev(d, 6, k, s, 1, NV)
    assert dev.get(d) == ref.encode([(u + k * v) % R for u, v in zip(x, y)])
    assert dev.intact(d) and dev.intact(s) and dev.get(s) == yb


@pytest.mark.parametrize("k", FACTORS, ids=["0", "1", "r-1", "rand"])
def test_scale_and_add_const(native, dev, vecs, k):
    xb, _, x, _ = vecs
    h = dev.load(xb, off=9)
    native.scalars_scale(h, 9, NV, k)
    kx = [k * u % R for u in x]
    assert dev.get(h) == ref.encode(kx)
    native.scalars_add_const(h, 9, NV, k)
    assert dev.get(h) == ref.encode([(u + k) % R for u in kx])
    assert dev.intact(h)


def test_vec_op_and_convert(native, dev, vecs):
    xb, yb, x, y = vecs
    a = dev.load(xb, off=2)
    b = dev.load(yb, off=11, seed=1)
    d = dev.zeros(NV, off=4)
    for op, f in ((0, lambda u, v: u + v), (1, lambda u, v: u - v), (2, lambda u, v: u * v)):
        native.vec_op_dev(op, d, 4, a, 2, b, 11, NV)
        assert dev.get(d) == ref.encode([f(u, v) % R for u, v in zip(x, y)]), op
    native.scalars_convert(a, 2, NV, True)
    assert dev.get(a) == ref.encode([u * M % R for u in x])
    native.scalars_convert(a, 2, NV, False)
    assert dev.get(a) == xb
    assert dev.intact(a) and dev.intact(b) and dev.intact(d)


# ------------------------------------------------------------------ Horner
POINTS = (0, 1, R - 1, W20, 0x6E5D4C3B2A1908F7E6D5C4B3A29180706F5E4D3C2B1A % R)


@pytest.mark.parametrize("n", [64, 65, 4096, 4097, 262144, 262145, BIG])
def test_poly_eval_dev(native, dev, n):
    cb = ref.rand_fr_bytes(50 + n, n)
    c = ref.decode(cb)
    h = dev.load(cb, off=13)
    for x in POINTS:
        assert native.fr_poly_eval_dev(h, 13, n, x) == ref.horner(c, x), x


def test_poly_eval_multi_dev(native, dev):
    """16 items of one call, lengths on both sides of every level boundary, 16 distinct points."""
    total = BIG + 40
    cb = ref.rand_fr_bytes(61, total)
    c = ref.decode(cb)
    h = dev.load(cb, off=0, tail=0)
    lens = [1, 2, 63, 64, 65, 4095, 4096, 4097, 262143, 262144, 262145, BIG, 100, 5000, 70000, 4160]
    offs = [(7 * i) % 40 for i in range(16)]
    pts = list(POINTS) + [pow(W20, 3 + i, R) * (i + 2) % R for i in range(11)]
    assert len(set(pts)) == 16
    items = [(h, o, m, x) for o, m, x in zip(offs, lens, pts)]
    assert native.fr_poly_eval_multi_dev(items) == [ref.horner(c[o:o + m], x) for o, m, x in zip(offs, lens, pts)]


def test_poly_eval_many_dev(native, dev):
    """Groups of mixed lengths across the level boundaries, per-proof strides and a shared vector, count 3,
    two point sets."""
    count = 3
    specs = [(1, 1, 0), (64, 64, 1), (65, 70, 0), (4096, 4096, 1), (4097, 4100, 0), (262145, 262145, 1),
             (262144, 0, 0), (BIG, 0, 1)]            # (length, stride, point set)
    handles, vals = [], []
    for g, (m, stride, _) in enumerate(specs):
        span = (count - 1) * stride + m
        b = ref.rand_fr_bytes(70 + g, span)
        handles.append(dev.load(b, off=g + 1, seed=g))
        vals.append(ref.decode(b))
    point_sets = [[0, R - 1, W20], [1, 0x51A7E5 * W20 % R, pow(W20, 1025, R)]]
    groups = [(h, g + 1, stride, m, sel) for g, (h, (m, stride, sel)) in enumerate(zip(handles, specs))]
    got = native.fr_poly_eval_many_dev(groups, count, point_sets)
    want = [[ref.horner(v[j * stride:j * stride + m], point_sets[sel][j]) for j in range(count)]
            for v, (m, stride, sel) in zip(vals, specs)]
    assert got == want


# ------------------------------------------------------------------ dot product
@pytest.mark.parametrize("which", ["cap-1", "cap", "cap+1", "2^20+5"])
def test_dot(native, dev, which):
    cap = 8 * 256 * native.device_info()["sm_count"]
    n = {"cap-1": cap - 1, "cap": cap, "cap+1": cap + 1, "2^20+5": (1 << 20) + 5}[which]
    ab, bb = ref.rand_fr_bytes(80 + n, n), ref.rand_fr_bytes(81 + n, n)
    a = dev.load(ab, off=3)
    b = dev.load(bb, off=17, seed=1)
    assert native.fr_dot_dev(a, 3, b, 17, n) == ref.dot(ref.decode(ab), ref.decode(bb))


# ------------------------------------------------------------------ division by (x - zeta)
ZETAS = (1, R - 1, W20, 0x7A6B5C4D3E2F1A0B9C8D7E6F5A4B3C2D1E0F % R)


@pytest.mark.parametrize("n", [2, 1024, 1025, 1026, (1 << 18) + 1, BIG])
def test_div_linear(native, dev, n):
    pb = ref.rand_fr_bytes(90 + n, n)
    p = ref.decode(pb)
    src = dev.load(pb)
    for z in ZETAS:
        dst = dev.load(bytes(32 * (n - 1)), off=4, tail=5, guard=b"zero")   # the padding beyond n - 1 stays zero
        native.div_linear_dev(src, OFF, n, z, dst, 4)
        assert dev.get(dst) == ref.encode(ref.div_linear(p, z)), z
        assert dev.intact(dst)
        dst.free()
    assert dev.intact(src) and dev.get(src) == pb


@pytest.mark.parametrize("zetas", [(1, W20, 0x1F2E3D4C5B6A798897A6B5C4D3E2F1 % R), (R - 1, 0, 5)])
def test_div_linear_many(native, dev, zetas):
    length, count, s_stride, d_stride = (1 << 18) + 1, len(zetas), (1 << 18) + 4, (1 << 18) + 2
    pb = ref.rand_fr_bytes(95, (count - 1) * s_stride + length)
    p = ref.decode(pb)
    src = dev.load(pb)
    dst = dev.zeros((count - 1) * d_stride + length - 1, off=2)
    native.div_linear_many_dev(src, OFF, s_stride, length, list(zetas), dst, 2, d_stride)
    got = ref.decode(dev.get(dst))
    for j, z in enumerate(zetas):
        assert got[j * d_stride:j * d_stride + length - 1] == ref.div_linear(p[j * s_stride:j * s_stride + length], z), j
        assert not any(got[j * d_stride + length - 1:(j + 1) * d_stride])           # gaps between outputs untouched
    assert dev.intact(dst)


# ------------------------------------------------------------------ NTT
@pytest.mark.parametrize("log_n", [10, 11, 13, 16, 17, 20, 21, 22])
def test_ntt_dev(native, dev, log_n):
    """Forward and coset-forward outputs through the fingerprint at two points; the inverse and the coset inverse
    applied to them must give back the input bit for bit."""
    n = 1 << log_n
    w = ref_path.get_root_of_unity(n)
    xb = ref.rand_fr_bytes(100 + log_n, n)
    x = ref.decode(xb)
    h = dev.load(xb)
    native.ntt_dev(h, OFF, log_n, w)
    y = ref.decode(dev.get(h))
    native.ntt_dev(h, OFF, log_n, w, inverse=True)
    assert dev.get(h) == xb
    native.ntt_dev(h, OFF, log_n, w, coset_shift=5)
    yc = ref.decode(dev.get(h))
    native.ntt_dev(h, OFF, log_n, w, inverse=True, coset_shift=5)
    assert dev.get(h) == xb
    assert dev.intact(h)
    for rho in RHO:
        dinv = ref.ntt_denominators(n, w, rho)
        assert ref.horner(y, rho) == ref.ntt_fingerprint(x, w, rho, dinv=dinv), rho
        assert ref.horner(yc, rho) == ref.ntt_fingerprint(x, w, rho, shift=5, dinv=dinv), rho


@pytest.mark.parametrize("count", [2, 3, 7])
@pytest.mark.parametrize("log_n", [0, 3, 9, 11, 14, 20])
def test_ntt_many_dev(native, dev, log_n, count):
    """Each block's fingerprint, bit-equality of each block with ntt_dev (plain and coset), the inverse giving back
    the input, and the guards before and after the blocks."""
    n = 1 << log_n
    w = ref_path.get_root_of_unity(n)
    xb = ref.rand_fr_bytes(200 + 10 * log_n + count, count * n)
    h = dev.load(xb, off=5, tail=3)
    single = dev.zeros(n)
    native.ntt_many_dev(h, 5, log_n, count, w)
    yb = dev.get(h)
    dinv = ref.ntt_denominators(n, w, RHO[0])
    for j in range(count):
        blk = slice(32 * j * n, 32 * (j + 1) * n)
        assert ref.horner(ref.decode(yb[blk]), RHO[0]) == ref.ntt_fingerprint(ref.decode(xb[blk]), w, RHO[0],
                                                                              dinv=dinv), j
        native.scalars_upload(single, OFF, xb[blk], n)
        native.ntt_dev(single, OFF, log_n, w)
        assert dev.get(single) == yb[blk], j
    native.ntt_many_dev(h, 5, log_n, count, w, inverse=True)
    assert dev.get(h) == xb
    native.ntt_many_dev(h, 5, log_n, count, w, coset_shift=5)
    cb = dev.get(h)
    for j in range(count):
        blk = slice(32 * j * n, 32 * (j + 1) * n)
        native.scalars_upload(single, OFF, xb[blk], n)
        native.ntt_dev(single, OFF, log_n, w, coset_shift=5)
        assert dev.get(single) == cb[blk], j
    assert dev.intact(h) and dev.intact(single)


# ------------------------------------------------------------------ products and division with remainder
@pytest.mark.parametrize("la,lb", [(1 << 15, 1 << 15), (1 << 14, (1 << 14) + 1), ((1 << 14) + 1, (1 << 14) + 1),
                                   (1 << 15, 1), (12345, 20000)])
def test_poly_mul(native, la, lb):
    a = ref.decode(ref.rand_fr_bytes(300 + la, la))
    b = ref.decode(ref.rand_fr_bytes(301 + lb, lb))
    c = ref.decode(native.fr_poly_mul(ref.encode(a), la, ref.encode(b), lb))
    assert ref.product_holds(a, b, c, RHO)


@pytest.mark.parametrize("la,lb,vanishing", [(1 << 15, (1 << 14) + 1, True), ((1 << 15) - 3, (1 << 12) + 1, True),
                                             (1 << 15, (1 << 14) + 3, False), (1 << 15, 2, False),
                                             (1 << 15, (1 << 15) - 5, False), ((1 << 15) + 1, 1 << 14, False)])
def test_poly_divmod(native, la, lb, vanishing):
    """Division by x^n - 1 (the fast path) and by random divisors: about half the dividend's length, a linear
    divisor (every Newton round) and a divisor almost as long as the dividend."""
    a = ref.decode(ref.rand_fr_bytes(400 + la, la))
    if vanishing:
        b = [R - 1] + [0] * (lb - 2) + [1]
    else:
        b = ref.decode(ref.rand_fr_bytes(401 + lb, lb))
        b[-1] = b[-1] or 1
    qb, rb = native.fr_poly_divmod(ref.encode(a), la, ref.encode(b), lb)
    q, r = ref.decode(qb), ref.decode(rb)
    assert ref.division_holds(a, b, q, r, RHO)
