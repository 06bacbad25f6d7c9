"""G1 / G2 MSM tests on tables of known discrete logs: entry i of a table is s_i * G, built on the device by the
fixed-base multiplication and spot-checked against the oracle, so an MSM with scalars k_i must return
(sum k_i s_i mod r) * G: one oracle scalar multiplication instead of n (the oracle's G2 MSM takes about 2 s per 200
points on a CPU).  -P has discrete log r - s and infinity has 0."""
from oracle import bn254

R = bn254.R


class Group:
    def __init__(self, native, name):
        g1 = name == "g1"
        self.native, self.name = native, name
        self.gen = bn254.G1 if g1 else bn254.G2
        self.size = 64 if g1 else 128
        self._mul = bn254.g1_mul if g1 else bn254.g2_mul
        self.gen_bytes = native.g1_bytes(self.gen) if g1 else native.g2_bytes(self.gen)
        self.decode = native.g1_from_bytes if g1 else native.g2_from_bytes
        self._fixed = native.g1_fixed_base_mul if g1 else native.g2_fixed_base_mul
        self._fixed_dev = native.g1_fixed_base_mul_dev if g1 else native.g2_fixed_base_mul_dev
        self._msm = native.g1_msm if g1 else native.g2_msm
        self.msm_table = native.g1_msm_table if g1 else native.g2_msm_table
        self.msm_dev = native.g1_msm_dev if g1 else native.g2_msm_dev

    def mul(self, k):
        return self._mul(self.gen, k % R)

    def want(self, dlogs, scalars):
        return self.mul(sum(s * k for s, k in zip(dlogs, scalars)))

    def entry(self, table, i):
        return self.decode(self.native.table_download(table, i, 1))

    def table(self, dlogs, spot=(0, -1)):
        """Plain device table with entry i = dlogs[i] * G; the entries at `spot` are checked against the oracle."""
        n = len(dlogs)
        t = self._fixed(self.gen_bytes, self.native.fr_vec_bytes([d % R for d in dlogs]), n)
        for i in spot:
            assert self.entry(t, i % n) == self.mul(dlogs[i])
        return t

    def table_dev(self, s_h, n, spot_dlogs=None):
        """Table of n entries s_i * G for the device scalars s_h (spot_dlogs: {index: s_i} to check)."""
        t = self._fixed_dev(self.gen_bytes, s_h, n)
        for i, s in (spot_dlogs or {}).items():
            assert self.entry(t, i) == self.mul(s)
        return t

    def msm_points(self, table, n, scalars):
        """The host-points entry point (zkp_g1_msm / zkp_g2_msm) over the first n entries of `table`."""
        pts = self.native.table_download(table, 0, n)
        return self._msm(pts, self.native.fr_vec_bytes(scalars), n)


def distinct_dlogs(rng, n):
    return [rng.randrange(1, R) for _ in range(n)]


def plus_minus(dlogs):
    """P_0, -P_0, P_1, -P_1, ...: pairs that cancel in every bucket they share."""
    out = []
    for s in dlogs:
        out += [s, R - s]
    return out


def auto_c(n):
    """The window width the engine picks for a plain table of n points (csrc/msm.cuh msm_plan)."""
    c = n.bit_length() - 1 - 4
    return min(max(c, 4), 16)


def part_cuts(n, parts):
    """Point ranges of a part-streamed MSM: ranges growing by 1.35x (csrc/msm.cuh MsmEngine::run)."""
    parts = min(parts, n)
    total, w = 0.0, 1.0
    for _ in range(parts):
        total += w
        w *= 1.35
    cut, acc, w = [0], 0.0, 1.0
    for p in range(parts):
        acc += w
        c = n if p + 1 == parts else int(n * (acc / total))
        c = max(c, cut[-1] + 1)
        cut.append(min(c, n))
        w *= 1.35
    return cut


def digit_scalars(c, windows=None):
    """Scalars whose signed c-bit digits stress the carries: every digit 2^c - 1 (each one becomes -1 plus a carry into
    the next window) and every digit 2^(c-1) (exactly the largest bucket), over all windows below 2^254 or over the
    lowest `windows` of them."""
    m = windows if windows is not None else 253 // c
    ones = sum(((1 << c) - 1) << (c * w) for w in range(m))
    half = sum((1 << (c - 1)) << (c * w) for w in range(m))
    return ones % R, half % R


def edge_cases(rng, n, c):
    """(name, dlogs, scalars) of the edge distributions, n >= 200 so that buckets hold more than one 64-entry task;
    c is the window width the MSM will use."""
    base = distinct_dlogs(rng, n)
    same = [base[0]] * n
    pm = plus_minus(base[:n // 2])
    with_inf = list(base)
    for i in (3, 77, 78, n - 1):
        with_inf[i] = 0
    ones, half = digit_scalars(c)
    ones1, half1 = digit_scalars(c, 1)
    rnd = lambda: [rng.randrange(R) for _ in range(n)]
    return [
        ("all zero", base, [0] * n),
        ("all one", base, [1] * n),
        ("all r - 1", base, [R - 1] * n),
        ("50% zeros", base, [rng.randrange(R) if i % 2 else 0 for i in range(n)]),
        ("all points equal", same, rnd()),
        ("same point, same scalar", same, [12345] * n),
        ("same point, same large scalar", same, [R - 12345] * n),
        ("P / -P pairs", pm, [777] * n),
        ("P / -P pairs, opposite scalars", pm, [777 if i % 2 == 0 else R - 777 for i in range(n)]),
        ("unreduced scalars", base, [(1 << 256) - 1, (1 << 255) + 5, R, R + 1, 2 * R + 3] + [1] * (n - 5)),
        ("infinity entries", with_inf, rnd()),
        ("infinity entries, one bucket", with_inf, [5] * n),
        ("digits 2^c - 1", base, [ones] * n),
        ("digits 2^c - 1, lowest window", base, [ones1] * n),
        ("digits 2^(c-1)", base, [half] * n),
        ("digits 2^(c-1), lowest window", base, [half1] * n),
        ("digit carries mixed", base, [(ones, half, ones1, half1)[i % 4] for i in range(n)]),
    ]
