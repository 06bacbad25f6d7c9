"""Thin Python layer over the C ABI: plain ints / tuples in, plain ints / tuples out.

Encoding at the boundary (include/zkp_b200.h): field elements are 32-byte little-endian canonical
integers; a G1 point is x||y; a G2 point is x.c0||x.c1||y.c0||y.c1; infinity (py_ecc ``None``) is
all zeros on input and an ``is_inf`` flag on output.
"""
import ctypes

from . import _lib
from ._lib import ZkpB200Error, NotDivisibleError, buf, check  # noqa: F401

R_MOD = 21888242871839275222246405745257275088548364400416034343698204186575808495617
P_MOD = 21888242871839275222246405745257275088696311157297823662689037894645226208583


# ------------------------------------------------------------------ encoders / decoders
def fe_bytes(x):
    return int(x).to_bytes(32, "little")


def fr_vec_bytes(xs):
    """list of int / FR (anything with __int__, already reduced) -> bytes."""
    return b"".join([int(x).to_bytes(32, "little") for x in xs])


def fr_vec_from_bytes(b, n=None):
    n = len(b) // 32 if n is None else n
    fb = int.from_bytes
    return [fb(b[32 * i:32 * i + 32], "little") for i in range(n)]


def g1_bytes(pt):
    if pt is None:
        return bytes(64)
    return int(pt[0]).to_bytes(32, "little") + int(pt[1]).to_bytes(32, "little")


def g1_vec_bytes(pts):
    return b"".join([g1_bytes(p) for p in pts])


def g2_bytes(pt):
    if pt is None:
        return bytes(128)
    (x, y) = pt
    xc = x.coeffs if hasattr(x, "coeffs") else x
    yc = y.coeffs if hasattr(y, "coeffs") else y
    return b"".join(int(v).to_bytes(32, "little") for v in (xc[0], xc[1], yc[0], yc[1]))


def g2_vec_bytes(pts):
    return b"".join([g2_bytes(p) for p in pts])


# Compressed points (csrc/point_codec.cuh): x plus a y-sign flag (bit 255) and an infinity flag (bit 254) in the last
# 32-byte field element.  Encoding a point the caller holds is one comparison; decoding needs a square root and is
# done on the device (g1_table_load_compressed / g2_table_load_compressed).
_HALF_P = (P_MOD - 1) // 2
_FLAG_SIGN, _FLAG_INF = 1 << 255, 1 << 254


def g1_compressed_bytes(pt):
    if pt is None:
        return _FLAG_INF.to_bytes(32, "little")
    x, y = int(pt[0]), int(pt[1])
    return (x | (_FLAG_SIGN if y > _HALF_P else 0)).to_bytes(32, "little")


def g1_vec_compressed_bytes(pts):
    return b"".join([g1_compressed_bytes(p) for p in pts])


def g2_compressed_bytes(pt):
    if pt is None:
        return bytes(32) + _FLAG_INF.to_bytes(32, "little")
    (x, y) = pt
    xc = x.coeffs if hasattr(x, "coeffs") else x
    yc = y.coeffs if hasattr(y, "coeffs") else y
    y0, y1 = int(yc[0]), int(yc[1])
    sign = y1 > _HALF_P if y1 else y0 > _HALF_P
    return int(xc[0]).to_bytes(32, "little") + (int(xc[1]) | (_FLAG_SIGN if sign else 0)).to_bytes(32, "little")


def g2_vec_compressed_bytes(pts):
    return b"".join([g2_compressed_bytes(p) for p in pts])


def g1_from_bytes(b, is_inf=False):
    if is_inf or b == bytes(64):
        return None
    return (int.from_bytes(b[:32], "little"), int.from_bytes(b[32:64], "little"))


def g2_from_bytes(b, is_inf=False):
    if is_inf or b == bytes(128):
        return None
    v = [int.from_bytes(b[32 * i:32 * i + 32], "little") for i in range(4)]
    return ((v[0], v[1]), (v[2], v[3]))


# ------------------------------------------------------------------ device info / timing
def device_info():
    l = _lib.lib()
    name = ctypes.create_string_buffer(128)
    sm, maj, mnr, khz = (ctypes.c_int() for _ in range(4))
    check(l.zkp_device_info(name, 128, ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mnr), ctypes.byref(khz)))
    return {"name": name.value.decode(), "sm_count": sm.value, "cc": (maj.value, mnr.value),
            "sm_clock_khz": khz.value}


def device_pci_bus_id():
    out = ctypes.create_string_buffer(32)
    check(_lib.lib().zkp_device_pci_bus_id(out, 32))
    return out.value.decode().lower()


def device_mem_info():
    f, t = ctypes.c_uint64(), ctypes.c_uint64()
    check(_lib.lib().zkp_device_mem_info(ctypes.byref(f), ctypes.byref(t)))
    return f.value, t.value


def launch_count():
    return int(_lib.lib().zkp_launch_count())


def timer_start():
    check(_lib.lib().zkp_timer_start())


def timer_stop():
    ms = ctypes.c_float()
    check(_lib.lib().zkp_timer_stop(ctypes.byref(ms)))
    return ms.value


def sync():
    check(_lib.lib().zkp_sync())


def imad_peak(variant=0):
    g = ctypes.c_double()
    clk = ctypes.c_double()
    check(_lib.lib().zkp_imad_peak(variant, ctypes.byref(g), ctypes.byref(clk)))
    return g.value


def latency_probe(mode):
    """ns per operation for a lone thread (see zkp_latency_probe)."""
    ns = ctypes.c_double()
    check(_lib.lib().zkp_latency_probe(mode, ctypes.byref(ns)))
    return ns.value


def msm_profile(enable):
    check(_lib.lib().zkp_msm_profile(1 if enable else 0))


def msm_last_profile(stage=None):
    """Device microseconds of the named stage(s) of the most recent MSM (None = whole MSM)."""
    us = ctypes.c_float()
    check(_lib.lib().zkp_msm_last_profile(stage.encode() if stage else None, ctypes.byref(us)))
    return us.value


class PinnedBuffer:
    """Page-locked host memory (cudaHostAlloc) exposed as a writable ctypes array."""

    def __init__(self, nbytes):
        p = ctypes.c_void_p()
        check(_lib.lib().zkp_pinned_alloc(nbytes, ctypes.byref(p)))
        self.addr = p.value
        self.nbytes = nbytes
        self.view = (ctypes.c_char * nbytes).from_address(self.addr)

    def write(self, data, offset=0):
        ctypes.memmove(self.addr + offset, data, len(data))

    def free(self):
        if self.addr:
            _lib.lib().zkp_pinned_free(self.addr)
            self.addr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def set_window_bits(c):
    check(_lib.lib().zkp_msm_set_window_bits(int(c)))


def msm_set_option(name, value):
    """Engine tunables for measurements ("sort", "split", "window_bits"; 0 = automatic)."""
    check(_lib.lib().zkp_msm_set_option(name.encode(), int(value)))


# ------------------------------------------------------------------ handles
class DeviceHandle:
    """Owns a device-resident table or scalar vector; freed on garbage collection."""

    def __init__(self, handle, n, kind):
        self.handle = handle
        self.n = n
        self.kind = kind

    def free(self):
        if self.handle:
            try:
                _lib.lib().zkp_free(self.handle)
            finally:
                self.handle = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _load(fn_name, data, n, kind):
    h = ctypes.c_uint64()
    check(getattr(_lib.lib(), fn_name)(buf(data), n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, kind)


def g1_table_load(pts_bytes, n):
    return _load("zkp_g1_table_load", pts_bytes, n, "g1")


def g2_table_load(pts_bytes, n):
    return _load("zkp_g2_table_load", pts_bytes, n, "g2")


def table_precompute(handle, window_bits=0):
    """Window-precomputed layout for a static table; window_bits = 0 lets the library pick the width
    for the table size (measured rule, csrc/msm.cuh msm_auto_precomputed_c)."""
    fn = _lib.lib().zkp_g1_table_precompute if handle.kind == "g1" else _lib.lib().zkp_g2_table_precompute
    check(fn(handle.handle, int(window_bits)))
    c = ctypes.c_int()
    check(_lib.lib().zkp_table_window_bits(handle.handle, ctypes.byref(c)))
    handle.pre_c = c.value
    return c.value


def scalars_load(sc_bytes, n):
    return _load("zkp_scalars_load", sc_bytes, n, "fr")


def scalars_generate(seed, n):
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_scalars_generate(seed, n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, "fr")


def scalars_download(handle, offset, n):
    out = bytearray(32 * n)
    check(_lib.lib().zkp_scalars_download(handle.handle, offset, n, buf(out)))
    return bytes(out)


def table_download(handle, offset, n):
    sz = 64 if handle.kind == "g1" else 128
    out = bytearray(sz * n)
    check(_lib.lib().zkp_table_download(handle.handle, offset, n, buf(out)))
    return bytes(out)


class InvalidPointError(ValueError):
    """A compressed encoding the device decoder rejected; `index` is the lowest such index of the call."""

    def __init__(self, msg, index):
        super().__init__(msg)
        self.index = index


def _load_compressed(what, enc, n, size, *extra):
    enc = bytes(enc)
    if len(enc) != size * n:
        raise ValueError("%s: %d compressed points need %d bytes, got %d" % (what, n, size * n, len(enc)))
    h, bad = ctypes.c_uint64(), ctypes.c_uint64()
    check(getattr(_lib.lib(), "zkp_" + what)(buf(enc) if n else None, n, *extra, ctypes.byref(h), ctypes.byref(bad)))
    if _first_bad(bad.value) is not None:
        raise InvalidPointError("%s: invalid compressed point at index %d" % (what, bad.value), bad.value)
    return DeviceHandle(h.value, n, "g1" if size == 32 else "g2")


def g1_table_load_compressed(enc, n):
    """n compressed G1 points (32 B each) -> a plain table, decoded on the device.  Raises ValueError naming the lowest
    index whose encoding is invalid (bad flags, x >= p, or no point with that x)."""
    return _load_compressed("g1_table_load_compressed", enc, n, 32)


def g2_table_load_compressed(enc, n, subgroup_check=True):
    """n compressed G2 points (64 B each) -> a plain table; with subgroup_check a point outside G2 is invalid too."""
    return _load_compressed("g2_table_load_compressed", enc, n, 64, 1 if subgroup_check else 0)


def table_download_compressed(handle, offset, n):
    """Points [offset, offset + n) of a G1 / G2 table as compressed encodings (32 / 64 B each)."""
    out = bytearray((32 if handle.kind == "g1" else 64) * n)
    check(_lib.lib().zkp_table_download_compressed(handle.handle, offset, n, buf(out)))
    return bytes(out)


def g1_fixed_base_mul(base_bytes, sc_bytes, n):
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_g1_fixed_base_mul(buf(base_bytes), buf(sc_bytes), n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, "g1")


def g2_fixed_base_mul(base_bytes, sc_bytes, n):
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_g2_fixed_base_mul(buf(base_bytes), buf(sc_bytes), n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, "g2")


def g2_fixed_base_mul_dev(base_bytes, scalars, n):
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_g2_fixed_base_mul_dev(buf(base_bytes), scalars.handle, n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, "g2")


def scalars_alloc(n):
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_scalars_alloc(n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, "fr")


def scalars_copy(dst, dst_off, src, src_off, n):
    check(_lib.lib().zkp_scalars_copy(dst.handle, dst_off, src.handle, src_off, n))


def scalars_upload(dst, dst_off, data, n):
    check(_lib.lib().zkp_scalars_upload(dst.handle, dst_off, buf(data), n))


def scalars_scale(h, off, n, k):
    check(_lib.lib().zkp_scalars_scale(h.handle, off, n, buf(fe_bytes(k))))


def fr_poly_eval_dev(h, off, n, x):
    out = bytearray(32)
    check(_lib.lib().zkp_fr_poly_eval_dev(h.handle, off, n, buf(fe_bytes(x)), buf(out)))
    return int.from_bytes(out, "little")


def groth16_quotient_dev(a, b, c, length, z, z_len, want_remainder=True):
    """(H, remainder) handles; with want_remainder=False only H is computed and (H, None) returned."""
    hq, hr = ctypes.c_uint64(), ctypes.c_uint64()
    check(_lib.lib().zkp_groth16_quotient_dev(a.handle, b.handle, c.handle, length, z.handle, z_len,
                                              ctypes.byref(hq), ctypes.byref(hr) if want_remainder else None))
    return (DeviceHandle(hq.value, 2 * length - z_len, "fr"),
            DeviceHandle(hr.value, z_len - 1, "fr") if want_remainder else None)


def groth16_quotient_batch_dev(a, b, c, length, count, z, z_len):
    """Handle of count quotients (2 * length - z_len coefficients each, back to back); proof j's a, b, c at j * length."""
    hq = ctypes.c_uint64()
    check(_lib.lib().zkp_groth16_quotient_batch_dev(a.handle, b.handle, c.handle, length, count, z.handle, z_len,
                                                    ctypes.byref(hq)))
    return DeviceHandle(hq.value, count * (2 * length - z_len), "fr")


def groth16_batch_scalars_dev(uA, uB, h, rx, k, m_priv, rs, ss):
    """(scA, scB, scC) handles of len(rs) proofs: uA | 1 | r, uB | 1 | s and r uB + s uA | r | rx | H | s | s r."""
    count = len(rs)
    ha, hb, hc = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
    check(_lib.lib().zkp_groth16_batch_scalars_dev(uA.handle, uB.handle, h.handle if h is not None else 0,
                                                   rx.handle if rx is not None else 0, k, m_priv, count,
                                                   buf(fr_vec_bytes(rs)), buf(fr_vec_bytes(ss)), ctypes.byref(ha),
                                                   ctypes.byref(hb), ctypes.byref(hc)))
    nC = 2 * k + 2 + m_priv
    return (DeviceHandle(ha.value, count * (k + 2), "fr"), DeviceHandle(hb.value, count * (k + 2), "fr"),
            DeviceHandle(hc.value, count * nC, "fr"))


def groth16_msms_dev(ta, sa, na, tb2, sb, nb, tc, sc, nc):
    """A (G1), B (G2), C' (G1) of one proof with the G2 MSM overlapped on a second stream."""
    oa, ob, oc = bytearray(64), bytearray(128), bytearray(64)
    inf = (ctypes.c_int * 3)()
    check(_lib.lib().zkp_groth16_msms_dev(ta.handle, sa.handle, na, tb2.handle, sb.handle, nb, tc.handle, sc.handle, nc,
                                          buf(oa), buf(ob), buf(oc), inf))
    return (g1_from_bytes(bytes(oa), bool(inf[0])), g2_from_bytes(bytes(ob), bool(inf[1])),
            g1_from_bytes(bytes(oc), bool(inf[2])))


def g1_fixed_base_mul_dev(base_bytes, scalars, n):
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_g1_fixed_base_mul_dev(buf(base_bytes), scalars.handle, n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, "g1")


def _table_scale(fn_name, table, offset, scalars, sc_offset, n):
    h = ctypes.c_uint64()
    check(getattr(_lib.lib(), fn_name)(table.handle, offset, scalars.handle, sc_offset, n, ctypes.byref(h)))
    return DeviceHandle(h.value, n, table.kind)


def g1_table_scale(table, offset, scalars, sc_offset, n):
    """New plain G1 table: out[i] = scalars[sc_offset + i] * table[offset + i] (scalars reduced mod r)."""
    return _table_scale("zkp_g1_table_scale", table, offset, scalars, sc_offset, n)


def g2_table_scale(table, offset, scalars, sc_offset, n):
    return _table_scale("zkp_g2_table_scale", table, offset, scalars, sc_offset, n)


def _first_bad(v):
    return None if v == (1 << 64) - 1 else v


def g1_table_validate(table, offset, n):
    """Lowest index in [offset, offset + n) whose point is not on the curve, or None (infinity is valid)."""
    bad = ctypes.c_uint64()
    check(_lib.lib().zkp_g1_table_validate(table.handle, offset, n, ctypes.byref(bad)))
    return _first_bad(bad.value)


def g2_table_validate(table, offset, n, subgroup_check=False):
    """Lowest index in [offset, offset + n) whose point is not on the twist or, with subgroup_check, not in G2;
    None if every point passes."""
    bad = ctypes.c_uint64()
    check(_lib.lib().zkp_g2_table_validate(table.handle, offset, n, 1 if subgroup_check else 0, ctypes.byref(bad)))
    return _first_bad(bad.value)


# ------------------------------------------------------------------ MSM
def _msm_out(group):
    return bytearray(64 if group == 1 else 128), ctypes.c_int()


def g1_msm(pts_bytes, sc_bytes, n):
    out, inf = _msm_out(1)
    check(_lib.lib().zkp_g1_msm(buf(pts_bytes), buf(sc_bytes), n, buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value))


def g2_msm(pts_bytes, sc_bytes, n):
    out, inf = _msm_out(2)
    check(_lib.lib().zkp_g2_msm(buf(pts_bytes), buf(sc_bytes), n, buf(out), ctypes.byref(inf)))
    return g2_from_bytes(bytes(out), bool(inf.value))


def g1_msm_table(table, offset, sc_bytes, n):
    out, inf = _msm_out(1)
    check(_lib.lib().zkp_g1_msm_table(table.handle, offset, buf(sc_bytes), n, buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value))


def g2_msm_table(table, offset, sc_bytes, n):
    out, inf = _msm_out(2)
    check(_lib.lib().zkp_g2_msm_table(table.handle, offset, buf(sc_bytes), n, buf(out), ctypes.byref(inf)))
    return g2_from_bytes(bytes(out), bool(inf.value))


def g1_msm_dev(table, offset, scalars, sc_offset, n):
    out, inf = _msm_out(1)
    check(_lib.lib().zkp_g1_msm_dev(table.handle, offset, scalars.handle, sc_offset, n, buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value))


def g2_msm_dev(table, offset, scalars, sc_offset, n):
    out, inf = _msm_out(2)
    check(_lib.lib().zkp_g2_msm_dev(table.handle, offset, scalars.handle, sc_offset, n, buf(out), ctypes.byref(inf)))
    return g2_from_bytes(bytes(out), bool(inf.value))


def g1_msm_dev_batch(table, items):
    """items: list of (scalars_handle, sc_offset, point_offset, n) -> list of points (pipelined on two streams)."""
    k = len(items)
    if k == 0:
        return []
    arr = lambda vals: (ctypes.c_uint64 * k)(*vals)
    out = bytearray(64 * k)
    inf = (ctypes.c_int * k)()
    check(_lib.lib().zkp_g1_msm_dev_batch(table.handle, k, arr([it[0].handle for it in items]), arr([it[1] for it in items]),
                                          arr([it[2] for it in items]), arr([it[3] for it in items]), buf(out), inf))
    return [g1_from_bytes(bytes(out[64 * i:64 * i + 64]), bool(inf[i])) for i in range(k)]


def msm_dev_many(table, offset, n, count, scalars, sc_offset=0):
    """count MSMs over the points [offset, offset + n) of `table` (G1 or G2 by its kind), vector j of scalars at
    sc_offset + j * n -> list of count points.  One Pippenger pass for the whole batch."""
    g1 = table.kind == "g1"
    sz = 64 if g1 else 128
    out = bytearray(sz * max(count, 1))
    inf = (ctypes.c_int * max(count, 1))()
    fn = _lib.lib().zkp_g1_msm_dev_many if g1 else _lib.lib().zkp_g2_msm_dev_many
    check(fn(table.handle, offset, n, count, scalars.handle, sc_offset, buf(out), inf))
    dec = g1_from_bytes if g1 else g2_from_bytes
    return [dec(bytes(out[sz * j:sz * j + sz]), bool(inf[j])) for j in range(count)]


def g1_msm_dev_partial(table, offset, scalars, sc_offset, n, out_addr=None):
    """XYZZ partial sum (128 B, Montgomery) of one rank's point range.  With `out_addr` (a host or
    device address on this GPU) the partial is written there and None returned."""
    if out_addr is not None:
        check(_lib.lib().zkp_g1_msm_dev_partial(table.handle, offset, scalars.handle, sc_offset, n, buf(int(out_addr))))
        return None
    out = bytearray(128)
    check(_lib.lib().zkp_g1_msm_dev_partial(table.handle, offset, scalars.handle, sc_offset, n, buf(out)))
    return bytes(out)


# ------------------------------------------------------------------ multi-GPU (one process per GPU)
COMM_ID_BYTES = 128


def comm_unique_id():
    """Rank 0: the 128-byte NCCL id every rank passes to comm_init."""
    out = bytearray(COMM_ID_BYTES)
    check(_lib.lib().zkp_comm_unique_id(buf(out)))
    return bytes(out)


def comm_init(rank, world, comm_id):
    if len(comm_id) != COMM_ID_BYTES:
        raise ValueError("a communicator id is %d bytes" % COMM_ID_BYTES)
    check(_lib.lib().zkp_comm_init(int(rank), int(world), buf(bytes(comm_id))))


def comm_info():
    r, w, v = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    check(_lib.lib().zkp_comm_info(ctypes.byref(r), ctypes.byref(w), ctypes.byref(v)))
    return {"rank": r.value, "world": w.value, "nccl_version": v.value}


def comm_barrier():
    check(_lib.lib().zkp_comm_barrier())


def comm_destroy():
    check(_lib.lib().zkp_comm_destroy())


def g1_msm_multi(table, offset, scalars, sc_offset, n):
    """Collective: this rank's shard of a sharded G1 MSM; every rank gets the affine result."""
    out, inf = _msm_out(1)
    check(_lib.lib().zkp_g1_msm_multi(table.handle, offset, scalars.handle, sc_offset, n, buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value))


def g1_msm_multi_table(table, offset, sc_bytes, n):
    """The same with this rank's scalars in host memory (bytes or a pinned address)."""
    out, inf = _msm_out(1)
    check(_lib.lib().zkp_g1_msm_multi_table(table.handle, offset, buf(sc_bytes), n, buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value))


def g2_msm_multi(table, offset, scalars, sc_offset, n):
    out, inf = _msm_out(2)
    check(_lib.lib().zkp_g2_msm_multi(table.handle, offset, scalars.handle, sc_offset, n, buf(out), ctypes.byref(inf)))
    return g2_from_bytes(bytes(out), bool(inf.value))


def msm_dev_begin(table, offset, scalars, sc_offset, n):
    """Asynchronous msm_dev on the library's second stream (G1 or G2 by the table's kind); msm_dev_end(kind)
    fetches the point.  What is called in between runs beside it."""
    fn = _lib.lib().zkp_g1_msm_dev_begin if table.kind == "g1" else _lib.lib().zkp_g2_msm_dev_begin
    check(fn(table.handle, offset, scalars.handle, sc_offset, n))


def msm_dev_end(kind):
    out, inf = _msm_out(1 if kind == "g1" else 2)
    fn = _lib.lib().zkp_g1_msm_dev_end if kind == "g1" else _lib.lib().zkp_g2_msm_dev_end
    check(fn(buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value)) if kind == "g1" else g2_from_bytes(bytes(out), bool(inf.value))


def msm_multi_begin(table, offset, scalars, sc_offset, n):
    """Collective, asynchronous: starts this rank's shard of a sharded MSM (G1 or G2 by the table's kind) on the
    library's second stream; msm_multi_end(kind) fetches the point."""
    fn = _lib.lib().zkp_g1_msm_multi_begin if table.kind == "g1" else _lib.lib().zkp_g2_msm_multi_begin
    check(fn(table.handle, offset, scalars.handle, sc_offset, n))


def msm_multi_end(kind):
    out, inf = _msm_out(1 if kind == "g1" else 2)
    fn = _lib.lib().zkp_g1_msm_multi_end if kind == "g1" else _lib.lib().zkp_g2_msm_multi_end
    check(fn(buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value)) if kind == "g1" else g2_from_bytes(bytes(out), bool(inf.value))


def g1_combine_partials(partials_bytes, count):
    out, inf = _msm_out(1)
    check(_lib.lib().zkp_g1_combine_partials(buf(partials_bytes), count, buf(out), ctypes.byref(inf)))
    return g1_from_bytes(bytes(out), bool(inf.value))


# ------------------------------------------------------------------ Fr vectors
def fr_ntt(data_bytes, log_n, omega, inverse=False, coset_shift=None):
    data = bytearray(data_bytes)
    cs = fe_bytes(coset_shift) if coset_shift is not None else None
    check(_lib.lib().zkp_fr_ntt(buf(data), log_n, buf(fe_bytes(omega)), 1 if inverse else 0, buf(cs)))
    return bytes(data)


def fr_vec_op(op, a_bytes, b_bytes, n):
    out = bytearray(32 * n)
    check(_lib.lib().zkp_fr_vec_op(op, buf(a_bytes), buf(b_bytes), n, buf(out)))
    return bytes(out)


def fr_vec_matrix(vec_bytes, mat_bytes, rows, cols):
    out = bytearray(32 * cols)
    check(_lib.lib().zkp_fr_vec_matrix(buf(vec_bytes), buf(mat_bytes), rows, cols, buf(out)))
    return bytes(out)


def fr_batch_inverse(a_bytes, n):
    out = bytearray(32 * n)
    check(_lib.lib().zkp_fr_batch_inverse(buf(a_bytes), n, buf(out)))
    return bytes(out)


def fr_prefix_product(a_bytes, n):
    out = bytearray(32 * n)
    check(_lib.lib().zkp_fr_prefix_product(buf(a_bytes), n, buf(out)))
    return bytes(out)


def fr_poly_eval(coeff_bytes, n, x):
    out = bytearray(32)
    check(_lib.lib().zkp_fr_poly_eval(buf(coeff_bytes), n, buf(fe_bytes(x)), buf(out)))
    return int.from_bytes(out, "little")


def fr_poly_mul(a_bytes, a_len, b_bytes, b_len):
    out = bytearray(32 * (a_len + b_len - 1))
    check(_lib.lib().zkp_fr_poly_mul(buf(a_bytes), a_len, buf(b_bytes), b_len, buf(out)))
    return bytes(out)


def fr_poly_divmod(a_bytes, a_len, b_bytes, b_len):
    q = bytearray(32 * (a_len - b_len + 1))
    r = bytearray(32 * max(b_len - 1, 1))
    check(_lib.lib().zkp_fr_poly_divmod(buf(a_bytes), a_len, buf(b_bytes), b_len, buf(q), buf(r)))
    return bytes(q), bytes(r[:32 * (b_len - 1)])


def groth16_quotient(a_bytes, b_bytes, c_bytes, length, z_bytes, z_len):
    h = bytearray(32 * (2 * length - 1 - z_len + 1))
    r = bytearray(32 * max(z_len - 1, 1))
    check(_lib.lib().zkp_groth16_quotient(buf(a_bytes), buf(b_bytes), buf(c_bytes), length, buf(z_bytes), z_len,
                                          buf(h), buf(r)))
    return bytes(h), bytes(r[:32 * (z_len - 1)])


# ------------------------------------------------------------------ pairings (verifier side)
def pairing(g2_b, g1_b):
    """e(Q, P) for one G2 point (128 B) and one G1 point (64 B) -> py_ecc's FQ12 coefficients (12 ints, w^0..w^11)."""
    out = bytearray(384)
    check(_lib.lib().zkp_pairing(buf(bytes(g2_b)), buf(bytes(g1_b)), buf(out)))
    return fr_vec_from_bytes(bytes(out), 12)


def pairing_check(g2_b, g1_b, n, scalars=None, g2_subgroup_check=False):
    """[ prod_i e(Q_i, k_i P_i) == 1 ] over n pairs (n x 128 B, n x 64 B; scalars: n x 32 B or None for k_i = 1)."""
    ok = ctypes.c_int()
    check(_lib.lib().zkp_pairing_check(buf(bytes(g2_b)) if n else None, buf(bytes(g1_b)) if n else None,
                                       buf(bytes(scalars)) if scalars is not None and n else None, n,
                                       1 if g2_subgroup_check else 0, ctypes.byref(ok)))
    return bool(ok.value)


def dbg_fp12_op(op, a_bytes, b_bytes, n):
    out = bytearray(384 * n)
    check(_lib.lib().zkp_dbg_fp12_op(op, buf(a_bytes), buf(b_bytes), n, buf(out)))
    return bytes(out)


# ------------------------------------------------------------------ diagnostics (tests)
def debug_check_guards():
    """(live device blocks, blocks whose canaries were overwritten) -- needs ZKP_B200_GUARD=1 in the environment."""
    live, bad = ctypes.c_uint64(), ctypes.c_uint64()
    check(_lib.lib().zkp_debug_check_guards(ctypes.byref(live), ctypes.byref(bad)))
    return live.value, bad.value


def dbg_field_op(field, op, a_bytes, b_bytes, n):
    out = bytearray((64 if field == 2 else 32) * n)
    check(_lib.lib().zkp_dbg_field_op(field, op, buf(a_bytes), buf(b_bytes), n, buf(out)))
    return bytes(out)


def dbg_point_add(group, a_bytes, b_bytes, n):
    sz = 64 if group == 0 else 128
    out = bytearray(sz * n)
    check(_lib.lib().zkp_dbg_point_add(group, buf(a_bytes), buf(b_bytes), n, buf(out)))
    return bytes(out)


# ------------------------------------------------------------------ device-resident vector ops (handles)
def vec_op_dev(op, dst, dst_off, a, a_off, b, b_off, n):
    check(_lib.lib().zkp_fr_vec_op_dev(op, dst.handle, dst_off, a.handle, a_off, b.handle, b_off, n))


def axpy_dev(dst, dst_off, k, src, src_off, n):
    check(_lib.lib().zkp_fr_axpy_dev(dst.handle, dst_off, buf(fe_bytes(k)), src.handle, src_off, n))


def fr_poly_eval_multi_dev(items):
    """items = [(handle, offset, length, x)] (at most 16) -> the values, one batched set of launches."""
    k = len(items)
    if not k:
        return []
    arr = lambda vals: (ctypes.c_uint64 * k)(*vals)
    out = bytearray(32 * k)
    xs = b"".join(fe_bytes(it[3]) for it in items)
    check(_lib.lib().zkp_fr_poly_eval_multi_dev(k, arr([it[0].handle for it in items]), arr([it[1] for it in items]),
                                                arr([it[2] for it in items]), buf(xs), buf(out)))
    return fr_vec_from_bytes(bytes(out))


def lincomb_dev(dst, dst_off, n, items):
    """dst[dst_off + i] = sum over items (coeff, handle, offset, length) of coeff * handle[offset + i], i < n."""
    k = len(items)
    arr = lambda vals: (ctypes.c_uint64 * max(k, 1))(*vals)
    check(_lib.lib().zkp_fr_lincomb_dev(dst.handle, dst_off, n, k, arr([it[1].handle for it in items]),
                                        arr([it[2] for it in items]), arr([it[3] for it in items]),
                                        buf(b"".join(fe_bytes(it[0]) for it in items)) if k else None))


def scalars_add_const(h, off, n, k):
    check(_lib.lib().zkp_scalars_add_const(h.handle, off, n, buf(fe_bytes(k))))


def scalars_fill_powers(h, off, n, first, base):
    check(_lib.lib().zkp_scalars_fill_powers(h.handle, off, n, buf(fe_bytes(first)), buf(fe_bytes(base))))


def scalars_convert(h, off, n, to_montgomery):
    check(_lib.lib().zkp_scalars_convert(h.handle, off, n, 1 if to_montgomery else 0))


def scalars_is_zero(h, off, n):
    flag = ctypes.c_int()
    check(_lib.lib().zkp_scalars_is_zero(h.handle, off, n, ctypes.byref(flag)))
    return bool(flag.value)


def batch_inverse_dev(h, off, n, montgomery=False):
    check(_lib.lib().zkp_fr_batch_inverse_dev(h.handle, off, n, 1 if montgomery else 0))


def scan_dev(op, dst, dst_off, src, src_off, n):
    check(_lib.lib().zkp_fr_scan_dev(op, dst.handle, dst_off, src.handle, src_off, n))


def fr_dot_dev(a, a_off, b, b_off, n):
    """sum_i a[a_off + i] * b[b_off + i] mod r of two device-resident canonical vectors."""
    out = bytearray(32)
    check(_lib.lib().zkp_fr_dot_dev(a.handle, a_off, b.handle, b_off, n, buf(out)))
    return int.from_bytes(out, "little")


def div_linear_dev(src, src_off, n, zeta, dst, dst_off):
    check(_lib.lib().zkp_fr_div_linear_dev(src.handle, src_off, n, buf(fe_bytes(zeta)), dst.handle, dst_off))


def ntt_dev(h, off, log_n, omega, inverse=False, coset_shift=None):
    cs = fe_bytes(coset_shift) if coset_shift is not None else None
    check(_lib.lib().zkp_fr_ntt_dev(h.handle, off, log_n, buf(fe_bytes(omega)), 1 if inverse else 0, buf(cs)))


def plonk_perm_terms_dev(a, b, c, s1, s2, s3, n, omega, beta, gamma, num, den):
    check(_lib.lib().zkp_plonk_perm_terms_dev(a.handle, b.handle, c.handle, s1.handle, s2.handle, s3.handle, n,
                                              buf(fe_bytes(omega)), buf(fe_bytes(beta)), buf(fe_bytes(gamma)),
                                              num.handle, den.handle))


def plonk_coset_setup_dev(n, ext, g, w8, x_out, l1f_out, zh8_out):
    check(_lib.lib().zkp_plonk_coset_setup_dev(n, ext, buf(fe_bytes(g)), buf(fe_bytes(w8)), buf(fe_bytes(pow(g, n, R_MOD))),
                                               buf(fe_bytes(pow(w8, n, R_MOD))), x_out.handle, l1f_out.handle,
                                               zh8_out.handle))


def plonk_quotient_dev(evals12, n, ext, x, l1f, zh8, beta, gamma, alpha, t_out):
    arr = (ctypes.c_uint64 * 12)(*[h.handle for h in evals12])
    check(_lib.lib().zkp_plonk_quotient_dev(arr, n, ext, x.handle, l1f.handle, zh8.handle, buf(fe_bytes(beta)),
                                            buf(fe_bytes(gamma)), buf(fe_bytes(alpha)), t_out.handle))


# ------------------------------------------------------------------ batch PLONK proving (count proofs per call)
def _u64s(vals):
    return (ctypes.c_uint64 * max(len(vals), 1))(*vals)


def _fr_rows(what, rows, count, width):
    """count rows of `width` scalars -> bytes (reduced mod r); the C side reads exactly count * width of them."""
    rows = [list(r) for r in rows]
    if len(rows) != count or any(len(r) != width for r in rows):
        raise ValueError("%s: expected %d rows of %d scalars" % (what, count, width))
    return fr_vec_bytes([int(x) % R_MOD for r in rows for x in r])


def ntt_many_dev(h, off, log_n, count, omega, inverse=False, coset_shift=None):
    """count contiguous transforms of 2^log_n elements from h[off] (ntt_dev each)."""
    cs = fe_bytes(coset_shift) if coset_shift is not None else None
    check(_lib.lib().zkp_fr_ntt_many_dev(h.handle, off, log_n, buf(fe_bytes(omega)), 1 if inverse else 0, buf(cs), count))


def plonk_blind_many_dev(src, src_off, src_stride, n, nvec, blinds, dst, dst_off, dst_stride):
    """dst_v = src_v + (b_v0 + b_v1 x + ...)(x^n - 1) at dst_stride, v < nvec; blinds: nvec lists of k scalars."""
    k = len(blinds[0]) if nvec else 0
    flat = _fr_rows("plonk_blind_many_dev: blinds", blinds, nvec, k)
    check(_lib.lib().zkp_plonk_blind_many_dev(src.handle, src_off, src_stride, n, nvec, buf(flat) if k else None, k,
                                              dst.handle, dst_off, dst_stride))


def plonk_perm_terms_many_dev(a, b, c, off, s1, s2, s3, n, omega, betas, gammas, num, den):
    """plonk_perm_terms_dev for len(betas) proofs, witness j at off + j * n of a, b, c."""
    count = len(betas)
    ch = _fr_rows("plonk_perm_terms_many_dev: betas, gammas", [betas, gammas], 2, count)
    check(_lib.lib().zkp_plonk_perm_terms_many_dev(a.handle, b.handle, c.handle, off, s1.handle, s2.handle, s3.handle, n,
                                                   count, buf(fe_bytes(omega)), buf(ch[:32 * count]),
                                                   buf(ch[32 * count:]), num.handle, den.handle))


def scan_many_dev(op, dst, dst_off, src, src_off, seg, count):
    """scan_dev over count segments of seg elements, each starting afresh (op 0 product, 1 sum)."""
    check(_lib.lib().zkp_fr_scan_many_dev(op, dst.handle, dst_off, src.handle, src_off, seg, count))


def plonk_coset_inputs_many_dev(wires, z, n, count, log_N, out):
    check(_lib.lib().zkp_plonk_coset_inputs_many_dev(wires.handle, z.handle, n, count, log_N, out.handle))


def plonk_quotient_many_dev(evals, circuit8, n, ext, x, l1f, zh8, betas, gammas, alphas, t_out):
    """plonk_quotient_dev for len(betas) proofs: evals holds the blocks a_*, b_*, c_*, z_* of N = ext * n each."""
    count = len(betas)
    if len(circuit8) != 8:
        raise ValueError("plonk_quotient_many_dev: 8 circuit coset evaluations, got %d" % len(circuit8))
    ch = _fr_rows("plonk_quotient_many_dev: betas, gammas, alphas", [betas, gammas, alphas], 3, count)
    check(_lib.lib().zkp_plonk_quotient_many_dev(evals.handle, _u64s([h.handle for h in circuit8]), n, ext, count,
                                                 x.handle, l1f.handle, zh8.handle, buf(ch[:32 * count]),
                                                 buf(ch[32 * count:64 * count]), buf(ch[64 * count:]), t_out.handle))


def plonk_divisible_many_dev(t, n, ext, count):
    """Lowest proof index whose quotient block has a non-zero coefficient at 3n + 6 or above, or None."""
    bad = ctypes.c_uint64()
    check(_lib.lib().zkp_plonk_divisible_many_dev(t.handle, n, ext, count, ctypes.byref(bad)))
    return _first_bad(bad.value)


def plonk_split_t_many_dev(t, n, ext, count, out):
    check(_lib.lib().zkp_plonk_split_t_many_dev(t.handle, n, ext, count, out.handle))


def fr_poly_eval_many_dev(groups, count, point_sets):
    """groups = [(handle, offset, stride, length, point_set)] (stride 0: shared by every proof), point_sets = lists of
    count points -> values[g][j] = p_g,j(point_sets[sel_g][j]).  One batched set of Horner launches."""
    g = len(groups)
    if not g or not count:
        return [[] for _ in range(g)]
    if any(not 0 <= it[4] < len(point_sets) for it in groups):
        raise ValueError("fr_poly_eval_many_dev: a group names a point set that is not given")
    out = bytearray(32 * g * count)
    sel = (ctypes.c_uint32 * g)(*[it[4] for it in groups])
    pts = _fr_rows("fr_poly_eval_many_dev: point_sets", point_sets, len(point_sets), count)
    check(_lib.lib().zkp_fr_poly_eval_many_dev(g, _u64s([it[0].handle for it in groups]), _u64s([it[1] for it in groups]),
                                               _u64s([it[2] for it in groups]), _u64s([it[3] for it in groups]), sel, count,
                                               len(point_sets), buf(pts), buf(out)))
    vals = fr_vec_from_bytes(bytes(out))
    return [vals[i * count:(i + 1) * count] for i in range(g)]


def lincomb_many_dev(dst, dst_off, dst_stride, n, count, sources, coeffs):
    """dst_j[i] = sum_k coeffs[j][k] * src_k,j[i] (+ coeffs[j][K] at i = 0), i < n; sources = [(handle, offset, stride,
    length)] with stride 0 for a vector shared by every proof; coeffs: count rows of K + 1 scalars."""
    K = len(sources)
    flat = _fr_rows("lincomb_many_dev: coeffs", coeffs, count, K + 1)
    check(_lib.lib().zkp_fr_lincomb_many_dev(dst.handle, dst_off, dst_stride, n, count, K, _u64s([s[0].handle for s in sources]),
                                             _u64s([s[1] for s in sources]), _u64s([s[2] for s in sources]),
                                             _u64s([s[3] for s in sources]), buf(flat) if count else None))


def div_linear_many_dev(src, src_off, src_stride, length, zetas, dst, dst_off, dst_stride):
    """div_linear_dev for len(zetas) polynomials of `length` coefficients at src_off + j * src_stride."""
    zs = fr_vec_bytes([int(z) % R_MOD for z in zetas])
    check(_lib.lib().zkp_fr_div_linear_many_dev(src.handle, src_off, src_stride, length, len(zetas),
                                                buf(zs) if zetas else None, dst.handle, dst_off, dst_stride))


def plonk_pi_scatter_many_dev(pub, off, stride, ell, n, count, dst, dst_off=0):
    """count blocks of n values at dst_off: proof j's ell public inputs (pub[off + j * stride ..]) at rows i < ell,
    zeros elsewhere.  pub may be None when ell = 0."""
    check(_lib.lib().zkp_plonk_pi_scatter_many_dev(pub.handle if pub is not None else 0, off, stride, ell, n, count,
                                                   dst.handle, dst_off))


def plonk_coset_inputs_pi_many_dev(wires, z, pi, pi_off, n, count, log_N, out):
    """plonk_coset_inputs_many_dev plus a fifth group: count blocks of n PI coefficients at pi_off."""
    check(_lib.lib().zkp_plonk_coset_inputs_pi_many_dev(wires.handle, z.handle, pi.handle, pi_off, n, count, log_N,
                                                        out.handle))


def plonk_quotient_pi_many_dev(evals, circuit8, n, ext, x, l1f, zh8, betas, gammas, alphas, t_out):
    """plonk_quotient_many_dev on 5 groups of blocks: a_*, b_*, c_*, z_*, PI_* (PI_j added to q_c)."""
    count = len(betas)
    if len(circuit8) != 8:
        raise ValueError("plonk_quotient_pi_many_dev: 8 circuit coset evaluations, got %d" % len(circuit8))
    ch = _fr_rows("plonk_quotient_pi_many_dev: betas, gammas, alphas", [betas, gammas, alphas], 3, count)
    check(_lib.lib().zkp_plonk_quotient_pi_many_dev(evals.handle, _u64s([h.handle for h in circuit8]), n, ext, count,
                                                    x.handle, l1f.handle, zh8.handle, buf(ch[:32 * count]),
                                                    buf(ch[32 * count:64 * count]), buf(ch[64 * count:]), t_out.handle))


def plonk_pi_eval_many_dev(pub, off, stride, ell, n, omega, zetas):
    """[PI_j(zeta_j) for j < len(zetas)]: PI_j = sum_{i < ell} x_j,i L_i over the n-th roots of unity of omega, proof j's
    inputs at pub[off + j * stride ..].  pub may be None when ell = 0."""
    count = len(zetas)
    out = bytearray(32 * max(count, 1))
    zs = fr_vec_bytes([int(z) % R_MOD for z in zetas])
    check(_lib.lib().zkp_plonk_pi_eval_many_dev(pub.handle if pub is not None else 0, off, stride, ell, n, count,
                                                buf(fe_bytes(omega)), buf(zs) if count else None, buf(out)))
    return fr_vec_from_bytes(bytes(out), count)


# ------------------------------------------------------------------ QAP over {1..k} at scale (SURVEY 8 f2)
def sparse_load(row_ptr, col_idx, values, rows, cols):
    """CSR matrix with Fr values -> device handle.  row_ptr: rows+1 offsets, col_idx: column of each
    entry (sequences or numpy uint32 arrays), values: ints (or already 32 B/entry canonical bytes)."""
    import numpy as np
    rp = np.ascontiguousarray(row_ptr, dtype=np.uint32)
    ci = np.ascontiguousarray(col_idx, dtype=np.uint32)
    if len(rp) != rows + 1:
        raise ValueError("sparse_load: row_ptr needs rows + 1 entries")
    nnz = len(ci)
    vb = values if isinstance(values, (bytes, bytearray)) else fr_vec_bytes(values)
    if len(vb) != 32 * nnz:
        raise ValueError("sparse_load: one value per column index")
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_sparse_load(rp.ctypes.data, ci.ctypes.data if nnz else None, buf(vb) if nnz else None,
                                     rows, cols, nnz, ctypes.byref(h)))
    out = DeviceHandle(h.value, rows, "sparse")
    out.cols, out.nnz = cols, nnz
    return out


def sparse_matvec_dev(matrix, vec, out, vec_off=0, out_off=0):
    """out[row] = sum_e value[e] * vec[col[e]] on device scalar handles (canonical)."""
    check(_lib.lib().zkp_sparse_matvec_dev(matrix.handle, vec.handle, vec_off, out.handle, out_off))


def fr_ap_interpolate_dev(values, k, out, scale=None, off=0, out_off=0):
    """out[0..k) = coefficients of the polynomial p of degree < k with p(j + 1) = values[j], times scale."""
    sc = fe_bytes(scale) if scale is not None else None
    check(_lib.lib().zkp_fr_ap_interpolate_dev(values.handle, off, k, buf(sc), out.handle, out_off))


def sparse_matvec_many_dev(matrix, vec, out, count, vec_off=0, out_off=0):
    """sparse_matvec_dev over count vectors: witness j at vec_off + j * cols, result j at out_off + j * rows."""
    check(_lib.lib().zkp_sparse_matvec_many_dev(matrix.handle, vec.handle, vec_off, out.handle, out_off, count))


def fr_ap_interpolate_many_dev(values, k, count, out, scale=None, off=0, out_off=0):
    """fr_ap_interpolate_dev over count value vectors of k entries each, back to back."""
    sc = fe_bytes(scale) if scale is not None else None
    check(_lib.lib().zkp_fr_ap_interpolate_many_dev(values.handle, off, k, count, buf(sc), out.handle, out_off))


def fr_ap_vanishing_dev(k):
    """Handle with the k + 1 coefficients of Z(x) = (x - 1)(x - 2)...(x - k)."""
    out = scalars_alloc(k + 1)
    check(_lib.lib().zkp_fr_ap_vanishing_dev(k, out.handle, 0))
    return out


def fr_ap_lagrange_dev(k, x):
    """Handle with l_1(x) .. l_k(x), the Lagrange basis of the points {1..k} at x."""
    out = scalars_alloc(k)
    check(_lib.lib().zkp_fr_ap_lagrange_dev(k, buf(fe_bytes(x)), out.handle, 0))
    return out


# ------------------------------------------------------------------ witness solving (zkp/witness.py)
def witness_program_load(row_ptr, col_idx, values, out_var, level_ptr, in_var, nvars):
    """Step program (include/zkp_b200.h zkp_witness_program_load) -> device handle.  row_ptr: 4 * steps + 1 offsets;
    col_idx / values: the entries of the four forms of every step; out_var: steps entries (0xFFFFFFFF = check)."""
    import numpy as np
    arr = lambda a: np.ascontiguousarray(a, dtype=np.uint32)
    rp, ci, ov, lp, iv = arr(row_ptr), arr(col_idx), arr(out_var), arr(level_ptr), arr(in_var)
    steps, nnz = len(ov), len(ci)
    if len(rp) != 4 * steps + 1 or len(lp) < 1:
        raise ValueError("witness_program_load: row_ptr needs 4 * steps + 1 entries and level_ptr at least one")
    vb = values if isinstance(values, (bytes, bytearray)) else fr_vec_bytes(values)
    if len(vb) != 32 * nnz:
        raise ValueError("witness_program_load: one value per column index")
    ptr = lambda a: a.ctypes.data if len(a) else None
    h = ctypes.c_uint64()
    check(_lib.lib().zkp_witness_program_load(rp.ctypes.data, ptr(ci), buf(vb) if nnz else None, nnz, ptr(ov), steps,
                                              lp.ctypes.data, len(lp) - 1, ptr(iv), len(iv), nvars, ctypes.byref(h)))
    out = DeviceHandle(h.value, nvars, "witness_program")
    out.steps, out.inputs = steps, len(iv)
    return out


def witness_solve_many_dev(program, inputs, count, out, in_off=0, out_off=0):
    """Solve count witnesses: inputs j at in_off + j * n_in, values j at out_off + j * nvars.  Returns the lowest
    j * steps + s whose step failed, or None."""
    bad = ctypes.c_uint64()
    check(_lib.lib().zkp_witness_solve_many_dev(program.handle, inputs.handle, in_off, count, out.handle, out_off,
                                                ctypes.byref(bad)))
    return _first_bad(bad.value)
