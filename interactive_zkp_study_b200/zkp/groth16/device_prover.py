"""Groth16 proving at scale: coefficient-vector entry points over device-resident keys.

The reference's `proof_a/b/c(sigma..., Ax, Rx, ...)` signatures take the dense numWires x numGates QAP
matrices, which cannot exist at 2^20 constraints (2^40 entries; SURVEY.md F12).  What the prover needs
from them is only the three coefficient vectors uA = R.Ax, uB = R.Bx, uC = R.Cx (numGates entries
each) -- this module is the same algebra as zkp/groth16/proving.py + poly_utils.hxr
(/root/reference/zkp/groth16/proving.py:23-75, poly_utils.py:116-125) on those vectors, with the CRS
resident on the GPU in three concatenated, window-precomputed tables so that each proof element is
ONE multi-scalar multiplication:

    TA  (G1) = [x^j]_1 (j < k) | alpha_1 | delta_1                  scalars  uA | 1 | r            -> A
    TB2 (G2) = [x^j]_2 (j < k) | beta_2  | delta_2                  scalars  uB | 1 | s            -> B
    TC  (G1) = [x^j]_1 (j < k) | beta_1 | sigma1_4[private] | sigma1_5 (k-1) | alpha_1 | delta_1
                                                       scalars  r*uB + s*uA | r | Rx_priv | H | s | s*r -> C

C = s*A + r*B1 - s*r*delta_1 + (wires) + (H) of proving.py:64-73 with A and B1 expanded over the SAME points [x^j]_1:
the s*A term becomes s*uA on the first k rows plus s*alpha_1 + s*r*delta_1, the -s*r*delta_1 cancels against
r*B1's s*r*delta_1, so C needs neither A's value nor a scalar multiplication -- the three elements are three
independent multi-scalar multiplications, and B (G2, the longest) starts before the quotient it does not need.
"""
from ... import native
from ...compat import G1, G2, curve_order, g1_from_ints, g2_from_ints

R = curve_order


class DeviceKey:
    def __init__(self, k, m_priv, TA, TB2, TC):
        self.k, self.m_priv, self.TA, self.TB2, self.TC = k, m_priv, TA, TB2, TC


def tc_rows(k, m_priv):
    """Rows of the C table: [x^j]_1 (k) | beta_1 | sigma1_4[private] (m_priv) | sigma1_5 (k-1) | alpha_1 | delta_1."""
    return k + 1 + m_priv + (k - 1) + 2


def _powers(x, count):
    return native.fr_prefix_product(native.fr_vec_bytes([x % R] * count), count)


def setup_from_toxic(k, alpha, beta, delta, x_val, zx_val, priv_vals, precompute=True):
    """CRS generation on the device (batched fixed-base multiplications; reference setup.py:15-69).
    priv_vals[i] = (beta*A_i(x) + alpha*B_i(x) + C_i(x)) / delta for the private wires, in order."""
    m_priv = len(priv_vals)
    pw = _powers(x_val, k)
    inv_delta = pow(delta % R, -1, R)
    s15 = native.fr_vec_op(3, pw[:32 * (k - 1)], native.fe_bytes(zx_val % R * inv_delta % R), k - 1) if k > 1 else b""
    enc = native.fr_vec_bytes
    scA = pw + enc([alpha % R, delta % R])
    scC = pw + enc([beta % R]) + enc([v % R for v in priv_vals]) + s15 + enc([alpha % R, delta % R])
    TA = native.g1_fixed_base_mul(native.g1_bytes(G1), scA, k + 2)
    TB2 = native.g2_fixed_base_mul(native.g2_bytes(G2), pw + enc([beta % R, delta % R]), k + 2)
    TC = native.g1_fixed_base_mul(native.g1_bytes(G1), scC, tc_rows(k, m_priv))
    if precompute:
        for t in (TA, TB2, TC):
            if t.n >= 2:
                native.table_precompute(t)
    return DeviceKey(k, m_priv, TA, TB2, TC)


def _scalars_ab(key, uA, uB, r, s):
    """Scalar vectors of the A and B elements (they need only uA, uB): uA | 1 | r and uB | 1 | s."""
    k = key.k
    one = native.fr_vec_bytes([1])
    scA = native.scalars_alloc(k + 2)
    native.scalars_copy(scA, 0, uA, 0, k)
    native.scalars_upload(scA, k, one + native.fe_bytes(r), 2)
    scB = native.scalars_alloc(k + 2)
    native.scalars_copy(scB, 0, uB, 0, k)
    native.scalars_upload(scB, k, one + native.fe_bytes(s), 2)
    return scA, scB


def _scalars_c(key, uA, uB, hq, rx_priv, r, s):
    """Scalar vector of C: r*uB + s*uA | r | Rx_priv | H | s | s*r  (see the table layout above)."""
    k, mp = key.k, key.m_priv
    nC = tc_rows(k, mp)
    scC = native.scalars_alloc(nC)
    native.scalars_copy(scC, 0, uB, 0, k)
    native.scalars_scale(scC, 0, k, r)
    native.axpy_dev(scC, 0, s, uA, 0, k)
    native.scalars_upload(scC, k, native.fe_bytes(r), 1)
    if mp:
        native.scalars_copy(scC, k + 1, rx_priv, 0, mp)
    if k > 1:
        native.scalars_copy(scC, k + 1 + mp, hq, 0, k - 1)
    native.scalars_upload(scC, nC - 2, native.fe_bytes(s) + native.fe_bytes(s * r % R), 2)
    return scC, nC


def prove(key, uA, uB, uC, Z, rx_priv, r, s, keep_quotient=False):
    """uA, uB, uC: device scalar handles with k coefficients; Z: handle with k+1 coefficients (monic
    divisor); rx_priv: handle with the private wires' witness values.  Returns (A, B, C) as the
    reference's point types (and the quotient / remainder handles when keep_quotient)."""
    k = key.k
    r, s = int(r) % R, int(s) % R
    # H: k-1 coefficients; the remainder (k coefficients, zero for a satisfied instance) only on request
    # B (G2, the longest of the three) needs only uB: it starts on the library's second stream and runs beside the
    # quotient; A and C follow on the first stream
    scA, scB = _scalars_ab(key, uA, uB, r, s)
    native.msm_dev_begin(key.TB2, 0, scB, 0, k + 2)
    hq, hr = native.groth16_quotient_dev(uA, uB, uC, k, Z, k + 1, want_remainder=keep_quotient)
    scC, nC = _scalars_c(key, uA, uB, hq, rx_priv, r, s)
    A = native.g1_msm_dev(key.TA, 0, scA, 0, k + 2)
    C = native.g1_msm_dev(key.TC, 0, scC, 0, nC)
    B = native.msm_dev_end("g2")
    for h in (scA, scB, scC):
        h.free()
    out = (g1_from_ints(A), g2_from_ints(B), g1_from_ints(C))
    if keep_quotient:
        return out + (hq, hr)
    hq.free()
    return out


# ------------------------------------------------------------------ many proofs of one circuit per pass
def _many_msm_shape(table, n):
    """(windows W, buckets per MSM) of a many-MSM pass over n rows of `table`: the table's own width when it is
    window-precomputed (all windows share one bucket set), else the automatic width of csrc/msm.cuh msm_plan."""
    c = getattr(table, "pre_c", 0)
    if not c:
        c = min(max(max(n, 1).bit_length() - 1 - 4, 4), 16)
    W = -(-255 // c)
    B = 1 << (c - 1)
    return W, (B if getattr(table, "pre_c", 0) else W * B)


def plan_chunk(key, count, free_bytes):
    """Largest number of proofs per pass of prove_batch: within the 32-bit entry and 31-bit bucket numbering of the
    many-MSM (count * W * n < 2^32, count * buckets < 2^31), the 32-bit batched transforms of the quotient, and half
    of `free_bytes` of device memory at the working set estimated below.  At least 1, at most count."""
    k, mp = key.k, key.m_priv
    nC = tc_rows(k, mp)
    lg1 = (2 * k - 2).bit_length()                     # transforms of 2^lg1 >= 2k - 1 points
    limit = ((1 << 32) - 1) >> lg1
    g1_ws = g2_ws = 0
    for table, n, xyzz in ((key.TA, k + 2, 128), (key.TB2, k + 2, 256), (key.TC, nC, 128)):
        W, per = _many_msm_shape(table, n)
        limit = min(limit, ((1 << 32) - 1) // (W * n), ((1 << 31) - 1) // per)
        ws = 8 * W * n + per * (3 * xyzz + 12)          # codes + sorted entries; buckets, partials, levels, counts
        if xyzz == 256:
            g2_ws = max(g2_ws, ws)
        else:
            g1_ws = max(g1_ws, ws)
    per_proof = (g1_ws + g2_ws                            # the G1 and the G2 engine keep their own workspace
                 + 32 * (2 * (k + 2) + nC)                # scalar vectors
                 + 32 * (5 << lg1)                        # quotient transforms
                 + 32 * (4 * k + mp))                     # chunk copies of uA, uB, uC, rx_priv and H
    limit = min(limit, (free_bytes // 2) // per_proof)
    return int(max(1, min(limit, count)))


def _slice(h, off, n):
    out = native.scalars_alloc(n)
    if n:
        native.scalars_copy(out, 0, h, off, n)
    return out


def prove_batch(key, uA, uB, uC, Z, rx_priv, rs, ss, keep_quotient=False, chunk=None):
    """count = len(rs) proofs of the circuit of `key`, bit-identical to count calls of prove: proof j from uA, uB, uC
    at offset j * k, rx_priv at offset j * m_priv, and (rs[j], ss[j]).  Per chunk of proofs: one batched quotient,
    one scalar assembly and three many-MSMs (TA, TB2, TC), so the launch count does not grow with count.
    chunk=None picks the largest chunk the 32-bit limits and the free device memory allow (plan_chunk); the
    result does not depend on it.  Returns the list of (A, B, C), and with keep_quotient also the handle of the
    count quotients (k - 1 coefficients each, back to back)."""
    k, mp = key.k, key.m_priv
    count = len(rs)
    if len(ss) != count:
        raise ValueError("prove_batch: rs and ss differ in length (%d, %d)" % (count, len(ss)))
    if chunk is not None and int(chunk) <= 0:
        raise ValueError("prove_batch: chunk must be positive")
    for name, h, need in (("uA", uA, count * k), ("uB", uB, count * k), ("uC", uC, count * k),
                          ("rx_priv", rx_priv, count * mp), ("Z", Z, k + 1)):
        if h is None or h.n < need:
            raise ValueError("prove_batch: %s holds %s values, needs %d" % (name, None if h is None else h.n, need))
    if count == 0:
        return []
    rs = [int(r) % R for r in rs]
    ss = [int(s) % R for s in ss]
    step = min(int(chunk), count) if chunk is not None else plan_chunk(key, count, native.device_mem_info()[0])
    nC = tc_rows(k, mp)
    H = native.scalars_alloc(count * (k - 1)) if keep_quotient else None
    proofs = []
    for j0 in range(0, count, step):
        cnt = min(step, count - j0)
        whole = cnt == count
        a, b, c = (h if whole else _slice(h, j0 * k, cnt * k) for h in (uA, uB, uC))
        x = rx_priv if whole or not mp else _slice(rx_priv, j0 * mp, cnt * mp)
        hq = native.groth16_quotient_batch_dev(a, b, c, k, cnt, Z, k + 1)
        scA, scB, scC = native.groth16_batch_scalars_dev(a, b, hq, x, k, mp, rs[j0:j0 + cnt], ss[j0:j0 + cnt])
        As = native.msm_dev_many(key.TA, 0, k + 2, cnt, scA)
        Bs = native.msm_dev_many(key.TB2, 0, k + 2, cnt, scB)
        Cs = native.msm_dev_many(key.TC, 0, nC, cnt, scC)
        if H is not None and k > 1:
            native.scalars_copy(H, j0 * (k - 1), hq, 0, cnt * (k - 1))
        for h in (scA, scB, scC, hq):
            h.free()
        if not whole:
            for h in (a, b, c) + ((x,) if mp else ()):
                h.free()
        proofs.extend((g1_from_ints(A), g2_from_ints(B), g1_from_ints(C)) for A, B, C in zip(As, Bs, Cs))
    return (proofs, H) if keep_quotient else proofs


# ------------------------------------------------------------------ the same proof over the GPUs of one box
class ShardedDeviceKey:
    """This rank's contiguous row range of each of the three CRS tables (sharded.shard_range of the
    concatenated table), resident and window-precomputed on this rank's GPU."""

    def __init__(self, k, m_priv, TA, TB2, TC, rA, rB, rC):
        self.k, self.m_priv, self.TA, self.TB2, self.TC = k, m_priv, TA, TB2, TC
        self.rA, self.rB, self.rC = rA, rB, rC        # (start, count) of this rank in each table


def setup_from_toxic_sharded(comm, k, alpha, beta, delta, x_val, zx_val, priv_vals, precompute=True):
    """setup_from_toxic with every table cut by point range over the ranks of `comm` (SURVEY 8e): a rank
    generates and keeps only its rows.  Same arguments on every rank."""
    from ... import sharded
    m_priv = len(priv_vals)
    pw = _powers(x_val, k)
    inv_delta = pow(delta % R, -1, R)
    s15 = native.fr_vec_op(3, pw[:32 * (k - 1)], native.fe_bytes(zx_val % R * inv_delta % R), k - 1) if k > 1 else b""
    enc = native.fr_vec_bytes
    scA = pw + enc([alpha % R, delta % R])
    scB = pw + enc([beta % R, delta % R])
    scC = pw + enc([beta % R]) + enc([v % R for v in priv_vals]) + s15 + enc([alpha % R, delta % R])
    out = []
    for sc, g2 in ((scA, False), (scB, True), (scC, False)):
        start, count = sharded.shard_range(len(sc) // 32, comm.rank, comm.world)
        part = sc[32 * start:32 * (start + count)]
        t = (native.g2_fixed_base_mul(native.g2_bytes(G2), part, count) if g2
             else native.g1_fixed_base_mul(native.g1_bytes(G1), part, count))
        if precompute and count >= 2:
            native.table_precompute(t)
        out.append((t, (start, count)))
    (TA, rA), (TB2, rB), (TC, rC) = out
    return ShardedDeviceKey(k, m_priv, TA, TB2, TC, rA, rB, rC)


def prove_sharded(comm, key, uA, uB, uC, Z, rx_priv, r, s):
    """prove() with each of the three multi-scalar multiplications sharded by point range over the ranks
    (zkp_g1_msm_multi / zkp_g2_msm_multi: local Pippenger -> one all-gather of the partial sums -> fold, inside
    the library).  Collective: every rank passes the same coefficient vectors and gets the same proof.  The
    quotient -- NTT work, which stays on one GPU (SURVEY 8e) -- is computed by every rank for itself: that
    costs no wall time and needs no 32 MiB broadcast of H; the A and B collectives run beside it on the second
    stream (zkp_g1/g2_msm_multi_begin / _end)."""
    k = key.k
    r, s = int(r) % R, int(s) % R
    # A and B need only uA, uB: their collectives start on the library's second stream and run beside the quotient
    scA, scB = _scalars_ab(key, uA, uB, r, s)
    native.msm_multi_begin(key.TA, 0, scA, key.rA[0], key.rA[1])
    native.msm_multi_begin(key.TB2, 0, scB, key.rB[0], key.rB[1])
    hq, _ = native.groth16_quotient_dev(uA, uB, uC, k, Z, k + 1, want_remainder=False)
    scC, _ = _scalars_c(key, uA, uB, hq, rx_priv, r, s)
    C = native.g1_msm_multi(key.TC, 0, scC, key.rC[0], key.rC[1])
    A = native.msm_multi_end("g1")
    B = native.msm_multi_end("g2")
    for h in (scA, scB, scC, hq):
        h.free()
    return (g1_from_ints(A), g2_from_ints(B), g1_from_ints(C))
