"""QAP construction and Groth16 setup / prove from a SPARSE R1CS at scale (SURVEY.md 8 f2).

The reference turns the R1CS into a QAP by Lagrange-interpolating every wire's column through the
points x = 1..numGates in floating point, scaled by the determinant of the Vandermonde matrix so the
coefficients come out integral (/root/reference/zkp/groth16/qap_creator_lcm.py:50-78,114-135), and
carries the dense numWires x numGates matrices Ax, Bx, Cx through setup (`ax_val`, poly_utils.py:86-106)
and proving (`R . Ax`, poly_utils.py:52-59, proving.py:27-31).  2^20 constraints would need 2^40 matrix
entries and exact arithmetic the floats cannot give.  Interpolation is linear, so

    R . Ax   = d * interp_{1..k}(A . w)              (one sparse mat-vec + one interpolation)
    Ax_i(x)  = d * sum_j A[j][i] * l_j(x) = d * (A^T . l(x))_i      (one transposed sparse mat-vec)

with d = det Vandermonde(1..k) = prod_{n<k} n! (d^2 for C, as in r1cs_to_qap_times_lcm) -- the same Fr
values the reference's pipeline produces at toy size (tests/golden/groth16_qap.json), exact at any size.
The proof elements then come from device_prover.prove (one MSM per element).
"""
import functools

import numpy as np

from ... import native
from ...compat import G1, G2, curve_order, g1_from_ints, g2_from_ints
from . import device_prover

R = curve_order


@functools.lru_cache(maxsize=16)
def vandermonde_det(k):
    """det of k_matrix(k) (qap_creator_lcm.py:97-108): prod_{1<=i<j<=k} (j - i) = prod_{n=1}^{k-1} n!  (mod r)."""
    d, f = 1, 1
    for n in range(1, k):
        f = f * n % R
        d = d * f % R
    return d


class SparseR1CS:
    """k constraints over m wires: (A.w) o (B.w) = C.w, each matrix as CSR (row_ptr, col_idx, values)."""

    def __init__(self, k, m, A, B, C):
        self.k, self.m = k, m
        self.mats = tuple((np.asarray(rp, dtype=np.uint32), np.asarray(ci, dtype=np.uint32), [int(v) % R for v in vals])
                          for rp, ci, vals in (A, B, C))

    @classmethod
    def from_dense(cls, A, B, C):
        """From the reference's R1CS (lists of rows, one row of numWires entries per gate:
        code_to_r1cs.py `code_to_r1cs_with_inputs` output)."""
        k, m = len(A), len(A[0])

        def csr(M):
            rp, ci, vals = [0], [], []
            for row in M:
                for j, v in enumerate(row):
                    if int(v) % R:
                        ci.append(j)
                        vals.append(int(v))
                rp.append(len(ci))
            return rp, ci, vals
        return cls(k, m, csr(A), csr(B), csr(C))

    @classmethod
    def from_rows(cls, k, m, rows_a, rows_b, rows_c):
        """rows_x[g] = {wire: coefficient} for gate g."""
        def csr(rows):
            rp, ci, vals = [0], [], []
            for row in rows:
                for j in sorted(row):
                    ci.append(j)
                    vals.append(row[j])
                rp.append(len(ci))
            return rp, ci, vals
        return cls(k, m, csr(rows_a), csr(rows_b), csr(rows_c))

    def transposed(self, which):
        """CSR of the transpose (m x k) of matrix `which` -- for the CRS terms A_i(x) = (A^T l(x))_i."""
        rp, ci, vals = self.mats[which]
        rows = np.repeat(np.arange(self.k, dtype=np.uint32), np.diff(rp).astype(np.int64))
        order = np.argsort(ci, kind="stable")
        t_rp = np.zeros(self.m + 1, dtype=np.uint32)
        t_rp[1:] = np.cumsum(np.bincount(ci.astype(np.int64), minlength=self.m))
        return t_rp, rows[order], [vals[i] for i in order]


class DeviceR1CS:
    """The three matrices (and, on demand, their transposes) resident on the GPU."""

    def __init__(self, r1cs):
        self.k, self.m, self.host = r1cs.k, r1cs.m, r1cs
        self.mats = [native.sparse_load(rp, ci, vals, r1cs.k, r1cs.m) for rp, ci, vals in r1cs.mats]
        self._t = None

    def transposes(self):
        if self._t is None:
            self._t = [native.sparse_load(*self.host.transposed(i), self.m, self.k) for i in range(3)]
        return self._t


def _scales(k, lcm):
    d = vandermonde_det(k) if lcm else 1
    return d, d, d * d % R


def witness_polys(dev, w, lcm=True):
    """uA = R.Ax, uB = R.Bx, uC = R.Cx as device coefficient vectors (k each) for the witness handle w
    (m canonical values, wire 0 = 1).  `lcm`: the reference's determinant scaling (d, d, d^2)."""
    out = []
    ev = native.scalars_alloc(dev.k)
    for mat, sc in zip(dev.mats, _scales(dev.k, lcm)):
        native.sparse_matvec_dev(mat, w, ev)
        u = native.scalars_alloc(dev.k)
        native.fr_ap_interpolate_dev(ev, dev.k, u, scale=sc if lcm else None)
        out.append(u)
    ev.free()
    return tuple(out)


def witness_polys_batch(dev, W, count, lcm=True, off=0):
    """witness_polys for count witnesses at once: witness j at W[off + j * m]; returns uA, uB, uC handles of
    count * k coefficients, proof j's at j * k.  Two launches of sparse products and two batched interpolations
    per matrix, whatever count is."""
    k = dev.k
    out = []
    ev = native.scalars_alloc(count * k)
    for mat, sc in zip(dev.mats, _scales(k, lcm)):
        native.sparse_matvec_many_dev(mat, W, ev, count, vec_off=off)
        u = native.scalars_alloc(count * k)
        native.fr_ap_interpolate_many_dev(ev, k, count, u, scale=sc if lcm else None)
        out.append(u)
    ev.free()
    return tuple(out)


class Keys:
    """Proving key (device tables of device_prover.DeviceKey) + the verifier's small CRS part."""

    def __init__(self, device_key, Z, pub_idx, priv_sel, sigma1_1, sigma1_3, sigma2_1, lcm):
        self.device_key, self.Z, self.pub_idx, self.priv_sel = device_key, Z, pub_idx, priv_sel
        self.priv_idx = priv_sel.idx
        self.sigma1_1, self.sigma1_3, self.sigma2_1, self.lcm = sigma1_1, sigma1_3, sigma2_1, lcm


class _Selection:
    """An index subset of a device vector; a contiguous run (the usual case: the public wires come first)
    is recognised once, at setup, and then gathered by a device copy."""

    def __init__(self, idx):
        self.idx = list(idx)
        n = len(self.idx)
        self.run = (self.idx[0], n) if n and self.idx[-1] - self.idx[0] == n - 1 and self.idx == list(range(self.idx[0], self.idx[0] + n)) else None

    def __len__(self):
        return len(self.idx)

    def gather(self, handle):
        n = len(self.idx)
        out = native.scalars_alloc(n)
        if self.run:
            native.scalars_copy(out, 0, handle, self.run[0], n)
        elif n:
            raw = native.scalars_download(handle, 0, handle.n)
            native.scalars_upload(out, 0, b"".join(raw[32 * i:32 * i + 32] for i in self.idx), n)
        return out


def setup(dev, alpha, beta, gamma, delta, x_val, pub_r_indexs=None, lcm=True, precompute=True):
    """CRS for a sparse R1CS from the toxic values (reference setup.py:15-69 with ax_val/bx_val/cx_val/zx_val
    of poly_utils.py:86-113), all vector work on the device."""
    k, m = dev.k, dev.m
    pub = [0, 1] if pub_r_indexs is None else list(pub_r_indexs)      # the reference's default (setup.py:26-27)
    pub_set = set(pub)
    priv = _Selection(i for i in range(m) if i not in pub_set)
    alpha, beta, gamma, delta, x_val = (int(v) % R for v in (alpha, beta, gamma, delta, x_val))
    sA, sB, sC = _scales(k, lcm)
    # val_i = beta*A_i(x) + alpha*B_i(x) + C_i(x) for every wire: three transposed sparse products of l(x)
    lag = native.fr_ap_lagrange_dev(k, x_val)
    val = native.scalars_alloc(m)
    tmp = native.scalars_alloc(m)
    for mat, coeff in zip(dev.transposes(), (beta * sA % R, alpha * sB % R, sC)):
        native.sparse_matvec_dev(mat, lag, tmp)
        native.axpy_dev(val, 0, coeff, tmp, 0, m)
    tmp.free()
    lag.free()
    Z = native.fr_ap_vanishing_dev(k)
    zx = native.fr_poly_eval_dev(Z, 0, k + 1, x_val)
    inv_delta, inv_gamma = pow(delta, -1, R), pow(gamma, -1, R)
    enc = native.fr_vec_bytes
    g1b, g2b = native.g1_bytes(G1), native.g2_bytes(G2)
    # TA = [x^j]_1 | alpha | delta ;  TB2 = [x^j]_2 | beta | delta ;
    # TC = [x^j]_1 | beta | sigma1_4[priv] | sigma1_5 | alpha | delta   (device_prover.tc_rows)
    mp = len(priv)
    scA = native.scalars_alloc(k + 2)
    native.scalars_fill_powers(scA, 0, k, 1, x_val)
    native.scalars_upload(scA, k, enc([alpha, delta]), 2)
    scB = native.scalars_alloc(k + 2)
    native.scalars_copy(scB, 0, scA, 0, k)
    native.scalars_upload(scB, k, enc([beta, delta]), 2)
    nC = device_prover.tc_rows(k, mp)
    scC = native.scalars_alloc(nC)
    native.scalars_copy(scC, 0, scA, 0, k)
    native.scalars_upload(scC, k, enc([beta]), 1)
    if mp:
        pv = priv.gather(val)
        native.scalars_scale(pv, 0, mp, inv_delta)
        native.scalars_copy(scC, k + 1, pv, 0, mp)
        pv.free()
    if k > 1:
        native.scalars_fill_powers(scC, k + 1 + mp, k - 1, zx * inv_delta % R, x_val)
    native.scalars_upload(scC, nC - 2, enc([alpha, delta]), 2)
    TA = native.g1_fixed_base_mul_dev(g1b, scA, k + 2)
    TB2 = native.g2_fixed_base_mul_dev(g2b, scB, k + 2)
    TC = native.g1_fixed_base_mul_dev(g1b, scC, nC)
    for h in (scA, scB, scC):
        h.free()
    if precompute:
        for t in (TA, TB2, TC):
            if t.n >= 2:
                native.table_precompute(t)
    # the verifier's part: sigma1_1, sigma2_1 and sigma1_3 on the public wires (placeholders elsewhere, setup.py:37)
    pub_vals = native.fr_vec_from_bytes(native.scalars_download(_Selection(pub).gather(val), 0, len(pub))) if pub else []
    val.free()
    s13_tab = native.g1_fixed_base_mul(g1b, enc([v * inv_gamma % R for v in pub_vals]), len(pub)) if pub else None
    s13_pts = [native.g1_from_bytes(native.table_download(s13_tab, i, 1)) for i in range(len(pub))]
    from ...compat import FQ
    sigma1_3 = [(FQ(0), FQ(0))] * m
    for i, p in zip(pub, s13_pts):
        sigma1_3[i] = g1_from_ints(p)
    t11 = native.g1_fixed_base_mul(g1b, enc([alpha, beta, delta]), 3)
    sigma1_1 = [g1_from_ints(native.g1_from_bytes(native.table_download(t11, i, 1))) for i in range(3)]
    t21 = native.g2_fixed_base_mul(g2b, enc([beta, gamma, delta]), 3)
    sigma2_1 = [g2_from_ints(native.g2_from_bytes(native.table_download(t21, i, 1))) for i in range(3)]
    key = device_prover.DeviceKey(k, mp, TA, TB2, TC)
    return Keys(key, Z, pub, priv, sigma1_1, sigma1_3, sigma2_1, lcm)


def prove(keys, dev, w, r, s, keep=False):
    """(A, B, C) for the witness handle w (m values).  The algebra of proving.py:23-75 + poly_utils.hxr."""
    uA, uB, uC = witness_polys(dev, w, keys.lcm)
    rx_priv = keys.priv_sel.gather(w)
    out = device_prover.prove(keys.device_key, uA, uB, uC, keys.Z, rx_priv, r, s, keep_quotient=keep)
    rx_priv.free()
    if keep:
        return out + (uA, uB, uC)
    for h in (uA, uB, uC):
        h.free()
    return out


def _selection_matrix(keys, m):
    """The private-wire selection as an m_priv x m 0/1 sparse matrix (cached on keys): one sparse product gathers the
    private wires of every witness of a batch."""
    if getattr(keys, "_sel_mat", None) is None:
        idx = keys.priv_idx
        keys._sel_mat = native.sparse_load(list(range(len(idx) + 1)), idx, [1] * len(idx), len(idx), m)
    return keys._sel_mat


def prove_batch(keys, dev, W, rs, ss, chunk=None):
    """[prove(keys, dev, w_j, rs[j], ss[j]) for each witness w_j = W[j * m : (j + 1) * m]] in batched passes:
    witness polynomials, private-wire gathers, quotients and the three MSMs of a chunk of proofs each run in a
    fixed number of launches (device_prover.prove_batch).  chunk=None: device_prover.plan_chunk."""
    count = len(rs)
    if len(ss) != count:
        raise ValueError("prove_batch: rs and ss differ in length (%d, %d)" % (count, len(ss)))
    if chunk is not None and int(chunk) <= 0:
        raise ValueError("prove_batch: chunk must be positive")
    if W is None or W.n < count * dev.m:
        raise ValueError("prove_batch: W holds %s values, needs %d" % (None if W is None else W.n, count * dev.m))
    if count == 0:
        return []
    key = keys.device_key
    mp = len(keys.priv_idx)
    step = min(int(chunk), count) if chunk is not None else device_prover.plan_chunk(key, count, native.device_mem_info()[0])
    sel = _selection_matrix(keys, dev.m) if mp else None
    proofs = []
    for j0 in range(0, count, step):
        cnt = min(step, count - j0)
        uA, uB, uC = witness_polys_batch(dev, W, cnt, keys.lcm, off=j0 * dev.m)
        rx = native.scalars_alloc(cnt * mp)
        if mp:
            native.sparse_matvec_many_dev(sel, W, rx, cnt, vec_off=j0 * dev.m)
        proofs.extend(device_prover.prove_batch(key, uA, uB, uC, keys.Z, rx, rs[j0:j0 + cnt], ss[j0:j0 + cnt], chunk=cnt))
        for h in (uA, uB, uC, rx):
            h.free()
    return proofs
