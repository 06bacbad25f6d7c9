"""Witness solving on the GPU: many inputs of one circuit per call, feeding the batch provers.

The reference computes every witness on the host: zkp/groth16/code_to_r1cs.py assigns the variables of the flattened
program, and zkp/plonk/circuit.py fills the wire vectors a, b, c while it builds the circuit.  Here a circuit is
compiled once, on the host, into a step program (csrc/witness.cuh): variables v_0 = 1, the caller's inputs, and one
step per constraint or gate,

    N = (alpha . v)(beta . v) + gamma . v,    D = delta . v,

that either solves one variable (v_out = N / D) or checks N = 0.  Steps are sorted by level, so one launch solves
`count` witnesses whatever the depth of the circuit.  A returned witness satisfies every constraint or gate;
otherwise solve_batch raises, naming the proof and the constraint.  There is no host evaluation path.

    prog = compile_r1cs(r1cs, inputs=[1])            # qap_device.SparseR1CS, caller-supplied wires
    W = solve_batch(prog, X, count)                  # X: count * len(inputs) scalars -> count * m values
    proofs = qap_device.prove_batch(keys, dev, W, rs, ss)

    prog = compile_plonk(n, selectors, sigma, inputs=[0])
    a, b, c = solve_batch(prog, X, count)            # count * n values each
    proofs = plonk.device_prover.prove_batch(key, a, b, c, count)

    prog = compile_plonk(n, selectors, sigma, inputs=[0], num_public_inputs=l)
    a, b, c, pub = solve_batch(prog, X, count)       # X rows: l public inputs, then the inputs; pub: count * l values
    proofs = plonk.device_prover.prove_batch(key, a, b, c, count, public_inputs=pub)
"""
import heapq

import numpy as np

from .. import native

R = native.R_MOD
CHECK = 0xFFFFFFFF       # out_var of a check step
ONE = {0: 1}             # delta of a step without division


def _add(form, var, coeff):
    c = (form.get(var, 0) + coeff) % R
    if c:
        form[var] = c
    else:
        form.pop(var, None)


def _scaled(form, k):
    k %= R
    return {v: c * k % R for v, c in form.items()} if k else {}


class WitnessProgram:
    """A compiled circuit: the step program (host arrays, uploaded to the device on first use) and how its variables
    map to the outputs.  kind "r1cs": variable i is wire i.  kind "plonk": variables are the copy classes of sigma that
    some gate uses (v_0 = 1 is not a class); pos_var[p] is the variable of wire position p, -1 for a class fixed at 0;
    pub_var: the variables of the public inputs (the first entries of each input row)."""

    def __init__(self, kind, nvars, in_var, steps, size, pos_var=None, pub_var=()):
        self.kind, self.nvars, self.size, self.pos_var = kind, nvars, size, pos_var
        self.pub_var = list(pub_var)
        self.in_var = np.asarray(in_var, dtype=np.uint32)
        steps = sorted(steps, key=lambda st: (st[0], st[1]))   # (level, source index, out_var, forms)
        self.step_src = [st[1] for st in steps]
        self.out_var = np.asarray([CHECK if st[2] is None else st[2] for st in steps], dtype=np.uint32)
        levels = [st[0] for st in steps]
        nlev = levels[-1] if levels else 0
        self.level_ptr = np.searchsorted(np.asarray(levels, dtype=np.int64), np.arange(1, nlev + 2), side="left").astype(np.uint32)
        rp, ci, vals = [0], [], []
        for st in steps:
            for form in st[3]:
                for v in sorted(form):
                    ci.append(v)
                    vals.append(form[v])
                rp.append(len(ci))
        self.row_ptr = np.asarray(rp, dtype=np.uint32)
        self.col_idx = np.asarray(ci, dtype=np.uint32)
        self.values = vals
        self.quotient = [st[2] is not None and st[3][3] != ONE for st in steps]
        self._dev = None
        self._sel = None

    @property
    def steps(self):
        return len(self.out_var)

    @property
    def levels(self):
        return len(self.level_ptr) - 1

    @property
    def n_in(self):
        return len(self.in_var)

    def form(self, s, f):
        """{variable: coefficient} of form f (0 alpha, 1 beta, 2 gamma, 3 delta) of step s."""
        lo, hi = self.row_ptr[4 * s + f], self.row_ptr[4 * s + f + 1]
        return {int(self.col_idx[e]): self.values[e] for e in range(lo, hi)}

    def device(self):
        if self._dev is None:
            self._dev = native.witness_program_load(self.row_ptr, self.col_idx, self.values, self.out_var, self.level_ptr,
                                                    self.in_var, self.nvars)
        return self._dev

    def selections(self):
        """PLONK: the n x nvars 0/1 matrices that gather a, b, c from the variables (an empty row gives 0), and with
        public inputs the l x nvars one that gathers them."""
        if self._sel is None:
            n = self.size
            self._sel = []
            parts = [self.pos_var[part * n:(part + 1) * n] for part in range(3)]
            for pv in parts + ([self.pub_var] if self.pub_var else []):
                rows = [[v] if v >= 0 else [] for v in pv]
                rp = np.cumsum([0] + [len(r) for r in rows]).astype(np.uint32)
                ci = [v for r in rows for v in r]
                self._sel.append(native.sparse_load(rp, ci, [1] * len(ci), len(pv), self.nvars))
        return self._sel

    def free(self):
        for h in ([self._dev] if self._dev is not None else []) + (self._sel or []):
            h.free()
        self._dev = self._sel = None


def _schedule(ncons, cons_vars, nvars, known, solve, check):
    """The deterministic worklist shared by both compilers: always take the lowest-index constraint with exactly one
    unknown variable u; solve(i, u) gives its forms or None (it cannot determine u).  Every constraint that solves
    nothing becomes a check.  Returns (steps, the set of variables left unknown)."""
    var_cons = [[] for _ in range(nvars)]
    unknown = [0] * ncons
    for i, vs in enumerate(cons_vars):
        for v in vs:
            var_cons[v].append(i)
            if not known[v]:
                unknown[i] += 1
    level = [0] * nvars
    heap = [i for i in range(ncons) if unknown[i] == 1]
    heapq.heapify(heap)
    used = [False] * ncons
    steps = []

    def step_level(forms):
        return 1 + max((level[v] for f in forms for v in f), default=0)

    while heap:
        i = heapq.heappop(heap)
        if unknown[i] != 1:
            continue
        u = next(v for v in cons_vars[i] if not known[v])
        forms = solve(i, u)
        if forms is None:
            continue
        used[i] = True
        known[u] = True
        level[u] = step_level(forms)
        steps.append((level[u], i, u, forms))
        for c in var_cons[u]:
            unknown[c] -= 1
            if unknown[c] == 1:
                heapq.heappush(heap, c)
    left = [v for v in range(nvars) if not known[v]]
    if not left:
        for i in range(ncons):
            if not used[i]:
                forms = check(i)
                steps.append((step_level(forms), i, None, forms))
    return steps, left


def compile_r1cs(r1cs, inputs):
    """Step program of a sparse R1CS (qap_device.SparseR1CS: (A.w) o (B.w) = C.w, wire 0 = 1).  `inputs`: the wires
    the caller supplies, in the order of each witness's input row.  A constraint with one unknown wire u solves it:
    u only in C gives u = (A'B' - C') / c_u; u in A only (or B only) gives the quotient u = (C' - A'B') / (a_u B' - c_u),
    checked for zero at run time; u in both A and B cannot be solved by that constraint.  ValueError for a bad input
    list or a wire no constraint determines."""
    m, k = r1cs.m, r1cs.k
    inputs = [int(i) for i in inputs]
    if any(not 1 <= i < m for i in inputs) or len(set(inputs)) != len(inputs):
        raise ValueError("compile_r1cs: inputs must be distinct wires in [1, %d) (wire 0 is the constant 1)" % m)
    rows = []
    for rp, ci, vals in r1cs.mats:
        rows.append([{} for _ in range(k)])
        for g in range(k):
            for e in range(int(rp[g]), int(rp[g + 1])):
                _add(rows[-1][g], int(ci[e]), vals[e])
    A, B, C = rows
    cons_vars = [sorted(set(A[g]) | set(B[g]) | set(C[g])) for g in range(k)]
    known = [False] * m
    known[0] = True
    for i in inputs:
        known[i] = True

    def solve(g, u):
        a_u, b_u, c_u = A[g].get(u, 0), B[g].get(u, 0), C[g].get(u, 0)
        if a_u and b_u:
            return None
        drop = lambda f: {v: c for v, c in f.items() if v != u}
        if not a_u and not b_u:
            inv = pow(c_u, -1, R)
            return (_scaled(drop(A[g]), inv), drop(B[g]), _scaled(drop(C[g]), R - inv), ONE)
        lin, other, coeff = (A[g], B[g], a_u) if a_u else (B[g], A[g], b_u)
        den = _scaled(drop(other), coeff)
        _add(den, 0, -c_u)
        alpha, beta, gamma = _scaled(drop(lin), R - 1), drop(other), drop(C[g])
        if set(den) <= {0}:
            if not den:
                return None
            inv = pow(den[0], -1, R)
            return (_scaled(alpha, inv), beta, _scaled(gamma, inv), ONE)
        return (alpha, beta, gamma, den)

    def check(g):
        return (dict(A[g]), dict(B[g]), _scaled(C[g], R - 1), ONE)

    steps, left = _schedule(k, cons_vars, m, known, solve, check)
    if left:
        raise ValueError("compile_r1cs: wire %d is not determined by the constraints (%d wires undetermined)" % (left[0], len(left)))
    return WitnessProgram("r1cs", m, inputs, steps, m)


def compile_plonk(n, selectors, sigma, inputs, num_public_inputs=0):
    """Step program of a PLONK circuit in the reference's layout: selectors = (q_l, q_r, q_o, q_m, q_c), n values each;
    sigma a permutation of the 3n wire positions (a_g at g, b_g at n + g, c_g at 2n + g); inputs: the positions the
    caller supplies.  Variables are the copy classes (cycles of sigma).  A gate q_l a + q_r b + q_o c + q_m a b + q_c = 0
    solves its single unknown class when the equation is of degree 1 in it; the coefficient may be a linear form
    (q_l + q_m b when the unknown is a).  A class no gate uses with a non-zero coefficient, and not an input, is 0.
    num_public_inputs: l public inputs x_0..x_{l-1}, fresh variables that come first in every input row; gate i < l
    gains + x_i (q_l a + q_r b + q_o c + q_m a b + q_c + x_i = 0, the PI term of device_prover's public inputs).
    ValueError for two inputs in one class, an undetermined class or l outside [0, n]."""
    n = int(n)
    ell = int(num_public_inputs)
    if not 0 <= ell <= n:
        raise ValueError("compile_plonk: num_public_inputs must be in [0, %d], got %d" % (n, ell))
    q = [[int(x) % R for x in s] for s in selectors]
    sigma = [int(s) for s in sigma]
    if len(q) != 5 or any(len(s) != n for s in q):
        raise ValueError("compile_plonk: five selectors of %d values" % n)
    if sorted(sigma) != list(range(3 * n)):
        raise ValueError("compile_plonk: sigma must be a permutation of the %d wire positions" % (3 * n))
    cls = [-1] * (3 * n)
    ncls = 0
    for p in range(3 * n):
        if cls[p] < 0:
            x = p
            while cls[x] < 0:
                cls[x] = ncls
                x = sigma[x]
            ncls += 1
    q_l, q_r, q_o, q_m, q_c = q
    slots = []                       # per gate: the class of a, b, c if that slot has a non-zero coefficient, else None
    for g in range(n):
        slots.append((cls[g] if q_l[g] or q_m[g] else None, cls[n + g] if q_r[g] or q_m[g] else None,
                      cls[2 * n + g] if q_o[g] else None))
    inputs = [int(p) for p in inputs]
    if any(not 0 <= p < 3 * n for p in inputs):
        raise ValueError("compile_plonk: input positions must be in [0, %d)" % (3 * n))
    in_cls = [cls[p] for p in inputs]
    if len(set(in_cls)) != len(in_cls):
        raise ValueError("compile_plonk: two inputs lie in one copy class (positions %s)" % inputs)
    used = set(in_cls) | {c for s in slots for c in s if c is not None}
    var_of = {c: i + 1 for i, c in enumerate(sorted(used))}
    pub_var = [len(used) + 1 + i for i in range(ell)]
    pub_of = lambda g: pub_var[g] if g < ell else None     # the public-input variable in gate g's equation
    nvars = len(used) + 1 + ell
    pos_var = [var_of.get(c, -1) for c in cls]
    gv = [tuple(var_of[c] if c is not None else None for c in s) for s in slots]
    cons_vars = [sorted({v for v in s if v is not None}) for s in gv]
    known = [False] * nvars
    known[0] = True
    for v in pub_var:
        known[v] = True
    for c in in_cls:
        known[var_of[c]] = True

    def solve(g, u):
        xa, xb, xc = gv[g]
        sa, sb, sc = xa == u, xb == u, xc == u
        if q_m[g] and sa and sb:
            return None
        coeff, alpha, beta, gamma = {}, {}, {}, {}
        _add(coeff, 0, q_l[g] * sa + q_r[g] * sb + q_o[g] * sc)
        if q_m[g]:
            if sa:
                _add(coeff, xb, q_m[g])
            elif sb:
                _add(coeff, xa, q_m[g])
            else:
                alpha, beta = {xa: R - q_m[g]}, {xb: 1}
        for x, s, sel in ((xa, sa, q_l[g]), (xb, sb, q_r[g]), (xc, sc, q_o[g])):
            if x is not None and not s and sel:
                _add(gamma, x, R - sel)
        _add(gamma, 0, R - q_c[g])
        if pub_of(g) is not None:
            _add(gamma, pub_of(g), R - 1)
        if set(coeff) <= {0}:
            if not coeff:
                return None
            inv = pow(coeff[0], -1, R)
            return (_scaled(alpha, inv), beta, _scaled(gamma, inv), ONE)
        return (alpha, beta, gamma, coeff)

    def check(g):
        xa, xb, xc = gv[g]
        gamma = {}
        for x, sel in ((xa, q_l[g]), (xb, q_r[g]), (xc, q_o[g])):
            if x is not None and sel:
                _add(gamma, x, sel)
        _add(gamma, 0, q_c[g])
        if pub_of(g) is not None:
            _add(gamma, pub_of(g), 1)
        return ({xa: q_m[g]} if q_m[g] else {}, {xb: 1} if q_m[g] else {}, gamma, ONE)

    steps, left = _schedule(n, cons_vars, nvars, known, solve, check)
    if left:
        p = pos_var.index(left[0])
        raise ValueError("compile_plonk: the copy class of %s_%d (position %d) is not determined by the gates "
                         "(%d classes undetermined)" % ("abc"[p // n], p % n, p, len(left)))
    return WitnessProgram("plonk", nvars, pub_var + [var_of[c] for c in in_cls], steps, n, pos_var, pub_var)


def solve_batch(program, X, count):
    """Solve `count` witnesses of `program` on the device from the scalar handle X (witness j's inputs at
    X[j * n_in], in the order of the compiler's `inputs`).  R1CS: returns W, count * m values (witness j at j * m),
    as qap_device.prove_batch takes it.  PLONK: returns the (a_vals, b_vals, c_vals) handles of count * n values each,
    as plonk.device_prover.prove_batch takes them, and for a program with l public inputs a fourth handle of count * l
    values (proof j's at j * l), its public_inputs.  One solving launch whatever count and the circuit depth are.
    ValueError naming the first failing proof and its constraint (gate) when a division by zero occurs or a
    constraint is not satisfied."""
    count = int(count)
    if count < 0:
        raise ValueError("solve_batch: count must be >= 0")
    if X is None or X.n < count * program.n_in:
        raise ValueError("solve_batch: X holds %s values, needs %d" % (None if X is None else X.n, count * program.n_in))
    W = native.scalars_alloc(count * program.nvars)
    bad = native.witness_solve_many_dev(program.device(), X, count, W)
    if bad is not None:
        W.free()
        j, s = divmod(bad, program.steps)
        what = "constraint" if program.kind == "r1cs" else "gate"
        reason = "division by zero" if program.quotient[s] else "constraint not satisfied"
        raise ValueError("solve_batch: proof %d, %s %d: %s" % (j, what, program.step_src[s], reason))
    if program.kind == "r1cs":
        return W
    out = []
    for sel in program.selections():
        h = native.scalars_alloc(count * sel.n)
        if count:
            native.sparse_matvec_many_dev(sel, W, h, count)
        out.append(h)
    W.free()
    return tuple(out)
