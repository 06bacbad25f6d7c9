"""Synthetic satisfiable PLONK circuits at any power-of-two size, built directly as the vectors the
prover consumes (selector evaluations, sigma, witness): alternating mul/add gates wired as a chain
(c_g == a_{g+1}), the same shape as tests/golden/make_golden.py::chain_circuit but without the
reference's Circuit class, so it also runs on the GPU box and at 2^20 gates."""
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from interactive_zkp_study_b200 import native as nat  # noqa: E402

R = nat.R_MOD


def chain_circuit(n, seed=1, break_witness=False):
    rng = random.Random(seed)
    a, b, c = [0] * n, [0] * n, [0] * n
    q_l, q_r, q_o, q_m, q_c = ([0] * n for _ in range(5))
    sigma = list(range(3 * n))
    prev = rng.randrange(1, 1 << 60)
    for g in range(n):
        other = rng.randrange(1, 1 << 60)
        a[g], b[g] = prev, other
        if g % 2 == 0:                      # multiplication gate: q_m = 1, q_o = -1
            q_m[g], q_o[g] = 1, R - 1
            c[g] = prev * other % R
        else:                               # addition gate: q_l = q_r = 1, q_o = -1
            q_l[g], q_r[g], q_o[g] = 1, 1, R - 1
            c[g] = (prev + other) % R
        if g > 0:                           # copy constraint c_{g-1} == a_g  (circuit.py:190-247 semantics)
            p1, p2 = 2 * n + (g - 1), g
            sigma[p1], sigma[p2] = sigma[p2], sigma[p1]
        prev = c[g]
    if break_witness:
        c[n // 2] = (c[n // 2] + 1) % R
    return {"n": n, "a": a, "b": b, "c": c, "sel": [q_l, q_r, q_o, q_m, q_c], "sigma": sigma}


def random_circuit(n, seed=1, witness_seed=None, break_witness=False):
    """A satisfiable circuit of n gates whose structure is drawn from `seed`: every gate is a multiplication
    (c = a b), an addition (c = a + b) or an addition of a constant (c = a + k, q_c = k), and each of its a and b is,
    with probability 1/2, a copy of the output of an earlier gate (a copy constraint) or a fresh input.  Two seeds give
    circuits with different selectors and sigma.  witness_seed (default: seed) draws the fresh inputs, so one circuit
    has many witnesses; break_witness adds 1 to one output."""
    rng = random.Random(seed)
    kinds, const, src_a, src_b = [], [], [], []
    for g in range(n):
        kinds.append(rng.randrange(3))
        const.append(rng.randrange(1, 1 << 60))
        src_a.append(rng.randrange(g) if g and rng.random() < 0.5 else None)
        src_b.append(rng.randrange(g) if g and rng.random() < 0.5 else None)
    vals = random.Random(seed if witness_seed is None else witness_seed)
    a, b, c = [0] * n, [0] * n, [0] * n
    q_l, q_r, q_o, q_m, q_c = ([0] * n for _ in range(5))
    cycles = {}                                          # gate p -> wire positions holding c_p (c_p itself first)
    for g in range(n):
        x = c[src_a[g]] if src_a[g] is not None else vals.randrange(1, 1 << 60)
        y = c[src_b[g]] if src_b[g] is not None else vals.randrange(1, 1 << 60)
        a[g], b[g] = x, y
        q_o[g] = R - 1
        if kinds[g] == 0:
            q_m[g], c[g] = 1, x * y % R
        elif kinds[g] == 1:
            q_l[g], q_r[g], c[g] = 1, 1, (x + y) % R
        else:
            q_l[g], q_c[g], c[g] = 1, const[g], (x + const[g]) % R
        for p, pos in ((src_a[g], g), (src_b[g], n + g)):
            if p is not None:
                cycles.setdefault(p, [2 * n + p]).append(pos)
    sigma = list(range(3 * n))
    for cyc in cycles.values():                          # each copy class one cycle of the permutation
        for i, pos in enumerate(cyc):
            sigma[pos] = cyc[(i + 1) % len(cyc)]
    if break_witness:
        c[n // 2] = (c[n // 2] + 1) % R
    return {"n": n, "a": a, "b": b, "c": c, "sel": [q_l, q_r, q_o, q_m, q_c], "sigma": sigma}


def prepend_public_gates(circ, tied, n=None, public_inputs=None):
    """The circuit `circ` (keys n, a, b, c, sel, sigma) behind len(tied) public-input gates, padded with zero gates to n
    gates (default: the smallest power of two that fits).  Gate i has q_l = -1, so with the PI term it reads
    x_i - a_i = 0, and a_i is copy-constrained to wire position tied[i] of circ; x_i defaults to that wire's value.
    Adds "num_public_inputs", "public_inputs" and "pos", the map from circ's wire positions to the new ones."""
    ell, m = len(tied), circ["n"]
    n = n or 1 << max(0, (m + ell - 1).bit_length())
    if n < m + ell:
        raise ValueError("prepend_public_gates: %d gates do not fit in %d" % (m + ell, n))
    pos = lambda p: (p // m) * n + ell + p % m
    sigma = list(range(3 * n))
    for p in range(3 * m):
        sigma[pos(p)] = pos(circ["sigma"][p])
    for i, p in enumerate(tied):                          # splice a_i into the copy cycle of the tied wire
        q = pos(p)
        sigma[i], sigma[q] = sigma[q], sigma[i]
    wires = circ["a"] + circ["b"] + circ["c"]
    x = [wires[p] for p in tied] if public_inputs is None else list(public_inputs)
    pad, zeros = [0] * (n - ell - m), [0] * ell
    a, b, c = (x + circ["a"] + pad, zeros + circ["b"] + pad, zeros + circ["c"] + pad)
    sel = [zeros + list(q) + pad for q in circ["sel"]]
    sel[0][:ell] = [R - 1] * ell
    return {"n": n, "a": a, "b": b, "c": c, "sel": sel, "sigma": sigma, "num_public_inputs": ell,
            "public_inputs": x, "pos": [pos(p) for p in range(3 * m)]}


def public_chain_circuit(n, ell, seed=1):
    """chain_circuit of n - ell gates behind ell public-input gates, public input i tied to b of chain gate i
    (2 ell <= n): the public inputs are the first ell free inputs of the chain.  "inputs": the wire positions a witness
    solver takes after the public inputs (a of the first chain gate, then the untied b's)."""
    if not 0 <= 2 * ell <= n:
        raise ValueError("public_chain_circuit: needs 2 * ell <= n")
    m = n - ell
    circ = prepend_public_gates(chain_circuit(m, seed), [m + i for i in range(ell)], n)
    circ["inputs"] = [ell] + [n + g for g in range(2 * ell, n)]
    return circ


def sigma_evals_bytes(sigma, n, omega):
    """Evaluations of S_sigma1..3 (permutation.py:44-86): position -> K * w^i, as three byte strings."""
    dom = nat.scalars_alloc(n)
    nat.scalars_fill_powers(dom, 0, n, 1, omega)
    d1 = nat.scalars_download(dom, 0, n)
    nat.scalars_scale(dom, 0, n, 2)
    d2 = nat.scalars_download(dom, 0, n)
    nat.scalars_fill_powers(dom, 0, n, 3, omega)
    d3 = nat.scalars_download(dom, 0, n)
    dom.free()
    table = d1 + d2 + d3
    out = []
    for part in range(3):
        out.append(b"".join(table[32 * sigma[part * n + i]:32 * sigma[part * n + i] + 32] for i in range(n)))
    return out


def device_srs(size, srs_tau=None, precompute=True):
    """An SRS table of `size` G1 powers tau^i G on the device (prefix product + fixed-base kernel) -> (table, tau)."""
    tau = srs_tau or 0x1d0c2e3f4a5b6c7d8e9fa0b1c2d3e4f5061728394a5b6c7d8e9f0011223344 % R
    powers = nat.fr_prefix_product(nat.fr_vec_bytes([tau] * size), size)
    srs = nat.g1_fixed_base_mul(nat.g1_bytes((1, 2)), powers, size)
    if precompute and size >= (1 << 12):
        nat.table_precompute(srs)
    return srs, tau


def device_key(circ, srs, srs_size):
    """The circuit uploaded and preprocessed against an existing SRS table -> (key, witness handles).  Keys made this
    way against one table can share the passes of device_prover.prove_batch_circuits."""
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import get_root_of_unity
    n = circ["n"]
    omega = int(get_root_of_unity(n))
    enc = nat.fr_vec_bytes
    sel_h = [nat.scalars_load(enc(v), n) for v in circ["sel"]]
    sig_h = [nat.scalars_load(bts, n) for bts in sigma_evals_bytes(circ["sigma"], n, omega)]
    key = dp.preprocess(n, sel_h, sig_h, srs, srs_size, num_public_inputs=circ.get("num_public_inputs", 0))
    return key, [nat.scalars_load(enc(circ[k]), n) for k in "abc"]


def device_setup_many(circs, srs_tau=None, precompute=True):
    """Several circuits of one size preprocessed against ONE SRS table (device_setup builds a table per call).
    Returns (keys, witness handles per circuit, tau)."""
    n = circs[0]["n"]
    if any(c["n"] != n for c in circs):
        raise ValueError("device_setup_many: the circuits differ in size")
    srs, tau = device_srs(n + 6, srs_tau, precompute)
    keys, wits = zip(*[device_key(c, srs, n + 6) for c in circs])
    return list(keys), list(wits), tau


def device_setup(circ, srs_tau=None, precompute=True, comm=None):
    """SRS on the device (tau^i G from a prefix-product + fixed-base kernel), the circuit uploaded, the
    device key preprocessed.  Returns (key, witness handles, tau).  comm: a sharded.Communicator -> every rank
    keeps only its row range of the SRS and all commitments are collective (same arguments on every rank).  A circuit
    with "num_public_inputs" (public_chain_circuit) gets a key bound to that many public inputs."""
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import get_root_of_unity
    n = circ["n"]
    tau = srs_tau or 0x1d0c2e3f4a5b6c7d8e9fa0b1c2d3e4f5061728394a5b6c7d8e9f0011223344 % R
    size = n + 6
    powers = nat.fr_prefix_product(nat.fr_vec_bytes([tau] * size), size)
    srs_range = None
    if comm is not None:
        from interactive_zkp_study_b200 import sharded
        srs_range = sharded.shard_range(size, comm.rank, comm.world)
        powers = powers[32 * srs_range[0]:32 * (srs_range[0] + srs_range[1])]
    rows = size if srs_range is None else srs_range[1]
    srs = nat.g1_fixed_base_mul(nat.g1_bytes((1, 2)), powers, rows)
    if precompute and rows >= (1 << 12):
        nat.table_precompute(srs)
    omega = int(get_root_of_unity(n))
    enc = nat.fr_vec_bytes
    sel_h = [nat.scalars_load(enc(v), n) for v in circ["sel"]]
    sig_h = [nat.scalars_load(bts, n) for bts in sigma_evals_bytes(circ["sigma"], n, omega)]
    key = dp.preprocess(n, sel_h, sig_h, srs, size, comm=comm, srs_range=srs_range,
                        num_public_inputs=circ.get("num_public_inputs", 0))
    wit = [nat.scalars_load(enc(circ[k]), n) for k in "abc"]
    return key, wit, tau
