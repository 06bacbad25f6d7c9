"""-m gpu: witness solving on the device (zkp/witness.py, csrc/witness.cuh).

(1) the golden code_to_r1cs programs solved bit for bit, and proved into the reference's proofs; (2) the golden PLONK
circuits solved into their a, b, c and proved with the golden blinds; (3) synthetic circuits against host witnesses,
and at 2^16 constraints every witness checked against the R1CS on the device; (4) a batch against count = 1 solves;
(5) a zero divisor and a violated constraint reported with their proof and constraint; (6) one solving launch
whatever the count and depth; (7) solve_batch -> prove_batch -> verify_batch for 128 distinct proofs of each system."""
import os
import random
import sys

import pytest

from oracle import bn254
from tests.util import g1, g2, ints, load

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

pytestmark = pytest.mark.gpu
R = bn254.R


def _vals(native, h):
    return native.fr_vec_from_bytes(native.scalars_download(h, 0, h.n))


def _load(native, xs):
    return native.scalars_load(native.fr_vec_bytes(xs), len(xs))


def _proof_ints(prf):
    A, B, C = prf
    return ((int(A[0]), int(A[1])), ((int(B[0].coeffs[0]), int(B[0].coeffs[1])), (int(B[1].coeffs[0]), int(B[1].coeffs[1]))),
            (int(C[0]), int(C[1])))


def _proof_dict(proof):
    return {k: (g1(v) if k.endswith("_comm") else int(v)) for k, v in vars(proof).items()}


def _host_r1cs_witnesses(ra, rb, count, seed):
    """tools/qap_large.circuit's witnesses for random inputs: w_{g+2} = (A_g . w)(B_g . w), as the host computes them."""
    rng = random.Random(seed)
    out = []
    for _ in range(count):
        w = [1, rng.randrange(2, 1 << 20)]
        for a, b in zip(ra, rb):
            w.append(sum(v * w[i] for i, v in a.items()) * sum(v * w[i] for i, v in b.items()) % R)
        out.append(w)
    return out


def _qap_program(k, seed=99):
    from qap_large import circuit
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs
    ra, rb, rc, _ = circuit(k, seed)
    r1cs = qd.SparseR1CS.from_rows(k, k + 2, ra, rb, rc)
    return ra, rb, r1cs, compile_r1cs(r1cs, [1])


def _chain_program(n):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    c0 = plonk_synth.chain_circuit(n, seed=1)
    return compile_plonk(n, c0["sel"], c0["sigma"], [0] + [n + g for g in range(n)])


def _chain_inputs(circs):
    return [x for c in circs for x in [c["a"][0]] + c["b"]]


@pytest.mark.parametrize("case", [0, 1])
def test_golden_r1cs_solved_and_proved(native, case):
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs, solve_batch
    c = load("groth16_qap.json")["cases"][case]
    r1cs = qd.SparseR1CS.from_dense(c["r1cs_A"], c["r1cs_B"], c["r1cs_C"])
    W = solve_batch(compile_r1cs(r1cs, [1]), _load(native, [c["witness"][1]]), 1)
    assert _vals(native, W) == ints(c["witness"])
    dev = qd.DeviceR1CS(r1cs)
    t = {key: int(v) for key, v in c["toxic"].items()}
    keys = qd.setup(dev, t["alpha"], t["beta"], t["gamma"], t["delta"], t["x_val"], pub_r_indexs=c["pub_r_indexs"],
                    precompute=False)
    got = _proof_ints(qd.prove(keys, dev, W, int(c["r"]), int(c["s"])))
    assert got == (g1(c["proof_a"]), g2(c["proof_b"]), g1(c["proof_c"]))


@pytest.mark.parametrize("name", ["plonk_n1.json", "plonk_x3.json", "plonk_chain16.json"])
def test_golden_plonk_solved_and_proved(native, name):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.witness import compile_plonk, solve_batch
    f = load(name)
    n = f["n"]
    sel = [ints(f["selectors"][k]) for k in ("q_l", "q_r", "q_o", "q_m", "q_c")]
    pos = {"plonk_x3.json": [0], "plonk_n1.json": [0, 1], "plonk_chain16.json": [0] + [n + g for g in range(13)]}[name]
    wires = ints(f["a_vals"]) + ints(f["b_vals"]) + ints(f["c_vals"])
    abc = solve_batch(compile_plonk(n, sel, f["sigma"], pos), _load(native, [wires[p] for p in pos]), 1)
    assert [_vals(native, h) for h in abc] == [ints(f[k + "_vals"]) for k in "abc"]
    pts = [g1(p) for p in f["g1_powers"]]
    srs = native.g1_table_load(native.g1_vec_bytes(pts), len(pts))
    sel_h = [native.scalars_load(native.fr_vec_bytes(s), n) for s in sel]
    sig_h = [native.scalars_load(b, n) for b in plonk_synth.sigma_evals_bytes(f["sigma"], n, int(f["omega"]))]
    key = dp.preprocess(n, sel_h, sig_h, srs, len(pts))
    proof = dp.prove(key, *abc, blinds=ints(f["blinds"]))
    assert _proof_dict(proof) == {k: (g1(v) if k.endswith("_comm") else int(v)) for k, v in f["proof"].items()}


def test_synthetic_r1cs_2_12_matches_host(native):
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    k, count = 1 << 12, 64
    ra, rb, _, prog = _qap_program(k)
    host = _host_r1cs_witnesses(ra, rb, count, 3)
    W = solve_batch(prog, _load(native, [w[1] for w in host]), count)
    assert _vals(native, W) == [x for w in host for x in w]


def test_synthetic_r1cs_2_16_satisfies_every_constraint(native):
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    k, count = 1 << 16, 32
    m = k + 2
    ra, rb, r1cs, prog = _qap_program(k, seed=7)
    rng = random.Random(16)
    xs = [rng.randrange(2, R) for _ in range(count)]
    W = solve_batch(prog, _load(native, xs), count)
    dev = qd.DeviceR1CS(r1cs)
    ev = [native.scalars_alloc(count * k) for _ in range(3)]
    for mat, e in zip(dev.mats, ev):
        native.sparse_matvec_many_dev(mat, W, e, count)
    native.vec_op_dev(2, ev[0], 0, ev[0], 0, ev[1], 0, count * k)
    native.vec_op_dev(1, ev[0], 0, ev[0], 0, ev[2], 0, count * k)
    assert native.scalars_is_zero(ev[0], 0, count * k)
    got = _vals(native, W)
    for j in (0, 1, 17, count - 1):
        w = [1, xs[j]]
        for a, b in zip(ra, rb):
            w.append(sum(v * w[i] for i, v in a.items()) * sum(v * w[i] for i, v in b.items()) % R)
        assert got[j * m:(j + 1) * m] == w


@pytest.mark.parametrize("log_n,count", [(12, 64), (14, 8)])
def test_synthetic_chain_matches_host(native, log_n, count):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    n = 1 << log_n
    prog = _chain_program(n)
    circs = [plonk_synth.chain_circuit(n, seed=50 + j) for j in range(count)]
    abc = solve_batch(prog, _load(native, _chain_inputs(circs)), count)
    for h, key in zip(abc, "abc"):
        assert _vals(native, h) == [x for c in circs for x in c[key]]


def test_batch_equals_single_solves(native):
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    k, count = 1 << 10, 12
    m = k + 2
    _, _, _, prog = _qap_program(k, seed=4)
    xs = [random.Random(j).randrange(R) for j in range(count)]
    batch = _vals(native, solve_batch(prog, _load(native, xs), count))
    for j in range(count):
        assert batch[j * m:(j + 1) * m] == _vals(native, solve_batch(prog, _load(native, [xs[j]]), 1))


def _division_program():
    """w3 = w1 / w2 (w3 * w2 = w1), w4 = w1 * w1, and the check w4 * 1 = w5 with w5 an input."""
    from interactive_zkp_study_b200.zkp.groth16.qap_device import SparseR1CS
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs
    r1cs = SparseR1CS.from_rows(3, 6, [{3: 1}, {1: 1}, {4: 1}], [{2: 1}, {1: 1}, {0: 1}], [{1: 1}, {4: 1}, {5: 1}])
    return compile_r1cs(r1cs, [1, 2, 5])


def test_failures_name_the_proof_and_the_constraint(native):
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    prog = _division_program()
    good = [[x, x + 1, x * x % R] for x in range(3, 11)]
    zero_div = [list(r) for r in good]
    zero_div[5][1] = 0
    unsat = [list(r) for r in good]
    unsat[3][2] += 1
    flat = lambda rows: _load(native, [x for r in rows for x in r])
    with pytest.raises(ValueError, match=r"proof 5, constraint 0: division by zero"):
        solve_batch(prog, flat(zero_div), 8)
    with pytest.raises(ValueError, match=r"proof 3, constraint 2: constraint not satisfied"):
        solve_batch(prog, flat(unsat), 8)
    both = [list(r) for r in zero_div]
    both[3] = unsat[3]
    with pytest.raises(ValueError, match=r"proof 3, constraint 2"):
        solve_batch(prog, flat(both), 8)
    others = [r for j, r in enumerate(both) if j not in (3, 5)]
    W = _vals(native, solve_batch(prog, flat(others), len(others)))
    for j, (x, y, z) in enumerate(others):
        assert W[6 * j:6 * j + 6] == [1, x, y, x * pow(y, -1, R) % R, x * x % R, z]


def test_one_solving_launch_whatever_count_and_depth(native):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    _, _, _, prog = _qap_program(1 << 12)
    per = {}
    for count in (1, 64, 1024):
        X = _load(native, list(range(2, count + 2)))
        solve_batch(prog, X, count)
        l0 = native.launch_count()
        solve_batch(prog, X, count)
        per[count] = native.launch_count() - l0
    assert per == {1: 1, 64: 1, 1024: 1}
    deep = {}
    for n in (16, 4096):
        prog = _chain_program(n)
        assert prog.levels == n
        X = _load(native, _chain_inputs([plonk_synth.chain_circuit(n, seed=j) for j in range(8)]))
        solve_batch(prog, X, 8)
        l0 = native.launch_count()
        solve_batch(prog, X, 8)
        deep[n] = native.launch_count() - l0
    assert deep[16] == deep[4096] == 4               # the solve and three selection products


def test_refusals_leave_the_library_usable(native):
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    prog = _division_program()
    dev = prog.device()
    X = _load(native, [3, 4, 9])
    out = native.scalars_alloc(6)
    with pytest.raises(native.ZkpB200Error):
        native.witness_solve_many_dev(dev, X, 2, out)                 # inputs too short
    with pytest.raises(native.ZkpB200Error):
        native.witness_solve_many_dev(dev, X, 1, out, out_off=1)      # output range too short
    with pytest.raises(native.ZkpB200Error):
        big = _load(native, [3, 4, 9] + [0] * 6)
        native.witness_solve_many_dev(dev, big, 1, big)               # outputs over the inputs
    with pytest.raises(native.ZkpB200Error):
        native.witness_program_load([0] * 5, [], [], [7], [0, 1], [], 6)  # a step writing past the variables
    with pytest.raises(native.ZkpB200Error):
        native.witness_program_load([0, 1, 1, 1, 1], [1], [1], [1], [0, 1], [], 2)  # a step reading its own output
    l0 = native.launch_count()
    assert native.witness_solve_many_dev(dev, X, 0, out) is None and native.launch_count() == l0
    assert _vals(native, solve_batch(prog, X, 1)) == [1, 3, 4, 3 * pow(4, -1, R) % R, 9, 9]


def test_solve_prove_verify_groth16_128(native):
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify_batch
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    k, count = 1 << 12, 128
    m = k + 2
    ra, rb, r1cs, prog = _qap_program(k)
    dev = qd.DeviceR1CS(r1cs)
    rng = random.Random(5)
    keys = qd.setup(dev, *(rng.randrange(1, R) for _ in range(5)), lcm=True, precompute=True)
    xs = [rng.randrange(2, 1 << 20) for _ in range(count)]
    rs = [rng.randrange(R) for _ in range(count)]
    ss = [rng.randrange(R) for _ in range(count)]
    proofs = qd.prove_batch(keys, dev, solve_batch(prog, _load(native, xs), count), rs, ss)
    vk = (keys.sigma1_1, keys.sigma1_3, keys.sigma2_1)
    pubs = [[(0, 1), (1, x)] for x in xs]
    assert keys.pub_idx == [0, 1]
    assert verify_batch(proofs, *vk, pubs, rng=random.Random(1)) is True
    w0 = [1, xs[0]]
    for a, b in zip(ra, rb):
        w0.append(sum(v * w0[i] for i, v in a.items()) * sum(v * w0[i] for i, v in b.items()) % R)
    assert _proof_ints(proofs[0]) == _proof_ints(qd.prove(keys, dev, _load(native, w0), rs[0], ss[0]))
    assert len({_proof_ints(p) for p in proofs}) == count and m == dev.m


def test_solve_prove_verify_plonk_128(native):
    import plonk_synth
    from interactive_zkp_study_b200.compat import G2, g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    from interactive_zkp_study_b200.zkp.witness import solve_batch
    n, count = 1 << 12, 128
    key, _, tau = plonk_synth.device_setup(plonk_synth.chain_circuit(n, seed=12))
    circs = [plonk_synth.chain_circuit(n, seed=2000 + j) for j in range(count)]
    abc = solve_batch(_chain_program(n), _load(native, _chain_inputs(circs)), count)
    rng = random.Random(8)
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(count)]
    proofs = dp.prove_batch(key, *abc, count, blinds=blinds)
    pp = type("PP", (), {})()
    pp.n, pp.omega = n, FR(key.omega)
    for name in dp.CIRCUIT_POLYS:
        setattr(pp, name + "_comm", key.comm[name])
    srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)
    assert verify_batch([(p, [], pp) for p in proofs], srs, rng=random.Random(1)) is True
    host0 = [_load(native, circs[0][k]) for k in "abc"]
    assert _proof_dict(proofs[0]) == _proof_dict(dp.prove(key, *host0, blinds=blinds[0]))
