"""CPU: the witness compilers of zkp/witness.py (host-only).  Their step programs are run here by a small interpreter
that follows the semantics of csrc/witness.cuh (v_0 = 1, inputs, steps in level order, N / D or N = 0, the lowest
failing step), and must reproduce the reference's witnesses: the golden code_to_r1cs programs, the golden PLONK
circuits with their padding gates and unused b slot, and the synthetic circuits of tools/."""
import os
import sys

import pytest

from tests.util import ints, load

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

R = 21888242871839275222246405745257275088548364400416034343698204186575808495617


def run(prog, inputs):
    """(values, index of the first failing step or None); checks the level order on the way."""
    from interactive_zkp_study_b200.zkp.witness import CHECK
    v = [None] * prog.nvars
    lvl = [None] * prog.nvars
    v[0], lvl[0] = 1, 0
    assert len(inputs) == prog.n_in
    for var, x in zip(prog.in_var, inputs):
        v[int(var)], lvl[int(var)] = int(x) % R, 0
    bad = None
    lp = [int(x) for x in prog.level_ptr]
    assert lp[0] == 0 and lp[-1] == prog.steps and lp == sorted(lp)
    for level in range(1, prog.levels + 1):
        for s in range(lp[level - 1], lp[level]):
            forms = [prog.form(s, f) for f in range(4)]
            for f in forms:
                for i in f:
                    assert lvl[i] is not None and lvl[i] < level, "step %d reads variable %d of level %s" % (s, i, lvl[i])
            dot = lambda f: sum(c * v[i] for i, c in f.items()) % R
            N = (dot(forms[0]) * dot(forms[1]) + dot(forms[2])) % R
            o = int(prog.out_var[s])
            if o == CHECK:
                ok = N == 0
            else:
                assert v[o] is None, "variable %d written twice" % o
                D = dot(forms[3])
                ok = D != 0
                v[o], lvl[o] = N * pow(D, -1, R) % R if D else 0, level
            if not ok and bad is None:
                bad = s
    assert None not in v
    return v, bad


def abc(prog, v):
    n = prog.size
    vals = [v[p] if p >= 0 else 0 for p in prog.pos_var]
    return vals[:n], vals[n:2 * n], vals[2 * n:]


def r1cs_of(case):
    from interactive_zkp_study_b200.zkp.groth16.qap_device import SparseR1CS
    return SparseR1CS.from_dense(case["r1cs_A"], case["r1cs_B"], case["r1cs_C"])


@pytest.mark.parametrize("idx", [0, 1])
def test_golden_r1cs_witness(idx):
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs
    case = load("groth16_qap.json")["cases"][idx]
    prog = compile_r1cs(r1cs_of(case), [1])
    v, bad = run(prog, [case["witness"][1]])
    assert bad is None and v == ints(case["witness"])
    assert prog.steps == case["numGates"] and prog.nvars == case["numWires"]


PLONK_INPUTS = {"plonk_x3.json": lambda n: [0], "plonk_n1.json": lambda n: [0, 1],
                "plonk_chain16.json": lambda n: [0] + [n + g for g in range(13)]}


def plonk_program(name):
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    f = load(name)
    n = f["n"]
    sel = [ints(f["selectors"][k]) for k in ("q_l", "q_r", "q_o", "q_m", "q_c")]
    pos = PLONK_INPUTS[name](n)
    wires = ints(f["a_vals"]) + ints(f["b_vals"]) + ints(f["c_vals"])
    return f, compile_plonk(n, sel, f["sigma"], pos), [wires[p] for p in pos]


@pytest.mark.parametrize("name", sorted(PLONK_INPUTS))
def test_golden_plonk_wires(name):
    f, prog, x = plonk_program(name)
    v, bad = run(prog, x)
    assert bad is None
    assert abc(prog, v) == (ints(f["a_vals"]), ints(f["b_vals"]), ints(f["c_vals"]))


def test_plonk_x3_unused_b_slot_is_zero_and_not_a_variable():
    f, prog, _ = plonk_program("plonk_x3.json")
    n = f["n"]
    assert prog.pos_var[n + 3] == -1                 # b_3: its gate has q_r = q_m = 0
    assert prog.nvars == 6                           # v_0 and the classes {x}, 9, 27, 30, 35


def test_synthetic_r1cs_matches_host_witness():
    import qap_large
    from interactive_zkp_study_b200.zkp.groth16.qap_device import SparseR1CS
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs
    k = 1 << 9
    ra, rb, rc, wit = qap_large.circuit(k, 5)
    prog = compile_r1cs(SparseR1CS.from_rows(k, k + 2, ra, rb, rc), [1])
    v, bad = run(prog, [wit[1]])
    assert bad is None and v == wit
    assert not any(prog.quotient)                    # constant denominators only: no inversion on the device
    assert prog.levels < 64                          # a random DAG is shallow


def test_synthetic_plonk_chain_matches_host_witness():
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    n = 1 << 8
    circ = plonk_synth.chain_circuit(n, seed=3)
    prog = compile_plonk(n, circ["sel"], circ["sigma"], [0] + [n + g for g in range(n)])
    wires = circ["a"] + circ["b"] + circ["c"]
    v, bad = run(prog, [wires[0]] + circ["b"])
    assert bad is None and abc(prog, v) == (circ["a"], circ["b"], circ["c"])
    assert prog.levels == n                          # a chain: one gate per level


def test_compilation_is_deterministic():
    import qap_large
    from interactive_zkp_study_b200.zkp.groth16.qap_device import SparseR1CS
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs
    k = 1 << 7
    ra, rb, rc, _ = qap_large.circuit(k, 11)
    p1, p2 = (compile_r1cs(SparseR1CS.from_rows(k, k + 2, ra, rb, rc), [1]) for _ in range(2))
    for name in ("row_ptr", "col_idx", "out_var", "level_ptr", "in_var"):
        assert list(getattr(p1, name)) == list(getattr(p2, name)), name
    assert p1.values == p2.values and p1.step_src == p2.step_src
    # within a level, steps come in constraint order
    lp = [int(x) for x in p1.level_ptr]
    for a, b in zip(lp, lp[1:]):
        assert p1.step_src[a:b] == sorted(p1.step_src[a:b])


def division_r1cs():
    """w3 = w1 / w2 (code_to_r1cs's division: w3 * w2 = w1), w4 = w3 + 1, and the redundant w4 * 1 = w3 + 1."""
    from interactive_zkp_study_b200.zkp.groth16.qap_device import SparseR1CS
    return SparseR1CS.from_rows(3, 5, [{3: 1}, {3: 1, 0: 1}, {4: 1}], [{2: 1}, {0: 1}, {0: 1}],
                                [{1: 1}, {4: 1}, {3: 1, 0: 1}])


def test_division_is_a_quotient_step_with_a_runtime_check():
    from interactive_zkp_study_b200.zkp.witness import CHECK, compile_r1cs
    prog = compile_r1cs(division_r1cs(), [1, 2])
    assert prog.quotient.count(True) == 1
    assert list(prog.out_var).count(CHECK) == 1 and prog.step_src[list(prog.out_var).index(CHECK)] == 2
    v, bad = run(prog, [10, 4])
    assert bad is None and v[3] == 10 * pow(4, -1, R) % R and v[4] == (v[3] + 1) % R
    _, bad = run(prog, [10, 0])
    assert prog.step_src[bad] == 0 and prog.quotient[bad]


def test_unsatisfied_redundant_constraint_is_reported():
    from interactive_zkp_study_b200.zkp.groth16.qap_device import SparseR1CS
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs
    # w2 = w1 * w1, then the check w2 * 1 = 4: only x = +-2 satisfies it
    prog = compile_r1cs(SparseR1CS.from_rows(2, 3, [{1: 1}, {2: 1}], [{1: 1}, {0: 1}], [{2: 1}, {0: 4}]), [1])
    assert run(prog, [2])[1] is None and run(prog, [R - 2])[1] is None
    _, bad = run(prog, [3])
    assert prog.step_src[bad] == 1 and not prog.quotient[bad]


def test_r1cs_refusals():
    from interactive_zkp_study_b200.zkp.groth16.qap_device import SparseR1CS
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs
    r = division_r1cs()
    with pytest.raises(ValueError, match="inputs"):
        compile_r1cs(r, [0, 1, 2])
    with pytest.raises(ValueError, match="inputs"):
        compile_r1cs(r, [1, 1, 2])
    with pytest.raises(ValueError, match="inputs"):
        compile_r1cs(r, [1, 5])
    with pytest.raises(ValueError, match="wire 2 "):
        compile_r1cs(r, [1])                         # w2 is in no constraint that can solve it
    # x * x = y with y given: quadratic in its only unknown, and nothing else determines x
    sq = SparseR1CS.from_rows(1, 3, [{1: 1}], [{1: 1}], [{2: 1}])
    with pytest.raises(ValueError, match="wire 1 "):
        compile_r1cs(sq, [2])
    assert compile_r1cs(sq, [1]).steps == 1


def test_plonk_refusals():
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    f = load("plonk_x3.json")
    n = f["n"]
    sel = [ints(f["selectors"][k]) for k in ("q_l", "q_r", "q_o", "q_m", "q_c")]
    with pytest.raises(ValueError, match="one copy class"):
        compile_plonk(n, sel, f["sigma"], [0, n])    # a_0 and b_0 both hold x
    with pytest.raises(ValueError, match="one copy class"):
        compile_plonk(n, sel, f["sigma"], [0, 0])
    with pytest.raises(ValueError, match="not determined"):
        compile_plonk(n, sel, f["sigma"], [])        # x is only ever squared
    with pytest.raises(ValueError, match="permutation"):
        compile_plonk(n, sel, [0] * (3 * n), [0])
    with pytest.raises(ValueError, match="positions"):
        compile_plonk(n, sel, f["sigma"], [3 * n])


def test_solve_batch_refuses_short_inputs_before_any_device_call():
    from interactive_zkp_study_b200.zkp.witness import compile_r1cs, solve_batch
    prog = compile_r1cs(division_r1cs(), [1, 2])
    with pytest.raises(ValueError, match="X holds"):
        solve_batch(prog, None, 1)
    with pytest.raises(ValueError, match="count"):
        solve_batch(prog, None, -1)
