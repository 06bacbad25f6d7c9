"""CPU: PLONK public inputs on the host side.  compile_plonk with num_public_inputs, run through the step-program
interpreter of tests/test_cpu_witness.py (the semantics of csrc/witness.cuh); the synthetic circuits of
tools/plonk_synth.py with public-input gates; and the ValueErrors of the verifier, the prover and compile_plonk that
fire before any device call."""
import os
import random
import sys

import pytest

from tests.test_cpu_witness import R, abc, run

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

X3 = {"n": 4, "a": [3, 9, 27, 30], "b": [3, 3, 3, 0], "c": [9, 27, 30, 35],
      "sel": [[0, 0, 1, 1], [0, 0, 1, 0], [R - 1] * 4, [1, 1, 0, 0], [0, 0, 0, 5]],
      "sigma": [6, 8, 9, 10, 0, 4, 5, 7, 1, 2, 3, 11]}


def _gates_hold(c, pub):
    q_l, q_r, q_o, q_m, q_c = c["sel"]
    a, b, cc = c["a"], c["b"], c["c"]
    return all((q_l[g] * a[g] + q_r[g] * b[g] + q_o[g] * cc[g] + q_m[g] * a[g] * b[g] + q_c[g]
                + (pub[g] if g < len(pub) else 0)) % R == 0 for g in range(c["n"]))


@pytest.mark.parametrize("n,ell", [(16, 1), (16, 3), (32, 16), (64, 0)])
def test_public_chain_solved_by_the_program(n, ell):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    c = plonk_synth.public_chain_circuit(n, ell, seed=7)
    assert _gates_hold(c, c["public_inputs"])
    prog = compile_plonk(n, c["sel"], c["sigma"], c["inputs"], num_public_inputs=ell)
    assert prog.n_in == ell + len(c["inputs"]) and len(prog.pub_var) == ell
    assert [int(v) for v in prog.in_var[:ell]] == prog.pub_var
    wires = c["a"] + c["b"] + c["c"]
    v, bad = run(prog, c["public_inputs"] + [wires[p] for p in c["inputs"]])
    assert bad is None
    assert list(abc(prog, v)) == [c["a"], c["b"], c["c"]]
    assert [v[i] for i in prog.pub_var] == c["public_inputs"]
    # gate i < ell reads its public input
    for s in range(prog.steps):
        g = prog.step_src[s]
        used = set().union(*(prog.form(s, f) for f in range(4)))
        assert (g < ell and prog.pub_var[g] in used) or (g >= ell and not used & set(prog.pub_var))


def test_other_public_inputs_give_another_satisfying_witness():
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    n, ell = 32, 4
    c = plonk_synth.public_chain_circuit(n, ell, seed=3)
    prog = compile_plonk(n, c["sel"], c["sigma"], c["inputs"], num_public_inputs=ell)
    rng = random.Random(4)
    pub = [rng.randrange(R) for _ in range(ell)]
    wires = c["a"] + c["b"] + c["c"]
    v, bad = run(prog, pub + [wires[p] for p in c["inputs"]])
    assert bad is None
    a, b, cc = abc(prog, v)
    got = dict(c, a=a, b=b, c=cc)
    assert _gates_hold(got, pub) and not _gates_hold(got, c["public_inputs"])
    assert all((a + b + cc)[p] == (a + b + cc)[c["sigma"][p]] for p in range(3 * n))


def test_x3_output_bound_to_its_public_input():
    """x^3 + x + 5 with a public-input gate on its output: the program checks the output against the input."""
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    c = plonk_synth.prepend_public_gates(X3, [11])
    assert c["n"] == 8 and c["public_inputs"] == [35] and _gates_hold(c, [35])
    prog = compile_plonk(8, c["sel"], c["sigma"], [c["pos"][0]], num_public_inputs=1)
    for x, out in ((3, 35), (4, 73)):
        v, bad = run(prog, [out, x])
        assert bad is None
        a, b, cc = abc(prog, v)
        assert _gates_hold(dict(c, a=a, b=b, c=cc), [out]) and cc[4] == out
    assert run(prog, [35, 4])[1] is not None
    assert run(prog, [73, 3])[1] is not None


def test_compile_plonk_refusals():
    from interactive_zkp_study_b200.zkp.witness import compile_plonk
    c = X3
    for ell in (-1, 5):
        with pytest.raises(ValueError, match="num_public_inputs"):
            compile_plonk(4, c["sel"], c["sigma"], [0], num_public_inputs=ell)


class _PP:
    n, omega, num_public_inputs = 8, 19540430494807482326159819597004422086093766032135589407132600596362845576832, 2


@pytest.mark.parametrize("bad", [[1], [1, 2, 3], [1, R], [1, -1], [1, 1.0], [1, "x"], [True, 1], None])
def test_verifier_refuses_public_inputs_before_any_device_call(bad):
    from interactive_zkp_study_b200.zkp.plonk.prover import Proof
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify, verify_batch
    with pytest.raises(ValueError):
        verify(Proof(), bad, _PP(), None, bind_public_inputs=True)
    with pytest.raises(ValueError):
        verify_batch([(Proof(), [1, 2], _PP()), (Proof(), bad, _PP())], None, bind_public_inputs=True)


def test_public_input_values_reads_ints_and_decimal_strings():
    from interactive_zkp_study_b200.zkp.plonk.device_prover import public_input_values
    assert public_input_values(["35", 0, R - 1], 3, "verify") == [35, 0, R - 1]
    assert public_input_values(None, 0, "verify") == []


def _fake_key(n, ell):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    key = dp.DeviceKey()
    key.n, key.log_n, key.omega, key.ext, key.num_public_inputs = n, n.bit_length() - 1, _PP.omega, 4, ell
    key.N8 = 4 * n
    return key


def test_prover_refusals_before_any_device_call():
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    with pytest.raises(ValueError, match="num_public_inputs"):
        dp.preprocess(8, [None] * 5, [None] * 3, None, 14, num_public_inputs=9)
    with pytest.raises(ValueError, match="sharded"):
        dp.preprocess(8, [None] * 5, [None] * 3, None, 14, comm=object(), srs_range=(0, 7), num_public_inputs=1)
    key = _fake_key(8, 2)
    with pytest.raises(ValueError, match="public inputs"):
        dp.prove(key, None, None, None, public_inputs=[1])
    with pytest.raises(ValueError, match="outside"):
        dp.prove(key, None, None, None, public_inputs=[1, R])
    with pytest.raises(ValueError, match="public_inputs"):
        dp.prove_batch(key, None, None, None, 4)
    with pytest.raises(ValueError, match="no public inputs"):
        dp.prove_batch(_fake_key(8, 0), None, None, None, 0, public_inputs=object())


def test_plan_chunk_counts_the_public_input_block():
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from tests.test_cpu_plonk_batch import _key
    key = _key(1 << 12)
    plain = dp.plan_chunk(key, 10 ** 9, 1 << 62)
    key.num_public_inputs = 64
    with_pi = dp.plan_chunk(key, 10 ** 9, 1 << 62)
    assert with_pi <= plain and 5 * with_pi * key.N8 < 1 << 32
    free = 8 << 30
    assert dp.plan_chunk(key, 10 ** 6, free) < dp.plan_chunk(_key(1 << 12), 10 ** 6, free)
