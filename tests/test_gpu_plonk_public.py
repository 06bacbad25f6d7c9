"""-m gpu: PLONK proofs bound to public inputs (device_prover with num_public_inputs, verifier bind_public_inputs).

(1) zkp_plonk_pi_eval_many_dev against utils.public_input_poly_eval, zeta on and off the domain; the scattered and
transformed PI blocks against oracle/ref_path; (2) single proofs accepted by verify(bind_public_inputs=True) and by a
plain-int restatement of the oracle's verifier with the transcript prefix and PI(zeta); rejected after changing or
swapping an input and under the reference protocol; (3) x^3 + x + 5 with its output public: each proof accepted only
with its own output, and the reference protocol's gap; (4) prove_batch against a loop of prove, a violated public
input named, and a 128-proof 2^12 batch from solve_batch through verify_batch; (5) l = 0 proofs equal the golden
ones; (6) launches independent of the batch size."""
import hashlib
import os
import random
import sys

import pytest

from oracle import bn254, ref_path
from oracle.plonk_verifier import K1, K2, _pairing
from tests.util import g1, g2, ints, load

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

pytestmark = pytest.mark.gpu
R = bn254.R
X3 = {"n": 4, "a": [3, 9, 27, 30], "b": [3, 3, 3, 0], "c": [9, 27, 30, 35],
      "sel": [[0, 0, 1, 1], [0, 0, 1, 0], [R - 1] * 4, [1, 1, 0, 0], [0, 0, 0, 5]],
      "sigma": [6, 8, 9, 10, 0, 4, 5, 7, 1, 2, 3, 11]}


def _pt(p):
    return None if p is None else (int(p[0]), int(p[1]))


def _proof_dict(proof):
    return {k: (_pt(v) if k.endswith("_comm") else int(v)) for k, v in vars(proof).items()}


def _load(native, xs):
    return native.scalars_load(native.fr_vec_bytes(xs), len(xs))


def _vals(native, h, off, m):
    return native.fr_vec_from_bytes(native.scalars_download(h, off, m))


class _Setup:
    """A device key for a circuit dict of tools/plonk_synth, with what the verifiers take."""

    def __init__(self, native, circ):
        import plonk_synth
        from interactive_zkp_study_b200.compat import G2, g2_from_ints
        from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
        from interactive_zkp_study_b200.zkp.plonk.field import FR
        from interactive_zkp_study_b200.zkp.plonk.srs import SRS
        self.circ = circ
        self.key, self.wit, tau = plonk_synth.device_setup(circ)
        n = self.n = circ["n"]
        self.pp = type("PP", (), {})()
        self.pp.n, self.pp.omega = n, FR(self.key.omega)
        self.pp.num_public_inputs = self.key.num_public_inputs
        for name in dp.CIRCUIT_POLYS:
            setattr(self.pp, name + "_comm", self.key.comm[name])
        self.g2p = [bn254.G2, bn254.g2_mul(bn254.G2, tau)]
        self.srs = SRS([], [G2, g2_from_ints(self.g2p[1])], n + 5)

    def prove(self, wit=None, pubs=None, blinds=None):
        from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
        return dp.prove(self.key, *(wit or self.wit), blinds=blinds,
                        public_inputs=self.circ.get("public_inputs", []) if pubs is None else pubs)

    def verify(self, proof, pubs, bind=True):
        from interactive_zkp_study_b200.zkp.pairing import pairing
        from interactive_zkp_study_b200.zkp.plonk.verifier import verify
        return verify(proof, pubs, self.pp, self.srs, pairing=pairing, bind_public_inputs=bind)

    def oracle_verify(self, proof, pubs):
        pre = {name: _pt(self.key.comm[name]) for name in ("q_l", "q_r", "q_o", "q_m", "q_c", "s_sigma1", "s_sigma2",
                                                            "s_sigma3")}
        return _oracle_verify_pi(_proof_dict(proof), pre, self.n, self.key.omega, self.g2p, pubs)


def _oracle_verify_pi(proof, pre_comm, n, omega, g2_powers, pubs):
    """oracle/plonk_verifier.verify over plain ints with the public-input protocol: append_scalar(b"public_input", x_i)
    before the first challenge and r0 + PI(zeta), PI(zeta) = sum_i x_i w^i (zeta^n - 1) / (n (zeta - w^i))."""
    add, mul, neg, inv = bn254.g1_add, bn254.g1_mul, bn254.g1_neg, lambda a: bn254.inv(a, R)
    mulr = lambda p, k: mul(p, k % R)
    state = bytearray(b"plonk")

    def chal(label):
        state.extend(label)
        h = hashlib.sha256(bytes(state)).digest()
        state.extend(h)
        return int.from_bytes(h, "big") % R

    def point(label, p):
        state.extend(label + (bytes(64) if p is None else p[0].to_bytes(32, "big") + p[1].to_bytes(32, "big")))

    for x in pubs:
        state.extend(b"public_input" + (x % R).to_bytes(32, "big"))
    for k in ("a_comm", "b_comm", "c_comm"):
        point(k.encode(), proof[k])
    beta, gamma = chal(b"beta"), chal(b"gamma")
    point(b"z_comm", proof["z_comm"])
    alpha = chal(b"alpha")
    for k in ("t_lo_comm", "t_mid_comm", "t_hi_comm"):
        point(k.encode(), proof[k])
    zeta = chal(b"zeta")
    for k in ("a_eval", "b_eval", "c_eval", "s_sigma1_eval", "s_sigma2_eval", "z_omega_eval"):
        state.extend(k.encode() + (proof[k] % R).to_bytes(32, "big"))
    v, u = chal(b"v"), chal(b"u")
    a_e, b_e, c_e = proof["a_eval"], proof["b_eval"], proof["c_eval"]
    s1_e, s2_e, zw_e = proof["s_sigma1_eval"], proof["s_sigma2_eval"], proof["z_omega_eval"]
    zh = (pow(zeta, n, R) - 1) % R
    den = (zeta - 1) % R
    l1 = 1 if den == 0 else inv(n) * zh % R * inv(den) % R
    pi = 0
    for i, x in enumerate(pubs):
        wi = pow(omega, i, R)
        pi = (pi + x * (1 if zeta == wi else wi * zh % R * inv(n * (zeta - wi) % R))) % R
    D = mulr(pre_comm["q_m"], a_e * b_e)
    D = add(D, mulr(pre_comm["q_l"], a_e))
    D = add(D, mulr(pre_comm["q_r"], b_e))
    D = add(D, mulr(pre_comm["q_o"], c_e))
    D = add(D, pre_comm["q_c"])
    perm_z = alpha * (a_e + beta * zeta + gamma) % R * (b_e + beta * K1 * zeta + gamma) % R * (c_e + beta * K2 * zeta + gamma) % R
    D = add(D, mulr(proof["z_comm"], perm_z))
    ab = (a_e + beta * s1_e + gamma) * (b_e + beta * s2_e + gamma) % R
    D = add(D, neg(mulr(pre_comm["s_sigma3"], alpha * ab % R * beta % R * zw_e)))
    D = add(D, mulr(proof["z_comm"], alpha * alpha % R * l1))
    r0 = (pi - alpha * ab % R * zw_e % R * (c_e + gamma) - alpha * alpha % R * l1) % R
    zn = pow(zeta, n, R)
    F = add(proof["t_lo_comm"], add(mulr(proof["t_mid_comm"], zn), mulr(proof["t_hi_comm"], zn * zn)))
    F = add(F, mulr(D, v))
    F = add(F, mulr(bn254.G1, v * r0))
    vp = v * v % R
    for key, src in (("a_comm", proof), ("b_comm", proof), ("c_comm", proof), ("s_sigma1", pre_comm), ("s_sigma2", pre_comm)):
        F = add(F, mulr(src[key], vp))
        vp = vp * v % R
    r_eval = proof["r_eval"]
    e = (r_eval * inv(zh) + v * r_eval) % R
    vp = v * v % R
    for ev in (a_e, b_e, c_e, s1_e, s2_e):
        e = (e + vp * ev) % R
        vp = vp * v % R
    e = (e + u * zw_e) % R
    A = add(proof["W_zeta_comm"], mulr(proof["W_zeta_omega_comm"], u))
    B = mulr(proof["W_zeta_comm"], zeta)
    B = add(B, mulr(proof["W_zeta_omega_comm"], u * zeta % R * omega))
    B = add(B, F)
    B = add(B, mulr(proof["z_comm"], u))
    B = add(B, neg(mulr(bn254.G1, e)))
    bn = _pairing()
    to1 = lambda p: None if p is None else (bn.FQ(p[0]), bn.FQ(p[1]))
    to2 = lambda p: (bn.FQ2([p[0][0], p[0][1]]), bn.FQ2([p[1][0], p[1][1]]))
    return bn.pairing(to2(g2_powers[1]), to1(A)) == bn.pairing(to2(g2_powers[0]), to1(B))


# ------------------------------------------------------------------ (1) the PI entries
@pytest.mark.parametrize("count", [1, 5, 256])
@pytest.mark.parametrize("ell", [1, 3, 64, "n"])
def test_pi_eval_equals_public_input_poly_eval(native, ell, count):
    from interactive_zkp_study_b200.zkp.plonk.field import FR, get_root_of_unity
    from interactive_zkp_study_b200.zkp.plonk.utils import public_input_poly_eval
    n = 128
    ell = n if ell == "n" else ell
    w = int(get_root_of_unity(n))
    rng = random.Random(ell * 1000 + count)
    stride = ell + 3                                      # inputs read in place from wider rows
    rows = [[rng.randrange(R) for _ in range(stride)] for _ in range(count)]
    zetas = [rng.randrange(R) for _ in range(count)]
    zetas[0] = pow(w, ell - 1, R)                         # on the domain, at a public-input row
    if count > 1:
        zetas[1] = pow(w, ell, R) if ell < n else 1       # on the domain, above the public inputs (or at row 0)
    if count > 2:
        zetas[2] = 0
    h = _load(native, [x for r in rows for x in r])
    got = native.plonk_pi_eval_many_dev(h, 0, stride, ell, n, w, zetas)
    want = [int(public_input_poly_eval(r[:ell], n, FR(w), FR(z))) for r, z in zip(rows, zetas)]
    assert got == want
    assert got[0] == rows[0][ell - 1]
    if count > 1 and ell < n:
        assert got[1] == 0
    assert native.plonk_pi_eval_many_dev(h, 0, stride, 0, n, w, zetas) == [0] * count


@pytest.mark.parametrize("n,ell,count", [(8, 3, 4), (16, 16, 3), (64, 5, 2)])
def test_pi_blocks_equal_ref_path_transforms(native, n, ell, count):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import get_root_of_unity
    w = int(get_root_of_unity(n))
    ext = 4 if n >= 8 else 8
    N = ext * n
    w8 = int(get_root_of_unity(N))
    rng = random.Random(n + ell)
    pubs = [[rng.randrange(R) for _ in range(ell)] for _ in range(count)]
    pub = _load(native, [x for p in pubs for x in p])
    ev = native.scalars_alloc(4 * count * n)
    native.plonk_pi_scatter_many_dev(pub, 0, ell, ell, n, count, ev, 3 * count * n)
    sparse = [p + [0] * (n - ell) for p in pubs]
    assert _vals(native, ev, 3 * count * n, count * n) == [x for s in sparse for x in s]
    native.ntt_many_dev(ev, 0, n.bit_length() - 1, 4 * count, w, inverse=True)
    coeffs = [ref_path.ifft(s, w) for s in sparse]
    assert _vals(native, ev, 3 * count * n, count * n) == [x for c in coeffs for x in c]
    wires, z = native.scalars_alloc(3 * count * (n + 2)), native.scalars_alloc(count * (n + 3))
    out = native.scalars_alloc(5 * count * N)
    native.plonk_coset_inputs_pi_many_dev(wires, z, ev, 3 * count * n, n, count, (N).bit_length() - 1, out)
    native.ntt_many_dev(out, 0, N.bit_length() - 1, 5 * count, w8, coset_shift=dp.COSET_SHIFT)
    native.scalars_convert(out, 4 * count * N, count * N, False)
    want = [x for c in coeffs for x in ref_path.coset_fft(c + [0] * (N - n), w8, dp.COSET_SHIFT)]
    assert _vals(native, out, 4 * count * N, count * N) == want


# ------------------------------------------------------------------ (2) single proofs
@pytest.fixture(scope="module")
def chain(native):
    import plonk_synth
    return _Setup(native, plonk_synth.public_chain_circuit(64, 5, seed=21))


def test_single_proof_accepted_and_bound(native, chain):
    pubs = chain.circ["public_inputs"]
    proof = chain.prove(blinds=list(range(1, 10)))
    assert chain.verify(proof, pubs) is True
    assert chain.oracle_verify(proof, pubs) is True
    changed = list(pubs)
    changed[3] = (changed[3] + 1) % R
    assert chain.verify(proof, changed) is False
    assert chain.oracle_verify(proof, changed) is False
    swapped = list(pubs)
    swapped[0], swapped[4] = swapped[4], swapped[0]
    assert swapped != pubs and chain.verify(proof, swapped) is False
    assert chain.verify(proof, pubs, bind=False) is False
    # the same proof key refuses a proof of other public inputs than the witness carries
    with pytest.raises(ValueError):
        chain.prove(pubs=changed)


def test_verify_batch_binds_each_proof(native, chain):
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    pubs = chain.circ["public_inputs"]
    proofs = [chain.prove() for _ in range(3)]
    items = [(p, pubs, chain.pp) for p in proofs]
    assert verify_batch(items, chain.srs, rng=random.Random(3), bind_public_inputs=True) is True
    assert verify_batch(items, chain.srs, rng=random.Random(3)) is False
    bad = list(pubs)
    bad[0] = (bad[0] + 1) % R
    assert verify_batch(items[:2] + [(proofs[2], bad, chain.pp)], chain.srs, rng=random.Random(3),
                        bind_public_inputs=True) is False


# ------------------------------------------------------------------ (3) x^3 + x + 5 with its output public
def test_x3_output_is_the_statement(native):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.witness import compile_plonk, solve_batch
    # the reference protocol: a proof of x = 4 (output 73) passes against "35"
    plain = _Setup(native, X3)
    x4 = [[4, 16, 64, 68], [4, 4, 4, 0], [16, 64, 68, 73]]
    proof4 = plain.prove(wit=[_load(native, v) for v in x4], pubs=[])
    plain.pp.num_public_inputs = 1
    assert plain.verify(proof4, ["35"], bind=False) is True
    # with a public-input gate on the output, each proof is accepted with its own output only
    circ = plonk_synth.prepend_public_gates(X3, [11])
    pi = _Setup(native, circ)
    prog = compile_plonk(circ["n"], circ["sel"], circ["sigma"], [circ["pos"][0]], num_public_inputs=1)
    a, b, c, pub = solve_batch(prog, _load(native, [35, 3, 73, 4]), 2)
    assert _vals(native, pub, 0, 2) == [35, 73]
    proofs = []
    for j, out in enumerate((35, 73)):
        wit = [native.scalars_alloc(8) for _ in range(3)]
        for dst, src in zip(wit, (a, b, c)):
            native.scalars_copy(dst, 0, src, 8 * j, 8)
        proofs.append(pi.prove(wit=wit, pubs=[out]))
    assert pi.verify(proofs[0], ["35"]) is True and pi.verify(proofs[0], ["73"]) is False
    assert pi.verify(proofs[1], ["73"]) is True and pi.verify(proofs[1], ["35"]) is False
    assert pi.oracle_verify(proofs[1], [73]) is True
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    batch = dp.prove_batch(pi.key, a, b, c, 2, public_inputs=pub)
    assert pi.verify(batch[0], [35]) is True and pi.verify(batch[1], [73]) is True


# ------------------------------------------------------------------ (4) batches
@pytest.mark.parametrize("log_n,ell,count", [(3, 1, 5), (6, 5, 7), (8, 128, 4)])
def test_prove_batch_equals_loop_of_prove(native, log_n, ell, count):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.witness import compile_plonk, solve_batch
    n = 1 << log_n
    s = _Setup(native, plonk_synth.public_chain_circuit(n, ell, seed=log_n))
    circ = s.circ
    prog = compile_plonk(n, circ["sel"], circ["sigma"], circ["inputs"], num_public_inputs=ell)
    rng = random.Random(log_n)
    wires = circ["a"] + circ["b"] + circ["c"]
    X = [x for _ in range(count) for x in [rng.randrange(R) for _ in range(ell)] + [wires[p] for p in circ["inputs"]]]
    a, b, c, pub = solve_batch(prog, _load(native, X), count)
    pubs = _vals(native, pub, 0, count * ell)
    assert len({tuple(pubs[j * ell:(j + 1) * ell]) for j in range(count)}) == count
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(count)]
    want = []
    for j in range(count):
        wit = [native.scalars_alloc(n) for _ in range(3)]
        for dst, src in zip(wit, (a, b, c)):
            native.scalars_copy(dst, 0, src, j * n, n)
        want.append(_proof_dict(s.prove(wit=wit, pubs=pubs[j * ell:(j + 1) * ell], blinds=blinds[j])))
    assert [_proof_dict(p) for p in dp.prove_batch(s.key, a, b, c, count, blinds=blinds, public_inputs=pub)] == want
    assert [_proof_dict(p) for p in dp.prove_batch(s.key, a, b, c, count, blinds=blinds, chunk=2,
                                                   public_inputs=pub)] == want
    # a public input that its gate does not satisfy
    bad = _load(native, pubs[:2 * ell] + [(pubs[2 * ell] + 1) % R] + pubs[2 * ell + 1:])
    with pytest.raises(ValueError, match="proof 2 "):
        dp.prove_batch(s.key, a, b, c, count, public_inputs=bad)
    with pytest.raises(ValueError, match="outside"):
        dp.prove_batch(s.key, a, b, c, count, public_inputs=_load(native, [R] + pubs[1:]))


def test_batch_2_12_from_solve_batch_through_verify_batch(native):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    from interactive_zkp_study_b200.zkp.witness import compile_plonk, solve_batch
    n, ell, count = 1 << 12, 16, 128
    s = _Setup(native, plonk_synth.public_chain_circuit(n, ell, seed=12))
    circ = s.circ
    prog = compile_plonk(n, circ["sel"], circ["sigma"], circ["inputs"], num_public_inputs=ell)
    rows = []
    for j in range(count):
        c = plonk_synth.public_chain_circuit(n, ell, seed=3000 + j)
        w = c["a"] + c["b"] + c["c"]
        rows.append(c["public_inputs"] + [w[p] for p in c["inputs"]])
    a, b, c, pub = solve_batch(prog, _load(native, [x for r in rows for x in r]), count)
    proofs = dp.prove_batch(s.key, a, b, c, count, public_inputs=pub)
    pubs = [r[:ell] for r in rows]
    assert len({tuple(p) for p in pubs}) == count
    items = [(p, x, s.pp) for p, x in zip(proofs, pubs)]
    assert verify_batch(items, s.srs, rng=random.Random(1), bind_public_inputs=True) is True
    items[77] = (proofs[77], pubs[78], s.pp)
    assert verify_batch(items, s.srs, rng=random.Random(1), bind_public_inputs=True) is False


# ------------------------------------------------------------------ (5) l = 0
@pytest.mark.parametrize("name", ["plonk_n1.json", "plonk_chain16.json"])
def test_no_public_inputs_keeps_the_golden_proofs(native, name):
    import plonk_synth
    from interactive_zkp_study_b200.compat import g2_from_ints
    from interactive_zkp_study_b200.zkp.pairing import pairing
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify
    f = load(name)
    n = f["n"]
    pts = [g1(p) for p in f["g1_powers"]]
    srs_t = native.g1_table_load(native.g1_vec_bytes(pts), len(pts))
    pad = lambda v: ints(v) + [0] * (n - len(v))
    sel_h = [_load(native, pad(f["selectors"][k])) for k in ("q_l", "q_r", "q_o", "q_m", "q_c")]
    sig_h = [native.scalars_load(bb, n) for bb in plonk_synth.sigma_evals_bytes(f["sigma"], n, int(f["omega"]))]
    key = dp.preprocess(n, sel_h, sig_h, srs_t, len(pts), num_public_inputs=0)
    wit = [_load(native, ints(f[k + "_vals"])) for k in "abc"]
    want = {k: (g1(v) if k.endswith("_comm") else int(v)) for k, v in f["proof"].items()}
    proof = dp.prove(key, *wit, blinds=ints(f["blinds"]), public_inputs=[])
    assert _proof_dict(proof) == want
    assert _proof_dict(dp.prove_batch(key, *wit, 1, blinds=[ints(f["blinds"])])[0]) == want
    pp = type("PP", (), {})()
    pp.n, pp.omega, pp.num_public_inputs = n, FR(key.omega), 0
    for nm in dp.CIRCUIT_POLYS:
        setattr(pp, nm + "_comm", key.comm[nm])
    srs = SRS([], [g2_from_ints(g2(p)) for p in f["g2_powers"][:2]], n + 5)
    assert verify(proof, [], pp, srs, pairing=pairing, bind_public_inputs=True) is True


# ------------------------------------------------------------------ (6) launches
def test_launches_do_not_grow_with_count(native):
    import plonk_synth
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    n, ell = 64, 8
    runs = {}
    for kind, circ in (("pi", plonk_synth.public_chain_circuit(n, ell, seed=5)), ("plain", plonk_synth.chain_circuit(n, seed=5))):
        key, wit, _ = plonk_synth.device_setup(circ)
        stack = lambda h: _load(native, _vals(native, h, 0, n) * 256)
        wit = [stack(h) for h in wit]
        pub = _load(native, circ["public_inputs"] * 256) if kind == "pi" else None
        for count in (16, 256, 16, 256):                # the first pair warms caches and workspaces
            before = native.launch_count()
            dp.prove_batch(key, *wit, count, public_inputs=pub)
            runs[kind, count] = native.launch_count() - before
    assert runs["pi", 256] <= 1.25 * runs["pi", 16], runs
    # what public inputs add is the same at any count
    assert runs["pi", 256] - runs["plain", 256] == runs["pi", 16] - runs["plain", 16], runs


def test_refusals_leave_the_library_usable(native):
    h = native.scalars_alloc(64)
    with pytest.raises(native.ZkpB200Error, match="more public inputs"):
        native.plonk_pi_eval_many_dev(h, 0, 17, 17, 16, 1, [1])
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.plonk_pi_eval_many_dev(h, 0, 20, 8, 16, 1, [1] * 4)
    with pytest.raises(native.ZkpB200Error, match="stride"):
        native.plonk_pi_scatter_many_dev(h, 0, 2, 3, 8, 4, native.scalars_alloc(64))
    with pytest.raises(native.ZkpB200Error, match="overlaps"):
        native.plonk_pi_scatter_many_dev(h, 0, 3, 3, 8, 4, h, 8)
    with pytest.raises(native.ZkpB200Error, match="2\\^32"):
        native.plonk_coset_inputs_pi_many_dev(h, h, h, 0, 8, 1 << 25, 5, h)
    from interactive_zkp_study_b200.zkp.plonk.field import FR, get_root_of_unity
    from interactive_zkp_study_b200.zkp.plonk.utils import public_input_poly_eval
    w = int(get_root_of_unity(16))
    got = native.plonk_pi_eval_many_dev(_load(native, [7, 9]), 0, 2, 2, 16, w, [5])
    assert got == [int(public_input_poly_eval([7, 9], 16, FR(w), FR(5)))]
