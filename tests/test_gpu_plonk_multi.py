"""-m gpu: batch PLONK proving over many circuits of one size (zkp/plonk/device_prover.prove_batch_circuits).

(1) golden proofs in a pass shared with other circuits on the fixture's SRS; (2) against a loop of prove under each
proof's own key, chunked and unchunked, with a repeated and an unused circuit; (3) one key equals prove_batch;
(4) each new entry against what it replaces: indexed permutation terms, indexed quotient (ext = 16 / 8 / 4, with and
without PI), the gather; (5) 128 proofs over 8 circuits at 2^12 through verify_batch and the oracle's verifier, a proof
against another circuit's data, a broken witness; (6) public inputs; (7) launches flat in C and in count;
(8) refusals leave the library usable."""
import os
import random
import sys

import pytest

from oracle import bn254, plonk_verifier
from tests.util import g1, ints, load

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))

pytestmark = pytest.mark.gpu
R = bn254.R


def _pt(p):
    return None if p is None else (int(p[0]), int(p[1]))


def _proof_dict(proof):
    return {k: (_pt(v) if k.endswith("_comm") else int(v)) for k, v in vars(proof).items()}


def _stack(native, rows, n):
    return native.scalars_load(native.fr_vec_bytes([x for r in rows for x in r]), len(rows) * n)


def _one(native, h, j, n):
    out = native.scalars_alloc(n)
    native.scalars_copy(out, 0, h, j * n, n)
    return out


def _get(native, h, off, m):
    return native.fr_vec_from_bytes(native.scalars_download(h, off, m))


def _rand(native, rng, m):
    vals = [rng.randrange(R) for _ in range(m)]
    return vals, native.scalars_load(native.fr_vec_bytes(vals), max(m, 1))


def _loop(native, keys, circuits, wit, blinds, pub=None):
    """prove of every proof under its own key (pub: one list of public inputs per proof)."""
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    n = keys[0].n
    return [_proof_dict(dp.prove(keys[c], *(_one(native, h, j, n) for h in wit), blinds=blinds[j],
                                 public_inputs=None if pub is None else pub[j]))
            for j, c in enumerate(circuits)]


def _multi_setup(native, log_n, seeds, circuits, wseed):
    """Keys of random_circuit(n, seed) for each seed on one SRS, and the witness of proof j: a fresh witness of its
    circuit (witness_seed = wseed + j)."""
    import plonk_synth
    n = 1 << log_n
    keys, _, tau = plonk_synth.device_setup_many([plonk_synth.random_circuit(n, s) for s in seeds])
    circs = [plonk_synth.random_circuit(n, seeds[c], witness_seed=wseed + j) for j, c in enumerate(circuits)]
    return keys, [_stack(native, [c[k] for c in circs], n) for k in "abc"], tau


def _pp(key):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    pp = type("PP", (), {})()
    pp.n, pp.omega = key.n, FR(key.omega)
    pp.num_public_inputs = key.num_public_inputs
    for name in dp.CIRCUIT_POLYS:
        setattr(pp, name + "_comm", key.comm[name])
    return pp


def _srs(n, tau):
    from interactive_zkp_study_b200.compat import G2, g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    return SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)


# ------------------------------------------------------------------ proofs
@pytest.mark.parametrize("name", ["plonk_x3.json", "plonk_chain16.json"])
def test_golden_proofs_in_a_pass_with_other_circuits(native, name):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    import plonk_synth
    f = load(name)
    n = f["n"]
    pts = [g1(p) for p in f["g1_powers"]]
    srs = native.g1_table_load(native.g1_vec_bytes(pts), len(pts))
    sel = f["selectors"]
    pad = lambda v: ints(v) + [0] * (n - len(v))
    sel_h = [native.scalars_load(native.fr_vec_bytes(pad(sel[k])), n) for k in ("q_l", "q_r", "q_o", "q_m", "q_c")]
    sig_h = [native.scalars_load(b, n) for b in plonk_synth.sigma_evals_bytes(f["sigma"], n, int(f["omega"]))]
    gold_key = dp.preprocess(n, sel_h, sig_h, srs, len(pts))
    others = [plonk_synth.random_circuit(n, 40 + s) for s in range(3)]
    keys = [plonk_synth.device_key(c, srs, len(pts))[0] for c in others[:2]]
    keys.insert(1, gold_key)
    keys.append(plonk_synth.device_key(others[2], srs, len(pts))[0])       # unused
    circuits = [1, 0, 2, 1, 0, 1]
    gold_w = {k: ints(f[k + "_vals"]) for k in "abc"}
    src = {0: others[0], 2: others[1]}
    wit = [_stack(native, [gold_w[k] if c == 1 else src[c][k] for c in circuits], n) for k in "abc"]
    rng = random.Random(n)
    gold = ints(f["blinds"])
    blinds = [gold if c == 1 and j != 3 else [rng.randrange(R) for _ in range(9)] for j, c in enumerate(circuits)]
    got = [_proof_dict(p) for p in dp.prove_batch_circuits(keys, circuits, *wit, blinds=blinds)]
    want = {k: (g1(v) if k.endswith("_comm") else int(v)) for k, v in f["proof"].items()}
    assert got[0] == want and got[5] == want
    assert got[3] != want
    assert got == _loop(native, keys, circuits, wit, blinds)


@pytest.mark.parametrize("log_n", [3, 8, 12])
def test_equals_loop_of_prove_under_each_key(native, log_n):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    circuits = [2, 0, 2, 1, 2, 0, 2]                     # circuit 2 repeated, circuit 3 unused, 7 proofs over 4 keys
    keys, wit, _ = _multi_setup(native, log_n, [10 * log_n + s for s in range(4)], circuits, 500)
    rng = random.Random(log_n)
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in circuits]
    blinds[1] = [0] * 9
    want = _loop(native, keys, circuits, wit, blinds)
    assert [_proof_dict(p) for p in dp.prove_batch_circuits(keys, circuits, *wit, blinds=blinds)] == want
    assert [_proof_dict(p) for p in dp.prove_batch_circuits(keys, circuits, *wit, blinds=blinds, chunk=3)] == want
    assert len({p["a_comm"] for p in want}) == len(circuits)


def test_one_key_equals_prove_batch(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    keys, wit, _ = _multi_setup(native, 5, [77], [0] * 6, 900)
    rng = random.Random(5)
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(6)]
    want = [_proof_dict(p) for p in dp.prove_batch(keys[0], *wit, 6, blinds=blinds)]
    assert [_proof_dict(p) for p in dp.prove_batch_circuits(keys, [0] * 6, *wit, blinds=blinds)] == want
    assert [_proof_dict(p) for p in dp.prove_batch_circuits(keys, [0] * 6, *wit, blinds=blinds, chunk=4)] == want


# ------------------------------------------------------------------ the new entries against what they replace
def test_indexed_perm_terms_equal_perm_terms_per_circuit(native):
    from interactive_zkp_study_b200.zkp.plonk.field import get_root_of_unity
    import plonk_synth
    n, circuits = 16, [2, 0, 2, 1, 0]
    count = len(circuits)
    w = int(get_root_of_unity(n))
    keys, _, _ = plonk_synth.device_setup_many([plonk_synth.random_circuit(n, s) for s in (1, 2, 3)])
    rng = random.Random(3)
    hs = [_rand(native, rng, count * n + 5)[1] for _ in range(3)]
    betas, gammas = [rng.randrange(R) for _ in circuits], [rng.randrange(R) for _ in circuits]
    num, den = native.scalars_alloc(count * n), native.scalars_alloc(count * n)
    native.plonk_perm_terms_multi_dev(*hs, 5, [k.sigma_evals for k in keys], circuits, n, w, betas, gammas, num, den)
    n1, d1 = native.scalars_alloc(n), native.scalars_alloc(n)
    for j, c in enumerate(circuits):
        native.plonk_perm_terms_many_dev(*hs, 5 + j * n, *keys[c].sigma_evals, n, w, betas[j:j + 1], gammas[j:j + 1],
                                         n1, d1)
        assert _get(native, num, j * n, n) == _get(native, n1, 0, n), j
        assert _get(native, den, j * n, n) == _get(native, d1, 0, n), j


@pytest.mark.parametrize("pi", [False, True])
@pytest.mark.parametrize("n", [1, 4, 16])
def test_indexed_quotient_equals_quotient_per_circuit(native, n, pi):
    """ext = 16 / 8 / 4 on random coset blocks: proof j of the indexed quotient equals the one-circuit quotient of its
    own blocks against its circuit's coset evaluations."""
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    import plonk_synth
    keys, _, _ = plonk_synth.device_setup_many([plonk_synth.random_circuit(n, s) for s in (4, 5, 6)])
    key, N = keys[0], keys[0].N8
    circuits = [1, 1, 0, 2]
    count, nblk = len(circuits), 5 if pi else 4
    rng = random.Random(n * 2 + pi)
    _, ev = _rand(native, rng, nblk * count * N)
    ch = [[rng.randrange(R) for _ in circuits] for _ in range(3)]
    t = native.scalars_alloc(count * N)
    multi = native.plonk_quotient_pi_multi_dev if pi else native.plonk_quotient_multi_dev
    many = native.plonk_quotient_pi_many_dev if pi else native.plonk_quotient_many_dev
    multi(ev, [[k.coset[p] for p in dp.CIRCUIT_POLYS] for k in keys], circuits, n, key.ext, key.x, key.l1f, key.zh8,
          *ch, t)
    ev1, t1 = native.scalars_alloc(nblk * N), native.scalars_alloc(N)
    for j, c in enumerate(circuits):
        for b in range(nblk):
            native.scalars_copy(ev1, b * N, ev, (b * count + j) * N, N)
        many(ev1, [keys[c].coset[p] for p in dp.CIRCUIT_POLYS], n, key.ext, key.x, key.l1f, key.zh8,
             [ch[0][j]], [ch[1][j]], [ch[2][j]], t1)
        assert _get(native, t, j * N, N) == _get(native, t1, 0, N), j


def test_gather_equals_per_proof_copies(native):
    rng = random.Random(8)
    n, K, circuits = 37, 3, [3, 0, 3, 1, 1, 0, 3]
    rows = [[_rand(native, rng, n + 2)[1] for _ in range(K)] for _ in range(5)]     # circuits 2 and 4 unused
    count = len(circuits)
    dst = native.scalars_alloc(K * count * n + 4)
    native.fr_gather_many_dev(rows, circuits, n, dst, 4)
    for k in range(K):
        for j, c in enumerate(circuits):
            one = native.scalars_alloc(n)
            native.scalars_copy(one, 0, rows[c][k], 0, n)
            assert _get(native, dst, 4 + (k * count + j) * n, n) == _get(native, one, 0, n), (k, j)


# ------------------------------------------------------------------ end to end, public inputs, launches, refusals
def test_end_to_end_2_12(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    import plonk_synth
    n, C, count = 1 << 12, 8, 128
    circuits = [(5 * j + j // 16) % C for j in range(count)]
    seeds = [1200 + s for s in range(C)]
    keys, wit, tau = _multi_setup(native, 12, seeds, circuits, 3000)
    proofs = dp.prove_batch_circuits(keys, circuits, *wit)
    pps, srs = [_pp(k) for k in keys], _srs(n, tau)
    items = [(p, [], pps[c]) for p, c in zip(proofs, circuits)]
    assert verify_batch(items, srs, rng=random.Random(1)) is True
    g2p = [bn254.G2, bn254.g2_mul(bn254.G2, tau)]
    for j in (0, 77, count - 1):
        pre = {k: keys[circuits[j]].comm[k] for k in dp.CIRCUIT_POLYS}
        assert plonk_verifier.verify(_proof_dict(proofs[j]), pre, n, keys[0].omega, g2p) is True
    other = (circuits[5] + 1) % C
    assert verify_batch([(proofs[5], [], pps[other])], srs, rng=random.Random(2)) is False
    assert verify_batch(items[:5] + [(proofs[5], [], pps[other])] + items[6:], srs, rng=random.Random(2)) is False
    # one broken witness at proof 40: prove_batch's ValueError naming the proof, chunked or not
    bad = plonk_synth.random_circuit(n, seeds[circuits[40]], witness_seed=3040, break_witness=True)
    native.scalars_upload(wit[2], 40 * n, native.fr_vec_bytes(bad["c"]), n)
    with pytest.raises(ValueError, match="나누어 떨어지지 않.*proof 40 "):
        dp.prove_batch_circuits(keys, circuits, *wit)
    with pytest.raises(ValueError, match="proof 40 "):
        dp.prove_batch_circuits(keys, circuits, *wit, chunk=16)


def test_public_inputs_bind_each_proof(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    import plonk_synth
    n, ell, seeds = 64, 4, (31, 32, 33)
    m = n - ell
    variant = lambda s, w: plonk_synth.prepend_public_gates(plonk_synth.random_circuit(m, s, witness_seed=w),
                                                            [m + i for i in range(ell)], n)
    srs, tau = plonk_synth.device_srs(n + 6)
    keys = [plonk_synth.device_key(variant(s, s), srs, n + 6)[0] for s in seeds]
    assert all(k.num_public_inputs == ell for k in keys)
    circuits = [0, 2, 2, 1, 0, 2]
    circs = [variant(seeds[c], 700 + j) for j, c in enumerate(circuits)]
    wit = [_stack(native, [c[k] for c in circs], n) for k in "abc"]
    pubs = [c["public_inputs"] for c in circs]
    assert len({tuple(p) for p in pubs}) == len(circuits)
    pub_h = _stack(native, pubs, ell)
    rng = random.Random(4)
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in circuits]
    proofs = dp.prove_batch_circuits(keys, circuits, *wit, blinds=blinds, public_inputs=pub_h)
    assert [_proof_dict(p) for p in proofs] == _loop(native, keys, circuits, wit, blinds, pubs)
    pps, vs = [_pp(k) for k in keys], _srs(n, tau)
    items = [(p, x, pps[c]) for p, x, c in zip(proofs, pubs, circuits)]
    assert verify_batch(items, vs, rng=random.Random(3), bind_public_inputs=True) is True
    items[2] = (proofs[2], pubs[3], pps[circuits[2]])                      # one input row replaced
    assert verify_batch(items, vs, rng=random.Random(3), bind_public_inputs=True) is False


def test_launches_do_not_grow_with_circuits_or_count(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    import plonk_synth
    n = 64
    keys, wits, _ = plonk_synth.device_setup_many([plonk_synth.random_circuit(n, 900 + s) for s in range(32)])
    vals = [[_get(native, w[i], 0, n) for i in range(3)] for w in wits]
    # proof j is of circuit j % C and carries that circuit's witness
    stacks = {C: [_stack(native, [vals[j % C][i] for j in range(256)], n) for i in range(3)] for C in (2, 32)}

    def run(C, count):
        before = native.launch_count()
        dp.prove_batch_circuits(keys[:C], [j % C for j in range(count)], *stacks[C])
        return native.launch_count() - before

    got = {}
    for C, count in ((2, 16), (32, 16), (2, 256), (32, 256)) * 2:        # the first round warms caches and workspaces
        got[C, count] = run(C, count)
    assert got[32, 256] <= 1.25 * got[32, 16], got
    assert got[2, 256] <= 1.25 * got[2, 16], got
    assert got[32, 256] <= 1.25 * got[2, 256], got
    assert got[32, 16] <= 1.25 * got[2, 16], got


def test_refusals_leave_the_library_usable(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    import plonk_synth
    n = 8
    keys, _, _ = plonk_synth.device_setup_many([plonk_synth.random_circuit(n, s) for s in (61, 62)])
    key, N = keys[0], keys[0].N8
    h = native.scalars_alloc(4 * n)
    out = native.scalars_alloc(4 * n)
    sig = [k.sigma_evals for k in keys]
    for bad in (2, 7, -1, 1 << 40):
        with pytest.raises(native.ZkpB200Error, match="circuit index out of range"):
            native.plonk_perm_terms_multi_dev(h, h, h, 0, sig, [0, bad, 1, 0], n, key.omega, [1] * 4, [2] * 4, out, out)
        with pytest.raises(native.ZkpB200Error, match="circuit index out of range"):
            native.fr_gather_many_dev([[k.coeffs["q_m"]] for k in keys], [0, bad], n, out)
    short = native.scalars_alloc(n - 1)
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.plonk_perm_terms_multi_dev(h, h, h, 0, [sig[0], [sig[1][0], short, sig[1][2]]], [0, 1, 1, 0], n, key.omega,
                                          [1] * 4, [2] * 4, out, out)
    ev = native.scalars_alloc(4 * 2 * N)
    t = native.scalars_alloc(2 * N)
    circ8 = [[k.coset[p] for p in dp.CIRCUIT_POLYS] for k in keys]
    with pytest.raises(native.ZkpB200Error, match="circuit index out of range"):
        native.plonk_quotient_multi_dev(ev, circ8, [0, 2], n, key.ext, key.x, key.l1f, key.zh8, [1, 2], [1, 2], [1, 2], t)
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.plonk_quotient_pi_multi_dev(ev, circ8, [0, 1], n, key.ext, key.x, key.l1f, key.zh8, [1, 2], [1, 2], [1, 2],
                                           t)                                  # 4 blocks where the PI form reads 5
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.plonk_quotient_multi_dev(ev, [circ8[0], circ8[1][:7] + [short]], [0, 1], n, key.ext, key.x, key.l1f,
                                        key.zh8, [1, 2], [1, 2], [1, 2], t)
    with pytest.raises(native.ZkpB200Error):                                # a G1 table where a vector belongs
        native.fr_gather_many_dev([[key.srs_table], [keys[1].coeffs["q_m"]]], [1, 1], n, out)
    with pytest.raises(native.ZkpB200Error, match="overlaps"):
        native.fr_gather_many_dev([[out], [keys[1].coeffs["q_m"]]], [1, 1], n, out)
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.fr_gather_many_dev([[keys[0].coeffs["q_m"]], [keys[1].coeffs["q_m"]]], [1] * 5, n, out)
    # a correct call afterwards
    native.fr_gather_many_dev([[keys[0].coeffs["q_m"]], [keys[1].coeffs["q_m"]]], [1, 0], n, out)
    assert _get(native, out, 0, n) == _get(native, keys[1].coeffs["q_m"], 0, n)
    assert _get(native, out, n, n) == _get(native, keys[0].coeffs["q_m"], 0, n)
    circuits = [1, 0, 1]
    wk, wit, _ = _multi_setup(native, 3, [61, 62], circuits, 40)
    blinds = [[j] * 9 for j in range(3)]
    got = [_proof_dict(p) for p in dp.prove_batch_circuits(wk, circuits, *wit, blinds=blinds)]
    assert got == _loop(native, wk, circuits, wit, blinds)
