"""-m gpu: batch PLONK proving -- many proofs of one circuit per pass (zkp/plonk/device_prover.prove_batch).

(1) the golden proofs at both ends of a batch; (2) prove_batch against a loop of prove, chunked and unchunked;
(3) every batched piece against its single-vector entry (segmented scans, segmented division by (x - zeta) with
zeta = 0 and 1, batched lincomb and Horner, the batched quotient at ext = 16 / 8 / 4, batched transforms) and a
zero-padded commitment; (4) a 128-proof 2^12-gate batch end to end through verify_batch and the oracle's verifier,
with a broken witness and a tampered evaluation; (5) launches independent of the batch size; (6) refusals."""
import copy
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


def _golden_key(native, name):
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
    return f, dp.preprocess(n, sel_h, sig_h, srs, len(pts))


def _stack(native, rows, n):
    return native.scalars_load(native.fr_vec_bytes([x for r in rows for x in r]), len(rows) * n)


def _one(native, h, j, n):
    out = native.scalars_alloc(n)
    native.scalars_copy(out, 0, h, j * n, n)
    return out


def _loop(native, key, wit, count, blinds):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    n = key.n
    return [_proof_dict(dp.prove(key, *(_one(native, h, j, n) for h in wit), blinds=blinds[j])) for j in range(count)]


@pytest.mark.parametrize("name", ["plonk_n1.json", "plonk_x3.json", "plonk_chain16.json"])
def test_golden_proofs_inside_a_batch(native, name):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    f, key = _golden_key(native, name)
    n, count = f["n"], 5
    rng = random.Random(n)
    gold = ints(f["blinds"])
    blinds = [gold] + [[rng.randrange(R) for _ in range(9)] for _ in range(count - 2)] + [gold]
    wit = [_stack(native, [ints(f[k + "_vals"])] * count, n) for k in "abc"]
    got = [_proof_dict(p) for p in dp.prove_batch(key, *wit, count, blinds=blinds)]
    want = {k: (g1(v) if k.endswith("_comm") else int(v)) for k, v in f["proof"].items()}
    assert got[0] == want and got[-1] == want
    assert got[1:-1] == _loop(native, key, wit, count, blinds)[1:-1]
    assert got[1] != got[0]


def _synthetic(native, log_n, count, seed):
    """The chain circuit of tools/plonk_synth at n = 2^log_n and count witnesses of it (one seed each)."""
    import plonk_synth
    n = 1 << log_n
    key, _, tau = plonk_synth.device_setup(plonk_synth.chain_circuit(n, seed=seed))
    circs = [plonk_synth.chain_circuit(n, seed=seed + 1 + j) for j in range(count)]
    wit = [_stack(native, [c[k] for c in circs], n) for k in "abc"]
    return key, wit, tau


@pytest.mark.parametrize("log_n,count", [(3, 7), (8, 7), (12, 5)])
def test_prove_batch_equals_loop_of_prove(native, log_n, count):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    key, wit, _ = _synthetic(native, log_n, count, 100 + log_n)
    rng = random.Random(log_n)
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(count)]
    blinds[1] = [0] * 9
    want = _loop(native, key, wit, count, blinds)
    assert [_proof_dict(p) for p in dp.prove_batch(key, *wit, count, blinds=blinds)] == want
    assert [_proof_dict(p) for p in dp.prove_batch(key, *wit, count, blinds=blinds, chunk=3)] == want
    assert len({p["a_comm"] for p in want}) == count           # different witnesses, different proofs


# ------------------------------------------------------------------ the pieces against the single-vector entries
def _rand(native, rng, m):
    vals = [rng.randrange(R) for _ in range(m)]
    return vals, native.scalars_load(native.fr_vec_bytes(vals), max(m, 1))


def _get(native, h, off, m):
    return native.fr_vec_from_bytes(native.scalars_download(h, off, m))


@pytest.mark.parametrize("op", [0, 1])
@pytest.mark.parametrize("seg,count", [(1, 5), (3, 700), (5, 1), (1000, 3), (1024, 3), (3000, 2), (4, 2000)])
def test_segmented_scan_equals_scan_per_segment(native, op, seg, count):
    rng = random.Random(seg * 31 + count + op)
    vals, src = _rand(native, rng, seg * count)
    if seg * count > 10:
        vals[7] = 0
        native.scalars_upload(src, 7, native.fe_bytes(0), 1)
    dst = native.scalars_alloc(seg * count)
    native.scan_many_dev(op, dst, 0, src, 0, seg, count)
    got = _get(native, dst, 0, seg * count)
    one = native.scalars_alloc(seg)
    for j in range(count):
        native.scan_dev(op, one, 0, src, j * seg, seg)
        assert got[j * seg:(j + 1) * seg] == _get(native, one, 0, seg), j
    if seg * count <= 4000:                                # and against the definition
        for j in range(0, count, max(1, count // 7)):
            acc = 1 if op == 0 else 0
            for i in range(seg):
                assert got[j * seg + i] == acc
                acc = acc * vals[j * seg + i] % R if op == 0 else (acc + vals[j * seg + i]) % R


@pytest.mark.parametrize("length,count", [(2, 3), (7, 5), (1030, 4), (4102, 3)])
def test_segmented_div_linear_equals_single(native, length, count):
    rng = random.Random(length)
    stride, dstride = length + 3, length + 1
    _, src = _rand(native, rng, stride * count)
    zetas = [0, 1] + [rng.randrange(R) for _ in range(count - 2)]
    dst = native.scalars_alloc(dstride * count)
    native.div_linear_many_dev(src, 0, stride, length, zetas, dst, 0, dstride)
    one = native.scalars_alloc(length - 1)
    for j, z in enumerate(zetas):
        native.div_linear_dev(src, j * stride, length, z, one, 0)
        assert _get(native, dst, j * dstride, length - 1) == _get(native, one, 0, length - 1), (j, z)
        assert _get(native, dst, j * dstride + length - 1, dstride - length + 1) == [0] * (dstride - length + 1)
    coeffs = _get(native, src, 0, length)                  # zeta = 0: the shift
    assert _get(native, dst, 0, length - 1) == coeffs[1:]


@pytest.mark.parametrize("n,count", [(1, 3), (16, 5), (1000, 4)])
def test_batched_lincomb_equals_lincomb(native, n, count):
    rng = random.Random(n + count)
    shared = [_rand(native, rng, n)[1] for _ in range(2)]
    _, per = _rand(native, rng, (n + 3) * count)
    sources = [(shared[0], 0, 0, n), (per, 0, n + 3, n + 3), (shared[1], 0, 0, max(n - 1, 1))]
    rows = [[rng.randrange(R) for _ in range(4)] for _ in range(count)]
    rows[0][1] = 0
    dst = native.scalars_alloc((n + 5) * count)
    native.lincomb_many_dev(dst, 0, n + 5, n + 3, count, sources, rows)
    one = native.scalars_alloc(n + 3)
    for j in range(count):
        items = [(rows[j][k], h, off + j * st, ln) for k, (h, off, st, ln) in enumerate(sources)]
        native.lincomb_dev(one, 0, n + 3, items)
        native.scalars_add_const(one, 0, 1, rows[j][3])
        assert _get(native, dst, j * (n + 5), n + 3) == _get(native, one, 0, n + 3), j


@pytest.mark.parametrize("n,count", [(1, 4), (16, 9), (4099, 3)])
def test_batched_horner_equals_single(native, n, count):
    rng = random.Random(n * 3 + count)
    _, shared = _rand(native, rng, n)
    _, per = _rand(native, rng, (n + 2) * count)
    pts = [[0, 1] + [rng.randrange(R) for _ in range(count - 2)], [rng.randrange(R) for _ in range(count)]]
    groups = [(per, 0, n + 2, n + 2, 0), (shared, 0, 0, n, 1), (per, 1, n + 2, n, 1)]
    got = native.fr_poly_eval_many_dev(groups, count, pts)
    for g, (h, off, st, ln, sel) in enumerate(groups):
        for j in range(count):
            assert got[g][j] == native.fr_poly_eval_dev(h, off + j * st, ln, pts[sel][j]), (g, j)


@pytest.mark.parametrize("n", [1, 4, 16])
def test_quotient_many_equals_single(native, n):
    """ext = 16 / 8 / 4: the batched coset inputs, transforms, quotient, divisibility check and split against the
    single path on random (so not divisible) wire and z coefficients."""
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    import plonk_synth
    key, _, _ = plonk_synth.device_setup(plonk_synth.chain_circuit(n, seed=5))
    N, count = key.N8, 3
    rng = random.Random(n)
    _, wires = _rand(native, rng, 3 * count * (n + 2))
    _, z = _rand(native, rng, count * (n + 3))
    ch = [[rng.randrange(R) for _ in range(count)] for _ in range(3)]
    ev = native.scalars_alloc(4 * count * N)
    native.plonk_coset_inputs_many_dev(wires, z, n, count, key.log_n + key.log_ext, ev)
    native.ntt_many_dev(ev, 0, key.log_n + key.log_ext, 4 * count, key.omega8, coset_shift=dp.COSET_SHIFT)
    t = native.scalars_alloc(count * N)
    native.plonk_quotient_many_dev(ev, [key.coset[k] for k in dp.CIRCUIT_POLYS], n, key.ext, key.x, key.l1f, key.zh8,
                                   *ch, t)
    got_t = _get(native, t, 0, count * N)
    native.ntt_many_dev(t, 0, key.log_n + key.log_ext, count, key.omega8, inverse=True, coset_shift=dp.COSET_SHIFT)
    assert native.plonk_divisible_many_dev(t, n, key.ext, count) == 0
    ts = native.scalars_alloc(3 * count * (n + 6))
    native.plonk_split_t_many_dev(t, n, key.ext, count, ts)
    for j in range(count):
        single = []
        for i, (h, off, ln) in enumerate([(wires, (w * count + j) * (n + 2), n + 2) for w in range(3)]
                                         + [(z, j * (n + 3), n + 3)]):
            e = native.scalars_alloc(N)
            native.scalars_copy(e, 0, h, off, ln)
            native.scalars_convert(e, 0, ln, True)
            native.ntt_dev(e, 0, key.log_n + key.log_ext, key.omega8, coset_shift=dp.COSET_SHIFT)
            assert _get(native, ev, (i * count + j) * N, N) == _get(native, e, 0, N), (j, i)
            single.append(e)
        t1 = native.scalars_alloc(N)
        native.plonk_quotient_dev(single + [key.coset[k] for k in dp.CIRCUIT_POLYS], n, key.ext, key.x, key.l1f, key.zh8,
                                  ch[0][j], ch[1][j], ch[2][j], t1)
        assert got_t[j * N:(j + 1) * N] == _get(native, t1, 0, N), j
        native.ntt_dev(t1, 0, key.log_n + key.log_ext, key.omega8, inverse=True, coset_shift=dp.COSET_SHIFT)
        native.scalars_convert(t1, 0, N, False)
        tc = _get(native, t1, 0, N)
        for part, ln in ((0, n), (1, n), (2, n + 6)):
            row = _get(native, ts, (part * count + j) * (n + 6), n + 6)
            assert row == tc[part * n:part * n + ln] + [0] * (n + 6 - ln), (j, part)
    # a divisible block: zero the top of proof 0 and 2, proof 1 stays the first failing one
    for j in (0, 2):
        native.scalars_upload(t, j * N + 3 * n + 6, bytes(32 * (N - 3 * n - 6)), N - 3 * n - 6)
    assert native.plonk_divisible_many_dev(t, n, key.ext, count) == 1
    native.scalars_upload(t, N + 3 * n + 6, bytes(32 * (N - 3 * n - 6)), N - 3 * n - 6)
    assert native.plonk_divisible_many_dev(t, n, key.ext, count) is None


def test_zero_padding_keeps_the_commitment(native):
    rng = random.Random(9)
    m, pad, count = 40, 6, 5
    t = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes([rng.randrange(1, R) for _ in range(m + pad)]),
                                 m + pad)
    vals = [[rng.randrange(R) for _ in range(m)] for _ in range(count)]
    padded = native.scalars_load(native.fr_vec_bytes([x for v in vals for x in v + [0] * pad]), count * (m + pad))
    tight = native.scalars_load(native.fr_vec_bytes([x for v in vals for x in v]), count * m)
    for table in (t,):
        assert native.msm_dev_many(table, 0, m + pad, count, padded) == native.msm_dev_many(table, 0, m, count, tight)
    native.table_precompute(t)
    assert native.msm_dev_many(t, 0, m + pad, count, padded) == [native.g1_msm_dev(t, 0, tight, j * m, m)
                                                                  for j in range(count)]


@pytest.mark.parametrize("log_n,count", [(0, 5), (4, 3), (10, 6)])
def test_ntt_many_equals_ntt(native, log_n, count):
    from interactive_zkp_study_b200.zkp.plonk.field import get_root_of_unity
    n = 1 << log_n
    w = int(get_root_of_unity(n))
    rng = random.Random(log_n)
    _, h = _rand(native, rng, count * n + 2)
    want = []
    for j in range(count):
        one = _one(native, h, 0, count * n + 2)
        native.ntt_dev(one, 2 + j * n, log_n, w, inverse=True, coset_shift=5)
        want += _get(native, one, 2 + j * n, n)
    native.ntt_many_dev(h, 2, log_n, count, w, inverse=True, coset_shift=5)
    assert _get(native, h, 2, count * n) == want


# ------------------------------------------------------------------ end to end, launches, refusals
def test_batch_end_to_end_2_12(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.compat import G2, g2_from_ints
    import plonk_synth
    log_n, count = 12, 128
    n = 1 << log_n
    key, _, tau = plonk_synth.device_setup(plonk_synth.chain_circuit(n, seed=12))
    circs = [plonk_synth.chain_circuit(n, seed=1000 + j) for j in range(count)]
    wit = [_stack(native, [c[k] for c in circs], n) for k in "abc"]
    proofs = dp.prove_batch(key, *wit, count)
    pp = type("PP", (), {})()
    pp.n, pp.omega = n, FR(key.omega)
    for name in dp.CIRCUIT_POLYS:
        setattr(pp, name + "_comm", key.comm[name])
    srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)
    items = [(p, [], pp) for p in proofs]
    assert verify_batch(items, srs, rng=random.Random(1)) is True
    pre = {k: key.comm[k] for k in dp.CIRCUIT_POLYS}
    g2p = [bn254.G2, bn254.g2_mul(bn254.G2, tau)]
    for j in (0, 77, count - 1):
        assert plonk_verifier.verify(_proof_dict(proofs[j]), pre, n, key.omega, g2p) is True
    bad = copy.deepcopy(proofs[40])
    bad.b_eval = bad.b_eval + FR(1)
    assert verify_batch(items[:40] + [(bad, [], pp)] + items[41:], srs, rng=random.Random(2)) is False
    # one broken witness at index 40: the reference's ValueError, naming the proof
    c40 = plonk_synth.chain_circuit(n, seed=1040, break_witness=True)
    native.scalars_upload(wit[2], 40 * n, native.fr_vec_bytes(c40["c"]), n)
    with pytest.raises(ValueError, match="나누어 떨어지지 않.*proof 40 "):
        dp.prove_batch(key, *wit, count)
    with pytest.raises(ValueError, match="proof 40 "):
        dp.prove_batch(key, *wit, count, chunk=16)


def test_launches_do_not_grow_with_count(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    key, wit, _ = _synthetic(native, 6, 256, 60)
    counts = {}
    for count in (16, 256, 16, 256):                    # the first pair warms caches and workspaces
        before = native.launch_count()
        dp.prove_batch(key, *wit, count)
        counts[count] = native.launch_count() - before
    assert counts[256] <= 1.25 * counts[16], counts


def test_refusals_leave_the_library_usable(native):
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    h = native.scalars_alloc(64)
    with pytest.raises(native.ZkpB200Error, match="2\\^32"):
        native.ntt_many_dev(h, 0, 20, 1 << 12, 5)           # 2^12 * 2^20 = 2^32
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.ntt_many_dev(h, 1, 4, 4, 5)                  # 64 elements from offset 1 of 64
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.scan_many_dev(0, native.scalars_alloc(64), 0, h, 0, 9, 8)
    with pytest.raises(native.ZkpB200Error, match="overlaps"):
        native.scan_many_dev(0, h, 0, h, 8, 8, 4)
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.div_linear_many_dev(h, 0, 20, 20, [1, 2, 3, 4], native.scalars_alloc(64), 0, 19)
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.lincomb_many_dev(native.scalars_alloc(64), 0, 16, 16, 5, [(h, 0, 16, 16)], [[1, 0]] * 5)
    with pytest.raises(native.ZkpB200Error, match="groups"):
        native.fr_poly_eval_many_dev([(h, 0, 0, 4, 0)] * 17, 2, [[1, 2]])
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.plonk_blind_many_dev(h, 0, 16, 16, 5, [[1, 2]] * 5, native.scalars_alloc(256), 0, 18)
    with pytest.raises(native.ZkpB200Error, match="range"):
        native.plonk_divisible_many_dev(h, 8, 4, 3)         # 3 blocks of 32 from a handle of 64
    with pytest.raises(native.ZkpB200Error, match="2\\^32"):
        native.plonk_coset_inputs_many_dev(h, h, 8, 1 << 25, 5, h)   # 4 * 2^25 * 2^5 = 2^32
    key, wit, _ = _synthetic(native, 3, 4, 33)
    # a correct call afterwards
    dst = native.scalars_alloc(64)
    native.scan_many_dev(1, dst, 0, h, 0, 16, 4)
    assert _get(native, dst, 0, 1) == [0]
    got = [_proof_dict(p) for p in dp.prove_batch(key, *wit, 4, blinds=[[j] * 9 for j in range(4)])]
    assert got == _loop(native, key, wit, 4, [[j] * 9 for j in range(4)])
