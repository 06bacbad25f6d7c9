"""-m gpu: compressed points (csrc/point_codec.cuh).  Device decoding and encoding against the oracle restatement
(tests/codec_oracle.py), planted invalid encodings rejected at the lowest index, the decoder's square roots on chosen
elements, round trips at 2^20 G1 / 2^16 G2 points, MSMs on compressed-loaded tables, and the wire formats: PLONK proofs,
SRSs decoded straight into device tables, and Groth16 proofs."""
import copy
import random

import pytest

from oracle import bn254
from tests import codec_oracle as co
from tests.util import g1, g2, ints, load

pytestmark = pytest.mark.gpu
P, R = bn254.P, bn254.R
rng = random.Random(4242)


def _g1_points(native, k):
    t = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes([rng.randrange(1, R) for _ in range(k)]), k)
    raw = native.table_download(t, 0, k)
    return [native.g1_from_bytes(raw[64 * i:64 * i + 64]) for i in range(k)]


def _g2_points(native, k):
    t = native.g2_fixed_base_mul(native.g2_bytes(bn254.G2), native.fr_vec_bytes([rng.randrange(1, R) for _ in range(k)]), k)
    raw = native.table_download(t, 0, k)
    return [native.g2_from_bytes(raw[128 * i:128 * i + 128]) for i in range(k)]


def _mixed(pts, neg):
    out = pts + [neg(p) for p in pts[:len(pts) // 2]]
    for i in (0, 7, len(out) - 1):
        out[i] = None
    return out


def _index_error(fn, *args):
    from interactive_zkp_study_b200 import native
    with pytest.raises(native.InvalidPointError) as e:
        fn(*args)
    return e.value.index


def test_g1_decode_matches_oracle(native):
    pts = _mixed(_g1_points(native, 2048), bn254.g1_neg)
    enc = b"".join(co.g1_compress(p) for p in pts)
    t = native.g1_table_load_compressed(enc, len(pts))
    got = native.table_download(t, 0, len(pts))
    assert got == native.g1_vec_bytes(pts)
    assert got == native.g1_vec_bytes([co.g1_decompress(enc[32 * i:32 * i + 32]) for i in range(len(pts))])
    assert native.g1_table_load_compressed(b"", 0).n == 0


def test_g2_decode_matches_oracle(native):
    pts = _mixed(_g2_points(native, 1024), bn254.g2_neg)
    enc = b"".join(co.g2_compress(p) for p in pts)
    want = native.g2_vec_bytes(pts)
    assert want == native.g2_vec_bytes([co.g2_decompress(enc[64 * i:64 * i + 64], subgroup_check=False)
                                        for i in range(len(pts))])
    for sub in (True, False):
        assert native.table_download(native.g2_table_load_compressed(enc, len(pts), sub), 0, len(pts)) == want


def test_invalid_encodings_rejected_at_the_lowest_index(native):
    good1 = [co.g1_compress(p) for p in _g1_points(native, 600)]
    bad1 = [e for e, _ in co.g1_invalid_encodings()] + [co.g1_no_point_x().to_bytes(32, "little")]
    for enc in bad1:
        for where in ([0], [599], [321], [450, 123]):
            v = list(good1)
            for i in where:
                v[i] = enc
            assert _index_error(native.g1_table_load_compressed, b"".join(v), len(v)) == min(where)
    good2 = [co.g2_compress(p) for p in _g2_points(native, 200)]
    for enc, why in co.g2_invalid_encodings():
        for where in ([0], [199], [150, 40]):
            v = list(good2)
            for i in where:
                v[i] = enc
            for sub in (True, False):
                assert _index_error(native.g2_table_load_compressed, b"".join(v), len(v), sub) == min(where), why
    # a twist point outside G2: rejected with the subgroup check, decoded without it
    outside = co.twist_point_outside_g2()
    v = list(good2)
    v[77] = co.g2_compress(outside)
    v[150] = co.g2_compress(outside)
    assert _index_error(native.g2_table_load_compressed, b"".join(v), len(v)) == 77
    t = native.g2_table_load_compressed(b"".join(v), len(v), subgroup_check=False)
    assert native.g2_from_bytes(native.table_download(t, 77, 1)) == outside
    assert native.g2_table_validate(t, 0, len(v), subgroup_check=True) == 77
    # the library stays usable after refusals
    assert native.table_download(native.g1_table_load_compressed(b"".join(good1), 600), 0, 1) == \
        native.g1_bytes(co.g1_decompress(good1[0]))


def test_square_roots_match_the_oracle(native):
    ones32 = b"\xff" * 32
    fp = [0, 1, 3, 4, P - 1, P - 4, 5] + [rng.randrange(P) for _ in range(200)] + \
         [pow(rng.randrange(P), 2, P) for _ in range(50)]
    got = native.dbg_field_op(0, 9, native.fr_vec_bytes(fp), None, len(fp))
    for i, a in enumerate(fp):
        y = co.fp_sqrt(a)
        assert got[32 * i:32 * i + 32] == (ones32 if y is None else y.to_bytes(32, "little")), a
    f2 = [(5, 0), (4, 0), (3, 0), (0, 7), (0, 1), (P - 1, 0), (0, P - 1), (0, 0), (1, 0)] + \
         [(rng.randrange(P), rng.randrange(P)) for _ in range(200)] + \
         [bn254.f2_mul(a, a) for a in [(rng.randrange(P), rng.randrange(P)) for _ in range(50)]] + \
         [(rng.randrange(P), 0) for _ in range(30)] + [(0, rng.randrange(P)) for _ in range(30)]
    got = native.dbg_field_op(2, 9, b"".join(native.fe_bytes(a) + native.fe_bytes(b) for a, b in f2), None, len(f2))
    roots = 0
    for i, a in enumerate(f2):
        y = co.f2_sqrt(a)
        want = b"\xff" * 64 if y is None else native.fe_bytes(y[0]) + native.fe_bytes(y[1])
        assert got[64 * i:64 * i + 64] == want, a
        roots += y is not None
    assert 0 < roots < len(f2)
    with pytest.raises(native.ZkpB200Error, match="error -3"):
        native.dbg_field_op(1, 9, native.fr_vec_bytes([4]), None, 1)


def test_compression_matches_host_encoders_and_oracle(native):
    pts = _mixed(_g1_points(native, 1500), bn254.g1_neg)
    n = len(pts)
    t = native.g1_table_load(native.g1_vec_bytes(pts), n)
    want = native.g1_vec_compressed_bytes(pts)
    assert want == b"".join(co.g1_compress(p) for p in pts)
    assert native.table_download_compressed(t, 0, n) == want
    assert native.table_download_compressed(t, 100, 333) == want[3200:32 * 433]
    native.table_precompute(t)
    assert native.table_download_compressed(t, 0, n) == want
    assert native.table_download_compressed(t, n - 5, 5) == want[32 * (n - 5):]
    q = _mixed(_g2_points(native, 300), bn254.g2_neg)
    t2 = native.g2_table_load(native.g2_vec_bytes(q), len(q))
    want2 = native.g2_vec_compressed_bytes(q)
    assert want2 == b"".join(co.g2_compress(p) for p in q)
    assert native.table_download_compressed(t2, 0, len(q)) == want2
    native.table_precompute(t2, 6)
    assert native.table_download_compressed(t2, 10, 20) == want2[640:64 * 30]
    with pytest.raises(native.ZkpB200Error, match="error -3"):
        native.table_download_compressed(t2, len(q) - 1, 2)
    sc = native.scalars_load(native.fr_vec_bytes([1]), 1)
    with pytest.raises(native.ZkpB200Error, match="error -4"):
        native.table_download_compressed(sc, 0, 1)


@pytest.mark.parametrize("group,log_n", [(1, 20), (2, 16)])
def test_round_trip_at_scale(native, group, log_n):
    n = 1 << log_n
    s = native.scalars_generate(70 + log_n, n)
    if group == 1:
        t = native.g1_fixed_base_mul_dev(native.g1_bytes(bn254.G1), s, n)
        back = native.g1_table_load_compressed(native.table_download_compressed(t, 0, n), n)
    else:
        t = native.g2_fixed_base_mul_dev(native.g2_bytes(bn254.G2), s, n)
        back = native.g2_table_load_compressed(native.table_download_compressed(t, 0, n), n)
    assert native.table_download(back, 0, n) == native.table_download(t, 0, n)


def test_compressed_tables_give_the_same_msms(native):
    pts = _mixed(_g1_points(native, 3000), bn254.g1_neg)
    n = len(pts)
    sc = native.fr_vec_bytes([rng.randrange(R) for _ in range(n)])
    plain = native.g1_table_load(native.g1_vec_bytes(pts), n)
    comp = native.g1_table_load_compressed(native.g1_vec_compressed_bytes(pts), n)
    want = native.g1_msm_table(plain, 0, sc, n)
    assert native.g1_msm_table(comp, 0, sc, n) == want
    native.table_precompute(comp)
    assert native.g1_msm_table(comp, 0, sc, n) == want
    q = _mixed(_g2_points(native, 64), bn254.g2_neg)
    sc2 = native.fr_vec_bytes([rng.randrange(R) for _ in q])
    comp2 = native.g2_table_load_compressed(native.g2_vec_compressed_bytes(q), len(q))
    assert native.g2_msm_table(comp2, 0, sc2, len(q)) == native.g2_msm(native.g2_vec_bytes(q), sc2, len(q))


def _norm(proof):
    return {k: (None if v is None else (int(v[0]), int(v[1]))) if k.endswith("_comm") else int(v)
            for k, v in vars(proof).items()}


def _golden(name):
    from interactive_zkp_study_b200.compat import g1_from_ints, g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk.field import FR as PFR
    from interactive_zkp_study_b200.zkp.plonk.prover import Proof
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    f = load(name)
    proof = Proof()
    for k, v in f["proof"].items():
        setattr(proof, k, g1_from_ints(g1(v)) if k.endswith("_comm") else PFR(int(v)))
    pp = type("PP", (), {})()
    pp.n, pp.omega, pp.num_public_inputs = f["n"], PFR(int(f["omega"])), 0
    for k, v in f["pre_comm"].items():
        setattr(pp, k + "_comm", g1_from_ints(g1(v)))
    srs = SRS([g1_from_ints(g1(p)) for p in f["g1_powers"]], [g2_from_ints(g2(p)) for p in f["g2_powers"]],
              f["srs_max_degree"])
    return f, proof, pp, srs


@pytest.mark.parametrize("name", ["plonk_n1.json", "plonk_x3.json", "plonk_chain16.json"])
def test_plonk_wire_golden_proofs(native, name):
    from interactive_zkp_study_b200.zkp.pairing import pairing
    from interactive_zkp_study_b200.zkp.plonk import wire
    from interactive_zkp_study_b200.zkp.plonk.ceremony import Contribution
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify
    f, proof, pp, srs = _golden(name)
    blob = wire.serialize_proof(proof, compressed=True)
    assert sum(len(p) for _, p in wire.loads(blob).values()) == 512
    back = wire.deserialize_proof(blob)
    assert _norm(back) == _norm(proof)
    assert verify(back, [], pp, srs, pairing=pairing) is True
    bad = copy.deepcopy(back)
    bad.a_eval = bad.a_eval + 1
    assert verify(bad, [], pp, srs, pairing=pairing) is False
    # a commitment replaced by an x with no point is refused, naming the record
    rec = wire.loads(blob)
    rec["z_comm"] = (wire.T_G1C, co.g1_no_point_x().to_bytes(32, "little"))
    with pytest.raises(ValueError, match="z_comm"):
        wire.deserialize_proof(wire.dumps([(k, t, p) for k, (t, p) in rec.items()]))
    # today's uncompressed blobs decode exactly as before; the compressed forms decode to the same objects
    assert _norm(wire.deserialize_proof(wire.serialize_proof(proof))) == _norm(proof)
    for compressed in (False, True):
        s2 = wire.deserialize_srs(wire.serialize_srs(srs, compressed=compressed))
        assert (s2.g1_powers, s2.g2_powers, s2.max_degree) == (srs.g1_powers, srs.g2_powers, srs.max_degree)
        c = Contribution(srs.g1_powers[-1], None, 12345)
        c2 = wire.deserialize_contribution(wire.serialize_contribution(c, compressed=compressed))
        assert (c2.s_g1, c2.R, c2.z) == (c.s_g1, c.R, c.z)


def test_plonk_wire_preprocessed(native):
    from interactive_zkp_study_b200.zkp.plonk import wire
    from interactive_zkp_study_b200.zkp.plonk.field import FR as PFR
    from interactive_zkp_study_b200.zkp.plonk.polynomial import Polynomial
    from interactive_zkp_study_b200.zkp.plonk.preprocessor import PreprocessedData
    f, _, _, _ = _golden("plonk_x3.json")
    pp = PreprocessedData()
    pp.n, pp.omega, pp.domain = f["n"], PFR(int(f["omega"])), [PFR(int(x)) for x in f["domain"]]
    for k in f["pre"]:
        setattr(pp, k + "_poly", Polynomial([PFR(int(x)) for x in f["pre"][k]]))
        setattr(pp, k + "_comm", g1(f["pre_comm"][k]))
    pp.q_c_comm = None
    pp.sigma, pp.num_public_inputs = [int(x) for x in f["sigma"]], 0
    plain = wire.serialize_preprocessed(pp)
    comp = wire.serialize_preprocessed(pp, compressed=True)
    assert len(plain) - len(comp) == 7 * 32
    for blob in (plain, comp):
        back = wire.deserialize_preprocessed(blob)
        for k in f["pre"]:
            got = getattr(back, k + "_comm")
            assert (None if got is None else (int(got[0]), int(got[1]))) == getattr(pp, k + "_comm"), k
            assert getattr(back, k + "_poly").coeffs == getattr(pp, k + "_poly").coeffs
        assert back.sigma == pp.sigma


def test_srs_decoded_into_a_device_table(native):
    from interactive_zkp_study_b200 import tables
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp, wire
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import plonk_synth
    d = (1 << 12) + 5
    srs = SRS.generate(d, seed=77)
    ref = native.table_download(tables.g1_table(srs.g1_powers), 0, d + 1)
    for compressed in (False, True):
        blob = wire.serialize_srs(srs, compressed=compressed)
        table, g2p, md = wire.deserialize_srs_to_table(blob)
        assert md == d and g2p == srs.g2_powers and table.n == d + 1 and getattr(table, "pre_c", 0) > 0
        assert native.table_download(table, 0, d + 1) == ref
        assert wire.serialize_srs_table(table, g2p, md, compressed=compressed) == blob
        plain, _, _ = wire.deserialize_srs_to_table(blob, precompute=False)
        assert getattr(plain, "pre_c", 0) == 0 and native.table_download(plain, 0, d + 1) == ref
    # a proof under the decoded table equals the proof under the list-based table (golden chain16 with its blinds)
    f, proof, _, srs16 = _golden("plonk_chain16.json")
    n = f["n"]
    pad = lambda v: ints(v) + [0] * (n - len(v))
    sel = [native.scalars_load(native.fr_vec_bytes(pad(f["selectors"][k])), n) for k in ("q_l", "q_r", "q_o", "q_m", "q_c")]
    sig = [native.scalars_load(b, n) for b in plonk_synth.sigma_evals_bytes(f["sigma"], n, int(f["omega"]))]
    wit = [native.scalars_load(native.fr_vec_bytes(ints(f[k + "_vals"])), n) for k in "abc"]
    size = len(srs16.g1_powers)
    got = []
    for table in (tables.g1_table(srs16.g1_powers), wire.deserialize_srs_to_table(wire.serialize_srs(srs16, True))[0]):
        key = dp.preprocess(n, sel, sig, table, size)
        got.append(_norm(dp.prove(key, *wit, blinds=ints(f["blinds"]))))
    assert got[0] == got[1] == _norm(proof)
    # one bad G1 power is refused, naming it, in either encoding
    pts = list(srs.g1_powers)
    off = bn254.g1_mul(bn254.G1, 3)
    blob = wire.serialize_srs(SRS(pts[:9] + [(off[0], off[1] + 1)] + pts[10:], srs.g2_powers, d))
    with pytest.raises(ValueError, match="G1 power 9 "):
        wire.deserialize_srs_to_table(blob)
    rec = wire.loads(wire.serialize_srs(srs, compressed=True))
    g1b = bytearray(rec["g1_powers"][1])
    g1b[32 * 4000:32 * 4001] = co.g1_no_point_x().to_bytes(32, "little")
    rec["g1_powers"] = (wire.T_G1CVEC, bytes(g1b))
    blob = wire.dumps([(k, t, p) for k, (t, p) in rec.items()])
    with pytest.raises(ValueError, match="G1 power 4000 "):
        wire.deserialize_srs_to_table(blob)
    with pytest.raises(ValueError):
        wire.deserialize_srs(blob)


def test_groth16_wire(native):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from qap_large import circuit
    from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd, wire as gwire
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify_batch
    k, count = 1 << 8, 128
    m = k + 2
    ra, rb, rc, _ = circuit(k, 7)
    dev = qd.DeviceR1CS(qd.SparseR1CS.from_rows(k, m, ra, rb, rc))
    keys = qd.setup(dev, *(rng.randrange(1, R) for _ in range(5)), lcm=True, precompute=True)
    ws = []
    for _ in range(count):
        w = [1, rng.randrange(2, 1 << 20)]
        for a, b in zip(ra, rb):
            w.append(sum(v * w[i] for i, v in a.items()) * sum(v * w[i] for i, v in b.items()) % R)
        ws.append(w)
    rs = [rng.randrange(R) for _ in range(count)]
    ss = [rng.randrange(R) for _ in range(count)]
    proofs = qd.prove_batch(keys, dev, native.scalars_load(native.fr_vec_bytes([x for w in ws for x in w]), count * m),
                            rs, ss)
    blob = gwire.serialize_proofs(proofs)
    assert len(blob) == 128 * count
    back = gwire.deserialize_proofs(blob)
    assert back == proofs
    assert [type(x) for x in back[0]] == [type(x) for x in proofs[0]]
    vk = (keys.sigma1_1, keys.sigma1_3, keys.sigma2_1)
    pubs = [[(i, w[i]) for i in keys.pub_idx] for w in ws]
    assert verify_batch(back, *vk, pubs, rng=random.Random(1)) is True
    flipped = bytearray(blob)
    flipped[128 * 50 + 95] ^= 0x80                   # B's y-sign of proof 50: -B, still in G2
    fb = gwire.deserialize_proofs(bytes(flipped))
    assert native.g2_bytes(fb[50][1]) == native.g2_bytes(bn254.g2_neg(native.g2_from_bytes(native.g2_bytes(proofs[50][1]))))
    assert verify_batch(fb, *vk, pubs, rng=random.Random(2)) is False
    outside = bytearray(blob)
    outside[128 * 90 + 32:128 * 90 + 96] = co.g2_compress(co.twist_point_outside_g2())
    with pytest.raises(ValueError, match="proof 90, element B"):
        gwire.deserialize_proofs(bytes(outside))
    bad_c = bytearray(blob)
    bad_c[128 * 3 + 96:128 * 4] = P.to_bytes(32, "little")
    with pytest.raises(ValueError, match="proof 3, element C"):
        gwire.deserialize_proofs(bytes(bad_c))
