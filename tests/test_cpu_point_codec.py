"""CPU: the compressed point encoding.  The oracle restatement (tests/codec_oracle.py) round-trips group elements of
both sign classes and infinity and rejects every invalid encoding; known bytes pin the layout; the package's host
encoders equal the oracle; wire records with the compressed tags parse, and malformed lengths are refused before
any device call."""
import random

import pytest

from oracle import bn254
from tests import codec_oracle as co

P, R = bn254.P, bn254.R
rng = random.Random(77)


def _g1_points(k):
    pts = [bn254.g1_mul(bn254.G1, rng.randrange(1, R)) for _ in range(k)]
    return pts + [bn254.g1_neg(p) for p in pts]


def _g2_points(k):
    pts = [bn254.g2_mul(bn254.G2, rng.randrange(1, R)) for _ in range(k)]
    return pts + [bn254.g2_neg(p) for p in pts]


def test_oracle_square_roots():
    for _ in range(50):
        a = rng.randrange(P)
        y = co.fp_sqrt(a)
        assert (y is not None) == (pow(a, (P - 1) // 2, P) in (0, 1))
        if y is not None:
            assert y * y % P == a
    assert co.fp_sqrt(0) == 0 and co.fp_sqrt(3) is None and co.fp_sqrt(P - 1) is None
    for _ in range(60):
        a = (rng.randrange(P), rng.randrange(P))
        y = co.f2_sqrt(a)
        norm = (a[0] * a[0] + a[1] * a[1]) % P
        assert (y is not None) == (pow(norm, (P - 1) // 2, P) == 1)
        if y is not None:
            assert bn254.f2_mul(y, y) == a
    # Fp inside Fp2, pure imaginary, zero, and the alpha = -1 branch (non-squares of Fp have imaginary roots)
    for a in [(5, 0), (4, 0), (0, 7), (P - 1, 0), (0, P - 1), (0, 0), (3, 0), (0, 1)]:
        y = co.f2_sqrt(a)
        assert y is not None and bn254.f2_mul(y, y) == a, a
    assert co.f2_sqrt((P - 1, 0)) in ((0, 1), (0, P - 1))


def test_g1_round_trip_and_known_bytes():
    pts = _g1_points(40) + [None, bn254.G1, bn254.g1_neg(bn254.G1)]
    signs = set()
    for p in pts:
        b = co.g1_compress(p)
        assert len(b) == 32 and co.g1_decompress(b) == p
        if p is not None:
            signs.add(co.g1_sign(p[1]))
    assert signs == {False, True}
    assert co.g1_compress(bn254.G1) == bytes([1]) + bytes(31)
    assert co.g1_compress(bn254.g1_neg(bn254.G1)) == bytes([1]) + bytes(30) + b"\x80"
    assert co.g1_compress(None) == bytes(31) + b"\x40"


def test_g2_round_trip():
    pts = _g2_points(6) + [None, bn254.G2]
    signs = set()
    for p in pts:
        b = co.g2_compress(p)
        assert len(b) == 64 and co.g2_decompress(b) == p
        if p is not None:
            signs.add(co.g2_sign(p[1]))
    assert signs == {False, True}
    assert co.g2_compress(None) == bytes(63) + b"\x40"
    outside = co.twist_point_outside_g2()
    enc = co.g2_compress(outside)
    assert co.g2_decompress(enc, subgroup_check=False) == outside
    with pytest.raises(ValueError):
        co.g2_decompress(enc)


def test_invalid_encodings_are_rejected():
    for enc, why in co.g1_invalid_encodings():
        with pytest.raises(ValueError):
            co.g1_decompress(enc)
    with pytest.raises(ValueError):
        co.g1_decompress(co.g1_no_point_x().to_bytes(32, "little"))
    for enc, why in co.g2_invalid_encodings():
        with pytest.raises(ValueError):
            co.g2_decompress(enc)


def test_host_encoders_equal_the_oracle():
    from interactive_zkp_study_b200 import native
    from interactive_zkp_study_b200.compat import g1_from_ints, g2_from_ints
    g1s, g2s = _g1_points(20) + [None], _g2_points(3) + [None]
    for p in g1s:
        assert native.g1_compressed_bytes(p) == co.g1_compress(p)
        assert native.g1_compressed_bytes(g1_from_ints(p)) == co.g1_compress(p)
    for p in g2s:
        assert native.g2_compressed_bytes(p) == co.g2_compress(p)
        assert native.g2_compressed_bytes(g2_from_ints(p)) == co.g2_compress(p)
    # y1 = 0: the sign comes from y0
    q = ((1, 2), (5, 0))
    assert native.g2_compressed_bytes(q)[63] & 0x80 == 0
    assert native.g2_compressed_bytes(((1, 2), (P - 5, 0)))[63] & 0x80 == 0x80
    assert native.g1_vec_compressed_bytes(g1s) == b"".join(co.g1_compress(p) for p in g1s)
    assert native.g2_vec_compressed_bytes(g2s) == b"".join(co.g2_compress(p) for p in g2s)


def _golden_proof():
    from interactive_zkp_study_b200.compat import g1_from_ints
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.prover import Proof
    from tests.util import g1, load
    f = load("plonk_x3.json")
    proof = Proof()
    for k, v in f["proof"].items():
        setattr(proof, k, g1_from_ints(g1(v)) if k.endswith("_comm") else FR(int(v)))
    return proof


def test_wire_records_with_compressed_tags():
    from interactive_zkp_study_b200 import native
    from interactive_zkp_study_b200.zkp.plonk import wire
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    proof = _golden_proof()
    blob = wire.serialize_proof(proof, compressed=True)
    rec = wire.loads(blob)
    comms = [n for n in rec if n.endswith("_comm")]
    assert len(comms) == 9 and all(rec[n][0] == wire.T_G1C and len(rec[n][1]) == 32 for n in comms)
    assert sum(len(p) for _, p in rec.values()) == 512
    assert sum(len(p) for _, p in wire.loads(wire.serialize_proof(proof)).values()) == 800
    for n in comms:
        assert rec[n][1] == native.g1_compressed_bytes(getattr(proof, n))
    pts = [bn254.g1_mul(bn254.G1, k) for k in (1, 2, 3)]
    g2p = [bn254.G2, bn254.g2_mul(bn254.G2, 9)]
    srs_rec = wire.loads(wire.serialize_srs(SRS(pts, g2p, 2), compressed=True))
    assert srs_rec["g1_powers"] == (wire.T_G1CVEC, native.g1_vec_compressed_bytes(pts))
    assert srs_rec["g2_powers"] == (wire.T_G2CVEC, native.g2_vec_compressed_bytes(g2p))
    # the default stays byte for byte what it was
    assert wire.serialize_srs(SRS(pts, g2p, 2)) == wire.dumps([
        ("g1_powers", wire.T_G1VEC, native.g1_vec_bytes(pts)), ("g2_powers", wire.T_G2VEC, native.g2_vec_bytes(g2p)),
        ("max_degree", wire.T_INT, (2).to_bytes(8, "little"))])
    # an uncompressed proof decodes on the host, as before
    back = wire.deserialize_proof(wire.serialize_proof(proof))
    assert all(getattr(back, n) == getattr(proof, n) for n in comms)


def test_malformed_lengths_are_refused_without_a_device(monkeypatch):
    from interactive_zkp_study_b200 import _lib
    from interactive_zkp_study_b200.zkp.groth16 import wire as gwire
    from interactive_zkp_study_b200.zkp.plonk import wire

    def no_device():
        raise AssertionError("a device call was made")
    monkeypatch.setattr(_lib, "lib", no_device)
    for n in (1, 127, 129, 200):
        with pytest.raises(ValueError, match="128-byte proofs"):
            gwire.deserialize_proofs(bytes(n))
    assert gwire.deserialize_proofs(b"") == []
    with pytest.raises(ValueError, match="32-byte"):
        wire.deserialize_srs(wire.dumps([("g1_powers", wire.T_G1CVEC, bytes(33)), ("g2_powers", wire.T_G2VEC, b""),
                                         ("max_degree", wire.T_INT, bytes(8))]))
    with pytest.raises(ValueError, match="64-byte"):
        wire.deserialize_srs(wire.dumps([("g1_powers", wire.T_G1VEC, b""), ("g2_powers", wire.T_G2CVEC, bytes(65)),
                                         ("max_degree", wire.T_INT, bytes(8))]))
    with pytest.raises(ValueError, match="32-byte"):
        wire.deserialize_srs_to_table(wire.dumps([("g1_powers", wire.T_G1CVEC, bytes(31)),
                                                  ("g2_powers", wire.T_G2VEC, b""), ("max_degree", wire.T_INT, bytes(8))]))
    with pytest.raises(ValueError, match="a compressed G1 point is 32"):
        wire.deserialize_proof(wire.dumps([("a_comm", wire.T_G1C, bytes(31))]))
    with pytest.raises(ValueError, match="a compressed G1 point is 32"):
        wire.deserialize_contribution(wire.dumps([("R", wire.T_G1C, bytes(64))]))
    from interactive_zkp_study_b200 import native
    with pytest.raises(ValueError, match="need 64 bytes"):
        native.g1_table_load_compressed(bytes(63), 2)
    with pytest.raises(ValueError, match="need 64 bytes"):
        native.g2_table_load_compressed(bytes(65), 1)
