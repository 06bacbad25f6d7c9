"""CPU: the host side of the powers-of-tau ceremony (zkp/plonk/ceremony.py) -- the wire record of a Contribution,
the Fiat-Shamir challenge bytes, and the shape checks, which must refuse a malformed SRS before any device call."""
import hashlib

import pytest

from oracle import bn254

R = bn254.R


def _pt(p):
    from interactive_zkp_study_b200.compat import g1_from_ints
    return g1_from_ints(p)


def _srs(d):
    """Points of an honest SRS built on the host (tau = 5), as compat tuples."""
    from interactive_zkp_study_b200.compat import g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    return SRS([_pt(bn254.g1_mul(bn254.G1, pow(5, i, R))) for i in range(d + 1)],
               [g2_from_ints(bn254.G2), g2_from_ints(bn254.g2_mul(bn254.G2, 5))], d)


@pytest.fixture
def no_device(monkeypatch):
    """Any call into the native library fails the test."""
    from interactive_zkp_study_b200 import _lib

    def refuse(*a, **k):
        raise AssertionError("a device call was made")
    monkeypatch.setattr(_lib, "lib", refuse)
    monkeypatch.setattr(_lib, "load_library", refuse)


def test_contribution_wire_round_trip():
    from interactive_zkp_study_b200.zkp.plonk import wire
    from interactive_zkp_study_b200.zkp.plonk.ceremony import Contribution
    c = Contribution(_pt(bn254.g1_mul(bn254.G1, 7)), _pt(bn254.g1_mul(bn254.G1, 11)), R - 3)
    blob = wire.serialize_contribution(c)
    assert blob.startswith(wire.MAGIC)
    back = wire.deserialize_contribution(blob)
    assert [int(v) for v in back.s_g1] == list(bn254.g1_mul(bn254.G1, 7))
    assert [int(v) for v in back.R] == list(bn254.g1_mul(bn254.G1, 11))
    assert back.z == R - 3
    assert wire.deserialize_contribution(wire.from_text(wire.to_text(blob))).z == R - 3
    inf = wire.deserialize_contribution(wire.serialize_contribution(Contribution(None, c.R, 0)))
    assert inf.s_g1 is None and inf.z == 0
    with pytest.raises(ValueError):
        wire.deserialize_contribution(blob[:-5])


def test_challenge_bytes():
    from interactive_zkp_study_b200.zkp.plonk.ceremony import challenge
    prev = _srs(3)
    s_g1, Rp = bn254.g1_mul(bn254.G1, 9), bn254.g1_mul(bn254.G1, 13)

    def le(v):
        return int(v).to_bytes(32, "little")
    t1 = bn254.g1_mul(bn254.G1, 5)
    t2 = bn254.g2_mul(bn254.G2, 5)
    msg = (b"zkp-b200 powers-of-tau v1" + le(t1[0]) + le(t1[1]) + le(t2[0][0]) + le(t2[0][1]) + le(t2[1][0]) +
           le(t2[1][1]) + le(s_g1[0]) + le(s_g1[1]) + le(Rp[0]) + le(Rp[1]))
    want = int.from_bytes(hashlib.sha256(msg).digest(), "big") % R
    assert challenge(prev, _pt(s_g1), _pt(Rp)) == want
    assert challenge(prev, _pt(Rp), _pt(s_g1)) != want
    # infinity is encoded as 64 zero bytes
    msg0 = msg[:-128] + bytes(64) + le(Rp[0]) + le(Rp[1])
    assert challenge(prev, None, _pt(Rp)) == int.from_bytes(hashlib.sha256(msg0).digest(), "big") % R


def test_malformed_srs_shapes_raise_before_any_device_call(no_device):
    from interactive_zkp_study_b200.zkp.plonk.ceremony import Contribution, contribute, verify_contribution, verify_srs
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    good = _srs(3)
    bad = [SRS(good.g1_powers[:3], good.g2_powers, 3),                  # one G1 power short
           SRS(good.g1_powers + [good.g1_powers[1]], good.g2_powers, 3),
           SRS(good.g1_powers, good.g2_powers[:1], 3),                  # [tau]_2 missing
           SRS(good.g1_powers, good.g2_powers * 2, 3),
           SRS(good.g1_powers[:1], good.g2_powers, 0)]                  # max_degree < 1
    proof = Contribution(_pt(bn254.G1), _pt(bn254.G1), 1)
    for srs in bad:
        with pytest.raises(ValueError):
            verify_srs(srs)
        with pytest.raises(ValueError):
            contribute(srs, secret=3)
        with pytest.raises(ValueError):
            verify_contribution(good, srs, proof)
        with pytest.raises(ValueError):
            verify_contribution(srs, good, proof)
    with pytest.raises(ValueError):
        contribute(good, secret=R)                                      # 0 mod r


def test_contribution_with_an_off_curve_or_infinite_s_is_refused_on_the_host(no_device):
    from interactive_zkp_study_b200.zkp.plonk.ceremony import Contribution, verify_contribution
    prev = _srs(3)
    g = bn254.g1_mul(bn254.G1, 4)
    for s_g1 in (None, (g[0], (g[1] + 1) % bn254.P)):
        assert verify_contribution(prev, prev, Contribution(_pt(s_g1), _pt(g), 1)) is False
