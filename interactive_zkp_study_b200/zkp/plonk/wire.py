"""Binary wire format for the PLONK objects (SURVEY.md 8 f3).

The reference moves every prover object between its Flask routes and TinyDB as JSON with one DECIMAL
STRING per field element (/root/reference/plonk_serializers.py:23-250; round trips per round in
plonk_routes.py:298-373).  At 2^20 gates that is ~80 bytes and two bignum <-> decimal conversions per
coefficient per round.  This module is the same set of functions -- same names, same objects in and
out -- over a binary encoding that is the C ABI's own layout, so a polynomial that lives on the GPU is
written and read without ever becoming Python integers:

    Fr      32 bytes little-endian, canonical
    G1      x | y, 64 bytes; the point at infinity (None) is 64 zero bytes
    G2      x.c0 | x.c1 | y.c0 | y.c1, 128 bytes; None is 128 zero bytes
    vectors the elements back to back

Composite objects (SRS, PreprocessedData, Proof, ceremony Contribution) are a flat container: magic, then (name, tag, length,
payload) records.  `to_text` / `from_text` wrap any payload as base64 for stores that only take strings
(TinyDB, JSON responses).

With `compressed=True` the serializers write points compressed (native.g1_compressed_bytes / g2_compressed_bytes:
x plus a y-sign and an infinity flag, 32 / 64 bytes) under their own record tags; uncompressed stays the default.
Every deserializer reads both.  Compressed points are decoded on the device, all G1 points of an object in one call
and all G2 points in another, which also checks them: a G1 point lies on the curve, a G2 point in G2.
"""
import base64
import struct

from ... import native, tables
from ...compat import FQ, FQ2, curve_order
from .ceremony import Contribution
from .field import FR
from .polynomial import Polynomial
from .preprocessor import PreprocessedData
from .prover import Proof
from .srs import SRS
from .transcript import Transcript

MAGIC = b"ZKPB\x01"
T_NONE, T_FR, T_G1, T_G2, T_FRVEC, T_INT, T_U32VEC, T_G1VEC, T_G2VEC, T_BYTES = range(10)
T_G1C, T_G2C, T_G1CVEC, T_G2CVEC = range(10, 14)  # compressed points


# ------------------------------------------------------------------ scalars and points
def serialize_fr(val):
    return (int(val) % curve_order).to_bytes(32, "little")


def deserialize_fr(b):
    return FR(int.from_bytes(b, "little"))


def serialize_g1(point):
    return native.g1_bytes(point)


def deserialize_g1(b):
    p = native.g1_from_bytes(bytes(b))
    return None if p is None else (FQ(p[0]), FQ(p[1]))


def serialize_g2(point):
    return native.g2_bytes(point)


def deserialize_g2(b):
    p = native.g2_from_bytes(bytes(b))
    return None if p is None else (FQ2([p[0][0], p[0][1]]), FQ2([p[1][0], p[1][1]]))


def serialize_fr_list(lst):
    return native.fr_vec_bytes(lst)


def deserialize_fr_list(b):
    return [FR(v) for v in native.fr_vec_from_bytes(bytes(b))]


def serialize_poly(poly):
    """Polynomial -> coefficient bytes (None stays None, as in the reference)."""
    return None if poly is None else native.fr_vec_bytes(poly.coeffs)


def deserialize_poly(b):
    return None if b is None else Polynomial(deserialize_fr_list(b))


# device-resident vectors: no Python integers on the way
def serialize_handle(handle, n=None, offset=0):
    """Device scalar vector (canonical form) -> the same bytes serialize_fr_list would give."""
    return native.scalars_download(handle, offset, handle.n - offset if n is None else n)


def deserialize_to_handle(b):
    return native.scalars_load(bytes(b), len(b) // 32)


def serialize_transcript(transcript):
    return bytes(transcript.state)


def deserialize_transcript(b):
    t = Transcript.__new__(Transcript)
    t.state = bytearray(b)
    return t


# ------------------------------------------------------------------ container
def dumps(fields):
    """fields: iterable of (name, tag, payload) -> one blob."""
    out = [MAGIC]
    for name, tag, payload in fields:
        nb = name.encode("ascii")
        payload = b"" if payload is None else payload
        out.append(struct.pack("<BBQ", len(nb), tag, len(payload)))
        out.append(nb)
        out.append(payload)
    return b"".join(out)


def loads(blob):
    """-> {name: (tag, payload)}; raises ValueError on a foreign or truncated blob."""
    blob = bytes(blob)
    if blob[:len(MAGIC)] != MAGIC:
        raise ValueError("not a zkp-b200 wire blob")
    pos, out = len(MAGIC), {}
    while pos < len(blob):
        if pos + 10 > len(blob):
            raise ValueError("truncated wire blob")
        nlen, tag, plen = struct.unpack_from("<BBQ", blob, pos)
        pos += 10
        if pos + nlen + plen > len(blob):
            raise ValueError("truncated wire blob")
        name = blob[pos:pos + nlen].decode("ascii")
        pos += nlen
        out[name] = (tag, blob[pos:pos + plen])
        pos += plen
    return out


def _g1f(name, p, compressed=False):
    if p is None:
        return (name, T_NONE, None)
    return (name, T_G1C, native.g1_compressed_bytes(p)) if compressed else (name, T_G1, serialize_g1(p))


def _frf(name, v):
    return (name, T_NONE, None) if v is None else (name, T_FR, serialize_fr(v))


def _split(what, payload, size):
    if len(payload) % size:
        raise ValueError("%s: %d bytes is not a whole number of %d-byte points" % (what, len(payload), size))
    return len(payload) // size


def _decode_compressed(what, payload, g2):
    """Compressed G1 / G2 points, back to back -> points as deserialize_g1 / g2 give them: one device decode (G2 with
    the subgroup check).  A rejected encoding raises native.InvalidPointError (a ValueError) with its index."""
    size = 64 if g2 else 32
    n = _split(what, payload, size)
    if not n:
        return []
    if g2:
        h = native.g2_table_load_compressed(payload, n, subgroup_check=True)
    else:
        h = native.g1_table_load_compressed(payload, n)
    raw = native.table_download(h, 0, n)
    h.free()
    dec, sz = (deserialize_g2, 128) if g2 else (deserialize_g1, 64)
    return [dec(raw[sz * i:sz * i + sz]) for i in range(n)]


def _get_g1s(rec, names, what):
    """{name: point} for the single-G1 records `names`; the compressed ones are decoded together."""
    out, comp = {}, []
    for name in names:
        tag, payload = rec.get(name, (T_NONE, b""))
        if tag == T_G1C:
            if len(payload) != 32:
                raise ValueError("%s: record %s holds %d bytes, a compressed G1 point is 32" % (what, name, len(payload)))
            comp.append((name, payload))
        else:
            out[name] = None if tag == T_NONE else deserialize_g1(payload)
    try:
        pts = _decode_compressed(what, b"".join(p for _, p in comp), False)
    except native.InvalidPointError as e:
        raise ValueError("%s: record %s is not a valid compressed G1 point" % (what, comp[e.index][0])) from e
    out.update(zip([name for name, _ in comp], pts))
    return out


def _g1_vec(rec, name, what):
    tag, payload = rec[name]
    if tag == T_G1CVEC:
        return _decode_compressed(what, payload, False)
    return [deserialize_g1(payload[i:i + 64]) for i in range(0, len(payload), 64)]


def _g2_vec(rec, name, what):
    tag, payload = rec[name]
    if tag == T_G2CVEC:
        return _decode_compressed(what, payload, True)
    return [deserialize_g2(payload[i:i + 128]) for i in range(0, len(payload), 128)]


def _get_fr(rec, name):
    tag, payload = rec.get(name, (T_NONE, b""))
    return None if tag == T_NONE else deserialize_fr(payload)


def to_text(blob):
    return base64.b64encode(blob).decode("ascii")


def from_text(text):
    return base64.b64decode(text.encode("ascii"))


# ------------------------------------------------------------------ SRS
def _srs_fields(g1_payload, g2_powers, max_degree, compressed):
    g2 = native.g2_vec_compressed_bytes(g2_powers) if compressed else native.g2_vec_bytes(g2_powers)
    return dumps([("g1_powers", T_G1CVEC if compressed else T_G1VEC, g1_payload),
                  ("g2_powers", T_G2CVEC if compressed else T_G2VEC, g2),
                  ("max_degree", T_INT, struct.pack("<q", max_degree))])


def serialize_srs(srs, compressed=False):
    """compressed=True: 32 bytes per G1 power and 64 per G2 power instead of 64 / 128."""
    g1 = native.g1_vec_compressed_bytes(srs.g1_powers) if compressed else native.g1_vec_bytes(srs.g1_powers)
    return _srs_fields(g1, srs.g2_powers, srs.max_degree, compressed)


def deserialize_srs(blob):
    rec = loads(blob)
    g1 = _g1_vec(rec, "g1_powers", "deserialize_srs")
    g2 = _g2_vec(rec, "g2_powers", "deserialize_srs")
    return SRS(g1, g2, struct.unpack("<q", rec["max_degree"][1])[0])


def deserialize_srs_to_table(blob, precompute=True):
    """SRS blob -> (G1 table handle, g2_powers, max_degree) without making the G1 powers Python integers.  A
    compressed G1 vector is decoded on the device (g1_table_load_compressed); an uncompressed one is uploaded and put
    through g1_table_validate, so either encoding is checked.  ValueError names the first G1 power that is not a
    point of the curve.  precompute=True gives the window-precomputed layout tables.g1_table gives a cached SRS; the
    handle goes straight to plonk.device_prover.preprocess(..., srs_table, srs_size)."""
    rec = loads(blob)
    tag, g1b = rec["g1_powers"]
    what = "deserialize_srs_to_table"
    if tag == T_G1CVEC:
        n = _split(what, g1b, 32)
        try:
            table = native.g1_table_load_compressed(g1b, n)
        except native.InvalidPointError as e:
            raise ValueError("%s: G1 power %d is not a valid compressed point" % (what, e.index)) from e
    elif tag == T_G1VEC:
        n = _split(what, g1b, 64)
        table = native.g1_table_load(g1b, n)
        bad = native.g1_table_validate(table, 0, n)
        if bad is not None:
            table.free()
            raise ValueError("%s: G1 power %d is not on the curve" % (what, bad))
    else:
        raise ValueError("%s: g1_powers is not a G1 vector record (tag %d)" % (what, tag))
    g2 = _g2_vec(rec, "g2_powers", what)
    if precompute:
        tables._maybe_precompute(table, n)
    return table, g2, struct.unpack("<q", rec["max_degree"][1])[0]


def serialize_srs_table(table, g2_powers, max_degree, compressed=False):
    """The inverse of deserialize_srs_to_table: a device-resident G1 table (SRS.generate's, a ceremony's) written as
    serialize_srs would write the same SRS, straight from the device (zkp_table_download[_compressed])."""
    dl = native.table_download_compressed if compressed else native.table_download
    return _srs_fields(dl(table, 0, table.n), g2_powers, max_degree, compressed)


# ------------------------------------------------------------------ powers-of-tau Contribution (ceremony.py)
def serialize_contribution(contribution, compressed=False):
    return dumps([_g1f("s_g1", contribution.s_g1, compressed), _g1f("R", contribution.R, compressed),
                  _frf("z", contribution.z)])


def deserialize_contribution(blob):
    rec = loads(blob)
    z = _get_fr(rec, "z")
    g1 = _get_g1s(rec, ("s_g1", "R"), "deserialize_contribution")
    return Contribution(g1["s_g1"], g1["R"], 0 if z is None else int(z))


# ------------------------------------------------------------------ PreprocessedData
_PP_POLYS = ("q_l", "q_r", "q_o", "q_m", "q_c", "s_sigma1", "s_sigma2", "s_sigma3")


def serialize_preprocessed(pp, compressed=False):
    fields = [("n", T_INT, struct.pack("<q", pp.n)), ("omega", T_FR, serialize_fr(pp.omega)),
              ("domain", T_FRVEC, serialize_fr_list(pp.domain))]
    for name in _PP_POLYS:
        fields.append((name + "_poly", T_FRVEC, serialize_poly(getattr(pp, name + "_poly"))))
        fields.append(_g1f(name + "_comm", getattr(pp, name + "_comm"), compressed))
    fields.append(("sigma", T_U32VEC, struct.pack("<%dI" % len(pp.sigma), *pp.sigma)))
    fields.append(("num_public_inputs", T_INT, struct.pack("<q", pp.num_public_inputs)))
    return dumps(fields)


def deserialize_preprocessed(blob):
    rec = loads(blob)
    pp = PreprocessedData()
    pp.n = struct.unpack("<q", rec["n"][1])[0]
    pp.omega = deserialize_fr(rec["omega"][1])
    pp.domain = deserialize_fr_list(rec["domain"][1])
    comms = _get_g1s(rec, [name + "_comm" for name in _PP_POLYS], "deserialize_preprocessed")
    for name in _PP_POLYS:
        setattr(pp, name + "_poly", deserialize_poly(rec[name + "_poly"][1]))
        setattr(pp, name + "_comm", comms[name + "_comm"])
    sb = rec["sigma"][1]
    pp.sigma = list(struct.unpack("<%dI" % (len(sb) // 4), sb))
    pp.num_public_inputs = struct.unpack("<q", rec["num_public_inputs"][1])[0]
    return pp


# ------------------------------------------------------------------ Proof
_PROOF_G1 = ("a_comm", "b_comm", "c_comm", "z_comm", "t_lo_comm", "t_mid_comm", "t_hi_comm", "W_zeta_comm",
             "W_zeta_omega_comm")
_PROOF_FR = ("a_eval", "b_eval", "c_eval", "s_sigma1_eval", "s_sigma2_eval", "z_omega_eval", "r_eval")


def serialize_proof(proof, compressed=False):
    """9 G1 points + 7 field elements: 800 bytes of payload for a complete proof, 512 compressed."""
    return dumps([_g1f(n, getattr(proof, n), compressed) for n in _PROOF_G1] +
                 [_frf(n, getattr(proof, n)) for n in _PROOF_FR])


def deserialize_proof(blob):
    rec = loads(blob)
    proof = Proof()
    g1 = _get_g1s(rec, _PROOF_G1, "deserialize_proof")
    for n in _PROOF_G1:
        setattr(proof, n, g1[n])
    for n in _PROOF_FR:
        setattr(proof, n, _get_fr(rec, n))
    return proof
