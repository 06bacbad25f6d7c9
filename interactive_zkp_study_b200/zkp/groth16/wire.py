"""Binary wire format for Groth16 proofs: 128 bytes per proof (A, B, C), A | B | C compressed (native.g1_compressed_bytes
/ g2_compressed_bytes: x plus a y-sign and an infinity flag; csrc/point_codec.cuh), proofs back to back.

Decoding runs on the device: one call decodes every A and C (on-curve by construction), one every B with the G2
subgroup check, so a blob that parses holds only valid group elements.
"""
from ... import native
from ...compat import g1_from_ints, g2_from_ints

PROOF_BYTES = 128


def serialize_proofs(proofs):
    """[(A, B, C)] as qap_device.prove / prove_batch return them -> 128 bytes per proof."""
    g1, g2 = native.g1_compressed_bytes, native.g2_compressed_bytes
    return b"".join([g1(a) + g2(b) + g1(c) for a, b, c in proofs])


def deserialize_proofs(blob):
    """The inverse of serialize_proofs: [(A, B, C)] in the types qap_device.prove returns.  ValueError names the proof
    and the element of an invalid encoding; a length that is not a multiple of 128 is refused before any device call."""
    blob = bytes(blob)
    if len(blob) % PROOF_BYTES:
        raise ValueError("deserialize_proofs: %d bytes is not a whole number of %d-byte proofs" % (len(blob), PROOF_BYTES))
    k = len(blob) // PROOF_BYTES
    if not k:
        return []
    ac = b"".join([blob[PROOF_BYTES * j:PROOF_BYTES * j + 32] + blob[PROOF_BYTES * j + 96:PROOF_BYTES * (j + 1)]
                   for j in range(k)])
    bs = b"".join([blob[PROOF_BYTES * j + 32:PROOF_BYTES * j + 96] for j in range(k)])
    try:
        t1 = native.g1_table_load_compressed(ac, 2 * k)
    except native.InvalidPointError as e:
        raise ValueError("deserialize_proofs: proof %d, element %s is not a valid compressed point"
                         % (e.index // 2, "AC"[e.index % 2])) from e
    try:
        t2 = native.g2_table_load_compressed(bs, k, subgroup_check=True)
    except native.InvalidPointError as e:
        raise ValueError("deserialize_proofs: proof %d, element B is not a valid compressed G2 point" % e.index) from e
    r1, r2 = native.table_download(t1, 0, 2 * k), native.table_download(t2, 0, k)
    t1.free()
    t2.free()
    return [(g1_from_ints(native.g1_from_bytes(r1[128 * j:128 * j + 64])),
             g2_from_ints(native.g2_from_bytes(r2[128 * j:128 * j + 128])),
             g1_from_ints(native.g1_from_bytes(r1[128 * j + 64:128 * j + 128]))) for j in range(k)]
