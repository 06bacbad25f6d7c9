#!/usr/bin/env python3
"""Compressed point encodings on the device (csrc/point_codec.cuh and the wire formats on top):
  - zkp_g1_table_load_compressed at 2^16 / 2^20 / 2^22 points, zkp_g2_table_load_compressed at 2^16 with and without
    the subgroup check, zkp_table_download_compressed at 2^20 G1 points, and zkp_table_download and
    zkp_g1_table_scale at 2^20 for comparison: CUDA events on the library stream around one call (the call's host
    copies included), after a warm-up call of the same size; median and minimum of --reps calls;
  - loading a 2^20-power SRS blob three ways (wall clock, whole call): plonk.wire.deserialize_srs_to_table on a
    compressed and on an uncompressed blob, and deserialize_srs + tables.g1_table (a Python point list, then the
    table);
  - groth16.wire.deserialize_proofs of 16 384 proofs (wall clock);
each wall-clock case is the median and minimum of --reps calls.
Every timed result is checked byte for byte against the table or points it came from.  Prints one JSON object (and
writes it to --out).

    python tools/point_codec_bench.py [--out FILE] [--reps N]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from interactive_zkp_study_b200 import native, tables  # noqa: E402
from oracle import bn254  # noqa: E402
from pairing_bench import card  # noqa: E402


def event_ms(fn, reps):
    fn()                                               # warm-up of the same size
    ts = []
    for _ in range(reps):
        native.timer_start()
        fn()
        ts.append(native.timer_stop())
    return statistics.median(ts), min(ts)


def wall_ms(fn, reps):
    ts, out = [], None
    for _ in range(reps):
        t = time.perf_counter()
        out = fn()
        ts.append((time.perf_counter() - t) * 1e3)
    return statistics.median(ts), min(ts), out


def source_table(group, n, seed):
    s = native.scalars_generate(seed, n)
    if group == 1:
        return native.g1_fixed_base_mul_dev(native.g1_bytes(bn254.G1), s, n)
    return native.g2_fixed_base_mul_dev(native.g2_bytes(bn254.G2), s, n)


def load_record(group, log_n, reps, subgroup=True):
    n = 1 << log_n
    src = source_table(group, n, 500 + log_n)
    enc = native.table_download_compressed(src, 0, n)
    if group == 1:
        load = lambda: native.g1_table_load_compressed(enc, n)
    else:
        load = lambda: native.g2_table_load_compressed(enc, n, subgroup_check=subgroup)
    med, best = event_ms(lambda: load().free(), reps)
    assert native.table_download(load(), 0, n) == native.table_download(src, 0, n), (group, log_n)
    rec = {"what": "zkp_g%d_table_load_compressed" % group, "points": n, "median_ms": med, "min_ms": best,
           "mpts_per_s": n / (med * 1e-3) / 1e6, "checked": True}
    if group == 2:
        rec["subgroup_check"] = subgroup
    return rec


def download_records(log_n, reps):
    """The compressed download beside the uncompressed one of the same table (both copy into a fresh host buffer)."""
    n = 1 << log_n
    src = source_table(1, n, 600 + log_n)
    out = []
    for what, fn in (("zkp_table_download_compressed", native.table_download_compressed),
                     ("zkp_table_download (for comparison)", native.table_download)):
        med, best = event_ms(lambda: fn(src, 0, n), reps)
        out.append({"what": what, "points": n, "median_ms": med, "min_ms": best, "mpts_per_s": n / (med * 1e-3) / 1e6})
    enc = native.table_download_compressed(src, 0, n)
    assert native.table_download(native.g1_table_load_compressed(enc, n), 0, n) == native.table_download(src, 0, n)
    out[0]["checked"] = True
    return out


def scale_record(log_n, reps):
    n = 1 << log_n
    src = source_table(1, n, 700 + log_n)
    k = native.scalars_generate(800 + log_n, n)
    med, best = event_ms(lambda: native.g1_table_scale(src, 0, k, 0, n).free(), reps)
    return {"what": "zkp_g1_table_scale (for comparison)", "points": n, "median_ms": med, "min_ms": best,
            "mpts_per_s": n / (med * 1e-3) / 1e6}


def srs_records(log_d, reps):
    from interactive_zkp_study_b200.zkp.plonk import wire
    n = 1 << log_d
    d = n - 1
    src = source_table(1, n, 900)
    want = native.table_download(src, 0, n)
    g2p = [bn254.G2, bn254.g2_mul(bn254.G2, 12345)]
    out = []
    for compressed in (True, False):
        blob = wire.serialize_srs_table(src, g2p, d, compressed=compressed)
        med, best, (table, _, _) = wall_ms(lambda: wire.deserialize_srs_to_table(blob), reps)
        assert native.table_download(table, 0, n) == want
        out.append({"what": "wire.deserialize_srs_to_table", "encoding": "compressed" if compressed else "uncompressed",
                    "powers": n, "blob_bytes": len(blob), "median_ms": med, "min_ms": best, "checked": True})
    blob = wire.serialize_srs_table(src, g2p, d)

    def list_path():
        srs = wire.deserialize_srs(blob)
        return native.table_download(tables.g1_table(srs.g1_powers), 0, n)
    med, best, got = wall_ms(list_path, reps)
    assert got == want
    out.append({"what": "wire.deserialize_srs + tables.g1_table", "encoding": "uncompressed", "powers": n,
                "blob_bytes": len(blob), "median_ms": med, "min_ms": best, "checked": True})
    tables.clear()
    return out


def groth16_record(count, reps):
    from interactive_zkp_study_b200.compat import g1_from_ints, g2_from_ints
    from interactive_zkp_study_b200.zkp.groth16 import wire as gwire
    ac = source_table(1, 2 * count, 1001)
    b = source_table(2, count, 1002)
    enc_ac, enc_b = native.table_download_compressed(ac, 0, 2 * count), native.table_download_compressed(b, 0, count)
    blob = b"".join(enc_ac[64 * j:64 * j + 32] + enc_b[64 * j:64 * j + 64] + enc_ac[64 * j + 32:64 * j + 64]
                    for j in range(count))
    med, best, proofs = wall_ms(lambda: gwire.deserialize_proofs(blob), reps)
    raw_ac, raw_b = native.table_download(ac, 0, 2 * count), native.table_download(b, 0, count)
    assert proofs == [(g1_from_ints(native.g1_from_bytes(raw_ac[128 * j:128 * j + 64])),
                       g2_from_ints(native.g2_from_bytes(raw_b[128 * j:128 * j + 128])),
                       g1_from_ints(native.g1_from_bytes(raw_ac[128 * j + 64:128 * j + 128]))) for j in range(count)]
    assert gwire.serialize_proofs(proofs) == blob
    return {"what": "groth16.wire.deserialize_proofs", "proofs": count, "blob_bytes": len(blob), "median_ms": med,
            "min_ms": best, "proofs_per_s": count / (med * 1e-3), "checked": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    info = native.device_info()
    res = {"device": info["name"], "nvidia_smi": card(), "records": []}
    for log_n in (16, 20, 22):
        res["records"].append(load_record(1, log_n, args.reps))
    for sub in (True, False):
        res["records"].append(load_record(2, 16, args.reps, subgroup=sub))
    res["records"].extend(download_records(20, args.reps))
    res["records"].append(scale_record(20, args.reps))
    res["records"].extend(srs_records(20, args.reps))
    res["records"].append(groth16_record(16384, args.reps))
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
