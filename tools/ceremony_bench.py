#!/usr/bin/env python3
"""Powers-of-tau timings on the device (zkp/plonk/ceremony.py and the entry points under it):
  - zkp_g1_table_scale at 2^16, 2^20, 2^22 points and zkp_g2_table_scale at 2^16: CUDA events on the library stream
    around one call, after a warm-up call of the same size; median and minimum of --reps calls;
  - verify_srs, contribute and verify_contribution on a 2^20-power SRS: the whole call (wall clock; it includes
    building the Python point list of the new SRS) and the part of it spent inside native-library calls, each of
    which ends in a device synchronisation (launches, device work, copies; the rest is host Python).
Every timed output is checked: a scaled table against the MSM identity sum_i c_i (k_i s_i G) = <c, k s> G with the
dot product on the device (and byte for byte against the fixed-base table of the products at 2^16); the contributed
SRS byte for byte against the fixed-base table of (tau s)^i; the verifications must accept, and reject a tampered z.
Prints one JSON object (and writes it to --out).

    python tools/ceremony_bench.py [--out FILE] [--reps N]
"""
import argparse
import hashlib
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from interactive_zkp_study_b200 import native  # noqa: E402
from oracle import bn254  # noqa: E402
from pairing_bench import card  # noqa: E402

R = bn254.R
_ENCODERS = {"fe_bytes", "fr_vec_bytes", "fr_vec_from_bytes", "g1_bytes", "g1_vec_bytes", "g2_bytes", "g2_vec_bytes",
             "g1_from_bytes", "g2_from_bytes"}


class NativeClock:
    """Wall time spent inside the public functions of `native` while active (nested calls counted once)."""

    def __enter__(self):
        self.seconds, self._depth, self._saved = 0.0, 0, {}
        for name in dir(native):
            fn = getattr(native, name)
            if (name.startswith("_") or name in _ENCODERS or isinstance(fn, type) or not callable(fn)
                    or getattr(fn, "__module__", None) != native.__name__):
                continue
            self._saved[name] = fn
            setattr(native, name, self._wrap(fn))
        return self

    def _wrap(self, fn):
        def timed_call(*a, **k):
            self._depth += 1
            t = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                self._depth -= 1
                if self._depth == 0:
                    self.seconds += time.perf_counter() - t
        return timed_call

    def __exit__(self, *exc):
        for name, fn in self._saved.items():
            setattr(native, name, fn)


def event_ms(fn, reps):
    fn().free()                                        # warm-up of the same size
    ts = []
    for _ in range(reps):
        native.timer_start()
        h = fn()
        ts.append(native.timer_stop())
        h.free()
    return statistics.median(ts), min(ts)


def scale_record(group, log_n, reps):
    n = 1 << log_n
    s = native.scalars_generate(100 + log_n, n)
    k = native.scalars_generate(200 + log_n, n)
    c = native.scalars_generate(300 + log_n, n)
    if group == 1:
        enc, fixed, scale, msm, mul = (native.g1_bytes, native.g1_fixed_base_mul_dev, native.g1_table_scale,
                                       native.g1_msm_dev, lambda e: bn254.g1_mul(bn254.G1, e))
    else:
        enc, fixed, scale, msm, mul = (native.g2_bytes, native.g2_fixed_base_mul_dev, native.g2_table_scale,
                                       native.g2_msm_dev, lambda e: bn254.g2_mul(bn254.G2, e))
    base = enc(bn254.G1 if group == 1 else bn254.G2)
    pts = fixed(base, s, n)
    med, best = event_ms(lambda: scale(pts, 0, k, 0, n), reps)
    out = scale(pts, 0, k, 0, n)
    prod = native.scalars_alloc(n)
    native.vec_op_dev(2, prod, 0, s, 0, k, 0, n)
    assert enc(msm(out, 0, c, 0, n)) == enc(mul(native.fr_dot_dev(c, 0, prod, 0, n))), (group, log_n)
    if log_n <= 16:
        assert native.table_download(out, 0, n) == native.table_download(fixed(base, prod, n), 0, n), (group, log_n)
    return {"what": "zkp_g%d_table_scale" % group, "points": n, "median_ms": med, "min_ms": best,
            "points_per_s": n / (med * 1e-3), "checked": True}


def timed_call(fn):
    with NativeClock() as clk:
        t = time.perf_counter()
        res = fn()
        wall = time.perf_counter() - t
    return res, wall * 1e3, clk.seconds * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    info = native.device_info()
    res = {"device": info["name"], "nvidia_smi": card(), "records": []}
    for group, log_n in ((1, 16), (1, 20), (1, 22), (2, 16)):
        res["records"].append(scale_record(group, log_n, args.reps))

    from interactive_zkp_study_b200.zkp.plonk.ceremony import Contribution, contribute, verify_contribution, verify_srs
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    d, seed, secret = 1 << 20, 2020, 0x5eed5eed5eed5eed5eed5eed5eed5eed5eed
    srs = SRS.generate(d, seed=seed)
    verify_srs(SRS.generate(4, seed=1))                # warm-up of every kernel on the path
    contribute(SRS.generate(4, seed=1), secret=3)

    ok, wall, nat = timed_call(lambda: verify_srs(srs))
    assert ok is True
    res["records"].append({"what": "verify_srs", "powers": d + 1, "wall_ms": wall, "native_ms": nat, "accepted": True})

    (nxt, proof), wall, nat = timed_call(lambda: contribute(srs, secret=secret))
    tau = int.from_bytes(hashlib.sha256(str(seed).encode()).digest(), "big") % R * secret % R
    powers = native.fr_prefix_product(native.fr_vec_bytes([tau] * (d + 1)), d + 1)
    want = native.table_download(native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), powers, d + 1), 0, d + 1)
    assert native.g1_vec_bytes(nxt.g1_powers) == want
    assert native.g2_bytes(nxt.g2_powers[1]) == native.g2_bytes(bn254.g2_mul(bn254.G2, tau))
    res["records"].append({"what": "contribute", "powers": d + 1, "wall_ms": wall, "native_ms": nat, "checked": True})

    ok, wall, nat = timed_call(lambda: verify_contribution(srs, nxt, proof))
    assert ok is True
    assert verify_contribution(srs, nxt, Contribution(proof.s_g1, proof.R, (proof.z + 1) % R)) is False
    res["records"].append({"what": "verify_contribution", "powers": d + 1, "wall_ms": wall, "native_ms": nat,
                           "accepted": True, "tampered_z_rejected": True})
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
