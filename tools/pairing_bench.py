#!/usr/bin/env python3
"""Pairing-side timings on the device: latency of one pairing check (2 and 4 pairs), Groth16 batch verification
(k = 1, 64, 1024, 16384 proofs, as proofs/s) and PLONK batch verification (k = 1, 64), next to one pairing of the
oracle's pure-Python py_ecc restatement on the host.  Every timed batch's decision is checked, and a batch with one
tampered proof must be rejected.  Prints one JSON object (and writes it to --out).

    python tools/pairing_bench.py [--out FILE] [--reps N]

Groth16 inputs are cheap and valid at any k: keys with known alpha, beta, gamma, delta and one public wire
(sigma1_3 = [s0 G1]); proof j is A = a G1, B = b G2, C = c G1 from the device's fixed-base multiplication with
c = (a b - alpha beta - x_j s0 gamma) / delta.  PLONK proofs come from the device prover on a 2^6-gate chain.
"""
import argparse
import copy
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from interactive_zkp_study_b200 import native  # noqa: E402
from oracle import bn254  # noqa: E402

R = bn254.R


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        res = fn()
        ts.append(time.perf_counter() - t)
    return res, statistics.median(ts), min(ts)


def device_points(g1_scalars, g2_scalars):
    n1, n2 = len(g1_scalars), len(g2_scalars)
    t1 = native.g1_fixed_base_mul(native.g1_bytes(bn254.G1), native.fr_vec_bytes(g1_scalars), n1)
    t2 = native.g2_fixed_base_mul(native.g2_bytes(bn254.G2), native.fr_vec_bytes(g2_scalars), n2)
    return native.table_download(t1, 0, n1), native.table_download(t2, 0, n2)


def synthetic_groth16(k, seed):
    from interactive_zkp_study_b200.compat import g1_from_ints, g2_from_ints
    rr = random.Random(seed)
    al, be, ga, de, s0 = (rr.randrange(1, R) for _ in range(5))
    a = [rr.randrange(1, R) for _ in range(k)]
    b = [rr.randrange(1, R) for _ in range(k)]
    x = [rr.randrange(R) for _ in range(k)]
    dinv = pow(de, -1, R)
    c = [(ai * bi - al * be - xi * s0 * ga) * dinv % R for ai, bi, xi in zip(a, b, x)]
    g1b, g2b = device_points(a + c + [al, s0], b + [be, ga, de])
    pt1 = [g1_from_ints(native.g1_from_bytes(g1b[64 * i:64 * i + 64])) for i in range(2 * k + 2)]
    pt2 = [g2_from_ints(native.g2_from_bytes(g2b[128 * i:128 * i + 128])) for i in range(k + 3)]
    proofs = [(pt1[j], pt2[j], pt1[k + j]) for j in range(k)]
    return proofs, ([pt1[2 * k]], [pt1[2 * k + 1]], pt2[k:k + 3]), [[(0, xi)] for xi in x]


def cancelling_pairs(n, seed):
    rr = random.Random(seed)
    a = [rr.randrange(1, R) for _ in range(n)]
    b = [rr.randrange(1, R) for _ in range(n - 1)]
    b.append((-sum(x * y for x, y in zip(a, b)) * pow(a[-1], -1, R)) % R)
    g1b, g2b = device_points(b, a)
    return g2b, g1b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    info = native.device_info()
    res = {"device": info["name"], "nvidia_smi": card(), "records": []}

    from oracle.shim.py_ecc import bn128 as bn
    t = time.perf_counter()
    bn.pairing(bn.G2, bn.G1)
    res["cpu_shim_pairing_s"] = time.perf_counter() - t

    for n in (2, 4):
        g2b, g1b = cancelling_pairs(n, n)
        ok, med, best = timed(lambda: native.pairing_check(g2b, g1b, n), max(args.reps, 10))
        assert ok is True
        res["records"].append({"what": "pairing_check", "pairs": n, "median_ms": med * 1e3, "min_ms": best * 1e3})

    from interactive_zkp_study_b200.compat import g1_from_ints
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify_batch
    for k in (1, 64, 1024, 16384):
        proofs, keys, pubs = synthetic_groth16(k, k)
        reps = args.reps if k <= 1024 else 2
        ok, med, best = timed(lambda: verify_batch(proofs, *keys, pubs), reps)
        assert ok is True, k
        bad = list(proofs)
        A, B, C = bad[k // 2]
        bad[k // 2] = (A, B, g1_from_ints(bn254.g1_add((int(C[0]), int(C[1])), bn254.G1)))
        assert verify_batch(bad, *keys, pubs) is False, k
        res["records"].append({"what": "groth16.verify_batch", "k": k, "median_ms": med * 1e3, "min_ms": best * 1e3,
                               "proofs_per_s": k / med, "tampered_rejected": True})

    import plonk_synth
    from interactive_zkp_study_b200.compat import G2, g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch as pverify_batch
    n = 1 << 6
    key, wit, tau = plonk_synth.device_setup(plonk_synth.chain_circuit(n, seed=3))
    pp = type("PP", (), {})()
    pp.n, pp.omega = n, FR(key.omega)
    for name in dp.CIRCUIT_POLYS:
        setattr(pp, name + "_comm", key.comm[name])
    srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)
    items = [(dp.prove(key, *wit), [], pp) for _ in range(64)]
    for k in (1, 64):
        ok, med, best = timed(lambda: pverify_batch(items[:k], srs), args.reps)
        assert ok is True, k
        bad = copy.deepcopy(items[0][0])
        bad.a_eval = bad.a_eval + FR(1)
        assert pverify_batch([(bad, [], pp)] + items[1:k], srs) is False, k
        res["records"].append({"what": "plonk.verify_batch", "k": k, "gates": n, "median_ms": med * 1e3,
                               "min_ms": best * 1e3, "proofs_per_s": k / med, "tampered_rejected": True})
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
