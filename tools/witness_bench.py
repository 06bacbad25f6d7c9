#!/usr/bin/env python3
"""Witness solving on the device: zkp.witness.solve_batch against the host path it replaces (the Python witness loop,
fr_vec_bytes and the upload), in witnesses/s, on the synthetic R1CS of tools/qap_large.py and the PLONK chain of
tools/plonk_synth.py at 1 .. 1024 witnesses per call; compile time per circuit and launches per call; and end to end,
inputs to proofs, for 256 distinct witnesses at 2^12 (Groth16 and PLONK), with every batch accepted by verify_batch.
Prints one JSON object (and writes it to --out).

    python tools/witness_bench.py [--out FILE] [--logk 12,16,20] [--logn 12,16] [--counts 1,16,256,1024]

The host path is timed over 16 witnesses at 2^12, 2 at 2^16 and 1 at 2^20: its rate does not depend on the batch
size.  The first two witnesses of every device batch are compared with host witnesses.
"""
import argparse
import json
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from interactive_zkp_study_b200 import native  # noqa: E402
from interactive_zkp_study_b200.zkp import witness as wz  # noqa: E402
from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd  # noqa: E402
from pairing_bench import card  # noqa: E402
from qap_large import circuit  # noqa: E402
import plonk_synth  # noqa: E402

R = native.R_MOD


def clock(fn):
    native.sync()
    t = time.perf_counter()
    res = fn()
    native.sync()
    return res, time.perf_counter() - t


def host_r1cs(ra, rb, xs):
    """The host witness computation of tools/groth16_batch_bench.py::witnesses, for given inputs."""
    out = []
    for x in xs:
        w = [1, x]
        for a, b in zip(ra, rb):
            w.append(sum(v * w[i] for i, v in a.items()) * sum(v * w[i] for i, v in b.items()) % R)
        out.append(w)
    return out


def host_upload(rows):
    """fr_vec_bytes + upload of host witnesses: what a user of prove_batch does today."""
    return native.scalars_load(native.fr_vec_bytes([x for r in rows for x in r]), sum(len(r) for r in rows))


def vals(h, off, n):
    return native.fr_vec_from_bytes(native.scalars_download(h, off, n))


def solve_rates(prog, make_inputs, counts, host_fn, host_n, check):
    """Device witnesses/s per count (best of 3 after a warm-up), launches per call, and the host path's rate."""
    out = {"device": []}
    for count in counts:
        X = native.scalars_load(native.fr_vec_bytes(make_inputs(count)), count * prog.n_in)
        res = wz.solve_batch(prog, X, count)
        del res
        best, launches = None, None
        for _ in range(3):
            l0 = native.launch_count()
            res, t = clock(lambda: wz.solve_batch(prog, X, count))
            launches = native.launch_count() - l0
            best = t if best is None else min(best, t)
        check(res, count)
        out["device"].append({"count": count, "ms": 1e3 * best, "witnesses_per_s": count / best, "launches": launches})
        del res
        X.free()
    t0 = time.perf_counter()
    up = host_fn(host_n)
    native.sync()
    t = time.perf_counter() - t0
    up.free()
    out["host"] = {"witnesses_timed": host_n, "ms_per_witness": 1e3 * t / host_n, "witnesses_per_s": host_n / t}
    return out


def r1cs_size(log_k, counts):
    k = 1 << log_k
    ra, rb, rc, _ = circuit(k, 99)
    r1cs = qd.SparseR1CS.from_rows(k, k + 2, ra, rb, rc)
    prog, t_compile = clock(lambda: wz.compile_r1cs(r1cs, [1]))
    _, t_load = clock(prog.device)
    rng = random.Random(log_k)
    xs = [rng.randrange(2, 1 << 20) for _ in range(max(counts))]
    host_n = 16 if log_k <= 12 else 2 if log_k <= 16 else 1
    ref = host_r1cs(ra, rb, xs[:2])

    def check(W, count):
        for j in range(min(count, 2)):
            if vals(W, j * (k + 2), k + 2) != ref[j]:
                raise SystemExit("R1CS k=2^%d count=%d: witness %d differs from the host" % (log_k, count, j))

    res = solve_rates(prog, lambda c: xs[:c], [c for c in counts if c * (k + 2) * 32 < 60e9], lambda h: host_upload(host_r1cs(ra, rb, xs[:h])),
                      host_n, check)
    res.update({"circuit": "qap_large", "log_k": log_k, "steps": prog.steps, "levels": prog.levels,
                "quotient_steps": sum(prog.quotient), "compile_s": t_compile, "program_upload_s": t_load})
    return res


def plonk_size(log_n, counts):
    n = 1 << log_n
    c0 = plonk_synth.chain_circuit(n, seed=1)
    pos = [0] + [n + g for g in range(n)]
    prog, t_compile = clock(lambda: wz.compile_plonk(n, c0["sel"], c0["sigma"], pos))
    _, t_load = clock(prog.device)
    circs = {}

    def circ(j):
        if j not in circs:
            circs[j] = plonk_synth.chain_circuit(n, seed=100 + j)
        return circs[j]

    rng = random.Random(log_n)
    seeds = [rng.randrange(1 << 60) for _ in range(max(counts))]

    def inputs(count):
        # distinct inputs per witness without building count host circuits: a random a_0 and b row per witness
        rows = []
        for j in range(count):
            if j < 2:
                c = circ(j)
                rows.extend([c["a"][0]] + c["b"])
            else:
                r = random.Random(seeds[j])
                rows.extend(r.randrange(1, 1 << 60) for _ in range(n + 1))
        return rows

    def check(abc, count):
        for j in range(min(count, 2)):
            for h, key in zip(abc, "abc"):
                if vals(h, j * n, n) != circ(j)[key]:
                    raise SystemExit("PLONK n=2^%d count=%d: %s of witness %d differs from the host" % (log_n, count, key, j))

    def host(h):
        t = [plonk_synth.chain_circuit(n, seed=500 + j) for j in range(h)]
        return host_upload([c[key] for c in t for key in "abc"])

    res = solve_rates(prog, inputs, counts, host, 16 if log_n <= 12 else 2, check)
    res.update({"circuit": "plonk_synth chain", "log_n": log_n, "steps": prog.steps, "levels": prog.levels,
                "quotient_steps": sum(prog.quotient), "compile_s": t_compile, "program_upload_s": t_load,
                "host_note": "chain_circuit builds the selectors and sigma with the witness"})
    return res


def e2e_times(solve, hostw, prove):
    """Inputs to proofs: solve_batch + prove_batch against host witnesses + upload + prove_batch (after a warm-up of
    both), and each part alone; the device timings are the best of three, the host path runs once."""
    prove(solve())
    best = lambda fn: min((clock(fn) for _ in range(3)), key=lambda r: r[1])
    wd, t_solve = best(solve)
    pd, t_prove = best(lambda: prove(wd))
    _, t_dev = best(lambda: prove(solve()))
    wh, t_hostw = clock(hostw)
    _, t_host = clock(lambda: prove(hostw()))
    ph = prove(wh)
    return {"solve_batch_ms": 1e3 * t_solve, "prove_batch_ms": 1e3 * t_prove, "device_path_ms": 1e3 * t_dev,
            "host_witnesses_and_upload_ms": 1e3 * t_hostw, "host_path_ms": 1e3 * t_host,
            "speedup": t_host / t_dev, "proofs": (pd, ph)}


def e2e_groth16(count=256):
    from interactive_zkp_study_b200.zkp.groth16.verifying import verify_batch
    k = 1 << 12
    ra, rb, rc, _ = circuit(k, 99)
    r1cs = qd.SparseR1CS.from_rows(k, k + 2, ra, rb, rc)
    dev = qd.DeviceR1CS(r1cs)
    rng = random.Random(12)
    keys = qd.setup(dev, *(rng.randrange(1, R) for _ in range(5)), lcm=True, precompute=True)
    prog = wz.compile_r1cs(r1cs, [1])
    xs = [rng.randrange(2, 1 << 20) for _ in range(count)]
    rs = [rng.randrange(R) for _ in range(count)]
    ss = [rng.randrange(R) for _ in range(count)]
    X = native.scalars_load(native.fr_vec_bytes(xs), count)
    vk = (keys.sigma1_1, keys.sigma1_3, keys.sigma2_1)
    pubs = [[(0, 1), (1, x)] for x in xs]
    solve = lambda: wz.solve_batch(prog, X, count)
    hostw = lambda: host_upload(host_r1cs(ra, rb, xs))
    prove = lambda W: qd.prove_batch(keys, dev, W, rs, ss)
    res = e2e_times(solve, hostw, prove)
    pd, ph = res.pop("proofs")
    ok = verify_batch(pd, *vk, pubs, rng=random.Random(1)) is True and verify_batch(ph, *vk, pubs, rng=random.Random(2)) is True
    same = [(p[0], p[2]) for p in pd] == [(p[0], p[2]) for p in ph]
    if not (ok and same):
        raise SystemExit("Groth16 end to end: verify %s, device and host proofs equal %s" % (ok, same))
    res.update({"system": "groth16", "k": k, "count": count, "distinct_witnesses": count, "verified": ok,
                "device_and_host_proofs_equal": same})
    return res


def e2e_plonk(count=256):
    from interactive_zkp_study_b200.compat import G2, g2_from_ints
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    from interactive_zkp_study_b200.zkp.plonk.field import FR
    from interactive_zkp_study_b200.zkp.plonk.srs import SRS
    from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch
    from oracle import bn254
    n = 1 << 12
    c0 = plonk_synth.chain_circuit(n, seed=12)
    key, _, tau = plonk_synth.device_setup(c0)
    prog = wz.compile_plonk(n, c0["sel"], c0["sigma"], [0] + [n + g for g in range(n)])
    seeds = [3000 + j for j in range(count)]
    circs = [plonk_synth.chain_circuit(n, seed=s) for s in seeds]
    X = native.scalars_load(native.fr_vec_bytes([x for c in circs for x in [c["a"][0]] + c["b"]]), count * (n + 1))
    rng = random.Random(13)
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(count)]

    def hostw():
        cs = [plonk_synth.chain_circuit(n, seed=s) for s in seeds]
        return tuple(host_upload([c[k] for c in cs]) for k in "abc")

    solve = lambda: wz.solve_batch(prog, X, count)
    prove = lambda abc: dp.prove_batch(key, *abc, count, blinds=blinds)
    res = e2e_times(solve, hostw, prove)
    pd, ph = res.pop("proofs")
    pp = type("PP", (), {})()
    pp.n, pp.omega = n, FR(key.omega)
    for name in dp.CIRCUIT_POLYS:
        setattr(pp, name + "_comm", key.comm[name])
    srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)
    ok = verify_batch([(p, [], pp) for p in pd], srs, rng=random.Random(1)) is True
    same = [str(vars(p)) for p in pd] == [str(vars(p)) for p in ph]
    if not (ok and same):
        raise SystemExit("PLONK end to end: verify %s, device and host proofs equal %s" % (ok, same))
    res.update({"system": "plonk", "n": n, "count": count, "distinct_witnesses": count, "verified": ok,
                "device_and_host_proofs_equal": same,
                "host_note": "host witnesses from plonk_synth.chain_circuit, which also builds the selectors and sigma"})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--logk", default="12,16,20")
    ap.add_argument("--logn", default="12,16")
    ap.add_argument("--counts", default="1,16,256,1024")
    a = ap.parse_args()
    counts = [int(x) for x in a.counts.split(",")]
    res = {"card": card(), "device": native.device_info()["name"], "solve": [], "end_to_end": []}
    for lk in (int(x) for x in a.logk.split(",") if x):
        res["solve"].append(r1cs_size(lk, counts))
        print(json.dumps(res["solve"][-1]), file=sys.stderr, flush=True)
    for ln in (int(x) for x in a.logn.split(",") if x):
        res["solve"].append(plonk_size(ln, counts))
        print(json.dumps(res["solve"][-1]), file=sys.stderr, flush=True)
    for fn in (e2e_groth16, e2e_plonk):
        res["end_to_end"].append(fn())
        print(json.dumps(res["end_to_end"][-1]), file=sys.stderr, flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
