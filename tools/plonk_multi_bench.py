#!/usr/bin/env python3
"""Batch PLONK proving over many circuits of one size: plonk.device_prover.prove_batch_circuits against a loop of
prove_batch (one call per circuit) and a loop of prove, for 256 proofs spread over C = 1, 4, 16, 64, 256 circuits
at n = 2^10, 2^12, 2^14 (proofs/s and kernel launches per call).  The circuits are tools/plonk_synth.random_circuit
with different seeds (different selectors and copy structure), all preprocessed against one SRS table; proof j is of
circuit j % C with that circuit's witness and its own blinds.  Every timed batch is checked: verify_batch must accept
the prove_batch_circuits batch and the per-circuit loop's proofs, each against its own circuit's preprocessed data,
and proof 0 must equal a lone prove with the same blinds.  Prints one JSON object (and writes it to --out) with the
card name and power limit read in the same run.

    python tools/plonk_multi_bench.py [--out FILE] [--logn 10,12,14] [--circuits 1,4,16,64,256] [--count 256]

The loop of prove does not depend on C: it is timed once per size, over 32 proofs of 32 different circuits.
"""
import argparse
import json
import os
import random
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from interactive_zkp_study_b200 import native  # noqa: E402
from interactive_zkp_study_b200.compat import G2, g2_from_ints  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk import device_prover as dp  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk.field import FR  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk.srs import SRS  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch  # noqa: E402
from oracle import bn254  # noqa: E402
from pairing_bench import card  # noqa: E402
import plonk_synth  # noqa: E402

R = native.R_MOD


def clock(fn):
    native.sync()
    t = time.perf_counter()
    res = fn()
    native.sync()
    return res, time.perf_counter() - t


def timed(fn, reps):
    """fn once to warm up, then reps timed calls -> (last result, times, launches of the last call)."""
    fn()
    times = []
    for _ in range(reps):
        l0 = native.launch_count()
        res, t = clock(fn)
        launches = native.launch_count() - l0
        times.append(t)
    return res, times, launches


def pdict(proof):
    return {k: ((int(v[0]), int(v[1])) if k.endswith("_comm") else int(v)) for k, v in vars(proof).items()}


def stacked(wits, order, n):
    """Three handles of len(order) * n wire values: circuit order[j]'s witness at offset j * n."""
    hs = []
    for w in range(3):
        h = native.scalars_alloc(len(order) * n)
        for j, c in enumerate(order):
            native.scalars_copy(h, j * n, wits[c][w], 0, n)
        hs.append(h)
    return hs


def pp_of(key):
    pp = type("PP", (), {})()
    pp.n, pp.omega = key.n, FR(key.omega)
    for name in dp.CIRCUIT_POLYS:
        setattr(pp, name + "_comm", key.comm[name])
    return pp


def run_size(log_n, cs, count, reps):
    n = 1 << log_n
    cmax = max(cs)
    keys, wits, tau = plonk_synth.device_setup_many([plonk_synth.random_circuit(n, 100000 * log_n + s)
                                                     for s in range(cmax)])
    pps = [pp_of(k) for k in keys]
    srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)
    rng = random.Random(log_n)
    out = {"n": n, "count": count, "circuits": []}
    nloop = min(32, cmax)
    lb = [[rng.randrange(R) for _ in range(9)] for _ in range(nloop)]
    dp.prove(keys[0], *wits[0], blinds=lb[0])
    lone, t = clock(lambda: [dp.prove(keys[j], *wits[j], blinds=lb[j]) for j in range(nloop)])
    out["loop_prove_proofs_per_s"] = nloop / t
    for C in cs:
        circuits = [j % C for j in range(count)]
        blinds = lb[:1] + [[rng.randrange(R) for _ in range(9)] for _ in range(count - 1)]
        wires = stacked(wits, circuits, n)
        proofs, times, launches = timed(lambda: dp.prove_batch_circuits(keys[:C], circuits, *wires, blinds=blinds), reps)
        for h in wires:
            h.free()
        # the same proofs by one prove_batch per circuit: circuit c's proofs are j = c, c + C, ...
        groups = [[j for j in range(count) if circuits[j] == c] for c in range(C)]
        per = [stacked(wits, [c] * len(g), n) for c, g in enumerate(groups)]
        loop, ltimes, llaunches = timed(lambda: [dp.prove_batch(keys[c], *per[c], len(g), blinds=[blinds[j] for j in g])
                                                 for c, g in enumerate(groups)], reps)
        for hs in per:
            for h in hs:
                h.free()
        items = [(p, [], pps[c]) for p, c in zip(proofs, circuits)]
        items += [(p, [], pps[c]) for c, ps in enumerate(loop) for p in ps]
        ok = verify_batch(items, srs, rng=random.Random(C)) is True
        same0 = pdict(proofs[0]) == pdict(lone[0])
        same_loop = all(pdict(p) == pdict(proofs[j]) for g, ps in zip(groups, loop) for j, p in zip(g, ps))
        if not (ok and same0 and same_loop):
            raise SystemExit("n=%d C=%d failed its check (verify %s, proof 0 %s, loop %s)" % (n, C, ok, same0, same_loop))
        best, lbest = min(times), min(ltimes)
        out["circuits"].append({
            "C": C, "chunk": dp.plan_chunk(keys[0], count, native.device_mem_info()[0], multi=True),
            "multi_s": best, "multi_s_median": statistics.median(times), "multi_proofs_per_s": count / best,
            "multi_launches": launches,
            "loop_prove_batch_s": lbest, "loop_prove_batch_proofs_per_s": count / lbest,
            "loop_prove_batch_launches": llaunches,
            "speedup_vs_loop_prove_batch": lbest / best,
            "speedup_vs_loop_prove": count / best / out["loop_prove_proofs_per_s"],
            "verified": ok, "proof0_equals_prove": same0, "loop_prove_batch_equal": same_loop})
        print(json.dumps(out["circuits"][-1]), file=sys.stderr, flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--logn", default="10,12,14")
    ap.add_argument("--circuits", default="1,4,16,64,256")
    ap.add_argument("--count", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    cs = [int(x) for x in a.circuits.split(",")]
    res = {"card": card(), "device": native.device_info()["name"], "sizes": []}
    for ln in (int(x) for x in a.logn.split(",")):
        res["sizes"].append(run_size(ln, cs, a.count, a.reps))
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
