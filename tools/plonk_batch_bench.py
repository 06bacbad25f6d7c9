#!/usr/bin/env python3
"""Batch PLONK proving throughput: plonk.device_prover.prove_batch against a loop of device_prover.prove on the chain
circuit of tools/plonk_synth.py, at n = 2^10 .. 2^16 gates (proofs/s; 256 proofs per batch, and 16 and 1024 at
2^12), kernel launches per call, and the time of each round of one prove_batch pass (each round ends in a device
synchronise).  Every timed batch is checked: verify_batch must accept it and proof 0 must equal a lone prove with the
same blinds.  Prints one JSON object (and writes it to --out) with the card name and power limit read in the same run.

    python tools/plonk_batch_bench.py [--out FILE] [--logn 10,12,14,16] [--counts 256] [--extra-counts 16,1024]

The batch holds WITNESSES distinct witnesses of the circuit (chain_circuit with different seeds), repeated, each
proof with its own blinds.  The sequential loop is timed over 16 proofs: its rate does not depend on the batch size.
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
from interactive_zkp_study_b200.compat import G2, g2_from_ints  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk import device_prover as dp  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk.field import FR  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk.srs import SRS  # noqa: E402
from interactive_zkp_study_b200.zkp.plonk.verifier import verify_batch  # noqa: E402
from oracle import bn254  # noqa: E402
from pairing_bench import card  # noqa: E402
import plonk_synth  # noqa: E402

R = native.R_MOD
WITNESSES = 4


def clock(fn):
    native.sync()
    t = time.perf_counter()
    res = fn()
    native.sync()
    return res, time.perf_counter() - t


def pdict(proof):
    return {k: ((int(v[0]), int(v[1])) if k.endswith("_comm") else int(v)) for k, v in vars(proof).items()}


def batch_wires(base, n, count):
    """count * n wire values per wire: witness j % WITNESSES at offset j * n."""
    hs = []
    for src in base:
        h = native.scalars_alloc(count * n)
        for j in range(count):
            native.scalars_copy(h, j * n, src, (j % WITNESSES) * n, n)
        hs.append(h)
    return hs


def setup(log_n):
    n = 1 << log_n
    key, _, tau = plonk_synth.device_setup(plonk_synth.chain_circuit(n, seed=log_n))
    circs = [plonk_synth.chain_circuit(n, seed=1000 * log_n + j) for j in range(WITNESSES)]
    base = [native.scalars_load(native.fr_vec_bytes([x for c in circs for x in c[k]]), WITNESSES * n) for k in "abc"]
    pp = type("PP", (), {})()
    pp.n, pp.omega = n, FR(key.omega)
    for name in dp.CIRCUIT_POLYS:
        setattr(pp, name + "_comm", key.comm[name])
    srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)
    return key, base, pp, srs


def run_size(log_n, counts, reps):
    n = 1 << log_n
    key, base, pp, srs = setup(log_n)
    rng = random.Random(log_n)
    out = {"n": n, "batches": []}
    single = [[native.scalars_alloc(n) for _ in range(3)] for _ in range(WITNESSES)]
    for i in range(WITNESSES):
        for w in range(3):
            native.scalars_copy(single[i][w], 0, base[w], i * n, n)
    nloop = 16
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(nloop)]
    dp.prove(key, *single[0], blinds=blinds[0])
    lone, t = clock(lambda: [dp.prove(key, *single[j % WITNESSES], blinds=blinds[j]) for j in range(nloop)])
    out["loop_proofs_per_s"] = nloop / t
    for count in counts:
        wires = batch_wires(base, n, count)
        bbl = blinds[:1] + [[rng.randrange(R) for _ in range(9)] for _ in range(count - 1)]
        dp.prove_batch(key, *wires, count, blinds=bbl)      # warm-up: workspaces, twiddles, power tables
        times = []
        for _ in range(reps):
            l0 = native.launch_count()
            proofs, t = clock(lambda: dp.prove_batch(key, *wires, count, blinds=bbl))
            launches = native.launch_count() - l0
            times.append(t)
        ok = verify_batch([(p, [], pp) for p in proofs], srs, rng=random.Random(count)) is True
        same0 = pdict(proofs[0]) == pdict(lone[0])
        if not (ok and same0):
            raise SystemExit("batch n=%d count=%d failed its check (verify %s, proof 0 %s)" % (n, count, ok, same0))
        best = min(times)
        out["batches"].append({"count": count, "chunk": dp.plan_chunk(key, count, native.device_mem_info()[0]),
                               "s": best, "proofs_per_s": count / best,
                               "speedup_vs_loop": count / best / out["loop_proofs_per_s"], "launches": launches,
                               "verified": ok, "proof0_equals_prove": same0})
        for h in wires:
            h.free()
    return out, key, base


def rounds(key, base, count):
    """One prove_batch pass cut at its rounds: prove_batch itself, with a device synchronise and a clock reading
    around each of its many-MSMs and after round 4's evaluations (wrappers around the native calls it makes)."""
    n = key.n
    wires = batch_wires(base, n, count)
    rng = random.Random(3)
    blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(count)]
    # a round ends with its commitment group (rounds 1, 2, 3, 5) or its evaluations (round 4)
    marks = []
    orig = native.msm_dev_many
    orig_eval = native.fr_poly_eval_many_dev
    msm = []

    def msm_mark(*a, **kw):
        native.sync()
        t = time.perf_counter()
        r = orig(*a, **kw)
        native.sync()
        marks.append(time.perf_counter())
        msm.append(marks[-1] - t)
        return r

    def eval_mark(*a, **kw):
        r = orig_eval(*a, **kw)
        native.sync()
        if len(a[0]) > 1:                                # round 4's six evaluations (round 5 evaluates r alone)
            marks.append(time.perf_counter())
        return r

    res = None
    native.msm_dev_many, native.fr_poly_eval_many_dev = msm_mark, eval_mark
    try:
        for _ in range(2):                                  # the second pass is the timed one
            marks.clear()
            msm.clear()
            native.sync()
            t0 = time.perf_counter()
            dp.prove_batch(key, *wires, count, blinds=blinds, chunk=count)
            t = [t0] + marks
            res = {"round1": t[1] - t[0], "round2": t[2] - t[1], "round3": t[3] - t[2], "round4": t[4] - t[3],
                   "round5": t[5] - t[4], "total": t[5] - t[0]}
            # the commitment group of each round (rounds 1, 2, 3, 5; round 4 commits nothing)
            res.update({"round%d_msm" % k: v for k, v in zip((1, 2, 3, 5), msm)})
    finally:
        native.msm_dev_many, native.fr_poly_eval_many_dev = orig, orig_eval
    for h in wires:
        h.free()
    return {k: 1e3 * v for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--logn", default="10,12,14,16")
    ap.add_argument("--counts", default="256")
    ap.add_argument("--extra-counts", default="16,1024", help="further batch sizes at n = 2^12")
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    counts = [int(x) for x in a.counts.split(",")]
    extra = [int(x) for x in a.extra_counts.split(",") if x]
    res = {"card": card(), "device": native.device_info()["name"], "witnesses_per_batch": WITNESSES, "sizes": []}
    for ln in (int(x) for x in a.logn.split(",")):
        cs = sorted(set(counts + (extra if ln == 12 else [])))
        out, key, base = run_size(ln, cs, a.reps)
        if ln == 12:
            res["rounds_ms_n4096_count256"] = rounds(key, base, 256)
        res["sizes"].append(out)
        print(json.dumps(out), file=sys.stderr, flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
