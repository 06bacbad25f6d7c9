#!/usr/bin/env python3
"""Cost of binding PLONK proofs to public inputs: plonk.device_prover.prove_batch at n = 2^12 gates with 256 proofs
per batch for l = 0, 1, 64, 1024 public inputs (proofs/s, the l > 0 runs alternated with l = 0 runs in one process),
verify_batch(bind_public_inputs=True) at k = 64 and 1024 proofs, and the PI-evaluation entry
(zkp_plonk_pi_eval_many_dev) alone.  l = 0 proves tools/plonk_synth.chain_circuit, l > 0 public_chain_circuit: the
same number of gates, so the same MSM sizes.  Every timed batch is checked: verify_batch must accept it (with its
public inputs bound) and proof 0 must equal a lone prove.  Prints one JSON object (and writes it to --out) with the
card name and power limit read in the same run.

    python tools/plonk_public_bench.py [--out FILE] [--ells 0,1,64,1024] [--reps 5]

The batch holds WITNESSES distinct witnesses (and input rows), repeated, each proof with its own blinds.
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
WITNESSES = 4
LOG_N, COUNT = 12, 256


def clock(fn):
    native.sync()
    t = time.perf_counter()
    res = fn()
    native.sync()
    return res, time.perf_counter() - t


def pdict(proof):
    return {k: ((int(v[0]), int(v[1])) if k.endswith("_comm") else int(v)) for k, v in vars(proof).items()}


def load(xs):
    return native.scalars_load(native.fr_vec_bytes(xs), len(xs))


class Case:
    """Key, COUNT-proof batch inputs and verifier data for one number of public inputs."""

    def __init__(self, ell):
        n = 1 << LOG_N
        self.ell, self.n = ell, n
        make = (lambda seed: plonk_synth.public_chain_circuit(n, ell, seed)) if ell else \
            (lambda seed: plonk_synth.chain_circuit(n, seed))
        self.key, _, tau = plonk_synth.device_setup(make(LOG_N))
        circs = [make(1000 + j) for j in range(WITNESSES)]
        self.pubs = [c.get("public_inputs", []) for c in circs]
        self.wires = [load([x for j in range(COUNT) for x in circs[j % WITNESSES][k]]) for k in "abc"]
        self.pub = load([x for j in range(COUNT) for x in self.pubs[j % WITNESSES]]) if ell else None
        self.single = [load(circs[0][k]) for k in "abc"]
        rng = random.Random(ell)
        self.blinds = [[rng.randrange(R) for _ in range(9)] for _ in range(COUNT)]
        self.pp = type("PP", (), {})()
        self.pp.n, self.pp.omega, self.pp.num_public_inputs = n, FR(self.key.omega), ell
        for name in dp.CIRCUIT_POLYS:
            setattr(self.pp, name + "_comm", self.key.comm[name])
        self.srs = SRS([], [G2, g2_from_ints(bn254.g2_mul(bn254.G2, tau))], n + 5)

    def prove_batch(self, count=COUNT):
        return dp.prove_batch(self.key, *self.wires, count, blinds=self.blinds[:count], public_inputs=self.pub)

    def items(self, proofs):
        return [(p, self.pubs[j % WITNESSES], self.pp) for j, p in enumerate(proofs)]


def prove_rates(cases, reps):
    """proofs/s of every case, the cases alternated rep by rep; each batch checked once."""
    times = {c.ell: [] for c in cases}
    launches = {}
    for c in cases:                                     # warm-up: workspaces, twiddles, power tables; and the checks
        proofs = c.prove_batch()
        lone = dp.prove(c.key, *c.single, blinds=c.blinds[0], public_inputs=c.pubs[0])
        ok = verify_batch(c.items(proofs), c.srs, rng=random.Random(c.ell), bind_public_inputs=True) is True
        if not (ok and pdict(proofs[0]) == pdict(lone)):
            raise SystemExit("l=%d: batch failed its check (verify %s)" % (c.ell, ok))
    for _ in range(reps):
        for c in cases:
            l0 = native.launch_count()
            _, t = clock(c.prove_batch)
            launches[c.ell] = native.launch_count() - l0
            times[c.ell].append(t)
    base = min(times[0]) if 0 in times else None
    out = []
    for c in cases:
        best = min(times[c.ell])
        row = {"ell": c.ell, "count": COUNT, "s_best": best, "s_median": statistics.median(times[c.ell]),
               "s_all": times[c.ell], "proofs_per_s": COUNT / best, "launches": launches[c.ell],
               "chunk": dp.plan_chunk(c.key, COUNT, native.device_mem_info()[0])}
        if base:
            row["rate_vs_ell0"] = base / best
        out.append(row)
    return out


def verify_rates(case, ks, reps):
    out = []
    proofs = case.prove_batch()
    for k in ks:
        reps_k = (k + COUNT - 1) // COUNT
        items = (case.items(proofs) * reps_k)[:k]
        verify_batch(items, case.srs, rng=random.Random(k), bind_public_inputs=True)
        ts = []
        for _ in range(reps):
            ok, t = clock(lambda: verify_batch(items, case.srs, rng=random.Random(k), bind_public_inputs=True))
            if ok is not True:
                raise SystemExit("verify_batch refused k=%d" % k)
            ts.append(t)
        unbound, t_plain = clock(lambda: verify_batch(items, case.srs, rng=random.Random(k)))
        out.append({"k": k, "ell": case.ell, "s_best": min(ts), "s_all": ts, "proofs_per_s": k / min(ts),
                    "s_reference_protocol": t_plain, "reference_protocol_accepts": unbound})
    return out


def pi_eval_rates(ells, count, iters):
    n = 1 << LOG_N
    out = []
    rng = random.Random(5)
    for ell in ells:
        h = load([rng.randrange(R) for _ in range(count * ell)])
        zetas = [rng.randrange(R) for _ in range(count)]
        w = int(dp.get_root_of_unity(n))
        native.plonk_pi_eval_many_dev(h, 0, ell, ell, n, w, zetas)
        _, t = clock(lambda: [native.plonk_pi_eval_many_dev(h, 0, ell, ell, n, w, zetas) for _ in range(iters)])
        out.append({"ell": ell, "count": count, "ms_per_call": 1e3 * t / iters, "terms": count * ell})
        h.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--ells", default="0,1,64,1024")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    ells = [int(x) for x in a.ells.split(",")]
    res = {"card": card(), "device": native.device_info()["name"], "n": 1 << LOG_N, "witnesses_per_batch": WITNESSES}
    cases = [Case(ell) for ell in ells]
    res["prove_batch"] = prove_rates(cases, a.reps)
    print(json.dumps(res["prove_batch"]), file=sys.stderr, flush=True)
    vcase = next((c for c in cases if c.ell == 64), cases[-1])
    res["verify_batch_bound"] = verify_rates(vcase, (64, 1024), a.reps)
    res["pi_eval"] = pi_eval_rates([1, 64, 1024], COUNT, 20)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
