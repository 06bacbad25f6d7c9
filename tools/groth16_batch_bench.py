#!/usr/bin/env python3
"""Batch Groth16 proving throughput: qap_device.prove_batch against a loop of qap_device.prove on the synthetic circuit
of tools/qap_large.py, at k = 2^10 .. 2^16 constraints and 1 .. 1024 proofs per batch (proofs/s); the many-MSM alone
against zkp_g1_msm_dev_batch over the same scalar vectors (Mpts/s); kernel launches per prove_batch call; and the
time of each stage of one device_prover.prove_batch pass.  Every timed batch is checked: verify_batch must accept it
and proof 0 must equal a lone prove.  Prints one JSON object (and writes it to --out).

    python tools/groth16_batch_bench.py [--out FILE] [--logk 10,12,14,16] [--counts 1,16,256,1024]

The batch holds WITNESSES distinct satisfying witnesses (different public inputs), repeated, each proof with its own
random r and s.  The sequential loop is timed over min(count, 16) proofs: its rate does not depend on the batch size.
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
from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp  # noqa: E402
from interactive_zkp_study_b200.zkp.groth16 import qap_device as qd  # noqa: E402
from interactive_zkp_study_b200.zkp.groth16.verifying import verify_batch  # noqa: E402
from pairing_bench import card  # noqa: E402
from qap_large import circuit  # noqa: E402

R = native.R_MOD
WITNESSES = 4


def witnesses(ra, rb, count, seed):
    rng = random.Random(seed)
    out = []
    for _ in range(count):
        w = [1, rng.randrange(2, 1 << 20)]
        for a, b in zip(ra, rb):
            w.append(sum(v * w[i] for i, v in a.items()) * sum(v * w[i] for i, v in b.items()) % R)
        out.append(w)
    return out


def clock(fn):
    native.sync()
    t = time.perf_counter()
    res = fn()
    native.sync()
    return res, time.perf_counter() - t


def ints(prf):
    A, B, C = prf
    return (int(A[0]), int(A[1])), tuple(tuple(int(v) for v in c.coeffs) for c in B), (int(C[0]), int(C[1]))


def run_size(log_k, counts, reps):
    k = 1 << log_k
    m = k + 2
    ra, rb, rc, _ = circuit(k, 99)
    dev = qd.DeviceR1CS(qd.SparseR1CS.from_rows(k, m, ra, rb, rc))
    rng = random.Random(log_k)
    keys = qd.setup(dev, *(rng.randrange(1, R) for _ in range(5)), lcm=True, precompute=True)
    base = witnesses(ra, rb, WITNESSES, log_k)
    wbase = native.scalars_load(native.fr_vec_bytes([x for w in base for x in w]), WITNESSES * m)
    vk = (keys.sigma1_1, keys.sigma1_3, keys.sigma2_1)
    out = {"k": k, "batches": []}
    # the sequential loop: proofs/s of qap_device.prove
    wl = [native.scalars_alloc(m) for _ in range(WITNESSES)]
    for i, h in enumerate(wl):
        native.scalars_copy(h, 0, wbase, i * m, m)
    nloop = 16
    rs = [rng.randrange(R) for _ in range(nloop)]
    ss = [rng.randrange(R) for _ in range(nloop)]
    qd.prove(keys, dev, wl[0], rs[0], ss[0])
    lone, t = clock(lambda: [qd.prove(keys, dev, wl[j % WITNESSES], rs[j], ss[j]) for j in range(nloop)])
    out["loop_proofs_per_s"] = nloop / t
    for count in counts:
        W = native.scalars_alloc(count * m)
        for j in range(count):
            native.scalars_copy(W, j * m, wbase, (j % WITNESSES) * m, m)
        brs = rs[:1] + [rng.randrange(R) for _ in range(count - 1)]
        bss = ss[:1] + [rng.randrange(R) for _ in range(count - 1)]
        qd.prove_batch(keys, dev, W, brs, bss)            # warm-up: workspaces, twiddles, divisor cache
        times = []
        for _ in range(reps):
            l0 = native.launch_count()
            proofs, t = clock(lambda: qd.prove_batch(keys, dev, W, brs, bss))
            launches = native.launch_count() - l0
            times.append(t)
        pubs = [[(i, base[j % WITNESSES][i]) for i in keys.pub_idx] for j in range(count)]
        ok = verify_batch(proofs, *vk, pubs, rng=random.Random(count)) is True
        same0 = ints(proofs[0]) == ints(lone[0])
        if not (ok and same0):
            raise SystemExit("batch k=%d count=%d failed its check (verify %s, proof 0 %s)" % (k, count, ok, same0))
        best = min(times)
        out["batches"].append({"count": count, "chunk": dp.plan_chunk(keys.device_key, count, native.device_mem_info()[0]),
                               "s": best, "proofs_per_s": count / best, "speedup_vs_loop": count / best / out["loop_proofs_per_s"],
                               "launches": launches, "verified": ok, "proof0_equals_prove": same0})
        W.free()
    return out, keys, dev, wbase


def stages(keys, dev, wbase, count):
    """One device_prover.prove_batch pass cut into its stages (each ends in a device synchronise)."""
    key, k, mp = keys.device_key, keys.device_key.k, keys.device_key.m_priv
    m = dev.m
    W = native.scalars_alloc(count * m)
    for j in range(count):
        native.scalars_copy(W, j * m, wbase, (j % WITNESSES) * m, m)
    rng = random.Random(3)
    rs = [rng.randrange(R) for _ in range(count)]
    ss = [rng.randrange(R) for _ in range(count)]
    res = {}
    for _ in range(2):                                  # the second round is the timed one
        (uA, uB, uC), res["witness_polys"] = clock(lambda: qd.witness_polys_batch(dev, W, count, keys.lcm))
        rx = native.scalars_alloc(count * mp)
        _, res["private_wires"] = clock(lambda: native.sparse_matvec_many_dev(qd._selection_matrix(keys, m), W, rx, count))
        hq, res["quotient"] = clock(lambda: native.groth16_quotient_batch_dev(uA, uB, uC, k, count, keys.Z, k + 1))
        (scA, scB, scC), res["scalars"] = clock(lambda: native.groth16_batch_scalars_dev(uA, uB, hq, rx, k, mp, rs, ss))
        _, res["msm_A"] = clock(lambda: native.msm_dev_many(key.TA, 0, k + 2, count, scA))
        _, res["msm_B_g2"] = clock(lambda: native.msm_dev_many(key.TB2, 0, k + 2, count, scB))
        _, res["msm_C"] = clock(lambda: native.msm_dev_many(key.TC, 0, dp.tc_rows(k, mp), count, scC))
    # the many-MSM against the two-stream pipeline of independent MSMs, same scalar vectors, table TA
    n = k + 2
    _, t_many = clock(lambda: native.msm_dev_many(key.TA, 0, n, count, scA))
    items = [(scA, j * n, 0, n) for j in range(count)]
    native.g1_msm_dev_batch(key.TA, items)
    _, t_batch = clock(lambda: native.g1_msm_dev_batch(key.TA, items))
    if native.msm_dev_many(key.TA, 0, n, count, scA) != native.g1_msm_dev_batch(key.TA, items):
        raise SystemExit("many-MSM and msm_dev_batch disagree")
    msm = {"points": n, "count": count, "window_bits": getattr(key.TA, "pre_c", 0),
           "many_ms": 1e3 * t_many, "many_mpts_per_s": count * n / t_many / 1e6,
           "dev_batch_ms": 1e3 * t_batch, "dev_batch_mpts_per_s": count * n / t_batch / 1e6}
    return {key_: 1e3 * v for key_, v in res.items()}, msm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--logk", default="10,12,14,16")
    ap.add_argument("--counts", default="1,16,256,1024")
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    counts = [int(x) for x in a.counts.split(",")]
    res = {"card": card(), "device": native.device_info()["name"], "witnesses_per_batch": WITNESSES, "sizes": []}
    for lk in (int(x) for x in a.logk.split(",")):
        out, keys, dev, wbase = run_size(lk, counts, a.reps)
        if lk == 12:
            st, msm = stages(keys, dev, wbase, 256)
            res["stages_ms_k4096_count256"] = st
            res["many_msm_vs_dev_batch"] = msm
        res["sizes"].append(out)
        print(json.dumps(out), file=sys.stderr, flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
