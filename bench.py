#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native prover hot path.

Metric (BASELINE.json): BN254 G1 MSM throughput, Mpts/s, 2^20 synthetic random points / scalars per
GPU (configs[1]); weak scaling over N GPUs (each rank owns a contiguous point range of the same
size; the library gathers one 128-byte partial sum per rank over NCCL and folds it -- SURVEY.md 8e).
Every line also carries `strong_2p26`: BASELINE configs[4], 2^26 points in total split over the N ranks
by point range (the >= 6x at 8 GPUs target), verified on the device at every N.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log-n 20] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `value` is timed with CUDA events on the library's stream with
points and scalars resident in HBM; `e2e` is the same MSM through the reference-facing C-ABI call
with the scalars in pinned HOST memory (H2D inside the timed region, affine result read back);
`roofline` is the bucket-accumulation kernel against the IMAD.WIDE peak measured live on the same
GPU (MEASURED_PEAKS.json carries no integer peak); `cpu_baseline` is the oracle's restatement of the
reference's CPU path (commit loop, fft, hxr, proof_a) timed on this box's host cores on bounded samples.
Every MSM that is timed is first checked against  sum_i k_i (s_i G) == <k, s> G  with the dot product
computed on the device (zkp_fr_dot_dev) and one oracle scalar multiplication: verification is on at
every size and every N.

torch appears here only as launcher plumbing (barrier and max-over-ranks of the timings, as the bench
contract prescribes); the product path -- including the NCCL exchange -- is inside libzkp_b200.so.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bn254_g1_msm_throughput"
UNIT = "Mpts/s"
SEED_SCALARS = 0x5EED0001
SEED_POINTS = 0x5EED0002
MACS_PER_FP_MUL = 136                      # 8-limb CIOS: 8*(8+1+8) limb-MACs   (SURVEY.md 8d)
MACS_PER_FP_SQR = 108                      # dedicated squaring: 36 + 72 (ff.cuh sqr_inline)
MACS_PER_MULSUB = 2 * 64 + 72              # a b - c d with one reduction (fp2.cuh fp_mulsub_outlined): 200 instead of 272
# XYZZ mixed addition 8M + 2S as the accumulate kernel executes it: 6 products, 2 squarings, and the Y coordinate
# R (Q - X3) - Y1 PPP as one lazily reduced pair = 1232 limb-MACs (1304 with every product reduced on its own)
MADD_MACS = 6 * MACS_PER_FP_MUL + 2 * MACS_PER_FP_SQR + MACS_PER_MULSUB
MADD_MACS_PLAIN = 8 * MACS_PER_FP_MUL + 2 * MACS_PER_FP_SQR
XYZZ_ADD_MACS = 12 * MACS_PER_FP_MUL + MACS_PER_MULSUB     # full addition in the compact flavour (squarings as products)


def BUCKETS_TOTAL(pre_c):
    """Buckets the reduction walks: one set of 2^(c-1) on a window-precomputed table, 16 sets of 2^15 on a plain one."""
    return (1 << (pre_c - 1)) if pre_c else 16 * (1 << 15)
MODEL_ACC_MACS_PER_POINT = 160 * MACS_PER_FP_MUL  # SURVEY model: 16 windows x 10 Fp-mul (XYZZ mixed add) = 21 760
M64 = (1 << 64) - 1


def windows_for(c):
    return (255 + c - 1) // c


def msm_macs_per_point(n):
    return MODEL_ACC_MACS_PER_POINT + 14 * MACS_PER_FP_MUL * (1 << 20) / n  # + bucket reduction, amortised


# ------------------------------------------------------------------ clocks sampling
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                power.append(float(r[3]))
            except ValueError:
                continue
            for name, val in zip(names, r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ reference arm (CPU)
def _ref_points(n):
    """n distinct valid G1 points, cheaply: P_0 = k*G, P_{i+1} = P_i + Q (one affine add each)."""
    from oracle import bn254
    p = bn254.g1_mul(bn254.G1, 0x1234567)
    q = bn254.g1_mul(bn254.G1, 0x7654321)
    out = []
    for _ in range(n):
        out.append(p)
        p = bn254.g1_add(p, q)
    return out


def _ref_worker(args):
    from oracle import bn254
    pts, scalars = args
    return bn254.g1_msm(pts, scalars)


def run_reference(args):
    """The reference's CPU path for this metric: kzg.commit's loop of affine double-and-add scalar
    multiplications (/root/reference/zkp/plonk/kzg.py:59-67 over py_ecc), as restated by
    oracle/bn254.g1_msm (py_ecc is not installable in this image: SURVEY F3), on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import bn254, synthetic
    cores = os.cpu_count() or 1
    steps, warmup = args.steps, args.warmup
    # size a step so the whole run takes about 60-90 s: ~13 ms per point per core
    per_point_s = 0.013
    budget_s = 75.0
    sample = int(budget_s * cores / ((steps + warmup) * per_point_s))
    sample = max(cores * 4, min(sample, 1 << 14))
    sample -= sample % cores
    pts = _ref_points(sample)
    scal = synthetic.scalars(SEED_SCALARS, sample)
    chunk = sample // cores
    jobs = [(pts[i * chunk:(i + 1) * chunk], scal[i * chunk:(i + 1) * chunk]) for i in range(cores)]
    with mp.Pool(cores) as pool:
        def step():
            parts = pool.map(_ref_worker, jobs)
            acc = None
            for p in parts:
                acc = bn254.g1_add(acc, p)
            return acc
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = step()
        dt = time.perf_counter() - t0
    assert bn254.g1_is_on_curve(res)
    value = sample * steps / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32x8 (254-bit modular integers)", "data": "synthetic",
        "config": {"workload": "BN254 G1 MSM, 2^%d synthetic points per GPU (configs[1])" % args.log_n,
                   "step": "bounded sample of %d points of that workload" % sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d points/step, oracle/bn254.g1_msm = commit()-style affine double-and-add "
                                   "(reference kzg.py:59-67 on py_ecc semantics; py_ecc itself is not installable here)" % sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ CPU legs of the metric (oracle = port of the reference)
def cpu_baseline(nat, table, scalars_handle):
    """Oracle (port of the reference's commit loop) on one host core, bounded sample; also a parity
    check of the GPU result on that sample.  Further legs: the reference's fft, hxr and proof_a (BASELINE.md 4)."""
    from oracle import bn254
    sample = 2048                        # ~10 s of single-core CPU work at ~5 ms per point
    raw = nat.table_download(table, 0, sample)
    pts = [nat.g1_from_bytes(raw[64 * i:64 * i + 64]) for i in range(sample)]
    scal = nat.fr_vec_from_bytes(nat.scalars_download(scalars_handle, 0, sample))
    t0 = time.perf_counter()
    want = bn254.g1_msm(pts, scal)
    dt = time.perf_counter() - t0
    got = nat.g1_msm_dev(table, 0, scalars_handle, 0, sample)
    if got != want:
        raise SystemExit("PARITY FAILURE: GPU MSM differs from the oracle on the cpu_baseline sample")
    out = {"value": sample / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port", "seconds": dt,
           "sample": "first %d points/scalars of the workload, oracle/bn254.g1_msm (reference kzg.commit loop, "
                     "affine double-and-add, py_ecc semantics); GPU result on the same sample is bit-identical" % sample}
    try:
        out["legs"] = cpu_legs(nat)
    except Exception as e:  # never lose the headline line
        out["legs_error"] = repr(e)
    return out


def cpu_legs(nat):
    """fft 2^14 (polynomial.py:292-341), hxr at numGates 64 (poly_utils.py:116-125), proof_a at 12 x 12
    (proving.py:23-33): oracle/ref_path restatements on one core, each compared with the GPU result."""
    import random
    from oracle import bn254, ref_path
    R = bn254.R
    rng = random.Random(41)
    legs = {}
    # ---- fft
    log_n = 14
    n = 1 << log_n
    vals = [rng.randrange(R) for _ in range(n)]
    w = ref_path.get_root_of_unity(n)
    t0 = time.perf_counter()
    want = ref_path.fft(vals, w)
    dt = time.perf_counter() - t0
    got = nat.fr_vec_from_bytes(nat.fr_ntt(nat.fr_vec_bytes(vals), log_n, w))
    legs["fft"] = {"n": n, "seconds": dt, "value": n / dt / 1e6, "unit": "Melem/s", "cores": 1, "kind": "port",
                   "reference": "zkp/plonk/polynomial.py:292-341 (recursive radix-2)", "gpu_bit_identical": got == want}
    # ---- hxr: numGates k, numWires m
    k, m = 64, 66
    Ax, Bx, Cx = ([[rng.randrange(R) for _ in range(k)] for _ in range(m)] for _ in range(3))
    Rv = [rng.randrange(R) for _ in range(m)]
    Z = [1]
    for j in range(1, k + 1):            # (x-1)...(x-k), qap_creator_lcm.py:128-135
        Z = ref_path.poly_mul(Z, [(-j) % R, 1])
    t0 = time.perf_counter()
    hx, rem = ref_path.hxr(Ax, Bx, Cx, Z, Rv)
    dt = time.perf_counter() - t0
    from interactive_zkp_study_b200.zkp.groth16 import poly_utils
    FR = poly_utils.FR
    t1 = time.perf_counter()
    ghx, grem = poly_utils.hxr([[FR(v) for v in row] for row in Ax], [[FR(v) for v in row] for row in Bx],
                               [[FR(v) for v in row] for row in Cx], [FR(v) for v in Z], [FR(v) for v in Rv])
    gdt = time.perf_counter() - t1
    legs["hxr"] = {"num_gates": k, "num_wires": m, "seconds": dt, "cores": 1, "kind": "port",
                   "reference": "zkp/groth16/poly_utils.py:116-125 (mat-vec + schoolbook product + long division)",
                   "gpu_mirror_seconds_incl_python_lists": gdt,
                   "gpu_bit_identical": [int(v) for v in ghx] == [v % R for v in hx] and [int(v) for v in grem] == [v % R for v in rem]}
    # ---- proof_a: the numWires x numGates loop of scalar multiplications
    k, m = 12, 12
    x = rng.randrange(1, R)
    sigma1_2 = [bn254.g1_mul(bn254.G1, pow(x, j, R)) for j in range(k)]
    sigma1_1 = [bn254.g1_mul(bn254.G1, rng.randrange(1, R)) for _ in range(3)]
    Ax = [[rng.randrange(R) for _ in range(k)] for _ in range(m)]
    Rv = [rng.randrange(R) for _ in range(m)]
    r = rng.randrange(R)
    t0 = time.perf_counter()
    want = ref_path.proof_a(sigma1_1, sigma1_2, Ax, Rv, r)
    dt = time.perf_counter() - t0
    from interactive_zkp_study_b200.zkp.groth16 import proving
    from interactive_zkp_study_b200.compat import FQ
    pt = lambda p: (FQ(p[0]), FQ(p[1]))
    t1 = time.perf_counter()
    got = proving.proof_a([pt(p) for p in sigma1_1], [pt(p) for p in sigma1_2], [[proving.FR(v) for v in row] for row in Ax],
                          [proving.FR(v) for v in Rv], r)
    gdt = time.perf_counter() - t1
    legs["proof_a"] = {"num_gates": k, "num_wires": m, "seconds": dt, "scalar_muls": m * k + m + 1, "cores": 1, "kind": "port",
                       "reference": "zkp/groth16/proving.py:23-33", "gpu_mirror_seconds_incl_table_upload": gdt,
                       "gpu_bit_identical": (int(got[0]), int(got[1])) == want}
    return legs


# ------------------------------------------------------------------ sub-records (other rows of the metric)
def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json"
        except Exception:
            pass
    return 6650.0, "fallback of B200_PROFILING.md (no MEASURED_PEAKS.json)"


def profile_traffic(kernel):
    """dram bytes per launch of `kernel` from the committed ncu capture of this round, or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(path)).get(kernel, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def ntt_record(nat, log_n, peak_tmacs):
    """Forward Fr NTT of 2^log_n resident elements: achieved integer and HBM rates (SURVEY 8d)."""
    from interactive_zkp_study_b200 import _lib
    n = 1 << log_n
    omega = pow(5, (nat.R_MOD - 1) >> log_n, nat.R_MOD)
    h = nat.scalars_generate(0x5EED0004, n)
    wb = nat.fe_bytes(omega)

    def go():
        nat.check(_lib.lib().zkp_fr_ntt_dev(h.handle, 0, log_n, nat.buf(wb), 0, None))
    for _ in range(3):
        go()
    best = 1e9
    for _ in range(10):
        nat.timer_start()
        go()
        best = min(best, nat.timer_stop())
    h.free()
    macs = 68.0 * n * log_n
    hbm, src = measured_hbm_peak()
    ach = macs / best / 1e9
    return {"n": n, "ms": best, "gelem_per_s": n / best / 1e6,
            "roofline": {"bound": "imad", "kernel": "ntt_pass_kernel", "achieved": ach, "peak": peak_tmacs,
                         "unit": "T limb-MAC/s", "frac": ach / peak_tmacs, "traffic": profile_traffic("ntt_pass_kernel"),
                         "algorithmic_macs": macs,
                         "hbm_view": {"algorithmic_bytes": 64.0 * n, "achieved_gbs": 64.0 * n / best / 1e6,
                                      "frac": 64.0 * n / best / 1e6 / hbm, "peak_gbs": hbm, "peak_source": src}},
            "note": "68*n*log2(n) limb-MACs ((n/2) log2 n products of 136) and 64 B/element (one read + one write); "
                    "the 254-bit NTT is integer bound (10.6 MAC/B needed)"}


def g2_record(nat, log_n, peak_tmacs):
    """G2 MSM of 2^log_n points on its window-precomputed table: the accumulation kernel's integer rate."""
    from oracle import bn254
    n = 1 << log_n
    s_h = nat.scalars_generate(0x5EED0003, n)
    k_h = nat.scalars_generate(SEED_SCALARS + 0x33, n)
    table = nat.g2_fixed_base_mul_dev(nat.g2_bytes(bn254.G2), s_h, n)
    c = nat.table_precompute(table)
    got = nat.g2_msm_dev(table, 0, k_h, 0, n)
    ok = got == bn254.g2_mul(bn254.G2, nat.fr_dot_dev(k_h, 0, s_h, 0, n))
    nat.msm_profile(True)
    best, acc = 1e9, 0.0
    for _ in range(4):
        nat.timer_start()
        nat.g2_msm_dev(table, 0, k_h, 0, n)
        ms = nat.timer_stop()
        if ms < best:
            best, acc = ms, nat.msm_last_profile("accumulate")
    nat.msm_profile(False)
    for h in (s_h, k_h, table):
        h.free()
    W = windows_for(c)
    # Fp2 product = Karatsuba on unreduced products, one reduction per component: 3 x 64 + 2 x 72 = 336 limb-MACs;
    # Fp2 squaring = 2 Fp products = 272: mixed addition 8 M2 + 2 S2 = 3232 limb-MACs
    madd2 = 8 * (3 * 64 + 2 * 72) + 2 * (2 * MACS_PER_FP_MUL)
    macs = n * W * madd2
    ach = macs / (acc * 1e-6) / 1e12
    return {"n": n, "ms": best, "value": n / best / 1e3, "unit": UNIT, "window_bits": c, "verified": bool(ok),
            "roofline": {"bound": "imad", "kernel": "msm_accumulate_kernel<Fp2>", "achieved": ach, "peak": peak_tmacs,
                         "unit": "T limb-MAC/s", "frac": ach / peak_tmacs, "kernel_ms": acc * 1e-3,
                         "traffic": profile_traffic("msm_accumulate_kernel<Fp2>"), "algorithmic_macs_per_launch": macs,
                         "algorithmic_note": "%d windows x (8 Fp2 products x 336 + 2 Fp2 squarings x 272 = 3232 limb-MAC per mixed addition); "
                                             "with every Fp2 product as 3 Fp products of 136 (SURVEY 8d, round 1) the figure is x %.3f" % (W, 28 * 136 / madd2)}}


def groth16_record(log_k, peak_tmacs, comm=None):
    """Second half of the BASELINE metric: Groth16 prove ms at 2^log_k constraints (config 3), with the
    SURVEY 8d work model as its roofline.  With a communicator the proof's MSMs are sharded over its ranks
    (every rank calls this)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import groth16_large
    res = groth16_large.run(log_k, 3, verify=True, quiet=True, comm=comm)
    if peak_tmacs is None:
        return res
    k = 1 << log_k
    # SURVEY 8d: 4 G1 MSMs + 1 G2 MSM at the model's per-point cost + ~1e10 for the quotient
    macs = 4 * k * msm_macs_per_point(k) + k * 3 * msm_macs_per_point(k) + 1.0e10 * k / (1 << 20)
    ach = macs / (res["prove_ms"] * 1e-3) / 1e12
    res["verified"] = bool(res.pop("verified_against_discrete_logs"))
    res["roofline"] = {"bound": "imad", "achieved": ach, "peak": peak_tmacs * res["n_gpus"], "unit": "T limb-MAC/s",
                       "frac": ach / (peak_tmacs * res["n_gpus"]),
                       "algorithmic_macs": macs,
                       "algorithmic_note": "SURVEY 8d model: 4 G1 MSMs + 1 G2 MSM (x3) of 2^%d points at 23 664 MAC/pt + 1e10 for the quotient; "
                                           "the prover here folds them into 2 G1 MSMs (k+2 and 3k points) + 1 G2 MSM started before the quotient" % log_k}
    return res


def dump_g1_point(out_dir, name, point):
    """Writes an affine G1 result as out_dir/<name>.npy: float64 of shape (2, 8), the 32-bit limbs of x and y,
    least significant first (every limb is exact in float64).  The point at infinity is all zeros, as in the
    library's byte encoding."""
    import numpy as np
    x, y = point if point is not None else (0, 0)
    limbs = [[(v >> (32 * j)) & 0xFFFFFFFF for j in range(8)] for v in (x, y)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), np.array(limbs, dtype=np.float64))


# ------------------------------------------------------------------ our arm (GPU)
def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = torch = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    os.environ.setdefault("ZKP_B200_DEVICE", str(local_rank))
    from interactive_zkp_study_b200 import native as nat
    from interactive_zkp_study_b200 import sharded
    from oracle import bn254
    info = nat.device_info()
    numa_node = sharded.bind_to_gpu_numa_node() if world > 1 else None   # before any pinned allocation

    def barrier():
        nat.sync()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks_int(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    comm = None
    if world > 1:
        # the library's own NCCL communicator; its 128-byte id rides on the launcher's process group
        def exchange(mine):
            box = [mine]
            dist.broadcast_object_list(box, src=0)
            return box[0]
        comm = sharded.Communicator(rank, world, exchange_id=exchange)

    def stream(seed, first, count):
        # element i of the global stream == element (i - first) of a stream with a shifted counter
        return nat.scalars_generate((seed + 64 * first) & M64, count)

    def expected_point(k, s, count):
        """(sum over ALL ranks of <k, s>) * G on rank 0: device dot products + one oracle scalar multiplication."""
        local = nat.fr_dot_dev(k, 0, s, 0, count)
        if dist is None:
            return bn254.g1_mul(bn254.G1, local)
        box = [None] * world
        dist.all_gather_object(box, local)
        return bn254.g1_mul(bn254.G1, sum(box) % bn254.R) if rank == 0 else None

    def msm_resident(table, k, count):
        if world == 1:
            return nat.g1_msm_dev(table, 0, k, 0, count)
        return nat.g1_msm_multi(table, 0, k, 0, count)

    def msm_from_host(table, addr, count):
        if world == 1:
            return nat.g1_msm_table(table, 0, addr, count)
        return nat.g1_msm_multi_table(table, 0, addr, count)

    n = 1 << args.log_n                 # points per GPU
    steps, warmup = args.steps, args.warmup
    G1 = nat.g1_bytes((1, 2))
    # this rank's point range [rank*n, (rank+1)*n): P_i = s_i * G with s_i from the synthetic stream
    # (known discrete logs -> O(1)-host check of any MSM), scalars k_i from a second stream
    s_h = stream(SEED_POINTS, rank * n, n)
    table = nat.g1_fixed_base_mul_dev(G1, s_h, n)
    plain_ms = None
    pre_c = 0
    precompute_s = 0.0
    if not args.plain:
        # first the plain-table number (no precomputation), for the record
        kk = stream(SEED_SCALARS + 0x9000, rank * n, n)
        for _ in range(3):
            nat.g1_msm_dev_partial(table, 0, kk, 0, n)
        nat.sync()
        nat.timer_start()
        for _ in range(5):
            nat.g1_msm_dev_partial(table, 0, kk, 0, n)
        plain_ms = nat.timer_stop() / 5
        kk.free()
        # static table -> window-precomputed layout, once (like loading the SRS)
        t0 = time.perf_counter()
        pre_c = nat.table_precompute(table)     # window width picked by the library for this table size
        precompute_s = time.perf_counter() - t0
    W_actual = windows_for(pre_c if pre_c else 16)
    n_vec = 4                            # rotate scalar vectors so no step reuses cached digits
    k_h = [stream(SEED_SCALARS + 0x1000 * v, rank * n, n) for v in range(n_vec)]

    def step_resident(i):
        return msm_resident(table, k_h[i % n_vec], n)

    # ---- correctness of the exact workload before timing (size-independent check, SURVEY 8d): every vector
    verified = None
    if args.verify:
        verified = True
        for v in range(n_vec):
            want = expected_point(k_h[v], s_h, n)
            got = step_resident(v)
            if rank == 0 and got != want:
                raise SystemExit("PARITY FAILURE: 2^%d x %d MSM != <k, s> * G (vector %d)" % (args.log_n, world, v))

    # clocks are sampled from here to the end of the timed region: the region itself lasts < 0.1 s and
    # nvidia-smi delivers a sample every ~50-100 ms, so the integer-peak microbenchmarks (also a
    # saturating integer load) and the warm-up steps are included to get a meaningful median
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    peak = {}
    if rank == 0:
        peak = {"imad_wide_u32": nat.imad_peak(0), "imad_lo": nat.imad_peak(1), "imad_hi_u32": nat.imad_peak(2),
                "fp_mul_chain": nat.imad_peak(3), "mad_wide_u32_register_factors": nat.imad_peak(4)}

    # ---- resident-input timing (value)
    for i in range(warmup):
        step_resident(i)
    nat.msm_profile(True)
    barrier()
    launches0 = nat.launch_count()
    acc_us = 0.0
    msm_us = 0.0
    nat.timer_start()
    for i in range(steps):
        last = step_resident(warmup + i)
        acc_us += nat.msm_last_profile("accumulate")
        msm_us += nat.msm_last_profile(None)
    ms = nat.timer_stop()
    barrier()
    launches = nat.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else {}
    ms = max_over_ranks(ms)
    launches = sum_over_ranks_int(launches)
    total_points = n * world
    value = total_points * steps / (ms * 1e-3) / 1e6

    nat.msm_profile(False)
    if args.dump_outputs and rank == 0:
        dump_g1_point(args.dump_outputs, "g1_msm", last)

    # for the record: the same MSMs submitted as ONE pipelined batch call (two streams: the tail of MSM k
    # overlaps the accumulation of MSM k+1), the call shape of a prover that commits in groups
    pipelined = None
    if world == 1:
        items = [(k_h[i % n_vec], 0, 0, n) for i in range(min(steps, 8))]
        nat.g1_msm_dev_batch(table, items)
        nat.timer_start()
        nat.g1_msm_dev_batch(table, items)
        bms = nat.timer_stop()
        pipelined = {"msms_per_call": len(items), "ms_per_msm": bms / len(items),
                     "value": n * len(items) / (bms * 1e-3) / 1e6, "unit": UNIT, "call": "zkp_g1_msm_dev_batch"}

    # ---- end-to-end timing: scalars in pinned host memory, H2D inside, affine result read back
    pinned = nat.PinnedBuffer(32 * n)
    pinned.write(nat.scalars_download(k_h[0], 0, n))
    e2e_want = step_resident(0)
    for _ in range(max(1, warmup // 2)):
        got = msm_from_host(table, pinned.addr, n)
    if got != e2e_want:
        raise SystemExit("PARITY FAILURE: host-scalar MSM differs from the resident one")
    barrier()
    nat.timer_start()
    for _ in range(steps):
        msm_from_host(table, pinned.addr, n)
    e2e_ms = nat.timer_stop()
    barrier()
    e2e_ms = max_over_ranks(e2e_ms)
    e2e_value = total_points * steps / (e2e_ms * 1e-3) / 1e6
    pinned.free()

    base = cpu_baseline(nat, table, k_h[0]) if (rank == 0 and world == 1 and args.cpu) else None
    for h in [table, s_h] + k_h:
        h.free()

    # ---- BASELINE configs[4]: 2^26 points in total, sharded by point range over the ranks (strong scaling)
    strong = None
    if args.strong_log_n:
        total_s = 1 << args.strong_log_n
        start, count = sharded.shard_range(total_s, rank, world)
        ss = stream(SEED_POINTS, start, count)
        tab = nat.g1_fixed_base_mul_dev(G1, ss, count)
        t0 = time.perf_counter()
        c_s = nat.table_precompute(tab)
        pre_s = time.perf_counter() - t0
        kv = [stream(SEED_SCALARS + 0x1000 * v, start, count) for v in range(2)]
        ok = True
        for v in range(2):
            want = expected_point(kv[v], ss, count)
            got = msm_resident(tab, kv[v], count)
            if rank == 0 and got != want:
                ok = False
        if rank == 0 and not ok:
            raise SystemExit("PARITY FAILURE: sharded 2^%d MSM over %d GPUs != <k, s> * G" % (args.strong_log_n, world))
        s_steps, s_warm = 4, 2
        for i in range(s_warm):
            msm_resident(tab, kv[i % 2], count)
        barrier()
        nat.timer_start()
        for i in range(s_steps):
            msm_resident(tab, kv[i % 2], count)
        sms = max_over_ranks(nat.timer_stop())
        barrier()
        # end to end: this rank's scalar shard from pinned host memory
        pin = nat.PinnedBuffer(32 * count)
        step_bytes = 1 << 28
        for off in range(0, 32 * count, step_bytes):
            m = min(step_bytes, 32 * count - off) // 32
            pin.write(nat.scalars_download(kv[0], off // 32, m), off)
        msm_from_host(tab, pin.addr, count)
        barrier()
        nat.timer_start()
        for _ in range(2):
            msm_from_host(tab, pin.addr, count)
        s_e2e = max_over_ranks(nat.timer_stop()) / 2
        barrier()
        pin.free()
        strong = {"workload": "BN254 G1 MSM, 2^%d points in total, sharded by contiguous point range (configs[4])" % args.strong_log_n,
                  "total_points": total_s, "points_per_gpu": count, "n_gpus": world, "scaling": "strong",
                  "ms_per_step": sms / s_steps, "value": total_s / (sms / s_steps) / 1e3, "unit": UNIT, "steps": s_steps,
                  "warmup": s_warm, "verified": True,
                  "verification": "result == (sum over ranks of <k, s> on the device) * G for both scalar vectors",
                  "e2e": {"ms_per_step": s_e2e, "value": total_s / s_e2e / 1e3, "unit": UNIT,
                          "h2d_bytes_per_step": 32 * total_s, "d2h_bytes_per_step": 64 * world},
                  "table": "window-precomputed, c = %d, %.1f GiB per GPU, built once in %.1f s" % (
                      c_s, windows_for(c_s) * count * 64 / 2**30, pre_s)}
        for h in [tab, ss] + kv:
            h.free()

    g16_sharded = None
    if comm is not None and args.extras and args.log_n <= 20 and os.environ.get("ZKP_BENCH_G16_SHARDED", "1") == "1":
        try:
            g16_sharded = groth16_record(args.log_n, None, comm=comm)
            g16_sharded["prove_ms"] = max_over_ranks(g16_sharded["prove_ms"])
        except Exception as e:  # never lose the headline line
            g16_sharded = {"error": repr(e)}
    plonk_sharded = None
    if comm is not None and args.extras and args.log_n <= 20 and os.environ.get("ZKP_BENCH_PLONK_SHARDED", "1") == "1":
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import plonk_large
            plonk_sharded = plonk_large.run(args.log_n, 3, verify=(rank == 0), quiet=True, comm=comm)
            plonk_sharded["prove_ms"] = max_over_ranks(plonk_sharded["prove_ms"])
        except Exception as e:  # never lose the headline line
            plonk_sharded = {"error": repr(e)}
    if comm is not None:
        comm.close()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (bucket accumulation) against the measured IMAD.WIDE peak
    peak_gmacs = peak["imad_wide_u32"]
    peak_t = peak_gmacs / 1e3
    acc_s = acc_us / steps * 1e-6
    acc_macs = n * W_actual * MADD_MACS          # the limb-MACs this launch really executes (squarings at 108, Y3 lazily reduced)
    achieved = acc_macs / acc_s / 1e12
    roofline = {
        "bound": "imad", "kernel": "msm_accumulate_kernel<Fp>", "achieved": achieved, "peak": peak_t,
        "unit": "T limb-MAC/s (one IMAD.WIDE.U32 = 32x32+64->64)", "frac": achieved / peak_t,
        "traffic": profile_traffic("msm_accumulate_kernel<Fp>"),
        "algorithmic_macs_per_launch": acc_macs,
        "algorithmic_note": "%d windows x (6 products x 136 + 2 squarings x 108 + the Y coordinate as one lazily reduced pair of "
                            "products, 200 = %d limb-MAC executed per XYZZ mixed addition) per point; with every product reduced on "
                            "its own (1304, round-2 records before this change) the figure is x %.4f, with squarings also counted as "
                            "products (SURVEY 8d: 1360) x %.4f"
                            % (W_actual, MADD_MACS, MADD_MACS_PLAIN / MADD_MACS, 1360.0 / MADD_MACS),
        "frac_survey_8d_units": (n * W_actual * 1360.0 / acc_s / 1e12) / peak_t,
        "kernel_ms": acc_s * 1e3, "kernel_share_of_step": acc_us / max(msm_us, 1e-9),
        "kernel_timing": "CUDA events on the library stream around the accumulate launch of every timed step",
        "peak_source": "measured live on this GPU by zkp_imad_peak(0): IMAD.WIDE.U32[.X] in the carry-chain form the field "
                       "arithmetic issues (mad.lo.cc / madc.hi.cc pairs), 4 independent 4-lane chains per thread, 1024 threads per SM, "
                       "no loop-invariant operand (checked in SASS); MEASURED_PEAKS.json has no integer peak",
        "peaks_gmacs": peak,
        "whole_msm": {"macs_per_point_model": msm_macs_per_point(n),
                      "frac": (n * msm_macs_per_point(n) / (msm_us / steps * 1e-6) / 1e12) / peak_t,
                      # the limb-MACs the whole MSM really executes: the mixed additions above + two full XYZZ additions
                      # (12 products + the lazily reduced pair = 1832) per bucket of the reduction
                      "macs_per_point_executed": W_actual * MADD_MACS + 2.0 * XYZZ_ADD_MACS * BUCKETS_TOTAL(pre_c) / n,
                      "frac_executed": ((n * W_actual * MADD_MACS + 2.0 * XYZZ_ADD_MACS * BUCKETS_TOTAL(pre_c))
                                        / (msm_us / steps * 1e-6) / 1e12) / peak_t,
                      "note": "SURVEY 8d model (16 windows + amortised bucket reduction, squarings as products) over the whole MSM time"},
        "hbm_view": {"algorithmic_bytes_per_launch": n * W_actual * 68,
                     "achieved_gbs": n * W_actual * 68 / acc_s / 1e9,
                     "note": "windows x (64 B point gather + 4 B index) per point: far below the HBM roof, the kernel is integer bound"},
    }
    sub = {}
    if world == 1 and args.extras and args.log_n <= 20:
        for name, fn in (("groth16_prove", lambda: groth16_record(args.log_n, peak_t)),
                         ("g2_msm", lambda: g2_record(nat, args.log_n, peak_t)),
                         ("fr_ntt", lambda: ntt_record(nat, args.log_n, peak_t))):
            try:
                sub[name] = fn()
            except Exception as e:  # never lose the headline line
                sub[name + "_error"] = repr(e)
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        try:
            import plonk_large
            sub["plonk_prove"] = plonk_large.run(args.log_n, 3, verify=True, quiet=True)
        except Exception as e:
            sub["plonk_prove_error"] = repr(e)
        try:   # last: its 1.3 GB subproduct-tree cache stays resident and crowds the buffer pool of whatever follows
            import qap_large
            sub["groth16_r1cs_prove"] = qap_large.run(args.log_n, 3, quiet=True)
        except Exception as e:
            sub["groth16_r1cs_prove_error"] = repr(e)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32x8 (254-bit modular integers, Montgomery)", "data": "synthetic", "verified": verified,
        "config": {
            "workload": "BN254 G1 MSM, 2^%d synthetic points per GPU (configs[1]); P_i = s_i*G, scalars uniform in [0,r)" % args.log_n,
            "points_per_gpu": n, "total_points": total_points,
            "sharding": ("contiguous point ranges; zkp_g1_msm_multi: local Pippenger -> ncclAllGather of one 128 B XYZZ partial per rank "
                         "-> fold, on the library's stream") if world > 1 else "single GPU",
            "table": ("window-precomputed static table T[w][i] = 2^(%d w) P_i, %d windows, %.0f MiB per GPU, built once in %.0f ms "
                      "(zkp_g1_table_precompute; SRS/CRS tables are fixed per circuit)" % (pre_c, W_actual, W_actual * n * 64 / 2**20, precompute_s * 1e3))
                     if pre_c else "plain affine table, 64 B/point",
            "plain_table": None if plain_ms is None else {"ms_per_step": plain_ms, "value": n / plain_ms / 1e3, "unit": UNIT,
                                                          "note": "same MSM without the precomputed windows (16 windows + Horner), this rank only"},
            "l2": "working set (point table + scalars + 2x100 MiB pair/index arrays + bucket partials) exceeds the 126 MB L2; "
                  "a different scalar vector every step",
            "verification": "every timed scalar vector: result == (sum over ranks of <k, s>, zkp_fr_dot_dev) * G",
            "device": info["name"],
        },
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms / steps,
                "h2d_bytes_per_step": 32 * n * world, "d2h_bytes_per_step": 64 * world,
                "path": ("zkp_g1_msm_table" if world == 1 else "zkp_g1_msm_multi_table") +
                        ": device-resident point table (static SRS), scalars from pinned host memory; part-streamed "
                        "(4 point ranges growing 1.35x: range p+1 is uploaded and sorted on a side lane while range p "
                        "accumulates into the one bucket set)",
                "numa_node_of_rank0": numa_node},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": base,
        "strong_2p%d" % args.strong_log_n if args.strong_log_n else "strong": strong,
        "pipelined_batch": pipelined,
    }
    if g16_sharded is not None:
        if "error" not in g16_sharded:
            k = 1 << args.log_n
            macs = 4 * k * msm_macs_per_point(k) + k * 3 * msm_macs_per_point(k) + 1.0e10 * k / (1 << 20)
            ach = macs / (g16_sharded["prove_ms"] * 1e-3) / 1e12
            g16_sharded["verified"] = bool(g16_sharded.pop("verified_against_discrete_logs"))
            g16_sharded["roofline"] = {"bound": "imad", "achieved": ach, "peak": peak_t * world, "unit": "T limb-MAC/s",
                                       "frac": ach / (peak_t * world), "algorithmic_macs": macs,
                                       "algorithmic_note": "SURVEY 8d model (4 G1 MSMs + 1 G2 MSM x3 + quotient) against %d x the one-GPU peak" % world}
        sub["groth16_prove"] = g16_sharded
    if plonk_sharded is not None:
        sub["plonk_prove"] = plonk_sharded
    line.update(sub)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline MSM and of its e2e record (the pipelined batch takes min(steps, 8)); "
                         "the other sub-records (strong scaling, Groth16, PLONK, G2, NTT) time their own fixed counts")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=20, help="log2 of the points per GPU")
    ap.add_argument("--strong-log-n", type=int, default=26, help="log2 of the TOTAL points of the sharded sub-record (0 = skip)")
    ap.add_argument("--no-verify", dest="verify", action="store_false", help="debugging only; no committed number uses it")
    ap.add_argument("--plain", action="store_true", help="do not precompute the window table")
    ap.add_argument("--no-extras", dest="extras", action="store_false", help="skip the Groth16 / PLONK / G2 / NTT sub-records")
    ap.add_argument("--no-cpu", dest="cpu", action="store_false", help="skip the CPU baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the affine point of the last timed headline MSM to DIR/g1_msm.npy (see dump_g1_point); "
                         "the inputs depend only on the arguments, so two builds can be compared output for output. "
                         "GPU arm only: --impl reference times a different, smaller sample and is refused")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
