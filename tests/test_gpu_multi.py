"""-m gpu: the multi-GPU entry points of the C ABI (zkp_comm_*, zkp_g1_msm_multi, zkp_g2_msm_multi), verified
at sizes the CPU cannot reach through the device-side identity  sum_i k_i (s_i G) == <k, s> G
(zkp_fr_dot_dev; SURVEY 8d/8e).

The communicator of the calling process is a one-rank NCCL world (the driver's GPU tier has one GPU):
local MSM -> ncclAllGather -> fold runs through exactly the code the 8-GPU runs use.  When two or more
GPUs are visible, a two-process world is exercised as well (one process per GPU, TCP rendezvous)."""
import os
import random
import socket
import subprocess
import sys

import pytest

from oracle import bn254, synthetic
from tests.msm_groups import Group

pytestmark = pytest.mark.gpu
R = bn254.R
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.fixture(scope="module")
def comm(native):
    from interactive_zkp_study_b200 import sharded
    c = sharded.Communicator(0, 1)
    yield c
    c.close()


def _known_dlog_table(native, n, seed_pts=0x5EED0002, seed_sc=0x5EED0001):
    s_h = native.scalars_generate(seed_pts, n)
    k_h = native.scalars_generate(seed_sc, n)
    table = native.g1_fixed_base_mul_dev(native.g1_bytes(bn254.G1), s_h, n)
    return table, s_h, k_h


def test_fr_dot_matches_python(native):
    rng = random.Random(11)
    for n in (1, 2, 255, 256, 257, 5000):
        a = [rng.randrange(R) for _ in range(n)]
        b = [rng.randrange(R) for _ in range(n)]
        a[0] = R - 1
        ha = native.scalars_load(native.fr_vec_bytes(a), n)
        hb = native.scalars_load(native.fr_vec_bytes(b), n)
        assert native.fr_dot_dev(ha, 0, hb, 0, n) == sum(x * y for x, y in zip(a, b)) % R
        if n > 2:
            assert native.fr_dot_dev(ha, 1, hb, 2, n - 2) == sum(x * y for x, y in zip(a[1:], b[2:])) % R
    assert native.fr_dot_dev(ha, 0, hb, 0, 0) == 0
    with pytest.raises(native.ZkpB200Error):
        native.fr_dot_dev(ha, 1, hb, 0, 5000)


def test_fr_dot_matches_synthetic_streams(native):
    n = 1 << 16
    s_h = native.scalars_generate(0x5EED0002, n)
    k_h = native.scalars_generate(0x5EED0001, n)
    s = synthetic.scalars(0x5EED0002, n)
    k = synthetic.scalars(0x5EED0001, n)
    assert native.fr_dot_dev(k_h, 0, s_h, 0, n) == sum(a * b for a, b in zip(k, s)) % R


def test_comm_world1_and_errors(native, comm):
    info = native.comm_info()
    assert (info["rank"], info["world"]) == (0, 1) and info["nccl_version"] >= 20000
    native.comm_barrier()
    with pytest.raises(native.ZkpB200Error):
        native.comm_init(0, 1, bytes(128))            # a communicator already exists
    with pytest.raises(ValueError):
        native.comm_init(0, 1, bytes(5))


def test_msm_multi_small_matches_oracle(native, comm):
    """One-rank world: the sharded entry point (device and host scalars, plain and precomputed tables, a
    sub-range, an all-zero vector, n = 0) returns the oracle's affine point."""
    from interactive_zkp_study_b200 import sharded
    rng = random.Random(91)
    n = 300
    base = [bn254.g1_mul(bn254.G1, rng.randrange(1, R)) for _ in range(3)]
    pts, acc = [], base[0]
    for i in range(n):
        acc = bn254.g1_add(acc, base[i % 3])
        pts.append(acc)
    scalars = [rng.randrange(R) for _ in range(n)]
    want = bn254.g1_msm(pts, scalars)
    table = native.g1_table_load(native.g1_vec_bytes(pts), n)
    sc = native.scalars_load(native.fr_vec_bytes(scalars), n)
    zero = native.scalars_alloc(n)
    for pre in (0, 9):
        if pre:
            native.table_precompute(table, pre)
        assert sharded.g1_msm_sharded(comm, table, sc, n) == want
        assert sharded.g1_msm_sharded(comm, table, native.fr_vec_bytes(scalars), n) == want
        assert native.g1_msm_multi(table, 40, sc, 10, 200) == bn254.g1_msm(pts[40:240], scalars[10:210])
        assert native.g1_msm_multi(table, 0, zero, 0, n) is None
        assert native.g1_msm_multi(table, 0, sc, 0, 0) is None
    with pytest.raises(native.ZkpB200Error):
        native.g1_msm_multi(table, 200, sc, 0, 200)


def test_g2_msm_multi_matches_oracle(native, comm):
    rng = random.Random(92)
    q = [bn254.g2_mul(bn254.G2, rng.randrange(1, 1 << 64)) for _ in range(12)]
    s2 = [rng.randrange(R) for _ in q]
    table = native.g2_table_load(native.g2_vec_bytes(q), len(q))
    sc = native.scalars_load(native.fr_vec_bytes(s2), len(q))
    assert native.g2_msm_multi(table, 0, sc, 0, len(q)) == bn254.g2_msm(q, s2)


def test_msm_multi_2p22_device_verified(native, comm):
    """partial -> all-gather -> combine at 2^22 points on the window-precomputed table; the expected point
    comes from the device dot product <k, s> and ONE oracle scalar multiplication."""
    n = 1 << 22
    table, s_h, k_h = _known_dlog_table(native, n)
    native.table_precompute(table)
    got = native.g1_msm_multi(table, 0, k_h, 0, n)
    assert got == bn254.g1_mul(bn254.G1, native.fr_dot_dev(k_h, 0, s_h, 0, n))
    # two "shards" of the same table folded by hand == the collective's answer
    half = n // 2
    parts = native.g1_msm_dev_partial(table, 0, k_h, 0, half) + native.g1_msm_dev_partial(table, half, k_h, half, half)
    assert native.g1_combine_partials(parts, 2) == got


@pytest.mark.parametrize("log_n,pre_c", [(17, 17), (18, 20), (20, 0), (20, 20)])
def test_large_msm_device_verified(native, log_n, pre_c):
    """Whole-table and offset sub-range MSMs at sizes the CPU cannot reach: result == <k, s> G with the dot
    product taken on the device, on a precomputed table (pre_c) or a plain one (pre_c = 0)."""
    n = 1 << log_n
    table, s_h, k_h = _known_dlog_table(native, n, 0x5EED0002 + log_n, 0x5EED0001 + log_n)
    if pre_c:
        native.table_precompute(table, pre_c)
    assert native.g1_msm_dev(table, 0, k_h, 0, n) == bn254.g1_mul(bn254.G1, native.fr_dot_dev(k_h, 0, s_h, 0, n))
    m = n // 2 + 3
    assert native.g1_msm_dev(table, 7, k_h, 5, m) == bn254.g1_mul(bn254.G1, native.fr_dot_dev(k_h, 5, s_h, 7, m))
    assert native.msm_set_option("window_bits", 0) is None
    with pytest.raises(native.ZkpB200Error):
        native.msm_set_option("no such option", 1)


def test_skewed_scalars_at_2p17(native):
    _skewed_scalars_at_2p17(native, "g1")


def test_g2_skewed_scalars_at_2p17(native):
    _skewed_scalars_at_2p17(native, "g2")


def _skewed_scalars_at_2p17(native, group):
    """Skewed digit distributions at a size where buckets are cut into many tasks: all scalars equal (every
    window's digits land in one bucket), half of them zero, tiny scalars (only the lowest window used), r - 1; on a
    plain and on a window-precomputed table.  Then all points equal under all scalars equal: every task's partial sum
    is 64 P, so the block-per-bucket fold adds equal sums (P + P) at every level of its tree."""
    n = 1 << 17
    grp = Group(native, group)
    s_h = native.scalars_generate(0x5EED0102, n)
    spot = {i: native.fr_vec_from_bytes(native.scalars_download(s_h, i, 1))[0] for i in (0, n - 1)}
    table = grp.table_dev(s_h, n, spot)
    rng = random.Random(4)
    k0 = rng.randrange(R)
    cases = {
        "all equal": [k0] * n,
        "half zero": [rng.randrange(R) if i & 1 else 0 for i in range(n)],
        "tiny": [rng.randrange(1, 1000) for _ in range(n)],
        "r - 1": [R - 1] * n,
    }
    same_h = native.scalars_load(native.fr_vec_bytes([k0] * n), n)
    same = grp.table_dev(same_h, n, {0: k0, n - 1: k0})      # every entry k0 * G
    for pre in (0, 17):
        if pre:
            native.table_precompute(table, pre)
            native.table_precompute(same, pre)
        for name, k in cases.items():
            k_h = native.scalars_load(native.fr_vec_bytes(k), n)
            want = grp.mul(native.fr_dot_dev(k_h, 0, s_h, 0, n))
            assert grp.msm_dev(table, 0, k_h, 0, n) == want, (name, pre)
            k_h.free()
        # all points equal, all scalars equal: n k0^2 * G
        assert grp.msm_dev(same, 0, same_h, 0, n) == grp.mul(n * k0 * k0), ("all points equal", pre)


def test_groth16_prove_sharded_equals_single_gpu(native, comm):
    """device_prover.prove_sharded (three MSMs through zkp_g1/g2_msm_multi on range-sharded CRS tables) returns
    the proof of device_prover.prove on the unsharded key; k = 2^10 constraints, random coefficient vectors."""
    from interactive_zkp_study_b200.zkp.groth16 import device_prover as dp
    rng = random.Random(31)
    k = 1 << 10
    mp = k - 2
    alpha, beta, delta, x = (rng.randrange(1, R) for _ in range(4))
    Z = native.scalars_generate(0x5EED0300, k + 1)
    native.scalars_upload(Z, k, native.fe_bytes(1), 1)
    zx = native.fr_poly_eval_dev(Z, 0, k + 1, x)
    priv = [rng.randrange(R) for _ in range(mp)]
    uA, uB, uC = (native.scalars_generate(0x5EED0100 + i, k) for i in range(3))
    rx = native.scalars_generate(0x5EED0200, mp)
    r, s = rng.randrange(R), rng.randrange(R)
    key = dp.setup_from_toxic(k, alpha, beta, delta, x, zx, priv)
    skey = dp.setup_from_toxic_sharded(comm, k, alpha, beta, delta, x, zx, priv)
    assert (skey.rA, skey.rB, skey.rC) == ((0, k + 2), (0, k + 2), (0, 3 * k))
    want = dp.prove(key, uA, uB, uC, Z, rx, r, s)
    got = dp.prove_sharded(comm, skey, uA, uB, uC, Z, rx, r, s)
    enc = lambda P: (native.g1_bytes(P[0]), native.g2_bytes(P[1]), native.g1_bytes(P[2]))
    assert enc(got) == enc(want)


def test_plonk_prove_with_sharded_srs_equals_single_gpu(native, comm):
    """PLONK device prover with the SRS held as a row range and every commitment a collective MSM: same proof
    as the unsharded prover for equal blinding scalars (n = 2^10 gates)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import plonk_synth
    from interactive_zkp_study_b200.zkp.plonk import device_prover as dp
    circ = plonk_synth.chain_circuit(1 << 10, seed=5)
    key, wit, _ = plonk_synth.device_setup(circ)
    skey, swit, _ = plonk_synth.device_setup(circ, comm=comm)
    assert skey.srs_range == (0, (1 << 10) + 6) and skey.ranks is comm
    assert {k: skey.comm[k] for k in dp.CIRCUIT_POLYS} == {k: key.comm[k] for k in dp.CIRCUIT_POLYS}
    blinds = list(range(101, 110))
    want = dp.prove(key, *wit, blinds=blinds)
    got = dp.prove(skey, *swit, blinds=blinds)
    flat = lambda pr: {k: (native.g1_bytes(v) if k.endswith("_comm") else int(v)) for k, v in vars(pr).items()}
    assert flat(got) == flat(want)


_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
rank, world, port, log_n = (int(x) for x in sys.argv[1:5])
os.environ["ZKP_B200_DEVICE"] = str(rank)
from interactive_zkp_study_b200 import native as nat, sharded
from oracle import bn254
comm = sharded.Communicator(rank, world, addr="127.0.0.1", port=port)
total = (1 << log_n) + 5
start, count = sharded.shard_range(total, rank, world)
M = (1 << 64) - 1
s_h = nat.scalars_generate((0x5EED0002 + 64 * start) & M, count)
k_h = nat.scalars_generate((0x5EED0001 + 64 * start) & M, count)
table = nat.g1_fixed_base_mul_dev(nat.g1_bytes(bn254.G1), s_h, count)
nat.table_precompute(table)
got = sharded.g1_msm_sharded(comm, table, k_h, count)
host = sharded.g1_msm_sharded(comm, table, nat.scalars_download(k_h, 0, count), count)
print("RESULT", rank, nat.fr_dot_dev(k_h, 0, s_h, 0, count), got[0], got[1], int(host == got), flush=True)
comm.barrier()
comm.close()
'''


def test_two_process_world_when_two_gpus_are_visible(native):
    """One process per GPU, TCP rendezvous, NCCL all-gather inside the library: both ranks return the same
    point, equal to (sum of the ranks' device dot products) * G."""
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        gpus = len([l for l in out.splitlines() if l.startswith("GPU ")])
    except Exception:
        gpus = 1
    if gpus < 2:
        pytest.skip("one GPU visible: the two-process world needs two (the one-rank world above covers the code path)")
    port = _free_port()
    code = _WORKER % {"root": ROOT}
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r), "2", str(port), "20"], stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = [p.communicate(timeout=600) for p in procs]
    for p, (so, se) in zip(procs, outs):
        assert p.returncode == 0, se[-2000:]
    rows = [[int(v) for v in line.split()[1:]] for so, _ in outs for line in so.splitlines() if line.startswith("RESULT")]
    assert len(rows) == 2
    dot = sum(r[1] for r in rows) % R
    want = bn254.g1_mul(bn254.G1, dot)
    for r in rows:
        assert (r[2], r[3]) == want and r[4] == 1
