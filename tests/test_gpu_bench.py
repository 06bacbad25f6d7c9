"""-m gpu: bench.py --dump-outputs writes the result of the last timed step, and --steps sets how many steps are
timed (the scalar vector of the last step depends on it)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import bn254

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_holds_the_last_timed_msm(native, tmp_path):
    import bench
    log_n, steps, warmup = 12, 3, 3
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--log-n", str(log_n), "--steps", str(steps),
           "--warmup", str(warmup), "--strong-log-n", "0", "--no-extras", "--no-cpu", "--dump-outputs", str(tmp_path)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["verified"] is True
    got = np.load(tmp_path / "g1_msm.npy")
    assert got.dtype == np.float64 and got.shape == (2, 8)
    x, y = (sum(int(v) << (32 * j) for j, v in enumerate(row)) for row in got)
    # step i uses scalar vector i mod 4; the last timed step is step warmup + steps - 1
    n = 1 << log_n
    s = native.scalars_generate(bench.SEED_POINTS, n)
    k = native.scalars_generate(bench.SEED_SCALARS + 0x1000 * ((warmup + steps - 1) % 4), n)
    want = bn254.g1_mul(bn254.G1, native.fr_dot_dev(k, 0, s, 0, n))
    s.free()
    k.free()
    assert (x, y) == want
