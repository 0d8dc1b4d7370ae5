"""bench.py on the device: --dump-outputs writes what the timed path computed in its last step (the oracle's
result on the same seeded workload, at the rows dump_rows picks), and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import iman_conover as oic

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, D = 500_000, 16  # more rows than a dump holds at d = 16: the sampled path


def _bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(N), "--d", str(D),
                        "--warmup", "1", "--e2e-steps", "0", "--cpu-rows", "0", "--graph-rows", "0", *args],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout)


def test_dump_outputs_holds_the_timed_result(tmp_path):
    import torch

    from bench import dump_rows, make_workload_device, target_matrix

    one = _bench("--steps", "1")
    three = _bench("--steps", "3", "--dump-outputs", str(tmp_path))
    assert one["steps"] == 1 and three["steps"] == 3
    assert three["gpu_launches"] == 3 * one["gpu_launches"] > 0
    assert [p.name for p in tmp_path.iterdir()] == ["Y.npy"]
    assert os.path.getsize(tmp_path / "Y.npy") <= 64_000_000
    got = np.load(tmp_path / "Y.npy")
    X = make_workload_device(N, D, seed=0, torch=torch).cpu().numpy()
    want = oic.iman_conover(X, target_matrix(D))[dump_rows(N, D)]
    assert got.dtype == np.float64 and got.shape == want.shape and got.shape[0] < N
    np.testing.assert_array_equal(got, want)
