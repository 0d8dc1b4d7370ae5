"""bench.py's contract that can be checked without a GPU: the reference arm prints exactly ONE JSON
line on stdout (anything else a library writes to file descriptor 1 goes to stderr) with the keys the
driver reads; the product arm refuses to run without the CUDA library / a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--ref-rows", "20000", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "iman_conover_samples_vars_per_s"
    assert line["unit"] == "samples*vars/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_dumps_the_result_of_its_last_step(tmp_path):
    import numpy as np

    from bench import dump_rows, make_workload_host, target_matrix
    from oracle import iman_conover as oic

    r = _run("--impl", "reference", "--ref-rows", "20000", "--steps", "2", "--warmup", "0",
             "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert [p.name for p in tmp_path.iterdir()] == ["Y.npy"]
    want = oic.iman_conover(make_workload_host(20000, 16, seed=0), target_matrix(16))[dump_rows(20000, 16)]
    got = np.load(tmp_path / "Y.npy")
    assert got.dtype == np.float64 and got.shape == (20000, 16)
    np.testing.assert_array_equal(got, want)


def test_dump_rows_are_a_fixed_sample_within_the_size_limit():
    import numpy as np

    from bench import DUMP_BYTES, dump_rows

    rows = dump_rows(100_000_000, 16)
    assert DUMP_BYTES <= 64_000_000 - 128 and len(rows) * 16 * 8 <= DUMP_BYTES
    assert len(rows) > 300_000 and np.all(np.diff(rows) > 0) and rows[-1] < 100_000_000
    np.testing.assert_array_equal(rows, dump_rows(100_000_000, 16))
    np.testing.assert_array_equal(dump_rows(1000, 16), np.arange(1000))


def test_steps_below_one_are_refused():
    r = _run("--impl", "reference", "--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr and r.stdout.strip() == ""


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present: the product arm would run")
    r = _run("--steps", "1", "--warmup", "0", "--rows", "1000", "--e2e-steps", "0", "--cpu-rows", "0",
             "--graph-rows", "0")
    assert r.returncode != 0
    assert r.stdout.strip() == ""  # no JSON line from a path that did not run on the device
    assert "no CUDA device" in r.stderr or "PblError" in r.stderr or "missing" in r.stderr
