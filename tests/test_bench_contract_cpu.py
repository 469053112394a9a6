"""bench.py's reference arm runs without a GPU: check the JSON contract the driver parses."""
import json
import os
import subprocess
import sys

from conftest import REPO

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "impl"]


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py")] + args, capture_output=True, text=True, env=e,
                       timeout=600, cwd=REPO)
    assert p.returncode == 0, p.stderr[-2000:]
    return p.stdout.strip().splitlines()


def test_reference_arm_prints_one_json_line():
    lines = _run(["--impl", "reference", "--n", "20000", "--steps", "2", "--warmup", "1", "--cpu-rows", "256"])
    assert len(lines) == 1
    r = json.loads(lines[0])
    for k in REQUIRED:
        assert k in r, k
    assert r["impl"] == "reference" and r["unit"] == "Gpairs/s" and r["higher_is_better"] is True
    assert r["metric"] == "gaussian_kernel_product_gpairs_per_s" and r["value"] > 0 and r["steps"] == 2
    from kernel_matrix_benchmarks_b200.harness import bootstrap

    # the reference's own class when its tree is staged (baseline/_ref) or mounted, the NumPy port otherwise
    assert r["cpu_baseline"]["kind"] == ("port" if bootstrap.find_reference() is None else "reference")
    assert r["cpu_baseline"]["cores"] >= 1 and r["cpu_baseline"]["value"] == r["value"]
    assert r["e2e"] == {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert r["config"]["N"] == 20000 and "workload" in r["config"] and r["vs_baseline"] is None
    assert r["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun only rank 0 runs and prints the reference arm."""
    lines = _run(["--impl", "reference", "--n", "20000", "--steps", "1", "--warmup", "1", "--gpus", "2"],
                 env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert lines == []


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=REPO)
    assert p.returncode == 2 and "--steps" in p.stderr


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones_the_same_way(tmp_path):
    import numpy as np
    import pytest

    import bench

    big = np.arange(2_000_000, dtype=np.float64).reshape(-1, 2)   # 32 MB, over the per-array limit
    small = np.linspace(0, 1, 10, dtype=np.float32).reshape(10, 1)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert np.array_equal(a, b) and a.dtype == np.float64 and a.shape[1] == 2
    assert 0 < a.nbytes <= bench.DUMP_ARRAY_BYTES and a.shape[0] >= bench.DUMP_ARRAY_BYTES // 16 - 1
    rows = a[:, 0] / 2   # whole rows of the original, in order
    assert np.array_equal(rows, np.round(rows)) and np.all(np.diff(rows) > 0) and np.array_equal(a[:, 1], a[:, 0] + 1)
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small)
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path / "c"), {"ints": np.arange(4)})
