"""bench.py on a B200: --dump-outputs writes what the timed paths returned (needs a B200)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO

pytestmark = pytest.mark.gpu


def _bench(*args):
    p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True, timeout=900,
                       cwd=REPO)
    assert p.returncode == 0, p.stderr[-2000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


def test_steps_sets_the_number_of_timed_steps():
    """gpu_launches counts the library's launches over the timed steps, so it grows with --steps, not with --warmup."""
    one, three = (_bench("--n", "20000", "--steps", k, "--warmup", w, "--no-cpu-baseline", "--no-e2e", "--no-configs")
                  for k, w in (("1", "2"), ("3", "1")))
    assert (one["steps"], three["steps"]) == (1, 3)
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]


def test_solve_workload_honours_steps(tmp_path):
    r = _bench("--workload", "solve", "--n", "20000", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert (r["steps"], r["warmup"]) == (2, 0) and r["converged"] and r["parity"]["ok"]
    x = np.load(tmp_path / "c5.npy")
    assert x.shape == (20000, 1) and x.dtype == np.float64


def test_dump_outputs_are_the_timed_results(tmp_path):
    n = 20000
    r = _bench("--n", str(n), "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--configs", "c1",
               "--dump-outputs", str(tmp_path))
    assert r["steps"] == 3 and r["parity"]["ok"]
    assert sorted(os.listdir(tmp_path)) == ["c1.npy", "e2e_product.npy", "product.npy"]
    got, e2e, c1 = (np.load(tmp_path / f) for f in ("product.npy", "e2e_product.npy", "c1.npy"))
    assert got.shape == (n, 1) and got.dtype == np.float32
    assert e2e.shape == (n, 1) and e2e.dtype == np.float64
    assert c1.shape == (10_000, 1) and c1.dtype == np.float64

    from kernel_matrix_benchmarks_b200 import datasets
    from oracle import c_oracle

    rows = np.arange(0, n, 97)
    for name, ds, out in (("product", datasets.config_c2(n), got), ("e2e_product", datasets.config_c2(n), e2e),
                          ("c1", datasets.config_c1(), c1)):
        want = c_oracle.kernel_product("gaussian", ds.source_points, None, ds.source_signal, rows=rows[rows < ds.N])
        rel = np.linalg.norm(out[rows[rows < ds.N]] - want) / np.linalg.norm(want)
        assert rel <= 1e-5, (name, rel)
