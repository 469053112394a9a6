"""The B200 plugin driven by the reference's own runner.run / results / metrics on a B200
(the drop-in claim of BASELINE.json's north star).  The runner tests need the reference tree (staged in baseline/_ref
or named by KMB_REFERENCE) and skip without it; the dataset tests run against the stand-in of
tests/reference_standin.py and the reference's outputs stored in tests/golden/."""
import os

import numpy as np
import pytest

from conftest import load_golden
from kernel_matrix_benchmarks_b200.harness import bootstrap
from reference_standin import standin_reference  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(bootstrap.find_reference() is None, reason="reference harness not staged")

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(dataset, task, dim, hardware="GPU", normalize_rows=False, kernel="gaussian"):
    bootstrap.activate()
    from kernel_matrix_benchmarks.datasets import get_dataset
    from kernel_matrix_benchmarks.definitions import get_definitions
    from kernel_matrix_benchmarks.plotting.utils import compute_all_metrics
    from kernel_matrix_benchmarks.results import load_all_results
    from kernel_matrix_benchmarks.runner import run

    defs = get_definitions(definition_file=os.path.join(REPO, "algos.yaml"), dimension=dim, dataset=dataset, task=task,
                           hardware=hardware, kernel=kernel, normalize_rows=normalize_rows)
    assert defs
    for d in defs:
        run(definition=d, dataset=dataset, runs=2)
    ds, _ = get_dataset(dataset)
    rows = []
    for props, f in load_all_results(dataset):
        m = compute_all_metrics(dataset=ds, run=f, properties=props)["metrics"]
        result, error = f["result"][:], f["error"][:]
        m["rel-l2"] = float(np.linalg.norm(error) / np.linalg.norm(result - error))
        m["props"] = props
        rows.append(m)
    ds.close()
    return rows


@needs_reference
def test_product_through_runner(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    rows = _run("product-ucube-D3-E1-M1000-N1000-gaussian", "product", 3)
    assert len(rows) == 4  # float32 path=auto / path=direct_diff, float64, float16
    for m in rows:
        name = m["props"]["name"]
        tol = 1e-12 if "float64" in name else 5e-3 if "float16" in name else 1e-5  # BASELINE.json: 1e-5 on the FP32 direct path
        assert m["rel-l2"] <= tol, m
        assert m["props"]["algo"] == "b200-product" and m["props"]["gpu_launches"] > 0
        assert m["query-time"] > 0 and m["build-time"] >= 0


@needs_reference
def test_solver_through_runner(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    rows = _run("solver-ucubelam1-D3-E1-M2000-N2000-gaussian", "solver", 3)
    assert len(rows) == 4  # (Nystrom-preconditioned, plain CG) x two query-arg groups (rtol 1e-4, 1e-6)
    best = min(m["rel-l2"] for m in rows)
    assert best <= 1e-4, rows
    assert all(m["props"]["cg_converged"] for m in rows)
    assert len({m["props"]["name"] for m in rows}) == 4  # the name carries the preconditioner and the swept rtol
    for m in rows:
        pc = m["props"]["preconditioner"]
        assert pc.startswith("nystrom") == ("nystrom" in m["props"]["name"]), m["props"]
        if "rtol=1e-06" in m["props"]["name"]:
            assert m["rel-l2"] <= 1e-4, m
    its = {m["props"]["name"]: m["props"]["cg_iterations"] for m in rows}
    pcg = min(v for k, v in its.items() if "nystrom" in k and "1e-06" in k)
    cg = min(v for k, v in its.items() if "nystrom" not in k and "1e-06" in k)
    assert pcg * 4 <= cg, its


@pytest.mark.parametrize("case, golden", [("product_d3", "product_absexp_cube_d3_e3_xy"),
                                           ("attention_d64", "attention_absoluteexponential_d64_e8"),
                                           ("solver_d3", "solver_gaussian_cube_d3_lam1")], ids=["product_d3", "attention_d64", "solver_d3"])
def test_gpu_written_ground_truth_equals_the_reference(tmp_path, monkeypatch, standin_reference, case, golden):
    """The BASELINE-size datasets (C2-C5) get their ``target_signal`` from kmb_product_f64; here the same writer on the
    reference's own float64 outputs stored in tests/golden (a product with independent targets and E = 3, row-normalised
    attention with D = 64, and the right-hand side K b + b of a solve): every row must agree to 1e-12."""
    import h5py

    from kernel_matrix_benchmarks_b200 import datasets as gen
    from kernel_matrix_benchmarks_b200.harness import datasets_ext

    g = load_golden(golden)
    ds = gen.KernelDataset(name=golden, task=g["task"], kernel=g["kernel"], source_points=g["source_points"],
                           target_points=g["source_points"] if g["same_points"] else g["target_points"],
                           source_signal=g["source_signal"], same_points=g["same_points"], normalize_rows=g["normalize_rows"])
    lam, want = (float(g["lam"]), g["rhs"]) if case == "solver_d3" else (0.0, g["truth"])
    monkeypatch.setattr(datasets_ext, "GPU_TRUTH_MIN_WORK", 1.0)
    monkeypatch.setattr(datasets_ext, "VERIFY_ROWS", 64)
    fn = str(tmp_path / "gpu_truth.hdf5")
    datasets_ext.write_dataset(fn, ds, label="ucube", lam=lam, verbose=False)
    f = h5py.File(fn, "r")
    assert "kmb_product_f64" in f.attrs["truth_source"] and "64 sampled target rows" in f.attrs["truth_source"]
    got = f["target_signal"][:]
    assert got.shape == want.shape
    assert np.linalg.norm(got - want) <= 1e-12 * np.linalg.norm(want)


def test_baseline_size_datasets_are_registered(standin_reference):
    """C2, C3, C4, C5 by the reference's naming contract (algos.yaml:38), with globs of this repo's algos.yaml matching."""
    from kernel_matrix_benchmarks.datasets import DATASETS

    for name in ("product-ucube-D3-E1-M1000000-N1000000-gaussian", "product-ucube-D784-E1-M60000-N10000-gaussian",
                 "attention-ucube-D64-E64-M262144-N262144-absolute-exponential", "solver-ucubelam1-D3-E1-M1000000-N1000000-gaussian"):
        assert name in DATASETS, name
