"""The offline harness layer (SURVEY.md section 8f ranks 1-2): the h5py stand-in, the extra dataset
writers and the plugin's algos.yaml as the *reference's own* parser sees it.  The dataset writers run against the
stand-in of tests/reference_standin.py and are compared with the reference's outputs stored in tests/golden/; the
tests that need the reference's parser or runner skip when its tree is neither staged (baseline/_ref) nor named by
KMB_REFERENCE."""
import os
import sys

import numpy as np
import pytest

from conftest import load_golden
from kernel_matrix_benchmarks_b200.harness import bootstrap, h5lite
from reference_standin import UPSTREAM_DATASET, standin_reference  # noqa: F401  (fixture)

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(bootstrap.find_reference() is None, reason="reference harness not available")


def test_h5lite_roundtrip(tmp_path):
    fn = tmp_path / "x.hdf5"
    a = np.arange(12.0).reshape(4, 3)
    with h5lite.File(fn, "w") as f:
        f.attrs["kernel"] = "gaussian"
        f.attrs["same_points"] = np.bool_(True)
        f["source_points"] = a
        f["target_points"] = f["source_points"]  # datasets.py:163 assigns one dataset to another key
    f = h5lite.File(fn, "r")
    assert f.attrs["kernel"] == "gaussian" and f.attrs["same_points"] is True
    assert f.attrs.get("normalize_rows", False) is False
    assert f["source_points"].shape == (4, 3) and int(f["source_points"].shape[-1]) == 3
    np.testing.assert_array_equal(f["target_points"][:], a)
    assert "source_points" in f and "nope" not in f
    with pytest.raises(OSError):
        f["z"] = a
    f.close()
    # the metrics cache of plotting/metrics.py:47-58: r+ mode, groups with attrs, delete
    f = h5lite.File(fn, "r+")
    g = f.create_group("metrics").create_group("errors")
    g.attrs["max"] = np.float64(1.5)
    f.close()
    f = h5lite.File(fn, "r+")
    assert f["metrics"]["errors"].attrs["max"] == 1.5
    del f["metrics"]
    f.close()
    assert "metrics" not in h5lite.File(fn, "r")


def test_h5lite_never_unpickles_and_rejects_foreign_files(tmp_path):
    """The stand-in parses only its own format (magic + npz read with allow_pickle=False): a pickle, a real HDF5
    file or a download that happens to sit at the dataset path is refused, never executed."""
    import pickle

    evil = tmp_path / "evil.hdf5"
    evil.write_bytes(pickle.dumps({"attrs": {}, "items": {}}))
    with pytest.raises(OSError, match="not an h5lite file"):
        h5lite.File(str(evil), "r")
    real = tmp_path / "real.hdf5"
    real.write_bytes(h5lite.HDF5_SIGNATURE + b"\0" * 64)
    with pytest.raises(OSError, match="real HDF5 file"):
        h5lite.File(str(real), "r")
    # object arrays (the one way to smuggle a pickle into an npz) cannot be written either
    with pytest.raises(TypeError):
        with h5lite.File(str(tmp_path / "o.hdf5"), "w") as f:
            f["x"] = np.array([{"a": 1}], dtype=object)
    # attributes survive as plain scalars / strings / arrays
    fn = str(tmp_path / "a.hdf5")
    with h5lite.File(fn, "w") as f:
        f.attrs["k"], f.attrs["n"], f.attrs["flag"], f.attrs["v"] = "gaussian", np.int64(3), np.bool_(True), np.arange(3.0)
        g = f.create_group("metrics")
        g.attrs["rmse"] = np.float64(0.5)
    f = h5lite.File(fn, "r")
    assert f.attrs["k"] == "gaussian" and f.attrs["n"] == 3 and f.attrs["flag"] is True
    assert np.array_equal(f.attrs["v"], np.arange(3.0)) and f["metrics"].attrs["rmse"] == 0.5


def test_offline_harness_refuses_to_download(tmp_path, standin_reference):
    """get_dataset (datasets.py:106-109) tries an HTTP download first; the offline harness must not.  activate() swaps
    the reference's ``datasets.download``; the stand-in's own ``download`` fails the test if the swap does not happen."""
    import kernel_matrix_benchmarks.datasets as ref_datasets

    with pytest.raises(OSError, match="not downloading"):
        ref_datasets.download("http://kernel-matrix-benchmarks.com/datasets/x.hdf5", str(tmp_path / "x.hdf5"))


def test_shims_do_not_shadow_real_modules():
    shimmed = bootstrap.install_import_shims()
    import numpy  # noqa: F401  (a real module is never replaced)

    for name in shimmed:
        assert name in ("h5py", "docker", "colors")
    assert "numpy" not in shimmed


def test_extra_datasets_are_registered_and_named_by_contract(standin_reference):
    from kernel_matrix_benchmarks.datasets import DATASETS

    from kernel_matrix_benchmarks_b200.harness import datasets_ext

    for name in datasets_ext.extra_datasets():
        assert name in DATASETS
        task, label, d, e, m, n, kernel = name.split("-", 6)  # algos.yaml:38
        assert task in ("product", "attention", "solver") and d[0] == "D" and e[0] == "E" and m[0] == "M" and n[0] == "N"
    assert DATASETS[UPSTREAM_DATASET].__name__ == "_upstream_writer"  # the reference's own are kept


def _golden_dataset(name):
    from kernel_matrix_benchmarks_b200 import datasets as gen

    g = load_golden(name)
    ds = gen.KernelDataset(name=name, task=g["task"], kernel=g["kernel"], source_points=g["source_points"],
                           target_points=g["source_points"] if g["same_points"] else g["target_points"],
                           source_signal=g["source_signal"], same_points=g["same_points"], normalize_rows=g["normalize_rows"],
                           density_estimation=g["density_estimation"])
    return g, ds


@pytest.mark.parametrize("name", ["product_gaussian_d16_e2", "product_gaussian_cube_d3", "product_absexp_cube_d3_e3_xy",
                                  "attention_absoluteexponential_d64_e8"])
def test_blocked_ground_truth_equals_the_reference_writer(tmp_path, monkeypatch, standin_reference, name):
    """write_dataset (blocked GroundTruth) == the reference's float64 result on the same arrays (tests/golden, written by
    the reference's BruteForceProductBLAS in float64 with difference-form distances, which is its GroundTruth)."""
    import h5py

    from kernel_matrix_benchmarks_b200.harness import datasets_ext

    g, ds = _golden_dataset(name)
    monkeypatch.setattr(datasets_ext, "TEMP_BYTES", 2 * 8 * ds.M * ds.D * 37)  # force blocks of 37 rows
    fn = str(tmp_path / "mine.hdf5")
    datasets_ext.write_dataset(fn, ds, label="ucube", verbose=False)
    a = h5py.File(fn, "r")
    for k in ("source_points", "target_points", "source_signal"):
        np.testing.assert_array_equal(a[k][:], g[k])
    got = a["target_signal"][:]
    assert got.shape == g["truth"].shape
    assert np.linalg.norm(got - g["truth"]) <= 1e-12 * np.linalg.norm(g["truth"])
    for k in ("kernel", "task", "normalize_rows", "same_points", "density_estimation"):
        assert a.attrs[k] == g[k], k
    assert a.attrs["point_type"] == "float" and "GroundTruth" in a.attrs["truth_source"]


def test_solver_dataset_rhs_is_lambda_consistent(tmp_path, standin_reference):
    import h5py

    from kernel_matrix_benchmarks_b200 import datasets as gen
    from kernel_matrix_benchmarks_b200.harness import datasets_ext

    ds = gen.uniform_cube(128, 3, 1.0, "gaussian", "solver")
    fn = str(tmp_path / "s.hdf5")
    datasets_ext.write_dataset(fn, ds, label="ucubelam1", lam=1.0, verbose=False)
    f = h5py.File(fn, "r")
    y, b, a = f["source_points"][:], f["source_signal"][:], f["target_signal"][:]
    K = np.exp(-((y[:, None, :] - y[None, :, :]) ** 2).sum(-1))
    np.testing.assert_allclose(a, K @ b + b, rtol=1e-12, atol=1e-12)
    assert f.attrs["task"] == "solver" and f.attrs["lam"] == 1.0
    # and the right-hand side the reference built for the same system (K b through its float64 product, + lam b)
    g, ds = _golden_dataset("solver_gaussian_cube_d3_lam1")
    datasets_ext.write_dataset(fn, ds, label="ucubelam1", lam=float(g["lam"]), verbose=False)
    a = h5py.File(fn, "r")["target_signal"][:]
    assert np.linalg.norm(a - g["rhs"]) <= 1e-12 * np.linalg.norm(g["rhs"])


@needs_reference
@pytest.mark.parametrize("dataset, task, dim, expect", [
    ("product-ucube-D3-E1-M10000-N10000-gaussian", "product", 3, {("b200-product", "auto"), ("b200-product", "direct_diff")}),
    ("product-ucube-D784-E1-M4000-N1000-gaussian", "product", 784, {("b200-product", "auto")}),
    ("attention-ucube-D64-E64-M4096-N4096-gaussian", "attention", 64, {("b200-product", "auto")}),
])
def test_algos_yaml_through_the_reference_parser(dataset, task, dim, expect):
    """definitions.get_definitions (definitions.py:90-168) on this repo's algos.yaml."""
    bootstrap.activate()
    from kernel_matrix_benchmarks.definitions import get_definitions

    defs = get_definitions(definition_file=os.path.join(REPO, "algos.yaml"), dimension=dim, dataset=dataset, task=task,
                           hardware="GPU", kernel="gaussian", normalize_rows=(task == "attention"))
    assert {(d.algorithm, d.arguments["path"]) for d in defs} == expect
    for d in defs:
        assert d.module == "kernel_matrix_benchmarks_b200.algorithms.b200" and d.constructor == "B200Product"
        assert d.arguments["kernel"] == "gaussian" and d.arguments["dimension"] == dim
    assert get_definitions(definition_file=os.path.join(REPO, "algos.yaml"), dimension=dim, dataset=dataset, task=task,
                           hardware="CPU", kernel="gaussian") == []


@needs_reference
def test_solver_run_groups():
    bootstrap.activate()
    from kernel_matrix_benchmarks.definitions import get_definitions

    def lams(dataset):
        defs = get_definitions(definition_file=os.path.join(REPO, "algos.yaml"), dimension=3, dataset=dataset,
                               task="solver", hardware="GPU", kernel="gaussian")
        return sorted(d.arguments["lam"] for d in defs), [d.query_argument_groups for d in defs]

    assert lams("solver-ucubelam1-D3-E1-M2000-N2000-gaussian")[0] == [1.0, 1.0]   # preconditioner "auto" and "nystrom"
    assert lams("solver-cube-D3-E1-M1000-N1000-gaussian")[0] == [0.0]
    assert all(len(g) == 2 for g in lams("solver-ucubelam1-D3-E1-M2000-N2000-gaussian")[1])


@needs_reference
def test_reference_harness_end_to_end_on_cpu(tmp_path, monkeypatch):
    """The unmodified runner.run -> results.store_result -> plotting.metrics chain, driven offline
    with the reference's own brute force as the algorithm (the B200 plugin takes the same road on
    the GPU box: tests/test_harness_gpu.py)."""
    bootstrap.activate()
    monkeypatch.chdir(tmp_path)  # data/ and results/ are cwd-relative
    from kernel_matrix_benchmarks.definitions import Definition
    from kernel_matrix_benchmarks.plotting.utils import compute_all_metrics
    from kernel_matrix_benchmarks.results import load_all_results
    from kernel_matrix_benchmarks.runner import run

    name = "product-ucube-D3-E1-M1000-N1000-gaussian"
    d = Definition(algorithm="bruteforce-product-blas", constructor="BruteForceProductBLAS",
                   module="kernel_matrix_benchmarks.algorithms.bruteforce", docker_tag="none",
                   arguments={"kernel": "gaussian", "dimension": 3, "normalize_rows": False, "precision": "float32",
                              "fast_sqdists": True},
                   query_argument_groups=[{}])
    run(definition=d, dataset=name, runs=1)
    res = list(load_all_results(name))
    assert len(res) == 1
    props, f = res[0]
    from kernel_matrix_benchmarks.datasets import get_dataset

    ds, dim = get_dataset(name)
    m = compute_all_metrics(dataset=ds, run=f, properties=props)["metrics"]
    assert dim == 3 and 0 < m["rmse-error"] < 1e-4 and m["total-time"] > 0
