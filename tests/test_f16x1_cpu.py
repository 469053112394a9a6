"""The one-term FP16 tensor path ("tensor_f16x1") without a GPU: the dispatch of every parity case of tests/f16x1_cases.py
(host-only plan query), what the path does not support, that "auto" never picks it, the plugin's and the solver's
checks, its algos.yaml run group, and the model of its arithmetic against the tolerance the GPU test holds it to."""
import ctypes
import fnmatch
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import dot_exponential_oracle as dxo
import f16x1_cases as fc
from conftest import REPO

PATH = fc.PATH


def _plan(case):
    from kernel_matrix_benchmarks_b200 import product

    return product.dispatch_plan(case.N, case.M, case.D, case.E, kernel=case.kernel, normalize_rows=case.norm,
                                 density_estimation=case.density, path=PATH, sms=148)


def _env_plans(cases):
    """dispatch_plan of cases that set environment knobs, in a child process with that environment (read once per process)."""
    plans = {}
    for env in sorted({c.env for c in cases}):
        script = ("import json, sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import f16x1_cases as fc; "
                  "from test_f16x1_cpu import _plan; env = tuple(map(tuple, json.loads(sys.argv[3]))); "
                  "print(json.dumps({c.name: _plan(c) for c in fc.all_cases() if c.env == env}))")
        res = subprocess.run([sys.executable, "-c", script, REPO, os.path.join(REPO, "tests"), json.dumps(env)],
                             env=dict(os.environ, **dict(env)), capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, res.stderr
        plans.update(json.loads(res.stdout.strip().splitlines()[-1]))
    return plans


@pytest.fixture(scope="module")
def plans():
    cases = fc.all_cases()
    out = {c.name: _plan(c) for c in cases if not c.env}
    out.update(_env_plans([c for c in cases if c.env]))
    return out


def test_every_case_reaches_its_family(plans):
    """Each case keeps the path it names and reaches its family, signal chunk and number of passes."""
    bad = []
    for c in fc.all_cases():
        p = plans[c.name]
        want = "fill" if (c.norm and c.density) else c.family
        if p["path"] != PATH or p["family"] != want:
            bad.append(f"{c.name}: {p['path']} / {p['family']}, expected {PATH} / {want}")
        elif want != "fill" and (p["chunk"], p["passes"]) != (c.chunk, c.passes):
            bad.append(f"{c.name}: {p['passes']} passes of {p['chunk']} columns, expected {c.passes} of {c.chunk}")
    assert not bad, "\n".join(bad)


def test_every_family_has_cases():
    """Every family (and the multi-pass route D > 128) x kernel x normalisation, density on every E <= 4 family, the
    single-CTA kernels under KMB_TENSOR_PAIR=0, EP = 1 / 2 / 4, and every D and E of the grid."""
    seen = set()
    for c in fc.all_cases():
        kind = "density" if c.density else f"n{int(c.norm)}"
        seen.add((c.covers, c.kernel, kind, "knob" if c.env else ""))
        seen |= {("D", c.D), ("E", c.E), ("chunk", c.chunk)}
    want = set()
    for kernel in fc.KERNELS:
        for kind in ("n0", "n1"):
            want |= {(f, kernel, kind, "") for f in fc.FAMILIES}
            want |= {(f, kernel, kind, "knob") for f in ("tensor", "pv16", "multipass")}
        want |= {(f, kernel, "density", "") for f in ("tensor", "tensor_pair")}
    want |= {("D", D) for D in fc.DIMS} | {("E", E) for E in fc.SIGNALS} | {("chunk", w) for w in (1, 2, 4, 64)}
    missing = sorted(want - seen, key=str)
    assert not missing, "one-term targets without a parity case:\n" + "\n".join(map(str, missing))
    assert {c.covers for c in fc.all_cases()} == set(fc.FAMILIES)


def test_pv_plan_is_the_three_term_plan():
    """The one-term P.B kernels run the launch plan of the three-term ones (same ring, stages, grid and wave plan)."""
    from kernel_matrix_benchmarks_b200 import product

    for N, M, D, E in ((401, 1500, 64, 64), (262144, 262144, 64, 64), (100, 1500, 16, 8), (4096, 4096, 128, 200)):
        for kernel in fc.KERNELS:
            kw = dict(kernel=kernel, normalize_rows=True, sms=148, smem_optin=232448)
            one, three = product.pv_plan(N, M, D, E, path=PATH, **kw), product.pv_plan(N, M, D, E, path="tensor_f16", **kw)
            assert one == three and one["family"].startswith("pv16"), (N, M, D, E, kernel, one, three)


def test_inverse_distance_and_tf32_family_shapes_are_unsupported():
    """1/|x - y| is rejected at every shape, E > 4 with D <= 128 included (where the three-term FP16 path takes the TF32
    P.B family), by every entry point that takes a path."""
    from kernel_matrix_benchmarks_b200 import _lib, product

    lib = _lib.load()
    kid, pid = _lib.KERNEL_IDS["inverse-distance"], _lib.PATH_IDS[PATH]
    for D, E in ((3, 1), (40, 4), (64, 64), (16, 8), (784, 1), (200, 64)):
        with pytest.raises(NotImplementedError, match="inverse-distance"):
            product.workspace_bytes(1000, 1000, D, E, kernel="inverse-distance", path=PATH)
        with pytest.raises(NotImplementedError, match="inverse-distance"):
            product.dispatch_plan(1000, 1000, D, E, kernel="inverse-distance", path=PATH)
        with pytest.raises(NotImplementedError):
            product.pv_plan(1000, 1000, D, E, kernel="inverse-distance", path=PATH, sms=148, smem_optin=232448)
    assert product.dispatch_plan(1000, 1000, 64, 64, kernel="inverse-distance", path="tensor_f16")["family"] == "pv"
    dummy = ctypes.c_void_p(256)   # never dereferenced: the kernel is rejected before any device work
    assert lib.kmb_product_f32(dummy, dummy, dummy, dummy, 10, 10, 64, 64, kid, 0, pid, 0, None, 0, None) == _lib.KMB_ERR_UNSUPPORTED
    assert lib.kmb_product_prepare_f32(dummy, dummy, 10, 10, 64, kid, 0, pid, None, 0, None) == _lib.KMB_ERR_UNSUPPORTED
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    with pytest.raises(NotImplementedError, match="inverse-distance"):
        B200Product(kernel="inverse-distance", dimension=64, path=PATH)


def test_the_path_id_and_its_bounds():
    from kernel_matrix_benchmarks_b200 import _lib, product

    lib = _lib.load()
    assert _lib.PATH_IDS[PATH] == 6
    need = ctypes.c_size_t(0)
    assert lib.kmb_product_workspace_bytes(1000, 1000, 64, 64, 0, 0, 7, ctypes.byref(need)) == _lib.KMB_ERR_INVALID
    assert lib.kmb_resolved_path(64, 64, 0, 7) == -1
    assert product.resolved_path(64, 64, "gaussian", PATH) == PATH


def test_auto_never_resolves_to_the_one_term_path():
    from kernel_matrix_benchmarks_b200 import product

    for kernel in ("gaussian", "absolute-exponential", "inverse-distance", "dot-exponential"):
        for D in (1, 3, 16, 17, 64, 128, 129, 784):
            for E in (1, 4, 5, 32, 64, 200):
                assert product.resolved_path(D, E, kernel) != PATH, (kernel, D, E)
                if kernel != "inverse-distance":
                    assert product.resolved_path(D, E, kernel, PATH) == PATH


def test_solver_rejects_the_path():
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Solver

    with pytest.raises(ValueError, match="tensor_f16x1"):
        B200Solver(kernel="gaussian", dimension=64, path=PATH)


def test_algos_yaml_run_group():
    """b200-product's fp16-single-term group: float16 inputs on the one-term path, D >= 17 and N >= 10^4 only."""
    import yaml

    with open(os.path.join(REPO, "algos.yaml")) as f:
        group = yaml.safe_load(f)["b200-product"]["run-groups"]["fp16-single-term"]
    assert group["args"] == [{"precision": "float16", "path": PATH}]
    match = lambda name: any(fnmatch.fnmatch(name, p) for p in group["datasets"])  # noqa: E731
    for D in list(range(1, 17)):
        for task, E in (("product", 1), ("attention", 64)):
            for n in (1000, 10_000, 262_144, 1_000_000):
                assert not match(f"{task}-ucube-D{D}-E{E}-M{n}-N{n}-gaussian"), D
    for D in (17, 18, 19, 20, 64, 99, 100, 784, 999):
        assert match(f"product-ucube-D{D}-E1-M60000-N10000-gaussian"), D
        assert not match(f"product-ucube-D{D}-E1-M4000-N1000-gaussian"), D
    assert match("product-ucube-D784-E1-M60000-N10000-gaussian")                        # C3
    assert match("attention-ucube-D64-E64-M262144-N262144-absolute-exponential")        # C4
    assert not match("attention-ucube-D64-E64-M4096-N4096-gaussian")


def _truth(kernel, x, y, b, norm):
    if kernel == "dot-exponential":
        return dxo.kernel_product(y, x, b, normalize_rows=norm)
    d2 = np.maximum((x * x).sum(1)[:, None] + (y * y).sum(1)[None, :] - 2 * x @ y.T, 0.0)
    L = -d2 if kernel == "gaussian" else -np.sqrt(d2)
    if norm:
        K = np.exp(L - L.max(1, keepdims=True))
        return (K @ b) / K.sum(1, keepdims=True)
    return np.exp(L) @ b


@pytest.mark.parametrize("name, kernel, D, E, norm", [
    ("C3", "gaussian", 784, 1, False),
    ("C4-gaussian", "gaussian", 64, 64, True),
    ("C4-absexp", "absolute-exponential", 64, 64, True),
    ("plain-D64-E64", "gaussian", 64, 64, False),
    ("D32-E3", "gaussian", 32, 3, False),
])
def test_model_of_the_arithmetic_leaves_the_tolerance_its_margin(name, kernel, D, E, norm):
    """The NumPy model of the one-term arithmetic (f16x1_cases.model_product) on C3- and C4-shaped data (the unit cube
    scaled by sqrt(3 / D), N = 256 rows against M = 8192 sources) against the float64 truth: 2.5x under the tolerance over
    the whole result and 4x under it on the worst row.  This is what fixes f16x1_cases.TOL / ROW_TOL without a GPU."""
    rng = np.random.RandomState(7)
    r = (3.0 / D) ** 0.5
    x, y, b = r * rng.rand(256, D), r * rng.rand(8192, D), rng.randn(8192, E)
    x, y, b = (a.astype(np.float32).astype(np.float64) for a in (x, y, b))
    err, row_err = fc.errors(fc.model_product(kernel, x, y, b, normalize_rows=norm), _truth(kernel, x, y, b, norm))
    assert 2.5 * err <= fc.TOL and 4 * row_err.max() <= fc.ROW_TOL, (name, err, row_err.max())
    assert err > 1e-7   # one term is float16-class: visibly less accurate than the three-term path


def test_model_of_the_arithmetic_on_every_case_stays_inside_the_tolerance():
    """The same model on the data of every parity case (the oracle in float64; the plain product, attention, density):
    what the GPU test demands of the kernels, with 2.5x (whole result) and 4x (worst row) to spare."""
    worst = []
    for c in fc.all_cases():
        if c.env or (c.norm and c.density) or c.D > 128:   # D > 128: E <= 4 arithmetic, the same as the D = 128 cases
            continue
        x, y, b = fc.make_data(c)
        if c.density:
            b = np.ones((c.M, 1))
        err, row_err = fc.errors(fc.model_product(c.kernel, x, y, b, normalize_rows=c.norm), _truth(c.kernel, x, y, b, c.norm))
        if 2.5 * err > fc.TOL or 4 * row_err.max() > fc.ROW_TOL:
            worst.append(f"{c.name}: {err:.2e} / worst row {row_err.max():.2e}")
    assert not worst, "\n".join(worst)
