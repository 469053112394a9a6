"""The dot-exponential kernel exp(<x, y>) (not in bruteforce.py) without a GPU: its float64 oracles, the dispatch of every
parity case of tests/dot_exponential_cases.py (host-only plan query), and what the kernel does not support."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import dot_exponential_cases as dxc
import dot_exponential_oracle as dxo
from conftest import REPO

KERNEL = dxc.KERNEL


def _small(seed, N=7, M=11, D=5, E=3, scale=1.0):
    rng = np.random.RandomState(seed)
    return scale * rng.randn(N, D), scale * rng.randn(M, D), rng.randn(M, E)


@pytest.mark.parametrize("impl", [dxo.kernel_product, dxo.kernel_product_c], ids=["numpy", "c"])
def test_oracle_is_the_literal_formula(impl):
    """exp(x y^T) b, its row sums and its row-normalised form, as written, on small inputs."""
    for seed in range(3):
        x, y, b = _small(seed)
        K = np.exp(x @ y.T)
        np.testing.assert_allclose(impl(y, x, b), K @ b, rtol=1e-13, atol=0)
        np.testing.assert_allclose(impl(y, x, None, density_estimation=True), K.sum(1, keepdims=True), rtol=1e-13, atol=0)
        np.testing.assert_allclose(impl(y, x, b, normalize_rows=True), (K @ b) / K.sum(1, keepdims=True), rtol=1e-13, atol=0)
        np.testing.assert_array_equal(impl(y, x, b, normalize_rows=True, density_estimation=True), np.ones((7, 1)))
        # targets None: the sources themselves; rows: a subset
        np.testing.assert_allclose(impl(y, None, b, rows=[0, 4]), (np.exp(y @ y.T) @ b)[[0, 4]], rtol=1e-13, atol=0)


@pytest.mark.parametrize("impl", [dxo.kernel_product, dxo.kernel_product_c], ids=["numpy", "c"])
def test_oracle_attention_stays_finite_where_exp_overflows(impl):
    """Rows whose largest <x, y> is ~1000: exp overflows float64, softmax(x y^T) b does not; it equals the attention of
    the same row shifted by any constant (here: computed with x scaled so that the logits stay small, times 1)."""
    x, y, b = _small(3, N=4, M=50, D=8, E=2)
    x *= 1000.0 / np.abs(x @ y.T).max()
    with np.errstate(over="ignore"):
        assert np.isinf(np.exp(x @ y.T)).any()
    got = impl(y, x, b, normalize_rows=True)
    s = x @ y.T
    w = np.exp(s - s.max(1, keepdims=True))
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, (w @ b) / w.sum(1, keepdims=True), rtol=1e-12, atol=0)
    assert np.isinf(impl(y, x, b[:, :1] ** 2)).any()   # the plain product overflows as the formula does


def test_numpy_and_c_oracles_agree():
    """NumPy (BLAS, blocked) against C (one source at a time) at 1e-12 on the parity data, every query mode."""
    for case in (c for c in dxc.all_cases() if c.N == 401 and c.E in (1, 64) and c.D in (3, 784) and c.path == "auto"):
        x, y, b = dxc.make_data(case)
        rows = np.arange(0, case.N, 13)
        kw = dict(normalize_rows=case.norm, density_estimation=case.density, rows=rows)
        want, got = dxo.kernel_product(y, x, b, **kw), dxo.kernel_product_c(y, x, b, **kw)
        err = np.linalg.norm(got - want) / np.linalg.norm(want)
        assert err <= 1e-12, (case.name, err)


def _plan(case):
    from kernel_matrix_benchmarks_b200 import product

    return product.dispatch_plan(case.N, case.M, case.D, case.E, kernel=KERNEL, normalize_rows=case.norm,
                                 density_estimation=case.density, path=case.path, sms=148)


def _env_plans(cases):
    """dispatch_plan of cases that set environment knobs, in a child process with that environment (read once per process)."""
    plans = {}
    for env in sorted({c.env for c in cases}):
        script = ("import json, sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import dot_exponential_cases as dxc; "
                  "from test_dot_exponential_cpu import _plan; env = tuple(map(tuple, json.loads(sys.argv[3]))); "
                  "print(json.dumps({c.name: _plan(c) for c in dxc.all_cases() if c.env == env}))")
        res = subprocess.run([sys.executable, "-c", script, REPO, os.path.join(REPO, "tests"), json.dumps(env)],
                             env=dict(os.environ, **dict(env)), capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, res.stderr
        plans.update(json.loads(res.stdout.strip().splitlines()[-1]))
    return plans


@pytest.fixture(scope="module")
def plans():
    cases = dxc.all_cases()
    out = {c.name: _plan(c) for c in cases if not c.env}
    out.update(_env_plans([c for c in cases if c.env]))
    return out


def test_every_case_reaches_its_family(plans):
    """Each case resolves to the tensor path it names ("auto": FP16 planes at every D) and reaches its family, signal chunk
    and number of passes."""
    bad = []
    for c in dxc.all_cases():
        p = plans[c.name]
        path = "tensor_f16" if c.path == "auto" else c.path
        want = "fill" if (c.norm and c.density) else c.family
        if p["path"] != path or p["family"] != want:
            bad.append(f"{c.name}: {p['path']} / {p['family']}, expected {path} / {want}")
        elif want != "fill" and (p["chunk"], p["passes"]) != (c.chunk, c.passes):
            bad.append(f"{c.name}: {p['passes']} passes of {p['chunk']} columns, expected {c.passes} of {c.chunk}")
    assert not bad, "\n".join(bad)


def test_every_family_has_cases(plans):
    """Every family (and the multi-pass route D > 128) x element type x normalisation, density on every E <= 4 family, the
    single-CTA FP16 kernels under KMB_TENSOR_PAIR=0, and every D, E and path of the grid."""
    seen = set()
    for c in dxc.all_cases():
        elt = "f16" if c.f16 else "tf32"
        kind = "density" if c.density else f"n{int(c.norm)}"
        seen.add((c.covers, elt, kind, "knob" if c.env else ""))
        seen |= {("D", c.D), ("E", c.E), ("path", c.path)}
    want = set()
    for kind in ("n0", "n1"):
        want |= {(f, "f16", kind, "") for f in ("tensor", "tensor_pair", "pv16", "pv16_pair", "multipass")}
        want |= {(f, "tf32", kind, "") for f in ("tensor", "pv", "multipass")}
        want |= {(f, "f16", kind, "knob") for f in ("tensor", "pv16", "multipass")}
    want |= {("tensor", "tf32", "density", ""), ("tensor", "f16", "density", ""), ("tensor_pair", "f16", "density", "")}
    want |= {("D", D) for D in dxc.DIMS} | {("E", E) for E in dxc.SIGNALS} | {("path", p) for p in dxc.PATHS}
    missing = sorted(want - seen, key=str)
    assert not missing, "dot-exponential targets without a parity case:\n" + "\n".join(map(str, missing))
    assert {c.covers for c in dxc.all_cases()} == set(dxc.FAMILIES)


def test_auto_resolves_to_the_fp16_tensor_path_at_every_d():
    from kernel_matrix_benchmarks_b200 import product

    for D in (1, 2, 3, 8, 15, 16, 17, 64, 128, 129, 784):
        for E in (1, 4, 5, 31, 32, 64, 200):
            assert product.resolved_path(D, E, KERNEL) == "tensor_f16", (D, E)
            assert product.resolved_path(D, E, KERNEL, "tensor_tf32") == "tensor_tf32"
    assert product.resolved_path(3, 1, "gaussian") == "direct"   # the other kernels keep their routing


def test_direct_and_symmetric_paths_are_rejected():
    from kernel_matrix_benchmarks_b200 import _lib, product

    lib = _lib.load()
    kid = _lib.KERNEL_IDS[KERNEL]
    assert kid == 3
    for path in ("direct", "direct_diff", "direct_sym"):
        with pytest.raises(NotImplementedError, match="tensor paths only"):
            product.workspace_bytes(1000, 1000, 3, 1, kernel=KERNEL, path=path)
        with pytest.raises(NotImplementedError):
            product.dispatch_plan(1000, 1000, 3, 1, kernel=KERNEL, path=path)
    dummy = ctypes.c_void_p(256)   # never dereferenced: the kernel is rejected before any device work
    assert lib.kmb_product_sym_f32(dummy, None, dummy, 1000, 3, kid, 0, 1, None, 0, None) == _lib.KMB_ERR_UNSUPPORTED
    assert lib.kmb_product_f32(dummy, dummy, dummy, dummy, 10, 10, 3, 1, kid, 0, _lib.PATH_IDS["direct"], 0, None, 0,
                               None) == _lib.KMB_ERR_UNSUPPORTED
    # the kernel ids after it stay unknown
    need = ctypes.c_size_t(0)
    for bad in (4, 7, 9):
        assert lib.kmb_product_workspace_bytes(10, 10, 3, 1, bad, 0, 0, ctypes.byref(need)) == _lib.KMB_ERR_UNSUPPORTED
        assert lib.kmb_resolved_path(3, 1, bad, 0) == -1


def test_symmetric_product_never_applies():
    """same_points data with D <= 3 and E == 1 would take the symmetric kernel for the kernels of bruteforce.py; exp(<x, y>)
    is not a function of |x - y| and has none."""
    import torch

    from kernel_matrix_benchmarks_b200 import product

    y = torch.zeros((40000, 3), dtype=torch.float32)
    assert product.symmetric_applies(y, y, "gaussian")
    assert not product.symmetric_applies(y, y, KERNEL)
    assert not product.symmetric_applies(y, y, KERNEL, density_estimation=True)


def test_solver_rejects_the_kernel():
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Solver

    with pytest.raises(NotImplementedError, match="dot-exponential"):
        B200Solver(kernel=KERNEL, dimension=3)
