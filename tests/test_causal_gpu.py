"""Causal products (KMB_FLAG_CAUSAL) on the GPU: every case of tests/causal_cases.py against the float64 oracle of
tests/causal_oracle.py, the float64 path, large attention logits, prepared points, repeatability, full visibility, the
plugin end to end and the multi-GPU row split."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import causal_cases as cc
import causal_oracle as co

from kernel_matrix_benchmarks_b200 import product as prod

pytestmark = pytest.mark.gpu

REL_L2, WORST_ROW = 1e-4, 1e-3
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(case, seed=0, prepared=False):
    x, y, b = case.data(seed)
    dev = torch.device("cuda", 0)
    xt = torch.tensor(x, dtype=torch.float32, device=dev)
    yt = torch.tensor(y, dtype=torch.float32, device=dev)
    bt = None if case.density else torch.tensor(b, dtype=torch.float32, device=dev)
    ws = prod.Workspace()
    token = None
    if prepared:
        need = prod.workspace_bytes(case.N, case.M, case.D, 1 if case.density else case.E, kernel=case.kernel,
                                    normalize_rows=case.norm, density_estimation=case.density, causal=True)
        token = prod.prepare_points(xt, yt, kernel=case.kernel, workspace=ws, min_bytes=need, causal=True)
    out = prod.kernel_product(xt, yt, bt, kernel=case.kernel, normalize_rows=case.norm, density_estimation=case.density,
                              row_offset=case.row_offset, workspace=ws, prepared=token, causal=True)
    torch.cuda.synchronize()
    assert prod.last_path == "tensor_f16"
    return out.double().cpu().numpy(), (x, y, b)


def _check(case, got, data):
    x, y, b = data
    want = co.causal_product(case.kernel, x, y, b, row_offset=case.row_offset, normalize_rows=case.norm,
                             density_estimation=case.density)
    assert np.all(np.isfinite(got)), case.id
    assert co.rel_l2(got, want) <= REL_L2, (case.id, co.rel_l2(got, want))
    assert co.worst_row(got, want) <= WORST_ROW, (case.id, co.worst_row(got, want))


@pytest.mark.parametrize("case", [c for c in cc.CASES if not c.env], ids=lambda c: c.id)
def test_case_against_oracle(case):
    got, data = _run(case)
    _check(case, got, data)


CHILD = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import numpy as np
import causal_cases as cc, causal_oracle as co
import test_causal_gpu as t
out = []
for c in cc.CASES:
    if c.env:
        got, (x, y, b) = t._run(c)
        want = co.causal_product(c.kernel, x, y, b, row_offset=c.row_offset, normalize_rows=c.norm, density_estimation=c.density)
        out.append([c.id, bool(np.all(np.isfinite(got))), co.rel_l2(got, want), co.worst_row(got, want)])
print(json.dumps(out))
"""


def test_cases_with_single_cta_kernels_forced():
    """KMB_TENSOR_PAIR=0 (read once per process): the single-CTA kernels on problems of several row tiles, in a child."""
    res = subprocess.run([sys.executable, "-c", CHILD, REPO, os.path.join(REPO, "tests")],
                         env=dict(os.environ, **dict(cc.PAIR_OFF)), capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    rows = json.loads(res.stdout.strip().splitlines()[-1])
    assert len(rows) == sum(1 for c in cc.CASES if c.env)
    for cid, finite, rel, worst in rows:
        assert finite and rel <= REL_L2 and worst <= WORST_ROW, (cid, rel, worst)


@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential", "inverse-distance", "dot-exponential"])
@pytest.mark.parametrize("D,E,norm,row_offset", [(3, 2, True, 77), (16, 9, False, 0), (64, 3, True, 128), (200, 70, True, 5)])
def test_f64_path_matches_oracle(kernel, D, E, norm, row_offset):
    rng = np.random.RandomState(D + E)
    N, M = 300, 500
    s = 1.0 / D ** 0.5
    x, y, b = s * rng.randn(N, D), s * rng.randn(M, D), 0.5 + rng.rand(M, E)
    dev = torch.device("cuda", 0)
    got = prod.kernel_product_f64(torch.tensor(x, device=dev), torch.tensor(y, device=dev), torch.tensor(b, device=dev),
                                  kernel=kernel, normalize_rows=norm, row_offset=row_offset, causal=True).cpu().numpy()
    with np.errstate(invalid="ignore"):
        want = co.causal_product(kernel, x, y, b, row_offset=row_offset, normalize_rows=norm)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("E", [4, 64])
def test_dot_attention_with_large_logits(E):
    """Logits <x_i, y_j> up to ~120: the online maximum keeps softmax finite, masked pairs must not enter it."""
    rng = np.random.RandomState(E)
    N, M, D = 500, 1500, 64
    x, y = rng.randn(N, D), rng.randn(M, D)
    x *= 11.0 / np.linalg.norm(x, axis=1, keepdims=True)
    y *= 11.0 / np.linalg.norm(y, axis=1, keepdims=True)
    y[3:N + 3] = x   # source j = i + 3 repeats target i: logit 121 on the last visible source of every row
    b = 0.5 + rng.rand(M, E)
    dev = torch.device("cuda", 0)
    got = prod.kernel_product(torch.tensor(x, dtype=torch.float32, device=dev), torch.tensor(y, dtype=torch.float32, device=dev),
                              torch.tensor(b, dtype=torch.float32, device=dev), kernel="dot-exponential", normalize_rows=True,
                              row_offset=3, causal=True).double().cpu().numpy()
    want = co.causal_product("dot-exponential", x, y, b, row_offset=3, normalize_rows=True)
    assert (x @ y.T).max() > 100
    assert np.all(np.isfinite(got))
    assert co.rel_l2(got, want) <= REL_L2 and co.worst_row(got, want) <= WORST_ROW


@pytest.mark.parametrize("case", [c for c in cc.CASES if not c.env and c.N >= 256][:4], ids=lambda c: c.id)
def test_prepared_equals_unprepared_and_repeats_bitwise(case):
    a, _ = _run(case)
    b, _ = _run(case)
    p, _ = _run(case, prepared=True)
    assert np.array_equal(a, b)
    assert np.array_equal(a, p)


@pytest.mark.parametrize("kernel,D,E", [("gaussian", 64, 1), ("dot-exponential", 64, 64), ("absolute-exponential", 784, 2)])
def test_rows_past_the_last_source_match_the_full_product(kernel, D, E):
    """row_offset >= M - 1: every row sees every source, the causal product is the full one (to tolerance)."""
    case = cc.CausalCase(kernel, 300, 700, D, E, True, 699, "any")
    x, y, b = case.data()
    dev = torch.device("cuda", 0)
    xt, yt, bt = (torch.tensor(a, dtype=torch.float32, device=dev) for a in (x, y, b))
    c = prod.kernel_product(xt, yt, bt, kernel=kernel, normalize_rows=True, row_offset=699, causal=True).double().cpu().numpy()
    f = prod.kernel_product(xt, yt, bt, kernel=kernel, normalize_rows=True, path="tensor_f16").double().cpu().numpy()
    assert co.rel_l2(c, f) <= REL_L2


@pytest.mark.parametrize("precision", ["float32", "float16", "float64"])
def test_plugin_end_to_end(precision):
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    rng = np.random.RandomState(5)
    N, D, E = 1000, 64, 64
    y = rng.randn(N, D) / D ** 0.5
    b = 0.5 + rng.rand(N, E)
    algo = B200Product(kernel="dot-exponential", dimension=D, normalize_rows=True, precision=precision, causal=True)
    assert "causal" in algo.name
    algo.prepare_data(source_points=y, target_points=y, same_points=True)
    algo.fit()
    algo.prepare_query(source_signal=b)
    algo.query()
    got = algo.get_result()
    yy = y.astype(np.float16).astype(np.float64) if precision == "float16" else y
    want = co.causal_product("dot-exponential", yy, yy, b.astype(np.float16).astype(np.float64) if precision == "float16" else b,
                             normalize_rows=True)
    tol = 1e-10 if precision == "float64" else REL_L2
    assert co.rel_l2(got, want) <= tol
    assert algo.get_additional()["path_used"] == ("direct_f64" if precision == "float64" else "tensor_f16")
    algo.done()


def test_plugin_rejects_paths_without_causal_kernels():
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    for path in ("direct", "tensor_tf32", "tensor_f16x1", "direct_sym"):
        with pytest.raises(NotImplementedError):
            B200Product(kernel="gaussian", dimension=3, path=path, causal=True)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_rows_mode():
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    rng = np.random.RandomState(9)
    N, D, E = 3000, 64, 8
    y = rng.randn(N, D) / D ** 0.5
    b = 0.5 + rng.rand(N, E)
    algo = B200Product(kernel="gaussian", dimension=D, normalize_rows=True, causal=True, n_gpus=2)
    algo.prepare_data(source_points=y, target_points=y, same_points=True)
    algo.fit()
    algo.prepare_query(source_signal=b)
    algo.query()
    got = algo.get_result()
    want = co.causal_product("gaussian", y, y, b, normalize_rows=True)
    assert co.rel_l2(got, want) <= REL_L2 and co.worst_row(got, want) <= WORST_ROW
    algo.done()
