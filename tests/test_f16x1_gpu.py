"""The one-term FP16 tensor path ("tensor_f16x1") on a B200: every parity case of tests/f16x1_cases.py against the float64
oracle, proof that the one-term kernels ran (the result differs from the three-term path's), prepared and repeated runs,
attention beyond FP32's exp range, and the plugin end to end."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import dot_exponential_oracle as dxo
import f16x1_cases as fc
from conftest import REPO
from oracle import c_oracle

pytestmark = pytest.mark.gpu

PATH = fc.PATH
CASES = [c for c in fc.all_cases() if not c.env]
ENV_CASES = [c for c in fc.all_cases() if c.env]


def _t(a):
    import torch

    return None if a is None else torch.tensor(a, dtype=torch.float32, device="cuda")


def oracle(kernel, x, y, b, *, normalize_rows=False, density_estimation=False):
    if kernel == "dot-exponential":
        return dxo.kernel_product(y, x, b, normalize_rows=normalize_rows, density_estimation=density_estimation)
    return c_oracle.kernel_product(kernel, y, x, b, normalize_rows=normalize_rows, density_estimation=density_estimation)


def run_case(case):
    """The case on cuda:0 with the one-term path -> (float64 result, facts about the run, the three-term result)."""
    from kernel_matrix_benchmarks_b200 import product

    x, y, b = fc.make_data(case)
    tx, ty, tb = _t(x), _t(y), _t(b)

    def once(path):
        return product.kernel_product(tx, ty, tb, kernel=case.kernel, normalize_rows=case.norm,
                                      density_estimation=case.density, path=path).cpu().numpy()

    got = once(PATH)
    info = {"last_path": product.last_path}
    dev = product.device_info(0)
    info["family"] = product.dispatch_plan(case.N, case.M, case.D, case.E, kernel=case.kernel, normalize_rows=case.norm,
                                           density_estimation=case.density, path=PATH, sms=dev["sm_count"])["family"]
    if case.repeat:
        info["bitwise_repeat"] = bool(np.array_equal(once(PATH).view(np.uint8), got.view(np.uint8)))
    three = once("tensor_f16")
    return got.astype(np.float64), info, three.astype(np.float64)


def check(case, got, info, three):
    x, y, b = fc.make_data(case)
    want = oracle(case.kernel, x, y, b, normalize_rows=case.norm, density_estimation=case.density)
    assert got.shape == want.shape
    assert np.isfinite(got).all(), f"{case.name}: non-finite results in rows {np.unique(np.nonzero(~np.isfinite(got))[0])[:10]}"
    assert info["last_path"] == PATH, (case.name, info)
    if case.norm and case.density:   # out = 1 on every path
        np.testing.assert_array_equal(got, 1.0)
        return
    err, row_err = fc.errors(got, want)
    assert err <= fc.TOL, f"{case.name}: rel-L2 {err:.3e} > {fc.TOL:g}"
    assert row_err.max() <= fc.ROW_TOL, f"{case.name}: row {row_err.argmax()} rel-L2 {row_err.max():.3e} > {fc.ROW_TOL:g}"
    assert info["family"] == case.family, (case.name, info)
    # the one-term kernels ran: float16-class, not the three-term path's FP32-class result
    diff = np.linalg.norm(got - three) / np.linalg.norm(three)
    assert diff > 1e-7, f"{case.name}: the one-term result equals the three-term one ({diff:.2e})"
    if case.repeat:
        assert info["bitwise_repeat"], f"{case.name}: a repeated run differs"


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_case_matches_oracle(case):
    check(case, *run_case(case))


CHILD = """
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import f16x1_cases as fc
from test_f16x1_gpu import run_case
env = tuple(map(tuple, json.loads(sys.argv[4])))
infos = {}
for c in fc.all_cases():
    if c.env == env:
        got, infos[c.name], three = run_case(c)
        np.save(f"{sys.argv[3]}/{c.name}.npy", got)
        np.save(f"{sys.argv[3]}/{c.name}.three.npy", three)
with open(f"{sys.argv[3]}/infos.json", "w") as f:
    json.dump(infos, f)
"""


@pytest.mark.parametrize("env", sorted({c.env for c in ENV_CASES}), ids=lambda env: ",".join("=".join(kv) for kv in env))
def test_cases_under_environment_knobs(env, tmp_path):
    """KMB_TENSOR_PAIR=0 (read once per process): a child process hands its results back through .npy files."""
    res = subprocess.run([sys.executable, "-c", CHILD, REPO, os.path.join(REPO, "tests"), str(tmp_path), json.dumps(env)],
                         env=dict(os.environ, **dict(env)), capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    infos = json.loads((tmp_path / "infos.json").read_text())
    cases = [c for c in ENV_CASES if c.env == env]
    assert sorted(infos) == sorted(c.name for c in cases)
    for c in cases:
        check(c, np.load(tmp_path / f"{c.name}.npy"), infos[c.name], np.load(tmp_path / f"{c.name}.three.npy"))


@pytest.mark.parametrize("kernel, D, E", [("gaussian", 3, 1), ("gaussian", 784, 1), ("absolute-exponential", 64, 64),
                                          ("dot-exponential", 3, 64), ("dot-exponential", 40, 4), ("gaussian", 200, 8)])
def test_prepared_run_is_bitwise_the_unprepared_run(kernel, D, E):
    """The prepass of fit() (product.prepare_points, at every D on this path) gives bitwise the product that does its own
    prepass, and a repeated run is bitwise identical."""
    from kernel_matrix_benchmarks_b200 import product

    case = fc.Case(f"prepared-{kernel}-D{D}-E{E}", kernel, N=401, M=1500, D=D, E=E, norm=True)
    x, y, b = fc.make_data(case)
    tx, ty, tb = _t(x), _t(y), _t(b)
    ws = product.Workspace()
    need = product.workspace_bytes(case.N, case.M, D, E, kernel=kernel, normalize_rows=True, path=PATH)
    token = product.prepare_points(tx, ty, kernel=kernel, path=PATH, workspace=ws, min_bytes=need)
    assert token is not None
    prepared = product.kernel_product(tx, ty, tb, kernel=kernel, normalize_rows=True, path=PATH, workspace=ws,
                                      prepared=token).cpu().numpy()
    assert ws.buf is token   # the workspace was not reallocated: the product skipped its prepass
    plain = [product.kernel_product(tx, ty, tb, kernel=kernel, normalize_rows=True, path=PATH).cpu().numpy() for _ in range(2)]
    assert np.array_equal(prepared.view(np.uint8), plain[0].view(np.uint8))
    assert np.array_equal(plain[0].view(np.uint8), plain[1].view(np.uint8))


@pytest.mark.parametrize("D,E", [(64, 64), (64, 4), (3, 64), (200, 8)])
def test_dot_attention_beyond_fp32_exp_range(D, E):
    """Attention rows whose largest <x, y> is about 120: exp overflows FP32 there; the online maximum keeps the one-term
    result finite and inside the tolerance."""
    from kernel_matrix_benchmarks_b200 import product

    case = fc.Case(f"far-D{D}-E{E}", "dot-exponential", N=401, M=1500, D=D, E=E, norm=True)
    x, y, b = fc.make_data(case)
    far = np.array([0, 1, 127, 128, 200, 400])
    s = x[far] @ y.T
    x[far] *= (120.0 / s.max(axis=1))[:, None]
    x = x.astype(np.float32).astype(np.float64)
    top = (x[far] @ y.T).max(axis=1)
    with np.errstate(over="ignore"):
        assert (top > 110).all() and np.isinf(np.exp(top.astype(np.float32))).all()
    got = product.kernel_product(_t(x), _t(y), _t(b), kernel="dot-exponential", normalize_rows=True, path=PATH).cpu().numpy()
    want = dxo.kernel_product(y, x, b, normalize_rows=True)
    assert np.isfinite(got).all()
    err, row_err = fc.errors(got, want)
    assert err <= fc.TOL and row_err.max() <= fc.ROW_TOL, (err, row_err[far])


def _plugin(kernel, x, y, b, *, precision="float32", norm=False, **kw):
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    algo = B200Product(kernel=kernel, dimension=y.shape[1], normalize_rows=norm, precision=precision, path=PATH, **kw)
    algo.prepare_data(source_points=y, target_points=x, same_points=False, density_estimation=False)
    algo.fit()
    algo.prepare_query(source_signal=b)
    algo.query()
    got, extra = algo.get_result(), algo.get_additional()
    algo.done()
    return got, extra


@pytest.mark.parametrize("precision", ["float32", "float16"])
@pytest.mark.parametrize("kernel, D, E, norm", [("gaussian", 784, 1, False), ("gaussian", 64, 64, True),
                                                ("absolute-exponential", 64, 64, True), ("dot-exponential", 64, 64, True),
                                                ("gaussian", 3, 1, False)])
def test_plugin_end_to_end(precision, kernel, D, E, norm):
    """B200Product(path="tensor_f16x1"): prepare_data / fit (prepass) / prepare_query / query / get_result.  float16
    rounds the inputs to half precision as the reference's astype does; the oracle sees the same rounded inputs."""
    case = fc.Case(f"plugin-{kernel}-D{D}-E{E}-n{int(norm)}", kernel, N=700, M=1500, D=D, E=E, norm=norm)
    x, y, b = fc.make_data(case)
    got, extra = _plugin(kernel, x, y, b, precision=precision, norm=norm)
    r = (lambda a: a.astype(np.float16).astype(np.float64)) if precision == "float16" else (lambda a: a)
    want = oracle(kernel, r(x), r(y), r(b), normalize_rows=norm)
    err, row_err = fc.errors(got, want)
    assert err <= fc.TOL and row_err.max() <= fc.ROW_TOL, (err, row_err.max(), extra)
    assert extra["path_used"] == PATH, extra


def test_two_gpus_rows_mode():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    case = fc.Case("two-gpus", "gaussian", N=1000, M=1500, D=64, E=64, norm=True)
    x, y, b = fc.make_data(case)
    got, extra = _plugin("gaussian", x, y, b, norm=True, n_gpus=2)
    assert extra["n_gpus"] == 2 and extra["path_used"] == PATH, extra
    want = oracle("gaussian", x, y, b, normalize_rows=True)
    err, row_err = fc.errors(got, want)
    assert err <= fc.TOL and row_err.max() <= fc.ROW_TOL, (err, row_err.max())
