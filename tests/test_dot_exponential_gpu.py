"""The dot-exponential kernel exp(<x, y>) (not in bruteforce.py) on a B200: every parity case of
tests/dot_exponential_cases.py against the float64 oracle (tests/dot_exponential_oracle.py), the float64 path, attention
beyond FP32's exp range, same_points, prepared runs and the plugin end to end."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import dot_exponential_cases as dxc
import dot_exponential_oracle as dxo
from conftest import REPO

pytestmark = pytest.mark.gpu

KERNEL = dxc.KERNEL
CASES = [c for c in dxc.all_cases() if not c.env]
ENV_CASES = [c for c in dxc.all_cases() if c.env]


def _t(a, dtype=None):
    import torch

    return None if a is None else torch.tensor(a, dtype=dtype or torch.float32, device="cuda")


def run_case(case):
    """The case's product on cuda:0 -> (float64 result, facts about the run)."""
    from kernel_matrix_benchmarks_b200 import product

    x, y, b = dxc.make_data(case)
    tx, ty, tb = _t(x), _t(y), _t(b)

    def once():
        return product.kernel_product(tx, ty, tb, kernel=KERNEL, normalize_rows=case.norm, density_estimation=case.density,
                                      path=case.path).cpu().numpy()

    got = once()
    info = {"last_path": product.last_path}
    dev = product.device_info(0)
    info["family"] = product.dispatch_plan(case.N, case.M, case.D, case.E, kernel=KERNEL, normalize_rows=case.norm,
                                           density_estimation=case.density, path=case.path, sms=dev["sm_count"])["family"]
    if case.repeat:
        info["bitwise_repeat"] = bool(np.array_equal(once().view(np.uint8), got.view(np.uint8)))
    return got.astype(np.float64), info


def _errors(got, want):
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    row_err = np.linalg.norm(got - want, axis=1) / np.linalg.norm(want, axis=1)
    return err, row_err


def check(case, got, info):
    x, y, b = dxc.make_data(case)
    want = dxo.kernel_product(y, x, b, normalize_rows=case.norm, density_estimation=case.density)
    assert got.shape == want.shape
    assert np.isfinite(got).all(), f"{case.name}: non-finite results in rows {np.unique(np.nonzero(~np.isfinite(got))[0])[:10]}"
    err, row_err = _errors(got, want)
    assert err <= dxc.TOL, f"{case.name}: rel-L2 {err:.3e} > {dxc.TOL:g}"
    assert row_err.max() <= 10 * dxc.TOL, f"{case.name}: row {row_err.argmax()} rel-L2 {row_err.max():.3e}"
    assert info["last_path"] == ("tensor_f16" if case.path == "auto" else case.path), (case.name, info)
    assert info["family"] == ("fill" if case.norm and case.density else case.family), (case.name, info)
    if case.repeat:
        assert info["bitwise_repeat"], f"{case.name}: a repeated run differs"


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_case_matches_oracle(case):
    got, info = run_case(case)
    check(case, got, info)


CHILD = """
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import dot_exponential_cases as dxc
from test_dot_exponential_gpu import run_case
env = tuple(map(tuple, json.loads(sys.argv[4])))
infos = {}
for c in dxc.all_cases():
    if c.env == env:
        got, infos[c.name] = run_case(c)
        np.save(f"{sys.argv[3]}/{c.name}.npy", got)
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
        check(c, np.load(tmp_path / f"{c.name}.npy"), infos[c.name])


@pytest.mark.parametrize("D,E", [(5, 1), (5, 3), (5, 11), (40, 1), (40, 64), (200, 70)])
@pytest.mark.parametrize("mode", ["plain", "norm", "density"])
def test_float64_path_matches_numpy_oracle(D, E, mode):
    """kmb_product_f64: one row per thread (D <= 16, signal chunks of 1, 2, 4, 8 columns) and the tiled kernel (D > 16)."""
    import torch

    from kernel_matrix_benchmarks_b200 import product

    case = dxc.Case(f"f64-D{D}-E{E}-{mode}", N=300, M=500, D=D, E=E, norm=mode == "norm", density=mode == "density")
    x, y, b = dxc.make_data(case)
    got = product.kernel_product_f64(_t(x, torch.float64), _t(y, torch.float64), _t(b, torch.float64), kernel=KERNEL,
                                     normalize_rows=case.norm, density_estimation=case.density).cpu().numpy()
    want = dxo.kernel_product(y, x, b, normalize_rows=case.norm, density_estimation=case.density)
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    assert err <= 1e-12, err
    blk = product.kernel_block_f64(_t(x[:50], torch.float64), _t(y[:70], torch.float64), kernel=KERNEL).cpu().numpy()
    np.testing.assert_allclose(blk, np.exp(x[:50] @ y[:70].T), rtol=1e-13, atol=0)


@pytest.mark.parametrize("D,E,path", [(64, 64, "auto"), (64, 64, "tensor_tf32"), (64, 4, "auto"), (64, 4, "tensor_tf32"),
                                      (3, 64, "auto"), (200, 8, "auto"), (200, 8, "tensor_tf32")])
def test_attention_beyond_fp32_exp_range(D, E, path):
    """Attention rows whose largest <x, y> is about 120: exp overflows FP32 there (and the plain product with it), the
    online maximum of the row-normalised kernels keeps the result finite and within the tensor-path tolerance."""
    from kernel_matrix_benchmarks_b200 import product

    case = dxc.Case(f"far-D{D}-E{E}-{path}", N=401, M=700, D=D, E=E, norm=True, path=path)
    x, y, b = dxc.make_data(case)
    far = np.array([0, 1, 127, 128, 200, 400])
    s = x[far] @ y.T
    x[far] *= (120.0 / s.max(axis=1))[:, None]          # the row's largest logit: ~120
    x = x.astype(np.float32).astype(np.float64)
    top = (x[far] @ y.T).max(axis=1)
    with np.errstate(over="ignore"):
        assert (top > 110).all() and np.isinf(np.exp(top.astype(np.float32))).all()
    got = product.kernel_product(_t(x), _t(y), _t(b), kernel=KERNEL, normalize_rows=True, path=path).cpu().numpy()
    want = dxo.kernel_product(y, x, b, normalize_rows=True)
    assert np.isfinite(got).all()
    err, row_err = _errors(got, want)
    assert err <= dxc.TOL and row_err[far].max() <= 10 * dxc.TOL, (err, row_err[far])


def _plugin(x, y, b, *, precision="float32", norm=False, density=False, same_points=False, **kw):
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    algo = B200Product(kernel=KERNEL, dimension=y.shape[1], normalize_rows=norm, precision=precision, **kw)
    algo.prepare_data(source_points=y, target_points=None if same_points else x, same_points=same_points,
                      density_estimation=density)
    algo.fit()
    algo.prepare_query(source_signal=None if density else b)
    algo.query()
    got, extra = algo.get_result(), algo.get_additional()
    algo.done()
    return got, extra


@pytest.mark.parametrize("precision", ["float32", "float16", "float64"])
@pytest.mark.parametrize("D,E,norm", [(3, 1, False), (64, 64, True), (40, 4, True), (784, 1, False)])
def test_plugin_end_to_end(precision, D, E, norm):
    """B200Product(kernel="dot-exponential"): prepare_data / fit (prepass) / prepare_query / query / get_result.  float16
    rounds the inputs to half precision as the reference's astype does; the oracle sees the same rounded inputs."""
    case = dxc.Case(f"plugin-D{D}-E{E}-n{int(norm)}", N=700, M=900, D=D, E=E, norm=norm)
    x, y, b = dxc.make_data(case)
    got, extra = _plugin(x, y, b, precision=precision, norm=norm)
    r = (lambda a: a.astype(np.float16).astype(np.float64)) if precision == "float16" else (lambda a: a)
    want = dxo.kernel_product(r(y), r(x), r(b), normalize_rows=norm)
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    assert err <= (1e-12 if precision == "float64" else dxc.TOL), (err, extra)
    assert extra["path_used"] == ("direct_f64" if precision == "float64" else "tensor_f16"), extra


def test_same_points_takes_the_tensor_path():
    """same_points with D = 3, E = 1 and N >= 32768: the kernels of bruteforce.py take the symmetric kernel here; this one
    must not."""
    case = dxc.Case("same-points", N=40000, M=40000, D=3, E=1)
    x, y, b = dxc.make_data(case)
    got, extra = _plugin(x, y, b, same_points=True)
    assert extra["path_used"] == "tensor_f16", extra
    rows = np.arange(0, 40000, 397)
    want = dxo.kernel_product_c(y, None, b, rows=rows)
    err = np.linalg.norm(got[rows] - want) / np.linalg.norm(want)
    assert err <= dxc.TOL, err


@pytest.mark.parametrize("D,E", [(3, 1), (3, 64), (40, 4), (64, 64), (200, 8)])
def test_prepared_run_is_bitwise_the_unprepared_run(D, E):
    """The prepass of fit() (product.prepare_points, at every D for this kernel) gives bitwise the product that does its
    own prepass, and a repeated run is bitwise identical."""
    from kernel_matrix_benchmarks_b200 import product

    case = dxc.Case(f"prepared-D{D}-E{E}", N=401, M=700, D=D, E=E, norm=True)
    x, y, b = dxc.make_data(case)
    tx, ty, tb = _t(x), _t(y), _t(b)
    ws = product.Workspace()
    need = product.workspace_bytes(case.N, case.M, D, E, kernel=KERNEL, normalize_rows=True)
    token = product.prepare_points(tx, ty, kernel=KERNEL, workspace=ws, min_bytes=need)
    assert token is not None
    prepared = product.kernel_product(tx, ty, tb, kernel=KERNEL, normalize_rows=True, workspace=ws, prepared=token)
    prepared = prepared.cpu().numpy()
    assert ws.buf is token   # the workspace was not reallocated: the product skipped its prepass
    plain = [product.kernel_product(tx, ty, tb, kernel=KERNEL, normalize_rows=True).cpu().numpy() for _ in range(2)]
    assert np.array_equal(prepared.view(np.uint8), plain[0].view(np.uint8))
    assert np.array_equal(plain[0].view(np.uint8), plain[1].view(np.uint8))


def test_density_with_normalisation_is_ones():
    case = dxc.Case("norm-density", N=300, M=500, D=64, E=1, norm=True, density=True)
    x, y, _ = dxc.make_data(case)
    got, _ = _plugin(x, y, None, norm=True, density=True)
    np.testing.assert_array_equal(got, np.ones((300, 1)))


def test_two_gpus_rows_mode():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    case = dxc.Case("two-gpus", N=1000, M=900, D=64, E=64, norm=True)
    x, y, b = dxc.make_data(case)
    got, extra = _plugin(x, y, b, norm=True, n_gpus=2)
    assert extra["n_gpus"] == 2, extra
    want = dxo.kernel_product(y, x, b, normalize_rows=True)
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    assert err <= dxc.TOL, err
