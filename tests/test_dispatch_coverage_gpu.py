"""Parity of every product kernel instantiation the dispatcher can reach (tests/dispatch_cases.py) with the float64 C
oracle, on the float32-rounded inputs (needs a B200).

Each case runs at device level (product.kernel_product / kernel_product_f64), so the path and the row offset are the
case's own, and the test checks that the run went where the case says (product.last_path; the Gaussian evaluation form
the device picked).  Tolerances are BASELINE.json's -- relative L2 <= 1e-5 on the direct path, <= 1e-4 on the tensor
path, <= 1e-12 in float64 -- over the whole result, and 10x that for the worst row and the worst column: a whole-matrix
norm over thousands of rows can hide one wrong row of a tile or one wrong column of a signal pass.  A zero signal column
must come out as exact zeros.  P.B cases also check that this device plans the launch the case was sized for (product.pv_plan
with the device's SM count and shared memory against dispatch_cases.SMS and SMEM_OPTIN).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import dispatch_cases as dc
from conftest import REPO
from oracle import c_oracle

pytestmark = pytest.mark.gpu

CASES = [c for c in dc.all_cases() if not c.env]
ENV_CASES = [c for c in dc.all_cases() if c.env]


def run_case(case):
    """The case's product on cuda:0 -> (result as float64 numpy, facts about the run)."""
    import torch

    from kernel_matrix_benchmarks_b200 import product

    x, y, b = dc.make_data(case)
    dt = torch.float64 if case.precision == "float64" else torch.float32
    t = lambda a: None if a is None else torch.tensor(a, dtype=dt, device="cuda")
    tx, ty, tb = t(x), t(y), t(b)

    def once():
        if case.precision == "float64":
            out = product.kernel_product_f64(tx, ty, tb, kernel=case.kernel, normalize_rows=case.norm,
                                             density_estimation=case.density, row_offset=case.row_offset)
        else:
            out = product.kernel_product(tx, ty, tb, kernel=case.kernel, normalize_rows=case.norm,
                                         density_estimation=case.density, path=case.path, row_offset=case.row_offset)
        return out.cpu().numpy()   # synchronises

    got = once()
    info = {"last_path": product.last_path}
    if case.family == "direct" and case.kernel == "gaussian":
        info["form"] = product.direct_stats()["form"]
    if case.family != "f64":
        dev = product.device_info(0)
        info["family"] = product.dispatch_plan(case.N, case.M, case.D, case.E, kernel=case.kernel, normalize_rows=case.norm,
                                               density_estimation=case.density, path=case.path, sms=dev["sm_count"])["family"]
    if case.group:   # the P.B launch on this device and the one at (SMS, SMEM_OPTIN) the case was sized for
        plan = lambda sms, smem: product.pv_plan(case.N, case.M, case.D, case.E, kernel=case.kernel,  # noqa: E731
                                                 normalize_rows=case.norm, path=case.path, sms=sms, smem_optin=smem)
        info["pv_plan"] = plan(dev["sm_count"], dev["smem_per_block_optin"])
        info["pv_plan_sized"] = plan(dc.SMS, dc.SMEM_OPTIN)
    if case.repeat:
        info["bitwise_repeat"] = bool(np.array_equal(once().view(np.uint8), got.view(np.uint8)))
    return got.astype(np.float64), info


def reference(case, rows):
    """float64 oracle on the same (rounded) inputs for the local rows `rows`, with the case's global row offset."""
    x, y, b = dc.make_data(case)
    if case.row_offset:   # the oracle's zeroing rule reads the global row index: place the shard at its offset
        x = np.concatenate((np.zeros((case.row_offset, case.D)), x))
    return c_oracle.kernel_product(case.kernel, y, x, b, normalize_rows=case.norm, density_estimation=case.density,
                                   rows=rows + case.row_offset)


def check(case, got, info):
    rows = dc.check_rows(case)
    want = reference(case, rows)
    got = got[rows]
    assert got.shape == want.shape
    bad = ~np.isfinite(got)
    assert not bad.any(), (f"{case.name}: non-finite results in rows {np.unique(np.nonzero(bad)[0])[:10]}, "
                           f"columns {np.unique(np.nonzero(bad)[1])[:10]}")
    zero = np.linalg.norm(want, axis=0) == 0   # a zero signal column: exact zeros
    assert not got[:, zero].any(), f"{case.name}: nonzero results in zero columns {np.nonzero(zero)[0]}"
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    row_err = np.linalg.norm(got - want, axis=1) / np.linalg.norm(want, axis=1)
    cols = np.nonzero(~zero)[0]
    col_err = np.linalg.norm(got[:, cols] - want[:, cols], axis=0) / np.linalg.norm(want[:, cols], axis=0)
    tol = case.tol
    assert err <= tol, f"{case.name}: rel-L2 {err:.3e} > {tol:g}"
    assert row_err.max() <= 10 * tol, f"{case.name}: row {rows[row_err.argmax()]} rel-L2 {row_err.max():.3e} > {10 * tol:g}"
    assert col_err.max() <= 10 * tol, f"{case.name}: column {cols[col_err.argmax()]} rel-L2 {col_err.max():.3e} > {10 * tol:g}"
    # the run went where the case says ("auto" with D <= 16: the direct kernel, unless the case targets the FP16 P.B kernel)
    if case.precision == "float64":
        want_path = "direct_f64"
    elif case.path == "auto":
        want_path = "tensor_f16" if case.D > 16 or case.family in ("pv16", "pv16_pair") else "direct"
    else:
        want_path = case.path
    assert info["last_path"] == want_path, (case.name, info)
    if case.family != "f64":
        assert info["family"] == case.family, (case.name, info)
    if "form" in info:
        assert info["form"] == case.form, (case.name, info)
    if case.repeat:
        assert info["bitwise_repeat"], f"{case.name}: a repeated run differs"
    if case.group:   # this device runs the launch the case was sized for
        assert info["pv_plan"] == info["pv_plan_sized"], (case.name, info["pv_plan"], info["pv_plan_sized"])


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_instantiation_matches_oracle(case):
    got, info = run_case(case)
    check(case, got, info)


CHILD = """
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import dispatch_cases as dc
from test_dispatch_coverage_gpu import run_case
env = tuple(map(tuple, json.loads(sys.argv[4])))
infos = {}
for c in dc.all_cases():
    if c.env == env:
        got, infos[c.name] = run_case(c)
        np.save(f"{sys.argv[3]}/{c.name}.npy", got)
with open(f"{sys.argv[3]}/infos.json", "w") as f:
    json.dump(infos, f)
"""


@pytest.mark.parametrize("env", sorted({c.env for c in ENV_CASES}), ids=lambda env: ",".join("=".join(kv) for kv in env))
def test_instantiations_under_environment_knobs(env, tmp_path):
    """Cases that set a run-time knob (KMB_TENSOR_PAIR=0: the single-CTA FP16 kernels on multi-tile problems;
    KMB_PV16_FLUSH_BLOCKS: the flush interval of kprod_tensor_pv16) run in a child process with that environment -- the
    library reads the knobs once per process -- and hand their results back through .npy files."""
    res = subprocess.run([sys.executable, "-c", CHILD, REPO, os.path.join(REPO, "tests"), str(tmp_path), json.dumps(env)],
                         env=dict(os.environ, **dict(env)), capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    infos = json.loads((tmp_path / "infos.json").read_text())
    cases = [c for c in ENV_CASES if c.env == env]
    assert sorted(infos) == sorted(c.name for c in cases)
    for c in cases:
        check(c, np.load(tmp_path / f"{c.name}.npy"), infos[c.name])
