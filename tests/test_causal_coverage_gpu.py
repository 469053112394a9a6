"""Causal products on the GPU: every case of tests/causal_coverage_cases.py against the float64 oracle of
tests/causal_oracle.py, row by row; repeat runs of the multi-wave cases bitwise; row shards on one GPU against the full
product; every float64 causal instantiation against NumPy.

Errors are measured per row against the row's norm under |b| -- the oracle with the signal's absolute values -- so that
signed data cannot hide an error behind a cancelling row (for a positive signal this is the row's own norm):
worst row <= 1e-3, and the relative L2 error over the checked rows <= 1e-4.  Large cases are checked on sampled rows
(causal_coverage_cases.sample_rows: both ends of every tile, every row whose diagonal is at a block or column-group
edge, 256 random rows)."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

import causal_coverage_cases as ccc
import causal_oracle as co

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = ccc.all_cases()
IN_PROCESS = [c for c in CASES if not c.env]


WORST = {}


@pytest.mark.parametrize("case", IN_PROCESS, ids=[c.name for c in IN_PROCESS])
def test_case_against_oracle(case):
    from kernel_matrix_benchmarks_b200 import product as prod

    assert prod.device_info(0)["sm_count"] == ccc.SMS, "the cases are sized for the B200's SM count"
    rel, worst, same = ccc.run_case(case)
    assert same is not False, f"{case.name}: a second run differs"
    WORST[case.target] = max(WORST.get(case.target, 0.0), worst)
    print(f"\nCAUSAL_COV {case.name} target={case.target} rel-L2 {rel:.2e} worst row {worst:.2e}"
          + ("" if same is None else " repeat bitwise"))


CHILD = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import causal_coverage_cases as ccc
out = []
for c in ccc.from_json(sys.argv[3]):
    try:
        rel, worst, same = ccc.run_case(c)
        out.append([c.name, None, rel, worst, same])
    except AssertionError as e:
        out.append([c.name, str(e), None, None, None])
print(json.dumps(out))
"""


@pytest.mark.parametrize("env", sorted({c.env for c in CASES if c.env}), ids=lambda e: ",".join("=".join(kv) for kv in e))
def test_knob_cases_against_oracle(env):
    """KMB_TENSOR_PAIR=0 and KMB_PV16_FLUSH_BLOCKS=1 are read once per process: their cases run in a child."""
    cases = ccc.to_json([c for c in CASES if c.env == env])
    res = subprocess.run([sys.executable, "-c", CHILD, REPO, os.path.join(REPO, "tests"), cases],
                         env=dict(os.environ, **dict(env)), capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    rows = json.loads(res.stdout.strip().splitlines()[-1])
    assert sorted(r[0] for r in rows) == sorted(c.name for c in CASES if c.env == env)
    for name, err, rel, worst, same in rows:
        assert err is None, err
        assert same is not False, f"{name}: a second run differs"
        print(f"\nCAUSAL_COV {name} rel-L2 {rel:.2e} worst row {worst:.2e}" + ("" if same is None else " repeat bitwise"))


# ---- row shards on one GPU ----------------------------------------------------------------------------------------------

SHARD_CASES = [c for c in IN_PROCESS if c.name in ("waves2-tensor-pair-empty-first-wave", "waves2-pv16-pair-split-odd-wave",
                                                    "waves6-tensor-pair-last-reversed-abs",
                                                    "inst-pv16_pair-epNone-absolute-exponential-plain-diagonal-absolute-exponential")]


def _cuts(N):
    from kernel_matrix_benchmarks_b200 import product as prod

    out = []
    for G in (2, 3, 8):
        out.append(("G%d" % G, [prod.causal_row_bounds(N, r, G) for r in range(G)]))
    edges = sorted({0, N, N // 3 + 1, N // 2 + 63, (2 * N) // 3 - 5})   # not on 128-row tiles
    out.append(("unaligned", list(zip(edges[:-1], edges[1:]))))
    return out


@pytest.mark.parametrize("case", SHARD_CASES, ids=[c.name for c in SHARD_CASES])
def test_row_shards_match_the_full_product(case):
    """Rows [lo, hi) run with row_offset + lo, as a row shard of a multi-GPU product does: they match the full product and
    the oracle at the sampled rows and at every shard's first and last row."""
    assert len(SHARD_CASES) == 4
    x, y, b = ccc.make_data(case)
    full = ccc.run(case, x, y, b)
    for label, bounds in _cuts(case.N):
        assert bounds[0][0] == 0 and bounds[-1][1] == case.N
        got = np.concatenate([ccc.run(case, x, y, b, lo, hi) for lo, hi in bounds if hi > lo])
        edge = [r for lo, hi in bounds if hi > lo for r in (lo, hi - 1)]
        rows = np.unique(np.concatenate([ccc.sample_rows(case), edge]))
        ccc.check(case, got[rows], rows, x, y, b, f" shards {label} {bounds}")
        want, scale = ccc.oracle_rows(case, x, y, b, rows)
        rel, worst, at = ccc.errors(got[rows], full[rows], scale)
        assert rel <= ccc.REL_L2 and worst <= ccc.WORST_ROW, f"{case.name} shards {label}: against the full product {rel:.2e} / {worst:.2e}"


# ---- float64 causal instantiations --------------------------------------------------------------------------------------

F64 = ccc.f64_cases()


@pytest.mark.parametrize("case", F64, ids=[c.name for c in F64])
def test_f64_instantiation_against_numpy(case):
    import torch

    from kernel_matrix_benchmarks_b200 import product as prod

    rng = np.random.RandomState(case.N + case.D + case.E)
    s = 1.0 / case.D ** 0.5
    x, y, b = s * rng.randn(case.N, case.D), s * rng.randn(case.M, case.D), rng.randn(case.M, case.E) + 0.25
    dev = torch.device("cuda", 0)
    got = prod.kernel_product_f64(torch.tensor(x, device=dev), torch.tensor(y, device=dev), torch.tensor(b, device=dev),
                                  kernel=case.kernel, normalize_rows=case.norm, row_offset=case.row_offset,
                                  causal=True).cpu().numpy()
    want = co.causal_product(case.kernel, x, y, b, row_offset=case.row_offset, normalize_rows=case.norm)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12 * np.abs(want).max(), err_msg=case.name)
