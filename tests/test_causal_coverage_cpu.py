"""Coverage of the causal-product cases (tests/causal_coverage_cases.py), host logic only: every case reaches the
instantiation and the schedule regimes it claims (product.dispatch_plan, product.causal_work); every causal tensor
instantiation, every float64 causal instantiation, every regime and every diagonal edge of every family has a case; and
the diagonal data make a mask one source off visible on every row the GPU test checks."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

import causal_coverage_cases as ccc
import causal_oracle as co

from kernel_matrix_benchmarks_b200 import product as prod

CASES = ccc.all_cases()
IN_PROCESS = [c for c in CASES if not c.env]
KNOB = [c for c in CASES if c.env]
WORST_ROW = ccc.WORST_ROW   # the GPU test's worst-row bound
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _plan(case):
    return prod.dispatch_plan(case.N, case.M, case.D, case.signal_cols, kernel=case.kernel,
                              normalize_rows=case.norm and not case.density, density_estimation=case.density, causal=True,
                              sms=ccc.SMS)


def _ep(chunk):
    """kprod_tensor's EP for the plan's chunk (launch_ep: 1, 2, else 4)."""
    return chunk if chunk in (1, 2) else 4


def _check_claims(case, plan, reached):
    assert plan["path"] == "tensor_f16", case.name
    assert plan["family"] == case.family, (case.name, plan["family"])
    assert plan["passes"] == case.passes, (case.name, plan["passes"])
    if case.family.startswith("tensor"):
        assert _ep(plan["chunk"]) == case.ep, (case.name, plan["chunk"])
    else:
        assert case.ep is None
    assert case.target in ccc.TARGETS, case.name
    missing = sorted(set(case.regimes) - reached)
    assert not missing, f"{case.name} does not reach {missing}; it reaches {sorted(reached)}"
    assert set(case.regimes) <= set(ccc.REGIMES)


@pytest.mark.parametrize("case", IN_PROCESS, ids=[c.name for c in IN_PROCESS])
def test_case_reaches_what_it_claims(case):
    _check_claims(case, _plan(case), ccc.reached(case))
    if case.data == "diagonal":   # the diagonal (+1) of every row is a real source
        assert case.row_offset + case.N <= case.M - 1, case.name


KNOB_CHILD = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import causal_coverage_cases as ccc
from kernel_matrix_benchmarks_b200 import product as prod
out = {}
for c in ccc.from_json(sys.argv[3]):
    plan = prod.dispatch_plan(c.N, c.M, c.D, c.signal_cols, kernel=c.kernel, normalize_rows=c.norm, causal=True, sms=ccc.SMS)
    fam = prod.causal_work(c.N, c.M, c.D, c.signal_cols, 0, 0, kernel=c.kernel, normalize_rows=c.norm, sms=ccc.SMS)["family"]
    assert fam == plan["family"]
    out[c.name] = [plan, sorted(ccc.reached(c, fam))]
print(json.dumps(out))
"""


def knob_plans():
    """{case name: (plan, reached regimes)} of the knob cases, each environment in a child process."""
    out = {}
    for env in sorted({c.env for c in KNOB}):
        cases = ccc.to_json([c for c in KNOB if c.env == env])
        res = subprocess.run([sys.executable, "-c", KNOB_CHILD, REPO, os.path.join(REPO, "tests"), cases],
                             env=dict(os.environ, **dict(env)), capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
        for name, (plan, reached) in json.loads(res.stdout.strip().splitlines()[-1]).items():
            out[name] = (plan, frozenset(reached))
    return out


def test_knob_cases_reach_what_they_claim():
    plans = knob_plans()
    assert sorted(plans) == sorted(c.name for c in KNOB)
    for c in KNOB:
        plan, reached = plans[c.name]
        _check_claims(c, plan, reached)


# ---- coverage -----------------------------------------------------------------------------------------------------------


def coverage_gaps(cases, knob_reached=None):
    """(instantiations without a positive-data case and a diagonal-data case at the diagonal edge G - 2, f64
    instantiations without a case, regimes without a case that claims and reaches them, (family, diagonal edge) without
    a diagonal-data case)."""
    knob_reached = knob_reached or {}

    def reach(c):
        return knob_reached[c.name] if c.env else ccc.reached(c)

    have = {}
    for c in cases:
        if c.data == "positive" or "diag_edge_m2" in reach(c):
            have.setdefault(c.target, set()).add(c.data)
    inst = [t for t in ccc.TARGETS if have.get(t, set()) != {"positive", "diagonal"}]
    f64 = set()
    for c in ccc.f64_cases():
        f64 |= {(c.kernel, ec) for ec in ccc.f64_instantiations(c.D, c.E)}
    f64_gaps = [t for t in ccc.F64_TARGETS if t not in f64]
    regimes, edges = set(), set()
    for c in cases:
        r = reach(c)
        regimes |= set(c.regimes) & r
        if c.data == "diagonal":
            edges |= {(c.family, e) for e in ccc.DIAG_EDGES if e in r}
    edge_gaps = [(f, e) for f in ccc.FAMILIES for e in ccc.DIAG_EDGES if (f, e) not in edges]
    return inst, f64_gaps, sorted(set(ccc.REGIMES) - regimes), edge_gaps


def test_every_instantiation_regime_and_diagonal_edge_has_a_case():
    knob = {n: r for n, (_, r) in knob_plans().items()}
    inst, f64, regimes, edges = coverage_gaps(CASES, knob)
    n_t, n_f = len(ccc.TARGETS), len(ccc.F64_TARGETS)
    print(f"\nCAUSAL_COVERAGE tensor instantiations {n_t - len(inst)} / {n_t} ({len(ccc.TENSOR_TARGETS)} kprod_tensor, "
          f"{len(ccc.PV16_TARGETS)} pv16), f64 causal instantiations {n_f - len(f64)} / {n_f}, "
          f"regimes {len(ccc.REGIMES) - len(regimes)} / {len(ccc.REGIMES)}, "
          f"diagonal edges {4 * len(ccc.DIAG_EDGES) - len(edges)} / {4 * len(ccc.DIAG_EDGES)}")
    assert n_t == 44 and n_f == 20
    assert not inst, f"instantiations without a positive-data case and a diagonal-data case at G - 2: {inst}"
    assert not f64, f"f64 causal instantiations without a case: {f64}"
    assert not regimes, f"regimes no case claims and reaches: {[(r, ccc.REGIMES[r]) for r in regimes]}"
    assert not edges, f"diagonal edges ({ccc.DIAG_EDGE_NOTE}) without a diagonal-data case: {edges}"
    # the report names what goes missing with the last case of a regime or an instantiation
    last = [c for c in CASES if "ro_above_2_31" in c.regimes]
    assert coverage_gaps([c for c in CASES if c not in last], knob)[2] == ["ro_above_2_31"]
    t = ("pv16", None, "absolute-exponential", False)
    assert coverage_gaps([c for c in CASES if c.target != t], knob)[0] == [t]


def test_f64_cases_span_several_ctas_off_the_cta_size():
    for c in ccc.f64_cases():
        rows = ccc.F64_WIDE_ROWS_PER_CTA if c.D > ccc.F64_MAX_D else ccc.F64_ROWS_PER_CTA
        assert c.N > 2 * rows and c.N % rows and c.row_offset % rows, c.name
        assert c.row_offset + c.N <= c.M, c.name


def test_sampled_rows_include_every_tile_edge():
    tm = ccc.geometry()[0]
    for c in CASES:
        if not c.sampled:
            continue
        rows = set(ccc.sample_rows(c).tolist())
        assert {0, c.N - 1} <= rows and len(rows) >= 256
        for t0 in range(0, c.N, tm):
            assert t0 in rows and min(t0 + tm, c.N) - 1 in rows, c.name


# ---- sensitivity of the diagonal data ---------------------------------------------------------------------------------


def masked_oracle(case, x, y, b, rows, shifts=(0,)):
    """The causal product at ``rows`` in float64 with the mask moved by ``shift`` sources -- row i sees j <= row_offset +
    i + shift -- and the inverse-distance zeroing rule left where it is.  Returns {shift: (out, out under |b|)}; a row
    that sees no source is NaN."""
    M, ro = case.M, case.row_offset
    norm = case.norm and not case.density
    bb = np.ones((M, 1)) if b is None else b
    res = {s: (np.empty((len(rows), bb.shape[1])), np.empty((len(rows), bb.shape[1]))) for s in shifts}
    at = 0
    for r0, r1 in ccc.runs(rows):
        jmax = int(min(M, max(0, ro + r1 + max(shifts))))
        i = ro + np.arange(r0, r1)[:, None]
        j = np.arange(jmax)[None, :]
        if case.kernel == "dot-exponential" and norm:
            s_full = x[r0:r1] @ y[:jmax].T
        else:
            k_full = co.kernel_matrix(case.kernel, x[r0:r1], y[:jmax], ro, r0, M)
        for s in shifts:
            vis = j <= i + s
            with np.errstate(invalid="ignore", divide="ignore"):
                if case.kernel == "dot-exponential" and norm:
                    sm = np.where(vis, s_full, -np.inf)
                    k = np.exp(sm - sm.max(axis=1, keepdims=True)) if jmax else np.zeros((r1 - r0, 0))
                    k = np.where(vis, k, 0.0)
                else:
                    k = np.where(vis, k_full, 0.0)
                out, out_abs = k @ bb[:jmax], k @ np.abs(bb[:jmax])
                if norm:
                    ks = k.sum(axis=1, keepdims=True)
                    out, out_abs = out / ks, out_abs / ks
            empty = ~vis.any(axis=1)
            out[empty], out_abs[empty] = np.nan, np.nan
            res[s][0][at:at + r1 - r0], res[s][1][at:at + r1 - r0] = out, out_abs
        at += r1 - r0
    return res


def test_masked_oracle_without_shift_is_the_oracle():
    tm = ccc.geometry()[0]
    for kernel in ccc.KERNELS:
        for norm in (False, True):
            c = ccc.Case(f"pin-{kernel}-{norm}", kernel, 2 * tm + 5, 3 * tm + 40, 16, 3, norm, 37, "any", data="diagonal")
            x, y, b = ccc.make_data(c)
            rows = np.array([0, 1, 2, 50, 51, 200, 2 * tm + 4])
            got = masked_oracle(c, x, y, b, rows)[0][0]
            want = co.causal_product(kernel, x, y, b, row_offset=c.row_offset, normalize_rows=norm)[rows]
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)


DIAG = [c for c in CASES if c.data == "diagonal"]


@pytest.mark.parametrize("case", DIAG, ids=[c.name for c in DIAG])
def test_diagonal_data_show_a_mask_one_source_off(case):
    """On every row the GPU test checks, the oracle with the mask moved by +1 or -1 source differs from the true oracle by
    more than the worst-row tolerance, and by 10x that on the median row.  The change is measured as the GPU test measures
    errors: per row, relative to the row's norm under |b|.

    Inverse distance, -1: the zeroing rule removes source (row_offset + i) mod (M + 1), which is the diagonal source of
    every row with row_offset + i <= M, so those rows are identical with the mask moved down by one -- in the kernel as in
    the oracle, no test can see it.  Such rows are exempt from the -1 check (and must be identical)."""
    x, y, b = ccc.make_data(case)
    rows = ccc.sample_rows(case)
    res = masked_oracle(case, x, y, b, rows, shifts=(0, 1, -1))
    want, scale = res[0]
    assert np.all(np.isfinite(want)), case.name
    report = []
    for s in (1, -1):
        got = res[s][0]
        with np.errstate(invalid="ignore"):
            ch = np.linalg.norm(got - want, axis=1) / np.linalg.norm(scale, axis=1)
        ch[~np.isfinite(ch)] = np.inf   # a row that sees nothing after the move
        check = np.ones(len(rows), dtype=bool)
        if s == -1 and case.kernel == "inverse-distance":
            zeroed_diag = (case.row_offset + rows) % (case.M + 1) == case.row_offset + rows
            assert np.all(ch[zeroed_diag] == 0.0), case.name
            check = ~zeroed_diag
        if check.any():
            assert ch[check].min() > WORST_ROW, (case.name, s, float(ch[check].min()), rows[check][np.argmin(ch[check])])
            assert np.median(ch[check]) >= 10 * WORST_ROW, (case.name, s, float(np.median(ch[check])))
            report.append(f"{s:+d}: min {ch[check].min():.2e} median {np.median(ch[check]):.2e}")
    print(f"\nCAUSAL_SENSITIVITY {case.name} ({len(rows)} rows) " + "; ".join(report))
