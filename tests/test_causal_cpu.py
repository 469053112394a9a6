"""Causal products (KMB_FLAG_CAUSAL) without a GPU: the float64 oracle against the literal masked formula, the plan of
every case, what is rejected, the causal wave schedule of the kernels (kmb_debug_causal_work) and the multi-GPU row split."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

import causal_cases as cc
import causal_oracle as co

from kernel_matrix_benchmarks_b200 import _lib
from kernel_matrix_benchmarks_b200 import product as prod

KERNELS = ("gaussian", "absolute-exponential", "inverse-distance", "dot-exponential")


# ---------------------------------------------------------------------------------------------------- oracle
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("row_offset", [0, 3, 40])
@pytest.mark.parametrize("shape", [(17, 23), (30, 11)])
def test_oracle_matches_literal_tril(kernel, row_offset, shape):
    N, M = shape
    rng = np.random.RandomState(N + M + row_offset)
    x, y, b = 0.7 * rng.randn(N, 5), 0.7 * rng.randn(M, 5), rng.randn(M, 3)
    K = co.kernel_matrix(kernel, x, y, row_offset)
    T = np.tril(K, row_offset)
    np.testing.assert_allclose(co.causal_product(kernel, x, y, b, row_offset=row_offset, block=7), T @ b, rtol=1e-12, atol=1e-12)
    with np.errstate(invalid="ignore"):   # inverse distance, row 0 at row_offset 0: its one visible source is zeroed, 0 / 0
        norm = co.causal_product(kernel, x, y, b, row_offset=row_offset, normalize_rows=True, block=7)
        want = (T @ b) / T.sum(1, keepdims=True)
    np.testing.assert_allclose(norm, want, rtol=1e-12, atol=1e-12)
    dens = co.causal_product(kernel, x, y, None, row_offset=row_offset, density_estimation=True, block=7)
    np.testing.assert_allclose(dens, T.sum(1, keepdims=True), rtol=1e-12, atol=1e-12)
    assert np.all(co.causal_product(kernel, x, y, None, normalize_rows=True, density_estimation=True) == 1.0)


def test_oracle_dot_exponential_subtracts_the_visible_row_maximum():
    rng = np.random.RandomState(3)
    x, y, b = 12.0 * rng.randn(20, 8), 12.0 * rng.randn(40, 8), rng.randn(40, 2)
    got = co.causal_product("dot-exponential", x, y, b, row_offset=5, normalize_rows=True, block=6)
    assert np.all(np.isfinite(got))
    s = x @ y.T
    for i in range(20):
        v = s[i, : 5 + i + 1]
        w = np.exp(v - v.max())
        np.testing.assert_allclose(got[i], w @ b[: 5 + i + 1] / w.sum(), rtol=1e-12, atol=1e-12)


# ---------------------------------------------------------------------------------------------------- plans
@pytest.mark.parametrize("case", [c for c in cc.CASES if not c.env], ids=lambda c: c.id)
def test_case_reaches_its_family(case):
    plan = prod.dispatch_plan(case.N, case.M, case.D, case.E, kernel=case.kernel, normalize_rows=case.norm,
                              density_estimation=case.density, causal=True)
    assert plan["path"] == "tensor_f16"
    assert plan["family"] == case.family
    assert plan["passes"] == case.passes


def test_pair_off_cases_reach_the_single_cta_families():
    cases = [c for c in cc.CASES if c.env == cc.PAIR_OFF]
    code = ("import json, sys; from kernel_matrix_benchmarks_b200 import product as p; cs = json.loads(sys.argv[1]); "
            "print(json.dumps([p.dispatch_plan(*c[:4], kernel=c[4], normalize_rows=c[5], causal=True)['family'] for c in cs]))")
    arg = json.dumps([[c.N, c.M, c.D, c.E, c.kernel, c.norm] for c in cases])
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", code, arg], env=dict(os.environ, **dict(cc.PAIR_OFF), PYTHONPATH=repo),
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    assert json.loads(res.stdout) == [c.family for c in cases]


@pytest.mark.parametrize("path", ["direct", "direct_diff", "direct_sym", "tensor_tf32", "tensor_f16x1"])
def test_paths_without_causal_kernels_are_rejected(path):
    with pytest.raises(NotImplementedError):
        prod.workspace_bytes(1000, 1000, 3, 1, path=path, causal=True)
    with pytest.raises(NotImplementedError):
        prod.dispatch_plan(1000, 1000, 64, 1, path=path, causal=True)


def test_tf32_pb_shape_is_rejected():
    """Inverse distance with E > 4, D <= 128: the FP16 path hands it to the TF32 P.B kernel, which has no causal form."""
    for call in (lambda: prod.workspace_bytes(500, 500, 64, 8, kernel="inverse-distance", causal=True),
                 lambda: prod.dispatch_plan(500, 500, 64, 8, kernel="inverse-distance", causal=True),
                 lambda: prod.pv_plan(500, 500, 64, 8, kernel="inverse-distance", causal=True, sms=148, smem_optin=232448)):
        with pytest.raises(NotImplementedError):
            call()
    # the same kernel at E <= 4 or D > 128 has one
    assert prod.dispatch_plan(500, 500, 64, 4, kernel="inverse-distance", causal=True)["family"] == "tensor_pair"
    assert prod.dispatch_plan(500, 500, 200, 8, kernel="inverse-distance", causal=True)["family"] == "tensor_pair"


def test_unsupported_codes_through_the_c_abi():
    import ctypes

    lib = _lib.load()
    need = ctypes.c_size_t(0)
    plan = (ctypes.c_int64 * 10)()
    for path in (1, 2, 3, 4, 6):
        assert lib.kmb_product_workspace_bytes(256, 256, 3, 1, 0, _lib.FLAG_CAUSAL, path, ctypes.byref(need)) == _lib.KMB_ERR_UNSUPPORTED
        assert lib.kmb_debug_product_plan(256, 256, 3, 1, 0, _lib.FLAG_CAUSAL, path, 148, plan) == _lib.KMB_ERR_UNSUPPORTED
    assert lib.kmb_debug_product_plan(256, 256, 3, 1, 0, _lib.FLAG_CAUSAL, 0, 148, plan) == _lib.KMB_OK
    assert lib.kmb_debug_product_plan(256, 256, 3, 1, 0, 16, 0, 148, plan) == _lib.KMB_ERR_INVALID   # bit 4 stays unknown


@pytest.mark.parametrize("D,E,kernel", [(3, 1, "gaussian"), (16, 2, "absolute-exponential"), (3, 64, "inverse-distance"),
                                        (64, 64, "gaussian"), (784, 1, "dot-exponential")])
def test_auto_resolves_to_tensor_f16(D, E, kernel):
    if kernel == "inverse-distance":
        E = 4
    assert prod.dispatch_plan(1000, 1000, D, E, kernel=kernel, causal=True)["path"] == "tensor_f16"
    assert prod.resolved_path(D, E, kernel, "auto", causal=True) == "tensor_f16"


def test_symmetric_never_applies_under_causal():
    class T:   # the attributes symmetric_applies looks at
        shape = (100000, 3)

        @staticmethod
        def data_ptr():
            return 1

    assert prod.symmetric_applies(T, T, "gaussian")
    assert not prod.symmetric_applies(T, T, "gaussian", causal=True)


# ---------------------------------------------------------------------------------------------------- schedule
def _schedule(N, M, D, E, kernel="gaussian", norm=True, row_offset=0, sms=148):
    """Every (wave, unit) work item of the causal kernel: {tile: [(sb_lo, sb_hi, c, Cw)]}, per-unit block totals."""
    first = prod.causal_work(N, M, D, E, 0, 0, kernel=kernel, normalize_rows=norm, row_offset=row_offset, sms=sms)
    tiles, order = {}, []
    per_unit, n_items = np.zeros(first["units"], dtype=np.int64), np.zeros(first["units"], dtype=np.int64)
    for w in range(first["waves"]):
        for u in range(first["units"]):
            ww = prod.causal_work(N, M, D, E, w, u, kernel=kernel, normalize_rows=norm, row_offset=row_offset, sms=sms)
            if ww["tile"] < 0:
                continue
            tiles.setdefault(ww["tile"], []).append((ww["sb_lo"], ww["sb_hi"], ww["c"], ww["Cw"]))
            per_unit[u] += ww["sb_hi"] - ww["sb_lo"]
            n_items[u] += 1
            if ww["c"] == 0:
                order.append(ww["tile"])
    return first, tiles, per_unit, order, n_items


@pytest.mark.parametrize("N,M,D,E,kernel,row_offset", [
    (262144, 262144, 64, 64, "dot-exponential", 0),     # C4: pv16_pair
    (65536, 65536, 64, 1, "gaussian", 0),                # tensor_pair
    (256, 65536, 64, 64, "gaussian", 0),                 # many ranges per tile, empty ones
    (256, 65536, 64, 1, "gaussian", 77),
    (1000, 3000, 64, 8, "gaussian", 1000),
    (100, 5000, 200, 4, "gaussian", 4000),               # one tile (single CTA)
    (5000, 300, 16, 2, "absolute-exponential", 129),
])
def test_causal_schedule_covers_exactly_the_visible_blocks(N, M, D, E, kernel, row_offset):
    first, tiles, _, order, _ = _schedule(N, M, D, E, kernel, True, row_offset)
    block = first["block"]
    pair = first["family"].endswith("_pair")
    rows_per_unit = 256 if pair else 128
    units_of_tiles = -(-N // rows_per_unit)
    nsb = -(-M // block)
    assert sorted(tiles) == list(range(units_of_tiles))
    assert sorted(order) == list(range(units_of_tiles))   # the serpentine visits every tile once
    for t, ranges in tiles.items():
        last_row = min(N, (t + 1) * rows_per_unit) - 1
        nb_t = min(nsb, (row_offset + last_row) // block + 1)
        ranges.sort(key=lambda r: r[2])
        Cw = ranges[0][3]
        assert [r[2] for r in ranges] == list(range(Cw))
        lo = 0
        for sb_lo, sb_hi, _, _ in ranges:   # disjoint, in order, covering [0, nb_t): nothing beyond the diagonal
            assert sb_lo == lo and sb_hi >= sb_lo
            lo = sb_hi
        assert lo == nb_t


def test_empty_ranges_occur():
    _, tiles, _, _, _ = _schedule(256, 65536, 64, 64, "gaussian", True, 0)
    assert any(lo == hi for ranges in tiles.values() for lo, hi, _, _ in ranges)


def test_c4_serpentine_balances_the_units():
    """At C4 the units that work on the same number of row tiles (the last wave is short, as in the full product) end
    within one wave's spread of each other, and the busiest unit has about half the blocks of the full product's."""
    N = 262144
    first, tiles, per_unit, _, n_items = _schedule(N, N, 64, 64, "dot-exponential", True, 0)
    rows = 256 if first["family"].endswith("_pair") else 128
    wave_spread = first["units"] * rows // first["block"]   # the first and last tile of a wave differ by this many blocks
    for k in set(n_items.tolist()):
        same = per_unit[n_items == k]
        assert same.max() - same.min() <= wave_spread
    nsb = -(-N // first["block"])
    assert abs(per_unit.sum() / (len(tiles) * nsb) - 0.5) < 0.01
    assert per_unit.max() / (n_items.max() * nsb) < 0.53


# ---------------------------------------------------------------------------------------------------- row split
@pytest.mark.parametrize("n,world", [(262144, 2), (262144, 8), (1000, 4), (100, 3), (5, 2)])
def test_causal_row_split(n, world):
    bounds = [prod.causal_row_bounds(n, r, world) for r in range(world)]
    assert bounds[0][0] == 0 and bounds[-1][1] == n
    for (a, b), (c, d) in zip(bounds, bounds[1:]):
        assert b == c and a <= b
    for lo, hi in bounds[:-1]:
        assert hi % 128 == 0 or hi == n
    if n >= 128 * world * 8:   # equal shares of the triangle, up to a tile
        work = [(hi * (hi + 1) - lo * (lo + 1)) / 2 for lo, hi in bounds]
        total = n * (n + 1) / 2
        for wk in work:
            assert abs(wk / total - 1 / world) < 2 * 128 / n * world
