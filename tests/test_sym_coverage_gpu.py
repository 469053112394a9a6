"""The symmetric (same_points) product, kprod_sym, against the float64 oracle row by row, for every case of
tests/sym_cases.py (needs a B200).

The bound is per row and relative to what the row sums: |got_i - want_i| <= tol (K|b|)_i + floor.  A global rel-L2 over
a dense signal lets cancellation and the sheer number of rows hide a misplaced tile or block; this bound does not.
  * spike signals (a few nonzero entries) and density: want_i and (K|b|)_i come from the float64 oracle for every row
    (spikes: sum_k c_k k(y_i, y_jk), O(N spikes); density: the C oracle), tol = 1e-5.
  * dense signals: every row against the general direct kernel run once with the two columns [b, |b|] (whose own accuracy
    the dispatch suite pins to the float64 oracle), tol = 2e-5; and rows of every source block (two each, every row of
    the first and the last block) against the float64 C oracle, tol = 1e-5.
  * floor = 2^-126 sum_j |b_j|: the kernel's exponentials flush results below FP32's smallest normal (2^-126) to zero,
    which moves each term k_ij b_j by at most 2^-126 |b_j|; nothing else is absolute.
Multi-part cases also check each part on its own: a part's output is the float64 sum over exactly the pairs its units
own (kmb_debug_sym_unit's unit list, split as kmb_debug_sym_plan says), zero elsewhere.
"""
import numpy as np
import pytest

import sym_cases as sc
from oracle import c_oracle

pytestmark = pytest.mark.gpu

CASES = sc.all_cases()
TOL, TOL_VS_DIRECT = 1e-5, 2e-5
FLUSH = 2.0 ** -126


def _t(a):
    import torch

    return None if a is None else torch.tensor(a, dtype=torch.float32, device="cuda").reshape(len(a), -1)


def _floor(b, N):
    return FLUSH * (N if b is None else np.abs(b).sum())


def run(case, ty, tb):
    """The case's product on cuda:0: (N,) float64 total, list of per-part (N,) outputs (n_parts > 1), Gaussian form."""
    from kernel_matrix_benchmarks_b200 import product

    if case.n_parts == 1:
        out = product.kernel_product(ty, ty, tb, kernel=case.kernel, density_estimation=tb is None, path="direct_sym")
        assert product.last_path == "direct_sym"
        parts = [out.cpu().numpy()[:, 0]]
    else:
        parts = [product.kernel_product_sym_part(ty, tb, p, case.n_parts, kernel=case.kernel).cpu().numpy()[:, 0]
                 for p in range(case.n_parts)]
    form = product.direct_stats()["form"] if case.kernel == "gaussian" else "difference"
    return parts, form


def check_rows(name, got, want, kabs, tol, floor, rows=None):
    """|got - want| <= tol kabs + floor on every row; returns the largest |err| / (K|b|) seen."""
    err = np.abs(got - want)
    bad = ~(err <= tol * kabs + floor)   # NaN fails too
    if bad.any():
        i = np.nonzero(bad)[0][:8]
        ids = i if rows is None else rows[i]
        raise AssertionError(f"{name}: {bad.sum()} rows over {tol:g} (K|b|)_i + {floor:.1e}; rows {ids.tolist()}: "
                             f"got {got[i].tolist()} want {want[i].tolist()} K|b| {kabs[i].tolist()}")
    return float(np.max(err / np.maximum(kabs, np.finfo(float).tiny))) if len(err) else 0.0


def unit_map(N, total_ctas):
    """U[tile, block] = index of unit (tile, block) in the strip-ordered list, by walking it segment by segment."""
    T, S, TB = sc.tiling()
    U = np.full((-(-N // T), -(-N // S)), -1, dtype=np.int64)
    u = 0
    while True:
        strip, tile, block, begin, length = sc.unit(N, total_ctas, u)
        if strip < 0:
            break
        U[tile, block:block + length] = np.arange(begin, begin + length)
        u = begin + length
    assert (U >= 0).sum() == u
    return U


def owner_parts(case, rows):
    """Part that owns pair (i, j_k) for every row i and spike row j_k: a pair with block(j) >= TB tile(i) is a row sum of
    unit (tile(i), block(j)), any other pair a column sum of unit (tile(j), block(i))."""
    T, S, TB = sc.tiling()
    N = case.N
    U = unit_map(N, sc.SMS * case.n_parts)
    i = np.arange(N)[:, None]
    ti, bi, tj, bj = i // T, i // S, rows[None, :] // T, rows[None, :] // S
    u = np.where(bj >= TB * ti, U[ti, bj], U[tj, bi])
    assert (u >= 0).all()
    ends = np.array([p["unit_end"] for p in sc.plans(N, case.D, case.kernel, case.n_parts)])
    return np.searchsorted(ends, u, side="right")


RATIOS = {}


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_symmetric_case_matches_oracle_row_by_row(case):
    from kernel_matrix_benchmarks_b200 import product

    assert product.device_info(0)["sm_count"] == sc.SMS, "the cases are sized for the B200's SM count"
    y = sc.make_points(case)
    b, rows = sc.make_signal(case)
    ty, tb = _t(y), _t(b)
    parts, form = run(case, ty, tb)
    assert form == case.form, (case.name, form)
    got = np.sum(np.stack(parts).astype(np.float64), axis=0)
    N, floor = case.N, _floor(b, case.N)

    if case.signal == "spike":
        K = sc.spike_terms(case, y, rows)
        c = b[rows]
        want, kabs = K @ c, K @ np.abs(c)
        ratio = check_rows(case.name, got, want, kabs, TOL, floor * case.n_parts)
        if case.n_parts > 1:
            owner = owner_parts(case, rows)
            for p, out in enumerate(parts):
                mine = owner == p
                check_rows(f"{case.name} part {p}", out.astype(np.float64), (K * mine) @ c, (K * mine) @ np.abs(c), TOL,
                           floor)
    elif case.signal == "density":
        want = c_oracle.kernel_product(case.kernel, y, None, None, density_estimation=True)[:, 0]
        ratio = check_rows(case.name, got, want, want, TOL, floor)
    else:
        # every row against the general direct kernel on [b, |b|]
        ref = product.kernel_product(ty, ty, _t(np.stack([b, np.abs(b)], 1)), kernel=case.kernel, path="direct")
        ref = ref.cpu().numpy().astype(np.float64)
        check_rows(f"{case.name} vs direct", got, ref[:, 0], ref[:, 1], TOL_VS_DIRECT, floor)
        # two rows of every source block and every row of the first and the last block against the float64 oracle
        T, S, TB = sc.tiling()
        rng = np.random.RandomState(7)
        blocks = np.arange(0, N, S)
        pick = (blocks[:, None] + rng.randint(0, S, size=(len(blocks), 2))) % N
        ids = np.unique(np.concatenate([pick.ravel(), np.arange(min(S, N)), np.arange(max(0, N - S), N)]))
        w = c_oracle.kernel_product(case.kernel, y, None, np.stack([b, np.abs(b)], 1), rows=ids)
        ratio = check_rows(f"{case.name} vs oracle", got[ids], w[:, 0], w[:, 1], TOL, floor, rows=ids)

    if case.repeat:
        again, _ = run(case, ty, tb)
        for p, (a1, a2) in enumerate(zip(parts, again)):
            assert np.array_equal(a1.view(np.uint32), a2.view(np.uint32)), f"{case.name}: part {p} differs on a second run"
    RATIOS[case.name] = ratio
    print(f"\nSYM_RATIO {case.name} DP{case.target[0]} {case.kernel} {case.form} max |err|/(K|b|) = {ratio:.3e}")


# ---- several GPUs: kmb_product_sym_multi_f32 through the plugin's n_gpus ----------------------------------------------


def _n_devices():
    import torch

    return torch.cuda.device_count()


@pytest.mark.parametrize("which", ["two", "all"])
def test_symmetric_product_on_several_gpus(which):
    """The unit list split over 2 GPUs and over every GPU of the box (at most 8), partial vectors added on the first
    device: every row against the float64 spike oracle."""
    have = _n_devices()
    if have < 2:
        pytest.skip("needs two or more GPUs in one box")
    n_gpus = 2 if which == "two" else min(have, 8)
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    case = next(c for c in CASES if c.name == "geo-mid")
    y = sc.make_points(case)
    b, rows = sc.make_signal(case)
    algo = B200Product(kernel=case.kernel, dimension=case.D, precision="float32", n_gpus=n_gpus)
    try:
        algo.prepare_data(source_points=y, target_points=y, same_points=True, density_estimation=False)
        algo.fit()
        algo.prepare_query(source_signal=b[:, None])
        algo.query()
        got, extra = algo.get_result()[:, 0], algo.get_additional()
    finally:
        algo.done()
    assert extra["n_gpus"] == n_gpus and extra["path_used"] == "direct_sym", extra
    K = sc.spike_terms(case, y, rows)
    c = b[rows]
    check_rows(f"{case.name} on {n_gpus} GPUs", got, K @ c, K @ np.abs(c), TOL, n_gpus * _floor(b, case.N))
