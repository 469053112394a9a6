"""Coverage of the symmetric-product cases (tests/sym_cases.py), host logic only: every case reaches the geometry regimes
it claims and targets the instantiation it names; every instantiation at every D and every regime has a case; the plan
query (kmb_debug_sym_plan) rejects what the launcher rejects and partitions the unit list that kmb_debug_sym_unit
describes.  The only launcher arithmetic restated here is the stream-K split u0 = ub + Ur c / G (sym_cases.cta_range)."""
import ctypes

import numpy as np
import pytest

import sym_cases as sc

CASES = sc.all_cases()


def _half_diag2(y):
    return float((((y.max(0) - y.min(0)) / 2) ** 2).sum())


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_case_reaches_what_it_claims(case):
    reached = sc.case_regimes(case)
    missing = sorted(set(case.regimes) - reached)
    assert not missing, f"{case.name} (N={case.N}, {case.n_parts} parts) does not reach {missing}; it reaches {sorted(reached)}"
    assert set(case.regimes) <= set(sc.REGIMES)
    DP, kernel, form = case.target
    assert (kernel, form) in sc.TARGETS and DP == sc.dp_of(case.D)
    plans = sc.plans(case.N, case.D, case.kernel, case.n_parts)
    assert all(form in p["forms"] for p in plans)
    assert plans[0]["forms"] == (("difference", "product") if kernel == "gaussian" else ("difference",))
    if kernel == "gaussian" and case.N > 1:
        # the device picks the product form when log2(e) * half-diagonal^2 <= 6: keep 0.5 % away from the edge
        r2 = sc.LOG2E * _half_diag2(sc.make_points(case))
        assert (r2 <= 0.995 * sc.PRODUCT_FORM_RADIUS2) if form == "product" else (r2 >= 1.005 * sc.PRODUCT_FORM_RADIUS2), (case.name, r2)
    if case.data == "below":
        assert r2 >= 0.98 * sc.PRODUCT_FORM_RADIUS2
    if case.signal == "spike":
        b, rows = sc.make_signal(case)
        assert len(rows) >= min(4, case.N) and np.count_nonzero(b) == len(rows)
        assert len(set(np.abs(b[rows]))) == len(rows) and (len(rows) < 2 or (b[rows] < 0).any())


def coverage_gaps(cases):
    """(instantiation x D without an off-diagonal case or without a density case, regimes without a case)."""
    inst = {}
    for c in cases:
        if c.regimes and "off_diag" in c.regimes and "off_diag" in sc.case_regimes(c):
            inst.setdefault((c.D, c.kernel, c.form), set()).add(c.signal)
    gaps = []
    for kernel, form in sc.TARGETS:
        for D in sc.DIMS:
            have = inst.get((D, kernel, form), set())
            if not have:
                gaps.append(f"Sym<{sc.dp_of(D)}, {kernel}, {form}> at D={D} (off-diagonal units)")
            elif "density" not in have:
                gaps.append(f"Sym<{sc.dp_of(D)}, {kernel}, {form}> at D={D} with density")
    regimes = set()
    for c in cases:
        regimes |= set(c.regimes) & sc.case_regimes(c)
    return gaps, sorted(set(sc.REGIMES) - regimes)


def test_every_instantiation_and_regime_has_a_case():
    gaps, regimes = coverage_gaps(CASES)
    assert not gaps, f"instantiations without a case: {gaps}"
    assert not regimes, f"geometry regimes no case claims and reaches: {[(r, sc.REGIMES[r]) for r in regimes]}"
    # the gap report names what is lost when the last case of a regime or an instantiation goes
    last = [c for c in CASES if "strip_cap" in c.regimes]
    assert coverage_gaps([c for c in CASES if c not in last])[1] == ["strip_cap"]
    inst = [c for c in CASES if (c.D, c.kernel, c.form) == (1, "inverse-distance", "difference")]
    assert any("D=1" in g and "inverse-distance" in g for g in coverage_gaps([c for c in CASES if c not in inst])[0])


def _plan(*args):
    from kernel_matrix_benchmarks_b200 import _lib

    out = (ctypes.c_int64 * 15)()
    return _lib.load().kmb_debug_sym_plan(*args, out)


def test_sym_plan_rejects_what_the_launcher_rejects():
    from kernel_matrix_benchmarks_b200 import _lib, product

    lib = _lib.load()
    assert len(product.SYM_PLAN_FIELDS) == 15
    assert _plan(1000, 3, 0, 0, 1, 148) == _lib.KMB_OK
    assert lib.kmb_debug_sym_plan(1000, 3, 0, 0, 1, 148, None) == _lib.KMB_ERR_INVALID
    for args in ((0, 3, 0, 0, 1, 148), (1000, 3, 0, 0, 1, 0), (1000, 3, 0, 2, 2, 148), (1000, 3, 0, -1, 2, 148),
                 (1000, 3, 0, 0, 0, 148)):
        assert _plan(*args) == _lib.KMB_ERR_INVALID, args
    for args in ((1000, 4, 0, 0, 1, 148), (1000, 0, 0, 0, 1, 148), (1000, 3, 3, 0, 1, 148), (1000, 3, 7, 0, 1, 148)):
        assert _plan(*args) == _lib.KMB_ERR_UNSUPPORTED, args
    with pytest.raises(NotImplementedError):
        product.sym_plan(1000, 3, kernel="dot-exponential")
    with pytest.raises(ValueError):
        product.sym_plan(1000, 3, part=3, n_parts=3)


@pytest.mark.parametrize("n, n_parts, sms", [(1, 1, 148), (4097, 13, 148), (50765, 3, 148), (85091, 5, 132),
                                             (300000, 8, 148), (1_000_000, 64, 148)])
def test_sym_plan_partitions_the_unit_list(n, n_parts, sms):
    """The parts tile the unit list of kmb_debug_sym_unit (same total, strips and strip width for sms x n_parts CTAs);
    each part's first segment / strip, segment and strip counts and grid are those of its units."""
    from kernel_matrix_benchmarks_b200 import _lib, product

    lib = _lib.load()
    head = (ctypes.c_int64 * 8)()
    _lib.check(lib.kmb_debug_sym_unit(n, sms * n_parts, -1, head))
    total, n_strips, Wb = head[:3]
    # every segment of the list, in order: (strip, tile, begin, length); its index is its slot number
    segs, u = [], 0
    while u < total:
        strip, tile, block, begin, length = sc.unit(n, sms * n_parts, u)
        segs.append((strip, tile, begin, length))
        u = begin + length
    begins = np.array([s[2] for s in segs])
    prev_end = 0
    for part in range(n_parts):
        p = product.sym_plan(n, 3, part=part, n_parts=n_parts, sms=sms)
        assert (p["units"], p["n_strips"], p["Wb"]) == (total, n_strips, Wb)
        assert p["tile_rows"] == p["TB"] * p["block_sources"]
        assert p["unit_begin"] == prev_end and p["unit_end"] >= p["unit_begin"]
        prev_end = p["unit_end"]
        units = p["unit_end"] - p["unit_begin"]
        assert p["grid"] == min(sms, units)
        if units == 0:
            assert (p["segments"], p["strips"]) == (0, 0)
            continue
        first = np.searchsorted(begins, p["unit_begin"], side="right") - 1
        last = np.searchsorted(begins, p["unit_end"] - 1, side="right") - 1
        assert p["seg_base"] == first and p["segments"] == last - first + 1
        assert p["strip_base"] == segs[first][0] and p["strips"] == segs[last][0] - segs[first][0] + 1
        # every CTA range is non-empty and inside the part
        for c in range(p["grid"]):
            c0, c1 = sc.cta_range(p, c)
            assert p["unit_begin"] <= c0 < c1 <= p["unit_end"]
    assert prev_end == total


def test_strip_cap_flag():
    from kernel_matrix_benchmarks_b200 import product

    assert not product.sym_plan(1_000_000, 3)["strip_cap"]
    capped = product.sym_plan(1_000_000, 3, n_parts=64)
    assert capped["strip_cap"]
