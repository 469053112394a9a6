"""Cases for the symmetric (same_points) product, kprod_sym (no GPU needed to import).

Each case names the instantiation it targets -- Sym<DP, kernel, form> of kprod_sym.cu -- and the geometry regimes of
the strip-ordered unit list it is sized to reach.  tests/test_sym_coverage_cpu.py checks with the host-only plan query
(product.sym_plan, kmb_debug_sym_plan) and the unit query (kmb_debug_sym_unit) that every case reaches what it claims
and that every instantiation at every D and every regime is the target of a case; tests/test_sym_coverage_gpu.py runs
them against the float64 oracle, row by row.

Sizes are derived from the launcher's own tiling (tile rows, sources per block, TB = blocks per row tile) and from the
partition the query reports, never written as literals, so a case stays on its edge when SymCfg's CTA shape changes.
SMS is the B200's SM count: the symmetric kernel runs one CTA per SM and part.
"""
from __future__ import annotations

import ctypes
import dataclasses
import functools
import math
import zlib

import numpy as np

SMS = 148
KERNELS = ("gaussian", "absolute-exponential", "inverse-distance")
LOG2E = 1.4426950408889634
PRODUCT_FORM_RADIUS2 = 6.0   # kprod_direct.cuh kProductFormRadius2: log2(e) * half-diagonal^2 at most this -> product form

# every instantiation the launcher can pick, as (kernel, Gaussian evaluation form); DP (2 or 3) follows from D
TARGETS = (("gaussian", "product"), ("gaussian", "difference"), ("absolute-exponential", "difference"),
           ("inverse-distance", "difference"))
DIMS = (1, 2, 3)

# Geometry regimes (reached() computes them from the plan and unit queries):
REGIMES = {
    "one_unit": "one unit in all (N <= sources per block)",
    "diag_only": "one row tile over several source blocks: diagonal units only",
    "first_off_diag": "exactly one off-diagonal unit (N = tile rows + 1)",
    "off_diag": "off-diagonal units: column sums",
    "partial_diag_tile": "source blocks not a multiple of TB: the last tile's diagonal is partial",
    "n_multiple_of_block": "N a multiple of the sources per block",
    "n_ragged": "N not a multiple of the sources per block: padded records and padded target rows",
    "grid_clamped": "a part with fewer units than SMs: its grid is clamped to its units",
    "cta_inside_segment": "a CTA range strictly inside one (strip, tile) segment",
    "cta_crosses_strip": "a CTA range over a strip boundary: it switches column slabs mid-range",
    "seg_cut_at_cta_start": "a segment that begins before a CTA and ends inside it (rowpart slot 0)",
    "seg_cut_at_cta_end": "a segment a CTA enters at its start and leaves unfinished (rowpart slot 1)",
    "one_strip": "a single strip",
    "narrow_last_strip": "a last strip narrower than the others",
    "last_strip_lt_TB": "a last strip narrower than TB blocks",
    "strip_cap": "the strip-count cap widens the strips beyond what the CTA count asks for",
    "part_mid_list": "a part whose first segment and first strip are not the list's first (seg_base, strip_base > 0)",
    "part_cut_in_segment": "a part boundary inside a segment",
    "empty_part": "a part with no units",
    "n_le_2": "N of 1 or 2 on the explicit direct_sym path",
}


def dp_of(D):
    """The instantiation's DP for D (kprod_sym.cu sym_launch_dp: D <= 2 runs Sym<2, ...> with zero-padded coordinates)."""
    return 2 if D <= 2 else 3


@dataclasses.dataclass(frozen=True)
class Case:
    name: str
    kernel: str
    D: int
    N: int
    form: str = "difference"   # the Gaussian evaluation form the data select on the device ("difference" otherwise)
    data: str = "unit"         # unit | below (product form, log2e half-diag^2 just below 6) | spread (just above 6) |
                               # grid (jittered grid on a 2^-22 lattice) | offset (around 10^3, spread 1) | dup (quantised)
    signal: str = "spike"      # spike | dense | density
    n_parts: int = 1
    repeat: bool = False       # run twice: bitwise identical
    regimes: tuple = ()        # REGIMES names the case is sized to reach

    @property
    def target(self):
        return dp_of(self.D), self.kernel, self.form


@functools.lru_cache(maxsize=None)
def tiling():
    """(tile rows, sources per block, TB) of the symmetric kernel (the same for every instantiation)."""
    from kernel_matrix_benchmarks_b200 import product

    p = product.sym_plan(1, 3)
    return p["tile_rows"], p["block_sources"], p["TB"]


@functools.lru_cache(maxsize=None)
def plans(N, D, kernel, n_parts):
    from kernel_matrix_benchmarks_b200 import product

    return tuple(product.sym_plan(N, D, kernel=kernel, part=p, n_parts=n_parts, sms=SMS) for p in range(n_parts))


def unit(N, total_ctas, u):
    """kmb_debug_sym_unit: (strip, tile, block, segment begin, segment length) of unit u."""
    from kernel_matrix_benchmarks_b200 import _lib

    o = (ctypes.c_int64 * 8)()
    _lib.check(_lib.load().kmb_debug_sym_unit(int(N), int(total_ctas), int(u), o))
    return tuple(o[3:8])


def cta_range(plan, c):
    """Units [u0, u1) of CTA c of a part: the stream-K split u0 = ub + Ur c / G that the kernel and the combine share."""
    ub, Ur, G = plan["unit_begin"], plan["unit_end"] - plan["unit_begin"], plan["grid"]
    return ub + Ur * c // G, ub + Ur * (c + 1) // G


def off_diagonal_units(N):
    T, S, TB = tiling()
    nsb, n_tiles = -(-N // S), -(-N // T)
    return sum(max(0, nsb - TB * (t + 1)) for t in range(n_tiles))


@functools.lru_cache(maxsize=None)
def reached(N, D, kernel, n_parts):
    """The REGIMES names this problem reaches on SMS SMs."""
    T, S, TB = tiling()
    ps = plans(N, D, kernel, n_parts)
    p0 = ps[0]
    nsb = -(-N // S)
    r = set()
    if N <= 2:
        r.add("n_le_2")
    if p0["units"] == 1:
        r.add("one_unit")
    off = off_diagonal_units(N)
    if off == 0 and nsb > 1:
        r.add("diag_only")
    if off == 1:
        r.add("first_off_diag")
    if off > 0:
        r.add("off_diag")
    if nsb % TB:
        r.add("partial_diag_tile")
    r.add("n_multiple_of_block" if N % S == 0 else "n_ragged")
    last_w = nsb - (p0["n_strips"] - 1) * p0["Wb"]
    if p0["n_strips"] == 1:
        r.add("one_strip")
    elif last_w < p0["Wb"]:
        r.add("narrow_last_strip")
        if last_w < TB:
            r.add("last_strip_lt_TB")
    if p0["strip_cap"]:
        r.add("strip_cap")
    total_ctas = SMS * n_parts
    for part, p in enumerate(ps):
        ub, ue = p["unit_begin"], p["unit_end"]
        if ue == ub:
            r.add("empty_part")
            continue
        if p["grid"] < SMS:
            r.add("grid_clamped")
        if p["seg_base"] > 0 and p["strip_base"] > 0:
            r.add("part_mid_list")
        if part > 0 and unit(N, total_ctas, ub)[3] < ub:
            r.add("part_cut_in_segment")
        for c in range(p["grid"]):
            c0, c1 = cta_range(p, c)
            f, l = unit(N, total_ctas, c0), unit(N, total_ctas, c1 - 1)
            f_end, l_end = f[3] + f[4], l[3] + l[4]
            if f[3] == l[3] and f[3] < c0 and f_end > c1:
                r.add("cta_inside_segment")
            if f[0] != l[0]:
                r.add("cta_crosses_strip")
            if f[3] < c0 and f_end <= c1:
                r.add("seg_cut_at_cta_start")
            if l[3] > c0 and l_end > c1:
                r.add("seg_cut_at_cta_end")
    return frozenset(r)


def case_regimes(case):
    return reached(case.N, case.D, case.kernel, case.n_parts)


# ---- the cases --------------------------------------------------------------------------------------------------------


def _sizes():
    """Named problem sizes, in units of the kernel's tiling and of the SMS-CTA partition."""
    T, S, TB = tiling()
    # one tile taller than the first-off-diagonal edge, ~4.5 units per CTA over a dozen row tiles: CTA ranges inside
    # segments, across strips, cutting segments at both ends; the last strip narrower than TB blocks
    mid = 12 * T + 3 * S + 77
    # CTA-count strips are wider than TB when the blocks exceed TB * sqrt(2 * SMS): the last strip is narrow but >= TB
    wt2 = (int(TB * math.sqrt(2 * SMS)) + 3 * TB + 5) * S + 99
    return dict(
        tiny1=1, tiny2=2,
        one_unit=S - 13, one_block=S,
        diag=T - S // 2 - 3, diag_full=T,
        first_off=T + 1,
        density=3 * T + T // 2 + 5,
        whole_tiles=5 * T,
        mid=mid, wt2=wt2,
        c2=1_000_000,
    )


def _instantiation_cases(sz):
    out = []
    for kernel, form in TARGETS:
        for D in DIMS:
            tag = f"inst-{kernel}-{form}-D{D}"
            data = "grid" if kernel == "inverse-distance" else "spread" if form == "difference" and kernel == "gaussian" else "unit"
            common = dict(kernel=kernel, D=D, form=form, data=data)
            out.append(Case(f"{tag}-spike", N=sz["mid"], signal="spike", regimes=("off_diag", "cta_crosses_strip"), **common))
            out.append(Case(f"{tag}-dense", N=sz["mid"], signal="dense", regimes=("off_diag",),
                            repeat=(D == 3), **common))
            out.append(Case(f"{tag}-density", N=sz["density"], signal="density", regimes=("off_diag",), **common))
    for D in DIMS:   # the least accurate product-form data: |2 u.v| up to 12
        out.append(Case(f"below-bound-gaussian-D{D}", "gaussian", D, sz["mid"], form="product", data="below",
                        regimes=("off_diag",)))
    for kernel, form in (("gaussian", "product"), ("absolute-exponential", "difference")):
        for D in (1, 3):
            out.append(Case(f"offset-{kernel}-D{D}", kernel, D, sz["mid"], form=form, data="offset", regimes=("off_diag",)))
        for signal in ("spike", "dense"):   # duplicated points: exact zeros of |x - y|
            out.append(Case(f"dup-{kernel}-D1-{signal}", kernel, 1, sz["mid"], form=form, data="dup", signal=signal,
                            regimes=("off_diag",)))
    return out


def _geometry_cases(sz):
    g = dict(kernel="gaussian", D=3, form="product")
    C = Case
    out = [
        C("geo-n1", N=sz["tiny1"], regimes=("n_le_2", "one_unit", "one_strip"), **g),
        C("geo-n2-invdist", "inverse-distance", 3, sz["tiny2"], data="grid", regimes=("n_le_2", "one_unit")),
        C("geo-one-unit", N=sz["one_unit"], regimes=("one_unit", "n_ragged", "grid_clamped"), repeat=True, **g),
        C("geo-one-block", N=sz["one_block"], signal="dense", regimes=("one_unit", "n_multiple_of_block"), **g),
        C("geo-diag-only", N=sz["diag"], regimes=("diag_only", "one_strip", "n_ragged"), **g),
        C("geo-diag-full-tile", N=sz["diag_full"], signal="dense", regimes=("diag_only", "n_multiple_of_block"), **g),
        C("geo-first-off-diag", N=sz["first_off"], regimes=("first_off_diag", "partial_diag_tile", "last_strip_lt_TB"), **g),
        C("geo-first-off-diag-invdist", "inverse-distance", 2, sz["first_off"], data="grid", regimes=("first_off_diag",)),
        C("geo-whole-tiles", N=sz["whole_tiles"], signal="dense", regimes=("n_multiple_of_block", "grid_clamped"), **g),
        C("geo-mid", N=sz["mid"], repeat=True,
          regimes=("cta_inside_segment", "cta_crosses_strip", "seg_cut_at_cta_start", "seg_cut_at_cta_end",
                   "last_strip_lt_TB", "partial_diag_tile"), **g),
        C("geo-wide-strips", N=sz["wt2"], regimes=("narrow_last_strip", "cta_crosses_strip", "seg_cut_at_cta_end"), **g),
        C("geo-wide-strips-dense", N=sz["wt2"], signal="dense", regimes=("narrow_last_strip",), **g),
        # parts
        C("parts-empty", N=sz["first_off"], n_parts=13, regimes=("empty_part", "grid_clamped"), **g),
        C("parts-3-mid", N=sz["mid"], n_parts=3, repeat=True,
          regimes=("part_mid_list", "part_cut_in_segment", "cta_crosses_strip"), **g),
        C("parts-3-mid-absexp", "absolute-exponential", 2, sz["mid"], n_parts=3, regimes=("part_mid_list",)),
        C("parts-5-wide", N=sz["wt2"], n_parts=5, regimes=("part_mid_list", "part_cut_in_segment"), **g),
        C("parts-5-wide-invdist", "inverse-distance", 3, sz["wt2"], data="grid", n_parts=5, regimes=("part_mid_list",)),
        # size anchors: the C2 shape, and the C2 shape over 64 parts, where the strip-count cap binds
        C("anchor-c2", N=sz["c2"], regimes=("narrow_last_strip", "cta_crosses_strip"), **g),
        C("anchor-c2-64-parts", N=sz["c2"], n_parts=64, regimes=("strip_cap", "part_mid_list", "part_cut_in_segment"), **g),
    ]
    return out


@functools.lru_cache(maxsize=None)
def all_cases():
    sz = _sizes()
    cases = _instantiation_cases(sz) + _geometry_cases(sz)
    names = [c.name for c in cases]
    assert len(set(names)) == len(names), "case names must be unique"
    return tuple(cases)


# ---- data and signals ---------------------------------------------------------------------------------------------------


def _grid_points(rng, n, D):
    """dispatch_cases._grid_points (every distance >= 0.8 grid steps) on a lattice of 2^-22: the kernel centres the
    coordinates in FP32 before it takes differences, and on this lattice the centring is exact, so the only rounding
    in 1/d is the kernel's own.  (Off the lattice, centring rounds a coordinate by up to 2^-25; at D = 1 with 5 10^4
    points the nearest neighbour is 5e-6 away, and 1/d of that pair would be off by ~1e-2.)"""
    import dispatch_cases

    return np.round(dispatch_cases._grid_points(rng, n, D) * 2.0 ** 22) / 2.0 ** 22


def _corners(y, lo, hi):
    """Pin the bounding box: one point at lo in every coordinate, one at hi."""
    y[0], y[-1] = lo, hi
    return y


def make_points(case):
    """The case's points as float64 holding float32 values (what the kernel and the oracle both see)."""
    rng = np.random.RandomState(zlib.crc32(case.name.encode()))
    N, D = case.N, case.D
    if case.data == "grid":
        y = _grid_points(rng, N, D)
    elif case.data in ("below", "spread"):
        # log2(e) * (half-diagonal)^2 = log2(e) D r^2 / 4, 1 % below / above the product-form bound
        r = math.sqrt(4 * PRODUCT_FORM_RADIUS2 * (0.99 if case.data == "below" else 1.01) / (LOG2E * D))
        y = _corners(r * rng.rand(N, D), 0.0, r) if N > 1 else r * rng.rand(N, D)
    elif case.data == "offset":
        y = 1000.0 + rng.rand(N, D)
    elif case.data == "dup":
        y = np.floor(rng.rand(N, D) * 64) / 64
    else:
        y = rng.rand(N, D)
    return y.astype(np.float32).astype(np.float64)


SPIKE_COEFFS = (1.5, -0.375, 3.25, -6.5, 0.8125, -1.75, 2.5, -0.21875)


def spike_rows(case):
    """Rows that carry the nonzero signal entries: row 0, the last row of the first tile, the first row of a strip (the
    second and the middle one), a row in a diagonal block of a later tile, row N - 1; then fillers up to four."""
    T, S, TB = tiling()
    N = case.N
    p0 = plans(N, case.D, case.kernel, case.n_parts)[0]
    n_tiles = -(-N // T)
    strip_rows = p0["Wb"] * S
    cand = [0, T - 1 if N > T else (N - 1) // 2, strip_rows, strip_rows * (p0["n_strips"] // 2),
            (n_tiles // 2) * T + S + 7, N - 1, N // 3, (2 * N) // 3]
    rows = []
    for r in cand:
        if 0 <= r < N and r not in rows:
            rows.append(r)
    return np.array(rows[:8], dtype=np.int64)


def make_signal(case):
    """(b as float64 holding float32 values, or None for density; spike rows or None)."""
    rng = np.random.RandomState(zlib.crc32(case.name.encode()) + 1)
    N = case.N
    if case.signal == "density":
        return None, None
    if case.signal == "spike":
        rows = spike_rows(case)
        b = np.zeros(N)
        b[rows] = SPIKE_COEFFS[:len(rows)]
        return b, rows
    # dense: source-dependent mean, mixed signs and magnitudes (2^-3 .. 2^3)
    b = (rng.randn(N) + np.linspace(-1.0, 2.0, N)) * 2.0 ** rng.randint(-3, 4, N)
    return b.astype(np.float32).astype(np.float64), None


def kernel_f64(kernel, d2):
    if kernel == "gaussian":
        return np.exp(-d2)
    if kernel == "absolute-exponential":
        return np.exp(-np.sqrt(d2))
    with np.errstate(divide="ignore"):
        return 1.0 / np.sqrt(d2)


def spike_terms(case, y, rows):
    """k(y_i, y_j) for every row i and every spike row j, in float64 (N x spikes); inverse distance zeroes i == j (the
    reference's rule with N == M)."""
    d2 = ((y[:, None, :] - y[None, rows, :]) ** 2).sum(-1)
    k = kernel_f64(case.kernel, d2)
    if case.kernel == "inverse-distance":
        k[rows, np.arange(len(rows))] = 0.0
    return k
