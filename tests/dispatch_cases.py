"""Parity cases for every product kernel instantiation the dispatcher can reach (no GPU needed to import).

Each case names the instantiation it targets; tests/test_dispatch_coverage_cpu.py checks with the host-only plan
query (product.dispatch_plan, kmb_debug_product_plan) that every direct table entry and every tensor family x signal
chunk x kernel x normalisation is the target of a case and that each case reaches what it claims -- for the P.B kernels
(E > 4) every launch shape that selects different code, with product.pv_plan (kmb_debug_pv_plan) -- and
tests/test_dispatch_coverage_gpu.py runs them against the float64 oracle.

Shapes are sized from the kernels' own tiling (kmb_debug_direct_entry), so a case stays at the edge it is meant to hit
when a tile size changes.  SMS is the B200's SM count: the direct cases that exercise the stream-K split are sized in
units of its resident grid (2 CTAs per SM).
"""
from __future__ import annotations

import dataclasses
import functools
import zlib

import numpy as np

SMS = 148
# opt-in shared memory per block of the B200 (kmb_get_device_info().smem_per_block_optin, read on the device): with SMS it
# decides the ring stages of the P.B kernels (product.pv_plan)
SMEM_OPTIN = 232448
KERNELS = ("gaussian", "absolute-exponential", "inverse-distance")

# direct tables in kmb_debug_direct_entry order: (kernel, normalised, Gaussian evaluation form)
DIRECT_TABLES = (
    ("gaussian", False, "difference"), ("gaussian", True, "difference"),
    ("absolute-exponential", False, None), ("absolute-exponential", True, None),
    ("inverse-distance", False, None), ("inverse-distance", True, None),
    ("gaussian", False, "product"), ("gaussian", True, "product"),
)
# D per template DP: DP itself and, for the wide ones, a D < DP (zero-padded coordinates)
DIRECT_DIMS = {2: (2,), 3: (3,), 4: (4,), 8: (8, 5), 16: (16, 11)}
# E per template EP: one the signal-chunk rule puts on that EP in a single full pass, and for EP >= 4 one that leaves a
# partial last pass (E = 3: one pass with a padded column; E = 17: 8 + 8 + 1; E = 25: 16 + 9)
DIRECT_SIGNALS = {1: (1,), 2: (2,), 4: (4, 3), 8: (8, 17), 16: (16, 25)}

TOL_DIRECT, TOL_TENSOR, TOL_F64 = 1e-5, 1e-4, 1e-12
TOL_FAR_ROWS = 2e-4   # rows far from every source: the exponent is ~1e3 ulps of FP32 away from zero (as in test_product_gpu)


@dataclasses.dataclass(frozen=True)
class Case:
    name: str
    kernel: str
    N: int
    M: int
    D: int
    E: int
    norm: bool = False
    density: bool = False
    path: str = "auto"
    row_offset: int = 0
    data: str = "unit"        # unit: r [0,1)^D, r^2 D = 3 | spread: Gaussian difference form under "auto" | grid: jittered
                              # grid (well separated points) | copy: x is a copy of y (grid) | magnitude, halves: unit points,
                              # signal columns of very different magnitudes (make_data)
    far_rows: bool = False    # a few target rows at d^2 > 104 from every source (FP32 exponentials underflow)
    sample_rows: int = 0      # check this many sampled rows (0: every row)
    precision: str = "float32"
    env: tuple = ()           # environment of a child process, e.g. (("KMB_TENSOR_PAIR", "0"),)
    repeat: bool = False      # run twice: the output must be bitwise identical
    # what the case targets
    family: str = "direct"    # KMB_FAMILY_* name (product.dispatch_plan), or "f64"
    entry: tuple = None       # direct: (table, DP, EP)
    form: str = None          # direct Gaussian: the evaluation form the data select
    chunk: int = None         # signal columns per pass of the targeted launch
    passes: int = None
    group: str = None         # P.B kernels: PB_GROUPS name
    edges: tuple = ()         # P.B kernels: the launch shapes (pb_edges names) the case is sized to reach

    @property
    def tol(self):
        if self.precision == "float64":
            return TOL_F64
        if self.far_rows:
            return TOL_FAR_ROWS
        return TOL_DIRECT if self.family == "direct" else TOL_TENSOR


@functools.lru_cache(maxsize=None)
def _direct_tables():
    from kernel_matrix_benchmarks_b200 import product

    return tuple(tuple(product.direct_entries(t)) for t in range(len(DIRECT_TABLES)))


def _tiling(table, DP, EP):
    """(TILE_ROWS, SB) of the table entry with this DP / EP; the widest tiling if there is none (the coverage test then
    names the missing entry)."""
    for e in _direct_tables()[table]:
        if e["DP"] == DP and e["EP"] == EP:
            return e["TILE_ROWS"], e["SB"]
    return 2048, 512


def _direct_cases():
    out = []
    for t, (kernel, norm, form) in enumerate(DIRECT_TABLES):
        # Gaussian difference form on unit data: only with the product form switched off
        path = "direct_diff" if form == "difference" else "direct"
        online_max = norm and kernel != "inverse-distance" and form != "product"
        data = "grid" if kernel == "inverse-distance" else "unit"
        tag = f"direct-t{t}-{kernel}-n{int(norm)}"
        for DP, dims in DIRECT_DIMS.items():
            for EP, signals in DIRECT_SIGNALS.items():
                T, S = _tiling(t, DP, EP)
                common = dict(kernel=kernel, norm=norm, path=path, data=data, far_rows=online_max, entry=(t, DP, EP),
                              form=form, chunk=EP)
                E = signals[0]
                # (a) one CTA holds the whole tile: fewer rows than a tile, at most one source block
                out.append(Case(f"{tag}-DP{DP}-EP{EP}-a-D{DP}-E{E}", N=T // 2 + 37, M=S - 13, D=DP, E=E, passes=1,
                                repeat=(DP == 3 and EP == 1), **common))
                # (b) 3 row tiles (the last ragged) x 4 source blocks (the last ragged): one unit per CTA, every tile is
                # split and combined by the last CTA to arrive
                shapes_b = [(DP, E)] + [(DP, e) for e in signals[1:]] + [(d, E) for d in dims[1:]]
                for D, e in shapes_b:
                    out.append(Case(f"{tag}-DP{DP}-EP{EP}-b-D{D}-E{e}", N=2 * T + T // 3 + 5, M=3 * S + S // 2 + 3, D=D,
                                    E=e, passes=-(-e // EP), **common))
            # (c) ~2 units per CTA of the resident grid over 7 source blocks per tile: CTA ranges start mid-tile and
            # end in the next tile (partial slots 0 and 1); checked on sampled rows
            T, S = _tiling(t, DP, 2)
            n_tiles = -(-4 * SMS // 7)
            out.append(Case(f"{tag}-DP{DP}-EP2-c-D{DP}-E2", N=(n_tiles - 1) * T + T // 2 + 1, M=7 * S - S // 3, D=DP, E=2,
                            sample_rows=256, kernel=kernel, norm=norm, path=path, data=data, far_rows=online_max,
                            entry=(t, DP, 2), form=form, chunk=2, passes=1))
    # the Gaussian difference form where "auto" picks it: spread-out data (log2 e * half-diagonal^2 > 6)
    for DP in DIRECT_DIMS:
        for norm in (False, True):
            T, S = _tiling(int(norm), DP, 1)
            out.append(Case(f"direct-spread-gaussian-n{int(norm)}-DP{DP}", "gaussian", N=T + 100, M=2 * S + 7, D=DP, E=1,
                            norm=norm, data="spread", entry=(int(norm), DP, 1), form="difference", chunk=1, passes=1))
    return out


TENSOR_DIMS = (40, 784)


def _tensor_cases():
    """The E <= 4 kernels (kprod_tensor, kprod_tensor_pair) at every signal chunk, the multi-pass route (D > 128, E > 4:
    the P.B kernels need D <= 128) and density estimation."""
    out = []
    small, multi = 100, 128 * 3 + 17   # one row tile (single CTA even with FP16 planes) / four row tiles (CTA pairs)
    variants = (("tensor_tf32", multi, "tensor"), ("tensor_f16", small, "tensor"), ("tensor_f16", multi, "tensor_pair"))
    for kernel in KERNELS:
        for norm in (False, True):
            for path, N, family in variants:
                for E in (1, 2, 3, 4):
                    for D in (TENSOR_DIMS if E >= 3 else TENSOR_DIMS[:1]):
                        out.append(Case(f"tensor-{path}-{family}-{kernel}-n{int(norm)}-N{N}-D{D}-E{E}", kernel, N=N, M=700,
                                        D=D, E=E, norm=norm, path=path, family=family, chunk=min(E, 4), passes=1,
                                        repeat=(kernel == "gaussian" and not norm and D == 40 and E == 3)))
                for D in (200, 784):
                    for E in (5, 10):
                        out.append(Case(f"tensor-{path}-{family}-multipass-{kernel}-n{int(norm)}-N{N}-D{D}-E{E}", kernel, N=N,
                                        M=700, D=D, E=E, norm=norm, path=path, family=family, chunk=4, passes=-(-E // 4)))
    for kernel in KERNELS:
        for path, N, family in variants:
            for D in TENSOR_DIMS:
                out.append(Case(f"tensor-density-{path}-{family}-{kernel}-N{N}-D{D}", kernel, N=N, M=700, D=D, E=1, density=True,
                                path=path, family=family, chunk=1, passes=1))
    # P.B kernels: one repeated case each for determinism (their launch shapes are the cases of _pb_cases)
    for path, family in (("tensor_tf32", "pv"), ("tensor_f16", "pv16_pair")):
        out.append(Case(f"tensor-{family}-repeat", "gaussian", N=multi, M=700, D=40, E=16, norm=True, path=path, family=family,
                        chunk=64, passes=1, repeat=True))
    return out


def _row_offset_cases():
    """Inverse distance with a row offset (a row shard of a larger target set): the zeroed column is (offset + i) mod
    (M + 1).  Offsets are not multiples of any tile; 'tall' has N > M + 1, so the zeroed column wraps inside the shard."""
    out = []
    for norm in (False, True):
        n = int(norm)
        for E in (1, 5):
            out.append(Case(f"offset-direct-n{n}-E{E}", "inverse-distance", N=2 * 2048 + 300, M=1000, D=3, E=E, norm=norm,
                            path="direct", row_offset=333, data="grid", entry=(4 + n, 3, 8 if E == 5 else 1),
                            chunk=8 if E == 5 else 1, passes=1))
        out.append(Case(f"offset-direct-tall-n{n}", "inverse-distance", N=3000, M=700, D=8, E=2, norm=norm, path="direct",
                        row_offset=1234, data="grid", entry=(4 + n, 8, 2), chunk=2, passes=1))
        for path, N, family in (("tensor_tf32", 300, "tensor"), ("tensor_f16", 100, "tensor"), ("tensor_f16", 300, "tensor_pair")):
            for E in (1, 3):
                out.append(Case(f"offset-{path}-{family}-n{n}-N{N}-E{E}", "inverse-distance", N=N, M=500, D=40, E=E, norm=norm,
                                path=path, row_offset=77 + 1000 * E, family=family, chunk=E, passes=1))
            out.append(Case(f"offset-{path}-{family}-tall-n{n}-N{N}", "inverse-distance", N=N, M=N // 2 - 9, D=40, E=2, norm=norm,
                            path=path, row_offset=45, family=family, chunk=2, passes=1))
        for path in ("tensor_tf32", "tensor_f16"):   # inverse distance never takes kprod_tensor_pv16 (it has no row offset)
            out.append(Case(f"offset-{path}-pv-n{n}", "inverse-distance", N=300, M=500, D=40, E=8, norm=norm, path=path,
                            row_offset=1077, family="pv", chunk=64, passes=1))
            out.append(Case(f"offset-{path}-pv-tall-n{n}", "inverse-distance", N=700, M=200, D=64, E=6, norm=norm, path=path,
                            row_offset=150, family="pv", chunk=64, passes=1))
    # x is a copy of y (other tensor, same values): a missed zeroing is 1/0 = inf, not a small shift
    out.append(Case("copy-direct", "inverse-distance", N=3000, M=3000, D=3, E=1, path="direct", data="copy", entry=(4, 3, 1),
                    chunk=1, passes=1))
    out.append(Case("copy-tensor-pair", "inverse-distance", N=300, M=300, D=40, E=2, path="tensor_f16", data="copy",
                    family="tensor_pair", chunk=2, passes=1))
    out.append(Case("copy-pv", "inverse-distance", N=300, M=300, D=40, E=8, path="tensor_f16", data="copy", family="pv",
                    chunk=64, passes=1))
    return out


PAIR_OFF = (("KMB_TENSOR_PAIR", "0"),)


def _env_cases():
    """KMB_TENSOR_PAIR=0: the single-CTA FP16 kernels on problems of several row tiles (read once per process, so these run
    in a child process)."""
    out = []
    for kernel in KERNELS:
        for norm in (False, True):
            for E in (1, 4):
                out.append(Case(f"pair-off-tensor-{kernel}-n{int(norm)}-E{E}", kernel, N=128 * 5 + 3, M=900, D=40, E=E,
                                norm=norm, path="tensor_f16", env=PAIR_OFF, family="tensor", chunk=E, passes=1,
                                repeat=(kernel == "gaussian" and E == 4 and not norm)))
        if kernel != "inverse-distance":
            for norm in (False, True):
                out.append(Case(f"pair-off-pv16-{kernel}-n{int(norm)}", kernel, N=128 * 5 + 3, M=900, D=64, E=16, norm=norm,
                                path="tensor_f16", env=PAIR_OFF, family="pv16", chunk=64, passes=1,
                                repeat=(kernel == "gaussian" and not norm)))
    return out


# ---- P.B kernels (E > 4, D <= 128): kprod_tensor_pv (TF32 planes), kprod_tensor_pv16 (FP16 planes), kprod_tensor_pv16_pair
# group -> (plan family, path, kernels it serves, environment, sources per block, default flush interval in blocks)
FLUSH_KNOB = "KMB_PV16_FLUSH_BLOCKS"
PB_GROUPS = {
    "pv": ("pv", "tensor_tf32", KERNELS, (), 64, 64),
    "pv16": ("pv16", "tensor_f16", KERNELS[:2], (), 128, 128),              # one row tile: CTA pairs need two
    "pv16_pair": ("pv16_pair", "tensor_f16", KERNELS[:2], (), 128, 128),
    "pv16_pair_off": ("pv16", "tensor_f16", KERNELS[:2], PAIR_OFF, 128, 128),   # single CTAs on several row tiles
}
PB_WIDTHS = (5, 31, 32, 33, 64, 65, 96, 129)   # one pass (ebp 32 / 64); passes whose last has 1, 32 and 1 columns
# every (K blocks, K steps of the last one) and ring-stage count of both kernels: FP16 K blocks of 64 (K steps of 16),
# TF32 K blocks of 32 (D zero-padded to whole K blocks)
PB_DIMS = (16, 17, 48, 64, 65, 96, 112, 128)
# signal magnitude kinds per column (data="magnitude"): largest |b| of the column, 0 (a zero column) or "dwarf" (one entry
# 1e6 times the rest)
MAGNITUDES = (1e-36, 1e-30, 1.0, 1e30, 1e35, 0.0, "dwarf")


def pb_group(plan, env):
    """PB_GROUPS name of a pv_plan (None for the other families)."""
    if plan["family"] == "pv16":
        return "pv16_pair_off" if plan["row_tiles"] >= 2 or dict(env).get("KMB_TENSOR_PAIR") == "0" else "pv16"
    return plan["family"] if plan["family"] in ("pv", "pv16_pair") else None


def range_blocks(plan):
    """Source blocks of the CTA ranges the wave plan makes (a row tile's nsb blocks split into C contiguous ranges)."""
    nsb = plan["source_blocks"]
    return {nsb * (c + 1) // Cw - nsb * c // Cw for Cw in {plan["C"], plan["C_last"]} for c in range(Cw)}


def pb_edges(plan, env):
    """The launch shapes a pv_plan reaches:
      ebp32 / ebp64   one signal pass, padded to 32 / 64 columns (CTA pairs: 16 / 32 per CTA)
      <p>pass-narrow  p passes, the last one narrower than 32 columns
      <p>pass-last<w> p passes, the last one w columns wide (32 or 64)
      stages<s>       s ring stages (set by D through the K blocks)
      k<b>x<s>        b K blocks, s K steps in the last one
      split           C > 1: row tiles split over several CTAs, merged by the last to arrive
      waves           W > 1
      ghost           CTA pairs on an odd number of row tiles: the last pair's second tile does not exist
      flush-1, flush, flush+1, 2flush+1   a CTA range of that many source blocks (flush = the flush interval)
      knob<F>         the flush interval F set by KMB_PV16_FLUSH_BLOCKS, on a CTA range longer than it"""
    e = set()
    if plan["passes"] == 1:
        e.add(f"ebp{plan['ebp_first']}")
    elif plan["eb_last"] < 32:
        e.add(f"{plan['passes']}pass-narrow")
    else:
        e.add(f"{plan['passes']}pass-last{plan['ebp_last']}")
    e.add(f"stages{plan['stages']}")
    e.add(f"k{plan['kblocks']}x{plan['ksteps_last']}")
    if plan["C"] > 1 or plan["C_last"] > 1:
        e.add("split")
    if plan["W"] > 1:
        e.add("waves")
    if plan["pair"] and plan["row_tiles"] % 2:
        e.add("ghost")
    F, blocks = plan["flush_blocks"], range_blocks(plan)
    if FLUSH_KNOB in dict(env):
        if max(blocks) > F:
            e.add(f"knob{F}")
    else:
        e |= {name for name, n in (("flush-1", F - 1), ("flush", F), ("flush+1", F + 1), ("2flush+1", 2 * F + 1)) if n in blocks}
    return e


def _pb_cases():
    """The P.B kernels at every launch shape that selects different code (pb_edges), for every kernel each serves and both
    normalisation settings.  Shapes are in the kernels' own units (SMS, sources per block, flush interval)."""
    out = []
    for group, (family, path, kernels, env, blk, F) in PB_GROUPS.items():
        pair = group == "pv16_pair"
        one_tile = group == "pv16"
        # row counts: one tile (N < 128), an even / odd number of tiles (odd: a ghost tile with pairs); never whole tiles
        n_a, n_b = (100, 100) if one_tile else (128 * 2 + 44, 100) if family == "pv" else (128 * 3 + 17, 128 * 5 + 103)
        for kernel in kernels:
            for norm in (False, True):
                tag = f"pb-{group}-{kernel}-n{int(norm)}"
                common = dict(kernel=kernel, norm=norm, path=path, env=env, family=family, chunk=64, group=group)

                def add(name, N, M, D, E, edges=(), **kw):
                    kw = dict(common, **kw)
                    out.append(Case(f"{tag}-{name}", N=N, M=M, D=D, E=E, passes=-(-E // 64), edges=tuple(edges), **kw))

                for E in PB_WIDTHS:
                    p, last = -(-E // 64), E - 64 * (-(-E // 64) - 1)
                    edge = f"ebp{32 if E <= 32 else 64}" if p == 1 else f"{p}pass-narrow" if last < 32 else f"{p}pass-last{last}"
                    add(f"N{n_a}-D64-E{E}", n_a, 700, 64, E, (edge, "split"))
                for D in PB_DIMS:
                    if D != 64:
                        add(f"N{n_b}-D{D}-E40", n_b, 700, D, 40, ("ebp64",))
                if pair:   # an odd number of row tiles: the second tile of the last pair does not exist
                    add("ghost-N557-D64-E64", 128 * 4 + 45, 700, 64, 64, ("ghost",))
                if family != "pv":   # D <= 16 and E >= 32: "auto" takes the FP16-plane P.B kernel
                    add(f"auto-N{n_b}-D3-E64", n_b, 700, 3, 64, ("ebp64",), path="auto")
                add(f"N{n_a}-D64-E40-M50", n_a, 50, 64, 40)   # fewer sources than a column group holds: one sees none
                if not one_tile:   # more row tiles than the resident grid (pairs: clusters) holds: two waves
                    add("waves-D64-E40", 128 * (SMS + 4) - 40, 700, 64, 40, ("waves",), sample_rows=256)
                    # the flush interval: ranges of F - 1, F, F + 1 and 2F + 1 source blocks, one range per row tile
                    # (as many row tiles as the grid has CTAs: C = 1)
                    for name, nsb in (("flush-1", F - 1), ("flush", F), ("flush+1", F + 1), ("2flush+1", 2 * F + 1)):
                        add(f"{name}-D16-E5", 128 * SMS - 50, nsb * blk - 7, 16, 5, (name,), sample_rows=256)
                if norm:   # rows far from every source: the running reference of the online max starts far below 0
                    add(f"far-N{n_a}-D64-E64", n_a, 700, 64, 64, far_rows=True)
                if group != "pv16_pair_off":
                    add(f"magnitude-N{n_a}-D64-E64", n_a, 700, 64, 64, data="magnitude")
                if pair:   # the two CTAs of a pair hold columns 0-31 and 32-63: 2^100 apart
                    add(f"halves-N{n_a}-D64-E64", n_a, 700, 64, 64, data="halves")
                # the flush knob (read once per process): small multi-tile problems whose CTA ranges cross it
                for knob in (() if family == "pv" else (1, 3) if group != "pv16_pair_off" else (3,)):
                    kenv = tuple(sorted(env + ((FLUSH_KNOB, str(knob)),)))
                    edges = (f"knob{knob}", "split")
                    if one_tile:
                        add(f"knob{knob}-N100-D16-E40", 100, 7 * SMS * blk + 5, 16, 40, edges, env=kenv)
                    elif pair:
                        add(f"knob{knob}-N{n_a}-D16-E40", n_a, 7 * (SMS // 4) * blk + 5, 16, 40, edges, env=kenv)
                    else:
                        add(f"knob{knob}-N557-D16-E40", 128 * 4 + 45, 7 * (SMS // 5) * blk + 5, 16, 40, edges, env=kenv)
    return out


# float64 kernel (D <= 16): signal chunks of <= 8 columns, each on the 1-, 2-, 4- or 8-column instantiation
F64_SIGNALS = (1, 2, 3, 4, 7, 8, 11)


def f64_buckets(E):
    """Column-chunk instantiations kmb_product_f64 launches for E signal columns (kprod_f64.cu: launch_f64)."""
    return [min(b for b in (1, 2, 4, 8) if b >= min(8, E - e0)) for e0 in range(0, E, 8)]


def _f64_cases():
    out = []
    for kernel in KERNELS:
        for norm in (False, True):
            for E in F64_SIGNALS:
                out.append(Case(f"f64-{kernel}-n{int(norm)}-E{E}", kernel, N=700, M=900, D=5, E=E, norm=norm,
                                precision="float64", data="grid" if kernel == "inverse-distance" else "unit",
                                row_offset=101 if kernel == "inverse-distance" else 0, family="f64",
                                passes=len(f64_buckets(E)), repeat=(E == 11 and not norm and kernel == "gaussian")))
    return out


@functools.lru_cache(maxsize=None)
def all_cases():
    cases = _direct_cases() + _tensor_cases() + _row_offset_cases() + _env_cases() + _pb_cases() + _f64_cases()
    names = [c.name for c in cases]
    assert len(set(names)) == len(names), "case names must be unique"
    return tuple(cases)


# ---- data ------------------------------------------------------------------------------------------------------------


def _grid_points(rng, n, D):
    """n distinct points of a jittered integer grid scaled into the unit cube: every distance is >= 0.8 grid steps, so
    FP32 rounding of the coordinates cannot dominate 1/d."""
    side = max(2, int(np.ceil((4.0 * n) ** (1.0 / D))))
    pts = np.zeros((0, D), dtype=np.int64)
    while len(pts) < n:
        pts = np.unique(np.concatenate([pts, rng.randint(0, side, size=(n, D))]), axis=0)
    pts = pts[rng.permutation(len(pts))[:n]]
    return (pts + 0.2 * (rng.rand(n, D) - 0.5)) / side


def far_row_ids(case):
    return np.array(sorted({1, case.N // 2, case.N - 1}), dtype=np.int64) if case.far_rows else np.zeros(0, dtype=np.int64)


def make_data(case):
    """(x, y, b) as float64 arrays holding values representable in the case's precision; b is None under density.
    Signal columns have distinct scales and signs and source-dependent means, so a wrong column offset, a column swap
    or a wrongly weighted source block changes the result well beyond the tolerance."""
    rng = np.random.RandomState(zlib.crc32(case.name.encode()))
    N, M, D, E = case.N, case.M, case.D, case.E
    if case.data in ("grid", "copy"):
        if D <= 16:
            pts = _grid_points(rng, M if case.data == "copy" else N + M, D)
        else:   # random points in high dimension are well separated (distances concentrate around sqrt(D / 6))
            pts = rng.rand(M if case.data == "copy" else N + M, D)
        y = pts[:M]
        x = pts.copy() if case.data == "copy" else pts[M:]
    else:
        r = 5.0 / D ** 0.5 if case.data == "spread" else (3.0 / max(D, 3)) ** 0.5
        y, x = r * rng.rand(M, D), r * rng.rand(N, D)
    if case.far_rows:
        x[far_row_ids(case), 0] += 12.0 if case.kernel == "gaussian" else 150.0
    b = None
    if case.data == "magnitude":   # column e: MAGNITUDES[e % 7] times values in [0.5, 1], sign (-1)^e
        b = (-1.0) ** np.arange(E) * (0.5 + 0.5 * rng.rand(M, E))
        for e in range(E):
            mag = MAGNITUDES[e % len(MAGNITUDES)]
            if mag == "dwarf":
                b[rng.randint(M), e] *= 1e6
            else:
                b[:, e] *= mag
    elif case.data == "halves":    # columns 0-31 and 32-63 at 2^-50 and 2^50
        b = (-1.0) ** np.arange(E) * (0.5 + 0.5 * rng.rand(M, E)) * np.where(np.arange(E) < 32, 2.0 ** -50, 2.0 ** 50)
    elif not case.density:
        scale = np.array([(-1.0) ** e * 2.0 ** (e % 5 - 2) for e in range(E)])
        b = scale * (0.5 + rng.rand(M, E) + np.linspace(0.0, 1.0, M)[:, None])
    dt = np.float64 if case.precision == "float64" else np.float32
    cast = lambda a: None if a is None else a.astype(dt).astype(np.float64)
    return cast(x), cast(y), cast(b)


def check_rows(case):
    """Rows (local indices) whose result is compared: all, or a sample that includes every far row and tile edges."""
    if not case.sample_rows:
        return np.arange(case.N)
    rng = np.random.RandomState(zlib.crc32(case.name.encode()) + 1)
    edges = [0, case.N - 1] + [t * s + d for s in (128, 1024, 2048) for t in range(1, 4) for d in (-1, 0)]
    edges += [128 * SMS * w + d for w in (1, 2) for d in (-1, 0)]   # the first row tiles of the tensor kernels' next waves
    rows = np.concatenate([rng.choice(case.N, case.sample_rows, replace=False), far_row_ids(case), edges])
    return np.unique(rows[(rows >= 0) & (rows < case.N)])
