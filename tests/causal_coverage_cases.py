"""Cases for causal products (KMB_FLAG_CAUSAL) that reach every causal kernel instantiation and every schedule regime
(no GPU needed to import).

Each case names the instantiation it targets -- family (kprod_tensor, _pair, pv16, pv16_pair), EP (kprod_tensor's
signal columns per pass), the epilogue kernel (tc::epilogue_kid: dot-exponential runs on the Gaussian instantiations)
and NORM (density runs NORM = false) -- and the regimes of the causal wave schedule it is sized to reach.
tests/test_causal_coverage_cpu.py checks with the library's own plan queries (product.dispatch_plan,
product.causal_work = kmb_debug_causal_work) that every case reaches what it claims and that every instantiation and
regime has a case; tests/test_causal_coverage_gpu.py runs them against the float64 oracle of tests/causal_oracle.py.

Sizes come from the queries (tile rows, source block, units per wave, the wave plan), never from literals, so a case
stays on its edge when the tiling or the wave plan changes.  SMS is the B200's SM count, which the plans depend on.

Two kinds of data:
  * "positive": points in a cube, a positive signal (rows of a plain product do not cancel);
  * "diagonal": sources on a closed curve of a torus, y_j = R / sqrt(K) (cos(w_k j), sin(w_k j))_k, K = D / 2,
    w_k in [0.05, 0.3]; target i sits at its own diagonal source, x_i = curve(row_offset + i) (absolute-exponential and
    inverse distance a fraction of a step further on: see DIAG_SHIFT), and the signal alternates in sign with zero mean.  Each
    row is then dominated by the few sources nearest its diagonal, so admitting or dropping one source at the diagonal
    changes the row by far more than the tolerance at any M (the CPU test checks this on every checked row).
"""
from __future__ import annotations

import collections
import dataclasses
import functools
import json
import zlib

import numpy as np

import causal_oracle as co

SMS = 148
TWO31 = 2 ** 31
KERNELS = ("gaussian", "absolute-exponential", "inverse-distance", "dot-exponential")
EPILOGUE_KID = {"gaussian": "gaussian", "dot-exponential": "gaussian", "absolute-exponential": "absolute-exponential",
                "inverse-distance": "inverse-distance"}

# every causal tensor instantiation: (family, EP, epilogue kernel, NORM); pv16 has no EP (None)
TENSOR_TARGETS = tuple((fam, ep, k, norm) for fam in ("tensor", "tensor_pair") for ep in (1, 2, 4)
                       for k in ("gaussian", "absolute-exponential", "inverse-distance") for norm in (False, True))
PV16_TARGETS = tuple((fam, None, k, norm) for fam in ("pv16", "pv16_pair") for k in ("gaussian", "absolute-exponential")
                     for norm in (False, True))
TARGETS = TENSOR_TARGETS + PV16_TARGETS
FAMILIES = ("tensor", "tensor_pair", "pv16", "pv16_pair")

# The float64 causal kernels of kprod_f64.cu: kprod_f64_causal_kernel<KID, EC> for D <= F64_MAX_D (one launch per EC
# bucket of at most F64_MAX_E signal columns), kprod_f64_wide_causal_kernel<KID> above.  No plan query reports them, so
# f64_instantiations restates the launcher's choice.
F64_MAX_D, F64_MAX_E, F64_ROWS_PER_CTA, F64_WIDE_ROWS_PER_CTA = 16, 8, 128, 64
F64_TARGETS = tuple((k, ec) for k in KERNELS for ec in (1, 2, 4, 8, "wide"))

REGIMES = {
    "waves_2": "two waves",
    "waves_3_last_reversed": "three or more waves, the last one odd (its tiles taken in reverse order)",
    "short_last_wave": "a last wave of fewer row tiles than the others (R_last < R)",
    "c_last_gt_1": "a last wave whose tiles are split over several ranges (C_last > 1)",
    "odd_wave_split": "a reversed odd wave whose tiles are split over several ranges (partial slots at the reversed index)",
    "empty_range": "a unit whose source range is empty",
    "empty_then_work": "a unit with an empty range in one wave and blocks in a later one",
    "fully_masked_rows": "rows that see none of the blocks of their unit's non-empty range",
    "pair_ghost": "CTA pairs over an odd number of row tiles (the last peer has no tile)",
    "n_mod_tile_1": "N one row past a multiple of the tile rows",
    "n_mod_tile_last": "N one row short of a multiple of the tile rows",
    "n_1": "a single target row",
    "n_gt_m": "more targets than sources",
    "ro_past_end": "row_offset >= M - 1: every row sees every source",
    "ro_above_2_31": "row_offset above 2^31",
    "ro_mod64_0": "row_offset = 0 mod 64", "ro_mod64_1": "row_offset = 1 mod 64",
    "ro_mod64_62": "row_offset = 62 mod 64", "ro_mod64_63": "row_offset = 63 mod 64",
    "ro_mod256_126": "row_offset = 126 mod 256", "ro_mod256_127": "row_offset = 127 mod 256",
    "ro_mod256_128": "row_offset = 128 mod 256", "ro_mod256_254": "row_offset = 254 mod 256",
    "ro_mod256_255": "row_offset = 255 mod 256",
    "pv16_passes": "pv16 over several signal passes (E > 64)",
    "tensor_passes": "kprod_tensor over several signal passes (D > 128, E > 4)",
    "knob_pair_off": "KMB_TENSOR_PAIR=0: single-CTA kernels on several row tiles",
    "knob_flush_1": "KMB_PV16_FLUSH_BLOCKS=1: pv16 flushes its accumulators after every block",
    "knob_multiwave": "a knob case over several waves",
}
# Diagonal positions: the first row of a tile, R0 = row_offset + first row, against the granularity G of the crossing
# test (kprod_tensor: a 256-source block, pv16: a column group of 64 sources).  A crossing test off by one moves the
# mask of that row only when R0 + 2 (test `> R0 + 1`) or R0 (test `> R0 - 1`) is a multiple of G.
DIAG_EDGES = {"diag_edge_m2": -2, "diag_edge_m1": -1, "diag_edge_0": 0, "diag_edge_p1": 1}
DIAG_EDGE_NOTE = "the first row of a tile at R0 = G - 2, G - 1, 0, 1 mod G (G: the crossing test's granularity)"

PAIR_OFF = (("KMB_TENSOR_PAIR", "0"),)
FLUSH_1 = (("KMB_PV16_FLUSH_BLOCKS", "1"),)


@dataclasses.dataclass(frozen=True)
class Case:
    name: str
    kernel: str
    N: int
    M: int
    D: int
    E: int
    norm: bool
    row_offset: int
    family: str                # the family the case targets
    ep: int | None = None      # kprod_tensor's EP (None for pv16)
    passes: int = 1
    data: str = "positive"     # positive | diagonal
    density: bool = False
    env: tuple = ()            # the environment of a child process (knobs read once per process)
    regimes: tuple = ()

    @property
    def target(self):
        return self.family, self.ep, EPILOGUE_KID[self.kernel], self.norm and not self.density

    @property
    def signal_cols(self):
        return 1 if self.density else self.E

    @property
    def sampled(self):
        """Large cases: compare sampled rows (sample_rows) rather than all of them."""
        return self.N * min(self.M, self.row_offset + self.N) > 40_000_000

    @property
    def multiwave(self):
        return waves_of(self) > 1


# ---- geometry from the plan queries ------------------------------------------------------------------------------------


@functools.lru_cache(maxsize=None)
def geometry():
    """(tile rows, kprod_tensor source block, pv16 source block, pv16 column group, clusters per wave)."""
    from kernel_matrix_benchmarks_b200 import product

    big = 1 << 20
    tm = big // product.dispatch_plan(big, 1000, 64, 1, causal=True)["row_tiles"]
    tn = product.causal_work(1000, 1000, 64, 1, 0, 0, sms=SMS)["block"]
    pv = product.causal_work(1000, 1000, 64, 64, 0, 0, sms=SMS)
    # pv16's epilogue tests the diagonal per column group: NG = 2 groups of half a block (kprod_tensor_pv16.cu CPT)
    return tm, tn, pv["block"], pv["block"] // 2, pv["units"]


def granularity(family):
    tm, tn, tns, cpt, _ = geometry()
    return tn if family.startswith("tensor") else cpt


@functools.lru_cache(maxsize=None)
def _schedule(N, M, D, E, kernel, norm, row_offset):
    """Every (wave, unit) work item: (first query, {(w, u): work dict with a tile})."""
    from kernel_matrix_benchmarks_b200 import product

    kw = dict(kernel=kernel, normalize_rows=norm, row_offset=row_offset, sms=SMS)
    first = product.causal_work(N, M, D, E, 0, 0, **kw)
    items = {}
    for w in range(first["waves"]):
        for u in range(first["units"]):
            ww = product.causal_work(N, M, D, E, w, u, **kw)
            if ww["tile"] >= 0:
                items[(w, u)] = ww
    return first, items


def schedule(case):
    return _schedule(case.N, case.M, case.D, case.signal_cols, case.kernel, case.norm and not case.density, case.row_offset)


def waves_of(case):
    return schedule(case)[0]["waves"]


def reached(case, family=None):
    """The REGIMES and DIAG_EDGES names this case reaches, from the schedule of the causal kernel (family: the family
    the plan reports, when the case runs with a knob the in-process query does not see)."""
    from kernel_matrix_benchmarks_b200 import product

    first, items = schedule(case)
    fam = family or first["family"]
    tm = geometry()[0]
    pair = fam.endswith("_pair")
    rows_per_unit = 2 * tm if pair else tm
    block = first["block"]
    W, N, M, ro = first["waves"], case.N, case.M, case.row_offset
    r = set()
    if W == 2:
        r.add("waves_2")
    if W >= 3 and (W - 1) % 2 == 1:
        r.add("waves_3_last_reversed")
    tiles_in = {}
    for (w, u), ww in items.items():
        tiles_in.setdefault(w, set()).add(ww["tile"])
    if W >= 2 and len(tiles_in.get(W - 1, ())) < len(tiles_in.get(0, ())):
        r.add("short_last_wave")
    for (w, u), ww in items.items():
        if W >= 2 and w == W - 1 and ww["Cw"] > 1:
            r.add("c_last_gt_1")
        if w % 2 == 1 and ww["Cw"] > 1:
            r.add("odd_wave_split")
        if ww["sb_lo"] == ww["sb_hi"]:
            r.add("empty_range")
            if any(items.get((w2, u)) and items[(w2, u)]["sb_lo"] < items[(w2, u)]["sb_hi"] for w2 in range(w + 1, W)):
                r.add("empty_then_work")
        elif ww["sb_lo"] > 0:
            # the unit's rows (pairs: both tiles); a row r sees nothing of [sb_lo, sb_hi) when ro + r < sb_lo * block
            row0 = ww["tile"] * rows_per_unit
            if row0 < N and ro + row0 < ww["sb_lo"] * block:
                r.add("fully_masked_rows")
    n_tiles = -(-N // tm)
    if pair and n_tiles % 2 == 1:
        r.add("pair_ghost")
    if N % tm == 1 and N > 1:
        r.add("n_mod_tile_1")
    if N % tm == tm - 1:
        r.add("n_mod_tile_last")
    if N == 1:
        r.add("n_1")
    if N > M:
        r.add("n_gt_m")
    if ro >= M - 1:
        r.add("ro_past_end")
    if ro > TWO31:
        r.add("ro_above_2_31")
    for m, res in ((64, (0, 1, 62, 63)), (256, (126, 127, 128, 254, 255))):
        if ro % m in res:
            r.add(f"ro_mod{m}_{ro % m}")
    plan = product.dispatch_plan(case.N, case.M, case.D, case.signal_cols, kernel=case.kernel,
                                 normalize_rows=case.norm and not case.density, density_estimation=case.density,
                                 causal=True, sms=SMS)
    if fam.startswith("pv16") and plan["passes"] > 1:
        r.add("pv16_passes")
    if fam.startswith("tensor") and plan["passes"] > 1:
        r.add("tensor_passes")
    env = dict(case.env)
    if env.get("KMB_TENSOR_PAIR") == "0" and n_tiles > 1:
        r.add("knob_pair_off")
    if env.get("KMB_PV16_FLUSH_BLOCKS") == "1" and fam.startswith("pv16"):
        r.add("knob_flush_1")
    if env and W > 1:
        r.add("knob_multiwave")
    # diagonal positions: a tile with rows whose first row sits at the edge, with the source just past it in range
    G = granularity(fam)
    for t in range(n_tiles):
        r0 = ro + t * tm
        if r0 + 1 >= M:
            break
        for name, k in DIAG_EDGES.items():
            if (r0 - k) % G == 0:
                r.add(name)
    return frozenset(r)


def f64_instantiations(D, E):
    """The float64 causal kernels kmb_product_f64 launches for (D, E): {("wide",)} or the EC buckets of its launches."""
    if D > F64_MAX_D:
        return {"wide"}
    out = set()
    for e0 in range(0, E, F64_MAX_E):
        ec = min(F64_MAX_E, E - e0)
        out.add(1 if ec <= 1 else 2 if ec <= 2 else 4 if ec <= 4 else 8)
    return out


# ---- the cases ----------------------------------------------------------------------------------------------------------


def _ep_signal(ep):
    return {1: 1, 2: 2, 4: 3}[ep]


def _first(pred, candidates):
    for c in candidates:
        if pred(c):
            return c
    raise AssertionError("no candidate reaches the regime")


# sources past N in the wave-sized problems: the diagonal of every row, row_offset + i + 1, stays a real source
PAD = 301


def _wave_sizes():
    """Problems of N targets and N + PAD sources sized in units of one wave of row tiles, picked by what their schedule
    reaches."""
    tm, tn, tns, cpt, units = geometry()
    wave_rows = units * 2 * tm   # one wave of CTA pairs with one tile each
    fr = tuple(round(wave_rows * f / 100) for f in range(40, 400, 5))

    def sched(n, E, reg):
        c = Case("probe", "gaussian", n, n + PAD, 64, E, True, 0, "")
        return reg(reached(c))
    t2 = _first(lambda n: sched(n, 1, lambda r: "waves_2" in r and "empty_then_work" in r), fr)
    t6 = _first(lambda n: sched(n, 1, lambda r: "waves_3_last_reversed" in r and "c_last_gt_1" in r and "odd_wave_split" in r), fr)
    p2 = _first(lambda n: sched(n, 64, lambda r: "waves_2" in r and "odd_wave_split" in r and "short_last_wave" in r), fr[::-1])
    p4 = _first(lambda n: sched(n, 64, lambda r: "waves_3_last_reversed" in r and "c_last_gt_1" in r), fr)
    # pv16: few row tiles over many sources, so that a first-wave range can be empty (searched over N, M)
    cand = tuple((k * tm, m * tns) for m in (512, 1024, 2048) for k in range(3, 13))
    pe = _first(lambda nm: "empty_then_work" in reached(Case("probe", "gaussian", nm[0], nm[1], 64, 64, True, 0, "")), cand)
    return dict(t2=t2, t6=t6, p2=p2, p4=p4, pe=pe)


# row offsets of the diagonal cases, per family.  _DIAG_RO_M2 puts the first row of some tile at G - 2 (DIAG_EDGES), where
# a crossing test off by one admits one source too many: every instantiation gets a diagonal case there.
# _DIAG_RO_EDGE walks the other diagonal edges (the dot-exponential diagonal cases).
_DIAG_RO_M2 = {"tensor": (254, 510, 254 + 256 * 5), "tensor_pair": (126, 254, 126 + 512, 254 + 256 * 3),
               "pv16": (62, 126, 254, 62 + 64 * 9), "pv16_pair": (62, 126, 254, 62 + 64 * 9)}
_DIAG_RO_EDGE = {"tensor": (255, 256, 257, 511, 512, 513), "tensor_pair": (127, 128, 129, 255, 256, 257),
                 "pv16": (63, 64), "pv16_pair": (63, 64)}
_POS_RO = (0, 77, 1, 63, 128, 43, 300, 1000)


def _instantiation_cases():
    tm, tn, tns, cpt, _ = geometry()
    out = []
    k_diag = collections.Counter()
    k_pos = 0
    for fam, ep, ekid, norm in TARGETS:
        pair = fam.endswith("_pair")
        pv = fam.startswith("pv16")
        kernels = ("gaussian", "dot-exponential") if ekid == "gaussian" else (ekid,)
        for n_shape, (data, kernel) in enumerate([("positive", kernels[0])] + [("diagonal", k) for k in kernels]):
            if pv:
                E = (8, 64, 40)[n_shape % 3]
                D = (64, 16, 128)[n_shape % 3]
            else:
                E = _ep_signal(ep) if ep < 4 else (3, 4, 4)[n_shape % 3]
                D = (64, 16, 32)[n_shape % 3]
            if pair:
                N = (2 * tm + 1, 3 * tm - 1, 4 * tm)[n_shape % 3]
            else:
                N = (tm, tm - 1, tm // 2 + 3)[n_shape % 3]
            if data == "diagonal":
                ros = _DIAG_RO_EDGE[fam] if kernel == "dot-exponential" else _DIAG_RO_M2[fam]
                ro = ros[k_diag[(fam, ros)] % len(ros)]
                k_diag[(fam, ros)] += 1
                M = ro + N + tn + 37   # sources past the last diagonal are never read
            else:
                ro = _POS_RO[k_pos % len(_POS_RO)]
                k_pos += 1
                M = (3 * tn + 11, 7 * tns + 5, 2 * N + 100)[k_pos % 3]
            name = f"inst-{fam}-ep{ep}-{ekid}-{'norm' if norm else 'plain'}-{data}-{kernel}"
            out.append(Case(name, kernel, N, M, D, E, norm, ro, fam, ep, data=data))
    # density (NORM = false, E = 1) on every E <= 4 family and epilogue kernel
    for fam in ("tensor", "tensor_pair"):
        for kernel in ("gaussian", "absolute-exponential", "inverse-distance"):
            N = 2 * tm + 1 if fam == "tensor_pair" else tm - 1
            out.append(Case(f"density-{fam}-{kernel}", kernel, N, 4 * tn, 16, 1, False, 77, fam, 1, density=True))
    return out


def _regime_cases():
    tm, tn, tns, cpt, _ = geometry()
    s = _wave_sizes()
    C = Case
    out = [
        # waves
        C("waves2-tensor-pair-empty-first-wave", "gaussian", s["t2"], s["t2"] + PAD, 64, 1, True, 0, "tensor_pair", 1,
          data="diagonal", regimes=("waves_2", "empty_range", "empty_then_work", "short_last_wave", "odd_wave_split",
                                    "ro_mod64_0")),
        C("waves6-tensor-pair-last-reversed", "gaussian", s["t6"], s["t6"] + PAD, 64, 2, False, 126, "tensor_pair", 2,
          data="diagonal", regimes=("waves_3_last_reversed", "c_last_gt_1", "odd_wave_split", "short_last_wave",
                                    "ro_mod256_126", "ro_mod64_62")),
        C("waves6-tensor-pair-last-reversed-abs", "absolute-exponential", s["t6"], s["t6"] + PAD, 32, 4, True, 255,
          "tensor_pair", 4, data="diagonal", regimes=("waves_3_last_reversed", "c_last_gt_1", "ro_mod256_255", "ro_mod64_63")),
        C("waves2-pv16-pair-split-odd-wave", "dot-exponential", s["p2"], s["p2"] + PAD, 64, 64, True, 62, "pv16_pair",
          data="diagonal", regimes=("waves_2", "odd_wave_split", "c_last_gt_1", "short_last_wave", "ro_mod64_62")),
        C("waves2-pv16-pair-plain-abs", "absolute-exponential", s["p2"], s["p2"] + PAD, 64, 16, False, 127, "pv16_pair",
          data="diagonal", regimes=("waves_2", "odd_wave_split", "ro_mod256_127", "ro_mod64_63")),
        C("waves4-pv16-pair-last-reversed", "gaussian", s["p4"], s["p4"] + PAD, 64, 64, True, 254, "pv16_pair",
          data="diagonal", regimes=("waves_3_last_reversed", "c_last_gt_1", "ro_mod256_254")),
        C("empty-then-work-pv16-pair", "gaussian", s["pe"][0], s["pe"][1], 64, 64, True, 0, "pv16_pair",
          regimes=("empty_range", "empty_then_work", "fully_masked_rows", "waves_2", "ro_mod64_0")),
        C("empty-then-work-pv16-pair-diag", "absolute-exponential", s["pe"][0], s["pe"][1], 64, 32, False, 1, "pv16_pair",
          data="diagonal", regimes=("empty_range", "empty_then_work", "fully_masked_rows", "ro_mod64_1")),
        # row offsets at and past the end, and above 2^31 (the causal product is the full product)
        C("ro-past-end-tensor-pair", "gaussian", 3 * tm - 1, 5 * tn + 3, 64, 1, True, 5 * tn + 2, "tensor_pair", 1,
          regimes=("ro_past_end", "pair_ghost", "n_mod_tile_last")),
        C("ro-past-end-pv16-pair", "absolute-exponential", 2 * tm + 1, 4 * tns, 64, 64, True, 4 * tns + 500, "pv16_pair",
          regimes=("ro_past_end", "pair_ghost", "n_mod_tile_1")),
        C("ro-above-2-31-tensor-pair", "inverse-distance", 2 * tm + 1, 3 * tn, 32, 4, True, TWO31 + 12345, "tensor_pair", 4,
          regimes=("ro_above_2_31", "ro_past_end")),
        C("ro-above-2-31-pv16", "dot-exponential", tm - 1, 5 * tns, 64, 64, True, TWO31 + 128, "pv16",
          regimes=("ro_above_2_31", "ro_past_end", "n_mod_tile_last", "ro_mod256_128")),
        # shape edges
        C("n1-tensor", "inverse-distance", 1, 2 * tn, 64, 2, False, 3 * tn - 2, "tensor", 2, regimes=("n_1", "ro_past_end")),
        C("n1-pv16", "gaussian", 1, 3 * tns, 64, 8, True, 129, "pv16", data="diagonal", regimes=("n_1",)),
        C("n1-tensor-diag", "gaussian", 1, 3 * tn, 64, 1, True, 254, "tensor", 1, data="diagonal",
          regimes=("n_1", "ro_mod256_254", "ro_mod64_62")),
        C("n-gt-m-tensor-pair", "absolute-exponential", 8 * tm + 1, 3 * tm, 16, 2, True, 0, "tensor_pair", 2,
          regimes=("n_gt_m", "n_mod_tile_1", "pair_ghost")),
        C("n-gt-m-pv16-pair", "gaussian", 7 * tm - 1, 2 * tm, 64, 64, False, 63, "pv16_pair",
          regimes=("n_gt_m", "n_mod_tile_last", "pair_ghost")),
        # several signal passes
        C("passes-pv16", "gaussian", tm - 1, 6 * tns, 64, 150, True, 62, "pv16", passes=3, data="diagonal",
          regimes=("pv16_passes", "ro_mod64_62")),
        C("passes-pv16-pair", "absolute-exponential", 3 * tm - 1, 9 * tns, 128, 100, False, 126, "pv16_pair", passes=2,
          data="diagonal", regimes=("pv16_passes", "pair_ghost", "ro_mod256_126")),
        C("passes-tensor", "inverse-distance", tm, 4 * tn, 200, 9, True, 254, "tensor", 4, passes=3, data="diagonal",
          regimes=("tensor_passes", "ro_mod256_254")),
        C("passes-tensor-pair", "dot-exponential", 3 * tm + 1, 6 * tn, 200, 8, True, 127, "tensor_pair", 4, passes=2,
          data="diagonal", regimes=("tensor_passes", "ro_mod256_127")),
        C("passes-tensor-pair-plain", "gaussian", 5 * tm, 3 * tn, 784, 6, False, 128, "tensor_pair", 4, passes=2,
          regimes=("tensor_passes", "ro_mod256_128", "ro_mod64_0")),
        # knobs (each read once per process: these run in a child process)
        C("knob-pair-off-tensor-waves", "gaussian", s["t2"], s["t2"] + PAD, 64, 2, True, 254, "tensor", 2, data="diagonal",
          env=PAIR_OFF, regimes=("knob_pair_off", "knob_multiwave")),
        C("knob-pair-off-tensor-abs", "absolute-exponential", 5 * tm + 1, 7 * tn, 64, 4, False, 126, "tensor", 4,
          data="diagonal", env=PAIR_OFF, regimes=("knob_pair_off",)),
        C("knob-pair-off-pv16-waves", "dot-exponential", s["p2"], s["p2"] + PAD, 64, 64, True, 62, "pv16", data="diagonal",
          env=PAIR_OFF, regimes=("knob_pair_off", "knob_multiwave")),
        C("knob-flush-1-pv16-pair-waves", "gaussian", s["p2"], s["p2"] + PAD, 64, 64, True, 63, "pv16_pair", data="diagonal",
          env=FLUSH_1, regimes=("knob_flush_1", "knob_multiwave")),
        C("knob-flush-1-pv16-plain", "absolute-exponential", tm, 8 * tns, 64, 70, False, 62, "pv16", passes=2,
          data="diagonal", env=FLUSH_1, regimes=("knob_flush_1",)),
    ]
    return out


@functools.lru_cache(maxsize=None)
def all_cases():
    cases = _instantiation_cases() + _regime_cases()
    names = [c.name for c in cases]
    assert len(set(names)) == len(names), "case names must be unique"
    return tuple(cases)


def to_json(cases):
    """The cases as JSON, for a child process that runs with a knob: sizes are derived from the default plans, which the
    knob would change there."""
    return json.dumps([dataclasses.asdict(c) for c in cases])


def from_json(text):
    out = []
    for d in json.loads(text):
        d["env"] = tuple(tuple(kv) for kv in d["env"])
        d["regimes"] = tuple(d["regimes"])
        out.append(Case(**d))
    return out


# ---- float64 cases: every kprod_f64 causal instantiation ------------------------------------------------------------------


@dataclasses.dataclass(frozen=True)
class F64Case:
    kernel: str
    N: int
    M: int
    D: int
    E: int
    norm: bool
    row_offset: int

    @property
    def name(self):
        return f"f64-{self.kernel}-N{self.N}-M{self.M}-D{self.D}-E{self.E}-{'norm' if self.norm else 'plain'}-ro{self.row_offset}"


def f64_cases():
    out = []
    for i, kernel in enumerate(KERNELS):
        for j, (D, E) in enumerate(((5, 1), (3, 2), (16, 3), (7, 8), (5, 11), (20, 3), (70, 70))):
            norm = (i + j) % 2 == 1
            rows = F64_WIDE_ROWS_PER_CTA if D > F64_MAX_D else F64_ROWS_PER_CTA
            N = 3 * rows + 37 + 10 * j                 # several CTAs, the last one partial
            ro = rows // 2 + 13 + 3 * i                # off the CTA size: a CTA's rows straddle its last source block
            out.append(F64Case(kernel, N, N + ro + 50 + 29 * j, D, E, norm, ro))
    return tuple(out)


# ---- data ---------------------------------------------------------------------------------------------------------------

# radius of the diagonal curve per kernel: the far sources of the curve must stay negligible against the near ones
DIAG_RADIUS = {"gaussian": 3.0, "dot-exponential": 5.5, "absolute-exponential": 15.0, "inverse-distance": 3.0}
# target i sits at curve(row_offset + i + DIAG_SHIFT): inverse distance keeps the zeroing rule off its nearest sources,
# and absolute-exponential keeps |x - y| away from 0, where sqrt amplifies the cancellation error of |x|^2 + |y|^2 - 2 x.y
# target i sits at curve(row_offset + i + DIAG_SHIFT).  Absolute-exponential: half a step, so |x - y| stays away from 0,
# where sqrt amplifies the cancellation error of |x|^2 + |y|^2 - 2 x.y.  Inverse distance: the zeroing rule removes the
# diagonal source itself, and 1/|x - y| has a heavy tail, so the target sits a quarter step before the first masked
# source (the one a mask off by +1 admits): its weight dominates the row.
DIAG_SHIFT = {"gaussian": 0.0, "dot-exponential": 0.0, "absolute-exponential": 0.5, "inverse-distance": 0.75}


def _seed(case):
    return zlib.crc32(case.name.encode())


def curve(index, D, radius, seed):
    """Points of the closed torus curve at (real) indices ``index``: (len(index), D) float64."""
    K = max(1, D // 2)
    omega = np.random.RandomState(seed).uniform(0.05, 0.3, K)
    ph = np.asarray(index, dtype=np.float64)[:, None] * omega[None, :]
    out = np.zeros((len(ph), D))
    s = radius / np.sqrt(K)
    out[:, 0:2 * K:2] = s * np.cos(ph)
    out[:, 1:2 * K:2] = s * np.sin(ph)
    return out


def make_data(case):
    """x (N, D), y (M, D), b (M, E) or None (density), as float64 holding float32 values (what the kernel and the oracle
    both see)."""
    rng = np.random.RandomState(_seed(case))
    N, M, D, E = case.N, case.M, case.D, case.E
    if case.data == "diagonal":
        seed = _seed(case) % 100000
        R = DIAG_RADIUS[case.kernel]
        y = curve(np.arange(M), D, R, seed)
        x = curve(case.row_offset + np.arange(N) + DIAG_SHIFT[case.kernel], D, R, seed)
        # alternating signs, zero mean: neighbouring sources pull a row in opposite directions
        sign = (-1.0) ** (np.arange(M)[:, None] + np.arange(E)[None, :])
        b = sign * (0.5 + rng.rand(M, E))
        b -= b.mean(axis=0, keepdims=True)
    else:
        if case.kernel == "dot-exponential":
            s = 1.5 / D ** 0.5
            x, y = s * rng.randn(N, D), s * rng.randn(M, D)
        else:
            r = (3.0 / D) ** 0.5
            x, y = r * rng.rand(N, D), r * rng.rand(M, D)
        b = 0.5 + rng.rand(M, E)
    f = lambda a: a.astype(np.float32).astype(np.float64)
    return f(x), f(y), (None if case.density else f(b))


def sample_rows(case, n_random=256):
    """Rows a large case is checked on: the first and last row of every tile, every row whose diagonal sits at a block
    or column-group edge (j0 - 1, j0, j0 + G - 1 for the crossing test's granularity G and for the source block), and
    n_random random rows; all rows of a small case."""
    if not case.sampled:
        return np.arange(case.N)
    tm = geometry()[0]
    first = schedule(case)[0]
    N, ro = case.N, case.row_offset
    rows = [np.arange(0, N, tm), np.minimum(np.arange(tm - 1, N + tm - 1, tm), N - 1)]
    for g in {first["block"], granularity(first["family"])}:
        j = ro + np.arange(N)
        rows.append(np.nonzero(np.isin(j % g, (g - 1, 0)))[0])
    rows.append(np.random.RandomState(_seed(case) + 1).randint(0, N, n_random))
    return np.unique(np.concatenate(rows))


def runs(rows):
    """Split sorted rows into runs of consecutive indices: [(start, stop), ...]."""
    rows = np.asarray(rows)
    if len(rows) == 0:
        return []
    cut = np.nonzero(np.diff(rows) != 1)[0] + 1
    return [(int(r[0]), int(r[-1]) + 1) for r in np.split(rows, cut)]


# ---- running a case on the GPU and checking it (tests/test_causal_coverage_gpu.py and its knob child processes) ---------

REL_L2, WORST_ROW = 1e-4, 1e-3


def run(case, x, y, b, lo=0, hi=None):
    """Rows [lo, hi) of the case's causal product on cuda:0 (row_offset + lo for their first row), as float64."""
    import torch

    from kernel_matrix_benchmarks_b200 import product as prod

    hi = case.N if hi is None else hi
    dev = torch.device("cuda", 0)
    t = lambda a: None if a is None else torch.tensor(a, dtype=torch.float32, device=dev)
    out = prod.kernel_product(t(x[lo:hi]), t(y), t(b), kernel=case.kernel, normalize_rows=case.norm and not case.density,
                              density_estimation=case.density, row_offset=case.row_offset + lo, causal=True)
    torch.cuda.synchronize()
    assert prod.last_path == "tensor_f16"
    return out.double().cpu().numpy()


def oracle_rows(case, x, y, b, rows):
    """(want, want under |b|) at ``rows`` from tests/causal_oracle.py, one call per run of consecutive rows."""
    norm = case.norm and not case.density
    want, scale = [], []
    for r0, r1 in runs(rows):
        kw = dict(row_offset=case.row_offset + r0, normalize_rows=norm, density_estimation=case.density)
        want.append(co.causal_product(case.kernel, x[r0:r1], y, b, **kw))
        scale.append(want[-1] if b is None else co.causal_product(case.kernel, x[r0:r1], y, np.abs(b), **kw))
    return np.concatenate(want), np.concatenate(scale)


def errors(got, want, scale):
    """(relative L2 error, worst row error, row of the worst), both relative to the norm under |b|."""
    num = np.linalg.norm(got - want, axis=1)
    den = np.maximum(np.linalg.norm(scale, axis=1), 1e-300)
    rel = float(np.linalg.norm(got - want) / max(np.linalg.norm(scale), 1e-300))
    per = num / den
    return rel, float(per.max()), int(np.argmax(per))


def check(case, got_rows, rows, x, y, b, what=""):
    assert np.all(np.isfinite(got_rows)), f"{case.name}{what}: non-finite output at rows {rows[~np.isfinite(got_rows).all(1)][:8]}"
    want, scale = oracle_rows(case, x, y, b, rows)
    rel, worst, at = errors(got_rows, want, scale)
    assert rel <= REL_L2 and worst <= WORST_ROW, f"{case.name}{what}: rel-L2 {rel:.2e}, worst row {worst:.2e} at row {rows[at]}"
    return rel, worst


def run_case(case):
    """Run, check against the oracle, repeat multi-wave cases: (rel, worst, bitwise repeat or None)."""
    x, y, b = make_data(case)
    got = run(case, x, y, b)
    rows = sample_rows(case)
    rel, worst = check(case, got[rows], rows, x, y, b)
    same = None
    if case.multiwave:
        again = run(case, x, y, b)
        same = bool(np.array_equal(got.view(np.uint64), again.view(np.uint64)))
    return rel, worst, same
