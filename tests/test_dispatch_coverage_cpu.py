"""Every product kernel instantiation the dispatcher can reach is the target of a parity case (tests/dispatch_cases.py),
and each case reaches what it claims: checked with the host-only plan query (kmb_debug_product_plan), no GPU needed.

A new direct table entry, a change of the signal-chunk rule or of a kernel family's applicability fails here, naming
what lost its case, until tests/dispatch_cases.py has a case for it (which tests/test_dispatch_coverage_gpu.py runs)."""
import json
import os
import subprocess
import sys

import pytest

import dispatch_cases as dc
from conftest import REPO


def _plan(case):
    """dispatch_plan of the case; P.B cases also get their pv_plan as plan["pv"]."""
    from kernel_matrix_benchmarks_b200 import product

    plan = product.dispatch_plan(case.N, case.M, case.D, case.E, kernel=case.kernel, normalize_rows=case.norm,
                                 density_estimation=case.density, path=case.path, sms=dc.SMS)
    if case.group:
        plan["pv"] = product.pv_plan(case.N, case.M, case.D, case.E, kernel=case.kernel, normalize_rows=case.norm,
                                     path=case.path, sms=dc.SMS, smem_optin=dc.SMEM_OPTIN)
    return plan


def _env_plans(cases):
    """dispatch_plan of cases that set environment knobs, each group in a child process with that environment (the
    knobs are read once per process)."""
    plans = {}
    for env in sorted({c.env for c in cases}):
        group = [c for c in cases if c.env == env]
        script = ("import json, sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import dispatch_cases as dc; "
                  "from test_dispatch_coverage_cpu import _plan; "
                  "print(json.dumps({c.name: _plan(c) for c in dc.all_cases() if c.env == tuple(map(tuple, json.loads(sys.argv[3])))}))")
        child_env = dict(os.environ, **dict(env))
        res = subprocess.run([sys.executable, "-c", script, REPO, os.path.join(REPO, "tests"), json.dumps(env)],
                             env=child_env, capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, res.stderr
        got = json.loads(res.stdout.strip().splitlines()[-1])
        assert sorted(got) == sorted(c.name for c in group)
        plans.update(got)
    return plans


@pytest.fixture(scope="module")
def plans():
    cases = dc.all_cases()
    out = {c.name: _plan(c) for c in cases if not c.env and c.family != "f64"}
    out.update(_env_plans([c for c in cases if c.env]))
    return out


def _mismatch(case, plan, tables):
    """Why the plan does not reach the case's target (None when it does)."""
    if plan["family"] != case.family:
        return f"family {plan['family']}, expected {case.family}"
    if plan["chunk"] != case.chunk or plan["passes"] != case.passes:
        return f"{plan['passes']} passes of {plan['chunk']} columns, expected {case.passes} of {case.chunk}"
    if case.family == "direct":
        table, DP, EP = case.entry
        key = "prod" if case.form == "product" else "diff"
        if plan[f"{key}_table"] != table:
            return f"{key}-form table {plan[f'{key}_table']}, expected {table}"
        ent = tables[table][plan[f"{key}_index"]]
        if (ent["DP"], ent["EP"]) != (DP, EP):
            return f"entry DP{ent['DP']}/EP{ent['EP']}, expected DP{DP}/EP{EP}"
        if case.form == "difference" and plan["prod_table"] != -1 and case.data != "spread":
            return "the product form is enqueued too: the unit-scale data would select it"
    return None


def _units(case, ent):
    """(row tiles, source blocks) of the case on a direct entry (the plan reports the difference form's; the product
    form's records are wider under row normalisation)."""
    return -(-case.N // ent["TILE_ROWS"]), -(-case.M // ent["SB"])


def test_every_case_reaches_its_target(plans):
    tables = dc._direct_tables()
    bad = [f"{c.name}: {m}" for c in dc.all_cases() if c.family != "f64" for m in [_mismatch(c, plans[c.name], tables)] if m]
    assert not bad, "\n".join(bad)


def test_every_direct_table_entry_has_a_case(plans):
    """All 8 tables x 25 entries; each entry with a case of its own D = DP, a single full pass, a split tile (3 row tiles x
    4 source blocks) and a CTA-contained tile."""
    tables = dc._direct_tables()
    assert len(tables) == len(dc.DIRECT_TABLES) == 8
    for t, (kernel, norm, form) in enumerate(dc.DIRECT_TABLES):
        for ent in tables[t]:
            assert (ent["NORM"], ent["FORM"]) == (int(norm), int(form == "product")), (t, ent)
    reached = {}
    tables_cases = [c for c in dc.all_cases() if c.family == "direct"]
    for c in tables_cases:
        p = plans[c.name]
        key = "prod" if c.form == "product" else "diff"
        ent = tables[p[f"{key}_table"]][p[f"{key}_index"]]
        tiles, blocks = _units(c, ent)
        kind = "contained" if tiles == 1 and blocks == 1 else "split" if tiles >= 2 and blocks >= 3 else "other"
        reached.setdefault((p[f"{key}_table"], ent["DP"], ent["EP"]), set()).add(kind)
    missing = []
    for t, entries in enumerate(tables):
        for ent in entries:
            kinds = reached.get((t, ent["DP"], ent["EP"]), set())
            for kind in ("contained", "split"):
                if kind not in kinds:
                    missing.append(f"table {t} {dc.DIRECT_TABLES[t]} DP={ent['DP']} EP={ent['EP']}: no {kind}-tile case")
    assert not missing, "direct entries without a parity case:\n" + "\n".join(missing)


def test_direct_edges_are_covered(plans):
    """Per table: multi-pass signals on EP 8 / 16, a partial last pass on every EP >= 4, zero-padded D < DP on DP 8 / 16,
    and per (table, DP) a case with more units than the resident grid (~2 units per CTA: partial slots 0 and 1)."""
    tables = dc._direct_tables()
    seen = set()
    for c in dc.all_cases():
        if c.family != "direct":
            continue
        p = plans[c.name]
        t, DP, EP = c.entry
        key = "prod" if c.form == "product" else "diff"
        tiles, blocks = _units(c, tables[p[f"{key}_table"]][p[f"{key}_index"]])
        if p["passes"] > 1:
            seen.add(("multipass", t, EP))
        if c.E % EP:
            seen.add(("partial", t, EP))
        if c.D < DP:
            seen.add(("padded", t, DP))
        units = tiles * blocks
        if 2 * dc.SMS < units <= 3 * 2 * dc.SMS and c.sample_rows:
            seen.add(("stream-k", t, DP))
    want = set()
    for t in range(len(tables)):
        want |= {("multipass", t, EP) for EP in (8, 16)} | {("partial", t, EP) for EP in (4, 8, 16)}
        want |= {("padded", t, DP) for DP in (8, 16)} | {("stream-k", t, DP) for DP in dc.DIRECT_DIMS}
    assert not sorted(want - seen), f"uncovered: {sorted(want - seen)}"


def test_gaussian_difference_form_is_reached_both_ways(plans):
    """The Gaussian difference-form tables run through path='direct_diff' on unit data and through 'auto' on spread data."""
    for t in (0, 1):
        ways = {(c.path, c.data) for c in dc.all_cases() if c.family == "direct" and c.entry[0] == t}
        assert ("direct_diff", "unit") in ways and ("auto", "spread") in ways, (t, ways)
        spread_dps = {c.entry[1] for c in dc.all_cases() if c.family == "direct" and c.entry[0] == t and c.data == "spread"}
        assert spread_dps == set(dc.DIRECT_DIMS), spread_dps


def test_tensor_families_are_covered(plans):
    """kprod_tensor (TF32 and FP16 single CTA, KMB_TENSOR_PAIR=0 included) and kprod_tensor_pair at every template EP
    (e_chunk 1, 2, 3 -> 4, 4) x kernel x normalisation; the multi-pass route (D > 128, E > 4) with both element types; density
    at D in {40, 784} on every E <= 4 family; pv16 with KMB_TENSOR_PAIR=0."""
    seen = set()
    for c in dc.all_cases():
        p = plans.get(c.name)
        if p is None or p["family"] not in ("tensor", "tensor_pair", "pv", "pv16", "pv16_pair"):
            continue
        ep = {1: 1, 2: 2, 3: 4, 4: 4}.get(p["chunk"], p["chunk"])
        elt = "f16" if p["path"] == "tensor_f16" else "tf32"
        if c.density:
            seen.add(("density", p["family"], elt, c.D))
        elif p["passes"] > 1:
            seen.add(("multipass", p["family"], elt, c.kernel, c.norm, c.D))
        else:
            seen.add((p["family"], elt, ep, c.kernel, c.norm, bool(c.env)))
    want = set()
    for kernel in dc.KERNELS:
        for norm in (False, True):
            for ep in (1, 2, 4):
                want |= {("tensor", "tf32", ep, kernel, norm, False), ("tensor", "f16", ep, kernel, norm, False),
                         ("tensor_pair", "f16", ep, kernel, norm, False)}
            want |= {("tensor", "f16", ep, kernel, norm, True) for ep in (1, 4)}
            for D in (200, 784):
                want |= {("multipass", "tensor", "tf32", kernel, norm, D), ("multipass", "tensor_pair", "f16", kernel, norm, D)}
            if kernel != "inverse-distance":
                want.add(("pv16", "f16", 64, kernel, norm, True))
    for D in dc.TENSOR_DIMS:
        want |= {("density", "tensor", "tf32", D), ("density", "tensor", "f16", D), ("density", "tensor_pair", "f16", D)}
    assert not sorted(want - seen, key=str), f"uncovered: {sorted(want - seen, key=str)}"


def test_inverse_distance_row_offsets_are_covered(plans):
    """row_offset != 0 (not a multiple of any tile) on the direct kernel, the E <= 4 tensor kernels (single CTA, CTA pairs)
    and kprod_tensor_pv, each also with N > M + 1 (the zeroed column wraps inside the shard); x a copy of y."""
    seen = set()
    for c in dc.all_cases():
        if c.kernel != "inverse-distance" or c.precision != "float32":
            continue
        fam = plans[c.name]["family"]
        if c.row_offset:
            assert c.row_offset % 128 and c.row_offset % 1024
            seen.add((fam, "offset"))
            if c.N > c.M + 1:
                seen.add((fam, "wrap"))
        if c.data == "copy":
            assert c.N == c.M
            seen.add((fam, "copy"))
    want = {(f, k) for f in ("direct", "tensor", "tensor_pair", "pv") for k in ("offset", "wrap")}
    want |= {("direct", "copy"), ("tensor_pair", "copy"), ("pv", "copy")}
    assert not sorted(want - seen), f"uncovered: {sorted(want - seen)}"


def test_every_pb_case_reaches_its_launch_shape(plans):
    """Each P.B case runs in the group it names (pv, pv16 on one row tile, pv16_pair, pv16 with KMB_TENSOR_PAIR=0) and
    reaches every launch shape it is sized for (dc.pb_edges)."""
    bad = []
    for c in dc.all_cases():
        if not c.group:
            continue
        pv = plans[c.name]["pv"]
        group = dc.pb_group(pv, c.env)
        missed = set(c.edges) - dc.pb_edges(pv, c.env)
        if group != c.group or missed:
            bad.append(f"{c.name}: group {group}, missed {sorted(missed)} ({pv})")
    assert not bad, "\n".join(bad)


def _pb_shapes(group):
    """Ring stages and (K blocks, K steps of the last one) the group's kernel takes over D = 1 .. 128."""
    from kernel_matrix_benchmarks_b200 import product

    family, path, kernels, env, blk, F = dc.PB_GROUPS[group]
    N = 401 if group == "pv16_pair" else 100   # pv16_pair_off: the single-CTA kernel's shapes (the pair knob is not set here)
    out = set()
    for D in range(1, 129):
        p = product.pv_plan(N, 700, D, 40, kernel=kernels[0], path=path, sms=dc.SMS, smem_optin=dc.SMEM_OPTIN)
        out |= {f"stages{p['stages']}", f"k{p['kblocks']}x{p['ksteps_last']}"}
    return out


def test_pb_launch_shapes_are_covered(plans):
    """Every (group, kernel, normalisation) of the P.B kernels has a parity case for each launch shape that selects different
    code: one pass padded to 32 and to 64 columns; two passes with a last pass of 1 and of 32 columns and three with a last
    of 1; every ring-stage count and (K blocks, K steps) D can select; row tiles split over CTAs; and, unless the problem
    has one row tile, two waves and CTA ranges of F - 1, F, F + 1 and 2F + 1 source blocks (F = the flush interval).  CTA
    pairs: an odd row-tile count (ghost tile).  FP16 planes: KMB_PV16_FLUSH_BLOCKS = 1 and 3 (3 only with
    KMB_TENSOR_PAIR=0).  Also: far rows under normalisation, signal columns of very different magnitudes (pv, pv16,
    pv16_pair) and, for pairs, columns 0-31 and 32-63 2^100 apart."""
    seen = set()
    for c in dc.all_cases():
        if c.group:
            key = (c.group, c.kernel, c.norm)
            seen |= {key + (e,) for e in dc.pb_edges(plans[c.name]["pv"], c.env)}
            if c.far_rows:
                seen.add(key + ("far",))
            if c.data in ("magnitude", "halves"):
                seen.add(key + (c.data,))
    want = set()
    for group, (family, path, kernels, env, blk, F) in dc.PB_GROUPS.items():
        edges = {"ebp32", "ebp64", "2pass-narrow", "2pass-last32", "3pass-narrow", "split"} | _pb_shapes(group)
        if group != "pv16":
            edges |= {"waves", "flush-1", "flush", "flush+1", "2flush+1"}
        if group == "pv16_pair":
            edges |= {"ghost", "halves"}
        if family != "pv":
            edges |= {"knob3"} if group == "pv16_pair_off" else {"knob1", "knob3"}
        if group != "pv16_pair_off":
            edges.add("magnitude")
        for kernel in kernels:
            for norm in (False, True):
                want |= {(group, kernel, norm, e) for e in edges | ({"far"} if norm else set())}
    missing = sorted(want - seen, key=str)
    assert not missing, "P.B launch shapes without a parity case:\n" + "\n".join(map(str, missing))


def test_pv_plan_query():
    """kmb_debug_pv_plan: argument checks, only the family for another family, and the fields it shares with
    kmb_debug_product_plan; the ring stages shrink with D and are fewer with less shared memory, and too little for the
    resident u tile is KMB_ERR_UNSUPPORTED."""
    import ctypes

    from kernel_matrix_benchmarks_b200 import _lib, product

    lib = _lib.load()
    out = (ctypes.c_int64 * len(product.PV_PLAN_FIELDS))()
    assert lib.kmb_debug_pv_plan(300, 700, 64, 64, 0, 0, 5, 0, dc.SMEM_OPTIN, out) == _lib.KMB_ERR_INVALID   # sms < 1
    assert lib.kmb_debug_pv_plan(300, 700, 64, 64, 0, 0, 5, dc.SMS, 0, out) == _lib.KMB_ERR_INVALID          # smem < 1
    assert lib.kmb_debug_pv_plan(300, 0, 64, 64, 0, 0, 5, dc.SMS, dc.SMEM_OPTIN, out) == _lib.KMB_ERR_INVALID     # M < 1
    assert lib.kmb_debug_pv_plan(300, 700, 64, 64, 0, 0, 5, dc.SMS, 100000, out) == _lib.KMB_ERR_UNSUPPORTED
    plan = lambda *a, **k: product.pv_plan(*a, sms=dc.SMS, smem_optin=dc.SMEM_OPTIN, **k)  # noqa: E731
    p = plan(100, 700, 64, 3)
    assert p["family"] == "tensor" and set(p.values()) == {"tensor", -1}
    for kernel in dc.KERNELS:
        for path in ("auto", "tensor_f16", "tensor_tf32"):
            for N, M, D, E in ((100, 700, 40, 5), (401, 50, 128, 129), (20000, 9000, 3, 64), (300, 700, 17, 96)):
                p, d = plan(N, M, D, E, kernel=kernel, path=path), product.dispatch_plan(N, M, D, E, kernel=kernel, path=path)
                assert p["family"] == d["family"], (kernel, path, N, M, D, E)
                if d["family"] not in ("pv", "pv16", "pv16_pair"):
                    continue
                assert (p["passes"], p["row_tiles"]) == (d["passes"], d["row_tiles"])
                assert p["pair"] == (d["family"] == "pv16_pair") and p["grid"] == dc.SMS
                blk = 64 if d["family"] == "pv" else 128
                assert p["source_blocks"] == -(-M // blk) and p["eb_first"] == min(E, 64)
                assert p["eb_last"] == E - 64 * (p["passes"] - 1) and p["ebp_last"] == -(-p["eb_last"] // 32) * 32
                assert p["flush_blocks"] == (64 if d["family"] == "pv" else 128)
    stages = [plan(100, 700, D, 40, path=path)["stages"] for path in ("tensor_tf32", "tensor_f16") for D in (16, 128)]
    assert stages[0] > stages[1] and stages[2] > stages[3], stages
    assert product.pv_plan(100, 700, 128, 40, path="tensor_tf32", sms=dc.SMS, smem_optin=dc.SMEM_OPTIN - 20000)["stages"] < stages[1]


def test_inverse_distance_never_resolves_to_pv16():
    """kprod_tensor_pv16 takes no row offset and has no inverse-distance form: inverse distance must go elsewhere."""
    from kernel_matrix_benchmarks_b200 import product

    for D in (1, 3, 16, 17, 64, 128, 129, 784):
        for E in (1, 4, 5, 31, 32, 64, 65, 200):
            for path in ("auto", "tensor_f16", "tensor_tf32"):
                for N in (1, 129, 10000):
                    fam = product.dispatch_plan(N, 500, D, E, kernel="inverse-distance", path=path)["family"]
                    assert fam not in ("pv16", "pv16_pair"), (D, E, path, N, fam)


def test_float64_instantiations_are_covered():
    """kprod_f64 (D <= 16): the 1-, 2-, 4- and 8-column instantiations x kernel x normalisation, and a two-pass signal."""
    seen, multipass = set(), set()
    for c in dc.all_cases():
        if c.family != "f64":
            continue
        assert c.D <= 16 and c.passes == len(dc.f64_buckets(c.E))
        seen |= {(c.kernel, c.norm, b) for b in dc.f64_buckets(c.E)}
        if c.passes > 1:
            multipass.add((c.kernel, c.norm))
    want = {(k, n, b) for k in dc.KERNELS for n in (False, True) for b in (1, 2, 4, 8)}
    assert not sorted(want - seen, key=str), f"uncovered: {sorted(want - seen, key=str)}"
    assert multipass == {(k, n) for k in dc.KERNELS for n in (False, True)}


def test_plan_query_arguments():
    """kmb_debug_product_plan / kmb_debug_direct_entry: argument checks, the fill and symmetric families, and a direct plan
    whose entry is what find_direct picks (the smallest DP >= D, then the smallest EP >= e_chunk)."""
    import ctypes

    from kernel_matrix_benchmarks_b200 import _lib, product

    lib = _lib.load()
    out = (ctypes.c_int64 * 10)()
    assert lib.kmb_debug_product_plan(10, 10, 3, 1, 0, 0, 0, 0, out) == _lib.KMB_ERR_INVALID          # sms < 1
    assert lib.kmb_debug_product_plan(10, 0, 3, 1, 0, 0, 0, 148, out) == _lib.KMB_ERR_INVALID         # M < 1
    assert lib.kmb_debug_product_plan(10, 10, 3, 1, 9, 0, 0, 148, out) == _lib.KMB_ERR_UNSUPPORTED    # kernel
    e = (ctypes.c_int32 * 11)()
    assert lib.kmb_debug_direct_entry(8, 0, e) == _lib.KMB_ERR_INVALID
    assert lib.kmb_debug_direct_entry(0, 25, e) == 0 and e[0] == 25 and e[1] == -1
    assert product.dispatch_plan(10, 10, 3, 1, normalize_rows=True, density_estimation=True)["family"] == "fill"
    assert product.dispatch_plan(10, 10, 3, 1, path="direct_sym")["family"] == "sym"
    assert product.dispatch_plan(10, 10, 17, 1, path="direct")["family"] == "unsupported"
    p = product.dispatch_plan(5000, 1000, 5, 6, kernel="gaussian")
    assert p["path"] == "direct" and p["chunk"] == 8 and p["passes"] == 1
    tables = dc._direct_tables()
    assert (tables[0][p["diff_index"]]["DP"], tables[0][p["diff_index"]]["EP"]) == (8, 8) and p["diff_table"] == 0
    assert p["prod_table"] == 6 and tables[6][p["prod_index"]]["DP"] == 8
    assert p["row_tiles"] == -(-5000 // tables[0][p["diff_index"]]["TILE_ROWS"])
    assert product.dispatch_plan(5000, 1000, 5, 6, path="direct_diff")["prod_table"] == -1
