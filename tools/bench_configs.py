#!/usr/bin/env python
"""The BASELINE.json configs beside the headline one (C2 is bench.py's own): C1, C3, C4, C5 through the plugin API.

    python tools/bench_configs.py [c1 c3 c4 c5]              # one JSON object per config on stdout
    bench.py imports run_config_block() and puts the same objects under "configs" of its JSON line.

Per config: device time of query() (CUDA events inside the plugin, max over ranks), the main kernel's time (events the
library records around it), the roofline of SURVEY.md section 8(d) for that kernel, and parity of the result on sampled
target rows against the float64 C oracle (rank 0; the oracle only checks, outside every timed region).  L2 is flushed
between timed queries.  Under torchrun (WORLD_SIZE > 1) the products run with distributed=True (target rows sharded,
sources replicated, no collective on the data path; the row blocks are gathered in get_result) and the solve runs
B200Solver(distributed=True) (symmetric matvec: unit list split over the ranks, one all-reduce of N floats per iteration).
"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

MUFU_PER_CLK_PER_SM = 16.0


def _max_over_ranks(values, dev, world):
    import torch
    import torch.distributed as dist

    t = torch.tensor(list(values), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def _oracle_rows(kernel, y, x, b, got_rows, rows, tol, normalize_rows=False):
    from oracle import c_oracle

    t0 = time.perf_counter()
    want = c_oracle.kernel_product(kernel, y, x, b, normalize_rows=normalize_rows, rows=rows)
    got = np.asarray(got_rows, dtype=np.float64).reshape(want.shape)
    rel = float(np.linalg.norm(got - want) / np.linalg.norm(want))
    return {"rel_l2": rel, "rows": int(len(rows)), "tol": tol, "ok": bool(rel <= tol),
            "checker": "oracle/kprod_ref.c float64, all sources", "seconds": round(time.perf_counter() - t0, 2)}


def _rows(n, k, seed=2):
    return np.sort(np.random.RandomState(seed).choice(n, int(min(n, k)), replace=False))


def run_product(name, ds, *, local_rank=0, rank=0, world=1, runs=5, warm=3, parity_rows=256, tol=1e-5, peaks=None, outputs=None,
                key=None, **kw):
    """One product / attention config through B200Product.  Returns the config's JSON object (rank 0) or None.  With
    `outputs` (a dict), rank 0 also stores the result of the last timed query there under `key`."""
    import torch

    from kernel_matrix_benchmarks_b200 import product as _product
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    dev = torch.device("cuda", local_rank)
    algo = B200Product(kernel=ds.kernel, dimension=ds.D, normalize_rows=ds.normalize_rows, precision="float32",
                       device=local_rank, distributed=world > 1, **kw)
    algo.prepare_data(source_points=ds.source_points, target_points=ds.target_points, same_points=ds.same_points)
    t0 = time.perf_counter()
    algo.fit()
    fit_ms = 1e3 * (time.perf_counter() - t0)
    algo.prepare_query(source_signal=ds.source_signal)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    _product.set_profiling(True)
    q_ms, k_ms = [], []
    for i in range(warm + runs):
        flush.fill_(1)
        torch.cuda.synchronize(dev)
        algo.query()
        if i >= warm:
            q_ms.append(algo.query_ms)
            try:
                k_ms.append(_product.last_main_kernel_ms())
            except Exception:   # paths without a profiled main kernel (float64)
                k_ms.append(algo.query_ms)
    _product.set_profiling(False)
    extra = algo.get_additional()
    res = algo.get_result()
    algo.done()
    del flush
    query_ms, kernel_ms, fit_ms = _max_over_ranks([sum(q_ms) / len(q_ms), sum(k_ms) / len(k_ms), fit_ms], dev, world)
    if rank != 0:
        return None
    if outputs is not None:
        outputs[key] = res
    pairs = float(ds.N) * ds.M
    rows = _rows(ds.N, parity_rows)
    out = {"workload": name, "kernel": ds.kernel, "N": ds.N, "M": ds.M, "D": ds.D, "E": ds.E, "normalize_rows": bool(ds.normalize_rows),
           "n_gpus": world, "ms": query_ms, "kernel_ms": kernel_ms, "fit_ms": fit_ms, "runs": runs, "warmup": warm,
           "gpairs_per_s": pairs / (query_ms * 1e-3) / 1e9, "path_used": extra.get("path_used"), "gpu_launches_per_query": extra.get("gpu_launches"),
           "l2": "flushed between timed queries (256 MiB write)",
           "parity": _oracle_rows(ds.kernel, ds.source_points, None if ds.same_points else ds.target_points, ds.source_signal,
                                  res[rows], rows, tol, normalize_rows=ds.normalize_rows)}
    peaks = peaks or {}
    info = _product.device_info(local_rank)
    sm_max = float(peaks.get("sm_max_mhz") or info["clock_khz"] / 1e3)
    if ds.D <= 16:
        peak = MUFU_PER_CLK_PER_SM * info["sm_count"] * sm_max * 1e6 / 1e9
        achieved = pairs / world / (kernel_ms * 1e-3) / 1e9
        out["roofline"] = {"bound": "fp32_mufu", "achieved": achieved, "peak": peak, "unit": "Gpairs/s", "frac": achieved / peak,
                           "traffic": None, "kernel_ms": kernel_ms,
                           "peak_basis": f"16 MUFU.EX2/clk/SM x {info['sm_count']} SMs x {sm_max:.0f} MHz, one evaluation per pair "
                                         "(general kernel); at this size the launch is latency-bound, not pipe-bound"
                                         if pairs < 1e10 else f"16 MUFU.EX2/clk/SM x {info['sm_count']} SMs x {sm_max:.0f} MHz"}
    else:
        pv = ds.E > 4 and ds.D <= 128   # second contraction on the tensor cores too
        flops = 2.0 * pairs * (ds.D + (ds.E if pv else 0))
        achieved = flops / world / (kernel_ms * 1e-3) / 1e12
        peak = float(peaks.get("bf16_tflops") or 1590.0)
        sustained = peaks.get("bf16_tflops_sustained")
        mufu_per_pair = 2.0 if ds.kernel == "absolute-exponential" else 1.0   # rsqrt + ex2 vs ex2
        mufu_floor_ms = 1e3 * mufu_per_pair * pairs / world / (MUFU_PER_CLK_PER_SM * info["sm_count"] * sm_max * 1e6)
        out["roofline"] = {
            "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": None, "kernel_ms": kernel_ms,
            "executed_tflops": 3.0 * achieved, "frac_executed": 3.0 * achieved / peak,
            "frac_executed_vs_sustained": (3.0 * achieved / sustained) if sustained else None,
            "mufu_floor_ms": mufu_floor_ms,
            "peak_basis": "algorithmic flops 2*N*M*(D" + ("+E" if pv else "") + ") / main-kernel time vs MEASURED_PEAKS.json bf16_tflops (burst; FP16 hi/lo "
                          "operand planes run at the bf16 rate); the three-term split executes 3x the algorithmic flops, so frac <= 1/3 "
                          "and frac_executed is the tensor-pipe figure; mufu_floor_ms = the exponentials alone at 16/clk/SM"}
    return out


def run_solver(name, n, *, lam=1.0, rtol=1e-6, local_rank=0, rank=0, world=1, parity_rows=128, peaks=None, runs=1, warm=1,
               outputs=None, key=None):
    """C5: (K + lam I) b = a through B200Solver; the right-hand side is built by the product under test (B200Product) and
    checked on sampled rows against the oracle, like the residual of the solution.  `warm` untimed solves, then `runs`
    timed ones (ms = their mean).  With `outputs` (a dict), rank 0 also stores the solution of the last timed query there
    under `key`."""
    import torch

    from kernel_matrix_benchmarks_b200 import datasets
    from kernel_matrix_benchmarks_b200 import product as _product
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product, B200Solver

    dev = torch.device("cuda", local_rank)
    ds = datasets.config_c5(n, lam)
    prod = B200Product(kernel="gaussian", dimension=3, precision="float32", device=local_rank, distributed=world > 1)
    prod.prepare_data(source_points=ds.source_points, target_points=ds.source_points, same_points=True)
    prod.fit()
    prod.prepare_query(source_signal=ds.source_signal)
    prod.query()
    rhs = prod.get_result() + lam * ds.source_signal
    prod.done()

    algo = B200Solver(kernel="gaussian", dimension=3, precision="float32", lam=lam, rtol=rtol, max_iter=500,
                      device=local_rank, distributed=world > 1)
    algo.prepare_data(source_points=ds.source_points)
    fits = []
    for _ in range(2):   # the first fit() of a process also pays the lazy cuSOLVER / cuBLAS set-up
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        algo.fit()
        fits.append(1e3 * (time.perf_counter() - t0))
    algo.prepare_query(target_signal=rhs)
    queries = []
    for _ in range(warm + runs):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        algo.query()
        queries.append((1e3 * (time.perf_counter() - t0), algo.query_ms))
    x = algo.get_result()
    extra = algo.get_additional()
    # end to end through the plugin: host float64 right-hand side in (cast + H2D), solve, host float64 solution out
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    algo.prepare_query(target_signal=rhs)
    algo.query()
    algo.get_result()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    algo.done()
    timed = [q[1] for q in queries[warm:]]
    fit_first, fit_ms, q_first, q_ms, e2e_ms = _max_over_ranks([fits[0], fits[1], queries[0][1], sum(timed) / len(timed), e2e_ms],
                                                               dev, world)
    if rank != 0:
        return None
    if outputs is not None:
        outputs[key] = x
    it = max(1, int(extra["cg_iterations"]))
    rows = _rows(n, parity_rows, seed=5)
    from oracle import c_oracle

    t0 = time.perf_counter()
    want_rhs = c_oracle.kernel_product("gaussian", ds.source_points, None, ds.source_signal, rows=rows) + lam * ds.source_signal[rows]
    resid = c_oracle.kernel_product("gaussian", ds.source_points, None, x, rows=rows) + lam * x[rows] - rhs[rows]
    info = _product.device_info(local_rank)
    sm_max = float((peaks or {}).get("sm_max_mhz") or info["clock_khz"] / 1e3)
    symmetric = extra["matvec"] == "symmetric"
    peak = MUFU_PER_CLK_PER_SM * info["sm_count"] * sm_max * 1e6 / 1e9 * (2.0 if symmetric else 1.0)
    pairs_per_gpu_per_iteration = float(n) * n / world
    ms_it = q_ms / it
    achieved = pairs_per_gpu_per_iteration / (ms_it * 1e-3) / 1e9
    return {
        "workload": name, "kernel": "gaussian", "N": n, "M": n, "D": 3, "E": 1, "lam": lam, "rtol": rtol, "n_gpus": world,
        "ms": q_ms, "first_query_ms": q_first, "fit_ms": fit_ms, "first_fit_ms": fit_first, "e2e_ms": e2e_ms,
        "iterations": it, "ms_per_iteration": ms_it, "converged": bool(extra["cg_converged"]),
        "rel_residual_recurrence": float(extra["cg_rel_residual"]), "matvec": extra["matvec"], "preconditioner": extra["preconditioner"],
        "collective": ("none (1 GPU)" if world == 1 else
                       "one NCCL all-reduce of N floats per matvec (symmetric unit list split over the ranks)" if symmetric else
                       "one NCCL all-gather of p (N*E floats) + two E-float all-reduces per iteration"),
        "rel_l2_vs_generating_b": float(np.linalg.norm(x - ds.source_signal) / np.linalg.norm(ds.source_signal)),
        "parity": {"rel_residual_oracle": float(np.linalg.norm(resid) / np.linalg.norm(rhs[rows])),
                   "rhs_rel_l2": float(np.linalg.norm(rhs[rows] - want_rhs) / np.linalg.norm(want_rhs)),
                   "rows": int(len(rows)), "tol": 2e-5, "ok": bool(np.linalg.norm(resid) / np.linalg.norm(rhs[rows]) <= 2e-5),
                   "checker": "oracle/kprod_ref.c float64: |(K + lam I) x - a| / |a| on sampled rows, a checked on the same rows",
                   "seconds": round(time.perf_counter() - t0, 2)},
        "roofline": {"bound": "fp32_mufu", "achieved": achieved, "peak": peak, "unit": "Gpairs/s", "frac": achieved / peak, "traffic": None,
                     "peak_basis": f"per iteration and GPU: N*M/n_gpus pairs / (query ms / iterations) vs 16 MUFU.EX2/clk/SM x {info['sm_count']} SMs x "
                                   f"{sm_max:.0f} MHz / {0.5 if symmetric else 1.0} evaluations per pair; the iteration also holds the preconditioner "
                                   "(two tall-skinny cuBLAS products) and the vector kernels"},
        "gpu_launches": int(extra["gpu_launches"]),
    }


def run_config_block(which, *, local_rank=0, rank=0, world=1, parity_rows=256, peaks=None, outputs=None):
    """bench.py's "configs" object: name -> result (rank 0), None elsewhere.  Every rank must call it (collectives).
    With `outputs` (a dict), rank 0 also stores each config's result there under its entry of `which` ("c1", ...)."""
    from kernel_matrix_benchmarks_b200 import datasets

    if isinstance(peaks, tuple):
        peaks = peaks[0]
    out = {}
    common = dict(local_rank=local_rank, rank=rank, world=world, peaks=peaks, outputs=outputs)
    if "c1" in which:
        out["C1"] = run_product("C1: gaussian product N=M=10^4, D=3, E=1", datasets.config_c1(), parity_rows=parity_rows, tol=1e-5,
                                runs=10, key="c1", **common)
    if "c3" in which:
        out["C3"] = run_product("C3: gaussian product M=60000, N=10000, D=784, E=1 (tcgen05, FP16 hi/lo planes, CTA pairs)",
                                datasets.config_c3(), parity_rows=min(parity_rows, 128), tol=1e-4, runs=10, key="c3", **common)
    if "c4" in which:
        out["C4"] = run_product("C4: absolute-exponential attention N=M=262144, D=64, E=64 (row-normalised; both contractions on tcgen05)",
                                datasets.config_c4(), parity_rows=min(parity_rows, 128), tol=1e-4, runs=3, warm=2, key="c4", **common)
    if "c4g" in which:
        out["C4-gaussian"] = run_product("C4 with the gaussian kernel", datasets.config_c4(kernel="gaussian"),
                                         parity_rows=min(parity_rows, 128), tol=1e-4, runs=3, warm=2, key="c4g", **common)
    if "c5" in which:
        out["C5"] = run_solver("C5: gaussian solve (K + I) b = a, N=M=10^6, D=3, preconditioned CG", 1_000_000,
                               parity_rows=min(parity_rows, 128), key="c5", **common)
    if "c5s" in which:
        out["C5-small"] = run_solver("C5 at N=10^5", 100_000, parity_rows=min(parity_rows, 128), key="c5s", **common)
    return out if rank == 0 else None


def main():
    import torch

    world, rank, local_rank = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", "1"), ("RANK", "0"), ("LOCAL_RANK", "0")))
    which = [a.lower() for a in sys.argv[1:]] or ["c1", "c3", "c4", "c5"]
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    peaks = {}
    try:
        with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    res = run_config_block(which, local_rank=local_rank, rank=rank, world=world, peaks=peaks)
    if rank == 0:
        for k, v in res.items():
            print(json.dumps({"config": k, **v}), flush=True)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
