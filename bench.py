#!/usr/bin/env python
"""Headline benchmark: Gaussian kernel product K.b, N = M = 1M, D = 3, E = 1 (BASELINE.json config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A step is one pass of the hot path over the whole synthetic problem: a_i = sum_j exp(-|x_i-y_j|^2) b_j
for all N targets.  The C2 dataset has targets == sources (datasets.uniform_cube, same_points), so the
default path is the symmetric kernel (kprod_sym: every kernel value feeds its row and its column).
With G > 1 GPUs the problem stays fixed (strong scaling): the triangular unit list is cut into G equal
ranges, one per rank, and the ranks' partial results are summed with one NCCL all-reduce of N floats
inside the timed step.  `--path direct` times the general (x != y) kernel instead, target rows sharded,
no collective.  Rank 0 prints ONE JSON line.

  value     Gpairs/s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       same metric through the plugin call sequence (runner.py:73-143) with HOST float64
            arrays: cast + H2D of points and signal, query, D2H of the result inside the timer
  roofline  the dominant kernel against the FP32/MUFU pipe roofline of SURVEY.md section 8(d):
            16 kernel evaluations/clk/SM x SMs x clocks.max.sm (this path is compute bound: its
            compulsory HBM traffic is 32 MB per 10^12 pairs).  The symmetric kernel needs one
            evaluation per TWO pairs, so its peak is 32 pairs/clk/SM; `frac` is against that and
            `frac_vs_one_eval_per_pair` against the 16 pairs/clk/SM figure of the general kernel
  cpu_baseline / --impl reference
            the reference's own BruteForceProductBLAS (float32, fast_sqdists=True), imported from the copy
            of the reference tree that __graft_entry__.build() stages in the git-ignored baseline/_ref
            (kind "reference"), on a bounded row sample with all host cores; the NumPy port in oracle/
            (kind "port") only when that tree is absent
  parity    sampled target rows of the TIMED output (and of the e2e result) against the float64 C oracle
            (oracle/kprod_ref.c -- the checker, never the thing measured), at every N: rel_l2, rows, tol
  --workload solve
            config C5 (the kernel solve) as the line's own metric (ms per solve, lower is better) with iterations, ms per
            iteration, fit() time and the collective -- for 1/2/4/8-GPU sweeps of the solve
  configs   the other BASELINE.json configs on the same line (skip with --no-configs): C1 (N=M=10^4), C3 (D=784,
            tensor path), C4 (D=E=64 attention, tensor path), C5 (CG solve, N=10^6) through the plugin API, each
            with ms, its roofline (SURVEY.md section 8d formulas) and oracle parity on sampled rows; under
            torchrun C3/C4 shard target rows and C5 runs the solver across the ranks
  --dump-outputs DIR
            after the run, what each timed path returned in its last step: product.npy (the device-resident output,
            float32), e2e_product.npy (the plugin's float64 result), and one file per config (c1.npy, c3.npy, c4.npy,
            c5.npy: the plugin's result).  Every file holds all N target rows, also under torchrun: bench.py gathers
            the row shards of the headline paths and the plugin's get_result gathers those of the configs.  The inputs
            are seeded, so two builds run with the same arguments can be compared file for file; an output over 6 MiB
            keeps a seeded sample of its rows, the same one in every run
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(1, os.path.join(REPO, "tools"))

METRIC = "gaussian_kernel_product_gpairs_per_s"
UNIT = "Gpairs/s"
PAIRS_PER_CLK_PER_SM = 16.0  # MUFU lanes per SM per clock == issue bound of the 8-slot pair (SURVEY.md 8d)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=1_000_000, help="N = M (default: the BASELINE config, 1M)")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU sample (0 = sized for ~15 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--path", default="auto", choices=["auto", "direct"],
                    help="auto: symmetric kernel (targets == sources); direct: general kernel, rows sharded")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1/C3/C4/C5 block")
    ap.add_argument("--configs", default="c1,c3,c4,c5", help="which of c1,c3,c4,c5 to run beside the headline")
    ap.add_argument("--parity-rows", type=int, default=256, help="sampled rows checked against the C oracle")
    ap.add_argument("--workload", default="product", choices=["product", "solve"],
                    help="product: the headline C2 product (default); solve: BASELINE config C5, (K + I) b = a at N = 10^6, as the line's own metric")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what each timed path returned in its last step as DIR/<name>.npy (float32 / float64) so that two "
                         "builds can be compared output for output; an output over 6 MiB is stored as a fixed, seeded sample of rows")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU paths; the reference arm keeps none")
    return args


def workload_config(n, n_gpus, path="auto"):
    sharding = (f"symmetric unit list over {n_gpus} GPU(s), points replicated, one all-reduce of N floats per step"
                if path == "auto" else f"target rows over {n_gpus} GPU(s), sources replicated, no collective")
    if path == "auto" and n_gpus == 1:
        sharding = "1 GPU, symmetric kernel (same_points), no collective"
    return {
        "workload": f"C2: gaussian kernel product N=M={n}, D=3, E=1 (datasets.uniform_cube semantics)",
        "kernel": "gaussian",
        "N": n,
        "M": n,
        "D": 3,
        "E": 1,
        "path": "symmetric (kprod_sym)" if path == "auto" else "general (kprod_direct)",
        "sharding": sharding,
        "l2": "flushed between timed steps (256 MiB write)",
    }


def read_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


def measured_traffic(n, world, sym):
    """dram__bytes_read.sum + dram__bytes_write.sum of the main kernel from the committed ncu capture
    (profiles/r*_traffic_*.json); only valid for the workload it was captured on."""
    try:
        name = "r2_traffic_sym_kernel.json" if sym else "r1_traffic_main_kernel.json"
        with open(os.path.join(REPO, "profiles", name)) as f:
            t = json.load(f)
        if t["N"] == n and world == 1:
            return t["dram_bytes_per_launch"], f"ncu-captured ({t['source']}), not measured in this run"
    except Exception:
        pass
    return None, "none: no ncu capture of this kernel on this workload"


def oracle_parity(kernel, y, x, b, got_rows, rows, tol, normalize_rows=False):
    """Sampled target rows of a GPU result against the float64 C oracle (oracle/kprod_ref.c, pinned to the reference's
    golden vectors by tests/test_oracle_c.py).  The oracle is the checker here, outside every timed region."""
    from oracle import c_oracle

    t0 = time.perf_counter()
    want = c_oracle.kernel_product(kernel, y, x, b, normalize_rows=normalize_rows, rows=rows)
    got = np.asarray(got_rows, dtype=np.float64).reshape(want.shape)
    rel = float(np.linalg.norm(got - want) / np.linalg.norm(want))
    return {"rel_l2": rel, "rows": int(len(rows)), "tol": tol, "ok": bool(rel <= tol),
            "checker": "oracle/kprod_ref.c float64, all sources", "seconds": round(time.perf_counter() - t0, 2)}


def sample_rows(n, k, seed=2):
    k = int(min(n, k))
    return np.sort(np.random.RandomState(seed).choice(n, k, replace=False))


DUMP_ARRAY_BYTES = 6 << 20    # at most eight outputs (product, e2e_product, c1, c3, c4, c4g, c5, c5s) stay under 64 MB
DUMP_TOTAL_BYTES = 64_000_000


def dump_outputs(directory, arrays):
    """--dump-outputs: name -> array as DIR/<name>.npy.  An array over DUMP_ARRAY_BYTES keeps as many rows as fit,
    chosen by sample_rows(..., seed=3): the same rows in every run with the same arguments."""
    os.makedirs(directory, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"output {name} is {a.dtype}, not float32 / float64")
        if a.nbytes > DUMP_ARRAY_BYTES:
            a = a[sample_rows(a.shape[0], DUMP_ARRAY_BYTES // (a.nbytes // a.shape[0]), seed=3)]
        path = os.path.join(directory, name + ".npy")
        np.save(path, a)
        total += os.path.getsize(path)
    if total > DUMP_TOTAL_BYTES:
        raise RuntimeError(f"--dump-outputs wrote {total} bytes, more than {DUMP_TOTAL_BYTES}")


# ------------------------------------------------------------------------------------ CPU arm


_REF_CLASS = "unset"


def reference_class():
    """The reference's own BruteForceProductBLAS (bruteforce.py:61-153), imported from the copy of the reference tree
    that __graft_entry__.build() stages in the git-ignored baseline/_ref (it travels to the GPU box with the
    snapshot; /root/reference is never read here).  None when the tree is not there: the NumPy port is timed instead."""
    global _REF_CLASS
    if _REF_CLASS == "unset":
        try:
            from kernel_matrix_benchmarks_b200.harness import bootstrap

            if bootstrap.find_reference() is None:
                raise ImportError("reference tree not staged")
            bootstrap.activate()
            from kernel_matrix_benchmarks.algorithms.bruteforce import BruteForceProductBLAS

            _REF_CLASS = BruteForceProductBLAS
        except Exception as e:  # noqa: BLE001
            print(f"[bench] reference class unavailable ({e}); timing the NumPy port", file=sys.stderr)
            _REF_CLASS = None
    return _REF_CLASS


def cpu_reference_sample(ds, rows, precision="float32", fast_sqdists=True, row_block=500):
    """The reference algorithm (bruteforce.py:25-58 + :153) on `rows` target rows x all sources, in its fastest
    configuration (float32, BLAS squared distances).  With the reference tree staged: the reference's own class,
    fed blocks of `row_block` target rows (a 500 x 10^6 float32 kernel block is 2 GB), timing fit() + query() as its
    harness does (runner.py:97-143); otherwise the NumPy port in oracle/.  Returns (seconds, kind)."""
    cls = reference_class()
    if cls is None:
        from oracle import bruteforce_oracle as orc

        t0 = time.perf_counter()
        orc.kernel_product(ds.kernel, ds.source_points, None, ds.source_signal, precision=precision,
                           fast_sqdists=fast_sqdists, rows=rows, row_block=64)
        return time.perf_counter() - t0, "port"
    secs = 0.0
    for lo in range(0, len(rows), row_block):
        algo = cls(kernel=ds.kernel, dimension=ds.D, normalize_rows=False, precision=precision, fast_sqdists=fast_sqdists)
        algo.prepare_data(source_points=ds.source_points, target_points=ds.source_points[rows[lo:lo + row_block]],
                          same_points=False, density_estimation=False)
        algo.prepare_query(source_signal=ds.source_signal)
        t0 = time.perf_counter()
        algo.fit()
        algo.query()
        secs += time.perf_counter() - t0
        algo.get_result()
        del algo
    return secs, "reference"


def _cpu_sample_text(kind):
    if kind == "reference":
        return ("the reference's own BruteForceProductBLAS (baseline/_ref, float32, fast_sqdists=True), fit() + query() on blocks "
                "of 500 target rows: OpenBLAS GEMM on all cores, exp/broadcast ufuncs single-threaded")
    return ("NumPy port of bruteforce.py float32 fast_sqdists=True: OpenBLAS GEMM on all cores, exp/broadcast ufuncs "
            "single-threaded")


def host_threads():
    """Threads the BLAS pool actually has (what `cores` reports)."""
    try:
        from threadpoolctl import threadpool_info

        n = [p["num_threads"] for p in threadpool_info() if p.get("user_api") == "blas"]
        return int(max(n)) if n else os.cpu_count()
    except Exception:
        return os.cpu_count()


def use_all_host_threads():
    """torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which would hold the reference's OpenBLAS calls to
    one thread (round 1: 0.247 instead of 0.317 Gpairs/s).  The CPU arm is meant to use every host core."""
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=os.cpu_count())
    except Exception as e:  # noqa: BLE001
        print(f"[bench] could not raise the BLAS thread limit ({e})", file=sys.stderr)


def cpu_baseline(ds, n_rows):
    use_all_host_threads()
    rows = np.random.RandomState(1).choice(ds.N, n_rows, replace=False)
    rows.sort()
    secs, kind = cpu_reference_sample(ds, rows)
    pairs = float(n_rows) * ds.M
    return {
        "value": pairs / secs / 1e9,
        "unit": UNIT,
        "cores": host_threads(),
        "kind": kind,
        "sample": f"{n_rows} target rows x {ds.M} sources ({pairs:.2e} pairs, {secs:.1f} s), " + _cpu_sample_text(kind),
    }


def pick_cpu_rows(ds, requested):
    if requested:
        return requested
    # ~1.5e8 pairs/s measured for this variant in the survey; aim at ~15 s
    return int(max(64, min(ds.N, 2.0e9 // ds.M)))


def run_reference_arm(args):
    """--impl reference: the reference's CPU algorithm on a bounded sample per step (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from kernel_matrix_benchmarks_b200 import datasets

    use_all_host_threads()
    ds = datasets.config_c2(args.n)
    n_rows = pick_cpu_rows(ds, args.cpu_rows)
    rows = np.sort(np.random.RandomState(1).choice(ds.N, n_rows, replace=False))
    for _ in range(args.warmup):
        cpu_reference_sample(ds, rows[: max(8, n_rows // 16)])
    runs = [cpu_reference_sample(ds, rows) for _ in range(args.steps)]
    secs, kind = [r[0] for r in runs], runs[0][1]
    ms = 1e3 * sum(secs) / len(secs)
    pairs = float(n_rows) * ds.M
    value = pairs / (ms * 1e-3) / 1e9
    sample = (f"each step = {n_rows} target rows x {ds.M} sources ({pairs:.2e} pairs) of the C2 workload; " + _cpu_sample_text(kind))
    print(json.dumps({
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": dict(workload_config(args.n, args.gpus, args.path),
                       path="reference CPU: BruteForceProductBLAS(float32, fast_sqdists=True), dense blocks of 500 target rows"
                       if kind == "reference" else "NumPy port of bruteforce.py (oracle/), float32, fast_sqdists=True",
                       sharding="host cores only (rank 0); no GPU on this arm", l2="n/a (CPU arm)"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": host_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------ GPU arm


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        clocks, powers, reasons, sm_max = [], [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [t.strip() for t in line.split(",")]
                if len(f) < 9:
                    continue
                clocks.append(float(f[1]))
                sm_max = float(f[2])
                powers.append(float(f[3]))
                for name, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if clocks:
            # "under load": samples at or above the median power
            med_p = float(np.median(powers))
            loaded = [c for c, p in zip(clocks, powers) if p >= med_p] or clocks
            out.update(sm_mhz=float(np.median(loaded)), sm_max_mhz=sm_max, reasons=sorted(reasons), samples=len(clocks),
                       power_w_max=max(powers))
        return out


def run_b200_arm(args):
    import torch
    import torch.distributed as dist

    from kernel_matrix_benchmarks_b200 import datasets, product
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product
    from kernel_matrix_benchmarks_b200.solver import shard_bounds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ds = datasets.config_c2(args.n)  # same seeded arrays on every rank
    N, M = ds.N, ds.M
    lo, hi, _ = shard_bounds(N, rank, world)
    pairs_total = float(N) * float(M)

    # ---- device-resident arm ---------------------------------------------------------------
    y = torch.from_numpy(ds.source_points.astype(np.float32)).to(dev)
    b = torch.from_numpy(ds.source_signal.astype(np.float32)).to(dev)
    sym = args.path == "auto"
    if sym and not product.symmetric_applies(y, y, "gaussian"):
        raise SystemExit("the symmetric path does not apply to this workload")
    x = y[lo:hi]
    out = torch.empty((N if sym else hi - lo, 1), dtype=torch.float32, device=dev)
    ws = product.Workspace()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        if not sym:
            product.kernel_product(x, y, b, kernel="gaussian", path="direct", row_offset=lo, out=out, workspace=ws)
        elif world == 1:
            product.kernel_product(y, y, b, kernel="gaussian", path="direct_sym", out=out, workspace=ws)
        else:
            product.kernel_product_sym_part(y, b, rank, world, out=out, workspace=ws)
            dist.all_reduce(out)   # the exchange step of the symmetric split: N floats

    product.set_profiling(True)
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms, launches = [], 0
    for e0, e1 in ev:
        flush.fill_(1)  # evict L2 between timed steps (outside the event bracket)
        e0.record()
        step()
        e1.record()
        kernel_ms.append(product.last_main_kernel_ms())
        launches += product.last_launch_count()   # the library's launches of this step's call
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    step_ms = sum(a.elapsed_time(b_) for a, b_ in ev) / args.steps
    step_ms = max_over_ranks(step_ms)
    main_ms = max_over_ranks(sum(kernel_ms) / len(kernel_ms))
    value = pairs_total / (step_ms * 1e-3) / 1e9

    # the general (x != y) kernel on the same data, rows sharded: what a caller without same_points gets
    general = None
    if sym:
        out_g = torch.empty((hi - lo, 1), dtype=torch.float32, device=dev)
        for _ in range(2):
            product.kernel_product(x, y, b, kernel="gaussian", path="direct", row_offset=lo, out=out_g, workspace=ws)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(2):
            product.kernel_product(x, y, b, kernel="gaussian", path="direct", row_offset=lo, out=out_g, workspace=ws)
        g1.record()
        barrier()
        g_ms = max_over_ranks(g0.elapsed_time(g1) / 2)
        g_main_ms = max_over_ranks(product.last_main_kernel_ms())
        general = {"value": pairs_total / (g_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": g_ms, "kernel_ms": g_main_ms,
                   "timed": "2 whole calls (bounding-box statistics + source packing + main kernel), L2 warm; kernel_ms = the main kernel alone",
                   "kernel": "kprod_direct_kernel<D=3,E=1,R=4,gaussian,product form,512 thr>, target rows sharded"}
        # parity of the two kernels on this rank's rows (the tests hold both to the oracle)
        diff = (out[lo:hi] - out_g).double().norm() / out_g.double().norm()
        general["rel_l2_symmetric_vs_general"] = float(diff)

    # ---- parity of the timed output against the float64 C oracle on sampled rows (every N) -----------
    prows = sample_rows(N, args.parity_rows)
    if sym or world == 1:
        timed_rows = out[torch.as_tensor(prows, device=dev)].cpu().numpy()
    else:   # row shards: bring the sampled rows together (untimed)
        mine = torch.zeros((len(prows), 1), dtype=torch.float32, device=dev)
        sel = torch.as_tensor(prows, device=dev)
        inside = (sel >= lo) & (sel < hi)
        mine[inside] = out[sel[inside] - lo]
        dist.all_reduce(mine)
        timed_rows = mine.cpu().numpy()
    parity = None
    if rank == 0:
        parity = oracle_parity("gaussian", ds.source_points, None, ds.source_signal, timed_rows, prows, tol=1e-5)
        parity["of"] = "the device-resident output of the last timed step"

    dumps = {} if args.dump_outputs else None

    def whole(part):
        """All N rows of an output whose rows [lo, hi) this rank holds (untimed; every rank must call it)."""
        if sym or world == 1:
            return part.cpu().numpy()
        full = torch.zeros((N,) + tuple(part.shape[1:]), dtype=part.dtype, device=dev)
        full[lo:hi] = part
        dist.all_reduce(full)
        return full.cpu().numpy()

    if dumps is not None:
        dumps["product"] = whole(out)

    # ---- end-to-end arm: plugin API, host float64 arrays in, host float64 result out ------------
    e2e = None
    if not args.no_e2e:
        xs_host = ds.source_points[lo:hi]

        phases = {}   # host seconds per plugin call, summed over the timed steps (this rank)

        def timed(name, fn, **kw):
            t = time.perf_counter()
            out = fn(**kw)
            phases[name] = phases.get(name, 0.0) + time.perf_counter() - t
            return out

        def e2e_step():
            algo = timed("construct", B200Product, kernel="gaussian", dimension=3, normalize_rows=False, precision="float32",
                         path=args.path, device=local_rank, distributed=(sym and world > 1))
            if world == 1 or sym:
                timed("prepare_data", algo.prepare_data, source_points=ds.source_points, target_points=ds.source_points, same_points=True)
            else:
                timed("prepare_data", algo.prepare_data, source_points=ds.source_points, target_points=xs_host, same_points=False)
            timed("fit", algo.fit)
            timed("prepare_query", algo.prepare_query, source_signal=ds.source_signal)
            timed("query", algo.query)
            res = timed("get_result", algo.get_result)
            timed("done", algo.done)
            return res

        for _ in range(max(1, min(2, args.warmup))):
            e2e_step()
        barrier()
        phases.clear()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = e2e_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        e2e_ms = max_over_ranks(1e3 * dt / args.steps)
        n_x = 0 if (world == 1 or sym) else (hi - lo) * 3
        n_out = N if sym else hi - lo
        e2e = {
            "value": pairs_total / (e2e_ms * 1e-3) / 1e9,
            "unit": UNIT,
            "ms_per_step": e2e_ms,
            "h2d_bytes_per_step": int(4 * (n_x + M * 3 + M * 1)),
            "d2h_bytes_per_step": int(4 * n_out),
            "api": "B200Product.prepare_data/fit/prepare_query/query/get_result, host float64 in/out",
            "host_ms_per_call": {k: round(1e3 * v / args.steps, 3) for k, v in phases.items()},   # rank 0's clock
        }
        assert res.shape == (n_out, 1)
        if dumps is not None:
            dumps["e2e_product"] = whole(torch.from_numpy(res).to(dev))
        if rank == 0:
            sel = prows if (sym or world == 1) else prows[prows < hi]
            e2e["parity"] = oracle_parity("gaussian", ds.source_points, None, ds.source_signal, res[sel], sel, tol=1e-5)

    if rank == 0:
        peaks, peaks_src = read_peaks()
        info = product.device_info(local_rank)
        sm_max = float(clocks.get("sm_max_mhz") or peaks.get("sm_max_mhz") or info["clock_khz"] / 1e3)
        evals_per_pair = 0.5 if sym else 1.0   # the symmetric kernel evaluates k once per two pairs
        peak_evals = PAIRS_PER_CLK_PER_SM * info["sm_count"] * sm_max * 1e6 / 1e9   # G kernel evaluations/s per GPU
        peak = peak_evals / evals_per_pair                                           # Gpairs/s per GPU
        pairs_per_launch = pairs_total / world  # every rank evaluates an equal share
        achieved = pairs_per_launch / (main_ms * 1e-3) / 1e9
        kernel_name = ("kprod_sym_kernel<D=3,512 thr x 8 rows,butterfly 16> + sym_combine_kernel" if sym
                       else "kprod_direct_kernel<D=3,E=1,R=4,gaussian,product form,512 thr>")
        roofline = {
            "bound": "fp32_mufu",
            "achieved": achieved,
            "peak": peak,
            "unit": UNIT,
            "frac": achieved / peak,
            "frac_vs_one_eval_per_pair": achieved / peak_evals,
            "kernel_evals_per_pair": evals_per_pair,
            "traffic": measured_traffic(args.n, world, sym)[0],
            "traffic_source": measured_traffic(args.n, world, sym)[1],
            "kernel": kernel_name,
            "kernel_ms": main_ms,
            "peak_basis": f"16 kernel evaluations (MUFU.EX2)/clk/SM x {info['sm_count']} SMs x {sm_max:.0f} MHz (clocks.max.sm) "
                          f"/ {evals_per_pair} evaluations per pair; MEASURED_PEAKS.json {peaks_src}: hbm {peaks.get('hbm_gbs')} GB/s "
                          f"not binding (algorithmic HBM bytes/launch = {4 * (N * 3 + M * 4 + N)})",
            "frac_at_sampled_clock": (achieved * evals_per_pair / (PAIRS_PER_CLK_PER_SM * info["sm_count"] * clocks["sm_mhz"] * 1e-3)
                                      if clocks.get("sm_mhz") else None),
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.n, world, args.path),
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "parity": parity,
        }
        if general is not None:
            line["general_kernel"] = general
    # ---- the other BASELINE configs, same process group, same line ---------------------------------
    del out, ws, flush
    configs = None
    if not args.no_configs:
        from bench_configs import run_config_block   # tools/bench_configs.py

        configs = run_config_block([c.strip() for c in args.configs.split(",") if c.strip()], local_rank=local_rank, rank=rank,
                                   world=world, parity_rows=args.parity_rows, peaks=read_peaks(), outputs=dumps)
    if rank == 0:
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(ds, pick_cpu_rows(ds, args.cpu_rows))
        if dumps is not None:
            dump_outputs(args.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_solve_workload(args):
    """--workload solve: config C5 (Gaussian solve (K + I) b = a, N = M = 10^6, preconditioned CG through B200Solver) as the
    line's metric, so that a 1/2/4/8-GPU sweep reports the solve like the product: time of query() (device, max over ranks),
    iterations, ms per iteration, fit() time, the collective, oracle-scored residual.  One step = one solve: --warmup untimed
    solves, then --steps timed ones."""
    import torch
    import torch.distributed as dist

    from bench_configs import run_solver   # tools/bench_configs.py

    rank, world, local_rank = (int(os.environ.get(k, "0" if k != "WORLD_SIZE" else "1")) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    peaks, _ = read_peaks()
    dumps = {} if args.dump_outputs else None
    c5 = run_solver("C5: gaussian solve (K + I) b = a, N=M=10^6, D=3, preconditioned CG", args.n, local_rank=local_rank, rank=rank,
                    world=world, parity_rows=min(args.parity_rows, 128), peaks=peaks, runs=args.steps, warm=args.warmup,
                    outputs=dumps, key="c5")
    if rank == 0:
        clocks = sampler.stop()
        if dumps is not None:
            dump_outputs(args.dump_outputs, dumps)
        n = args.n
        print(json.dumps({
            "metric": "gaussian_kernel_solve_ms", "value": c5["ms"], "unit": "ms", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": c5["ms"], "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": c5["workload"], "N": n, "M": n, "D": 3, "E": 1, "lam": c5["lam"], "rtol": c5["rtol"],
                       "matvec": c5["matvec"], "preconditioner": c5["preconditioner"], "collective": c5["collective"],
                       "l2": "the 32 MB of records per matvec are L2-resident by design; nothing is flushed inside a solve"},
            "clocks": clocks, "iterations": c5["iterations"], "ms_per_iteration": c5["ms_per_iteration"], "fit_ms": c5["fit_ms"],
            "first_fit_ms": c5["first_fit_ms"], "converged": c5["converged"],
            "e2e": {"value": c5["e2e_ms"], "unit": "ms", "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": 4 * n,
                    "api": "B200Solver.prepare_query/query/get_result, host float64 in/out"},
            "gpu_launches": c5["gpu_launches"], "roofline": c5["roofline"], "parity": c5["parity"],
        }))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "solve":
        run_solve_workload(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
