"""The one-term FP16 tensor path ("tensor_f16x1") against the three-term one ("tensor_f16") at C3 and C4.

    python tools/bench_f16x1.py [--rounds 10] [--out FILE]

Workloads (datasets.config_c3 / config_c4 points and signals, the same inputs for both arms):
  C3          N = 10^4 targets, M = 6 10^4 sources, D = 784, E = 1, Gaussian, plain product
  C4-gaussian N = M = 262144, D = E = 64, Gaussian, row-normalised
  C4-absexp   the same with the absolute-exponential kernel
Both arms run kernel_product on cuda:0 with the points prepared in advance (product.prepare_points on the arm's own
workspace: what B200Product.fit() does), so a pass is the query: signal planes + main kernel.  The arms alternate in one
process (A B, then B A, ...), every pass preceded by a write of 512 MB that evicts the 126 MB L2.  Per pass: the main
kernel's time (kmb_set_profiling / kmb_last_main_kernel_ms, CUDA events around the dominant kernel) and the query's
(CUDA events around kernel_product).  After the timed rounds, sampled rows of each arm's last output are compared with the
float64 C oracle (oracle/c_oracle.py).  Prints the device name and power limit read in the same run and one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "tests")]

ARMS = ("tensor_f16", "tensor_f16x1")


def device_facts(index=0):
    """name, power limit [W] and max SM clock [MHz] of GPU `index` (nvidia-smi query, read only)."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                          str(index)], capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (f.strip() for f in out.split(","))
    return {"device": name, "power_limit_w": float(power), "sm_clock_max_mhz": float(clock)}


def workloads():
    from kernel_matrix_benchmarks_b200 import datasets

    c4 = lambda kernel: datasets.config_c4(n=262_144, d=64, e=64, kernel=kernel)  # noqa: E731
    return (("C3", "gaussian", False, lambda: datasets.config_c3(60_000, 10_000, 784)),
            ("C4-gaussian", "gaussian", True, lambda: c4("gaussian")),
            ("C4-absexp", "absolute-exponential", True, lambda: c4("absolute-exponential")))


def bench(name, kernel, norm, ds, rounds, parity_rows, flush):
    import torch

    from kernel_matrix_benchmarks_b200 import product
    from oracle import c_oracle

    t = lambda a: torch.tensor(np.ascontiguousarray(a), dtype=torch.float32, device="cuda")  # noqa: E731
    x, y, b = t(ds.target_points), t(ds.source_points), t(ds.source_signal)
    (N, D), (M, E) = x.shape, b.shape
    ws, token, out = {}, {}, {}
    for arm in ARMS:   # fit(): the points-only prepass into the arm's own workspace
        ws[arm] = product.Workspace()
        need = product.workspace_bytes(N, M, D, E, kernel=kernel, normalize_rows=norm, path=arm)
        token[arm] = product.prepare_points(x, y, kernel=kernel, path=arm, workspace=ws[arm], min_bytes=need)
        assert token[arm] is not None

    def run(arm):
        return product.kernel_product(x, y, b, kernel=kernel, normalize_rows=norm, path=arm, workspace=ws[arm],
                                      prepared=token[arm])

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    product.set_profiling(True)
    for arm in ARMS:   # warm-up: module load, tensor maps
        for _ in range(2):
            out[arm] = run(arm)
    torch.cuda.synchronize()
    query_ms, main_ms = {a: [] for a in ARMS}, {a: [] for a in ARMS}
    for r in range(rounds):
        for arm in (ARMS if r % 2 == 0 else ARMS[::-1]):
            flush.fill_(r & 0xFF)   # overwrite L2 with data the product does not read
            ev0.record()
            out[arm] = run(arm)
            ev1.record()
            ev1.synchronize()
            query_ms[arm].append(ev0.elapsed_time(ev1))
            main_ms[arm].append(product.last_main_kernel_ms())
            assert ws[arm].buf is token[arm]   # the prepared head was used, not redone
    product.set_profiling(False)

    rng = np.random.RandomState(1)
    rows = np.unique(np.concatenate([rng.choice(N, min(parity_rows, N), replace=False), [0, 127, 128, N - 1]]))
    f64 = lambda a: a.astype(np.float32).astype(np.float64)  # noqa: E731
    want = c_oracle.kernel_product(kernel, f64(ds.source_points), f64(ds.target_points), f64(ds.source_signal),
                                   normalize_rows=norm, rows=rows)
    sms = product.device_info(0)["sm_count"]
    res = {"kernel": kernel, "normalize_rows": norm, "N": N, "M": M, "D": D, "E": E, "rounds": rounds}
    for arm in ARMS:
        got = out[arm].cpu().numpy().astype(np.float64)[rows]
        q, m = np.array(query_ms[arm]), np.array(main_ms[arm])
        res[arm] = {"main_kernel_median_ms": float(np.median(m)), "main_kernel_min_ms": float(m.min()),
                    "main_kernel_max_ms": float(m.max()), "query_median_ms": float(np.median(q)),
                    "query_min_ms": float(q.min()), "query_max_ms": float(q.max()),
                    "family": product.dispatch_plan(N, M, D, E, kernel=kernel, normalize_rows=norm, path=arm, sms=sms)["family"],
                    "parity_rows": int(len(rows)),
                    "parity_rel_l2": float(np.linalg.norm(got - want) / np.linalg.norm(want))}
        print(f"{name:>12} {arm:>13}: main kernel median {res[arm]['main_kernel_median_ms']:.3f} ms "
              f"(min {res[arm]['main_kernel_min_ms']:.3f}, max {res[arm]['main_kernel_max_ms']:.3f}), query median "
              f"{res[arm]['query_median_ms']:.3f} ms, {res[arm]['family']}, rel-L2 vs float64 oracle on {len(rows)} rows "
              f"{res[arm]['parity_rel_l2']:.2e}", flush=True)
    res["main_kernel_speedup"] = res[ARMS[0]]["main_kernel_median_ms"] / res[ARMS[1]]["main_kernel_median_ms"]
    res["query_speedup"] = res[ARMS[0]]["query_median_ms"] / res[ARMS[1]]["query_median_ms"]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=10, help="timed passes per arm (alternating)")
    ap.add_argument("--parity-rows", type=int, default=256)
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if args.rounds < 10:
        raise SystemExit("at least 10 passes per arm")
    facts = device_facts(0)
    print(f"device: {facts['device']}, power limit {facts['power_limit_w']:.0f} W, max SM clock {facts['sm_clock_max_mhz']:.0f} MHz")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    res = dict(facts, method="points prepared in advance; arms alternate in one process; L2 overwritten (512 MB) before "
                              "every pass; main kernel: CUDA events around the dominant kernel; query: CUDA events around "
                              "kernel_product")
    for name, kernel, norm, make in workloads():
        res[name] = bench(name, kernel, norm, make(), args.rounds, args.parity_rows, flush)
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
