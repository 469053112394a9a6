"""Softmax attention (the dot-exponential kernel exp(<x, y>), row-normalised) against the Gaussian kernel at the C4 shape.

    python tools/bench_dot_attention.py [--rounds 10] [--out FILE]

C4: N = M = 262144 targets and sources, D = 64, E = 64, row-normalised (datasets.config_c4 points and signal, the same
inputs for both kernels).  Both run kernel_product as a user calls it (prepass included, FP16-plane tensor path) on
cuda:0.  The two kernels alternate in one process (A B, then B A, ...), each pass timed with CUDA events and preceded by
a write of 512 MB that evicts the 126 MB L2.  After the timed rounds, sampled rows of each kernel's last output are
compared with the float64 C oracles (tests/dot_exponential_oracle.py for exp(<x, y>), oracle/c_oracle.py for the
Gaussian).  Prints the device name and power limit read in the same run and one JSON line.
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


def device_facts(index=0):
    """name, power limit [W] and max SM clock [MHz] of GPU `index` (nvidia-smi query, read only)."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                          str(index)], capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (f.strip() for f in out.split(","))
    return {"device": name, "power_limit_w": float(power), "sm_clock_max_mhz": float(clock)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=10, help="timed passes per kernel (alternating)")
    ap.add_argument("--n", type=int, default=262_144)
    ap.add_argument("--parity-rows", type=int, default=256)
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch

    import dot_exponential_oracle as dxo
    from kernel_matrix_benchmarks_b200 import datasets, product
    from oracle import c_oracle

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    facts = device_facts(0)
    print(f"device: {facts['device']}, power limit {facts['power_limit_w']:.0f} W, max SM clock {facts['sm_clock_max_mhz']:.0f} MHz")
    ds = datasets.config_c4(n=args.n, kernel="gaussian")
    t = lambda a: torch.tensor(np.ascontiguousarray(a), dtype=torch.float32, device="cuda")  # noqa: E731
    x, y, b = t(ds.target_points), t(ds.source_points), t(ds.source_signal)
    kernels = ("dot-exponential", "gaussian")
    ws = {k: product.Workspace() for k in kernels}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = {}

    def run(kernel):
        return product.kernel_product(x, y, b, kernel=kernel, normalize_rows=True, workspace=ws[kernel])

    for k in kernels:   # warm-up: module load, workspace allocation, tensor maps
        for _ in range(2):
            out[k] = run(k)
    torch.cuda.synchronize()
    times = {k: [] for k in kernels}
    for r in range(args.rounds):
        for k in (kernels if r % 2 == 0 else kernels[::-1]):
            flush.fill_(r & 0xFF)   # overwrite L2 with data the product does not read
            ev0.record()
            out[k] = run(k)
            ev1.record()
            ev1.synchronize()
            times[k].append(ev0.elapsed_time(ev1))
    paths = {k: product.resolved_path(64, b.shape[1], k) for k in kernels}

    rng = np.random.RandomState(1)
    rows = np.unique(np.concatenate([rng.choice(args.n, args.parity_rows, replace=False), [0, 127, 128, args.n - 1]]))
    b64 = ds.source_signal.astype(np.float32).astype(np.float64)
    y64, x64 = (a.astype(np.float32).astype(np.float64) for a in (ds.source_points, ds.target_points))
    want = {"dot-exponential": dxo.kernel_product_c(y64, x64, b64, normalize_rows=True, rows=rows),
            "gaussian": c_oracle.kernel_product("gaussian", y64, x64, b64, normalize_rows=True, rows=rows)}
    res = dict(facts, workload=f"attention N=M={args.n}, D=64, E=64 (C4 points and signal), row-normalised, kernel_product "
                                "with prepass, L2 overwritten before every pass", rounds=args.rounds)
    for k in kernels:
        got = out[k].cpu().numpy().astype(np.float64)[rows]
        ms = np.array(times[k])
        res[k] = {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()), "path": paths[k],
                  "family": product.dispatch_plan(args.n, args.n, 64, b.shape[1], kernel=k, normalize_rows=True,
                                                  sms=product.device_info(0)["sm_count"])["family"],
                  "parity_rows": int(len(rows)),
                  "parity_rel_l2": float(np.linalg.norm(got - want[k]) / np.linalg.norm(want[k]))}
        print(f"{k:>16}: median {res[k]['median_ms']:.2f} ms (min {res[k]['min_ms']:.2f}, max {res[k]['max_ms']:.2f}) over "
              f"{args.rounds} passes, {res[k]['family']}, rel-L2 vs float64 oracle on {len(rows)} rows {res[k]['parity_rel_l2']:.2e}")
    res["ratio_dot_over_gaussian"] = res["dot-exponential"]["median_ms"] / res["gaussian"]["median_ms"]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
