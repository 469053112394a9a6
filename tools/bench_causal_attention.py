"""Causal against full kernel products on the FP16 tensor path: C4 attention and one E = 1 product.

    python tools/bench_causal_attention.py [--rounds 10] [--out FILE]

Workloads (C4 = datasets.config_c4 points and signal, N = M = 262144, D = 64, E = 64, row-normalised):
    dot-exponential C4   softmax attention, pv16 family, causal (row i sees sources j <= i) and full
    gaussian C4          the same inputs with the Gaussian kernel
    gaussian E=1         N = M = 65536, D = 64, E = 1, row-normalised: the kprod_tensor family
The causal and full product of each workload alternate in one process (A B, then B A, ...); every pass is preceded by a
write of 512 MB that evicts the 126 MB L2 and timed twice: the main kernel alone (kmb_set_profiling /
kmb_last_main_kernel_ms: CUDA events around the last pass's main kernel) and the whole call (CUDA events, prepass
included).  Sampled rows of each causal output are compared with the float64 causal oracle (tests/causal_oracle.py).
Prints the device name and power limit read in the same run and one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "tests"), os.path.join(REPO, "tools")]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=10, help="timed passes per variant (alternating)")
    ap.add_argument("--n", type=int, default=262_144)
    ap.add_argument("--n-e1", type=int, default=65_536)
    ap.add_argument("--parity-rows", type=int, default=64)
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch

    import causal_oracle as co
    from bench_dot_attention import device_facts
    from kernel_matrix_benchmarks_b200 import datasets, product

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    facts = device_facts(0)
    print(f"device: {facts['device']}, power limit {facts['power_limit_w']:.0f} W, max SM clock {facts['sm_clock_max_mhz']:.0f} MHz")
    t = lambda a: torch.tensor(np.ascontiguousarray(a), dtype=torch.float32, device="cuda")  # noqa: E731
    ds = datasets.config_c4(n=args.n, kernel="gaussian")
    c4 = (ds.target_points, ds.source_points, ds.source_signal)
    rng = np.random.RandomState(3)
    r = (3.0 / 64) ** 0.5
    e1 = (r * rng.rand(args.n_e1, 64), r * rng.rand(args.n_e1, 64), 0.5 + rng.rand(args.n_e1, 1))
    workloads = {"dot-exponential C4": ("dot-exponential", c4), "gaussian C4": ("gaussian", c4), "gaussian E=1": ("gaussian", e1)}
    sms = product.device_info(0)["sm_count"]
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = dict(facts, rounds=args.rounds, method="causal and full alternate in one process, L2 overwritten before each pass; "
                                                "main kernel: kmb_last_main_kernel_ms; call: CUDA events around kernel_product")
    for name, (kernel, (x, y, b)) in workloads.items():
        xt, yt, bt = t(x), t(y), t(b)
        N, M, E = x.shape[0], y.shape[0], b.shape[1]
        ws = {c: product.Workspace() for c in (True, False)}
        out = {}

        def run(causal):
            return product.kernel_product(xt, yt, bt, kernel=kernel, normalize_rows=True, workspace=ws[causal], causal=causal)

        for c in (True, False):   # warm-up
            for _ in range(2):
                out[c] = run(c)
        torch.cuda.synchronize()
        main_ms, call_ms = {True: [], False: []}, {True: [], False: []}
        product.set_profiling(True)
        for i in range(args.rounds):
            for c in ((True, False) if i % 2 == 0 else (False, True)):
                flush.fill_(i & 0xFF)
                ev0.record()
                out[c] = run(c)
                ev1.record()
                ev1.synchronize()
                call_ms[c].append(ev0.elapsed_time(ev1))
                main_ms[c].append(product.last_main_kernel_ms())
        product.set_profiling(False)
        rows = np.unique(np.concatenate([rng.choice(N, args.parity_rows, replace=False), [0, 1, 127, 128, 255, N - 1]]))
        x64, y64, b64 = (a.astype(np.float32).astype(np.float64) for a in (x, y, b))
        got = out[True].cpu().numpy().astype(np.float64)[rows]
        want = np.concatenate([co.causal_product(kernel, x64[i:i + 1], y64, b64, row_offset=int(i), normalize_rows=True) for i in rows])
        entry = {"kernel": kernel, "N": N, "M": M, "D": 64, "E": E,
                 "family": product.dispatch_plan(N, M, 64, E, kernel=kernel, normalize_rows=True, sms=sms, causal=True)["family"],
                 "parity_rows": int(len(rows)), "parity_rel_l2": co.rel_l2(got, want), "parity_worst_row": co.worst_row(got, want),
                 "finite": bool(torch.isfinite(out[True]).all().item())}
        for c, tag in ((True, "causal"), (False, "full")):
            entry[tag] = {"main_kernel_median_ms": float(np.median(main_ms[c])), "main_kernel_min_ms": float(np.min(main_ms[c])),
                          "call_median_ms": float(np.median(call_ms[c]))}
        entry["main_kernel_ratio_causal_over_full"] = entry["causal"]["main_kernel_median_ms"] / entry["full"]["main_kernel_median_ms"]
        res[name] = entry
        print(f"{name:>20}: main kernel causal {entry['causal']['main_kernel_median_ms']:.2f} ms, full "
              f"{entry['full']['main_kernel_median_ms']:.2f} ms, ratio {entry['main_kernel_ratio_causal_over_full']:.3f} "
              f"({entry['family']}); parity rel-L2 {entry['parity_rel_l2']:.2e}, worst row {entry['parity_worst_row']:.2e}")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
