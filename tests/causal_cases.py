"""Causal-product cases (KMB_FLAG_CAUSAL) that reach every kernel family with a causal instantiation -- kprod_tensor,
kprod_tensor_pair, pv16, pv16_pair, and the multi-pass kprod_tensor route (D > 128, E > 4) -- through the plan the
library itself reports (tests/test_causal_cpu.py) and on the GPU against tests/causal_oracle.py (test_causal_gpu.py).
Shapes cover N < M, N > M, N not a multiple of 128, N = 1, row offsets 0 / a multiple of 128 / 77 / >= M - 1, and plans
with several ranges per row tile and empty ranges (N = 256, M = 65536)."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass(frozen=True)
class CausalCase:
    kernel: str
    N: int
    M: int
    D: int
    E: int
    norm: bool
    row_offset: int
    family: str               # what dispatch_plan reports (148 SMs)
    density: bool = False
    env: tuple = ()           # environment of a child process, e.g. (("KMB_TENSOR_PAIR", "0"),)
    passes: int = 1

    @property
    def id(self):
        mode = "density" if self.density else ("norm" if self.norm else "plain")
        env = "-" + ",".join("=".join(kv) for kv in self.env) if self.env else ""
        return f"{self.family}-{self.kernel}-N{self.N}-M{self.M}-D{self.D}-E{self.E}-{mode}-ro{self.row_offset}{env}"

    def data(self, seed=0):
        """x (N, D), y (M, D), b (M, E) in float64: points in a cube of half-diagonal ~1 (dot-exponential: Gaussian
        points with |<x, y>| of a few units), a positive signal (rows of a plain product do not cancel)."""
        rng = np.random.RandomState(seed + self.N + 7 * self.M + 31 * self.D + self.E + self.row_offset)
        if self.kernel == "dot-exponential":
            s = 1.5 / self.D ** 0.5
            x, y = s * rng.randn(self.N, self.D), s * rng.randn(self.M, self.D)
        else:
            r = (3.0 / self.D) ** 0.5
            x, y = r * rng.rand(self.N, self.D), r * rng.rand(self.M, self.D)
        b = 0.5 + rng.rand(self.M, self.E)
        return x, y, b


PAIR_OFF = (("KMB_TENSOR_PAIR", "0"),)

CASES = [
    # kprod_tensor: one row tile (no pair), E <= 4
    CausalCase("gaussian", 100, 300, 3, 1, False, 0, "tensor"),
    CausalCase("absolute-exponential", 128, 1000, 16, 2, True, 77, "tensor"),
    CausalCase("inverse-distance", 120, 1000, 64, 3, True, 128, "tensor"),
    CausalCase("dot-exponential", 1, 5000, 200, 4, True, 4000, "tensor"),
    CausalCase("gaussian", 1, 300, 16, 1, False, 0, "tensor", density=True),
    # kprod_tensor_pair
    CausalCase("gaussian", 1000, 700, 64, 1, False, 0, "tensor_pair", density=True),
    CausalCase("gaussian", 640, 3000, 784, 2, True, 256, "tensor_pair"),
    CausalCase("dot-exponential", 256, 65536, 64, 1, True, 0, "tensor_pair"),
    CausalCase("inverse-distance", 300, 300, 128, 4, False, 0, "tensor_pair"),
    CausalCase("absolute-exponential", 400, 300, 3, 4, True, 299, "tensor_pair"),
    # pv16: one row tile
    CausalCase("gaussian", 100, 2000, 64, 8, True, 77, "pv16"),
    CausalCase("absolute-exponential", 1, 500, 16, 64, True, 0, "pv16"),
    CausalCase("dot-exponential", 128, 4000, 128, 200, True, 128, "pv16", passes=4),
    # pv16_pair
    CausalCase("dot-exponential", 256, 65536, 64, 64, True, 0, "pv16_pair"),
    CausalCase("gaussian", 1000, 1500, 128, 200, False, 128, "pv16_pair", passes=4),
    CausalCase("absolute-exponential", 700, 400, 3, 64, True, 1000, "pv16_pair"),
    CausalCase("gaussian", 300, 5000, 64, 64, True, 77, "pv16_pair"),
    # kprod_tensor over several signal passes (D > 128, E > 4)
    CausalCase("gaussian", 500, 900, 200, 8, True, 77, "tensor_pair", passes=2),
    CausalCase("absolute-exponential", 100, 700, 784, 64, False, 0, "tensor", passes=16),
    # KMB_TENSOR_PAIR=0: the single-CTA kernels on problems of several row tiles
    CausalCase("gaussian", 1000, 2000, 64, 2, True, 77, "tensor", env=PAIR_OFF),
    CausalCase("dot-exponential", 1000, 3000, 64, 64, True, 0, "pv16", env=PAIR_OFF),
    CausalCase("absolute-exponential", 256, 65536, 64, 8, True, 0, "pv16", env=PAIR_OFF),
]
