"""Parity cases of the dot-exponential kernel exp(<x, y>) (not in bruteforce.py) on every tensor-core family it runs on
(no GPU needed to import).

tests/test_dot_exponential_cpu.py checks with the host-only plan query (product.dispatch_plan) that each case reaches the
family it names and that every family has a case; tests/test_dot_exponential_gpu.py runs them against the float64
oracle (tests/dot_exponential_oracle.py).

The kernel has no direct kernel: "auto" resolves to the FP16-plane tensor path at every D.  The family follows from the
element type, the signal width and D: E > 4 and D <= 128 take a P.B kernel (pv16 / pv16_pair with FP16 planes, pv with
TF32 planes), everything else the E <= 4 kernels, D > 128 with E > 4 in several signal passes of 4 columns (the
multi-pass route).  FP16 planes use CTA pairs from two row tiles on, unless KMB_TENSOR_PAIR=0.
"""
from __future__ import annotations

import dataclasses
import functools
import zlib

import numpy as np

KERNEL = "dot-exponential"
DIMS = (3, 16, 40, 64, 200, 784)
SIGNALS = (1, 2, 3, 4, 8, 64, 200)
PATHS = ("auto", "tensor_f16", "tensor_tf32")
PAIR_OFF = (("KMB_TENSOR_PAIR", "0"),)
# every family the kernel can reach (product.dispatch_plan names; "multipass": D > 128, E > 4 on the E <= 4 kernels)
FAMILIES = ("tensor", "tensor_pair", "pv", "pv16", "pv16_pair", "multipass")
TOL = 1e-4   # BASELINE's tensor-path tolerance (relative L2); the worst row within 10x


@dataclasses.dataclass(frozen=True)
class Case:
    name: str
    N: int
    M: int
    D: int
    E: int
    norm: bool = False
    density: bool = False
    path: str = "auto"
    env: tuple = ()
    repeat: bool = False   # run twice: the output must be bitwise identical

    @property
    def f16(self):
        return self.path != "tensor_tf32"

    @property
    def family(self):
        """The family the case targets (product.dispatch_plan name)."""
        pair = self.f16 and self.N > 128 and dict(self.env).get("KMB_TENSOR_PAIR") != "0"
        if self.E > 4 and self.D <= 128:
            return ("pv16_pair" if pair else "pv16") if self.f16 else "pv"
        return "tensor_pair" if pair else "tensor"

    @property
    def chunk(self):
        return 64 if self.family.startswith("pv") else min(self.E, 4)

    @property
    def passes(self):
        return -(-self.E // self.chunk)

    @property
    def covers(self):
        """Coverage key: the family, or "multipass" for the D > 128 route."""
        return "multipass" if self.D > 128 and self.E > 4 else self.family


@functools.lru_cache(maxsize=None)
def all_cases():
    out = []
    add = lambda name, **kw: out.append(Case(f"dotexp-{name}", **kw))  # noqa: E731
    # the full grid on four row tiles (FP16: CTA pairs) and M = 700 sources (not a multiple of any source block)
    for D in DIMS:
        for E in SIGNALS:
            for norm in (False, True):
                for path in PATHS:
                    add(f"{path}-n{int(norm)}-D{D}-E{E}", N=401, M=700, D=D, E=E, norm=norm, path=path,
                        repeat=(D == 64 and E in (4, 64) and not norm))
        for path in PATHS:
            add(f"density-{path}-D{D}", N=401, M=700, D=D, E=1, density=True, path=path)
    # one row tile: the single-CTA FP16 kernels
    for D in (3, 40, 784):
        for E in (1, 4, 64):
            for norm in (False, True):
                add(f"single-n{int(norm)}-D{D}-E{E}", N=100, M=700, D=D, E=E, norm=norm)
        add(f"single-density-D{D}", N=100, M=700, D=D, E=1, density=True)
    # fewer sources than one source block
    for E in (2, 64):
        add(f"few-sources-E{E}", N=401, M=50, D=64, E=E, norm=True)
    # KMB_TENSOR_PAIR=0 (read once per process: a child process): the single-CTA FP16 kernels on several row tiles
    for D in (3, 64, 200):
        for E in (4, 64):
            for norm in (False, True):
                add(f"pair-off-n{int(norm)}-D{D}-E{E}", N=401, M=700, D=D, E=E, norm=norm, path="tensor_f16", env=PAIR_OFF,
                    repeat=(D == 64 and not norm))
    names = [c.name for c in out]
    assert len(set(names)) == len(names), "case names must be unique"
    return tuple(out)


def make_data(case):
    """(x, y, b) as float64 arrays of float32-representable values.  Coordinates N(0, s^2) with s^2 sqrt(D) = 2, so that
    <x, y> has a standard deviation of 2 at every D and the kernel values span about e^-8 .. e^8; signal columns of
    distinct scales and signs with source-dependent means (see dispatch_cases.make_data)."""
    rng = np.random.RandomState(zlib.crc32(case.name.encode()))
    s = (2.0 / case.D ** 0.5) ** 0.5
    y, x = s * rng.randn(case.M, case.D), s * rng.randn(case.N, case.D)
    b = None
    if not case.density:
        scale = np.array([(-1.0) ** e * 2.0 ** (e % 5 - 2) for e in range(case.E)])
        b = scale * (0.5 + rng.rand(case.M, case.E) + np.linspace(0.0, 1.0, case.M)[:, None])
    cast = lambda a: None if a is None else a.astype(np.float32).astype(np.float64)  # noqa: E731
    return cast(x), cast(y), cast(b)
