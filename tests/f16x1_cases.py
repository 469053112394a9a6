"""Parity cases of the one-term FP16 tensor path ("tensor_f16x1", KMB_PATH_TENSOR_1XF16) on every family it reaches, and a
NumPy model of its arithmetic (no GPU needed to import).

tests/test_f16x1_cpu.py checks with the host-only plan query (product.dispatch_plan) that each case reaches the family it
names and that the model of the one-term arithmetic stays inside the tolerance; tests/test_f16x1_gpu.py runs every case
against the float64 oracle (oracle/c_oracle.py; tests/dot_exponential_oracle.py for exp(<x, y>)).

The path reaches the FP16-plane families of "tensor_f16" and no other: E > 4 with D <= 128 takes pv16 (pv16_pair from two
row tiles on, unless KMB_TENSOR_PAIR=0), everything else the E <= 4 kernels (tensor / tensor_pair), D > 128 with E > 4 in
several signal passes of 4 columns (the multi-pass route).  The inverse-distance kernel is not supported.
"""
from __future__ import annotations

import dataclasses
import functools
import zlib

import numpy as np

PATH = "tensor_f16x1"
KERNELS = ("gaussian", "absolute-exponential", "dot-exponential")
DIMS = (3, 16, 40, 64, 128, 200, 784)
SIGNALS = (1, 2, 3, 4, 8, 64, 200)
PAIR_OFF = (("KMB_TENSOR_PAIR", "0"),)
FAMILIES = ("tensor", "tensor_pair", "pv16", "pv16_pair", "multipass")
# Fixed before any GPU measurement, with at least 2.5x margin over the model of the arithmetic (model_product) on C3- and
# C4-shaped data and 4x on the worst row.  One FP16 term is float16-class: S carries 11 significand bits per operand, and
# for E > 4 the weights P and the signal b are rounded to one FP16 plane each.
TOL = 2e-3        # relative L2 over the whole result
ROW_TOL = 1e-2    # relative L2 of the worst row


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
    env: tuple = ()
    repeat: bool = False   # run twice: the output must be bitwise identical

    @property
    def family(self):
        """The family the case targets (product.dispatch_plan name)."""
        pair = self.N > 128 and dict(self.env).get("KMB_TENSOR_PAIR") != "0"
        if self.E > 4 and self.D <= 128:
            return "pv16_pair" if pair else "pv16"
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


_SHORT = {"gaussian": "gauss", "absolute-exponential": "absexp", "dot-exponential": "dotexp"}


@functools.lru_cache(maxsize=None)
def all_cases():
    out = []

    def add(name, kernel, **kw):
        out.append(Case(f"f16x1-{_SHORT[kernel]}-{name}", kernel, **kw))

    # the full grid on four row tiles (CTA pairs) and M = 1500 sources (not a multiple of any source block)
    for kernel in KERNELS:
        for D in DIMS:
            for E in SIGNALS:
                for norm in (False, True):
                    add(f"n{int(norm)}-D{D}-E{E}", kernel, N=401, M=1500, D=D, E=E, norm=norm,
                        repeat=(D == 64 and E in (4, 64) and not norm))
            add(f"density-D{D}", kernel, N=401, M=1500, D=D, E=1, density=True)
        # one row tile: the single-CTA kernels
        for D in (3, 64, 784):
            for E in (1, 4, 64):
                for norm in (False, True):
                    add(f"single-n{int(norm)}-D{D}-E{E}", kernel, N=100, M=1500, D=D, E=E, norm=norm)
            add(f"single-density-D{D}", kernel, N=100, M=1500, D=D, E=1, density=True)
        # KMB_TENSOR_PAIR=0 (read once per process: a child process): the single-CTA kernels on several row tiles
        for D in (3, 64, 200):
            for E in (2, 4, 64):
                for norm in (False, True):
                    add(f"pair-off-n{int(norm)}-D{D}-E{E}", kernel, N=401, M=1500, D=D, E=E, norm=norm, env=PAIR_OFF,
                        repeat=(D == 64 and E == 64 and not norm))
    names = [c.name for c in out]
    assert len(set(names)) == len(names), "case names must be unique"
    return tuple(out)


def make_data(case):
    """(x, y, b) as float64 arrays of float32-representable values.  Gaussian / exponential: the unit cube scaled by
    sqrt(3 / D) (E|x - y|^2 = 0.5 at every D, as the C3 / C4 datasets).  Dot-exponential: coordinates uniform in [-r, r]
    with r^2 sqrt(D) = 3, so that <x, y> has a standard deviation of 1 at every D.  (The exponent error of one FP16 term
    grows with max |x_d| |y|: Gaussian coordinates at D = 3 put the model of the plain product at 3e-3, over the
    tolerance; bounded ones at 2e-4.)  Signal columns of distinct scales and signs with source-dependent means, so a wrong
    column or source block shows."""
    rng = np.random.RandomState(zlib.crc32(case.name.encode()))
    if case.kernel == "dot-exponential":
        r = (3.0 / case.D ** 0.5) ** 0.5
        y, x = r * (2 * rng.rand(case.M, case.D) - 1), r * (2 * rng.rand(case.N, case.D) - 1)
    else:
        r = (3.0 / max(case.D, 3)) ** 0.5
        y, x = r * rng.rand(case.M, case.D), r * rng.rand(case.N, case.D)
    b = None
    if not case.density:
        scale = np.array([(-1.0) ** e * 2.0 ** (e % 5 - 2) for e in range(case.E)])
        b = scale * (0.5 + rng.rand(case.M, case.E) + np.linspace(0.0, 1.0, case.M)[:, None])
    cast = lambda a: None if a is None else a.astype(np.float32).astype(np.float64)  # noqa: E731
    return cast(x), cast(y), cast(b)


# ---- model of the one-term arithmetic -------------------------------------------------------------------------------


def _f16(a):
    return a.astype(np.float16).astype(np.float64)


def _pow2_into(m, lo_exp):
    """2^p with 2^p m in [2^lo_exp, 2^(lo_exp + 1))."""
    return 2.0 ** (lo_exp - np.floor(np.log2(m)))


def model_product(kernel, x, y, b, *, normalize_rows=False, density_estimation=False):
    """What the one-term kernels compute, in NumPy: the data centred on the source mean (dot-exponential: not centred),
    scaled by one power of two into [2^13, 2^14) and rounded to FP16 once; S = hi.hi exactly (FP32 accumulation of
    products of 11-bit operands is exact enough to ignore here); squared norms in FP32.  E <= 4 (and D > 128): weights and
    sums in FP32 on the CUDA cores.  E > 4 with D <= 128: P (relative to the row maximum) and b (per-column power of two) rounded to one FP16 plane
    each, and the row sum of the rounded weights."""
    if density_estimation:
        b = np.ones((y.shape[0], 1))
    if kernel == "dot-exponential":
        c = np.zeros(x.shape[1])
    else:
        c = y.mean(0)
    u, v = x - c, y - c
    s = _pow2_into(max(np.abs(u).max(), np.abs(v).max()), 13)
    S = (_f16(u * s) @ _f16(v * s).T) / (s * s)
    if kernel == "dot-exponential":
        L = S
    else:
        un = (u * u).sum(1).astype(np.float32).astype(np.float64)
        vn = (v * v).sum(1).astype(np.float32).astype(np.float64)
        d2 = np.maximum(un[:, None] + vn[None, :] - 2 * S, 0.0)
        L = -d2 if kernel == "gaussian" else -np.sqrt(d2)
    ref = L.max(1, keepdims=True)
    P = np.exp(L - ref)
    if b.shape[1] > 4 and x.shape[1] <= 128:   # the P.B kernels (D > 128: the E <= 4 kernels, pass by pass)
        q = _pow2_into(np.abs(b).max(0), 13)
        Ph = _f16(P)
        O, den = (Ph @ _f16(b * q)) / q, Ph.sum(1, keepdims=True)
    else:
        P32 = P.astype(np.float32).astype(np.float64)
        O, den = P32 @ b, P32.sum(1, keepdims=True)
    return O / den if normalize_rows else O * np.exp(ref)


def errors(got, want):
    """(relative L2 over the whole result, relative L2 of each row)."""
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    row_err = np.linalg.norm(got - want, axis=1) / np.linalg.norm(want, axis=1)
    return err, row_err
