"""float64 oracles of the dot-exponential kernel k(x, y) = exp(<x, y>) -- TEST INFRASTRUCTURE ONLY.

The kernel is not in bruteforce.py (an extension of the plugin), so the reference has no formula or golden vector for
it; this restates one.  Same contract as oracle.bruteforce_oracle.kernel_product without the kernel argument:
    plain product   sum_j exp(<x_i, y_j>) b_j            (inf where exp overflows float64, as the literal formula)
    density         sum_j exp(<x_i, y_j>)
    normalize_rows  softmax(x y^T) b, with the row maximum of <x_i, y_j> subtracted before exp: finite for any row
Two implementations, pinned against each other (tests/test_dot_exponential_cpu.py) and against the literal formula
np.exp(x @ y.T) @ b on small inputs: ``kernel_product`` (NumPy, blocked over target rows) and ``kernel_product_c``
(tests/dot_exponential_ref.c through ctypes, compiled on first use into a temporary directory).
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "dot_exponential_ref.c")


def _prepare(source_points, target_points, source_signal, density_estimation, rows):
    y = np.ascontiguousarray(source_points, dtype=np.float64)
    x = y if target_points is None else np.ascontiguousarray(target_points, dtype=np.float64)
    if rows is not None:
        x = np.ascontiguousarray(x[np.asarray(rows, dtype=np.int64)])
    b = None if density_estimation else np.ascontiguousarray(source_signal, dtype=np.float64)
    return x, y, b


def kernel_product(source_points, target_points, source_signal, *, normalize_rows=False, density_estimation=False,
                   rows=None, block=1024):
    """NumPy float64 oracle (rows: evaluate only these target rows)."""
    x, y, b = _prepare(source_points, target_points, source_signal, density_estimation, rows)
    if normalize_rows and density_estimation:   # bruteforce.py:134-138
        return np.ones((x.shape[0], 1))
    E = 1 if b is None else b.shape[1]
    out = np.empty((x.shape[0], E))
    with np.errstate(over="ignore"):
        for i0 in range(0, x.shape[0], block):
            s = x[i0:i0 + block] @ y.T
            m = s.max(axis=1, keepdims=True) if normalize_rows else 0.0
            k = np.exp(s - m)
            a = k.sum(axis=1, keepdims=True) if b is None else k @ b
            out[i0:i0 + block] = a / k.sum(axis=1, keepdims=True) if normalize_rows else a
    return out


_lib = None


def _load():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        so = os.path.join(tempfile.gettempdir(), f"kmb_dotexp_oracle_{os.getuid()}_{hashlib.sha1(src).hexdigest()[:12]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.run(["cc", "-O2", "-shared", "-fPIC", "-pthread", "-o", tmp, _SRC, "-lm"], check=True)
            os.replace(tmp, so)
        lib = ctypes.CDLL(so)
        lib.kmb_dotexp_oracle_f64.restype = ctypes.c_int
        _lib = lib
    return _lib


def kernel_product_c(source_points, target_points, source_signal, *, normalize_rows=False, density_estimation=False,
                     rows=None):
    """The C float64 oracle (tests/dot_exponential_ref.c), same contract as kernel_product."""
    x, y, b = _prepare(source_points, target_points, source_signal, density_estimation, rows)
    n, (M, D) = x.shape[0], y.shape
    if normalize_rows and density_estimation:
        return np.ones((n, 1))
    E = 1 if b is None else b.shape[1]
    out = np.empty((n, E))
    p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    rc = _load().kmb_dotexp_oracle_f64(p(x), p(y), p(b), p(out), ctypes.c_int64(n), ctypes.c_int64(M), ctypes.c_int(D),
                                       ctypes.c_int(E), ctypes.c_int(int(normalize_rows)))
    if rc != 0:
        raise ValueError(f"kmb_dotexp_oracle_f64: bad arguments (rc={rc})")
    return out
