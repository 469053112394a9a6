"""float64 oracle of causal kernel products -- TEST INFRASTRUCTURE ONLY.

    out[i] = sum_{j <= row_offset + i} k(x_i, y_j) b_j

for every kernel of the library (bruteforce.py:18-22 and the dot-exponential extension), with the query modes of
bruteforce.py:130-153 restricted to the visible sources: normalize_rows divides by the masked row sum (for the
dot-exponential kernel after subtracting the row's largest visible <x_i, y_j>, so softmax attention stays finite),
density sums the masked kernel values, both together fill ones.  The inverse-distance zeroing rule (flat index
(row_offset + i) (M + 1), bruteforce.py:12-14) applies on top of the mask.  Blocked over target rows; pinned to the
literal np.tril(K, row_offset) @ b at small sizes (tests/test_causal_cpu.py).
"""
from __future__ import annotations

import numpy as np


def kernel_matrix(kernel, x, y, row_offset=0, row0=0, n_sources=None):
    """K[i, j] = k(x_i, y_j) in float64 for rows row0 .. row0 + len(x) - 1 of a target set starting at row_offset; y may be
    the first columns of a source set of n_sources points (the inverse-distance zeroing rule depends on it)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    if kernel == "dot-exponential":
        with np.errstate(over="ignore"):
            return np.exp(x @ y.T)
    d2 = np.maximum((x * x).sum(1)[:, None] + (y * y).sum(1)[None, :] - 2.0 * (x @ y.T), 0.0)
    if kernel == "gaussian":
        return np.exp(-d2)
    if kernel == "absolute-exponential":
        return np.exp(-np.sqrt(np.maximum(d2, 0.0)))
    if kernel == "inverse-distance":
        with np.errstate(divide="ignore"):
            k = 1.0 / np.sqrt(np.maximum(d2, 0.0))
        rows = row_offset + row0 + np.arange(x.shape[0])
        zj = rows % ((y.shape[0] if n_sources is None else n_sources) + 1)
        hit = zj < y.shape[0]
        k[np.arange(x.shape[0])[hit], zj[hit]] = 0.0
        return k
    raise ValueError(kernel)


def causal_product(kernel, x, y, b, *, row_offset=0, normalize_rows=False, density_estimation=False, block=64):
    """The causal product in float64 (b ignored under density_estimation)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    N, M = x.shape[0], y.shape[0]
    if normalize_rows and density_estimation:
        return np.ones((N, 1))
    b = np.ones((M, 1)) if density_estimation else np.asarray(b, dtype=np.float64)
    out = np.empty((N, b.shape[1]))
    for r0 in range(0, N, block):
        r1 = min(N, r0 + block)
        jmax = min(M, row_offset + r1)            # sources beyond the block's last row are never seen
        rows = row_offset + np.arange(r0, r1)
        visible = np.arange(jmax)[None, :] <= rows[:, None]
        if kernel == "dot-exponential" and normalize_rows:
            s = x[r0:r1] @ y[:jmax].T
            s = np.where(visible, s, -np.inf)
            k = np.exp(s - s.max(axis=1, keepdims=True))
        else:
            k = np.where(visible, kernel_matrix(kernel, x[r0:r1], y[:jmax], row_offset, r0, M), 0.0)
        out[r0:r1] = k @ b[:jmax]
        if normalize_rows:
            out[r0:r1] /= k.sum(axis=1, keepdims=True)
    return out


def rel_l2(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-300))


def worst_row(got, want):
    """Largest per-row relative L2 error."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    num = np.linalg.norm(got - want, axis=1)
    den = np.maximum(np.linalg.norm(want, axis=1), 1e-300)
    return float((num / den).max())
