"""Several GPUs behind ONE plugin object in ONE process.

The reference harness drives a plugin from a single Python thread: ``runner.run`` calls ``query()`` and times it with
``time.time()`` (/root/reference/kernel_matrix_benchmarks/runner.py:118-148; one worker, main.py:299-308).  To sweep
1/2/4/8 GPUs through that unmodified harness (``query-args: [{n_gpus: 1}, {n_gpus: 2}, ...]`` in algos.yaml) the plugin
itself has to drive the devices -- torchrun-style process groups cannot exist inside ``run.py --local``.

``DeviceGroup`` owns the per-device replicas and workspaces; the launches go through the library's multi-device entry
points (``kmb_product_rows_multi_f32`` / ``kmb_product_sym_multi_f32``, include/kmb_b200.h), which fork/join on the
first device's stream and move partial results through NVLink peer memory: no NCCL, no host synchronisation until
the caller synchronises the first device.  PyTorch provides memory and streams only.
"""
from __future__ import annotations

import ctypes
import warnings

import torch

from . import _lib
from .product import SYM_MIN_POINTS, Workspace, _check_f32, prepare_points, symmetric_applies, workspace_bytes
from .solver import CudaShardOps, shard_bounds


def available_gpus():
    return torch.cuda.device_count()


def clamp_gpus(requested, first_device=0):
    """``n_gpus`` as requested by the harness, limited to what this box has (a warning, not an error: runner.run would
    otherwise abort every remaining query-argument group of the definition, runner.py:110-174)."""
    have = max(1, available_gpus() - int(first_device))
    n = max(1, int(requested))
    if n > have:
        warnings.warn(f"n_gpus={n} requested but only {have} CUDA device(s) from cuda:{first_device} on: using {have}")
        n = have
    return n


class DeviceGroup:
    """``n`` consecutive CUDA devices starting at ``first_device``, peer access enabled among them."""

    def __init__(self, first_device, n):
        self.devices = [torch.device("cuda", int(first_device) + i) for i in range(int(n))]
        self.n = len(self.devices)
        ids = (ctypes.c_int * self.n)(*[d.index for d in self.devices])
        if self.n > 1:
            _lib.check(_lib.load().kmb_enable_peer_access(ids, self.n))
        self.workspaces = [Workspace() for _ in self.devices]
        self.parts = [None] * self.n       # symmetric mode: per-device partial N-vectors
        self.prepared = None               # rows mode: per-device tokens of the tensor path's prepass
        self.launches = 0

    def replicate(self, t0):
        """``t0`` (on the first device) -> one tensor per device (peer copies over NVLink; element 0 is ``t0`` itself)."""
        out = [t0]
        for d in self.devices[1:]:
            out.append(t0.to(d, non_blocking=True))
        return out

    def shard_rows(self, x0, bounds=None):
        """Contiguous row blocks of ``x0`` (first device), block i copied to device i.  Returns (blocks, bounds).
        ``bounds(n, i, n_devices) -> (lo, hi)``: the split (default: equal blocks, solver.shard_bounds)."""
        n = x0.shape[0]
        split = bounds if bounds is not None else (lambda n_, i_, g_: shard_bounds(n_, i_, g_)[:2])
        blocks, bounds = [], []
        for i, d in enumerate(self.devices):
            lo, hi = split(n, i, self.n)
            blocks.append(x0[lo:hi] if i == 0 else x0[lo:hi].to(d, non_blocking=True).contiguous())
            bounds.append((lo, hi))
        return blocks, bounds

    def synchronize(self):
        for d in self.devices:
            torch.cuda.synchronize(d)

    def _stream(self, i):
        return torch.cuda.current_stream(self.devices[i]).cuda_stream

    # ------------------------------------------------------------------------------------------------ rows mode

    def prepare_rows(self, xs, ys, *, kernel, path, causal=False):
        """Per-device prepass of the tensor path (kmb_product_prepare_f32) for each device's row block; returns the
        tokens ``product_rows`` wants (None entries where nothing was prepared)."""
        tokens = []
        for i, d in enumerate(self.devices):
            with torch.cuda.device(d):
                tokens.append(prepare_points(xs[i], ys[i], kernel=kernel, path=path, workspace=self.workspaces[i], causal=causal)
                              if xs[i].shape[0] else None)
        self.prepared = tokens
        return tokens

    def product_rows(self, xs, bounds, ys, bs, out0, *, kernel, normalize_rows=False, density_estimation=False, path="auto",
                     prepared=None, causal=False):
        """Device i computes rows ``bounds[i]`` of the product and stores them straight into ``out0`` (N, E) on the
        first device through peer memory.  ``bs``: the signal per device (a list), or one tensor on the first device that
        the other devices read over NVLink.  Asynchronous; ordered on the first device's current stream."""
        lib = _lib.load()
        M, D = ys[0].shape
        flags = ((_lib.FLAG_NORMALIZE_ROWS if normalize_rows else 0) | (_lib.FLAG_DENSITY if density_estimation else 0)
                 | (_lib.FLAG_CAUSAL if causal else 0))
        if density_estimation:
            E, bs = 1, [None] * self.n
        else:
            if not isinstance(bs, (list, tuple)):
                bs = [bs] * self.n
            E = bs[0].shape[1]
        _check_f32("out", out0, E)
        shards = (_lib.DeviceShard * self.n)()
        for i, d in enumerate(self.devices):
            lo, hi = bounds[i]
            need = workspace_bytes(max(hi - lo, 1), M, D, E, kernel=kernel, normalize_rows=normalize_rows,
                                   density_estimation=density_estimation, path=path, causal=causal)
            ws = self.workspaces[i].get(need, d)
            if prepared is not None and prepared[i] is not None and prepared[i] is not ws:
                # the workspace had to grow for a wider signal: prepare once more, inside this (timed) query
                with torch.cuda.device(d):
                    prepared[i] = prepare_points(xs[i], ys[i], kernel=kernel, path=path, workspace=self.workspaces[i], min_bytes=need,
                                                 causal=causal)
                ws = self.workspaces[i].get(need, d)
            sh = shards[i]
            sh.device = d.index
            sh.flags = _lib.FLAG_PREPARED if (prepared is not None and prepared[i] is not None and prepared[i] is ws) else 0
            sh.x = xs[i].data_ptr() if hi > lo else None
            sh.y = ys[i].data_ptr()
            sh.b = None if density_estimation else bs[i].data_ptr()
            sh.out = out0.data_ptr() + 4 * E * lo if hi > lo else None
            sh.n_targets, sh.row_offset = hi - lo, lo
            sh.workspace, sh.workspace_bytes = ws.data_ptr(), ws.numel()
            sh.stream = self._stream(i)
        _lib.check(lib.kmb_product_rows_multi_f32(shards, self.n, M, D, E, _lib.KERNEL_IDS[kernel], flags, _lib.PATH_IDS[path]))
        self.launches = int(lib.kmb_last_launch_count())
        return out0

    # ------------------------------------------------------------------------------------------- symmetric mode

    def symmetric_applies(self, y0, kernel, normalize_rows, density_estimation, E, path):
        return (path == "auto" and y0.shape[0] >= SYM_MIN_POINTS
                and symmetric_applies(y0, y0, kernel, normalize_rows, density_estimation, E))

    def product_sym(self, ys, bs, out0, kernel="gaussian"):
        """Product with targets == sources: device i evaluates range i of the triangular unit list, the first
        device adds the partial vectors (peer reads) into ``out0`` (n, 1).  ``bs`` as in product_rows (None: density)."""
        lib = _lib.load()
        n, D = ys[0].shape
        if bs is not None and not isinstance(bs, (list, tuple)):
            bs = [bs] * self.n
        _check_f32("out", out0, 1)
        shards = (_lib.DeviceShard * self.n)()
        for i, d in enumerate(self.devices):
            need = ctypes.c_size_t(0)
            _lib.check(lib.kmb_product_sym_workspace_bytes(n, D, i, self.n, ctypes.byref(need)))
            ws = self.workspaces[i].get(need.value, d)
            if self.n > 1 and (self.parts[i] is None or self.parts[i].shape[0] != n):
                self.parts[i] = torch.empty((n, 1), dtype=torch.float32, device=d)
            sh = shards[i]
            sh.device = d.index
            sh.y = ys[i].data_ptr()
            sh.b = None if bs is None else bs[i].data_ptr()
            sh.out = self.parts[i].data_ptr() if self.n > 1 else out0.data_ptr()
            sh.workspace, sh.workspace_bytes = ws.data_ptr(), ws.numel()
            sh.stream = self._stream(i)
        _lib.check(lib.kmb_product_sym_multi_f32(shards, self.n, ctypes.c_void_p(out0.data_ptr()), n, D, _lib.KERNEL_IDS[kernel]))
        self.launches = int(lib.kmb_last_launch_count())
        return out0


# ---------------------------------------------------------------------------------------------------------
# CG matvecs on a device group: all CG vectors live on the first device (N floats each: their updates cost
# microseconds); only the matvec -- 10^12 pairs -- is spread over the GPUs.  The search direction p is read by the
# other devices straight from the first device's memory (one pass of the packing kernel, 4 MB over NVLink), the
# result comes back through peer memory as in the plugin's product.  Use with solver.LocalComm.
# ---------------------------------------------------------------------------------------------------------


class MultiDeviceSymmetricOps(CudaShardOps):
    """Symmetric matvec (kprod_sym) split over the group's devices: one peer-memory reduction of N floats per matvec."""

    def __init__(self, group, ys, kernel):
        super().__init__(ys[0], kernel, 0, ys[0].shape[0])
        self.group, self.ys = group, ys

    def matvec(self, p_full):
        if p_full.shape[1] != 1:
            raise NotImplementedError("the symmetric matvec takes one right-hand side")
        self._ap(1)
        self.group.product_sym(self.ys, p_full, self.Ap, kernel=self.kernel)
        self.launches += self.group.launches
        return self.Ap


class MultiDeviceRowOps(CudaShardOps):
    """Row-sharded matvec: device i computes its block of rows of K p and stores it into Ap on the first device."""

    def __init__(self, group, ys, kernel, path="auto"):
        n = ys[0].shape[0]
        super().__init__(ys[0], kernel, 0, n, path=path)
        self.group, self.ys = group, ys
        self.bounds = [shard_bounds(n, i, group.n)[:2] for i in range(group.n)]
        self.xs = [ys[i][lo:hi] for i, (lo, hi) in enumerate(self.bounds)]
        self.prepared = group.prepare_rows(self.xs, ys, kernel=kernel, path=path)

    def matvec(self, p_full):
        self._ap(p_full.shape[1])
        self.group.product_rows(self.xs, self.bounds, self.ys, p_full, self.Ap, kernel=self.kernel, path=self.path,
                                prepared=self.prepared)
        self.launches += self.group.launches
        return self.Ap
