"""B200 plugins for kernel-matrix-benchmarks: drop-ins for the brute-force path.

``B200Product`` stands where ``BruteForceProductBLAS`` stands
(/root/reference/kernel_matrix_benchmarks/algorithms/bruteforce.py:61-153) and
``B200Solver`` where ``BruteForceSolverLAPACK`` stands (:156-207): same
constructor keywords, same prepare_data / fit / prepare_query / query /
get_result sequence driven by ``runner.run`` (runner.py:70-176), same error
behaviour (``NotImplementedError`` for an unknown kernel, :82-85).  Registered in
``algos.yaml`` with ``hardware: GPU``.

What differs is *where* the work happens: the reference builds the dense kernel
matrix in ``fit()`` and multiplies in ``query()``; here the matrix is never
built, ``fit()`` only sizes device buffers and all arithmetic happens inside
``query()`` in hand-written sm_100a kernels (libkmb_b200.so).  Compare the two
on total time (build + query), the harness's default x-axis.

The timer around fit()/query() is host wall-clock (runner.py:97-99, 138-140), so
both end with a device synchronise.  There is no CPU fallback: constructing
either class without the CUDA library or a GPU raises.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib
from .. import multigpu as _multigpu
from .. import product as _product
from ..product import Workspace, device_info, kernel_product, kernel_product_sym_part, last_launch_count
from ..solver import (CudaShardOps, CudaSymmetricOps, LocalComm, NystromPreconditioner, ReplicatedComm, TorchDistComm, cg_solve,
                      landmark_indices, pcg_solve, shard_bounds)
from .base import BaseProduct, BaseSolver


def _check_precision(precision, who, allowed=(np.float32,)):
    """The reference accepts a numpy dtype or its name (algos.yaml:156-162 passes strings)."""
    dt = np.dtype(precision)
    if dt not in [np.dtype(a) for a in allowed]:
        names = ", ".join(np.dtype(a).name for a in allowed)
        raise NotImplementedError(f"{who} supports precision in {{{names}}} (got precision={precision}).")
    return dt


def _cast_threads():
    """Host threads of one cast (numpy releases the GIL inside copyto): 4, fewer when several ranks share the host's cores
    (torchrun's LOCAL_WORLD_SIZE) -- eight ranks with four threads each on sixteen cores only get in each other's way."""
    import os

    local = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1))
    return max(1, min(4, (os.cpu_count() or 4) // local))


_CAST_THREADS = _cast_threads()
_CAST_MIN_BYTES = 2 << 20    # below this a single pass is faster than handing out slices (C2: the 4 MB result and signal are above it)
_cast_pool = None


def _cast_into(dst, src):
    """dst[...] = src (float64 -> working precision) in one pass over the data, large arrays on a few host threads: the
    cast is memory-bound and single-threaded in NumPy (4-5 ms for the 24 MB of C2's points -- as long as 3 % of the product)."""
    global _cast_pool
    if src.nbytes < _CAST_MIN_BYTES or src.shape[0] < _CAST_THREADS:
        np.copyto(dst, src, casting="unsafe")
        return
    if _cast_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _cast_pool = ThreadPoolExecutor(max_workers=_CAST_THREADS)
    step = -(-src.shape[0] // _CAST_THREADS)
    list(_cast_pool.map(lambda lo: np.copyto(dst[lo:lo + step], src[lo:lo + step], casting="unsafe"), range(0, src.shape[0], step)))


def _to_device(array, device, precision=np.float32, comm=None):
    """float64 host array (owned by the runner, never mutated) -> device tensor in the working precision.

    ``comm`` with world > 1 (one process per GPU, every rank handed the same array): each rank casts and copies only its
    1 / world slice of the rows and the slices are all-gathered on the devices (NVLink) -- the host cast and the PCIe copy of
    the replicated array do not grow with the number of ranks sharing the host.

    float32: cast as bruteforce.py:100-106 casts.  float64: kept.  float16: the inputs are rounded to half
    precision exactly as the reference's ``astype(float16)`` rounds them, then widened to float32 -- the
    arithmetic itself runs in FP32 (the reference's float16 run also accumulates in half precision, which
    costs it another ~1e-3; this variant only carries the input rounding)."""
    dt = np.dtype(precision)
    a = np.asarray(array)
    if dt == np.float16:
        a = a.astype(np.float16).astype(np.float32)
    work = np.float64 if dt == np.float64 else np.float32
    if a.ndim == 1:
        a = a[:, None]
    world = comm.world if comm is not None else 1
    if world > 1 and a.nbytes >= _CAST_MIN_BYTES and dt != np.float16:
        lo, hi, per = shard_bounds(a.shape[0], comm.rank, world)
        stage = _staging((per,) + a.shape[1:], work)
        _cast_into(stage.numpy()[: hi - lo], a[lo:hi])
        mine = stage[: hi - lo].to(device, non_blocking=True)
        with torch.cuda.device(device):
            out = comm.all_gather(mine, a.shape[0]).clone()   # the communicator's gather buffer is reused by the next call
        torch.cuda.current_stream(device).synchronize()
        return out
    # cast straight into a cached pinned staging buffer (one pass over the data, no per-call pinning)
    stage = _staging(a.shape, work)
    _cast_into(stage.numpy(), a)
    out = stage.to(device, non_blocking=True)
    torch.cuda.current_stream(device).synchronize()   # the staging buffer is reused by the next call
    return out


def _to_host_f64(t):
    """Device result -> fresh float64 host array (base.py:116 / :167): one copy into pinned memory, one widening pass."""
    if t.dtype not in (torch.float32, torch.float64) or t.numel() == 0:
        return np.ascontiguousarray(t.cpu().numpy(), dtype=np.float64)
    stage = _staging(tuple(t.shape), np.float64 if t.dtype == torch.float64 else np.float32)
    stage.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    out = np.empty(tuple(t.shape), dtype=np.float64)
    _cast_into(out, stage.numpy())
    return out


_STAGING = {}


def _staging(shape, dtype):
    key = (tuple(shape), np.dtype(dtype).str)
    buf = _STAGING.get(key)
    if buf is None:
        if len(_STAGING) > 16:
            _STAGING.clear()
        buf = torch.empty(tuple(shape), dtype=torch.float64 if np.dtype(dtype) == np.float64 else torch.float32).pin_memory()
        _STAGING[key] = buf
    return buf


class _GpuTimer:
    def __init__(self):
        self.start, self.stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def __enter__(self):
        self.start.record()
        return self

    def __exit__(self, *exc):
        self.stop.record()

    def ms(self):
        self.stop.synchronize()
        return self.start.elapsed_time(self.stop)


class B200Product(BaseProduct):
    """On-the-fly kernel product / density / attention on one B200."""

    def __init__(self, *, kernel, dimension, normalize_rows=False, precision="float32", path="auto", device=0,
                 distributed=False, n_gpus=1, causal=False):
        """``causal=True``: row i of the result sums the sources j <= i only (autoregressive attention; an extension, not in
        the reference).  It runs on the FP16 tensor path ("auto" or "tensor_f16") and in float64; the other paths raise
        NotImplementedError here.  With several GPUs each device gets an equal share of the triangle, not of the rows.

        ``n_gpus=G`` (constructor argument, or ``query-args: [{n_gpus: G}]`` through ``set_query_arguments``): this ONE
        process drives devices ``device .. device+G-1`` -- the harness calls the plugin from a single thread
        (runner.py:118-148), so this is how ``run.py --local --hardware GPU`` sweeps 1/2/4/8 GPUs.  With ``same_points``
        Gaussian data the devices split the symmetric unit list and the first device adds the partial vectors through
        NVLink peer memory; otherwise they split the target rows and store them straight into the first device's result
        (multigpu.DeviceGroup; no NCCL).

        ``distributed=True``: one process per GPU under torch.distributed (NCCL).  Every rank is handed
        the same arrays; with ``same_points`` data the ranks split the symmetric unit list and all-reduce
        the result, otherwise they split the target rows and ``get_result`` gathers them.  Every rank
        returns the whole (N, E) result."""
        super().__init__(kernel=kernel, dimension=dimension, normalize_rows=normalize_rows, precision=precision)
        if kernel not in _lib.KERNEL_IDS:
            raise NotImplementedError(f"B200Product doesn't support kernel {kernel}.")
        if path not in _lib.PATH_IDS:
            raise ValueError(f"unknown path {path!r} (expected one of {sorted(_lib.PATH_IDS)})")
        if path == "tensor_f16x1" and kernel == "inverse-distance":   # 1/|x - y| amplifies the error of a one-term S
            raise NotImplementedError("B200Product doesn't support kernel inverse-distance on path tensor_f16x1.")
        self.causal = bool(causal)
        if self.causal and path not in ("auto", "tensor", "tensor_f16"):
            raise NotImplementedError(f"B200Product doesn't support causal products on path {path}.")
        self.dtype = _check_precision(precision, "B200Product", (np.float32, np.float64, np.float16))
        _lib.load()  # fail here, loudly, if the CUDA library is absent
        if not torch.cuda.is_available():
            raise RuntimeError("B200Product needs a CUDA device; there is no CPU fallback.")
        self.path = path
        self.device = torch.device("cuda", int(device))
        self.comm = TorchDistComm() if distributed else LocalComm()
        if distributed and int(n_gpus) > 1:
            raise ValueError("distributed=True (one process per GPU) and n_gpus > 1 (one process, several GPUs) exclude each other")
        self.n_gpus = _multigpu.clamp_gpus(n_gpus, self.device.index)
        self._group = None
        self._set_name()
        self.path_used = None
        self.workspace = Workspace()
        self.query_ms = None
        self.launches = 0
        self.res = None

    def _set_name(self):
        gpus = self.comm.world if self.comm.world > 1 else self.n_gpus
        extra = (", causal" if self.causal else "") + (f", gpus={gpus}" if gpus > 1 else "")
        self.name = f"B200Product({self.dtype.name}, path={self.path}{extra})"

    def set_query_arguments(self, n_gpus=None, **kwargs):
        """``query-args`` of algos.yaml (runner.py:123, after fit() and before prepare_query()): ``n_gpus`` re-targets the
        same fitted object at another number of GPUs; the replicas are made in prepare_query() (untimed, like every
        host->device copy), points-only prepasses of the tensor path inside the first query with that GPU count."""
        if n_gpus is not None:
            if self.comm.world > 1:
                raise ValueError("n_gpus cannot be combined with distributed=True")
            self.n_gpus = _multigpu.clamp_gpus(n_gpus, self.device.index)
            self._set_name()   # the name labels the stored result (runner.py:155)

    def _multi(self):
        return self.n_gpus > 1 and self.dtype != np.float64

    def _setup_group(self):
        """Replicas of the points on the group's devices (peer copies from the first device), row blocks of the targets."""
        g = self._group
        if g is None or g.n != self.n_gpus:
            g = _multigpu.DeviceGroup(self.device.index, self.n_gpus)
            self._ys = g.replicate(self.source_points)
            if self.same_points:
                self._bounds = [self._row_bounds(self.source_points.shape[0], i, g.n) for i in range(g.n)]
                self._xs = [self._ys[i][lo:hi] for i, (lo, hi) in enumerate(self._bounds)]
            else:
                self._xs, self._bounds = g.shard_rows(self.target_points, bounds=self._row_bounds)
            g.synchronize()
            self._group = g
        return g

    def _row_bounds(self, n, rank, world):
        """Row block of a device or rank: equal rows, or under causal equal shares of the triangle (one helper for the
        n_gpus rows mode and distributed=True)."""
        if self.causal:
            return _product.causal_row_bounds(n, rank, world)
        return shard_bounds(n, rank, world)[:2]

    def prepare_data(self, *, source_points, target_points, same_points=False, density_estimation=False):
        """Untimed host->device copy (base.py:64-67), cast to float32 as bruteforce.py:100-106 casts."""
        self._group = None
        self.source_points = _to_device(source_points, self.device, self.dtype, self.comm)
        self.same_points = bool(same_points)
        self.target_points = self.source_points if self.same_points else _to_device(target_points, self.device, self.dtype, self.comm)
        self.density_estimation = bool(density_estimation)
        torch.cuda.synchronize(self.device)

    def fit(self):
        """Timed (the harness books it as build time).  K is never materialised (bruteforce.py:113-120 builds it here);
        what depends on the points alone -- the tensor path's prepass: centre, scale, FP16 operand planes, squared
        norms -- is done here and kept in the workspace (product.prepare_points), so that query() is the product only."""
        N = self.target_points.shape[0]
        self._out_rows = N
        self._prepared = None
        if self._multi():   # n_gpus given to the constructor: replicate and prepare every device's row block here
            g = self._setup_group()
            g.prepare_rows(self._xs, self._ys, kernel=self.kernel, path=self.path, causal=self.causal)
            g.synchronize()
        elif self.dtype != np.float64:
            with torch.cuda.device(self.device):
                self._prepared = _product.prepare_points(self._my_rows(), self.source_points, kernel=self.kernel,
                                                         path=self.path, workspace=self.workspace, causal=self.causal)
        torch.cuda.synchronize(self.device)

    def _my_rows(self):
        """The target rows this process evaluates (all of them, or its block under distributed=True)."""
        if self.comm.world == 1:
            return self.target_points
        lo, hi = self._row_bounds(self.target_points.shape[0], self.comm.rank, self.comm.world)
        return self.target_points[lo:hi]

    def _prepared_token(self, E):
        """The prepass of fit() is still valid if the workspace did not have to grow for this signal width; otherwise
        grow it first and prepare once more (paid by the first query with a wider signal only)."""
        if getattr(self, "_prepared", None) is None:
            return None
        x = self._my_rows()
        need = _product.workspace_bytes(x.shape[0], self.source_points.shape[0], x.shape[1], E, kernel=self.kernel,
                                        normalize_rows=bool(self.normalize_rows), density_estimation=self.density_estimation,
                                        path=self.path, causal=self.causal)
        if self.workspace.get(need, x.device) is not self._prepared:
            self._prepared = _product.prepare_points(x, self.source_points, kernel=self.kernel, path=self.path,
                                                     workspace=self.workspace, min_bytes=need, causal=self.causal)
        return self._prepared

    def prepare_query(self, *, source_signal):
        """Untimed host->device copy of the signal (bruteforce.py:122-128)."""
        self.source_signal = None if self.density_estimation else _to_device(source_signal, self.device, self.dtype, self.comm)
        if self._multi():
            g = self._setup_group()
            self._bs = None if self.density_estimation else g.replicate(self.source_signal)
            g.synchronize()
        torch.cuda.synchronize(self.device)

    def _query_multi(self):
        """n_gpus > 1 in this process (multigpu.DeviceGroup): symmetric unit list or target rows split over the devices;
        the result is complete on the first device when its stream gets there."""
        g = self._group
        y0 = self.source_points
        E = 1 if self.density_estimation else self.source_signal.shape[1]
        N = self.target_points.shape[0]
        self.res_device = torch.empty((N, E), dtype=torch.float32, device=self.device)
        if (self.same_points and not self.causal
                and g.symmetric_applies(y0, self.kernel, bool(self.normalize_rows), self.density_estimation, E, self.path)):
            g.product_sym(self._ys, self._bs, self.res_device, kernel=self.kernel)
            self.path_used = "direct_sym"
        else:
            if g.prepared is None:   # n_gpus arrived as a query argument: the first query with this GPU count prepares
                g.prepare_rows(self._xs, self._ys, kernel=self.kernel, path=self.path, causal=self.causal)
            g.product_rows(self._xs, self._bounds, self._ys, self._bs, self.res_device, kernel=self.kernel,
                           normalize_rows=bool(self.normalize_rows), density_estimation=self.density_estimation, path=self.path,
                           prepared=g.prepared, causal=self.causal)
            self.path_used = _product.resolved_path(y0.shape[1], E, self.kernel, self.path, self.causal)
        self.launches = g.launches

    def query(self):
        """Timed: the whole product, ending with a device synchronise."""
        with torch.cuda.device(self.device):
            with _GpuTimer() as t:
                if self.dtype == np.float64:
                    lo, hi = self._row_bounds(self.target_points.shape[0], self.comm.rank, self.comm.world)
                    mine = _product.kernel_product_f64(
                        self.target_points[lo:hi], self.source_points, self.source_signal, kernel=self.kernel,
                        normalize_rows=bool(self.normalize_rows), density_estimation=self.density_estimation, row_offset=lo,
                        causal=self.causal)
                    self.launches = last_launch_count()
                    self.path_used = "direct_f64"
                    self.res_device = mine if self.comm.world == 1 else self._gather_rows(mine)
                elif self.comm.world > 1:
                    self._query_distributed()
                elif self._multi():
                    self._query_multi()
                else:
                    E = 1 if self.density_estimation else self.source_signal.shape[1]
                    self.res_device = kernel_product(
                        self.target_points,
                        self.source_points,
                        self.source_signal,
                        kernel=self.kernel,
                        normalize_rows=bool(self.normalize_rows),
                        density_estimation=self.density_estimation,
                        path=self.path,
                        workspace=self.workspace,
                        prepared=self._prepared_token(E),
                        causal=self.causal,
                    )
                    self.path_used = _product.last_path
                    self.launches = last_launch_count()
            torch.cuda.synchronize(self.device)
        self.query_ms = t.ms()

    def _query_distributed(self):
        """world > 1.  same_points + Gaussian + D <= 3: this rank's range of the symmetric unit list, then
        one all-reduce of N floats.  Otherwise: this rank's block of target rows, gathered afterwards."""
        rank, world = self.comm.rank, self.comm.world
        y, b = self.source_points, self.source_signal
        E = 1 if self.density_estimation else b.shape[1]
        sym = (self.path == "auto" and self.same_points and y.shape[0] >= _product.SYM_MIN_POINTS and
               _product.symmetric_applies(y, y, self.kernel, bool(self.normalize_rows), self.density_estimation, E, self.causal))
        if sym:
            self.res_device = kernel_product_sym_part(y, b, rank, world, kernel=self.kernel, workspace=self.workspace)
            self.launches = last_launch_count()
            self.comm.all_reduce(self.res_device)
            self.path_used = "direct_sym"
            return
        lo, hi = self._row_bounds(self.target_points.shape[0], rank, world)
        mine = kernel_product(self.target_points[lo:hi], y, b, kernel=self.kernel, normalize_rows=bool(self.normalize_rows),
                              density_estimation=self.density_estimation, path=self.path, row_offset=lo,
                              workspace=self.workspace, prepared=self._prepared_token(E), causal=self.causal)
        self.launches = last_launch_count()
        self.path_used = _product.last_path
        self.res_device = self._gather_rows(mine)

    def _gather_rows(self, mine):
        """All ranks' row blocks (self._row_bounds) in row order on every rank.  The equal blocks of the non-causal split
        are what comm.all_gather expects; the causal blocks are padded to the largest and cut back out."""
        n, world = self.target_points.shape[0], self.comm.world
        if not self.causal:
            return self.comm.all_gather(mine, n)
        bounds = [self._row_bounds(n, r, world) for r in range(world)]
        per = max(hi - lo for lo, hi in bounds)
        full = self.comm.all_gather(mine, per * world)
        return torch.cat([full[r * per: r * per + (hi - lo)] for r, (lo, hi) in enumerate(bounds)])

    def get_result(self):
        """Untimed device->host copy; float64 contiguous as base.py:116."""
        self.res = _to_host_f64(self.res_device.contiguous())
        return self.res

    def get_additional(self):
        """Extra attrs stored with the result (runner.py:162 -> results.py:116-117)."""
        if self.query_ms is None:
            return {}
        pairs = float(self.target_points.shape[0]) * float(self.source_points.shape[0])
        return {
            "gpu_query_ms": float(self.query_ms),
            "gpairs_per_s": pairs / (self.query_ms * 1e-3) / 1e9,
            "gpu_launches": int(self.launches),
            "path": self.path,
            "path_used": str(self.path_used),
            "form": self._form(),
            "n_gpus": int(self.comm.world if self.comm.world > 1 else (self.n_gpus if self._multi() else 1)),
        }

    def _form(self):
        if self.source_points.shape[1] > 16 or (self.normalize_rows and self.density_estimation) or self.dtype == np.float64:
            return "n/a"
        E = 1 if self.density_estimation else self.source_signal.shape[1]
        if self.path_used != "direct_sym" and _product.resolved_path(self.source_points.shape[1], E, self.kernel, self.path).startswith("tensor"):
            return "n/a"   # wide signal: the tensor-core kernel ran (no direct-path statistics in the workspace)
        from ..product import direct_stats

        return direct_stats(self._group.workspaces[0] if self._multi() else self.workspace)["form"]

    def get_memory_usage(self):
        """Host RSS as the reference reports, plus device bytes in kB."""
        return super().get_memory_usage() + torch.cuda.memory_allocated(self.device) / 1024

    def done(self):
        for k in ("source_points", "target_points", "source_signal", "res_device", "res", "_prepared", "_group", "_ys", "_xs", "_bs"):
            self.__dict__.pop(k, None)
        self._group = None
        self.workspace = Workspace()

    def __del__(self):  # runner.py keeps only the fastest-fit instance; the others are just dropped
        try:
            self.done()
        except Exception:
            pass


class B200Solver(BaseSolver):
    """Kernel solve (K + lam I) b = a by conjugate gradients on the on-the-fly product.

    ``lam = 0`` is the reference's system K b = a (bruteforce.py:205-207); for the
    Gaussian kernel that matrix is singular to working precision (cond ~ 1e20), so
    the BASELINE solve config uses lam = 1 and scores the residual.
    """

    def __init__(self, *, kernel, dimension, normalize_rows=False, precision="float32", lam=0.0, rtol=1e-6,
                 max_iter=500, path="auto", device=0, distributed=False, preconditioner="auto", precond_rank=1024, n_gpus=1):
        """``n_gpus`` / ``distributed`` as for B200Product.  With ``n_gpus=G`` all CG vectors and the preconditioner live on
        the first device; only the matvec (10^12 pairs at config C5) is spread over the G devices of this process
        (multigpu.MultiDeviceSymmetricOps / MultiDeviceRowOps)."""
        super().__init__(kernel=kernel, dimension=dimension, normalize_rows=normalize_rows, precision=precision)
        if kernel not in _lib.KERNEL_IDS or kernel == "dot-exponential":   # exp(<x, y>): product / attention only
            raise NotImplementedError(f"B200Solver doesn't support kernel {kernel}.")
        if path == "tensor_f16x1":
            raise ValueError("B200Solver doesn't support path tensor_f16x1: its matvec error (~3e-4 relative) cannot reach "
                             "the solver's tolerances (rtol 1e-6); use path 'auto' or 'tensor_f16'.")
        if preconditioner not in ("auto", "nystrom", "none"):
            raise ValueError(f"unknown preconditioner {preconditioner!r} (expected 'auto', 'nystrom' or 'none')")
        self.preconditioner, self.precond_rank = preconditioner, int(precond_rank)
        self.dtype = _check_precision(precision, "B200Solver", (np.float32, np.float64, np.float16))
        _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("B200Solver needs a CUDA device; there is no CPU fallback.")
        self.lam, self.rtol, self.max_iter, self.path = float(lam), float(rtol), int(max_iter), path
        self.comm = TorchDistComm() if distributed else LocalComm()
        self.device = torch.device("cuda", int(device))
        if distributed and int(n_gpus) > 1:
            raise ValueError("distributed=True (one process per GPU) and n_gpus > 1 (one process, several GPUs) exclude each other")
        self.n_gpus = _multigpu.clamp_gpus(n_gpus, self.device.index)
        self._group = None
        self.precision_name = np.dtype(precision).name
        self._set_name()
        self.info = None
        self.res = None

    PRECOND_MIN_POINTS = 65536

    def _set_name(self):
        pc = f", nystrom{self.precond_rank}" if self.preconditioner == "nystrom" else ", plain" if self.preconditioner == "none" else ""
        gpus = self.comm.world if self.comm.world > 1 else self.n_gpus
        pc += f", gpus={gpus}" if gpus > 1 else ""
        self.name = f"B200Solver({self.precision_name}, lam={self.lam:g}, rtol={self.rtol:g}{pc})"

    def set_query_arguments(self, **kwargs):
        """``query-args`` of algos.yaml (runner.py:123): rtol / max_iter / lam can be swept without refitting."""
        for k in ("rtol", "lam"):
            if k in kwargs:
                setattr(self, k, float(kwargs[k]))
        if "max_iter" in kwargs:
            self.max_iter = int(kwargs["max_iter"])
        if kwargs.get("n_gpus") is not None:
            if self.comm.world > 1:
                raise ValueError("n_gpus cannot be combined with distributed=True")
            n = _multigpu.clamp_gpus(kwargs["n_gpus"], self.device.index)
            if n != self.n_gpus:
                self.n_gpus = n
                self._ops = {}   # matvec objects are per GPU count; the preconditioner (first device) is kept
        self._set_name()  # the name labels the result (runner.py:155)

    _warmed = set()

    def _warm_libraries(self):
        """Once per process and device: a small preconditioner with the real landmark count, so that the first timed fit()
        does not pay the lazy loading of the cuSOLVER / cuBLAS kernels it uses (1.1 s against 0.2 s, measured) -- library
        start-up, which the reference's timers do not see either (its NumPy / LAPACK are loaded at import)."""
        key = (self.device.index, self.precond_rank)
        if key in B200Solver._warmed or not self._use_precond():
            return
        B200Solver._warmed.add(key)
        n = min(self.source_points.shape[0], 4 * self.precond_rank)
        pts = self.source_points[:n]
        idx = landmark_indices(n, min(self.precond_rank, n // 2)).to(self.device)
        with torch.cuda.device(self.device):
            pc = NystromPreconditioner(pts, pts[idx], self.kernel, max(self.lam, 1.0), LocalComm(), dtype=self.source_points.dtype)
            pc.apply(torch.ones((n, 1), dtype=self.source_points.dtype, device=self.device))
            torch.cuda.synchronize(self.device)

    def prepare_data(self, *, source_points):
        """float32: the production path.  float64: double-precision matvec (kmb_product_f64) and vector kernels.  float16: the
        inputs are rounded to half precision as the reference's astype does (bruteforce.py:186-203), arithmetic in FP32."""
        self.source_points = _to_device(source_points, self.device, self.dtype, self.comm)
        if self.comm.world > 1:
            self.comm.warm(self.device)
        self._warm_libraries()
        torch.cuda.synchronize(self.device)

    def _multi(self):
        return self.n_gpus > 1 and self.dtype != np.float64

    def fit(self):
        """Timed (the harness books it as build time).  The system itself is never factorised -- it is applied
        through the on-the-fly product -- but the Nystrom preconditioner (solver.NystromPreconditioner: m landmark
        columns of K, an m x m eigendecomposition) depends on the points only and is built here."""
        self._ops, self._precond = {}, {}
        with torch.cuda.device(self.device):
            with _GpuTimer() as t:
                if self._use_precond():
                    self._precond_for(self._mode(1))
            torch.cuda.synchronize(self.device)
        self.fit_ms = t.ms()

    def _mode(self, E):
        symmetric = self.path == "auto" and CudaSymmetricOps.applies(self.source_points, self.kernel, E)
        return "symmetric" if symmetric else "rows"

    def _use_precond(self):
        """'auto': from PRECOND_MIN_POINTS points on (below that, building it costs more than the iterations it saves:
        at N = 10^4 plain CG takes 7 ms, the 0.2 s Nystrom build is only repaid from ~10^5 points)."""
        n = self.source_points.shape[0]
        if self.preconditioner == "none" or self.kernel == "inverse-distance" or self.precond_rank <= 0 or n < 64:
            return False
        return self.preconditioner == "nystrom" or n >= self.PRECOND_MIN_POINTS

    def _precond_for(self, key):
        """Symmetric matvec: every rank holds all rows (no collective inside the preconditioner); row-sharded
        matvec: each rank holds its rows of U and the small products are all-reduced."""
        if self._multi():
            key = "symmetric"   # all CG vectors on the first device: the preconditioner holds all rows there
        if key not in self._precond:
            n = self.source_points.shape[0]
            idx = landmark_indices(n, min(self.precond_rank, n // 2)).to(self.device)   # small data sets: half the points
            landmarks = self.source_points[idx]
            # built from this rank's rows (1 / world of the landmark block, the triangular solve and the Gram matrix; one
            # all-reduce of m x m doubles); the symmetric matvec then wants every row of U on every rank: one all-gather
            lo, hi, _ = shard_bounds(n, self.comm.rank, self.comm.world)
            pc = NystromPreconditioner(self.source_points[lo:hi], landmarks, self.kernel, self.lam, self.comm, dtype=self.source_points.dtype)
            self._precond[key] = pc.replicate(n) if key == "symmetric" else pc
        pc = self._precond[key]
        pc.set_shift(self.lam)   # lam may have been changed by set_query_arguments
        return pc

    def _ops_for(self, E):
        """The matvec of the solve always has targets == sources: the symmetric product applies whenever
        the kernel is Gaussian, D <= 3 and there is one right-hand side (every rank then holds all CG
        vectors and the ranks share the unit list); otherwise the rows of the system are sharded."""
        n = self.source_points.shape[0]
        key = self._mode(E)
        symmetric = key == "symmetric"
        if key not in self._ops:
            if self._multi():
                g = self._setup_group()
                self.rows = (0, n)
                self._ops[key] = (_multigpu.MultiDeviceSymmetricOps(g, self._ys, self.kernel) if symmetric
                                  else _multigpu.MultiDeviceRowOps(g, self._ys, self.kernel, path=self.path))
            elif symmetric:
                self._ops[key] = CudaSymmetricOps(self.source_points, self.kernel, self.comm)
            else:
                lo, hi, _ = shard_bounds(n, self.comm.rank, self.comm.world)
                self.rows = (lo, hi)
                self._ops[key] = CudaShardOps(self.source_points, self.kernel, lo, hi, path=self.path)
        self.symmetric, self.ops = symmetric, self._ops[key]
        return self.ops

    def _setup_group(self):
        g = self._group
        if g is None or g.n != self.n_gpus:
            g = self._group = _multigpu.DeviceGroup(self.device.index, self.n_gpus)
            self._ys = g.replicate(self.source_points)
            g.synchronize()
        return g

    def prepare_query(self, *, target_signal):
        self.target_signal = _to_device(target_signal, self.device, self.dtype, self.comm)
        if self._multi():
            self._setup_group()   # replicas of the points on the other devices: an untimed copy like the one above
        torch.cuda.synchronize(self.device)

    def query(self):
        n = self.source_points.shape[0]
        with torch.cuda.device(self.device):
            with _GpuTimer() as t:
                self._ops_for(self.target_signal.shape[1])
                pc = self._precond_for("symmetric" if self.symmetric else "rows") if self._use_precond() else None
                self.precond_rank_used = pc.rank if pc is not None else 0
                if self.symmetric or self._multi():  # vectors replicated / on the first device; the exchange is inside ops.matvec
                    comm, rhs = ReplicatedComm(self.comm), self.target_signal
                else:
                    lo, hi = self.rows
                    comm, rhs = self.comm, self.target_signal[lo:hi].contiguous()
                if pc is not None:
                    self.info = pcg_solve(self.ops, comm, rhs, n, pc, lam=self.lam, rtol=self.rtol, max_iter=self.max_iter)
                else:
                    self.info = cg_solve(self.ops, comm, rhs, n, lam=self.lam, rtol=self.rtol, max_iter=self.max_iter)
                self.x_full = self.info.x if (self.symmetric or self._multi()) else self.comm.all_gather(self.info.x, n)
            torch.cuda.synchronize(self.device)
        self.query_ms = t.ms()

    def get_result(self):
        self.res = _to_host_f64(self.x_full.contiguous())
        return self.res

    def get_additional(self):
        if self.info is None:
            return {}
        return {
            "gpu_query_ms": float(self.query_ms),
            "cg_iterations": int(self.info.iterations),
            "cg_rel_residual": float(self.info.rel_residual),
            "cg_converged": bool(self.info.converged),
            "matvec": "symmetric" if self.symmetric else "rows",
            "preconditioner": f"nystrom(rank={self.precond_rank_used})" if self.precond_rank_used else "none",
            "gpu_fit_ms": float(getattr(self, "fit_ms", 0.0)),
            "gpu_launches": int(self.ops.launches),
            "n_gpus": int(self.comm.world if self.comm.world > 1 else (self.n_gpus if self._multi() else 1)),
        }

    def get_memory_usage(self):
        return super().get_memory_usage() + torch.cuda.memory_allocated(self.device) / 1024

    def done(self):
        for k in ("source_points", "target_signal", "ops", "_ops", "_precond", "x_full", "res", "_group", "_ys"):
            self.__dict__.pop(k, None)
        self._group = None

    def __del__(self):
        try:
            self.done()
        except Exception:
            pass
