"""Device-level entry points: torch tensors in, torch tensors out, libkmb_b200 kernels inside.

PyTorch only provides device memory and streams here; every FLOP of the hot
path runs in the hand-written sm_100a kernels behind the C ABI.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _flags(normalize_rows=False, density_estimation=False, causal=False):
    return ((_lib.FLAG_NORMALIZE_ROWS if normalize_rows else 0) | (_lib.FLAG_DENSITY if density_estimation else 0)
            | (_lib.FLAG_CAUSAL if causal else 0))


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check_f32(name, t, cols=None):
    if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.dim() == 2):
        raise ValueError(f"{name} must be a contiguous 2-D float32 CUDA tensor")
    if cols is not None and t.shape[1] != cols:
        raise ValueError(f"{name} has {t.shape[1]} columns, expected {cols}")


class Workspace:
    """A grow-only device buffer handed to the C ABI (the library never allocates)."""

    def __init__(self):
        self.buf = None

    def get(self, nbytes, device):
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        return self.buf


_default_ws = {}

# below this many points the symmetric kernel's extra passes (column-sum buffers, combine kernel) cost
# more than the exponentials it saves
SYM_MIN_POINTS = 32768


last_path = None  # the path the last kernel_product call took ("auto" resolved: direct_sym here, otherwise kmb_resolved_path)


# the kernels of bruteforce.py:18-22: functions of |x - y|, so K is symmetric when the targets are the sources
SYMMETRIC_KERNELS = ("gaussian", "absolute-exponential", "inverse-distance")


def symmetric_applies(x, y, kernel, normalize_rows=False, density_estimation=False, E=1, causal=False):
    """targets *are* the sources (same tensor), plain product or density of a kernel of bruteforce.py (all of :18-22 are
    functions of |x - y|, so K is symmetric; dot-exponential has no symmetric kernel), D <= 3, E == 1, not causal (the
    masked matrix is triangular, not symmetric)."""
    return (x.data_ptr() == y.data_ptr() and x.shape == y.shape and kernel in SYMMETRIC_KERNELS and not normalize_rows
            and E == 1 and x.shape[1] <= 3 and not causal)


def causal_row_bounds(n, rank, world, tile=128):
    """Row block of ``rank`` of ``world`` for a causal product over rows 0 .. n - 1: row i costs about i + 1 sources, so
    equal shares of the triangle end near n sqrt(g / world); boundaries on ``tile``-row tiles.  Returns (lo, hi)."""
    def edge(g):
        if g >= world:
            return n
        return min(n, int(round(n * (g / world) ** 0.5 / tile)) * tile)
    return edge(rank), max(edge(rank), edge(rank + 1))


def workspace_bytes(N, M, D, E, *, kernel="gaussian", normalize_rows=False, density_estimation=False, path="auto", causal=False):
    """kmb_product_workspace_bytes for this shape."""
    flags = _flags(normalize_rows, density_estimation, causal)
    need = ctypes.c_size_t(0)
    _lib.check(_lib.load().kmb_product_workspace_bytes(int(N), int(M), int(D), int(E), _lib.KERNEL_IDS[kernel], flags,
                                                       _lib.PATH_IDS[path], ctypes.byref(need)))
    return int(need.value)


def resolved_path(D, E, kernel="gaussian", path="auto", causal=False):
    """The name of the path ``path`` stands for with this D, E and kernel (kmb_resolved_path; "auto" -> what the C library picks).
    A causal product resolves "auto" to "tensor_f16" at every D."""
    if causal and path == "auto":
        return "tensor_f16"
    pid = int(_lib.load().kmb_resolved_path(int(D), int(E), _lib.KERNEL_IDS[kernel], _lib.PATH_IDS[path]))
    names = {v: k for k, v in _lib.PATH_IDS.items() if k != "tensor"}
    if pid not in names:
        raise ValueError(f"bad arguments D={D} E={E} kernel={kernel} path={path}")
    return names[pid]


PLAN_FIELDS = ("path", "family", "diff_table", "diff_index", "prod_table", "prod_index", "chunk", "passes", "row_tiles",
               "source_blocks")


def dispatch_plan(N, M, D, E, *, kernel="gaussian", normalize_rows=False, density_estimation=False, path="auto", sms=148,
                  causal=False):
    """What kernel_product would launch for this problem on a device with ``sms`` SMs (kmb_debug_product_plan, host logic
    only, no GPU needed): a dict of PLAN_FIELDS, ``path`` and ``family`` as names, -1 where a field does not apply."""
    flags = _flags(normalize_rows, density_estimation, causal)
    out = (ctypes.c_int64 * len(PLAN_FIELDS))()
    _lib.check(_lib.load().kmb_debug_product_plan(int(N), int(M), int(D), int(E), _lib.KERNEL_IDS[kernel], flags,
                                                  _lib.PATH_IDS[path], int(sms), out))
    plan = dict(zip(PLAN_FIELDS, (int(v) for v in out)))
    plan["path"] = {v: k for k, v in _lib.PATH_IDS.items() if k != "tensor"}[plan["path"]]
    plan["family"] = _lib.FAMILIES[plan["family"]]
    return plan


PV_PLAN_FIELDS = ("family", "pair", "grid", "stages", "kblocks", "ksteps_last", "passes", "eb_first", "ebp_first", "eb_last",
                  "ebp_last", "row_tiles", "source_blocks", "R", "C", "W", "R_last", "C_last", "flush_blocks")


def pv_plan(N, M, D, E, *, kernel="gaussian", normalize_rows=False, path="auto", sms, smem_optin, causal=False):
    """How the P.B kernel (families pv, pv16, pv16_pair) would run this problem on a device with ``sms`` SMs and
    ``smem_optin`` bytes of opt-in shared memory per block (kmb_debug_pv_plan, the launchers' own plan; host logic only,
    no GPU needed): a dict of PV_PLAN_FIELDS, ``family`` as a name, ``pair`` as a bool.  With CTA pairs R and R_last
    count pairs of row tiles.  Another family only fills ``family`` (the rest are -1)."""
    flags = _flags(normalize_rows, False, causal)
    out = (ctypes.c_int64 * len(PV_PLAN_FIELDS))()
    _lib.check(_lib.load().kmb_debug_pv_plan(int(N), int(M), int(D), int(E), _lib.KERNEL_IDS[kernel], flags,
                                             _lib.PATH_IDS[path], int(sms), int(smem_optin), out))
    plan = dict(zip(PV_PLAN_FIELDS, (int(v) for v in out)))
    plan["family"] = _lib.FAMILIES[plan["family"]]
    if plan["pair"] >= 0:
        plan["pair"] = bool(plan["pair"])
    return plan


CAUSAL_WORK_FIELDS = ("family", "waves", "units", "block", "tile", "sb_lo", "sb_hi", "c", "Cw")


def causal_work(N, M, D, E, wave, unit, *, kernel="gaussian", normalize_rows=False, path="auto", row_offset=0, sms=148,
                smem_optin=232448):
    """The work of ``unit`` (a CTA, or a cluster of two for the CTA-pair kernels) in wave ``wave`` of the causal kernel
    kernel_product(..., causal=True) would launch (kmb_debug_causal_work, the kernels' own schedule; host logic only, no GPU
    needed): a dict of CAUSAL_WORK_FIELDS, ``family`` as a name; ``tile`` (a pair index for CTA pairs) and the source-block
    range [sb_lo, sb_hi) of range c of Cw are -1 when the unit has no row tile in that wave."""
    out = (ctypes.c_int64 * len(CAUSAL_WORK_FIELDS))()
    _lib.check(_lib.load().kmb_debug_causal_work(int(N), int(M), int(D), int(E), _lib.KERNEL_IDS[kernel],
                                                 _flags(normalize_rows, False, True), _lib.PATH_IDS[path], int(row_offset),
                                                 int(sms), int(smem_optin), int(wave), int(unit), out))
    work = dict(zip(CAUSAL_WORK_FIELDS, (int(v) for v in out)))
    work["family"] = _lib.FAMILIES[work["family"]]
    return work


SYM_PLAN_FIELDS = ("tile_rows", "block_sources", "TB", "units", "unit_begin", "unit_end", "grid", "n_strips", "Wb",
                   "seg_base", "strip_base", "segments", "strips", "forms", "strip_cap")


def sym_plan(n, D, *, kernel="gaussian", part=0, n_parts=1, sms=148):
    """How kernel_product_sym_part would run part ``part`` of ``n_parts`` on a device with ``sms`` SMs (kmb_debug_sym_plan,
    the launcher's own geometry and partition; host logic only, no GPU needed): a dict of SYM_PLAN_FIELDS, ``forms`` as
    the tuple of evaluation forms enqueued ("difference", and "product" for the Gaussian), ``strip_cap`` as a bool."""
    out = (ctypes.c_int64 * len(SYM_PLAN_FIELDS))()
    _lib.check(_lib.load().kmb_debug_sym_plan(int(n), int(D), _lib.KERNEL_IDS[kernel], int(part), int(n_parts), int(sms), out))
    plan = dict(zip(SYM_PLAN_FIELDS, (int(v) for v in out)))
    plan["forms"] = tuple(name for bit, name in ((1, "difference"), (2, "product")) if plan["forms"] & bit)
    plan["strip_cap"] = bool(plan["strip_cap"])
    return plan


DIRECT_ENTRY_FIELDS =("KID", "NORM", "FORM", "DP", "EP", "R", "TILE_ROWS", "SB", "RECV", "PS")


def direct_entries(table):
    """Every entry of direct-kernel table ``table`` (0..7, kmb_debug_direct_entry) as dicts of DIRECT_ENTRY_FIELDS."""
    lib = _lib.load()
    out = (ctypes.c_int32 * 11)()
    _lib.check(lib.kmb_debug_direct_entry(int(table), -1, out))
    entries = []
    for i in range(out[0]):
        _lib.check(lib.kmb_debug_direct_entry(int(table), i, out))
        entries.append(dict(zip(DIRECT_ENTRY_FIELDS, out[1:])))
    return entries


def prepare_points(x, y, *, kernel="gaussian", path="auto", workspace=None, min_bytes=0, causal=False):
    """The points-only part of a product (kmb_product_prepare_f32): for the FP16 tensor path the prepass (centre, scale,
    operand planes, squared norms) is written to the head of ``workspace``.  Returns the buffer it was written to: a
    later ``kernel_product(..., prepared=token)`` on the same x, y, kernel, path and workspace skips the prepass as long
    as the workspace has not been reallocated since (``token`` is compared with the buffer in use; otherwise the
    product silently does the prepass itself).  No-op (returns None) on the other paths.  The dot-exponential kernel
    takes the FP16 tensor path at every D, so it is prepared at every D, and so is every kernel on "tensor_f16x1" and every
    causal product (``causal`` as for kernel_product)."""
    lib = _lib.load()
    _check_f32("target points", x)
    _check_f32("source points", y, x.shape[1])
    N, D = x.shape
    M = y.shape[0]
    three_term = _lib.PATH_IDS[path] in (_lib.PATH_IDS["auto"], _lib.PATH_IDS["tensor_f16"])
    if path != "tensor_f16x1" and (not three_term or (D <= 16 and kernel != "dot-exponential" and not causal)):
        return None
    kid, pid = _lib.KERNEL_IDS[kernel], _lib.PATH_IDS[path]
    flags = _flags(causal=causal)
    need = ctypes.c_size_t(0)
    _lib.check(lib.kmb_product_workspace_bytes(N, M, D, 1, kid, flags, pid, ctypes.byref(need)))
    if workspace is None:
        workspace = _default_ws.setdefault(x.device, Workspace())
    ws = workspace.get(max(need.value, int(min_bytes)), x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.kmb_product_prepare_f32(_ptr(x), _ptr(y), N, M, D, kid, flags, pid, _ptr(ws), ws.numel(), _stream()))
    return ws


def kernel_product(x, y, b, *, kernel="gaussian", normalize_rows=False, density_estimation=False, path="auto",
                   row_offset=0, out=None, workspace=None, prepared=None, causal=False):
    """a_i = sum_j k(x_i, y_j) b_j on the current CUDA device (kmb_product_f32).

    x (N, D), y (M, D), b (M, E) float32 CUDA tensors; b is ignored (may be None)
    under ``density_estimation``.  Asynchronous on the current stream.  ``prepared``: the token of
    ``prepare_points`` for these points (see there).  ``causal``: a_i = sum_{j <= row_offset + i} k(x_i, y_j) b_j
    (KMB_FLAG_CAUSAL; the three-term FP16 tensor path, other paths raise NotImplementedError).
    """
    lib = _lib.load()
    if kernel not in _lib.KERNEL_IDS:
        raise NotImplementedError(f"B200 kernel product doesn't support kernel {kernel}.")
    _check_f32("target points", x)
    _check_f32("source points", y, x.shape[1])
    N, D = x.shape
    M = y.shape[0]
    flags = _flags(normalize_rows, density_estimation, causal)
    if density_estimation:
        b, E = None, 1
    else:
        _check_f32("source signal", b)
        if b.shape[0] != M:
            raise ValueError("source signal and source points disagree on M")
        E = b.shape[1]
    if out is None:
        out = torch.empty((N, E), dtype=torch.float32, device=x.device)
    else:
        _check_f32("out", out, E)
    if path == "auto" and N >= SYM_MIN_POINTS and symmetric_applies(x, y, kernel, normalize_rows, density_estimation, E, causal):
        path = "direct_sym"  # same_points: each kernel value serves its row and its column (kprod_sym.cuh)
    global last_path
    last_path = path if path == "direct_sym" else resolved_path(D, E, kernel, path, causal)   # what "auto" stood for
    kid, pid = _lib.KERNEL_IDS[kernel], _lib.PATH_IDS[path]
    need = ctypes.c_size_t(0)
    _lib.check(lib.kmb_product_workspace_bytes(N, M, D, E, kid, flags, pid, ctypes.byref(need)))
    if workspace is None:
        workspace = _default_ws.setdefault(x.device, Workspace())
    ws = workspace.get(need.value, x.device)
    if prepared is not None and prepared is ws:   # same buffer as at prepare time: its head holds the operand planes
        flags |= _lib.FLAG_PREPARED
    with torch.cuda.device(x.device):
        _lib.check(lib.kmb_product_f32(_ptr(x), _ptr(y), _ptr(b), _ptr(out), N, M, D, E, kid, flags, pid, int(row_offset),
                                       _ptr(ws), ws.numel(), _stream()))
    return out


def kernel_product_sym_part(y, b, part, n_parts, *, kernel="gaussian", out=None, workspace=None):
    """This part's share of the product with targets == sources (kmb_product_sym_f32).

    Returns an (n, 1) tensor; the shares of all ``n_parts`` parts add up to K b (the caller
    all-reduces them when every part runs on its own GPU).  Asynchronous on the current stream.
    """
    lib = _lib.load()
    _check_f32("points", y)
    n, D = y.shape
    if b is not None:  # None: density estimation (b == 1)
        _check_f32("signal", b, 1)
        if b.shape[0] != n:
            raise ValueError("signal and points disagree on n")
    if out is None:
        out = torch.empty((n, 1), dtype=torch.float32, device=y.device)
    else:
        _check_f32("out", out, 1)
    need = ctypes.c_size_t(0)
    _lib.check(lib.kmb_product_sym_workspace_bytes(n, D, int(part), int(n_parts), ctypes.byref(need)))
    if workspace is None:
        workspace = _default_ws.setdefault(y.device, Workspace())
    ws = workspace.get(need.value, y.device)
    with torch.cuda.device(y.device):
        _lib.check(lib.kmb_product_sym_f32(_ptr(y), _ptr(b), _ptr(out), n, D, _lib.KERNEL_IDS[kernel], int(part),
                                           int(n_parts), _ptr(ws), ws.numel(), _stream()))
    return out


def kernel_product_f64(x, y, b, *, kernel="gaussian", normalize_rows=False, density_estimation=False, row_offset=0, out=None,
                       causal=False):
    """The float64 variant (kmb_product_f64): x (N, D), y (M, D), b (M, E) float64 CUDA tensors, any D; ``causal`` as for
    kernel_product (every kernel)."""
    lib = _lib.load()
    if kernel not in _lib.KERNEL_IDS:
        raise NotImplementedError(f"B200 kernel product doesn't support kernel {kernel}.")
    for name, t in (("target points", x), ("source points", y)) + ((("source signal", b),) if not density_estimation else ()):
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.dim() == 2):
            raise ValueError(f"{name} must be a contiguous 2-D float64 CUDA tensor")
    N, D = x.shape
    M = y.shape[0]
    if y.shape[1] != D:
        raise ValueError("target and source points disagree on D")
    E = 1 if density_estimation else b.shape[1]
    if not density_estimation and b.shape[0] != M:
        raise ValueError("source signal and source points disagree on M")
    flags = _flags(normalize_rows, density_estimation, causal)
    if out is None:
        out = torch.empty((N, E), dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.kmb_product_f64(_ptr(x), _ptr(y), None if density_estimation else _ptr(b), _ptr(out), N, M, D, E,
                                       _lib.KERNEL_IDS[kernel], flags, int(row_offset), _stream()))
    global last_path
    last_path = "direct_f64"
    return out


def kernel_block_f64(x, y, *, kernel="gaussian"):
    """Explicit (n, m) block k(x_i, y_j) of the kernel matrix in float64 (kmb_kernel_block_f64): the landmark
    columns of the Nystrom preconditioner.  x (n, D), y (m, D): float64 CUDA tensors."""
    lib = _lib.load()
    if kernel not in _lib.KERNEL_IDS:
        raise NotImplementedError(f"B200 kernel product doesn't support kernel {kernel}.")
    for name, t in (("points", x), ("landmarks", y)):
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.dim() == 2):
            raise ValueError(f"{name} must be a contiguous 2-D float64 CUDA tensor")
    if x.shape[1] != y.shape[1]:
        raise ValueError("points and landmarks disagree on D")
    out = torch.empty((x.shape[0], y.shape[0]), dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.kmb_kernel_block_f64(_ptr(x), _ptr(y), _ptr(out), x.shape[0], y.shape[0], x.shape[1],
                                            _lib.KERNEL_IDS[kernel], _stream()))
    return out


def direct_stats(workspace=None, device=None):
    """What the device-side statistics pass of the last direct-path product decided (synchronises):
    bounding-box centre, log2(e)*half-diagonal^2 and the evaluation form of the Gaussian kernel."""
    import struct

    if workspace is None:
        workspace = _default_ws[torch.device(device) if device is not None else next(iter(_default_ws))]
    raw = bytes(workspace.buf[:80].cpu().numpy())
    vals = struct.unpack("16f f i I i", raw)
    return {"center": vals[:16], "radius2": vals[16], "form": "product" if vals[17] else "difference"}


def last_launch_count():
    return int(_lib.load().kmb_last_launch_count())


def device_info(device=0):
    info = _lib.DeviceInfo()
    _lib.check(_lib.load().kmb_get_device_info(int(device), ctypes.byref(info)))
    return {f: getattr(info, f) for f, _ in info._fields_}


def set_profiling(enabled):
    _lib.check(_lib.load().kmb_set_profiling(int(bool(enabled))))


def last_main_kernel_ms():
    ms = ctypes.c_float(0)
    _lib.check(_lib.load().kmb_last_main_kernel_ms(ctypes.byref(ms)))
    return float(ms.value)
