"""ctypes binding of libkmb_b200.so (include/kmb_b200.h).

There is deliberately no fallback: if the shared library is missing or a call
fails, this raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
(or ``make -C kernel_matrix_benchmarks_b200/csrc``).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# KMB_B200_LIB: another build of the same library (instrumented or A/B variants made by csrc/Makefile with EXTRA=...)
LIB_PATH = os.environ.get("KMB_B200_LIB") or os.path.join(_HERE, "libkmb_b200.so")

KMB_OK, KMB_ERR_INVALID, KMB_ERR_UNSUPPORTED, KMB_ERR_WORKSPACE, KMB_ERR_CUDA = range(5)

# "dot-exponential" is exp(<x, y>) (softmax attention under normalize_rows): not in bruteforce.py, an extension
KERNEL_IDS = {"gaussian": 0, "absolute-exponential": 1, "inverse-distance": 2, "dot-exponential": 3}
# FLAG_CAUSAL: row i sees sources j <= row_offset + i (an extension, not in bruteforce.py)
FLAG_NORMALIZE_ROWS, FLAG_DENSITY, FLAG_PREPARED, FLAG_CAUSAL = 1, 2, 4, 8
# "tensor_f16x1": the FP16 tensor path with one hi.hi term (float16-class accuracy; only when asked for, never "auto")
PATH_IDS = {"auto": 0, "direct": 1, "tensor": 5, "tensor_tf32": 2, "tensor_f16": 5, "direct_diff": 3, "direct_sym": 4,
            "tensor_f16x1": 6}
# KMB_FAMILY_* of kmb_debug_product_plan, by value
FAMILIES = ("direct", "sym", "tensor", "tensor_pair", "pv", "pv16", "pv16_pair", "fill", "unsupported")


class DeviceInfo(ctypes.Structure):
    _fields_ = [
        ("sm_count", c_int),
        ("cc_major", c_int),
        ("cc_minor", c_int),
        ("clock_khz", c_int),
        ("l2_bytes", c_int),
        ("smem_per_block_optin", c_int),
        ("total_mem", c_size_t),
    ]


class DeviceShard(ctypes.Structure):
    """kmb_device_shard (include/kmb_b200.h)."""

    _fields_ = [
        ("device", c_int),
        ("flags", c_int),
        ("x", c_void_p),
        ("y", c_void_p),
        ("b", c_void_p),
        ("out", c_void_p),
        ("n_targets", c_int64),
        ("row_offset", c_int64),
        ("workspace", c_void_p),
        ("workspace_bytes", c_size_t),
        ("stream", c_void_p),
    ]


# every symbol include/kmb_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "kmb_abi_version": (c_int, []),
    "kmb_last_error": (c_char_p, []),
    "kmb_last_launch_count": (c_int, []),
    "kmb_get_device_info": (c_int, [c_int, POINTER(DeviceInfo)]),
    "kmb_product_workspace_bytes": (c_int, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, POINTER(c_size_t)]),
    "kmb_product_f32": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_int64,
         c_void_p, c_size_t, c_void_p],
    ),
    "kmb_product_prepare_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "kmb_product_sym_workspace_bytes": (c_int, [c_int64, c_int, c_int, c_int, POINTER(c_size_t)]),
    "kmb_product_sym_f32": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p],
    ),
    "kmb_enable_peer_access": (c_int, [POINTER(c_int), c_int]),
    "kmb_product_rows_multi_f32": (c_int, [POINTER(DeviceShard), c_int, c_int64, c_int, c_int, c_int, c_int, c_int]),
    "kmb_product_sym_multi_f32": (c_int, [POINTER(DeviceShard), c_int, c_void_p, c_int64, c_int, c_int]),
    "kmb_reduce_parts_f32": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_int64, c_void_p]),
    "kmb_product_f64": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int64, c_void_p],
    ),
    "kmb_kernel_block_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p]),
    "kmb_debug_plan_waves": (c_int, [c_int64, c_int64, c_int, c_size_t, POINTER(c_int64)]),
    "kmb_debug_sym_unit": (c_int, [c_int64, c_int64, c_int64, POINTER(c_int64)]),
    "kmb_debug_sym_plan": (c_int, [c_int64, c_int, c_int, c_int, c_int, c_int, POINTER(c_int64)]),
    "kmb_resolved_path": (c_int, [c_int, c_int, c_int, c_int]),
    "kmb_debug_product_plan": (c_int, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, POINTER(c_int64)]),
    "kmb_debug_direct_entry": (c_int, [c_int, c_int, POINTER(c_int32)]),
    "kmb_debug_causal_work": (
        c_int,
        [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, POINTER(c_int64)],
    ),
    "kmb_debug_pv_plan": (c_int, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, POINTER(c_int64)]),
    "kmb_set_profiling": (c_int, [c_int]),
    "kmb_last_main_kernel_ms": (c_int, [POINTER(c_float)]),
    "kmb_cg_scratch_bytes": (c_size_t, []),
    "kmb_cg_init_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "kmb_cg_shift_dot_f32": (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "kmb_cg_update_f32": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p],
    ),
    "kmb_cg_direction_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "kmb_cg_init_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "kmb_cg_shift_dot_f64": (c_int, [c_void_p, c_void_p, c_double, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "kmb_cg_update_f64": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p],
    ),
    "kmb_cg_direction_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
}

_lib = None


class KmbError(RuntimeError):
    pass


def load():
    """Load libkmb_b200.so; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the B200 plugin has no CPU fallback. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` first."
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the header and the library disagree
            fn.restype, fn.argtypes = res, args
        if lib.kmb_abi_version() != 1:
            raise ImportError(f"libkmb_b200.so ABI {lib.kmb_abi_version()} != 1")
        _lib = lib
    return _lib


def check(rc):
    """Map a KMB_ERR_* return code to the exception the reference's callers expect."""
    if rc == KMB_OK:
        return
    msg = load().kmb_last_error().decode()
    if rc == KMB_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)  # bruteforce.py:82-85 raises the same for unknown kernels
    if rc == KMB_ERR_INVALID:
        raise ValueError(msg)
    raise KmbError(f"libkmb_b200 error {rc}: {msg}")
