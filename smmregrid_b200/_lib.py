"""ctypes binding of the C ABI declared in ``include/smmregrid_b200.h``.

The library must exist (``python -m smmregrid_b200._build`` or ``__graft_entry__.build()``);
a missing library is a hard error -- this package has no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes
import os

from . import _build

SMM_OK, SMM_ERR_INVALID, SMM_ERR_RANGE, SMM_ERR_CUDA, SMM_ERR_ALLOC, SMM_ERR_DTYPE = range(6)
SMM_F32, SMM_F64, SMM_I16, SMM_F16, SMM_BF16 = 0, 1, 2, 3, 4
SMM_KERNEL_STAGED, SMM_KERNEL_GATHER, SMM_KERNEL_COMPACT = 1, 2, 3
KERNEL_NAMES = {SMM_KERNEL_STAGED: "staged", SMM_KERNEL_GATHER: "gather"}
KERNEL_CODES = {None: 0, "auto": 0, "staged": SMM_KERNEL_STAGED, "gather": SMM_KERNEL_GATHER,
                "compact": SMM_KERNEL_COMPACT}
SMM_SUM_AUTO, SMM_SUM_FAST, SMM_SUM_REFERENCE = 0, 1, 2
SUMMATION_CODES = {None: SMM_SUM_AUTO, "auto": SMM_SUM_AUTO, "fast": SMM_SUM_FAST, "reference": SMM_SUM_REFERENCE}
SUMMATION_NAMES = {SMM_SUM_FAST: "fast", SMM_SUM_REFERENCE: "reference"}

i32, i64, f64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_double
vp = ctypes.c_void_p
P = ctypes.POINTER


class SmmInfo(ctypes.Structure):
    _fields_ = [
        ("n_src", i64), ("n_dst", i64), ("nnz", i64),
        ("n_levels", i32), ("kernel", i32), ("lanes_per_row", i32), ("links_per_lane", i32),
        ("rows_per_tile", i32), ("n_tiles", i32), ("max_row_nnz", i32), ("max_tile_segments", i32),
        ("consumer_threads", i32), ("rows_reordered", i32), ("packed_rows", i32), ("summation", i32),
        ("max_tile_elems", i64), ("sum_tile_elems", i64), ("touched_src", i64), ("device_bytes", i64),
        ("plan_cache_hit", i32), ("gather_rows", i32),
    ]

    def asdict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["kernel_name"] = KERNEL_NAMES.get(self.kernel, "?")
        d["summation_name"] = SUMMATION_NAMES.get(self.summation, "?")
        return d


class SmmCreateOpts(ctypes.Structure):
    """``smm_create_opts``: zero-initialised = defaults."""
    _fields_ = [("summation", i32), ("reserved", i32), ("plan_cache_dir", ctypes.c_char_p)]


class SmmDecode(ctypes.Structure):
    """``smm_decode``: CF unpacking of 16-bit source data (x_dtype ``SMM_I16``)."""
    _fields_ = [("dtype", i32), ("is_unsigned", i32), ("scale_factor", f64), ("add_offset", f64),
                ("n_fill", i32), ("fill", i32 * 4)]


class SmmApplyOpts(ctypes.Structure):
    """``smm_apply_opts``: zero-initialised = defaults (automatic kernel, reference semantics)."""
    _fields_ = [("kernel", i32), ("renormalize", i32), ("min_valid_fraction", f64), ("decode", P(SmmDecode))]


def create_opts(summation=None, plan_cache_dir=None):
    """``smm_create_opts`` for ``smm_create*`` (None when everything is default)."""
    code = SUMMATION_CODES[summation] if not isinstance(summation, int) else summation
    if code == SMM_SUM_AUTO and not plan_cache_dir:
        return None
    return SmmCreateOpts(code, 0, os.fsencode(plan_cache_dir) if plan_cache_dir else None)


def apply_opts(kernel=None, renormalize=None, decode=None):
    """``smm_apply_opts`` for one call (None when everything is default).  ``kernel``: None |
    'auto' | 'staged' | 'gather' | 'compact' (or the SMM_KERNEL_* code); ``renormalize``: None
    (reference semantics) or the minimum valid weight fraction of the opt-in extension;
    ``decode``: an ``SmmDecode`` for x_dtype ``SMM_I16`` (the options keep it alive)."""
    code = kernel if isinstance(kernel, int) else KERNEL_CODES[kernel]
    if code == 0 and renormalize is None and decode is None:
        return None
    o = SmmApplyOpts(code, 0 if renormalize is None else 1, 0.0 if renormalize is None else float(renormalize),
                     ctypes.pointer(decode) if decode is not None else None)
    o._decode = decode
    return o


# name -> (restype, argtypes): every symbol the header declares
SIGNATURES = {
    "smm_create": (ctypes.c_int, [i64, i64, i64, vp, vp, vp, i32, i32, i32, P(SmmCreateOpts), P(vp)]),
    "smm_create_levels": (ctypes.c_int, [i32, vp, i64, i64, i64, vp, vp, vp, i32, i32, i32, P(SmmCreateOpts), P(vp)]),
    "smm_destroy": (ctypes.c_int, [vp]),
    "smm_get_info": (ctypes.c_int, [vp, i32, P(SmmInfo)]),
    "smm_mask_sum": (ctypes.c_int, [vp, i32, vp, vp, P(i32)]),
    "smm_set_dst_mask": (ctypes.c_int, [vp, i32, vp, vp]),
    "smm_apply": (ctypes.c_int, [vp, i32, vp, i32, i64, i64, vp, i32, i64, i32, f64, P(SmmApplyOpts), vp]),
    "smm_apply_levels": (ctypes.c_int, [vp, i32, vp, vp, i32, i64, i64, i64, vp, i32, i64, i64, vp, f64,
                                        P(SmmApplyOpts), vp]),
    "smm_apply_host": (ctypes.c_int, [vp, i32, vp, i32, i64, i64, vp, i32, i64, i32, f64, P(SmmApplyOpts), i64]),
    "smm_apply_levels_host": (ctypes.c_int, [vp, i32, vp, vp, i32, i64, vp, i32, vp, f64, P(SmmApplyOpts), i64]),
    "smm_nan_variation": (ctypes.c_int, [vp, i32, i64, i64, i64, P(i64), vp]),
    "smm_host_plan_build": (ctypes.c_int, [i64, i64, i64, vp, vp, vp, i32, i32, P(SmmCreateOpts), P(vp)]),
    "smm_host_plan_info": (ctypes.c_int, [vp, P(SmmInfo), P(i64)]),
    "smm_host_plan_copy": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, vp, vp]),
    "smm_host_plan_rowmap": (ctypes.c_int, [vp, vp]),
    "smm_host_plan_rowslot": (ctypes.c_int, [vp, vp]),
    "smm_host_plan_gather_rows": (ctypes.c_int, [vp, vp]),
    "smm_host_plan_compact": (ctypes.c_int, [vp, P(i64), P(i64), vp, vp, vp]),
    "smm_host_plan_free": (None, [vp]),
    "smm_copy_ceiling": (ctypes.c_int, [i32, vp, i64, i32, i32, P(f64)]),
    "smm_launch_count": (i64, []),
    "smm_last_error": (ctypes.c_char_p, []),
    "smm_version": (ctypes.c_char_p, []),
}

_lib = None


class SmmError(RuntimeError):
    pass


def lib_path() -> str:
    """In-tree library; SMM_LIB_PATH points at an alternative build (experiments)."""
    return os.environ.get("SMM_LIB_PATH") or _build.LIB_PATH


def load():
    """Load the shared library (never builds silently, never falls back)."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not os.path.exists(path):
            raise SmmError(
                f"{path} is missing: build it with `python -m smmregrid_b200._build` "
                "(nvcc, sm_100a). smmregrid_b200 has no CPU fallback.")
        lib = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


_EXC = {SMM_ERR_INVALID: ValueError, SMM_ERR_RANGE: ValueError, SMM_ERR_CUDA: SmmError,
        SMM_ERR_ALLOC: MemoryError, SMM_ERR_DTYPE: TypeError}


def check(rc: int):
    """Map a status code to the exception type the reference would raise."""
    if rc != SMM_OK:
        msg = load().smm_last_error().decode("utf-8", "replace")
        raise _EXC.get(rc, SmmError)(msg)
