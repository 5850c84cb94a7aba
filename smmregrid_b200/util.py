"""Device mirror of ``smmregrid/util.py:detect_nan_variation_dims`` (SURVEY.md §8 f4).

The reference uses this probe (``regrid.py:630-653``, ``check_nan=True``) to find out along which
extra dimensions the missing-value pattern of a field changes, i.e. which dimension needs
per-level masked weights.  The test itself -- does NaN-ness change anywhere along an axis -- is
one pass over the first time step; here it runs in ``nan_variation_kernel`` through the C ABI
(``smm_nan_variation``), on the data where it already lives (CUDA tensor) or after one copy.
"""
from __future__ import annotations

import ctypes
from typing import Sequence, Union

import numpy as np

from . import _lib


def _first_step(field, time_axis):
    if time_axis is None:
        return field
    return field[(slice(None),) * time_axis + (0,)]


def nan_variation_count(field, axis: int, device=None) -> int:
    """Positions (over the other axes) whose NaN-ness changes somewhere along ``axis``:
    ``isnull().astype('int8').diff(dim).astype(bool).any(dim).sum()`` (``util.py:75-78``)."""
    import torch
    lib = _lib.load()
    if isinstance(field, torch.Tensor):
        t = field if field.is_cuda else field.to(f"cuda:{0 if device is None else device}")
    else:
        a = np.asarray(field)
        if a.dtype not in (np.float16, np.float32, np.float64):
            return 0                                        # integer data has no NaN (isnull is all False)
        t = torch.from_numpy(np.ascontiguousarray(a)).to(f"cuda:{0 if device is None else device}")
    if t.dtype in (torch.float16, torch.bfloat16):
        t = t.to(torch.float32)                             # widening keeps NaN-ness exactly; the kernel reads f32 / f64
    if t.dtype not in (torch.float32, torch.float64):
        return 0
    t = t.contiguous()
    axis = axis % t.dim()
    shape = tuple(t.shape)
    outer = int(np.prod(shape[:axis], dtype=np.int64))
    inner = int(np.prod(shape[axis + 1:], dtype=np.int64))
    count = ctypes.c_int64()
    with torch.cuda.device(t.device):
        _lib.check(lib.smm_nan_variation(t.data_ptr(), _lib.SMM_F32 if t.dtype == torch.float32 else _lib.SMM_F64,
                                         outer, shape[axis], inner, ctypes.byref(count),
                                         torch.cuda.current_stream().cuda_stream))
    return int(count.value)


def detect_nan_variation_dims(field, time_dim, check_dims: Sequence[Union[int, str]], device=None):
    """``smmregrid/util.py:57-85``: the members of ``check_dims`` along which the NaN pattern of
    ``field`` varies, looking at the first step of ``time_dim`` only.

    ``field`` is a numpy array / torch tensor (dims are axis numbers of ``field``; ``time_dim``
    an axis number, a 1-element list as the reference passes it, or None / []) or, when xarray
    is installed, a ``DataArray`` (dims are names).
    """
    if isinstance(time_dim, (list, tuple)):
        time_dim = time_dim[0] if len(time_dim) else None
    if hasattr(field, "dims") and hasattr(field, "isel"):                 # xarray.DataArray
        if time_dim is not None and time_dim in field.dims:
            field = field.isel({time_dim: 0}, drop=True)
        names = list(field.dims)
        data = np.asarray(field.values)
        return [d for d in check_dims if nan_variation_count(data, names.index(d), device) > 0]
    ndim = field.dim() if hasattr(field, "dim") else np.ndim(field)
    time_axis = None if time_dim is None else int(time_dim) % ndim
    first = _first_step(field, time_axis)
    out = []
    for d in check_dims:
        ax = int(d) % ndim
        if time_axis is not None:
            if ax == time_axis:
                continue                                     # removed with the time step
            ax -= ax > time_axis
        if nan_variation_count(first, ax, device) > 0:
            out.append(d)
    return out
