"""Regridder -- host-side mirror of ``smmregrid/regrid.py`` for the weight-application path.

Same class / method names, argument meaning and error behaviour as the reference for the
part of the API that sits on the hot path (``Regridder(weights=...)``, ``regrid``,
``regrid_array``, ``regrid2d``, ``regrid3d``, ``apply_weights``, module-level ``regrid``).
Weight *generation* (``Regridder(source_grid, target_grid)`` -> CDO subprocess) is out of
scope here and raises ``NotImplementedError``: generate the weights with CDO / the reference's
``CdoGenerate`` and pass them in.

Data may be

* an ``xarray.DataArray`` / ``Dataset`` (anything with the same surface: ``dims``, ``coords``,
  ``attrs``, ``name``, ``data``, ``isel``, ``transpose``; xarray itself is never imported).
  Horizontal and mask dimensions are recognised by NAME exactly as the reference's
  ``GridType`` does (``gridtype.py:6-13`` + ``horizontal_dims=`` / ``mask_dim=``).  The field
  is **never materialised as a whole**: dask-backed arrays stay lazy
  (``dask.array.map_blocks`` over chunks of the kept dims, like ``regrid.py:538-550``), any
  other backing is streamed through the device in blocks of the leading kept dim
  (``host_block_bytes``), so peak host memory is one block plus the (50-100x smaller) result.
* a numpy array or torch tensor (CPU or CUDA): the horizontal axes are the trailing ones
  (``[..., nlat, nlon]`` or ``[..., ncell]``) and, for 3-D weights, ``mask_dim`` is the axis
  just before them unless ``level_axis`` says otherwise.

The numeric core always runs in the sm_100a kernels through the C ABI; there is no CPU path.
Everything that varies per call (kernel family, the renormalising extension) travels as an
argument of the C call (``smm_apply_opts``), never as state of the shared device handle.

CF-packed 16-bit data (``packing=``, see ``packing.CFPacking``) reaches the kernels raw and is
decoded there: a ``CFPacking`` for arrays and tensors, ``"cf"`` to take it from each variable's own
attributes (as opened with ``mask_and_scale=False``).
"""
from __future__ import annotations

import ctypes
import logging
import math
from typing import Optional, Sequence

import numpy as np

from . import _lib
from .packing import PACKING_ATTRS, RAW_DTYPES, CFPacking
from .weights import (CdoWeights, WeightsMatrix, check_mask, compute_weights_matrix,
                      compute_weights_matrix3d, mask_weights, _device_index)

DEFAULT_AREA_MIN = 0.5  # default minimum area for conservative remapping (regrid.py:49)
LEVEL_TOLERANCE = 1e-3  # regrid.py:390

# dimension names the reference recognises (smmregrid/gridtype.py:6-13)
DEFAULT_DIMS = {
    'horizontal': ['i', 'j', 'x', 'y', 'lon', 'lat', 'longitude', 'latitude',
                   'cell', 'cells', 'ncells', 'values', 'value', 'nod2', 'pix', 'elem',
                   'nav_lon', 'nav_lat', 'rgrid'],
    'mask': ['lev', 'nz1', 'nz', 'depth', 'depth_full', 'depth_half'],
    'time': ['time', 'time_counter', 'valid_time', 'forecast_time'],
}


def _logger(level):
    log = logging.getLogger("smmregrid.Regrid")
    log.setLevel(getattr(logging, str(level).upper(), logging.WARNING))
    return log


def _torch():
    import torch
    return torch


def _np_dtype_code(dt) -> int:
    dt = np.dtype(dt)
    if dt == np.float32:
        return _lib.SMM_F32
    if dt == np.float64:
        return _lib.SMM_F64
    raise TypeError(f"only float32/float64 data can be regridded, got {dt}")


def _tolist(value):
    """``smmregrid/util.py:47``."""
    if value is None:
        return []
    return value if isinstance(value, list) else [value]


def select_level(weight_levels, lev, name="lev") -> int:
    """Nearest weights level within 1e-3, else ValueError (``regrid.py:386-395``)."""
    wl = np.asarray(weight_levels, dtype=np.float64)
    d = np.abs(wl - float(lev))
    widx = int(np.argmin(d))
    if not d[widx] <= LEVEL_TOLERANCE:
        raise ValueError(f"{lev} not found in mask_dim {name}. Available levels: {list(wl)}")
    return widx


def _is_dataset(obj) -> bool:
    return hasattr(obj, "data_vars") and hasattr(obj, "attrs") and hasattr(obj, "map")


def _is_dataarray(obj) -> bool:
    return (hasattr(obj, "dims") and hasattr(obj, "coords") and hasattr(obj, "attrs")
            and hasattr(obj, "isel") and not hasattr(obj, "data_vars"))


def _is_bounds(name) -> bool:
    """``GridInspector._is_bounds`` (``gridinspector.py:199-203``)."""
    name = str(name)
    return (name.endswith('_bnds') or name.endswith('_bounds') or name == 'vertices') and 'time' not in name


def _is_dask(array) -> bool:
    return type(array).__module__.split(".")[0] == "dask"


_PREFAULT_MIN_BYTES = 16 << 20
_MADV_POPULATE_WRITE = 23          # Linux >= 5.14: make the pages present and writable, contents untouched


def _prefault(addr: int, nbytes: int):
    try:
        libc = ctypes.CDLL(None)   # the process's own symbols: madvise of the C library
        page = 4096
        lo = (addr + page - 1) // page * page
        hi = (addr + nbytes) // page * page
        if hi > lo:
            libc.madvise(ctypes.c_void_p(lo), ctypes.c_size_t(hi - lo), ctypes.c_int(_MADV_POPULATE_WRITE))
    except Exception:              # an older kernel or another libc: the pages are faulted in by the copies instead
        pass


class _PinnedResults:
    """Small pool of page-locked result buffers.  A result in pinned memory is written by the
    device-to-host copies directly; a pageable one goes through the library's bounce buffers and
    a host memcpy that, with 4-8 ranks sharing the host's memory system, costs 8 ms of a 74 ms
    step (C4, 128 steps).  Allocating pinned memory per call is worse (3.6 ms for 66 MB), so
    buffers are kept and handed out again once the caller has dropped the previous result: a
    buffer is free when its storage has no user but the pool (views, and numpy arrays made from
    them, count as users).  Page-locking is expensive in a process that already holds tens of GB
    (~100 ms for 66 MB next to the bench's 28 GB slab), so the pool only serves a result size it
    has been asked for before (a loop), keeps at most two buffers per size -- what
    ``y = rg.regrid(x)`` in a loop needs -- and is capped; everything else, and every torch
    build without the storage-use-count hook, gets ordinary pageable arrays."""

    cap_bytes = 1 << 30
    min_bytes = 8 << 20
    per_size = 2

    def __init__(self):
        import threading
        self._bufs = []            # (flat uint8 pinned tensor, its storage use count when idle)
        self._asked = {}           # result size -> times requested
        self._lock = threading.Lock()

    @staticmethod
    def _alloc(nbytes):
        return _torch().empty(nbytes, dtype=_torch().uint8, pin_memory=True)

    @staticmethod
    def _users(t) -> int:
        return _torch()._C._storage_Use_Count(t.untyped_storage()._cdata)

    def take(self, shape, dtype):
        """pinned torch tensor of that shape / numpy dtype, or None (small result, cap reached, no hook)"""
        torch = _torch()
        nbytes = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
        if nbytes < self.min_bytes or nbytes > self.cap_bytes or not hasattr(torch._C, "_storage_Use_Count"):
            return None
        with self._lock:
            # (idle count measured per buffer when it is created: the tensor itself, the temporary
            # storage handle and whatever the allocator of this torch build keeps)
            self._asked[nbytes] = self._asked.get(nbytes, 0) + 1
            fits = [(t, idle) for t, idle in self._bufs if nbytes <= t.numel() <= 2 * nbytes]
            base = next((t for t, idle in fits if self._users(t) <= idle), None)
            if base is None:
                if self._asked[nbytes] < 2 or len(fits) >= self.per_size or \
                        sum(t.numel() for t, _ in self._bufs) + nbytes > self.cap_bytes:
                    return None
                try:
                    base = self._alloc(nbytes)
                except RuntimeError:
                    return None
                self._bufs.append((base, self._users(base)))
            tdt = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}[np.dtype(dtype)]
            return base[:nbytes].view(tdt).reshape(tuple(int(n) for n in shape))


_pinned_results = _PinnedResults()


def _new_host_result(shape, dtype) -> np.ndarray:
    """Pageable result array.  Its pages are new to the process: the first write to each makes the
    kernel map and zero-fill it (~7 ms for the 66 MB of a 128-step C4 result when the ranks of an
    8-GPU box all do that at once), and those first writes would be the library's result copies,
    in line with the device pipeline.  A helper thread asks the kernel to populate the pages
    (``madvise(MADV_POPULATE_WRITE)``: contents untouched, so it is safe next to the copies) while
    the first chunks are still on their way to the device."""
    a = np.empty(shape, dtype=dtype)
    if a.nbytes >= _PREFAULT_MIN_BYTES:
        import threading
        threading.Thread(target=_prefault, args=(a.ctypes.data, a.nbytes), daemon=True).start()
    return a


def remove_degenerate_axes(values, dims):
    """``smmregrid/dimension.py:22-37`` on a bare array: every axis along which all values
    are identical is averaged away.  Returns ``(values, dims)``."""
    values, dims = np.asarray(values), list(dims)
    for d in list(dims):
        ax = dims.index(d)
        if np.allclose(values.max(axis=ax) - values.min(axis=ax), 0):
            values = values.mean(axis=ax)
            dims.pop(ax)
    return values, dims


class Regridder(object):
    """Main regridding class (reference: ``smmregrid/regrid.py:52``), weights-initialised.

    Keywords beyond the reference's: ``device`` (CUDA device index), ``out_dtype`` (float32 to
    round the float64 result once at the store), ``renormalize`` (opt-in extension, see
    ``smm_apply_opts``), ``kernel`` (None | 'staged' | 'gather' | 'compact': force a kernel
    family, testing aid), ``summation`` (None = automatic | 'fast' | 'reference': see
    ``SMM_SUM_*`` in the header), ``plan_cache_dir`` (on-disk cache of the operator
    construction) and ``host_block_bytes`` (source bytes per streamed block of host data).
    """

    def __init__(self, source_grid=None, target_grid=None, weights=None,
                 method='con', remap_area_min=DEFAULT_AREA_MIN, transpose=True, mask_dim=None,
                 vertical_dim=None, horizontal_dims=None, cdo_extra=None, cdo_options=None,
                 check_nan=False, cdo='cdo', loglevel='WARNING',
                 device=None, out_dtype=None, renormalize=None, kernel=None, summation=None,
                 plan_cache_dir=None, host_block_bytes=1 << 30):
        if (source_grid is None or target_grid is None) and (weights is None):
            raise ValueError("Either weights or source_grid/target_grid must be supplied")
        if vertical_dim is not None:      # deprecated alias (util.py:26-39)
            import warnings
            warnings.warn("vertical_dim is deprecated and will be removed in future versions. "
                          "Please use mask_dim instead.", DeprecationWarning, stacklevel=2)
            if mask_dim is None:
                mask_dim = vertical_dim
        self.loggy = _logger(loglevel)
        self.loglevel = loglevel
        self.transpose = transpose
        self.remap_area_min = float(remap_area_min)
        if self.remap_area_min < 0.0 or self.remap_area_min > 1.0:
            raise ValueError('The remap_area_min provided must be between 0.0 and 1.0')
        if weights is None:
            raise NotImplementedError(
                "smmregrid_b200 accelerates weight *application*; generate weights with CDO "
                "(reference CdoGenerate) and pass weights=")
        self.init_mode = 'weights'
        self.device = _device_index(device)
        self.out_dtype = None if out_dtype is None else np.dtype(out_dtype)
        if kernel not in _lib.KERNEL_CODES:
            raise ValueError(f"kernel must be one of {sorted(k for k in _lib.KERNEL_CODES if k)} or None")
        # per-Regridder call options (never stored on the shared device handle)
        self.kernel = kernel
        # extension beyond the reference (off by default): time-varying missing values are
        # excluded and the remaining weights renormalised, NaN below `renormalize` valid fraction
        self.renormalize = renormalize
        self.host_block_bytes = int(host_block_bytes)

        mask_dim = mask_dim[0] if isinstance(mask_dim, list) and mask_dim else (None if isinstance(mask_dim, list) else mask_dim)
        w = CdoWeights.from_any(weights, mask_dim=mask_dim)
        self.mask_dim = w.mask_dim if w.is3d else None
        # names GridType extends its defaults with (regrid.py:111-118, 217)
        self.extra_dims = {'mask': _tolist(self.mask_dim if w.is3d else mask_dim),
                           'horizontal': _tolist(horizontal_dims)}
        if w.is3d:
            self.weights_matrix = compute_weights_matrix3d(w, self.mask_dim, device=self.device,
                                                           summation=summation, plan_cache_dir=plan_cache_dir)
        else:
            self.weights_matrix = compute_weights_matrix(w, device=self.device, summation=summation,
                                                         plan_cache_dir=plan_cache_dir)
        # destination mask: precomputed flag or compute it now (regrid.py:196-203)
        if "dst_grid_masked" in w:
            self.masked = np.asarray(w["dst_grid_masked"]).astype(bool)
            if not w.is3d:
                self.masked = bool(self.masked)
        else:
            w = mask_weights(w, self.weights_matrix, self.mask_dim)
            self.masked = check_mask(w, self.mask_dim)
        self.weights = w
        n = w.sizes
        self.n_src, self.n_dst = n["src_grid_size"], n["dst_grid_size"]
        self.src_grid_shape = tuple(int(v) for v in np.atleast_1d(w["src_grid_dims"]))[::-1] \
            if "src_grid_dims" in w else (self.n_src,)
        dgd = tuple(int(v) for v in np.atleast_1d(w["dst_grid_dims"])) if "dst_grid_dims" in w else (self.n_dst,)
        rank = len(dgd)
        if rank == 2:                      # regrid.py:572-574
            self.tgt_shape, self.tgt_dims = (dgd[1], dgd[0]), ["i", "j"]
        elif rank == 1:
            self.tgt_shape, self.tgt_dims = (dgd[0],), ["cell"]
        else:
            raise ValueError('Unknown dimensional target grid')

    # ------------------------------------------------------------------ public API

    def regrid(self, source_data, level_axis: Optional[int] = None, levels: Optional[Sequence[float]] = None,
               packing=None):
        """Regrid an array / DataArray / Dataset (reference: ``regrid.py:233-271``).  ``packing``:
        None, a ``CFPacking`` (raw int16 / uint16 data decoded in the kernels) or ``"cf"`` (each
        DataArray / Dataset variable's packing from its own attributes; unpacked variables as
        without it)."""
        if _is_dataset(source_data):
            # the reference refuses data on several grids when initialised from weights (regrid.py:253-259)
            grids = []
            for name in source_data.data_vars:
                if _is_bounds(name):
                    continue
                key = self._grid_dims(source_data[name].dims)
                if key and key not in grids:
                    grids.append(key)
            if len(grids) > 1 and self.init_mode == 'weights':
                raise ValueError(f'Cannot process data with {len(grids)} GridType initializing from weights')
            out = source_data.map(lambda v: self.regrid_array(v, packing=packing), keep_attrs=True)
            degen = [v for v in out.data_vars if out[v].dims == ()]      # regrid.py:265-266
            out = out.drop_vars(degen)
            if packing is not None:           # (keep_attrs copies the packed variables' attributes back)
                for name in out.data_vars:
                    if _packing_of(source_data[name], packing) is not None:
                        for k in PACKING_ATTRS:
                            out[name].attrs.pop(k, None)
            return out
        if _is_dataarray(source_data):
            return self.regrid_array(source_data, packing=packing)
        if isinstance(source_data, np.ndarray) or _is_tensor(source_data):
            return self.regrid_array(source_data, level_axis=level_axis, levels=levels, packing=packing)
        if isinstance(source_data, dict):
            # plain-array counterpart of Dataset.map (regrid.py:262): one entry per variable;
            # bounds variables are dropped except time bounds (regrid.py:482-490)
            out = {}
            for name, arr in source_data.items():
                if any(sub in str(name) for sub in ("bnds", "bounds", "vertices")):
                    if 'time' in str(name):
                        out[name] = arr
                    continue
                out[name] = self.regrid_array(arr, level_axis=level_axis, levels=levels, packing=packing)
            return out
        raise TypeError('The object provided is not a Xarray object!')

    def regrid_array(self, source_data, level_axis=None, levels=None, packing=None):
        """2-D or 3-D dispatch on the presence of ``mask_dim`` (reference: ``regrid.py:273-312``)."""
        if _is_dataarray(source_data):
            return self._regrid_dataarray(source_data, packing)
        if self.mask_dim:
            return self.regrid3d(source_data, level_axis=level_axis, levels=levels, packing=packing)
        return self.regrid2d(source_data, packing=packing)

    def regrid2d(self, source_data, datagridtype=None, packing=None):
        """Single apply with the 2-D operator (reference: ``regrid.py:429-456``)."""
        if _is_dataarray(source_data):
            return self._regrid_dataarray(source_data, packing)
        return self.apply_weights(source_data, self.weights, weights_matrix=self.weights_matrix,
                                  masked=self.masked, packing=packing)

    def regrid3d(self, source_data, datagridtype=None, level_axis=None, levels=None, out=None, transpose=None,
                 packing=None):
        """Per-level apply for level-varying masks (reference: ``regrid.py:339-427``), issued as
        one grouped launch that writes every level at its final position.  ``transpose``
        overrides ``self.transpose`` for this call; ``out`` (host data only): contiguous numpy
        array that receives the ``[kept..., L, tgt...]`` result."""
        if _is_dataarray(source_data):
            return self._regrid_dataarray(source_data, packing)
        torch = _torch()
        transpose = self.transpose if transpose is None else bool(transpose)
        source_data, opts = self._source(source_data, packing)
        nh = self._n_horizontal_axes(source_data.shape)
        nkept = source_data.ndim - nh
        if nkept < 1:
            raise ValueError(f"3-D weights need a {self.mask_dim} axis in the data")
        la = nkept - 1 if level_axis is None else (level_axis % source_data.ndim)
        if la >= nkept:
            raise ValueError("level_axis must be one of the non-horizontal axes")
        Ld = source_data.shape[la]
        wl = self.weights.levels
        if levels is None:
            if Ld != len(wl):
                raise ValueError(f"data has {Ld} levels, weights {len(wl)}: pass levels= to select")
            levels = wl
        if len(levels) != Ld:
            raise ValueError("levels must have one value per data level")
        widx = np.array([select_level(wl, lev, self.mask_dim) for lev in levels], dtype=np.int32)
        masked = np.ascontiguousarray(np.asarray(self.masked)[widx], dtype=np.uint8)

        was_numpy = isinstance(source_data, np.ndarray)
        x = torch.from_numpy(np.ascontiguousarray(source_data)) if was_numpy else source_data
        host_in = not x.is_cuda
        if host_in:
            return self._regrid3d_host(x, la, nkept, Ld, widx, masked, was_numpy, opts, transpose, out)
        dev = torch.device("cuda", self.device)
        # canonical layout [T, L, n_src]: level axis last among the kept ones
        x = torch.movedim(x, la, nkept - 1)
        kept_shape = tuple(x.shape[:nkept - 1])
        T = int(np.prod(kept_shape)) if kept_shape else 1
        x = x.reshape(T, Ld, self.n_src).contiguous()
        ydt = self._out_torch_dtype(x.dtype)
        if transpose:
            y = torch.empty((T, Ld, self.n_dst), dtype=ydt, device=dev)
            ybs, yls = Ld * self.n_dst, self.n_dst
        else:
            y = torch.empty((Ld, T, self.n_dst), dtype=ydt, device=dev)
            ybs, yls = self.n_dst, T * self.n_dst
        lib = _lib.load()
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.smm_apply_levels(
                self.weights_matrix.handle, Ld, widx.ctypes.data_as(ctypes.c_void_p),
                ctypes.c_void_p(x.data_ptr()), _x_code(x.dtype), T,
                Ld * self.n_src, self.n_src,
                ctypes.c_void_p(y.data_ptr()), _np_dtype_code(_np_of(y.dtype)), ybs, yls,
                masked.ctypes.data_as(ctypes.c_void_p), self.remap_area_min, opts, ctypes.c_void_p(stream)))
        if transpose:           # [kept..., L, tgt...]  (regrid.py:420-427)
            y = y.reshape(kept_shape + (Ld,) + self.tgt_shape)
        else:                   # concat on a new leading axis (regrid.py:410)
            y = y.reshape((Ld,) + kept_shape + self.tgt_shape)
        return y

    def _regrid3d_host(self, x, la, nkept, Ld, widx, masked, was_numpy, opts, transpose, out=None):
        """regrid3d for host data: streamed through the library in chunks of the leading kept
        axes (pinned bounce buffers for pageable arrays), never holding the whole field on the
        device.  ``out`` (numpy ``[T, L, n_dst]``-shaped, contiguous): write the canonical
        ``[kept..., L, n_dst]`` result there instead of allocating."""
        torch = _torch()
        x = torch.movedim(x, la, nkept - 1)                    # canonical [T, L, n_src]
        kept_shape = tuple(x.shape[:nkept - 1])
        T = int(np.prod(kept_shape)) if kept_shape else 1
        x = x.reshape(T, Ld, self.n_src).contiguous()
        if out is not None:
            if not (transpose and out.flags.c_contiguous):
                raise ValueError("out= needs transpose=True and a C-contiguous array")
            y = torch.from_numpy(out.reshape(T, Ld, self.n_dst))
        else:
            y = _pinned_results.take((T, Ld, self.n_dst), self._out_np_dtype())
            if y is None:
                y = torch.from_numpy(_new_host_result((T, Ld, self.n_dst), self._out_np_dtype()))
        _lib.check(_lib.load().smm_apply_levels_host(
            self.weights_matrix.handle, Ld, widx.ctypes.data_as(ctypes.c_void_p),
            ctypes.c_void_p(x.data_ptr()), _x_code(x.dtype), T,
            ctypes.c_void_p(y.data_ptr()), _np_dtype_code(_np_of(y.dtype)),
            masked.ctypes.data_as(ctypes.c_void_p), self.remap_area_min, opts, 0))
        if out is not None:
            return out
        if transpose:           # [kept..., L, tgt...]  (regrid.py:420-427)
            y = y.reshape(kept_shape + (Ld,) + self.tgt_shape)
        else:                   # level axis first, as xarray.concat leaves it (regrid.py:410)
            y = torch.movedim(y, 1, 0).reshape((Ld,) + kept_shape + self.tgt_shape)
        return y.numpy() if was_numpy else y

    def apply_weights(self, source_data, weights=None, weights_matrix=None, masked=True,
                      horizontal_dims=None, level: int = 0, out=None, packing=None):
        """Numeric core of the reference's ``apply_weights`` (``regrid.py:536-584``):
        reshape to ``[kept, n_src]``, non-finite -> 1e20, sparse matmul, destination mask,
        ``dst_grid_frac < remap_area_min``, ``> 1e19 -> NaN``, reshape to the target grid.
        ``out`` (host data only): numpy array of the result's size to write into.  ``packing``: a
        ``CFPacking`` for raw int16 / uint16 data (decoded in the kernels)."""
        if _is_dataarray(source_data):
            return self._regrid_dataarray(source_data, packing)
        torch = _torch()
        wm = weights_matrix if weights_matrix is not None else self.weights_matrix
        parent, lvl = (wm.parent, wm.level) if hasattr(wm, "parent") else (wm, level)
        source_data, opts = self._source(source_data, packing)
        nh = self._n_horizontal_axes(source_data.shape)
        kept_shape = tuple(source_data.shape[:source_data.ndim - nh])
        B = int(np.prod(kept_shape)) if kept_shape else 1
        lib = _lib.load()
        masked = 1 if bool(masked) else 0

        if isinstance(source_data, np.ndarray) or not source_data.is_cuda:
            # host data: chunked H2D -> kernel -> D2H pipeline inside the library
            was_numpy = isinstance(source_data, np.ndarray)
            xt = torch.from_numpy(np.ascontiguousarray(source_data)) if was_numpy else source_data.contiguous()
            xt = xt.reshape(B, self.n_src)
            if out is not None:
                if not out.flags.c_contiguous:
                    raise ValueError("out= must be a C-contiguous array")
                y = torch.from_numpy(out.reshape(B, self.n_dst))
            else:
                # a recycled pinned buffer (the device-to-host copies write it directly), else
                # pageable memory: the library then returns the result through its own pinned bounce
                # buffers -- a pinned allocation per call costs more than that (3.6 ms for 66 MB)
                y = _pinned_results.take((B, self.n_dst), self._out_np_dtype())
                if y is None:
                    y = torch.from_numpy(_new_host_result((B, self.n_dst), self._out_np_dtype()))
            _lib.check(lib.smm_apply_host(
                parent.handle, lvl, ctypes.c_void_p(xt.data_ptr()), _x_code(xt.dtype), B,
                self.n_src, ctypes.c_void_p(y.data_ptr()), _np_dtype_code(_np_of(y.dtype)), self.n_dst,
                masked, self.remap_area_min, opts, 0))
            if out is not None:
                return out
            y = y.reshape(kept_shape + self.tgt_shape)
            return y.numpy() if was_numpy else y

        dev = source_data.device
        x = source_data.reshape(B, self.n_src)
        if not x.is_contiguous():
            x = x.contiguous()
        y = torch.empty((B, self.n_dst), dtype=self._out_torch_dtype(x.dtype), device=dev)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.smm_apply(
                parent.handle, lvl, ctypes.c_void_p(x.data_ptr()), _x_code(x.dtype), B,
                self.n_src, ctypes.c_void_p(y.data_ptr()), _np_dtype_code(_np_of(y.dtype)), self.n_dst,
                masked, self.remap_area_min, opts, ctypes.c_void_p(stream)))
        return y.reshape(kept_shape + self.tgt_shape)

    # ------------------------------------------------------------------ helpers

    def _source(self, data, packing):
        """The data as the kernels read it and the options of the call: floating-point data
        (``_floating``), or with a ``CFPacking`` the raw 16 bits (as int16: the packing says how
        they read) and the options that decode them."""
        if packing is None:
            return self._floating(data), _lib.apply_opts(self.kernel, self.renormalize)
        if isinstance(packing, str):
            raise ValueError('packing="cf" reads the attributes of a DataArray / Dataset variable; '
                             'pass a CFPacking with array data')
        if not isinstance(packing, CFPacking):
            raise TypeError(f"packing must be None, 'cf' or a CFPacking, got {type(packing).__name__}")
        if isinstance(data, np.ndarray) and data.dtype in RAW_DTYPES:
            data = data.view(np.int16)
        elif not (_is_tensor(data) and data.dtype == _torch().int16):
            raise TypeError(f"packed data must be a numpy int16 / uint16 array or a torch int16 tensor, "
                            f"got {getattr(data, 'dtype', type(data).__name__)}")
        return data, _lib.apply_opts(self.kernel, self.renormalize, packing.to_c())

    def _floating(self, data):
        """The reference computes in ``result_type(data, float64 weights)``: integer and bool
        data are promoted to float64 (they hold no missing values), float16 is widened to
        float32 before the 1e20 fill."""
        if isinstance(data, np.ndarray):
            if data.dtype in (np.float32, np.float64):
                return data
            if data.dtype == np.float16:
                return data.astype(np.float32)
            if data.dtype.kind in "iub":
                return data.astype(np.float64)
            raise TypeError(f"cannot regrid data of dtype {data.dtype}")
        torch = _torch()
        if data.dtype in (torch.float32, torch.float64):
            return data
        if data.dtype in (torch.float16, torch.bfloat16):
            return data.to(torch.float32)
        if not data.dtype.is_floating_point and not data.dtype.is_complex:
            return data.to(torch.float64)
        raise TypeError(f"cannot regrid data of dtype {data.dtype}")

    def _out_np_dtype(self):
        return np.dtype(np.float64) if self.out_dtype is None else self.out_dtype

    def _out_torch_dtype(self, x_dtype):
        """Reference output dtype is result_type(data, float64 weights) = float64
        (SURVEY §0.3); ``out_dtype=float32`` rounds once at the store."""
        torch = _torch()
        if self.out_dtype is None:
            return torch.float64
        return torch.float32 if self.out_dtype == np.float32 else torch.float64

    def _n_horizontal_axes(self, shape) -> int:
        shape = tuple(int(s) for s in shape)
        gs = self.src_grid_shape
        if len(shape) >= len(gs) and shape[-len(gs):] == gs:
            return len(gs)
        if len(shape) >= 1 and shape[-1] == self.n_src:
            return 1
        raise KeyError('Dimensions mismatch')          # regrid.py:524

    # ------------------------------------------------------------------ xarray front end

    def _dim_names(self, axis):
        return set(DEFAULT_DIMS[axis]) | set(self.extra_dims.get(axis) or [])

    def _grid_dims(self, dims):
        """``GridType.dims`` of a variable: its horizontal dims + its mask dim (``gridtype.py:55-57``);
        frozen so that grids compare like ``GridType.__eq__``.  More than one mask dim is an error
        (``gridtype.py:165-167``)."""
        hor = [d for d in dims if d in self._dim_names('horizontal')]
        mask = [d for d in dims if d in self._dim_names('mask')]
        if len(mask) > 1:
            raise ValueError(f'Only one masked dimension can be processed at the time: check {mask}')
        return frozenset(hor + mask)

    def _regrid_dataarray(self, da, packing=None):
        """``regrid_array`` + ``regrid2d`` / ``regrid3d`` + the xarray side of ``apply_weights``
        (``regrid.py:273-312, 339-456, 476-626``) for one variable."""
        packing = _packing_of(da, packing)
        name = "" if da.name is None else str(da.name)
        cls = type(da)
        scalars = [k for k, c in da.coords.items() if c.dims == ()]          # regrid.py:289-295
        if scalars:
            self.loggy.warning(
                "Found scalar coordinates %s. If have selected a along a masked dimensions,"
                "regridding might fail. Please consider subsetting with [] or with slice", scalars)
        if _is_bounds(name) or not self._grid_dims(da.dims):
            return cls(data=None)                      # no gridtype: dropped from a Dataset (regrid.py:309-312)
        if any(s in name for s in ("bnds", "bounds", "vertices")):          # regrid.py:482-490
            if 'time' in name:
                self.loggy.info('%s will not be interpolated in the output', name)
                return da
            return cls(data=None)
        hor_names = self._dim_names('horizontal')
        horizontal = [d for d in da.dims if d in hor_names]
        if not horizontal:                             # regrid.py:518-524
            self.loggy.error("None of dimensions on which we can interpolate is found in the DataArray.")
            raise KeyError('Dimensions mismatch')
        lev_dim = None
        if self.mask_dim:
            if self.mask_dim not in da.dims:
                # per-level weights cannot serve a variable without that dimension (a surface field
                # next to 3-D ones): excluded from the output like a variable of another grid
                self.loggy.info('%s will be excluded from the output', name)
                return cls(data=None)
            lev_dim = self.mask_dim
        other = [d for d in da.dims if d not in horizontal and d != lev_dim]
        # the reference reshapes without transposing (regrid.py:538-541): horizontal dims must trail
        order = other + ([lev_dim] if lev_dim else []) + horizontal
        if list(da.dims) != order:
            da = da.transpose(*order)
        sizes = dict(zip(da.dims, da.shape))
        hshape = tuple(sizes[d] for d in horizontal)
        if int(np.prod(hshape)) != self.n_src:
            raise KeyError('Dimensions mismatch')
        levels = None
        if lev_dim:
            levels = np.asarray(da.coords[lev_dim].values if lev_dim in da.coords else self.weights.levels,
                                dtype=np.float64)
            for lev in levels:                         # fail before any work is queued (regrid.py:390-395)
                select_level(self.weights.levels, lev, lev_dim)
        kept_canon = other + ([lev_dim] if lev_dim else [])           # order the numeric core produces
        kept_shape = tuple(sizes[d] for d in kept_canon)
        out_dt = self._out_np_dtype()

        # `.chunks` is None unless the variable is dask-backed; `.data` of a lazily indexed backend
        # array would load the whole field, so it is only touched for dask
        if getattr(da, "chunks", None):
            values = self._dask_apply(da.data, len(horizontal), levels, out_dt, packing)
        else:
            values = self._stream_blocks(da, other, lev_dim, levels, kept_shape, out_dt, packing)
        out_dims = kept_canon
        if lev_dim and not self.transpose:             # level axis first, as xarray.concat leaves it (regrid.py:410)
            values = _moveaxis(values, len(other), 0)
            out_dims = [lev_dim] + other
        return self._dress(cls, da, values, out_dims, drop_packing=packing is not None)

    def _block_apply(self, block, levels, out=None, packing=None):
        """numeric core on one host block laid out ``[other..., (lev,) horizontal...]``; returns /
        fills ``[other..., (lev,) tgt...]``."""
        block = np.asarray(block)
        if packing is None:
            block = self._floating(block)
        n_kept = block.ndim - self._n_horizontal_axes(block.shape)
        if levels is not None:     # level axis last among the kept ones; the caller moves it if asked to
            res = self.regrid3d(block, level_axis=n_kept - 1, levels=levels, out=out, transpose=True, packing=packing)
        else:
            res = self.apply_weights(block, self.weights, weights_matrix=self.weights_matrix, masked=self.masked, out=out,
                                     packing=packing)
        if out is not None:
            return out
        return np.asarray(res).reshape(block.shape[:n_kept] + self.tgt_shape)

    def _stream_blocks(self, da, other, lev_dim, levels, kept_shape, out_dt, packing=None):
        """Host-backed (numpy or lazily indexed) data: blocks of the leading kept dim are read,
        pushed through the device pipeline and written straight into the result, so no more than
        ``host_block_bytes`` of the source is ever held (``regrid.py:538-550`` keeps the field lazy)."""
        out = _new_host_result(kept_shape + self.tgt_shape, out_dt)
        if not other or da.shape[0] <= 1:
            self._block_apply(da.values, levels, out=out, packing=packing)
            return out
        lead, n_lead = other[0], da.shape[0]
        row_bytes = max(1, int(np.prod(da.shape[1:])) * np.dtype(da.dtype).itemsize)
        step = int(max(1, min(n_lead, self.host_block_bytes // row_bytes)))
        for a in range(0, n_lead, step):
            b = min(n_lead, a + step)
            self._block_apply(da.isel({lead: slice(a, b)}).values, levels, out=out[a:b], packing=packing)
        return out

    def _dask_apply(self, data, n_hor, levels, out_dt, packing=None):
        """dask-backed data stays lazy: one ``map_blocks`` task per chunk of the kept dims, each
        feeding the device pipeline (the handle is shared read-only by the worker threads)."""
        import dask.array as dka
        nd = data.ndim
        single = list(range(nd - n_hor, nd)) + ([nd - n_hor - 1] if levels is not None else [])
        data = data.rechunk({ax: -1 for ax in single})
        hor_axes = list(range(nd - n_hor, nd))
        new_axes = list(range(nd - n_hor, nd - n_hor + len(self.tgt_shape)))
        chunks = tuple(data.chunks[:nd - n_hor]) + tuple((n,) for n in self.tgt_shape)
        return dka.map_blocks(lambda blk: self._block_apply(blk, levels, packing=packing).astype(out_dt, copy=False), data,
                              dtype=out_dt, chunks=chunks, drop_axis=hor_axes, new_axis=new_axes,
                              meta=np.empty((0,) * (nd - n_hor + len(self.tgt_shape)), dtype=out_dt))

    def _dress(self, cls, da, values, kept_dims, drop_packing=False):
        """Output DataArray of ``apply_weights`` (``regrid.py:586-626``): kept coordinates, target
        lat/lon (degrees, rounded; degenerate axes removed), ``i/j -> lat/lon`` for regular
        targets, coordinate and variable attributes (``drop_packing``: without the CF packing
        attributes, which xarray moves to ``.encoding`` when it decodes)."""
        w = self.weights
        tgt_dims = list(self.tgt_dims)
        coords = {k: v for k, v in da.coords.items() if set(v.dims).issubset(kept_dims)}
        lat_lon = {}
        if "dst_grid_center_lat" in w and "dst_grid_center_lon" in w:
            scale = 180.0 / math.pi                    # weight lat/lon are in radians
            meta = {"lat": {"units": "degrees_north", "standard_name": "latitude", "axis": "Y"},
                    "lon": {"units": "degrees_east", "standard_name": "longitude", "axis": "X"}}
            for key in ("lat", "lon"):
                centre = np.asarray(w["dst_grid_center_" + key], dtype=np.float64)
                centre = centre.reshape(-1, self.n_dst)[0].reshape(self.tgt_shape)   # 3-D weights: one copy per level
                vals, dims = remove_degenerate_axes(centre, tgt_dims)
                lat_lon[key] = (dims, np.round(vals * scale, 10), meta[key])
            if tgt_dims == ["i", "j"] and lat_lon["lat"][1].ndim == 1 and lat_lon["lon"][1].ndim == 1 \
                    and lat_lon["lat"][0] == ["i"] and lat_lon["lon"][0] == ["j"]:
                tgt_dims = ["lat", "lon"]              # regular grid: drop the 'i' and 'j' dimensions
                lat_lon = {"lat": (["lat"], lat_lon["lat"][1], meta["lat"]),
                           "lon": (["lon"], lat_lon["lon"][1], meta["lon"])}
        for key, (dims, vals, attrs) in lat_lon.items():
            coords[key] = (tuple(dims), vals, attrs)
        attrs = dict(da.attrs)
        attrs.pop('CDI_grid_type', None)               # regrid.py:624
        if drop_packing:
            for k in PACKING_ATTRS:
                attrs.pop(k, None)
        return cls(values, dims=list(kept_dims) + tgt_dims, coords=coords, name=da.name, attrs=attrs)


def regrid(source_data, target_grid=None, weights=None, transpose=True, cdo='cdo', **kwargs):
    """One-shot helper (reference: ``regrid.py:656-677``)."""
    regridder = Regridder(source_data if weights is None else None, target_grid=target_grid,
                          weights=weights, cdo=cdo, transpose=transpose, **kwargs)
    return regridder.regrid(source_data)


def _moveaxis(values, src, dst):
    if _is_dask(values):
        import dask.array as dka
        return dka.moveaxis(values, src, dst)
    return np.moveaxis(values, src, dst)


def _is_tensor(obj) -> bool:
    try:
        return isinstance(obj, _torch().Tensor)
    except ImportError:
        return False


def _packing_of(da, packing):
    """CFPacking of one DataArray: ``packing`` itself, or from its attributes for ``"cf"``."""
    if isinstance(packing, str):
        if packing != "cf":
            raise ValueError(f"packing must be None, 'cf' or a CFPacking, got {packing!r}")
        return CFPacking.from_attrs(da.attrs, da.dtype)
    return packing


def _x_code(torch_dtype) -> int:
    """x_dtype code of the tensor handed to the library (int16: raw CF-packed values, which only
    ``Regridder._source`` lets through)."""
    if torch_dtype == _torch().int16:
        return _lib.SMM_I16
    return _np_dtype_code(_np_of(torch_dtype))


def _np_of(torch_dtype):
    torch = _torch()
    if torch_dtype == torch.float32:
        return np.float32
    if torch_dtype == torch.float64:
        return np.float64
    raise TypeError(f"only float32/float64 data can be regridded, got {torch_dtype}")
