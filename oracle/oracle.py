"""CPU ORACLE for the smmregrid weight-application hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package
(``smmregrid_b200``) never does.

PARITY STATUS: **parity unpinned** at the sparse/dask boundary.  The reference's
arithmetic lives in pydata ``sparse`` + ``dask`` (unpinned in
``/root/reference/pyproject.toml:26,29``), neither installable here, and the reference
holds no golden vectors (all its numeric tests call the ``cdo`` binary).  What is pinned:
``tests/golden/make_golden.py`` executes the reference's *own* ``smmregrid/weights.py``
source under numpy-backed stand-ins for ``dask``/``sparse`` and stores the outputs; this
module and ``smm_oracle.c`` are checked against those fixtures and against each other.

Two independent restatements live here:

* ``*_np``   -- numpy/scipy, literal transcription of the reference call sites with
  ``dask.array`` -> ``numpy`` and ``sparse.COO`` -> explicit sorted/deduplicated COO.
* ``*_c``    -- ctypes calls into ``libsmm_oracle.so`` (``smm_oracle.c``), the loop-order
  faithful port that is also the timed CPU baseline.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

FILL = 1e20          # np.ma default float fill value (regrid.py:545)
THRESH = 1e19        # regrid.py:570


def build(force: bool = False) -> str:
    """Compile ``libsmm_oracle.so`` with the committed Makefile (gcc)."""
    so = os.path.join(_HERE, "libsmm_oracle.so")
    src = os.path.join(_HERE, "smm_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return so


def _lib():
    """The library as it is when present: bench.py may run from a read-only tree, so rebuilding a
    stale one is left to build() (__graft_entry__.build() and the test fixture call it)."""
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "libsmm_oracle.so")
        lib = ctypes.CDLL(so if os.path.exists(so) else build())
        i64, i32p, f64p, vp = ctypes.c_int64, ctypes.POINTER(ctypes.c_int32), \
            ctypes.POINTER(ctypes.c_double), ctypes.c_void_p
        lib.orc_coo_build.restype = i64
        lib.orc_coo_build.argtypes = [i64, i64, i64, i32p, i32p, f64p, ctypes.c_int,
                                      ctypes.c_int, i32p, i32p, f64p]
        lib.orc_mask_sum.restype = None
        lib.orc_mask_sum.argtypes = [i64, i64, i32p, i32p, f64p, i32p, i32p, f64p]
        lib.orc_apply.restype = ctypes.c_int
        lib.orc_apply.argtypes = [i64, i64, i64, i32p, i32p, f64p, vp, ctypes.c_int, i64, i64,
                                  f64p, i64, i32p, f64p, ctypes.c_double, ctypes.c_int]
        _LIB = lib
    return _LIB


def _p(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


class CooMatrix:
    """What ``sparse.COO([src, dst], w, shape=(n_src, n_dst))`` holds after construction:
    coordinates sorted src-major, duplicates summed (weights.py:37-39)."""

    def __init__(self, src, dst, w, n_src, n_dst):
        self.src = np.ascontiguousarray(src, dtype=np.int32)
        self.dst = np.ascontiguousarray(dst, dtype=np.int32)
        self.w = np.ascontiguousarray(w, dtype=np.float64)
        self.shape = (int(n_src), int(n_dst))

    @property
    def nnz(self):
        return self.w.size

    def todense(self):
        d = np.zeros(self.shape, dtype=np.float64)
        np.add.at(d, (self.src, self.dst), self.w)
        return d


# --------------------------------------------------------------------------- weights.py


def compute_weights_matrix_np(src_address, dst_address, remap_matrix, n_src, n_dst):
    """weights.py:25-44 with sparse.COO semantics restated in numpy."""
    src = np.asarray(src_address).astype(np.int64) - 1          # weights.py:31
    dst = np.asarray(dst_address).astype(np.int64) - 1          # weights.py:32
    rm = np.asarray(remap_matrix, dtype=np.float64)
    w = rm[:, 0] if rm.ndim == 2 else rm                         # weights.py:33
    if src.size and (src.min() < 0 or src.max() >= n_src or dst.min() < 0 or dst.max() >= n_dst):
        raise ValueError("address out of range")
    lin = src * n_dst + dst
    order = np.argsort(lin, kind="stable")
    lin, w = lin[order], w[order]
    if lin.size:
        first = np.concatenate(([True], lin[1:] != lin[:-1]))
        starts = np.flatnonzero(first)
        # np.add.reduceat is pairwise for long runs; duplicates are sequentially summed here
        wsum = np.empty(starts.size, dtype=np.float64)
        ends = np.concatenate((starts[1:], [lin.size]))
        simple = (ends - starts) == 1
        wsum[simple] = w[starts[simple]]
        for i in np.flatnonzero(~simple):
            acc = 0.0
            for v in w[starts[i]:ends[i]]:
                acc = acc + v
            wsum[i] = acc
        lin = lin[starts]
        w = wsum
    return CooMatrix(lin // n_dst, lin % n_dst, w, n_src, n_dst)


def compute_weights_matrix_c(src_address, dst_address, remap_matrix, n_src, n_dst):
    src_address = np.ascontiguousarray(src_address, dtype=np.int32)
    dst_address = np.ascontiguousarray(dst_address, dtype=np.int32)
    rm = np.ascontiguousarray(remap_matrix, dtype=np.float64)
    num_wgts = rm.shape[1] if rm.ndim == 2 else 1
    nnz = src_address.size
    s = np.empty(nnz, np.int32); d = np.empty(nnz, np.int32); w = np.empty(nnz, np.float64)
    m = _lib().orc_coo_build(n_src, n_dst, nnz, _p(src_address, ctypes.c_int32),
                             _p(dst_address, ctypes.c_int32), _p(rm, ctypes.c_double),
                             num_wgts, 1, _p(s, ctypes.c_int32), _p(d, ctypes.c_int32),
                             _p(w, ctypes.c_double))
    if m < 0:
        raise ValueError("address out of range")
    return CooMatrix(s[:m].copy(), d[:m].copy(), w[:m].copy(), n_src, n_dst)


def compute_weights_matrix3d_np(src_address, dst_address, remap_matrix, link_length, n_src, n_dst,
                                builder=None):
    """weights.py:7-23: level i uses links [0:link_length[i]) of the padded [L, nl_max] arrays."""
    builder = builder or compute_weights_matrix_np
    out = []
    for i, nl in enumerate(np.asarray(link_length)):
        nl = int(nl)
        out.append(builder(src_address[i, :nl], dst_address[i, :nl], remap_matrix[i, :nl],
                           n_src, n_dst))
    return out


def mask_tensordot_np(src_mask, mat: CooMatrix):
    """weights.py:47-52."""
    t = np.zeros(mat.shape[1], dtype=np.float64)
    prod = np.asarray(src_mask)[mat.src].astype(np.float64) * mat.w
    for k in range(mat.nnz):                         # COO order accumulation (small cases only)
        t[mat.dst[k]] += prod[k]
    return np.where(t < 0.5, 0, 1).astype(np.int32), t


def mask_tensordot_c(src_mask, mat: CooMatrix):
    src_mask = np.ascontiguousarray(src_mask, dtype=np.int32)
    out = np.empty(mat.shape[1], np.int32)
    t = np.empty(mat.shape[1], np.float64)
    _lib().orc_mask_sum(mat.shape[1], mat.nnz, _p(mat.src, ctypes.c_int32),
                        _p(mat.dst, ctypes.c_int32), _p(mat.w, ctypes.c_double),
                        _p(src_mask, ctypes.c_int32), _p(out, ctypes.c_int32),
                        _p(t, ctypes.c_double))
    return out, t


def check_mask_np(dst_grid_imask):
    """weights.py:103-120: scalar for 2-D, bool[L] for [L, n_dst]."""
    m = np.asarray(dst_grid_imask)
    if m.ndim == 2:
        return ~(m == 1).all(axis=1)
    return bool(~(m == 1).all())


# ---------------------------------------------------------------------------- regrid.py


def apply_weights_np(x, mat: CooMatrix, dst_imask=None, dst_frac=None, remap_area_min=0.5,
                     masked=True):
    """regrid.py:536-570 with dask.array -> numpy and the sparse matmul through scipy CSR.

    x: [..., n_src] float32/float64.  Returns [..., n_dst] in result_type(x, float64).
    Summation order differs from the reference loop (scipy CSR), so use the C version
    when bit-level agreement of the `> 1e19` decision matters.
    """
    import scipy.sparse as sp

    x = np.asarray(x)
    kept = x.shape[:-1]
    xa = x.reshape(-1, x.shape[-1])
    xa = np.ma.filled(np.ma.fix_invalid(xa))                         # :545-547
    W = sp.csr_matrix((mat.w, (mat.src, mat.dst)), shape=mat.shape)
    y = np.asarray((W.T @ xa.astype(np.result_type(xa.dtype, np.float64)).T).T)  # :550
    if masked:
        y = np.where(np.asarray(dst_imask).reshape(1, -1).astype(bool), y, np.nan)  # :553-559
    if remap_area_min > 0.0:
        y = np.where(np.broadcast_to(dst_frac, y.shape) < remap_area_min, np.nan, y)  # :562-565
    with np.errstate(invalid="ignore"):
        y = np.where(y > THRESH, np.nan, y)                           # :570
    return y.reshape(kept + (mat.shape[1],))


def apply_weights_c(x, mat: CooMatrix, dst_imask=None, dst_frac=None, remap_area_min=0.5,
                    masked=True, nthreads=1, out=None):
    """Loop-order faithful port (smm_oracle.c: orc_apply)."""
    x = np.asarray(x)
    if x.dtype not in (np.float32, np.float64):
        raise TypeError("float32/float64 only")
    kept = x.shape[:-1]
    xa = np.ascontiguousarray(x.reshape(-1, x.shape[-1]))
    B = xa.shape[0]
    n_src, n_dst = mat.shape
    assert xa.shape[1] == n_src
    y = out if out is not None else np.empty((B, n_dst), dtype=np.float64)
    im = None
    if masked:
        im = np.ascontiguousarray(dst_imask, dtype=np.int32)
    fr = None
    if remap_area_min > 0.0:
        fr = np.ascontiguousarray(dst_frac, dtype=np.float64)
    rc = _lib().orc_apply(n_src, n_dst, mat.nnz, _p(mat.src, ctypes.c_int32),
                          _p(mat.dst, ctypes.c_int32), _p(mat.w, ctypes.c_double),
                          xa.ctypes.data_as(ctypes.c_void_p), 0 if xa.dtype == np.float32 else 1,
                          B, n_src, _p(y, ctypes.c_double), n_dst,
                          _p(im, ctypes.c_int32) if im is not None else None,
                          _p(fr, ctypes.c_double) if fr is not None else None,
                          float(remap_area_min), int(nthreads))
    if rc != 0:
        raise RuntimeError("orc_apply failed")
    return y.reshape(kept + (n_dst,))


def select_level_np(weight_levels, lev, tol=1e-3):
    """regrid.py:386-395: pandas Index.get_indexer([lev], method='nearest', tolerance=1e-3)."""
    wl = np.asarray(weight_levels, dtype=np.float64)
    d = np.abs(wl - float(lev))
    widx = int(np.argmin(d))            # first minimum; pandas picks the larger index only on exact ties
    if not d[widx] <= tol:
        raise ValueError(f"{lev} not found in mask_dim. Available levels: {list(wl)}")
    return widx


def regrid3d_np(x, level_axis, data_levels, weight_levels, mats, dst_imask, dst_frac, masked,
                remap_area_min=0.5, apply=apply_weights_c):
    """regrid.py:387-427: per-level apply, concat on a new axis 0, then move that axis to just
    before the horizontal one (transpose=True).  x: [..., L_data, ..., n_src]."""
    x = np.asarray(x)
    outs = []
    for idx, lev in enumerate(data_levels):
        widx = select_level_np(weight_levels, lev)
        xa = np.take(x, idx, axis=level_axis)
        fr = dst_frac[widx] if np.ndim(dst_frac) == 2 else dst_frac
        outs.append(apply(xa, mats[widx], dst_imask[widx], fr, remap_area_min, bool(masked[widx])))
    y = np.stack(outs, axis=0)
    return np.moveaxis(y, 0, -2)


def apply_weights_renorm_np(x, mat: CooMatrix, dst_imask=None, dst_frac=None, remap_area_min=0.5,
                            masked=True, min_valid=0.5):
    """Checker for the opt-in renormalising EXTENSION (not reference behaviour): non-finite
    sources are excluded; a destination that saw missing sources becomes
    sum_valid(w x) * sum_all(w) / sum_valid(w), or NaN when |sum_valid(w)| < min_valid*|sum_all(w)|;
    destinations without missing sources keep the plain sum."""
    import scipy.sparse as sp
    x = np.asarray(x)
    kept = x.shape[:-1]
    xa = x.reshape(-1, x.shape[-1]).astype(np.float64)
    fin = np.isfinite(xa)
    W = sp.csr_matrix((mat.w, (mat.src, mat.dst)), shape=mat.shape).T.tocsr()
    wx = np.asarray((W @ np.where(fin, xa, 0.0).T).T)
    wv = np.asarray((W @ fin.astype(np.float64).T).T)
    wa = np.asarray(W @ np.ones(mat.shape[0]))[None, :]
    missing = np.asarray((abs(W) @ (~fin).astype(np.float64).T).T) > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        ren = np.where((np.abs(wv) >= min_valid * np.abs(wa)) & (wv != 0), wx * (wa / wv), np.nan)
    y = np.where(missing, ren, wx)
    if masked:
        y = np.where(np.asarray(dst_imask).reshape(1, -1).astype(bool), y, np.nan)
    if remap_area_min > 0.0:
        y = np.where(np.broadcast_to(dst_frac, y.shape) < remap_area_min, np.nan, y)
    return y.reshape(kept + (mat.shape[1],))


def nan_variation_count_np(field, axis):
    """util.py:75-78: `nan_mask.astype("int8").diff(dim).astype(bool).any(dim).sum()`."""
    nan_mask = np.isnan(np.asarray(field))
    if nan_mask.shape[axis] < 2:
        return 0
    return int(np.diff(nan_mask.astype(np.int8), axis=axis).astype(bool).any(axis=axis).sum())


def detect_nan_variation_dims_np(field, time_axis, check_axes):
    """util.py:57-85 on a bare array: drop the time axis at its first step (util.py:69-71), then
    report the members of check_axes (numbered on the ORIGINAL array) with count > 0."""
    field = np.asarray(field)
    out = []
    if time_axis is not None:
        field = np.take(field, 0, axis=time_axis)
    for d in check_axes:
        ax = d
        if time_axis is not None:
            if d == time_axis:
                continue
            ax = d - (d > time_axis)
        if nan_variation_count_np(field, ax) > 0:
            out.append(d)
    return out
