"""CF-packed int16 / uint16 sources decoded inside the kernels (x_dtype SMM_I16, smm_decode).

Every result is compared with the float path of the same handle applied to this file's own numpy
decode of the raw field (xarray's CF decoding: fill values -> NaN, then v * scale + offset in the
decoded dtype D, each operation rounded once): the two must be bit-identical.  The variant list
and its operator recipes are test_gpu_variants.py's, so every compiled kernel variant is reached
with packed sources as well.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))      # refshim

from test_gpu_variants import (BY_ID, KERNEL_COMPACT, KERNEL_GATHER, KERNEL_STAGED, VARIANTS, _create,
                               _diff, _operator, _oracle_result, _same_bits)

F32, F64 = np.float32, np.float64
PACKED_B = (1, 37, 200)


# ------------------------------------------------------------------ the decode, restated in numpy

def np_decode(raw, scale, offset, fills, D, unsigned):
    """xarray's CF decoding of raw 16-bit values: _FillValue / missing_value -> NaN, then the
    scale and offset, each in D."""
    v = raw.view(np.uint16 if unsigned else np.int16)
    x = v.astype(D)
    with np.errstate(over="ignore", invalid="ignore"):
        if scale is not None:
            x = x * D(scale)
        if offset is not None:
            x = x + D(offset)
    if len(fills):
        x[np.isin(v.astype(np.int64), np.asarray(fills, np.int64))] = np.nan
    return x


class Case:
    def __init__(self, name, D, scale=None, offset=None, fills=(), unsigned=False):
        self.name, self.D, self.scale, self.offset, self.fills, self.unsigned = name, D, scale, offset, list(fills), unsigned

    def packing(self):
        from smmregrid_b200 import CFPacking
        return CFPacking(self.scale, self.offset, self.fills, dtype=self.D, unsigned=self.unsigned)

    def decode(self, raw):
        return np_decode(raw, self.scale, self.offset, self.fills, self.D, self.unsigned)

    def __repr__(self):
        return self.name


# 0, 1, 2 and 4 fill values; fills at -32768 and 32767; unsigned data; a negative scale; an absent
# offset (raw 0 times a negative scale is -0.0 and must stay so); a float32 scale whose products
# overflow to +-inf (then filled with 1e20)
CASES_F32 = [Case("f32-scale-offset", F32, np.float32(0.0125), np.float32(250.0), [-32767]),
             Case("f32-unsigned-negscale-nooffset", F32, np.float32(-0.5), None, [1, 2, 3, 65535], unsigned=True),
             Case("f32-overflow", F32, np.float32(3e34), None, [])]
CASES_F64 = [Case("f64-scale-offset", F64, -0.0025, 280.0, [-32768, 32767]),
             Case("f64-unsigned", F64, 0.01, -100.0, [40000], unsigned=True)]


def _raw_field(op, case, B, seed):
    """Raw values over the whole 16-bit range; fill values in scattered cells, in the whole middle
    batch row, and on the zero-weight row's missing source."""
    rng = np.random.default_rng(seed)
    raw = rng.integers(0, 1 << 16, size=(B, op.n_src)).astype(np.uint16)
    if case.fills:
        fv = np.array(case.fills, np.int64) & 0xFFFF
        hit = rng.random(raw.shape) < 0.02
        raw[hit] = fv[rng.integers(len(fv), size=int(hit.sum()))]
        raw[B // 2, :] = fv[0]
        raw[:, op.zero_cols[0]] = fv[-1]
    raw[:, 0] = 0                                   # (-0.0 with a negative scale and no offset)
    return raw.view(np.int16)


def _dev(a, ldx, offset_elems=0):
    """Device copy with row stride ldx, starting offset_elems into its allocation."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a))
    buf = torch.zeros(a.shape[0] * ldx + offset_elems + 8, dtype=t.dtype, device="cuda")
    view = buf[offset_elems:offset_elems + a.shape[0] * ldx].view(a.shape[0], ldx)
    view[:, :a.shape[1]] = t.cuda()
    return buf, view


def _code(dt):
    return 0 if np.dtype(dt) == np.float32 else 1


def _apply(lib, h, op, xview, x_code, ydt, B, ldx, kernel, decode=None, renorm=None, n_dst=None):
    import torch
    from smmregrid_b200 import _lib
    y = torch.full((B, op.n_dst), -7.0, dtype=torch.float64 if ydt == F64 else torch.float32, device="cuda")
    _lib.check(lib.smm_apply(h, 0, xview.data_ptr(), x_code, B, ldx, y.data_ptr(), _code(ydt), op.n_dst,
                             int(op.masked), op.amin, _lib.apply_opts(kernel, renorm, decode), None))
    torch.cuda.synchronize()
    return y.cpu().numpy()


def _ldx(v, op):
    # 2-byte rows: bulk (TMA) copies of the compact path need ldx % 8 == 0; the element variant keeps its odd ldx
    return op.ldx if v.ldx_pad else -(-op.n_src // 8) * 8


def _packed_vs_float(lib, v, op, h, case, ydt, B, seed, kernel=None, renorm=None):
    raw = _raw_field(op, case, B, seed)
    ldx = _ldx(v, op)
    _, xr = _dev(raw, ldx)
    _, xf = _dev(case.decode(raw), ldx)
    k = v.kernel if kernel is None else kernel
    yp = _apply(lib, h, op, xr, 2, ydt, B, ldx, k, case.packing().to_c(), renorm)
    yf = _apply(lib, h, op, xf, _code(case.D), ydt, B, ldx, k, None, renorm)
    return raw, yp, yf


# ------------------------------------------------------------------ every variant

@pytest.mark.gpu
@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_packed_variant_matches_float_path(smm_lib, oracle, cuda, v):
    """int16 / uint16 with D = float32 and float64, y = float32 and float64, B = 1, 37, 200: bit-identical
    to the float path on the numpy decode.  One variant per family is also held to the oracle."""
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    bad = []
    try:
        for i, B in enumerate(PACKED_B):
            for case in (CASES_F32[(i + len(v.id)) % 3], CASES_F64[(i + len(v.id)) % 2]):
                for ydt in (F64, F32):
                    raw, yp, yf = _packed_vs_float(smm_lib, v, op, h, case, ydt, B, seed=len(v.id) * 100 + B)
                    if not _same_bits(yp, yf):
                        bad.append(f"{case} B={B} y={np.dtype(ydt).name}: " + _diff(yp, yf))
                    if ydt == F64 and v.id in ORACLE_IDS and v.ref_order:
                        ref = _oracle_result(oracle, op, case.decode(raw))
                        if not _same_bits(yp, ref):
                            bad.append(f"{case} B={B} oracle: " + _diff(yp, ref))
    finally:
        smm_lib.smm_destroy(h)
    assert not bad, f"{v.id}: " + "; ".join(bad)


# one variant per family (reference-order ones: the oracle is bit-exact there)
ORACLE_IDS = {"staged-l2k14-n256-ord", "staged-packed-n256-ord", "ordered-r64-t1", "gather-ord", "compact-bulk-raw"}


@pytest.mark.gpu
@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_packed_threshold_is_reference_order(smm_lib, oracle, cuda, v):
    """Fill values carrying 10 % of a row's weight decode to NaN, are filled with 1e20 and put the
    row's sum within rounding of 1e19: the NaN decisions (the fast variants' replay decodes the row
    again) and the values near 1e19 are the oracle's, bit for bit."""
    op = _operator(v, "threshold")
    B = 16
    case = Case("threshold", F64, 2000.0 / 65535.0, 1000.0, [-32768])
    rng = np.random.default_rng(len(v.id))
    raw = rng.integers(-32767, 32768, size=(B, op.n_src)).astype(np.int16)
    src0, dst0 = op.src.astype(np.int64) - 1, op.dst.astype(np.int64) - 1
    for b in range(B):
        raw[b, src0[op.nan_link & ((dst0 + b) % 3 != 0)]] = -32768
    x = case.decode(raw)
    ref = _oracle_result(oracle, op, x)
    h = _create(smm_lib, v, op)
    try:
        ldx = _ldx(v, op)
        _, xr = _dev(raw, ldx)
        y = _apply(smm_lib, h, op, xr, 2, F64, B, ldx, v.kernel, case.packing().to_c())
    finally:
        smm_lib.smm_destroy(h)
    near = np.abs(ref - 1e19) < 1e10
    assert near.sum() >= 10 and np.isnan(ref).sum() >= 10, (v.id, int(near.sum()))
    assert np.array_equal(np.isnan(y), np.isnan(ref)), f"{v.id}: NaN decisions, " + _diff(y, ref)
    assert _same_bits(y[near], ref[near]), f"{v.id}: values near 1e19, " + _diff(y[near], ref[near])


RENORM_IDS = ["staged-l1k12-n256-fast", "staged-l4k16-n512-fast", "staged-l2k14-n256-ord", "gather-lpr4", "gather-ord"]


@pytest.mark.gpu
@pytest.mark.parametrize("vid", RENORM_IDS)
def test_packed_renormalize_matches_float_path(smm_lib, cuda, vid):
    """The renormalising extension excludes decoded fill values exactly as it excludes NaN."""
    v = BY_ID[vid]
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    try:
        for case in (CASES_F32[0], CASES_F64[0]):
            for ydt in (F64, F32):
                _, yp, yf = _packed_vs_float(smm_lib, v, op, h, case, ydt, 37, seed=5, renorm=0.3)
                assert _same_bits(yp, yf), f"{vid} {case}: " + _diff(yp, yf)
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ alignment fallbacks

@pytest.mark.gpu
@pytest.mark.parametrize("vid,what", [("staged-l1k12-n256-fast", "x+2B"), ("staged-packed-n256-fast", "x+2B"),
                                      ("staged-l2k14-n256-ord", "ldx%8=4"), ("compact-bulk-raw", "x+2B"),
                                      ("compact-element-raw", "odd-ldx")])
def test_packed_alignment_fallbacks(smm_lib, cuda, vid, what):
    """Rows that are not 16-byte aligned as 2-byte elements (x 2 bytes into its allocation, a row
    stride of 8k + 4 elements, an odd stride) run -- staged levels on the gather kernel, the compact
    path with element copies -- and equal the float path forced to the same kernel family."""
    v = BY_ID[vid]
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    try:
        case = CASES_F32[0]
        B = 37
        raw = _raw_field(op, case, B, 11)
        ldx = {"x+2B": -(-op.n_src // 8) * 8, "ldx%8=4": -(-op.n_src // 8) * 8 + 4, "odd-ldx": op.n_src | 1}[what]
        off = 1 if what == "x+2B" else 0
        _, xr = _dev(raw, ldx, off)
        _, xf = _dev(case.decode(raw), ldx, off)
        family = KERNEL_COMPACT if v.family == "compact" else KERNEL_GATHER
        if v.family != "compact":
            with pytest.raises(ValueError):
                _apply(smm_lib, h, op, xr, 2, F64, B, ldx, KERNEL_STAGED, case.packing().to_c())
        yp = _apply(smm_lib, h, op, xr, 2, F64, B, ldx, None if v.family == "staged" else family, case.packing().to_c())
        yf = _apply(smm_lib, h, op, xf, 0, F64, B, ldx, family)
        assert _same_bits(yp, yf), f"{vid} {what}: " + _diff(yp, yf)
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ host streaming

def _host(a, pinned, keep):
    import torch
    if not pinned:
        return np.ascontiguousarray(a)
    t = torch.empty(a.shape, dtype=torch.from_numpy(np.ascontiguousarray(a)).dtype, pin_memory=True)
    t.numpy()[...] = a
    keep.append(t)
    return t.numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("vid", ["staged-l1k12-n256-fast", "staged-packed-n256-ord", "gather-lpr4", "compact-bulk-raw"])
def test_packed_host_streaming_matches_device_apply(smm_lib, cuda, vid):
    """smm_apply_host with pinned and pageable int16, chunk_rows 0, 1, 7 and B, and a padded ldx:
    equal to the device apply of the same rows."""
    from smmregrid_b200 import _lib
    v = BY_ID[vid]
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    try:
        case = CASES_F32[1]
        dec = case.packing().to_c()
        B = 37
        ldx = -(-op.n_src // 8) * 8 + 8
        raw = _raw_field(op, case, B, 3)
        _, xr = _dev(raw, ldx)
        want = _apply(smm_lib, h, op, xr, 2, F64, B, ldx, v.kernel, dec)
        for pinned in (False, True):
            keep = []
            padded = np.zeros((B, ldx), np.int16)
            padded[:, :op.n_src] = raw
            xh = _host(padded, pinned, keep)
            for chunk in (0, 1, 7, B):
                y = np.full((B, op.n_dst), -7.0)
                _lib.check(smm_lib.smm_apply_host(h, 0, xh.ctypes.data, 2, B, ldx, y.ctypes.data, 1, op.n_dst,
                                                  int(op.masked), op.amin, _lib.apply_opts(v.kernel, None, dec), chunk))
                # chunks of 1 or 7 rows are separate applies: equal for every kernel family, since rows
                # never depend on the batching (test_gpu_variants.test_rows_do_not_depend_on_batching)
                assert _same_bits(y, want), f"{vid} pinned={pinned} chunk={chunk}: " + _diff(y, want)
    finally:
        smm_lib.smm_destroy(h)


@pytest.mark.gpu
def test_packed_split_plan_matches_float_path(smm_lib, cuda):
    """A split plan (short rows packed, the long ones gathered next to the staged launch) with
    packed sources: both launches decode, bit-identical to the float path."""
    import ctypes
    from smmregrid_b200 import _lib
    from test_gpu_levels_host import SPLIT, _split_operator
    from test_gpu_variants import _create_env
    op = _split_operator()
    h = ctypes.c_void_p()
    with _create_env(SPLIT.env):
        _lib.check(smm_lib.smm_create(op.n_src, op.n_dst, op.src.size, op.src.ctypes.data, op.dst.ctypes.data,
                                      op.w.ctypes.data, 1, 1, 0, None, ctypes.byref(h)))
    try:
        _lib.check(smm_lib.smm_set_dst_mask(h, 0, op.imask.ctypes.data, op.frac.ctypes.data))
        inf = _lib.SmmInfo()
        _lib.check(smm_lib.smm_get_info(h, 0, ctypes.byref(inf)))
        assert inf.kernel == KERNEL_STAGED and inf.packed_rows == 1 and inf.gather_rows > 0
        for case in (CASES_F32[0], CASES_F32[1], CASES_F64[0]):
            for B in (1, 37):
                raw = _raw_field(op, case, B, 17)
                _, xr = _dev(raw, op.n_src)
                _, xf = _dev(case.decode(raw), op.n_src)
                for ydt in (F64, F32):
                    yp = _apply(smm_lib, h, op, xr, 2, ydt, B, op.n_src, None, case.packing().to_c())
                    yf = _apply(smm_lib, h, op, xf, _code(case.D), ydt, B, op.n_src, None)
                    assert _same_bits(yp, yf), f"split {case} B={B}: " + _diff(yp, yf)
    finally:
        smm_lib.smm_destroy(h)


@pytest.mark.gpu
def test_packed_levels_host_matches_device_apply(smm_lib, cuda):
    """smm_apply_levels_host with pinned and pageable int16, chunk_rows 0, 1, 7 and B, over a
    repeated level selection: equal to smm_apply_levels of the same rows on the device."""
    import torch
    from smmregrid_b200 import Regridder, _lib, synth
    w3 = synth.ocean3d_weights(36, 18, 12, 6, n_levels=4, seed=3, level_values=[5.0, 15.0, 30.0, 60.0])
    rg = Regridder(weights=w3, remap_area_min=0.5)
    n_src, n_dst = rg.n_src, rg.n_dst
    sel = np.array([3, 2, 0, 0, 1], np.int32)
    masked = np.ascontiguousarray(np.asarray(rg.masked)[sel], dtype=np.uint8)
    case = CASES_F32[1]
    dec = case.packing().to_c()
    opts = _lib.apply_opts(None, None, dec)
    B = 37
    rng = np.random.default_rng(23)
    raw = rng.integers(0, 1 << 16, size=(B, sel.size, n_src)).astype(np.uint16).view(np.int16)
    raw.view(np.uint16)[:, :, ::17] = 65535
    xd = torch.from_numpy(raw).cuda()
    yd = torch.empty((B, sel.size, n_dst), dtype=torch.float64, device="cuda")
    _lib.check(smm_lib.smm_apply_levels(rg.weights_matrix.handle, sel.size, sel.ctypes.data, xd.data_ptr(), 2, B,
                                        sel.size * n_src, n_src, yd.data_ptr(), 1, sel.size * n_dst, n_dst,
                                        masked.ctypes.data, 0.5, opts, None))
    torch.cuda.synchronize()
    want = yd.cpu().numpy()
    # the float path on the decoded field agrees as well
    xf = torch.from_numpy(case.decode(raw)).cuda()
    yf = torch.empty_like(yd)
    _lib.check(smm_lib.smm_apply_levels(rg.weights_matrix.handle, sel.size, sel.ctypes.data, xf.data_ptr(), 0, B,
                                        sel.size * n_src, n_src, yf.data_ptr(), 1, sel.size * n_dst, n_dst,
                                        masked.ctypes.data, 0.5, None, None))
    torch.cuda.synchronize()
    assert _same_bits(want, yf.cpu().numpy())
    for pinned in (False, True):
        keep = []
        xh = _host(raw, pinned, keep)
        for chunk in (0, 1, 7, B):
            y = np.full((B, sel.size, n_dst), -7.0)
            _lib.check(smm_lib.smm_apply_levels_host(rg.weights_matrix.handle, sel.size, sel.ctypes.data, xh.ctypes.data,
                                                     2, B, y.ctypes.data, 1, masked.ctypes.data, 0.5, opts, chunk))
            assert _same_bits(y, want), f"pinned={pinned} chunk={chunk}: " + _diff(y, want)


# ------------------------------------------------------------------ front end

def _front_weights():
    from smmregrid_b200 import synth
    return synth.conservative_latlon(36, 18, 12, 6)


@pytest.mark.gpu
def test_front_end_arrays_and_tensors(smm_lib, cuda):
    """numpy int16 / uint16 and CUDA int16 tensors with a CFPacking: equal to the decoded float
    path, through regrid, regrid2d and apply_weights; other dtypes with a packing raise TypeError."""
    import torch
    from smmregrid_b200 import Regridder
    rg = Regridder(weights=_front_weights(), remap_area_min=0.5)
    rng = np.random.default_rng(1)
    for case in CASES_F32[:2] + CASES_F64[:1]:
        raw = rng.integers(-32768, 32768, size=(5, 18, 36)).astype(np.int16)
        raw.view(np.uint16)[1, 3:7, 10:20] = case.fills[0] & 0xFFFF
        want = rg.regrid(case.decode(raw))
        p = case.packing()
        for got in (rg.regrid(raw, packing=p), rg.regrid(raw.view(np.uint16), packing=p),
                    rg.regrid2d(raw, packing=p), rg.apply_weights(raw, packing=p),
                    rg.regrid(torch.from_numpy(raw).cuda(), packing=p).cpu().numpy()):
            assert _same_bits(np.asarray(got), want), f"{case}: " + _diff(np.asarray(got), want)
    p = CASES_F32[0].packing()
    for bad in (np.zeros((2, 18, 36), np.int8), np.zeros((2, 18, 36), np.int32), np.zeros((2, 18, 36), np.float32),
                torch.zeros((2, 18, 36), dtype=torch.float32, device="cuda")):
        with pytest.raises(TypeError, match="int16"):
            rg.regrid(bad, packing=p)
    with pytest.raises(ValueError, match="cf"):
        rg.regrid(raw, packing="cf")


def _cf_attrs(case):
    """Attributes of a signed packed variable as netCDF stores them."""
    a = {"units": "K", "long_name": "packed"}
    if case.scale is not None:
        a["scale_factor"] = case.scale
    if case.offset is not None:
        a["add_offset"] = case.offset
    if case.fills:
        a["_FillValue"] = np.int16(case.fills[0])
        if len(case.fills) > 1:
            a["missing_value"] = np.array(case.fills[1:], np.int64)
    return a


@pytest.mark.gpu
def test_front_end_dataarray_dataset_lazy_levels(smm_lib, cuda):
    """packing="cf": a raw int16 DataArray equals, bit for bit and in dims, coords and attrs,
    regridding the decoded DataArray without the packing attributes; a Dataset with a packed and a
    float variable; a lazily read DataArray streamed in several blocks; a 3-D variable with levels
    (grouped launches, both layouts, a repeated level selection)."""
    import refshim
    import torch
    from smmregrid_b200 import Regridder, synth
    rg = Regridder(weights=_front_weights(), remap_area_min=0.5)
    case = Case("era5-like", F64, 0.0021, 270.5, [-32767])
    rng = np.random.default_rng(2)
    raw = rng.integers(-32768, 32768, size=(6, 18, 36)).astype(np.int16)
    raw[2, 5:9, :] = -32767
    coords = {"time": np.arange(6.0)}
    attrs = _cf_attrs(case)
    da = refshim.DataArray(raw, ("time", "lat", "lon"), coords=coords, name="t2m", attrs=attrs)
    plain_attrs = {k: v for k, v in attrs.items() if k not in ("scale_factor", "add_offset", "_FillValue",
                                                               "missing_value", "_Unsigned")}
    dec = refshim.DataArray(case.decode(raw), ("time", "lat", "lon"), coords=coords, name="t2m", attrs=plain_attrs)
    got, want = rg.regrid(da, packing="cf"), rg.regrid(dec)
    assert got.dims == want.dims and sorted(got.coords) == sorted(want.coords) and dict(got.attrs) == dict(want.attrs)
    for k in want.coords:
        assert np.array_equal(np.asarray(got.coords[k].data), np.asarray(want.coords[k].data)), k
    assert _same_bits(np.asarray(got.data), np.asarray(want.data)), _diff(np.asarray(got.data), np.asarray(want.data))
    # Dataset: one packed, one float variable
    tas = refshim.DataArray(rng.standard_normal((6, 18, 36)).astype(np.float32), ("time", "lat", "lon"), coords=coords,
                            attrs={"units": "K"})
    out = rg.regrid(refshim.Dataset({"t2m": da, "tas": tas}, attrs={"title": "demo"}), packing="cf")
    assert _same_bits(np.asarray(out["t2m"].data), np.asarray(want.data))
    assert dict(out["t2m"].attrs) == plain_attrs and out["tas"].attrs == {"units": "K"}
    assert _same_bits(np.asarray(out["tas"].data), np.asarray(rg.regrid(tas).data))
    # lazily read, several blocks
    lazy = refshim.LazyDataArray(raw, ("time", "lat", "lon"), coords=coords, name="t2m", attrs=attrs)
    rgb = Regridder(weights=_front_weights(), remap_area_min=0.5, host_block_bytes=2 * 18 * 36 * 2 + 10)
    res = rgb.regrid(lazy, packing="cf")
    assert len(lazy.reads) == 3 and max(lazy.reads) == 2 * 18 * 36 * 2
    assert _same_bits(np.asarray(res.data), np.asarray(want.data))
    # 3-D: levels (grouped launches), both layouts, a repeated selection, host and device data
    w3 = synth.ocean3d_weights(36, 18, 12, 6, n_levels=4, seed=3, level_values=[5.0, 15.0, 30.0, 60.0])
    raw3 = rng.integers(-32768, 32768, size=(3, 5, 18, 36)).astype(np.int16)
    raw3[:, :, 0, :] = -32767
    lev = [30.0, 5.0, 5.0, 60.0, 15.0]
    p = case.packing()
    for transpose in (True, False):
        rg3 = Regridder(weights=w3, remap_area_min=0.5, transpose=transpose)
        want3 = rg3.regrid3d(case.decode(raw3), levels=lev)
        for got3 in (rg3.regrid3d(raw3, levels=lev, packing=p),
                     rg3.regrid3d(torch.from_numpy(raw3).cuda(), levels=lev, packing=p).cpu().numpy()):
            assert _same_bits(np.asarray(got3), np.asarray(want3)), f"transpose={transpose}: " + _diff(got3, want3)
    so = refshim.DataArray(raw3[:, :4], ("time", "lev", "lat", "lon"),
                           coords={"time": np.arange(3.0), "lev": np.array([5.0, 15.0, 30.0, 60.0])}, name="so",
                           attrs=attrs)
    rg3 = Regridder(weights=w3, remap_area_min=0.5)
    got_so = rg3.regrid(so, packing="cf")
    want_so = rg3.regrid3d(case.decode(raw3[:, :4]))
    assert got_so.dims == ("time", "lev", "lat", "lon") and _same_bits(np.asarray(got_so.data), np.asarray(want_so))


@pytest.mark.gpu
def test_abi_rejects_bad_decode(smm_lib, cuda):
    """SMM_I16 without decode, decode with float x, n_fill outside 0-4, a non-finite scale, an
    inexact float32 scale: SMM_ERR_INVALID; SMM_I16 as y_dtype: SMM_ERR_DTYPE."""
    import torch
    from smmregrid_b200 import _lib
    v = BY_ID["staged-l1k12-n256-fast"]
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    try:
        x = torch.zeros((2, op.ldx), dtype=torch.int16, device="cuda")
        y = torch.zeros((2, op.n_dst), dtype=torch.float64, device="cuda")

        def call(x_code, y_code, dec):
            o = _lib.apply_opts(None, None, dec) if dec is not None else None
            return smm_lib.smm_apply(h, 0, x.data_ptr(), x_code, 2, op.ldx, y.data_ptr(), y_code, op.n_dst, 0, 0.0, o, None)

        good = CASES_F32[0].packing().to_c()
        assert call(2, 1, good) == _lib.SMM_OK
        assert call(2, 1, None) == _lib.SMM_ERR_INVALID
        assert call(0, 1, good) == _lib.SMM_ERR_INVALID
        assert call(1, 2, None) == _lib.SMM_ERR_DTYPE
        for field, val in (("n_fill", 5), ("n_fill", -1), ("scale_factor", float("inf")), ("add_offset", float("nan")),
                           ("scale_factor", 0.1), ("dtype", 7)):
            d = CASES_F32[0].packing().to_c()
            setattr(d, field, val)
            assert call(2, 1, d) == _lib.SMM_ERR_INVALID, (field, val)
        torch.cuda.synchronize()
    finally:
        smm_lib.smm_destroy(h)
