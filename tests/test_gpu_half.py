"""float16 and bfloat16 sources read by the kernels (x_dtype SMM_F16 / SMM_BF16).

Contract: every result with half data is bit-identical to the same call on the float32 widening of
that data, for every kernel family, plan kind, summation order, kernel option, the renormalising
extension, grouped levels and host streaming.  The variant list and its operator recipes are
test_gpu_variants.py's, so every compiled kernel variant is reached with half sources as well.
"""
from __future__ import annotations

import copy
import ctypes
import os
import sys
import threading

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))      # refshim

from test_gpu_packed import CASES_F32, RENORM_IDS, _apply, _dev, _host, _ldx
from test_gpu_variants import (BY_ID, KERNEL_COMPACT, KERNEL_GATHER, KERNEL_STAGED, VARIANTS, _create, _diff,
                               _operator, _oracle_result, _same_bits)

F32, F64 = np.float32, np.float64
HALF_B = (1, 37, 200)
KINDS = ("f16", "bf16")
CODE = {"f16": 3, "bf16": 4}

# bit patterns: -0.0, subnormals, the largest finite values, NaN with several payloads, +-inf
SPECIAL = {
    "f16": dict(neg0=0x8000, sub=[0x0001, 0x03FF, 0x8001, 0x83FF], big=[0x7BFF, 0xFBFF],
                nan=[0x7E00, 0xFE00, 0x7C01, 0xFD55], inf=0x7C00, ninf=0xFC00),
    "bf16": dict(neg0=0x8000, sub=[0x0001, 0x007F, 0x8001, 0x807F], big=[0x7F7F, 0xFF7F],
                 nan=[0x7FC0, 0xFFC0, 0x7F81, 0xFF81], inf=0x7F80, ninf=0xFF80),
}


# ------------------------------------------------------------------ half values in numpy

def _to_bits(x32, kind):
    """Finite float32 values rounded to the nearest half value, as uint16 bits."""
    if kind == "f16":
        return x32.astype(np.float16).view(np.uint16)
    u = x32.astype(np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def _widen(bits, kind):
    """The exact float32 widening of half bits."""
    if kind == "f16":
        return bits.view(np.float16).astype(np.float32)
    return (bits.astype(np.uint32) << 16).view(np.float32)


def _half_field(op, kind, B, seed):
    """Both signs, -0.0, subnormals, the largest finite values, NaN with several payloads and +-inf
    in scattered cells, a whole NaN batch row, NaN on the zero-weight row's source."""
    rng = np.random.default_rng(seed)
    bits = _to_bits((100.0 * rng.standard_normal((B, op.n_src))).astype(np.float32), kind)
    sp = SPECIAL[kind]
    u = rng.random(bits.shape)
    p = min(0.02, 0.5 / max(op.max_row, 1))
    for lo, hi, pool in ((0.0, p, sp["nan"]), (p, p + 0.01, sp["sub"] + [sp["neg0"]]), (p + 0.01, p + 0.012, sp["big"])):
        m = (u >= lo) & (u < hi)
        bits[m] = rng.choice(np.array(pool, np.uint16), size=int(m.sum()))
    bits[0, rng.integers(op.n_src)] = sp["inf"]
    bits[B // 2, rng.integers(op.n_src)] = sp["ninf"]
    if B >= 3:
        bits[B // 3, :] = sp["nan"][2]
    if hasattr(op, "zero_cols"):
        bits[:, op.zero_cols[0]] = sp["nan"][1]
    return bits


def _pair(op, kind, B, seed, ldx, off=0):
    """Device copies (row stride ldx) of a half field, `off` elements into its allocation, and of its
    float32 widening (16-byte aligned)."""
    bits = _half_field(op, kind, B, seed)
    _, xh = _dev(bits.view(np.int16), ldx, off)
    _, xf = _dev(_widen(bits, kind), ldx)
    return bits, xh, xf


def _launches(lib, fn):
    n0 = lib.smm_launch_count()
    out = fn()
    return out, lib.smm_launch_count() - n0


# ------------------------------------------------------------------ 1. every variant

@pytest.mark.gpu
@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_half_variant_matches_float32(smm_lib, oracle, cuda, v):
    """float16 and bfloat16, y float64 and float32, B = 1, 37, 200: bit-identical to the float32
    widening with the same kernel option; reference-order variants also equal the oracle."""
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    ldx = _ldx(v, op)
    bad = []
    try:
        for B in HALF_B:
            for kind in KINDS:
                bits, xh, xf = _pair(op, kind, B, len(v.id) * 1000 + B, ldx)
                for ydt in (F64, F32):
                    yh = _apply(smm_lib, h, op, xh, CODE[kind], ydt, B, ldx, v.kernel)
                    yf = _apply(smm_lib, h, op, xf, 0, ydt, B, ldx, v.kernel)
                    if not _same_bits(yh, yf):
                        bad.append(f"{kind} B={B} y={np.dtype(ydt).name}: " + _diff(yh, yf))
                    if ydt == F64 and v.ref_order:
                        ref = _oracle_result(oracle, op, _widen(bits, kind))
                        if not _same_bits(yh, ref):
                            bad.append(f"{kind} B={B} oracle: " + _diff(yh, ref))
    finally:
        smm_lib.smm_destroy(h)
    assert not bad, f"{v.id}: " + "; ".join(bad)


# ------------------------------------------------------------------ 2. the 1e19 threshold

FILL32 = float(np.float32(1e20))          # 1.00000002004e20: the float32 fill as a float64


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_half_threshold_is_float32_fill(smm_lib, oracle, cuda, v, kind):
    """NaN sources carry 10 % of a row's weight, scaled so that the FLOAT32 fill puts the sums within
    rounding of 1e19: the NaN decisions and the values near 1e19 are the oracle's on the float32
    widening, bit for bit (a float64 1e20 fill would leave every such sum 2e11 below 1e19)."""
    op = copy.copy(_operator(v, "threshold"))
    op.__dict__.pop("mat", None)
    op.w = op.w * (1e20 / FILL32)
    B = 16
    rng = np.random.default_rng(len(v.id))
    bits = _to_bits(rng.uniform(0, 2000, size=(B, op.n_src)).astype(np.float32), kind)
    src0, dst0 = op.src.astype(np.int64) - 1, op.dst.astype(np.int64) - 1
    for b in range(B):
        bits[b, src0[op.nan_link & ((dst0 + b) % 3 != 0)]] = SPECIAL[kind]["nan"][b % 4]
    ref = _oracle_result(oracle, op, _widen(bits, kind))
    h = _create(smm_lib, v, op)
    try:
        ldx = _ldx(v, op)
        _, xh = _dev(bits.view(np.int16), ldx)
        y = _apply(smm_lib, h, op, xh, CODE[kind], F64, B, ldx, v.kernel)
    finally:
        smm_lib.smm_destroy(h)
    near = np.abs(ref - 1e19) < 1e10
    assert near.sum() >= 10 and np.isnan(ref).sum() >= 10, (v.id, int(near.sum()))
    assert np.array_equal(np.isnan(y), np.isnan(ref)), f"{v.id}: NaN decisions, " + _diff(y, ref)
    assert _same_bits(y[near], ref[near]), f"{v.id}: values near 1e19, " + _diff(y[near], ref[near])


# ------------------------------------------------------------------ 3. renormalising extension

@pytest.mark.gpu
@pytest.mark.parametrize("vid", RENORM_IDS)
def test_half_renormalize_matches_float32(smm_lib, cuda, vid):
    """The renormalising extension excludes non-finite half sources exactly as float32 ones."""
    v = BY_ID[vid]
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    ldx = _ldx(v, op)
    try:
        for kind in KINDS:
            _, xh, xf = _pair(op, kind, 37, 5, ldx)
            for ydt in (F64, F32):
                yh = _apply(smm_lib, h, op, xh, CODE[kind], ydt, 37, ldx, v.kernel, renorm=0.3)
                yf = _apply(smm_lib, h, op, xf, 0, ydt, 37, ldx, v.kernel, renorm=0.3)
                assert _same_bits(yh, yf), f"{vid} {kind}: " + _diff(yh, yf)
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ 4. family choice and fallback

def _op_variant(vid, what):
    """The variant's parity operator; "nsrc%8=4" drops the last 4 (untouched) source columns."""
    op = _operator(BY_ID[vid], "parity")
    if what == "nsrc%8=4":
        op = copy.copy(op)
        op.__dict__.pop("mat", None)
        op.n_src -= 4
        op.ldx = op.n_src
    return op


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["nsrc%8=4", "ldx%8=4", "x+2B"])
@pytest.mark.parametrize("vid", ["staged-l1k12-n256-fast", "staged-packed-n256-fast", "staged-l2k14-n256-ord",
                                 "ordered-r64-t1"])
def test_half_unstageable_rows_take_float32_family(smm_lib, cuda, vid, what):
    """Staged levels whose 2-byte rows cannot be staged (n_src or the row stride 8k + 4 elements, x
    2 bytes into its allocation) while float32 rows can: automatic and forced-staged calls (and forced
    compact ones, which leave staged levels staged) run the float32 path on widened rows (one
    widening launch more) and equal float32 bit for bit; forced gather calls read the 2-byte rows
    and equal float32 forced the same way."""
    v = BY_ID[vid]
    op = _op_variant(vid, what)
    assert op.n_src % 4 == 0
    h = _create(smm_lib, v, op)
    try:
        ldx = op.n_src + 4 if what == "ldx%8=4" else -(-op.n_src // 8) * 8
        off = 1 if what == "x+2B" else 0
        assert (ldx % 8 == 4) or (op.n_src % 8 == 4) or off
        B = 37
        for kind in KINDS:
            _, xh, xf = _pair(op, kind, B, 7, ldx, off)
            for kernel in (None, KERNEL_STAGED, KERNEL_COMPACT):
                yh, nh = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xh, CODE[kind], F64, B, ldx, kernel))
                yf, nf = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xf, 0, F64, B, ldx, kernel))
                assert _same_bits(yh, yf), f"{vid} {what} {kind} kernel={kernel}: " + _diff(yh, yf)
                assert nh == nf + 1, (nh, nf)
            for kernel in (KERNEL_GATHER,):
                yh, nh = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xh, CODE[kind], F32, B, ldx, kernel))
                yf, nf = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xf, 0, F32, B, ldx, kernel))
                assert _same_bits(yh, yf), f"{vid} {what} {kind} kernel={kernel}: " + _diff(yh, yf)
                assert nh == nf, (nh, nf)
    finally:
        smm_lib.smm_destroy(h)


def _create_plain(lib, n_src, n_dst, src, dst, w):
    from smmregrid_b200 import _lib
    h = ctypes.c_void_p()
    _lib.check(lib.smm_create(n_src, n_dst, src.size, src.ctypes.data, dst.ctypes.data, w.ctypes.data, 1, 1, 0, None,
                              ctypes.byref(h)))
    info = _lib.SmmInfo()
    _lib.check(lib.smm_get_info(h, 0, ctypes.byref(info)))
    return h, info


@pytest.mark.gpu
def test_half_compact_cost_uses_float32_size(smm_lib, cuda):
    """A scattered operator whose compact-path cost lies between the 2-byte and the 4-byte figure
    (1 M random-order sources, 7 500 destinations of 4 links, B = 64): half data takes float32's
    choice, the gather kernel, and equals both the float32 call and the half call forced to gather."""
    rng = np.random.default_rng(42)
    n_src, n_dst, k = 1 << 20, 7500, 4
    src = np.concatenate([np.sort(rng.choice(n_src, size=k, replace=False)) for _ in range(n_dst)]).astype(np.int32) + 1
    dst = np.repeat(np.arange(n_dst, dtype=np.int32), k) + 1
    w = rng.random((src.size, 1))
    h, info = _create_plain(smm_lib, n_src, n_dst, src, dst, w)
    try:
        assert info.kernel == KERNEL_GATHER
        gather_cost = info.nnz * 120.0
        compact = 1.2 * (n_src + info.touched_src + info.nnz)
        assert compact * 2 < gather_cost < compact * 4, (compact, gather_cost)
        op = copy.copy(_operator(BY_ID["gather-lpr4"], "parity"))
        op.n_src, op.n_dst, op.max_row, op.masked, op.amin = n_src, n_dst, k, False, 0.0
        del op.zero_cols
        B = 64
        for kind in KINDS:
            _, xh, xf = _pair(op, kind, B, 9, n_src)
            yh, nh = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xh, CODE[kind], F64, B, n_src, None))
            yf, nf = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xf, 0, F64, B, n_src, None))
            yg = _apply(smm_lib, h, op, xh, CODE[kind], F64, B, n_src, KERNEL_GATHER)
            assert nh == nf == 1, (nh, nf)            # one gather launch, no two-pass launches
            assert _same_bits(yh, yf), f"{kind}: " + _diff(yh, yf)
            assert _same_bits(yh, yg), f"{kind}: " + _diff(yh, yg)
    finally:
        smm_lib.smm_destroy(h)


@pytest.mark.gpu
def test_half_widening_in_several_chunks(smm_lib, cuda):
    """Unstageable 2-byte rows of a large field are widened in bounded chunks (80 rows of 1 M
    sources: two chunks): still equal to the float32 call."""
    n_dst = 1 << 18
    n_src = 4 * n_dst + 4                           # n_src % 8 == 4
    rng = np.random.default_rng(3)
    src = (4 * np.repeat(np.arange(n_dst), 4) + np.tile(np.arange(4), n_dst)).astype(np.int32) + 1
    dst = np.repeat(np.arange(n_dst, dtype=np.int32), 4) + 1
    w = rng.random((src.size, 1))
    h, info = _create_plain(smm_lib, n_src, n_dst, src, dst, w)
    try:
        assert info.kernel == KERNEL_STAGED
        op = copy.copy(_operator(BY_ID["staged-l1k12-n256-fast"], "parity"))
        op.n_src, op.n_dst, op.max_row, op.masked, op.amin = n_src, n_dst, 4, False, 0.0
        del op.zero_cols
        B = 80
        _, xh, xf = _pair(op, "f16", B, 4, n_src)
        yh, nh = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xh, CODE["f16"], F32, B, n_src, None))
        yf, nf = _launches(smm_lib, lambda: _apply(smm_lib, h, op, xf, 0, F32, B, n_src, None))
        assert _same_bits(yh, yf), _diff(yh, yf)
        assert nh > nf + 1, (nh, nf)                # several widening launches and staged applies
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ 5. host streaming, grouped levels

@pytest.mark.gpu
@pytest.mark.parametrize("vid,what", [("staged-l1k12-n256-fast", ""), ("staged-l1k12-n256-fast", "nsrc%8=4"),
                                      ("staged-packed-n256-ord", ""), ("gather-lpr4", ""), ("compact-bulk-raw", "")])
def test_half_host_streaming_matches_device_apply(smm_lib, cuda, vid, what):
    """smm_apply_host with pinned and pageable float16 / bfloat16, chunk_rows 0, 1, 7 and B, and a
    padded ldx: equal to the device apply of the same rows (2 bytes per point over PCIe)."""
    from smmregrid_b200 import _lib
    v = BY_ID[vid]
    op = _op_variant(vid, what)
    h = _create(smm_lib, v, op)
    try:
        B = 37
        ldx = -(-op.n_src // 8) * 8 + 8
        for kind in KINDS:
            bits, xh, xf = _pair(op, kind, B, 3, ldx)
            want = _apply(smm_lib, h, op, xh, CODE[kind], F64, B, ldx, v.kernel)
            assert _same_bits(want, _apply(smm_lib, h, op, xf, 0, F64, B, ldx, v.kernel))
            for pinned in (False, True):
                keep = []
                padded = np.zeros((B, ldx), np.int16)
                padded[:, :op.n_src] = bits.view(np.int16)
                xhost = _host(padded, pinned, keep)
                for chunk in (0, 1, 7, B):
                    y = np.full((B, op.n_dst), -7.0)
                    _lib.check(smm_lib.smm_apply_host(h, 0, xhost.ctypes.data, CODE[kind], B, ldx, y.ctypes.data, 1,
                                                      op.n_dst, int(op.masked), op.amin, _lib.apply_opts(v.kernel), chunk))
                    assert _same_bits(y, want), f"{vid} {kind} pinned={pinned} chunk={chunk}: " + _diff(y, want)
    finally:
        smm_lib.smm_destroy(h)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_half_levels_grouped_and_host(smm_lib, cuda, kind):
    """Grouped 3-D smm_apply_levels with a repeated level selection and strided y (levels first,
    batch rows inside): half data equals its float32 widening; smm_apply_levels_host with pinned and
    pageable half data, chunk_rows 0, 1, 7 and B, equals the device apply."""
    import torch
    from smmregrid_b200 import Regridder, _lib, synth
    w3 = synth.ocean3d_weights(36, 18, 12, 6, n_levels=4, seed=3, level_values=[5.0, 15.0, 30.0, 60.0])
    rg = Regridder(weights=w3, remap_area_min=0.5)
    n_src, n_dst = rg.n_src, rg.n_dst
    sel = np.array([3, 2, 0, 0, 1], np.int32)
    L = sel.size
    masked = np.ascontiguousarray(np.asarray(rg.masked)[sel], dtype=np.uint8)
    B = 37
    op = copy.copy(_operator(BY_ID["staged-l1k12-n256-fast"], "parity"))
    op.n_src, op.max_row = L * n_src, 8
    del op.zero_cols
    bits = _half_field(op, kind, B, 23).reshape(B, L, n_src)
    xh = torch.from_numpy(bits.view(np.int16)).cuda()
    xf = torch.from_numpy(_widen(bits, kind)).cuda()
    hdl = rg.weights_matrix.handle

    def levels(x, code, ybs, yls, shape):
        y = torch.full(shape, -7.0, dtype=torch.float64, device="cuda")
        _lib.check(smm_lib.smm_apply_levels(hdl, L, sel.ctypes.data, x.data_ptr(), code, B, L * n_src, n_src, y.data_ptr(),
                                            1, ybs, yls, masked.ctypes.data, 0.5, None, None))
        torch.cuda.synchronize()
        return y.cpu().numpy()

    for ybs, yls, shape in ((L * n_dst, n_dst, (B, L, n_dst)), (n_dst, B * n_dst, (L, B, n_dst))):
        got, want = levels(xh, CODE[kind], ybs, yls, shape), levels(xf, 0, ybs, yls, shape)
        assert _same_bits(got, want), f"ybs={ybs}: " + _diff(got, want)
    want = levels(xh, CODE[kind], L * n_dst, n_dst, (B, L, n_dst))
    for pinned in (False, True):
        keep = []
        xhost = _host(bits.view(np.int16), pinned, keep)
        for chunk in (0, 1, 7, B):
            y = np.full((B, L, n_dst), -7.0)
            _lib.check(smm_lib.smm_apply_levels_host(hdl, L, sel.ctypes.data, xhost.ctypes.data, CODE[kind], B,
                                                     y.ctypes.data, 1, masked.ctypes.data, 0.5, None, chunk))
            assert _same_bits(y, want), f"pinned={pinned} chunk={chunk}: " + _diff(y, want)


# ------------------------------------------------------------------ 6. front end

class _Spy:
    """Stands in for the loaded library: records the x_dtype of every apply call."""
    X_ARG = {"smm_apply": 3, "smm_apply_host": 3, "smm_apply_levels": 4, "smm_apply_levels_host": 4}

    def __init__(self, lib):
        self._lib, self.codes = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name not in self.X_ARG:
            return fn

        def call(*args):
            self.codes.append(int(args[self.X_ARG[name]]))
            return fn(*args)
        return call


def _np(a):
    import torch
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


@pytest.mark.gpu
def test_front_end_half_inputs(smm_lib, cuda, monkeypatch):
    """numpy float16, torch float16 / bfloat16 on the CPU (pinned and pageable) and on the device,
    contiguous and not: each result equals today's route (regrid of the float32 widening) bit for
    bit, with the same type, dtype and shape, and the library receives the half data itself."""
    import torch
    from smmregrid_b200 import Regridder, _lib, synth
    rg = Regridder(weights=synth.conservative_latlon(36, 18, 12, 6), remap_area_min=0.5)
    rng = np.random.default_rng(1)
    x32 = (280.0 + 20.0 * rng.standard_normal((5, 18, 40))).astype(np.float32)
    x32[1, 3:7, 10:20] = np.nan
    x32[2, 0, 0] = np.inf
    inputs = []
    a16 = x32[..., :36].astype(np.float16)
    inputs.append(("numpy", a16, a16.astype(np.float32)))
    for dt in (torch.float16, torch.bfloat16):
        full = torch.from_numpy(x32).to(dt)
        for where in ("cpu", "pinned", "cuda"):
            t = full.pin_memory() if where == "pinned" else full.cuda() if where == "cuda" else full
            for contiguous in (True, False):
                x = t[..., :36].contiguous() if contiguous else t[..., :36]
                if where == "pinned" and contiguous:
                    x = x.pin_memory()
                assert x.is_contiguous() == contiguous
                inputs.append((f"{dt} {where} contiguous={contiguous}", x, x.float()))
    real = _lib.load()
    for name, x, x_wide in inputs:
        want = rg.regrid(x_wide)
        spy = _Spy(real)
        monkeypatch.setattr(_lib, "load", lambda: spy)
        try:
            got = rg.regrid(x)
        finally:
            monkeypatch.setattr(_lib, "load", lambda: real)
        half_code = _lib.SMM_BF16 if getattr(x, "dtype", None) == torch.bfloat16 else _lib.SMM_F16
        assert spy.codes and set(spy.codes) == {half_code}, (name, spy.codes)
        assert type(got) is type(want) and got.dtype == want.dtype and tuple(got.shape) == tuple(want.shape), name
        if isinstance(got, torch.Tensor):
            assert got.device == want.device, name
        assert _same_bits(_np(got), _np(want)), f"{name}: " + _diff(_np(got), _np(want))


@pytest.mark.gpu
def test_front_end_half_dataarray_dataset_dask(smm_lib, cuda, monkeypatch):
    """A float16 DataArray, a Dataset with a float16 and a float32 variable, and a dask-backed
    float16 DataArray: the same data, dims and coordinates as regridding the float32 widening, and
    the library receives float16 data."""
    import refshim
    from smmregrid_b200 import Regridder, _lib, synth
    rg = Regridder(weights=synth.conservative_latlon(36, 18, 12, 6), remap_area_min=0.5)
    rng = np.random.default_rng(2)
    x16 = (280.0 + 20.0 * rng.standard_normal((6, 18, 36))).astype(np.float16)
    x16[2, 5:9, :] = np.nan
    coords = {"time": np.arange(6.0)}
    da = refshim.DataArray(x16, ("time", "lat", "lon"), coords=coords, name="tas", attrs={"units": "K"})
    da32 = refshim.DataArray(x16.astype(np.float32), ("time", "lat", "lon"), coords=coords, name="tas",
                             attrs={"units": "K"})
    pr = refshim.DataArray(rng.standard_normal((6, 18, 36)).astype(np.float32), ("time", "lat", "lon"), coords=coords)

    def same(got, want, what):
        assert got.dims == want.dims and sorted(got.coords) == sorted(want.coords), what
        for k in want.coords:
            assert np.array_equal(np.asarray(got.coords[k].data), np.asarray(want.coords[k].data)), (what, k)
        g, w = np.asarray(got.data), np.asarray(want.data)
        assert g.dtype == w.dtype and _same_bits(g, w), f"{what}: " + _diff(g, w)

    real = _lib.load()
    spy = _Spy(real)
    want = rg.regrid(da32)
    monkeypatch.setattr(_lib, "load", lambda: spy)
    same(rg.regrid(da), want, "DataArray")
    out = rg.regrid(refshim.Dataset({"tas": da, "pr": pr}, attrs={"title": "demo"}))
    monkeypatch.setattr(_lib, "load", lambda: real)
    same(out["tas"], want, "Dataset tas")
    same(out["pr"], rg.regrid(pr), "Dataset pr")
    assert _lib.SMM_F16 in spy.codes and set(spy.codes) <= {_lib.SMM_F16, _lib.SMM_F32}, spy.codes
    refshim.install_fake_dask()
    try:
        lazy = refshim.FakeDaskArray(x16, chunks=((2, 4), (18,), (36,)))
        dl = refshim.DataArray(lazy, ("time", "lat", "lon"), coords=coords, name="tas")
        spy = _Spy(real)
        monkeypatch.setattr(_lib, "load", lambda: spy)
        res = rg.regrid(dl)
        y = res.data.compute()
        monkeypatch.setattr(_lib, "load", lambda: real)
        assert res.dims == ("time", "lat", "lon") and set(spy.codes) == {_lib.SMM_F16}, spy.codes
        assert _same_bits(y, np.asarray(want.data)), _diff(y, np.asarray(want.data))
    finally:
        for m in ("dask", "dask.array"):
            sys.modules.pop(m, None)


# ------------------------------------------------------------------ 7. concurrency

@pytest.mark.gpu
def test_half_widening_concurrent_streams(smm_lib, cuda):
    """Two threads on two streams apply one handle to misaligned float16 data (x 2 bytes into its
    allocation), so both take float32 copies from the handle's pool: bit-identical to serial calls."""
    import torch
    from smmregrid_b200 import _lib
    v = BY_ID["staged-l1k12-n256-fast"]
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    try:
        B, ldx = 200, op.n_src
        xs = [_pair(op, "f16", B, 30 + i, ldx, 1)[1] for i in range(2)]
        serial = [_apply(smm_lib, h, op, x, CODE["f16"], F64, B, ldx, None) for x in xs]
        streams = [torch.cuda.Stream() for _ in xs]
        ys = [[torch.full((B, op.n_dst), -7.0, dtype=torch.float64, device="cuda") for _ in range(6)] for _ in xs]
        torch.cuda.synchronize()
        errors = []

        def work(i):
            try:
                for y in ys[i]:
                    _lib.check(smm_lib.smm_apply(h, 0, xs[i].data_ptr(), CODE["f16"], B, ldx, y.data_ptr(), 1, op.n_dst,
                                                 int(op.masked), op.amin, None, ctypes.c_void_p(streams[i].cuda_stream)))
            except BaseException as e:          # reported by the main thread
                errors.append(e)

        threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        torch.cuda.synchronize()
        assert not errors, errors
        for i in range(2):
            for y in ys[i]:
                assert _same_bits(y.cpu().numpy(), serial[i]), f"thread {i}: " + _diff(y.cpu().numpy(), serial[i])
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ 8. ABI

@pytest.mark.gpu
def test_half_abi_errors(smm_lib, cuda):
    """A half y_dtype: TypeError; a decode with SMM_F16 data: ValueError; smm_nan_variation with the
    half codes: TypeError."""
    import torch
    from smmregrid_b200 import _lib
    v = BY_ID["staged-l1k12-n256-fast"]
    op = _operator(v, "parity")
    h = _create(smm_lib, v, op)
    try:
        x = torch.zeros((2, op.ldx), dtype=torch.float16, device="cuda")
        y = torch.zeros((2, op.n_dst), dtype=torch.float64, device="cuda")

        def call(x_code, y_code, opts=None):
            _lib.check(smm_lib.smm_apply(h, 0, x.data_ptr(), x_code, 2, op.ldx, y.data_ptr(), y_code, op.n_dst, 0, 0.0,
                                         opts, None))

        call(_lib.SMM_F16, _lib.SMM_F64)
        call(_lib.SMM_BF16, _lib.SMM_F32)
        for yc in (_lib.SMM_F16, _lib.SMM_BF16):
            with pytest.raises(TypeError):
                call(_lib.SMM_F16, yc)
        for xc in (_lib.SMM_F16, _lib.SMM_BF16):
            with pytest.raises(ValueError):
                call(xc, _lib.SMM_F64, _lib.apply_opts(None, None, CASES_F32[0].packing().to_c()))
            count = ctypes.c_int64(-1)
            with pytest.raises(TypeError):
                _lib.check(smm_lib.smm_nan_variation(x.data_ptr(), xc, 1, 2, op.ldx, ctypes.byref(count), None))
        torch.cuda.synchronize()
    finally:
        smm_lib.smm_destroy(h)
