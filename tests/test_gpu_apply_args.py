"""Argument checks of the four apply entry points (smm_apply, smm_apply_levels, smm_apply_host,
smm_apply_levels_host).

Each row of the table below is one call with a single invalid argument; every other argument is
that of a call that succeeds.  The call must return the row's SMM_ERR_* code, smm_last_error()
must contain the row's message, and y must be left as it was.  Calls with B == 0 or n_sel == 0
must return SMM_OK whatever the data pointers are, and leave y alone.

The handles have two levels and no destination mask or area fraction set, so that a masked call
or a remap_area_min > 0 is a fault; one has staged plans, the other gather-family plans.
"""
from __future__ import annotations

import ctypes
import math

import numpy as np
import pytest

from test_gpu_variants import BY_ID, KERNEL_GATHER, KERNEL_STAGED, _create_env, _operator

SMM_OK, SMM_ERR_INVALID, SMM_ERR_DTYPE = 0, 1, 5
SMM_F32, SMM_F64, SMM_I16, SMM_F16, SMM_BF16 = 0, 1, 2, 3, 4
B = 3
SENTINEL = -7.0
N_LEVELS = 2

SINGLE = ("smm_apply", "smm_apply_host")
GROUPED = ("smm_apply_levels", "smm_apply_levels_host")
ENTRY_POINTS = SINGLE + GROUPED

GOOD_DECODE = dict(dtype=SMM_F64, is_unsigned=0, scale_factor=1.0, add_offset=0.0, n_fill=0)


def _dec(**fields):
    return dict(x_dtype=SMM_I16, decode={**GOOD_DECODE, **fields})


BAD_X = "x_dtype must be SMM_F32 (0)"
BAD_Y = "y_dtype SMM_F32 or SMM_F64"
BAD_KERNEL = "smm_apply_opts.kernel must be 0, SMM_KERNEL_STAGED, SMM_KERNEL_GATHER or SMM_KERNEL_COMPACT"
BAD_FRACTION = "smm_apply_opts.min_valid_fraction must be within [0, 1]"
ONLY_I16 = "smm_apply_opts.decode is only valid with x_dtype SMM_I16"
BAD_N_FILL = "smm_decode.n_fill must be within [0, 4]"
NOT_FINITE = "smm_decode.scale_factor and add_offset must be finite"
BAD_AREA = "The remap_area_min provided must be between 0.0 and 1.0"
NULL_SINGLE, NULL_GROUPED = "null x or y", "null level_index, x or y"

# (id, entry points, arguments that differ from a good call, code, message)
FAULTS = [
    ("null-handle", ENTRY_POINTS, dict(h=None), SMM_ERR_INVALID, "null handle"),
    ("level-past-end", SINGLE, dict(level=2), SMM_ERR_INVALID, "level 2 out of range [0, 2)"),
    ("level-negative", SINGLE, dict(level=-1), SMM_ERR_INVALID, "level -1 out of range [0, 2)"),
    ("level-index-past-end", GROUPED, dict(level_index=[0, 2]), SMM_ERR_INVALID, "level 2 out of range [0, 2)"),
    ("level-index-negative", GROUPED, dict(level_index=[-1, 1]), SMM_ERR_INVALID, "level -1 out of range [0, 2)"),
    ("x-dtype-5", ENTRY_POINTS, dict(x_dtype=5), SMM_ERR_DTYPE, BAD_X),
    ("x-dtype-negative", ENTRY_POINTS, dict(x_dtype=-1), SMM_ERR_DTYPE, BAD_X),
    ("y-dtype-i16", ENTRY_POINTS, dict(y_dtype=SMM_I16), SMM_ERR_DTYPE, BAD_Y),
    ("y-dtype-f16", ENTRY_POINTS, dict(y_dtype=SMM_F16), SMM_ERR_DTYPE, BAD_Y),
    ("y-dtype-bf16", ENTRY_POINTS, dict(y_dtype=SMM_BF16), SMM_ERR_DTYPE, BAD_Y),
    ("y-dtype-5", ENTRY_POINTS, dict(y_dtype=5), SMM_ERR_DTYPE, BAD_Y),
    ("kernel-4", ENTRY_POINTS, dict(kernel=4), SMM_ERR_INVALID, BAD_KERNEL),
    ("kernel-negative", ENTRY_POINTS, dict(kernel=-1), SMM_ERR_INVALID, BAD_KERNEL),
    ("min-valid-negative", ENTRY_POINTS, dict(renormalize=-0.1), SMM_ERR_INVALID, BAD_FRACTION),
    ("min-valid-above-1", ENTRY_POINTS, dict(renormalize=1.5), SMM_ERR_INVALID, BAD_FRACTION),
    ("min-valid-nan", ENTRY_POINTS, dict(renormalize=math.nan), SMM_ERR_INVALID, BAD_FRACTION),
    ("i16-without-decode", ENTRY_POINTS, dict(x_dtype=SMM_I16), SMM_ERR_INVALID,
     "x_dtype SMM_I16 needs smm_apply_opts.decode"),
    ("decode-with-f32", ENTRY_POINTS, dict(decode=GOOD_DECODE), SMM_ERR_INVALID, ONLY_I16),
    ("decode-with-f16", ENTRY_POINTS, dict(x_dtype=SMM_F16, decode=GOOD_DECODE), SMM_ERR_INVALID, ONLY_I16),
    ("decode-dtype", ENTRY_POINTS, _dec(dtype=7), SMM_ERR_INVALID, "smm_decode.dtype must be SMM_F32 or SMM_F64"),
    ("decode-n-fill-5", ENTRY_POINTS, _dec(n_fill=5), SMM_ERR_INVALID, BAD_N_FILL),
    ("decode-n-fill-negative", ENTRY_POINTS, _dec(n_fill=-1), SMM_ERR_INVALID, BAD_N_FILL),
    ("decode-scale-inf", ENTRY_POINTS, _dec(scale_factor=math.inf), SMM_ERR_INVALID, NOT_FINITE),
    ("decode-offset-nan", ENTRY_POINTS, _dec(add_offset=math.nan), SMM_ERR_INVALID, NOT_FINITE),
    ("decode-inexact-f32", ENTRY_POINTS, _dec(dtype=SMM_F32, scale_factor=0.1), SMM_ERR_INVALID,
     "smm_decode: scale_factor and add_offset must be exact float32 values when dtype is SMM_F32"),
    ("B-negative", SINGLE, dict(B=-1), SMM_ERR_INVALID, "B must be >= 0"),
    ("B-negative", GROUPED, dict(B=-1), SMM_ERR_INVALID, "n_sel and B must be >= 0"),
    ("n-sel-negative", GROUPED, dict(n_sel=-1), SMM_ERR_INVALID, "n_sel and B must be >= 0"),
    ("null-x", SINGLE, dict(x=None), SMM_ERR_INVALID, NULL_SINGLE),
    ("null-x", GROUPED, dict(x=None), SMM_ERR_INVALID, NULL_GROUPED),
    ("null-y", SINGLE, dict(y=None), SMM_ERR_INVALID, NULL_SINGLE),
    ("null-y", GROUPED, dict(y=None), SMM_ERR_INVALID, NULL_GROUPED),
    ("null-level-index", GROUPED, dict(level_index=None), SMM_ERR_INVALID, NULL_GROUPED),
    ("ldx-short", SINGLE, dict(ldx=-1), SMM_ERR_INVALID, "ldx < n_src or ldy < n_dst"),
    ("ldy-short", SINGLE, dict(ldy=-1), SMM_ERR_INVALID, "ldx < n_src or ldy < n_dst"),
    ("area-min-negative", ENTRY_POINTS, dict(remap_area_min=-0.1), SMM_ERR_INVALID, BAD_AREA),
    ("area-min-above-1", ENTRY_POINTS, dict(remap_area_min=1.5), SMM_ERR_INVALID, BAD_AREA),
    ("area-min-nan", ENTRY_POINTS, dict(remap_area_min=math.nan), SMM_ERR_INVALID, BAD_AREA),
    # the single-level calls apply level 1, the grouped ones levels (0, 1)
    ("masked-without-mask", SINGLE, dict(masked=1), SMM_ERR_INVALID,
     "masked apply but dst_grid_imask was never set for level 1"),
    ("masked-without-mask", GROUPED, dict(masked=[0, 1]), SMM_ERR_INVALID,
     "masked apply but dst_grid_imask was never set for level 1"),
    ("area-min-without-frac", SINGLE, dict(remap_area_min=0.5), SMM_ERR_INVALID,
     "remap_area_min > 0 but dst_grid_frac was never set for level 1"),
    ("area-min-without-frac", GROUPED, dict(remap_area_min=0.5), SMM_ERR_INVALID,
     "remap_area_min > 0 but dst_grid_frac was never set for level 0"),
    ("staged-forced-on-gather-level", SINGLE, dict(h="gather", kernel=KERNEL_STAGED), SMM_ERR_INVALID,
     "staged kernel forced but unavailable for level 1: "),
    ("staged-forced-on-gather-level", GROUPED, dict(h="gather", kernel=KERNEL_STAGED), SMM_ERR_INVALID,
     "staged kernel forced but unavailable for level 0: "),
]

# calls with nothing to apply: SMM_OK before any pointer is looked at
EMPTY = [
    ("B-zero-null-data", ENTRY_POINTS, dict(B=0, x=None, y=None)),
    ("B-zero-null-x", ENTRY_POINTS, dict(B=0, x=None)),
    ("n-sel-zero-null-data", GROUPED, dict(n_sel=0, level_index=None, x=None, y=None)),
    ("n-sel-zero-null-x", GROUPED, dict(n_sel=0, level_index=None, x=None)),
]


def _cases(table):
    return [pytest.param(ep, row, id=f"{ep}-{row[0]}") for row in table for ep in row[1]]


class _Setup:
    """Two handles of two levels each (staged | gather plans) and the buffers of B batch rows."""

    def __init__(self, lib):
        import torch
        from smmregrid_b200 import _lib
        self.lib = lib
        self.handles, self.sizes = {}, {}
        for name, vid, kernel in (("staged", "staged-l1k12-n256-fast", KERNEL_STAGED),
                                  ("gather", "gather-lpr4", KERNEL_GATHER)):
            v = BY_ID[vid]
            op = _operator(v, "parity")
            ll = np.full(N_LEVELS, op.src.size, np.int64)
            sa, da, rm = (np.tile(a.ravel(), N_LEVELS) for a in (op.src, op.dst, op.w))
            h = ctypes.c_void_p()
            with _create_env(v.env):
                _lib.check(lib.smm_create_levels(N_LEVELS, ll.ctypes.data, op.src.size, op.n_src, op.n_dst,
                                                 sa.ctypes.data, da.ctypes.data, rm.ctypes.data, 1, 1, 0, None,
                                                 ctypes.byref(h)))
            self.handles[name] = h
            self.sizes[name] = (op.n_src, op.n_dst)
            for level in range(N_LEVELS):
                info = _lib.SmmInfo()
                _lib.check(lib.smm_get_info(h, level, ctypes.byref(info)))
                assert info.kernel == kernel, (name, info.asdict())
        # float64 elements: room for B x N_LEVELS rows of any x or y dtype and either handle
        n_src, n_dst = (max(s[i] for s in self.sizes.values()) for i in (0, 1))
        self.x_dev = torch.zeros(B * N_LEVELS * n_src, dtype=torch.float64, device="cuda")
        self.y_dev = torch.full((B * N_LEVELS * n_dst,), SENTINEL, dtype=torch.float64, device="cuda")
        self.x_host = np.zeros(B * N_LEVELS * n_src)
        self.y_host = np.full(B * N_LEVELS * n_dst, SENTINEL)

    def close(self):
        for h in self.handles.values():
            self.lib.smm_destroy(h)

    def y_untouched(self, ep):
        import torch
        if ep in ("smm_apply", "smm_apply_levels"):
            torch.cuda.synchronize()
            return bool((self.y_dev == SENTINEL).all())
        return bool((self.y_host == SENTINEL).all())

    def reset_y(self):
        self.y_dev.fill_(SENTINEL)
        self.y_host.fill(SENTINEL)

    def call(self, ep, **changes):
        """The entry point's call with `changes` to the arguments of a call that succeeds."""
        from smmregrid_b200 import _lib
        host = ep.endswith("_host")
        a = dict(h="staged", level=1, level_index=[0, 1], n_sel=N_LEVELS, x="x", x_dtype=SMM_F32, B=B, ldx=0, y="y",
                 y_dtype=SMM_F64, ldy=0, masked=None, remap_area_min=0.0, kernel=0, renormalize=None, decode=None)
        a.update(changes)
        h = self.handles[a["h"]] if a["h"] else None
        n_src, n_dst = self.sizes[a["h"] or "staged"]
        x = None if a["x"] is None else (self.x_host.ctypes.data if host else self.x_dev.data_ptr())
        y = None if a["y"] is None else (self.y_host.ctypes.data if host else self.y_dev.data_ptr())
        ldx, ldy = n_src + a["ldx"], n_dst + a["ldy"]      # ldx / ldy: offsets from n_src / n_dst
        dec = None
        if a["decode"] is not None:
            dec = _lib.SmmDecode()
            for k, val in a["decode"].items():
                setattr(dec, k, val)
        opts = _lib.apply_opts(a["kernel"], a["renormalize"], dec)
        B_, amin = a["B"], a["remap_area_min"]
        if ep in SINGLE:
            masked = a["masked"] or 0
            if host:
                return self.lib.smm_apply_host(h, a["level"], x, a["x_dtype"], B_, ldx, y, a["y_dtype"], ldy, masked,
                                               amin, opts, 0)
            return self.lib.smm_apply(h, a["level"], x, a["x_dtype"], B_, ldx, y, a["y_dtype"], ldy, masked, amin,
                                      opts, None)
        sel = None if a["level_index"] is None else np.array(a["level_index"], np.int32)
        masked = None if a["masked"] is None else np.array(a["masked"], np.uint8)
        sel_p = None if sel is None else sel.ctypes.data
        masked_p = None if masked is None else masked.ctypes.data
        if host:
            return self.lib.smm_apply_levels_host(h, a["n_sel"], sel_p, x, a["x_dtype"], B_, y, a["y_dtype"],
                                                  masked_p, amin, opts, 0)
        return self.lib.smm_apply_levels(h, a["n_sel"], sel_p, x, a["x_dtype"], B_, N_LEVELS * n_src, n_src, y,
                                         a["y_dtype"], N_LEVELS * n_dst, n_dst, masked_p, amin, opts, None)


@pytest.fixture(scope="module")
def setup(smm_lib, cuda):
    s = _Setup(smm_lib)
    yield s
    s.close()


def _last_error(lib):
    return lib.smm_last_error().decode("utf-8", "replace")


@pytest.mark.gpu
@pytest.mark.parametrize("ep", ENTRY_POINTS)
def test_good_call_succeeds(setup, ep):
    """The call every fault below differs from by one argument is valid and writes y."""
    setup.reset_y()
    assert setup.call(ep) == SMM_OK, _last_error(setup.lib)
    assert not setup.y_untouched(ep)
    setup.reset_y()


@pytest.mark.gpu
@pytest.mark.parametrize("ep, row", _cases(FAULTS))
def test_single_fault_is_rejected(setup, ep, row):
    _, _, changes, code, message = row
    setup.reset_y()
    assert setup.call(ep, **changes) == code
    assert message in _last_error(setup.lib)
    assert setup.y_untouched(ep)


@pytest.mark.gpu
@pytest.mark.parametrize("ep, row", _cases(EMPTY))
def test_empty_call_returns_ok(setup, ep, row):
    setup.reset_y()
    assert setup.call(ep, **row[2]) == SMM_OK, _last_error(setup.lib)
    assert setup.y_untouched(ep)
