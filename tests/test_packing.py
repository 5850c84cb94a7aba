"""CF packing on the host (no GPU): the decoded-dtype table, the attributes CFPacking reads, and the
layout of the C structs against their ctypes mirrors.

Values are checked against a numpy decode written here (xarray's CF decoding restated), never
against CFPacking itself: the kernels' decode is emulated from the smm_decode struct CFPacking
builds -- fill values compared on the raw 16 bits, v * scale + offset in the decoded dtype -- and
must give the numpy decode bit for bit.
"""
from __future__ import annotations

import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def np_decode(raw, attrs):
    """xarray (CFMaskCoder + CFScaleOffsetCoder) on raw int16 / uint16 data with these attributes."""
    unsigned = raw.dtype == np.uint16 or str(attrs.get("_Unsigned", "")).lower() == "true"
    v = raw.view(np.uint16 if unsigned else np.int16)
    sf, ao = attrs.get("scale_factor"), attrs.get("add_offset")
    if sf is not None and ao is not None:
        t = np.asarray(sf).dtype
        D = t.type if t == np.asarray(ao).dtype and t in (np.float32, np.float64) else np.float64
    elif ao is not None:
        D = np.float64
    elif sf is not None:
        D = np.asarray(sf).dtype.type
    else:
        D = np.float32
    fills = []
    for k in ("_FillValue", "missing_value"):
        if k in attrs:
            a = np.atleast_1d(np.asarray(attrs[k])).astype(np.int64)
            fills.extend((a & 0xFFFF) if unsigned else a)
    x = v.astype(D)
    with np.errstate(over="ignore"):
        if sf is not None:
            x = x * D(np.asarray(sf).reshape(-1)[0])
        if ao is not None:
            x = x + D(np.asarray(ao).reshape(-1)[0])
    x[np.isin(v.astype(np.int64), fills)] = np.nan
    return x


def emulate_kernel(raw, d):
    """The kernels' decode from the smm_decode struct alone."""
    D = np.float32 if d.dtype == 0 else np.float64
    r = raw.view(np.uint16).astype(np.int64)
    v = (r ^ (0 if d.is_unsigned else 0x8000)) - (0 if d.is_unsigned else 0x8000)
    with np.errstate(over="ignore"):
        x = v.astype(D) * D(d.scale_factor) + D(d.add_offset)
    lo, hi = (0, 65535) if d.is_unsigned else (-32768, 32767)
    for f in list(d.fill)[:d.n_fill]:
        if lo <= f <= hi:
            x[r == (f & 0xFFFF)] = np.nan
    return x


def _same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a[~np.isnan(a)].view(np.uint32 if a.dtype == np.float32 else np.uint64),
                       b[~np.isnan(b)].view(np.uint32 if b.dtype == np.float32 else np.uint64))


ALL_RAW = np.arange(-32768, 32768, dtype=np.int64).astype(np.int16)

TABLE = [
    ("f32 pair", {"scale_factor": np.float32(0.01), "add_offset": np.float32(273.15), "_FillValue": np.int16(-32767)},
     np.int16, np.float32),
    ("f64 pair", {"scale_factor": np.float64(0.0021), "add_offset": np.float64(250.5)}, np.int16, np.float64),
    ("python floats", {"scale_factor": 0.0021, "add_offset": 250.5}, np.int16, np.float64),
    ("types differ", {"scale_factor": np.float32(0.5), "add_offset": 10.0}, np.int16, np.float64),
    ("scale only f32", {"scale_factor": np.float32(0.25)}, np.int16, np.float32),
    ("scale only python", {"scale_factor": -0.25}, np.int16, np.float64),
    ("offset only", {"add_offset": np.float32(100.0)}, np.int16, np.float64),
    ("fill only", {"_FillValue": np.int16(-1)}, np.int16, np.float32),
    ("missing_value array", {"scale_factor": np.float32(2.0), "missing_value": np.array([-32768, 32767, 0], np.int16)},
     np.int16, np.float32),
    ("_Unsigned", {"scale_factor": np.float32(0.5), "add_offset": np.float32(-3.0), "_Unsigned": "true",
                   "_FillValue": np.int16(-1)}, np.int16, np.float32),
    ("uint16", {"scale_factor": 0.1, "_FillValue": np.uint16(65535), "missing_value": np.uint16(0)}, np.uint16,
     np.float64),
    ("valid_range ignored", {"scale_factor": np.float32(0.5), "add_offset": np.float32(1.0),
                             "valid_range": np.array([-100, 100], np.int16)}, np.int16, np.float32),
    ("overflow", {"scale_factor": np.float32(3e36)}, np.int16, np.float32),
]


@pytest.mark.parametrize("name,attrs,raw_dt,D", TABLE, ids=[t[0] for t in TABLE])
def test_decoded_dtype_and_values(name, attrs, raw_dt, D):
    from smmregrid_b200 import CFPacking
    p = CFPacking.from_attrs(attrs, raw_dt)
    raw = ALL_RAW.view(raw_dt)
    want = np_decode(raw, attrs)
    assert want.dtype == D and p.dtype == D
    got = emulate_kernel(raw, p.to_c())
    assert _same(got, want), name


def test_unpacked_and_unsupported():
    from smmregrid_b200 import CFPacking
    assert CFPacking.from_attrs({"units": "K"}, np.int16) is None
    assert CFPacking.from_attrs({"_FillValue": np.float32(1e20)}, np.float32) is None
    for dt in (np.int8, np.int32, np.uint8):
        with pytest.raises(TypeError, match="int16"):
            CFPacking.from_attrs({"scale_factor": 0.5}, dt)
    with pytest.raises(ValueError, match="at most 4"):
        CFPacking.from_attrs({"_FillValue": np.int16(1), "missing_value": np.array([2, 3, 4, 5], np.int16)}, np.int16)
    # repeated fill values count once
    assert len(CFPacking.from_attrs({"_FillValue": np.int16(1), "missing_value": np.array([1, 2, 3, 4])},
                                    np.int16).fill_values) == 4
    with pytest.raises(ValueError, match="float32"):
        CFPacking(scale_factor=0.1, dtype=np.float32)
    with pytest.raises(ValueError, match="finite"):
        CFPacking(scale_factor=np.inf)


def test_absent_offset_keeps_negative_zero():
    from smmregrid_b200 import CFPacking
    d = CFPacking(scale_factor=np.float32(-2.0)).to_c()
    assert d.add_offset == 0.0 and np.signbit(d.add_offset) and d.scale_factor == -2.0 and d.n_fill == 0
    x = emulate_kernel(np.zeros(1, np.int16), d)
    assert x[0] == 0.0 and np.signbit(x[0])


def test_nc4_variable_packing(tmp_path):
    """Variable.packing(): None for the float variables of a real file; for an int16 variable with
    CF attributes (the reader's metadata record built by hand), the packing of its attributes."""
    from smmregrid_b200 import nc4
    path = os.path.join(ROOT, "tests", "golden", "data", "regional.nc")
    with nc4.File(path) as f:
        for v in f.variables.values():
            p = v.packing()
            if v.dtype is not None and v.dtype.kind == "f":
                assert p is None
    attrs = {"scale_factor": np.float32(0.01), "add_offset": np.float32(273.15), "_FillValue": np.int16(-32767),
             "missing_value": np.int16(-32766), "units": "K"}
    var = nc4.Variable(None, "t2m", {"shape": (2, 3), "dtype": np.empty(0, ">i2"), "attrs": attrs})
    p = var.packing()
    raw = ALL_RAW
    assert p.dtype == np.float32 and _same(emulate_kernel(raw, p.to_c()), np_decode(raw, attrs))


def test_c_struct_layout_matches_ctypes(tmp_path):
    """sizeof / offsetof of smm_decode and smm_apply_opts, compiled from the header by the C compiler."""
    import ctypes
    import shutil
    from smmregrid_b200 import _lib
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text("""
#include <stdio.h>
#include <stddef.h>
#include "smmregrid_b200.h"
#define F(T, m) printf("%s.%s %zu\\n", #T, #m, offsetof(T, m));
int main(void) {
    printf("smm_decode %zu\\n", sizeof(smm_decode));
    printf("smm_apply_opts %zu\\n", sizeof(smm_apply_opts));
    F(smm_decode, dtype) F(smm_decode, is_unsigned) F(smm_decode, scale_factor) F(smm_decode, add_offset)
    F(smm_decode, n_fill) F(smm_decode, fill)
    F(smm_apply_opts, kernel) F(smm_apply_opts, renormalize) F(smm_apply_opts, min_valid_fraction)
    F(smm_apply_opts, decode)
    printf("SMM_I16 %d\\n", SMM_I16);
    return 0;
}
""")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(line.rsplit(" ", 1) for line in subprocess.run([str(exe)], check=True, capture_output=True,
                                                              text=True).stdout.splitlines())
    assert int(out["smm_decode"]) == ctypes.sizeof(_lib.SmmDecode)
    assert int(out["smm_apply_opts"]) == ctypes.sizeof(_lib.SmmApplyOpts)
    for cls, name in ((_lib.SmmDecode, "smm_decode"), (_lib.SmmApplyOpts, "smm_apply_opts")):
        for field, _ in cls._fields_:
            assert int(out[f"{name}.{field}"]) == getattr(cls, field).offset, (name, field)
    assert int(out["SMM_I16"]) == _lib.SMM_I16
