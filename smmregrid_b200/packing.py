"""CF-packed 16-bit source data, decoded inside the kernels (``smm_decode`` in the C header).

Much reanalysis data (ERA5, NCEP) is stored as ``int16`` with ``scale_factor`` / ``add_offset`` /
``_FillValue`` / ``missing_value`` attributes.  Handing the raw 16-bit values to the kernels moves
half the bytes of float32 over PCIe and through HBM.  The result equals decoding the field the way
xarray does and regridding the decoded field: bit for bit with reference-order sums or when both
take the same kernel family; otherwise (fast sums, where 2-byte and 4-byte rows may pick different
kernel families) to the rounding of the fast sums.
"""
from __future__ import annotations

import numpy as np

from . import _lib

PACKING_ATTRS = ("scale_factor", "add_offset", "_FillValue", "missing_value", "_Unsigned")
RAW_DTYPES = (np.dtype(np.int16), np.dtype(np.uint16))


def _attr_dtype(value) -> np.dtype:
    """Type of an attribute value as xarray sees it: numpy scalars / arrays keep theirs, a Python
    float counts as float64."""
    return np.asarray(value).dtype


def _attr_value(value) -> float:
    return float(np.asarray(value).reshape(-1)[0])


def choose_dtype(scale_factor=None, add_offset=None) -> np.dtype:
    """Decoded dtype of 16-bit packed data: xarray's ``_choose_float_dtype`` for 16-bit integers.
    ``scale_factor`` and ``add_offset`` of the same float type: that type; only ``scale_factor``:
    its type (float64 unless float32); ``add_offset`` present and the types differ or
    ``scale_factor`` is missing: float64; neither: float32."""
    if scale_factor is not None and add_offset is not None:
        st, ot = _attr_dtype(scale_factor), _attr_dtype(add_offset)
        if st == ot and st in (np.float32, np.float64):
            return np.dtype(st)
        return np.dtype(np.float64)
    if add_offset is not None:
        return np.dtype(np.float64)
    if scale_factor is not None:
        st = _attr_dtype(scale_factor)
        return np.dtype(np.float32) if st == np.float32 else np.dtype(np.float64)
    return np.dtype(np.float32)


class CFPacking:
    """How raw 16-bit values decode (the semantics of ``smm_decode``, include/smmregrid_b200.h).

    For a raw element ``r``: ``v`` = ``r`` as int16, or as uint16 when ``unsigned``; ``v`` equal to
    one of ``fill_values`` (at most 4: ``_FillValue`` and every ``missing_value``) is NaN; else
    ``x = D(D(v) * scale_factor) + add_offset``, each operation rounded once in the decoded dtype
    ``D`` (no FMA).  An absent ``scale_factor`` is 1.0, an absent ``add_offset`` -0.0 (adding it
    leaves every value, -0.0 included, unchanged).  Then the reference's apply: non-finite -> 1e20
    in ``D`` (a decode that overflowed to +-inf included), float64 products and sums.
    ``dtype=None`` picks ``D`` as xarray does (``choose_dtype``); ``valid_min`` / ``valid_max`` /
    ``valid_range`` are ignored, as xarray ignores them.  Fill values are given in the raw type's
    range (for unsigned data a negative value is taken as its 16-bit pattern); a value that no raw
    element can hold matches nothing.
    """

    def __init__(self, scale_factor=None, add_offset=None, fill_values=(), dtype=None, unsigned=False):
        self.dtype = choose_dtype(scale_factor, add_offset) if dtype is None else np.dtype(dtype)
        if self.dtype not in (np.float32, np.float64):
            raise ValueError(f"decoded dtype must be float32 or float64, got {self.dtype}")
        self.scale_factor = None if scale_factor is None else _attr_value(scale_factor)
        self.add_offset = None if add_offset is None else _attr_value(add_offset)
        for name, v in (("scale_factor", self.scale_factor), ("add_offset", self.add_offset)):
            if v is None:
                continue
            if not np.isfinite(v):
                raise ValueError(f"{name} must be finite, got {v}")
            if self.dtype == np.float32 and float(np.float32(v)) != v:
                raise ValueError(f"{name} {v!r} is not exactly representable in the decoded dtype float32")
        self.unsigned = bool(unsigned)
        lo, hi = (0, 65535) if self.unsigned else (-32768, 32767)
        fills = []
        for f in np.asarray(fill_values, dtype=np.float64).ravel():
            if not np.isfinite(f) or f != np.floor(f):
                continue                                   # no integer raw value equals it
            f = int(f)
            if self.unsigned and -32768 <= f < 0:
                f &= 0xFFFF                                # the 16-bit pattern of a signed attribute
            if lo <= f <= hi and f not in fills:
                fills.append(f)
        if len(fills) > 4:
            raise ValueError(f"at most 4 distinct fill values are supported, got {len(fills)}: {fills}")
        self.fill_values = tuple(fills)

    @classmethod
    def from_attrs(cls, attrs, raw_dtype):
        """Packing of a variable opened without decoding (``mask_and_scale=False``): None when it
        is not packed (no ``scale_factor`` / ``add_offset`` / ``_FillValue`` / ``missing_value``, or
        floating-point data).  TypeError for packed integer data other than int16 / uint16."""
        raw = np.dtype(raw_dtype)
        keys = ("scale_factor", "add_offset", "_FillValue", "missing_value")
        if not any(attrs.get(k) is not None for k in keys) or raw.kind == "f":
            return None
        if raw not in RAW_DTYPES:
            raise TypeError(f"CF-packed data is supported as int16 or uint16, got {raw}")
        unsigned = raw == np.uint16 or str(attrs.get("_Unsigned", "")).lower() == "true"
        fills = []
        for k in ("_FillValue", "missing_value"):
            if attrs.get(k) is not None:
                fills.extend(np.atleast_1d(np.asarray(attrs[k], dtype=np.float64)).ravel().tolist())
        return cls(attrs.get("scale_factor"), attrs.get("add_offset"), fills, unsigned=unsigned)

    def to_c(self) -> "_lib.SmmDecode":
        """The ``smm_decode`` struct of the C ABI."""
        d = _lib.SmmDecode()
        d.dtype = _lib.SMM_F32 if self.dtype == np.float32 else _lib.SMM_F64
        d.is_unsigned = 1 if self.unsigned else 0
        d.scale_factor = 1.0 if self.scale_factor is None else self.scale_factor
        d.add_offset = -0.0 if self.add_offset is None else self.add_offset
        d.n_fill = len(self.fill_values)
        for i, f in enumerate(self.fill_values):
            d.fill[i] = f
        return d

    def __repr__(self):
        return (f"CFPacking(scale_factor={self.scale_factor!r}, add_offset={self.add_offset!r}, "
                f"fill_values={self.fill_values!r}, dtype={self.dtype.name!r}, unsigned={self.unsigned!r})")
