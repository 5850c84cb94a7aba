"""float16 / bfloat16 sources on the host side (no device): the ABI codes and the front end's
hand-over of half data to the library without a float32 copy."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "smmregrid_b200.h")


def _header_defines():
    with open(HEADER) as f:
        return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(SMM_\w+)\s+(-?\d+)", f.read())}


def test_header_dtype_codes_match_binding():
    from smmregrid_b200 import _lib
    d = _header_defines()
    for name in ("SMM_F32", "SMM_F64", "SMM_I16", "SMM_F16", "SMM_BF16"):
        assert d[name] == getattr(_lib, name), name
    assert (d["SMM_F16"], d["SMM_BF16"]) == (3, 4)
    assert len({d[n] for n in ("SMM_F32", "SMM_F64", "SMM_I16", "SMM_F16", "SMM_BF16")}) == 5


def _bare_regridder():
    from smmregrid_b200 import Regridder
    return Regridder.__new__(Regridder)       # _floating reads no state: no weights, no device


def test_x_code_maps_half_dtypes():
    import torch
    from smmregrid_b200 import _lib
    from smmregrid_b200.regrid import _x_code
    assert _x_code(torch.float16) == _lib.SMM_F16
    assert _x_code(torch.bfloat16) == _lib.SMM_BF16
    assert _x_code(torch.float32) == _lib.SMM_F32
    assert _x_code(torch.float64) == _lib.SMM_F64
    assert _x_code(torch.int16) == _lib.SMM_I16


def test_floating_passes_half_data_unchanged():
    import torch
    rg = _bare_regridder()
    a = np.arange(12, dtype=np.float16).reshape(3, 4)
    out = rg._floating(a)
    assert out is a and out.dtype == np.float16
    for dt in (torch.float16, torch.bfloat16):
        t = torch.arange(12, dtype=dt).reshape(3, 4)
        assert rg._floating(t) is t
        s = t[:, ::2]                                   # non-contiguous views pass as they are, too
        assert rg._floating(s) is s
    # the other promotions are unchanged
    assert rg._floating(np.zeros(3, np.int32)).dtype == np.float64
    assert rg._floating(torch.zeros(3, dtype=torch.int16)).dtype == torch.float64
