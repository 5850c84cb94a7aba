"""GPU parity tests: the sm_100a kernels, called through the C ABI, against the CPU oracle.

Bar (BASELINE.md §4): bit-exact NaN pattern; values within 1e-12 relative for float64 output
and 1e-6 relative for float32 output.
"""
import ctypes

import numpy as np
import pytest

from helpers import assert_parity, random_links

pytestmark = pytest.mark.gpu

RTOL_F64 = 1e-12
RTOL_F32 = 1e-6


def _create(lib, src, dst, rm, n_src, n_dst, summation=None):
    from smmregrid_b200 import _lib
    opts = _lib.create_opts(summation)
    h = ctypes.c_void_p()
    src = np.ascontiguousarray(src, np.int32)
    dst = np.ascontiguousarray(dst, np.int32)
    rm = np.ascontiguousarray(rm, np.float64)
    _lib.check(lib.smm_create(n_src, n_dst, src.size, src.ctypes.data, dst.ctypes.data, rm.ctypes.data,
                              rm.shape[1], 1, 0, opts, ctypes.byref(h)))
    return h


def _apply(lib, h, x_np, n_dst, ydtype, masked, amin, imask=None, frac=None, kernel=0, level=0, renormalize=None):
    import torch
    from smmregrid_b200 import _lib
    if imask is not None or frac is not None:
        im = None if imask is None else np.ascontiguousarray(imask, np.int32)
        fr = None if frac is None else np.ascontiguousarray(frac, np.float64)
        _lib.check(lib.smm_set_dst_mask(h, level, None if im is None else im.ctypes.data,
                                        None if fr is None else fr.ctypes.data))
    opts = _lib.apply_opts(kernel, renormalize)          # per call: nothing is stored on the handle
    x = torch.from_numpy(x_np).cuda()
    B = x.shape[0]
    y = torch.full((B, n_dst), -7.0, dtype=torch.float64 if ydtype == np.float64 else torch.float32, device="cuda")
    _lib.check(lib.smm_apply(h, level, x.data_ptr(), 0 if x_np.dtype == np.float32 else 1, B, x.shape[1],
                             y.data_ptr(), 1 if ydtype == np.float64 else 0, n_dst, int(masked), float(amin), opts,
                             torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return y.cpu().numpy()


def _info(lib, h, level=0):
    from smmregrid_b200 import _lib
    inf = _lib.SmmInfo()
    _lib.check(lib.smm_get_info(h, level, ctypes.byref(inf)))
    return inf.asdict()


@pytest.mark.parametrize("xdt", [np.float32, np.float64])
@pytest.mark.parametrize("ydt", [np.float64, np.float32])
@pytest.mark.parametrize("kernel", [0, 2])
@pytest.mark.parametrize("nnz_per_row", [1, 3, 7, 12, 30, 60, 120, 200])
def test_random_matrix(smm_lib, oracle, cuda, xdt, ydt, kernel, nnz_per_row):
    """Random links over a locally ordered source: every lane configuration, both kernels."""
    rng = np.random.default_rng(100 + nnz_per_row)
    n_src, n_dst, B = 4096, 700, 37
    counts = rng.integers(0, nnz_per_row + 1, size=n_dst)
    counts[5] = nnz_per_row                      # pin the lane configuration
    dst = np.repeat(np.arange(n_dst), counts)
    centre = (dst * n_src) // n_dst
    src = np.clip(centre + rng.integers(-300, 300, size=dst.size), 0, n_src - 1)
    w = rng.random(dst.size)
    o = np.lexsort((src, dst))
    src, dst, w = src[o] + 1, dst[o] + 1, w[o].reshape(-1, 1)
    x = (280 + 20 * rng.standard_normal((B, n_src))).astype(xdt)
    x[rng.random(x.shape) < 0.02] = np.nan
    x[3, 100] = np.inf
    x[4, 200] = -np.inf
    imask = (rng.random(n_dst) > 0.1).astype(np.int32)
    frac = rng.random(n_dst)
    mat = oracle.compute_weights_matrix_c(src, dst, w, n_src, n_dst)
    y_ref = oracle.apply_weights_c(x, mat, imask, frac, 0.5, True)
    h = _create(smm_lib, src, dst, w, n_src, n_dst)
    try:
        y = _apply(smm_lib, h, x, n_dst, ydt, True, 0.5, imask, frac, kernel)
        if ydt == np.float32:
            y_ref = y_ref.astype(np.float32)
        assert_parity(y, y_ref, RTOL_F64 if ydt == np.float64 else RTOL_F32, f"nnz{nnz_per_row}")
    finally:
        smm_lib.smm_destroy(h)


@pytest.mark.parametrize("cfg,scale,B", [("C1", 1, 12), ("C2", 4, 40), ("C4", 5, 24), ("C4", 10, 130)])
@pytest.mark.parametrize("nan_mode", ["none", "static", "step"])
def test_named_configs(smm_lib, oracle, cuda, cfg, scale, B, nan_mode):
    """BASELINE.json configurations at reduced size, float32 in, float64 and float32 out."""
    from smmregrid_b200 import synth
    w = synth.config_weights(cfg, scale)
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    x = synth.synthetic_field((B, n_src), np.float32, seed=5, nan_mode=nan_mode)
    mat = oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    imask, _ = oracle.mask_tensordot_c(w["src_grid_imask"], mat)
    y_ref = oracle.apply_weights_c(x, mat, imask, w["dst_grid_frac"], 0.5, True, nthreads=4)
    h = _create(smm_lib, w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    try:
        assert _info(smm_lib, h)["kernel_name"] == "staged"
        for kernel in (0, 2):
            y = _apply(smm_lib, h, x, n_dst, np.float64, True, 0.5, imask, w["dst_grid_frac"], kernel)
            assert_parity(y, y_ref, RTOL_F64, f"{cfg} f64 kernel{kernel}")
        y32 = _apply(smm_lib, h, x, n_dst, np.float32, True, 0.5, imask, w["dst_grid_frac"], 0)
        assert_parity(y32, y_ref.astype(np.float32), RTOL_F32, f"{cfg} f32")
    finally:
        smm_lib.smm_destroy(h)


def test_mask_sum_matches_oracle(smm_lib, oracle, cuda):
    """mask_tensordot: bit-exact 0/1 destination mask and any-masked flag on a conservative
    operator.  (None of its row sums lands on 0.5: the boundary is tested in
    test_gpu_init_kernels.py.)"""
    from smmregrid_b200 import _lib, synth
    w = synth.conservative_latlon(360, 180, 36, 18)
    n_src, n_dst = 360 * 180, 36 * 18
    rng = np.random.default_rng(3)
    src_mask = (rng.random(n_src) > 0.5).astype(np.int32)
    src_mask[: n_src // 3] = 0
    mat = oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    ref, _ = oracle.mask_tensordot_c(src_mask, mat)
    h = _create(smm_lib, w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    try:
        out = np.empty(n_dst, np.int32)
        flag = ctypes.c_int32(-1)
        _lib.check(smm_lib.smm_mask_sum(h, 0, src_mask.ctypes.data, out.ctypes.data, ctypes.byref(flag)))
        assert np.array_equal(out, ref)
        assert flag.value == int((ref == 0).any())
    finally:
        smm_lib.smm_destroy(h)


def test_threshold_replay_is_reference_order(smm_lib, oracle, cuda):
    """Rows whose filled sum lands within rounding of 1e19: the NaN decision must be the
    reference's (ascending-src order, separate multiply and add), not the tree order's."""
    rng = np.random.default_rng(9)
    n_src, n_dst, B = 2048, 512, 16
    k = 40
    dst = np.repeat(np.arange(n_dst), k)
    src = (np.repeat(np.arange(n_dst) * 3, k) + np.tile(np.arange(k), n_dst)) % n_src
    w = np.full(dst.size, 1.0 / k)
    w += rng.uniform(-1e-17, 1e-17, size=w.size)         # perturb the last bits
    o = np.lexsort((src, dst))
    src, dst, w = src[o] + 1, dst[o] + 1, w[o].reshape(-1, 1)
    x = rng.uniform(0, 2000, size=(B, n_src))          # float64: the fill is exactly 1e20
    # exactly 4 of 40 links NaN -> filled sum = 0.1 * 1e20 +- rounding, right at the threshold
    for d in range(n_dst):
        cols = (d * 3 + rng.choice(k, size=4, replace=False)) % n_src
        x[d % B, cols] = np.nan
    mat = oracle.compute_weights_matrix_c(src, dst, w, n_src, n_dst)
    y_ref = oracle.apply_weights_c(x, mat, None, None, 0.0, False)
    assert 0 < np.isnan(y_ref).sum() < y_ref.size
    # the case is discriminating: a lane-split + tree summation of the same terms (what the
    # fast path does) would flip hundreds of NaN decisions
    xf = np.where(np.isfinite(x), x, 1e20)
    o2 = np.lexsort((mat.src, mat.dst))
    terms = xf[:, mat.src[o2].reshape(n_dst, k)] * mat.w[o2].reshape(1, n_dst, k)
    t = sum(terms[:, :, j * 8:(j + 1) * 8] for j in range(k // 8))
    while t.shape[-1] > 1:
        t = t[..., ::2] + t[..., 1::2]
    assert ((t[..., 0] > 1e19) != np.isnan(y_ref)).sum() > 50
    h = _create(smm_lib, src, dst, w, n_src, n_dst)
    try:
        for kernel in (0, 2):
            y = _apply(smm_lib, h, x, n_dst, np.float64, False, 0.0, kernel=kernel)
            assert np.array_equal(np.isnan(y), np.isnan(y_ref)), kernel
            near = np.abs(y_ref - 1e19) < 1e10
            assert near.any()
            assert np.array_equal(y[near], y_ref[near]), "replayed rows must be bit-identical"
    finally:
        smm_lib.smm_destroy(h)


def test_reference_quirks(smm_lib, oracle, cuda):
    """SURVEY §7 quirks: 0.05-weight NaN leaks 5e18; negative weights never trip; > 1e19 data -> NaN;
    identity weights are exact; all-NaN row -> all-NaN; only column 0 of remap_matrix is used."""
    n = 64
    src = np.arange(1, n + 1, dtype=np.int32)
    dst = src.copy()
    rm = np.ones((n, 3))
    rm[:, 1:] = 99.0
    rm[0, 0] = 0.05
    rm[1, 0] = -0.5
    x = np.linspace(1, 2, 3 * n, dtype=np.float32).reshape(3, n)
    x[0, 0] = np.nan
    x[0, 1] = np.nan
    x[1, 5] = 3e19
    x[2, :] = np.nan
    mat = oracle.compute_weights_matrix_c(src, dst, rm, n, n)
    y_ref = oracle.apply_weights_c(x, mat, None, None, 0.0, False)
    h = _create(smm_lib, src, dst, rm, n, n)
    try:
        y = _apply(smm_lib, h, x, n, np.float64, False, 0.0)
    finally:
        smm_lib.smm_destroy(h)
    assert np.array_equal(np.isnan(y), np.isnan(y_ref))
    assert y[0, 0] == np.float64(np.float32(1e20)) * 0.05 and np.isfinite(y[0, 0])
    assert y[0, 1] == np.float64(np.float32(1e20)) * -0.5
    assert np.isnan(y[1, 5])
    assert np.isnan(y[2, 2:]).all()
    assert np.array_equal(y[1, 6:], x[1, 6:].astype(np.float64))


def test_levels_grouped_apply(smm_lib, oracle, cuda):
    """3-D ocean weights: one grouped launch over all levels == per-level oracle; subset of
    levels == slicing the full result (tests/levels_test.py in the reference)."""
    import torch
    from smmregrid_b200 import Regridder, synth
    w = synth.ocean3d_weights(72, 36, 36, 18, n_levels=30)
    n_src, n_dst, L, T = 72 * 36, 36 * 18, 30, 5
    x = synth.synthetic_field((T, L, n_src), np.float32, seed=2)
    x[:, w["src_grid_imask"] == 0] = np.nan
    mats = oracle.compute_weights_matrix3d_np(w["src_address"], w["dst_address"], w["remap_matrix"],
                                              w["link_length"], n_src, n_dst,
                                              builder=oracle.compute_weights_matrix_c)
    imask = np.stack([oracle.mask_tensordot_c(w["src_grid_imask"][l], mats[l])[0] for l in range(L)])
    masked = oracle.check_mask_np(imask)
    y_ref = oracle.regrid3d_np(x, 1, w.levels, w.levels, mats, imask, w["dst_grid_frac"], masked, 0.5)
    rg = Regridder(weights=w, remap_area_min=0.5)
    assert np.array_equal(np.asarray(rg.masked), masked)
    assert np.array_equal(rg.weights["dst_grid_imask"], imask)
    y = rg.regrid(torch.from_numpy(x).cuda()).cpu().numpy().reshape(T, L, n_dst)
    assert_parity(y, y_ref, RTOL_F64, "3d")
    sel = [14, 15, 17]
    ys = rg.regrid(x[:, sel], levels=w.levels[sel]).reshape(T, len(sel), n_dst)
    assert_parity(ys, y_ref[:, sel], RTOL_F64, "3d subset")
    with pytest.raises(ValueError):
        rg.regrid(x[:, :2], levels=[1e9, 2e9])
    # transpose=False keeps the level axis first (regrid.py:410)
    rg2 = Regridder(weights=w, remap_area_min=0.5, transpose=False)
    y2 = rg2.regrid(x).reshape(L, T, n_dst)
    assert_parity(np.moveaxis(y2, 0, 1), y_ref, RTOL_F64, "3d no transpose")


def test_host_apply_and_strides(smm_lib, oracle, cuda):
    """smm_apply_host (chunked H2D/D2H pipeline) and non-trivial ldx/ldy."""
    import torch
    from smmregrid_b200 import _lib, synth
    w = synth.config_weights("C2", 8)
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    B = 101
    x = synth.synthetic_field((B, n_src), np.float32, seed=8, nan_mode="random")
    mat = oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    y_ref = oracle.apply_weights_c(x, mat, None, w["dst_grid_frac"], 0.5, False, nthreads=4)
    h = _create(smm_lib, w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    try:
        fr = np.ascontiguousarray(w["dst_grid_frac"], np.float64)
        _lib.check(smm_lib.smm_set_dst_mask(h, 0, None, fr.ctypes.data))
        y = np.zeros((B, n_dst), np.float64)
        _lib.check(smm_lib.smm_apply_host(h, 0, x.ctypes.data, 0, B, n_src, y.ctypes.data, 1, n_dst, 0, 0.5, None, 16))
        assert_parity(y, y_ref, RTOL_F64, "host")
        # padded strides on the device path (ldx = n_src + 4 keeps 16-byte rows for TMA)
        xp = torch.zeros((B, n_src + 4), dtype=torch.float32, device="cuda")
        xp[:, :n_src] = torch.from_numpy(x).cuda()
        yp = torch.full((B, n_dst + 3), 5.0, dtype=torch.float64, device="cuda")
        _lib.check(smm_lib.smm_apply(h, 0, xp.data_ptr(), 0, B, n_src + 4, yp.data_ptr(), 1, n_dst + 3, 0, 0.5, None, None))
        torch.cuda.synchronize()
        assert_parity(yp[:, :n_dst].cpu().numpy(), y_ref, RTOL_F64, "strided")
        assert (yp[:, n_dst:] == 5.0).all()
        # odd ldx breaks the 16-byte row alignment: must still be right (gather kernel)
        xo = torch.zeros((B, n_src + 1), dtype=torch.float32, device="cuda")
        xo[:, :n_src] = torch.from_numpy(x).cuda()
        yo = torch.empty((B, n_dst), dtype=torch.float64, device="cuda")
        _lib.check(smm_lib.smm_apply(h, 0, xo.data_ptr(), 0, B, n_src + 1, yo.data_ptr(), 1, n_dst, 0, 0.5, None, None))
        torch.cuda.synchronize()
        assert_parity(yo.cpu().numpy(), y_ref, RTOL_F64, "unaligned")
    finally:
        smm_lib.smm_destroy(h)


def test_full_size_properties(smm_lib, cuda):
    """C4 at full grid size (6.48 M -> 64 800, 7.1 M links): size-independent properties.
    Constant field -> constant (rows sum to 1); linearity; NaN step -> NaN row; staged == gather."""
    import torch
    from smmregrid_b200 import Regridder, synth
    w = synth.config_weights("C4")
    rg = Regridder(weights=w, remap_area_min=0.5)
    n_src, n_dst = rg.n_src, rg.n_dst
    assert rg.weights_matrix.info()["kernel_name"] == "staged"
    B = 48
    g = torch.Generator(device="cuda").manual_seed(1234)
    x1 = 280 + 20 * torch.randn((B, n_src), generator=g, device="cuda", dtype=torch.float32)
    x2 = 5 * torch.randn((B, n_src), generator=g, device="cuda", dtype=torch.float32)
    const = torch.full((2, n_src), 3.25, device="cuda", dtype=torch.float32)
    yc = rg.regrid(const).reshape(2, n_dst)
    assert torch.allclose(yc, torch.full_like(yc, 3.25), rtol=1e-13, atol=0)
    y1 = rg.regrid(x1).reshape(B, n_dst)
    y2 = rg.regrid(x2).reshape(B, n_dst)
    y12 = rg.regrid((x1.double() + 2 * x2.double())).reshape(B, n_dst)
    assert torch.allclose(y12, y1 + 2 * y2, rtol=1e-11, atol=1e-9)
    # mean preservation: area-weighted mean of a conservative remap equals that of the source
    x1[7] = float("nan")
    y1n = rg.regrid(x1).reshape(B, n_dst)
    assert torch.isnan(y1n[7]).all() and not torch.isnan(y1n[6]).any()
    rg.kernel = "gather"
    yg = rg.regrid(x1).reshape(B, n_dst)
    rg.kernel = None
    assert torch.equal(torch.isnan(yg), torch.isnan(y1n))
    ok = ~torch.isnan(yg)
    assert torch.allclose(yg[ok], y1n[ok], rtol=1e-12, atol=0)


def test_errors(smm_lib, cuda):
    from smmregrid_b200 import Regridder, synth
    w = synth.config_weights("C1")
    with pytest.raises(ValueError):
        Regridder(weights=w, remap_area_min=1.5)
    with pytest.raises(ValueError):
        Regridder()
    rg = Regridder(weights=w)
    with pytest.raises(KeyError):
        rg.regrid(np.zeros((3, 17), np.float32))
    with pytest.raises(TypeError):
        rg.regrid("not an array")
    bad = w.assign(src_address=w["src_address"] + 10**6)
    with pytest.raises(ValueError):
        Regridder(weights=bad)


@pytest.mark.parametrize("k", [1, 4])
def test_healpix_nested_reordered_plan(smm_lib, oracle, cuda, k):
    """HEALPix-nested source: the staged plan tiles rows re-ordered by mean source address
    (row map indirection in the kernel); results must not depend on it."""
    from smmregrid_b200 import synth
    w = synth.healpix_weights(64, 180, 90, k)
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    B = 21
    x = synth.synthetic_field((B, n_src), np.float32, seed=3, nan_mode="random")
    frac = np.random.default_rng(0).random(n_dst)
    imask = (np.random.default_rng(1).random(n_dst) > 0.1).astype(np.int32)
    mat = oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    y_ref = oracle.apply_weights_c(x, mat, imask, frac, 0.5, True)
    h = _create(smm_lib, w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    try:
        info = _info(smm_lib, h)
        assert info["kernel_name"] == "staged" and (info["rows_reordered"] == 1 or info["packed_rows"] == 1)
        for kernel in (0, 2):
            y = _apply(smm_lib, h, x, n_dst, np.float64, True, 0.5, imask, frac, kernel)
            assert_parity(y, y_ref, RTOL_F64, f"healpix k={k} kernel={kernel}")
    finally:
        smm_lib.smm_destroy(h)


def test_c3_full_size_levels(smm_lib, oracle, cuda):
    """BASELINE config C3 at full size (ORCA1-like 362x292, 75 levels with level-varying masks):
    grouped launches over all levels against the per-level oracle, host (numpy) and device paths."""
    import torch
    from smmregrid_b200 import Regridder, synth
    w = synth.config_weights("C3")
    L, n_src, n_dst, T = 75, 362 * 292, 360 * 180, 3
    x = synth.synthetic_field((T, L, n_src), np.float32, seed=4)
    x[:, w["src_grid_imask"] == 0] = np.nan
    mats = oracle.compute_weights_matrix3d_np(w["src_address"], w["dst_address"], w["remap_matrix"],
                                              w["link_length"], n_src, n_dst, builder=oracle.compute_weights_matrix_c)
    imask = np.stack([oracle.mask_tensordot_c(w["src_grid_imask"][l], mats[l])[0] for l in range(L)])
    masked = oracle.check_mask_np(imask)
    y_ref = oracle.regrid3d_np(x, 1, w.levels, w.levels, mats, imask, w["dst_grid_frac"], masked, 0.5)
    rg = Regridder(weights=w, remap_area_min=0.5)
    assert np.array_equal(np.asarray(rg.masked), masked)
    assert np.array_equal(rg.weights["dst_grid_imask"], imask)
    y_host = rg.regrid(x).reshape(T, L, n_dst)                         # smm_apply_levels_host
    assert_parity(y_host, y_ref, RTOL_F64, "C3 host")
    y_dev = rg.regrid(torch.from_numpy(x).cuda()).cpu().numpy().reshape(T, L, n_dst)   # smm_apply_levels
    assert_parity(y_dev, y_ref, RTOL_F64, "C3 device")
    # the deeper the level the more destination cells are masked
    nan_per_level = np.isnan(y_ref[0]).sum(axis=1)
    assert nan_per_level[-1] > nan_per_level[0]


def test_c2_full_size_properties(smm_lib, cuda):
    """C2 (1440x721 -> r360x180 remapcon) at full grid size: constants are preserved, the
    area-weighted mean is conserved, staged == gather."""
    import torch
    from smmregrid_b200 import Regridder, synth
    w = synth.config_weights("C2")
    rg = Regridder(weights=w, remap_area_min=0.5)
    assert rg.weights_matrix.info()["kernel_name"] == "staged"
    B = 33
    g = torch.Generator(device="cuda").manual_seed(7)
    x = 280 + 20 * torch.randn((B, rg.n_src), generator=g, device="cuda", dtype=torch.float32)
    y = rg.regrid(x).reshape(B, 180, 360)
    yc = rg.regrid(torch.full((1, rg.n_src), -1.5, device="cuda", dtype=torch.float64))
    assert torch.allclose(yc, torch.full_like(yc, -1.5), rtol=1e-13, atol=0)
    # first-order conservative remapping conserves the area integral
    lat_s = torch.linspace(-90, 90, 721, device="cuda", dtype=torch.float64)
    edges = torch.clamp(torch.cat([lat_s[:1], 0.5 * (lat_s[1:] + lat_s[:-1]), lat_s[-1:]]), -90, 90)
    a_s = (torch.sin(torch.deg2rad(edges[1:])) - torch.sin(torch.deg2rad(edges[:-1])))[:, None].expand(721, 1440)
    e_d = torch.linspace(-90, 90, 181, device="cuda", dtype=torch.float64)
    a_d = (torch.sin(torch.deg2rad(e_d[1:])) - torch.sin(torch.deg2rad(e_d[:-1])))[:, None].expand(180, 360)
    mean_s = (x.double().reshape(B, 721, 1440) * a_s).sum((1, 2)) / a_s.sum()
    mean_d = (y * a_d).sum((1, 2)) / a_d.sum()
    assert torch.allclose(mean_s, mean_d, rtol=1e-11, atol=0)
    rg.kernel = "gather"
    yg = rg.regrid(x).reshape(B, 180, 360)
    assert torch.allclose(yg, y, rtol=1e-12, atol=0)


def test_operator_cache_reuses_handle(smm_lib, cuda):
    import smmregrid_b200 as sb
    from smmregrid_b200 import synth
    w = synth.config_weights("C1")
    sb.enable_operator_cache(2)
    try:
        a = sb.Regridder(weights=w)
        b = sb.Regridder(weights=synth.config_weights("C1"))          # same content, new object
        assert a.weights_matrix is b.weights_matrix
        c = sb.Regridder(weights=synth.config_weights("C2", 8))
        assert c.weights_matrix is not a.weights_matrix
        x = synth.synthetic_field((2, a.n_src), np.float32)
        assert np.array_equal(a.regrid(x), b.regrid(x), equal_nan=True)
    finally:
        sb.enable_operator_cache(0)
    d = sb.Regridder(weights=w)
    assert d.weights_matrix is not a.weights_matrix


def test_concurrent_applies_on_streams(smm_lib, oracle, cuda):
    """The header promises smm_apply is re-entrant across host threads and streams: four
    threads, each on its own stream, hammer one handle; every result must be exact."""
    import threading
    import torch
    from smmregrid_b200 import _lib, synth
    w = synth.config_weights("C2", 4)
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    mat = oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    h = _create(smm_lib, w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    fr = np.ascontiguousarray(w["dst_grid_frac"], np.float64)
    _lib.check(smm_lib.smm_set_dst_mask(h, 0, None, fr.ctypes.data))
    errors = []

    def worker(seed):
        try:
            B = 17 + seed
            x = synth.synthetic_field((B, n_src), np.float32, seed=seed, nan_mode="random")
            y_ref = oracle.apply_weights_c(x, mat, None, fr, 0.5, False)
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                xd = torch.from_numpy(x).cuda()
                for _ in range(20):
                    yd = torch.empty((B, n_dst), dtype=torch.float64, device="cuda")
                    _lib.check(smm_lib.smm_apply(h, 0, xd.data_ptr(), 0, B, n_src, yd.data_ptr(), 1, n_dst, 0, 0.5,
                                                 None, st.cuda_stream))
                st.synchronize()
                assert_parity(yd.cpu().numpy(), y_ref, RTOL_F64, f"thread {seed}")
        except Exception as e:          # noqa: BLE001
            errors.append(repr(e))

    threads = [threading.Thread(target=worker, args=(s,)) for s in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    smm_lib.smm_destroy(h)
    assert not errors, errors


def test_dict_of_variables(smm_lib, cuda):
    from smmregrid_b200 import Regridder, synth
    rg = Regridder(weights=synth.config_weights("C1"))
    x = synth.synthetic_field((3, 73, 144), np.float32)
    out = rg.regrid({"tas": x, "pr": 2 * x, "lat_bnds": np.zeros((73, 2)), "time_bnds": np.zeros((3, 2))})
    assert set(out) == {"tas", "pr", "time_bnds"}
    assert out["tas"].shape == (3, 90, 180) and np.allclose(out["pr"], 2 * out["tas"], rtol=1e-13)


@pytest.mark.parametrize("xdt", [np.float32, np.float64])
def test_renormalising_extension(smm_lib, oracle, cuda, xdt):
    """Opt-in extension (off by default): time-varying missing values are excluded and the
    remaining weights renormalised.  Reference mode on the same handle must be unaffected."""
    from smmregrid_b200 import Regridder, synth
    w = synth.config_weights("C2", 4)
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    rng = np.random.default_rng(5)
    B = 9
    x = (280 + 20 * rng.standard_normal((B, n_src))).astype(xdt)
    for b in range(B):                                   # a different blob of missing data per step
        c = rng.integers(0, n_src)
        x[b, max(0, c - 3000):c + 3000] = np.nan
    x[0, rng.random(n_src) < 0.3] = np.nan
    x[1, 5] = np.inf
    mat = oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    imask = np.ones(n_dst, np.int32)
    for min_valid in (0.0, 0.5, 0.9):
        ref = oracle.apply_weights_renorm_np(x, mat, imask, w["dst_grid_frac"], 0.5, False, min_valid)
        rg = Regridder(weights=w, remap_area_min=0.5, renormalize=min_valid)
        for kernel in (None, "gather"):
            rg.kernel = kernel
            y = rg.regrid(x).reshape(B, n_dst)
            assert_parity(y, ref, 1e-12, f"renorm {min_valid} {kernel}")
        # fewer NaNs than the reference semantics, and values stay in the data range
        y_ref_mode = Regridder(weights=w, remap_area_min=0.5).regrid(x).reshape(B, n_dst)
        assert np.isnan(y).sum() <= np.isnan(y_ref_mode).sum()
        assert np.nanmax(y) < 400 and np.nanmin(y) > 150
    # off again: bit-identical NaN pattern with the oracle's reference semantics
    y0 = Regridder(weights=w, remap_area_min=0.5).regrid(x).reshape(B, n_dst)
    assert_parity(y0, oracle.apply_weights_c(x, mat, None, w["dst_grid_frac"], 0.5, False), 1e-12, "reference mode")


def test_levels_mixed_kernels_and_empty_level(smm_lib, oracle, cuda):
    """A 3-D weight set whose levels need different kernel families (structured -> staged,
    scattered -> gather) plus a level without any link; B = 1 as well."""
    from smmregrid_b200 import CdoWeights, Regridder, synth
    n_lon_s, n_lat_s, n_lon_d, n_lat_d = 576, 288, 72, 36
    n_src, n_dst = n_lon_s * n_lat_s, n_lon_d * n_lat_d
    con = synth.conservative_latlon(n_lon_s, n_lat_s, n_lon_d, n_lat_d)
    sca = synth.scattered_weights(n_src, n_lon_d, n_lat_d, links_per_row=4, ordering="random", seed=2)
    parts = [con, sca, None, con]                          # level 2 has no links at all
    ll = np.array([0 if p is None else p["src_address"].size for p in parts], np.int64)
    nl = int(ll.max())
    sa = np.zeros((4, nl), np.int32); da = np.zeros((4, nl), np.int32); rm = np.zeros((4, nl, 1))
    for l, p in enumerate(parts):
        if p is not None:
            sa[l, :ll[l]], da[l, :ll[l]], rm[l, :ll[l]] = p["src_address"], p["dst_address"], p["remap_matrix"]
    v = dict(con.vars)
    v.update(src_address=sa, dst_address=da, remap_matrix=rm, link_length=ll,
             src_grid_imask=np.ones((4, n_src), np.int32), dst_grid_imask=np.ones((4, n_dst), np.int32),
             dst_grid_frac=np.ones((4, n_dst)))
    w = CdoWeights(v, mask_dim="lev", levels=[1.0, 2.0, 3.0, 4.0])
    rg = Regridder(weights=w, remap_area_min=0.0)
    kinds = [rg.weights_matrix.info(l)["kernel_name"] for l in range(4)]
    assert kinds[0] == "staged" and kinds[1] == "gather" and kinds[3] == "staged", kinds
    mats = oracle.compute_weights_matrix3d_np(sa, da, rm, ll, n_src, n_dst, builder=oracle.compute_weights_matrix_c)
    imask = np.stack([oracle.mask_tensordot_c(np.ones(n_src, np.int32), m)[0] for m in mats])
    masked = oracle.check_mask_np(imask)
    assert masked.tolist() == [False, False, True, False] and np.array_equal(np.asarray(rg.masked), masked)
    for T in (1, 7):
        x = synth.synthetic_field((T, 4, n_src), np.float32, seed=T, nan_mode="random")
        y_ref = oracle.regrid3d_np(x, 1, w.levels, w.levels, mats, imask, v["dst_grid_frac"], masked, 0.0)
        for kernel in (None, "compact"):                   # compact: the scattered level takes the two-pass path
            rg.kernel = kernel
            y = rg.regrid(x).reshape(T, 4, n_dst)
            assert_parity(y, y_ref, RTOL_F64, f"mixed T={T} {kernel}")
            assert np.isnan(y[:, 2]).all()                 # no links -> masked level -> NaN everywhere
    # many time steps, device data with the level stride (the scattered level may go two-pass by itself)
    import torch
    rg.kernel = None
    x = synth.synthetic_field((40, 4, n_src), np.float32, seed=9, nan_mode="random")
    y_ref = oracle.regrid3d_np(x, 1, w.levels, w.levels, mats, imask, v["dst_grid_frac"], masked, 0.0)
    y = rg.regrid(torch.from_numpy(x).cuda()).cpu().numpy().reshape(40, 4, n_dst)
    assert_parity(y, y_ref, RTOL_F64, "mixed T=40")


def _short_row_links(rng, n_src, n_dst, choices, spread=6):
    counts = rng.choice(choices, size=n_dst)
    dst = np.repeat(np.arange(n_dst), counts)
    src = np.clip((dst * n_src) // n_dst + rng.integers(-spread, spread + 1, size=dst.size), 0, n_src - 1)
    w = rng.random(dst.size) + 0.05
    o = np.lexsort((src, dst))
    return src[o] + 1, dst[o] + 1, w[o].reshape(-1, 1)


@pytest.mark.parametrize("xdt", [np.float32, np.float64])
@pytest.mark.parametrize("ydt", [np.float64, np.float32])
@pytest.mark.parametrize("n_dst", [3001, 420000])
def test_packed_rows_parity(smm_lib, oracle, cuda, xdt, ydt, n_dst):
    """Short-row operators run the packed-rows layout (a thread owns up to 4 rows): missing
    values (static and per step), masks, frac, both output types, one tile and many tiles."""
    rng = np.random.default_rng(n_dst)
    n_src = n_dst * 3 // 2 + 8
    B = 37 if n_dst < 10000 else 5
    src, dst, w = _short_row_links(rng, n_src, n_dst, [0, 1, 2, 3, 4, 4, 4, 5, 6, 9, 16])
    x = (280 + 20 * rng.standard_normal((B, n_src))).astype(xdt)
    x[:, rng.random(n_src) < 0.05] = np.nan                # static mask
    x[rng.random(x.shape) < 0.002] = np.nan                # per-step holes
    x[1, 77] = np.inf
    x[2, 99] = -np.inf
    imask = (rng.random(n_dst) > 0.1).astype(np.int32)
    frac = rng.random(n_dst)
    mat = oracle.compute_weights_matrix_c(src, dst, w, n_src, n_dst)
    y_ref = oracle.apply_weights_c(x, mat, imask, frac, 0.5, True, nthreads=4)
    h = _create(smm_lib, src, dst, w, n_src, n_dst)
    try:
        inf = _info(smm_lib, h)
        assert inf["kernel_name"] == "staged" and inf["packed_rows"] == 1, inf
        assert inf["consumer_threads"] == 256, inf            # packed plans: two CTAs per SM
        y = _apply(smm_lib, h, x, n_dst, ydt, True, 0.5, imask, frac)
        if ydt == np.float32:
            y_ref = y_ref.astype(np.float32)
        assert_parity(y, y_ref, RTOL_F64 if ydt == np.float64 else RTOL_F32, "packed")
    finally:
        smm_lib.smm_destroy(h)


def test_packed_rows_threshold_replay_and_renorm(smm_lib, oracle, cuda):
    """Packed plans: sums within rounding of 1e19 are replayed in the reference order (rows that
    span two sub-rows included); the renormalising extension falls back to the gather kernel."""
    rng = np.random.default_rng(21)
    n_src, n_dst, B, k = 4096, 1500, 16, 8
    dst = np.repeat(np.arange(n_dst), k)
    src = (np.repeat(np.arange(n_dst) * 2, k) + np.tile(np.arange(k), n_dst)) % n_src
    w = np.full(dst.size, 1.0 / k) + rng.uniform(-1e-17, 1e-17, size=dst.size)
    # two of three rows are short, so the operator packs; every third keeps its 8 links
    keep = (dst % 3 == 0) | (np.tile(np.arange(k), n_dst) < 2)
    src, dst, w = src[keep], dst[keep], w[keep]
    w[dst % 3 != 0] = 0.05 + rng.uniform(-1e-17, 1e-17, size=(dst % 3 != 0).sum())
    o = np.lexsort((src, dst))
    src, dst, w = src[o] + 1, dst[o] + 1, w[o].reshape(-1, 1)
    x = rng.uniform(0, 2000, size=(B, n_src))              # float64: the fill is exactly 1e20
    for d in range(n_dst):                                 # missing links put sums at 0.1 * 1e20 +- rounding
        nbad = 2 if d % 3 else 1
        cols = (d * 2 + rng.choice(2 if d % 3 else k, size=nbad, replace=False)) % n_src
        x[d % B, cols] = np.nan
    mat = oracle.compute_weights_matrix_c(src, dst, w, n_src, n_dst)
    y_ref = oracle.apply_weights_c(x, mat, None, None, 0.0, False)
    near = np.abs(y_ref - 1e19) < 1e10
    assert near.sum() > 100 and 0 < np.isnan(y_ref).sum() < y_ref.size
    h = _create(smm_lib, src, dst, w, n_src, n_dst)
    try:
        assert _info(smm_lib, h)["packed_rows"] == 1
        y = _apply(smm_lib, h, x, n_dst, np.float64, False, 0.0)
        assert np.array_equal(np.isnan(y), np.isnan(y_ref))
        assert np.array_equal(y[near], y_ref[near]), "replayed rows must be bit-identical"
        assert_parity(y, y_ref, RTOL_F64, "packed threshold")
        # renormalising extension on a packed plan
        from smmregrid_b200 import _lib
        n0 = smm_lib.smm_launch_count()
        yr = _apply(smm_lib, h, x, n_dst, np.float64, False, 0.0, renormalize=0.3)
        assert smm_lib.smm_launch_count() == n0 + 1
        ref = oracle.apply_weights_renorm_np(x, mat, np.ones(n_dst, np.int32), None, 0.0, False, 0.3)
        assert_parity(yr, ref, 1e-12, "packed renorm -> gather")
        assert_parity(_apply(smm_lib, h, x, n_dst, np.float64, False, 0.0), y_ref, RTOL_F64, "back to reference mode")
    finally:
        smm_lib.smm_destroy(h)


def test_nan_variation_probe(smm_lib, oracle, cuda):
    """detect_nan_variation_dims on the device against the reference-made fixture and the oracle."""
    import os
    import torch
    from smmregrid_b200 import detect_nan_variation_dims
    from smmregrid_b200.util import nan_variation_count
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "nan_variation.npz"))
    for k in [k for k in g.files if not k.endswith("_dims")]:
        want = g[k + "_dims"].tolist()
        assert detect_nan_variation_dims(g[k], 0, [1, 2]) == want, k
        assert detect_nan_variation_dims(g[k], [0], [1, 2]) == want, k            # the reference passes a list
        assert detect_nan_variation_dims(torch.from_numpy(g[k]).cuda(), 0, [1, 2]) == want, k
        assert detect_nan_variation_dims(g[k][0], None, [0, 1]) == [d - 1 for d in want], k
    # counts, every axis, odd sizes, against the oracle
    rng = np.random.default_rng(8)
    for dt in (np.float32, np.float64):
        f = rng.standard_normal((3, 7, 33, 5)).astype(dt)
        f[rng.random(f.shape) < 0.05] = np.nan
        f[0, 0, 0, 0] = np.inf
        for ax in range(4):
            assert nan_variation_count(f, ax) == oracle.nan_variation_count_np(f, ax), (dt, ax)
    assert nan_variation_count(np.zeros((4, 1, 3), np.float32), 1) == 0           # nothing to diff
    assert nan_variation_count(np.arange(12).reshape(3, 4), 0) == 0               # integers have no NaN


def test_more_levels_than_one_launch_holds(smm_lib, oracle, cuda):
    """140 levels: more than the 128 a grouped launch takes, so the apply is split in two
    balanced launches; device and host entry points."""
    import torch
    from smmregrid_b200 import Regridder, synth
    L, T = 140, 3
    w = synth.ocean3d_weights(36, 18, 24, 12, n_levels=L, seed=5)
    n_src, n_dst = 36 * 18, 24 * 12
    x = synth.synthetic_field((T, L, n_src), np.float32, seed=4)
    x[:, w["src_grid_imask"] == 0] = np.nan
    mats = oracle.compute_weights_matrix3d_np(w["src_address"], w["dst_address"], w["remap_matrix"],
                                              w["link_length"], n_src, n_dst,
                                              builder=oracle.compute_weights_matrix_c)
    imask = np.stack([oracle.mask_tensordot_c(w["src_grid_imask"][l], mats[l])[0] for l in range(L)])
    y_ref = oracle.regrid3d_np(x, 1, w.levels, w.levels, mats, imask, w["dst_grid_frac"],
                               oracle.check_mask_np(imask), 0.5)
    rg = Regridder(weights=w, remap_area_min=0.5)
    n0 = smm_lib.smm_launch_count()
    y = rg.regrid(torch.from_numpy(x).cuda()).cpu().numpy().reshape(T, L, n_dst)
    assert smm_lib.smm_launch_count() - n0 == 2
    assert_parity(y, y_ref, RTOL_F64, "140 levels, device")
    assert_parity(rg.regrid(x).reshape(T, L, n_dst), y_ref, RTOL_F64, "140 levels, host")


@pytest.mark.parametrize("xdt", [np.float32, np.float64])
@pytest.mark.parametrize("ydt", [np.float64, np.float32])
@pytest.mark.parametrize("B", [1, 37, 64, 130])
def test_compact_two_pass_path(smm_lib, oracle, cuda, xdt, ydt, B):
    """Scattered sources: the two-pass path (touched columns transposed into a compact buffer,
    links applied with lanes over the batch) sums in the reference's own order, so float64
    results are BIT-IDENTICAL to the reference-order oracle."""
    rng = np.random.default_rng(1000 + B)
    n_src, n_dst = 400001, 3001                   # odd sizes: partial column block, partial row block
    src, dst, w = random_links(rng, n_src, n_dst, 3, dup_frac=0.05, sort=False, negative=True)
    x = (280 + 20 * rng.standard_normal((B, n_src))).astype(xdt)
    x[rng.random(x.shape) < 0.03] = np.nan
    x[0, src[0] - 1] = np.inf
    imask = (rng.random(n_dst) > 0.1).astype(np.int32)
    frac = rng.random(n_dst)
    mat = oracle.compute_weights_matrix_c(src, dst, w, n_src, n_dst)
    y_ref = oracle.apply_weights_c(x, mat, imask, frac, 0.5, True)
    h = _create(smm_lib, src, dst, w, n_src, n_dst)
    try:
        assert _info(smm_lib, h)["kernel_name"] == "gather"
        n0 = smm_lib.smm_launch_count()
        y = _apply(smm_lib, h, x, n_dst, ydt, True, 0.5, imask, frac, kernel=3)
        assert smm_lib.smm_launch_count() - n0 == 2 * ((B + 63) // 64)          # two passes per 64 batch rows
        if ydt == np.float64:
            assert_parity(y, y_ref, RTOL_F64, "compact f64 out")
            diff = ~((y == y_ref) | (np.isnan(y) & np.isnan(y_ref)))
            assert not diff.any(), (int(diff.sum()), y[diff][:4], y_ref[diff][:4])
        else:
            assert_parity(y, y_ref.astype(np.float32), RTOL_F32, "compact f32 out")
        # automatic choice (direct gathers here: few links per source column).  The weights of this
        # case change sign, so the operator is summed in the reference's order on every path
        assert _info(smm_lib, h)["summation_name"] == "reference"
        y_auto = _apply(smm_lib, h, x, n_dst, ydt, True, 0.5, imask, frac, kernel=0)
        assert_parity(y_auto, y_ref.astype(ydt), RTOL_F64 if ydt == np.float64 else RTOL_F32, "auto")
    finally:
        smm_lib.smm_destroy(h)


def test_compact_path_is_chosen_for_dense_scattered_operators(smm_lib, oracle, cuda):
    """Scattered sources (random source order): with >= 16 batch rows of float32 the apply takes the
    two-pass path by itself -- C5dis-like (4 links per row) and, since its first pass moves the slab
    with TMA bulk copies, nn-like operators too; float64 input doubles the slab the first pass has
    to move, there a sparse nn-like operator keeps the direct gathers."""
    from smmregrid_b200 import synth
    for cfg, xdt, expect_compact in (("C5dis", np.float32, True), ("C5nn", np.float32, True), ("C5nn", np.float64, False)):
        w = synth.config_weights(cfg, 8)
        n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
        x = synth.synthetic_field((40, n_src), xdt, seed=3, nan_mode="random")
        mat = oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
        y_ref = oracle.apply_weights_c(x, mat, None, None, 0.0, False, nthreads=4)
        h = _create(smm_lib, w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
        try:
            n0 = smm_lib.smm_launch_count()
            y = _apply(smm_lib, h, x, n_dst, np.float64, False, 0.0)
            assert (smm_lib.smm_launch_count() - n0 >= 2) == expect_compact, (cfg, xdt)
            assert_parity(y, y_ref, RTOL_F64, cfg)
            n0 = smm_lib.smm_launch_count()
            y8 = _apply(smm_lib, h, np.ascontiguousarray(x[:8]), n_dst, np.float64, False, 0.0)   # few rows: direct gathers
            assert smm_lib.smm_launch_count() - n0 == 1
            assert_parity(y8, y_ref[:8], RTOL_F64, cfg + " B=8")
        finally:
            smm_lib.smm_destroy(h)


def test_c5_full_size_properties(smm_lib, cuda):
    """C5dis (20.97 M randomly ordered cells -> 0.25 deg, 4 inverse-distance links per cell) at
    full size: the compact path is chosen for 48 steps, constants are preserved (weights of a
    cell sum to 1), results lie between the extremes of the linked sources, compact == direct
    gathers, and a NaN source poisons exactly the cells linked to it."""
    import torch
    from smmregrid_b200 import Regridder, synth
    w = synth.config_weights("C5dis")
    rg = Regridder(weights=w, remap_area_min=0.0)
    assert rg.weights_matrix.info()["kernel_name"] == "gather" and rg.n_src == 20971520
    B = 48
    g = torch.Generator(device="cuda").manual_seed(11)
    x = 280 + 20 * torch.randn((B, rg.n_src), generator=g, device="cuda", dtype=torch.float32)
    n0 = smm_lib.smm_launch_count()
    y = rg.regrid(x).reshape(B, -1)
    assert smm_lib.smm_launch_count() - n0 == 2                    # two passes, one chunk of <= 64 steps
    rg.kernel = "gather"
    yg = rg.regrid(x).reshape(B, -1)
    rg.kernel = None
    assert torch.allclose(y, yg, rtol=1e-12, atol=0) and not torch.isnan(y).any()
    yc = rg.regrid(torch.full((16, rg.n_src), 3.25, device="cuda", dtype=torch.float64)).reshape(16, -1)
    assert torch.allclose(yc, torch.full_like(yc, 3.25), rtol=1e-13, atol=0)
    src = torch.from_numpy(np.asarray(w["src_address"]).astype(np.int64) - 1).cuda().reshape(-1, 4)
    dst = torch.from_numpy(np.asarray(w["dst_address"]).astype(np.int64) - 1).cuda().reshape(-1, 4)
    assert (dst == dst[:, :1]).all()                                # 4 consecutive links per destination cell
    xs = x[0].double()[src]
    lo, hi = xs.min(1).values, xs.max(1).values
    assert ((y[0][dst[:, 0]] >= lo - 1e-9) & (y[0][dst[:, 0]] <= hi + 1e-9)).all()
    # one missing source cell -> NaN exactly in the destination cells linked to it (1e20 fill, > 1e19 rule
    # needs weight > 0.1; smaller weights leak a huge finite value instead, as in the reference)
    c = int(src[12345, 0])
    x[3, c] = float("nan")
    y3 = rg.regrid(x[3:4]).reshape(-1)
    wts = torch.from_numpy(np.asarray(w["remap_matrix"])[:, 0]).cuda().reshape(-1, 4)
    hit = (src == c)
    big = (hit & (wts > 0.1)).any(1)
    assert torch.isnan(y3[dst[big, 0]]).all() and big.any()
    untouched = ~hit.any(1)
    assert torch.allclose(y3[dst[untouched, 0]], y[3][dst[untouched, 0]], rtol=1e-12, atol=0)   # (direct gathers at B = 1)
