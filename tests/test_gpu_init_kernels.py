"""The two init-time kernels against the oracle, at the edges where they go wrong.

mask_sum_kernel (smm_mask_sum; weights.mask_tensordot / mask_weights / check_mask) writes the 0/1
destination mask that every later apply of the level reads in its epilogue: one wrong decision is
a destination cell that stays NaN for the rest of the run, or one that should be masked and is
not.  The reference decides `t < 0.5` on a float64 sum taken in ascending-source order with
separate multiplies and adds (weights.py:47-52), so the kernel has to reproduce that sum bit for
bit.  The operators here are built to tell summation orders apart:

  * boundary rows: Dirichlet weights x 0.5 whose ascending sum is exactly 0.5 while the reversed
    sum or a pairwise tree is not, or whose ascending sum is one ulp off 0.5 while the reversed
    sum or the tree lands on it.  The source mask switches other links of the row off, so the sum that lands
    on 0.5 is a subset sum;
  * cancelling rows: 0.5 x cubic-convolution taps, weights of both signs (bicubic-like weights);
  * duplicate links, merged in input order like sparse.COO's sum_duplicates, with magnitudes that
    make the merged weight depend on that order;
  * rows without links, a one-row operator, partial last blocks, all-zero and all-one masks.

CPU checks show that the constructions discriminate.  GPU checks run them through every plan
kind, 3-D sets, the plan cache, a second mask on the same handle and the full-size constructors.

nan_variation_kernel (smm_nan_variation; util.nan_variation_count / detect_nan_variation_dims)
counts the positions whose NaN-ness changes along an axis (util.py:57-85): ranks 1-5, every axis,
partial warps and blocks, axes of 0-3 and 1000 elements, NaN at the first or only at the last
index, NaN payloads (negative, signalling), +-inf, every input dtype and container, and more than
2**31 positions.
"""
import ctypes
import zlib

import numpy as np
import pytest

from test_gpu_levels_host import SPLIT
from test_gpu_variants import BY_ID, KERNEL_GATHER, KERNEL_STAGED, SCATTER, SUM_FAST, SUM_REFERENCE, _create_env, \
    _same_bits

BELOW = float(np.nextafter(0.5, 0.0))           # 0.49999999999999994
ABOVE = float(np.nextafter(0.5, 1.0))           # 0.5000000000000001


# ------------------------------------------------------------------ summation orders

def _ascending(p):
    """Left-to-right sums over the last axis, one rounded add at a time (the reference's order)."""
    t = np.zeros(p.shape[:-1])
    for j in range(p.shape[-1]):
        t = t + p[..., j]
    return t


def _reversed(p):
    return _ascending(p[..., ::-1])


def _tree(p):
    """Pairwise tree over the last axis, padded with zeros to a power of two (the fast lanes' order)."""
    n = 1 << max(0, p.shape[-1] - 1).bit_length()
    t = np.concatenate([p, np.zeros(p.shape[:-1] + (n - p.shape[-1],))], axis=-1)
    while t.shape[-1] > 1:
        t = t[..., ::2] + t[..., 1::2]
    return t[..., 0]


# ------------------------------------------------------------------ mask operators

class MaskOp:
    """Links (1-based, CDO layout), the designed source mask and the kind of every row."""

    def weights(self, mask=None):
        from smmregrid_b200 import CdoWeights
        return CdoWeights({"src_address": self.src, "dst_address": self.dst, "remap_matrix": self.w,
                           "src_grid_imask": self.mask if mask is None else mask,
                           "dst_grid_imask": np.ones(self.n_dst, np.int32), "dst_grid_frac": np.ones(self.n_dst)})


def _candidates(layout, n_dst, rng):
    """Per destination row, the sorted source cells it may link, and n_src."""
    if layout in ("band", "split"):
        span = 24 if layout == "band" else 40
        return [r + np.arange(span) for r in range(n_dst)], n_dst + span + 8
    if layout == "scattered":                       # touched columns 64 apart: no staged segment pays
        pool = 512
        out = []
        for _ in range(n_dst):
            j = np.sort(rng.choice(pool, size=28, replace=False))
            out.append(SCATTER * j + j % 7)
        return out, SCATTER * pool + 100
    assert layout == "healpix"                      # HEALPix nested source (nside 128) -> 2-degree cells
    from smmregrid_b200 import synth
    nside, nlon, nlat = 128, 180, 90
    assert n_dst == nlon * nlat
    f = (np.arange(4) + 0.5) / 4                    # the pixels of 4 x 4 points in the cell
    lat = -90.0 + 2.0 * (np.arange(nlat)[:, None, None, None] + f[None, None, :, None])
    lon = 2.0 * (np.arange(nlon)[None, :, None, None] + f[None, None, None, :])
    pix = synth.ang2pix_nest(nside, lat + 0 * lon, lon + 0 * lat).reshape(n_dst, 16)
    return [np.unique(p) for p in pix], 12 * nside * nside


N_DST = {"band": 1237, "split": 1237, "scattered": 1237, "healpix": 180 * 90}   # partial last 32- and 256-row blocks
KINDS = ("exact", "below", "above", "cancel", "exact", "exact", "below", "cancel", "exact", "above", "exact", "exact")
M = 512                                             # candidate draws per row


def _draw(kind, p_on, n_links, rng, off_w):
    """Weights of one row (ascending source order) whose on-links (positions p_on) sum as `kind`
    wants; off-links (masked-out sources) get off_w.  Returns (weights, kind achieved)."""
    from smmregrid_b200 import synth
    k = len(p_on)
    for attempt in range(20):
        if kind == "cancel" and k == 4:
            g = 0.5 * synth._cubic_taps(rng.random(M))
        else:
            g = 0.5 * rng.dirichlet(np.ones(k), M)
        P = np.zeros((M, n_links))
        P[:, p_on] = g
        a, r, t = _ascending(P), _reversed(P), _tree(P)
        if kind in ("exact", "cancel"):
            ok = (a == 0.5) & ((r != 0.5) | (t != 0.5))
        elif kind == "below":
            ok = (a == BELOW) & ((r == 0.5) | (t == 0.5))
        else:
            ok = (a == ABOVE) & ((r == 0.5) | (t == 0.5))
        if ok.any():
            w = off_w.copy()
            w[p_on] = g[np.argmax(ok)]
            return w, kind
        if attempt >= 3 and kind != "cancel":
            kind = "exact"                          # one-ulp-off draws are rarer: settle for an exact row
    raise AssertionError(f"no draw of kind {kind} for {k} links")


_OPS = {}


def _boundary_op(layout, n_dst=None):
    """Boundary rows of every kind over one layout: 3-8 on-links (4 for cancelling rows) and up to
    16 links in all; every 13th row has no links; in the split layout every 40th row has 20."""
    key = (layout, n_dst)
    if key in _OPS:
        return _OPS[key]
    n_dst = N_DST[layout] if n_dst is None else n_dst
    rng = np.random.default_rng(zlib.crc32(f"{layout}/{n_dst}".encode()))
    cands, n_src = _candidates(layout, n_dst, rng)
    mask = (rng.random(n_src) < 0.55).astype(np.int32)
    src, dst, w, kinds = [], [], [], []
    for r in range(n_dst):
        c = cands[r]
        on_c, off_c = c[mask[c] == 1], c[mask[c] == 0]
        kind = KINDS[r % len(KINDS)]
        if (r % 13 == 0 and n_dst > 1) or len(on_c) < 3:
            kinds.append("empty" if r % 13 == 0 or len(c) == 0 else "plain")
            if kinds[-1] == "plain":
                links = np.sort(rng.choice(c, size=min(len(c), 6), replace=False))
                src.append(links); dst.append(np.full(links.size, r)); w.append(rng.uniform(0.05, 0.5, links.size))
            continue
        k_on = 4 if kind == "cancel" else int(rng.integers(3, 9))
        k_on = min(k_on, len(on_c))
        total = 20 if layout == "split" and r % 40 == 1 else int(rng.integers(k_on, 17))
        k_off = min(len(off_c), total - k_on)
        on = rng.choice(on_c, size=k_on, replace=False)
        links = np.concatenate([on, rng.choice(off_c, size=k_off, replace=False)])
        order = np.argsort(links)
        links = links[order]
        p_on = np.flatnonzero(np.isin(links, on))
        off_w = rng.uniform(-0.5, 0.5, links.size) if kind == "cancel" else rng.uniform(0.05, 0.5, links.size)
        wr, got = _draw(kind, p_on, links.size, rng, off_w)
        src.append(links); dst.append(np.full(links.size, r)); w.append(wr); kinds.append(got)
    op = MaskOp()
    op.layout, op.n_src, op.n_dst, op.mask = layout, int(n_src), int(n_dst), mask
    op.src = (np.concatenate(src) + 1).astype(np.int32)
    op.dst = (np.concatenate(dst) + 1).astype(np.int32)
    op.w = np.concatenate(w).reshape(-1, 1)
    op.kinds = np.array(kinds)
    _OPS[key] = op
    return op


def _duplicates_op(shuffled):
    """Rows whose one on-link appears 2-4 times (the merged weight is 0.5 or one ulp below it,
    depending on the order the copies are added in), plus 0-3 masked-out links: source cell 2r is
    row r's on-link, odd cells are masked out.  The same links in CDO order (dst-major, copies
    adjacent) or shuffled."""
    key = ("dups", shuffled)
    if key in _OPS:
        return _OPS[key]
    rng = np.random.default_rng(4242)
    n_dst = 611
    n_src = 2 * n_dst + 16
    src, dst, w = [], [], []
    for r in range(n_dst):
        m = 2 + r % 3
        big = 0.5 * rng.dirichlet(np.ones(m - 1)) if r % 2 else np.full(m - 1, 0.5 / (m - 1))
        tiny = -rng.choice([2.0 ** -55, 2.0 ** -54, 3 * 2.0 ** -56])
        links = [(2 * r, v) for v in rng.permutation(np.concatenate([big, [tiny]]))]
        links += [(2 * r + 1 + 2 * int(j), rng.uniform(0.1, 0.5)) for j in rng.choice(6, size=r % 4, replace=False)]
        links.sort(key=lambda sv: sv[0])          # stable: the copies keep their order
        src += [s for s, _ in links]
        dst += [r] * len(links)
        w += [v for _, v in links]
    src, dst, w = np.array(src), np.array(dst), np.array(w)
    if shuffled:
        o = np.random.default_rng(99).permutation(src.size)
        src, dst, w = src[o], dst[o], w[o]
    op = MaskOp()
    op.layout, op.n_src, op.n_dst = "dups", n_src, n_dst
    op.src, op.dst = (src + 1).astype(np.int32), (dst + 1).astype(np.int32)
    op.w = w.reshape(-1, 1)
    op.mask = (np.arange(n_src) % 2 == 0).astype(np.int32)
    op.kinds = np.array(["dup"] * n_dst)
    _OPS[key] = op
    return op


MASK_CASES = {
    "boundary-band": lambda: _boundary_op("band"),
    "boundary-scattered": lambda: _boundary_op("scattered"),
    "boundary-healpix": lambda: _boundary_op("healpix"),
    "boundary-split": lambda: _boundary_op("split"),
    "duplicates-cdo-order": lambda: _duplicates_op(False),
    "duplicates-shuffled": lambda: _duplicates_op(True),
    "one-row": lambda: _boundary_op("band", n_dst=1),
    "33-rows": lambda: _boundary_op("band", n_dst=33),
}


def _masks(op):
    """The designed source mask, all zero, all one, and a random one."""
    rng = np.random.default_rng(op.n_dst)
    return {"designed": op.mask, "zeros": np.zeros(op.n_src, np.int32), "ones": np.ones(op.n_src, np.int32),
            "random": (rng.random(op.n_src) < 0.7).astype(np.int32)}


def _matrix(oracle, op):
    if not hasattr(op, "mat"):
        op.mat = oracle.compute_weights_matrix_c(op.src, op.dst, op.w, op.n_src, op.n_dst)
    return op.mat


def _row_sums(mat, mask):
    """Per destination row: the ascending, reversed and pairwise-tree sums of mask[src] * w."""
    o = np.lexsort((mat.src, mat.dst))
    p = mask[mat.src[o]] * mat.w[o]
    b = np.searchsorted(mat.dst[o], np.arange(mat.shape[1] + 1))
    rows = [p[b[r]:b[r + 1]][None] for r in range(mat.shape[1])]
    return tuple(np.array([f(q)[0] for q in rows]) for f in (_ascending, _reversed, _tree))


# ------------------------------------------------------------------ 1a. the constructions discriminate (CPU)

@pytest.mark.parametrize("layout", ["band", "split", "scattered", "healpix"])
def test_boundary_rows_tell_summation_orders_apart(oracle, layout):
    """On the designed mask: >= 20 rows whose reference sum is exactly 0.5, >= 20 rows whose 0/1
    decision flips when the links are summed in reversed order, >= 20 when they are summed as a
    pairwise tree; one-ulp-off rows that another order puts on 0.5; cancelling rows on 0.5; rows
    without links.  A kernel summing in another order, or deciding `t <= 0.5`, fails on them."""
    op = _boundary_op(layout)
    mat = _matrix(oracle, op)
    ref, t = oracle.mask_tensordot_c(op.mask, mat)
    asc, rev, tree = _row_sums(mat, op.mask)
    assert np.array_equal(asc, t)                                   # the oracle sums in ascending-source order
    assert (t == 0.5).sum() >= 20
    assert ((rev < 0.5) != (t < 0.5)).sum() >= 20
    assert ((tree < 0.5) != (t < 0.5)).sum() >= 20
    other_on_half = (rev == 0.5) | (tree == 0.5)
    assert ((t == BELOW) & other_on_half).sum() >= 20 and ((t == ABOVE) & other_on_half).sum() >= 20
    assert ((t == 0.5) & (op.kinds == "cancel")).sum() >= 20
    assert (mat.w < 0).any()
    linkless = np.bincount(mat.dst, minlength=op.n_dst) == 0
    assert linkless.sum() >= 20 and (ref[linkless] == 0).all()
    assert 0 < ref.sum() < op.n_dst


def test_duplicate_links_merge_order_matters(oracle):
    """The same links in CDO order and shuffled: duplicates are merged in input order, and the
    merged weights -- and with them >= 20 mask decisions -- differ between the two orders."""
    a, b = _duplicates_op(False), _duplicates_op(True)
    ma, mb = _matrix(oracle, a), _matrix(oracle, b)
    assert np.array_equal(ma.src, mb.src) and np.array_equal(ma.dst, mb.dst)
    assert ma.nnz < a.src.size
    assert (ma.w != mb.w).sum() >= 20
    ra, ta = oracle.mask_tensordot_c(a.mask, ma)
    rb, tb = oracle.mask_tensordot_c(b.mask, mb)
    assert (ra != rb).sum() >= 20 and ((ta == 0.5) | (tb == 0.5)).sum() >= 100


# ------------------------------------------------------------------ 1b. plan kinds (CPU host plans, GPU handles)

class _Reordered:
    id, env = "reordered-rows", {}


PLAN_KINDS = [(BY_ID["staged-packed-n256-fast"], "band"), (BY_ID["staged-packed-n256-ord"], "band"),
              (BY_ID["staged-l1k16-n256-fast"], "band"), (BY_ID["staged-l1k16-n256-ord"], "band"),
              (BY_ID["ordered-r64-t2"], "band"), (SPLIT, "split"), (_Reordered(), "healpix"),
              (BY_ID["gather-lpr4"], "scattered"), (BY_ID["gather-ord"], "scattered"),
              (BY_ID["compact-bulk-raw"], "scattered")]
PLAN_IDS = [v.id for v, _ in PLAN_KINDS]


def _plan_ok(vid, info):
    """The plan of the recipe: packing, lanes, summation order, kernel family."""
    s = {"kernel": info["kernel"], "packed": info["packed_rows"], "lanes": info["lanes_per_row"],
         "sum": info["summation"], "nct": info["consumer_threads"], "gather_rows": info["gather_rows"],
         "reordered": info["rows_reordered"]}
    staged = s["kernel"] == KERNEL_STAGED
    return {
        "staged-packed-n256-fast": staged and s["packed"] == 1 and s["sum"] == SUM_FAST,
        "staged-packed-n256-ord": staged and s["packed"] == 1 and s["sum"] == SUM_REFERENCE,
        "staged-l1k16-n256-fast": staged and not s["packed"] and s["lanes"] == 1 and info["links_per_lane"] == 16
        and s["sum"] == SUM_FAST,
        "staged-l1k16-n256-ord": staged and not s["packed"] and s["lanes"] == 1 and s["sum"] == SUM_REFERENCE,
        "ordered-r64-t2": staged and not s["packed"] and s["nct"] == 64 and s["sum"] == SUM_REFERENCE,
        SPLIT.id: staged and s["packed"] == 1 and s["gather_rows"] > 0,
        "reordered-rows": staged and s["reordered"] == 1,
        "gather-lpr4": s["kernel"] == KERNEL_GATHER and s["sum"] == SUM_FAST,
        "gather-ord": s["kernel"] == KERNEL_GATHER and s["sum"] == SUM_REFERENCE,
        "compact-bulk-raw": s["kernel"] == KERNEL_GATHER,
    }[vid]


@pytest.mark.parametrize("v,layout", PLAN_KINDS, ids=PLAN_IDS)
def test_boundary_operator_takes_each_plan_kind(smm_lib, v, layout):
    """Host plan (no GPU) of the boundary operator under each recipe: the plan kind it names."""
    from smmregrid_b200 import _lib
    op = _boundary_op(layout)
    h = ctypes.c_void_p()
    with _create_env(v.env):
        _lib.check(smm_lib.smm_host_plan_build(op.n_src, op.n_dst, op.src.size, op.src.ctypes.data, op.dst.ctypes.data,
                                               op.w.ctypes.data, 1, 1, None, ctypes.byref(h)))
    try:
        inf = _lib.SmmInfo()
        _lib.check(smm_lib.smm_host_plan_info(h, ctypes.byref(inf), None))
        info = inf.asdict()
    finally:
        smm_lib.smm_host_plan_free(h)
    assert _plan_ok(v.id, info), (v.id, info)


# ------------------------------------------------------------------ 1c. masks on the device (GPU)

def _mask_sum(lib, wm, level, mask):
    from smmregrid_b200 import _lib
    out = np.full(wm.shape[1], -1, np.int32)
    flag = ctypes.c_int32(-1)
    m = np.ascontiguousarray(mask, np.int32)
    _lib.check(lib.smm_mask_sum(wm.handle, level, m.ctypes.data, out.ctypes.data, ctypes.byref(flag)))
    return out, flag.value


def _check_masks(lib, oracle, op, wm, what):
    """For each source mask: smm_mask_sum's mask and any_masked flag, then mask_weights /
    check_mask on a fresh copy of the weights, against the oracle."""
    from smmregrid_b200 import check_mask, mask_weights
    mat = _matrix(oracle, op)
    for name, mask in _masks(op).items():
        ref, _ = oracle.mask_tensordot_c(mask, mat)
        out, flag = _mask_sum(lib, wm, 0, mask)
        assert np.array_equal(out, ref), f"{what} {name}: {int((out != ref).sum())} of {op.n_dst} decisions differ"
        assert flag == int((ref == 0).any()), (what, name, flag)
        w = mask_weights(op.weights(mask), wm)
        assert np.array_equal(w["dst_grid_imask"], ref), (what, name)
        assert check_mask(w) == oracle.check_mask_np(ref), (what, name)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MASK_CASES))
def test_mask_sum_at_the_boundary(smm_lib, oracle, cuda, case):
    """mask_tensordot: the 0/1 destination mask and the any-masked flag bit for bit, with the
    designed, all-zero, all-one and a random source mask."""
    from smmregrid_b200 import compute_weights_matrix
    op = MASK_CASES[case]()
    wm = compute_weights_matrix(op.weights())
    try:
        _check_masks(smm_lib, oracle, op, wm, case)
    finally:
        wm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("v,layout", PLAN_KINDS, ids=PLAN_IDS)
def test_mask_sum_on_every_plan_kind(smm_lib, oracle, cuda, v, layout):
    """The boundary operator built under each plan kind: the mask reads the CSR every plan keeps."""
    from smmregrid_b200 import compute_weights_matrix
    op = _boundary_op(layout)
    with _create_env(v.env):
        wm = compute_weights_matrix(op.weights())
    try:
        assert _plan_ok(v.id, wm.info()), (v.id, wm.info())
        _check_masks(smm_lib, oracle, op, wm, v.id)
    finally:
        wm.close()


LINKLESS = 2


def _levels(op):
    """A 3-D set over the band boundary operator: all its links; those of its first 600 rows
    (link_length < nl_max); none; all again.  The designed source mask on levels 0 and 1, other
    masks on 2 and 3."""
    from smmregrid_b200 import CdoWeights
    n = op.src.size
    ll = np.array([n, int((op.dst <= 600).sum()), 0, n], np.int64)
    sa, da = np.zeros((4, n), np.int32), np.zeros((4, n), np.int32)
    rm = np.zeros((4, n, 1))
    for l in range(4):
        sa[l, :ll[l]], da[l, :ll[l]], rm[l, :ll[l]] = op.src[:ll[l]], op.dst[:ll[l]], op.w[:ll[l]]
    rng = np.random.default_rng(5)
    masks = np.stack([op.mask, op.mask, (rng.random(op.n_src) < 0.5), np.roll(op.mask, 3)]).astype(np.int32)
    w = CdoWeights({"src_address": sa, "dst_address": da, "remap_matrix": rm, "link_length": ll,
                    "src_grid_imask": masks, "dst_grid_imask": np.ones((4, op.n_dst), np.int32),
                    "dst_grid_frac": np.ones((4, op.n_dst))}, mask_dim="lev", levels=[1.0, 2.0, 3.0, 4.0])
    return w, masks


def _level_refs(oracle, op, w, masks):
    mats = oracle.compute_weights_matrix3d_np(w["src_address"], w["dst_address"], w["remap_matrix"], w["link_length"],
                                              op.n_src, op.n_dst, builder=oracle.compute_weights_matrix_c)
    return mats, np.stack([oracle.mask_tensordot_c(m, mat)[0] for m, mat in zip(masks, mats)])


@pytest.mark.gpu
def test_mask_sum_on_3d_levels_and_from_the_plan_cache(smm_lib, oracle, cuda, tmp_path):
    """mask_weights / check_mask over the levels of a 3-D set (link_length < nl_max, a linkless
    level), built fresh and restored from the plan cache."""
    from smmregrid_b200 import check_mask, compute_weights_matrix3d, mask_weights
    op = _boundary_op("band")
    w, masks = _levels(op)
    _, ref = _level_refs(oracle, op, w, masks)
    assert (ref[LINKLESS] == 0).all() and not np.array_equal(ref[0], ref[1])
    for hit in (0, 1):
        wm = compute_weights_matrix3d(w, "lev", plan_cache_dir=str(tmp_path / "plans"))
        try:
            assert [wm.info(l)["plan_cache_hit"] for l in range(4)] == [hit] * 4
            w2 = mask_weights(w, wm, "lev")
            assert np.array_equal(w2["dst_grid_imask"], ref), [int((w2["dst_grid_imask"][l] != ref[l]).sum())
                                                               for l in range(4)]
            assert np.array_equal(check_mask(w2, "lev"), oracle.check_mask_np(ref))
            for l in range(4):
                assert _mask_sum(smm_lib, wm, l, masks[l])[1] == int((ref[l] == 0).any())
        finally:
            wm.close()


def _apply(lib, wm, level, x):
    """smm_apply of one level, float64 in and out, masked, no frac test."""
    import torch
    from smmregrid_b200 import _lib
    xd = torch.from_numpy(x).cuda()
    y = torch.full((x.shape[0], wm.shape[1]), -7.0, dtype=torch.float64, device="cuda")
    _lib.check(lib.smm_apply(wm.handle, level, xd.data_ptr(), 1, x.shape[0], x.shape[1], y.data_ptr(), 1, wm.shape[1],
                             1, 0.0, None, None))
    torch.cuda.synchronize()
    return y.cpu().numpy()


def _field(n_src, seed):
    rng = np.random.default_rng(seed)
    x = 100.0 * rng.standard_normal((5, n_src))
    x[rng.random(x.shape) < 0.01] = np.nan
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("layout,kernel", [("band", KERNEL_STAGED), ("scattered", KERNEL_GATHER)])
def test_apply_reads_the_latest_mask(smm_lib, oracle, cuda, layout, kernel):
    """mask_weights twice on one handle with different source masks: a masked apply in reference
    order is bit for bit the oracle's apply under the second mask."""
    from smmregrid_b200 import compute_weights_matrix, mask_weights
    op = _boundary_op(layout)
    mat = _matrix(oracle, op)
    second = _masks(op)["random"]
    ref_first, ref_second = oracle.mask_tensordot_c(op.mask, mat)[0], oracle.mask_tensordot_c(second, mat)[0]
    assert (ref_first != ref_second).sum() >= 100
    wm = compute_weights_matrix(op.weights(), summation="reference")
    try:
        assert wm.info()["kernel"] == kernel
        mask_weights(op.weights(), wm)
        mask_weights(op.weights(second), wm)
        x = _field(op.n_src, 1)
        want = oracle.apply_weights_c(x, mat, ref_second, None, 0.0, True)
        y = _apply(smm_lib, wm, 0, x)
        assert _same_bits(y, want), f"{int((np.isnan(y) != np.isnan(want)).sum())} NaN cells differ"
    finally:
        wm.close()


@pytest.mark.gpu
def test_mask_sum_on_one_level_keeps_the_others(smm_lib, oracle, cuda):
    """smm_mask_sum on level 1 of a 3-D handle replaces that level's mask only: every level's
    apply is the oracle's under its own latest mask."""
    from smmregrid_b200 import compute_weights_matrix3d, mask_tensordot, mask_weights
    op = _boundary_op("band")
    w, masks = _levels(op)
    mats, ref = _level_refs(oracle, op, w, masks)
    other = _masks(op)["random"]
    ref = ref.copy()
    ref[1] = oracle.mask_tensordot_c(other, mats[1])[0]
    wm = compute_weights_matrix3d(w, "lev", summation="reference")
    try:
        mask_weights(w, wm, "lev")
        assert np.array_equal(mask_tensordot(other, wm[1]), ref[1])
        x = _field(op.n_src, 2)
        for l in range(4):
            want = oracle.apply_weights_c(x, mats[l], ref[l], None, 0.0, True)
            y = _apply(smm_lib, wm, l, x)
            assert _same_bits(y, want), f"level {l}: {int((np.isnan(y) != np.isnan(want)).sum())} NaN cells differ"
    finally:
        wm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["C4", "C3tri"])
def test_constructor_masks_at_full_size(smm_lib, oracle, cuda, tmp_path, cfg):
    """Regridder(weights=...) at full size with a land/sea source mask: its dst_grid_imask per
    level and its `masked` flags are the oracle's; C4 a second time from the plan cache.  C3tri
    (75 tripolar levels) takes the sea mask of the level below, so that coastal cells are only
    partly covered."""
    from smmregrid_b200 import Regridder, synth
    w = synth.config_weights(cfg)
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    if cfg == "C4":
        masks = synth.ocean_masks(3600, 1800, 4, seed=3)[2:3]      # ~60 % sea, long fractal coasts
        w = w.assign(src_grid_imask=masks[0])
        mats = [oracle.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)]
    else:
        masks = np.roll(w["src_grid_imask"], -1, axis=0)
        w = w.assign(src_grid_imask=masks)
        mats = oracle.compute_weights_matrix3d_np(w["src_address"], w["dst_address"], w["remap_matrix"],
                                                  w["link_length"], n_src, n_dst, builder=oracle.compute_weights_matrix_c)
    sums = [oracle.mask_tensordot_c(m, mat) for m, mat in zip(masks, mats)]
    ref = np.stack([r for r, _ in sums])
    t = np.stack([s for _, s in sums])
    assert ((t > 0.05) & (t < 0.95)).sum() >= 100 and 0 < ref.sum() < ref.size
    for run in range(2 if cfg == "C4" else 1):
        rg = Regridder(weights=w, plan_cache_dir=str(tmp_path / "plans") if cfg == "C4" else None)
        if cfg == "C4":
            assert rg.weights_matrix.info()["plan_cache_hit"] == run
            assert np.array_equal(rg.weights["dst_grid_imask"], ref[0])
            assert rg.masked == oracle.check_mask_np(ref[0]) and rg.masked
        else:
            got = rg.weights["dst_grid_imask"]
            assert np.array_equal(got, ref), [int((got[l] != ref[l]).sum()) for l in range(len(ref))]
            assert np.array_equal(np.asarray(rg.masked), oracle.check_mask_np(ref))
        del rg


# ------------------------------------------------------------------ 2. nan_variation_kernel

NAN_BITS = {                                    # quiet, negative, signalling, negative signalling (, max payload)
    "float16": np.array([0x7e00, 0xfe00, 0x7c01, 0xfc01], np.uint16),
    "bfloat16": np.array([0x7fc0, 0xffc0, 0x7f81, 0xff81], np.uint16),
    "float32": np.array([0x7fc00000, 0xffc00000, 0x7f800001, 0xff800001, 0x7fbfffff], np.uint32),
    "float64": np.array([0x7ff8000000000000, 0xfff8000000000000, 0x7ff0000000000001, 0xfff0000000000001,
                         0x7ff7ffffffffffff], np.uint64),
}
PATTERNS = ("none", "first", "last", "all", "alternate", "inf", "random")


def _pattern(name, outer, n, inner, rng):
    """(NaN cells, +-inf cells as +1 / -1 / 0) of a field viewed as [outer, n, inner].  The
    patterned positions are a random half of them and always the last one (the tail of the last
    warp and block)."""
    nan = np.zeros((outer, n, inner), bool)
    inf = np.zeros((outer, n, inner), np.int8)
    if n == 0:
        return nan, inf
    sel = rng.random((outer, inner)) < 0.5
    sel[-1, -1] = True
    if name == "first":
        nan[:, 0, :] = sel
    elif name == "last":
        nan[:, -1, :] = sel
    elif name == "all":
        nan[:] = True
    elif name == "alternate":
        nan[:, ::2, :] = sel[:, None, :]
    elif name == "inf":                             # +-inf is not missing
        inf[:] = np.where(rng.random(inf.shape) < 0.3, rng.choice(np.array([-1, 1], np.int8), size=inf.shape), 0)
    elif name == "random":
        nan = rng.random(nan.shape) < 0.05
        inf[(rng.random(inf.shape) < 0.02) & ~nan] = 1
    else:
        assert name == "none"
    return nan, inf


def _materialize(nan, inf, dtype, rng):
    """(data, the array the oracle sees): finite values, +-inf, and NaN with payloads drawn from
    NAN_BITS[dtype].  bfloat16 data are uint16 bits; integer data ignore the pattern."""
    if dtype.startswith("int"):
        x = rng.integers(-1000, 1000, size=nan.shape).astype(dtype)
        return x, x
    x = (100.0 * rng.standard_normal(nan.shape)).astype("float32" if dtype == "bfloat16" else dtype)
    x[inf != 0] = inf[inf != 0] * np.inf
    if dtype == "bfloat16":
        bits = (x.view(np.uint32) >> 16).astype(np.uint16)
        bits[nan] = rng.choice(NAN_BITS[dtype], size=int(nan.sum()))
        return bits, (bits.astype(np.uint32) << 16).view(np.float32)
    x.view(NAN_BITS[dtype].dtype)[nan] = rng.choice(NAN_BITS[dtype], size=int(nan.sum()))
    return x, x


def _container(raw, dtype, kind):
    """raw as a numpy array, a CPU tensor, a CUDA tensor, or a non-contiguous CUDA tensor with the
    same values: reversed strides, or every other element of a larger tensor whose other elements
    are NaN (integers: large numbers)."""
    import torch
    if kind == "numpy":
        return raw
    t = torch.from_numpy(raw.view(np.int16)).view(torch.bfloat16) if dtype == "bfloat16" else torch.from_numpy(raw)
    if kind == "cpu":
        return t
    if kind == "cuda":
        return t.cuda()
    if kind == "cuda-transposed":
        perm = tuple(reversed(range(t.dim())))
        return t.permute(perm).contiguous().cuda().permute(perm)
    assert kind == "cuda-strided"                   # every other element along the first and the last axis
    ends = (0, t.dim() - 1)
    sl = tuple(slice(None, None, 2) if d in ends else slice(None) for d in range(t.dim()))
    shape = [2 * n if d in ends else n for d, n in enumerate(t.shape)]
    big = torch.full(shape, 7777 if dtype.startswith("int") else float("nan"), dtype=t.dtype)
    big[sl] = t
    return big.cuda()[sl]


FACTORS = {1: [(), (1, 1)], 31: [(31,)], 32: [(4, 8)], 33: [(3, 11)], 255: [(3, 5, 17)], 256: [(2, 2, 4, 16)],
           257: [(257,)], 4099: [(4099,)]}
N_AXIS = (0, 1, 2, 3, 1000)
SHAPE_CASES = [(p, n) for p in FACTORS for n in N_AXIS]


@pytest.mark.gpu
@pytest.mark.parametrize("positions,n_axis", SHAPE_CASES, ids=[f"pos{p}-n{n}" for p, n in SHAPE_CASES])
def test_nan_variation_count_shapes(smm_lib, oracle, cuda, positions, n_axis):
    """outer * inner positions in {1, 31, 32, 33, 255, 256, 257, 4099} (partial warps, partial
    blocks, several blocks) along an axis of 0, 1, 2, 3 or 1000 elements, that axis at every place of
    ranks 1-5, given as a positive and as a negative axis; every pattern; float32 and float64 with
    NaN payloads."""
    from smmregrid_b200.util import nan_variation_count
    rng = np.random.default_rng(positions * 7919 + n_axis)
    checked = 0
    for fac in FACTORS[positions]:
        for split in range(len(fac) + 1):
            outer_dims, inner_dims = fac[:split], fac[split:]
            outer, inner = int(np.prod(outer_dims)), int(np.prod(inner_dims))
            shape = tuple(outer_dims) + (n_axis,) + tuple(inner_dims)
            for name in PATTERNS:
                nan, inf = _pattern(name, outer, n_axis, inner, rng)
                for dtype in ("float32", "float64"):
                    raw, ref = _materialize(nan, inf, dtype, rng)
                    raw, ref = raw.reshape(shape), ref.reshape(shape)
                    want = oracle.nan_variation_count_np(ref, split)
                    if name in ("none", "all", "inf") or n_axis < 2:
                        assert want == 0
                    elif name in ("first", "last"):
                        assert want == int(nan[:, 0 if name == "first" else -1, :].sum()) and want > 0
                    for axis in (split, split - len(shape)):
                        got = nan_variation_count(raw, axis)
                        assert got == want, (shape, axis, name, dtype, got, want)
                        checked += 1
    assert checked >= 28


INPUTS = ([("float32", c) for c in ("numpy", "cpu", "cuda", "cuda-transposed", "cuda-strided")]
          + [("float64", c) for c in ("numpy", "cpu", "cuda", "cuda-transposed", "cuda-strided")]
          + [("float16", c) for c in ("numpy", "cpu", "cuda", "cuda-transposed", "cuda-strided")]
          + [("bfloat16", c) for c in ("cpu", "cuda", "cuda-transposed", "cuda-strided")]
          + [("int32", "numpy"), ("int64", "cpu"), ("int32", "cuda")])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,container", INPUTS, ids=[f"{d}-{c}" for d, c in INPUTS])
def test_nan_variation_count_inputs(smm_lib, oracle, cuda, dtype, container):
    """Every input dtype (half precision is widened, integers have no NaN) in every container, on
    every axis of three shapes and every pattern, against the oracle on the same values."""
    from smmregrid_b200.util import nan_variation_count
    rng = np.random.default_rng(zlib.crc32(f"{dtype}/{container}".encode()))
    varied = 0
    for shape in ((5, 3, 70), (257, 2), (2, 33, 4)):
        for axis in range(len(shape)):
            outer, inner = int(np.prod(shape[:axis])), int(np.prod(shape[axis + 1:]))
            for name in PATTERNS:
                nan, inf = _pattern(name, outer, shape[axis], inner, rng)
                raw, ref = _materialize(nan, inf, dtype, rng)
                raw, ref = raw.reshape(shape), ref.reshape(shape)
                want = oracle.nan_variation_count_np(ref, axis)
                x = _container(raw, dtype, container)
                got = nan_variation_count(x, axis - len(shape) if name == "alternate" else axis)
                assert got == want, (shape, axis, name, got, want)
                varied += want > 0
    assert (varied > 0) == (not dtype.startswith("int"))


TIME_DIMS = [None, 0, [0], -4, 2, [-2], []]


@pytest.mark.gpu
@pytest.mark.parametrize("container", ["numpy", "cuda"])
@pytest.mark.parametrize("time_dim", TIME_DIMS, ids=[repr(t).replace(" ", "") for t in TIME_DIMS])
def test_detect_nan_variation_dims_time_dim(smm_lib, oracle, cuda, container, time_dim):
    """detect_nan_variation_dims with time_dim None, an int, a one-element list (as the reference
    passes it), a negative int or an empty list: the first step of the time axis is probed, and
    check_dims given as positive and negative axes come back as given."""
    import torch
    from smmregrid_b200 import detect_nan_variation_dims
    rng = np.random.default_rng(11)
    f = rng.standard_normal((3, 4, 5, 6))
    f[0, -1, :, :3] = np.nan                   # step 0: varies along axes 1 and 3
    f[1:, :, 0, :] = np.nan                    # later steps: along axis 2
    f[2, 1, 1, 1] = np.inf
    x = f if container == "numpy" else torch.from_numpy(f).cuda()
    t = time_dim[0] if isinstance(time_dim, list) and time_dim else (None if isinstance(time_dim, list) else time_dim)
    t_axis = None if t is None else t % 4
    check = [0, 1, 2, 3, -1, -3]
    norm = [d % 4 for d in check]
    ref = oracle.detect_nan_variation_dims_np(f, t_axis, sorted(set(norm)))
    want = [d for d, n in zip(check, norm) if n in ref]
    assert detect_nan_variation_dims(x, time_dim, check) == want
    assert want                                 # something varies in every probe


@pytest.mark.gpu
def test_nan_variation_beyond_2_31_positions(smm_lib, cuda):
    """float32 [32771, 2, 65536] (17 GB): 2 147 680 256 positions, beyond 2**31.  NaN placed
    beyond position 2**31 give a count known by construction; then a count beyond 2**31 itself."""
    import torch
    from smmregrid_b200.util import nan_variation_count
    if torch.cuda.mem_get_info()[0] < 40 * 2 ** 30:
        pytest.skip("needs 40 GB of free device memory")
    outer, inner = 2 ** 15 + 3, 2 ** 16
    npos = outer * inner
    assert npos > 2 ** 31
    x = torch.zeros((outer, 2, inner), dtype=torch.float32, device="cuda")
    try:
        def at(pos, k):
            return int(pos // inner), k, int(pos % inner)

        varying = [2 ** 31, 2 ** 31 + 1, 2 ** 31 + 65535, 2 ** 31 + 65536 * 2 + 17, npos - 1]
        steady = [2 ** 31 + 5, npos - 2]             # NaN at both indices: no variation
        for p in varying[:3]:
            x[at(p, 1)] = float("nan")
        for p in varying[3:]:
            x[at(p, 0)] = float("nan")
        for p in steady:
            x[at(p, 0)] = float("nan")
            x[at(p, 1)] = float("nan")
        x[at(2 ** 31 + 9, 1)] = float("inf")
        assert nan_variation_count(x, 1) == len(varying)
        assert nan_variation_count(x, -2) == len(varying)
        x[:, 1, :] = float("nan")                    # now every position varies but the NaN-at-index-0 ones
        assert nan_variation_count(x, 1) == npos - len(varying[3:]) - len(steady)
    finally:
        del x
        torch.cuda.empty_cache()
