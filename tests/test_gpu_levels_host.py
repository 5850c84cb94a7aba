"""Every kernel variant through grouped level launches, the host streaming pipeline and the
plan cache.

test_gpu_variants.py pins each compiled variant to the oracle through smm_apply: one level,
device pointers, a freshly built handle.  Most calls take other routes, each with its own logic
in smm_api.cu:

  * a 3-D weight set runs as grouped launches (smm_apply_levels): up to 128 levels share one
    grid, the group's segment table, footprint and chunking are the maximum over its levels,
    gather launches find their level through item offsets, split plans add a pass over per-level
    row lists, compact launches run one level at a time, and a level whose x is not 16-byte
    aligned leaves the staged group for the gather group of the same call;
  * numpy input streams through smm_apply_host / smm_apply_levels_host: pinned or pageable x and
    y, strided rows, threaded row copies above 4 MB, a ring of device slots that grows with the
    chunk size, a partial last chunk;
  * plan_cache_dir hands back a handle rebuilt from a file.

Every variant of test_gpu_variants.VARIANTS, plus a split plan (short rows packed, long rows
gathered), becomes a 3-D set: its parity operator and two variations of it with the same longest
row, so that the recipe still gives its plan, and a level without links.  Each route must give
the bits smm_apply gives for the same level and rows, and so match the oracle.
"""
import ctypes

import numpy as np
import pytest

from test_gpu_variants import (BY_ID, KERNEL_GATHER, KERNEL_STAGED, SUM_FAST, SUM_REFERENCE, VARIANTS, ZERO_ROW, Op,
                               _backward_scale, _create_env, _diff, _field_parity, _operator, _oracle_result,
                               _same_bits, _seed, expected_info)

F32, F64 = np.float32, np.float64
SENTINEL = -7.0


# ------------------------------------------------------------------ the split recipe

class SplitRecipe:
    """Short rows (<= 16 links) packed, the few long ones (20 links) listed for the gather kernel.
    No compiled variant of its own (the staged part is the packed kernel), so not in VARIANTS."""
    family, id, kernel, ref_order, ldx_pad = "split", "split-packed-fast", KERNEL_STAGED, False, 0
    env = {"SMM_SPLIT": "1", "SMM_SUMMATION": "fast"}
    LONG = 20

    def __repr__(self):
        return self.id


SPLIT = SplitRecipe()
ALL = VARIANTS + [SPLIT]
ALL_BY_ID = {**BY_ID, SPLIT.id: SPLIT}


def _split_operator():
    """Band operator of 0-8 link rows and every 40th row with 20 links, with the special rows of
    the parity operators (a weight-0 missing source, a sum below -3.4e38)."""
    if "split" in _SPLIT_OP:
        return _SPLIT_OP["split"]
    rng = np.random.default_rng(_seed(SPLIT.id, "parity"))
    n_dst = 3001
    counts = rng.integers(0, 9, size=n_dst)
    counts[::40] = SplitRecipe.LONG
    counts[ZERO_ROW], counts[n_dst - 2] = 2, 4
    span = SplitRecipe.LONG + 9
    src = np.concatenate([r + np.sort(rng.choice(span, size=n, replace=False)) for r, n in enumerate(counts)])
    dst = np.repeat(np.arange(n_dst), counts)
    w = rng.random(dst.size)
    starts = np.concatenate([[0], np.cumsum(counts)])
    w[starts[ZERO_ROW]] = 0.0
    w[starts[n_dst - 2]:starts[n_dst - 1]] = 0.9
    op = Op()
    op.n_dst, op.n_src = n_dst, -(-(n_dst + span) // 8) * 8 + 8
    op.zero_cols = src[starts[ZERO_ROW]:starts[ZERO_ROW + 1]]
    op.big_cols = src[starts[n_dst - 2]:starts[n_dst - 1]]
    op.imask = (rng.random(n_dst) > 0.1).astype(np.int32)
    op.frac = rng.uniform(0.4, 1.0, n_dst)
    for r in (ZERO_ROW, n_dst - 2):
        op.imask[r], op.frac[r] = 1, 1.0
    op.src, op.dst, op.w = (src + 1).astype(np.int32), (dst + 1).astype(np.int32), w.reshape(-1, 1)
    op.counts, op.max_row = counts, int(counts.max())
    op.masked, op.amin, op.ldx = True, 0.5, op.n_src
    _SPLIT_OP["split"] = op
    return op


_SPLIT_OP = {}


def _expected(v):
    if v is SPLIT:
        return dict(kernel=KERNEL_STAGED, packed_rows=1, lanes_per_row=1, links_per_lane=16, consumer_threads=256,
                    rows_per_tile=1024, summation=SUM_FAST)
    return expected_info(v)


def _base_operator(v):
    return _split_operator() if v is SPLIT else _operator(v, "parity")


# ------------------------------------------------------------------ 3-D weight sets

N_LEVELS = 4
EMPTY = 3                       # the level without links


def _level_op(base, src0, dst0, w, imask, frac, masked):
    op = Op()
    op.n_src, op.n_dst, op.ldx, op.amin = base.n_src, base.n_dst, base.ldx, base.amin
    o = np.lexsort((src0, dst0))
    op.src, op.dst, op.w = (src0[o] + 1).astype(np.int32), (dst0[o] + 1).astype(np.int32), w[o].reshape(-1, 1)
    op.imask, op.frac, op.masked = imask.astype(np.int32), frac, masked
    op.counts = np.bincount(dst0, minlength=base.n_dst)
    return op


_LEVELS = {}


def _level_ops(v):
    """Level 0: the variant's parity operator.  Level 1: every odd row (every row of a packed
    plan: fewer sub-rows, fewer tiles) that is shorter than the longest keeps the first half of its
    links, other weights and masks, not masked.  Level 2: the rows permuted (some plans then tile
    them re-ordered), other weights, another mask.  Level 3: no links, every cell masked (what
    mask_sum makes of it).  Every data level has the same longest row."""
    if v.id in _LEVELS:
        return _LEVELS[v.id]
    base = _base_operator(v)
    rng = np.random.default_rng(_seed(v.id, "levels"))
    src0, dst0, w0 = base.src.astype(np.int64) - 1, base.dst.astype(np.int64) - 1, base.w[:, 0]
    n_dst = base.n_dst
    counts = np.bincount(dst0, minlength=n_dst)
    starts = np.concatenate([[0], np.cumsum(counts)])
    keep = np.ones(src0.size, bool)
    packed = v.family == "staged" and v.key[3]
    for r in range(0 if packed else 1, n_dst, 1 if packed else 2):
        if 2 <= counts[r] < base.max_row and r not in (ZERO_ROW, n_dst - 2):
            keep[starts[r] + (counts[r] + 1) // 2:starts[r + 1]] = False
    perm = rng.permutation(n_dst)
    ops = [
        _level_op(base, src0, dst0, w0, base.imask, base.frac, True),
        _level_op(base, src0[keep], dst0[keep], w0[keep] * rng.uniform(0.5, 1.5, keep.sum()),
                  np.roll(base.imask, 7), rng.uniform(0.4, 1.0, n_dst), False),
        _level_op(base, src0, perm[dst0], w0 * rng.uniform(0.5, 1.5, w0.size),
                  (rng.random(n_dst) > 0.2).astype(np.int32), rng.uniform(0.4, 1.0, n_dst), True),
        _level_op(base, np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0), np.zeros(n_dst, np.int32),
                  np.ones(n_dst), True),
    ]
    for op in ops[:3]:
        assert op.counts.max() == base.max_row
    _LEVELS[v.id] = ops
    return ops


def _create_levels(lib, v, ops, cache_dir=None, summation=None):
    from smmregrid_b200 import _lib
    ll = np.array([op.src.size for op in ops], np.int64)
    nl = max(int(ll.max()), 1)
    sa = np.zeros((len(ops), nl), np.int32)
    da = np.zeros((len(ops), nl), np.int32)
    rm = np.zeros((len(ops), nl, 1))
    for l, op in enumerate(ops):
        sa[l, :ll[l]], da[l, :ll[l]], rm[l, :ll[l]] = op.src, op.dst, op.w
    h = ctypes.c_void_p()
    with _create_env(v.env):
        _lib.check(lib.smm_create_levels(len(ops), ll.ctypes.data, nl, ops[0].n_src, ops[0].n_dst, sa.ctypes.data,
                                         da.ctypes.data, rm.ctypes.data, 1, 1, 0,
                                         _lib.create_opts(summation, cache_dir), ctypes.byref(h)))
    try:
        for l, op in enumerate(ops):
            _lib.check(lib.smm_set_dst_mask(h, l, op.imask.ctypes.data, op.frac.ctypes.data))
    except BaseException:
        lib.smm_destroy(h)
        raise
    return h


def _infos(lib, h, n):
    from smmregrid_b200 import _lib
    out = []
    for l in range(n):
        inf = _lib.SmmInfo()
        _lib.check(lib.smm_get_info(h, l, ctypes.byref(inf)))
        out.append(inf.asdict())
    return out


def _check_plans(v, ops, infos):
    """Every data level has the recipe's plan; packed and split levels differ in tile count."""
    want = _expected(v)
    for l, (op, got) in enumerate(zip(ops, infos)):
        if l == EMPTY:
            assert got["nnz"] == 0 and got["summation"] == want["summation"], (v.id, got)
            continue
        assert {k: got[k] for k in want} == want, (v.id, l, got)
        if v.family in ("staged", "ordered"):
            assert got["gather_rows"] == 0, (v.id, l, got)
        if v is SPLIT:
            assert got["gather_rows"] == int((op.counts > 16).sum()) > 0, (v.id, l, got)
    if infos[0]["packed_rows"]:
        assert len({infos[l]["n_tiles"] for l in range(3)}) > 1, (v.id, [i["n_tiles"] for i in infos])


# ------------------------------------------------------------------ device calls

def _dt(d):
    return 0 if d == F32 else 1


def _torch_dt(d):
    import torch
    return torch.float32 if d == F32 else torch.float64


def _slot_fields(v, xdt, B, n):
    """Data of n slots: the parity field, rolled over the batch and scaled, one per slot, so that
    a slot that reads or writes another slot's rows shows."""
    base = _field_parity(_base_operator(v), v, F64, B)
    out = []
    with np.errstate(over="ignore"):
        for i in range(n):
            out.append((np.roll(base, i, axis=0) * ((-1.0) ** i * (1.0 + 0.25 * i))).astype(xdt))
    return out


def _apply_one(lib, h, kernel, op, level, x_dev_ptr, xdt, ydt, B, ldx):
    """smm_apply of one level into a fresh [B, n_dst] device array (kernel: SMM_KERNEL_*, 0 = automatic)."""
    import torch
    from smmregrid_b200 import _lib
    y = torch.full((B, op.n_dst), SENTINEL, dtype=_torch_dt(ydt), device="cuda")
    _lib.check(lib.smm_apply(h, level, x_dev_ptr, _dt(xdt), B, ldx, y.data_ptr(), _dt(ydt), op.n_dst,
                             int(op.masked), op.amin, _lib.apply_opts(kernel), None))
    return y


def _apply_grouped(lib, h, kernel, ops, sel, fields, xdt, ydt, B, layout, level_pad=0):
    """smm_apply_levels of data slots i = 0.. (weight level sel[i], data fields[i]) in the
    [B, L, n] or [L, B, n] layout; level_pad elements between levels of x ([L, B, n] only).
    Returns y as [L, B, n_dst] (numpy) and the launches it took."""
    import torch
    from smmregrid_b200 import _lib
    n, ldx, n_dst = len(sel), ops[0].ldx, ops[0].n_dst
    if layout == "BLn":
        assert level_pad == 0
        xs = torch.zeros((B, n, ldx), dtype=_torch_dt(xdt), device="cuda")
        for i in range(n):
            xs[:, i, :ops[0].n_src] = torch.from_numpy(fields[i]).cuda()
        xbs, xls = n * ldx, ldx
        y = torch.full((B, n, n_dst), SENTINEL, dtype=_torch_dt(ydt), device="cuda")
        ybs, yls = n * n_dst, n_dst
    else:
        xls = B * ldx + level_pad
        xs = torch.zeros(n * xls, dtype=_torch_dt(xdt), device="cuda")
        for i in range(n):
            xs[i * xls:i * xls + B * ldx].view(B, ldx)[:, :ops[0].n_src] = torch.from_numpy(fields[i]).cuda()
        xbs = ldx
        y = torch.full((n, B, n_dst), SENTINEL, dtype=_torch_dt(ydt), device="cuda")
        ybs, yls = n_dst, B * n_dst
    idx = np.asarray(sel, np.int32)
    masked = np.array([ops[l].masked for l in sel], np.uint8)
    torch.cuda.synchronize()
    n0 = lib.smm_launch_count()
    _lib.check(lib.smm_apply_levels(h, n, idx.ctypes.data, xs.data_ptr(), _dt(xdt), B, xbs, xls, y.data_ptr(),
                                    _dt(ydt), ybs, yls, masked.ctypes.data, ops[0].amin, _lib.apply_opts(kernel),
                                    None))
    torch.cuda.synchronize()
    launches = lib.smm_launch_count() - n0
    y = y.cpu().numpy()
    return (np.moveaxis(y, 1, 0) if layout == "BLn" else y), launches, xs, xls


def _check_against_oracle(oracle, ref_order, op, x, y64, what):
    """Bits for reference-order sums, 1e-12 sum |w| |x_filled| for fast ones."""
    ref = _oracle_result(oracle, op, x)
    assert np.array_equal(np.isnan(y64), np.isnan(ref)), what + ": NaN pattern, " + _diff(y64, ref)
    if ref_order:
        assert _same_bits(y64, ref), what + ": " + _diff(y64, ref)
        return
    assert np.array_equal(np.isinf(y64), np.isinf(ref)), what
    fin = ~np.isnan(ref) & np.isfinite(ref)
    err = np.abs(y64[fin] - ref[fin])
    assert np.all(err <= 1e-12 * np.maximum(_backward_scale(op, x)[fin], 1e-300)), (what, err.max())


# ------------------------------------------------------------------ 1-2. grouped device launches (GPU)

GROUP_B = (1, 7, 37)
GROUP_DTYPES = [(F32, F64), (F64, F32)]
SELECTIONS = {"all": [0, 1, 2, 3], "permuted": [3, 2, 0, 0, 1]}


@pytest.mark.gpu
@pytest.mark.parametrize("xdt,ydt", GROUP_DTYPES, ids=["f32-f64", "f64-f32"])
@pytest.mark.parametrize("v", ALL, ids=[v.id for v in ALL])
def test_grouped_levels_match_single_levels(smm_lib, oracle, cuda, v, xdt, ydt):
    """smm_apply_levels over all levels, and over a permuted selection with a repeated level, in
    both stride layouts: every data slot is bit-identical to smm_apply of its level on the same
    rows (and so within the oracle's bound, or bit-identical to it in reference order); the
    linkless level is all NaN.  At B = 7 also: x levels that are not 16-byte aligned (staged and
    gather launches in one call), and more than 128 selected levels (two launches per group)."""
    import torch
    ops = _level_ops(v)
    h = _create_levels(smm_lib, v, ops)
    try:
        _check_plans(v, ops, _infos(smm_lib, h, N_LEVELS))
        for B in GROUP_B:
            fields = _slot_fields(v, xdt, B, 5)
            dev = [None] * 5
            single = {}

            def reference(level, i, kernel=v.kernel):
                """smm_apply of weight level `level` on slot i's data; with the recipe's kernel,
                checked against the oracle (float64 output) the first time it is asked for."""
                if (level, i, kernel) not in single:
                    if dev[i] is None:
                        dev[i] = torch.zeros((B, ops[0].ldx), dtype=_torch_dt(xdt), device="cuda")
                        dev[i][:, :ops[0].n_src] = torch.from_numpy(fields[i]).cuda()
                    op = ops[level]
                    y = _apply_one(smm_lib, h, kernel, op, level, dev[i].data_ptr(), xdt, ydt, B, op.ldx)
                    if level != EMPTY and kernel == v.kernel:
                        y64 = _apply_one(smm_lib, h, kernel, op, level, dev[i].data_ptr(), xdt, F64, B, op.ldx)
                        _check_against_oracle(oracle, v.ref_order, op, fields[i], y64.cpu().numpy(),
                                              f"{v.id} B={B} level {level} slot {i}")
                    torch.cuda.synchronize()
                    single[(level, i, kernel)] = y.cpu().numpy()
                return single[(level, i, kernel)]

            for name, sel in SELECTIONS.items():
                for layout in ("BLn", "LBn"):
                    y = _apply_grouped(smm_lib, h, v.kernel, ops, sel, fields, xdt, ydt, B, layout)[0]
                    for i, level in enumerate(sel):
                        what = f"{v.id} B={B} {name} {layout} slot {i} (level {level})"
                        assert _same_bits(y[i], reference(level, i)), what + ": " + _diff(y[i], reference(level, i))
                        if level == EMPTY:
                            assert np.isnan(y[i]).all(), what
            if B != 7:
                continue
            # The automatic kernel choice from here on: a staged level whose x is not 16-byte
            # aligned moves to the gather kernel (forcing the staged kernel would fail), and the
            # launch count below is that of the grouped launches (a forced compact path runs
            # level by level).  Levels 1 element apart beyond B rows: only level 0 stays aligned.
            sel = SELECTIONS["all"]
            y, _, xs, xls = _apply_grouped(smm_lib, h, 0, ops, sel, fields, xdt, ydt, B, "LBn", level_pad=1)
            # (at B = 7 the compact recipes take the gather kernel with fast sums)
            ref_order = v.ref_order and v.family != "compact"
            for i, level in enumerate(sel):
                what = f"{v.id} B={B} unaligned slot {i}"
                ptr = xs.data_ptr() + i * xls * xs.element_size()
                yi = _apply_one(smm_lib, h, 0, ops[level], level, ptr, xdt, ydt, B, ops[0].ldx)
                torch.cuda.synchronize()
                yi = yi.cpu().numpy()
                assert _same_bits(y[i], yi), what + ": " + _diff(y[i], yi)
                if ref_order or level == EMPTY or i == 0:
                    want = reference(level, i, 0)
                    assert _same_bits(y[i], want), what + ": " + _diff(y[i], want)
                elif ydt == F64:
                    _check_against_oracle(oracle, False, ops[level], fields[i], y[i], what)
            # 130 selected levels: each group is split in two launches
            many = [i % 3 for i in range(130)]
            n64 = _apply_grouped(smm_lib, h, 0, ops, many[:64], [fields[i % 3] for i in range(64)],
                                 xdt, ydt, B, "BLn")[1]
            y, n130, _, _ = _apply_grouped(smm_lib, h, 0, ops, many, [fields[i % 3] for i in range(130)],
                                           xdt, ydt, B, "BLn")
            assert n64 in (1, 2) and n130 == 2 * n64, (v.id, n64, n130)
            for i, level in enumerate(many):
                want = reference(level, level, 0)
                assert _same_bits(y[i], want), f"{v.id} 130 levels, slot {i}: " + _diff(y[i], want)
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ 3. host streaming (GPU)

HOST_VARIANTS = ["staged-l1k12-n256-fast", "staged-l2k14-n256-ord", "staged-packed-n256-fast", SPLIT.id,
                 "ordered-r64-t2", "gather-lpr4", "compact-bulk-raw"]
HOST_B = (1, 37, 200)
HOST_SEL = [3, 2, 0, 0, 1]


def _host_array(shape, dtype, pinned, keep, offset=0):
    """A zeroed host array, pinned (page-locked through torch) or pageable, starting `offset`
    elements into its allocation."""
    import torch
    n = int(np.prod(shape)) + offset
    if pinned:
        t = torch.zeros(n, dtype=_torch_dt(dtype), pin_memory=True)
        keep.append(t)
        flat = t.numpy()
    else:
        flat = np.zeros(n, dtype)
    return flat[offset:].reshape(shape)


def _chunks(B):
    return list(dict.fromkeys((0, 1, 7, B - 1, B)))          # (B = 1: B - 1 = 0, the automatic size)


def _rows_per_chunk(chunk_rows, B, row_bytes, x_pinned):
    """The pipeline's chunk: chunk_rows, or for 0 about 128 MB (pinned x) / 64 MB (pageable x) of
    source, at least 4 rows; never more than B."""
    if chunk_rows <= 0:
        chunk_rows = max(4, ((128 if x_pinned else 64) << 20) // row_bytes)
    return min(chunk_rows, B)


def _device_chunked(fn, B, chunk):
    """Rows [0, B) as the pipeline cuts them: one device apply per chunk."""
    return np.concatenate([fn(b0, min(chunk, B - b0)) for b0 in range(0, B, chunk)])


@pytest.mark.gpu
@pytest.mark.parametrize("vid", HOST_VARIANTS)
def test_host_streaming_matches_device_apply(smm_lib, cuda, vid):
    """smm_apply_host (f32 -> f64, padded and contiguous rows) and smm_apply_levels_host (f64 ->
    f32, a permuted selection with a repeated level) with x and y each pinned or pageable, at
    chunk_rows 0 (automatic), 1, 7, B - 1 and B: every output is bit-identical to the device
    apply of the same chunks of rows, and padding cells of y keep their sentinel.  Chunks grow
    from call to call on one handle, so the slot ring is reallocated along the way."""
    import torch
    from smmregrid_b200 import _lib
    v = ALL_BY_ID[vid]
    ops = _level_ops(v)
    n_src, n_dst = ops[0].n_src, ops[0].n_dst
    h = _create_levels(smm_lib, v, ops)
    keep = []
    try:
        for B in HOST_B:
            fields = _slot_fields(v, F64, B, len(HOST_SEL))
            x32 = fields[0].astype(F32)
            x32_dev = torch.from_numpy(x32).cuda()
            xl = np.stack(fields, axis=1)                                 # [B, n_sel, n_src] float64
            xl_dev = torch.from_numpy(xl).cuda()
            idx = np.asarray(HOST_SEL, np.int32)
            masked = np.array([ops[l].masked for l in HOST_SEL], np.uint8)
            nsel = len(HOST_SEL)

            def dev_one(b0, nb):
                y = _apply_one(smm_lib, h, v.kernel, ops[0], 0, x32_dev[b0:].data_ptr(), F32, F64, nb, n_src)
                torch.cuda.synchronize()
                return y.cpu().numpy()

            def dev_levels(b0, nb):
                y = torch.full((nb, nsel, n_dst), SENTINEL, dtype=torch.float32, device="cuda")
                _lib.check(smm_lib.smm_apply_levels(h, nsel, idx.ctypes.data, xl_dev[b0:].data_ptr(), 1, nb,
                                                    nsel * n_src, n_src, y.data_ptr(), 0, nsel * n_dst, n_dst,
                                                    masked.ctypes.data, ops[0].amin, _lib.apply_opts(v.kernel), None))
                torch.cuda.synchronize()
                return y.cpu().numpy()

            refs1, refsl = {}, {}
            for chunk in _chunks(B):
                for x_pin in (False, True):
                    c1 = _rows_per_chunk(chunk, B, n_src * 4, x_pin)
                    cl = _rows_per_chunk(chunk, B, nsel * n_src * 8, x_pin)
                    if c1 not in refs1:
                        refs1[c1] = _device_chunked(dev_one, B, c1)
                    if cl not in refsl:
                        refsl[cl] = _device_chunked(dev_levels, B, cl)
                    want1, wantl = refs1[c1], refsl[cl]
                    for y_pin in (False, True):
                        what = f"{vid} B={B} chunk_rows={chunk} x {'pinned' if x_pin else 'pageable'} " \
                               f"y {'pinned' if y_pin else 'pageable'}"
                        for ldx, ldy in ((n_src, n_dst), (n_src + 3, n_dst + 5)):
                            x = _host_array((B, ldx), F32, x_pin, keep)
                            x[:, :n_src] = x32
                            y = _host_array((B, ldy), F64, y_pin, keep)
                            y[:] = SENTINEL
                            _lib.check(smm_lib.smm_apply_host(h, 0, x.ctypes.data, 0, B, ldx, y.ctypes.data, 1, ldy,
                                                              int(ops[0].masked), ops[0].amin,
                                                              _lib.apply_opts(v.kernel), chunk))
                            assert _same_bits(y[:, :n_dst], want1), f"{what} ldx={ldx}: " + _diff(y[:, :n_dst], want1)
                            assert (y[:, n_dst:] == SENTINEL).all(), f"{what} ldy={ldy}: padding overwritten"
                        x = _host_array(xl.shape, F64, x_pin, keep)
                        x[:] = xl
                        y = _host_array((B, nsel, n_dst), F32, y_pin, keep)
                        y[:] = SENTINEL
                        _lib.check(smm_lib.smm_apply_levels_host(h, nsel, idx.ctypes.data, x.ctypes.data, 1, B,
                                                                 y.ctypes.data, 0, masked.ctypes.data, ops[0].amin,
                                                                 _lib.apply_opts(v.kernel), chunk))
                        assert _same_bits(y, wantl), f"{what} levels: " + _diff(y, wantl)
                        assert np.isnan(y[:, 0]).all(), what           # slot 0 is the linkless level
                        keep.clear()
    finally:
        smm_lib.smm_destroy(h)


@pytest.mark.gpu
def test_host_streaming_threaded_copies(smm_lib, cuda):
    """Chunks above 4 MB of pageable x are staged by several threads with non-temporal stores.
    Rows of 131 472 bytes (not a multiple of 64), a source pointer 4 bytes into its allocation, a
    padded row stride, a partial last chunk below 4 MB; then a second call with larger chunks on
    the same handle.  Bit-identical to the device apply of the same chunks."""
    import torch
    from smmregrid_b200 import _lib
    v = BY_ID["gather-lpr4"]
    ops = _level_ops(v)
    op = ops[0]
    n_src, n_dst, B = op.n_src, op.n_dst, 64
    assert (n_src * 4) % 64 != 0 and 40 * n_src * 4 > 4 << 20 > 24 * n_src * 4
    x32 = _slot_fields(v, F32, B, 1)[0]
    x_dev = torch.from_numpy(x32).cuda()
    h = _create_levels(smm_lib, v, ops)
    keep = []
    try:
        def dev_one(b0, nb):
            y = _apply_one(smm_lib, h, 0, op, 0, x_dev[b0:].data_ptr(), F32, F32, nb, n_src)
            torch.cuda.synchronize()
            return y.cpu().numpy()

        ldx, ldy = n_src + 3, n_dst + 1
        x = _host_array((B, ldx), F32, False, keep, offset=1)
        assert x.ctypes.data % 8 == 4
        x[:, :n_src] = x32
        for chunk in (40, B):
            want = _device_chunked(dev_one, B, chunk)
            for y_pin in (False, True):
                y = _host_array((B, ldy), F32, y_pin, keep, offset=1)
                y[:] = SENTINEL
                _lib.check(smm_lib.smm_apply_host(h, 0, x.ctypes.data, 0, B, ldx, y.ctypes.data, 0, ldy,
                                                  int(op.masked), op.amin, None, chunk))
                what = f"chunk_rows={chunk} y {'pinned' if y_pin else 'pageable'}"
                assert _same_bits(y[:, :n_dst], want), what + ": " + _diff(y[:, :n_dst], want)
                assert (y[:, n_dst:] == SENTINEL).all(), what
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ 4. plan cache

CACHE_VARIANTS = ["staged-l1k12-n256-fast", "staged-l4k16-n512-fast", "staged-l2k14-n256-ord",
                  "staged-packed-n256-fast", "staged-packed-n256-ord", SPLIT.id, "ordered-r64-t2", "ordered-r256-t1",
                  "gather-lpr4", "gather-ord", "compact-bulk-raw", "compact-element-fill"]


def _strip(info):
    return {k: val for k, val in info.items() if k != "plan_cache_hit"}


@pytest.mark.gpu
@pytest.mark.parametrize("vid", CACHE_VARIANTS)
def test_plan_cache_restores_every_plan_kind_as_3d_set(smm_lib, cuda, tmp_path, vid):
    """Created twice under the recipe's switches with one cache directory: the second handle is
    a hit on every level, reports the same plans and gives the same bits."""
    v = ALL_BY_ID[vid]
    ops = _level_ops(v)
    cache = str(tmp_path / "plans")
    infos, outs = [], []
    for _ in range(2):
        h = _create_levels(smm_lib, v, ops, cache_dir=cache)
        try:
            infos.append(_infos(smm_lib, h, N_LEVELS))
            fields = _slot_fields(v, F32, 37, 5)
            outs.append(_apply_grouped(smm_lib, h, v.kernel, ops, SELECTIONS["permuted"], fields, F32, F64, 37,
                                       "BLn")[0])
        finally:
            smm_lib.smm_destroy(h)
    assert [i["plan_cache_hit"] for i in infos[0]] == [0] * N_LEVELS
    assert [i["plan_cache_hit"] for i in infos[1]] == [1] * N_LEVELS
    _check_plans(v, ops, infos[1])
    assert [_strip(i) for i in infos[0]] == [_strip(i) for i in infos[1]]
    assert _same_bits(outs[0], outs[1]), vid + ": " + _diff(outs[0], outs[1])


class _LongRows:
    id, env, kernel, ref_order = "long-rows", {}, 0, True


def _long_row_ops():
    """Two levels with weights of both signs; level 0 has rows of 513 and 600 links, which no
    staged layout holds, so the whole set is served by the gather kernel."""
    rng = np.random.default_rng(513)
    n_src, n_dst = 4096, 300
    ops = []
    for level in range(2):
        counts = rng.integers(0, 41, size=n_dst)
        if level == 0:
            counts[5], counts[17] = 513, 600
        dst = np.repeat(np.arange(n_dst), counts)
        src = np.concatenate([np.sort(rng.choice(n_src, size=n, replace=False)) for n in counts])
        op = Op()
        op.n_src, op.n_dst, op.ldx, op.amin, op.masked = n_src, n_dst, n_src, 0.0, False
        op.src, op.dst = (src + 1).astype(np.int32), (dst + 1).astype(np.int32)
        op.w = rng.standard_normal((dst.size, 1))
        op.imask, op.frac = np.ones(n_dst, np.int32), np.ones(n_dst)
        ops.append(op)
    return ops


@pytest.mark.gpu
@pytest.mark.parametrize("summation", [None, "reference"])
def test_long_rows_keep_reference_order_from_the_cache(smm_lib, oracle, cuda, tmp_path, summation):
    """Rows over 512 links with weights of both signs: gather kernel, reference-order sums, built
    fresh and rebuilt from the plan cache; bit-identical to the oracle with the gather kernel
    forced and by default, for float32 and float64 input."""
    import torch
    from smmregrid_b200 import _lib
    v = _LongRows()
    ops = _long_row_ops()
    cache = str(tmp_path / "plans")
    rng = np.random.default_rng(600)
    for hit in (0, 1):
        h = _create_levels(smm_lib, v, ops, cache_dir=cache, summation=summation)
        try:
            for l, info in enumerate(_infos(smm_lib, h, 2)):
                assert info["plan_cache_hit"] == hit and info["kernel"] == KERNEL_GATHER, (hit, l, info)
                assert info["summation"] == SUM_REFERENCE, (hit, l, info)
            for xdt in (F32, F64):
                x = (100.0 * rng.standard_normal((9, ops[0].n_src))).astype(xdt)
                x[rng.random(x.shape) < 0.01] = np.nan
                xd = torch.from_numpy(x).cuda()
                for l, op in enumerate(ops):
                    ref = _oracle_result(oracle, op, x)
                    for kernel in (0, KERNEL_GATHER):
                        y = _apply_one(smm_lib, h, kernel, op, l, xd.data_ptr(), xdt, F64, x.shape[0], op.ldx)
                        torch.cuda.synchronize()
                        y = y.cpu().numpy()
                        assert _same_bits(y, ref), f"cache hit {hit} level {l} {np.dtype(xdt).name} kernel {kernel}: " \
                            + _diff(y, ref)
        finally:
            smm_lib.smm_destroy(h)


def _host_plan_info(lib, op, cache_dir, env, summation=None):
    from smmregrid_b200 import _lib
    h = ctypes.c_void_p()
    with _create_env(env):
        _lib.check(lib.smm_host_plan_build(op.n_src, op.n_dst, op.src.size, op.src.ctypes.data, op.dst.ctypes.data,
                                           op.w.ctypes.data, 1, 1, _lib.create_opts(summation, cache_dir),
                                           ctypes.byref(h)))
    try:
        inf = _lib.SmmInfo()
        _lib.check(lib.smm_host_plan_info(h, ctypes.byref(inf), None))
        return inf.asdict()
    finally:
        lib.smm_host_plan_free(h)


@pytest.mark.parametrize("switch,value", [("SMM_SPLIT", "0"), ("SMM_ORDLONG", "0"), ("SMM_ORD_ROWS", "64"),
                                          ("SMM_SUMMATION", "fast"), ("SMM_SUMMATION", "reference"),
                                          ("SMM_FORCE_LANES", "8,16"), ("SMM_CONSUMER_THREADS", "512"),
                                          ("SMM_PACKED", "0")])
def test_plan_cache_key_covers_plan_switches(smm_lib, tmp_path, switch, value):
    """A switch that shapes the plan, changed between two builds, is a cache miss; the file
    written under it then serves exactly the plan a build without the cache gives."""
    op = _split_operator()
    neg = Op()
    neg.__dict__.update(op.__dict__)
    neg.w = op.w * np.where(np.arange(op.w.shape[0]) % 5 == 0, -1.0, 1.0)[:, None]     # reference order by default
    cache = str(tmp_path / "plans")
    for o in (op, neg):
        first = _host_plan_info(smm_lib, o, cache, {})
        assert first["plan_cache_hit"] == 0
        assert _host_plan_info(smm_lib, o, cache, {})["plan_cache_hit"] == 1
        fresh = _host_plan_info(smm_lib, o, None, {switch: value})
        miss = _host_plan_info(smm_lib, o, cache, {switch: value})
        hit = _host_plan_info(smm_lib, o, cache, {switch: value})
        assert miss["plan_cache_hit"] == 0 and hit["plan_cache_hit"] == 1, (switch, value)
        assert _strip(hit) == _strip(fresh) == _strip(miss), (switch, value)
        assert _strip(_host_plan_info(smm_lib, o, cache, {})) == _strip(first)


@pytest.mark.parametrize("summation", [None, "reference", "fast"])
def test_long_row_plan_reports_its_summation(smm_lib, tmp_path, summation):
    """Rows over 512 links (no staged plan) with weights of both signs sum in reference order by
    default: the host plan says so, built fresh and from the plan cache."""
    op = _long_row_ops()[0]
    want = SUM_FAST if summation == "fast" else SUM_REFERENCE
    cache = str(tmp_path / "plans")
    for hit in (0, 1):
        info = _host_plan_info(smm_lib, op, cache, {}, summation)
        assert info["plan_cache_hit"] == hit and info["kernel"] == KERNEL_GATHER, info
        assert info["summation"] == want, (hit, info)
