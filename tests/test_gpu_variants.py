"""Every compiled kernel variant against the oracle.

The dispatch tables of smmregrid_b200/csrc/smm_launch.cuh instantiate many staged and ordered
kernels, and the launch logic adds gather and two-pass compact variants.  Which of them a call
reaches depends on the operator (longest row, mean row length, source layout), on create-time
switches (SMM_FORCE_LANES, SMM_PACKED, SMM_CONSUMER_THREADS, SMM_SUMMATION, SMM_ORDLONG,
SMM_ORD_ROWS), on the batch size and on a few process-wide switches.  This file keeps one explicit
list of the variants with the recipe that reaches each of them and checks:

  * (CPU) the list matches the SMM_CASE / SMM_ORD_CASE instantiations exactly, and every recipe
    gives the host plan it is meant to give;
  * every variant x (x, y) dtype pair against the oracle: fast sums within 1e-12 of the backward
    bound sum |w| |x_filled|, reference-order sums bit-identical;
  * float32 output is the float64 result rounded once: y32 == float32(y64), bit for bit;
  * the `> 1e19` threshold is decided on the reference's own sum for every variant;
  * a row's bits do not depend on scheduling: batch size, sub-slabs, NaN patterns that steer the
    sticky-fill state of the consumers, and the process-wide staging / chunking switches (run in
    child processes, since they are read once per process).

Run as a script (`python test_gpu_variants.py SPEC OUT`), the file is the child of those tests.
"""
import contextlib
import ctypes
import json
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAUNCH_CUH = os.path.join(ROOT, "smmregrid_b200", "csrc", "smm_launch.cuh")

# smm_tuning.h: PlanSettings, read by each smm_create | LaunchSettings, read once per process
CREATE_ENV = ("SMM_FORCE_LANES", "SMM_PACKED", "SMM_CONSUMER_THREADS", "SMM_SUMMATION", "SMM_ORDLONG",
              "SMM_ORD_ROWS", "SMM_SPLIT")
PROCESS_ENV = ("SMM_ROWS_PER_STAGE", "SMM_MAX_STAGES", "SMM_MIN_ROWS_PER_ITEM", "SMM_WAVES", "SMM_ORD_TPR",
               "SMM_COMPACT_F64_ROWS")

KERNEL_STAGED, KERNEL_GATHER, KERNEL_COMPACT = 1, 2, 3
SUM_FAST, SUM_REFERENCE = 1, 2
ALL_B = (1, 7, 37, 200)
DTYPE_PAIRS = [(np.float32, np.float32), (np.float32, np.float64), (np.float64, np.float32), (np.float64, np.float64)]
ORD_K = 20                      # longest row of the ordered-kernel operators (> 16: no staged lane plan looks alike)
ZERO_ROW = 4                    # its only missing source has weight 0


# ------------------------------------------------------------------ the variant matrix

class Variant:
    """One compiled variant and the recipe that reaches it.

    family  staged | ordered | gather | compact
    key     staged (lanes per row, links per lane, consumer threads, packed, reference order),
            ordered (rows per tile, threads per row), gather (lanes per row, reference order),
            compact (pass-1 copies, pass-2 form)
    env     create-time switches
    runs    ((process-wide switches, batch sizes), ...): the ordered kernel's threads per row
            follow from B, or from SMM_ORD_TPR, which only a child process can set
    """

    def __init__(self, family, key, env, kernel, runs=(({}, ALL_B),), ldx_pad=0):
        self.family, self.key, self.env, self.kernel, self.runs, self.ldx_pad = family, key, env, kernel, runs, ldx_pad
        if family == "staged":
            L, K, N, P, O = key
            self.id = f"staged-{'packed' if P else f'l{L}k{K}'}-n{N}-{'ord' if O else 'fast'}"
            self.ref_order = O
        elif family == "ordered":
            self.id = f"ordered-r{key[0]}-t{key[1]}"
            self.ref_order = True
        elif family == "gather":
            self.id = "gather-ord" if key[1] else f"gather-lpr{key[0]}"
            self.ref_order = key[1]
        else:
            self.id = f"compact-{key[0]}-{key[1]}"
            self.ref_order = True                 # pass 2 always sums in the reference's order

    def __repr__(self):
        return self.id


# SMM_CASE(L, K) of launch_staged_t: fast sums at 256 and 512 consumer threads, reference order at 256
LANES = [(1, 4), (2, 4), (1, 8), (1, 12), (1, 16), (2, 12), (2, 14), (2, 16), (4, 12), (4, 16), (8, 12), (8, 14),
         (8, 16), (16, 16), (32, 16)]
# SMM_CASE_PO(1, 16, N, true, O): packed rows
PACKED = [(256, False), (512, False), (256, True)]
# SMM_ORD_CASE_T(R, T) of launch_ordered_t.  Two threads per row need >= 2 batch rows, and R <= 128
# unless SMM_ORD_TPR overrides the choice
ORDERED = [
    (32, 1, (({}, (1,)), ({"SMM_ORD_TPR": "1"}, (7, 37, 200)))),
    (32, 2, (({}, (7, 37, 200)),)),
    (64, 1, (({}, (1,)), ({"SMM_ORD_TPR": "1"}, (7, 37, 200)))),
    (64, 2, (({}, (7, 37, 200)),)),
    (128, 1, (({}, (1,)), ({"SMM_ORD_TPR": "1"}, (7, 37, 200)))),
    (128, 2, (({}, (7, 37, 200)),)),
    (256, 1, (({}, ALL_B),)),
    (256, 2, (({"SMM_ORD_TPR": "2"}, (7, 37, 200)),)),
]
# gather_kernel<LPR, ORD>: LPR from the mean row length (<= 2, <= 24, more), ORD always LPR 1
GATHER = [(1, False), (4, False), (32, False), (1, True)]
# compact path: pass 1 with bulk (TMA) or element copies (x rows not 16-byte aligned); pass 2 raw
# first (>= 2 links per row), with the fill in line (fewer), or with the links read from global
# memory (a 32-row block holds more than 1024 links)
COMPACT = [("bulk", "raw"), ("bulk", "fill"), ("element", "raw"), ("element", "fill"), ("bulk", "long")]


def _variants():
    out = []
    for L, K in LANES:
        base = {"SMM_FORCE_LANES": f"{L},{K}", "SMM_PACKED": "0", "SMM_SPLIT": "0"}
        out.append(Variant("staged", (L, K, 256, False, False),
                           {**base, "SMM_CONSUMER_THREADS": "256", "SMM_SUMMATION": "fast"}, KERNEL_STAGED))
        out.append(Variant("staged", (L, K, 512, False, False),
                           {**base, "SMM_CONSUMER_THREADS": "512", "SMM_SUMMATION": "fast"}, KERNEL_STAGED))
        out.append(Variant("staged", (L, K, 256, False, True),
                           {**base, "SMM_SUMMATION": "reference", "SMM_ORDLONG": "0"}, KERNEL_STAGED))
    for N, O in PACKED:
        env = {"SMM_PACKED": "1", "SMM_SUMMATION": "reference" if O else "fast"}
        if not O:
            env["SMM_CONSUMER_THREADS"] = str(N)
        out.append(Variant("staged", (1, 16, N, True, O), env, KERNEL_STAGED))
    for R, T, runs in ORDERED:
        out.append(Variant("ordered", (R, T), {"SMM_SUMMATION": "reference", "SMM_PACKED": "0", "SMM_SPLIT": "0",
                                               "SMM_ORD_ROWS": str(R)}, KERNEL_STAGED, runs))
    for lpr, ordr in GATHER:
        out.append(Variant("gather", (lpr, ordr), {"SMM_SUMMATION": "reference" if ordr else "fast"}, KERNEL_GATHER))
    for p1, p2 in COMPACT:
        out.append(Variant("compact", (p1, p2), {"SMM_SUMMATION": "fast"}, KERNEL_COMPACT,
                           ldx_pad=1 if p1 == "element" else 0))
    return out


VARIANTS = _variants()
BY_ID = {v.id: v for v in VARIANTS}
assert len(BY_ID) == len(VARIANTS)


def ordered_threads_per_row(R, B, tpr_env):
    """What size_staged picks for an ordered-kernel plan of R rows per tile (two batch rows per
    stage fit whenever B >= 2 for these operators)."""
    return 2 if B >= 2 and (tpr_env == 2 or (tpr_env == 0 and R <= 128)) else 1


def gather_lanes(mean_row, ref_order):
    return 1 if ref_order or mean_row <= 2.0 else (4 if mean_row <= 24.0 else 32)


def expected_info(v):
    """smm_info fields of the plan the recipe is meant to give."""
    if v.family == "staged":
        L, K, N, P, O = v.key
        return dict(kernel=KERNEL_STAGED, lanes_per_row=L, links_per_lane=K, consumer_threads=N, packed_rows=int(P),
                    summation=SUM_REFERENCE if O else SUM_FAST, rows_per_tile=4 * N if P else N // L)
    if v.family == "ordered":
        R = v.key[0]
        return dict(kernel=KERNEL_STAGED, lanes_per_row=1, links_per_lane=ORD_K, consumer_threads=R, packed_rows=0,
                    summation=SUM_REFERENCE, rows_per_tile=R)
    # (the compact path sums in the reference's order whatever the handle's summation is)
    return dict(kernel=KERNEL_GATHER, summation=SUM_REFERENCE if v.env["SMM_SUMMATION"] == "reference" else SUM_FAST)


# ------------------------------------------------------------------ operators and fields

class Op:
    pass


def _shape(v, purpose):
    """(n_dst, shortest row, longest row, layout).  Parity operators have 2.5 tiles (row blocks),
    scheduling operators ~12, so that default chunks span several tiles' batch loops."""
    tiles = 12 if purpose == "sched" else 2
    if v.family == "staged":
        L, K, N, P, O = v.key
        if P:
            return (24 if purpose == "sched" else 6) * N + 37, 0, 16, "band"
        R = N // L
        return tiles * R + R // 2 + 1, 0, L * K, "band"
    if v.family == "ordered":
        R = v.key[0]
        return tiles * R + R // 2 + 1, 0, ORD_K, "band"
    if v.family == "gather":
        lo, hi = {(1, False): (0, 3), (4, False): (0, 30), (32, False): (0, 100), (1, True): (0, 30)}[v.key]
        rpb = 256 // (1 if v.key[1] else v.key[0])
        return tiles * rpb + rpb // 2 + 1, lo, hi, "scattered"
    lo, hi = {"raw": (0, 6), "fill": (0, 2), "long": (20, 60)}[v.key[1]]
    return (1000 if purpose == "sched" else 200), lo, hi, "scattered"


def _threshold_counts(v, n_dst):
    """Row lengths of the threshold construction: as long as the layout takes (>= 2 links, so
    that 10 % of the weight can sit on the missing sources), within the variant's class."""
    if v.family == "staged":
        L, K, N, P, O = v.key
        k = [2, 4, 8, 12, 16] if P else [L * K]
    elif v.family == "ordered":
        k = [ORD_K]
    elif v.family == "gather":
        k = [{1: 2, 4: 20, 32: 40}[v.key[0]] if not v.key[1] else 20]
    else:
        k = {"raw": [20], "fill": [1, 2], "long": [40]}[v.key[1]]
    return np.resize(np.array(k), n_dst)


SCATTER = 64                    # scattered layouts: touched columns 64 apart never share a staged segment
_OPS = {}


def _operator(v, purpose):
    """Links, masks and the special rows of the operator a test of variant v uses.  purpose:
    parity | sched (weights scaled by 1e-3: a filled source stays far below 1e19) | threshold."""
    key = (v.id, purpose)
    if key in _OPS:
        return _OPS[key]
    rng = np.random.default_rng(zlib.crc32(f"{v.id}/{purpose}".encode()))
    n_dst, lo, hi, layout = _shape(v, purpose)
    op = Op()
    op.n_dst = n_dst
    if purpose == "threshold":
        counts = _threshold_counts(v, n_dst)
    else:
        counts = rng.integers(lo, hi + 1, size=n_dst)
        if v.family in ("staged", "ordered"):
            # empty, full and padded rows, the last row in the partial last tile
            counts[0], counts[1], counts[2], counts[3], counts[-1] = 0, hi, 1, max(hi - 1, 1), hi
        counts[ZERO_ROW] = max(2, lo)
        counts[n_dst - 2] = max(4, lo)
    dst = np.repeat(np.arange(n_dst), counts)
    cols = []
    if purpose == "threshold":
        # disjoint rows: a row's missing sources are its own
        pos = np.arange(dst.size)
        if layout == "band":
            src = pos
            n_src = -(-dst.size // 8) * 8 + 8
        else:
            src = SCATTER * pos + pos % 7
            n_src = SCATTER * dst.size + 100
    elif layout == "band":
        span = hi + hi // 4 + 4
        for r, n in enumerate(counts):
            cols.append(r + np.sort(rng.choice(span, size=n, replace=False)))
        src = np.concatenate(cols).astype(np.int64)
        n_src = -(-(n_dst + span) // 8) * 8 + 8
    else:
        pool = 512
        for n in counts:
            j = np.sort(rng.choice(pool, size=n, replace=False))
            cols.append(SCATTER * j + j % 7)
        src = np.concatenate(cols).astype(np.int64)
        n_src = SCATTER * pool + 100            # n_src % 256 = 100: a partial last pass-1 block
    w = rng.random(dst.size)
    if purpose == "threshold":
        # 10 % of each row's weight on n_nan links, which the fields make missing; every weight
        # perturbed in its last bits so that the summation order decides the `> 1e19` test
        op.nan_link = np.zeros(dst.size, bool)
        a = 0
        for n in counts:
            n_nan = max(1, int(round(n / 10)))
            pick = a + rng.choice(n, size=n_nan, replace=False)
            op.nan_link[pick] = True
            w[a:a + n] = 0.9 / (n - n_nan) if n > n_nan else 0.0
            w[pick] = 0.1 / n_nan
            a += n
        w += rng.uniform(-1e-17, 1e-17, size=w.size)
        op.imask = np.ones(n_dst, np.int32)
        op.frac = np.ones(n_dst)
    else:
        starts = np.concatenate([[0], np.cumsum(counts)])
        w[starts[ZERO_ROW]] = 0.0
        op.zero_cols = src[starts[ZERO_ROW]:starts[ZERO_ROW + 1]]
        op.big_cols = src[starts[n_dst - 2]:starts[n_dst - 1]]
        w[starts[n_dst - 2]:starts[n_dst - 1]] = 0.9     # a sum below -3.4e38 in the last batch row
        if purpose == "sched":
            w *= 1e-3
        op.imask = (rng.random(n_dst) > 0.1).astype(np.int32)
        op.frac = rng.uniform(0.4, 1.0, n_dst)
        for r in (ZERO_ROW, n_dst - 2):
            op.imask[r], op.frac[r] = 1, 1.0
    op.n_src = int(n_src)
    op.src = (src + 1).astype(np.int32)
    op.dst = (dst + 1).astype(np.int32)
    op.w = w.reshape(-1, 1)
    op.counts = counts
    op.max_row = int(counts.max())
    op.masked, op.amin = (purpose != "threshold"), (0.0 if purpose == "threshold" else 0.5)
    op.ldx = op.n_src + v.ldx_pad
    _OPS[key] = op
    return op


def _seed(*parts):
    return zlib.crc32("/".join(str(p) for p in parts).encode())


def _field_parity(op, v, xdt, B):
    """Fields of both signs with NaN, +-inf, the weight-0 row's lone missing source and a row
    whose sum is below -3.4e38 (float32 output: -inf)."""
    rng = np.random.default_rng(_seed(v.id, "parity", B))
    x = 100.0 * rng.standard_normal((B, op.n_src))
    x[rng.random(x.shape) < min(0.02, 0.5 / max(op.max_row, 1))] = np.nan
    x[0, rng.integers(op.n_src)] = np.inf
    x[B // 2, rng.integers(op.n_src)] = -np.inf
    x[:, op.zero_cols] = 100.0 * rng.standard_normal((B, op.zero_cols.size))
    x[:, op.zero_cols[0]] = np.nan
    big = op.big_cols[op.big_cols != op.zero_cols[0]]
    x[B - 1, big] = -3e38
    return x.astype(xdt)


PATTERNS = ("random", "row0", "first17", "probe16", "alternate")


def _field_sched(op, v, xdt, B, pattern):
    """NaN patterns over the batch rows that steer the consumers' sticky-fill state: only in row
    0, first in row 17, on the 16-row re-probe boundary, in alternate rows (or scattered)."""
    rng = np.random.default_rng(_seed(v.id, "sched", B))
    x = 100.0 * rng.standard_normal((B, op.n_src))
    rows = np.arange(B)
    nan_rows = {"random": np.zeros(B, bool), "row0": rows == 0, "first17": rows >= 17,
                "probe16": rows % 16 == 0, "alternate": rows % 2 == 0}[pattern]
    if pattern == "random":
        x[rng.random(x.shape) < 0.01] = np.nan
        x[rng.integers(B), rng.integers(op.n_src)] = np.inf
        x[rng.integers(B), rng.integers(op.n_src)] = -np.inf
    x[np.ix_(nan_rows, np.arange(op.n_src) % 11 == 3)] = np.nan
    return x.astype(xdt)


def _field_threshold(op, v, B):
    """float64 data; in a batch row, a row's missing links are NaN in two of every three rows."""
    rng = np.random.default_rng(_seed(v.id, "threshold", B))
    x = rng.uniform(0, 2000, size=(B, op.n_src))
    src0, dst0 = op.src.astype(np.int64) - 1, op.dst.astype(np.int64) - 1
    for b in range(B):
        hit = op.nan_link & ((dst0 + b) % 3 != 0)
        x[b, src0[hit]] = np.nan
    return x


# ------------------------------------------------------------------ C ABI

@contextlib.contextmanager
def _create_env(env):
    saved = {k: os.environ.get(k) for k in CREATE_ENV}
    for k in CREATE_ENV:
        os.environ.pop(k, None)
    os.environ.update(env)
    try:
        yield
    finally:
        for k, val in saved.items():
            if val is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = val


def _create(lib, v, op):
    """Handle of the operator under the variant's create-time switches; asserts the plan."""
    from smmregrid_b200 import _lib
    h = ctypes.c_void_p()
    with _create_env(v.env):
        _lib.check(lib.smm_create(op.n_src, op.n_dst, op.src.size, op.src.ctypes.data, op.dst.ctypes.data,
                                  op.w.ctypes.data, 1, 1, 0, None, ctypes.byref(h)))
    try:
        _lib.check(lib.smm_set_dst_mask(h, 0, op.imask.ctypes.data, op.frac.ctypes.data))
        inf = _lib.SmmInfo()
        _lib.check(lib.smm_get_info(h, 0, ctypes.byref(inf)))
        got = inf.asdict()
        want = expected_info(v)
        assert {k: got[k] for k in want} == want, (v.id, got)
        if v.family in ("staged", "ordered"):
            assert got["n_tiles"] >= 3 and got["gather_rows"] == 0, (v.id, got)
    except BaseException:
        lib.smm_destroy(h)
        raise
    return h


def _to_device(x, ldx):
    import torch
    xd = torch.zeros((x.shape[0], ldx), dtype=torch.from_numpy(x).dtype, device="cuda")
    xd[:, :x.shape[1]] = torch.from_numpy(x).cuda()
    return xd


def _apply(lib, h, v, op, xd, ydt, B, row0=0, y=None, yrow0=0):
    """smm_apply of batch rows [row0, row0 + B) of xd into rows [yrow0, yrow0 + B) of y."""
    import torch
    from smmregrid_b200 import _lib
    if y is None:
        y = torch.full((B, op.n_dst), -7.0, dtype=torch.float64 if ydt == np.float64 else torch.float32, device="cuda")
    xp = xd.data_ptr() + row0 * op.ldx * xd.element_size()
    yp = y.data_ptr() + yrow0 * op.n_dst * y.element_size()
    _lib.check(lib.smm_apply(h, 0, xp, 0 if xd.dtype == torch.float32 else 1, B, op.ldx,
                             yp, 1 if ydt == np.float64 else 0, op.n_dst, int(op.masked), op.amin,
                             _lib.apply_opts(v.kernel), None))
    return y


def _run(lib, v, purpose, xdt, B, pattern=None, ydts=(np.float64, np.float32), split=False):
    """Outputs of one case from one handle and one input: "y64" / "y32" = all B rows in one call
    in float64 / float32; with split, also the same rows applied one call each ("_single") and a
    sub-slab at a row offset ("_slab")."""
    import torch
    op = _operator(v, purpose)
    if purpose == "parity":
        x = _field_parity(op, v, xdt, B)
    elif purpose == "threshold":
        x = _field_threshold(op, v, B)
    else:
        x = _field_sched(op, v, xdt, B, pattern)
    xd = _to_device(x, op.ldx)
    h = _create(lib, v, op)
    try:
        out = {}
        for ydt in ydts:
            tag = "y64" if ydt == np.float64 else "y32"
            out[tag] = _apply(lib, h, v, op, xd, ydt, B)
            if split:
                single = torch.full_like(out[tag], -7.0)
                for b in range(B):
                    _apply(lib, h, v, op, xd, ydt, 1, row0=b, y=single, yrow0=b)
                out[tag + "_single"] = single
                r0, n = 3, min(50, B - 3)
                out[tag + "_slab"] = _apply(lib, h, v, op, xd, ydt, n, row0=r0)
        torch.cuda.synchronize()
        return {k: t.cpu().numpy() for k, t in out.items()}
    finally:
        lib.smm_destroy(h)


# ------------------------------------------------------------------ child processes

def _spawn(jobs, proc_env, tmp_path, name):
    """Run the jobs in a child process with the process-wide switches proc_env; returns one dict
    of outputs per job.  The child is awaited (with a time limit) before this returns."""
    tmp_path = str(tmp_path)
    spec = os.path.join(tmp_path, f"{name}.json")
    out = os.path.join(tmp_path, f"{name}.npz")
    with open(spec, "w") as f:
        json.dump({"jobs": jobs}, f)
    env = {k: val for k, val in os.environ.items() if k not in CREATE_ENV + PROCESS_ENV}
    env.update(proc_env)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), spec, out]
    proc = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, f"child {proc_env} failed:\n{proc.stdout[-3000:]}\n{proc.stderr[-3000:]}"
    res = [dict() for _ in jobs]
    with np.load(out) as z:
        for k in z.files:
            i, tag = k.split("_", 1)
            res[int(i)][tag] = z[k]
    os.remove(out)
    return res


def _child_main(spec, out):
    sys.path.insert(0, ROOT)
    from smmregrid_b200 import _lib
    lib = _lib.load()
    with open(spec) as f:
        jobs = json.load(f)["jobs"]
    arrays = {}
    for i, j in enumerate(jobs):
        r = _run(lib, BY_ID[j["variant"]], j["purpose"], np.dtype(j["xdt"]).type, j["B"], j.get("pattern"),
                 tuple(np.dtype(t).type for t in j["ydts"]))
        for tag, a in r.items():
            arrays[f"{i}_{tag}"] = a
    np.savez(out, **arrays)


# ------------------------------------------------------------------ comparisons

def _same_bits(a, b):
    """Bit-identical values; NaN at the same cells (any payload)."""
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    u = np.uint64 if a.dtype == np.float64 else np.uint32
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(u), b[~nb].view(u))


def _diff(a, b):
    na, nb = np.isnan(a), np.isnan(b)
    bad = (na != nb) | (~na & ~nb & (a != b))
    return f"{int(bad.sum())} of {a.size} cells differ (first at {np.argwhere(bad)[:3].tolist()})"


def _f32(a):
    with np.errstate(over="ignore"):
        return a.astype(np.float32)


# ------------------------------------------------------------------ 1. the matrix (CPU)

def _launch_instantiations():
    """(staged keys, ordered keys) instantiated by smm_launch.cuh: SMM_CASE / SMM_CASE_PO and
    SMM_ORD_CASE / SMM_ORD_CASE_T invocations, with the wrapper macros expanded as defined there."""
    text = open(LAUNCH_CUH).read()
    text = re.sub(r"//[^\n]*|/\*.*?\*/", "", text, flags=re.S).replace("\\\n", " ")
    defs, body = {}, []
    for line in text.splitlines():
        m = re.match(r"\s*#\s*define\s+(\w+)\(([^)]*)\)(.*)", line)
        if m:
            defs[m.group(1)] = ([p.strip() for p in m.group(2).split(",")], m.group(3))
        elif not line.lstrip().startswith("#"):
            body.append(line)
    leaves = {"SMM_CASE_PO": [], "SMM_ORD_CASE_T": []}
    call = re.compile(r"\b(SMM_CASE_PO|SMM_CASE|SMM_ORD_CASE_T|SMM_ORD_CASE)\s*\(([^()]*)\)")

    def expand(src):
        for name, args in call.findall(src):
            args = [a.strip() for a in args.split(",")]
            if name in leaves:
                leaves[name].append(tuple(args))
            else:
                params, tmpl = defs[name]
                assert len(params) == len(args), (name, args)
                for p, a in zip(params, args):
                    tmpl = re.sub(rf"\b{p}\b", a, tmpl)
                expand(tmpl)

    expand("\n".join(body))
    b = {"true": True, "false": False}
    staged = [(int(L), int(K), int(N), b[P], b[O]) for L, K, N, P, O in leaves["SMM_CASE_PO"]]
    ordered = [(int(R), int(T)) for R, T in leaves["SMM_ORD_CASE_T"]]
    return staged, ordered


def test_variant_list_matches_dispatch_tables():
    staged, ordered = _launch_instantiations()
    assert len(staged) == len(set(staged)) and len(ordered) == len(set(ordered))
    listed_staged = sorted(v.key for v in VARIANTS if v.family == "staged")
    listed_ordered = sorted(v.key for v in VARIANTS if v.family == "ordered")
    assert listed_staged == sorted(staged), (set(staged) ^ set(listed_staged))
    assert listed_ordered == sorted(ordered), (set(ordered) ^ set(listed_ordered))
    assert len(staged) == 48 and len(ordered) == 8


def _host_info(lib, v, op):
    from smmregrid_b200 import _lib
    h = ctypes.c_void_p()
    with _create_env(v.env):
        _lib.check(lib.smm_host_plan_build(op.n_src, op.n_dst, op.src.size, op.src.ctypes.data, op.dst.ctypes.data,
                                           op.w.ctypes.data, 1, 1, None, ctypes.byref(h)))
    inf = _lib.SmmInfo()
    ns = ctypes.c_int64()
    try:
        _lib.check(lib.smm_host_plan_info(h, ctypes.byref(inf), ctypes.byref(ns)))
        info = inf.asdict()
        tiles = np.empty((max(info["n_tiles"], 1), 8), np.int32)
        _lib.check(lib.smm_host_plan_copy(h, None, None, None, tiles.ctypes.data, None, None, None))
    finally:
        lib.smm_host_plan_free(h)
    return info, tiles


@pytest.mark.parametrize("purpose", ["parity", "sched", "threshold"])
def test_recipes_give_the_intended_plans(smm_lib, purpose):
    """Every recipe builds the plan it names (host plan, no GPU): lanes, links per lane,
    consumer threads, packing, summation order, rows per tile; >= 3 tiles with a partial last
    one; for gather and compact variants the class that picks the kernel."""
    for v in VARIANTS:
        op = _operator(v, purpose)
        info, tiles = _host_info(smm_lib, v, op)
        want = expected_info(v)
        assert {k: info[k] for k in want} == want, (v.id, purpose, info)
        if v.family in ("staged", "ordered"):
            assert info["n_tiles"] >= 3 and info["gather_rows"] == 0, (v.id, purpose, info)
            if not info["packed_rows"]:
                assert tiles[-1, 1] < info["rows_per_tile"], (v.id, purpose, "last tile is full")
            if purpose != "threshold":
                assert op.max_row == _shape(v, purpose)[2] and op.counts.min() == 0, v.id
        mean = op.src.size / op.n_dst
        if v.family == "gather":
            assert gather_lanes(mean, v.ref_order) == v.key[0], (v.id, purpose, mean)
        if v.family == "compact":
            raw = op.src.size >= 2 * op.n_dst
            blocks = np.add.reduceat(op.counts, np.arange(0, op.n_dst, 32))
            if v.key[1] == "raw":
                assert raw and blocks.max() <= 1024, (v.id, purpose)
            elif v.key[1] == "fill":
                assert not raw, (v.id, purpose)
            else:
                assert raw and blocks.max() > 1024, (v.id, purpose)
            assert (op.ldx * 4) % 16 == (0 if v.key[0] == "bulk" else 4), v.id
    for v in VARIANTS:
        if v.family == "ordered":
            R, T = v.key
            for proc_env, batches in v.runs:
                for B in batches:
                    assert ordered_threads_per_row(R, B, int(proc_env.get("SMM_ORD_TPR", 0))) == T, (v.id, B)


# ------------------------------------------------------------------ 2-4. oracle parity (GPU)

_RESULTS = {}
_CHILD_RUNS = {}


def _env_key(env):
    return tuple(sorted(env.items()))


def _threshold_run(v):
    proc_env, batches = v.runs[0]
    return proc_env, (16 if max(batches) >= 16 else 1)


def _results(lib, v, purpose, xdt, B, proc_env, tmp_path):
    """Outputs of a parity / threshold case, in this process or -- when the variant needs a
    process-wide switch -- from the one child that runs every such case of that switch."""
    key = (v.id, purpose, np.dtype(xdt).name, B)
    if not proc_env:
        if key not in _RESULTS:
            _RESULTS[key] = _run(lib, v, purpose, xdt, B, ydts=(np.float64,) if purpose == "threshold"
                                 else (np.float64, np.float32))
        return _RESULTS[key]
    ek = _env_key(proc_env)
    if ek not in _CHILD_RUNS:
        jobs = []
        for u in VARIANTS:
            for penv, batches in u.runs:
                if _env_key(penv) != ek:
                    continue
                for x in ("float32", "float64"):
                    for b in batches:
                        jobs.append(dict(variant=u.id, purpose="parity", xdt=x, B=b, ydts=["float64", "float32"]))
            tenv, tb = _threshold_run(u)
            if _env_key(tenv) == ek:
                jobs.append(dict(variant=u.id, purpose="threshold", xdt="float64", B=tb, ydts=["float64"]))
        outs = _spawn(jobs, proc_env, tmp_path, "variants_" + "_".join(f"{k}{val}" for k, val in ek))
        _CHILD_RUNS[ek] = {(j["variant"], j["purpose"], j["xdt"], j["B"]): o for j, o in zip(jobs, outs)}
    return _CHILD_RUNS[ek][key]


def _backward_scale(op, x):
    import scipy.sparse as sp
    xf = np.abs(np.where(np.isfinite(x), x, x.dtype.type(1e20)).astype(np.float64))
    W = sp.csr_matrix((np.abs(op.w[:, 0]), (op.src - 1, op.dst - 1)), shape=(op.n_src, op.n_dst))
    return np.asarray((W.T @ xf.T).T)


def _oracle_result(oracle, op, x):
    if not hasattr(op, "mat"):
        op.mat = oracle.compute_weights_matrix_c(op.src, op.dst, op.w, op.n_src, op.n_dst)
    return oracle.apply_weights_c(x, op.mat, op.imask, op.frac, op.amin, op.masked)


@pytest.mark.gpu
@pytest.mark.parametrize("xdt,ydt", DTYPE_PAIRS, ids=["f32-f32", "f32-f64", "f64-f32", "f64-f64"])
@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_variant_matches_oracle(smm_lib, oracle, cuda, tmp_path, v, xdt, ydt):
    """Fast sums within 1e-12 of sum |w| |x_filled|; reference-order sums bit-identical.
    float32 output: exactly float32 of the float64 output (same handle, same input), hence
    bit-identical to float32(oracle) in reference order and within one float32 ulp of it where
    the float64 bound is below half a float32 ulp."""
    op = _operator(v, "parity")
    checked = 0
    for proc_env, batches in v.runs:
        for B in batches:
            x = _field_parity(op, v, xdt, B)
            ref = _oracle_result(oracle, op, x)
            r = _results(smm_lib, v, "parity", xdt, B, proc_env, tmp_path)
            y64, y32 = r["y64"], r["y32"]
            what = f"{v.id} B={B} {proc_env}"
            assert np.array_equal(np.isnan(y64), np.isnan(ref)), what + ": NaN pattern, " + _diff(y64, ref)
            assert np.isnan(ref).any() and (~np.isnan(ref)).any()
            scale = _backward_scale(op, x)
            if ydt == np.float64:
                if v.ref_order:
                    assert _same_bits(y64, ref), what + ": " + _diff(y64, ref)
                else:
                    ok = ~np.isnan(ref)
                    assert np.array_equal(np.isinf(y64), np.isinf(ref)), what
                    fin = ok & np.isfinite(ref)
                    err = np.abs(y64[fin] - ref[fin])
                    assert np.all(err <= 1e-12 * np.maximum(scale[fin], 1e-300)), (what, err.max())
                assert ZERO_ROW < op.n_dst and np.isfinite(y64[:, ZERO_ROW]).all(), what
            else:
                # rounded once at the store: exactly float32 of the float64 result, NaN cells included
                assert _same_bits(y32, _f32(y64)), what + ": y32 != float32(y64), " + _diff(y32, _f32(y64))
                r32 = _f32(ref)
                assert np.isneginf(y32[-1, op.n_dst - 2]) and np.isfinite(y64[-1, op.n_dst - 2]), what
                if v.ref_order:
                    assert _same_bits(y32, r32), what + ": " + _diff(y32, r32)
                else:
                    with np.errstate(invalid="ignore", over="ignore"):
                        tight = np.isfinite(r32) & (1e-12 * scale <= 0.5 * np.spacing(np.abs(r32)).astype(np.float64))
                    near = ((y32 == r32) | (y32 == np.nextafter(r32, np.float32(np.inf)))
                            | (y32 == np.nextafter(r32, np.float32(-np.inf))))
                    assert tight.sum() > 0.5 * np.isfinite(r32).sum(), what
                    assert near[tight].all(), what + f": {int((~near & tight).sum())} cells beyond 1 float32 ulp"
            checked += 1
    assert checked >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_variant_threshold_is_reference_order(smm_lib, oracle, cuda, tmp_path, v):
    """Rows whose filled sum lands within rounding of 1e19 (10 % of the weight on NaN sources,
    float64 data, last-bit weight perturbations): the NaN decision and every value within 1e10
    of 1e19 are the reference's, bit for bit."""
    proc_env, B = _threshold_run(v)
    op = _operator(v, "threshold")
    x = _field_threshold(op, v, B)
    ref = _oracle_result(oracle, op, x)
    y = _results(smm_lib, v, "threshold", np.float64, B, proc_env, tmp_path)["y64"]
    near = np.abs(ref - 1e19) < 1e10
    assert near.sum() >= 10 and np.isnan(ref).sum() >= 10, (v.id, int(near.sum()))
    assert np.array_equal(np.isnan(y), np.isnan(ref)), f"{v.id}: NaN decisions, " + _diff(y, ref)
    assert _same_bits(y[near], ref[near]), f"{v.id}: values near 1e19, " + _diff(y[near], ref[near])


# ------------------------------------------------------------------ 5. scheduling invariance (GPU)

SCHED = ["staged-packed-n256-fast", "staged-l1k12-n256-fast", "staged-l4k16-n512-fast", "staged-l2k14-n256-ord",
         "ordered-r64-t2", "gather-lpr4", "compact-bulk-raw"]
SCHED_B = 200


@pytest.mark.gpu
@pytest.mark.parametrize("xdt,ydt", DTYPE_PAIRS, ids=["f32-f32", "f32-f64", "f64-f32", "f64-f64"])
@pytest.mark.parametrize("vid", SCHED)
def test_rows_do_not_depend_on_batching(smm_lib, cuda, vid, xdt, ydt):
    """All B rows in one call == the same rows one call each == a 16-byte aligned sub-slab at a
    row offset, bit for bit, under NaN patterns that exercise the sticky-fill state (first row
    only, first in row 17, on the 16-row re-probe boundary, alternate rows)."""
    v = BY_ID[vid]
    tag = "y64" if ydt == np.float64 else "y32"
    bad = []
    for pattern in PATTERNS:
        r = _run(smm_lib, v, "sched", xdt, SCHED_B, pattern, ydts=(ydt,), split=True)
        y, single, slab = r[tag], r[tag + "_single"], r[tag + "_slab"]
        assert np.isnan(y).any() and (~np.isnan(y)).any()
        if not _same_bits(y, single):
            bad.append(f"{pattern}: one call vs single rows, " + _diff(y, single))
        if not _same_bits(y[3:3 + slab.shape[0]], slab):
            bad.append(f"{pattern}: sub-slab, " + _diff(y[3:3 + slab.shape[0]], slab))
    assert not bad, f"{vid}: " + "; ".join(bad)


SETTINGS = [{"SMM_ROWS_PER_STAGE": "1"}, {"SMM_ROWS_PER_STAGE": "3"}, {"SMM_ROWS_PER_STAGE": "8"},
            {"SMM_MAX_STAGES": "2"}, {"SMM_MIN_ROWS_PER_ITEM": "1"},
            {"SMM_MIN_ROWS_PER_ITEM": "200"},          # one chunk: whole-batch loops, many trips round the stage ring
            {"SMM_WAVES": "1"}, {"SMM_WAVES": "32"}, {"SMM_ORD_TPR": "1"}, {"SMM_ORD_TPR": "2"},
            {"SMM_COMPACT_F64_ROWS": "64"}]
SETTING_CASES = [(vid, x, y, p) for vid in SCHED for x, y in ((np.float32, np.float64), (np.float64, np.float32))
                 for p in ("random", "alternate")]
_SCHED_FULL = {}


@pytest.mark.gpu
@pytest.mark.parametrize("proc_env", SETTINGS, ids=["-".join(f"{k}={val}" for k, val in s.items()) for s in SETTINGS])
def test_rows_do_not_depend_on_process_switches(smm_lib, cuda, tmp_path, proc_env):
    """The process-wide staging / chunking switches (read once per process, so set in a child
    process) change how the batch is cut into work items and stages, never a row's bits."""
    jobs = [dict(variant=vid, purpose="sched", xdt=np.dtype(x).name, B=SCHED_B, pattern=p, ydts=[np.dtype(y).name])
            for vid, x, y, p in SETTING_CASES]
    outs = _spawn(jobs, proc_env, tmp_path, "sched")
    for (vid, x, y, p), out in zip(SETTING_CASES, outs):
        key = (vid, x, y, p)
        if key not in _SCHED_FULL:
            _SCHED_FULL[key] = _run(smm_lib, BY_ID[vid], "sched", x, SCHED_B, p, ydts=(y,))
        tag = "y64" if y == np.float64 else "y32"
        mine, theirs = _SCHED_FULL[key][tag], out[tag]
        assert _same_bits(mine, theirs), f"{vid} {p} {np.dtype(x).name}->{np.dtype(y).name} {proc_env}: " + _diff(mine, theirs)


if __name__ == "__main__":
    _child_main(sys.argv[1], sys.argv[2])
