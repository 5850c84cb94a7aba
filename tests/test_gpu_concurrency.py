"""Concurrent callers of one operator: every kernel family, every entry point and the front end.

include/smmregrid_b200.h promises that smm_apply* are re-entrant across threads and streams and
that one handle can be shared by any number of callers.  The front end relies on it: dask's
worker threads share one Regridder, torch callers apply on their own streams, and the pinned
result pool hands buffers to whichever thread asks.  A concurrent call must give the bits of the
same call made alone: fast sums do not depend on batching or scheduling
(test_gpu_variants.test_rows_do_not_depend_on_batching), so nothing less is right.

The first launches of a kernel are the delicate ones: each raises the kernel's shared-memory
opt-in, whose size follows B.  This pytest process has long raised them, so that test runs in a
child process: run as a script (`python test_gpu_concurrency.py OUT`), this file is that child.
"""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from test_gpu_levels_host import SPLIT, _base_operator, _create_levels, _host_array, _infos, _level_ops, _slot_fields
from test_gpu_packed import CASES_F32, CASES_F64, _dev, _ldx, _raw_field
from test_gpu_variants import (ALL_B, BY_ID, CREATE_ENV, PROCESS_ENV, ROOT, _backward_scale, _create, _diff, _f32,
                               _field_parity, _oracle_result, _same_bits, _seed)

F32, F64 = np.float32, np.float64

# ------------------------------------------------------------------ first launches, racing

# one handle per kernel family: staged fast sums with 1, 2, 8 and 32 lanes per row, staged reference
# order, packed rows (fast and reference order), the ordered kernel with one thread per row (R = 256
# at every B) and two (R = 64 from B = 2), a split plan, gathers with 1, 4 and 32 lanes and in
# reference order, and the two-pass compact path
RACE_IDS = ["staged-l1k12-n256-fast", "staged-l2k14-n512-fast", "staged-l8k16-n256-fast", "staged-l32k16-n256-fast",
            "staged-l2k14-n256-ord", "staged-packed-n256-fast", "staged-packed-n256-ord", "ordered-r256-t1",
            "ordered-r64-t2", SPLIT.id, "gather-lpr1", "gather-lpr4", "gather-lpr32", "gather-ord", "compact-bulk-raw"]
# x: float32, float64, or int16 decoded to float32 / float64 (test_gpu_packed's cases); y: float32, float64
X_KINDS = [("f32", F32, None), ("f64", F64, None), ("i16f32", None, CASES_F32[0]), ("i16f64", None, CASES_F64[0])]
COMBOS = [(xk, ydt) for xk in X_KINDS for ydt in (F32, F64)]
N_THREADS = 8


def _recipe(rid):
    return SPLIT if rid == SPLIT.id else BY_ID[rid]


def _thread_B(t):
    # threads 2k and 2k + 1 share B; with the combo parity below every (B, combo) pair is one thread's
    return ALL_B[(t // 2) % len(ALL_B)]


def _thread_combo(t, h):
    # per handle, the four threads of one parity apply the same kernel instantiation at B = 1, 7, 37, 200
    return COMBOS[(h + t % 2) % len(COMBOS)]


def _thread_order(t):
    # every thread its own order: threads 2k and 2k + 1 start at handle 2k and 2k + 1 and go forwards
    # for even k, backwards for odd k; with an odd number of handles every forward thread then meets
    # every backward one on one handle at the same step
    n = len(RACE_IDS)
    assert n % 2 == 1
    step = 1 if (t // 2) % 2 == 0 else -1
    return [(t + step * k) % n for k in range(n)]


def _race_input(v, op, xkind, B):
    """(data as applied, float data the oracle reads, x code, packing case)."""
    name, xdt, case = xkind
    if case is None:
        x = _field_parity(op, v, xdt, B)
        return x, x, 0 if xdt == F32 else 1, None
    raw = _raw_field(op, case, B, _seed(v.id, case.name, B))
    return raw, case.decode(raw), 2, case


def _race_handle(lib, v, op):
    from smmregrid_b200 import _lib
    if v is not SPLIT:
        return _create(lib, v, op)
    h = _create_levels(lib, v, [op])
    info = _infos(lib, h, 1)[0]
    assert info["packed_rows"] == 1 and info["gather_rows"] > 0 and info["summation"] == _lib.SMM_SUM_FAST, info
    return h


def _race_main(out):
    """Child: every handle created, every input on the device; then N_THREADS threads released at
    once, each on its own stream with its own B, apply every handle once in its own order; then the
    same calls one after the other.  Saves both results and each concurrent call's status."""
    sys.path.insert(0, ROOT)
    import torch
    from smmregrid_b200 import _lib
    lib = _lib.load()
    ops = [_base_operator(_recipe(rid)) for rid in RACE_IDS]
    handles = [_race_handle(lib, _recipe(rid), op) for rid, op in zip(RACE_IDS, ops)]
    jobs = {}                                  # (t, h) -> (x view, x code, ldx, y dtype, B, opts)
    keep = []
    for t in range(N_THREADS):
        B = _thread_B(t)
        for h, rid in enumerate(RACE_IDS):
            v, op = _recipe(rid), ops[h]
            xkind, ydt = _thread_combo(t, h)
            x, _, code, case = _race_input(v, op, xkind, B)
            ldx = _ldx(v, op)
            buf, view = _dev(x, ldx)
            keep.append(buf)
            opts = _lib.apply_opts(v.kernel, None, case.packing().to_c() if case else None)
            jobs[(t, h)] = (view, code, ldx, ydt, B, opts)
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(N_THREADS)]

    def call(t, h, stream):
        """smm_apply of job (t, h) on a torch stream (None: the current one), y filled there too"""
        view, code, ldx, ydt, B, opts = jobs[(t, h)]
        op = ops[h]
        with torch.cuda.stream(stream):
            y = torch.full((B, op.n_dst), -7.0, dtype=torch.float32 if ydt == F32 else torch.float64, device="cuda")
            rc = lib.smm_apply(handles[h], 0, view.data_ptr(), code, B, ldx, y.data_ptr(), 0 if ydt == F32 else 1,
                               op.n_dst, int(op.masked), op.amin, opts, torch.cuda.current_stream().cuda_stream)
        return y, rc, lib.smm_last_error().decode() if rc else ""

    conc, status = {}, {}
    barrier = threading.Barrier(N_THREADS)

    def worker(t):
        st = streams[t]
        try:
            barrier.wait()
            for h in _thread_order(t):
                y, rc, msg = call(t, h, st)
                conc[(t, h)] = y
                status[(t, h)] = (rc, msg)
            st.synchronize()
        except Exception as e:                 # noqa: BLE001
            status[(t, -1)] = (-1, repr(e))

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(N_THREADS)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    torch.cuda.synchronize()
    arrays = {}
    for (t, h), y in conc.items():
        arrays[f"conc_{t}_{h}"] = y.cpu().numpy()
    for (t, h) in jobs:
        y, rc, msg = call(t, h, None)
        _lib.check(rc)
        torch.cuda.synchronize()
        arrays[f"seq_{t}_{h}"] = y.cpu().numpy()
    arrays["status"] = np.array([f"{t} {h} {rc} {msg}" for (t, h), (rc, msg) in sorted(status.items())])
    for h in handles:
        lib.smm_destroy(h)
    np.savez(out, **arrays)


def _spawn_race(tmp_path):
    out = os.path.join(str(tmp_path), "race.npz")
    env = {k: val for k, val in os.environ.items() if k not in CREATE_ENV + PROCESS_ENV}
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), out]
    proc = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, f"child failed:\n{proc.stdout[-3000:]}\n{proc.stderr[-3000:]}"
    with np.load(out) as z:
        return {k: z[k] for k in z.files}


def _check_oracle(oracle, ref_order, op, x, y, what):
    """Bits of the oracle (rounded once to float32 for float32 y) in reference order; fast sums
    within 1e-12 sum |w| |x_filled| of it, plus the float32 rounding for float32 y."""
    ref = _oracle_result(oracle, op, x)
    assert np.array_equal(np.isnan(y), np.isnan(ref)), what + ": NaN pattern, " + _diff(y, ref)
    r = _f32(ref) if y.dtype == F32 else ref
    if ref_order:
        assert _same_bits(y, r), what + ": " + _diff(y, r)
        return
    assert np.array_equal(np.isinf(y), np.isinf(r)), what
    fin = np.isfinite(r)
    tol = 1e-12 * _backward_scale(op, x)[fin]
    if y.dtype == F32:
        tol = tol + np.spacing(np.abs(r[fin])).astype(F64)
    err = np.abs(y[fin].astype(F64) - ref[fin])
    assert np.all(err <= np.maximum(tol, 1e-300)), (what, float(err.max()))


@pytest.mark.gpu
def test_first_launches_race_in_a_fresh_process(smm_lib, oracle, cuda, tmp_path):
    """8 threads, B = 1, 7, 37 and 200, every family x (f32, f64, int16 -> f32, int16 -> f64) x
    (f32, f64), first launches of every kernel racing: every call returns SMM_OK and gives the bits
    of the same call made alone, which match the oracle."""
    res = _spawn_race(tmp_path)
    errors = [s for s in res["status"] if s.split(" ", 3)[2] != "0"]
    assert not errors, "concurrent calls failed:\n" + "\n".join(errors)
    assert len(res["status"]) == N_THREADS * len(RACE_IDS)
    ops = [_base_operator(_recipe(rid)) for rid in RACE_IDS]
    bad = []
    for t in range(N_THREADS):
        B = _thread_B(t)
        for h, rid in enumerate(RACE_IDS):
            v, op = _recipe(rid), ops[h]
            xkind, ydt = _thread_combo(t, h)
            what = f"thread {t} {rid} B={B} {xkind[0]}->{np.dtype(ydt).name}"
            conc, seq = res[f"conc_{t}_{h}"], res[f"seq_{t}_{h}"]
            if not _same_bits(conc, seq):
                bad.append(what + ": concurrent != alone, " + _diff(conc, seq))
            _, x, _, _ = _race_input(v, op, xkind, B)
            _check_oracle(oracle, v.ref_order, op, x, seq, what)
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------ every entry point on one 3-D handle

MIXED_IDS = ["staged-l1k12-n256-fast", "compact-bulk-raw"]
MIXED_B = 37
MIXED_SEL = [3, 2, 0, 0, 1]
MIXED_REPEAT = 3


@pytest.mark.gpu
@pytest.mark.parametrize("vid", MIXED_IDS)
def test_entry_points_run_together_on_one_3d_handle(smm_lib, cuda, vid):
    """smm_apply and smm_apply_levels on user streams, smm_apply_host and smm_apply_levels_host
    with pinned and pageable data, two callers of each, all at once on one 3-D handle, three
    calls each: every result is bit-identical to the same call made alone.  On the compact set
    every device call takes its transposed buffer from the handle's pool on its own stream."""
    import torch
    from smmregrid_b200 import _lib
    v = BY_ID[vid]
    ops = _level_ops(v)
    n_src, n_dst = ops[0].n_src, ops[0].n_dst
    nsel = len(MIXED_SEL)
    idx = np.asarray(MIXED_SEL, np.int32)
    masked = np.array([ops[l].masked for l in MIXED_SEL], np.uint8)
    opts = _lib.apply_opts(v.kernel)
    fields = _slot_fields(v, F64, MIXED_B, nsel)
    x32 = fields[0].astype(F32)
    xl = np.stack(fields, axis=1)                                  # [B, nsel, n_src] float64
    x32_dev, xl_dev = torch.from_numpy(x32).cuda(), torch.from_numpy(xl).cuda()
    torch.cuda.synchronize()
    keep = []
    h = _create_levels(smm_lib, v, ops)
    try:
        def dev_apply(stream):
            ys = []
            with torch.cuda.stream(stream):
                for l in range(3):
                    y = torch.full((MIXED_B, n_dst), -7.0, dtype=torch.float64, device="cuda")
                    _lib.check(smm_lib.smm_apply(h, l, x32_dev.data_ptr(), 0, MIXED_B, n_src, y.data_ptr(), 1, n_dst,
                                                 int(ops[l].masked), ops[l].amin, opts, stream.cuda_stream))
                    ys.append(y)
            stream.synchronize()
            return np.stack([y.cpu().numpy() for y in ys])

        def dev_levels(stream):
            with torch.cuda.stream(stream):
                y = torch.full((MIXED_B, nsel, n_dst), -7.0, dtype=torch.float32, device="cuda")
                _lib.check(smm_lib.smm_apply_levels(h, nsel, idx.ctypes.data, xl_dev.data_ptr(), 1, MIXED_B,
                                                    nsel * n_src, n_src, y.data_ptr(), 0, nsel * n_dst, n_dst,
                                                    masked.ctypes.data, ops[0].amin, opts, stream.cuda_stream))
            stream.synchronize()
            return y.cpu().numpy()

        def host_apply(pinned):
            x = _host_array((MIXED_B, n_src), F32, pinned, keep)
            x[:] = x32
            y = _host_array((MIXED_B, n_dst), F64, pinned, keep)
            y[:] = -7.0
            _lib.check(smm_lib.smm_apply_host(h, 0, x.ctypes.data, 0, MIXED_B, n_src, y.ctypes.data, 1, n_dst,
                                              int(ops[0].masked), ops[0].amin, opts, 7))
            return np.array(y)

        def host_levels(pinned):
            x = _host_array(xl.shape, F64, pinned, keep)
            x[:] = xl
            y = _host_array((MIXED_B, nsel, n_dst), F32, pinned, keep)
            y[:] = -7.0
            _lib.check(smm_lib.smm_apply_levels_host(h, nsel, idx.ctypes.data, x.ctypes.data, 1, MIXED_B,
                                                     y.ctypes.data, 0, masked.ctypes.data, ops[0].amin, opts, 7))
            return np.array(y)

        callers = [("apply", dev_apply, True), ("apply", dev_apply, True), ("levels", dev_levels, True),
                   ("levels", dev_levels, True), ("host", host_apply, True), ("host", host_apply, False),
                   ("levels_host", host_levels, True), ("levels_host", host_levels, False)]
        args = [torch.cuda.Stream() if name in ("apply", "levels") else pinned for name, _, pinned in callers]
        alone = {name: fn(torch.cuda.Stream() if name in ("apply", "levels") else True) for name, fn, _ in callers}
        assert np.isnan(alone["levels"][:, 0]).all() and np.isnan(alone["levels_host"][:, 0]).all()
        assert _same_bits(alone["host"], alone["apply"][0]) and _same_bits(alone["levels_host"], alone["levels"])
        got = [[] for _ in callers]
        errors = []
        barrier = threading.Barrier(len(callers))

        def worker(i):
            name, fn, _ = callers[i]
            try:
                barrier.wait()
                for _ in range(MIXED_REPEAT):
                    got[i].append(fn(args[i]))
            except Exception as e:          # noqa: BLE001
                errors.append(f"{name} #{i}: {e!r}")

        threads = [threading.Thread(target=worker, args=(i,)) for i in range(len(callers))]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        assert not errors, errors
        bad = []
        for i, (name, _, pinned) in enumerate(callers):
            assert len(got[i]) == MIXED_REPEAT
            for k, y in enumerate(got[i]):
                if not _same_bits(y, alone[name]):
                    bad.append(f"{vid} {name} #{i} (pinned={pinned}) call {k}: " + _diff(y, alone[name]))
        assert not bad, "\n".join(bad)
    finally:
        smm_lib.smm_destroy(h)


# ------------------------------------------------------------------ smm_last_error

@pytest.mark.gpu
def test_last_error_stays_with_its_thread(smm_lib, cuda):
    """Threads that pass a level out of range each read back their own message -- also after a
    later successful call -- while the other threads' applies succeed with the right bits."""
    import torch
    from smmregrid_b200 import _lib
    lib = smm_lib
    v = BY_ID["staged-l1k12-n256-fast"]
    ops = _level_ops(v)
    op = ops[0]
    B = 37
    x = torch.from_numpy(_slot_fields(v, F32, B, 1)[0]).cuda()
    torch.cuda.synchronize()
    h = _create_levels(lib, v, ops)
    try:
        def apply(level, stream):
            with torch.cuda.stream(stream):
                y = torch.full((B, op.n_dst), -7.0, dtype=torch.float64, device="cuda")
                rc = lib.smm_apply(h, level, x.data_ptr(), 0, B, op.n_src, y.data_ptr(), 1, op.n_dst, int(op.masked),
                                   op.amin, None, stream.cuda_stream)
            return rc, y

        st0 = torch.cuda.Stream()
        rc, want = apply(0, st0)
        assert rc == _lib.SMM_OK
        st0.synchronize()
        want = want.cpu().numpy()
        n = 8
        barrier = threading.Barrier(n)
        bad = []

        def worker(t):
            st = torch.cuda.Stream()
            try:
                barrier.wait()
                for i in range(20):
                    if t % 2:
                        rc, y = apply(0, st)
                        st.synchronize()
                        if rc != _lib.SMM_OK or not _same_bits(y.cpu().numpy(), want):
                            bad.append(f"thread {t} call {i}: rc {rc}")
                        continue
                    level = 1000 + 10 * t + i % 3
                    rc, _ = apply(level, st)
                    msg = lib.smm_last_error().decode()
                    if rc != _lib.SMM_ERR_INVALID or f"level {level} out of range" not in msg:
                        bad.append(f"thread {t} call {i}: rc {rc}, {msg!r}")
                    rc, _ = apply(0, st)
                    st.synchronize()
                    msg2 = lib.smm_last_error().decode()
                    if rc != _lib.SMM_OK or msg2 != msg:
                        bad.append(f"thread {t} call {i}: after a success {msg2!r} (was {msg!r})")
            except Exception as e:          # noqa: BLE001
                bad.append(f"thread {t}: {e!r}")

        threads = [threading.Thread(target=worker, args=(t,)) for t in range(n)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        assert not bad, "\n".join(bad[:20])
    finally:
        lib.smm_destroy(h)


# ------------------------------------------------------------------ front end

# results of 8.8 MB (2-D) and 10.4 MB (3-D) float64: the pinned result pool serves them
FRONT_B, FRONT_T = 17, 5
FRONT_THREADS = 3
FRONT_CALLS = 6


def _front_regridders():
    from smmregrid_b200 import Regridder, synth
    rg = Regridder(weights=synth.conservative_latlon(36, 18, 360, 180), remap_area_min=0.5)
    w3 = synth.ocean3d_weights(36, 18, 360, 180, n_levels=4, seed=3, level_values=[5.0, 15.0, 30.0, 60.0])
    return rg, Regridder(weights=w3, remap_area_min=0.5)


@pytest.mark.gpu
def test_front_end_threads_share_one_regridder(smm_lib, cuda):
    """Threads share one 2-D and one 3-D Regridder and call them in a loop, all at once: numpy
    input whose results the pinned pool serves from the second call on, CUDA tensors under each
    thread's own torch stream, and regrid3d on numpy input.  Each thread holds its last two
    results; every result, checked when it arrives and again at the end, equals the result of
    the same call made alone.  A pool buffer handed out while a thread still holds it would be
    overwritten by another thread's result."""
    import torch
    import importlib
    from smmregrid_b200 import synth
    regrid_mod = importlib.import_module("smmregrid_b200.regrid")     # (the package exports a function of that name)
    rg, rg3 = _front_regridders()
    xs = [synth.synthetic_field((FRONT_B, 18, 36), F32, seed=10 + t, nan_mode="random") for t in range(FRONT_THREADS)]
    x3s = [synth.synthetic_field((FRONT_T, 4, 18, 36), F64, seed=20 + t, nan_mode="random")
           for t in range(FRONT_THREADS)]
    # results made alone (copies: the pool's buffers go back to it)
    want = [np.array(rg.regrid(x), copy=True) for x in xs]
    want3 = [np.array(rg3.regrid3d(x), copy=True) for x in x3s]
    assert want[0].nbytes >= 8 << 20 and want3[0].nbytes >= 8 << 20
    x_devs = [torch.from_numpy(x).cuda() for x in xs]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(FRONT_THREADS)]

    def numpy_2d(t):
        return rg.regrid(xs[t]), want[t]

    def tensor_2d(t):
        with torch.cuda.stream(streams[t]):
            y = rg.regrid(x_devs[t])
        streams[t].synchronize()
        return y.cpu().numpy(), want[t]

    def numpy_3d(t):
        return rg3.regrid3d(x3s[t]), want3[t]

    kinds = [("numpy", numpy_2d), ("tensor", tensor_2d), ("regrid3d", numpy_3d)]
    callers = [(name, fn, t) for name, fn in kinds for t in range(FRONT_THREADS)]
    barrier = threading.Barrier(len(callers))
    held = [[] for _ in callers]
    bad = []

    def worker(i):
        name, fn, t = callers[i]
        try:
            barrier.wait()
            for k in range(FRONT_CALLS):
                y, w = fn(t)
                if not _same_bits(np.asarray(y), w):
                    bad.append(f"{name} thread {t} call {k}: " + _diff(np.asarray(y), w))
                held[i] = (held[i] + [(k, y, w)])[-2:]
        except Exception as e:              # noqa: BLE001
            bad.append(f"{name} thread {t}: {e!r}")

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(len(callers))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    for i, (name, _, t) in enumerate(callers):
        for k, y, w in held[i]:
            if not _same_bits(np.asarray(y), w):
                bad.append(f"{name} thread {t} call {k}, held to the end: " + _diff(np.asarray(y), w))
    assert not bad, "\n".join(bad[:20])
    # the loop did go through the pool: pinned buffers of both result sizes exist
    sizes = [t.numel() for t, _ in regrid_mod._pinned_results._bufs]
    for nbytes in (want[0].nbytes, want3[0].nbytes):
        assert any(nbytes <= s <= 2 * nbytes for s in sizes), (nbytes, sizes)


@pytest.mark.gpu
def test_dask_uneven_chunks_on_threads(smm_lib, cuda):
    """A dask-backed DataArray with uneven chunks, computed by the threaded scheduler (one task
    per chunk, the tasks sharing the Regridder): equal to the eager result."""
    dask_array = pytest.importorskip("dask.array")
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import refshim
    from smmregrid_b200 import synth
    rg, _ = _front_regridders()
    x = synth.synthetic_field((FRONT_B, 18, 36), F32, seed=3, nan_mode="random")
    want = np.array(rg.regrid(x), copy=True)
    lazy = dask_array.from_array(x, chunks=((3, 5, 1, 8), 18, 36))
    da = refshim.DataArray(lazy, ("time", "lat", "lon"), coords={"time": np.arange(float(FRONT_B))}, name="tas")
    out = rg.regrid(da)
    got = np.asarray(out.data.compute(scheduler="threads"))
    assert _same_bits(got.reshape(want.shape), want), _diff(got.reshape(want.shape), want)


if __name__ == "__main__":
    _race_main(sys.argv[1])
