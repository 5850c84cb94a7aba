#!/usr/bin/env python
"""bench.py -- headline benchmark of the weight-application path (BASELINE.json metric).

Workload: BASELINE config C4, 0.1 deg global (3600x1800 = 6.48 M source points) -> r360x180
first-order conservative (110 links/row, 7.128 M links, float64 weights), float32 fields,
float64 accumulate/output (the reference's result_type).  The 8760-step batch shards over
the GPUs of one box with replicated weights and no data-path collective: every rank holds
`--batch` (default 1095 = 8760/8) resident time steps, so N = 8 is exactly C4 and N < 8 is
the same per-GPU work (weak scaling).  One *step* = one smm_apply over the rank's whole
resident slab (28.4 GB of source, far larger than the 126 MB L2, so no flush is needed).

Prints ONE JSON line (rank 0).  `value` = source points regridded per second over all GPUs
with inputs resident in HBM (CUDA events, max over ranks); `e2e` = same metric through the
public API (`Regridder.regrid`) from pinned HOST buffers, H2D + D2H inside the timed region;
`roofline` = algorithmic bytes / measured launch time against MEASURED_PEAKS.json;
`cpu_baseline` = the reference's CPU algorithm (oracle C port, all host threads) on a
bounded sample.  `--impl reference` times that CPU port as its own arm.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "regridded source points/sec, 0.1deg->1deg remapcon"
UNIT = "points/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", help="C4 (default) | C2 | C4s<k> (C4 grids scaled down k x)")
    ap.add_argument("--batch", type=int, default=0, help="resident batch rows per GPU (0 = workload default)")
    ap.add_argument("--e2e-batch", type=int, default=128, help="host batch rows per e2e step")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--strong-rows", type=int, default=8760,
                    help="fixed total batch rows of the strong-scaling sub-record (the north-star year); 0 = skip")
    ap.add_argument("--strong-steps", type=int, default=3)
    ap.add_argument("--no-others", action="store_true", help="skip the other_configs records (N = 1 only)")
    ap.add_argument("--xdtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--ydtype", default="f64", choices=["f32", "f64"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--kernel", default="auto", choices=["auto", "staged", "gather", "compact"])
    ap.add_argument("--nan", default="none", choices=["none", "land", "random"],
                    help="missing values in the synthetic slab: none | land (static smooth land mask, ~35%%) | random (30%% of points)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step to DIR/y.npy (rank 0; a fixed sample of its rows "
                         "when larger than 48 MiB), so that two builds can be compared output for output")
    return ap.parse_args()


def workload(name):
    from smmregrid_b200 import synth
    if name == "C4":
        return synth.config_weights("C4"), 1095, "C4 0.1deg 3600x1800 -> r360x180 remapcon (110 links/row), synthetic CDO-shaped weights"
    if name == "C2":
        return synth.config_weights("C2"), 3441, "C2 ERA5-like 1440x721 -> r360x180 remapcon (25 links/row), synthetic CDO-shaped weights"
    if name.startswith("C4s"):
        k = int(name[3:])
        return synth.config_weights("C4", k), 64, f"C4 scaled 1/{k}: {3600 // k}x{1800 // k} -> {360 // k}x{180 // k} remapcon"
    if name == "C3":          # ORCA1-like 362x292, 75 levels with level-varying mask -> 1 deg remapcon
        return synth.config_weights("C3"), 96, "C3 ORCA-like 362x292 x 75 levels (level-varying mask) -> r360x180 remapcon, per-level weights"
    if name == "C3tri":       # the same with a tripolar (north-fold) curvilinear index space
        return synth.config_weights("C3tri"), 96, "C3tri ORCA-like TRIPOLAR 362x292 x 75 levels (level-varying mask, north fold) -> r360x180 conservative-like, per-level weights"
    if name == "C2bic":       # bicubic-like: 16 links per row, weights of both signs
        return synth.config_weights("C2bic"), 3441, "C2bic ERA5-like 1440x721 -> r360x180 bicubic-like (16 links/row, weights of both signs)"
    if name in ("C5hpnn", "C5hpdis"):
        return synth.config_weights(name), 64, f"{name}: HEALPix nside 1024 NESTED (12.58M cells) -> 0.25deg, {'1' if name == 'C5hpnn' else '4'} link(s)/row"
    if name in ("C5nn", "C5dis"):
        return synth.config_weights(name), 64, f"{name}: 20.97M unstructured cells -> 0.25deg, {'1' if name == 'C5nn' else '4'} link(s)/row, random source order"
    if name.startswith("con:"):          # con:<nlon_s>x<nlat_s>:<nlon_d>x<nlat_d>  (experiments)
        _, a, b = name.split(":")
        (ls, ts), (ld, td) = [tuple(int(v) for v in g.split("x")) for g in (a, b)]
        return synth.conservative_latlon(ls, ts, ld, td), 1024, f"remapcon {ls}x{ts} -> {ld}x{td}"
    if name.startswith("bil:"):          # bil:<nlon_s>x<nlat_s>:<nlon_d>x<nlat_d>  (experiments)
        _, a, b = name.split(":")
        (ls, ts), (ld, td) = [tuple(int(v) for v in g.split("x")) for g in (a, b)]
        return synth.bilinear_latlon(ls, ts, ld, td), 256, f"remapbil {ls}x{ts} -> {ld}x{td}"
    raise SystemExit(f"unknown workload {name}")


def kernel_source_hash():
    """sha1 over the kernel sources: ties an ncu capture (profiles/traffic.json) to the code it
    was taken from (the GPU box has no .git)."""
    import hashlib
    h = hashlib.sha1()
    d = os.path.join(ROOT, "smmregrid_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".h", ".cpp")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(workload_name, batch_rows, xdtype, ydtype):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the ncu capture of this exact
    configuration, or None -- also None when the capture predates the current kernel sources
    (scripts/round_evidence.sh regenerates profiles/traffic.json and records the hash)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if t.get("kernel_source_hash") != kernel_source_hash():
            return None
        for c in t["captures"]:
            if (c["workload"], c["batch_rows"], c["x_dtype"], c["y_dtype"]) == (workload_name, batch_rows, xdtype, ydtype):
                return c["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


def algorithmic_bytes(info, B, sx, sy, masked, area_min):
    """BASELINE.md §2: CSR values+cols+rowptr (+imask, +frac) + source slab read + destination slab written."""
    b = info["nnz"] * (8 + 4) + (info["n_dst"] + 1) * 4
    if masked:
        b += info["n_dst"] * 1
    if area_min > 0:
        b += info["n_dst"] * 8
    return b + B * info["n_src"] * sx + B * info["n_dst"] * sy


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout):
        """Block until the first sample has arrived, so the timed region is certain to be covered."""
        t_end = time.perf_counter() + timeout
        while self.proc and not self.lines and time.perf_counter() < t_end:
            time.sleep(0.02)
        time.sleep(0.05)

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            f = [s.strip() for s in line.split(",")]
            if len(f) < 7:
                continue
            try:
                clk, mx = float(f[0]), float(f[1])
            except ValueError:
                continue
            smax = mx
            if t0 - 0.05 <= ts <= t1 + 0.05:
                sm.append(clk)
                for n, v in zip(names, f[3:7]):
                    if v == "Active":
                        reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 48 << 20


def dump_output(out_dir, y):
    """--dump-outputs: ``y`` (torch tensor or numpy array) as ``out_dir/y.npy``.  An output larger
    than DUMP_BYTES is viewed as rows of its last axis and a fixed sample of those rows (seed 0,
    kept in order) is written as a 2-D array."""
    import numpy as np
    rows = y.reshape(-1, y.shape[-1])
    k = DUMP_BYTES // (rows.shape[1] * rows.dtype.itemsize)
    out = y
    if k < rows.shape[0]:
        out = rows[np.sort(np.random.default_rng(0).choice(rows.shape[0], max(1, k), replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "y.npy"), out.cpu().numpy() if hasattr(out, "cpu") else out)


def cpu_port_throughput(w, n_threads, rows, reps, seed=99):
    """The reference's CPU algorithm (oracle C port: fill + COO-order loop + 3 where passes,
    one pthread per batch chunk like dask's threaded scheduler) on `rows` batch rows.
    Returns (points/s of the best rep, seconds of every rep, the last rep's result)."""
    import numpy as np
    from oracle import oracle as orc
    from smmregrid_b200 import synth
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    mat = orc.compute_weights_matrix_c(w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst)
    x = synth.synthetic_field((rows, n_src), np.float32, seed=seed)
    y = np.empty((rows, n_dst), np.float64)
    imask = np.ones(n_dst, np.int32)
    best = float("inf")
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        orc.apply_weights_c(x, mat, imask, w["dst_grid_frac"], 0.5, True, nthreads=n_threads, out=y)
        dt = time.perf_counter() - t0
        times.append(dt)
        best = min(best, dt)
    return rows * n_src / best, times, y


def run_reference(args):
    """--impl reference: the reference's own CPU path.  The reference package cannot be
    installed here (xarray/dask/sparse absent, no network: see DESIGN.md), so this arm times
    the oracle C port of its algorithm with every host thread, on rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w, _, desc = workload(args.workload)
    cores = len(os.sched_getaffinity(0))
    rows = max(cores, min(4 * cores, 512))
    for _ in range(args.warmup):
        cpu_port_throughput(w, cores, min(rows, cores), 1)
    tput, times, y = cpu_port_throughput(w, cores, rows, max(1, args.steps))
    if args.dump_outputs:
        dump_output(args.dump_outputs, y)
    n_src = w.sizes["src_grid_size"]
    ms = 1e3 * sum(times) / len(times)
    val = rows * n_src / (sum(times) / len(times))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "sample_rows_per_step": rows, "x_dtype": "f32", "y_dtype": "f64"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{rows} batch rows per step, {args.steps} steps, mean"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_3d(args, rg, w, T, xdt, ydt, sx, sy, area_min, dev, g, world, rank, desc):
    """BASELINE config C3: [T, L, n_src] ocean-like field, one grouped launch over all levels
    (Regridder.regrid3d -> smm_apply_levels).  Reported like the 2-D line; single GPU."""
    import numpy as np
    import torch
    from smmregrid_b200 import _lib
    L, n_src, n_dst = rg.weights_matrix.n_levels, rg.n_src, rg.n_dst
    x = torch.empty((T, L, n_src), dtype=xdt, device=dev)
    x.normal_(10.0, 2.0, generator=g)
    land = torch.from_numpy(np.asarray(w["src_grid_imask"]).reshape(L, n_src) == 0).to(dev)
    x[:, land] = float("nan")
    lib = _lib.load()
    for _ in range(max(3, args.warmup)):
        y = rg.regrid(x)
    torch.cuda.synchronize(dev)
    l0 = lib.smm_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        y = rg.regrid(x)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_output(args.dump_outputs, y)
    infos = [rg.weights_matrix.info(l) for l in range(L)]
    nnz = sum(i["nnz"] for i in infos)
    abytes = nnz * 12 + L * ((n_dst + 1) * 4 + n_dst * 9) + T * L * (n_src * sx + n_dst * sy)
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = abytes / (ms * 1e-3) / 1e9
    traffic = measured_traffic(args.workload, T, args.xdtype, args.ydtype)
    print(json.dumps({
        "metric": METRIC, "value": T * L * n_src / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "time_steps": T, "levels": L, "n_src": n_src, "n_dst": n_dst, "nnz_all_levels": nnz,
                   "kernels": sorted({i["kernel_name"] for i in infos}), "lanes_per_row": infos[0]["lanes_per_row"],
                   "nan_cells": int(torch.isnan(y).sum().item()), "x_dtype": args.xdtype, "y_dtype": args.ydtype},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "algorithmic_bytes_per_launch": abytes},
        "gpu_launches": int(lib.smm_launch_count() - l0)}), flush=True)


def other_configs(dev, peak):
    """The other BASELINE configurations on the same box, a few launches each (device-resident
    slab, CUDA events): ms, GB/s and fraction of the measured peak for both byte models."""
    import numpy as np
    import torch
    from smmregrid_b200 import Regridder, _lib, synth
    lib = _lib.load()
    out = []
    specs = [("C2", "C2", 3441, "none"), ("C2 + static land mask (35 % of sources NaN)", "C2", 3441, "land"),
             ("C3", "C3", 96, "levels"), ("C3 on a tripolar (north-fold) index space", "C3tri", 96, "levels"),
             ("C2 bicubic-like (16 links/row, both signs: reference-order sums)", "C2bic", 3441, "none"),
             ("C5nn", "C5nn", 64, "none"), ("C5dis", "C5dis", 64, "none"),
             ("C4 with reference-order sums forced (bit-identical values; SMM_SUM_REFERENCE)", "C4", 256, "none", "reference")]
    for label, name, B, nan, *rest in specs:
        t_build = time.perf_counter()
        w, _, desc = workload(name)
        rg = Regridder(weights=w, remap_area_min=0.5, device=dev.index, summation=rest[0] if rest else None)
        t_build = time.perf_counter() - t_build
        L = rg.weights_matrix.n_levels
        infos = [rg.weights_matrix.info(l) for l in range(L)]
        n_src, n_dst = rg.n_src, rg.n_dst
        g = torch.Generator(device=dev).manual_seed(77)
        shape = (B, L, n_src) if rg.mask_dim else (B, n_src)
        x = torch.empty(shape, dtype=torch.float32, device=dev)
        x.normal_(280.0, 20.0, generator=g)
        if nan == "land":
            ii = torch.arange(n_src, device=dev, dtype=torch.float32)
            nlon = float(np.atleast_1d(w["src_grid_dims"])[0])
            lon, lat = (ii % nlon) / nlon * 6.2832, torch.floor(ii / nlon) / (n_src / nlon) * 3.1416
            x[:, (torch.sin(2 * lon + 0.5) * torch.sin(lat) + 0.6 * torch.cos(3 * lon - 1.0) * torch.sin(2 * lat)) > 0.25] = float("nan")
        elif nan == "levels":
            x[:, torch.from_numpy(np.asarray(w["src_grid_imask"]).reshape(L, n_src) == 0).to(dev)] = float("nan")
        for _ in range(3):
            y = rg.regrid(x)
        torch.cuda.synchronize(dev)
        l0 = lib.smm_launch_count()
        steps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            y = rg.regrid(x)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        launches = (lib.smm_launch_count() - l0) // steps
        nnz = sum(i["nnz"] for i in infos)
        masked = bool(np.any(rg.masked))
        fixed = nnz * 12 + L * ((n_dst + 1) * 4 + n_dst * 8 + (n_dst if masked else 0))
        touched = sum(i["touched_src"] for i in infos)
        ab = fixed + B * L * (n_src * 4 + n_dst * 8)
        ab_t = fixed + B * (touched * 4 + L * n_dst * 8)
        kern = infos[0]["kernel_name"]
        if kern == "gather" and launches >= 2:
            kern = "compact_kernel + compact_apply_kernel"
        out.append({"config": label, "workload": desc, "batch_rows": B, "levels": L, "x_dtype": "f32", "y_dtype": "f64",
                    "ms_per_launch_group": ms, "launches_per_apply": int(launches), "kernel": kern,
                    "packed_rows": infos[0]["packed_rows"], "lanes_per_row": infos[0]["lanes_per_row"],
                    "summation": infos[0]["summation_name"],
                    "achieved_gbs": ab / (ms * 1e-3) / 1e9, "frac": ab / (ms * 1e-3) / 1e9 / peak,
                    "achieved_touched_src_gbs": ab_t / (ms * 1e-3) / 1e9, "frac_touched_src": ab_t / (ms * 1e-3) / 1e9 / peak,
                    "src_points_per_s": B * L * n_src / (ms * 1e-3), "operator_build_s": round(t_build, 2),
                    "nan_cells_out": int(torch.isnan(y).sum().item())})
        del x, y, rg, w
        torch.cuda.empty_cache()
    return out


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from smmregrid_b200 import Regridder, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from smmregrid_b200.shard import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local) if world > 1 else None      # host staging stays on the GPU's socket
    # the library is the one build() left in the tree: a run compiles nothing (the tree may be read-only)

    w, B_default, desc = workload(args.workload)
    B = args.batch or B_default
    xdt = torch.float32 if args.xdtype == "f32" else torch.float64
    ydt = np.float32 if args.ydtype == "f32" else np.float64
    sx, sy = (4 if args.xdtype == "f32" else 8), (4 if args.ydtype == "f32" else 8)
    area_min = 0.5
    rg = Regridder(weights=w, remap_area_min=area_min, device=local, out_dtype=ydt,
                   kernel=None if args.kernel == "auto" else args.kernel)
    info = rg.weights_matrix.info()
    n_src, n_dst = rg.n_src, rg.n_dst
    masked = bool(np.any(rg.masked))

    is3d = bool(rg.mask_dim)
    L = rg.weights_matrix.n_levels
    # synthetic slab generated on the device (seeded per rank), resident for the whole run
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    if is3d:
        return run_3d(args, rg, w, B, xdt, ydt, sx, sy, area_min, dev, g, world, rank, desc)
    x = torch.empty((B, n_src), dtype=xdt, device=dev)
    for b0 in range(0, B, 64):
        xb = x[b0:b0 + 64]
        xb.normal_(280.0, 20.0, generator=g)
    if args.nan != "none" and not is3d:
        if args.nan == "random":
            m = torch.rand(n_src, generator=g, device=dev) < 0.3
        else:       # smooth, contiguous "continents" (SURVEY 8d variant ii): same cells every step
            ii = torch.arange(n_src, device=dev, dtype=torch.float32)
            nlon = float(np.atleast_1d(w["src_grid_dims"])[0])
            lon, lat = (ii % nlon) / nlon * 6.2832, torch.floor(ii / nlon) / (n_src / nlon) * 3.1416
            m = (torch.sin(2 * lon + 0.5) * torch.sin(lat) + 0.6 * torch.cos(3 * lon - 1.0) * torch.sin(2 * lat)) > 0.25
        x[:, m] = float("nan")
        nan_frac = float(m.float().mean().item())
    else:
        nan_frac = 0.0
    y = torch.empty((B, n_dst), dtype=torch.float32 if args.ydtype == "f32" else torch.float64, device=dev)
    lib = _lib.load()
    stream = torch.cuda.current_stream(dev)
    xcode, ycode = (0 if args.xdtype == "f32" else 1), (0 if args.ydtype == "f32" else 1)

    opts = _lib.apply_opts(rg.kernel)

    def step():
        _lib.check(lib.smm_apply(rg.weights_matrix.handle, 0, x.data_ptr(), xcode, B, n_src,
                                 y.data_ptr(), ycode, n_dst, int(masked), area_min, opts, stream.cuda_stream))

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first(5.0)         # nvidia-smi can take a second to come up on a cold box
    launches0 = lib.smm_launch_count()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    evs[0].record(stream)
    for i in range(args.steps):
        step()
        evs[i + 1].record(stream)
    torch.cuda.synchronize(dev)
    t1 = time.perf_counter()
    launches = lib.smm_launch_count() - launches0
    total_ms = evs[0].elapsed_time(evs[-1])
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms_max = float(tt.item())
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, y)

    # ---- e2e: public API from HOST memory, H2D + D2H inside the timed region
    def all_max(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_regrids(xin, steps):
        """`steps` calls of Regridder.regrid(host array), all ranks at once; max-over-ranks seconds."""
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0e = time.perf_counter()
        for _ in range(steps):
            yh = rg.regrid(xin)
        torch.cuda.synchronize(dev)
        dt = all_max(time.perf_counter() - t0e)
        assert tuple(yh.shape[:1]) == (xin.shape[0],)
        return dt

    e2e = None
    if not args.no_e2e:
        Be = min(args.e2e_batch, B)
        h2d_bytes, d2h_bytes = Be * n_src * sx, Be * n_dst * sy
        xh = torch.empty((Be, n_src), dtype=xdt, pin_memory=True)
        xh.copy_(x[:Be])
        rg.regrid(xh[: min(Be, 8)])                               # warm the staging buffers
        yw = None
        for _ in range(3):                                        # and the pool of pinned result buffers: a loop that
            yw = rg.regrid(xh)                                    # keeps its last result, like the timed one, needs two
        del yw
        te = timed_regrids(xh, args.e2e_steps)
        e2e_val = world * Be * n_src * args.e2e_steps / te
        # what the PCIe links themselves sustain: bare cudaMemcpyAsync of the same pinned bytes,
        # all ranks at the same time (and the result's bytes in the other direction)
        sec = ctypes.c_double()
        if world > 1:
            dist.barrier()
        _lib.check(lib.smm_copy_ceiling(local, xh.data_ptr(), h2d_bytes, 0, 5, ctypes.byref(sec)))
        h2d_s = all_max(sec.value)
        yh_pin = torch.empty((Be, n_dst), dtype=y.dtype, pin_memory=True)
        if world > 1:
            dist.barrier()
        _lib.check(lib.smm_copy_ceiling(local, yh_pin.data_ptr(), d2h_bytes, 1, 5, ctypes.byref(sec)))
        d2h_s = all_max(sec.value)
        # the same through the C ABI alone (smm_apply_host into a preallocated pinned result):
        # separates the pipeline inside the library from the Python layer above it
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        tc0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            _lib.check(lib.smm_apply_host(rg.weights_matrix.handle, 0, xh.data_ptr(), xcode, Be, n_src,
                                          yh_pin.data_ptr(), ycode, n_dst, int(masked), area_min, opts, 0))
        tc = all_max(time.perf_counter() - tc0)
        ceiling_gbs = world * h2d_bytes / h2d_s / 1e9
        e2e_h2d_gbs = world * h2d_bytes * args.e2e_steps / te / 1e9
        # second figure: PAGEABLE numpy input, what Regridder.regrid(DataArray / ndarray) is handed
        # in practice (goes through pinned bounce buffers filled by host threads)
        xp = xh.numpy().copy()
        yw = rg.regrid(xp)
        yw = rg.regrid(xp)
        del yw
        p_steps = max(3, args.e2e_steps // 2)
        tp = timed_regrids(xp, p_steps)
        e2e = {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": d2h_bytes, "batch_rows_per_step": Be, "steps": args.e2e_steps,
               "ms_per_step": 1e3 * te / args.e2e_steps,
               "api": "Regridder.regrid(pinned host tensor) -> smm_apply_host -> new host array", "numa_node": numa,
               "h2d_gbs": e2e_h2d_gbs,
               "h2d_ceiling_gbs": ceiling_gbs,
               "d2h_ceiling_gbs": world * d2h_bytes / d2h_s / 1e9,
               "frac_of_ceiling": e2e_h2d_gbs / ceiling_gbs,
               "pinned_result_buffers": len(sys.modules["smmregrid_b200.regrid"]._pinned_results._bufs),
               "c_abi_only": {"h2d_gbs": world * h2d_bytes * args.e2e_steps / tc / 1e9, "ms_per_step": 1e3 * tc / args.e2e_steps,
                              "api": "smm_apply_host(pinned x, preallocated pinned y)"},
               "ceiling": f"bare pinned cudaMemcpyAsync of the same bytes, 5 back-to-back copies, all {world} rank(s) concurrently, max over ranks",
               "pageable": {"value": world * Be * n_src * p_steps / tp, "unit": UNIT, "steps": p_steps,
                            "ms_per_step": 1e3 * tp / p_steps, "h2d_gbs": world * h2d_bytes * p_steps / tp / 1e9,
                            "api": "Regridder.regrid(pageable numpy array): pinned bounce buffers filled by host threads"}}
        del xp, yh_pin

    # ---- strong scaling: the fixed north-star job (8760 steps) over the ranks of this run, with
    # the final host gather over NCCL inside the timed region
    strong = None
    if args.strong_rows > 0 and not is3d:
        from smmregrid_b200.shard import HostGather, batch_shard, gather_to_host
        Bs = args.strong_rows
        r0, r1 = batch_shard(Bs, world, rank)
        rows = r1 - r0
        y_full = torch.empty((rows, n_dst), dtype=y.dtype, device=dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # destinations of the gather, allocated once like an application would: a pinned array on
        # rank 0 (NCCL route) and a shared-memory array every rank maps (direct route)
        host_pin = torch.empty((Bs, n_dst), dtype=y.dtype, pin_memory=True) if rank == 0 else None
        hg = HostGather(Bs, (n_dst,), y.dtype, dst=0)

        def strong_step(via):
            """this rank's block of the year in resident chunks of <= B rows, then the gather"""
            ev0.record(stream)
            for c0 in range(0, rows, B):
                nb = min(B, rows - c0)
                _lib.check(lib.smm_apply(rg.weights_matrix.handle, 0, x.data_ptr(), xcode, nb, n_src,
                                         y_full[c0:].data_ptr(), ycode, n_dst, int(masked), area_min, opts,
                                         stream.cuda_stream))
            ev1.record(stream)
            return gather_to_host(y_full, Bs, dst=0, via=via, out=hg if via == "shm" else host_pin)

        def strong_run(via):
            full = strong_step(via)                               # warm-up (NCCL channels, page faults of the result)
            if rank == 0:
                assert tuple(full.shape) == (Bs, n_dst)
            apply_ms, total_s = [], []
            for _ in range(args.strong_steps):
                torch.cuda.synchronize(dev)
                if world > 1:
                    dist.barrier()
                ts0 = time.perf_counter()
                full = strong_step(via)
                torch.cuda.synchronize(dev)
                total_s.append(all_max(time.perf_counter() - ts0))
                apply_ms.append(all_max(ev0.elapsed_time(ev1)))
            if rank == 0 and via == "shm":                        # the two routes deliver the same array ...
                assert torch.equal(full[:: max(1, Bs // 64)].nan_to_num(), host_pin[:: max(1, Bs // 64)].nan_to_num())
                assert torch.equal(full[:3].nan_to_num(), y_full[:3].cpu().nan_to_num())     # ... which starts with rank 0's rows
            return sum(total_s) / len(total_s), 1e-3 * sum(apply_ms) / len(apply_ms)

        tot_n, app_n = strong_run("nccl")
        tot, app = strong_run("shm")
        strong = {"scaling": "strong", "total_batch_rows": Bs, "rows_per_rank": -(-Bs // world),
                  "value": Bs * n_src / tot, "unit": UNIT, "ms_per_step": 1e3 * tot, "steps": args.strong_steps,
                  "apply_ms": 1e3 * app, "gather_ms": 1e3 * (tot - app), "gather_frac": (tot - app) / tot,
                  "gather_bytes": Bs * n_dst * sy,
                  "gather": "shard.gather_to_host(via='shm'): every rank copies its [rows, n_dst] block device->host "
                            "over its own PCIe link into its rows of one shared-memory [%d, n_dst] array "
                            "(registered with the driver once), then a barrier" % Bs,
                  "nccl_route": {"ms_per_step": 1e3 * tot_n, "apply_ms": 1e3 * app_n, "gather_ms": 1e3 * (tot_n - app_n),
                                 "value": Bs * n_src / tot_n,
                                 "gather": ("shard.gather_to_host(via='nccl'): NCCL gather of the ranks' blocks to rank 0 over "
                                            "NVLink + device->host copy into one pinned array (the whole result crosses ONE PCIe link)")
                                 if world > 1 else "device->host copy of the result into one pinned array"},
                  "data": "every resident chunk re-reads the rank's synthetic %d-row slab (%.1f GB >> L2); "
                          "results go to distinct rows" % (B, B * n_src * sx / 1e9),
                  "value_apply_only": Bs * n_src / app}
        hg.close()
        del y_full, host_pin

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)"
    abytes = algorithmic_bytes(info, B, sx, sy, masked, area_min)
    traffic = measured_traffic(args.workload, B, args.xdtype, args.ydtype)
    avg_launch_s = 1e-3 * sum(per_launch_ms) / len(per_launch_ms)
    achieved = abytes / avg_launch_s / 1e9
    value = world * B * n_src * args.steps / (total_ms_max * 1e-3)

    cpu = None
    if world == 1 and not args.no_cpu:
        cores = len(os.sched_getaffinity(0))
        rows = max(cores, min(2 * cores, 256))
        tput, times, _ = cpu_port_throughput(w, cores, rows, 3)
        cpu = {"value": tput, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{rows} batch rows of the same workload, best of 3 ({min(times) * 1e3:.0f} ms)"}

    others = None
    if world == 1 and not args.no_others and args.workload == "C4":
        del x, y
        torch.cuda.empty_cache()
        others = other_configs(dev, peak)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "batch_rows_per_gpu": B, "global_batch_rows": B * world,
                   "n_src": n_src, "n_dst": n_dst, "nnz": info["nnz"], "x_dtype": args.xdtype,
                   "y_dtype": args.ydtype, "weights_dtype": "f64", "remap_area_min": area_min,
                   "kernel": info["kernel_name"], "lanes_per_row": info["lanes_per_row"],
                   "nan": args.nan, "nan_fraction_of_source": round(nan_frac, 3),
                   "parallelism": f"batch-sharded x{world}, weights replicated, no collective",
                   "l2": "resident slab (%.1f GB) >> 126 MB L2, no flush" % (B * n_src * sx / 1e9)},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "traffic_source": ("profiles/traffic.json (ncu --set full of this configuration, kernel sources %s)" % kernel_source_hash())
                     if traffic is not None else "no ncu capture of the current kernel sources",
                     "algorithmic_bytes_per_launch": abytes, "avg_launch_ms": avg_launch_s * 1e3,
                     "kernel": "smm::staged_kernel" if info["kernel_name"] == "staged"
                     else ("smm::gather_kernel" if launches <= args.steps
                           else "smm::compact_kernel + smm::compact_apply_kernel (two passes per 64 batch rows)"),
                     # stricter touched-source model (BASELINE.md §2): only source columns with >= 1 link
                     "achieved_touched_src": (abytes - B * (n_src - info["touched_src"]) * sx) / avg_launch_s / 1e9},
        "dst_points_per_s": world * B * n_dst * args.steps / (total_ms_max * 1e-3),
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if strong is not None:
        line["strong"] = strong
    if others is not None:
        line["other_configs"] = others
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
