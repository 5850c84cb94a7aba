"""CF-packed int16 sources against float32 sources: device-resident and end-to-end throughput.

    python scripts/packed_throughput.py --out DIR [--configs C4,C2,...] [--reps 5]

Writes DIR/r03a_packed_device.json and DIR/r03a_packed_e2e.json, each with the GPU name and power
limit of the run.

Device-resident runs: the raw int16 slab (values over the whole int16 range, 1 % fill values) and
its decoded float32 (and, for C4, float64) slab both live in HBM; they are timed interleaved with
CUDA events around `launches` calls of Regridder.regrid each, after a warm-up, and every slab is
larger than the 126 MB L2.  The decoded slab is made on the device with the decode's own
arithmetic (separate multiply and add in the decoded dtype, fill values -> NaN), and every int16
output is compared bit for bit with the float path's output on it.  Bytes per call = B x L x
(n_src x source itemsize + n_dst x 8); GB/s over 6499 GB/s (the measured B200 copy peak) is the
fraction reported.

End to end: Regridder.regrid of 128 host rows, 10 steps, pinned and pageable, int16 against
float32, next to smm_copy_ceiling of the same pinned bytes.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

COPY_PEAK_GBS = 6499.0
CONFIGS = {"C4": 1095, "C2": 3441, "C3": 96, "C2bic": 3441, "C5dis": 64}
SCALE, OFFSET, FILL = 0.0125, 250.0, -32767


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = out[0].split(", ")
        return {"gpu": name, "power_limit": power}
    except Exception as e:                          # noqa: BLE001 - recorded, not fatal
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def decode_torch(raw, D):
    """int16 -> D with the decode's arithmetic: D(v) * D(scale), then + D(offset), fill -> NaN."""
    import torch
    f32 = D == torch.float32
    x = raw.to(D)
    x.mul_(float(np.float32(SCALE)) if f32 else SCALE)          # separate kernels: each rounded once in D
    x.add_(float(np.float32(OFFSET)) if f32 else OFFSET)
    x[raw == FILL] = float("nan")
    return x


def same_bits(a, b):
    import torch
    na, nb = torch.isnan(a), torch.isnan(b)
    return bool(torch.equal(na, nb)) and bool(torch.equal(a[~na], b[~nb]))


def time_calls(fn, launches):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def device_runs(names, reps, launches):
    import torch
    from smmregrid_b200 import CFPacking, Regridder, synth
    out = []
    for name in names:
        B = CONFIGS[name]
        w = synth.config_weights(name)
        rg = Regridder(weights=w, remap_area_min=0.5, device=0)
        n_src, n_dst = rg.n_src, rg.n_dst
        L = w.n_levels if rg.mask_dim else 1
        shape = (B, L, n_src) if L > 1 else (B, n_src)
        g = torch.Generator(device="cuda").manual_seed(1)
        raw = torch.randint(-32768, 32768, shape, dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
        raw[torch.rand(shape, device="cuda", generator=g) < 0.01] = FILL
        for D in ((torch.float32, torch.float64) if name == "C4" else (torch.float32,)):
            pk = CFPacking(np.float32(SCALE) if D == torch.float32 else SCALE,
                           np.float32(OFFSET) if D == torch.float32 else OFFSET, [FILL])
            xf = decode_torch(raw, D)
            run_f = lambda: rg.regrid(xf)                               # noqa: E731
            run_p = lambda: rg.regrid(raw, packing=pk)                  # noqa: E731
            yf, yp = run_f(), run_p()                                   # warm-up (and the output check)
            torch.cuda.synchronize()
            ok = same_bits(yf, yp)
            del yf, yp
            tf, tp = [], []
            for _ in range(reps):                                       # interleaved
                tf.append(time_calls(run_f, launches))
                tp.append(time_calls(run_p, launches))
            ms_f, ms_p = float(np.median(tf)), float(np.median(tp))
            points = B * L * n_src
            sxf = 4 if D == torch.float32 else 8
            by_f, by_p = B * L * (n_src * sxf + n_dst * 8), B * L * (n_src * 2 + n_dst * 8)
            rec = {"config": name, "B": B, "levels": L, "n_src": n_src, "n_dst": n_dst,
                   "decoded_dtype": str(D).replace("torch.", ""), "bits_identical": ok,
                   "float": {"ms": ms_f, "points_per_s": points / ms_f * 1e3, "gbs": by_f / ms_f / 1e6,
                             "frac_of_copy_peak": by_f / ms_f / 1e6 / COPY_PEAK_GBS, "ms_reps": tf},
                   "int16": {"ms": ms_p, "points_per_s": points / ms_p * 1e3, "gbs": by_p / ms_p / 1e6,
                             "frac_of_copy_peak": by_p / ms_p / 1e6 / COPY_PEAK_GBS, "ms_reps": tp},
                   "speedup": ms_f / ms_p}
            print(json.dumps({k: rec[k] for k in ("config", "decoded_dtype", "bits_identical", "speedup")}
                             | {"ms_float": ms_f, "ms_int16": ms_p}), flush=True)
            out.append(rec)
            del xf
        del raw
        torch.cuda.empty_cache()
    return out


def e2e_runs(steps, rows):
    import torch
    from smmregrid_b200 import CFPacking, Regridder, _lib, synth
    w = synth.config_weights("C4")
    rg = Regridder(weights=w, remap_area_min=0.5, device=0)
    n_src = rg.n_src
    pk = CFPacking(np.float32(SCALE), np.float32(OFFSET), [FILL])
    g = torch.Generator().manual_seed(2)
    raw = torch.randint(-32768, 32768, (rows, n_src), dtype=torch.int32, generator=g).to(torch.int16)
    xf = decode_torch(raw.cuda(), torch.float32).cpu()
    lib = _lib.load()
    res = {"config": "C4", "rows_per_step": rows, "steps": steps}
    for pinned in (True, False):
        if pinned:
            rp, fp = raw.pin_memory(), xf.pin_memory()
        else:
            rp, fp = raw.numpy(), xf.numpy()
        for tag, fn in (("float32", lambda: rg.regrid(fp)), ("int16", lambda: rg.regrid(rp, packing=pk))):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            key = ("pinned" if pinned else "pageable") + "_" + tag
            res[key] = {"points_per_s": rows * n_src * steps / dt, "ms_per_step": 1e3 * dt / steps,
                        "h2d_gbs": rows * n_src * (4 if tag == "float32" else 2) * steps / dt / 1e9}
            print(key, json.dumps(res[key]), flush=True)
        if pinned:
            sec = ctypes.c_double()
            _lib.check(lib.smm_copy_ceiling(0, fp.data_ptr(), fp.numel() * 4, 0, 5, ctypes.byref(sec)))
            res["h2d_ceiling_gbs"] = fp.numel() * 4 / sec.value / 1e9
    ok = np.array_equal(np.asarray(rg.regrid(raw.numpy(), packing=pk)), np.asarray(rg.regrid(xf.numpy())),
                        equal_nan=True)
    res["bits_identical"] = bool(ok)
    for tag in ("float32", "int16"):
        res[f"pinned_{tag}"]["frac_of_h2d_ceiling"] = res[f"pinned_{tag}"]["h2d_gbs"] / res["h2d_ceiling_gbs"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-rows", type=int, default=128)
    ap.add_argument("--no-e2e", action="store_true", help="device-resident runs only")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("packed_throughput.py measures on a CUDA device; none is available")
    os.makedirs(args.out, exist_ok=True)
    ident = gpu_identity()
    dev = {"measured_on": ident, "copy_peak_gbs": COPY_PEAK_GBS,
           "runs": device_runs([c for c in args.configs.split(",") if c], args.reps, args.launches)}
    with open(os.path.join(args.out, "r03a_packed_device.json"), "w") as f:
        json.dump(dev, f, indent=1)
    if args.no_e2e:
        return
    e2e = {"measured_on": ident, **e2e_runs(args.e2e_steps, args.e2e_rows)}
    with open(os.path.join(args.out, "r03a_packed_e2e.json"), "w") as f:
        json.dump(e2e, f, indent=1)


if __name__ == "__main__":
    main()
