"""float16 / bfloat16 sources read by the kernels against float32 sources and against widening
first: device-resident and end-to-end throughput.

    python scripts/half_throughput.py --out DIR [--configs C4,C2,...] [--reps 5]

Writes DIR/r03b_half_device.json and DIR/r03b_half_e2e.json, each with the GPU name and power limit
of the run.

Device-resident runs, for float16 and for bfloat16: a half slab (280 + 20 N(0, 1), 1 % NaN) and its
float32 widening both live in HBM, every slab larger than the 126 MB L2.  Three arms are timed
interleaved with CUDA events around `launches` calls of Regridder.regrid each, after a warm-up:
  float32   regrid of the float32 slab;
  native    regrid of the half slab (the kernels read 2 bytes per point);
  widen     regrid(x.float()), the route before half sources were read natively: the widening
            copy is inside the timed region.
Every native output is compared bit for bit with the float32 output on the widened slab.  For C4 and
float16 a fourth arm, `fallback`, regrids a copy of the half slab that starts 2 bytes into its
allocation: its rows cannot be staged as 2-byte rows, so the library widens them into float32
chunks from the handle's pool and stages those (timed interleaved with `native`, output checked
against the float32 output too); the device memory the pool keeps after it is recorded.  Bytes per
call = B x L x (n_src x source itemsize + n_dst x 8); for the native and widen arms the source is
counted at 2 bytes (the bytes a caller's field occupies).  GB/s over 6499 GB/s (the measured B200
copy peak) is the fraction reported.

End to end: Regridder.regrid of 128 host rows, 10 steps, pinned and pageable, float16 against
float32, next to smm_copy_ceiling of the same pinned float32 bytes.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.packed_throughput import COPY_PEAK_GBS, gpu_identity, same_bits, time_calls   # noqa: E402

CONFIGS = {"C4": 1095, "C2": 3441, "C3": 96, "C2bic": 3441, "C5dis": 64}


def half_slab(shape, dt, seed):
    """280 + 20 N(0, 1) in dt, 1 % NaN, made on the device in float32 pieces of at most 2**28 values."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.empty(shape, dtype=dt, device="cuda")
    flat = x.view(-1)
    step = 1 << 28
    for a in range(0, flat.numel(), step):
        n = min(step, flat.numel() - a)
        v = torch.randn(n, device="cuda", generator=g).mul_(20.0).add_(280.0)
        v[torch.rand(n, device="cuda", generator=g) < 0.01] = float("nan")
        flat[a:a + n] = v.to(dt)
        del v
    return x


def fallback_run(rg, xh, xw, shape, reps, launches):
    """The half slab 2 bytes into its allocation (float32 chunks widened by the library) against
    the aligned half slab: ms per call and the device memory the pool keeps."""
    import torch
    buf = torch.empty(xh.numel() + 8, dtype=xh.dtype, device="cuda")
    xm = buf[1:1 + xh.numel()].view(shape)
    xm.copy_(xh)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    ym = rg.regrid(xm)
    torch.cuda.synchronize()
    ok = same_bits(ym, rg.regrid(xw))
    del ym
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    kept = free0 - torch.cuda.mem_get_info()[0]
    t_mis, t_nat = [], []
    for _ in range(reps):
        t_mis.append(time_calls(lambda: rg.regrid(xm), launches))
        t_nat.append(time_calls(lambda: rg.regrid(xh), launches))
    del xm, buf
    torch.cuda.empty_cache()
    m, n = float(np.median(t_mis)), float(np.median(t_nat))
    print(json.dumps({"fallback_ms": m, "native_ms": n, "bits_identical": ok, "pool_bytes_kept": kept}), flush=True)
    return {"ms": m, "native_ms_same_reps": n, "ms_reps": t_mis, "bits_identical": ok,
            "pool_bytes_kept_after_call": int(kept), "vs_native": n / m}


def device_runs(names, reps, launches):
    import torch
    from smmregrid_b200 import Regridder, synth
    out = []
    for name in names:
        B = CONFIGS[name]
        w = synth.config_weights(name)
        rg = Regridder(weights=w, remap_area_min=0.5, device=0)
        n_src, n_dst = rg.n_src, rg.n_dst
        L = w.n_levels if rg.mask_dim else 1
        shape = (B, L, n_src) if L > 1 else (B, n_src)
        for dt in (torch.float16, torch.bfloat16):
            xh = half_slab(shape, dt, 1)
            xw = xh.float()
            arms = {"float32": lambda: rg.regrid(xw), "native": lambda: rg.regrid(xh),
                    "widen": lambda: rg.regrid(xh.float())}
            yw, yh = arms["float32"](), arms["native"]()          # warm-up (and the output check)
            arms["widen"]()
            torch.cuda.synchronize()
            ok = same_bits(yw, yh)
            del yw, yh
            ms = {k: [] for k in arms}
            for _ in range(reps):                                  # interleaved
                for k, fn in arms.items():
                    ms[k].append(time_calls(fn, launches))
            points = B * L * n_src
            rec = {"config": name, "B": B, "levels": L, "n_src": n_src, "n_dst": n_dst,
                   "source_dtype": str(dt).replace("torch.", ""), "bits_identical": ok}
            for k, t in ms.items():
                m = float(np.median(t))
                sx = 4 if k == "float32" else 2
                by = B * L * (n_src * sx + n_dst * 8)
                rec[k] = {"ms": m, "points_per_s": points / m * 1e3, "gbs": by / m / 1e6,
                          "frac_of_copy_peak": by / m / 1e6 / COPY_PEAK_GBS, "ms_reps": t}
            if name == "C4" and dt == torch.float16:
                rec["fallback"] = fallback_run(rg, xh, xw, shape, reps, launches)
            rec["speedup_vs_float32"] = rec["float32"]["ms"] / rec["native"]["ms"]
            rec["speedup_vs_widen"] = rec["widen"]["ms"] / rec["native"]["ms"]
            print(json.dumps({k: rec[k] for k in ("config", "source_dtype", "bits_identical", "speedup_vs_float32",
                                                  "speedup_vs_widen")}
                             | {f"ms_{k}": rec[k]["ms"] for k in arms}), flush=True)
            out.append(rec)
            del xh, xw, arms
            torch.cuda.empty_cache()
    return out


def e2e_runs(steps, rows):
    import torch
    from smmregrid_b200 import Regridder, _lib, synth
    w = synth.config_weights("C4")
    rg = Regridder(weights=w, remap_area_min=0.5, device=0)
    n_src = rg.n_src
    xh = half_slab((rows, n_src), torch.float16, 2).cpu()
    xf = xh.float()
    lib = _lib.load()
    res = {"config": "C4", "rows_per_step": rows, "steps": steps}
    for pinned in (True, False):
        if pinned:
            hp, fp = xh.pin_memory(), xf.pin_memory()
        else:
            hp, fp = xh.numpy(), xf.numpy()
        for tag, fn in (("float32", lambda: rg.regrid(fp)), ("float16", lambda: rg.regrid(hp))):
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
    yh, yf = np.asarray(rg.regrid(xh.numpy())), np.asarray(rg.regrid(xf.numpy()))
    res["bits_identical"] = bool(np.array_equal(np.isnan(yh), np.isnan(yf)) and
                                 np.array_equal(yh[~np.isnan(yh)].view(np.uint64), yf[~np.isnan(yf)].view(np.uint64)))
    for tag in ("float32", "float16"):
        res[f"pinned_{tag}"]["frac_of_h2d_ceiling"] = res[f"pinned_{tag}"]["h2d_gbs"] / res["h2d_ceiling_gbs"]
    res["points_per_s_ratio_pinned"] = res["pinned_float16"]["points_per_s"] / res["pinned_float32"]["points_per_s"]
    res["points_per_s_ratio_pageable"] = res["pageable_float16"]["points_per_s"] / res["pageable_float32"]["points_per_s"]
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
        sys.exit("half_throughput.py measures on a CUDA device; none is available")
    os.makedirs(args.out, exist_ok=True)
    ident = gpu_identity()
    dev = {"measured_on": ident, "copy_peak_gbs": COPY_PEAK_GBS,
           "runs": device_runs([c for c in args.configs.split(",") if c], args.reps, args.launches)}
    with open(os.path.join(args.out, "r03b_half_device.json"), "w") as f:
        json.dump(dev, f, indent=1)
    if args.no_e2e:
        return
    e2e = {"measured_on": ident, **e2e_runs(args.e2e_steps, args.e2e_rows)}
    with open(os.path.join(args.out, "r03b_half_e2e.json"), "w") as f:
        json.dump(e2e, f, indent=1)


if __name__ == "__main__":
    main()
