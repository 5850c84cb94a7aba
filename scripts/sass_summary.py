#!/usr/bin/env python
"""Per-kernel SASS mnemonic counts of the built library (cuobjdump -sass), for profiles/.

Usage: python scripts/sass_summary.py > profiles/r02_sass_summary.txt
Counts are static instruction counts of each kernel instantiation the benchmarks run; the
mnemonics are the ones B200_PROFILING.md lists as evidence (UBLKCP = 1-D TMA bulk copy,
UTMALDG / UTMASTG = tensor-map TMA, SYNCS = mbarrier operations) plus the per-link instructions
of the consumer loop (LDS, F2F.F64.F32, DFMA / DMUL / DADD) and the uniform-datapath share.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "smmregrid_b200", "build")
KERNELS = [
    ("smm_inst_f32_f64.o", "ordered_kernel<float, double, 64>", "C4 with reference-order sums (thread per row)"),
    ("smm_inst_f32_f64.o", "staged_kernel<float, double, 8, 14, 512, false, false>", "C4 / bench headline"),
    ("smm_inst_f32_f64.o", "staged_kernel<float, double, 2, 14, 512, false, false>", "C2"),
    ("smm_inst_f32_f64.o", "staged_kernel<float, double, 1, 16, 256, true, false>", "C3 (packed rows)"),
    ("smm_inst_f32_f64.o", "staged_kernel<float, double, 1, 16, 256, true, true>", "bicubic-like (packed, reference order)"),
    ("smm_inst_f32_f64.o", "staged_kernel<float, double, 8, 14, 256, false, true>", "C4 forced to reference order"),
    ("smm_inst_f32_f64.o", "gather_kernel<float, double, 1, false>", "C5nn"),
    ("smm_inst_f32_f64.o", "gather_kernel<float, double, 4, false>", "C5dis, few batch rows"),
    ("smm_inst_f32_f64.o", "compact_kernel<float>", "C5dis pass 1"),
    ("smm_inst_f32_f64.o", "compact_apply_kernel<float, double>", "C5dis pass 2"),
    # CF-packed int16 sources decoded to float32 (per link: LDS.U16 + decode instead of LDS.32)
    ("smm_inst_i16f32_f64.o", "staged_kernel<smm::I16F32, double, 8, 14, 512, false, false>", "C4, int16 -> float32"),
    ("smm_inst_i16f32_f64.o", "staged_kernel<smm::I16F32, double, 2, 14, 512, false, false>", "C2, int16 -> float32"),
    ("smm_inst_i16f32_f64.o", "staged_kernel<smm::I16F32, double, 1, 16, 256, true, false>", "C3, int16 -> float32"),
]
MNEMONICS = ["UBLKCP", "UTMALDG", "UTMASTG", "SYNCS", "LDGSTS", "LDS", "F2F", "DFMA", "DMUL", "DADD", "IMAD", "LEA", "SHFL",
             "STG", "LDG", "USETMAXREG", "FMUL", "FADD", "ISETP", "FSEL", "LOP3", "I2F"]


def main():
    print("# static SASS instruction counts per kernel instantiation (cuobjdump -sass, sm_100a)")
    print("# UBLKCP = cp.async.bulk (1-D TMA), UTMALDG/UTMASTG = tensor-map TMA, SYNCS = mbarrier ops,")
    print("# 'U*' = instructions on the uniform datapath (loop control, stage addressing)")
    print(f"{'kernel':<66} " + " ".join(f"{m:>8}" for m in MNEMONICS) + f" {'U*':>6} {'total':>6}  use")
    for obj, name, use in KERNELS:
        out = subprocess.run(["cuobjdump", "-sass", os.path.join(OBJ, obj)], capture_output=True, text=True).stdout
        # split per function
        blocks = re.split(r"\n\s*Function : ", out)
        want = re.sub(r"\s+", "", name)
        hit = None
        for b in blocks[1:]:
            mangled = b.split("\n", 1)[0].strip()
            dem = subprocess.run(["c++filt", mangled], capture_output=True, text=True).stdout.strip()
            if re.sub(r"\s+", "", dem).startswith("voidsmm::" + want + "("):
                hit = b
                break
        if hit is None:
            print(f"{name:<66} (not found)")
            continue
        ops = re.findall(r"^\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", hit, flags=re.M)
        cnt = collections.Counter()
        for op in ops:
            base = op.split(".")[0]
            cnt[base] += 1
        uni = sum(v for k, v in cnt.items() if k.startswith("U") and k not in ("UBLKCP", "UTMALDG", "UTMASTG", "USETMAXREG"))
        print(f"{name:<66} " + " ".join(f"{cnt.get(m, 0):>8}" for m in MNEMONICS) + f" {uni:>6} {len(ops):>6}  {use}")


if __name__ == "__main__":
    main()
