"""In-tree build of ``libsmmregrid_b200.so`` (nvcc, sm_100a only).

The shared library is a plain C-ABI object (``include/smmregrid_b200.h``): no torch, no
pybind.  It is built into ``smmregrid_b200/lib/`` so it travels with the source tree.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
LIB_DIR = os.path.join(_PKG, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsmmregrid_b200.so")
# one translation unit per (x, y) element-type pair of the kernels (x: float32, float64, CF-packed
# 16 bits decoding to either, float16 or bfloat16), compiled in parallel
SOURCES = ["smm_api.cu", "smm_plan.cpp", "smm_plan_cache.cpp", "smm_tuning.cpp",
           "smm_inst_f32_f32.cu", "smm_inst_f32_f64.cu", "smm_inst_f64_f32.cu", "smm_inst_f64_f64.cu",
           "smm_inst_i16f32_f32.cu", "smm_inst_i16f32_f64.cu", "smm_inst_i16f64_f32.cu", "smm_inst_i16f64_f64.cu",
           "smm_inst_f16_f32.cu", "smm_inst_f16_f64.cu", "smm_inst_bf16_f32.cu", "smm_inst_bf16_f64.cu"]
HEADERS = ["smm_common.h", "smm_internal.h", "smm_kernels.cuh", "smm_launch.cuh", "smm_aux_kernels.cuh", "smm_plan.h", "smm_tuning.h",
           os.path.join("..", "..", "include", "smmregrid_b200.h")]
OBJ_DIR = os.path.join(_PKG, "build")

NVCC_FLAGS = [
    "-Xcompiler", "-fPIC", "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: smmregrid_b200 needs the CUDA toolkit to build "
                       "(there is no CPU fallback)")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, variant: str = "", flags=()) -> str:
    """Compile the library if sources are newer than the binary.  Returns its path.
    ``variant`` / ``flags``: an experimental build with extra nvcc flags (``-DSMM_...``) next to
    the default one, as ``lib/libsmmregrid_b200_<variant>.so`` (select it with ``SMM_LIB_PATH``)."""
    lib_path = LIB_PATH if not variant else os.path.join(LIB_DIR, f"libsmmregrid_b200_{variant}.so")
    obj_dir = OBJ_DIR if not variant else OBJ_DIR + "_" + variant
    if not variant and not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = _nvcc()
    extra = (["-Xptxas", "-v"] if verbose else []) + list(flags)
    if os.environ.get("SMM_NVCC_FLAGS"):
        extra += os.environ["SMM_NVCC_FLAGS"].split()

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", "-o", obj, os.path.join(CSRC, src)]
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        return src, obj, proc.returncode, proc.stdout

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    log = "".join(f"--- {src}\n{out}" for src, _, _, out in results if out)
    bad = [src for src, _, rc, _ in results if rc != 0]
    if bad:
        raise RuntimeError(f"nvcc failed on {bad}:\n" + log)
    tmp = lib_path + ".tmp"
    proc = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] +
                          [obj for _, obj, _, _ in results],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        raise RuntimeError("link failed:\n" + proc.stdout)
    os.replace(tmp, lib_path)
    if verbose:
        print(log)
    return lib_path


if __name__ == "__main__":
    print(build(force=True, verbose=True))
