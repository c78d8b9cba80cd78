"""Builds the sm_100a CUDA library of radiorust_b200 in-tree with nvcc.

Outputs (git-ignored, but they travel to the GPU box with gpurun):
  radiorust_b200/lib/libradiorust_b200.so   -- the C ABI of include/radiorust_b200.h
  radiorust_b200/lib/libradiorust_b200.a    -- the same objects as a static archive
                                               (what a Rust build.rs links, INTEGRATION.md)

nvcc cross-compiles without a GPU.  Objects are rebuilt only when a source or
header is newer.  `python -m radiorust_b200.build [-j N] [--force]`.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "lib")
SO = os.path.join(LIB, "libradiorust_b200.so")
AR = os.path.join(LIB, "libradiorust_b200.a")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr",
]

F32_SIZES = [64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384]
F64_SIZES = [64, 128, 256, 512, 1024, 2048, 4096]


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")


def translation_units():
    """(object name, source, extra flags)"""
    tus = [
        ("rr_design.o", "rr_design.cpp", []),
        ("rr_chain.o", "rr_chain.cu", []),
        ("rr_stage_kernels.o", "rr_stage_kernels.cu", []),
        ("rr_chunk_kernels.o", "rr_chunk_kernels.cu", []),
        ("rr_metering.o", "rr_metering.cu", []),
        ("rr_big_os.o", "rr_big_os.cu", []),
        ("rr_long_os.o", "rr_long_os.cu", []),
        ("rr_chain_os_dispatch.o", "rr_chain_os_dispatch.cu", []),
        ("rr_poly.o", "rr_poly.cu", []),
        ("rr_poly2.o", "rr_poly2.cu", []),
        ("rr_front.o", "rr_front.cu", []),
        ("rr_front_wide.o", "rr_front_wide.cu", []),
        ("rr_fused.o", "rr_fused.cu", []),
        ("rr_fourier.o", "rr_fourier.cu", []),
        ("rr_synth.o", "rr_synth.cu", []),
    ]
    for t, tn in (("float", "f32"), ("double", "f64")):
        for k in (256, 512, 1024):
            for g in (8, 10):
                tus.append((f"rr_poly_{tn}_{k}_{g}.o", "rr_poly_inst.cu", [f"-DRR_T={t}", f"-DRR_K={k}", f"-DRR_G={g}"]))
    for n in F32_SIZES:
        tus.append((f"rr_chain_os_f32_{n}.o", "rr_chain_os_inst.cu", ["-DRR_T=float", f"-DRR_N={n}"]))
        tus.append((f"rr_fourier_f32_{n}.o", "rr_fourier_inst.cu", ["-DRR_T=float", f"-DRR_N={n}"]))
    for n in F64_SIZES:
        tus.append((f"rr_chain_os_f64_{n}.o", "rr_chain_os_inst.cu", ["-DRR_T=double", f"-DRR_N={n}"]))
        tus.append((f"rr_fourier_f64_{n}.o", "rr_fourier_inst.cu", ["-DRR_T=double", f"-DRR_N={n}"]))
    return [t for t in tus if os.path.exists(os.path.join(CSRC, t[1]))]


def _newest_header() -> float:
    m = 0.0
    for d in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(d):
            if f.endswith((".h", ".cuh", ".hpp")):
                m = max(m, os.path.getmtime(os.path.join(d, f)))
    return max(m, os.path.getmtime(os.path.abspath(__file__)))


def _compile(nvcc, obj, src, extra, verbose):
    cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", os.path.join(OBJ, obj)]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src} {extra}:\n{r.stdout}\n{r.stderr}")
    return obj, r.stderr


def build(jobs: int | None = None, force: bool = False, verbose: bool = False) -> str:
    nvcc = nvcc_path()
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIB, exist_ok=True)
    hdr = _newest_header()
    todo = []
    tus = translation_units()
    for obj, src, extra in tus:
        o = os.path.join(OBJ, obj)
        stale = force or not os.path.exists(o) or os.path.getmtime(o) < max(hdr, os.path.getmtime(os.path.join(CSRC, src)))
        if stale:
            todo.append((obj, src, extra))
    if todo:
        jobs = jobs or max(1, (os.cpu_count() or 2))
        with cf.ThreadPoolExecutor(max_workers=jobs) as ex:
            futs = [ex.submit(_compile, nvcc, o, s, e, verbose) for o, s, e in todo]
            for f in cf.as_completed(futs):
                obj, log = f.result()
                if verbose and log:
                    sys.stderr.write(f"== {obj}\n{log}\n")
    objs = [os.path.join(OBJ, t[0]) for t in tus]
    newest_obj = max(os.path.getmtime(o) for o in objs)
    if force or todo or not os.path.exists(SO) or os.path.getmtime(SO) < newest_obj:
        r = subprocess.run([nvcc, "-shared", "-o", SO] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
        if os.path.exists(AR):
            os.remove(AR)
        r = subprocess.run(["ar", "rcs", AR] + objs, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"ar failed:\n{r.stdout}\n{r.stderr}")
    return SO


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("-j", type=int, default=None)
    ap.add_argument("--force", action="store_true")
    ap.add_argument("-v", action="store_true")
    a = ap.parse_args()
    print(build(a.j, a.force, a.v))
