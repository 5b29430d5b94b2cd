"""Build libvitok_b200.so (sm_100a only) in-tree with nvcc.

    python vitok-release_b200/build.py [--force] [--ptxas-v]

No torch headers are involved: the library is a plain C-ABI CUDA shared object
(include/vitok_b200.h) that the Python host layer loads with ctypes.
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "vitok_b200")
LIB = os.path.join(OUT_DIR, "libvitok_b200.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["vtk_api.cu", "vtk_gemm.cu", "vtk_attention.cu", "vtk_elementwise.cu", "vtk_pp.cu", "vtk_train.cu", "vtk_attention_bwd.cu", "vtk_ssim.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr",
]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libvitok_b200.so cannot be built")
    return exe


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, ptxas_v: bool = False) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "vitok_b200.h"))
    headers.append(os.path.abspath(__file__))
    flags = NVCC_FLAGS + (["-Xptxas", "-v"] if ptxas_v else [])

    def compile_one(src: str):
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            cmd = [nvcc()] + flags + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
            if verbose or ptxas_v:
                sys.stderr.write(r.stderr)
        return o

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--ptxas-v", action="store_true")
    a = ap.parse_args()
    print(build(force=a.force, verbose=True, ptxas_v=a.ptxas_v))
