"""Build libtbk.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot).

    python -m tbmodels_b200.build [--force] [--verbose]

Each .cu is compiled to an object in parallel, then linked into ``tbmodels_b200/libtbk.so``.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libtbk.so")
SOURCES = ["tbk_api.cu", "hk_gemm.cu", "hk_gemm_i8.cu", "hk_small.cu", "hk_mesh.cu", "expand.cu", "kdotp_construct.cu", "supercell_pack.cu", "eig_tridiag.cu", "eig_tridiag_reg.cu", "eig_tridiag_panel.cu", "eig_ql.cu", "eig_vectors.cu", "band_velocity.cu", "berry_curvature.cu", "eig_band.cu", "microbench.cu"]
HEADERS = ["tbk_kernels.h", "tbk_math.cuh", "jacobi_eig.cuh", "tcgen05.cuh", os.path.join("..", "..", "include", "tbk.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libtbk.so cannot be built (there is no CPU fallback)")
    return exe


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    os.makedirs(BUILD, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(BUILD, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc, *ARCH, *FLAGS, *os.environ.get("TBK_BUILD_DEFINES", "").split(), "-c", s, "-o", o]  # debug -D flags
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        return cmd, r

    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for cmd, r in ex.map(run, jobs):
                if verbose or r.returncode != 0:
                    sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed for {cmd[-3]}")
    if jobs or force or _stale(LIB, objs):
        cmd = [nvcc, *ARCH, "-shared", "-o", LIB, *objs]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
            raise RuntimeError("link of libtbk.so failed")
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
