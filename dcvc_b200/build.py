"""In-tree build of libdcvc_b200.so (sm_100a only) with nvcc.

The shared library is the C-ABI drop-in boundary (include/dcvc_b200.h).  It is built in-tree so the
`.so` travels with the repository snapshot; nothing is installed into site-packages.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(ROOT, "csrc")
OBJ_DIR = os.path.join(CSRC, "build")
LIB_DIR = os.path.join(ROOT, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libdcvc_b200.so")

SOURCES = [
    "pw_gemm.cu",
    "dcb_tail.cu",
    "elementwise.cu",
    "frame_io.cu",
    "metrics.cu",
    "rate.cu",
    "family_ops.cu",
    "rans_host.cpp",
    "c_api_ops.cu",
    "codec.cu",
    "codec_hts.cu",
    "codec_ld.cu",
    "codec_htl.cu",
]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libdcvc_b200.so cannot be built")


def _stamp(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _all_inputs():
    ins = []
    for name in os.listdir(CSRC):
        if name.endswith((".cu", ".cuh", ".cpp", ".h")):
            ins.append(os.path.join(CSRC, name))
    ins.append(os.path.join(ROOT, "..", "include", "dcvc_b200.h"))
    return ins


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA/C++ source for sm_100a and link libdcvc_b200.so.  Returns its path."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    stamp_file = os.path.join(OBJ_DIR, "stamp.txt")
    stamp = _stamp(_all_inputs())
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp_file):
        with open(stamp_file) as f:
            if f.read().strip() == stamp:
                return LIB_PATH
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + ["-x", "cu", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-lpthread", "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
