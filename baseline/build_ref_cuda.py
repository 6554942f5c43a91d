"""Build the REFERENCE's own CUDA inference extension (CUTLASS / CuTe path) for sm_100a, from the sources where they lie
under /root/reference, into baseline/_ref/ (git-ignored; the built .so travels to the GPU box with the snapshot).

COMPARATOR ONLY.  Nothing in the product (dcvc_b200/, inference_extensions_cuda/, include/) imports or links this.  It is
what `north_star` names as the target ("decode >= reference CUTLASS build FPS on 1 GPU") and what pins the parity of the
product against the reference's CUDA proxy on the same box: `bench.py` times it beside the product (`"reference_cuda"`),
`tests/test_reference_cuda_gpu.py` compares streams and reconstructions.

What the reference does (src/layers/extensions/inference/setup.py:15-75): a torch CUDAExtension over every .cpp / .cu under
that directory + src/cpp/py_rans/{rans,py_rans}.cpp, `-DCURRENT_DEVICE_SM=100 -O3 --use_fast_math
--extra-device-vectorization -gencode arch=compute_100a,code=sm_100a -DCUTLASS_ENABLE_GDC_FOR_SM100=1`, CUTLASS from
third_party/cutlass (un-vendored in the snapshot: the README pins 4.4.1).  Here: the same flags and file list through a
ninja file we write (setup.py asks torch.cuda for the device capability, which a GPU-less container cannot answer), and
CUTLASS 4.5.0 headers from site-packages/flashinfer/data/cutlass — a 4.4.1 -> 4.5.0 drift, recorded in DESIGN.md.

The module is built under the name `inference_extensions_cuda_ref` (pybind's TORCH_EXTENSION_NAME) so that it can sit in
one process with the product's `inference_extensions_cuda` package; `load_as_plugin()` installs it in sys.modules under the
reference's own name for the processes that drive the unmodified reference models with the reference's kernels.

The reference's Python surface that drives it is the byte-code oracle/build_ref.py emits into oracle/_ref/py.
"""
from __future__ import annotations

import glob
import importlib.util
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
EXT = os.path.join(REF, "src/layers/extensions/inference")
RANS = os.path.join(REF, "src/cpp/py_rans")
OUT = os.path.join(HERE, "_ref")
OBJ = os.path.join(OUT, "obj")
MODNAME = "inference_extensions_cuda_ref"


def module_path() -> str:
    return os.path.join(OUT, MODNAME + sysconfig.get_config_var("EXT_SUFFIX"))


def cutlass_root() -> str | None:
    import site
    for sp in site.getsitepackages():
        for rel in ("flashinfer/data/cutlass", "tilelang/3rdparty/cutlass"):
            p = os.path.join(sp, rel)
            if os.path.exists(os.path.join(p, "include/cutlass/cutlass.h")):
                return p
    return None


def _sources():
    cpp = sorted(glob.glob(os.path.join(EXT, "**/*.cpp"), recursive=True))
    cu = sorted(glob.glob(os.path.join(EXT, "**/*.cu"), recursive=True))
    cpp += [os.path.join(RANS, "rans.cpp"), os.path.join(RANS, "py_rans.cpp")]
    return cpp, cu


def write_ninja(jobs_split: int = 2) -> str:
    import torch
    from torch.utils.cpp_extension import include_paths, library_paths
    cl = cutlass_root()
    if cl is None:
        raise RuntimeError("no CUTLASS header tree found in site-packages")
    os.makedirs(OBJ, exist_ok=True)
    incs = [os.path.join(cl, "include"), os.path.join(cl, "tools/util/include"), RANS, EXT]
    incs += include_paths("cuda") + [sysconfig.get_paths()["include"]]
    inc = " ".join("-I" + i for i in incs)
    common = (f"-DTORCH_EXTENSION_NAME={MODNAME} -DTORCH_API_INCLUDE_EXTENSION_H "
              f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)} -std=c++17")
    cxx = f"{common} -O3 -Wno-deprecated-declarations -fPIC {inc}"
    nvcc = (f"{common} -DCURRENT_DEVICE_SM=100 -O3 --use_fast_math --extra-device-vectorization "
            f"-gencode arch=compute_100a,code=sm_100a -Wno-deprecated-declarations --split-compile={jobs_split} "
            f"-DCUTLASS_ENABLE_GDC_FOR_SM100=1 -D__CUDA_NO_HALF_OPERATORS__ -D__CUDA_NO_HALF_CONVERSIONS__ "
            f"-D__CUDA_NO_BFLOAT16_CONVERSIONS__ -D__CUDA_NO_HALF2_OPERATORS__ --expt-relaxed-constexpr "
            f"--compiler-options -fPIC {inc}")
    libdirs = library_paths("cuda")
    ld = (" ".join("-L" + d for d in libdirs) + " " + " ".join("-Wl,-rpath," + d for d in libdirs) +
          " -lc10 -lc10_cuda -ltorch_cpu -ltorch_cuda -ltorch -ltorch_python -lcudart -lcuda -lpthread")
    cpp, cu = _sources()
    lines = ["ninja_required_version = 1.3",
             f"cxxflags = {cxx}", f"nvccflags = {nvcc}", f"ldflags = {ld}", "",
             "rule cxx", "  command = g++ -MMD -MF $out.d $cxxflags -c $in -o $out", "  depfile = $out.d", "  deps = gcc", "",
             "rule nvcc", "  command = /usr/local/cuda/bin/nvcc $nvccflags -c $in -o $out", "",
             "rule link", "  command = g++ -shared $in $ldflags -o $out", ""]
    objs = []
    for s in cpp:
        o = os.path.join(OBJ, os.path.relpath(s, REF).replace("/", "_") + ".o")
        lines.append(f"build {o}: cxx {s}")
        objs.append(o)
    for s in cu:
        o = os.path.join(OBJ, os.path.relpath(s, REF).replace("/", "_") + ".o")
        lines.append(f"build {o}: nvcc {s}")
        objs.append(o)
    lines.append(f"build {module_path()}: link {' '.join(objs)}")
    lines.append(f"default {module_path()}")
    path = os.path.join(OBJ, "build.ninja")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    return path


def build_ref_cuda(force: bool = False, jobs: int | None = None) -> str | None:
    """Returns the path of the built module; None if the reference tree is absent and nothing is prebuilt."""
    out = module_path()
    if os.path.exists(out) and not force:
        return out
    if not os.path.isdir(EXT):
        return None
    nj = write_ninja()
    jobs = jobs or max(1, min(6, (os.cpu_count() or 4) - 2))
    r = subprocess.run(["ninja", "-f", nj, "-j", str(jobs)], cwd=OBJ)
    if r.returncode != 0:
        raise RuntimeError("reference CUDA extension build failed (see ninja output)")
    return out


def load(as_plugin: bool = False):
    """import the reference extension from baseline/_ref; with as_plugin=True also register it as
    `inference_extensions_cuda` (the name the reference's models import) for THIS process."""
    p = module_path()
    if not os.path.exists(p):
        return None
    import torch  # noqa: F401  (libtorch must be loaded first)
    spec = importlib.util.spec_from_file_location(MODNAME, p)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.modules[MODNAME] = mod
    if as_plugin:
        sys.modules["inference_extensions_cuda"] = mod
    return mod


if __name__ == "__main__":
    print("[baseline] reference CUDA extension:", build_ref_cuda(force="--force" in sys.argv))
