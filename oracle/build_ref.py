"""Build the reference's own host entropy coder (MLCodec_extensions_cpp) from the sources where
they lie under /root/reference, into oracle/_ref/ (git-ignored; travels to the GPU box as a built
.so).  TEST INFRASTRUCTURE ONLY: used to pin the oracle and to check that the product's rANS
streams are bit-identical to the reference's.  Reference sources are never copied into this repo.

The reference's own build (src/cpp/setup.py) is a 3-file pybind11 extension; we invoke g++ on
those files directly.

Also emits sourceless byte-code of the reference's Python surface (src/, test_video.py,
test_compress_time.py) into oracle/_ref/py: a build output like the .so, so that the tests can import
the *unmodified* reference models on a machine without the reference tree.  No reference source text
is copied into the repository.
"""
from __future__ import annotations

import glob
import os
import py_compile
import shutil
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
REF_SRC = os.path.join(REF, "src/cpp/py_rans")
OUT_DIR = os.path.join(HERE, "_ref")
PY_OUT = os.path.join(OUT_DIR, "py")


def ref_module_path() -> str:
    suffix = sysconfig.get_config_var("EXT_SUFFIX")
    return os.path.join(OUT_DIR, "MLCodec_extensions_cpp" + suffix)


def shim_module_path() -> str:
    suffix = sysconfig.get_config_var("EXT_SUFFIX")
    return os.path.join(OUT_DIR, "dcvc_ref_rans" + suffix)


def build_ref(force: bool = False) -> str | None:
    """Returns the path of the built module, or None if the reference tree is absent and no
    prebuilt module exists."""
    out = ref_module_path()
    shim = shim_module_path()
    shim_src = os.path.join(HERE, "ref_shim.cpp")
    fresh = os.path.exists(out) and os.path.exists(shim) and os.path.getmtime(shim) >= os.path.getmtime(shim_src)
    if fresh and not force:
        return out
    if os.path.exists(out) and os.path.exists(shim) and not os.path.isdir(REF_SRC):
        return out      # GPU box: no reference tree to rebuild from, the prebuilt files are what there is
    if not os.path.isdir(REF_SRC):
        return None
    import pybind11
    os.makedirs(OUT_DIR, exist_ok=True)
    srcs = [os.path.join(REF_SRC, f) for f in ("bind.cpp", "py_rans.cpp", "rans.cpp")]
    cmd = ["g++", "-O3", "-std=c++17", "-shared", "-fPIC", "-Wall", "-Wextra",
           "-I", pybind11.get_include(), "-I", sysconfig.get_paths()["include"],
           "-I", REF_SRC] + srcs + ["-o", out, "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("reference rANS build failed:\n" + r.stderr)
    # the same reference sources + our extra binding (oracle/ref_shim.cpp) exposing the decoder output
    srcs2 = [os.path.join(HERE, "ref_shim.cpp")] + [os.path.join(REF_SRC, f) for f in ("py_rans.cpp", "rans.cpp")]
    cmd2 = ["g++", "-O3", "-std=c++17", "-shared", "-fPIC",
            "-I", pybind11.get_include(), "-I", sysconfig.get_paths()["include"],
            "-I", REF_SRC] + srcs2 + ["-o", shim, "-lpthread"]
    r = subprocess.run(cmd2, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("reference rANS shim build failed:\n" + r.stderr)
    return out


def build_py_surface() -> str | None:
    """Sourceless byte-code of the reference's Python surface -> oracle/_ref/py.  Returns that directory, or None
    if the reference tree is absent and nothing is prebuilt."""
    if not os.path.isdir(REF):
        return PY_OUT if os.path.isdir(PY_OUT) else None
    files = [os.path.join(REF, "test_video.py"), os.path.join(REF, "test_compress_time.py")]
    files += sorted(glob.glob(os.path.join(REF, "src/**/*.py"), recursive=True))
    for f in files:
        rel = os.path.relpath(f, REF)
        if rel.startswith("src/cpp") or "extensions" in rel and rel.endswith("setup.py"):
            continue
        dst = os.path.join(PY_OUT, rel + "c")
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if not os.path.exists(dst) or os.path.getmtime(dst) < os.path.getmtime(f):
            py_compile.compile(f, cfile=dst, dfile=rel, doraise=True)
    # the reference's test configuration (JSON, data not code) is read by test_video.py at run time
    cfg_src, cfg_dst = os.path.join(REF, "test_cfg"), os.path.join(PY_OUT, "test_cfg")
    if os.path.isdir(cfg_src) and not os.path.isdir(cfg_dst):
        shutil.copytree(cfg_src, cfg_dst)
    return PY_OUT


def py_surface_root() -> str | None:
    """oracle/_ref/py when it holds the reference's models (for sys.path), else None."""
    return PY_OUT if os.path.isdir(os.path.join(PY_OUT, "src", "models")) else None


def import_ref():
    """import MLCodec_extensions_cpp from oracle/_ref (None if unavailable)."""
    p = build_ref()
    if p is None:
        return None
    if OUT_DIR not in sys.path:
        sys.path.insert(0, OUT_DIR)
    import MLCodec_extensions_cpp  # noqa
    return MLCodec_extensions_cpp


def import_ref_shim():
    """import dcvc_ref_rans (reference coder + decoded-symbol getter) from oracle/_ref."""
    p = build_ref()
    if p is None or not os.path.exists(shim_module_path()):
        return None
    if OUT_DIR not in sys.path:
        sys.path.insert(0, OUT_DIR)
    import dcvc_ref_rans  # noqa
    return dcvc_ref_rans


if __name__ == "__main__":
    print(build_ref(force="--force" in sys.argv))
    print(build_py_surface())
