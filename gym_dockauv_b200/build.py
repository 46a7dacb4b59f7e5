"""Builds libdockauv_b200.so (the C-ABI library of include/dockauv.h) in-tree with nvcc for sm_100a.

    python -m gym_dockauv_b200.build [--force]

The three translation units (C API, FP64 kernels, FP32 kernels) are compiled in parallel and linked into
gym_dockauv_b200/_lib/libdockauv_b200.so (git-ignored; the directory is created on the first build).
"""
import os
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.environ.get("DOCKAUV_LIB_OUT") or os.path.join(LIB_DIR, "libdockauv_b200.so")   # override: tuning builds
UNITS = ["dockauv_capi.cu", "dockauv_kernels_f64.cu", "dockauv_kernels_f32.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")
    return exe


def _sources():
    out = [os.path.join(HERE, "..", "include", "dockauv.h")]
    for f in os.listdir(CSRC):
        if f.endswith((".cu", ".cuh", ".h", ".inl")):
            out.append(os.path.join(CSRC, f))
    return out


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in _sources())


def build_library(force=False, verbose=False):
    if not force and not is_stale():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
    env = dict(os.environ)
    # the image's $CC/$CXX point at a gcc without libgomp; nvcc should use the system g++
    host_cxx = shutil.which("g++") or "g++"

    # objects go to a private temporary directory: none land in the tree, and builds by different users or of
    # different library paths never share one
    with tempfile.TemporaryDirectory(prefix="dockauv_b200_obj_") as obj_dir:
        def compile_unit(unit):
            extra = os.environ.get("DOCKAUV_NVCC_EXTRA", "").split()
            obj = os.path.join(obj_dir, unit.replace(".cu", ".o"))
            cmd = [nvcc, "-ccbin", host_cxx, *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, unit), "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            r = subprocess.run(cmd, capture_output=True, text=True, env=env)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {unit}:\n{r.stdout}\n{r.stderr}")
            return obj, r.stderr

        with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
            results = list(ex.map(compile_unit, UNITS))
        objs = [o for o, _ in results]
        tmp = LIB_PATH + ".tmp"
        link = [nvcc, "-ccbin", host_cxx, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp, *objs,
                "-cudart", "shared"]
        r = subprocess.run(link, capture_output=True, text=True, env=env)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB_PATH)
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    return LIB_PATH


if __name__ == "__main__":
    path = build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
