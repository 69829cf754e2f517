"""Build libcngp.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

Usage: python -m corenav_gp_b200.build [--force]
The built .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "_obj")
LIB = os.path.join(HERE, "libcngp.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
if os.environ.get("CNGP_VAR_TUNE"):   # tuning builds: extra gp_var_kernel group shapes (CNGP_VAR_VARIANT at run time)
    COMMON.append("-DCNGP_VAR_TUNE")

# translation unit -> extra flags
UNITS = {
    "cngp_api.cu": [],
    "zupt_lookahead.cu": ["-fmad=false"],   # explicit fma() only: same operation order as the C oracle
}
OPTIONAL_UNITS = {"chol_large.cu": [], "gp_slip.cu": [], "ragged.cu": [], "slip_record.cu": ["-fmad=false"], "ekf_context.cu": []}


def _sources():
    units = dict(UNITS)
    for k, v in OPTIONAL_UNITS.items():
        if os.path.exists(os.path.join(CSRC, k)):
            units[k] = v
    return units


def _newest_dep():
    t = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include"), os.path.join(HERE, "host")):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h", ".hpp", ".cpp")):
                t = max(t, os.path.getmtime(os.path.join(root, f)))
    return t


def build(force: bool = False, verbose: bool = False) -> str:
    units = _sources()
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_dep():
        if not os.path.exists(HOST_LIB) or os.path.getmtime(HOST_LIB) < os.path.getmtime(LIB):
            build_host()
        return LIB
    os.makedirs(OBJ, exist_ok=True)

    def compile_one(item):
        src, extra = item
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC, *ARCH, *COMMON, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    objs = []
    with concurrent.futures.ThreadPoolExecutor(max_workers=4) as ex:
        for src, obj, r in ex.map(compile_one, units.items()):
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError(f"nvcc failed on {src}")
            if verbose:
                sys.stderr.write(r.stderr)
            with open(os.path.join(OBJ, src + ".ptxas.log"), "w") as f:
                f.write(r.stderr)
            objs.append(obj)
    cmd = [NVCC, *ARCH, "-shared", "-o", LIB, *objs, "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    build_host()
    return LIB


HOST_LIB = os.path.join(HERE, "libgp_predictor_b200.so")


def build_host() -> str:
    """The C++ host side above the C ABI: the ROS-free GpPredictor class (include/gp_predictor_b200.hpp)."""
    srcs = [os.path.join(HERE, "host", "gp_predictor.cpp"), os.path.join(HERE, "host", "gp_slip_predict.cpp")]
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", HOST_LIB, *srcs, LIB, "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("host library build failed")
    return HOST_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
