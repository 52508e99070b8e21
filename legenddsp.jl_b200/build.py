"""In-tree build of liblgdsp_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OUT = os.path.join(_HERE, "liblgdsp_b200.so")
SOURCES = ("lgdsp_api.cu", "lgdsp_icpc.cu", "lgdsp_sipm.cu", "lgdsp_codec.cu", "lgdsp_synth.cu", "lgdsp_host_filters.cpp")
HEADERS = ("lgdsp_device.cuh", "lgdsp_kernels.h", "lgdsp_synth.cuh", "lgdsp_icpc_split.cuh", "lgdsp_sweep_warp.cuh", os.path.join("..", "..", "include", "lgdsp_b200.h"))
NVCC_FLAGS = ["-O3", "-std=c++17", "--threads", "4", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    extra = os.environ.get("LGDSP_NVCC_EXTRA", "").split()   # extra flags of experiment builds, never set for a release build
    cmd = ([nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT] + list(SOURCES))
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building liblgdsp_b200.so")
    if verbose:
        sys.stderr.write(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
