"""Build liboverflow_b200.so in-tree with nvcc for sm_100a.

    python -m overflow_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The library links the static CUDA runtime and
resolves cuTensorMapEncodeTiled through cudaGetDriverEntryPoint, so it has no
link-time dependency on libcuda.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "liboverflow_b200.so")
SOURCES = ["runtime.cu", "direction.cu", "direction_generic.cu", "accumulation.cu", "flats.cu", "pits.cu", "synth.cu", "basins.cu", "api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",  # never contract a*b+c: the direction arithmetic must round like the reference
    "-Xcompiler", "-fPIC,-O2,-Wall",
    "-cudart", "static",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; liboverflow_b200 cannot be built")


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "overflow_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    extra = os.environ.get("OFL_NVCC_EXTRA", "").split()  # e.g. -DOFL_DIR_RB=4 for tuning sweeps
    cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-shared", "-o", LIB] + srcs
    env = dict(os.environ)
    env.pop("CC", None)  # the image exports a gcc wrapper that nvcc should not pick up
    env.pop("CXX", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building liboverflow_b200.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
