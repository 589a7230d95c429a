"""In-tree build of the CUDA library (nvcc, sm_100a only).

    python -m rayopt_b200.build          # rebuild if sources are newer

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librtx.so")
SOURCES = ["rtx.cu"]
HEADERS = ["rtx_device.cuh", "rtx_psf.cuh", os.path.join("..", "..", "include", "rtx.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
]


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found")
    return exe


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t
               for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    cmd = [nvcc()] + NVCC_FLAGS
    if os.environ.get("RTX_TUNING_SPACE"):      # extra kernel variants for sweeps
        cmd += ["-DRTX_TUNING_SPACE"]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
