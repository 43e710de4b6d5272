"""In-tree build of the CUDA library (sm_100a only).  `python schnorr-sig_b200/build.py`"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(CSRC, "libschnorr_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC",
              "-diag-suppress", "550"]


def sources():
    deps = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    deps += [os.path.join(HERE, "..", "include", f) for f in ("schnorr_b200.h", "cheetah_params.h")]
    return deps


def is_stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(f) > t for f in sources())


def build(force=False, verbose=False):
    if not force and not is_stale():
        return SO
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO, os.path.join(CSRC, "schnorr_b200.cu")]
    subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
