"""Build recipe of the C-ABI library pcl_tracking_b200/lib/libpft.so (nvcc, sm_100a only).

-fmad=false is part of the arithmetic contract (DESIGN.md): every fp32/fp64 add and multiply is
rounded on its own, exactly as the x86-64 default-march build of PCL does it, which is what lets
nearest-neighbour indices be compared bit-for-bit with the CPU oracle.
"""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libpft.so")
SOURCES = ["pft_api.cu", "pft_filters.cu", "pft_cluster.cu", "pft_tracker.cu"]
HEADERS = ["pft_common.cuh", "pft_internal.h", "pft_tracker_kernels.cuh", os.path.join("..", "..", "include", "pft", "pft.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
         "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared"]


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile libpft.so if it is missing or older than its sources.  Returns its path."""
    if os.environ.get("PFT_LIB"):
        return os.environ["PFT_LIB"]  # a tuning build chosen explicitly: never rebuilt behind the caller's back
    if not (force or _stale()):
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH] + SOURCES + ["-ldl"]
    subprocess.check_call(cmd, cwd=CSRC)
    return LIB_PATH


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
