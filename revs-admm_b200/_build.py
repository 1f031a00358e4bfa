"""Build the C-ABI shared library (hand-written CUDA for sm_100a) in-tree.

    python revs-admm_b200/_build.py        ->  revs-admm_b200/librevs_admm.so

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the tree.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librevs_admm.so")
SOURCES = ["contract_f64.cu", "home_solve.cu", "dual_update.cu", "utility_qp.cu", "utility_qp_warp.cu", "tree_newton.cu",
           "feeder_build.cu", "network_check.cu", "repair.cu", "central.cu", "certify.cu", "hosting.cu", "screen_bf16.cu", "screen_tc5.cu",
           "revs_capi.cu"]
HEADERS = ["common.cuh", "kernels.cuh", os.path.join("..", "..", "include", "revs_admm.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--threads", "0",
              "-shared", "-Xcompiler", "-fPIC"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every CUDA source of the package for sm_100a.  Returns the .so path."""
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
        ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
