"""Build recipe for the in-tree CUDA library (librbf_b200.so).  nvcc cross-compiles for
sm_100a without a GPU; the .so travels to the GPU box with the repo snapshot."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "librbf_b200.so")
SOURCES = ["rbf_kernels.cu", "rbf_api.cu"]
HEADERS = ["rbf_hash.cuh", "rbf_kernels.cuh", "rbf_k1_threshold.cuh", "rbf_k1_binarize.cuh", "rbf_k2_insert.cuh", "rbf_k3_query.cuh", "rbf_k3b_witness.cuh",
           "rbf_aux_kernels.cuh", os.path.join("..", "..", "include", "rbf_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall",
    "--fmad=true",           # device integer code only; host float maths is guarded by -ffp-contract=off
    "-shared", "-cudart", "shared",
]


def needs_build() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return SO
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", SO] + [os.path.join(CSRC, f) for f in SOURCES] + ["-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building %s" % SO)
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
