"""In-tree build of the sm_100a C-ABI library (include/pgi.h) — `python -m pose_graph_initialization_b200.build`.

nvcc cross-compiles without a GPU; the resulting libpgi.so lives next to this file (git-ignored, but it
travels with the gpurun snapshot).  -fmad=false: every FP64 expression on the path is decision-bearing and
must round like the reference's SSE2 host build (CMakeLists.txt:28-34, SURVEY App. A.8/A.9).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpgi.so")
SOURCES = ["pgi_api.cu", "pgb_host.cpp"]  # pgb_host.cpp includes pgb_tracklets.cpp
DEPS = ["pgi_api.cu", "pgi_kernels.cuh", "pgi_math.cuh", "pgi_astar.cuh", "pgi_matcher.cuh", "pgi_guided_batch.cuh", "pgi_guided_nn.h", "pgi_match_scene.cuh", "pgi_nn2.h", "pgi_atan2.h", "pgi_nvtx.h", "pgb_host.cpp", "pgb_tracklets.cpp", os.path.join("..", "..", "include", "pgi.h"),
        os.path.join("..", "..", "include", "pgb.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo", "-fmad=false",
              "-Xcompiler", "-fPIC,-O3,-ffp-contract=off,-pthread", "-shared"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.exists(os.path.join(CSRC, d)) and os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building libpgi.so")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
