"""In-tree build of libb200reg.so (hand-written sm_100a CUDA behind the C ABI of include/b200reg.h)."""
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(PKG, "csrc")
REPO = os.path.dirname(PKG)
SOURCES = ["api.cu", "index_build.cu", "gicp.cu", "quatro.cu", "assemble.cu", "batch.cu", "map.cu"]
EXTRA = {"quatro.cu": ["-fmad=false"],    # fixed fp32 operation order for the FPFH / matcher arithmetic
         "assemble.cu": ["-fmad=false"],  # transformPcd / VoxelGrid / candidate distances as the (FMA-free) reference computes them
         "map.cu": ["-fmad=false"]}       # the same transformPcd / VoxelGrid over the whole keyframe store
HEADERS = ["internal.cuh", "voxel.cuh", "knn.cuh", "smallmath.cuh", "fpfh_basis.cuh", os.path.join(REPO, "include", "b200reg.h")]
LIB = os.path.join(CSRC, "libb200reg.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
         "-ccbin", "/usr/bin/g++"]


def _mtime(p):
    return os.path.getmtime(p) if os.path.exists(p) else 0.0


def build_native(force=False, verbose=False):
    """Compile every .cu of the package for sm_100a and link libb200reg.so.  Returns the path."""
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    if not force and os.path.exists(LIB) and all(_mtime(d) <= _mtime(LIB) for d in deps):
        return LIB
    if not os.path.exists(NVCC):
        raise RuntimeError("nvcc not found at %s and no prebuilt %s" % (NVCC, LIB))

    def cc(src):
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + EXTRA.get(src, []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr))
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(len(SOURCES)) as ex:
        objs = list(ex.map(cc, SOURCES))
    # libdl for the run-time NCCL binding (b200reg_comm_*), pthread for the batch driver's worker threads
    r = subprocess.run([NVCC, "-shared", "-o", LIB, "-ccbin", "/usr/bin/g++"] + objs + ["-ldl", "-lpthread"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build_native(force=True, verbose=True))
