"""Builds libgraphmarl_b200.so IN-TREE with nvcc for sm_100a (cross-compiles without a GPU).

    python -m graph_marl_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libgraphmarl_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = ["runtime.cu", "routing_env.cu", "simple_env.cu", "netmon.cu", "gemm_dispatch.cu", "linear_simt.cu",
           "gemm_sm100.cu", "dqn.cu", "replay.cu", "replay_sampler.cu", "train.cu", "learner.cu", "eval_metrics.cu", "topology.cu", "host_topology.cpp", "collective.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-x", "cu",
              "--expt-relaxed-constexpr", "-I", INCLUDE]
# e.g. GM_NVCC_EXTRA="-DGM_TC_PROBES=1" builds the timing probes of gemm_sm100.cu (GM_TC_DEBUG / GM_LN_DEBUG)
NVCC_FLAGS += os.environ.get("GM_NVCC_EXTRA", "").split()


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _digest():
    h = hashlib.sha256()
    for root in (CSRC, INCLUDE):
        for f in sorted(os.listdir(root)):
            with open(os.path.join(root, f), "rb") as fh:
                h.update(f.encode()), h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "build.stamp")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJDIR, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    # the CUDA runtime comes from libcudart.so.12 (torch has it loaded already; the rpath covers hosts that link the
    # library without torch), so the library carries no runtime of its own
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "shared",
                                                 "-Xlinker", "-rpath=/usr/local/cuda/lib64", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as fh:
        fh.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
