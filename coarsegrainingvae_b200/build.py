"""Build libcgvae_sm100.so in-tree with nvcc for sm_100a (B200).  No other arch, no JIT cache.

    python -m coarsegrainingvae_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcgvae_sm100.so")
SOURCES = ["graph.cu", "geom.cu", "gemm.cu", "gemm_tc.cu", "gemm_stream.cu", "message.cu", "message_tc.cu", "message_geom.cu", "nodewise.cu", "loss.cu", "metrics.cu", "optim.cu", "wgrad.cu", "collate.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "cgvae_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        subprocess.run(cmd, check=True)
        objs.append(obj)
    subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
