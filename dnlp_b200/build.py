"""Build the CUDA C-ABI library in-tree (nvcc, sm_100a)."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
LIB = os.path.join(PKG, "libdnlp_b200.so")
SOURCES = [os.path.join(PKG, "csrc", "dnlp_cabi.cu"), os.path.join(PKG, "csrc", "dnlp_batch.cu"),
           os.path.join(PKG, "csrc", "dnlp_shard.cu")]
HEADERS = [os.path.join(PKG, "csrc", "dnlp_kernels.cuh"), os.path.join(PKG, "csrc", "dnlp_engine.h"), os.path.join(PKG, "csrc", "dnlp_batch_kernels.cuh"),
           os.path.join(PKG, "csrc", "dnlp_batch_kkt.cuh"),
           os.path.join(PKG, "csrc", "dnlp_batch_qn.cuh"), os.path.join(ROOT, "include", "dnlp_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC,-fopenmp", "-Xptxas", "-v", "-lgomp", "-ldl"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not is_stale():
        return LIB
    cmd = [nvcc_path()] + NVCC_FLAGS + ["-o", LIB] + SOURCES
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building %s" % LIB)
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
