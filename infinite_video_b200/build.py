"""Builds libinfltm.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libinfltm.so")
SOURCES = ["pool.cu", "consolidate.cu", "sticky.cu", "attn.cu", "attn_fast.cu", "attn_tc.cu", "attn_g16.cu", "gemm_simt.cu", "gemm_tcgen05.cu", "ridge.cu", "stm.cu",
           "capi.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC"]


def _stale():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "infltm.h"),
                                                                  os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    objs, procs = [], []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    subprocess.check_call([nvcc, "-shared", "-o", LIB] + objs + FLAGS[:2])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
