"""Build liboem_b200.so (hand-written sm_100a CUDA + C++ host drivers behind the C ABI of
include/oem_b200.h) with nvcc, in-tree under oem_b200/lib/ so that it travels to the GPU box."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "liboem_b200.so")
SOURCES = ["runtime.cu", "gram_syrk.cu", "colstats.cu", "assemble.cu", "path_kernel.cu", "host_common.cu",
           "entries.cu", "entry_logistic.cu", "entry_xval.cu", "entry_xval_logistic.cu", "entry_sparse.cu", "cvscore.cu", "logit_slab.cu", "comm.cu", "ingest.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(HERE, "..", "include", "oem_b200.h"))
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs, procs = [], []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {s} ---\n{out}\n")
        failed = failed or pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if procs or force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
