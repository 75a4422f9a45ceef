"""Build the C-ABI shared library in-tree (nvcc cross-compiles sm_100a without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libptq4vit_b200.so")
SOURCES = ["runtime.cu", "sweep_tc.cu", "sweep_simt.cu", "prep.cu", "gram.cu", "gram_gemm.cu", "linear_api.cu", "matmul_api.cu",
           "conv_api.cu", "export.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "ptq4vit_b200.h"))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        if not os.path.exists(s):
            continue
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + os.environ.get("P4V_NVCC_EXTRA", "").split() + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    if force or procs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
