"""Build libdaisyrec_b200.so (hand-written sm_100a CUDA + the C ABI) in-tree with nvcc.

No torch involvement: the library is a plain CUDA shared object (static cudart) exposing
the extern "C" entry points of include/daisyrec_b200.h.  The .so lands in
daisyrec_b200/lib/ (git-ignored, shipped to the GPU box by gpurun).
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
SO = os.path.join(LIBDIR, "libdaisyrec_b200.so")
SOURCES = ["capi.cu", "mf_bpr.cu", "sampler.cu", "rank.cu", "shard.cu", "lightgcn.cu", "neumf.cu", "comm.cu", "metrics.cu", "csr.cu", "randperm.cu", "p2p.cu", "ngcf.cu", "nfm.cu", "vae.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--threads", "4"]


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libdaisyrec_b200.so cannot be built")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "daisyrec_b200.h"))
    objs, procs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc()] + ARCH + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose:
            sys.stderr.write(out)
    if force or procs or _stale(SO, objs):
        cmd = [nvcc()] + ARCH + ["-shared", "-cudart", "static", "-o", SO] + objs + ["-ldl"]
        subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
