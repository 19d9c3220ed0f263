"""In-tree build of the CUDA engine (sm_100a only) with nvcc. No torch headers, no JIT cache: the resulting
`lq_mpc_b200/_lib/liblqmpc_b200.so` travels with the repo snapshot to the GPU box."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "_lib")
OBJDIR = os.path.join(PKG, "_lib", "obj")
LIB = os.path.join(LIBDIR, "liblqmpc_b200.so")
SOURCES = ["c_api.cu", "k_eval.cu", "k_clqr.cu", "k_pclqr.cu", "k_bounds.cu", "k_stats.cu", "k_tiled.cu", "k_sampler.cu", "k_dyn.cu", "k_group.cu",
           "k_worst.cu", "k_worst_inf.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]
NVCC_FLAGS += os.environ.get("LQMPC_NVCC_EXTRA", "").split()     # development switches, e.g. -DLQ_K4_PROFILE


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found; the engine has no CPU fallback and cannot be built without it")
    return p


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(os.path.dirname(PKG), "include", "lqmpc_b200.h"))
    return hs


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every translation unit for sm_100a and link the shared library. Returns its path."""
    os.makedirs(OBJDIR, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    stamp = os.path.join(LIBDIR, "build.stamp")
    dig = _digest(srcs + _headers())
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return LIB
    nvcc = nvcc_path()
    hdig = _digest(_headers())

    def compile_one(src):
        obj = os.path.join(OBJDIR, os.path.basename(src) + ".o")
        ostamp = obj + ".stamp"
        d = _digest([src]) + hdig
        if not force and os.path.exists(obj) and os.path.exists(ostamp) and open(ostamp).read() == d:
            return obj, ""
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        with open(ostamp, "w") as f:
            f.write(d)
        with open(obj + ".ptxas.log", "w") as f:
            f.write(r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        results = list(ex.map(compile_one, srcs))
    objs = [o for o, _ in results]
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
