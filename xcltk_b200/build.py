"""In-tree build of libxcltk_b200.so (host decoder + sm_100a kernels + C-ABI).

nvcc cross-compiles for sm_100a without a GPU; the .so stays inside the package
directory so that it travels with the repo snapshot and is the library the tests,
smoke() and bench.py load.
"""

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.environ.get("XG_LIBDIR") or os.path.join(HERE, "_lib")    # XG_LIBDIR: side builds for debugging
LIB = os.path.join(LIBDIR, "libxcltk_b200.so")

CU = ["ctx.cu", "basefc.cu", "baf.cu", "discover.cu", "synth.cu", "gpu_decode.cu", "phase.cu"]
CPP = ["decode.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC,-O3,-Wall", "-Xptxas", "-v"]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _newer(src_list, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in src_list)


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(os.path.dirname(HERE), "include", "xcltk_b200.h"), __file__]
    if not force and not _newer(deps, LIB):
        return LIB
    nvcc = _nvcc()
    objs = []
    log = []
    for f in CU:
        src = os.path.join(CSRC, f)
        if not os.path.exists(src):
            continue
        obj = os.path.join(LIBDIR, f + ".o")
        cmd = [nvcc] + NVCC_FLAGS + os.environ.get("XG_NVCC_EXTRA", "").split() + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + log[-1])
        objs.append(obj)
    for f in CPP:
        src = os.path.join(CSRC, f)
        obj = os.path.join(LIBDIR, f + ".o")
        cmd = ["g++", "-O3", "-std=c++17", "-fPIC", "-Wall", "-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("g++ failed:\n" + log[-1])
        objs.append(obj)
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-lz", "-lpthread", "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + log[-1])
    with open(os.path.join(LIBDIR, "build.log"), "w") as fp:
        fp.write("\n".join(log))
    if verbose:
        sys.stderr.write("\n".join(log) + "\n")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
