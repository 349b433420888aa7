"""Build libbbk.so (the sm_100a kernels + C ABI) in-tree with nvcc.

    python -m blueberry_b200.build [--force]

Cross-compiles without a GPU.  The library lands in blueberry_b200/lib/libbbk.so (git-ignored, but it
travels to the GPU box with the repository snapshot).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libbbk.so")
IO_LIB = os.path.join(LIBDIR, "libbbkio.so")      # host-side file formats (include/bbk_io.h): g++ + zlib, no CUDA
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--threads", "0"]
# (source, extra flags).  fit_stage.cu: FMA contraction off - its knot search must round like the CPU library.
SOURCES = [
    ("api.cu", []),
    ("hist.cu", []),
    ("fit_stage.cu", ["-fmad=false"]),
    ("pvalue.cu", []),
    ("bh.cu", []),
    ("pack.cu", []),
    ("extract.cu", []),
    ("band.cu", []),
    ("decimate.cu", []),
    ("contactmap.cu", []),
    ("synth.cu", []),
]


def _newest_source_mtime():
    m = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(root):
            m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def build_io(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    src = os.path.join(CSRC, "io_host.cpp")
    deps = [src] + [os.path.join(os.path.dirname(HERE), "include", h) for h in ("bbk_io.h", "bbk.h")]
    if not force and os.path.exists(IO_LIB) and os.path.getmtime(IO_LIB) >= max(os.path.getmtime(f) for f in deps):
        return IO_LIB
    cmd = [os.environ.get("CXX", "g++"), "-O3", "-std=c++17", "-fPIC", "-shared", "-o", IO_LIB, src, "-lz", "-lpthread"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return IO_LIB


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    build_io(force, verbose)
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_source_mtime():
        return LIB
    nvcc = nvcc_path()
    objs = []
    procs = []
    for src, extra in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + ARCH + COMMON + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out.decode()))
    cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
