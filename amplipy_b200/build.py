"""Compile the CUDA extension in-tree for sm_100a (explicit nvcc; no JIT cache involved)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libamplipy_b200.so")
SOURCES = ["amp_abi.cu"]
HEADERS = ["amp_core.cuh", "amp_kernels.cuh", "amp_warp.cuh", "amp_call.cuh", "amp_bgzf.cuh", "amp_ont.cuh", "amp_deflate.cuh", "amp_ivar.cuh", "amp_contig.cuh", "amp_annot.cuh", "amp_exchange.cuh", "amp_dels.cuh", os.path.join("..", "..", "include", "amplipy_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build amplipy_b200's CUDA extension")


def is_stale():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build_extension(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> amplipy_b200/csrc/libamplipy_b200.so"""
    if not force and not is_stale():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    env = dict(os.environ)
    if os.path.isfile("/usr/bin/g++"):
        cmd += ["-ccbin", "/usr/bin/g++"]
    r = subprocess.run(cmd, cwd=CSRC, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building %s" % LIB)
    with open(os.path.join(CSRC, "ptxas_info.txt"), "w") as f:
        f.write(r.stdout)
    return LIB


HOSTIO_LIB = os.path.join(CSRC, "libamplipy_hostio.so")


def build_hostio(force=False):
    """g++ -O2 -fopenmp amp_hostio.cpp -lz -> amplipy_b200/csrc/libamplipy_hostio.so (CPU-only BGZF/BAM codec)."""
    src = os.path.join(CSRC, "amp_hostio.cpp")
    if not force and os.path.isfile(HOSTIO_LIB) and os.path.getmtime(HOSTIO_LIB) >= os.path.getmtime(src):
        return HOSTIO_LIB
    gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
    base = [gxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-o", HOSTIO_LIB, src, "-lz"]
    r = subprocess.run(base[:1] + ["-fopenmp"] + base[1:], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:   # toolchain without libgomp: single-threaded codec
        r = subprocess.run(base, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        print(r.stdout)
        raise RuntimeError("g++ failed building %s" % HOSTIO_LIB)
    return HOSTIO_LIB


if __name__ == "__main__":
    print(build_hostio(force=True))
    print(build_extension(force=True, verbose=True))
