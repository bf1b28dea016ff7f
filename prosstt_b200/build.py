"""In-tree build of the CUDA library (nvcc -> prosstt_b200/libprosstt_b200.so).

sm_100a only; the .so is git-ignored but travels to the GPU box with the snapshot."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libprosstt_b200.so")
SOURCES = ["pst_index.cu", "pst_lineage.cu", "pst_counts.cu", "pst_epilogue.cu", "pst_deflate.cu"]
HOST_SOURCES = ["pst_host.cpp"]          # host side of the device->host path (threads, no CUDA)
HOST_FLAGS = ["-O3", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-pthread", "-Wall", "-Wextra"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xptxas=-v", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(PKG), "include", "prosstt_b200.h"))
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library.  Returns its path."""
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    os.makedirs(os.path.join(PKG, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(PKG, "build", src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + os.environ.get("PST_NVCC_DEFS", "").split() + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed on %s" % src)
        objs.append(obj)
    cxx = os.environ.get("CXX", "g++")
    for src in HOST_SOURCES:
        obj = os.path.join(PKG, "build", src.replace(".cpp", ".o"))
        cmd = [cxx] + HOST_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("%s failed on %s" % (cxx, src))
        objs.append(obj)
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
