"""Build libantiz_b200.so (hand-written sm_100a kernels + C ABI) and the `uncomp` host program, in-tree."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libantiz_b200.so")
UNCOMP = os.path.join(HERE, "uncomp")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CU = ["api.cu", "scan.cu", "inflate.cu", "chains.cu", "deflate.cu", "png.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-O2,-Wall"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "antiz_b200.h"), __file__]
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    if force or _newer(LIB, deps):
        procs = []
        for f in CU:
            o = os.path.join(HERE, "build", f.replace(".cu", ".o"))
            objs.append(o)
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, f), "-o", o]
            procs.append((cmd, subprocess.Popen(cmd)))
        for cmd, p in procs:
            if p.wait() != 0:
                raise RuntimeError("nvcc failed: " + " ".join(cmd))
        subprocess.check_call([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    host = os.path.join(HERE, "host", "uncomp.cpp")
    if os.path.exists(host) and (force or _newer(UNCOMP, [host, LIB] + [os.path.join(HERE, "host", f) for f in os.listdir(os.path.join(HERE, "host"))])):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(HERE, "host"),
                               host, "-o", UNCOMP, "-L", HERE, "-lantiz_b200", "-Wl,-rpath,$ORIGIN", "-lpthread"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
