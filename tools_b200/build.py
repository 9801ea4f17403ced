"""Build the CUDA shared library in-tree: tools_b200/libqfall_b200.so (sm_100a only)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libqfall_b200.so")
SOURCES = ["api.cu", "gemm_f64.cu", "elementwise.cu", "lattice.cu", "compress.cu", "ring_ntt.cu", "setup.cu", "gemm_i8.cu", "ring_small.cu", "gemm_i8_fused.cu", "encodings.cu", "domain_code.cu", "offline_online.cu"]
HEADERS = ["common.cuh", "domain_code.cuh", "kernels.h", "tc05.cuh", os.path.join("..", "..", "include", "qfall_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--threads", "4",
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for s in SOURCES:
        o = os.path.join(HERE, "build", s.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            print(" ".join(cmd))
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out.decode())
            raise RuntimeError(f"nvcc failed on {s}")
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "shared"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
