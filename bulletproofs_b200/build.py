"""In-tree builds: the sm_100a CUDA library (product), the C oracle and the host-emulation test library
(both test infrastructure).  nvcc cross-compiles without a GPU; the built .so files are git-ignored but
travel to the GPU box with the gpurun snapshot."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bulletproofs_b200", "csrc")
LIB = os.path.join(ROOT, "bulletproofs_b200", "libbpmsm.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--shared", "-Xcompiler", "-fPIC", "-diag-suppress", "177,550"]


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _run(cmd, cwd=None):
    print("+", " ".join(cmd), flush=True)
    subprocess.run(cmd, cwd=cwd, check=True)


def build_cuda(force=False, verbose=False):
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", f) for f in ("bpmsm.h", "bpmsm_ct.h")]
    if not force and _newer(LIB, srcs):
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    flags = NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else [])
    _run([nvcc] + flags + ["-o", LIB, os.path.join(CSRC, "bpmsm.cu")])
    return LIB


def build_host(force=False):
    """C++ mirror of the reference API (bulletproofs_b200/host), linked against libbpmsm.so"""
    hdir = os.path.join(ROOT, "bulletproofs_b200", "host")
    lib = os.path.join(ROOT, "bulletproofs_b200", "libbulletproofs_host.so")
    srcs = [os.path.join(hdir, f) for f in os.listdir(hdir)] + [os.path.join(CSRC, f) for f in ("sc.cuh", "merlin.cuh", "fe.cuh")] + [LIB]
    if force or not _newer(lib, srcs):
        _run(["g++", "-O2", "-std=c++17", "-pthread", "-shared", "-fPIC", "-DBP_HOST_REQUIRE_CT", "-o", lib, os.path.join(hdir, "bulletproofs.cpp"), os.path.join(hdir, "r1cs.cpp"), os.path.join(hdir, "mpc.cpp"),
              "-L" + os.path.join(ROOT, "bulletproofs_b200"), "-lbpmsm", "-Wl,-rpath,$ORIGIN"])
    return lib


def build_oracle(force=False):
    odir = os.path.join(ROOT, "oracle")
    lib = os.path.join(odir, "liboracle.so")
    srcs = [os.path.join(odir, f) for f in ("bp_oracle.c", "fe51.h", "sc.h", "ge.h", "hashes.h", "r1cs.h", "mpc.h")]
    if force or not _newer(lib, srcs):
        _run(["make", "-B", "-C", odir, "liboracle.so"])
    return lib


def build_emul(force=False):
    edir = os.path.join(ROOT, "tests", "host_emul")
    lib = os.path.join(edir, "libemul.so")
    srcs = [os.path.join(edir, "emul.cpp")] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    if force or not _newer(lib, srcs):
        _run(["g++", "-O2", "-std=c++17", "-pthread", "-shared", "-fPIC", "-o", lib, os.path.join(edir, "emul.cpp")])
    return lib


if __name__ == "__main__":
    build_cuda(force="--force" in sys.argv, verbose="-v" in sys.argv)
    build_host()
    build_oracle()
    build_emul()
