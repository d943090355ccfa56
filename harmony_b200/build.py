"""harmony_b200/build.py -- in-tree builds (no JIT cache): the CUDA product library and the CPU oracle.

    libhbls.so          nvcc -gencode arch=compute_100a,code=sm_100a   (product; harmony_b200/lib/)
    hbls_host_test      g++  (C++ host mirror hbls_host.hpp + restated reference tests; links libhbls.so)
    libhbls_oracle.so   gcc  (oracle/: TEST INFRASTRUCTURE, never loaded by the product path)
"""
import os, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "harmony_b200", "csrc")
LIBDIR = os.path.join(ROOT, "harmony_b200", "lib")
LIB = os.path.join(LIBDIR, "libhbls.so")
HOSTTEST = os.path.join(LIBDIR, "hbls_host_test")
ORACLE_LIB = os.path.join(ROOT, "oracle", "libhbls_oracle.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)

def _sources(d, exts):
    out = []
    for base, _, files in os.walk(d):
        out += [os.path.join(base, f) for f in files if f.endswith(exts)]
    return out

def build_cuda(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    srcs = _sources(CSRC, (".cu", ".cuh", ".h", ".hpp")) + [os.path.join(ROOT, "include", "hbls.h")]
    if not force and _newer(LIB, srcs):
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB, os.path.join(CSRC, "hbls.cu")]
    subprocess.check_call(cmd)
    return LIB

def build_host(force=False):
    """C++ host mirror (header-only hbls_host.hpp) + its test driver, linked against libhbls.so."""
    hd = os.path.join(ROOT, "harmony_b200", "host")
    src = os.path.join(hd, "hbls_host_test.cpp")
    srcs = [src, os.path.join(hd, "hbls_host.hpp"), os.path.join(hd, "hbls_consensus.hpp"), os.path.join(hd, "hbls_keyfile.hpp"), os.path.join(ROOT, "include", "hbls.h")]
    if not force and _newer(HOSTTEST, srcs) and os.path.getmtime(HOSTTEST) >= os.path.getmtime(LIB):
        return HOSTTEST
    cmd = ["g++", "-O2", "-std=c++17", "-Wall", "-o", HOSTTEST, src, "-L" + LIBDIR, "-lhbls", "-Wl,-rpath,$ORIGIN", "-pthread", "-ldl", "-lrt"]
    subprocess.check_call(cmd)
    return HOSTTEST

def build_oracle(force=False):
    od = os.path.join(ROOT, "oracle")
    srcs = [os.path.join(od, f) for f in ("hbls_oracle.c", "ho_curve_tmpl.h", "ho_constants.h")]
    if not force and _newer(ORACLE_LIB, srcs):
        return ORACLE_LIB
    cmd = ["gcc", "-O3", "-march=x86-64-v3", "-fPIC", "-shared", "-fvisibility=hidden", "-Wno-misleading-indentation",
           "-pthread", "-o", ORACLE_LIB, srcs[0]]
    subprocess.check_call(cmd)
    return ORACLE_LIB

def build_all(force=False, verbose=False):
    build_cuda(force, verbose)
    build_host(force)
    build_oracle(force)

if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built:", LIB, ORACLE_LIB)
