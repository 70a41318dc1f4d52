"""Builds libusflow_b200.so (sm_100a) in-tree with nvcc.  No torch headers are involved: the library is
plain CUDA C++ behind the C ABI of include/usflow_b200.h."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libusflow_b200.so")
SOURCES = ["usf_api.cu", "usf_simt.cu", "usf_tc.cu", "usf_trsm.cu", "usf_small.cu", "usf_grad.cu", "usf_host.cpp"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _newer(a, b):
    return not os.path.exists(b) or os.path.getmtime(a) > os.path.getmtime(b)


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(os.path.dirname(HERE), "include", "usflow_b200.h")]
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIBDIR, os.path.splitext(src)[0] + ".o")
        objs.append(o)
        if force or any(_newer(d, o) for d in deps):
            jobs.append([NVCC, *FLAGS, "-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        return cmd, r

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        for cmd, r in ex.map(run, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for " + cmd[-3])
            with open(cmd[-1].replace(".o", ".ptxas.log"), "w") as f:
                f.write(r.stderr)
    if force or jobs or not os.path.exists(LIB):
        cmd = [NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-pthread"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
