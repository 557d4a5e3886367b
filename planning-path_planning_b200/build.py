"""In-tree build of the native libraries (no JIT cache: the .so files travel with the tree).

    libdymu_cuda.so  <- csrc/*.cu            nvcc, sm_100a only, -fmad=false (the reference
                                             arithmetic contains no fused multiply-adds)
    libdymu_b200.so  <- src/*.cpp + capi/    g++; the drop-in DyMuPathPlanner class on top of
                                             the C ABI of include/dymu_cuda.h

Run as ``python planning-path_planning_b200/build.py [--force] [--verbose]``.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
INCLUDE = os.path.join(ROOT, "include")
BUILD = os.path.join(ROOT, "build")
CUDA_SO = os.path.join(HERE, "libdymu_cuda.so")
HOST_SO = os.path.join(HERE, "libdymu_b200.so")

NVCC = os.environ.get("DYMU_NVCC", "/usr/local/cuda/bin/nvcc")
CXX = os.environ.get("DYMU_CXX", "/usr/bin/g++")  # not $CXX: see oracle/Makefile

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false", "-Xcompiler", "-fPIC", "-ccbin", CXX, "-I", INCLUDE,
]
CXX_FLAGS = ["-O2", "-std=c++14", "-fPIC", "-Wall", "-ffp-contract=off", "-I", INCLUDE,
             "-I", os.path.join(HERE, "src"), "-I", os.path.join(HERE, "shim")]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("build step failed: " + " ".join(cmd[:3]) + " ...")
    if verbose and r.stdout:
        print(r.stdout)
    return r.stdout


def cuda_sources():
    d = os.path.join(HERE, "csrc")
    return sorted(os.path.join(d, f) for f in os.listdir(d) if f.endswith(".cu"))


def host_sources():
    d = os.path.join(HERE, "src")
    srcs = sorted(os.path.join(d, f) for f in os.listdir(d) if f.endswith(".cpp"))
    srcs.append(os.path.join(HERE, "capi", "planner_capi.cpp"))
    return srcs


def build_cuda(force=False, verbose=False, ptxas_v=False):
    os.makedirs(BUILD, exist_ok=True)
    headers = [os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc"))
               if f.endswith((".cuh", ".h"))] + [os.path.join(INCLUDE, "dymu_cuda.h")]
    objs = []
    log = ""
    for src in cuda_sources():
        obj = os.path.join(BUILD, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if force or _newer(obj, [src] + headers):
            extra = ["-Xptxas", "-v"] if ptxas_v else []
            if os.environ.get("DYMU_FIM_PROFILE"):
                extra.append("-DDYMU_FIM_PROFILE")
            if os.environ.get("DYMU_LOCAL_PROFILE"):
                extra.append("-DDYMU_LOCAL_PROFILE")
            if os.environ.get("DYMU_PATH_PROFILE"):
                extra.append("-DDYMU_PATH_PROFILE")
            log += _run([NVCC] + NVCC_FLAGS + extra + ["-c", src, "-o", obj], verbose)
    if force or _newer(CUDA_SO, objs):
        _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", CXX,
              "-o", CUDA_SO] + objs + ["-cudart", "shared"], verbose)
    return log


def build_host(force=False, verbose=False):
    srcs = host_sources()
    hdrs = [os.path.join(HERE, "src", f) for f in os.listdir(os.path.join(HERE, "src"))
            if f.endswith((".hpp", ".h"))]
    hdrs += [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]
    if force or _newer(HOST_SO, srcs + hdrs + [CUDA_SO]):
        _run([CXX] + CXX_FLAGS + ["-shared", "-DDYMU_CAPI_B200"] + srcs +
             ["-o", HOST_SO, "-L", HERE, "-ldymu_cuda", "-Wl,-rpath,$ORIGIN"], verbose)


def build_all(force=False, verbose=False, ptxas_v=False):
    log = build_cuda(force, verbose, ptxas_v)
    if os.path.exists(os.path.join(HERE, "src", "DyMu.hpp")):
        build_host(force, verbose)
    return log


if __name__ == "__main__":
    out = build_all(force="--force" in sys.argv, verbose="--verbose" in sys.argv,
                    ptxas_v="--ptxas" in sys.argv)
    if "--ptxas" in sys.argv:
        print(out)
    print("built", CUDA_SO, "and", HOST_SO if os.path.exists(HOST_SO) else "(host lib pending)")
