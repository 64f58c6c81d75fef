"""Builds libvsom_b200.so (the C-ABI library of include/vsom_b200.h) in-tree with nvcc for sm_100a only."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIB_DIR, "libvsom_b200.so")
HOST_LIB = os.path.join(LIB_DIR, "libvsom_host.so")
API_DRIVER = os.path.join(REPO, "tests", "cpp", "api_driver_b200")
MNIST_TEST = os.path.join(REPO, "tests", "cpp", "mnist_loader_test")
TOPO_DRIVER = os.path.join(REPO, "tests", "cpp", "topo_driver")
LININIT_DRIVER = os.path.join(REPO, "tests", "cpp", "lininit_driver")
CLUSTER_DRIVER = os.path.join(REPO, "tests", "cpp", "cluster_driver")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # parity: the reference CPU build has no FMA; never let nvcc contract a*b+c (see csrc/common.cuh)
    "-fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fvisibility=hidden",
    "-Xptxas", "-v",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def up_to_date() -> bool:
    outputs = (LIB, HOST_LIB, API_DRIVER, MNIST_TEST, TOPO_DRIVER, LININIT_DRIVER, CLUSTER_DRIVER)
    if not all(os.path.exists(o) for o in outputs):
        return False
    t = min(os.path.getmtime(o) for o in outputs)
    deps = sources() + glob.glob(os.path.join(REPO, "tests", "cpp", "*.cpp")) + glob.glob(os.path.join(REPO, "include", "compat", "Eigen", "*")) + glob.glob(os.path.join(PKG, "host", "*.cpp")) + glob.glob(os.path.join(REPO, "include", "*.hpp")) + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(REPO, "include", "*.h")) + [os.path.abspath(__file__)]
    return all(os.path.getmtime(d) <= t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into lib/libvsom_b200.so.  Cross-compiles without a GPU."""
    if not force and up_to_date():
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    objs = []
    procs = []
    for src in sources():
        obj = os.path.join(LIB_DIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc_path(), *NVCC_FLAGS, "-I", os.path.join(REPO, "include"), "-I", CSRC, "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {os.path.basename(src)}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    # link the shared libstdc++ by name: this image's g++ would otherwise embed a private static copy
    # (its libstdc++.so symlink dangles), which clashes with the one already loaded into Python.
    stdcxx = ["-Xlinker", "-l:libstdc++.so.6"] if os.path.exists("/usr/lib/x86_64-linux-gnu/libstdc++.so.6") else []
    cmd = [nvcc_path(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", *stdcxx]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if out.returncode != 0:
        raise RuntimeError(f"link failed:\n{out.stdout}")
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    build_host()
    return LIB




def build_host() -> str:
    """The drop-in C++ classes (include/SOM.hpp, ...) on top of the C-ABI, and the API driver of tests/cpp."""
    cxx = shutil.which("g++") or "g++"
    eigen = "/usr/include/eigen3" if os.path.exists("/usr/include/eigen3/Eigen/Dense") else os.path.join(REPO, "include", "compat")
    flags = ["-std=c++20", "-O2", "-fPIC", "-ffp-contract=off", "-msse2", "-I", os.path.join(REPO, "include"), "-I", eigen]
    stdcxx = ["-nostdlib++", "-l:libstdc++.so.6"] if os.path.exists("/usr/lib/x86_64-linux-gnu/libstdc++.so.6") else []
    srcs = sorted(glob.glob(os.path.join(PKG, "host", "*.cpp")))
    cmd = [cxx, *flags, "-shared", "-o", HOST_LIB, *srcs, "-L", LIB_DIR, "-lvsom_b200", "-Wl,-rpath,$ORIGIN", *stdcxx]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if out.returncode != 0:
        raise RuntimeError(f"host library failed to build:\n{out.stdout}")
    for src, exe, defs in ((os.path.join(REPO, "tests", "cpp", "api_driver.cpp"), API_DRIVER, ["-DVSOM_B200_API"]),
                           (os.path.join(REPO, "tests", "cpp", "mnist_loader_test.cpp"), MNIST_TEST, []),
                           (os.path.join(REPO, "tests", "cpp", "topo_driver.cpp"), TOPO_DRIVER, []),
                           (os.path.join(REPO, "tests", "cpp", "lininit_driver.cpp"), LININIT_DRIVER, []),
                           (os.path.join(REPO, "tests", "cpp", "cluster_driver.cpp"), CLUSTER_DRIVER, [])):
        if os.path.exists(src):
            cmd = [cxx, *flags, *defs, src, "-o", exe, "-L", LIB_DIR, "-lvsom_host", "-lvsom_b200", f"-Wl,-rpath,{LIB_DIR}", *stdcxx]
            out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            if out.returncode != 0:
                raise RuntimeError(f"{os.path.basename(src)} failed to build:\n{out.stdout}")
    return HOST_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
