"""Build libcrl_b200.so (the C-ABI library, include/crl_b200.h) in-tree with nvcc for sm_100a.

    python competitive-rl_b200/build.py [--force] [--verbose]

Every .cu is compiled to an object file (in parallel, only when it or a header changed) and linked into the
shared library.  The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
OUT = os.path.join(HERE, "libcrl_b200.so")
SOURCES = ["crl_abi.cu", "pong_step.cu", "pong_raster.cu", "pong_raster_fast.cu", "crl_car_abi.cu",
           "car_physics.cu", "car_raster.cu", "pong_opponent.cu"]
HEADERS = ["pong_common.cuh", "pong_raster_dev.cuh", "car_common.cuh", "car_contact.cuh", "car_spans.cuh", "crl_host.h",
           os.path.join("..", "..", "include", "crl_b200.h")]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-fmad=false",            # cv2's area resize, the fp64 ball physics and Box2D's fp32 solver are un-fused mul/add
    "-Xcompiler", "-fPIC",
]


def _newer(path, deps):
    if not os.path.exists(path):
        return True
    t = os.path.getmtime(path)
    return any(os.path.getmtime(d) > t for d in deps)


def needs_build():
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return _newer(OUT, deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    common = [os.path.join(CSRC, f) for f in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    for f in SOURCES:
        src, obj = os.path.join(CSRC, f), os.path.join(OBJ, f[:-3] + ".o")
        if force or _newer(obj, [src] + common):
            jobs.append([nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj])

    def run(cmd):
        if verbose:
            print(" ".join(cmd))
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        return cmd, r.returncode, r.stdout

    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        for cmd, rc, out in ex.map(run, jobs):
            if out.strip() and (verbose or rc != 0):
                print(out)
            if rc != 0:
                raise subprocess.CalledProcessError(rc, cmd)
    link = [nvcc, "-shared", "-cudart", "shared", "-gencode", "arch=compute_100a,code=sm_100a"] + \
           [os.path.join(OBJ, f[:-3] + ".o") for f in SOURCES] + ["-o", OUT]
    subprocess.check_call(link)
    return OUT


EXT_SRC = os.path.join(CSRC, "crl_torch.cpp")
EXT_NAME = "_crl_torch"
EXT_OUT = os.path.join(HERE, EXT_NAME + ".so")


def build_torch_ext(force=False, verbose=False):
    """The host layer's torch C++ extension (csrc/crl_torch.cpp): g++ against torch's headers, linked to libcrl_b200.so
    next to it (rpath $ORIGIN).  In-tree like the library, so it travels to the GPU box with the snapshot."""
    build(force=False, verbose=verbose)
    deps = [EXT_SRC, os.path.join(CSRC, "..", "..", "include", "crl_b200.h"), os.path.abspath(__file__)]
    if not force and not _newer(EXT_OUT, deps):
        return EXT_OUT
    import sysconfig
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import torch
        from torch.utils import cpp_extension as ce
    inc = ce.include_paths() + [sysconfig.get_paths()["include"], "/usr/local/cuda/include"]
    libdir = ce.library_paths()[0]
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-deprecated-declarations",
           "-DTORCH_EXTENSION_NAME=" + EXT_NAME, "-DTORCH_API_INCLUDE_EXTENSION_H",
           "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI)]
    for i in inc:
        cmd += ["-isystem", i]
    cmd += [EXT_SRC, "-o", EXT_OUT, "-L" + libdir, "-L" + HERE, "-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch", "-ltorch_python",
            "-l:libcrl_b200.so", "-Wl,-rpath,$ORIGIN", "-Wl,-rpath," + libdir]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return EXT_OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
    print(build_torch_ext(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
