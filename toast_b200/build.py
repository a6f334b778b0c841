"""Build libtoastb200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python -m toast_b200.build [--force]

nvcc cross-compiles without a GPU.  ``-fmad=false`` keeps every a*b+c in the pointing chain
double-rounded like the reference's x86-64 build (bit-exact pixels); the built library is
git-ignored but travels to the GPU box with the repository snapshot.
"""

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("TB_LIB_PATH", os.path.join(HERE, "libtoastb200.so"))
SOURCES = ["tb_runtime.cu", "tb_ops.cu", "tb_solver.cu", "tb_blocked.cu", "tb_peer.cu",
           "tb_sort.cu", "tb_prior.cu"]
HEADERS = ["tb_math.cuh", "tb_device.cuh", "tb_runtime.cuh", "tb_prior.cuh", "tb_obs.cuh", "tb_wcs.cuh",
           "tb_pixelise.cuh",
           "../../include/toast_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in HEADERS]
    if not force and not _stale(LIB, deps):
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for s in srcs:
        o = os.path.join(objdir, os.path.basename(s) + ".o")
        objs.append(o)
        extra = os.environ.get("TB_EXTRA_NVCC_FLAGS", "").split()
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd)))
    for cmd, p in procs:
        if p.wait() != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    cmd = [nvcc, "-shared", "-o", LIB] + objs
    subprocess.check_call(cmd)
    return LIB


def _host_cxx():
    """The system g++ (the compiler nvcc uses as host compiler).  $CXX is deliberately ignored:
    this image sets it to a second GCC whose static libstdc++ breaks C++ exception unwinding
    across the pybind11 boundary."""
    for cand in ("/usr/bin/g++", "g++"):
        if os.path.exists(cand) or cand == "g++":
            return cand


def build_pybind(force=False):
    """Compile the `_libtoast` pybind11 module (host C++ above the C ABI), linked against
    libtoastb200.so in the same directory ($ORIGIN rpath)."""
    import sysconfig

    import pybind11

    ext = sysconfig.get_config_var("EXT_SUFFIX")
    target = os.path.join(HERE, "_libtoast" + ext)
    src = os.path.join(CSRC, "pybind_module.cpp")
    deps = [src, os.path.join(HERE, "..", "include", "toast_b200.h"), LIB]
    if not force and not _stale(target, deps):
        return target
    cmd = [
        _host_cxx(), "-O2", "-std=c++17", "-fPIC", "-shared",
        "-fvisibility=hidden", "-o", target, src,
        "-I" + sysconfig.get_paths()["include"], "-I" + pybind11.get_include(),
        "-L" + HERE, "-ltoastb200", "-Wl,-rpath,$ORIGIN",
    ]
    subprocess.check_call(cmd)
    return target


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_pybind(force="--force" in sys.argv))
