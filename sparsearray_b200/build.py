"""In-tree build of the native pieces (no JIT cache: the .so files travel with
the repository snapshot to the GPU box).

  sparsearray_b200/libsvtgpu.so     CUDA kernels + C ABI (include/svtgpu.h),
                                    nvcc, sm_100a only, static cudart
  rshim/librshim.so                 stand-in for libR (R is not installed)
  sparsearray_b200/libsvt_rglue.so  the R-facing .Call entry points (plain C),
                                    compiled against the shim here and against
                                    real R headers in an R installation
"""
import os
import subprocess
import sys

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
_CSRC = os.path.join(_PKG, "csrc")
_RGLUE = os.path.join(_PKG, "rglue")
_SHIM = os.path.join(_ROOT, "rshim")

LIBSVTGPU = os.path.join(_PKG, "libsvtgpu.so")
LIBRGLUE = os.path.join(_PKG, "libsvt_rglue.so")
LIBRSHIM = os.path.join(_SHIM, "librshim.so")

CUDA_SOURCES = ["svtgpu_matrix.cu", "svtgpu_colstats.cu", "svtgpu_rowstats.cu",
                "svtgpu_crossprod.cu", "svtgpu_transpose.cu",
                "svtgpu_groupsum.cu", "svtgpu_gen.cu", "svtgpu_ewise.cu",
                "svtgpu_medians.cu", "svtgpu_ewise2.cu", "svtgpu_subset.cu"]
RGLUE_SOURCES = ["svt_flatten.c", "rglue_common.c", "rglue_matrixStats.c",
                 "rglue_mult.c", "rglue_summarization.c", "rglue_rowsum.c",
                 "rglue_bridge.c", "rglue_ewise.c", "rglue_subset.c",
                 "rglue_init.c"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
              "-std=c++17", "-Xcompiler", "-fPIC,-fopenmp"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)


def nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def build_rshim(force=False, verbose=False):
    src = os.path.join(_SHIM, "rshim.c")
    deps = [src, os.path.join(_SHIM, "include", "Rinternals.h")]
    if force or _newer(LIBRSHIM, deps):
        _run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-o", LIBRSHIM,
              src, "-lm"], verbose)
    return LIBRSHIM


def build_svtgpu(force=False, verbose=False):
    from concurrent.futures import ThreadPoolExecutor
    headers = [os.path.join(_CSRC, h) for h in
               ("svtgpu_internal.h", "svt_semantics.h", "svt_ptx.cuh")]
    headers.append(os.path.join(_ROOT, "include", "svtgpu.h"))
    objs, jobs = [], []
    for name in CUDA_SOURCES:
        src = os.path.join(_CSRC, name)
        obj = os.path.join(_CSRC, name[:-3] + ".o")
        if force or _newer(obj, [src] + headers):
            jobs.append([nvcc()] + NVCC_FLAGS + ["-c", src, "-o", obj])
        objs.append(obj)
    if jobs:   # one nvcc per translation unit, side by side
        with ThreadPoolExecutor(max_workers=min(len(jobs),
                                                os.cpu_count() or 1)) as ex:
            list(ex.map(lambda cmd: _run(cmd, verbose), jobs))
    if jobs or not os.path.exists(LIBSVTGPU):
        _run([nvcc(), "-shared", "-o", LIBSVTGPU] + objs +
             ["-Xcompiler", "-fopenmp", "-lgomp"], verbose)
    return LIBSVTGPU


def build_rglue(force=False, verbose=False):
    build_rshim(force, verbose)
    srcs = [os.path.join(_RGLUE, s) for s in RGLUE_SOURCES]
    deps = srcs + [os.path.join(_RGLUE, "svt_flatten.h"),
                   os.path.join(_RGLUE, "rglue_common.h"),
                   os.path.join(_CSRC, "svt_semantics.h"),
                   os.path.join(_ROOT, "include", "svtgpu.h"), LIBSVTGPU]
    if force or _newer(LIBRGLUE, deps):
        _run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-fopenmp", "-Wall",
              "-shared", "-I", os.path.join(_SHIM, "include"),
              "-o", LIBRGLUE] + srcs +
             ["-L", _PKG, "-lsvtgpu", "-L", _SHIM, "-lrshim",
              # -Bsymbolic: the registration table must bind to OUR entry
              # points even when the reference build (oracle/_ref), which
              # exports the same names, is loaded in the same process
              "-Wl,-Bsymbolic", "-Wl,-rpath,$ORIGIN:$ORIGIN/../rshim", "-lm"],
             verbose)
    return LIBRGLUE


def build_all(force=False, verbose=False):
    build_svtgpu(force, verbose)
    build_rglue(force, verbose)
    return LIBSVTGPU, LIBRGLUE


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose=True)
