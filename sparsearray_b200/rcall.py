"""`.Call` into the GPU glue (libsvt_rglue.so) the way R does.

Mirrors SparseArray.Call() (R/thread-control.R:87-92): routines are resolved
only through the table registered by R_init_SparseArray()
(src/R_init_SparseArray.c:149-155), and C_set_max_threads is invoked around
every call.  R itself is not installed here, so SEXPs come from the R-API shim
(rshim/); with real R the same shared object is loaded by useDynLib().
"""
import ctypes
import os
import sys

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from rshim import rshim  # noqa: E402
from . import _native  # noqa: E402

GLUE_PATH = os.path.join(_PKG, "libsvt_rglue.so")


class _DllInfo(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("call_methods", ctypes.c_void_p),
                ("n_call_methods", ctypes.c_int),
                ("use_dynamic_symbols", ctypes.c_int)]


_glue = None
_info = None
_nthread = None


def glue():
    """Load the glue and run its R_init_SparseArray()."""
    global _glue, _info
    if _glue is None:
        if not os.path.exists(GLUE_PATH):
            raise ImportError(
                "%s is missing: run `python -m sparsearray_b200.build`"
                % GLUE_PATH)
        _native.lib()
        rshim.lib()
        G = ctypes.CDLL(GLUE_PATH, mode=ctypes.RTLD_LOCAL)
        info = _DllInfo(b"SparseArray", None, 0, 1)
        G.R_init_SparseArray(ctypes.byref(info))
        _glue, _info = G, info
    return _glue


def registered_routines():
    """{name: arity} of the registered .Call routines."""
    glue()
    L = rshim.lib()
    L.rshim_lookup_call_routine.restype = ctypes.c_void_p
    L.rshim_lookup_call_routine.argtypes = [ctypes.c_void_p, ctypes.c_char_p,
                                            ctypes.POINTER(ctypes.c_int)]
    out = {}
    for name in ("C_get_num_procs", "C_get_max_threads", "C_set_max_threads",
                 "C_colStats_SVT", "C_rowStats_SVT", "C_crossprod2_SVT_mat",
                 "C_crossprod2_mat_SVT", "C_crossprod2_SVT_SVT",
                 "C_crossprod1_SVT", "C_matmul_SVT_mat",
                 "C_summarize_SVT", "C_rowsum_SVT", "C_colsum_SVT",
                 "C_rowMoments_SVT", "C_rowStatsT_SVT",
                 "C_colMedians_SVT", "C_rowMedians_SVT",
                 "C_svtgpu_last_timings", "C_svtgpu_resident_SVT",
                 "C_svtgpu_release", "C_svtgpu_from_CSC", "C_svtgpu_to_CSC",
                 "C_svtgpu_set_cache",
                 "C_svtgpu_cache_stats", "C_svtgpu_Arith_SVT",
                 "C_svtgpu_Math_SVT", "C_svtgpu_Compare_SVT",
                 "C_svtgpu_is_SVT", "C_svtgpu_Ops_SVT_SVT",
                 "C_svtgpu_subset_SVT"):
        n = ctypes.c_int(-1)
        p = L.rshim_lookup_call_routine(ctypes.byref(_info), name.encode(),
                                        ctypes.byref(n))
        if p:
            out[name] = n.value
    return out


def _routine(name, nargs):
    glue()
    L = rshim.lib()
    L.rshim_lookup_call_routine.restype = ctypes.c_void_p
    L.rshim_lookup_call_routine.argtypes = [ctypes.c_void_p, ctypes.c_char_p,
                                            ctypes.POINTER(ctypes.c_int)]
    n = ctypes.c_int(-1)
    p = L.rshim_lookup_call_routine(ctypes.byref(_info), name.encode(),
                                    ctypes.byref(n))
    if not p:
        raise rshim.RError('"%s" not available for .Call() for package '
                           '"SparseArray"' % name)
    if n.value != nargs:
        raise rshim.RError("Incorrect number of arguments (%d), expecting %d "
                           "for '%s'" % (nargs, n.value, name))
    return p


def dot_call(name, args):
    """.Call(name, ...) -> (SEXP, warnings); caller releases the SEXP."""
    return rshim.dot_call(_routine(name, len(args)), list(args))


def get_SparseArray_nthread():
    """R/thread-control.R:46-67: default = min(max threads, procs %/% 3)."""
    global _nthread
    if _nthread is None:
        ans, _ = dot_call("C_get_num_procs", [])
        procs = int(rshim.to_numpy(ans)[0][0])
        rshim.lib().rshim_release_tree(ans)
        ans, _ = dot_call("C_get_max_threads", [])
        mx = int(rshim.to_numpy(ans)[0][0])
        rshim.lib().rshim_release_tree(ans)
        _nthread = max(1, min(mx, procs // 3))
    return _nthread


def set_SparseArray_nthread(nthread=None):
    global _nthread
    prev = get_SparseArray_nthread()
    if nthread is None:
        _nthread = None
        get_SparseArray_nthread()
    else:
        _nthread = max(1, int(nthread))
    return prev


# running totals over every GPU .Call of this process (bench.py reads them)
totals = {"calls": 0, "h2d_bytes": 0.0, "d2h_bytes": 0.0, "flatten_ms": 0.0,
          "h2d_ms": 0.0, "kernel_ms": 0.0, "d2h_ms": 0.0, "launches": 0.0}


def _accumulate():
    t = last_timings()
    totals["calls"] += 1
    for k in ("h2d_bytes", "d2h_bytes", "flatten_ms", "h2d_ms", "kernel_ms",
              "d2h_ms", "launches"):
        totals[k] += t[k]


def SparseArray_Call(name, *args):
    """SparseArray.Call(), R/thread-control.R:87-92."""
    nthread = get_SparseArray_nthread()
    a = rshim.integer([nthread])
    prev, _ = dot_call("C_set_max_threads", [a])
    prev_n = int(rshim.to_numpy(prev)[0][0])
    rshim.lib().rshim_release_tree(prev)
    try:
        res = dot_call(name, args)
        _accumulate()
        return res
    finally:
        b = rshim.integer([prev_n])
        r, _ = dot_call("C_set_max_threads", [b])
        rshim.lib().rshim_release_tree(r)


def last_timings():
    """Phase timings (ms / bytes) of the most recent GPU .Call."""
    ans, _ = dot_call("C_svtgpu_last_timings", [])
    v = rshim.to_numpy(ans)[0]
    rshim.lib().rshim_release_tree(ans)
    keys = ("flatten_ms", "h2d_ms", "kernel_ms", "d2h_ms", "h2d_bytes",
            "d2h_bytes", "launches")
    return dict(zip(keys, (float(x) for x in v)))


def set_gpu_cache(on):
    """options(SparseArray.gpu.cache = on) -> .Call("C_svtgpu_set_cache", on):
    keep the device CSC of the most recent SVT in HBM and reuse it while the
    next calls present the same object (validated by a fingerprint over all
    leaves on every call; see rglue/rglue_common.c for the caveat).  None =
    just drop the cached matrix.  Returns the previous setting."""
    a = rshim.logical([rshim.NA_INTEGER if on is None else int(bool(on))])
    ans, _ = dot_call("C_svtgpu_set_cache", [a])
    prev = bool(rshim.to_numpy(ans)[0][0])
    rshim.lib().rshim_release_tree(ans)
    a.release()
    return prev


def gpu_cache_stats():
    """(hits, misses) of the device cache since the glue was loaded"""
    ans, _ = dot_call("C_svtgpu_cache_stats", [])
    v = rshim.to_numpy(ans)[0]
    rshim.lib().rshim_release_tree(ans)
    return int(v[0]), int(v[1])
