"""ctypes binding of the C ABI in include/svtgpu.h (libsvtgpu.so).

There is no CPU fallback: a missing library raises at import of this module's
`lib()`, a missing device raises SvtGpuError(NO_DEVICE) from the first call.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libsvtgpu.so")

OK, ERR_NO_DEVICE, ERR_CUDA, ERR_ARG, ERR_UNSUPPORTED, ERR_NOMEM = range(6)
LGL, INT, DOUBLE = 10, 13, 14
HAS_OFFS, HAS_VALS = 1, 2

OPCODES = {"anyNA": 1, "countNAs": 2, "any": 3, "all": 4, "min": 5, "max": 6,
           "range": 7, "sum": 8, "prod": 9, "mean": 10, "centered_X2_sum": 11,
           "sum_X_X2": 12, "var1": 13, "var2": 14, "sd1": 15, "sd2": 16}
RTYPE = {"logical": LGL, "integer": INT, "double": DOUBLE}


class SvtGpuError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("svtgpu status %d: %s" % (status, message))
        self.status = status
        self.message = message


class Timings(ctypes.Structure):
    _fields_ = [("h2d_ms", ctypes.c_double), ("kernel_ms", ctypes.c_double),
                ("d2h_ms", ctypes.c_double), ("h2d_bytes", ctypes.c_double),
                ("d2h_bytes", ctypes.c_double), ("launches", ctypes.c_int)]


_c = ctypes
_P = _c.c_void_p
_I64 = _c.c_int64
_INT = _c.c_int
_DBL = _c.c_double

# name -> (restype, argtypes); every symbol include/svtgpu.h declares
SIGNATURES = {
    "svtgpu_last_error": (_c.c_char_p, []),
    "svtgpu_device_count": (_INT, [_c.POINTER(_INT)]),
    "svtgpu_set_device": (_INT, [_INT]),
    "svtgpu_get_device": (_INT, [_c.POINTER(_INT)]),
    "svtgpu_device_info": (_INT, [_c.c_char_p, _INT, _c.POINTER(_INT),
                                  _c.POINTER(_I64)]),
    "svtgpu_release_cached_memory": (_INT, []),
    "svtgpu_launch_count": (_I64, []),
    "svtgpu_matrix_create": (_INT, [_c.POINTER(_P), _I64, _I64, _I64, _INT,
                                    _INT]),
    "svtgpu_matrix_wrap_device": (_INT, [_c.POINTER(_P), _I64, _I64, _I64,
                                         _INT, _P, _P, _P]),
    "svtgpu_matrix_free": (_INT, [_P]),
    "svtgpu_matrix_set_leaf_ptr": (_INT, [_P, _P]),
    "svtgpu_matrix_stage_capacity": (_INT, [_P, _c.POINTER(_I64)]),
    "svtgpu_matrix_stage": (_INT, [_P, _I64, _c.POINTER(_P),
                                   _c.POINTER(_P)]),
    "svtgpu_matrix_commit": (_INT, [_P, _I64, _I64]),
    "svtgpu_matrix_commit_packed": (_INT, [_P, _I64, _I64, _INT, _INT]),
    "svtgpu_matrix_finish_upload": (_INT, [_P]),
    "svtgpu_matrix_upload": (_INT, [_P, _P, _P, _P]),
    "svtgpu_matrix_fold_rows": (_INT, [_P, _I64]),
    "svtgpu_matrix_set_leaf_base": (_INT, [_P, _I64]),
    "svtgpu_matrix_download": (_INT, [_P, _P, _P, _P]),
    "svtgpu_matrix_transposed": (_INT, [_P, _c.POINTER(_P)]),
    "svtgpu_matrix_info": (_INT, [_P, _c.POINTER(_I64), _c.POINTER(_I64),
                                  _c.POINTER(_I64), _c.POINTER(_INT),
                                  _c.POINTER(_INT)]),
    "svtgpu_matrix_timings": (_INT, [_P, _c.POINTER(Timings)]),
    "svtgpu_matrix_compact_bytes": (_INT, [_P, _c.POINTER(_I64)]),
    "svtgpu_colstats": (_INT, [_P, _INT, _INT, _DBL, _I64, _P,
                               _c.POINTER(_INT)]),
    "svtgpu_colstats_dev": (_INT, [_P, _INT, _INT, _DBL, _I64, _P, _P, _P]),
    "svtgpu_colstats_out_is_int": (_INT, [_INT, _INT]),
    "svtgpu_rowstats": (_INT, [_P, _INT, _INT, _P, _P, _c.POINTER(_INT)]),
    "svtgpu_rowstats_via_transpose": (_INT, [_P, _INT, _INT, _DBL, _P,
                                             _c.POINTER(_INT)]),
    "svtgpu_rowsum": (_INT, [_P, _P, _INT, _INT, _P, _c.POINTER(_INT)]),
    "svtgpu_colsum": (_INT, [_P, _P, _INT, _INT, _P, _c.POINTER(_INT)]),
    "svtgpu_colmedians": (_INT, [_P, _INT, _P]),
    "svtgpu_colmedians_dev": (_INT, [_P, _INT, _P, _P]),
    "svtgpu_rowmedians": (_INT, [_P, _INT, _P]),
    "svtgpu_colmedians_selected": (_INT, [_P, _c.POINTER(_I64),
                                          _c.POINTER(_I64)]),
    "svtgpu_summarize_supported": (_INT, [_INT, _INT]),
    "svtgpu_summarize": (_INT, [_P, _INT, _INT, _DBL, _c.POINTER(_DBL),
                                _c.POINTER(_INT)]),
    "svtgpu_rowstats_state_layout": (_INT, [_INT, _INT, _c.POINTER(_INT),
                                            _c.POINTER(_INT)]),
    "svtgpu_rowstats_accumulate_dev": (_INT, [_P, _INT, _INT, _P, _P]),
    "svtgpu_rowstats_finalize_dev": (_INT, [_INT, _INT, _INT, _I64, _I64, _P,
                                            _P, _P, _P, _P]),
    "svtgpu_rowmoments": (_INT, [_P, _INT, _P, _P]),
    "svtgpu_rowmoments_accumulate_dev": (_INT, [_P, _INT, _P, _P]),
    "svtgpu_rowmoments_finalize_dev": (_INT, [_INT, _INT, _I64, _I64, _P, _P,
                                              _P, _P]),
    "svtgpu_crossprod": (_INT, [_P, _P, _INT, _I64, _I64, _INT, _INT, _P]),
    "svtgpu_crossprod_svt": (_INT, [_P, _P, _P]),
    "svtgpu_crossprod_dev": (_INT, [_P, _P, _INT, _I64, _P, _P]),
    "svtgpu_matmul": (_INT, [_P, _P, _INT, _I64, _P]),
    "svtgpu_matmul_dev": (_INT, [_P, _P, _INT, _I64, _P, _P]),
    "svtgpu_gen_count": (_INT, [_I64, _I64, _I64, _c.c_uint64, _c.c_uint32,
                                _P, _P]),
    "svtgpu_gen_fill": (_INT, [_I64, _I64, _I64, _c.c_uint64, _c.c_uint32,
                               _c.c_uint32, _P, _INT, _INT, _P, _P, _P, _P]),
    "svtgpu_exclusive_scan": (_INT, [_P, _I64, _P, _P]),
    "svtgpu_ewise": (_INT, [_P, _INT, _P, _INT, _I64, _INT, _INT,
                            _c.POINTER(_P), _c.POINTER(_INT)]),
}

# element-wise opcodes (SVTGPU_EW_*) and warning bits
EW_OPCODES = {"*": 1, "/": 2, "abs": 11, "sign": 12, "sqrt": 13, "floor": 14,
              "ceiling": 15, "trunc": 16, "log1p": 17, "expm1": 18,
              ">": 21, ">=": 22, "<": 23, "<=": 24, "==": 25, "!=": 26,
              "is.na": 31, "is.nan": 32, "is.infinite": 33}
EW_COMPARE = (">", ">=", "<", "<=", "==", "!=")
EW_WARN_INT_OVERFLOW, EW_WARN_NAN = 1, 2
EW_WARNINGS = ((EW_WARN_INT_OVERFLOW, "NAs produced by integer overflow"),
               (EW_WARN_NAN, "NaNs produced"))

_lib = None


def lib():
    """The loaded C-ABI library (raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s is missing: run `python -m sparsearray_b200.build` "
                "(there is no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status != OK:
        raise SvtGpuError(status, lib().svtgpu_last_error().decode())


def device_count():
    n = _INT(0)
    rc = lib().svtgpu_device_count(ctypes.byref(n))
    return n.value if rc == OK else 0


def launch_count():
    return int(lib().svtgpu_launch_count())
