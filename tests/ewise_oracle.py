"""TEST INFRASTRUCTURE -- ctypes front-end to tests/ewise_oracle.c, the CPU
restatement of the element-wise operations (x * v, x / v, Math) on flat CSC
arrays.  The library is compiled on first use into a temporary directory,
so the repository tree is never written.  Never imported by the product."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ewise_oracle.c")
RTYPE = {"logical": 10, "integer": 13, "double": 14}


class _Csc(ctypes.Structure):
    _fields_ = [("nrow", ctypes.c_int64), ("nleaf", ctypes.c_int64),
                ("leaf_ptr", ctypes.c_void_p), ("offs", ctypes.c_void_p),
                ("vals", ctypes.c_void_p), ("val_type", ctypes.c_int),
                ("lacunar", ctypes.c_void_p)]


def _csc(nrow, nleaf, ptr, offs, vals, type_, lacunar):
    ptr = np.ascontiguousarray(ptr, dtype=np.int64)
    offs = np.ascontiguousarray(offs, dtype=np.int32)
    keep = [ptr, offs]
    c = _Csc()
    c.nrow, c.nleaf = int(nrow), int(nleaf)
    c.leaf_ptr = ptr.ctypes.data
    c.offs = offs.ctypes.data
    c.val_type = RTYPE[type_]
    c.vals = None
    if vals is not None:
        vals = np.ascontiguousarray(
            vals, dtype=np.float64 if type_ == "double" else np.int32)
        keep.append(vals)
        c.vals = vals.ctypes.data
    c.lacunar = None
    if lacunar is not None:
        lacunar = np.ascontiguousarray(lacunar, dtype=np.uint8)
        keep.append(lacunar)
        c.lacunar = lacunar.ctypes.data
    return c, keep


_lib = None
_tmp = None


def lib():
    global _lib, _tmp
    if _lib is None:
        _tmp = tempfile.TemporaryDirectory(prefix="ewise_oracle_")
        so = os.path.join(_tmp.name, "libewise_oracle.so")
        subprocess.check_call(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared",
                               "-o", so, _SRC, "-lm"])
        _lib = ctypes.CDLL(so)
    return _lib


EW_OPCODES = {"*": 1, "/": 2, "abs": 11, "sign": 12, "sqrt": 13, "floor": 14,
              "ceiling": 15, "trunc": 16, "log1p": 17, "expm1": 18}


def ewise(nrow, nleaf, ptr, offs, vals, type_, op, v=None, v_type=None,
          margin=0, lacunar=None):
    """op(x) or x op v (v a numpy vector of v_type) that keeps zeros at zero:
    (ptr, offs, vals, result type, warn bits)."""
    c, keep = _csc(nrow, nleaf, ptr, offs, vals, type_, lacunar)
    vp, vt = None, 0
    if v is not None:
        v = np.ascontiguousarray(
            v, dtype=np.float64 if v_type == "double" else np.int32)
        keep.append(v)
        vp, vt = v.ctypes.data_as(ctypes.c_void_p), RTYPE[v_type]
    tp, to, tv = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
    otype, warn = ctypes.c_int(0), ctypes.c_int(0)
    L = lib()
    rc = L.ewise_oracle(ctypes.byref(c), EW_OPCODES[op], vp, vt,
                            int(margin), ctypes.byref(tp), ctypes.byref(to),
                            ctypes.byref(tv), ctypes.byref(otype),
                            ctypes.byref(warn))
    if rc != 0:
        raise ValueError("ewise_oracle: unsupported op %r" % (op,))
    t_out = "double" if otype.value == 14 else "integer"
    vt_np = np.float64 if t_out == "double" else np.int32

    def take(p, n, dt):
        if n == 0:
            return np.zeros(0, dtype=dt)
        buf = (ctypes.c_char * (n * np.dtype(dt).itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=dt).copy()

    p = take(tp, nleaf + 1, np.int64)
    n = int(p[-1])
    out = (p, take(to, n, np.int32), take(tv, n, vt_np), t_out, warn.value)
    libc = ctypes.CDLL(None)
    libc.free.argtypes = [ctypes.c_void_p]
    for q in (tp, to, tv):
        libc.free(q)
    return out
