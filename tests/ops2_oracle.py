"""TEST INFRASTRUCTURE -- ctypes front-end to tests/ops2_oracle.c, the CPU
restatement of `x op y` between two SVTs on flat CSC arrays.  The library is
compiled on first use into a temporary directory, so the repository tree is
never written.  Never imported by the product."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from ewise_oracle import _csc

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ops2_oracle.c")
OPS = ("+", "-", "*", "&", "|", ">", "<", "!=")
OPCODES = {"+": 3, "-": 4, "*": 1, "&": 41, "|": 42, ">": 21, "<": 23,
           "!=": 26}
TYPES = {10: "logical", 13: "integer", 14: "double"}

_lib = None
_tmp = None


def lib():
    global _lib, _tmp
    if _lib is None:
        _tmp = tempfile.TemporaryDirectory(prefix="ops2_oracle_")
        so = os.path.join(_tmp.name, "libops2_oracle.so")
        subprocess.check_call(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared",
                               "-ffp-contract=off", "-o", so, _SRC, "-lm"])
        _lib = ctypes.CDLL(so)
    return _lib


def _take(p, n, dt):
    if n == 0:
        return np.zeros(0, dtype=dt)
    buf = (ctypes.c_char * (n * np.dtype(dt).itemsize)).from_address(p.value)
    return np.frombuffer(buf, dtype=dt).copy()


def ops2(nrow, nleaf, x, y, op):
    """x and y: (ptr, offs, vals, type, lacunar) of the two operands.
    Returns (ptr, offs, vals, result type, warn bits); vals of a logical
    result hold 1 / NA_integer_ (None when no NA is stored, as the device
    stores it)."""
    cx, kx = _csc(nrow, nleaf, *x[:2], x[2], x[3], x[4])
    cy, ky = _csc(nrow, nleaf, *y[:2], y[2], y[3], y[4])
    tp, to, tv = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
    otype, warn = ctypes.c_int(0), ctypes.c_int(0)
    rc = lib().ops2_oracle(ctypes.byref(cx), ctypes.byref(cy), OPCODES[op],
                           ctypes.byref(tp), ctypes.byref(to),
                           ctypes.byref(tv), ctypes.byref(otype),
                           ctypes.byref(warn))
    if rc != 0:
        raise ValueError("ops2_oracle: unsupported op %r or geometry" % (op,))
    t_out = TYPES[otype.value]
    p = _take(tp, nleaf + 1, np.int64)
    n = int(p[-1])
    v = _take(tv, n, np.float64 if t_out == "double" else np.int32)
    if t_out == "logical" and not (v == -2**31).any():
        v = None
    out = (p, _take(to, n, np.int32), v, t_out, warn.value)
    libc = ctypes.CDLL(None)
    libc.free.argtypes = [ctypes.c_void_p]
    for q in (tp, to, tv):
        libc.free(q)
    del kx, ky
    return out


def of_svt(s):
    """(ptr, offs, vals, type, lacunar) of an SVT_SparseArray."""
    return (s.ptr, s.offs, s.vals, s.type, s.lacunar)
