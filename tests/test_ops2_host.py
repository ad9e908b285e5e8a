"""`x op y` between two SVTs without a GPU: the rules of svt_semantics.h
compiled for the host and the CPU oracle (tests/ops2_oracle.c), both held to
numpy's dense `a op b` over a grid of special values and on random inputs;
the refusals and their messages; registration; the C ABI's argument checks
before any device work."""
import ctypes
import itertools
import os
import subprocess
import tempfile

import numpy as np
import pytest

import ops2_oracle
import sparsearray_b200 as sa
from sparsearray_b200 import _native, rcall
from sparsearray_b200.rcall import rshim

NA_I = -2**31
INT_MAX = 2**31 - 1
NA_R = sa.NA_REAL
NAN_PAYLOAD = np.array([0x7FF8000000000123], np.uint64).view(np.float64)[0]
NAN_NEG = np.array([0xFFF8000000000456], np.uint64).view(np.float64)[0]
CANON = 0x7FF8000000000000
NA_BITS = int(np.array([NA_R]).view(np.uint64)[0])
OPS = ops2_oracle.OPS
HERE = os.path.dirname(os.path.abspath(__file__))
NO_DEVICE = "no usable CUDA device"

GRID = {
    "logical": np.array([0, 1, NA_I], np.int32),
    "integer": np.array([0, 1, -1, INT_MAX, -INT_MAX, NA_I], np.int32),
    "double": np.array([0.0, 1.0, -1.0, float(INT_MAX), float(-INT_MAX),
                        -0.0, np.inf, -np.inf, NA_R, NAN_PAYLOAD, NAN_NEG,
                        5e-324, 1.7976931348623157e308,
                        -1.7976931348623157e308, float(2**53 + 1), 1e-200]),
}


# ---- numpy's dense definition ---------------------------------------------

def _as_double(a, t):
    if t == "double":
        return a.astype(np.float64)
    d = a.astype(np.float64)
    d[a == NA_I] = NA_R
    return d


def _is_nan(a, t):
    return np.isnan(a) if t == "double" else a == NA_I


def dense(a, ta, b, tb, op):
    """(values, kind) of `a op b`: kind 0 value, 1 NA, 2 NaN (double
    results; NaN / NA values are then not compared by bits here); logical
    results hold 1 / NA_integer_ / 0."""
    arith = op in ("+", "-", "*")
    if arith and ta != "double" and tb != "double":
        x, y = a.astype(np.int64), b.astype(np.int64)
        z = x + y if op == "+" else x - y if op == "-" else x * y
        na = (a == NA_I) | (b == NA_I) | (z > INT_MAX) | (z < -INT_MAX)
        return np.where(na, NA_I, z).astype(np.int32), na.astype(int)
    if arith:
        x, y = _as_double(a, ta), _as_double(b, tb)
        with np.errstate(all="ignore"):
            z = x + y if op == "+" else x - y if op == "-" else x * y
        xn, yn = np.isnan(x), np.isnan(y)
        first_na = np.where(xn, sa.is_na_real(x),
                            np.where(yn, sa.is_na_real(y), False))
        kind = np.where(np.isnan(z), np.where(first_na, 1, 2), 0)
        return z, kind
    na = _is_nan(a, ta) | _is_nan(b, tb)
    if op in ("&", "|"):
        ta_ = ~_is_nan(a, ta) & (a != 0)
        tb_ = ~_is_nan(b, tb) & (b != 0)
        fa = ~_is_nan(a, ta) & (a == 0)
        fb = ~_is_nan(b, tb) & (b == 0)
        if op == "&":
            true, false = ta_ & tb_, fa | fb
        else:
            true, false = ta_ | tb_, fa & fb
        na = ~true & ~false
    else:
        x, y = _as_double(a, ta), _as_double(b, tb)
        with np.errstate(all="ignore"):
            true = {">": x > y, "<": x < y, "!=": x != y}[op] & ~na
    out = np.where(na, NA_I, true.astype(np.int32)).astype(np.int32)
    return out, na.astype(int)


def dense_csc(a, ta, b, tb, op):
    """the dense result with zeros dropped, column-major CSC"""
    z, kind = dense(a, ta, b, tb, op)
    keep = (z != 0) | (kind != 0)
    ptr = np.concatenate([[0], np.cumsum(keep.sum(axis=0))]).astype(np.int64)
    rows = np.nonzero(keep.T)
    return ptr, rows[1].astype(np.int32), z.T[rows], kind.T[rows]


def svt(a, t):
    return sa.SVT_SparseArray.from_dense(a, t)


def check_oracle(a, ta, b, tb, op):
    x, y = svt(a, ta), svt(b, tb)
    p, o, v, t, w = ops2_oracle.ops2(a.shape[0], a.shape[1],
                                     ops2_oracle.of_svt(x),
                                     ops2_oracle.of_svt(y), op)
    ep, eo, ev, ek = dense_csc(a, ta, b, tb, op)
    assert np.array_equal(p, ep) and np.array_equal(o, eo), (op, ta, tb)
    if t == "double":
        assert np.array_equal(sa.is_na_real(v), ek == 1)
        assert np.array_equal(np.isnan(v) & ~sa.is_na_real(v), ek == 2)
        fin = ek == 0
        assert np.array_equal(v[fin].view(np.uint64),
                              ev[fin].astype(np.float64).view(np.uint64))
    elif t == "logical":
        assert v is None if not (ev == NA_I).any() else \
            np.array_equal(v, ev)
    else:
        assert np.array_equal(v, ev)
    return w


TYPE_PAIRS = list(itertools.product(GRID, GRID))


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("ta,tb", TYPE_PAIRS)
def test_oracle_matches_numpy_on_the_special_value_grid(op, ta, tb):
    xs, ys = GRID[ta], GRID[tb]
    a = np.repeat(xs, ys.size).reshape(-1, 1)
    b = np.tile(ys, xs.size).reshape(-1, 1)
    w = check_oracle(a, ta, b, tb, op)
    if op in ("+", "-", "*") and ta != "double" and tb != "double":
        ok = (a != NA_I) & (b != NA_I)
        x, y = a.astype(np.int64), b.astype(np.int64)
        z = x + y if op == "+" else x - y if op == "-" else x * y
        assert bool(w & 1) == bool((ok & (np.abs(z) > INT_MAX)).any())
    else:
        assert w == 0


def _random(t, shape, rng, dens=0.3):
    m = rng.random(shape) < dens
    if t == "double":
        a = np.where(m, np.round(rng.standard_normal(shape) * 3, 1), 0.0)
        a.reshape(-1)[rng.integers(0, a.size, 12)] = np.resize(
            [NA_R, np.nan, np.inf, -np.inf, -0.0, NAN_PAYLOAD], 12)
        return a
    if t == "logical":
        a = m.astype(np.int32)
        a.reshape(-1)[rng.integers(0, a.size, 4)] = NA_I
        return a
    a = np.where(m, rng.integers(-4, 5, shape), 0).astype(np.int32)
    a.reshape(-1)[rng.integers(0, a.size, 6)] = np.resize(
        [NA_I, INT_MAX, -INT_MAX], 6)
    return a


@pytest.mark.parametrize("op", OPS)
def test_oracle_matches_numpy_on_random_inputs(op):
    rng = np.random.Generator(np.random.PCG64(11))
    for ta, tb in TYPE_PAIRS:
        a, b = _random(ta, (40, 9), rng), _random(tb, (40, 9), rng)
        a[:, 2] = 0
        b[:, 3] = 0
        check_oracle(a, ta, b, tb, op)
        check_oracle(a, ta, a, ta, op)          # x op x


# NaN bits, each with its R expression (x first, implicit zeros as 0)
NAN_VECTORS = [
    ("NA_real_ + NaN", NA_R, NAN_PAYLOAD, "+", NA_BITS),
    ("NaN - NA_real_", NAN_PAYLOAD, NA_R, "-", 0x7FF8000000000123),
    ("1 - NaN (not negated)", 1.0, NAN_PAYLOAD, "-", 0x7FF8000000000123),
    ("-NaN * 0", NAN_NEG, 0.0, "*", 0xFFF8000000000456),
    ("0 - -NaN", 0.0, NAN_NEG, "-", 0xFFF8000000000456),
    ("Inf - Inf", np.inf, np.inf, "-", CANON),
    ("Inf * 0", np.inf, 0.0, "*", CANON),
    ("0 * -Inf", 0.0, -np.inf, "*", CANON),
    ("-Inf + Inf", -np.inf, np.inf, "+", CANON),
    ("NaN + NA_real_", NAN_PAYLOAD, NA_R, "+", 0x7FF8000000000123),
]


@pytest.mark.parametrize("name,x,y,op,want", NAN_VECTORS)
def test_oracle_nan_bits(name, x, y, op, want):
    a, b = np.array([[x]]), np.array([[y]])
    p, o, v, t, w = ops2_oracle.ops2(1, 1, ops2_oracle.of_svt(svt(a, "double")),
                                     ops2_oracle.of_svt(svt(b, "double")), op)
    assert list(o) == [0], name
    assert int(v.view(np.uint64)[0]) == want, name


def test_oracle_integer_na_becomes_na_real():
    a = np.array([[NA_I]], np.int32)
    b = np.array([[NAN_PAYLOAD]])
    p, o, v, t, w = ops2_oracle.ops2(1, 1, ops2_oracle.of_svt(svt(a, "integer")),
                                     ops2_oracle.of_svt(svt(b, "double")), "+")
    assert int(v.view(np.uint64)[0]) == NA_BITS


# ---- the rules, compiled for the host ---------------------------------------

@pytest.fixture(scope="module")
def sem():
    tmp = tempfile.TemporaryDirectory(prefix="ops2_host_")
    so = os.path.join(tmp.name, "libops2_host.so")
    subprocess.check_call(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared",
                           "-ffp-contract=off", "-o", so,
                           os.path.join(HERE, "ops2_host.c"), "-lm"])
    L = ctypes.CDLL(so)
    L.e2_opcode.argtypes = [ctypes.c_char_p]
    L.e2_int.argtypes = [ctypes.c_int, ctypes.c_int32, ctypes.c_int32,
                         ctypes.POINTER(ctypes.c_uint32)]
    L.e2_int.restype = ctypes.c_int32
    L.e2_dbl.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_int,
                         ctypes.c_double, ctypes.c_int]
    L.e2_dbl.restype = ctypes.c_double
    L.e2_lgl.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_int,
                         ctypes.c_double, ctypes.c_int]
    L.e2_msg.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    yield L
    tmp.cleanup()


def _rule(sem, op, a, ta, b, tb):
    """the product's rule for one pair, in the oracle's encoding"""
    code = ops2_oracle.OPCODES[op]
    rt = sem.e2_result_type(code, _native.RTYPE[ta], _native.RTYPE[tb])
    if rt == _native.INT:
        fl = ctypes.c_uint32(0)
        return int(sem.e2_int(code, int(a), int(b), ctypes.byref(fl))), \
            fl.value & 1
    xa, xn = (float(a), 0) if ta == "double" else (float(a), int(a == NA_I))
    ya, yn = (float(b), 0) if tb == "double" else (float(b), int(b == NA_I))
    if ta == "double":
        xn = int(sa.is_na_real(np.array([a]))[0])
    if tb == "double":
        yn = int(sa.is_na_real(np.array([b]))[0])
    if rt == _native.DOUBLE:
        return sem.e2_dbl(code, xa, xn, ya, yn), 0
    c = sem.e2_lgl(code, xa, xn, ya, yn)
    return {0: 0, 1: 1, 2: NA_I}[c], 0


@pytest.mark.parametrize("op", OPS)
def test_rules_match_numpy_on_the_grid(sem, op):
    for ta, tb in TYPE_PAIRS:
        for a, b in itertools.product(GRID[ta], GRID[tb]):
            z, kind = dense(np.array([a]), ta, np.array([b]), tb, op)
            got, _ = _rule(sem, op, a, ta, b, tb)
            if isinstance(got, float):
                if kind[0] == 0:
                    assert np.array([got]).view(np.uint64)[0] == \
                        np.array([z[0]], np.float64).view(np.uint64)[0], \
                        (op, a, b)
                else:
                    assert bool(sa.is_na_real(np.array([got]))[0]) == \
                        (kind[0] == 1), (op, a, b)
            else:
                assert got == z[0], (op, ta, a, tb, b)


@pytest.mark.parametrize("name,x,y,op,want", NAN_VECTORS)
def test_rule_nan_bits(sem, name, x, y, op, want):
    xn = int(sa.is_na_real(np.array([x]))[0])
    yn = int(sa.is_na_real(np.array([y]))[0])
    got = sem.e2_dbl(ops2_oracle.OPCODES[op], x, xn, y, yn)
    assert int(np.array([got]).view(np.uint64)[0]) == want, name


def test_rule_integer_overflow_flag(sem):
    fl = ctypes.c_uint32(0)
    assert sem.e2_int(3, INT_MAX, 1, ctypes.byref(fl)) == NA_I
    assert fl.value & _native.EW_WARN_INT_OVERFLOW
    fl = ctypes.c_uint32(0)
    assert sem.e2_int(4, -INT_MAX, 1, ctypes.byref(fl)) == NA_I   # -2^31
    assert fl.value & _native.EW_WARN_INT_OVERFLOW
    fl = ctypes.c_uint32(0)
    assert sem.e2_int(1, NA_I, 0, ctypes.byref(fl)) == NA_I      # NA * 0L
    assert sem.e2_int(4, 7, 7, ctypes.byref(fl)) == 0
    assert fl.value == 0


def test_result_types_and_opcodes(sem):
    L, I, D = _native.LGL, _native.INT, _native.DOUBLE
    for op in ("+", "-", "*"):
        c = sem.e2_opcode(op.encode())
        assert c == _native.EW2_OPCODES[op]
        assert sem.e2_result_type(c, L, L) == I
        assert sem.e2_result_type(c, L, I) == I
        assert sem.e2_result_type(c, I, D) == D
        assert sem.e2_result_type(c, D, L) == D
    for op in ("&", "|", ">", "<", "!="):
        c = sem.e2_opcode(op.encode())
        assert c == _native.EW2_OPCODES[op]
        assert sem.e2_result_type(c, D, D) == L
    for op in ("/", "^", "%%", "%/%", "==", ">=", "<=", "&&", "!", ""):
        assert sem.e2_opcode(op.encode()) == 0


# ---- refusals, registration, the C ABI --------------------------------------

def _x(type_="integer", shape=(3, 4)):
    a = np.zeros(shape, np.float64 if type_ == "double" else np.int32)
    a.reshape(-1)[::3] = 2
    return svt(a, type_)


def _ops(x, op, y, x_type=None):
    t = [rshim.string(op)]
    xt = x.r_type if x_type is None else rshim.string(x_type)
    if x_type is not None:
        t.append(xt)
    try:
        return rcall.SparseArray_Call("C_svtgpu_Ops_SVT_SVT", x.r_dim, xt,
                                      x.r_SVT, t[0], y.r_dim, y.r_type,
                                      y.r_SVT)
    finally:
        for o in t:
            o.release()


ZEROS = {"/": r"NaN \(0 / 0\)", "^": r"1 \(0 \^ 0\)", "%%": r"NA \(0 %%",
         "%/%": r"NA \(0 %%", "==": r"TRUE \(0 == 0\)",
         ">=": r"TRUE \(0 >= 0\)", "<=": r"TRUE \(0 <= 0\)"}


@pytest.mark.parametrize("op", list(ZEROS))
def test_refused_operators_name_what_the_zeros_would_become(op):
    x = _x()
    msg = (r'operator "%s" between two SparseArray objects is not supported '
           r'on the GPU path: the implicit zeros of the result would become '
           % op.replace("^", r"\^")) + ZEROS[op]
    with pytest.raises(rshim.RError, match=msg):
        _ops(x, op, x)


def test_refusals_through_the_python_interface():
    x, y = _x(), _x("double")
    with pytest.raises(rshim.RError, match=r'operator "/" between two'):
        x / y
    with pytest.raises(rshim.RError, match=r'operator "==" between two'):
        sa.Compare(x, "==", y)
    with pytest.raises(rshim.RError, match=r'operator "<=" between two'):
        x <= y
    with pytest.raises(rshim.RError, match=r'operator "&&" between two .*'
                       r'\(supported: "\+", "-", "\*", "&", "\|", ">", "<", '
                       r'"!="\)'):
        sa.Logic(x, "&&", y)
    with pytest.raises(TypeError):
        x & True
    # a scalar keeps the existing path and its message
    with pytest.raises(rshim.RError, match=r'Arith operator "\+" is not '
                       r'supported on a SparseArray'):
        x + 1
    with pytest.raises(rshim.RError, match=r'Arith operator "-"'):
        1 - x
    with pytest.raises(rshim.RError, match=r'Arith operator "-"'):
        sa.sweep(x, 2, np.ones(4), "-")


def test_non_conformable_and_bad_types():
    with pytest.raises(rshim.RError, match="non-conformable arrays"):
        _x() + _x(shape=(4, 3))
    with pytest.raises(rshim.RError, match="non-conformable arrays"):
        _x() * svt(np.ones((3, 4, 1), np.int32), "integer")
    with pytest.raises(rshim.RError, match=r'"\+": SparseArray objects of '
                       r'type\(\) "complex" are not supported'):
        _ops(_x(), "+", _x(), x_type="complex")


def test_entry_point_registered_with_its_arity():
    r = rcall.registered_routines()
    assert r["C_svtgpu_Ops_SVT_SVT"] == 7
    assert r["C_svtgpu_Arith_SVT"] == 7


class _MatrixHead(ctypes.Structure):
    """The leading fields of struct svtgpu_matrix (svtgpu_internal.h): all
    that svtgpu_ewise2() reads before it asks for a device."""
    _fields_ = [("nrow", ctypes.c_int64), ("nleaf", ctypes.c_int64),
                ("nnz", ctypes.c_int64), ("val_type", ctypes.c_int),
                ("flags", ctypes.c_int), ("pad", ctypes.c_char * 4096)]


def _ewise2(x, y, op):
    out, warn = ctypes.c_void_p(), ctypes.c_int()
    return _native.lib().svtgpu_ewise2(
        None if x is None else ctypes.byref(x),
        None if y is None else ctypes.byref(y), op, ctypes.byref(out),
        ctypes.byref(warn))


def test_cabi_refuses_before_device():
    L = _native.lib()
    x = _MatrixHead(3, 4, 0, _native.INT, 0)
    y = _MatrixHead(3, 4, 0, _native.DOUBLE, 0)
    for op in (2, 25, 22, 24, 0, 11, 31, 99):       # "/", "==", ">=", ...
        assert _ewise2(x, y, op) == _native.ERR_ARG
        assert "is not an operation between two matrices" in \
            L.svtgpu_last_error().decode()
    z = _MatrixHead(4, 3, 0, _native.INT, 0)
    assert _ewise2(x, z, 3) == _native.ERR_ARG
    assert "non-conformable" in L.svtgpu_last_error().decode()
    c = _MatrixHead(3, 4, 0, 15, 0)                  # complex
    assert _ewise2(x, c, 3) == _native.ERR_ARG
    assert _ewise2(None, y, 3) == _native.ERR_ARG


def test_scalar_path_still_refuses_the_new_opcodes():
    L = _native.lib()
    m = _MatrixHead(3, 4, 0, _native.INT, 0)
    v = np.array([1], np.int32)
    for op in ("+", "-", "&", "|"):
        rc = L.svtgpu_ewise(ctypes.byref(m), _native.EW2_OPCODES[op],
                            v.ctypes.data, _native.INT, 1, 0, 0,
                            ctypes.byref(ctypes.c_void_p()),
                            ctypes.byref(ctypes.c_int()))
        assert rc == _native.ERR_ARG
        assert "is not supported on a SparseArray on the GPU path" in \
            L.svtgpu_last_error().decode()


@pytest.mark.skipif(_native.device_count() > 0, reason="needs a GPU-less box")
def test_valid_call_without_device_fails_loudly():
    x, y = _x(), _x("double")
    for call in (lambda: x + y, lambda: x - x, lambda: x * y,
                 lambda: x & y, lambda: x | y, lambda: x > y,
                 lambda: x < y, lambda: sa.Compare(x, "!=", y)):
        with pytest.raises(rshim.RError, match=NO_DEVICE):
            call()
    a = _MatrixHead(3, 4, 0, _native.INT, 0)
    assert _ewise2(a, a, 3) == _native.ERR_NO_DEVICE
