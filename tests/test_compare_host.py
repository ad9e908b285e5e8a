"""Comparisons (x op v) and is.na / is.nan / is.infinite without a GPU: the
admission rule of the .Call entry points and the C ABI (refused before any
device work, with R-style messages), the value rule svt_ew_cmp() compiled for
the host and held to numpy, and the registration of the entry points."""
import ctypes
import itertools
import os
import subprocess
import tempfile

import numpy as np
import pytest

import compare_ref as cr
import sparsearray_b200 as sa
from sparsearray_b200 import _native, rcall
from sparsearray_b200.rcall import rshim

NA_I = -2**31
INT_MAX = 2**31 - 1
NA_R = sa.NA_REAL
OPS = cr.COMPARE
HERE = os.path.dirname(os.path.abspath(__file__))
NO_DEVICE = "no usable CUDA device"


@pytest.fixture(scope="module")
def sem():
    tmp = tempfile.TemporaryDirectory(prefix="compare_host_")
    so = os.path.join(tmp.name, "libcompare_host.so")
    subprocess.check_call(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared",
                           "-o", so, os.path.join(HERE, "compare_host.c"),
                           "-lm"])
    L = ctypes.CDLL(so)
    L.cmp_host.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_int,
                           ctypes.c_double]
    L.cmp_host.restype = ctypes.c_int
    L.check_host.argtypes = [ctypes.c_int] * 3 + [ctypes.c_int64] + \
        [ctypes.c_int] * 3 + [ctypes.c_int64] * 2 + \
        [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]
    L.check_host.restype = ctypes.c_int
    yield L
    tmp.cleanup()


def _x(type_="integer"):
    a = np.array([[0, 3, 0, 1], [2, 0, 0, -4], [0, 5, 7, 0]])
    return sa.SVT_SparseArray.from_dense(
        a.astype(np.float64 if type_ == "double" else np.int32), type_)


def _compare(x, op, y, margin=0, on_left=False):
    yv = sa.svt._operand(y)
    t = [rshim.string(op), rshim.integer([margin]),
         rshim.logical([int(on_left)])]
    try:
        return rcall.SparseArray_Call("C_svtgpu_Compare_SVT", x.r_dim,
                                      x.r_type, x.r_SVT, t[0], yv, t[1],
                                      t[2])
    finally:
        for o in t + [yv]:
            o.release()


def _passes_admission(call):
    """True when `call` got past the admission check: it ran (a GPU is
    present) or failed only for want of a device."""
    try:
        call()
    except rshim.RError as e:
        if NO_DEVICE in str(e):
            return True
        raise
    return True


# name -> (numpy operand, R printing of the value)
SCALARS = {
    "0": (np.array([0.0]), "0"), "-0": (np.array([-0.0]), "-0"),
    "1": (np.array([1.0]), "1"), "-1": (np.array([-1.0]), "-1"),
    "0.5": (np.array([0.5]), "0.5"), "Inf": (np.array([np.inf]), "Inf"),
    "-Inf": (np.array([-np.inf]), "-Inf"),
    "TRUE": (np.array([True]), "TRUE"), "FALSE": (np.array([False]), "FALSE"),
    "NA_integer_": (np.array([NA_I], dtype=np.int32), "NA"),
    "NA_real_": (np.array([NA_R]), "NA"), "NaN": (np.array([np.nan]), "NaN"),
}


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", list(SCALARS))
def test_admission_of_scalars(op, name):
    v, shown = SCALARS[name]
    x = _x()
    if cr.admitted(op, v):
        assert _passes_admission(lambda: _compare(x, op, v))
        return
    zeros = "NA" if shown in ("NA", "NaN") else "TRUE"
    msg = ('operator "%s": element 1 of the operand is %s, so the implicit '
           'zeros of the result would be %s' % (op, shown, zeros))
    with pytest.raises(rshim.RError) as e:
        _compare(x, op, v)
    assert msg in str(e.value)


def test_admission_table():
    """The issue's table, stated per operator on a few values."""
    allowed = {">": [0.0, -0.0, 2.0, np.inf], ">=": [1e-300, 3.0, np.inf],
               "<": [0.0, -0.0, -2.0, -np.inf], "<=": [-1e-300, -np.inf],
               "==": [1.0, -1.0, np.inf], "!=": [0.0, -0.0]}
    refused = {">": [-1e-300, -np.inf], ">=": [0.0, -0.0, -1.0],
               "<": [1e-300, np.inf], "<=": [0.0, -0.0, 1.0],
               "==": [0.0, -0.0], "!=": [1.0, -np.inf]}
    for op in OPS:
        for v in allowed[op]:
            assert cr.admitted(op, np.array([v])), (op, v)
        for v in refused[op] + [np.nan, NA_R]:
            assert not cr.admitted(op, np.array([v])), (op, v)


def test_offending_element_of_vectors_is_named():
    x = _x()     # 3 x 4
    with pytest.raises(rshim.RError, match=r'operator ">=": element 3 of the '
                       r'operand is 0, so the implicit zeros of the result '
                       r'would be TRUE'):
        _compare(x, ">=", np.array([1, 2, 0], dtype=np.int32), margin=1)
    with pytest.raises(rshim.RError, match=r'operator ">": element 2 of the '
                       r'operand is -0.5, so the implicit zeros'):
        _compare(x, ">", np.array([1.0, -0.5, 2.0]), margin=1)
    with pytest.raises(rshim.RError, match=r'operator "<": element 4 of the '
                       r'operand is 5, so'):
        sa.sweep(x, 2, np.array([0, -1, -2, 5], dtype=np.int32), "<")
    with pytest.raises(rshim.RError, match=r'operator "==": element 2 of the '
                       r'operand is NA, so the implicit zeros of the result '
                       r'would be NA'):
        sa.sweep(x, 2, np.array([1.0, NA_R, 2.0, 3.0]), "==")
    with pytest.raises(rshim.RError, match=r'element 1 of the operand is '
                       r'FALSE'):
        sa.Compare(x, "==", np.array([False, True, True]))
    with pytest.raises(rshim.RError, match=r'element 3 of the operand is NaN'):
        x > np.array([1.0, 2.0, np.nan])


def test_operand_on_the_left_is_mirrored():
    x = _x()
    # 0 < x is x > 0: admitted; 1 > x is x < 1: 0 < 1 is TRUE, refused
    assert _passes_admission(lambda: _compare(x, "<", [0], on_left=True))
    assert _passes_admission(lambda: _compare(x, ">=", [-1], on_left=True))
    with pytest.raises(rshim.RError, match=r'operator ">": element 1 of the '
                       r'operand is 1, so the implicit zeros of the result '
                       r'would be TRUE'):
        _compare(x, ">", [1], on_left=True)
    with pytest.raises(rshim.RError, match=r'operator "<=": element 1'):
        _compare(x, "<=", [0], on_left=True)          # 0 <= 0
    # Python reflects `2 < x` to x.__gt__(2) and `-1 >= x` to x.__le__(-1)
    with pytest.raises(rshim.RError, match=r'operator ">": element 1 of the '
                       r'operand is -1'):
        -1 < x
    with pytest.raises(rshim.RError, match=r'operator "<=": element 1 of the '
                       r'operand is 1'):
        1 >= x
    assert _passes_admission(lambda: sa.Compare(3, "<", x))      # x > 3
    with pytest.raises(rshim.RError, match=r'operator ">": element 1'):
        sa.Compare(3, ">", x)                                    # x < 3


def test_mirrored_refusal_matches_mirrored_admission(sem):
    for op, v in itertools.product(OPS, [0.0, -0.0, 1.0, -1.0, np.inf]):
        a = np.array([v])
        bad = ctypes.c_int64(0)
        code_left = sem.check_host(_native.EW_OPCODES[op], _native.INT,
                                   _native.DOUBLE, 1, 0, 1, 2, 3, 4,
                                   a.ctypes.data, ctypes.byref(bad))
        assert (code_left == 0) == cr.admitted(cr.MIRROR[op], a), (op, v)


@pytest.mark.parametrize("call,msg", [
    (lambda x: _compare(x, ">", [1, 2]), r'length 2, a scalar operand'),
    (lambda x: _compare(x, ">", [1, 2], margin=1), r'length nrow\(x\) = 3'),
    (lambda x: _compare(x, ">", [1, 2, 3], margin=2), r'length ncol\(x\) = 4'),
    (lambda x: _compare(x, ">", [1], margin=3), r"MARGIN must be 0"),
    (lambda x: _compare(x, "<>", [1]), r'Compare operator "<>" is not '
     r'supported'),
    (lambda x: _compare(x, "+", [1]), r'Compare operator "\+"'),
    (lambda x: x > np.ones(5), r'length nrow\(x\) = 3'),
    (lambda x: sa.sweep(x, 2, np.ones(3), ">"), r'length ncol\(x\) = 4'),
    (lambda x: sa.sweep(x, 2, np.ones(4), "-"), r'Arith operator "-"'),
    (lambda x: sa.sweep(x, 2, np.ones(4), "+"), r'Arith operator "\+"'),
    (lambda x: sa.svt._arith_call(x, ">", [1], 0, False),
     r'Arith operator ">" is not supported'),
])
def test_refusals_before_device(call, msg):
    with pytest.raises(rshim.RError, match=msg):
        call(_x())


def test_margin_2_needs_a_matrix():
    a = np.zeros((2, 3, 2), dtype=np.int32)
    a[1, 2, 1] = 4
    x = sa.SVT_SparseArray.from_dense(a)
    with pytest.raises(rshim.RError, match="MARGIN must be 0"):
        _compare(x, ">", [1, 2, 3], margin=2)


@pytest.mark.parametrize("fun", ["is.finite", "is.null", "anyNA", "is.na<-",
                                 "isna", ""])
def test_is_refuses_other_names(fun):
    x = _x("double")
    t = rshim.string(fun)
    try:
        with pytest.raises(rshim.RError, match=r'"%s" is not supported on a '
                           r'SparseArray on the GPU path' % fun.replace(
                               ".", r"\.")):
            rcall.SparseArray_Call("C_svtgpu_is_SVT", x.r_dim, x.r_type,
                                   x.r_SVT, t)
    finally:
        t.release()


# ---- the value rule, compiled for the host -------------------------------

INT_VALUES = [0, 1, -1, 2, 7, INT_MAX, -INT_MAX, NA_I, 2**24 + 1]
DBL_VALUES = [0.0, -0.0, 1.0, -1.0, 0.5, 7.0, np.inf, -np.inf, NA_R, np.nan,
              np.array([0x7FF8000000000123], np.uint64).view(np.float64)[0],
              np.array([0xFFF0000000000001], np.uint64).view(np.float64)[0],
              5e-324, -5e-324, 2.2250738585072e-308, float(INT_MAX),
              float(INT_MAX) + 0.5, float(-INT_MAX), 2.0**53, 2.0**53 + 2,
              float(2**53 + 1)]
V_INT = [0, 1, -1, 7, INT_MAX, -INT_MAX]
V_DBL = [0.0, -0.0, 1.0, -1.0, 0.5, 7.0, np.inf, -np.inf, 5e-324, -5e-324,
         float(INT_MAX), float(INT_MAX) + 0.5, float(2**53 + 1), 2.0**53 + 2]
CODE = {False: 0, True: 1}


def _expect(op, x, x_int, v, v_int):
    if x_int:
        if x == NA_I:
            return 2
        xs = np.int32(x)
    else:
        if np.isnan(x):
            return 2
        xs = np.float64(x)
    vs = np.int32(v) if v_int else np.float64(v)
    return CODE[bool(cr._NP[op](xs, vs))]


@pytest.mark.parametrize("op", OPS)
def test_value_rule_matches_numpy(sem, op):
    code = _native.EW_OPCODES[op]
    n = 0
    for x_int, xs in ((True, INT_VALUES), (False, DBL_VALUES)):
        for v_int, vs in ((True, V_INT), (False, V_DBL)):
            for x, v in itertools.product(xs, vs):
                x_na = (x == NA_I) if x_int else bool(sa.is_na_real(
                    np.array([x]))[0])
                got = sem.cmp_host(code, float(x), int(x_na), float(v))
                assert got == _expect(op, x, x_int, v, v_int), (op, x, v)
                n += 1
    assert n == len(INT_VALUES) * (len(V_INT) + len(V_DBL)) + \
        len(DBL_VALUES) * (len(V_INT) + len(V_DBL))


def test_int_against_2_53_plus_1(sem):
    """2^53 + 1 as a double is 2^53; an int compares with it after an
    exact conversion to double, as R does."""
    v = float(2**53 + 1)
    for op in OPS:
        got = sem.cmp_host(_native.EW_OPCODES[op], float(INT_MAX), 0, v)
        assert got == CODE[bool(cr._NP[op](np.int32(INT_MAX),
                                           np.float64(v)))]


@pytest.mark.parametrize("fun", ["is.na", "is.nan", "is.infinite"])
def test_predicates_match_numpy(sem, fun):
    code = _native.EW_OPCODES[fun]
    for x in DBL_VALUES:
        na = bool(sa.is_na_real(np.array([x]))[0])
        exp = {"is.na": np.isnan(x), "is.nan": np.isnan(x) and not na,
               "is.infinite": np.isinf(x)}[fun]
        assert sem.cmp_host(code, float(x), int(na), 0.0) == int(exp), x
    for x in INT_VALUES:
        exp = fun == "is.na" and x == NA_I
        assert sem.cmp_host(code, float(x), int(x == NA_I), 0.0) == int(exp)


def test_dense_reference_vectors():
    """compare_ref's dense definition on hand-written vectors."""
    a = np.array([[3], [NA_I], [1], [0]], dtype=np.int32)
    val, na = cr.dense(a, "integer", ">", [1], "integer")
    assert list(val[:, 0]) == [True, False, False, False]
    assert list(na[:, 0]) == [False, True, False, False]
    p, i, x = cr.to_csc(val, na)
    assert list(p) == [0, 2] and list(i) == [0, 1] and list(x) == [1, NA_I]
    d = np.array([[np.inf], [NA_R], [np.nan], [-2.0]])
    for fun, rows in (("is.na", [1, 2]), ("is.nan", [2]),
                      ("is.infinite", [0])):
        p, i, x = cr.to_csc(*cr.dense(d, "double", fun))
        assert list(i) == rows and x is None


# ---- registration and the C ABI -------------------------------------------

def test_entry_points_registered_with_their_arity():
    r = rcall.registered_routines()
    assert r["C_svtgpu_Compare_SVT"] == 7
    assert r["C_svtgpu_is_SVT"] == 4
    assert r["C_svtgpu_Arith_SVT"] == 7


class _MatrixHead(ctypes.Structure):
    """The leading fields of struct svtgpu_matrix (svtgpu_internal.h): all
    that svtgpu_ewise() reads before it asks for a device."""
    _fields_ = [("nrow", ctypes.c_int64), ("nleaf", ctypes.c_int64),
                ("nnz", ctypes.c_int64), ("val_type", ctypes.c_int),
                ("flags", ctypes.c_int), ("pad", ctypes.c_char * 4096)]


def test_cabi_refuses_before_device():
    L = _native.lib()
    for nm in OPS + ("is.na", "is.nan", "is.infinite"):
        assert _native.EW_OPCODES[nm] > 0
    m = _MatrixHead(3, 4, 0, _native.INT, 0)
    v = np.array([0.0])
    out, warn = ctypes.c_void_p(), ctypes.c_int()
    rc = L.svtgpu_ewise(ctypes.byref(m), _native.EW_OPCODES[">="],
                        v.ctypes.data, _native.DOUBLE, 1, 0, 0,
                        ctypes.byref(out), ctypes.byref(warn))
    assert rc == _native.ERR_ARG
    assert 'operator ">=": element 1 of the operand is 0' in \
        L.svtgpu_last_error().decode()
    # mirrored: 0 < x is x > 0, admitted; 0 > x is x < 0 ... admitted too;
    # 1 > x is x < 1, refused
    v1 = np.array([1.0])
    rc = L.svtgpu_ewise(ctypes.byref(m), _native.EW_OPCODES[">"],
                        v1.ctypes.data, _native.DOUBLE, 1, 0, 1,
                        ctypes.byref(out), ctypes.byref(warn))
    assert rc == _native.ERR_ARG


@pytest.mark.skipif(_native.device_count() > 0, reason="needs a GPU-less box")
def test_valid_call_without_device_fails_loudly():
    x = _x("double")
    for call in (lambda: x > 0, lambda: sa.Compare(x, "!=", 0),
                 lambda: sa.sweep(x, 2, np.arange(1, 5.0), "=="),
                 lambda: sa.is_na(x), lambda: sa.is_nan(x),
                 lambda: sa.is_infinite(x)):
        with pytest.raises(rshim.RError, match=NO_DEVICE):
            call()
    L = _native.lib()
    m = _MatrixHead(3, 4, 0, _native.INT, 0)
    v = np.array([1.0])
    rc = L.svtgpu_ewise(ctypes.byref(m), _native.EW_OPCODES[">"],
                        v.ctypes.data, _native.DOUBLE, 1, 0, 0,
                        ctypes.byref(ctypes.c_void_p()),
                        ctypes.byref(ctypes.c_int()))
    assert rc == _native.ERR_NO_DEVICE
