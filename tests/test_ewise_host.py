"""Element-wise operations (x * v, x / v, Math) without a GPU: the oracle's
restatement against base R's dense definition computed with numpy, the
hand-written rule vectors (each with the R expression it restates), the
refusals of the .Call entry points (raised before any device work) and their
registration."""
import ctypes

import numpy as np
import pytest

import ewise_oracle
import sparsearray_b200 as sa
from sparsearray_b200 import _native, rcall
from sparsearray_b200.rcall import rshim

NA_I = -2**31
INT_MAX = 2**31 - 1
NA_R = sa.NA_REAL
NAN_BITS = 0x7FF8000000000000
_LIBM = ctypes.CDLL("libm.so.6")
for _f in ("log1p", "expm1"):
    getattr(_LIBM, _f).restype = ctypes.c_double
    getattr(_LIBM, _f).argtypes = [ctypes.c_double]

MATH = ["abs", "sign", "sqrt", "floor", "ceiling", "trunc", "log1p", "expm1"]


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def dense_ref(a, type_, op, v=None, v_type=None, margin=0):
    """f(as.matrix(x)) with base R's rules, as (dense result, type, warn)."""
    nrow = a.shape[0]
    a = a.reshape((nrow, int(np.prod(a.shape[1:]))), order="F")
    if type_ == "double":
        xd = a.astype(np.float64)
        na = sa.is_na_real(xd).reshape(xd.shape)
    else:
        na = a == NA_I
        xd = a.astype(np.float64)
        xd[na] = np.nan
    nan_in = np.isnan(xd) & ~na
    V = None
    if v is not None:
        v = np.asarray(v)
        V = v.reshape(1, 1) if margin == 0 else \
            v.reshape(-1, 1) if margin == 1 else v.reshape(1, -1)
        V = np.broadcast_to(V, a.shape)
    x_int = type_ != "double"
    if (op == "*" and x_int and v_type != "double") or (op == "abs" and x_int):
        z = np.abs(a.astype(np.int64)) if op == "abs" else \
            a.astype(np.int64) * V.astype(np.int64)
        ov = ~na & ((z > INT_MAX) | (z <= NA_I))
        r = np.where(na | ov, NA_I, np.where(ov, 0, z)).astype(np.int32)
        return r, "integer", int(ov.any())
    with np.errstate(all="ignore"):
        if op == "*":
            r = xd * V.astype(np.float64)
        elif op == "/":
            r = xd / V.astype(np.float64)
        elif op in ("log1p", "expm1"):
            f = getattr(_LIBM, op)
            r = np.frompyfunc(lambda t: f(float(t)), 1, 1)(xd).astype(
                np.float64)
        else:
            r = {"abs": np.abs, "sign": np.sign, "sqrt": np.sqrt,
                 "floor": np.floor, "ceiling": np.ceil,
                 "trunc": np.trunc}[op](xd)
    r = np.array(r, dtype=np.float64)
    made = np.isnan(r) & ~np.isnan(xd)
    warn = 2 if (op in MATH and made.any()) else 0
    rb = r.view(np.uint64)
    rb[made] = NAN_BITS
    rb[nan_in] = a.astype(np.float64).view(np.uint64)[nan_in] \
        if type_ == "double" else rb[nan_in]
    r[na] = NA_R
    return r, "double", warn


def to_csc(r):
    nleaf = r.shape[1]
    ptr = np.zeros(nleaf + 1, dtype=np.int64)
    offs, vals = [], []
    for l in range(nleaf):
        nz = np.flatnonzero(r[:, l] != 0)
        ptr[l + 1] = ptr[l] + nz.size
        offs.append(nz.astype(np.int32))
        vals.append(r[nz, l])
    return (ptr, np.concatenate(offs) if offs else np.zeros(0, np.int32),
            np.concatenate(vals) if vals else np.zeros(0, r.dtype))


def oracle_of(x, op, v=None, v_type=None, margin=0):
    nrow = x.dim[0]
    nleaf = x.ptr.size - 1
    return ewise_oracle.ewise(nrow, nleaf, x.ptr, x.offs, x.vals, x.type, op, v,
                      v_type, margin, x.lacunar)


def assert_same(got, exp_dense, exp_type, exp_warn):
    p, o, vals, t, w = got
    ep, eo, ev = to_csc(exp_dense)
    assert t == exp_type
    assert w == exp_warn
    assert np.array_equal(p, ep)
    assert np.array_equal(o, eo)
    if t == "double":
        assert np.array_equal(bits(vals), bits(ev))
    else:
        assert np.array_equal(vals, ev)


def random_dense(rng, nrow, ncol, type_, density=0.3, specials=True):
    m = rng.random((nrow, ncol)) < density
    if type_ == "double":
        a = np.where(m, rng.standard_normal((nrow, ncol)) * 3, 0.0)
        if specials and a.size:
            sp = [NA_R, np.nan, np.inf, -np.inf, 1e-310, -1e-310, 0.25,
                  -0.5, -1.0, -2.0, 1e308, 0.999]
            k = rng.integers(0, a.size, size=min(a.size, 2 * len(sp)))
            a.reshape(-1)[k] = np.resize(np.array(sp), k.size)
        return a
    if type_ == "logical":
        a = np.where(m, 1, 0).astype(np.int32)
    else:
        a = np.where(m, rng.integers(-50, 50, (nrow, ncol)), 0).astype(
            np.int32)
        if specials and a.size:
            sp = [NA_I, INT_MAX, -INT_MAX, 70000, -46341, 46341]
            k = rng.integers(0, a.size, size=min(a.size, 2 * len(sp)))
            a.reshape(-1)[k] = np.resize(np.array(sp), k.size)
    if specials and a.size:
        a.reshape(-1)[rng.integers(0, a.size)] = NA_I
    return a


def operand(rng, op, n, v_type):
    if v_type == "double":
        v = rng.standard_normal(n) * 2
        v[rng.random(n) < 0.2] = np.inf if op == "/" else 0.0
        if n:
            v[0] = 1e-320 if op == "*" else -np.inf   # underflow / 0 / -Inf
        return v
    if v_type == "logical":
        return np.ones(n, dtype=np.int32) if op == "/" else \
            (rng.random(n) < 0.7).astype(np.int32)
    v = rng.integers(-3, 4, n).astype(np.int32)
    if op == "/":
        v[v == 0] = 5
    elif n:
        v[0] = 65536                                 # overflow with 70000
    return v


@pytest.mark.parametrize("type_", ["integer", "logical", "double"])
@pytest.mark.parametrize("shape", [(7, 9), (40, 13), (0, 5), (6, 0), (1, 1)])
def test_oracle_math_matches_dense_definition(type_, shape):
    rng = np.random.Generator(np.random.PCG64(sum(shape) + len(type_)))
    a = random_dense(rng, *shape, type_)
    x = sa.SVT_SparseArray.from_dense(a, type_)
    for op in MATH:
        r, t, w = dense_ref(a, type_, op)
        assert_same(oracle_of(x, op), r, t, w)


@pytest.mark.parametrize("type_", ["integer", "logical", "double"])
@pytest.mark.parametrize("v_type", ["integer", "logical", "double"])
@pytest.mark.parametrize("margin", [0, 1, 2])
@pytest.mark.parametrize("op", ["*", "/"])
def test_oracle_arith_matches_dense_definition(type_, v_type, margin, op):
    rng = np.random.Generator(np.random.PCG64(
        7 * margin + len(type_) + 3 * len(v_type) + (op == "*")))
    for shape in [(30, 11), (0, 4), (5, 0)]:
        a = random_dense(rng, *shape, type_)
        x = sa.SVT_SparseArray.from_dense(a, type_)
        n = 1 if margin == 0 else shape[0] if margin == 1 else shape[1]
        v = operand(rng, op, n, v_type)
        r, t, w = dense_ref(a, type_, op, v, v_type, margin)
        assert_same(oracle_of(x, op, v, v_type, margin), r, t, w)


def test_oracle_lacunar_and_mixed_leaves():
    a = np.zeros((6, 5), dtype=np.int32)
    a[[0, 2], 0] = 1          # lacunar leaf
    a[[1, 4], 1] = [3, -2]    # regular leaf
    a[5, 3] = 1               # lacunar leaf (column 2 and 4 empty)
    mixed = sa.SVT_SparseArray.from_dense(a, "integer")
    assert mixed.lacunar is not None and mixed.vals is not None
    allones = sa.SVT_SparseArray.from_dense((a != 0).astype(np.int32),
                                            "logical")
    assert allones.vals is None
    for x, src in ((mixed, a), (allones, (a != 0).astype(np.int32))):
        for op in MATH:
            r, t, w = dense_ref(src, x.type, op)
            assert_same(oracle_of(x, op), r, t, w)
        for op, v, vt in (("*", [2], "integer"), ("*", [0.5], "double"),
                          ("/", [4.0], "double"), ("*", [0], "integer")):
            r, t, w = dense_ref(src, x.type, op, np.array(v), vt, 0)
            assert_same(oracle_of(x, op, np.array(v), vt, 0), r, t, w)


def one(op, xs, type_, v=None, v_type=None):
    """op applied to the column vector xs (one leaf): (values, type, warn)
    at the kept positions, and the kept offsets."""
    a = np.array(xs, dtype=np.float64 if type_ == "double" else np.int32)
    x = sa.SVT_SparseArray.from_dense(a.reshape(-1, 1), type_,
                                      lacunar=False)
    p, o, vals, t, w = oracle_of(x, op, None if v is None else np.array(v),
                                 v_type, 0)
    return vals, t, w, o


def test_rule_vectors():
    # sqrt(c(-1, NA, NaN, 4))  ->  NaN NA NaN 2, warning "NaNs produced"
    v, t, w, o = one("sqrt", [-1, NA_R, np.nan, 4], "double")
    assert t == "double" and w == 2
    assert np.isnan(v[0]) and not sa.is_na_real(v[:1])[0]
    assert sa.is_na_real(v[1:2])[0] and np.isnan(v[2]) and v[3] == 2
    # sqrt(NaN) alone does not warn: the NaN was not produced
    assert one("sqrt", [np.nan], "double")[2] == 0
    # .Machine$integer.max * 2L  ->  NA, "NAs produced by integer overflow"
    v, t, w, o = one("*", [INT_MAX], "integer", [2], "integer")
    assert t == "integer" and w == 1 and v[0] == NA_I
    # -46341L * 46341L  ->  NA (below -.Machine$integer.max: INT_MIN is NA)
    v, t, w, o = one("*", [-46341], "integer", [46341], "integer")
    assert w == 1 and v[0] == NA_I
    # 46340L * 46340L  ->  2147395600L, no warning
    v, t, w, o = one("*", [46340], "integer", [46340], "integer")
    assert w == 0 and v[0] == 2147395600
    # c(3L, NA) * 0L  ->  0 NA: the 0 is dropped, the NA kept
    v, t, w, o = one("*", [3, NA_I], "integer", [0], "integer")
    assert list(o) == [1] and v[0] == NA_I and w == 0
    # TRUE * TRUE  ->  1L (integer)
    v, t, w, o = one("*", [1], "logical", [1], "logical")
    assert t == "integer" and v[0] == 1
    # 5L / 2L  ->  2.5 (double); NA_integer_ / 2L  ->  NA_real_
    v, t, w, o = one("/", [5, NA_I], "integer", [2], "integer")
    assert t == "double" and v[0] == 2.5 and sa.is_na_real(v[1:2])[0]
    # 3 / Inf  ->  0 (dropped); Inf / Inf -> NaN, no warning
    v, t, w, o = one("/", [3, np.inf], "double", [np.inf], "double")
    assert list(o) == [1] and np.isnan(v[0]) and w == 0
    # c(Inf, 2) * 0  ->  NaN 0: kept NaN, dropped 0
    v, t, w, o = one("*", [np.inf, 2], "double", [0.0], "double")
    assert list(o) == [0] and np.isnan(v[0])
    # 1e-300 * 1e-300  ->  0 (underflow, dropped)
    assert one("*", [1e-300], "double", [1e-300], "double")[3].size == 0
    # -2 * 0  ->  -0, compares equal to 0: dropped
    assert one("*", [-2.0], "double", [0.0], "double")[3].size == 0
    # log1p(-1)  ->  -Inf, no warning; log1p(-2) -> NaN with the warning
    v, t, w, o = one("log1p", [-1.0], "double")
    assert v[0] == -np.inf and w == 0
    v, t, w, o = one("log1p", [-2.0], "double")
    assert np.isnan(v[0]) and w == 2
    # trunc(-0.5), ceiling(-0.5)  ->  -0: dropped; floor(0.5) -> 0: dropped
    for op, xv in (("trunc", -0.5), ("ceiling", -0.5), ("floor", 0.5)):
        assert one(op, [xv], "double")[3].size == 0
    # floor(-0.5)  ->  -1
    assert one("floor", [-0.5], "double")[0][0] == -1
    # abs(c(-3L, NA))  ->  3L NA (integer, do_abs()); abs(TRUE) -> 1L
    v, t, w, o = one("abs", [-3, NA_I], "integer")
    assert t == "integer" and list(v) == [3, NA_I]
    assert one("abs", [1], "logical")[1] == "integer"
    # sign(-2L)  ->  -1 (double); sign(NA_integer_) -> NA_real_
    v, t, w, o = one("sign", [-2, NA_I], "integer")
    assert t == "double" and v[0] == -1 and sa.is_na_real(v[1:2])[0]
    # expm1(NA_real_) -> NA; expm1(-800) -> -1
    v, t, w, o = one("expm1", [NA_R, -800.0], "double")
    assert sa.is_na_real(v[:1])[0] and v[1] == -1
    # a NaN with a payload keeps its bits through Math (math1())
    odd = np.array([0x7FF8000000000123], dtype=np.uint64).view(np.float64)
    v, t, w, o = one("floor", [odd[0]], "double")
    assert bits(v)[0] == 0x7FF8000000000123


# ---- the .Call entry points: refusals come before any device work --------

def _arith(x, op, y, margin=0, on_left=False):
    yv = sa.svt._operand(y)
    t = [rshim.string(op), rshim.integer([margin]),
         rshim.logical([int(on_left)])]
    try:
        return rcall.SparseArray_Call("C_svtgpu_Arith_SVT", x.r_dim,
                                      x.r_type, x.r_SVT, t[0], yv, t[1], t[2])
    finally:
        for o in t + [yv]:
            o.release()


def _x():
    return sa.SVT_SparseArray.from_dense(
        np.arange(12, dtype=np.int32).reshape(3, 4), "integer")


@pytest.mark.parametrize("call,msg", [
    (lambda x: _arith(x, "+", [1]), r'Arith operator "\+" is not supported'),
    (lambda x: _arith(x, "^", [2]), r'Arith operator "\^"'),
    (lambda x: _arith(x, "%%", [2]), r'Arith operator "%%"'),
    (lambda x: _arith(x, "/", [2], on_left=True),
     r'operator "/" with the SparseArray on the right'),
    (lambda x: _arith(x, "*", [np.inf]), r'element 1 of the operand is Inf'),
    (lambda x: _arith(x, "*", [-np.inf]), r'element 1 of the operand is -Inf'),
    (lambda x: _arith(x, "*", [1.0, np.nan, 2.0], margin=1),
     r'"\*": element 2 of the operand is NaN'),
    (lambda x: _arith(x, "*", [1, 2, NA_I], margin=1),
     r'element 3 of the operand is NA'),
    (lambda x: _arith(x, "*", [NA_R]), r'element 1 of the operand is NA'),
    (lambda x: _arith(x, "/", [1, 2, 3, 0], margin=2),
     r'"/": element 4 of the operand is 0'),
    (lambda x: _arith(x, "/", [0.0]), r'element 1 of the operand is 0'),
    (lambda x: _arith(x, "/", [np.nan]), r'element 1 of the operand is NaN'),
    (lambda x: _arith(x, "/", [NA_I]), r'element 1 of the operand is NA'),
    (lambda x: _arith(x, "/", [False]), r'element 1 of the operand is 0'),
    (lambda x: _arith(x, "*", [1, 2]), r'length 2, a scalar operand'),
    (lambda x: _arith(x, "*", [1, 2], margin=1), r'length nrow\(x\) = 3'),
    (lambda x: _arith(x, "*", [1, 2, 3], margin=2), r'length ncol\(x\) = 4'),
    (lambda x: _arith(x, "*", [1], margin=3), r"MARGIN must be 0"),
    (lambda x: sa.Math(x, "exp"), r'Math function "exp" is not supported'),
    (lambda x: sa.Math(x, "log"), r'Math function "log"'),
    (lambda x: sa.Math(x, "cos"), r'Math function "cos"'),
    (lambda x: sa.Math(x, "round"), r'Math function "round"'),
    (lambda x: sa.Math(x, "cumsum"), r'Math function "cumsum"'),
    (lambda x: 2 / x, r'operator "/" with the SparseArray on the right'),
    (lambda x: x * np.array([1.0, np.inf, 1.0]),
     r'element 2 of the operand is Inf'),
    (lambda x: sa.sweep(x, 2, np.array([1.0, 2.0, 0.0, 1.0]), "/"),
     r'element 3 of the operand is 0'),
    (lambda x: sa.sweep(x, 2, np.ones(4)), r'Arith operator "-"'),
    (lambda x: x * np.ones(4), r'length nrow\(x\) = 3'),
])
def test_refusals_before_device(call, msg):
    with pytest.raises(rshim.RError, match=msg):
        call(_x())


def test_margin_2_needs_a_matrix():
    a = np.zeros((2, 3, 2), dtype=np.int32)
    a[1, 2, 1] = 4
    x = sa.SVT_SparseArray.from_dense(a)
    with pytest.raises(rshim.RError, match="MARGIN must be 0"):
        _arith(x, "*", [1, 2, 3], margin=2)


def test_refusal_of_unsupported_x_type():
    x = _x()
    with pytest.raises(rshim.RError, match="not supported by the SparseArray"):
        rcall.SparseArray_Call("C_svtgpu_Math_SVT", x.r_dim,
                               rshim.string("complex"), x.r_SVT,
                               rshim.string("abs"))


def test_ndarray_operand_defers_to_the_svt():
    """ndarray * x must reach x.__rmul__ (and its checks), not broadcast."""
    with pytest.raises(rshim.RError, match=r"length nrow\(x\) = 3"):
        np.ones(5) * _x()


def test_entry_points_registered_with_their_arity():
    r = rcall.registered_routines()
    assert r["C_svtgpu_Arith_SVT"] == 7
    assert r["C_svtgpu_Math_SVT"] == 4


def test_cabi_refuses_before_device():
    """svtgpu_ewise applies the same rules (the checks run before it asks for
    a device, so an invalid operand is an argument error everywhere)."""
    L = _native.lib()
    for nm in ("abs", "log1p", "*", "/"):
        assert _native.EW_OPCODES[nm] > 0
    assert "svtgpu_ewise" in _native.SIGNATURES
    assert L.svtgpu_ewise(None, 1, None, _native.DOUBLE, 1, 0, 0,
                          ctypes.byref(ctypes.c_void_p()),
                          ctypes.byref(ctypes.c_int())) == _native.ERR_ARG


@pytest.mark.skipif(_native.device_count() > 0, reason="needs a GPU-less box")
def test_valid_call_without_device_fails_loudly():
    x = _x()
    with pytest.raises(rshim.RError, match="no usable CUDA device"):
        sa.Math(x, "sqrt")
    with pytest.raises(rshim.RError, match="no usable CUDA device"):
        x * 2
    with pytest.raises(rshim.RError, match="no usable CUDA device"):
        sa.sweep(x, 2, np.arange(1, 5, dtype=np.float64), "/")
