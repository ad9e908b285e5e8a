"""colMedians() / rowMedians() without a GPU: the median rules of
svt_semantics.h (plan from counts, midpoint, order-preserving keys) compiled
for the host and held to numpy, the registration of the .Call entry points,
their R errors, and the failure without a device.

`ref_colmedians` below is the reference the GPU tests hold the device to:
base R's median() of every dense column, written from its definition with
np.partition (not np.median, whose midpoint and NaN rules differ)."""
import ctypes
import fractions
import os
import subprocess
import tempfile

import numpy as np
import pytest

import sparsearray_b200 as sa
from sparsearray_b200 import _native, rcall
from sparsearray_b200.rcall import rshim

NA_I = -2**31
INT_MAX = 2**31 - 1
NA_R = sa.NA_REAL
DBL_MAX = np.finfo(np.float64).max
DENORM = 5e-324
HERE = os.path.dirname(os.path.abspath(__file__))
NO_DEVICE = "no usable CUDA device"
MED_NA, MED_ZERO, MED_SELECT = 0, 1, 2
NEG, POS = 0, 1
SECOND_NONE, SECOND_ZERO, SECOND_NEXT = 0, 1, 2


# ---- the reference ---------------------------------------------------------

def _bits(x):
    return np.float64(x).view(np.uint64)


def ref_mid(a, b):
    """Correctly rounded (a + b) / 2 of two doubles: (a + b) / 2 when the sum
    is finite, a/2 + b/2 when it overflows; -Inf and +Inf give NaN."""
    with np.errstate(all="ignore"):
        s = np.float64(a) + np.float64(b)
        if np.isnan(s):
            return np.float64(np.nan)
        if np.isinf(s) and np.isfinite(a) and np.isfinite(b):
            return np.float64(a) / 2 + np.float64(b) / 2
        return s / 2


def ref_median(v, type_, na_rm):
    """median(v, na.rm) of one dense column (int32 with NA_integer_, or
    float64 with NA_real_ / NaN) as a double."""
    v = np.asarray(v)
    if type_ == "double":
        miss = np.isnan(v)
        vals = v[~miss].astype(np.float64)
    else:
        miss = v == NA_I
        vals = v[~miss].astype(np.float64)
    if miss.any() and not na_rm:
        return NA_R
    n = vals.size
    if n == 0:
        return NA_R
    lo, hi = (n - 1) // 2, n // 2
    part = np.partition(vals, [lo, hi])
    r = part[lo] if lo == hi else ref_mid(part[lo], part[hi])
    return np.float64(r) + 0.0       # a zero median is +0


def ref_colmedians(dense, type_, na_rm):
    """Column medians of a dense nrow x ncol matrix (logical as 0 / 1)."""
    dense = np.asarray(dense)
    out = np.empty(dense.shape[1], dtype=np.float64)
    for j in range(dense.shape[1]):
        out[j] = ref_median(dense[:, j], type_, na_rm)
    return out


def assert_bit_exact(got, want):
    """Bit-exact, except that a NaN result only has to be NaN and not NA."""
    got = np.asarray(got, dtype=np.float64).reshape(-1)
    want = np.asarray(want, dtype=np.float64).reshape(-1)
    assert got.shape == want.shape
    wna = sa.is_na_real(want)
    wnan = np.isnan(want) & ~wna
    assert np.array_equal(sa.is_na_real(got), wna)
    assert np.array_equal(np.isnan(got) & ~sa.is_na_real(got), wnan)
    ok = ~np.isnan(want)
    bad = np.flatnonzero(got[ok].view(np.uint64) != want[ok].view(np.uint64))
    assert bad.size == 0, "first mismatches at %s: got %r, want %r" % (
        np.flatnonzero(ok)[bad[:5]], got[ok][bad[:5]], want[ok][bad[:5]])


# ---- the rules compiled for the host ---------------------------------------

@pytest.fixture(scope="module")
def sem():
    tmp = tempfile.TemporaryDirectory(prefix="medians_host_")
    so = os.path.join(tmp.name, "libmedians_host.so")
    subprocess.check_call(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared",
                           "-o", so, os.path.join(HERE, "medians_host.c"),
                           "-lm"])
    L = ctypes.CDLL(so)
    c = ctypes
    L.plan_host.argtypes = [c.c_int64] * 4 + [c.c_int] + \
        [c.POINTER(c.c_int)] * 3 + [c.POINTER(c.c_int64)]
    L.plan_host.restype = None
    L.mid_host.argtypes = [c.c_double, c.c_double]
    L.mid_host.restype = c.c_double
    L.key_i32_host.argtypes = [c.c_int32, c.POINTER(c.c_uint32)]
    L.key_i32_host.restype = c.c_int
    L.unkey_i32_host.argtypes = [c.c_uint32]
    L.unkey_i32_host.restype = c.c_int32
    L.key_f64_host.argtypes = [c.c_double, c.POINTER(c.c_uint64)]
    L.key_f64_host.restype = c.c_int
    L.unkey_f64_host.argtypes = [c.c_uint64]
    L.unkey_f64_host.restype = c.c_double
    yield L
    tmp.cleanup()


def plan(L, nrow, nneg, npos, nna, narm):
    k, s, sec, r = (ctypes.c_int(), ctypes.c_int(), ctypes.c_int(),
                    ctypes.c_int64())
    L.plan_host(nrow, nneg, npos, nna, int(narm), ctypes.byref(k),
                ctypes.byref(s), ctypes.byref(sec), ctypes.byref(r))
    return k.value, s.value, sec.value, r.value


def key(L, x, type_):
    if type_ == "double":
        k = ctypes.c_uint64()
        ok = L.key_f64_host(float(x), ctypes.byref(k))
    else:
        k = ctypes.c_uint32()
        ok = L.key_i32_host(int(x), ctypes.byref(k))
    return k.value if ok else None


def unkey(L, k, type_):
    return L.unkey_f64_host(k) if type_ == "double" else \
        float(L.unkey_i32_host(k))


def median_by_rules(L, col, type_, na_rm):
    """What the kernels compute for one column with nrow = len(col): counts
    -> plan; a selection sorts the side's keys and takes the rank; NEXT is
    the smallest stored nonzero key above the first."""
    col = np.asarray(col)
    keys = [key(L, x, type_) for x in col]
    vals = col.astype(np.float64)
    neg = [k for k, x in zip(keys, vals) if k is not None and x < 0]
    pos = [k for k, x in zip(keys, vals) if k is not None and x > 0]
    nna = sum(k is None for k in keys)
    kind, side, second, rank = plan(L, len(col), len(neg), len(pos), nna,
                                    na_rm)
    if kind == MED_NA:
        return NA_R
    if kind == MED_ZERO:
        return 0.0
    s = sorted(neg if side == NEG else pos)
    a = s[rank]
    va = unkey(L, a, type_)
    if second == SECOND_NONE:
        return va
    if second == SECOND_ZERO:
        return L.mid_host(va, 0.0)
    b = min(k for k in neg + pos if k > a) if rank + 1 >= len(s) or \
        s[rank + 1] != a else a
    return L.mid_host(va, unkey(L, b, type_))


# (R expression, column, type): each column's median as R prints it is in the
# comment; the tests hold the rules to ref_median on all of them
VECTORS = [
    # median(c(0L, 0L, 3L)) = 0: the middle rank is a zero
    ([0, 0, 3], "integer"),
    # median(c(-5L, -2L, 0L, 7L)) = -1: -2 and 0 straddle neg / zero
    ([-5, -2, 0, 7], "integer"),
    # median(c(-5L, 0L, 4L, 7L)) = 2: 0 and 4 straddle zero / pos
    ([-5, 0, 4, 7], "integer"),
    # median(c(-3L, 5L)) = 1: -3 and 5, no zeros between the sides
    ([-3, 5], "integer"),
    # median(c(-3L, -1L, 2L)) = -1: odd, last negative
    ([-3, -1, 2], "integer"),
    # median(c(-9L, -7L, -3L, -1L, 0L)) = -3: odd, inside the negatives
    ([-9, -7, -3, -1, 0], "integer"),
    # median(c(0L, 1L, 2L, 3L, 4L, 5L)) = 2.5: even, inside the positives
    ([0, 1, 2, 3, 4, 5], "integer"),
    # median(c(2L, 2L, 2L, 9L)) = 2: ties
    ([2, 2, 2, 9], "integer"),
    # median(c(1L, NA, 3L)) = NA; with na.rm = TRUE 2
    ([1, NA_I, 3], "integer"),
    # median(c(NA_integer_, NA)) = NA either way (nothing left)
    ([NA_I, NA_I], "integer"),
    # median(c(2147483647L, 2147483647L)) = 2147483647
    ([INT_MAX, INT_MAX], "integer"),
    # median(c(-2147483647L, 2147483647L)) = 0
    ([-INT_MAX, INT_MAX], "integer"),
    # median(c(2147483646L, 2147483647L)) = 2147483646.5 (exact in double)
    ([INT_MAX - 1, INT_MAX], "integer"),
    # median(c(.Machine$double.xmax, .Machine$double.xmax)) = 1.797693e+308
    # (a + b overflows: a/2 + b/2)
    ([DBL_MAX, DBL_MAX], "double"),
    # median(c(-.Machine$double.xmax, -.Machine$double.xmax, 1)) = -xmax
    ([-DBL_MAX, -DBL_MAX, 1.0], "double"),
    # median(c(-.Machine$double.xmax, .Machine$double.xmax)) = 0
    ([-DBL_MAX, DBL_MAX], "double"),
    # median(c(-Inf, Inf)) = NaN (not NA)
    ([-np.inf, np.inf], "double"),
    # median(c(-Inf, 0, 0, 1, Inf)) = 0
    ([-np.inf, 0.0, 0.0, 1.0, np.inf], "double"),
    # median(c(Inf, Inf, 0)) = Inf
    ([np.inf, np.inf, 0.0], "double"),
    # median(c(-Inf, 1)) = -Inf
    ([-np.inf, 1.0], "double"),
    # median(c(-0, -0, 5)) = 0 (+0, never -0)
    ([-0.0, -0.0, 5.0], "double"),
    # median(c(-1, -0)) = -0.5
    ([-1.0, -0.0], "double"),
    # median(c(4.9e-324, 0)) = 0 (the halved denormal rounds to even)
    ([DENORM, 0.0], "double"),
    # median(c(4.9e-324, 1.5e-323)) = 9.9e-324
    ([DENORM, 3 * DENORM], "double"),
    # median(c(NaN, 1)) = NA (never NaN); na.rm = TRUE: 1
    ([np.nan, 1.0], "double"),
    # median(c(NA, NaN, 2, 3)) = NA; na.rm = TRUE: 2.5
    ([NA_R, np.nan, 2.0, 3.0], "double"),
    # median(c(0.1, 0.2)) = 0.15 as (0.1 + 0.2) / 2
    ([0.1, 0.2], "double"),
    # median(c(-0.3, 0, 0, 0.7, 1e300)) = 0
    ([-0.3, 0.0, 0.0, 0.7, 1e300], "double"),
    # median(c(-2.5, -1e-300, 0)) = -1e-300
    ([-2.5, -1e-300, 0.0], "double"),
    # median(numeric(0)) = NA
    ([], "double"),
]


@pytest.mark.parametrize("na_rm", [False, True])
@pytest.mark.parametrize("i", range(len(VECTORS)))
def test_rules_match_reference(sem, i, na_rm):
    col, type_ = VECTORS[i]
    col = np.array(col, dtype=np.float64 if type_ == "double" else np.int32)
    assert_bit_exact([median_by_rules(sem, col, type_, na_rm)],
                     [ref_median(col, type_, na_rm)])


def test_reference_on_hand_vectors():
    """ref_median itself against the values R prints."""
    i32 = lambda v: np.array(v, dtype=np.int32)  # noqa: E731
    f64 = lambda v: np.array(v, dtype=np.float64)  # noqa: E731
    assert ref_median(i32([-5, -2, 0, 7]), "integer", False) == -1.0
    assert ref_median(i32([-3, 5]), "integer", False) == 1.0
    assert ref_median(i32([INT_MAX - 1, INT_MAX]), "integer", False) == \
        2147483646.5
    assert ref_median(f64([DBL_MAX, DBL_MAX]), "double", False) == DBL_MAX
    assert sa.is_na_real(ref_median(f64([np.nan, 1.0]), "double", False))
    assert ref_median(f64([np.nan, 1.0]), "double", True) == 1.0
    r = ref_median(f64([-np.inf, np.inf]), "double", False)
    assert np.isnan(r) and not sa.is_na_real(r)
    r = ref_median(f64([-0.0, -0.0, 5.0]), "double", False)
    assert r == 0.0 and not np.signbit(r)


@pytest.mark.parametrize("na_rm", [False, True])
def test_rules_on_random_columns(sem, na_rm):
    rng = np.random.Generator(np.random.PCG64(7))
    for t in range(300):
        n = int(rng.integers(0, 12))
        if t % 2:
            col = rng.choice(np.array([-3, -1, 0, 0, 0, 1, 2, 2, 5, NA_I],
                                      dtype=np.int32), n)
            type_ = "integer"
        else:
            col = rng.choice(np.array([-np.inf, -2.5, -0.0, 0.0, 0.0, 1e-310,
                                       0.5, 3.0, np.inf, np.nan]), n)
            type_ = "double"
        assert_bit_exact([median_by_rules(sem, col, type_, na_rm)],
                         [ref_median(col, type_, na_rm)])


def test_plan_straddles(sem):
    # 2 negatives, 3 zeros (nrow 7 - 4 stored), 2 positives: rank 3 is a zero
    assert plan(sem, 7, 2, 2, 0, False)[0] == MED_ZERO
    # nrow 4, values -5 -2 0 7: ranks 1, 2 = last negative and a zero
    assert plan(sem, 4, 2, 1, 0, False) == (MED_SELECT, NEG, SECOND_ZERO, 1)
    # nrow 4, values -5 0 4 7: ranks 1, 2 = a zero and the first positive
    assert plan(sem, 4, 1, 2, 0, False) == (MED_SELECT, POS, SECOND_ZERO, 0)
    # nrow 2, values -3 5: last negative, next is the first positive
    assert plan(sem, 2, 1, 1, 0, False) == (MED_SELECT, NEG, SECOND_NEXT, 0)
    # nrow 6, 0 1 2 3 4 5: ranks 2, 3 = positives 1 and 2 (in-side ranks)
    assert plan(sem, 6, 0, 5, 0, False) == (MED_SELECT, POS, SECOND_NEXT, 1)
    # odd: nrow 5, -9 -7 -3 -1 0 -> rank 2 of the negatives, one value
    assert plan(sem, 5, 4, 0, 0, False) == (MED_SELECT, NEG, SECOND_NONE, 2)
    # NA without na.rm; with na.rm the NA leaves n_eff = 2
    assert plan(sem, 3, 0, 2, 1, False)[0] == MED_NA
    assert plan(sem, 3, 0, 2, 1, True) == (MED_SELECT, POS, SECOND_NEXT, 0)
    # nothing left, and nrow 0
    assert plan(sem, 2, 0, 0, 2, True)[0] == MED_NA
    assert plan(sem, 0, 0, 0, 0, False)[0] == MED_NA
    # C2-like column: 33538 rows, 7 % stored -> the zeros decide
    assert plan(sem, 33538, 0, 2348, 3, True)[0] == MED_ZERO


def test_midpoint_is_correctly_rounded(sem):
    rng = np.random.Generator(np.random.PCG64(3))
    a = np.concatenate([rng.standard_normal(2000) * 10.0 **
                        rng.integers(-300, 308, 2000),
                        [DBL_MAX, -DBL_MAX, DBL_MAX * 0.75, DENORM,
                         3 * DENORM, 2.0**-1022, 1.0, -1.0]])
    b = np.concatenate([rng.standard_normal(2000) * 10.0 **
                        rng.integers(-300, 308, 2000),
                        [DBL_MAX, -DBL_MAX * 0.5, DBL_MAX, 0.0,
                         DENORM, 2.0**-1022 + DENORM, 1.0 + 2**-52, 3.0]])
    for x, y in zip(a, b):
        got = sem.mid_host(x, y)
        exact = (fractions.Fraction(float(x)) + fractions.Fraction(float(y))) \
            / 2
        assert _bits(got) == _bits(float(exact) + 0.0), (x, y)
        assert _bits(got) == _bits(ref_mid(x, y) + 0.0)
    # -Inf and +Inf: NaN, not NA; same-signed infinities stay
    r = sem.mid_host(-np.inf, np.inf)
    assert np.isnan(r) and not sa.is_na_real(r)
    assert sem.mid_host(np.inf, np.inf) == np.inf
    assert sem.mid_host(-np.inf, 5.0) == -np.inf
    # DBL_MAX + DBL_MAX overflows; the midpoint is DBL_MAX
    assert sem.mid_host(DBL_MAX, DBL_MAX) == DBL_MAX


def test_int_keys(sem):
    # NA_integer_ (INT_MIN) is not a key
    assert key(sem, NA_I, "integer") is None
    xs = [-INT_MAX, -70000, -1, 0, 1, 2, 65536, INT_MAX]
    ks = [key(sem, x, "integer") for x in xs]
    assert all(k is not None and k >= 1 for k in ks)
    assert ks == sorted(ks) and len(set(ks)) == len(ks)
    assert [unkey(sem, k, "integer") for k in ks] == [float(x) for x in xs]


def test_double_keys(sem):
    xs = [-np.inf, -DBL_MAX, -1.0, -2.0**-1022, -DENORM, -0.0, 0.0, DENORM,
          2.0**-1022 - DENORM, 2.0**-1022, 1.0, 1.0 + 2**-52, DBL_MAX, np.inf]
    ks = [key(sem, x, "double") for x in xs]
    assert all(k is not None for k in ks)
    assert all(a < b for a, b in zip(ks, ks[1:]))
    for x, k in zip(xs, ks):
        assert _bits(unkey(sem, k, "double")) == _bits(x)
    # neither NA nor any NaN is a key
    assert key(sem, NA_R, "double") is None
    assert key(sem, np.nan, "double") is None
    assert key(sem, -np.nan, "double") is None


# ---- registration, R errors, no device --------------------------------------

def _x(type_="integer"):
    a = np.array([[0, 3, 0, 1], [2, 0, 0, -4], [0, 5, 7, 0]])
    return sa.SVT_SparseArray.from_dense(
        a.astype(np.float64 if type_ == "double" else np.int32), type_)


def test_entry_points_registered_with_their_arity():
    r = rcall.registered_routines()
    assert r["C_colMedians_SVT"] == 5
    assert r["C_rowMedians_SVT"] == 5


def _raw(entry, x, na_rm, type_=None):
    t = [rshim.logical(na_rm) if isinstance(na_rm, list) else na_rm]
    ty = rshim.string(type_) if type_ is not None else None
    try:
        return rcall.SparseArray_Call(entry, x.r_dim, None,
                                      ty if ty is not None else x.r_type,
                                      x.r_SVT, t[0])
    finally:
        for o in t + ([ty] if ty is not None else []):
            o.release()


@pytest.mark.parametrize("entry", ["C_colMedians_SVT", "C_rowMedians_SVT"])
def test_r_errors(entry):
    x = _x()
    with pytest.raises(rshim.RError, match="'na.rm' must be TRUE or FALSE"):
        _raw(entry, x, rshim.integer([1]))
    with pytest.raises(rshim.RError, match="'na.rm' must be TRUE or FALSE"):
        _raw(entry, x, [1, 0])
    with pytest.raises(rshim.RError, match=r'type\(\) "complex" are not '
                       r'supported by the SparseArray GPU path'):
        _raw(entry, x, [0], type_="complex")
    with pytest.raises(rshim.RError, match="invalid 'x_type' value"):
        _raw(entry, x, [0], type_="matrix")
    a = np.zeros((2, 3, 2), dtype=np.int32)
    a[1, 2, 1] = 4
    x3 = sa.SVT_SparseArray.from_dense(a)
    fun = "colMedians" if "col" in entry else "rowMedians"
    with pytest.raises(rshim.RError, match=r"%s\(\): only matrices" % fun):
        _raw(entry, x3, [0])


def test_python_argument_checks():
    x = _x()
    with pytest.raises(ValueError, match="'na.rm' must be TRUE or FALSE"):
        sa.colMedians(x, na_rm=1)
    with pytest.raises(ValueError, match="'useNames' must be TRUE or FALSE"):
        sa.rowMedians(x, useNames="yes")
    with pytest.raises(TypeError):
        sa.colMedians(np.zeros((2, 2)))


def test_empty_extents_need_no_device():
    """ncol == 0 gives a length-0 result, nrow == 0 NA for every column
    (and the mirror for rows), decided before any device work."""
    e = sa.SVT_SparseArray.from_dense(np.zeros((0, 3), dtype=np.int32))
    assert_bit_exact(sa.colMedians(e), [NA_R] * 3)
    assert np.asarray(sa.rowMedians(e)).size == 0
    f = sa.SVT_SparseArray.from_dense(np.zeros((4, 0), dtype=np.float64),
                                      "double")
    assert np.asarray(sa.colMedians(f)).size == 0
    assert_bit_exact(sa.rowMedians(f, na_rm=True), [NA_R] * 4)


class _MatrixHead(ctypes.Structure):
    _fields_ = [("nrow", ctypes.c_int64), ("nleaf", ctypes.c_int64),
                ("nnz", ctypes.c_int64), ("val_type", ctypes.c_int),
                ("flags", ctypes.c_int), ("pad", ctypes.c_char * 4096)]


@pytest.mark.skipif(_native.device_count() > 0, reason="needs a GPU-less box")
def test_valid_call_without_device_fails_loudly():
    x = _x("double")
    for call in (lambda: sa.colMedians(x), lambda: sa.rowMedians(x),
                 lambda: sa.colMedians(x, na_rm=True)):
        with pytest.raises(rshim.RError, match=NO_DEVICE):
            call()
    L = _native.lib()
    m = _MatrixHead(3, 4, 0, _native.INT, 0)
    out = np.zeros(4)
    for fn in (L.svtgpu_colmedians, L.svtgpu_rowmedians):
        assert fn(ctypes.byref(m), 0, out.ctypes.data) == \
            _native.ERR_NO_DEVICE
    assert L.svtgpu_colmedians_dev(ctypes.byref(m), 0, out.ctypes.data,
                                   None) == _native.ERR_NO_DEVICE
