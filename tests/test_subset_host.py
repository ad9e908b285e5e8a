"""`x[i, j, ...]` without a GPU: the numpy oracle (tests/subset_oracle.py)
and the conversion of numpy-style keys held to numpy's `a[np.ix_(...)]` on
hand-written keys; every refusal of C_svtgpu_subset_SVT with its message;
registration; the C ABI's range checks before any device work."""
import ctypes

import numpy as np
import pytest

import subset_oracle
import sparsearray_b200 as sa
from sparsearray_b200 import _native, rcall
from sparsearray_b200.rcall import rshim
from sparsearray_b200.svt import _numpy_key_to_subscript

NA_I = -2**31
NO_DEVICE = "no usable CUDA device"


def _dense(shape=(7, 6), seed=1):
    rng = np.random.Generator(np.random.PCG64(seed))
    a = np.where(rng.random(shape) < 0.4, rng.integers(-5, 6, shape), 0)
    return a.astype(np.int32)


KEYS = [
    (slice(None), slice(None)),
    ([3, 3, 0, 6, 3], slice(None)),                # duplicates
    (slice(None, None, -1), [5, 4, 3, 2, 1, 0]),   # reversed
    ([], slice(None)),                             # empty
    (slice(None), []),
    (slice(1, 7, 2), slice(None, None, 3)),        # slices with steps
    (np.array([True, False, True, True, False, False, True]),
     np.array([False, True, True, False, False, True])),
    ([-1, 0, -7], [2, -6, 2]),
    (4, 0),                                        # ints keep the dimension
    ([1, 2, 2, 5], [5, 5, 0]),
]


def _ix(a, key):
    sub = [np.arange(n)[k] if not isinstance(k, (int, np.integer))
           else np.array([k % n]) for k, n in zip(key, a.shape)]
    return a[np.ix_(*[np.atleast_1d(s) for s in sub])]


def _nindex(key, shape):
    return [_numpy_key_to_subscript(k, n) for k, n in zip(key, shape)]


@pytest.mark.parametrize("key", KEYS, ids=range(len(KEYS)))
def test_oracle_and_key_conversion_match_numpy(key):
    a = _dense()
    x = sa.SVT_SparseArray.from_dense(a, lacunar=False)
    nidx = _nindex(key, a.shape)
    rows = None if nidx[0] is None else nidx[0] - 1
    cols = None if nidx[1] is None else nidx[1] - 1
    p, o, v = subset_oracle.subset(a.shape[0], *subset_oracle.csc_of(x),
                                   rows, cols)
    want = _ix(a, key)
    got = sa.SVT_SparseArray(want.shape, "integer", p, o, v).to_dense()
    assert np.array_equal(got, want)


def test_oracle_on_nd_arrays_and_lacunar_input():
    rng = np.random.Generator(np.random.PCG64(4))
    a = (rng.random((6, 4, 3)) < 0.4).astype(np.int32)
    x = sa.SVT_SparseArray.from_dense(a, "logical")
    assert x.vals is None
    i, j, k = [4, 0, 0], [3, 1], [2, 0, 1, 2]
    leaves = [jj + 4 * kk for kk in k for jj in j]   # column-major product
    p, o, v = subset_oracle.subset(6, *subset_oracle.csc_of(x), i, leaves)
    assert v is None
    want = a[np.ix_(i, j, k)]
    got = sa.SVT_SparseArray(want.shape, "logical", p, o, None).to_dense()
    assert np.array_equal(got, want)


def test_key_conversion_refusals():
    with pytest.raises(IndexError, match="out of bounds"):
        _numpy_key_to_subscript(7, 7)
    with pytest.raises(IndexError, match="out of bounds"):
        _numpy_key_to_subscript([0, -8], 7)
    with pytest.raises(IndexError, match="does not match"):
        _numpy_key_to_subscript(np.ones(6, bool), 7)
    with pytest.raises(IndexError, match="integers or booleans"):
        _numpy_key_to_subscript(np.array([1.0]), 7)
    with pytest.raises(IndexError, match="1-D"):
        _numpy_key_to_subscript(np.zeros((2, 2), int), 7)
    assert _numpy_key_to_subscript(slice(None), 7) is None
    assert _numpy_key_to_subscript(slice(0, 7), 7) is None
    assert list(_numpy_key_to_subscript(slice(None, None, -1), 3)) == [3, 2, 1]
    x = sa.SVT_SparseArray.from_dense(_dense())
    with pytest.raises(IndexError, match="too many indices"):
        x[0, 0, 0]


# ---- refusals of the entry point, raised before any device work -----------

def _call(x, nidx_robj):
    try:
        return rcall.SparseArray_Call("C_svtgpu_subset_SVT", x.r_dim,
                                      x.r_type, x.r_SVT, nidx_robj)
    finally:
        nidx_robj.release()


def _x():
    return sa.SVT_SparseArray.from_dense(_dense())


def test_refusals_and_their_messages():
    x = _x()
    wrong = r"'Nindex' must be a list with one element per dimension"
    with pytest.raises(rshim.RError, match=wrong):
        _call(x, rshim.integer([1, 2]))
    with pytest.raises(rshim.RError, match=wrong):
        sa.subset(x, [None])
    with pytest.raises(rshim.RError, match=wrong):
        sa.subset(x, [None, None, None])
    with pytest.raises(rshim.RError, match=wrong):
        sa.subset(x, "a")
    notint = r"subscript 2 of 'Nindex' must be NULL or an integer vector"
    with pytest.raises(rshim.RError, match=notint):
        sa.subset(x, [None, np.array([1.0])])
    with pytest.raises(rshim.RError, match=notint):
        sa.subset(x, [None, np.array([True, False])])
    with pytest.raises(rshim.RError, match=r"^subscript contains NAs$"):
        sa.subset(x, [np.array([1, NA_I], np.int32), None])
    with pytest.raises(rshim.RError,
                       match=r"^subscript contains out-of-bounds indices$"):
        sa.subset(x, [np.array([8]), None])
    with pytest.raises(rshim.RError,
                       match=r"^subscript contains out-of-bounds indices$"):
        sa.subset(x, [None, np.array([0])])
    with pytest.raises(rshim.RError,
                       match=r"^subscript contains out-of-bounds indices$"):
        sa.subset(x, [None, np.array([-1])])
    c = sa.SVT_SparseArray.from_dense(_dense())
    t = rshim.string("complex")
    try:
        with pytest.raises(rshim.RError, match=r'type\(\) "complex" are not'):
            rcall.SparseArray_Call("C_svtgpu_subset_SVT", c.r_dim, t, c.r_SVT,
                                   rshim.rlist([None, None]))
    finally:
        t.release()


def test_entry_point_registered_with_its_arity():
    assert rcall.registered_routines()["C_svtgpu_subset_SVT"] == 4


class _MatrixHead(ctypes.Structure):
    """The leading fields of struct svtgpu_matrix (svtgpu_internal.h): all
    that svtgpu_subset() reads before it asks for a device."""
    _fields_ = [("nrow", ctypes.c_int64), ("nleaf", ctypes.c_int64),
                ("nnz", ctypes.c_int64), ("val_type", ctypes.c_int),
                ("flags", ctypes.c_int), ("pad", ctypes.c_char * 4096)]


def _subset(x, rows, leaves, n_rows=None, n_leaves=None):
    r = None if rows is None else np.asarray(rows, np.int32)
    l = None if leaves is None else np.asarray(leaves, np.int64)
    out = ctypes.c_void_p()
    return _native.lib().svtgpu_subset(
        None if x is None else ctypes.byref(x),
        None if r is None else r.ctypes.data_as(ctypes.c_void_p),
        (0 if r is None else r.size) if n_rows is None else n_rows,
        None if l is None else l.ctypes.data_as(ctypes.c_void_p),
        (0 if l is None else l.size) if n_leaves is None else n_leaves,
        ctypes.byref(out))


def test_cabi_refuses_bad_ranges_before_device():
    L = _native.lib()
    x = _MatrixHead(5, 4, 0, _native.INT, 0)
    for rows, leaves, what in (([5], None, "row subscript"),
                               ([-1], None, "row subscript"),
                               (None, [4], "leaf subscript"),
                               (None, [0, -2], "leaf subscript")):
        assert _subset(x, rows, leaves) == _native.ERR_ARG
        assert what in L.svtgpu_last_error().decode()
    assert _subset(x, [0], None, n_rows=-1) == _native.ERR_ARG
    assert _subset(x, None, [0], n_leaves=-1) == _native.ERR_ARG
    assert _subset(x, None, [0], n_leaves=2**31) == _native.ERR_UNSUPPORTED
    assert "2^31 - 2 result leaves" in L.svtgpu_last_error().decode()
    c = _MatrixHead(5, 4, 0, 15, 0)                 # complex
    assert _subset(c, None, None) == _native.ERR_ARG
    assert _subset(None, None, None) == _native.ERR_ARG


@pytest.mark.skipif(_native.device_count() > 0, reason="needs a GPU-less box")
def test_valid_call_without_device_fails_loudly():
    x = _x()
    for call in (lambda: x[[1, 0], 2:], lambda: x[:, [True] * 6],
                 lambda: sa.subset(x, [None, None]),
                 lambda: sa.subset(x, [np.array([7, 1]), np.array([2])])):
        with pytest.raises(rshim.RError, match=NO_DEVICE):
            call()
    a = _MatrixHead(5, 4, 0, _native.INT, 0)
    assert _subset(a, [4, 0], [3]) == _native.ERR_NO_DEVICE
    assert _subset(a, None, None) == _native.ERR_NO_DEVICE
