"""colMedians() / rowMedians() on the device, bit-exact against base R's
median() of every dense column or row (ref_colmedians in
tests/test_medians_host.py): every input kind with na.rm both ways, NA and
NaN, the zero block, extreme values, tiny and empty extents, long leaves,
resident handles and derived matrices, column shards, the compact copy, and
a matrix above 2^31 nonzeros where every column needs selection."""
import ctypes

import numpy as np
import pytest

import sparsearray_b200 as sa
from sparsearray_b200 import _native, sharded, synth
from test_medians_host import assert_bit_exact, ref_colmedians, ref_median

pytestmark = pytest.mark.gpu

NA_I = -2**31
INT_MAX = 2**31 - 1
NA_R = sa.NA_REAL
DBL_MAX = np.finfo(np.float64).max
KINDS = ["integer", "double", "logical", "lacunar"]


def make_input(kind, nrow=1500, ncol=64, seed=1):
    """Signed values with per-column densities from 0.02 to 1, so medians
    fall among the negatives, in the zero block and among the positives;
    column 5 is empty, column 7 fully stored, column 9 one repeated value."""
    rng = np.random.Generator(np.random.PCG64(seed))
    dens = np.linspace(0.02, 1.0, ncol)
    mask = rng.random((nrow, ncol)) < dens
    mask[:, 5] = False
    mask[:, 7] = True
    mask[:, 9] = rng.random(nrow) < 0.8
    # the share of negatives varies too
    negshare = np.linspace(0.0, 1.0, ncol)[rng.permutation(ncol)]
    sign = np.where(rng.random((nrow, ncol)) < negshare, -1, 1)
    if kind == "double":
        a = np.where(mask, sign * np.round(rng.exponential(3.0, (nrow, ncol)),
                                           rng.integers(0, 4)), 0.0)
        a[mask & (a == 0)] = 0.25
        a[:, 9] = np.where(mask[:, 9], 2.5, 0.0)
        return sa.SVT_SparseArray.from_dense(a, "double"), a
    if kind in ("logical", "lacunar"):
        a = mask.astype(np.int32)
        if kind == "logical":
            a[3, 11] = NA_I
            a[0, 12] = NA_I
        return sa.SVT_SparseArray.from_dense(a, "logical"), a
    a = np.where(mask, sign * rng.integers(1, 9, (nrow, ncol)), 0) \
        .astype(np.int32)
    a[:, 9] = np.where(mask[:, 9], 3, 0)
    a[2, 13] = NA_I
    return sa.SVT_SparseArray.from_dense(a, "integer"), a


def check(x, dense, type_, na_rm):
    assert_bit_exact(sa.colMedians(x, na_rm=na_rm),
                     ref_colmedians(dense, type_, na_rm))
    assert_bit_exact(sa.rowMedians(x, na_rm=na_rm),
                     ref_colmedians(np.asarray(dense).T, type_, na_rm))


@pytest.mark.parametrize("na_rm", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_kinds(kind, na_rm):
    x, a = make_input(kind)
    t = "double" if kind == "double" else "integer"
    check(x, a, t, na_rm)
    # negated integers through the device (x * -1L)
    if kind == "integer":
        y = sa.Arith(sa.to_device(x), "*", np.array([-1], np.int32))
        neg = np.where(a == NA_I, NA_I, -a).astype(np.int32)
        check(y, neg, "integer", na_rm)


def _csc(nrow, cols, type_):
    """An SVT from explicit columns (stored zeros kept as given)."""
    ptr = np.zeros(len(cols) + 1, np.int64)
    offs, vals = [], []
    for j, (rows, v) in enumerate(cols):
        ptr[j + 1] = ptr[j] + len(rows)
        offs += list(rows)
        vals += list(v)
    dt = np.float64 if type_ == "double" else np.int32
    x = sa.SVT_SparseArray((nrow, len(cols)), type_, ptr,
                           np.array(offs, np.int32), np.array(vals, dt))
    dense = np.zeros((nrow, len(cols)), dt)
    for j, (rows, v) in enumerate(cols):
        dense[list(rows), j] = v
    return x, dense


@pytest.mark.parametrize("na_rm", [False, True])
def test_edges_double(na_rm):
    nan2 = np.array([0x7FF8000000000123], np.uint64).view(np.float64)[0]
    cols = [
        ([0, 1], [NA_R, 1.0]),                   # NA alone
        ([0, 1], [np.nan, 1.0]),                 # NaN alone
        ([0, 1, 2], [NA_R, nan2, 3.0]),          # both
        ([0, 1, 2, 3], [0.0, -0.0, 0.0, -0.0]),  # stored zeros only
        ([0, 1, 2, 3], [-0.0, -0.0, 5.0, 7.0]),  # -0 and positives
        ([0, 1, 2, 3], [DBL_MAX, DBL_MAX, DBL_MAX, DBL_MAX]),
        ([0, 1, 2, 3], [-DBL_MAX, -DBL_MAX, -DBL_MAX, -DBL_MAX]),
        ([0, 1, 2, 3], [-DBL_MAX, -DBL_MAX, DBL_MAX, DBL_MAX]),
        ([0, 1, 2, 3], [-np.inf, -np.inf, np.inf, np.inf]),
        ([0, 1, 2, 3], [np.inf, np.inf, np.inf, 1.0]),
        ([0, 1, 2, 3], [5e-324, 5e-324, 1.5e-323, 1e-323]),
        ([0, 1, 2, 3], [-1.0, -2.0, -3.0, -4.0]),
        ([1, 2], [-3.0, 5.0]),
        ([], []),
    ]
    x, a = _csc(4, cols, "double")
    check(x, a, "double", na_rm)


@pytest.mark.parametrize("na_rm", [False, True])
def test_edges_integer(na_rm):
    cols = [
        ([0, 1], [INT_MAX, INT_MAX]),
        ([0, 1], [-INT_MAX, -INT_MAX]),
        ([0, 1], [-INT_MAX, INT_MAX]),
        ([0, 1, 2, 3], [INT_MAX, INT_MAX - 1, INT_MAX, INT_MAX - 1]),
        ([0, 1, 2, 3], [0, 0, 0, 4]),            # stored zeros
        ([0, 3], [NA_I, 2]),
        ([0, 1, 2, 3], [NA_I, NA_I, NA_I, NA_I]),
        ([0, 1, 2, 3], [-2, -2, -2, -2]),
        ([0, 1, 2], [-5, -1, 6]),
        ([], []),
    ]
    x, a = _csc(4, cols, "integer")
    check(x, a, "integer", na_rm)


@pytest.mark.parametrize("nrow", [0, 1, 2])
def test_tiny_extents(nrow):
    rng = np.random.Generator(np.random.PCG64(nrow))
    a = rng.integers(-2, 3, (nrow, 7)).astype(np.int32)
    x = sa.SVT_SparseArray.from_dense(a, "integer")
    for na_rm in (False, True):
        check(x, a, "integer", na_rm)
    d = sa.SVT_SparseArray.from_dense(np.zeros((5, 0)), "double")
    assert np.asarray(sa.colMedians(d)).size == 0
    assert_bit_exact(sa.rowMedians(d), [NA_R] * 5)


def test_heavy_ties_and_long_leaves():
    """Leaves far longer than a CTA pass (and any staging size), ties
    everywhere, middles at bucket edges of every radix round."""
    rng = np.random.Generator(np.random.PCG64(5))
    nrow = 300_000
    a = np.zeros((nrow, 6), np.int32)
    a[:, 0] = rng.integers(1, 4, nrow)                     # ties
    a[:, 1] = rng.integers(-3_000_000, 3_000_000, nrow)   # wide range
    a[:, 2] = np.where(rng.random(nrow) < 0.55, rng.integers(1, 2**31 - 1,
                                                             nrow), 0)
    a[:, 3] = np.where(rng.random(nrow) < 0.7, -2048 * rng.integers(1, 5,
                                                                    nrow), 0)
    a[:, 4] = np.where(rng.random(nrow) < 0.5, 2047, 2049)
    a[:, 5] = -rng.integers(1, 2**31 - 1, nrow)
    x = sa.SVT_SparseArray.from_dense(a, "integer")
    assert_bit_exact(sa.colMedians(x), ref_colmedians(a, "integer", False))
    d = a.astype(np.float64) * np.array([0.1, 1e-300, 3.5, 1e300, -0.25, 7])
    xd = sa.SVT_SparseArray.from_dense(d, "double")
    assert_bit_exact(sa.colMedians(xd), ref_colmedians(d, "double", False))
    # a row of 1e5 columns: one leaf of the transpose
    b = np.where(rng.random((3, 100_000)) < 0.9,
                 rng.standard_normal((3, 100_000)), 0.0)
    xb = sa.SVT_SparseArray.from_dense(b, "double")
    assert_bit_exact(sa.rowMedians(xb), ref_colmedians(b.T, "double", False))


def test_compare_result_median_is_one_half():
    a = np.zeros((10, 3), np.int32)
    a[:5, 0] = 4                 # x > 0: five TRUE, five FALSE -> 0.5
    a[:6, 1] = 1                 # 0.6 stored share -> 1
    a[:4, 2] = -1                # no TRUE -> 0
    r = sa.Compare(sa.to_device(sa.SVT_SparseArray.from_dense(a)), ">", 0)
    assert_bit_exact(sa.colMedians(r), [0.5, 1.0, 0.0])
    assert_bit_exact(sa.rowMedians(r), ref_colmedians((a > 0).T.astype(
        np.int32), "integer", False))


@pytest.mark.parametrize("kind", ["integer", "double", "lacunar"])
def test_resident_and_names(kind):
    x0, a = make_input(kind, seed=3)
    t = "double" if kind == "double" else "integer"
    dn = (["r%d" % i for i in range(a.shape[0])],
          ["c%d" % j for j in range(a.shape[1])])
    x = sa.SVT_SparseArray.from_dense(a, x0.type, dimnames=dn)
    h = sa.to_device(x)
    for na_rm in (False, True):
        c, ch = sa.colMedians(x, na_rm=na_rm), sa.colMedians(h, na_rm=na_rm)
        assert_bit_exact(ch, c)
        assert list(c.names) == dn[1]
        r, rh = sa.rowMedians(x, na_rm=na_rm), sa.rowMedians(h, na_rm=na_rm)
        assert_bit_exact(rh, r)
        assert_bit_exact(rh, ref_colmedians(a.T, t, na_rm))
        assert list(r.names) == dn[0]
    assert sa.colMedians(x, useNames=False).names is None
    # from_csc handles
    p, o, v = x.ptr, x.offs, x.vals
    if v is not None:
        hc = sa.from_csc(a.shape, p, v, o)
        assert_bit_exact(sa.colMedians(hc), ref_colmedians(a, t, False))


def test_row_medians_equal_col_medians_of_transpose():
    x, a = make_input("double", nrow=700, ncol=900, seed=8)
    xt = sa.SVT_SparseArray.from_dense(np.ascontiguousarray(a.T), "double")
    for na_rm in (False, True):
        assert_bit_exact(sa.rowMedians(x, na_rm=na_rm),
                         sa.colMedians(xt, na_rm=na_rm))


def test_column_shards_and_device_results():
    from sparsearray_b200.device import DeviceSVT, plan_column_shards
    x, a = make_input("integer", ncol=90, seed=4)
    whole = DeviceSVT.from_host(x)
    for na_rm in (False, True):
        ref = ref_colmedians(a, "integer", na_rm)
        assert_bit_exact(whole.colmedians(na_rm=na_rm).cpu().numpy(), ref)
        parts = [DeviceSVT.from_host(x, r).colmedians(na_rm=na_rm)
                 .cpu().numpy() for r in plan_column_shards(90, 4, x.ptr)]
        assert_bit_exact(np.concatenate(parts), ref)
        assert_bit_exact(whole.rowmedians(na_rm=na_rm),
                         ref_colmedians(a.T, "integer", na_rm))
        assert_bit_exact(sharded.colMedians(x, na_rm=na_rm), ref)
    with pytest.raises(ValueError, match="does not compose"):
        DeviceSVT.from_host(x, (0, 30)).rowmedians()
    # derived handles: ewise results of a shard
    y = whole.ewise("*", np.array([-3], np.int32))
    neg = np.where(a == NA_I, NA_I, -3 * a).astype(np.int32)
    assert_bit_exact(y.colmedians().cpu().numpy(),
                     ref_colmedians(neg, "integer", False))


def test_unchanged_after_compact_copy():
    from sparsearray_b200.device import DeviceSVT
    x, a = make_input("integer", seed=6)
    d = DeviceSVT.from_host(x)
    before = [d.colmedians(na_rm=r).cpu().numpy() for r in (False, True)]
    for _ in range(3):
        d.colstats("sum")
    nb = ctypes.c_int64(0)
    _native.check(_native.lib().svtgpu_matrix_compact_bytes(
        d._h, ctypes.byref(nb)))
    assert nb.value > 0
    for r, b in zip((False, True), before):
        assert_bit_exact(d.colmedians(na_rm=r).cpu().numpy(), b)
        assert_bit_exact(b, ref_colmedians(a, "integer", r))


# ---- at scale ---------------------------------------------------------------

NROW, NCOL, DENS, SEED = 33538, 110_000, 0.6, 11


def _release():
    import gc
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    _native.lib().svtgpu_release_cached_memory()


def test_scale_above_2_31_every_column_selected():
    from sparsearray_b200.device import DeviceSVT
    x = DeviceSVT.generate_poisson(NROW, NCOL, DENS, seed=SEED, na_rate=1e-6)
    assert x.nnz > 2**31
    out = np.zeros(NCOL)
    for na_rm in (True, False):
        _native.check(_native.lib().svtgpu_colmedians(
            x._h, int(na_rm), out.ctypes.data_as(ctypes.c_void_p)))
        sel = x.median_selected()[0]
        if na_rm:
            assert sel == NCOL                   # every column selects
            res_rm = out.copy()
    res = out.copy()
    dev = x.colmedians(na_rm=True).cpu().numpy()
    assert_bit_exact(dev, res_rm)
    ptr = x.leaf_ptr.cpu().numpy()
    l31 = int(np.searchsorted(ptr, 2**31, side="right")) - 1
    rng = np.random.Generator(np.random.PCG64(23))
    leaves = sorted({0, NCOL - 1, l31} |
                    set(int(v) for v in rng.integers(0, NCOL, 2000)))
    for l in leaves:
        p, o, v = synth.poisson_csc(NROW, 1, DENS, seed=SEED, na_rate=1e-6,
                                    leaf0=l)
        col = np.zeros(NROW, np.int32)
        col[o] = v
        for na_rm, got in ((True, res_rm), (False, res)):
            assert_bit_exact([got[l]], [ref_median(col, "integer", na_rm)])
    rows = x.rowmedians(na_rm=True)
    for i in sorted(set(int(v) for v in rng.integers(0, NROW, 150))):
        c, v, na = synth.poisson_row(NROW, NCOL, i, DENS, seed=SEED,
                                     na_rate=1e-6)
        row = np.zeros(NCOL, np.int32)
        row[c] = np.where(na, NA_I, v)
        assert_bit_exact([rows[i]], [ref_median(row, "integer", True)])
    del x
    _release()


def test_c2_medians_are_zero_without_selection():
    from sparsearray_b200.device import DeviceSVT
    x = DeviceSVT.generate_poisson(33538, 1_000_000, 0.07, seed=2,
                                   na_rate=1e-6)
    assert x.nnz > 2**31
    out = np.full(1_000_000, 7.0)
    _native.check(_native.lib().svtgpu_colmedians(
        x._h, 1, out.ctypes.data_as(ctypes.c_void_p)))
    assert x.median_selected() == (0, 0)
    assert np.all(out == 0.0) and not np.any(np.signbit(out))
    del x
    _release()
