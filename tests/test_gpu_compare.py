"""Comparisons (x op v) and is.na / is.nan / is.infinite on the device
against base R's dense definition computed with numpy (tests/compare_ref.py):
structure and values of every result, its type and whether it carries a
value array; leaf and tile edges; the statistics run on the results; column
shards; and the benchmark's C2 matrix above 2^31 nonzeros."""
import ctypes

import numpy as np
import pytest

import compare_ref as cr
import sparsearray_b200 as sa
from sparsearray_b200 import _native, synth

pytestmark = pytest.mark.gpu

NA_I = -2**31
NA_R = sa.NA_REAL
OPS = cr.COMPARE
KINDS = ["integer", "logical", "double", "lacunar", "mixed"]
PREDS = ["is.na", "is.nan", "is.infinite"]


def make_input(kind, nrow=1500, ncol=60, seed=1, shape=None):
    """int / logical / double / lacunar / mixed SVT with NA, NaN, +-Inf,
    denormals and an empty leaf; more than one 32,768-entry tile."""
    rng = np.random.Generator(np.random.PCG64(seed))
    shape = shape or (nrow, ncol)
    mask = rng.random(shape) < 0.3
    mask.reshape(shape[0], -1, order="F")[:, 5] = False   # an empty leaf
    if kind == "double":
        a = np.where(mask, np.round(rng.standard_normal(shape) * 4, 1), 0.0)
        k = rng.integers(0, a.size, 80)
        a.reshape(-1)[k] = np.resize(
            [NA_R, np.nan, np.inf, -np.inf, 5e-324, -5e-324, 0.5, 1.0, 2.0,
             np.array([0x7FF8000000000123], np.uint64).view(np.float64)[0]],
            k.size)
        a[mask == 0] = 0.0
        return sa.SVT_SparseArray.from_dense(a, "double"), a
    if kind in ("logical", "lacunar"):
        a = mask.astype(np.int32)
        if kind == "logical":
            a.reshape(-1)[np.flatnonzero(mask)[rng.integers(
                0, mask.sum(), 10)]] = NA_I
        return sa.SVT_SparseArray.from_dense(a, "logical"), a
    a = np.where(mask, rng.integers(-6, 7, shape), 0).astype(np.int32)
    nz = np.flatnonzero(a)
    a.reshape(-1)[nz[rng.integers(0, nz.size, 30)]] = np.resize(
        [NA_I, 2**31 - 1, -(2**31 - 1)], 30)
    if kind == "mixed":
        a2 = a.reshape(shape[0], -1, order="F")
        m2 = mask.reshape(shape[0], -1, order="F")
        a2[:, 1::3] = m2[:, 1::3]                        # lacunar leaves
        a = a2.reshape(shape, order="F")
    return sa.SVT_SparseArray.from_dense(a, "integer"), a


POOL = {"integer": np.arange(-3, 4, dtype=np.int32),
        "logical": np.array([False, True]),
        "double": np.array([-2.5, -1.0, -0.5, -0.0, 0.0, 0.5, 1.0, 2.5,
                            np.inf, -np.inf, 5e-324, -5e-324])}


def operand(op, n, vt, seed=3):
    """n admissible elements of type vt for `x op v`, or None."""
    pool = [p for p in POOL[vt] if cr.admitted(op, np.array([p]))]
    if not pool:
        return None
    rng = np.random.Generator(np.random.PCG64(seed + n))
    return np.array(pool, dtype=POOL[vt].dtype)[rng.integers(0, len(pool), n)]


def expected(a, type_, op, v=None, margin=0, on_left=False):
    vt = None
    if v is not None:
        vt = "double" if np.asarray(v).dtype.kind == "f" else "integer"
    return cr.to_csc(*cr.dense(a, type_, cr.MIRROR[op] if on_left else op,
                               None if v is None else np.asarray(v), vt,
                               margin))


def check(r, exp):
    ep, eo, ev = exp
    assert r.type == "logical"
    p, o, v = sa.to_csc(r)
    assert np.array_equal(p.astype(np.int64), ep)
    assert np.array_equal(o, eo)
    assert np.array_equal(v, np.ones(eo.size, np.int32) if ev is None else ev)


def device_flags(x, op, v=None, margin=0, on_left=False):
    from sparsearray_b200.device import DeviceSVT
    y = DeviceSVT.from_host(x).ewise(op, v, margin=margin,
                                     operand_on_left=on_left)
    fl = ctypes.c_int(0)
    _native.check(_native.lib().svtgpu_matrix_info(
        y._h, None, None, None, None, ctypes.byref(fl)))
    assert y.val_type == "logical"
    return y, fl.value


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("margin", [0, 1, 2])
@pytest.mark.parametrize("vt", ["integer", "logical", "double"])
@pytest.mark.parametrize("op", OPS)
def test_compare_vs_dense(kind, margin, vt, op):
    x, a = make_input(kind)
    h = sa.to_device(x)
    n = 1 if margin == 0 else x.dim[0] if margin == 1 else x.dim[1]
    v = operand(op, n, vt)
    if v is None:
        pytest.skip("no %s value v makes 0 %s v FALSE" % (vt, op))
    if margin == 2:
        r = sa.sweep(h, 2, v, op)
    else:
        r = sa.Compare(h, op, v)
    exp = expected(a, x.type, op, v, margin)
    check(r, exp)
    # the same on the left: v op' x with the mirrored operator
    if margin < 2:
        check(sa.Compare(v, cr.MIRROR[op], h), exp)
    # a value array exactly when the result holds an NA
    y, fl = device_flags(x, op, v, margin)
    assert bool(fl & _native.HAS_VALS) == (exp[2] is not None)
    assert y.nnz == exp[1].size


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("fun", PREDS)
def test_predicates_vs_dense(kind, fun):
    x, a = make_input(kind)
    r = {"is.na": sa.is_na, "is.nan": sa.is_nan,
         "is.infinite": sa.is_infinite}[fun](sa.to_device(x))
    exp = expected(a, x.type, fun)
    assert exp[2] is None
    check(r, exp)
    y, fl = device_flags(x, fun)
    assert not fl & _native.HAS_VALS


def test_operators_on_the_python_object():
    x, a = make_input("double", seed=5)
    h = sa.to_device(x)
    check(h > 0.5, expected(a, "double", ">", [0.5]))
    check(h >= 1, expected(a, "double", ">=", [1]))
    check(h < -1, expected(a, "double", "<", [-1]))
    check(h <= -0.5, expected(a, "double", "<=", [-0.5]))
    check(2 < h, expected(a, "double", ">", [2]))            # reflected
    check(-2 >= h, expected(a, "double", "<=", [-2]))
    check(sa.Compare(h, "==", 1.0), expected(a, "double", "==", [1.0]))
    check(sa.Compare(h, "!=", 0), expected(a, "double", "!=", [0]))
    # == and != stay identity comparisons of the Python objects
    assert (h == h) is True and (h != h) is False
    assert {h: 1}[h] == 1


@pytest.mark.parametrize("margin", [0, 1])
@pytest.mark.parametrize("kind", ["integer", "double"])
def test_n_dimensional(margin, kind):
    x, a = make_input(kind, shape=(40, 7, 9), seed=11)
    v = operand(">", 1 if margin == 0 else 40, "double", seed=4)
    r = sa.Compare(sa.to_device(x), ">", v)
    check(r, expected(a, kind, ">", v, margin))
    assert r.dim == (40, 7, 9)


def test_leaf_and_tile_edges():
    nrow = 100_000
    a = np.zeros((nrow, 9), dtype=np.int32)
    rng = np.random.Generator(np.random.PCG64(21))
    a[:3, 0] = [1, 2, 3]                    # 3 entries: leaf 1 starts at 3
    a[:, 1] = rng.integers(1, 4, nrow)      # 100,000 entries, > 3 tiles
    a[::7, 1] = 0
    a[5, 2] = 2                             # single-entry leaf
    # leaf 3 empty
    a[:70_001:1, 4] = rng.integers(-2, 3, 70_001)
    a[:2, 5] = [NA_I, 2]
    a[10:13, 6] = [3, 1, 2]
    a[::2, 7] = 1
    a[nrow - 1, 8] = 9
    x = sa.SVT_SparseArray.from_dense(a, "integer", lacunar=False)
    assert x.ptr[1] % 4 == 3                # the long leaf starts unaligned
    h = sa.to_device(x)
    for op, v in ((">", 1), (">", 0), (">=", 2), ("==", 2), ("!=", 0),
                  ("<", 0), ("<=", -1), (">", 100)):
        check(sa.Compare(h, op, v), expected(a, "integer", op, [v]))
    for fun in PREDS:
        check({"is.na": sa.is_na, "is.nan": sa.is_nan,
               "is.infinite": sa.is_infinite}[fun](h),
              expected(a, "integer", fun))
    # nnz < 4, with and without an NA
    for tiny in (np.array([[0, 5], [3, 0]], np.int32),
                 np.array([[NA_I], [0], [2]], np.int32)):
        t = sa.to_device(sa.SVT_SparseArray.from_dense(tiny, "integer"))
        for op, v in ((">", 2), (">", 0), ("==", 3), ("<", 0)):
            check(sa.Compare(t, op, v), expected(tiny, "integer", op, [v]))


def test_kept_all_nothing_and_one_na():
    a = np.zeros((500, 30), dtype=np.int32)
    rng = np.random.Generator(np.random.PCG64(2))
    m = rng.random(a.shape) < 0.2
    a[m] = rng.integers(1, 5, m.sum())
    x = sa.SVT_SparseArray.from_dense(a, "integer")
    y, fl = device_flags(x, ">", np.array([0]))             # everything kept
    assert y.nnz == x.nnz and not fl & _native.HAS_VALS
    p, o, v = y.download()
    assert np.array_equal(p, x.ptr) and np.array_equal(o, x.offs)
    assert v is None
    y, fl = device_flags(x, ">", np.array([10]))            # nothing kept
    assert y.nnz == 0
    p, _, _ = y.download()
    assert not p.any()
    check(sa.Compare(sa.to_device(x), ">", 10),
          expected(a, "integer", ">", [10]))
    a[np.flatnonzero(m.reshape(-1, order="F"))[77] % 500,
      np.flatnonzero(m.reshape(-1, order="F"))[77] // 500] = NA_I
    x = sa.SVT_SparseArray.from_dense(a, "integer")
    y, fl = device_flags(x, ">", np.array([0]))             # one NA
    assert fl & _native.HAS_VALS
    p, o, v = y.download()
    assert (v == NA_I).sum() == 1 and (v == 1).sum() == x.nnz - 1
    check(sa.Compare(sa.to_device(x), ">", 0),
          expected(a, "integer", ">", [0]))
    # lacunar input with a scalar: a constant predicate
    lac = sa.SVT_SparseArray.from_dense((a != 0).astype(np.int32), "logical")
    assert lac.vals is None
    for op, v in ((">", 0), (">", 1), ("==", 1), (">=", 2), ("!=", 0)):
        check(sa.Compare(sa.to_device(lac), op, v),
              expected((a != 0).astype(np.int32), "logical", op, [v]))


def _stat_close(got, exp):
    got, exp = np.asarray(got, np.float64), np.asarray(exp, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(exp))
    m = ~np.isnan(exp)
    assert np.allclose(got[m], exp[m], rtol=1e-12, atol=0)


def test_statistics_of_results():
    x = synth.poisson_svt(3000, 200, 0.15, seed=12, na_rate=2e-3)
    a = np.zeros(x.dim, dtype=np.int32)
    for l in range(x.dim[1]):
        a[x.offs[x.ptr[l]:x.ptr[l + 1]], l] = x.vals[x.ptr[l]:x.ptr[l + 1]]
    h = sa.to_device(x)
    for y, (val, na) in ((h > 1, cr.dense(a, "integer", ">", [1], "integer")),
                         (h > 0, cr.dense(a, "integer", ">", [0], "integer")),
                         (sa.is_na(h), cr.dense(a, "integer", "is.na"))):
        d = cr.dense_logical(val, na)
        nan = np.isnan(d)
        dz = np.where(nan, 0.0, d)
        for na_rm in (False, True):
            def ref_sum(axis):
                s = dz.sum(axis=axis)
                if not na_rm:
                    s[nan.any(axis=axis)] = np.nan
                return s
            _stat_close(sa.colSums(y, na_rm=na_rm), ref_sum(0))
            _stat_close(sa.rowSums(y, na_rm=na_rm), ref_sum(1))
            _stat_close(sa.rowSums(y, na_rm=na_rm), ref_sum(1))  # compact copy
            cnt1 = (~nan).sum(axis=1) if na_rm else np.full(x.dim[0],
                                                            x.dim[1])
            _stat_close(sa.rowMeans(y, na_rm=na_rm), ref_sum(1) / cnt1)
            if na_rm:
                cv = np.nanvar(np.where(nan, np.nan, d), axis=0, ddof=1)
                rv = np.nanvar(np.where(nan, np.nan, d), axis=1, ddof=1)
            else:
                cv = d.var(axis=0, ddof=1)
                rv = d.var(axis=1, ddof=1)
            _stat_close(sa.colVars(y, na_rm=na_rm), cv)
            _stat_close(sa.rowVars(y, na_rm=na_rm), rv)
            # sum() of a logical is an integer: NA_integer_ when an NA counts
            tot = dz.sum() if (na_rm or not nan.any()) else np.nan
            got = np.asarray(sa.svt_sum(y, na_rm=na_rm)).reshape(-1)[:1]
            got = np.where(got == NA_I, np.nan, got.astype(np.float64))
            _stat_close(got, [tot])


def test_shards_equal_the_whole():
    from sparsearray_b200.device import DeviceSVT
    x = synth.poisson_svt(3000, 90, 0.1, seed=8, na_rate=1e-3)
    v = np.arange(90, dtype=np.float64) % 4
    for na in (True, False):
        if not na:
            x = synth.poisson_svt(3000, 90, 0.1, seed=8)
        whole = DeviceSVT.from_host(x).ewise(">", v, margin=2)
        parts = [DeviceSVT.from_host(x, r).ewise(">", v, margin=2)
                 for r in ((0, 37), (37, 90))]
        wp, wo, wv = whole.download()
        (p0, o0, v0), (p1, o1, v1) = parts[0].download(), parts[1].download()
        assert np.array_equal(wp, np.concatenate([p0, p1[1:] + p0[-1]]))
        assert np.array_equal(wo, np.concatenate([o0, o1]))
        if wv is None:
            assert v0 is None and v1 is None
        else:
            # a shard without an NA stores no values: its entries are TRUE
            vv = [np.ones(o.size, np.int32) if u is None else u
                  for u, o in ((v0, o0), (v1, o1))]
            assert np.array_equal(wv, np.concatenate(vv))


def test_scale_above_2_31_nonzeros():
    """C2 as the benchmark generates it (2.348e9 nonzeros, NA rate 1e-6)."""
    from sparsearray_b200.device import DeviceSVT
    nrow, ncol, dens, seed, na = 33538, 1_000_000, 0.07, 2, 1e-6
    x = DeviceSVT.generate_poisson(nrow, ncol, dens, seed=seed, na_rate=na)
    assert x.nnz > 2**31
    xlens = np.diff(x.leaf_ptr.cpu().numpy())
    nas = x.colstats("countNAs")[0].cpu().numpy().astype(np.int64)
    assert 1000 < nas.sum() < 4000
    # x > 1: about 3.6 % kept, below INT_MAX, so downloaded whole
    y, fl = None, ctypes.c_int(0)
    y = x.ewise(">", np.array([1], np.int32))
    assert 0.03 * x.nnz < y.nnz < 0.045 * x.nnz
    p, o, v = y.download()
    assert v is not None and (v == NA_I).sum() == nas.sum()
    cs = y.colstats("sum", na_rm=True)[0].cpu().numpy()
    cn = y.colstats("countNAs")[0].cpu().numpy()
    assert np.array_equal(cs + cn, np.diff(p).astype(np.float64))
    # about 2,000 leaves, with the one holding entry 2^31, bit for bit
    big = int(np.searchsorted(np.cumsum(xlens), 2**31, side="right"))
    rng = np.random.Generator(np.random.PCG64(5))
    leaves = sorted(set(rng.integers(0, ncol, 2000).tolist()) |
                    {0, big, ncol - 1})
    for l in leaves:
        _, oo, vv = synth.poisson_csc(nrow, 1, dens, seed=seed, na_rate=na,
                                      leaf0=l)
        keep = (vv > 1) | (vv == NA_I)
        assert np.array_equal(o[p[l]:p[l + 1]], oo[keep]), l
        assert np.array_equal(v[p[l]:p[l + 1]],
                              np.where(vv[keep] == NA_I, NA_I, 1)), l
    del y, p, o, v
    # x > 0 keeps every entry, more than INT_MAX: checked by identities
    y0 = x.ewise(">", np.array([0], np.int32))
    _native.check(_native.lib().svtgpu_matrix_info(
        y0._h, None, None, None, None, ctypes.byref(fl)))
    assert y0.nnz == x.nnz and fl.value & _native.HAS_VALS
    cs0 = y0.colstats("sum", na_rm=True)[0].cpu().numpy()
    assert np.array_equal(cs0, (xlens - nas).astype(np.float64))
    rs = y0.rowstats("sum", na_rm=True)[0].cpu().numpy()
    for i in np.linspace(0, nrow - 1, 150).astype(np.int64):
        c, _, isna = synth.poisson_row(nrow, ncol, int(i), dens, seed=seed,
                                       na_rate=na)
        assert rs[i] == c.size - isna.sum(), i
    assert rs.sum() == cs0.sum() == x.nnz - nas.sum()
    del y0, x
    # the same generator without NA: the result carries no value array
    x0 = DeviceSVT.generate_poisson(nrow, ncol, dens, seed=seed)
    y = x0.ewise(">", np.array([0], np.int32))
    _native.check(_native.lib().svtgpu_matrix_info(
        y._h, None, None, None, None, ctypes.byref(fl)))
    assert y.nnz == x0.nnz and not fl.value & _native.HAS_VALS
    assert y.colstats("sum")[0].sum().item() == x0.nnz
