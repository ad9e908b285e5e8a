"""`x[i, j, ...]` on the device against the numpy oracle
(tests/subset_oracle.py), bit for bit with doubles compared as uint64: every
input kind and derived handle, every route of the row subscript on rows and
columns, N-d arrays, edge geometries, results in every entry point, x left
intact with its caches, the device cache, shards, and C2 above 2^31 entries
against the counter-based generator."""
import ctypes
import gc

import numpy as np
import pytest

import subset_oracle
import sparsearray_b200 as sa
from sparsearray_b200 import _native as N, rcall, synth
from sparsearray_b200.device import DeviceSVT
from test_gpu_ewise import KINDS, make_input

pytestmark = pytest.mark.gpu

NA_I = -2**31


def _same(got, want):
    p, o, v = got
    ep, eo, ev = want
    assert np.array_equal(np.asarray(p, np.int64), ep)
    assert np.array_equal(o, eo)
    if ev is None:
        return
    if ev.dtype == np.float64:
        assert np.array_equal(v.view(np.uint64), ev.view(np.uint64))
    else:
        assert np.array_equal(v, ev)


def expected(x, rows, leaves):
    """the oracle on x's CSC; for N-d arrays `leaves` are leaf numbers"""
    p, o, v = subset_oracle.csc_of(x)
    ep, eo, ev = subset_oracle.subset(x.dim[0], p, o, v, rows, leaves)
    if ev is None:                      # to_CSC gives a lacunar matrix ones
        ev = np.ones(eo.size, np.float64 if x.type == "double" else np.int32)
    return ep, eo, ev


def check(r, x, rows, cols):
    """r = x[rows, cols] (0-based or None) of a matrix"""
    n_r = x.dim[0] if rows is None else len(rows)
    n_c = x.dim[1] if cols is None else len(cols)
    assert r.dim == (n_r, n_c) and r.type == x.type
    _same(sa.to_csc(r), expected(x, rows, cols))


def nidx(rows, cols):
    return [None if rows is None else np.asarray(rows) + 1,
            None if cols is None else np.asarray(cols) + 1]


def subscripts(n, seed=0):
    """one subscript per route: missing, sorted, sorted with duplicates,
    unsorted, unsorted with duplicates, empty"""
    rng = np.random.Generator(np.random.PCG64(seed))
    srt = np.sort(rng.choice(n, max(1, n // 3), replace=False))
    dup = np.sort(np.concatenate([srt, srt[::2], srt[:3]]))
    uns = rng.permutation(srt)
    udp = rng.permutation(dup)
    return {"missing": None, "sorted": srt, "sorted_dup": dup,
            "unsorted": uns, "unsorted_dup": udp,
            "empty": np.zeros(0, np.int64)}


ROUTES = list(subscripts(10))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("rroute", ROUTES)
@pytest.mark.parametrize("croute", ["missing", "sorted", "unsorted_dup",
                                    "empty"])
def test_kinds_and_routes_vs_oracle(kind, rroute, croute):
    x, _ = make_input(kind)
    rows = subscripts(x.dim[0], 1)[rroute]
    cols = subscripts(x.dim[1], 2)[croute]
    check(sa.subset(sa.to_device(x), nidx(rows, cols)), x, rows, cols)
    if kind == "double":
        check(sa.subset(x, nidx(rows, cols)), x, rows, cols)   # plain SVT


def test_columns_with_routes_on_every_kind():
    for kind in KINDS:
        x, _ = make_input(kind)
        h = sa.to_device(x)
        for cr, cols in subscripts(x.dim[1], 3).items():
            check(sa.subset(h, nidx(None, cols)), x, None, cols)


def test_double_values_bit_for_bit():
    bits = np.array([0x7FF00000000007A2,          # NA_real_
                     0x7FF8000000000123, 0xFFF8000000000456,   # NaN payloads
                     0x8000000000000000,          # -0 (stored)
                     0x0000000000000001, 0x7FF0000000000000,
                     0xFFF0000000000000, 0x3FF0000000000000], np.uint64)
    vals = bits.view(np.float64)
    ptr = np.array([0, 4, 8], np.int64)
    offs = np.array([0, 2, 5, 9, 1, 3, 5, 7], np.int32)
    x = sa.SVT_SparseArray((10, 2), "double", ptr, offs, vals)
    for rows in (None, [9, 5, 2, 1, 0], [0, 0, 5, 5, 9], [3, 7, 1]):
        for cols in (None, [1, 0, 1]):
            check(sa.subset(sa.to_device(x), nidx(rows, cols)), x, rows, cols)


def _flags(d):
    fl = ctypes.c_int(0)
    N.check(N.lib().svtgpu_matrix_info(d._h, None, None, None, None,
                                       ctypes.byref(fl)))
    return fl.value


def double_mask(seed=7):
    rng = np.random.Generator(np.random.PCG64(seed))
    m = (rng.random((500, 40)) < 0.3).astype(np.float64)
    m[:, 5] = 0
    x = sa.SVT_SparseArray.from_dense(m, "double")
    assert x.vals is None
    return x


@pytest.mark.parametrize("kind", ["lacunar", "double_mask", "mixed"])
def test_value_array_presence(kind):
    x = double_mask() if kind == "double_mask" else make_input(kind)[0]
    d = DeviceSVT.from_host(x)
    for rows in (None, [7, 3, 3, 1], [1, 3, 3, 7]):
        r = d.subset(rows, [4, 0, 4, 2])
        assert bool(_flags(r) & N.HAS_VALS) == (x.vals is not None)
        assert r.val_type == x.type
        p, o, v = r.download()
        ep, eo, ev = subset_oracle.subset(x.dim[0], *subset_oracle.csc_of(x),
                                          rows, [4, 0, 4, 2])
        assert np.array_equal(p, ep) and np.array_equal(o, eo)
        assert (v is None) == (ev is None)
        if v is not None:
            assert np.array_equal(v, ev)


def test_nd_arrays_all_dimensions_subscripted():
    rng = np.random.Generator(np.random.PCG64(3))
    shape = (30, 4, 5)
    a = np.where(rng.random(shape) < 0.3, rng.integers(-3, 4, shape),
                 0).astype(np.int32)
    x = sa.SVT_SparseArray.from_dense(a, lacunar=False)
    h = sa.to_device(x)
    for i, j, k in (([29, 0, 4, 4], [3, 1], [4, 0, 2, 2]),
                    ([1, 2, 5], None, [3]),
                    (None, [0, 0], None),
                    ([], [1], [0, 1]),
                    (np.arange(29, -1, -1), [2, 3, 0], [1, 4])):
        key = [None if s is None else np.asarray(s) + 1 for s in (i, j, k)]
        r = sa.subset(h, key)
        jj = np.arange(4) if j is None else np.asarray(j)
        kk = np.arange(5) if k is None else np.asarray(k)
        leaves = (jj[None, :] + 4 * kk[:, None]).reshape(-1)
        want_dim = tuple(n if s is None else len(s)
                         for s, n in zip((i, j, k), shape))
        assert r.dim == want_dim
        _same(sa.to_csc(r), expected(x, i, leaves))
        ii = np.arange(30) if i is None else np.asarray(i, np.int64)
        got = np.asarray(sa.to_csc(r)[1])
        assert got.size == np.count_nonzero(a[np.ix_(ii, jj, kk)])
    # numpy-style keys on the same array
    r = h[[3, 3, 0], 1:, ::-2]
    assert r.dim == (3, 3, 3)
    leaves = (np.array([1, 2, 3])[None, :] + 4 * np.array([4, 2, 0])[:, None])
    _same(sa.to_csc(r), expected(x, [3, 3, 0], leaves.reshape(-1)))


def _csc_svt(nrow, cols, type_="integer"):
    ptr = np.concatenate([[0], np.cumsum([len(c[0]) for c in cols])])
    offs = np.concatenate([np.asarray(c[0], np.int32) for c in cols]) \
        if cols else np.zeros(0, np.int32)
    vals = np.concatenate([np.asarray(c[1], np.int32) for c in cols]) \
        if cols else np.zeros(0, np.int32)
    return sa.SVT_SparseArray((nrow, len(cols)), type_, ptr, offs, vals)


def test_empty_and_long_leaves():
    nrow = 600_000
    ev = np.arange(0, nrow, 2)
    x = _csc_svt(nrow, [([], []), (ev, np.arange(1, ev.size + 1)), ([], []),
                        ([5, nrow - 1], [7, 8]), ([], []),
                        (np.arange(1, nrow, 2), -np.ones(ev.size)), ([], [])])
    h = sa.to_device(x)
    rng = np.random.Generator(np.random.PCG64(5))
    for rows in (None, np.arange(1000, 400_000), np.arange(nrow - 1, -1, -1),
                 np.sort(rng.integers(0, nrow, 50_000)),
                 rng.integers(0, nrow, 50_000)):
        for cols in (None, [0, 2, 4, 6], [6, 1, 1, 0, 5, 3]):
            check(sa.subset(h, nidx(rows, cols)), x, rows, cols)


@pytest.mark.parametrize("shape", [(0, 5), (1, 300), (70_000, 3), (50, 0)])
def test_extreme_shapes(shape):
    rng = np.random.Generator(np.random.PCG64(2))
    a = np.where(rng.random(shape) < 0.4, rng.integers(-3, 4, shape), 0)
    x = sa.SVT_SparseArray.from_dense(a.astype(np.int32), "integer")
    h = sa.to_device(x)
    nr, nc = shape
    for rows in (None, [], list(range(nr))[::-1][:7], [0] * min(nr, 3)):
        if nr == 0 and rows:
            continue
        for cols in (None, [], [nc - 1, 0] if nc else []):
            r = sa.subset(h, nidx(rows, cols))
            check(r, x, rows, cols)


def _derived():
    x, a = make_input("integer")
    y, _ = make_input("double", seed=9)
    hx, hy = sa.to_device(x), sa.to_device(y)
    p, i, v = sa.to_csc(y)
    out = {"from_csc": (sa.from_csc(y.dim, p, v, i), y)}
    sc = hx * -1
    out["arith"] = (sc, sa.SVT_SparseArray.from_dense(
        np.where(a == NA_I, NA_I, -a).astype(np.int32), "integer"))
    gt = hx > 1
    out["compare"] = (gt, sa.SVT_SparseArray.from_dense(
        np.where(a == NA_I, NA_I, (a > 1)).astype(np.int32), "logical"))
    s = hx - hx * 2                          # ewise2: x - 2x = -x
    out["ewise2"] = (s, out["arith"][1])
    return out, hy


def test_derived_handles():
    out, _ = _derived()
    for name, (h, ref) in out.items():
        rows = subscripts(ref.dim[0], 4)
        for rr in ("missing", "sorted_dup", "unsorted"):
            check(sa.subset(h, nidx(rows[rr], [3, 0, 69, 3])), ref, rows[rr],
                  [3, 0, 69, 3])
    # an input carrying its compact copy
    xs = synth.poisson_svt(3000, 40, 0.2, seed=4)
    hs = sa.to_device(xs)
    sa.colSums(hs)
    sa.colSums(hs)
    d = DeviceSVT.from_host(xs)
    d.colstats("sum")
    d.colstats("sum")
    cb = ctypes.c_int64(0)
    N.check(N.lib().svtgpu_matrix_compact_bytes(d._h, ctypes.byref(cb)))
    assert cb.value > 0
    for rows in (None, np.arange(0, 3000, 3), np.arange(2999, -1, -7)):
        check(sa.subset(hs, nidx(rows, np.arange(39, -1, -2))), xs, rows,
              np.arange(39, -1, -2))
        r = d.subset(rows, np.arange(39, -1, -2))
        N.check(N.lib().svtgpu_matrix_compact_bytes(r._h, ctypes.byref(cb)))
        assert cb.value == 0                 # the result carries no copy


def test_dimnames_and_getitem():
    x, a = make_input("integer")
    xn = sa.SVT_SparseArray(x.dim, x.type, x.ptr, x.offs, x.vals, x.lacunar,
                            dimnames=[None, ["c%d" % k for k in range(70)]])
    r = sa.subset(sa.to_device(xn), [np.array([5, 1]), np.array([3, 3, 70])])
    assert r.dimnames == [None, ["c2", "c2", "c69"]]
    h = sa.to_device(x)
    keep = np.zeros(70, bool)
    keep[::3] = True
    for key, rows, cols in (((slice(None), keep), None, np.flatnonzero(keep)),
                            ((slice(10, 40, 3),), np.arange(10, 40, 3), None),
                            ((7, [2, -1]), [7], [2, 69]),
                            ((slice(None, None, -1), 5), np.arange(1999, -1,
                                                                   -1), [5])):
        check(h[key], x, rows, cols)


def test_results_feed_every_statistic():
    x = synth.poisson_svt(3000, 80, 0.1, seed=4, na_rate=1e-3)
    h = sa.to_device(x)
    rng = np.random.Generator(np.random.PCG64(6))
    for rows in (None, np.sort(rng.choice(3000, 900, replace=False)),
                 rng.integers(0, 3000, 1200)):
        cols = rng.integers(0, 80, 50)
        r = sa.subset(h, nidx(rows, cols))
        ep, eo, ev = expected(x, rows, cols)
        ref = sa.SVT_SparseArray(r.dim, "integer", ep, eo, ev)
        for na_rm in (False, True):
            for f in (sa.colSums, sa.rowSums, sa.rowVars, sa.colMedians):
                assert np.array_equal(np.asarray(f(r, na_rm=na_rm)),
                                      np.asarray(f(ref, na_rm=na_rm)),
                                      equal_nan=True)
        assert np.array_equal(np.asarray(sa.crossprod(r)),
                              np.asarray(sa.crossprod(ref)), equal_nan=True)
        _same(sa.to_csc(r), (ep, eo, ev))


def test_x_and_its_caches_survive():
    x = synth.poisson_svt(3000, 60, 0.1, seed=2, na_rate=1e-3)
    h = sa.to_device(x)
    rm0 = np.asarray(sa.rowMedians(h))            # builds the transpose
    sa.colSums(h)
    cs0 = np.asarray(sa.colSums(h))               # builds the compact copy
    rs0 = np.asarray(sa.rowSums(h))
    p0 = sa.to_csc(h)
    for rows in (None, np.arange(0, 3000, 2), np.arange(2999, -1, -1)):
        sa.subset(h, nidx(rows, np.arange(59, -1, -1)))
    assert np.array_equal(np.asarray(sa.rowMedians(h)), rm0, equal_nan=True)
    assert np.array_equal(np.asarray(sa.colSums(h)), cs0, equal_nan=True)
    assert np.array_equal(np.asarray(sa.rowSums(h)), rs0, equal_nan=True)
    for got, want in zip(sa.to_csc(h), p0):
        assert np.array_equal(got, want)


def test_device_cache_on():
    x = synth.poisson_svt(2000, 60, 0.1, seed=1, na_rate=1e-3)
    prev = rcall.set_gpu_cache(True)
    try:
        sa.colSums(x)                             # x is the cached matrix
        for rows in (None, np.arange(0, 2000, 5), np.arange(1999, -1, -3)):
            r = sa.subset(x, nidx(rows, [59, 0, 0]))
            check(r, x, rows, [59, 0, 0])
            del r
            gc.collect()                          # the result is freed ...
        # ... and the cached x still answers
        assert np.array_equal(np.asarray(sa.colSums(x)),
                              np.asarray(sa.colSums(sa.to_device(x))),
                              equal_nan=True)
        check(sa.subset(x, [None, None]), x, None, None)
    finally:
        rcall.set_gpu_cache(None)
        rcall.set_gpu_cache(prev)


def test_column_shards():
    x = synth.poisson_svt(3000, 90, 0.1, seed=8, na_rate=1e-3)
    rows = np.arange(2999, 0, -4)
    for r0, r1 in ((0, 37), (37, 90)):
        d = DeviceSVT.from_host(x, (r0, r1))
        loc = np.array([3, 0, 3, r1 - r0 - 1])
        p, o, v = d.subset(rows, loc).download()
        ep, eo, ev = subset_oracle.subset(3000, *subset_oracle.csc_of(x),
                                          rows, loc + r0)
        assert np.array_equal(p, ep) and np.array_equal(o, eo)
        assert np.array_equal(v, ev)
    with pytest.raises(N.SvtGpuError, match="leaf subscript"):
        DeviceSVT.from_host(x, (0, 37)).subset(None, [37])


# ---- C2: 33,538 x 1e6 integer counts generated in HBM ----------------------

NROW, NCOL, DENS, SEED, NA_RATE = 33538, 1_000_000, 0.07, 2, 1e-6
BLOCK = 250


def _leaf_ptr(d):
    p = np.zeros(d.nleaf + 1, np.int64)
    N.check(N.lib().svtgpu_matrix_download(
        d._h, p.ctypes.data_as(ctypes.c_void_p), None, None))
    return p


def _leaf_entries(d, p, l0, n):
    """(offs, vals) of d's leaves [l0, l0 + n), downloaded through a
    one-leaf-range subset of d"""
    r = d.subset(None, np.arange(l0, l0 + n))
    q, o, v = r.download()
    return q, o, v


def test_scale_c2_above_2_31():
    import torch
    total = torch.cuda.get_device_properties(0).total_memory
    if total < 120e9:
        pytest.skip("needs 120 GB of device memory, the device has %.0f"
                    % (total / 1e9))
    x = DeviceSVT.generate_poisson(NROW, NCOL, DENS, seed=SEED,
                                   na_rate=NA_RATE)
    assert x.nnz > 2**31
    rng = np.random.Generator(np.random.PCG64(11))
    keep = np.flatnonzero(rng.random(NCOL) < 0.95)
    r = x.subset(None, keep)
    assert r.nnz > 2**31
    rp = _leaf_ptr(r)
    xp = _leaf_ptr(x)
    assert np.array_equal(np.diff(rp), np.diff(xp)[keep])
    k31 = int(np.searchsorted(rp, 2**31, side="right")) - 1
    starts = [0, keep.size - BLOCK, k31 - BLOCK // 2]
    starts += [int(s) for s in rng.integers(0, keep.size - BLOCK, 5)]
    checked = 0
    for k0 in starts:                     # ~2,000 result columns
        q, o, v = _leaf_entries(r, rp, k0, BLOCK)
        for k in range(BLOCK):
            l = int(keep[k0 + k])
            hp, ho, hv = synth.poisson_csc(NROW, 1, DENS, seed=SEED,
                                           na_rate=NA_RATE, leaf0=l)
            assert np.array_equal(o[q[k]:q[k + 1]], ho), (k0, k)
            assert np.array_equal(v[q[k]:q[k + 1]], hv), (k0, k)
            checked += 1
    assert checked >= 2000
    # colSums(x[, j]) == colSums(x)[j], exactly
    cs, _ = x.colstats("sum", na_rm=True)
    rs, _ = r.colstats("sum", na_rm=True)
    assert torch.equal(rs, cs[torch.as_tensor(keep, device=cs.device)])
    del r, rs
    gc.collect()

    # x[rev(seq_len(nrow)), ]: the unsorted route, above 2^31 entries
    rev = np.arange(NROW - 1, -1, -1)
    t = x.subset(rev, None)
    assert t.nnz == x.nnz
    tp = _leaf_ptr(t)
    assert np.array_equal(tp, xp)
    l31 = int(np.searchsorted(tp, 2**31, side="right")) - 1
    for l0 in (0, l31 - 4, NCOL - 8):
        q, o, v = _leaf_entries(t, tp, l0, 8)
        for k in range(8):
            hp, ho, hv = synth.poisson_csc(NROW, 1, DENS, seed=SEED,
                                           na_rate=NA_RATE, leaf0=l0 + k)
            assert np.array_equal(o[q[k]:q[k + 1]], NROW - 1 - ho[::-1])
            assert np.array_equal(v[q[k]:q[k + 1]], hv[::-1])
    # rowSums(x[i, ]) == rowSums(x)[i], exactly
    rsx, _ = x.rowstats("sum", na_rm=True)
    rst, _ = t.rowstats("sum", na_rm=True)
    assert torch.equal(rst, torch.flip(rsx, [0]))
    del t
    gc.collect()
    i = np.sort(rng.choice(NROW, 2000, replace=False))
    s = x.subset(i, None)
    rss, _ = s.rowstats("sum", na_rm=True)
    assert torch.equal(rss, rsx[torch.as_tensor(i, device=rsx.device)])
