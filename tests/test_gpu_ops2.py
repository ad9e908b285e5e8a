"""`x op y` between two SVTs on the device against the CPU oracle
(tests/ops2_oracle.c, itself held to numpy's dense definition by
test_ops2_host.py), bit for bit: structure, values, NA vs NaN, result type
and the overflow warning; every input kind, operator and order; N-d arrays;
edge geometries; derived inputs and results in every entry point; the device
cache; column shards; and C2 against a second generator matrix, whose union
passes 2^31 entries."""
import ctypes
import gc

import numpy as np
import pytest

import ops2_oracle
import sparsearray_b200 as sa
from sparsearray_b200 import _native as N, rcall, synth
from test_gpu_ewise import KINDS, make_input

pytestmark = pytest.mark.gpu

NA_I = -2**31
OPS = ops2_oracle.OPS
OVF = "NAs produced by integer overflow"


def oracle(x, y, op):
    return ops2_oracle.ops2(x.dim[0], x.ptr.size - 1, ops2_oracle.of_svt(x),
                            ops2_oracle.of_svt(y), op)


def run(x, op, y):
    if op in ("+", "-", "*"):
        return sa.Arith(x, op, y)
    if op in ("&", "|"):
        return sa.Logic(x, op, y)
    return sa.Compare(x, op, y)


def check(r, exp):
    ep, eo, ev, et, ew = exp
    assert r.type == et
    assert r.warnings == ([OVF] if ew & 1 else [])
    p, o, v = sa.to_csc(r)
    assert np.array_equal(p.astype(np.int64), ep)
    assert np.array_equal(o, eo)
    if et == "logical" and ev is None:
        ev = np.ones(eo.size, np.int32)
    if et == "double":
        assert np.array_equal(v.view(np.uint64), ev.view(np.uint64))
    else:
        assert np.array_equal(v, ev)


def second(kind, seed=5):
    """another input of the same shape; rows shifted so patterns overlap
    partly"""
    return make_input(kind, seed=seed)[0]


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("kx", KINDS)
@pytest.mark.parametrize("ky", KINDS)
def test_kinds_ops_orders_vs_oracle(op, kx, ky):
    x, y = make_input(kx)[0], second(ky)
    hx, hy = sa.to_device(x), sa.to_device(y)
    check(run(hx, op, hy), oracle(x, y, op))
    check(run(hy, op, hx), oracle(y, x, op))
    if kx == ky == "double":
        check(run(x, op, y), oracle(x, y, op))          # plain SVTs


def double_mask(seed=7):
    """a double 0 / 1 mask: every leaf all ones, so the matrix is stored
    without a value array yet has type "double" (`x * keep`)"""
    rng = np.random.Generator(np.random.PCG64(seed))
    m = (rng.random((2000, 70)) < 0.3).astype(np.float64)
    m[:, 5] = 0
    x = sa.SVT_SparseArray.from_dense(m, "double")
    assert x.type == "double" and x.vals is None
    return x


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("ky", KINDS + ["double_mask"])
def test_double_mask_against_every_kind(op, ky):
    x = double_mask()
    y = double_mask(seed=8) if ky == "double_mask" else second(ky)
    hx, hy = sa.to_device(x), sa.to_device(y)
    check(run(hx, op, hy), oracle(x, y, op))
    check(run(hy, op, hx), oracle(y, x, op))
    check(run(x, op, y), oracle(x, y, op))              # plain SVTs


def test_double_mask_plus_int_max_is_double():
    m = sa.SVT_SparseArray.from_dense(np.array([[1.0], [0.0], [1.0]]),
                                      "double")
    k = sa.SVT_SparseArray.from_dense(
        np.array([[2**31 - 1], [3], [NA_I]], np.int32), "integer")
    for r, sign in ((sa.to_device(m) + sa.to_device(k), 1),
                    (sa.to_device(k) - sa.to_device(m), -1)):
        assert r.type == "double" and r.warnings == []
        p, o, v = sa.to_csc(r)
        assert list(o) == [0, 1, 2]
        assert v[0] == 2.0**31 - 1 + sign and v[1] == 3.0
        assert sa.is_na_real(v[2:3])[0]


@pytest.mark.parametrize("op", OPS)
def test_nd_arrays_and_same_operand(op):
    rng = np.random.Generator(np.random.PCG64(3))
    a = np.where(rng.random((30, 4, 5)) < 0.3,
                 rng.integers(-3, 4, (30, 4, 5)), 0).astype(np.int32)
    b = np.where(rng.random((30, 4, 5)) < 0.3,
                 rng.integers(-3, 4, (30, 4, 5)), 0).astype(np.int32)
    x = sa.SVT_SparseArray.from_dense(a, lacunar=False)
    y = sa.SVT_SparseArray.from_dense(b, lacunar=False)
    r = run(sa.to_device(x), op, y)
    assert r.dim == (30, 4, 5)
    check(r, oracle(x, y, op))
    h = sa.to_device(x)
    check(run(h, op, h), oracle(x, x, op))              # one handle
    check(run(x, op, x), oracle(x, x, op))              # one SVT


def test_x_minus_x_is_empty_and_usable():
    x, _ = make_input("integer")
    h = sa.to_device(x)
    z = h - h
    p, o, v = sa.to_csc(z)
    nas = int(np.sum(x.vals == NA_I))
    assert o.size == nas                       # NA - NA stays NA
    e = sa.to_device(sa.SVT_SparseArray.from_dense(
        np.where(x.to_dense() == NA_I, 3, x.to_dense()).astype(np.int32)))
    z = e - e
    assert sa.to_csc(z)[1].size == 0
    assert np.array_equal(np.asarray(sa.colSums(z)), np.zeros(x.dim[1]))
    assert np.array_equal(np.asarray(sa.rowSums(z)), np.zeros(x.dim[0]))
    assert np.array_equal(np.asarray(sa.colMedians(z)), np.zeros(x.dim[1]))
    assert np.array_equal(np.asarray(sa.rowVars(z)), np.zeros(x.dim[0]))


def _csc_svt(nrow, cols, type_="integer"):
    """an SVT from a list of (offsets, values) per column"""
    ptr = np.concatenate([[0], np.cumsum([len(c[0]) for c in cols])])
    offs = np.concatenate([np.asarray(c[0], np.int32) for c in cols]) \
        if cols else np.zeros(0, np.int32)
    vals = np.concatenate([np.asarray(c[1]) for c in cols]) \
        if cols else np.zeros(0)
    return sa.SVT_SparseArray((nrow, len(cols)), type_, ptr, offs, vals)


def test_edge_leaves():
    nrow = 100_000
    rng = np.random.Generator(np.random.PCG64(8))
    long_ = np.sort(rng.choice(nrow, 60_000, replace=False))
    lo = np.arange(0, 4000)
    hi = np.arange(90_000, 96_000)
    cols_x = [(long_, rng.integers(1, 9, long_.size)), ([], []),
              (lo, np.ones(lo.size, np.int32)), (hi, -np.ones(hi.size)),
              ([0, nrow - 1], [5, 6]), ([], [])]
    cols_y = [([], []), (long_, rng.integers(-9, -1, long_.size)),
              (hi, np.full(hi.size, 2)), (lo, np.full(lo.size, 7)),
              ([nrow - 1], [-6]), ([], [])]
    x = _csc_svt(nrow, cols_x)
    y = _csc_svt(nrow, cols_y)
    for op in OPS:
        check(run(sa.to_device(x), op, sa.to_device(y)), oracle(x, y, op))
        check(run(sa.to_device(y), op, sa.to_device(x)), oracle(y, x, op))


def test_two_interleaved_300k_leaves():
    nrow = 600_000
    ev, od = np.arange(0, nrow, 2), np.arange(1, nrow, 2)
    x = _csc_svt(nrow, [(ev, np.arange(1, ev.size + 1)), (od, np.ones(od.size))])
    y = _csc_svt(nrow, [(od, np.full(od.size, 3)), (ev, np.arange(ev.size) % 5)])
    y = sa.SVT_SparseArray.from_dense(y.to_dense(), "integer")
    for op in OPS:
        check(run(sa.to_device(x), op, sa.to_device(y)), oracle(x, y, op))


@pytest.mark.parametrize("shape", [(1, 300), (70_000, 3), (50, 0)])
def test_extreme_shapes(shape):
    rng = np.random.Generator(np.random.PCG64(2))
    a = np.where(rng.random(shape) < 0.4, rng.integers(-3, 4, shape), 0)
    b = np.where(rng.random(shape) < 0.4, rng.standard_normal(shape), 0.0)
    x = sa.SVT_SparseArray.from_dense(a.astype(np.int32), "integer")
    y = sa.SVT_SparseArray.from_dense(b, "double")
    for op in OPS:
        r = run(sa.to_device(x), op, sa.to_device(y))
        assert r.dim == shape
        if shape[1] > 0 and shape[0] > 0:
            check(r, oracle(x, y, op))


def test_overflow_warns_once():
    a = np.array([[2**31 - 1, 5], [-(2**31 - 1), 0], [3, 2**31 - 1]],
                 np.int32)
    x = sa.SVT_SparseArray.from_dense(a, "integer")
    r = sa.to_device(x) + sa.to_device(x)
    assert r.warnings == [OVF]
    check(r, oracle(x, x, "+"))
    r = sa.to_device(x) - sa.to_device(x)
    assert r.warnings == []


def test_derived_inputs_and_dimnames():
    from sparsearray_b200.device import DeviceSVT
    x, a = make_input("integer")
    y, b = make_input("double", seed=9)
    hx = sa.to_device(x)
    gt = hx > 1                                    # Compare result
    lg = sa.SVT_SparseArray.from_dense(
        np.where(a == NA_I, NA_I, (a > 1)).astype(np.int32), "logical")
    sc = hx * -1                                   # Arith result
    scs = sa.SVT_SparseArray.from_dense(
        np.where(a == NA_I, NA_I, -a).astype(np.int32), "integer")
    p, i, v = sa.to_csc(y)
    fc = sa.from_csc(y.dim, p, v, i)              # from_csc handle
    for op in OPS:
        check(run(gt, op, fc), oracle(lg, y, op))
        check(run(sc, op, gt), oracle(scs, lg, op))
    # a compact copy on x (two statistic calls build it)
    xs = synth.poisson_svt(3000, 40, 0.2, seed=4)
    hs = sa.to_device(xs)
    sa.colSums(hs)
    sa.colSums(hs)
    ys = synth.poisson_svt(3000, 40, 0.1, seed=5)
    check(hs + sa.to_device(ys), oracle(xs, ys, "+"))
    # a result carries no compact copy, even from an input that has one
    dx = DeviceSVT.from_host(xs)
    dx.colstats("sum")
    dx.colstats("sum")
    cb = ctypes.c_int64(-1)
    dr = dx.ewise_svt("+", DeviceSVT.from_host(ys))
    N.check(N.lib().svtgpu_matrix_compact_bytes(dr._h, ctypes.byref(cb)))
    assert cb.value == 0
    dr.colstats("sum")
    dr.colstats("sum")
    s, _ = dr.colstats("sum")
    t = oracle(xs, ys, "+")
    assert np.array_equal(s.cpu().numpy(), np.asarray(sa.colSums(
        sa.SVT_SparseArray(xs.dim, "integer", t[0], t[1], t[2]))))
    # dimnames from e1, else from e2
    xn = sa.SVT_SparseArray(x.dim, x.type, x.ptr, x.offs, x.vals, x.lacunar,
                            dimnames=[None, ["c%d" % k for k in range(70)]])
    assert (x + xn).dimnames == xn.dimnames
    assert (xn - x).dimnames == xn.dimnames
    assert (x * x).dimnames == [None, None]


def test_results_feed_every_statistic():
    x = synth.poisson_svt(3000, 80, 0.1, seed=4, na_rate=1e-3)
    y = synth.poisson_svt(3000, 80, 0.05, seed=6, na_rate=1e-3)
    r = sa.to_device(x) - sa.to_device(y)
    t = oracle(x, y, "-")
    ref = sa.SVT_SparseArray(x.dim, "integer", t[0], t[1], t[2])
    for na_rm in (False, True):
        for f in (sa.colSums, sa.rowSums, sa.rowVars, sa.colMedians):
            assert np.array_equal(np.asarray(f(r, na_rm=na_rm)),
                                  np.asarray(f(ref, na_rm=na_rm)),
                                  equal_nan=True)
    p, i, v = sa.to_csc(r)
    assert np.array_equal(p, t[0]) and np.array_equal(i, t[1])
    m = (sa.to_device(x) > 1) | (sa.to_device(y) > 0)
    assert m.type == "logical"
    t = oracle(sa.SVT_SparseArray(x.dim, "logical", *_gt(x.ptr, x.offs,
                                                         x.vals, 1)),
               sa.SVT_SparseArray(y.dim, "logical", *_gt(y.ptr, y.offs,
                                                         y.vals, 0)), "|")
    check(m, t)


def test_device_cache_on():
    x = synth.poisson_svt(2000, 60, 0.1, seed=1, na_rate=1e-3)
    y = synth.poisson_svt(2000, 60, 0.1, seed=2, na_rate=1e-3)
    prev = rcall.set_gpu_cache(True)
    try:
        for _ in range(2):
            check(x + y, oracle(x, y, "+"))        # plain SVTs both sides
        sa.colSums(x)                              # x is now the cached one
        check(x * y, oracle(x, y, "*"))
        check(y - x, oracle(y, x, "-"))
        check(x - x, oracle(x, x, "-"))
        sa.colSums(y)                              # y is now the cached one
        check(x + y, oracle(x, y, "+"))
        assert np.array_equal(np.asarray(sa.colSums(x)),
                              np.asarray(sa.colSums(sa.to_device(x))),
                              equal_nan=True)
    finally:
        rcall.set_gpu_cache(None)
        rcall.set_gpu_cache(prev)


def test_column_shards():
    from sparsearray_b200.device import DeviceSVT
    x = synth.poisson_svt(3000, 90, 0.1, seed=8, na_rate=1e-3)
    y = synth.poisson_svt(3000, 90, 0.1, seed=3, na_rate=1e-3)
    for op in ("+", "*", "!="):
        whole = DeviceSVT.from_host(x).ewise_svt(op, DeviceSVT.from_host(y))
        parts = [DeviceSVT.from_host(x, r).ewise_svt(op,
                                                     DeviceSVT.from_host(y, r))
                 for r in ((0, 37), (37, 90))]
        wp, wo, wv = whole.download()
        (p0, o0, v0), (p1, o1, v1) = parts[0].download(), parts[1].download()
        assert np.array_equal(wp, np.concatenate([p0, p1[1:] + p0[-1]]))
        assert np.array_equal(wo, np.concatenate([o0, o1]))
        t = oracle(x, y, op)
        assert np.array_equal(wp, t[0]) and np.array_equal(wo, t[1])
        if wv is not None:
            assert np.array_equal(wv, np.concatenate([v0, v1]))
    with pytest.raises(ValueError):
        DeviceSVT.from_host(x, (0, 37)).ewise_svt("+",
                                                  DeviceSVT.from_host(y, (1, 38)))


# ---- C2 and a second generator matrix: the union passes 2^31 ---------------

NROW, NCOL, DENS, SEED, NA_RATE = 33538, 1_000_000, 0.07, 2, 1e-6
Y_DENS, Y_SEED = 0.01, 7
BLOCK = 250


def _leaf_ptr(d):
    p = np.zeros(d.nleaf + 1, np.int64)
    N.check(N.lib().svtgpu_matrix_download(
        d._h, p.ctypes.data_as(ctypes.c_void_p), None, None))
    return p


def _gt(p, o, v, thr):
    """x > thr of an integer CSC, as the logical CSC the device keeps"""
    keep = (v > thr) | (v == NA_I)
    q = np.concatenate([[0], np.cumsum(keep)]).astype(np.int64)[p]
    w = np.where(v[keep] == NA_I, NA_I, 1).astype(np.int32)
    return q, o[keep], w


def test_scale_union_above_2_31():
    import torch
    from sparsearray_b200.device import DeviceSVT
    total = torch.cuda.get_device_properties(0).total_memory
    if total < 60e9:
        pytest.skip("needs 60 GB of device memory, the device has %.0f"
                    % (total / 1e9))
    x = DeviceSVT.generate_poisson(NROW, NCOL, DENS, seed=SEED,
                                   na_rate=NA_RATE)
    y = DeviceSVT.generate_poisson(NROW, NCOL, Y_DENS, seed=Y_SEED)
    assert x.nnz > 2**31
    xp = x.leaf_ptr.cpu().numpy()
    rng = np.random.Generator(np.random.PCG64(1))
    starts = [0, NCOL - BLOCK,
              int(np.searchsorted(xp, 2**31, side="right")) - BLOCK // 2]
    starts += [int(s) for s in rng.integers(0, NCOL - BLOCK, 4)]
    gx, gy = {}, {}

    def host(l0):
        if l0 not in gx:
            gx[l0] = synth.poisson_csc(NROW, BLOCK, DENS, seed=SEED,
                                       na_rate=NA_RATE, leaf0=l0)
            gy[l0] = synth.poisson_csc(NROW, BLOCK, Y_DENS, seed=Y_SEED,
                                       leaf0=l0)
        return gx[l0], gy[l0]

    def verify(r, make_ref, blocks):
        rp = _leaf_ptr(r)
        s, _ = r.colstats("sum", na_rm=True)
        na, _ = r.colstats("countNAs")
        s, na = s.cpu().numpy(), na.cpu().numpy()
        for l0 in blocks:
            t = make_ref(l0)
            sl = slice(l0, l0 + BLOCK)
            assert np.array_equal(np.diff(rp[l0:l0 + BLOCK + 1]),
                                  np.diff(t[0])), l0
            v = t[2] if t[2] is not None else np.ones(t[1].size, np.int32)
            ok = v != NA_I
            col = np.repeat(np.arange(BLOCK), np.diff(t[0]))
            es = np.bincount(col[ok], v[ok].astype(np.float64), BLOCK)
            en = np.bincount(col[~ok], minlength=BLOCK)
            assert np.array_equal(s[sl], es), l0
            assert np.array_equal(na[sl], en), l0
        return rp

    r = x.ewise_svt("+", y)
    assert r.nnz > 2**31 and r.val_type == "integer"
    rp = _leaf_ptr(r)
    blocks = starts + [int(np.searchsorted(rp, 2**31, side="right"))
                       - BLOCK // 2]

    def ref_add(l0):
        (p, o, v), (q, oo, w) = host(l0)
        return ops2_oracle.ops2(NROW, BLOCK, (p, o, v, "integer", None),
                                (q, oo, w, "integer", None), "+")
    verify(r, ref_add, blocks)
    del r
    gc.collect()

    def ref_mul(l0):
        (p, o, v), (q, oo, w) = host(l0)
        return ops2_oracle.ops2(NROW, BLOCK, (p, o, v, "integer", None),
                                (q, oo, w, "integer", None), "*")
    r = x.ewise_svt("*", y)
    verify(r, ref_mul, blocks)
    del r
    gc.collect()

    def ref_or(l0):
        (p, o, v), (q, oo, w) = host(l0)
        a, b = _gt(p, o, v, 1), _gt(q, oo, w, 0)
        return ops2_oracle.ops2(NROW, BLOCK,
                                (a[0], a[1], a[2], "logical", None),
                                (b[0], b[1], b[2], "logical", None), "|")
    gx1, gy0 = x.ewise(">", 1), y.ewise(">", 0)
    r = gx1.ewise_svt("|", gy0)
    assert r.val_type == "logical"
    verify(r, ref_or, blocks)
