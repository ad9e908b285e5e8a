"""Element-wise operations on the device against the oracle's restatement
(tests/ewise_oracle.c, itself held to base R's dense definition by
test_ewise_host.py): structure and values bit for bit (log1p / expm1 within
2 ulp), NA vs NaN, result type and warnings; the compaction path; derived
handles in every entry point; column shards; one run above 2^31 nonzeros."""
import numpy as np
import pytest

import ewise_oracle
import sparsearray_b200 as sa
from oracle import port
from sparsearray_b200 import synth

pytestmark = pytest.mark.gpu

NA_I = -2**31
MATH = ["abs", "sign", "sqrt", "floor", "ceiling", "trunc", "log1p", "expm1"]
WARN = {1: "NAs produced by integer overflow", 2: "NaNs produced"}


def make_input(kind, nrow=2000, ncol=70, seed=1):
    """int / logical / double / lacunar / mixed SVT with NA, NaN, +-Inf,
    overflow-prone integers and empty leaves; >1 tile of 32,768 entries."""
    rng = np.random.Generator(np.random.PCG64(seed))
    mask = rng.random((nrow, ncol)) < 0.3
    mask[:, 5] = False                              # an empty leaf
    if kind == "double":
        a = np.where(mask, rng.standard_normal((nrow, ncol)) * 4, 0.0)
        k = rng.integers(0, a.size, 60)
        a.reshape(-1)[k] = np.resize(
            [sa.NA_REAL, np.nan, np.inf, -np.inf, -1.0, -2.5, 1e-310, 0.5],
            k.size)
        a[:, 5] = 0
        return sa.SVT_SparseArray.from_dense(a, "double"), a
    if kind in ("logical", "lacunar"):
        a = mask.astype(np.int32)
        if kind == "logical":
            a.reshape(-1)[rng.integers(0, a.size, 10)] = NA_I
        a[:, 5] = 0
        return sa.SVT_SparseArray.from_dense(a, "logical"), a
    a = np.where(mask, rng.integers(-40, 40, (nrow, ncol)), 0).astype(np.int32)
    a.reshape(-1)[rng.integers(0, a.size, 40)] = np.resize(
        [NA_I, 2**31 - 1, 70000, -46341], 40)
    if kind == "mixed":
        a[:, 1::3] = mask[:, 1::3]                  # lacunar leaves
    a[:, 5] = 0
    return sa.SVT_SparseArray.from_dense(a, "integer"), a


KINDS = ["integer", "logical", "double", "lacunar", "mixed"]


def oracle(x, op, v=None, vt=None, margin=0):
    return ewise_oracle.ewise(x.dim[0], x.ptr.size - 1, x.ptr, x.offs,
                              x.vals, x.type,
                      op, v, vt, margin, x.lacunar)


def download(r):
    p, i, v = sa.to_csc(r)
    return p.astype(np.int64), i, v


def check(r, exp, op):
    ep, eo, ev, et, ew = exp
    assert r.type == et
    assert sorted(r.warnings) == sorted(WARN[b] for b in (1, 2) if ew & b)
    p, o, v = download(r)
    assert np.array_equal(p, ep)
    assert np.array_equal(o, eo)
    if et == "integer":
        assert np.array_equal(v, ev)
        return
    vb, eb = v.view(np.uint64), ev.view(np.uint64)
    assert np.array_equal(sa.is_na_real(v), sa.is_na_real(ev))
    assert np.array_equal(np.isnan(v), np.isnan(ev))
    if op in ("log1p", "expm1"):
        fin = ~np.isnan(ev)
        d = np.abs(vb[fin].astype(np.int64) - eb[fin].astype(np.int64))
        assert d.max(initial=0) <= 2
        assert np.array_equal(vb[~fin], eb[~fin])
    else:
        assert np.array_equal(vb, eb)


def operand(x, op, margin, vt, seed=3):
    rng = np.random.Generator(np.random.PCG64(seed))
    n = 1 if margin == 0 else x.dim[0] if margin == 1 else x.dim[1]
    if vt == "double":
        v = rng.standard_normal(n) * 3
        if op == "/":
            v[rng.random(n) < 0.1] = np.inf
        else:
            v[rng.random(n) < 0.1] = 0.0
        return v
    if vt == "logical":
        return np.ones(n, bool) if op == "/" else rng.random(n) < 0.7
    v = rng.integers(-3, 4, n).astype(np.int32)
    if op == "/":
        v[v == 0] = 2
    elif n > 1:
        v[::7] = 65536
    return v


def run_arith(x, op, v, margin, on_left):
    if margin == 2:
        return sa.sweep(x, 2, v, op)
    if on_left:
        return sa.Arith(v, op, x)
    return sa.Arith(x, op, v)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("margin", [0, 1, 2])
@pytest.mark.parametrize("vt", ["integer", "logical", "double"])
@pytest.mark.parametrize("op,on_left", [("*", False), ("*", True),
                                        ("/", False)])
def test_arith_vs_oracle(kind, margin, vt, op, on_left):
    if margin == 2 and on_left:
        pytest.skip("sweep() has the SVT on the left")
    x, _ = make_input(kind)
    v = operand(x, op, margin, vt)
    np_vt = np.asarray(v)
    vtype = "logical" if np_vt.dtype == bool else vt
    vv = np_vt.astype(np.int32) if np_vt.dtype == bool else np_vt
    r = run_arith(sa.to_device(x), op, v, margin, on_left)
    check(r, oracle(x, op, vv, vtype, margin), op)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("op", MATH)
def test_math_vs_oracle(kind, op):
    x, _ = make_input(kind)
    check(sa.Math(sa.to_device(x), op), oracle(x, op), op)


def test_host_input_matches_handle_input_and_input_unchanged():
    x, _ = make_input("double")
    h = sa.to_device(x)
    before = download(h)
    sf = np.linspace(0.5, 2.0, x.dim[1])
    a = sa.Math(sa.sweep(h, 2, sf, "/"), "log1p")
    b = sa.Math(sa.sweep(x, 2, sf, "/"), "log1p")
    for u, w in zip(download(a), download(b)):
        assert np.array_equal(np.asarray(u).view(np.uint8),
                              np.asarray(w).view(np.uint8))
    after = download(h)
    for u, w in zip(before, after):
        assert np.array_equal(np.asarray(u).view(np.uint8),
                              np.asarray(w).view(np.uint8))


def test_compaction_cases():
    a = np.zeros((100, 6), dtype=np.int32)
    a[::3, 0] = 4
    a[1::2, 1] = 1            # 1 // ... floor(1/3) empties this leaf
    a[[2, 50], 2] = [NA_I, 5]
    a[:, 4] = np.arange(1, 101)
    x = sa.SVT_SparseArray.from_dense(a, "integer", lacunar=False)
    h = sa.to_device(x)
    # a leaf that empties; dropped and kept entries interleave
    y = sa.Math(sa.Arith(h, "/", 3), "floor")
    y3 = oracle(x, "/", np.array([3.0]), "double")
    ys = sa.SVT_SparseArray((100, 6), "double", y3[0], y3[1], y3[2])
    check(y, oracle(ys, "floor"), "floor")
    assert download(y)[0][2] == download(y)[0][1]          # leaf 1 empty
    # x * 0L keeps only the NA
    z = h * 0
    p, o, v = download(z)
    assert list(o) == [2] and list(v) == [NA_I] and z.type == "integer"
    # everything dropped: nnz == 0 still answers colSums / rowSums
    b = np.where(a == NA_I, 7, a)
    e = sa.to_device(sa.SVT_SparseArray.from_dense(b, "integer")) * 0
    assert download(e)[1].size == 0
    assert np.array_equal(np.asarray(sa.colSums(e)), np.zeros(6))
    assert np.array_equal(np.asarray(sa.rowSums(e)), np.zeros(100))


def test_compaction_across_tile_boundaries():
    x = synth.poisson_svt(8000, 60, 0.3, seed=9, na_rate=1e-3)
    assert x.nnz > 3 * 32768
    y = sa.Math(sa.sweep(sa.to_device(x), 2,
                         np.arange(2, 62, dtype=np.float64), "/"), "floor")
    s = oracle(x, "/", np.arange(2, 62, dtype=np.float64), "double", 2)
    xs = sa.SVT_SparseArray((8000, 60), "double", s[0], s[1], s[2])
    check(y, oracle(xs, "floor"), "floor")


def _close(a, b, exact=False):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    m = ~np.isnan(b)
    if exact:
        assert np.array_equal(a[m], b[m])
    else:
        assert np.allclose(a[m], b[m], rtol=1e-12, atol=1e-300)


def _close_scaled(a, b, scale):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    m = ~np.isnan(b)
    assert np.all(np.abs(a[m] - b[m]) <= 1e-12 * (scale[m] + 1e-300))


def test_derived_handles_work_everywhere():
    x = synth.poisson_svt(3000, 80, 0.1, seed=4, na_rate=1e-3)
    cs = np.asarray(sa.colSums(x, na_rm=True))
    sf = cs / cs.mean()
    y = sa.Math(sa.sweep(sa.to_device(x), 2, sf, "/"), "log1p")
    t1 = oracle(x, "/", sf, "double", 2)
    x1 = sa.SVT_SparseArray(x.dim, "double", t1[0], t1[1], t1[2])
    t2 = oracle(x1, "log1p")
    ref = sa.SVT_SparseArray(x.dim, "double", t2[0], t2[1], t2[2])
    nrow, ncol = x.dim
    for na_rm in (False, True):
        _close(sa.colSums(y, na_rm=na_rm),
               port.colstats(nrow, ncol, *t2[:3], "double", "sum", na_rm)[0])
        _close(sa.colVars(y, na_rm=na_rm),
               port.colstats(nrow, ncol, *t2[:3], "double", "var1", na_rm)[0])
        _close(sa.rowSums(y, na_rm=na_rm),
               port.rowstats(nrow, ncol, *t2[:3], "double", "sum", na_rm)[0])
        _close(sa.rowMaxs(y, na_rm=na_rm),
               port.rowstats(nrow, ncol, *t2[:3], "double", "max", na_rm)[0])
        _close(sa.rowVars(y, na_rm=na_rm), sa.rowVars(ref, na_rm=na_rm))
    g = (np.arange(nrow) % 5) + 1
    _close(sa.rowsum(y, g), sa.rowsum(ref, g))
    # products: terms of both signs cancel, so the tolerance is relative to
    # the sum of the absolute values of the terms
    dense = np.zeros((nrow, ncol))
    for l in range(ncol):
        a, b = t2[0][l], t2[0][l + 1]
        dense[t2[1][a:b], l] = np.abs(np.nan_to_num(t2[2][a:b]))
    d = np.random.Generator(np.random.PCG64(2)).standard_normal((nrow, 8))
    _close_scaled(sa.crossprod(y, d),
                  port.crossprod(nrow, ncol, *t2[:3], "double", d),
                  dense.T @ np.abs(d))
    dd = np.random.Generator(np.random.PCG64(3)).standard_normal((ncol, 8))
    _close_scaled(sa.matmul(y, dd), sa.matmul(ref, dd), dense @ np.abs(dd))
    m, v = sa.rowMoments(y)
    _close(v, sa.rowVars(ref))
    p, i, vals = sa.to_csc(y)
    assert np.array_equal(p, t2[0]) and np.array_equal(i, t2[1])


def test_no_inherited_value_bound():
    """x uploaded int8-narrowed (|x| <= 127 known for free) must not hand
    that bound to x * 1000L."""
    x = synth.poisson_svt(4000, 50, 0.2, seed=6)
    assert x.vals.max() <= 127
    h = sa.to_device(x)
    y = h * 1000
    t = oracle(x, "*", np.array([1000], np.int32), "integer", 0)
    nrow, ncol = x.dim
    _close(sa.colVars(y),
           port.colstats(nrow, ncol, *t[:3], "integer", "var1")[0])
    _close(sa.rowVars(y), sa.rowVars(
        sa.SVT_SparseArray(x.dim, "integer", t[0], t[1], t[2])))
    _close(sa.rowMaxs(y),
           port.rowstats(nrow, ncol, *t[:3], "integer", "max")[0], exact=True)
    _close(sa.colSums(y), 1000.0 * np.asarray(sa.colSums(h)), exact=True)


def test_two_shards_equal_the_whole():
    from sparsearray_b200.device import DeviceSVT
    x = synth.poisson_svt(3000, 90, 0.1, seed=8, na_rate=1e-3)
    sf = np.linspace(0.3, 3.0, 90)
    whole = DeviceSVT.from_host(x).ewise("/", sf, margin=2)
    parts = [DeviceSVT.from_host(x, r).ewise("/", sf, margin=2)
             for r in ((0, 37), (37, 90))]
    wp, wo, wv = whole.download()
    (p0, o0, v0), (p1, o1, v1) = parts[0].download(), parts[1].download()
    assert np.array_equal(wp, np.concatenate([p0, p1[1:] + p0[-1]]))
    assert np.array_equal(wo, np.concatenate([o0, o1]))
    assert np.array_equal(wv.view(np.uint64),
                          np.concatenate([v0, v1]).view(np.uint64))


def test_scale_above_2_31_nonzeros():
    import torch
    from sparsearray_b200.device import DeviceSVT
    nrow, ncol, dens, seed, na = 33538, 1_000_000, 0.07, 2, 1e-6
    x = DeviceSVT.generate_poisson(nrow, ncol, dens, seed=seed, na_rate=na)
    assert x.nnz > 2**31
    cs, _ = x.colstats("sum", na_rm=True)
    y = x.ewise("*", np.array([2], np.int32))
    assert y.val_type == "integer" and y.nnz == x.nnz
    ycs, _ = y.colstats("sum", na_rm=True)
    assert torch.equal(ycs, 2 * cs)
    del y
    csh = cs.cpu().numpy()
    sf = csh / csh.mean()
    z = x.ewise("/", sf, margin=2)
    assert z.val_type == "double" and z.nnz == x.nnz
    got = {op: z.colstats(op)[0].cpu().numpy()
           for op in ("max", "min", "countNAs")}
    for l0 in (0, ncol - 1000):
        p, o, v = synth.poisson_csc(nrow, 1000, dens, seed=seed, na_rate=na,
                                    leaf0=l0)
        t = ewise_oracle.ewise(nrow, 1000, p, o, v, "integer", "/",
                       sf[l0:l0 + 1000], "double", 2)
        for op in ("max", "min", "countNAs"):
            exp = port.colstats(nrow, 1000, *t[:3], "double", op)[0]
            _close(got[op][l0:l0 + 1000], exp, exact=True)
