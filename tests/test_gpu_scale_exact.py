"""Every row and every column of the benchmark's matrices against exact host
answers.

bench.py times C2 (33,538 x 1e6 counts, d = 0.07, 2.35e9 nonzeros) and C5
(100,000 x 2e6 lacunar, d = 0.01).  Several code paths run only at that
scale or are chosen from the data: cyclic tiles with several tiles per
block, entry indices above 2^31, chunk-relative 32-bit strip positions, and
the accumulator classes launch_class() (csrc/svtgpu_rowstats.cu) picks from
max|x|.  This file holds each of them to exact values, not to identities.

The reference: one host pass over the matrix the device generated (chunks of
leaves sliced from the DeviceSVT tensors) collects exact integer histograms
per row and per column, from which sums, sums of squares, NA counts and
maxima follow exactly.  That pass reads device-made data, so the data are
checked on their own against the counter-based formula (synth.poisson_csc
for whole leaves, synth.poisson_row for single rows).

Run with -s to see the time of each stage and the largest variance error in
ulps."""
import concurrent.futures as cf
import ctypes
import gc
import math
import os
import time

import numpy as np
import pytest
import torch

import ewise_oracle
import sparsearray_b200 as sa
from sparsearray_b200 import _native as N
from sparsearray_b200 import synth
from sparsearray_b200.device import DeviceSVT
from sparsearray_b200.svt import SVT_SparseArray

pytestmark = pytest.mark.gpu

# the benchmark's matrices and operands (bench.py)
NROW, NCOL, DENS, SEED, NA_RATE = 33538, 1_000_000, 0.07, 2, 1e-6
C5_NROW, C5_NCOL, C5_DENS, C5_SEED = 100_000, 2_000_000, 0.01, 5
K_DENSE = 50
CHUNK = 10_000            # leaves per host chunk
NCODE = 16                # histogram slots: 0 = NA, 1..15 = the value
NA_INT = -2**31

TIMES = {}
VAR_ULP = {}              # largest ulp distance of each variance family


class _stage:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        self.t = time.perf_counter()
        return self

    def __exit__(self, *exc):
        dt = time.perf_counter() - self.t
        TIMES[self.name] = TIMES.get(self.name, 0.0) + dt
        print("[scale] %-44s %7.1f s" % (self.name, dt), flush=True)


def _release():
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    N.check(N.lib().svtgpu_release_cached_memory())


def _need(gb):
    total = torch.cuda.get_device_properties(0).total_memory
    if total < gb * 1e9:
        pytest.skip("needs %d GB of device memory, the device has %.0f"
                    % (gb, total / 1e9))


def _pool():
    return cf.ThreadPoolExecutor(max_workers=max(1, min(16, os.cpu_count())))


def _chunks(nleaf):
    return [(l0, min(l0 + CHUNK, nleaf)) for l0 in range(0, nleaf, CHUNK)]


def _moments(h):
    """Exact per-line quantities from an (n, NCODE) histogram."""
    h = np.asarray(h, dtype=np.int64)
    c = np.arange(h.shape[1], dtype=np.int64)
    rev = h[:, 1:][:, ::-1] > 0
    return {"nna": h[:, 0].copy(), "nval": h[:, 1:].sum(1), "s1": h @ c,
            "s2": h @ (c * c),
            "vmax": np.where(rev.any(1), h.shape[1] - 1 - rev.argmax(1), 0)}


def _leaf_index(ptr, l0, l1):
    return torch.repeat_interleave(
        torch.arange(l1 - l0), torch.from_numpy(np.diff(ptr[l0:l1 + 1])))


# ---------------------------------------------------------------------------
# exact references

def _c2_chunk(x, ptr, l0, l1, rg, cg):
    e0, e1 = int(ptr[l0]), int(ptr[l1])
    nl = l1 - l0
    o = x.offs[e0:e1].cpu().to(torch.int64)
    v = x.vals[e0:e1].cpu()
    na = v == NA_INT
    code = torch.where(na, 0, v).to(torch.int64)
    assert bool((na | ((code >= 1) & (code < NCODE))).all()), (l0, l1)
    leaf = _leaf_index(ptr, l0, l1)
    rowh = torch.bincount((o * 8 + cg[l0 + leaf]) * NCODE + code,
                          minlength=NROW * 8 * NCODE)
    colh = torch.bincount((leaf * 12 + rg[o]) * NCODE + code,
                          minlength=nl * 12 * NCODE).view(nl, 12, NCODE)
    cv = torch.arange(NCODE, dtype=torch.int64)
    gs1 = (colh * cv).sum(2).numpy()
    gna = colh[:, :, 0].numpy()
    return l0, rowh, _moments(colh.sum(1).numpy()), gs1, gna


def _c2_reference(x, rg, cg):
    ptr = x.leaf_ptr.cpu().numpy()
    rg_t = torch.from_numpy(rg.astype(np.int64) - 1)
    cg_t = torch.from_numpy(cg.astype(np.int64) - 1)
    rowh = torch.zeros(NROW * 8 * NCODE, dtype=torch.int64)
    col = {k: np.zeros(NCOL, np.int64)
           for k in ("nna", "nval", "s1", "s2", "vmax")}
    rowsum_s1 = np.zeros((12, NCOL), np.int64)
    rowsum_na = np.zeros((12, NCOL), np.int64)
    with _pool() as ex:
        futs = [ex.submit(_c2_chunk, x, ptr, l0, l1, rg_t, cg_t)
                for l0, l1 in _chunks(NCOL)]
        for f in cf.as_completed(futs):
            l0, rh, cm, gs1, gna = f.result()
            rowh += rh
            l1 = l0 + gs1.shape[0]
            for k in col:
                col[k][l0:l1] = cm[k]
            rowsum_s1[:, l0:l1] = gs1.T
            rowsum_na[:, l0:l1] = gna.T
    rowh = rowh.view(NROW, 8, NCODE).numpy()
    cv = np.arange(NCODE, dtype=np.int64)
    return {"ptr": ptr, "row": _moments(rowh.sum(1)), "col": col,
            "rowsum": (rowsum_s1, rowsum_na),
            "colsum": (rowh @ cv, rowh[:, :, 0].copy())}


def _c5_chunk(x, ptr, l0, l1, rg, cg):
    e0, e1 = int(ptr[l0]), int(ptr[l1])
    nl = l1 - l0
    o = x.offs[e0:e1].cpu().to(torch.int64)
    leaf = _leaf_index(ptr, l0, l1)
    rowh = torch.bincount(o * 8 + cg[l0 + leaf], minlength=C5_NROW * 8)
    colg = torch.bincount(leaf * 12 + rg[o], minlength=nl * 12).view(nl, 12)
    return l0, rowh, colg.numpy()


def _c5_reference(x, rg, cg):
    ptr = x.leaf_ptr.cpu().numpy()
    rg_t = torch.from_numpy(rg.astype(np.int64) - 1)
    cg_t = torch.from_numpy(cg.astype(np.int64) - 1)
    rowh = torch.zeros(C5_NROW * 8, dtype=torch.int64)
    rowsum = np.zeros((12, C5_NCOL), np.int64)
    with _pool() as ex:
        futs = [ex.submit(_c5_chunk, x, ptr, l0, l1, rg_t, cg_t)
                for l0, l1 in _chunks(C5_NCOL)]
        for f in cf.as_completed(futs):
            l0, rh, cgc = f.result()
            rowh += rh
            rowsum[:, l0:l0 + cgc.shape[0]] = cgc.T
    rowh = rowh.view(C5_NROW, 8).numpy()
    return {"ptr": ptr, "row_count": rowh.sum(1), "col_count": np.diff(ptr),
            "colsum": rowh, "rowsum": rowsum}


def _sample_rows(nrow, extra, rng, n):
    rows = {0, 1, nrow - 1}
    for t in range(2, 9):
        for j in range(1, t):
            m = (nrow * j // t) // 32
            rows.update((32 * m - 1, 32 * m))
    rows.update(int(r) for r in extra)
    while len(rows) < n:
        rows.add(int(rng.integers(0, nrow)))
    return sorted(r for r in rows if 0 <= r < nrow)


def _sample_leaves(ptr, nleaf, rng, n):
    l31 = int(np.searchsorted(ptr, 2**31, side="right")) - 1
    assert ptr[l31] <= 2**31 < ptr[l31 + 1]
    leaves = {0, nleaf - 1, l31}
    while len(leaves) < n:
        leaves.add(int(rng.integers(0, nleaf)))
    return sorted(leaves), l31


@pytest.fixture(scope="module")
def c2():
    _need(120)
    rng = np.random.Generator(np.random.PCG64(3))
    rg = rng.integers(1, 13, size=NROW).astype(np.int32)
    cg = rng.integers(1, 9, size=NCOL).astype(np.int32)
    with _stage("C2 generate"):
        x = DeviceSVT.generate_poisson(NROW, NCOL, DENS, seed=SEED,
                                       na_rate=NA_RATE)
    assert x.nnz > 2**31
    with _stage("C2 host reference pass"):
        ref = _c2_reference(x, rg, cg)
    ref["rg"], ref["cg"] = rg, cg
    ref["M0"] = int(ref["row"]["vmax"].max())
    ref["rows"] = _sample_rows(
        NROW, np.flatnonzero(ref["row"]["nna"])[:12],
        np.random.Generator(np.random.PCG64(17)), 150)
    yield x, ref
    del x
    _release()


@pytest.fixture(scope="module")
def c5():
    _need(60)
    rng = np.random.Generator(np.random.PCG64(3))
    rg = rng.integers(1, 13, size=C5_NROW).astype(np.int32)
    cg = rng.integers(1, 9, size=C5_NCOL).astype(np.int32)
    with _stage("C5 generate"):
        x = DeviceSVT.generate_poisson(C5_NROW, C5_NCOL, C5_DENS,
                                       seed=C5_SEED, lacunar=True)
    with _stage("C5 host reference pass"):
        ref = _c5_reference(x, rg, cg)
    ref["rg"], ref["cg"] = rg, cg
    yield x, ref
    del x
    _release()


# ---------------------------------------------------------------------------
# expectations and comparisons

def _expect(m, n_other, op, na_rm, k=1):
    """R's answer for the lines of y = k * x from x's exact line quantities
    (m = _moments()); every line also holds implicit zeros.  Variances come
    back in long double, the exact rational rounded to 64 bits."""
    nna, s1, s2, vmax = m["nna"], m["s1"], m["s2"], m["vmax"]
    n = n_other - nna if na_rm else np.full_like(nna, n_other)
    if op == "countNAs":
        return nna.astype(np.float64)
    if op == "sum":
        e = (k * s1).astype(np.float64)
    elif op == "mean":
        e = (k * s1).astype(np.float64) / n.astype(np.float64)
    elif op == "var1":
        num = n * s2 - s1 * s1
        e = num.astype(np.longdouble) * np.longdouble(k * k) / \
            (n.astype(np.longdouble) * (n - 1))
    elif op == "max":
        e = (k * vmax if k > 0 else 0 * vmax).astype(np.float64)
    elif op == "min":
        e = (0 * vmax if k > 0 else k * vmax).astype(np.float64)
    else:
        raise ValueError(op)
    if not na_rm:
        e[nna > 0] = np.nan
    return e


def _f64(t):
    a = t.cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
    if a.dtype == np.int32:
        out = a.astype(np.float64)
        out[a == NA_INT] = np.nan
        return out
    return a.astype(np.float64)


def _exact(got, exp, what):
    got = _f64(got)
    exp = np.asarray(exp, dtype=np.float64)
    assert got.shape == exp.shape, (what, got.shape, exp.shape)
    bad = ~((got == exp) | (np.isnan(got) & np.isnan(exp)))
    if bad.any():
        i = np.flatnonzero(bad)
        raise AssertionError("%s: %d of %d differ; first at %s: got %r, "
                             "exact %r" % (what, i.size, got.size, i[:5],
                                           got[i[:5]], exp[i[:5]]))


def _var_close(got, exp_ld, what, family):
    """<= 1e-12 relative to the exact value; records the ulp distance."""
    got = _f64(got)
    exp = exp_ld.astype(np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(exp)), what
    ok = ~np.isnan(exp)
    g, e, el = got[ok], exp[ok], exp_ld[ok]
    assert (e >= 0).all() and (g >= 0).all(), what
    rel = np.abs(g.astype(np.longdouble) - el) / \
        np.where(el == 0, 1, el)
    ulp = int(np.abs(g.view(np.int64) - e.view(np.int64)).max()) \
        if g.size else 0
    VAR_ULP[family] = max(VAR_ULP.get(family, 0), ulp)
    worst = float(rel.max()) if rel.size else 0.0
    assert worst <= 1e-12, "%s: relative error %.3g at %s" % (
        what, worst, np.flatnonzero(ok)[int(np.argmax(rel))])


def _check(got, m, n_other, op, na_rm, what, k=1, family="var"):
    exp = _expect(m, n_other, op, na_rm, k)
    if op == "var1":
        _var_close(got, exp, what, family)
    else:
        _exact(got, exp, what)


COL_OPS = ("sum", "mean", "var1", "max", "min", "countNAs")
ROW_OPS = ("sum", "max", "min", "countNAs")


def _check_cols(x, ref, tag, k=1, ops=COL_OPS):
    for na_rm in (False, True):
        for op in ops:
            _check(x.colstats(op, na_rm=na_rm)[0], ref["col"], NROW, op,
                   na_rm, "%s col %s na_rm=%s" % (tag, op, na_rm), k,
                   "colVars")


def _check_rows(x, ref, tag, k=1):
    for na_rm in (False, True):
        for op in ROW_OPS:
            _check(x.rowstats(op, na_rm=na_rm)[0], ref["row"], NCOL, op,
                   na_rm, "%s row %s na_rm=%s" % (tag, op, na_rm), k)
        mean, var = x.rowmoments(na_rm=na_rm)
        _check(mean, ref["row"], NCOL, "mean", na_rm,
               "%s rowMeans na_rm=%s" % (tag, na_rm), k)
        _check(var, ref["row"], NCOL, "var1", na_rm,
               "%s rowVars na_rm=%s" % (tag, na_rm), k, family="rowVars")


def _check_rows_hist_on_off(x, ref, tag, monkeypatch, k=1):
    _check_rows(x, ref, tag + " [hist auto]", k)
    with monkeypatch.context() as mp:
        mp.setenv("SVTGPU_ROW_HIST", "off")
        _check_rows(x, ref, tag + " [hist off]", k)


# ---------------------------------------------------------------------------
# 1. the reference against the generator's formula

def test_c2_reference_matches_formula(c2):
    x, ref = c2
    ptr = ref["ptr"]
    with _stage("C2 reference vs formula"):
        leaves, l31 = _sample_leaves(
            ptr, NCOL, np.random.Generator(np.random.PCG64(19)), 203)
        for l in leaves:
            p, o, v = synth.poisson_csc(NROW, 1, DENS, seed=SEED,
                                        na_rate=NA_RATE, leaf0=l)
            e0, e1 = int(ptr[l]), int(ptr[l + 1])
            assert e1 - e0 == p[1], l
            assert np.array_equal(x.offs[e0:e1].cpu().numpy(), o), l
            assert np.array_equal(x.vals[e0:e1].cpu().numpy(), v), l
        m = ref["row"]
        for i in ref["rows"]:
            c, v, na = synth.poisson_row(NROW, NCOL, i, DENS, seed=SEED,
                                         na_rate=NA_RATE)
            got = (m["nna"][i], m["nval"][i], m["s1"][i], m["s2"][i],
                   m["vmax"][i])
            w = v[~na]
            exp = (na.sum(), w.size, w.sum(), (w * w).sum(),
                   w.max() if w.size else 0)
            assert got == exp, (i, got, exp)
    # the rows and columns all hold implicit zeros (the expectations of
    # min / max rely on it) and the sample holds rows with NAs
    assert (m["nval"] + m["nna"] < NCOL).all()
    assert (ref["col"]["nval"] + ref["col"]["nna"] < NROW).all()
    assert any(m["nna"][i] > 0 for i in ref["rows"])
    assert int(m["nna"].sum()) == int(ref["col"]["nna"].sum()) > 0
    assert int(m["s1"].sum()) == int(ref["col"]["s1"].sum())


def test_c5_reference_matches_formula(c5):
    x, ref = c5
    ptr = ref["ptr"]
    with _stage("C5 reference vs formula"):
        rng = np.random.Generator(np.random.PCG64(23))
        leaves = {0, C5_NCOL - 1} | set(rng.integers(0, C5_NCOL, 200).tolist())
        for l in sorted(leaves):
            p, o, _ = synth.poisson_csc(C5_NROW, 1, C5_DENS, seed=C5_SEED,
                                        leaf0=l, lacunar=True)
            e0, e1 = int(ptr[l]), int(ptr[l + 1])
            assert np.array_equal(x.offs[e0:e1].cpu().numpy(), o), l
        rng = np.random.Generator(np.random.PCG64(29))
        rows = _sample_rows(C5_NROW, [65535, 65536, C5_NROW - 2] +
                            rng.integers(65536, C5_NROW, 30).tolist(),
                            rng, 100)
        assert sum(r >= 65536 for r in rows) >= 30
        for i in rows:
            c, _, _ = synth.poisson_row(C5_NROW, C5_NCOL, i, C5_DENS,
                                        seed=C5_SEED)
            assert ref["row_count"][i] == c.size, i
    assert int(ref["row_count"].sum()) == int(ptr[-1])


# ---------------------------------------------------------------------------
# 2. statistics at C2, every entry

def test_c2_statistics(c2, monkeypatch):
    x, ref = c2
    with _stage("C2 statistics"):
        _check_cols(x, ref, "C2")
        _check_rows_hist_on_off(x, ref, "C2", monkeypatch)


def test_c2_group_sums(c2):
    x, ref = c2
    with _stage("C2 rowsum / colsum"):
        for na_rm in (False, True):
            got, ov, _ = x.rowsum(ref["rg"], 12, na_rm=na_rm)
            assert not ov
            s1, nna = ref["rowsum"]
            exp = s1.astype(np.float64)
            if not na_rm:
                exp[nna > 0] = np.nan
            _exact(got, exp, "C2 rowsum(rg, 12) na_rm=%s" % na_rm)
            got, ov, _ = x.colsum(ref["cg"], 8, na_rm=na_rm)
            assert not ov
            s1, nna = ref["colsum"]
            exp = s1.astype(np.float64)
            if not na_rm:
                exp[nna > 0] = np.nan
            _exact(got, exp, "C2 colsum(cg, 8) na_rm=%s" % na_rm)


# ---------------------------------------------------------------------------
# 3. a ladder of value ranges: y = x * k

def _colvar_bound_32bit():
    """Largest known bound B for which the column kernels accumulate sums
    of squares in 32 bits (svtgpu_colstats: a lane sees at most
    nrow / 32 + 2 values)."""
    per_lane = NROW // 32 + 2
    b = 0
    while per_lane < 0x7FFFFFFF // ((b + 1) * (b + 1) + 1):
        b += 1
    return b


def _ladder(M0):
    """[(limit, inclusive, what)] and the k that land on both sides."""
    table = [
        (22, True, "row_hist moments / packed strip moments (M^2 * 64 <= "
                   "32767)"),
        (_colvar_bound_32bit(), True, "32-bit colVars sums of squares "
                                      "once max|x| is cached"),
        (5792, True, "int32 sum-of-squares row accumulators (F >= 64)"),
        (65535, False, "packed row min / max strips"),
        (65536, False, "one-pass integer colVars guard"),
        (33554431, True, "int32 row sum accumulators with F >= 64"),
    ]
    ks = set()
    for lim, incl, _ in table:
        k_in = (lim if incl else lim - 1) // M0
        assert k_in >= 1
        ks.update((k_in, k_in + 1))
    ks.add((2**31 - 1) // M0)          # double accumulators, no overflow
    ks.add(-max(1, 22 // M0))          # vmin < 0: no histogram, no packing
    return table, sorted(ks)


def test_c2_value_ladder(c2, monkeypatch):
    x, ref = c2
    M0 = ref["M0"]
    table, ks = _ladder(M0)
    print("\n[scale] M0 = max|x| = %d; k = %s" % (M0, ks))
    for lim, incl, what in table:
        inside = [k for k in ks if (abs(k) * M0 <= lim if incl
                                    else abs(k) * M0 < lim)]
        outside = [k for k in ks if k > 0 and k not in inside]
        below = max(k * M0 for k in inside if k > 0)
        above = min(k * M0 for k in outside)
        print("[scale]   %s %-9d %s: k*M0 = %d inside, %d outside"
              % ("<=" if incl else "< ", lim, what, below, above))
        assert (below <= lim if incl else below < lim)
        assert (above > lim if incl else above >= lim)
    top = max(ks) * M0
    assert 33554431 < top <= 2**31 - 1
    assert min(ks) < 0
    for k in ks:
        with _stage("C2 ladder"):
            y = x.ewise("*", np.array([k], np.int32))
            assert y.val_type == "integer" and y.nnz == x.nnz
            assert y.warnings == [], (k, y.warnings)
            tag = "C2*%d" % k
            # colVars on the fresh result (no cached bound), then the row
            # operations (which cache max|y|), then colVars again
            _check_cols(y, ref, tag, k, ops=("var1",))
            _check_rows_hist_on_off(y, ref, tag, monkeypatch, k)
            _check_cols(y, ref, tag + " [bound cached]", k)
            del y
            _release()


# ---------------------------------------------------------------------------
# 4. C2 as double, and the double element-wise chain

def test_c2_as_double(c2):
    x, ref = c2
    with _stage("C2 double generate"):
        xd = DeviceSVT.generate_poisson(NROW, NCOL, DENS, seed=SEED,
                                        na_rate=NA_RATE, val_type="double")
    assert xd.nnz == x.nnz
    with _stage("C2 double statistics"):
        for na_rm in (False, True):
            for op in COL_OPS:
                _check(xd.colstats(op, na_rm=na_rm)[0], ref["col"], NROW, op,
                       na_rm, "C2d col %s na_rm=%s" % (op, na_rm),
                       family="colVars (double)")
        for na_rm in (False, True):
            for op in ROW_OPS:
                _check(xd.rowstats(op, na_rm=na_rm)[0], ref["row"], NCOL, op,
                       na_rm, "C2d row %s na_rm=%s" % (op, na_rm))
            mean, var = xd.rowmoments(na_rm=na_rm)
            _check(mean, ref["row"], NCOL, "mean", na_rm,
                   "C2d rowMeans na_rm=%s" % na_rm)
            _check(var, ref["row"], NCOL, "var1", na_rm,
                   "C2d rowVars na_rm=%s" % na_rm,
                   family="rowVars (double)")
    del xd
    _release()


def _ulps_within(got, exp, n, what, ptr):
    ulp = np.abs(got.view(np.int64) - exp.view(np.int64))
    bad = np.flatnonzero(ulp > n)
    if bad.size:
        raise AssertionError(
            "%s: %d columns beyond %d ulp; first %s: got %r, exact %r, "
            "entries %r" % (what, bad.size, n, bad[:8], got[bad[:8]],
                            exp[bad[:8]], ptr[bad[:8]]))


def _max_skipping_na(w, starts):
    # NA_real_ is a signalling NaN, which numpy's fmax reduction does not
    # reliably skip (it restarts the running maximum), so mask it first
    return np.maximum.reduceat(np.where(np.isnan(w), -np.inf, w), starts)


def _chain_chunk(x, ptr, l0, l1, sf):
    e0, e1 = int(ptr[l0]), int(ptr[l1])
    p = ptr[l0:l1 + 1] - e0
    o = x.offs[e0:e1].cpu().numpy()
    v = x.vals[e0:e1].cpu().numpy()
    t = ewise_oracle.ewise(NROW, l1 - l0, p, o, v, "integer", "/",
                           sf[l0:l1], "double", 2)
    zmax = _max_skipping_na(t[2], p[:-1])
    t = ewise_oracle.ewise(NROW, l1 - l0, *t[:3], "double", "log1p")
    w = t[2]
    assert np.array_equal(t[0], p)
    starts = p[:-1]
    wz = np.where(np.isnan(w), 0.0, w)
    return (l0, zmax, _max_skipping_na(w, starts),
            np.add.reduceat(wz.astype(np.longdouble), starts),
            np.add.reduceat(np.abs(wz), starts))


def test_c2_log1p_sweep_chain(c2):
    x, ref = c2
    ptr = ref["ptr"]
    assert (np.diff(ptr) > 0).all()          # reduceat needs no empty leaf
    with _stage("C2 chain on device"):
        cs = x.colstats("sum", na_rm=True)[0].cpu().numpy()
        sf = cs / cs.mean()
        z = x.ewise("/", sf, margin=2)
        w = z.ewise("log1p")
        z_max = z.colstats("max", na_rm=True)[0].cpu().numpy()
        w_max0 = w.colstats("max", na_rm=True)[0].cpu().numpy()
        del z                  # w must not depend on its operand's arrays
        _release()
        got_max = w.colstats("max", na_rm=True)[0].cpu().numpy()
        got_min = w.colstats("min", na_rm=True)[0].cpu().numpy()
        got_sum = w.colstats("sum", na_rm=True)[0].cpu().numpy()
        got_cna = w.colstats("countNAs")[0].cpu().numpy()
        got_rows = w.rowstats("sum", na_rm=True)[0].cpu().numpy()
        del w
        _release()
    errors = []

    def check(fn, *args):
        try:
            fn(*args)
        except AssertionError as e:
            errors.append(str(e))

    check(_exact, got_max, w_max0, "chain colMaxs after its operand was freed")
    check(_exact, got_cna, ref["col"]["nna"], "chain colCountNAs")
    with _stage("C2 chain host reference"):
        ewise_oracle.lib()
        e_max = np.empty(NCOL)
        e_zmax = np.empty(NCOL)
        e_sum = np.empty(NCOL, np.longdouble)
        e_abs = np.empty(NCOL)
        with _pool() as ex:
            for l0, zmx, mx, s, a in ex.map(
                    lambda c: _chain_chunk(x, ptr, c[0], c[1], sf),
                    _chunks(NCOL)):
                n = mx.size
                e_zmax[l0:l0 + n], e_max[l0:l0 + n] = zmx, mx
                e_sum[l0:l0 + n], e_abs[l0:l0 + n] = s, a
    check(_ulps_within, z_max, e_zmax, 0, "x / sf colMaxs", ptr)
    check(_ulps_within, got_max, e_max, 2, "chain colMaxs", ptr)
    check(_exact, got_min, np.zeros(NCOL), "chain colMins")
    err = np.abs(got_sum.astype(np.longdouble) - e_sum)
    bad = np.flatnonzero(err > 1e-12 * e_abs)
    if bad.size:
        errors.append("chain colSums: %d columns, first %s" % (bad.size,
                                                              bad[:8]))
    assert not errors, "\n".join(errors)
    with _stage("C2 chain sampled rows"):
        for i in ref["rows"]:
            c, v, na = synth.poisson_row(NROW, NCOL, i, DENS, seed=SEED,
                                         na_rate=NA_RATE)
            p = np.zeros(NCOL + 1, np.int64)
            p[c + 1] = 1
            p = np.cumsum(p)
            vi = np.where(na, NA_INT, v).astype(np.int32)
            t = ewise_oracle.ewise(1, NCOL, p, np.zeros(c.size, np.int32),
                                   vi, "integer", "/", sf, "double", 2)
            t = ewise_oracle.ewise(1, NCOL, *t[:3], "double", "log1p")
            terms = [float(u) for u in t[2] if not math.isnan(u)]
            exp = math.fsum(terms)
            bound = 1e-12 * math.fsum(abs(u) for u in terms)
            assert abs(got_rows[i] - exp) <= bound, (i, got_rows[i], exp)


# ---------------------------------------------------------------------------
# 5. C5, every entry

def test_c5_statistics(c5, monkeypatch):
    x, ref = c5
    cnt = ref["row_count"]
    m = {"nna": np.zeros_like(cnt), "s1": cnt, "s2": cnt,
         "vmax": (cnt > 0).astype(np.int64)}
    assert (cnt < C5_NCOL).all() and (ref["col_count"] < C5_NROW).all()
    with _stage("C5 statistics"):
        _exact(x.colstats("sum")[0], ref["col_count"], "C5 colSums")
        for hist in ("auto", "off"):
            with monkeypatch.context() as mp:
                mp.setenv("SVTGPU_ROW_HIST", hist)
                tag = "C5 [hist %s]" % hist
                _check(x.rowstats("sum")[0], m, C5_NCOL, "sum", False,
                       tag + " rowSums")
                _check(x.rowstats("max")[0], m, C5_NCOL, "max", False,
                       tag + " rowMaxs")
                mean, var = x.rowmoments()
                _check(mean, m, C5_NCOL, "mean", False, tag + " rowMeans")
                _check(var, m, C5_NCOL, "var1", False, tag + " rowVars",
                       family="rowVars (C5)")
                got, ov, _ = x.colsum(ref["cg"], 8)
                assert not ov
                _exact(got, ref["colsum"], tag + " colsum(cg5, 8)")
                got, ov, _ = x.rowsum(ref["rg"], 12)
                assert not ov
                _exact(got, ref["rowsum"], tag + " rowsum(rg5, 12)")


# ---------------------------------------------------------------------------
# 6. products and the transpose at C2 (double)

def test_c2_products_and_transpose(c2):
    x, ref = c2
    ptr = ref["ptr"]
    rng = np.random.Generator(np.random.PCG64(7))
    Yh = np.asfortranarray(rng.standard_normal((NROW, K_DENSE)))
    Dh = np.asfortranarray(rng.standard_normal((NCOL, K_DENSE)))
    with _stage("C2 double generate"):
        xd = DeviceSVT.generate_poisson(NROW, NCOL, DENS, seed=SEED,
                                        na_rate=NA_RATE, val_type="double")
    with _stage("C2 crossprod"):
        Y = torch.from_numpy(np.ascontiguousarray(Yh)).cuda()
        cp = xd.crossprod(Y).view(K_DENSE, NCOL)
        srng = np.random.Generator(np.random.PCG64(31))
        leaves, l31 = _sample_leaves(ptr, NCOL, srng, 1500)
        for mm in srng.integers(1, NCOL // 512, 250):
            leaves += [512 * int(mm) - 1, 512 * int(mm)]
        leaves = sorted(set(leaves))
        got = cp[:, torch.tensor(leaves, device="cuda")].cpu().numpy()
        del cp, Y
        Yl = Yh.astype(np.longdouble)
        for j, l in enumerate(leaves):
            e0, e1 = int(ptr[l]), int(ptr[l + 1])
            o = xd.offs[e0:e1].cpu().numpy()
            v = xd.vals[e0:e1].cpu().numpy()
            if np.isnan(v).any():
                assert np.isnan(got[:, j]).all(), l
                continue
            exp = v.astype(np.longdouble) @ Yl[o]
            bound = 1e-12 * (np.abs(v) @ np.abs(Yh[o]))
            err = np.abs(got[:, j] - exp)
            assert (err <= bound).all(), ("crossprod leaf", l)
    with _stage("C2 matmul"):
        D = torch.from_numpy(np.ascontiguousarray(Dh)).cuda()
        mm_ = xd.matmul(D).view(NROW, K_DENSE)
        rows = ref["rows"]
        got = mm_[torch.tensor(rows, device="cuda")].cpu().numpy()
        del mm_, D
        for j, i in enumerate(rows):
            c, v, na = synth.poisson_row(NROW, NCOL, i, DENS, seed=SEED,
                                         na_rate=NA_RATE)
            if na.any():
                assert np.isnan(got[j]).all(), i
                continue
            exp = v.astype(np.longdouble) @ Dh[c].astype(np.longdouble)
            bound = 1e-12 * (np.abs(v) @ np.abs(Dh[c]))
            assert (np.abs(got[j] - exp) <= bound).all(), ("matmul row", i)
    with _stage("C2 rowstats via transpose"):
        L = N.lib()
        for na_rm in (False, True):
            for op in ("sum", "max", "var1"):
                out = np.zeros(NROW, np.float64)
                warn = ctypes.c_int(0)
                N.check(L.svtgpu_rowstats_via_transpose(
                    xd._h, N.OPCODES[op], int(na_rm),
                    ctypes.c_double(synth.NA_REAL),
                    out.ctypes.data_as(ctypes.c_void_p), ctypes.byref(warn)))
                _check(out, ref["row"], NCOL, op, na_rm,
                       "C2d via transpose %s na_rm=%s" % (op, na_rm),
                       family="rowVars (transpose)")
    del xd
    _release()


# ---------------------------------------------------------------------------
# 7. the upload path at scale

def _upload_and_check(svt, x, nrow, ncol, exp_rows, exp_cols, exp_var,
                      tag, extra=()):
    with _stage(tag + " to_device"):
        r = sa.to_device(svt)
    svt.release()
    with _stage(tag + " R-level statistics"):
        _exact(np.asarray(sa.rowSums(r, na_rm=True)), exp_rows,
               tag + " rowSums")
        _exact(np.asarray(sa.colSums(r, na_rm=True)), exp_cols,
               tag + " colSums")
        _var_close(np.asarray(sa.rowVars(r, na_rm=True), dtype=np.float64),
                   exp_var, tag + " rowVars", "rowVars (" + tag + ")")
        for fn, exp, what in extra:
            _exact(np.asarray(fn(r)), exp, tag + " " + what)
    if x.nnz > 2**31 - 1:
        # R's dgCMatrix holds at most INT_MAX nonzeros: to_csc refuses, as
        # as(x, "dgCMatrix") does
        with pytest.raises(Exception, match="too many nonzero values"):
            sa.to_csc(r)
        r.release()
        del r
        _release()
        return
    with _stage(tag + " to_csc"):
        p, i, v = sa.to_csc(r)
        r.release()
        del r
        ptr = x.leaf_ptr.cpu().numpy()
        assert np.array_equal(np.asarray(p, dtype=np.int64), ptr)
        for l0, l1 in _chunks(ncol):
            e0, e1 = int(ptr[l0]), int(ptr[l1])
            assert np.array_equal(i[e0:e1], x.offs[e0:e1].cpu().numpy()), l0
            if x.vals is not None:
                assert np.array_equal(v[e0:e1], x.vals[e0:e1].cpu().numpy())
            elif v is not None:
                assert (v[e0:e1] == 1).all()
        del p, i, v
    _release()


def test_c2_upload(c2):
    x, ref = c2
    with _stage("C2 host SVT"):
        svt = SVT_SparseArray((NROW, NCOL), "integer",
                              x.leaf_ptr.cpu().numpy(),
                              x.offs[:x.nnz].cpu().numpy(),
                              x.vals[:x.nnz].cpu().numpy())
    _upload_and_check(svt, x, NROW, NCOL,
                      _expect(ref["row"], NCOL, "sum", True),
                      _expect(ref["col"], NROW, "sum", True),
                      _expect(ref["row"], NCOL, "var1", True), "C2",
                      extra=[(lambda r: sa.colMaxs(r), _expect(
                                  ref["col"], NROW, "max", False), "colMaxs"),
                             (lambda r: sa.rowMaxs(r), _expect(
                                  ref["row"], NCOL, "max", False), "rowMaxs"),
                             (lambda r: sa.colCountNAs(r),
                              ref["col"]["nna"], "colCountNAs"),
                             (lambda r: sa.rowCountNAs(r),
                              ref["row"]["nna"], "rowCountNAs")])
    del svt
    gc.collect()


def test_c5_upload(c5):
    x, ref = c5
    cnt = ref["row_count"]
    m = {"nna": np.zeros_like(cnt), "s1": cnt, "s2": cnt,
         "vmax": (cnt > 0).astype(np.int64)}
    with _stage("C5 host SVT"):
        svt = SVT_SparseArray((C5_NROW, C5_NCOL), "integer",
                              x.leaf_ptr.cpu().numpy(),
                              x.offs[:x.nnz].cpu().numpy(), None)
    _upload_and_check(svt, x, C5_NROW, C5_NCOL, cnt.astype(np.float64),
                      ref["col_count"].astype(np.float64),
                      _expect(m, C5_NCOL, "var1", True), "C5")
    del svt
    gc.collect()


def test_zz_report():
    """Prints the stage times and the largest variance ulp distances."""
    print("\n[scale] stage times (s): " + ", ".join(
        "%s %.1f" % kv for kv in TIMES.items()))
    print("[scale] total %.1f s" % sum(TIMES.values()))
    print("[scale] largest variance distance (ulp): " + ", ".join(
        "%s %d" % kv for kv in VAR_ULP.items()))
