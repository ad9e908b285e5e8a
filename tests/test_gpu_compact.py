"""The compact copy of a device matrix (int8 values, uint16 row offsets):
when it is built, which arrays it holds, and that colSums / colMeans /
rowSums / rowMeans / rowVars read from it are bit-identical to the wide
kernels that run on the first call of a fresh handle."""
import ctypes

import numpy as np
import pytest
import torch

from sparsearray_b200 import _native as N
from sparsearray_b200 import synth
from sparsearray_b200.device import DeviceSVT

pytestmark = pytest.mark.gpu

NA_INT = -2 ** 31
PAD = 64
TILE = 32768        # row_hist entries per cyclic tile
BATCH = 16384       # entries per batch of the compact row_hist


def compact_bytes(d):
    b = ctypes.c_int64(-1)
    N.check(N.lib().svtgpu_matrix_compact_bytes(d._h, ctypes.byref(b)))
    return b.value


def structure(nrow, ncol, seed):
    """leaf_ptr and row offsets with empty leaves, one-entry leaves, leaves
    of every length (so leaf starts fall anywhere in a 16-byte word) and nnz
    that is a multiple of neither 16 nor a tile."""
    rng = np.random.default_rng(seed)
    dens = rng.uniform(0.0, 0.4, size=ncol)
    dens[rng.random(ncol) < 0.05] = 0.0
    lens = rng.binomial(nrow, dens)
    lens[rng.random(ncol) < 0.05] = 1
    offs = np.empty(int(lens.sum()), dtype=np.int32)
    ptr = np.zeros(ncol + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(lens)
    for j in range(ncol):
        k = int(lens[j])
        if k == nrow:
            offs[ptr[j]:ptr[j + 1]] = np.arange(nrow)
        elif k:
            offs[ptr[j]:ptr[j + 1]] = np.sort(
                rng.choice(nrow, size=k, replace=False))
    nnz = int(ptr[-1])
    if nnz % 16 == 0 or nnz % TILE == 0:
        # drop the last entry of the last non-empty leaf
        j = int(np.flatnonzero(lens)[-1])
        lens[j] -= 1
        ptr[j + 1:] -= 1
        offs = offs[:-1]
    return ptr, offs


def values(ptr, kind, seed):
    """kind: "signed" (every value in [-127, 127] \\ {0}, both ends present),
    "small" (1..22, the packed row moments), "logical"; NA at the first and
    last entry of some leaves and around every tile and batch edge."""
    rng = np.random.default_rng(seed)
    nnz = int(ptr[-1])
    if kind == "signed":
        v = rng.integers(1, 128, size=nnz).astype(np.int32)
        v *= np.where(rng.random(nnz) < 0.5, -1, 1).astype(np.int32)
        v[:2] = (127, -127)
    elif kind == "small":
        v = rng.integers(1, 23, size=nnz).astype(np.int32)
    else:
        v = (rng.random(nnz) < 0.7).astype(np.int32)
    na = rng.random(nnz) < 1e-3
    firsts = ptr[:-1][np.diff(ptr) > 0]
    lasts = ptr[1:][np.diff(ptr) > 0] - 1
    na[firsts[::7]] = True
    na[lasts[::5]] = True
    for step in (BATCH, TILE):
        for d in (-1, 0, 1):
            e = np.arange(step, nnz, step) + d
            na[e[(e >= 0) & (e < nnz)]] = True
    v[na] = NA_INT
    return v


def on_device(nrow, ptr, offs, vals, vtype):
    def dev(a, dtype):
        t = torch.zeros(len(a) + PAD, dtype=dtype, device="cuda")
        t[:len(a)] = torch.from_numpy(np.ascontiguousarray(a))
        return t
    lp = torch.from_numpy(ptr).cuda()
    o = dev(offs, torch.int32)
    v = None if vals is None else dev(
        vals, torch.float64 if vtype == "double" else torch.int32)
    return lp, o, v


OPS = ("colSums", "colMeans", "rowSums", "rowMoments")


def run(d, op, na_rm):
    if op == "colSums":
        return [d.colstats("sum", na_rm=na_rm)[0]]
    if op == "colMeans":
        return [d.colstats("mean", na_rm=na_rm)[0]]
    if op == "rowSums":
        return [d.rowstats("sum", na_rm=na_rm)[0]]
    return list(d.rowmoments(na_rm=na_rm))


def bits(ts):
    out = []
    for t in ts:
        a = t.cpu().numpy()
        out.append(a.view(np.int64) if a.dtype == np.float64 else a)
    return out


def same(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.fixture(scope="module")
def big():
    """30,000 x 4,000, ~24e6 entries: enough tiles for the cyclic row_hist
    and full batches in the chunked one."""
    nrow, ncol = 30000, 4000
    ptr, offs = structure(nrow, ncol, seed=5)
    assert ptr[-1] > 4 * 148 * TILE
    return nrow, ncol, ptr, offs


@pytest.mark.parametrize("tiles", ["cyclic", "chunked"])
@pytest.mark.parametrize("kind", ["signed", "small", "logical"])
def test_compact_equals_wide(big, kind, tiles, monkeypatch):
    monkeypatch.setenv("SVTGPU_ROW_HIST_TILES", tiles)
    nrow, ncol, ptr, offs = big
    vals = values(ptr, kind, seed=len(kind))
    vtype = "logical" if kind == "logical" else "integer"
    lp, o, v = on_device(nrow, ptr, offs, vals, vtype)
    nnz = int(ptr[-1])

    def fresh():
        return DeviceSVT(nrow, ncol, nnz, vtype, lp, o, v)

    for na_rm in (False, True):
        # the first call on a fresh handle runs wide and builds nothing
        wide = {}
        for op in OPS:
            d = fresh()
            wide[op] = bits(run(d, op, na_rm))
            assert compact_bytes(d) == 0, op
            d.free()
        # the second eligible call builds; from then on the compact kernels
        d = fresh()
        assert same(bits(run(d, "colSums", na_rm)), wide["colSums"])
        assert compact_bytes(d) == 0
        assert same(bits(run(d, "colSums", na_rm)), wide["colSums"])
        assert compact_bytes(d) == 3 * (nnz + PAD)
        for op in OPS:
            assert same(bits(run(d, op, na_rm)), wide[op]), (op, na_rm)
        d.free()
        # the row kernels count towards the build as well
        d = fresh()
        assert same(bits(run(d, "rowSums", na_rm)), wide["rowSums"])
        assert compact_bytes(d) == 0
        assert same(bits(run(d, "rowSums", na_rm)), wide["rowSums"])
        assert compact_bytes(d) == 3 * (nnz + PAD)
        for op in OPS:
            assert same(bits(run(d, op, na_rm)), wide[op]), (op, na_rm)
        d.free()

    # and the wide answer is the right one
    x = vals.astype(np.int64)
    isna = vals == NA_INT
    leaf = np.repeat(np.arange(ncol), np.diff(ptr))
    cs = np.bincount(leaf, weights=np.where(isna, 0, x), minlength=ncol)
    assert np.array_equal(wide["colSums"][0].view(np.float64), cs)
    rs = np.bincount(offs, weights=np.where(isna, 0, x), minlength=nrow)
    assert np.array_equal(wide["rowSums"][0].view(np.float64), rs)


def test_compact_nrow_65536():
    nrow, ncol = 65536, 3000
    d = DeviceSVT.generate_poisson(nrow, ncol, 0.12, seed=9, na_rate=1e-4)
    wide = {}
    for op in OPS:
        f = DeviceSVT(nrow, ncol, d.nnz, "integer", d.leaf_ptr, d.offs, d.vals)
        wide[op] = bits(run(f, op, True))
        f.free()
    run(d, "colSums", True)
    run(d, "colSums", True)
    assert compact_bytes(d) == 3 * (d.nnz + PAD)
    for op in OPS:
        assert same(bits(run(d, op, True)), wide[op]), op


def small_case(nrow, ncol, vals_fn, vtype="integer", seed=3):
    ptr, offs = structure(nrow, ncol, seed)
    nnz = int(ptr[-1])
    vals = None if vals_fn is None else vals_fn(nnz)
    lp, o, v = on_device(nrow, ptr, offs, vals, vtype)
    return DeviceSVT(nrow, ncol, nnz, vtype, lp, o, v), nnz


@pytest.mark.parametrize("name,nrow,vals_fn,vtype", [
    ("stored -128", 500, lambda n: np.where(np.arange(n) == n // 2, -128,
                                            np.arange(n) % 50 + 1), "integer"),
    ("value 128", 500, lambda n: np.where(np.arange(n) == n // 3, 128,
                                          np.arange(n) % 50 + 1), "integer"),
    ("double", 500, lambda n: (np.arange(n) % 5 + 1).astype(np.float64),
     "double"),
    ("lacunar", 500, None, "integer"),
])
def test_ineligible_builds_nothing(name, nrow, vals_fn, vtype):
    def make():
        return small_case(nrow, 300, None if vals_fn is None else
                          (lambda n: vals_fn(n).astype(
                              np.float64 if vtype == "double" else np.int32)),
                          vtype)[0]
    wide = {}
    for op in OPS:
        f = make()
        wide[op] = bits(run(f, op, True))
    d = make()
    for _ in range(2):
        for op in OPS:
            assert same(bits(run(d, op, True)), wide[op]), (name, op)
    assert compact_bytes(d) == 0, name


def test_values_only_above_65536_rows():
    nrow = 65537
    make = lambda: small_case(nrow, 200, lambda n: (np.arange(n) % 9 + 1)
                              .astype(np.int32), seed=4)
    wide = {}
    for op in OPS:
        wide[op] = bits(run(make()[0], op, False))
    d, nnz = make()
    run(d, "colSums", False)
    run(d, "colSums", False)
    assert compact_bytes(d) == nnz + PAD
    for op in OPS:
        assert same(bits(run(d, op, False)), wide[op]), op


def test_fold_rows_drops_the_copy():
    nrow, ncol, fold = 300, 48, 4
    x = synth.poisson_svt(nrow, ncol, 0.2, seed=21, na_rate=1e-2)
    d = DeviceSVT.from_host(x)
    run(d, "colSums", True)
    run(d, "colSums", True)
    assert compact_bytes(d) > 0
    N.check(N.lib().svtgpu_matrix_fold_rows(d._h, fold))
    assert compact_bytes(d) == 0
    d.nrow, d.nleaf = nrow * fold, ncol // fold
    d.nleaf_total = d.nleaf
    v = np.asarray(x.vals, dtype=np.int64)
    ok = v != NA_INT
    leaf = np.repeat(np.arange(ncol), np.diff(x.ptr))
    rows = np.asarray(x.offs) + nrow * (leaf % fold)
    want = np.bincount(rows[ok], weights=v[ok], minlength=nrow * fold)
    for _ in range(3):   # wide, then built again on the folded rows
        got = d.rowstats("sum", na_rm=True)[0].cpu().numpy()
        assert np.array_equal(got, want)
    assert compact_bytes(d) == 3 * (x.ptr[-1] + PAD)
