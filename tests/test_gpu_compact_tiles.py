"""The compact copy on leaf layouts that put every kind of leaf bound on a
32,768-entry tile edge: leading and trailing empty leaves, empty leaves
exactly at a tile edge, leaves that start or end exactly on one, leaves
longer than several tiles, a partial last tile with nnz a multiple of
neither 16 nor the tile, and NA bytes at tile and word edges.  The compact
row histogram streams each CTA's tiles back to back (the next tile's first
batch is in flight while the piece check runs); column sums, column means,
row sums and row moments are bit-identical to the wide kernels of a fresh
handle and to host sums, in the cyclic and the chunked row form."""
import numpy as np
import pytest

from sparsearray_b200.device import DeviceSVT
from test_gpu_compact import (NA_INT, PAD, TILE, bits, compact_bytes,
                              on_device, run, same, values)

pytestmark = pytest.mark.gpu


def edge_lengths(nrow, n_target, seed, long_leaves=0):
    """leaf lengths: 3 empty leaves first and last; at every third tile edge
    a leaf that ends exactly there followed by two empty leaves (so the next
    leaf starts on the edge); `long_leaves` leaves of 5.5 tiles; otherwise
    lengths 1 .. min(nrow, 5000)"""
    rng = np.random.default_rng(seed)
    lens = [0, 0, 0]
    p, edge, n_long = 0, TILE, 0
    while p < n_target:
        if n_long < long_leaves and edge // TILE == 7 + 40 * n_long:
            k = TILE * 5 + TILE // 2 + 13
            n_long += 1
        elif edge - p <= min(nrow, 5000) and (edge // TILE) % 3 == 0:
            k = edge - p
            lens += [k, 0, 0]
            p += k
            edge += TILE
            continue
        else:
            k = int(rng.integers(1, min(nrow, 5000) + 1))
        lens.append(k)
        p += k
        while edge <= p:
            edge += TILE
    lens = np.asarray(lens + [0, 0, 0], dtype=np.int64)
    return odd_nnz(lens)


def odd_nnz(lens):
    """nnz a multiple of neither 16 nor the tile"""
    while lens.sum() % 16 == 0 or lens.sum() % TILE == 0:
        lens[np.flatnonzero(lens > 1)[-1]] -= 1
    return lens


def layout(nrow, lens, seed):
    rng = np.random.default_rng(seed)
    ptr = np.zeros(len(lens) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(lens)
    offs = np.empty(int(ptr[-1]), dtype=np.int32)
    for j, k in enumerate(lens):
        k = int(k)
        if k == 0:
            continue
        if k * 4 >= nrow:
            offs[ptr[j]:ptr[j + 1]] = np.sort(
                rng.permutation(nrow)[:k]).astype(np.int32)
        else:
            offs[ptr[j]:ptr[j + 1]] = np.sort(
                rng.choice(nrow, size=k, replace=False))
    return ptr, offs


def word_edge_nas(v, nnz, seed):
    """NA at both sides of random 16-byte word bounds"""
    rng = np.random.default_rng(seed)
    w = rng.integers(1, nnz // 16, size=2000) * 16
    v[w] = NA_INT
    v[w - 1] = NA_INT
    return v


def check(nrow, ptr, offs, vals, vtype, ops, na_rm):
    lp, o, v = on_device(nrow, ptr, offs, vals, vtype)
    nnz, ncol = int(ptr[-1]), len(ptr) - 1

    def fresh():
        return DeviceSVT(nrow, ncol, nnz, vtype, lp, o, v)

    wide = {}
    for op in ops:
        d = fresh()
        wide[op] = bits(run(d, op, na_rm))
        d.free()
    # the second call builds the copy; later calls read it
    d = fresh()
    run(d, "colSums", na_rm)
    for _ in range(2):
        for op in ops:
            assert same(bits(run(d, op, na_rm)), wide[op]), (op, na_rm)
    assert compact_bytes(d) > 0
    d.free()
    return wide


@pytest.fixture(scope="module")
def edges():
    nrow = 30000
    lens = edge_lengths(nrow, 4 * 148 * TILE + 5 * TILE + 777, seed=11)
    ptr, offs = layout(nrow, lens, seed=12)
    nnz = int(ptr[-1])
    assert nnz % 16 and nnz % TILE
    # the tile-edge layouts are really there
    starts = ptr[:-1]
    assert np.sum((lens == 0) & (starts % TILE == 0) & (starts > 0)) > 100
    assert np.sum((lens > 0) & (starts % TILE == 0)) > 100
    assert np.sum((lens > 0) & (ptr[1:] % TILE == 0)) > 100
    return nrow, ptr, offs


@pytest.mark.parametrize("tiles", ["cyclic", "chunked"])
@pytest.mark.parametrize("kind", ["signed", "small", "logical"])
def test_tile_edges(edges, kind, tiles, monkeypatch):
    monkeypatch.setenv("SVTGPU_ROW_HIST_TILES", tiles)
    nrow, ptr, offs = edges
    nnz = int(ptr[-1])
    vals = word_edge_nas(values(ptr, kind, seed=len(kind) + 7), nnz, 3)
    vtype = "logical" if kind == "logical" else "integer"
    for na_rm in (False, True):
        wide = check(nrow, ptr, offs, vals, vtype,
                     ("colSums", "colMeans", "rowSums", "rowMoments"), na_rm)
    x = vals.astype(np.int64)
    isna = vals == NA_INT
    leaf = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
    cs = np.bincount(leaf, weights=np.where(isna, 0, x),
                     minlength=len(ptr) - 1)
    assert np.array_equal(wide["colSums"][0].view(np.float64), cs)
    rs = np.bincount(offs, weights=np.where(isna, 0, x), minlength=nrow)
    assert np.array_equal(wide["rowSums"][0].view(np.float64), rs)


def test_long_leaves_values_only():
    """nrow > 65,536 (values-only copy): leaves of 5.5 tiles, and one leaf
    whose sum passes 2^31"""
    nrow = 18_000_000
    big = 17_500_000
    lens = edge_lengths(200_000, 4 * 148 * TILE + 3 * TILE + 99, seed=21,
                        long_leaves=4)
    lens = odd_nnz(np.concatenate([lens[:5], [big], lens[5:]]))
    ptr = np.zeros(len(lens) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(lens)
    nnz = int(ptr[-1])
    # offsets: the first k rows of each leaf (the column kernels never read
    # them)
    offs = (np.arange(nnz, dtype=np.int64) -
            np.repeat(ptr[:-1], lens)).astype(np.int32)
    vals = np.full(nnz, 127, dtype=np.int32)
    rng = np.random.default_rng(5)
    small = rng.integers(-127, 128, size=nnz).astype(np.int32)
    vals[:ptr[5]] = small[:ptr[5]]
    vals[ptr[6]:] = small[ptr[6]:]
    for d in (-1, 0, 1):
        e = np.arange(TILE, nnz, TILE) + d
        vals[e[e < nnz]] = NA_INT
    vals = word_edge_nas(vals, nnz, 4)
    isna = vals == NA_INT
    leaf = np.repeat(np.arange(len(lens)), lens)
    cs = np.bincount(leaf, weights=np.where(isna, 0, vals.astype(np.int64)),
                     minlength=len(lens))
    assert cs[5] > 2 ** 31
    for na_rm in (False, True):
        wide = check(nrow, ptr, offs, vals, "integer",
                     ("colSums", "colMeans"), na_rm)
    assert np.array_equal(wide["colSums"][0].view(np.float64), cs)
