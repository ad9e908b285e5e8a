"""Column sums and means from the compact copy on leaf layouts the tile-edge
tests do not build: runs of leaves of 0-3 entries (leaves whose first and
last 16-byte word is the same, and words shared by several leaves), a
matrix of fewer 32,768-entry tiles than SMs, one smaller than a tile, and
segments of `group` consecutive leaves (N-d arrays).  Each is bit-identical
to the wide kernels of a fresh handle and to host sums, and each reaches the
compact copy."""
import ctypes

import numpy as np
import pytest
import torch

from sparsearray_b200 import _native as N
from sparsearray_b200 import synth
from sparsearray_b200.device import DeviceSVT, _ptr, _stream_ptr
from test_gpu_compact import (NA_INT, TILE, compact_bytes, on_device,
                              values)
from test_gpu_compact_tiles import (check, edge_lengths, layout, odd_nnz,
                                    word_edge_nas)

pytestmark = pytest.mark.gpu


def mixed_lengths(n_target, seed):
    """runs of tiny leaves (0-3 entries: tens of thousands in one tile, 1-2
    tiles per run) between runs of leaves of 1..5000 entries (3-5 tiles)"""
    rng = np.random.default_rng(seed)
    parts, p, tiny = [], 0, True
    while p < n_target:
        span = int(rng.integers(TILE, 2 * TILE) if tiny
                   else rng.integers(3 * TILE, 5 * TILE))
        k = rng.integers(0, 4, size=span) if tiny else \
            rng.integers(1, 5001, size=span // 2000)
        k = k[:np.searchsorted(np.cumsum(k), span) + 1]
        parts.append(k)
        p += int(k.sum())
        tiny = not tiny
    return odd_nnz(np.concatenate(parts).astype(np.int64))


def spread_layout(nrow, lens, seed):
    """leaf_ptr and ascending row offsets of leaves of at most nrow // 6
    entries, without a loop over the leaves: entry i of a leaf goes to row
    6 i + (0..5)"""
    rng = np.random.default_rng(seed)
    ptr = np.zeros(len(lens) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(lens)
    i = np.arange(int(ptr[-1]), dtype=np.int64) - np.repeat(ptr[:-1], lens)
    assert i.max() < nrow // 6
    return ptr, (6 * i + rng.integers(0, 6, size=len(i))).astype(np.int32)


def column_layout(name):
    """leaf lengths: tiny leaves mixed with larger ones over more tiles than
    SMs, a matrix of fewer tiles than SMs, one smaller than a tile"""
    if name == "tiny leaves":
        lens = mixed_lengths(3 * 148 * TILE // 2, seed=31)
    elif name == "few tiles":
        lens = edge_lengths(30000, 20 * TILE + 123, seed=32)
    else:
        lens = odd_nnz(np.random.default_rng(33).integers(0, 60, size=500))
        assert lens.sum() < TILE
    return lens


@pytest.mark.parametrize("name", ["tiny leaves", "few tiles", "below a tile"])
@pytest.mark.parametrize("kind", ["signed", "logical"])
def test_column_layouts(name, kind):
    """column sums, means and row sums from the compact copy where one tile
    holds thousands of leaves, where the matrix has fewer tiles than SMs and
    where it is smaller than one tile"""
    nrow = 30000
    lens = column_layout(name)
    ptr, offs = spread_layout(nrow, lens, seed=34)
    nnz = int(ptr[-1])
    assert nnz % 16
    vals = values(ptr, kind, seed=35)
    vtype = "logical" if kind == "logical" else "integer"
    for na_rm in (False, True):
        wide = check(nrow, ptr, offs, vals, vtype,
                     ("colSums", "colMeans", "rowSums"), na_rm)
    isna = vals == NA_INT
    leaf = np.repeat(np.arange(len(lens)), lens)
    cs = np.bincount(leaf, weights=np.where(isna, 0, vals.astype(np.int64)),
                     minlength=len(lens))
    assert np.array_equal(wide["colSums"][0].view(np.float64), cs)


def colstats_group(d, op, na_rm, group):
    """colstats_dev over segments of `group` consecutive leaves"""
    code = N.OPCODES[op]
    out = torch.empty(d.nleaf // group, device="cuda", dtype=torch.float64)
    warn = torch.zeros(4, dtype=torch.int32, device="cuda")
    N.check(N.lib().svtgpu_colstats_dev(
        d._h, code, int(na_rm), ctypes.c_double(synth.NA_REAL), int(group),
        _ptr(out), _ptr(warn), _stream_ptr()))
    return out.cpu().numpy().view(np.int64)


@pytest.fixture(scope="module")
def edges():
    nrow = 30000
    lens = edge_lengths(nrow, 4 * 148 * TILE + 5 * TILE + 777, seed=11)
    ptr, offs = layout(nrow, lens, seed=12)
    return nrow, ptr, offs


@pytest.mark.parametrize("group", [2, 7])
def test_group_segments(edges, group):
    """segments of `group` leaves (N-d arrays) on a handle that holds the
    compact copy: equal to the wide kernel and to host sums"""
    nrow, ptr, offs = edges
    nleaf = (len(ptr) - 1) // group * group
    ptr = ptr[:nleaf + 1]
    offs = offs[:ptr[-1]]
    nnz = int(ptr[-1])
    vals = word_edge_nas(values(ptr, "signed", seed=36), nnz, 6)
    lp, o, v = on_device(nrow, ptr, offs, vals, "integer")

    def fresh():
        return DeviceSVT(nrow, nleaf, nnz, "integer", lp, o, v)

    for na_rm in (False, True):
        for op in ("sum", "mean"):
            f = fresh()
            wide = colstats_group(f, op, na_rm, group)
            f.free()
            d = fresh()
            colstats_group(d, op, na_rm, group)
            assert compact_bytes(d) == 0
            for _ in range(2):
                assert np.array_equal(colstats_group(d, op, na_rm, group),
                                      wide), (op, na_rm)
            assert compact_bytes(d) > 0
            d.free()
            if op == "sum" and na_rm:
                isna = vals == NA_INT
                seg = np.repeat(np.arange(nleaf), np.diff(ptr)) // group
                cs = np.bincount(seg, weights=np.where(
                    isna, 0, vals.astype(np.int64)),
                    minlength=nleaf // group)
                assert np.array_equal(wide.view(np.float64), cs)
