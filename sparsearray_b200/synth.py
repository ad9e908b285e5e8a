"""Synthetic SVT inputs with the distributions of the reference's generators.

R's RNG is not available, so the data are defined by our own seeded,
counter-based formula (documented in include/svtgpu.h next to
svtgpu_gen_count/fill, which evaluate the very same formula in HBM):

  poisson_svt()  -- poissonSparseArray(dim, density)
                    (R/randomSparseArray.R:62-81, src/randomSparseArray.c:
                    91-158): every cell iid Poisson(lambda = -log(1-density)),
                    zeros dropped, type integer.
  random_svt()   -- randomSparseArray(dim, density) (R/randomSparseArray.R:
                    11-38): floor(prod(dim) * density) nonzeros at distinct
                    uniformly random cells, values signif(rnorm(.), 2),
                    type double.

The host versions here serve the parity tests (small sizes); benchmarks call
the device generator through the C ABI.
"""
import math

import numpy as np

from .svt import SVT_SparseArray, NA_INTEGER, NA_REAL

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)
GOLDEN = np.uint64(0x9E3779B97F4A7C15)
SALT2 = np.uint64(0xD1B54A32D192ED03)


def mix64(z):
    """splitmix64 finaliser on uint64 arrays."""
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return z


def poisson_thresholds(density, max_value=12):
    """(nz_threshold, value_thresholds): P(cell != 0) = density and the
    zero-truncated Poisson(lambda) CDF, both scaled to 2^32."""
    if not 0.0 < density < 1.0:
        raise ValueError("density must be in (0, 1)")
    lam = -math.log1p(-density)
    nz_threshold = min(int(round(density * 2.0 ** 32)), 2 ** 32 - 1)
    p0 = math.exp(-lam)
    cdf, term, out = 0.0, p0, []
    for k in range(1, max_value):
        term = term * lam / k
        cdf += term / (1.0 - p0)          # P(1 <= X <= k | X >= 1)
        t = min(int(round(cdf * 2.0 ** 32)), 2 ** 32 - 1)
        out.append(t)
        if t >= 2 ** 32 - 1:
            break
    return nz_threshold, np.array(out, dtype=np.uint32)


def na_threshold(rate):
    return min(int(round(rate * 2.0 ** 32)), 2 ** 32 - 1)


def poisson_csc(nrow, nleaf, density, seed=0, na_rate=0.0, leaf0=0,
                type="integer", lacunar=False):
    """Host evaluation of the device generator's formula: (ptr, offs, vals)."""
    nz_thr, vthr = poisson_thresholds(density)
    na_thr = np.uint64(na_threshold(na_rate))
    ptr = np.zeros(nleaf + 1, dtype=np.int64)
    offs_l, vals_l = [], []
    i = np.arange(nrow, dtype=np.uint64)
    with np.errstate(over="ignore"):
        for l in range(nleaf):
            cell = np.uint64(leaf0 + l) * np.uint64(nrow) + i
            h = mix64(np.uint64(seed) + (cell + np.uint64(1)) * GOLDEN)
            hit = (h >> np.uint64(32)) < np.uint64(nz_thr)
            idx = np.flatnonzero(hit)
            ptr[l + 1] = ptr[l] + idx.size
            offs_l.append(idx.astype(np.int32))
            if lacunar:
                continue
            h2 = mix64(h[idx] ^ SALT2)
            u = (h2 >> np.uint64(32)).astype(np.uint64)
            v = 1 + (u[:, None] >= vthr[None, :].astype(np.uint64)).sum(axis=1)
            is_na = (h2 & np.uint64(0xFFFFFFFF)) < na_thr
            if type == "double":
                v = v.astype(np.float64)
                v[is_na] = NA_REAL
            else:
                v = v.astype(np.int32)
                v[is_na] = NA_INTEGER
            vals_l.append(v)
    offs = np.concatenate(offs_l) if offs_l else np.zeros(0, np.int32)
    if lacunar:
        return ptr, offs, None
    dt = np.float64 if type == "double" else np.int32
    vals = np.concatenate(vals_l) if vals_l else np.zeros(0, dt)
    return ptr, offs, vals


def poisson_row(nrow, nleaf, i, density, seed=0, na_rate=0.0, leaf0=0):
    """Row i of the matrix poisson_csc() makes, evaluated on its own (cell
    (i, l) depends only on l * nrow + i): (leaves, values, is_na), leaves
    relative to leaf0 and ascending, values int64 (those under is_na are
    the draws that became NA).  The values of a lacunar matrix are ignored."""
    nz_thr, vthr = poisson_thresholds(density)
    na_thr = np.uint64(na_threshold(na_rate))
    l = np.arange(leaf0, leaf0 + nleaf, dtype=np.uint64)
    with np.errstate(over="ignore"):
        h = mix64(np.uint64(seed) +
                  (l * np.uint64(nrow) + np.uint64(i) + np.uint64(1)) * GOLDEN)
        cols = np.flatnonzero((h >> np.uint64(32)) < np.uint64(nz_thr))
        h2 = mix64(h[cols] ^ SALT2)
        v = 1 + np.searchsorted(vthr.astype(np.uint64), h2 >> np.uint64(32),
                                side="right")
        is_na = (h2 & np.uint64(0xFFFFFFFF)) < na_thr
    return cols, v.astype(np.int64), is_na


def poisson_svt(nrow, ncol, density, seed=0, na_rate=0.0, type="integer",
                lacunar=False):
    ptr, offs, vals = poisson_csc(nrow, ncol, density, seed, na_rate, 0, type,
                                  lacunar)
    return SVT_SparseArray((nrow, ncol), type, ptr, offs, vals)


def _signif2(x):
    """signif(x, 2)"""
    x = np.asarray(x, dtype=np.float64)
    out = np.zeros_like(x)
    nzm = x != 0
    mag = np.floor(np.log10(np.abs(x[nzm])))
    scale = 10.0 ** (1 - mag)
    out[nzm] = np.round(x[nzm] * scale) / scale
    return out


def random_svt(nrow, ncol, density, seed=0):
    """randomSparseArray(c(nrow, ncol), density): exact nonzero count, distinct
    uniformly random cells, values signif(rnorm(.), 2) (zeros re-drawn as the
    smallest representable step so the count stays exact)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    total = nrow * ncol
    nnz = int(math.floor(total * density))
    cells = np.sort(rng.choice(total, size=nnz, replace=False))
    vals = _signif2(rng.standard_normal(nnz))
    vals[vals == 0] = 0.01
    cols = cells // nrow
    offs = (cells - cols * nrow).astype(np.int32)
    ptr = np.zeros(ncol + 1, dtype=np.int64)
    np.add.at(ptr, cols + 1, 1)
    ptr = np.cumsum(ptr)
    return SVT_SparseArray((nrow, ncol), "double", ptr, offs, vals)
