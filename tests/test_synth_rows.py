"""synth.poisson_row() -- one row of the counter-based generator's matrix --
against the whole matrix that synth.poisson_csc() builds.  The scale tests
(test_gpu_scale_exact.py) use poisson_row to check rows of matrices far too
large to build on the host."""
import numpy as np
import pytest

from sparsearray_b200 import synth


@pytest.mark.parametrize("nrow,nleaf,density,seed,na_rate,leaf0", [
    (997, 301, 0.07, 2, 1e-2, 13),
    (64, 500, 0.3, 5, 0.1, 0),
    (1, 200, 0.5, 0, 0.0, 7),
    (300, 1, 0.9, 11, 0.5, 123456),
])
def test_poisson_row_equals_poisson_csc(nrow, nleaf, density, seed, na_rate,
                                        leaf0):
    p, o, v = synth.poisson_csc(nrow, nleaf, density, seed=seed,
                                na_rate=na_rate, leaf0=leaf0)
    dense = np.zeros((nrow, nleaf), np.int64)
    for l in range(nleaf):
        dense[o[p[l]:p[l + 1]], l] = v[p[l]:p[l + 1]]
    na = dense == synth.NA_INTEGER
    nna = 0
    for i in range(nrow):
        c, rv, rna = synth.poisson_row(nrow, nleaf, i, density, seed=seed,
                                       na_rate=na_rate, leaf0=leaf0)
        assert np.array_equal(c, np.flatnonzero(dense[i])), i
        assert np.array_equal(rna, na[i, c]), i
        assert np.array_equal(rv[~rna], dense[i, c][~rna]), i
        assert ((rv >= 1) & (rv <= 12)).all()
        nna += int(rna.sum())
    assert nna == int(na.sum())
    if na_rate >= 1e-2 and nrow * nleaf > 10000:
        assert nna > 0            # the NA branch was exercised


def test_poisson_row_lacunar_pattern():
    p, o, _ = synth.poisson_csc(1000, 40, 0.01, seed=5, leaf0=3,
                                lacunar=True)
    rows = np.concatenate([np.full(p[l + 1] - p[l], l) for l in range(40)])
    for i in np.unique(o)[:50]:
        c, _, _ = synth.poisson_row(1000, 40, int(i), 0.01, seed=5, leaf0=3)
        assert np.array_equal(c, np.sort(rows[o == i]))
