"""GPU parity: the CUDA path, called through the reference-facing API
(.Call glue -> C ABI -> kernels), against the outputs of the reference's own C
(golden.npz) and against the oracle port on seeded inputs.

Bar: bit-exact for integer/logical results, counts, NA handling, min/max and
sums of integer input; 1e-12 relative for double sums / means / variances
(summation order differs)."""
import ctypes
import os

import numpy as np
import pytest

import cases
import fixtures as fx
import runners
from rcompare import assert_identical, assert_close
import sparsearray_b200 as sa
from sparsearray_b200 import synth, _native
import test_semantics_host as tsh
import conditioning as C

pytestmark = pytest.mark.gpu

STAT = cases.stat_cases()


def rcall_last():
    from sparsearray_b200 import rcall
    return rcall.last_timings()


CP = cases.crossprod_cases()
MM = cases.matmul_cases()
RTOL = 1e-12


def _exact(x, op, exp):
    if exp.dtype.kind != "f":
        return True
    return x.type != "double" and op in ("sum", "countNAs", "mean")


@pytest.mark.parametrize("name", sorted(STAT))
def test_colstats_vs_reference(name):
    G = runners.golden()
    x = STAT[name]
    for op, na_rm, center, dims in cases.col_requests(x):
        k = runners.key_col(name, op, na_rm, center, dims)
        if k + "|error" in G:
            with pytest.raises(Exception):
                runners.api_col(x, op, na_rm, center, dims)
            continue
        v, w = runners.api_col(x, op, na_rm, center, dims)
        exp = G[k]
        if _exact(x, op, exp):
            assert_identical(v, exp, k)
        else:
            assert_close(v, exp, rtol=RTOL, what=k,
                         cond=C.cond(x, "col", op, center, dims, exp=exp))
        assert bool(G[k + "|warn"]) == w, k


@pytest.mark.parametrize("name", sorted(STAT))
def test_summarize_vs_reference(name):
    """C_summarize_SVT (sum/mean/var/range/... of the whole array): value,
    result type and warning against the reference's outputs."""
    G = runners.golden()
    x = STAT[name]
    for op, na_rm, center in cases.summarize_requests(x):
        k = runners.key_summ(name, op, na_rm, center)
        v, w = runners.api_summarize(x, op, na_rm, center)
        exp = G[k].reshape(-1)
        assert classes_match(v, exp), (k, v.dtype, exp.dtype)
        if exp.dtype.kind != "f" or (x.type != "double" and
                                     op in ("sum", "countNAs", "mean")):
            assert_identical(v, exp, k)
        else:
            # the whole array as one column: reduce over every axis
            assert_close(v, exp, rtol=RTOL, what=k,
                         cond=C.cond(x, "col", op, center, len(x.dim),
                                     exp=exp))
        assert bool(G[k + "|warn"]) == w, k


def classes_match(v, exp):
    return v.dtype.kind == exp.dtype.kind or \
        {v.dtype.kind, exp.dtype.kind} <= {"i", "b"}


@pytest.mark.parametrize("name", sorted(STAT))
def test_rowstats_vs_reference(name):
    G = runners.golden()
    x = STAT[name]
    if len(x.dim) < 2:
        return
    # rows holding an NA / NaN AND an infinity: the reference's running
    # centered_X2_sum then depends on Inf * (Inf - 2c) and Inf - Inf accidents
    # (DESIGN.md section 2); the only rows left out, and only for that op
    na_inf = tsh._rows_with_na_and_inf(x)
    for op, na_rm, kind in cases.row_requests(x):
        k = runners.key_row(name, op, na_rm, kind)
        exp = G[k].reshape(-1)
        center = cases.row_center(x, kind)
        v, w = runners.api_row(x, op, na_rm, center)
        v = v.reshape(-1)
        if _exact(x, op, exp):
            assert_identical(v, exp, k)
        else:
            keep = ~na_inf if (op == "centered_X2_sum" and not na_rm) \
                else np.ones(x.dim[0], bool)
            cond = C.cond(x, "row", op, center, 1, exp=exp)
            assert_close(v[keep], exp[keep], rtol=RTOL, what=k,
                         cond=None if cond is None else cond[keep])
        assert bool(G[k + "|warn"]) == w, k


@pytest.mark.parametrize("name", sorted(n for n in STAT
                                        if len(STAT[n].dim) == 2))
def test_row_compositions_vs_reference(name):
    """rowMeans / rowVars / rowSds composed as the R methods compose them,
    and the one-pass rowMoments extension."""
    G = runners.golden()
    x = STAT[name]
    na_inf = tsh._rows_with_na_and_inf(x)
    opof = {"rowMeans": "mean", "rowVars": "var1", "rowSds": "sd1"}
    for na_rm in (False, True):
        keep = ~na_inf if not na_rm else np.ones(x.dim[0], bool)
        for fn, key in ((sa.rowMeans, "rowMeans"), (sa.rowVars, "rowVars"),
                        (sa.rowSds, "rowSds")):
            exp = G["stat|%s|%s|%d" % (name, key, na_rm)].reshape(-1)
            cur = np.asarray(fn(x, na_rm=na_rm)).reshape(-1)
            if x.type != "double" and key == "rowMeans":
                assert_identical(cur, exp, key)
            else:
                # 1e-12 of the magnitudes the reference's c^2 * ncol +
                # sum x(x - 2c) adds up (tests/conditioning.py)
                cond = C.cond(x, "row", opof[key], None, 1, exp=exp)
                assert_close(cur[keep], exp[keep], rtol=RTOL,
                             cond=cond[keep],
                             what="%s %s %s" % (name, key, na_rm),
                             na_nan_strict=False)
        if x.dim[0] == 0:
            continue
        mean, var = sa.rowMoments(x, na_rm=na_rm)
        em = G["stat|%s|rowMeans|%d" % (name, na_rm)].reshape(-1)
        ev = G["stat|%s|rowVars|%d" % (name, na_rm)].reshape(-1)
        assert_close(np.asarray(mean)[keep], em[keep], rtol=RTOL,
                     cond=C.cond(x, "row", "mean")[keep],
                     what=name + " moments mean", na_nan_strict=False)
        fin = np.isfinite(ev) & keep
        assert_close(np.asarray(var)[fin], ev[fin], rtol=RTOL,
                     cond=C.cond(x, "row", "var1")[fin],
                     what=name + " moments var")


@pytest.mark.parametrize("name", sorted(CP))
def test_crossprod_vs_reference(name):
    G = runners.golden()
    x, y, ty = CP[name]
    left = np.asarray(sa.crossprod(x, y, transpose_y=ty))
    right = np.asarray(sa.crossprod(y, x, transpose_y=ty))
    el, er = G["cp|%s|left" % name], G["cp|%s|right" % name]
    if x.type == "integer":
        assert_identical(left, el, name)
        assert_identical(right, er, name)
    else:
        atol = 0.0
        if x.vals is not None and x.vals.size and np.isfinite(y).any():
            atol = 1e-12 * float(np.abs(y[np.isfinite(y)]).max()) * \
                float(np.abs(x.vals[np.isfinite(x.vals)]).max()) * x.dim[0]
        assert_close(left, el, rtol=RTOL, atol=atol, what=name)
        assert_close(right, er, rtol=RTOL, atol=atol, what=name)


@pytest.mark.parametrize("name", sorted(MM))
def test_matmul_vs_reference(name):
    """`svt %*% dense` without the reference's t(svt)."""
    G = runners.golden()
    x, d = MM[name]
    cur = np.asarray(sa.matmul(x, d))
    exp = G["mm|%s" % name]
    if x.type == "integer":
        assert_identical(cur, exp, name)
    else:
        atol = 1e-12 * float(np.abs(d[np.isfinite(d)]).max()) * 100 * x.dim[1]
        assert_close(cur, exp, rtol=RTOL, atol=atol, what=name)


def test_names_and_dimnames_propagate():
    m1, dn = fx.ms_m1()
    x = sa.SVT_SparseArray.from_dense(m1, "integer", dimnames=dn)
    assert sa.colSums(x).names == dn[1]
    assert sa.rowSums(x).names == dn[0]
    assert sa.colMaxs(x, useNames=False).names is None
    assert sa.colMaxs(x).rtype == "integer"
    assert sa.colAnyNAs(x).rtype == "logical"
    y = np.arange(8, dtype=np.int32).reshape(4, 2)
    cp = sa.crossprod(x, y, y_dimnames=(None, ["u", "v"]))
    assert cp.dimnames == [dn[1], ["u", "v"]]
    assert cp.shape == (5, 2) and cp.rtype == "double"


def test_zero_row_minmax_warns():
    """tests/testthat/test-SparseArray-matrixStats.R:173-189"""
    x = STAT["ms_m1_zero_rows"]
    r = sa.colMins(x)
    assert any("NAs introduced by coercion of infinite values to integers"
               in w for w in r.warnings)
    assert_identical(np.asarray(r), np.full(5, fx.NA_I, dtype=np.int32))


def test_rejected_inputs_raise():
    x = STAT["ms_m1"]
    from sparsearray_b200.rcall import rshim
    with pytest.raises(rshim.RError, match="must be one of"):
        sa.svt._colStats("median", x)
    with pytest.raises(rshim.RError):
        sa.svt._colStats("range", x)      # not served by the GPU path


# ---- seeded mid-size inputs against the oracle port -----------------------

@pytest.fixture(scope="module")
def mid_int():
    return synth.poisson_svt(33538, 96, 0.07, seed=2, na_rate=1e-4)


@pytest.fixture(scope="module")
def mid_dbl():
    return synth.random_svt(20000, 300, 0.05, seed=1)


@pytest.mark.parametrize("op", ["sum", "mean", "var1", "sd1", "max", "min",
                                "countNAs", "anyNA"])
@pytest.mark.parametrize("na_rm", [False, True])
def test_mid_int_colstats(mid_int, op, na_rm):
    x = mid_int
    v, w = runners.api_col(x, op, na_rm, None, 1)
    e, ew = runners.port_col(x, op, na_rm, None, 1)
    if op in ("var1", "sd1"):
        assert_close(v, e, rtol=RTOL, what=op)
    else:
        assert_identical(v, e, op)
    assert w == ew


@pytest.mark.parametrize("op", ["sum", "min", "max", "countNAs",
                                "centered_X2_sum"])
@pytest.mark.parametrize("na_rm", [False, True])
def test_mid_int_rowstats(mid_int, op, na_rm):
    x = mid_int
    center = None
    if op == "centered_X2_sum":
        center = np.linspace(0.0, 1.0, x.dim[0])
    v, w = runners.api_row(x, op, na_rm, center)
    e, ew = runners.port_row(x, op, na_rm, center)
    if op == "centered_X2_sum":
        assert_close(v, e, rtol=RTOL, what=op,
                     cond=C.cond(x, "row", op, center))
    else:
        assert_identical(v, e, op)
    assert w == ew


@pytest.mark.parametrize("op", ["sum", "mean", "var1", "sd1", "range",
                                "prod", "countNAs", "anyNA", "any", "all"])
@pytest.mark.parametrize("na_rm", [False, True])
def test_mid_int_summarize(mid_int, op, na_rm):
    """many slices per pass (225k stored values): slice reduction + combine"""
    x = mid_int
    v, w = runners.api_summarize(x, op, na_rm, None)
    e, ew = runners.port_summarize(x, op, na_rm, None)
    if op in ("var1", "sd1") and na_rm:
        # The reference adds 225k nearly identical squares one after the
        # other: its own rounding error grows like n * eps (measured 4e-12
        # here), beyond the 1e-12 bar.  Integer data has an exact answer:
        # hold the GPU result to 1e-12 of THAT, the reference to n * eps.
        from fractions import Fraction
        reg = x.vals[x.vals != fx.NA_I].astype(object)
        n = int(np.prod(x.dim)) - int((x.vals == fx.NA_I).sum())
        s1, s2 = int(reg.sum()), int((reg * reg).sum())
        exact = Fraction(n * s2 - s1 * s1, n * (n - 1))
        exact = float(exact) if op == "var1" else float(exact) ** 0.5
        assert abs(v[0] - exact) <= RTOL * exact, (v, exact)
        assert abs(e[0] - exact) <= x.vals.size * 2.3e-16 * exact, (e, exact)
    elif op in ("var1", "sd1", "prod"):
        assert_close(v, e, rtol=RTOL, what=op)
    else:
        assert_identical(v, e, op)
    assert w == ew


@pytest.mark.parametrize("op", ["sum", "mean", "var1", "range"])
def test_mid_dbl_summarize(mid_dbl, op):
    x = mid_dbl
    v, _ = runners.api_summarize(x, op, False, None)
    e, _ = runners.port_summarize(x, op, False, None)
    if op == "range":
        assert_identical(v, e, op)
    else:
        assert_close(v, e, rtol=RTOL, what=op,
                     cond=C.cond(x, "col", op, None, len(x.dim), exp=e))


@pytest.mark.parametrize("op", ["sum", "mean", "var1", "max", "min"])
def test_mid_dbl_colstats(mid_dbl, op):
    x = mid_dbl
    v, _ = runners.api_col(x, op, False, None, 1)
    e, _ = runners.port_col(x, op, False, None, 1)
    if op in ("max", "min"):
        assert_identical(v, e, op)
    else:
        assert_close(v, e, rtol=RTOL, what=op,
                     cond=C.cond(x, "col", op, exp=e))


def test_mid_dbl_rowsums_crossprod(mid_dbl):
    x = mid_dbl
    v, _ = runners.api_row(x, "sum", False, None)
    e, _ = runners.port_row(x, "sum", False, None)
    assert_close(v, e, rtol=RTOL, what="rowSums", cond=C.cond(x, "row", "sum"))
    rng = np.random.Generator(np.random.PCG64(9))
    y = rng.standard_normal((x.dim[0], 50))
    cur = np.asarray(sa.crossprod(x, y))
    exp = runners.port_crossprod(x, y, False, True)
    assert_close(cur, exp, rtol=RTOL, what="crossprod", cond=C.dot_cond(x, y))
    d = rng.standard_normal((x.dim[1], 50))
    cur = np.asarray(sa.matmul(x, d))
    exp = runners.port_matmul(x, d)
    assert_close(cur, exp, rtol=RTOL, what="matmul", cond=C.matmul_cond(x, d))


@pytest.mark.parametrize("impl_env", [("SVTGPU_COLSTATS_IMPL", "direct"),
                                      ("SVTGPU_COLSTATS_IMPL", "tma"),
                                      ("SVTGPU_COL_STAGE_KB", "4"),
                                      ("SVTGPU_ROW_IMPL", "flat"),
                                      ("SVTGPU_ROW_IMPL", "tiles"),
                                      ("SVTGPU_ROW_IMPL", "f64acc"),
                                      ("SVTGPU_ROW_IMPL", "acc32"),
                                      ("SVTGPU_ROW_IMPL", "hist"),
                                      ("SVTGPU_ROW_HIST", "off"),
                                      ("SVTGPU_ROW_SLOTS", "2"),
                                      ("SVTGPU_ROW_WARPS", "5"),
                                      ("SVTGPU_ROW_NTILES", "3")])
def test_kernel_variants_agree(mid_int, impl_env, monkeypatch):
    """Every kernel variant (TMA-staged / direct, tiled / flat, multi-chunk
    leaves, forced row tiling) gives the same answers."""
    monkeypatch.setenv(*impl_env)
    x = mid_int
    for op in ("sum", "var1", "max"):
        v, _ = runners.api_col(x, op, True, None, 1)
        e, _ = runners.port_col(x, op, True, None, 1)
        if op == "var1":
            assert_close(v, e, rtol=RTOL, what=op)
        else:
            assert_identical(v, e, op)
    for op in ("sum", "max", "min"):
        v, _ = runners.api_row(x, op, True, None)
        e, _ = runners.port_row(x, op, True, None)
        assert_identical(v, e, op)


_MULTISLOT = r"""
import os, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np
import sparsearray_b200 as sa
import runners
import conditioning as C
from rcompare import assert_identical, assert_close
rng = np.random.Generator(np.random.PCG64(77))
m = np.zeros((3000, 400), dtype=np.int32)
mask = rng.random(m.shape) < 0.4
m[mask] = rng.integers(1, 9, size=mask.sum())
m[5, 3] = -2**31                      # NA travels as -128
m[:, 300:][mask[:, 300:]] = 1000      # later slots do not fit int8
x = sa.SVT_SparseArray.from_dense(m, "integer", lacunar=False)
assert x.nnz > 3 * 131072             # > 3 staging slots of 1 MB
for na_rm in (False, True):
    v, _ = runners.api_col(x, "sum", na_rm, None, 1)
    assert_identical(v, runners.port_col(x, "sum", na_rm, None, 1)[0])
    v, _ = runners.api_row(x, "sum", na_rm, None)
    assert_identical(v, runners.port_row(x, "sum", na_rm, None)[0])
    v, _ = runners.api_row(x, "max", na_rm, None)
    assert_identical(v, runners.port_row(x, "max", na_rm, None)[0])
xd = x.with_type("double")
y = rng.standard_normal((3000, 7))
assert_close(np.asarray(sa.crossprod(xd, y)),
             runners.port_crossprod(xd, y, False, True), rtol=1e-12,
             cond=C.dot_cond(xd, y))
t = sa.last_timings()
print("ok", t["h2d_bytes"], x.nnz)
"""


_WRAPPED = r"""
import os, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np
import sparsearray_b200 as sa
import runners
from rcompare import assert_identical
rng = np.random.Generator(np.random.PCG64(78))
nrow, ncol = 200000, 260
cols = []
for j in range(ncol):
    d = 0.02 if j %% 7 else 0.2
    o = np.nonzero(rng.random(nrow) < d)[0].astype(np.int32)
    if j == 5:
        o = np.array([], dtype=np.int32)            # empty column
    if j == 9:
        o = np.arange(nrow, dtype=np.int32)         # every row
    if j == 11:
        o = np.array([70000], dtype=np.int32) if %d else o   # first > 65535
    if j == 200:
        o = np.array([3, 10, 90000, 199999], dtype=np.int32) if %d else o  # a step > 65535
    cols.append(o)
ptr = np.zeros(ncol + 1, dtype=np.int64)
ptr[1:] = np.cumsum([o.size for o in cols])
offs = np.concatenate(cols)
lac = bool(%d)
vals = None if lac else rng.integers(1, 100, size=offs.size).astype(np.int32)
x = sa.SVT_SparseArray((nrow, ncol), "integer", ptr, offs, vals)
assert x.nnz > 3 * 131072                            # several 1 MB slots
for na_rm in (False, True):
    v, _ = runners.api_row(x, "sum", na_rm, None)
    assert_identical(v, runners.port_row(x, "sum", na_rm, None)[0])
    v, _ = runners.api_col(x, "sum", na_rm, None, 1)
    assert_identical(v, runners.port_col(x, "sum", na_rm, None, 1)[0])
sa.rowSums(x)
t = sa.last_timings()
gp, gi, gx = sa.to_csc(x)          # to_device() then C_svtgpu_to_CSC
assert np.array_equal(np.asarray(gi), offs), "offsets differ after the upload"
assert np.array_equal(np.asarray(gp), ptr)
print("ok", t["h2d_bytes"], x.nnz)
"""


@pytest.mark.parametrize("lacunar", [0, 1])
@pytest.mark.parametrize("unfit", [0, 1])
@pytest.mark.parametrize("narrow", ["1", "0"])
def test_wrapped_16bit_offsets_upload(narrow, unfit, lacunar):
    """200,000 rows: offsets travel as their low 16 bits and the device
    rebuilds the high halves leaf by leaf (SVTGPU_OFFS_U16_WRAPPED), across
    several staging slots, with leaves that straddle slots, an empty and a
    full column; with `unfit` a leaf starts above 65535 and another steps by
    more than 65535, so their slots are re-sent as int32 and the rest of the
    matrix follows in int32.  The uploaded offsets are read back bit for
    bit."""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, SVTGPU_STAGE_MB="1", SVTGPU_NARROW=narrow)
    r = subprocess.run([sys.executable, "-c",
                        _WRAPPED % (os.path.dirname(here), here, unfit,
                                    unfit, lacunar)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.strip().startswith("ok")
    if narrow == "1" and not unfit and lacunar:
        sent, nnz = r.stdout.split()[1:3]
        assert float(sent) < 2.2 * float(nnz)       # 2 bytes per offset


@pytest.mark.parametrize("narrow", ["1", "0"])
def test_multislot_narrowed_upload(narrow):
    """Several staging slots, int8/uint16 narrowing that stops fitting half
    way through the matrix (and the same with narrowing disabled)."""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, SVTGPU_STAGE_MB="1", SVTGPU_NARROW=narrow)
    r = subprocess.run([sys.executable, "-c",
                        _MULTISLOT % (os.path.dirname(here), here)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.strip().startswith("ok")


def test_colvars_int_single_pass_and_fallback():
    """Integer variance runs in one pass from exact integer sums; columns with
    |x| >= 65536 take the two-pass form.  Both against the oracle."""
    rng = np.random.Generator(np.random.PCG64(123))
    m = np.zeros((4000, 24), dtype=np.int32)
    mask = rng.random(m.shape) < 0.3
    m[mask] = rng.integers(-60000, 60000, size=mask.sum())
    m[:, 5][mask[:, 5]] = rng.integers(-2**30, 2**30, size=mask[:, 5].sum())
    m[:, 6] = 1_000_000 + rng.integers(-1, 2, size=4000)   # mean >> spread
    m[:, 7] = 30_000 + rng.integers(-1, 2, size=4000)      # same, one pass
    m[3, 8] = fx.NA_I
    x = sa.SVT_SparseArray.from_dense(m, "integer")
    for op in ("var1", "sd1", "centered_X2_sum"):
        for na_rm in (False, True):
            v, _ = runners.api_col(x, op, na_rm, None, 1)
            e, _ = runners.port_col(x, op, na_rm, None, 1)
            assert_close(v, e, rtol=1e-12, what="%s %s" % (op, na_rm))


@pytest.mark.parametrize("nonneg", ["on", "off"])
def test_colvars_of_counts_with_known_bound(nonneg, monkeypatch):
    """Once the handle knows max |x| and that no value is negative (the row
    kernels compute both), integer colVars sums a lane's values as unsigned
    64-bit -- #NA * 2^31 + sum -- and lets NA^2 vanish mod 2^32: columns that
    are all NA, hold one NA, none, or nothing at all, against the reference;
    `off` = the signed form with the explicit NA test."""
    monkeypatch.setenv("SVTGPU_COLVAR_NONNEG", nonneg)
    x = synth.poisson_svt(5000, 300, 0.07, seed=21, na_rate=2e-3)
    vals = x.vals.copy()
    ptr = x.ptr
    vals[ptr[3]:ptr[4]] = fx.NA_I                  # column 3: nothing but NA
    vals[ptr[5]:ptr[6]] = np.where(vals[ptr[5]:ptr[6]] == fx.NA_I, 1,
                                   vals[ptr[5]:ptr[6]])   # column 5: no NA
    x = sa.SVT_SparseArray(x.dim, "integer", ptr, x.offs, vals)
    h = sa.to_device(x)
    sa.rowSums(h)                                  # caches max |x| and the sign
    for op in ("var1", "sd1", "centered_X2_sum"):
        for na_rm in (False, True):
            v, w = runners.api_col(h, op, na_rm, None, 1)
            e, ew = runners.port_col(x, op, na_rm, None, 1)
            assert_close(v, e, rtol=1e-12, what="%s %s" % (op, na_rm),
                         cond=C.cond(x, "col", op))
            assert w == ew
    # var() / sd() of the whole array take the same form per slice
    for op in ("var1", "sd1", "mean", "sum"):
        for na_rm in (False, True):
            v, w = runners.api_summarize(h, op, na_rm, None)
            e, ew = runners.port_summarize(x, op, na_rm, None)
            assert_close(v, np.asarray(e).reshape(-1), rtol=1e-10,
                         what="summarize %s %s" % (op, na_rm))
            assert w == ew
    h.release()


@pytest.mark.parametrize("name", ["ms_m1", "ms_m2_lgl", "rand_int_na",
                                  "rand_dbl_special", "rand_lacunar_int",
                                  "rand_mixed_lacunar", "all_zero",
                                  "poisson_small", "one_row"])
def test_non_native_rowstats_via_device_transpose(name):
    """rowProds / rowMeans2 / rowAnys / rowAlls / row var1: the reference
    computes colStats(aperm(x)) (.OLD_rowStats_SparseArray); here the
    transpose happens on the device.  Oracle: the same composition."""
    from oracle import port
    x = STAT[name]
    nrow, ncol = x.dim
    tp, to, tv = port.transpose(nrow, ncol, x.ptr, x.offs, x.vals, x.type,
                                x.lacunar)
    ops = ["prod", "mean", "var1", "sd1"]
    if x.type != "double":
        ops += ["any", "all"]
    for op in ops:
        for na_rm in (False, True):
            e, ew = port.colstats(ncol, nrow, tp, to, tv, x.type, op, na_rm)
            r = sa.svt._rowStats(op, x, na_rm=na_rm, useNames=False)
            v = np.asarray(r).reshape(-1)
            what = "%s %s %s" % (name, op, na_rm)
            if e.dtype.kind != "f" or (x.type != "double" and op == "mean"):
                assert_identical(v, e, what)
            else:
                assert_close(v, e, rtol=1e-12, what=what,
                             cond=C.cond(x, "row", op, exp=e))
            assert (len(r.warnings) > 0) == ew, what


def test_tcrossprod_matches_reference_formulation():
    """tcrossprod(svt, M) against crossprod2(t(x), M, transpose.y=TRUE) as the
    reference runs it (tests/testthat/test-SparseMatrix-mult.R:231-241)."""
    from oracle import port
    _, _, m2, m3 = fx.cp_double()
    tx = sa.SVT_SparseArray.from_dense(np.ascontiguousarray(m2.T), "double")
    tm3 = np.ascontiguousarray(m3.T)
    cur = np.asarray(sa.tcrossprod(tx, tm3))
    # reference: crossprod2_SVT_mat(t(tx) = m2 as SVT, tm3, transpose_y)
    x = sa.SVT_SparseArray.from_dense(m2, "double")
    exp = port.crossprod(x.dim[0], x.dim[1], x.ptr, x.offs, x.vals, "double",
                         tm3, True, True, x.lacunar)
    assert_close(cur, exp, rtol=1e-12, what="tcrossprod")


# ---- device-resident handles (upload once, run many) ----------------------

def _same(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape, what
    if a.dtype.kind == "f":
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), what
    else:
        assert np.array_equal(a, b), what


@pytest.mark.parametrize("name", ["ms_m1", "rand_dbl_special", "ms_a3d",
                                  "poisson_small", "ms_m2_lgl", "all_zero",
                                  "rand_mixed_lacunar", "torture_3d_int_j0"])
def test_resident_handle_equals_per_call_upload(name):
    """x_SVT may be the external pointer of C_svtgpu_resident_SVT: every
    entry point then answers exactly as with the SVT list."""
    x = STAT[name]
    before = _native.lib().svtgpu_launch_count()
    r = sa.to_device(x)
    assert isinstance(r, sa.ResidentSVT)
    for op, na_rm, center, dims in cases.col_requests(x)[::3]:
        k = runners.key_col(name, op, na_rm, center, dims)
        if k + "|error" in runners.golden():
            continue
        a = runners.api_col(x, op, na_rm, center, dims)
        b = runners.api_col(r, op, na_rm, center, dims)
        _same(a[0], b[0], k)
        assert a[1] == b[1]
    for op, na_rm, kind in cases.row_requests(x):
        c = cases.row_center(x, kind)
        a = runners.api_row(x, op, na_rm, c)
        b = runners.api_row(r, op, na_rm, c)
        _same(a[0], b[0], (op, na_rm, kind))
        assert a[1] == b[1]
    for op, na_rm, center in cases.summarize_requests(x)[::2]:
        a = runners.api_summarize(x, op, na_rm, center)
        b = runners.api_summarize(r, op, na_rm, center)
        _same(a[0], b[0], (op, na_rm, center))
    if len(x.dim) == 2:
        _same(sa.rowVars(x, na_rm=True), sa.rowVars(r, na_rm=True), "rowVars")
        _same(sa.rowProds(x), sa.rowProds(r), "rowProds")
        ma, va = sa.rowMoments(x, na_rm=True)
        mb, vb = sa.rowMoments(r, na_rm=True)
        _same(ma, mb, "rowMoments mean")
        _same(va, vb, "rowMoments var")
    assert _native.lib().svtgpu_launch_count() > before
    r.release()
    r.release()     # idempotent


def test_resident_handle_products():
    x, y, ty = CP["dbl_m2_tm3"]
    r = sa.to_device(x)
    _same(sa.svt._crossprod2_SVT_mat(x, y, transpose_y=ty),
          sa.svt._crossprod2_SVT_mat(r, y, transpose_y=ty), "SVT_mat")
    _same(sa.svt._crossprod2_mat_SVT(y, x, transpose_x=ty),
          sa.svt._crossprod2_mat_SVT(y, r, transpose_x=ty), "mat_SVT")
    xm, d = next(iter(MM.values()))
    rm = sa.to_device(xm)
    a = sa.matmul(xm, d)
    for _ in range(2):            # the second call reuses the cached t(x)
        assert_close(np.asarray(sa.matmul(rm, d)), np.asarray(a), rtol=RTOL,
                     cond=C.matmul_cond(xm, d), what="matmul")
    r.release()
    rm.release()


def test_device_cache_reuses_and_invalidates():
    """options(SparseArray.gpu.cache=TRUE): consecutive .Calls on the same SVT
    reuse one upload (rowVars = 3 calls, 1 upload); another object, a changed
    leaf or dims >= 2 (row folding modifies the device matrix) do not; results
    are bit-identical to the stateless path."""
    x = synth.poisson_svt(3000, 200, 0.1, seed=5, na_rate=1e-3)
    exp = {"colSums": sa.colSums(x, na_rm=True),
           "rowSums": sa.rowSums(x), "rowVars": sa.rowVars(x, na_rm=True),
           "colVars": sa.colVars(x)}
    prev = sa.set_gpu_cache(True)
    try:
        h0, m0 = sa.gpu_cache_stats()
        _same(sa.colSums(x, na_rm=True), exp["colSums"], "colSums")   # miss
        assert rcall_last()["h2d_bytes"] > 0
        _same(sa.rowSums(x), exp["rowSums"], "rowSums")               # hit
        assert rcall_last()["h2d_bytes"] == 0
        _same(sa.rowVars(x, na_rm=True), exp["rowVars"], "rowVars")   # 3 hits
        _same(sa.colVars(x), exp["colVars"], "colVars")               # hit
        h1, m1 = sa.gpu_cache_stats()
        assert (h1 - h0, m1 - m0) == (5, 1)
        # the same values in a NEW object (new leaf vectors): a miss
        y = sa.SVT_SparseArray(x.dim, x.type, x.ptr.copy(), x.offs.copy(),
                               x.vals.copy())
        _same(sa.rowSums(y), exp["rowSums"], "rowSums y")
        assert sa.gpu_cache_stats()[1] - m1 == 1
        # a leaf changed in place (R code cannot do this; C code could): the
        # first / last elements of every leaf are part of the fingerprint
        a = int(y.ptr[3])
        y.vals[a] += 1
        cur = sa.colSums(y, na_rm=True)
        assert sa.gpu_cache_stats()[1] - m1 == 2
        sa.set_gpu_cache(False)
        _same(cur, sa.colSums(y, na_rm=True), "changed leaf")
        assert cur[3] != exp["colSums"][3]
        sa.set_gpu_cache(True)
        # dims >= 2 folds rows in place on its own private upload
        x3 = STAT["ms_a3d"]
        e3 = sa.rowSums(x3, dims=2)
        sa.set_gpu_cache(True)
        _same(sa.rowSums(x3, dims=2), e3, "dims=2")
        _same(sa.rowSums(x3), sa.rowSums(x3), "dims=1 twice")
        # a resident handle owns its own upload: it neither takes the cached
        # matrix nor enters the cache (the cache would free it behind the
        # handle's back, and the other way round)
        _same(sa.rowSums(x), exp["rowSums"], "x cached again")
        h = sa.to_device(x)
        _same(sa.rowSums(h), exp["rowSums"], "handle")
        _same(sa.colVars(x), exp["colVars"], "cached x beside the handle")
        h.release()
        _same(sa.rowSums(x), exp["rowSums"], "cached x after the release")
        h = sa.to_device(x)
        sa.set_gpu_cache(False)           # drops the cached copy, not h's
        _same(sa.rowSums(h), exp["rowSums"], "handle after the cache is gone")
        h.release()
        sa.set_gpu_cache(True)
    finally:
        sa.set_gpu_cache(False)
        sa.set_gpu_cache(prev)
    # off again: every call uploads
    sa.rowSums(x)
    assert rcall_last()["h2d_bytes"] > 0


def test_resident_handle_is_checked():
    x = STAT["ms_m1"]
    r = sa.to_device(x)
    other = sa.SVT_SparseArray.from_dense(
        np.ones((x.dim[0] + 1, x.dim[1]), dtype=np.int32))
    wrong = sa.ResidentSVT.__new__(sa.ResidentSVT)
    wrong.__dict__.update(other.__dict__)
    wrong._robjs = dict(other._build_robjs())
    wrong._robjs["SVT"] = r._robjs["SVT"]
    with pytest.raises(Exception, match="does not match"):
        sa.colSums(wrong)
    wrong._robjs = None
    # a released handle is refused, not dereferenced
    from sparsearray_b200 import rcall
    rcall.SparseArray_Call("C_svtgpu_release", r.r_SVT)
    with pytest.raises(Exception, match="has been released"):
        sa.colSums(r)
    r.release()


@pytest.mark.parametrize("hist", ["auto", "off"])
def test_packed_row_moments_flush_when_rows_fill(hist, monkeypatch):
    """8 nearly dense rows x 1,200,000 columns of small counts: the packed
    (sum | sum of squares) accumulators of rowVars reach their guard bits
    inside a chunk, so the on-chip look-ahead must really flush -- in the
    histogram kernel and in the strip kernel."""
    monkeypatch.setenv("SVTGPU_ROW_HIST", hist)
    rng = np.random.Generator(np.random.PCG64(5))
    nrow, ncol = 8, 1200000
    mask = rng.random((ncol, nrow)) < 0.9
    cnt = mask.sum(axis=1)
    ptr = np.zeros(ncol + 1, dtype=np.int64)
    np.cumsum(cnt, out=ptr[1:])
    offs = np.nonzero(mask)[1].astype(np.int32)
    vals = rng.integers(1, 6, size=offs.size).astype(np.int32)
    vals[rng.random(offs.size) < 1e-5] = fx.NA_I
    x = sa.SVT_SparseArray((nrow, ncol), "integer", ptr, offs, vals)
    for na_rm in (False, True):
        for op, center in (("sum", None), ("centered_X2_sum", None),
                           ("centered_X2_sum", np.full(nrow, 2.5)),
                           ("max", None), ("min", None)):
            v, w = runners.api_row(x, op, na_rm, center)
            e, ew = runners.port_row(x, op, na_rm, center)
            if op == "centered_X2_sum":
                # 1.2e6 terms per row: 1e-12 of the magnitudes the
                # reference adds (c^2 * ncol + sum |x||x - 2c|)
                s1 = np.bincount(offs[vals != fx.NA_I], minlength=nrow,
                                 weights=np.abs(vals[vals != fx.NA_I]))
                s2_ = np.bincount(offs[vals != fx.NA_I], minlength=nrow,
                                  weights=vals[vals != fx.NA_I].astype(
                                      np.float64) ** 2)
                cc = np.abs(center) if center is not None else s1 / ncol
                assert_close(v, e, rtol=RTOL, what=(op, na_rm),
                             cond=s2_ + 2 * cc * s1 + cc * cc * ncol)
            else:
                assert_identical(v, e, (op, na_rm))
    m, v = sa.rowMoments(x, na_rm=True)
    ok = vals != fx.NA_I
    dense_sum = np.zeros(nrow)
    np.add.at(dense_sum, offs[ok], vals[ok])
    nn = ncol - np.bincount(offs[~ok], minlength=nrow)
    assert_close(np.asarray(m), dense_sum / nn, rtol=RTOL, what="mean")
    s2 = np.zeros(nrow)
    np.add.at(s2, offs[ok], vals[ok].astype(np.float64) ** 2)
    var = (s2 - dense_sum ** 2 / nn) / (nn - 1)
    # (this numpy formula itself cancels: sum x^2 - (sum x)^2 / n)
    assert_close(np.asarray(v), var, rtol=RTOL, what="var",
                 cond=(s2 + dense_sum ** 2 / nn) / (nn - 1))


@pytest.mark.parametrize("hist", ["auto", "off"])
def test_row_max_of_counts_edge_rows(hist, monkeypatch):
    """rowMaxs of non-negative integers runs as one shared-memory atomic max
    per nonzero without the exact coverage count (row_hist<HIST_MAX32>): the
    rows where coverage decides -- stored in every column and all NA, stored
    in every column and regular, never stored, only stored zeros, NA next to
    regular values -- against the reference's update_out_for_rowMinsMaxs
    semantics (src/SparseArray_matrixStats.c:900-990), with the strip kernel
    (exact coverage) as the second arm."""
    monkeypatch.setenv("SVTGPU_ROW_HIST", hist)
    nrow, ncol = 7, 40
    rng = np.random.Generator(np.random.PCG64(11))
    cols = []
    for j in range(ncol):
        o = [0, 1, 3]                 # rows 0, 1: every column; 3: zeros
        v = [fx.NA_I, int(rng.integers(2, 9)), 0]
        if j % 3 == 0:
            o.append(4); v.append(fx.NA_I if j % 2 else int(rng.integers(1, 5)))
        if j % 5 == 0:
            o.append(5); v.append(int(rng.integers(0, 3)))
        if j == 7:
            o.append(6); v.append(fx.NA_I)      # row 6: one NA, nothing else
        cols.append((o, v))
    ptr = np.zeros(ncol + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([len(o) for o, _ in cols])
    offs = np.concatenate([np.asarray(o, dtype=np.int32) for o, _ in cols])
    vals = np.concatenate([np.asarray(v, dtype=np.int32) for _, v in cols])
    x = sa.SVT_SparseArray((nrow, ncol), "integer", ptr, offs, vals)
    for na_rm in (False, True):
        for op in ("max", "min"):
            v, w = runners.api_row(x, op, na_rm, None)
            e, ew = runners.port_row(x, op, na_rm, None)
            assert_identical(v, e, (op, na_rm))
            assert w == ew


@pytest.mark.parametrize("tiles", ["cyclic", "chunks"])
def test_row_hist_tiles_with_flushes(tiles, monkeypatch):
    """The histogram row kernels take the entry range in tiles, round-robin
    over the SMs (cyclic form), and look at their cells before the leaves
    touched since the last look can overflow one: 64 nearly dense rows x
    330,000 columns (19 million entries, ~550 leaves per tile) make the packed
    moments reach their guard bits many times per SM, so the on-chip look
    really flushes; sums, maxima, counts and moments against the reference,
    and the chunked form as the second arm."""
    monkeypatch.setenv("SVTGPU_ROW_HIST_TILES", tiles)
    rng = np.random.Generator(np.random.PCG64(19))
    nrow, ncol = 64, 330000
    mask = rng.random((ncol, nrow)) < 0.9
    cnt = mask.sum(axis=1)
    ptr = np.zeros(ncol + 1, dtype=np.int64)
    np.cumsum(cnt, out=ptr[1:])
    offs = np.nonzero(mask)[1].astype(np.int32)
    vals = rng.integers(1, 6, size=offs.size).astype(np.int32)
    vals[rng.random(offs.size) < 1e-5] = fx.NA_I
    x = sa.SVT_SparseArray((nrow, ncol), "integer", ptr, offs, vals)
    for na_rm in (False, True):
        for op in ("sum", "max", "countNAs"):
            v, w = runners.api_row(x, op, na_rm, None)
            e, ew = runners.port_row(x, op, na_rm, None)
            assert_identical(v, e, (op, na_rm))
    m, v = sa.rowMoments(x, na_rm=True)
    ok = vals != fx.NA_I
    s1 = np.bincount(offs[ok], weights=vals[ok], minlength=nrow)
    s2 = np.bincount(offs[ok], weights=vals[ok].astype(np.float64) ** 2,
                     minlength=nrow)
    nn = ncol - np.bincount(offs[~ok], minlength=nrow)
    assert_close(np.asarray(m), s1 / nn, rtol=RTOL, what="mean")
    assert_close(np.asarray(v), (s2 - s1 ** 2 / nn) / (nn - 1), rtol=RTOL,
                 what="var", cond=(s2 + s1 ** 2 / nn) / (nn - 1))
    xl = sa.SVT_SparseArray((nrow, ncol), "integer", ptr, offs, None)
    v, w = runners.api_row(xl, "sum", False, None)
    assert_identical(v, np.bincount(offs, minlength=nrow).astype(np.float64),
                     "lacunar counts")


# ---- rowsum() / colsum() ---------------------------------------------------

GS = cases.groupsum_cases()


@pytest.mark.parametrize("name", sorted(GS))
def test_groupsum_vs_reference(name):
    G = runners.golden()
    x, rg, nrg, cg, ncg = GS[name]
    for na_rm in (False, True):
        for what, fn, g, ng in (("rowsum", runners.api_rowsum, rg, nrg),
                                ("colsum", runners.api_colsum, cg, ncg)):
            k = "gs|%s|%s|%d" % (name, what, na_rm)
            v, w = fn(x, g, ng, na_rm)
            exp = G[k]
            assert v.shape == exp.shape and v.dtype == exp.dtype, k
            if x.type == "integer":
                assert_identical(v, exp, k)
            else:
                assert_close(v, exp, rtol=RTOL, what=k,
                             cond=C.groupsum_cond(x, what, g, ng))
            assert bool(G[k + "|warn"]) == w, k


def test_groupsum_r_level_methods():
    """rowsum(x, group, reorder=) / colsum(): labels, dimnames, a resident
    handle, and the argument errors of R/rowsum-methods.R + check_group()."""
    m = np.zeros((6, 4))
    m[:, 0] = [8.55, np.inf, fx.NA_R, 0, fx.NaN, -np.inf]
    m[:, 2] = [0.6, -11.99, 0, 4.44, 0, 0]
    m[:, 3] = [1, 2, 3, 4, 5, 6]
    x = sa.SVT_SparseArray.from_dense(m, "double",
                                      dimnames=[None, list("abcd")])
    group = ["B", "A", "B", "B", "B", "A"]
    r = sa.rowsum(x, group)
    assert r.dimnames == [["A", "B"], list("abcd")]
    exp = np.array([[fx.NaN, 0, -11.99, 8.0],
                    [fx.NaN, 0, 5.04, 13.0]])
    exp[0, 0] = np.inf - np.inf
    assert_close(np.asarray(r), exp, rtol=RTOL, what="rowsum",
                 na_nan_strict=False)
    r2 = sa.rowsum(x, group, reorder=False, na_rm=True)
    assert r2.dimnames[0] == ["B", "A"]
    assert_close(np.asarray(r2)[:, 2:], exp[::-1, 2:], rtol=RTOL, what="ro")
    assert np.asarray(r2)[0, 0] == 8.55 and np.isnan(np.asarray(r2)[1, 0])
    t = sa.SVT_SparseArray.from_dense(m.T.copy(), "double")
    c = sa.colsum(t, group)
    assert_close(np.asarray(c), exp.T, rtol=RTOL, what="colsum",
                 na_nan_strict=False)
    h = sa.to_device(t)
    assert_close(np.asarray(sa.colsum(h, group)), np.asarray(c), rtol=RTOL,
                 what="resident")
    h.release()
    with pytest.raises(Exception, match="one element per row"):
        runners.api_rowsum(x, [1, 1], 1, False)
    with pytest.raises(Exception, match=">= 1 and <= 'ngroup'"):
        runners.api_rowsum(x, [1, 2, 3, 1, 1, 1], 2, False)
    lg = sa.SVT_SparseArray.from_dense(m != 0, "logical")
    with pytest.raises(Exception, match="do not support"):
        runners.api_rowsum(lg, [1] * 6, 1, False)


def test_groupsum_mid_size_against_port(mid_int, mid_dbl):
    rng = np.random.Generator(np.random.PCG64(9))
    for x in (mid_int, mid_dbl):
        rg = rng.integers(1, 13, size=x.dim[0]).astype(np.int32)
        cg = rng.integers(1, 6, size=x.dim[1]).astype(np.int32)
        for na_rm in (False, True):
            v, w = runners.api_rowsum(x, rg, 12, na_rm)
            e, ew = runners.port_rowsum(x, rg, 12, na_rm)
            if x.type == "integer":
                assert_identical(v, e, "rowsum")
            else:
                assert_close(v, e, rtol=RTOL, what="rowsum",
                             cond=C.groupsum_cond(x, "rowsum", rg, 12))
            v, w = runners.api_colsum(x, cg, 5, na_rm)
            e, ew = runners.port_colsum(x, cg, 5, na_rm)
            if x.type == "integer":
                assert_identical(v, e, "colsum")
            else:
                assert_close(v, e, rtol=RTOL, what="colsum",
                             cond=C.groupsum_cond(x, "colsum", cg, 5))
            assert w == ew


@pytest.mark.parametrize("env", [{"SVTGPU_ROWSUM_IMPL": "atomic"},
                                 {"SVTGPU_ROWSUM_IMPL": "private"},
                                 {"SVTGPU_COLSUM_IMPL": "l2"},
                                 {"SVTGPU_COLSUM_IMPL": "exact64"}])
@pytest.mark.parametrize("name", ["rand_int_na_g3", "rand_dbl_special_g3",
                                  "poisson_small_g40", "rand_lacunar_int_g3",
                                  "int_overflow_rows", "int_overflow_cols"])
def test_groupsum_other_kernels(name, env, monkeypatch):
    """the shared-memory-atomic rowsum and the 64-bit colsum (taken when
    there are many groups / no bound on the values) answer the same"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    test_groupsum_vs_reference(name)


@pytest.mark.parametrize("env", [{"SVTGPU_ROW_LACUNAR": "full"},
                                 {"SVTGPU_ROW_HIST": "off"},
                                 {"SVTGPU_ROW_LACUNAR": "full",
                                  "SVTGPU_ROW_HIST": "off"}])
@pytest.mark.parametrize("name", ["rand_lacunar_int", "rand_lacunar_lgl",
                                  "rand_lacunar_dbl", "ms_m2_lgl"])
def test_lacunar_row_kernels_full(name, env, monkeypatch):
    """lacunar matrices normally get all their row statistics from one
    counting pass (a shared-memory histogram); the strip kernels and the
    dedicated lacunar variants must agree"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    test_rowstats_vs_reference(name)
    test_row_compositions_vs_reference(name)


# ---- crossprod of two sparse matrices / crossprod(x) ----------------------

CPS = cases.sparse_crossprod_cases()


@pytest.mark.parametrize("name", sorted(CPS))
def test_sparse_crossprod_vs_reference(name):
    """C_crossprod2_SVT_SVT / C_crossprod1_SVT against the reference's
    outputs (NA vs NaN included: the same operand is made dense)"""
    G = runners.golden()
    x, y = CPS[name]
    for key, a, b in (("xy", x, y), ("yx", y, x), ("xx", x, None)):
        exp = G["cps|%s|%s" % (name, key)]
        cur = runners.api_crossprod_svt(a, b)
        assert cur.shape == exp.shape, (name, key)
        bb = a if b is None else b
        assert_close(cur, exp, rtol=RTOL, what="%s %s" % (name, key),
                     cond=C.dot_cond(a, bb.to_dense()))


def test_sparse_crossprod_blocks_and_handles():
    """more than one 64-leaf block on the dense side, both orientations, and
    resident handles on either side"""
    rng = np.random.Generator(np.random.PCG64(21))
    a = (rng.random((300, 150)) < 0.1) * rng.integers(1, 9, (300, 150))
    b = (rng.random((300, 70)) < 0.4) * rng.integers(1, 9, (300, 70))
    x = sa.SVT_SparseArray.from_dense(a.astype(np.float64), "double")
    y = sa.SVT_SparseArray.from_dense(b.astype(np.float64), "double")
    exp = a.T.astype(np.float64) @ b
    assert_close(np.asarray(sa.crossprod(x, y)), exp, rtol=RTOL, what="xy")
    assert_close(np.asarray(sa.crossprod(y, x)), exp.T, rtol=RTOL, what="yx")
    assert_close(np.asarray(sa.crossprod(x)), a.T.astype(np.float64) @ a,
                 rtol=RTOL, what="xx")
    hx, hy = sa.to_device(x), sa.to_device(y)
    assert_close(np.asarray(sa.crossprod(hx, hy)), exp, rtol=RTOL, what="h")
    assert_close(np.asarray(sa.crossprod(hx, y)), exp, rtol=RTOL, what="hx")
    assert_close(np.asarray(sa.crossprod(x, hy)), exp, rtol=RTOL, what="hy")
    assert_close(np.asarray(sa.crossprod(hx)), a.T.astype(np.float64) @ a,
                 rtol=RTOL, what="hxx")
    xi = sa.SVT_SparseArray.from_dense(a.astype(np.int32), "integer")
    yi = sa.SVT_SparseArray.from_dense(b.astype(np.int32), "integer")
    assert_identical(np.asarray(sa.crossprod(xi, yi)), exp, "int")
    hx.release()
    hy.release()
    with pytest.raises(Exception, match="non-conformable"):
        sa.crossprod(x, sa.SVT_SparseArray.from_dense(np.ones((3, 2)),
                                                      "double"))


# ---- row*(x, dims >= 2) on arrays -------------------------------------------

@pytest.mark.parametrize("name", sorted(n for n in STAT
                                        if len(STAT[n].dim) >= 3))
def test_rowstats_nd_vs_reference(name):
    G = runners.golden()
    x = STAT[name]
    for op, na_rm, dims in cases.row_requests_nd(x):
        k = runners.key_row_nd(name, op, na_rm, dims)
        v, w = runners.api_row_nd(x, op, na_rm, dims)
        exp = G[k]
        assert v.shape == exp.shape and v.dtype == exp.dtype, k
        if exp.dtype.kind != "f" or x.type != "double":
            assert_identical(v, exp, k)
        else:
            assert_close(v, exp, rtol=RTOL, what=k,
                         cond=C.cond(x, "row", op, None, dims, exp=exp))
        assert bool(G[k + "|warn"]) == w, k
    r = sa.to_device(x)
    with pytest.raises(Exception, match="resident"):
        runners.api_row_nd(r, "sum", False, 2)
    r.release()


@pytest.mark.parametrize("name", ["rand_int_na", "rand_int_dense_cols",
                                  "rand_int_big_leaves", "poisson_small",
                                  "rand_lacunar_int", "rand_lacunar_lgl",
                                  "ms_m1", "torture_2d_1"])
def test_row_hist_short_pieces(name, monkeypatch):
    """the histogram kernels cut a chunk into pieces that cannot overflow a
    cell; forcing 3-leaf pieces runs the flush, re-zero and guard-bit paths
    of all three modes on the small fixtures"""
    monkeypatch.setenv("SVTGPU_ROW_HIST_PIECE", "3")
    test_rowstats_vs_reference(name)
    test_row_compositions_vs_reference(name)
    x = STAT[name]
    if len(x.dim) == 2 and x.type != "double":
        m, v = sa.rowMoments(x, na_rm=True)
        monkeypatch.setenv("SVTGPU_ROW_HIST", "off")
        m2, v2 = sa.rowMoments(x, na_rm=True)
        assert_close(np.asarray(m), np.asarray(m2), rtol=RTOL, what="mean")
        assert_close(np.asarray(v), np.asarray(v2), rtol=RTOL, what="var",
                     cond=C.cond(x, "row", "var1"))


def test_colsum_many_pieces_per_group():
    """40,000 short columns in 3 groups: every group is summed in ~200
    shared-memory pieces (and rowsum runs 40,000 tiny leaves)"""
    rng = np.random.Generator(np.random.PCG64(31))
    nrow, ncol = 50, 40000
    mask = rng.random((ncol, nrow)) < 0.3
    cnt = mask.sum(axis=1)
    ptr = np.zeros(ncol + 1, dtype=np.int64)
    np.cumsum(cnt, out=ptr[1:])
    offs = np.nonzero(mask)[1].astype(np.int32)
    vals = rng.integers(-9, 10, size=offs.size).astype(np.int32)
    vals[vals == 0] = 3
    vals[rng.random(offs.size) < 1e-4] = fx.NA_I
    x = sa.SVT_SparseArray((nrow, ncol), "integer", ptr, offs, vals)
    cg = rng.integers(1, 4, size=ncol).astype(np.int32)
    rg = rng.integers(1, 6, size=nrow).astype(np.int32)
    for na_rm in (False, True):
        v, w = runners.api_colsum(x, cg, 3, na_rm)
        e, ew = runners.port_colsum(x, cg, 3, na_rm)
        assert_identical(v, e, "colsum")
        assert w == ew
        v, w = runners.api_rowsum(x, rg, 5, na_rm)
        e, ew = runners.port_rowsum(x, rg, 5, na_rm)
        assert_identical(v, e, "rowsum")


@pytest.mark.parametrize("lacunar", [False, True])
def test_colsum_many_rows_16bit_cells(lacunar):
    """60,000 rows do not fit one SM as int32 cells: non-negative counts go
    through 16-bit halves"""
    x = synth.poisson_svt(60000, 1500, 0.02, seed=8, na_rate=1e-4,
                          lacunar=lacunar)
    rng = np.random.Generator(np.random.PCG64(2))
    cg = rng.integers(1, 5, size=x.dim[1]).astype(np.int32)
    for na_rm in (False, True):
        v, w = runners.api_colsum(x, cg, 4, na_rm)
        e, ew = runners.port_colsum(x, cg, 4, na_rm)
        assert_identical(v, e, "colsum")
        assert w == ew


@pytest.mark.parametrize("impl", ["packed", "old"])
@pytest.mark.parametrize("ngroup", [1, 5, 12, 16, 17])
def test_rowsum_lacunar_packed_paths(impl, ngroup, monkeypatch):
    """rowsum() of a lacunar matrix keeps a leaf's group counts in packed
    registers (rowsum_lacunar_packed, <= 16 groups): leaves of 0, 1, 255 x 32
    and > 8,160 entries (the 8-bit fields must spill inside a leaf), every
    group count up to the limit and one past it (other kernel), groups that
    never occur, against the reference's compute_rowsum_ints
    (src/rowsum_methods.c:44-84); the lane-private shared-memory kernel is
    the second arm."""
    monkeypatch.setenv("SVTGPU_ROWSUM_LACUNAR", impl)
    rng = np.random.Generator(np.random.PCG64(17 + ngroup))
    nrow = 40000
    dens = [0.0, 1.0 / nrow, 0.01, 0.01, 8160.0 / nrow, 0.25, 0.6, 1.0,
            0.003, 0.0, 0.3] + [0.02] * 70
    cols = []
    for d in dens:
        if d >= 1.0:
            o = np.arange(nrow, dtype=np.int32)
        else:
            o = np.nonzero(rng.random(nrow) < d)[0].astype(np.int32)
        cols.append(o)
    ptr = np.zeros(len(cols) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([o.size for o in cols])
    offs = np.concatenate(cols)
    x = sa.SVT_SparseArray((nrow, len(cols)), "integer", ptr, offs, None)
    rg = rng.integers(1, max(ngroup, 2), size=nrow).astype(np.int32)
    rg = np.minimum(rg, ngroup)          # the last group may stay empty
    for na_rm in (False, True):
        v, w = runners.api_rowsum(x, rg, ngroup, na_rm)
        e, ew = runners.port_rowsum(x, rg, ngroup, na_rm)
        assert_identical(v, e, ("rowsum", ngroup, na_rm))
        assert w == ew
    assert int(np.asarray(v).sum()) == int(offs.size)


@pytest.mark.parametrize("mode", ["auto", "twopass"])
def test_colvars_double_one_pass_and_fallbacks(mode, monkeypatch):
    """colVars / colSds / centered_X2_sum of doubles finish sparse columns
    from the sums of one pass (S2 - 2 c S1 + n c^2, rho = n_reg / n <= 1/4)
    and take the reference's second pass (src/SparseArray_summarization.c:
    89-102) for dense columns, an explicit centre and sums of squares near
    the ends of the double range: columns on both sides of rho = 1/4,
    a large common offset (mean >> sd), values ~1e+-160 (squares overflow /
    underflow), +-Inf, NA, NaN -- against the reference at 1e-12 with the
    conditioning bound, both modes."""
    monkeypatch.setenv("SVTGPU_COLVAR_DOUBLE", mode)
    rng = np.random.Generator(np.random.PCG64(23))
    nrow = 4000
    cols = []

    def col(density, scale=1.0, shift=0.0, special=None):
        o = np.nonzero(rng.random(nrow) < density)[0].astype(np.int32)
        v = (rng.standard_normal(o.size) + shift) * scale
        v[v == 0] = scale
        if special is not None and o.size > 3:
            v[1] = special
        cols.append((o, v))

    for d in (0.01, 0.1, 0.2, 0.245, 0.255, 0.3, 0.6, 1.0):
        col(d)
        col(d, shift=1000.0)
    col(0.05, scale=1e160)
    col(0.05, scale=1e-160)
    col(0.05, scale=1e100)
    col(0.05, scale=1e-100)
    col(0.05, special=np.inf)
    col(0.05, special=-np.inf)
    col(0.05, special=fx.NA_R)
    col(0.05, special=np.nan)
    col(0.0)
    col(1.0 / nrow * 1.5)
    ptr = np.zeros(len(cols) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([o.size for o, _ in cols])
    offs = np.concatenate([o for o, _ in cols])
    vals = np.concatenate([v for _, v in cols]).astype(np.float64)
    x = sa.SVT_SparseArray((nrow, len(cols)), "double", ptr, offs, vals)
    for na_rm in (False, True):
        for op, center in (("var1", None), ("sd1", None),
                           ("centered_X2_sum", None),
                           ("centered_X2_sum", 0.5)):
            with np.errstate(all="ignore"):
                v, w = runners.api_col(x, op, na_rm, center, 1)
                e, ew = runners.port_col(x, op, na_rm, center, 1)
                assert_close(v, e, rtol=RTOL, what=(op, na_rm, center),
                             cond=C.cond(x, "col", op, center))
            assert w == ew


@pytest.mark.parametrize("name", ["rand_int_na", "poisson_small", "ms_m1",
                                  "rand_int_big_leaves", "torture_3d_int"])
def test_summarize_int_var_two_pass_form(name, monkeypatch):
    """var() / sd() of integer arrays normally come from exact 64-bit sums in
    one pass; the two-pass form (mean first) must agree"""
    monkeypatch.setenv("SVTGPU_SUMMARIZE_VAR", "twopass")
    test_summarize_vs_reference(name)


# ---- CSC <-> device-resident SVT bridges ------------------------------------

CSC_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)),
                          "golden", "csc_bridges.npz")


@pytest.mark.parametrize("dtype,one_based,shuffle,zeros", cases.CSC_CASES)
def test_csc_bridges_vs_reference(dtype, one_based, shuffle, zeros):
    """C_svtgpu_from_CSC against the reference's C_build_SVT_from_CSC (zeros
    dropped, entries ordered by row, 0- / 1-based indices, integer / double
    indptr), C_svtgpu_to_CSC against its
    C_from_SVT_SparseMatrix_to_CsparseMatrix, and the statistics of the
    handle against the reference's on the SVT it builds (inputs and expected
    outputs stored by tests/golden/make_csc_golden.py)."""
    nrow, ncol = cases.CSC_DIM
    key = cases.csc_key(dtype, one_based, shuffle, zeros) + "|"
    with np.load(CSC_GOLDEN, allow_pickle=False) as f:
        G = {k[len(key):]: f[k] for k in f.files if k.startswith(key)}
    p, i, x = G["p"], G["i"], G["x"]
    ep, ei, ex = G["ep"], G["ei"], G["ex"]
    for ip in (p.astype(np.int32), p.astype(np.float64)):
        h = sa.from_csc((nrow, ncol), ip, x, i, one_based)
        gp, gi, gx = sa.to_csc(h)
        assert np.array_equal(gp, ep) and np.array_equal(gi, ei)
        assert np.array_equal(np.asarray(gx).view(np.uint8),
                              np.asarray(ex).view(np.uint8))
        assert sa.to_csc(h, as_ngCMatrix=True)[2] is None
        for op in ("sum", "max"):
            for na_rm in (False, True):
                e = G["col|%s|%d" % (op, na_rm)]
                v = np.asarray(sa.svt._colStats(op, h, na_rm=na_rm,
                                                useNames=False))
                if dtype == np.int32 or op == "max":
                    assert_identical(v, e, ("col", op, na_rm))
                else:
                    assert_close(v, e, rtol=RTOL, what=("col", op, na_rm),
                                 cond=np.add.reduceat(
                                     np.append(np.abs(np.nan_to_num(ex)), 0),
                                     np.minimum(ep[:-1], ex.size)) *
                                 (np.diff(ep) > 0))
                e = G["row|%s|%d" % (op, na_rm)]
                v = np.asarray(sa.svt._rowStats(op, h, na_rm=na_rm,
                                                useNames=False))
                if dtype == np.int32 or op == "max":
                    assert_identical(v, e, ("row", op, na_rm))
                else:
                    assert_close(v, e, rtol=RTOL, what=("row", op, na_rm),
                                 cond=np.bincount(
                                     ei, weights=np.abs(np.nan_to_num(ex)),
                                     minlength=nrow))
        h.release()
    # a host SVT goes the same way: to_device() then to_CSC
    xs = sa.SVT_SparseArray((nrow, ncol), "double" if dtype == np.float64
                            else "integer", ep, ei, ex)
    gp, gi, gx = sa.to_csc(xs)
    assert np.array_equal(gp, ep) and np.array_equal(gi, ei)


def test_csc_bridge_rejects_bad_input():
    p = np.array([0, 2, 3], dtype=np.int32)
    x = np.array([1.0, 2.0, 3.0])
    with pytest.raises(Exception, match="outside the matrix"):
        sa.from_csc((4, 2), p, x, np.array([0, 4, 1], dtype=np.int32))
    with pytest.raises(Exception, match="duplicates"):
        sa.from_csc((4, 2), p, x, np.array([1, 1, 1], dtype=np.int32))
    with pytest.raises(Exception, match="invalid 'slotp'"):
        sa.from_csc((4, 2), np.array([1, 2, 3], dtype=np.int32), x,
                    np.array([0, 1, 1], dtype=np.int32))
    with pytest.raises(Exception, match="invalid 'indices'"):
        sa.from_csc((4, 2), p, x, np.array([0, 1], dtype=np.int32))


def test_malformed_leaf_offsets_are_refused():
    """A leaf whose nzoffs leave [0, nrow) or do not ascend strictly must not
    reach the kernels (they index shared-memory cells with the offsets): the
    flattener checks every offset it copies and the call fails with an R
    error.  Column statistics never look at the offsets and still work."""
    x = synth.poisson_svt(500, 40, 0.1, seed=2)
    good = np.asarray(sa.colSums(x))
    for what in ("range", "order"):
        y = sa.SVT_SparseArray(x.dim, x.type, x.ptr.copy(), x.offs.copy(),
                               x.vals.copy())
        a = int(y.ptr[7])
        if what == "range":
            y.offs[a + 1] = 500
        else:
            y.offs[a + 1] = y.offs[a]
        with pytest.raises(Exception, match="invalid SVT leaf"):
            sa.rowSums(y)
        with pytest.raises(Exception, match="invalid SVT leaf"):
            sa.crossprod(y.with_type("double"), np.ones((500, 3)))
        assert_identical(np.asarray(sa.colSums(y)), good, "colSums")
    assert_identical(np.asarray(sa.rowSums(x)),
                     runners.port_row(x, "sum", False, None)[0], "after")
