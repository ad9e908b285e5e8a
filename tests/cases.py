"""The parity case list shared by tests/golden/make_golden.py (which runs the
reference's compiled C on every case and stores its outputs), the oracle tests
and the GPU parity tests."""
import numpy as np

import fixtures as fx
from sparsearray_b200.svt import SVT_SparseArray
from sparsearray_b200 import synth

COL_OPS_NUM = ["sum", "mean", "var1", "sd1", "min", "max", "countNAs",
               "anyNA", "prod"]
COL_OPS_INT_ONLY = ["any", "all"]
ROW_OPS = ["sum", "countNAs", "anyNA", "min", "max", "centered_X2_sum"]


def _rand_int(nrow, ncol, density, seed, na_rate=0.02, lo=-50, hi=50):
    rng = np.random.Generator(np.random.PCG64(seed))
    m = np.zeros((nrow, ncol), dtype=np.int32)
    mask = rng.random((nrow, ncol)) < density
    v = rng.integers(lo, hi, size=mask.sum()).astype(np.int32)
    v[v == 0] = 7
    m[mask] = v
    na = mask & (rng.random((nrow, ncol)) < na_rate)
    m[na] = fx.NA_I
    return m


def _rand_dbl(nrow, ncol, density, seed, special_rate=0.03):
    rng = np.random.Generator(np.random.PCG64(seed))
    m = np.zeros((nrow, ncol), dtype=np.float64)
    mask = rng.random((nrow, ncol)) < density
    v = synth._signif2(rng.standard_normal(mask.sum()) * 10)
    v[v == 0] = 0.5
    m[mask] = v
    idx = np.argwhere(mask)
    k = max(4, int(len(idx) * special_rate))
    pick = idx[rng.choice(len(idx), size=min(k, len(idx)), replace=False)]
    specials = [fx.NA_R, fx.NaN, fx.Inf, -fx.Inf]
    for n, (i, j) in enumerate(pick):
        m[i, j] = specials[n % 4]
    return m


def stat_cases():
    """name -> SVT_SparseArray"""
    out = {}
    m1, dn = fx.ms_m1()
    out["ms_m1"] = SVT_SparseArray.from_dense(m1, "integer", dimnames=dn)
    out["ms_m1_zero_rows"] = SVT_SparseArray.from_dense(
        m1[:0, :], "integer", dimnames=[None, dn[1]])
    m2, dn = fx.ms_m2_logical()
    out["ms_m2_lgl"] = SVT_SparseArray.from_dense(m2, "logical", dimnames=dn)
    out["ms_m2_lgl_zero_rows"] = SVT_SparseArray.from_dense(
        m2[:0, :], "logical", dimnames=[None, dn[1]])
    out["ms_m0_man"] = SVT_SparseArray.from_dense(fx.ms_m0_man(), "integer")
    out["ms_a3d"] = SVT_SparseArray.from_dense(fx.ms_a3d(), "double")
    for i, m in enumerate(fx.ms_torture_2d()):
        out["torture_2d_%d" % i] = SVT_SparseArray.from_dense(m, "integer")
    for dbl in (False, True):
        a = fx.ms_torture_3d(dbl)
        t = "double" if dbl else "integer"
        tag = "dbl" if dbl else "int"
        out["torture_3d_" + tag] = SVT_SparseArray.from_dense(a, t)
        out["torture_3d_%s_k0" % tag] = SVT_SparseArray.from_dense(
            a[:, :, :0], t)
        out["torture_3d_%s_j0" % tag] = SVT_SparseArray.from_dense(
            a[:, :0, :], t)
        out["torture_3d_%s_i0" % tag] = SVT_SparseArray.from_dense(
            a[:0, :, :], t)
    out["rand_int_na"] = SVT_SparseArray.from_dense(
        _rand_int(211, 67, 0.12, 11), "integer")
    out["rand_int_dense_cols"] = SVT_SparseArray.from_dense(
        _rand_int(64, 33, 1.0, 12, na_rate=0.0), "integer")
    out["rand_int_big_leaves"] = SVT_SparseArray.from_dense(
        _rand_int(9000, 5, 0.8, 13, na_rate=0.001, lo=-1000, hi=1000),
        "integer")
    out["rand_dbl_special"] = SVT_SparseArray.from_dense(
        _rand_dbl(157, 43, 0.15, 21), "double")
    out["rand_dbl_clean"] = SVT_SparseArray.from_dense(
        _rand_dbl(300, 29, 0.3, 22, special_rate=0.0)[:, :], "double",
        lacunar=False)
    out["rand_dbl_big_leaves"] = SVT_SparseArray.from_dense(
        _rand_dbl(7001, 4, 0.9, 23, special_rate=0.0005), "double")
    lac = (_rand_int(300, 50, 0.1, 31, na_rate=0.0) != 0).astype(np.int32)
    out["rand_lacunar_int"] = SVT_SparseArray.from_dense(lac, "integer")
    out["rand_lacunar_lgl"] = SVT_SparseArray.from_dense(lac, "logical")
    out["rand_lacunar_dbl"] = SVT_SparseArray.from_dense(
        lac.astype(np.float64), "double")
    mixed = _rand_int(120, 40, 0.2, 32, na_rate=0.01, lo=0, hi=3)
    mixed[:, ::3] = (mixed[:, ::3] != 0)
    out["rand_mixed_lacunar"] = SVT_SparseArray.from_dense(mixed, "integer")
    out["poisson_small"] = synth.poisson_svt(500, 64, 0.07, seed=2,
                                             na_rate=1e-2)
    out["poisson_small_dbl"] = synth.poisson_svt(400, 48, 0.07, seed=3,
                                                 na_rate=5e-3, type="double")
    out["random_small"] = synth.random_svt(2000, 50, 0.05, seed=1)
    out["all_zero"] = SVT_SparseArray.from_dense(
        np.zeros((7, 5), dtype=np.int32), "integer")
    out["one_row"] = SVT_SparseArray.from_dense(
        np.array([[3, 0, fx.NA_I, -2]], dtype=np.int32), "integer")
    out["one_col_dbl"] = SVT_SparseArray.from_dense(
        np.array([[1.5], [0.0], [fx.NaN], [-2.0]]), "double")
    return out


def col_requests(x):
    """(op, na_rm, center, dims) tuples to run on case x."""
    ops = list(COL_OPS_NUM)
    if x.type != "double":
        ops += COL_OPS_INT_ONLY
    reqs = []
    for dims in range(1, len(x.dim) + 1):
        if dims > 2 and len(x.dim) > 3:
            break
        for op in ops:
            for na_rm in (False, True):
                reqs.append((op, na_rm, None, dims))
        for na_rm in (False, True):
            reqs.append(("centered_X2_sum", na_rm, None, dims))
            reqs.append(("centered_X2_sum", na_rm, 0.5, dims))
            reqs.append(("var1", na_rm, -1.25, dims))
    return reqs


def summarize_requests(x):
    """(op, na_rm, center) for the whole-array summaries (C_summarize_SVT)."""
    ops = ["sum", "prod", "mean", "var1", "sd1", "min", "max", "range",
           "countNAs", "anyNA"]
    if x.type != "double":
        ops += COL_OPS_INT_ONLY
    reqs = []
    for op in ops:
        for na_rm in (False, True):
            reqs.append((op, na_rm, None))
    for na_rm in (False, True):
        reqs.append(("centered_X2_sum", na_rm, None))
        reqs.append(("centered_X2_sum", na_rm, 0.5))
        reqs.append(("var1", na_rm, -1.25))
    return reqs


def row_requests(x):
    """(op, na_rm, center_kind) with center_kind in None / "half" / "mean"."""
    if len(x.dim) < 2:
        return []
    reqs = []
    for op in ROW_OPS:
        for na_rm in (False, True):
            if op in ("countNAs", "anyNA") and na_rm:
                continue
            reqs.append((op, na_rm, None))
            if op == "centered_X2_sum":
                reqs.append((op, na_rm, "half"))
    return reqs


def row_requests_nd(x):
    """(op, na_rm, dims) for row*(x, dims >= 2) on arrays of >= 3 dimensions:
    the strata are head(dim, dims)-shaped."""
    if len(x.dim) < 3:
        return []
    reqs = []
    for dims in range(2, len(x.dim)):
        for op in ROW_OPS:
            for na_rm in (False, True):
                if op in ("countNAs", "anyNA") and na_rm:
                    continue
                reqs.append((op, na_rm, dims))
    return reqs


def row_center(x, kind):
    if kind is None:
        return None
    n = x.dim[0]
    return 0.5 + 0.25 * np.arange(n, dtype=np.float64)


def groupsum_cases():
    """name -> (x, row_group, n_row_groups, col_group, n_col_groups) for
    rowsum() / colsum(): 1-based labels, NA_INTEGER = the last group."""
    out = {}
    st = stat_cases()
    rng = np.random.Generator(np.random.PCG64(77))
    for name in ("ms_m1", "ms_m1_zero_rows", "torture_2d_0", "torture_2d_1",
                 "rand_int_na", "rand_int_dense_cols", "rand_int_big_leaves",
                 "rand_dbl_special", "rand_dbl_clean", "rand_dbl_big_leaves",
                 "rand_lacunar_int", "rand_lacunar_dbl", "rand_mixed_lacunar",
                 "poisson_small", "poisson_small_dbl", "random_small",
                 "all_zero", "one_row", "one_col_dbl"):
        x = st[name]
        if len(x.dim) != 2 or x.type not in ("integer", "double"):
            continue
        for ng in (1, 3, 40):
            rg = rng.integers(1, ng + 1, size=x.dim[0]).astype(np.int32)
            cg = rng.integers(1, ng + 1, size=x.dim[1]).astype(np.int32)
            if ng == 3:         # NA labels fall into the last group
                rg[rng.random(rg.size) < 0.2] = fx.NA_I
                cg[rng.random(cg.size) < 0.2] = fx.NA_I
            out["%s_g%d" % (name, ng)] = (x, rg, ng, cg, ng)
    # partial sums that leave the integer range, in both orders, and an NA
    # met before / after the overflow
    big = np.array([[2000000000, 2000000000, -2000000000, 5],
                    [2000000000, -2000000000, 2000000000, fx.NA_I],
                    [fx.NA_I, 2000000000, 2000000000, 1],
                    [2000000000, 2000000000, fx.NA_I, 1],
                    [-2147483647, -1, 0, 3],
                    [1500000000, 600000000, 47483647, 0]],
                   dtype=np.int32)
    ones4 = np.ones(4, dtype=np.int32)
    ones6 = np.ones(6, dtype=np.int32)
    out["int_overflow_rows"] = (SVT_SparseArray.from_dense(big.T.copy(),
                                                           "integer"),
                                ones4, 1, np.array([1, 2, 1, 2, 1, 2],
                                                   dtype=np.int32), 2)
    out["int_overflow_cols"] = (SVT_SparseArray.from_dense(big, "integer"),
                                ones6, 1, ones4, 1)
    return out


def crossprod_cases():
    """name -> (x SVT, y dense ndarray of x's type, transpose_y)"""
    out = {}
    m0, m1, m2, m3 = fx.cp_double()
    S = SVT_SparseArray.from_dense
    out["dbl_m2_m3"] = (S(m2, "double"), m3, False)
    out["dbl_m3_m2"] = (S(m3, "double"), m2, False)
    out["dbl_m2_tm3"] = (S(m2, "double"), np.ascontiguousarray(m3.T), True)
    out["dbl_m0_m0"] = (S(m0, "double"), m0, False)
    out["dbl_m1_m1"] = (S(m1, "double"), m1, False)
    out["dbl_m3_m3"] = (S(m3, "double"), m3, False)
    out["dbl_zero_rows"] = (S(np.zeros((0, 3)), "double"), np.zeros((0, 2)),
                            False)
    out["dbl_zero_cols_y"] = (S(m3, "double"), np.zeros((6, 0)), False)
    out["dbl_zero_cols_x"] = (S(np.zeros((6, 0)), "double"), m3, False)
    i2, i3 = fx.cp_int(False)
    out["int_m2_m3"] = (S(i2, "integer"), i3, False)
    out["int_m3_m2"] = (S(i3, "integer"), i2, False)
    out["int_m2_m2"] = (S(i2, "integer"), i2, False)
    n2, n3 = fx.cp_int(True)
    out["int_na_m2_m3"] = (S(n2, "integer"), n3, False)
    out["int_na_m3_m2"] = (S(n3, "integer"), n2, False)
    i1 = fx.cp_int_m1()
    out["int_m1_m1"] = (S(i1, "integer"), i1, False)
    out["int_zero_rows"] = (S(np.zeros((0, 3), np.int32), "integer"),
                            np.zeros((0, 3), np.int32), False)
    out["int_m3_zero_cols"] = (S(i3, "integer"), np.zeros((6, 0), np.int32),
                               False)
    # seeded random: finite and non-finite dense columns, K not a multiple
    # of the kernel's column tile
    xd = _rand_dbl(157, 43, 0.15, 41, special_rate=0.01)
    rng = np.random.Generator(np.random.PCG64(42))
    y = rng.standard_normal((157, 70))
    out["rand_dbl_finite_y"] = (S(xd, "double"), y, False)
    y2 = y.copy()
    y2[3, 1] = fx.Inf
    y2[10, 5] = fx.NaN
    y2[20, 9] = fx.NA_R
    y2[7, 64] = -fx.Inf
    out["rand_dbl_nonfinite_y"] = (S(xd, "double"), y2, False)
    out["rand_dbl_ty"] = (S(xd, "double"), np.ascontiguousarray(y2.T), True)
    xi = _rand_int(211, 37, 0.12, 43, na_rate=0.003)
    yi = rng.integers(-9, 9, size=(211, 13)).astype(np.int32)
    out["rand_int_y"] = (S(xi, "integer"), yi, False)
    yi2 = yi.copy()
    yi2[5, 2] = fx.NA_I
    out["rand_int_na_y"] = (S(xi, "integer"), yi2, False)
    lac = (_rand_int(300, 50, 0.1, 31, na_rate=0.0) != 0)
    out["lacunar_dbl_y"] = (S(lac.astype(np.float64), "double"),
                            rng.standard_normal((300, 50)), False)
    out["lacunar_int_y"] = (S(lac.astype(np.int32), "integer"),
                            rng.integers(-5, 5, (300, 7)).astype(np.int32),
                            False)
    p = synth.poisson_svt(500, 64, 0.07, seed=2, na_rate=0.0, type="double")
    out["poisson_dbl_y50"] = (p, rng.standard_normal((500, 50)), False)
    # leaves holding both an NA and a NaN: the first one decides
    # (`ans += v * y` on a register accumulator, SparseVec_dotprod.c:36-41)
    out["dbl_na_nan_order"] = (S(_na_nan_order(), "double"),
                               np.arange(1.0, 13.0).reshape(6, 2), False)
    return out


def sparse_crossprod_cases():
    """name -> (x, y) for crossprod of two SVT_SparseMatrix objects: the
    SVT x dense cases with the dense operand made sparse, plus operands with
    NULL SVTs and lacunar / mixed leaves."""
    out = {}
    for name, (x, y, ty) in crossprod_cases().items():
        y = np.ascontiguousarray(y.T if ty else y)
        if y.shape[0] != x.dim[0]:
            continue
        out[name] = (x, SVT_SparseArray.from_dense(y, x.type, lacunar=False))
    st = stat_cases()
    for a, b in (("rand_dbl_special", "rand_dbl_clean"),
                 ("rand_int_na", "rand_int_dense_cols"),
                 ("rand_lacunar_int", "rand_int_na"),
                 ("rand_lacunar_dbl", "rand_dbl_special"),
                 ("poisson_small", "poisson_small")):
        xa, xb = st[a], st[b]
        if xa.dim[0] == xb.dim[0] and xa.type == xb.type:
            out["%s_x_%s" % (a, b)] = (xa, xb)
    inf = np.zeros((5, 3))
    inf[1, 0] = np.inf
    inf[2, 1] = fx.NA_R
    inf[4, 2] = 2.0
    zero = np.zeros((5, 2))
    out["zero_x_nonfinite"] = (SVT_SparseArray.from_dense(zero, "double"),
                               SVT_SparseArray.from_dense(inf, "double"))
    out["nonfinite_x_zero"] = (SVT_SparseArray.from_dense(inf, "double"),
                               SVT_SparseArray.from_dense(zero, "double"))
    # a NULL SVT against leaves that hold a NaN BEFORE an NA: the reference's
    # "fictive matrix of zeros" routines (crossprod2_SVT_mat0_double() /
    # crossprod2_mat0_SVT_double(), src/SparseMatrix_mult.c:558-591) answer NA
    # wherever the NA stands, unlike a dense column of zeros
    nn = np.zeros((6, 4))
    nn[:, 0] = [0, fx.NaN, 3, fx.NA_R, 0, 1]      # NaN first, then NA
    nn[:, 1] = [fx.NA_R, 0, fx.NaN, 0, 0, 2]      # NA first
    nn[:, 2] = [0, fx.Inf, 0, 0, fx.NaN, 0]       # no NA
    nn[:, 3] = [1, 0, 2, 0, 3, 0]                 # clean
    z64 = np.zeros((6, 3))
    out["nan_na_x_null"] = (SVT_SparseArray.from_dense(nn, "double"),
                            SVT_SparseArray.from_dense(z64, "double"))
    out["null_x_nan_na"] = (SVT_SparseArray.from_dense(z64, "double"),
                            SVT_SparseArray.from_dense(nn, "double"))
    ni = np.zeros((6, 3), dtype=np.int32)
    ni[:, 0] = [0, 4, fx.NA_I if hasattr(fx, "NA_I") else -2**31, 0, 1, 0]
    ni[:, 2] = [1, 0, 2, 0, 3, 0]
    zi = np.zeros((6, 2), dtype=np.int32)
    out["int_na_x_null"] = (SVT_SparseArray.from_dense(ni, "integer"),
                            SVT_SparseArray.from_dense(zi, "integer"))
    out["null_x_int_na"] = (SVT_SparseArray.from_dense(zi, "integer"),
                            SVT_SparseArray.from_dense(ni, "integer"))
    return out


def _na_nan_order():
    m = np.zeros((6, 4))
    m[:, 0] = [1, fx.NA_R, 0, fx.NaN, 2, 0]       # NA first
    m[:, 1] = [1, fx.NaN, 0, fx.NA_R, 2, 0]       # NaN first
    m[:, 2] = [0, fx.NaN, 0, fx.NaN, fx.NA_R, 3]
    m[:, 3] = [fx.NA_R, 0, fx.NA_R, 0, 0, fx.NaN]
    return m


def matmul_cases():
    """name -> (x SVT, d dense of x's type): x %*% d"""
    out = {}
    S = SVT_SparseArray.from_dense
    rng = np.random.Generator(np.random.PCG64(333))
    m1 = fx.mm_m1()
    out["mm_m1_runif"] = (S(m1, "integer").with_type("double"),
                          rng.random((6, 2)))
    out["mm_m1_int"] = (S(m1, "integer"),
                        rng.integers(-4, 4, (6, 3)).astype(np.int32))
    xd = _rand_dbl(157, 43, 0.15, 51, special_rate=0.01)
    d = rng.standard_normal((43, 70))
    out["rand_dbl_finite_d"] = (S(xd, "double"), d)
    d2 = d.copy()
    d2[3, 1] = fx.Inf
    d2[10, 5] = fx.NaN
    d2[20, 9] = fx.NA_R
    out["rand_dbl_nonfinite_d"] = (S(xd, "double"), d2)
    xi = _rand_int(211, 37, 0.12, 53, na_rate=0.003)
    di = rng.integers(-9, 9, size=(37, 13)).astype(np.int32)
    out["rand_int_d"] = (S(xi, "integer"), di)
    di2 = di.copy()
    di2[5, 2] = fx.NA_I
    out["rand_int_na_d"] = (S(xi, "integer"), di2)
    lac = (_rand_int(300, 50, 0.1, 31, na_rate=0.0) != 0)
    out["lacunar_dbl_d"] = (S(lac.astype(np.float64), "double"),
                            rng.standard_normal((50, 9)))
    # rows holding both an NA and a NaN (column order decides)
    out["dbl_na_nan_order_mm"] = (S(np.ascontiguousarray(_na_nan_order().T),
                                    "double"),
                                  np.arange(1.0, 13.0).reshape(6, 2))
    return out


# CSC <-> SVT bridges: (dtype, one_based, shuffle, zeros) of the stored cases
# (tests/golden/csc_bridges.npz, written by tests/golden/make_csc_golden.py)
CSC_DIM = (211, 57)
CSC_CASES = [(np.float64, False, False, True), (np.int32, True, True, True),
             (np.float64, True, True, False), (np.int32, False, False, False)]


def csc_key(dtype, one_based, shuffle, zeros):
    return "%s|%d|%d|%d" % (np.dtype(dtype).name, one_based, shuffle, zeros)


def csc_fixture(seed, nrow, ncol, dtype, one_based, shuffle, zeros):
    """CSC arrays with explicit zeros in @x and (optionally) unsorted row
    indices inside the columns"""
    rng = np.random.Generator(np.random.PCG64(seed))
    cnt = rng.binomial(nrow, 0.2, size=ncol)
    cnt[rng.integers(0, ncol, 3)] = 0
    p = np.zeros(ncol + 1, dtype=np.int64)
    np.cumsum(cnt, out=p[1:])
    i = np.concatenate([np.sort(rng.choice(nrow, size=c, replace=False))
                        for c in cnt] + [np.zeros(0, np.int64)]).astype(np.int32)
    if dtype == np.float64:
        x = np.round(rng.standard_normal(i.size), 2)
        x[rng.random(i.size) < 0.01] = fx.NA_R
        x[rng.random(i.size) < 0.01] = np.nan
    else:
        x = rng.integers(-5, 6, size=i.size).astype(np.int32)
        x[rng.random(i.size) < 0.01] = fx.NA_I
    if zeros:
        x[rng.random(i.size) < 0.1] = 0
    else:
        x[x == 0] = 1
    if shuffle:
        for j in range(ncol):
            q = rng.permutation(cnt[j])
            i[p[j]:p[j + 1]] = i[p[j]:p[j + 1]][q]
            x[p[j]:p[j + 1]] = x[p[j]:p[j + 1]][q]
    return p, i + (1 if one_based else 0), x
