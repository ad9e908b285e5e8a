"""TEST INFRASTRUCTURE -- comparisons (x op v) and is.na / is.nan /
is.infinite by base R's dense definition, computed with numpy on the dense
matrix and turned into the CSC a logical SparseArray stores: an entry for
every TRUE or NA, values 1 / NA_integer_, and no value array at all when the
result holds no NA.  Never imported by the product."""
import numpy as np

import sparsearray_b200 as sa

NA_I = -2**31
COMPARE = (">", ">=", "<", "<=", "==", "!=")
MIRROR = {">": "<", ">=": "<=", "<": ">", "<=": ">=", "==": "==", "!=": "!="}
_NP = {">": np.greater, ">=": np.greater_equal, "<": np.less,
       "<=": np.less_equal, "==": np.equal, "!=": np.not_equal}


def admitted(op, v):
    """`0 op v` is FALSE for every element (NA and NaN never)."""
    v = np.asarray(v)
    if v.dtype.kind == "f":
        if np.isnan(v).any():
            return False
    elif (v.astype(np.int64) == NA_I).any():
        return False
    return not _NP[op](np.zeros(1, dtype=v.dtype), v).any()


def dense(a, type_, op, v=None, v_type=None, margin=0):
    """(value, na) of the dense logical result: value True where TRUE."""
    nrow = a.shape[0]
    a = a.reshape((nrow, int(np.prod(a.shape[1:]))), order="F")
    if type_ == "double":
        x = a.astype(np.float64)
        na = np.isnan(x)                       # NA and NaN alike
        is_na = sa.is_na_real(x.reshape(-1)).reshape(x.shape)
    else:
        x = a.astype(np.int32)
        na = x == NA_I
        is_na = na
    if op == "is.na":
        return na, np.zeros_like(na)
    if op == "is.nan":
        return na & ~is_na, np.zeros_like(na)
    if op == "is.infinite":
        return (np.isinf(x) if type_ == "double" else np.zeros_like(na)), \
            np.zeros_like(na)
    v = np.asarray(v)
    v = v.astype(np.float64 if v_type == "double" else np.int32)
    V = v.reshape(1, 1) if margin == 0 else \
        v.reshape(-1, 1) if margin == 1 else v.reshape(1, -1)
    with np.errstate(invalid="ignore"):
        r = _NP[op](x, V)                     # int32 vs float64 -> float64
    return r & ~na, na


def to_csc(val, na):
    """(p, i, x) of the logical result; x None when it holds no NA."""
    keep = val | na
    nleaf = keep.shape[1]
    ptr = np.zeros(nleaf + 1, dtype=np.int64)
    offs, vals = [], []
    for l in range(nleaf):
        nz = np.flatnonzero(keep[:, l])
        ptr[l + 1] = ptr[l] + nz.size
        offs.append(nz.astype(np.int32))
        vals.append(np.where(na[nz, l], NA_I, 1).astype(np.int32))
    offs = np.concatenate(offs) if offs else np.zeros(0, np.int32)
    vals = np.concatenate(vals) if vals else np.zeros(0, np.int32)
    return ptr, offs, (vals if na.any() else None)


def dense_logical(val, na):
    """The dense logical matrix as doubles (NA as NA_real_), for statistics
    held to numpy."""
    out = val.astype(np.float64)
    out[na] = sa.NA_REAL
    return out
