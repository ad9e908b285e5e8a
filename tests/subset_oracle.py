"""TEST INFRASTRUCTURE -- the numpy restatement of `x[i, j, drop = FALSE]` on
flat CSC arrays, written leaf by leaf from the definition (look every
requested row up in the source leaf, in the order requested) rather than
from the device's routes.  Never imported by the product."""
import numpy as np


def csc_of(x):
    """(ptr, offs, vals) of an SVT_SparseArray as the device holds it: a
    mixed SVT's lacunar leaves hold ones, vals is None when every leaf is
    lacunar."""
    vals = x.vals
    if vals is not None and x.lacunar is not None:
        vals = vals.copy()
        for l in np.flatnonzero(x.lacunar):
            vals[x.ptr[l]:x.ptr[l + 1]] = 1
    return x.ptr.astype(np.int64), x.offs, vals


def subset(nrow, ptr, offs, vals, rows=None, leaves=None):
    """rows / leaves: 0-based positions (None = all, in order).  Returns
    (ptr, offs, vals) of the result; vals None when the input has none."""
    nleaf = ptr.size - 1
    rows = np.arange(nrow) if rows is None else np.asarray(rows, np.int64)
    leaves = np.arange(nleaf) if leaves is None else \
        np.asarray(leaves, np.int64)
    where = np.full(nrow, -1, np.int64)    # position of row r in the leaf
    out_p = np.zeros(leaves.size + 1, np.int64)
    out_o, out_v = [], []
    for k, l in enumerate(leaves):
        a, b = int(ptr[l]), int(ptr[l + 1])
        where[offs[a:b]] = np.arange(a, b)
        hit = where[rows]
        keep = np.flatnonzero(hit >= 0)
        out_o.append(keep.astype(np.int32))
        if vals is not None:
            out_v.append(vals[hit[keep]])
        out_p[k + 1] = out_p[k] + keep.size
        where[offs[a:b]] = -1
    o = np.concatenate(out_o) if out_o else np.zeros(0, np.int32)
    v = None
    if vals is not None:
        v = np.concatenate(out_v) if out_v else np.zeros(0, vals.dtype)
    return out_p, o, v
