"""Host-side mirror of the reference's R interface for the SVT hot path.

`SVT_SparseArray` plays the role of the S4 object of
R/SVT_SparseArray-class.R:29-48 (slots dim, dimnames, type, SVT); the
functions below are the matrixStats / multiplication methods of
R/SparseArray-matrixStats.R and R/SparseMatrix-mult.R with the same names,
argument meaning and error behaviour.  Each one normalises its arguments as
the R method does and then performs the very `.Call` the R method performs
(SparseArray.Call -> C_colStats_SVT / C_rowStats_SVT / C_crossprod2_SVT_mat /
C_crossprod2_mat_SVT), served by the GPU glue in libsvt_rglue.so.  Nothing is
computed in Python except the R-level compositions the reference itself does
in R (rowMeans = sums / nvals, rowVars = X2 / (nvals - 1), rowSds = sqrt).
"""
import numpy as np

from . import rcall
from .rcall import rshim

NA_INTEGER = rshim.NA_INTEGER
NA_REAL = rshim.NA_REAL
is_na_real = rshim.is_na_real

_NP = {"logical": np.int32, "integer": np.int32, "double": np.float64}
_RT = {"logical": rshim.LGLSXP, "integer": rshim.INTSXP,
       "double": rshim.REALSXP}
_TYPE_OF_SEXP = {rshim.LGLSXP: "logical", rshim.INTSXP: "integer",
                 rshim.REALSXP: "double"}


class RArray(np.ndarray):
    """An R vector/array result: values + names/dimnames + R type."""

    def __new__(cls, a, names=None, dimnames=None, rtype=None,
                warnings=()):
        obj = np.asarray(a).view(cls)
        obj.names = names
        obj.dimnames = dimnames
        obj.rtype = rtype
        obj.warnings = list(warnings)
        return obj

    def __array_finalize__(self, obj):
        self.names = getattr(obj, "names", None)
        self.dimnames = getattr(obj, "dimnames", None)
        self.rtype = getattr(obj, "rtype", None)
        self.warnings = getattr(obj, "warnings", [])


def _wmsg_stop(msg):
    raise ValueError(msg)


class SVT_SparseArray:
    """dim / dimnames / type / SVT, the SVT held as a flat CSC over leaves.

    ptr[nleaf+1] (int64), offs[nnz] (int32, ascending per leaf), vals[nnz]
    (int32 or float64; None when every leaf is lacunar), lacunar[nleaf]
    (uint8, optional per-leaf flags for mixed SVTs).  Leaf l of an N-d array
    is the column at [, i1, i2, ...] with l = i1 + d1 * (i2 + d2 * ...).
    """

    def __init__(self, dim, type, ptr, offs, vals=None, lacunar=None,
                 dimnames=None):
        self.dim = tuple(int(d) for d in dim)
        if type not in _NP:
            raise ValueError("unsupported type(): %r" % (type,))
        self.type = type
        self.ptr = np.ascontiguousarray(ptr, dtype=np.int64)
        self.offs = np.ascontiguousarray(offs, dtype=np.int32)
        self.vals = None if vals is None else \
            np.ascontiguousarray(vals, dtype=_NP[type])
        self.lacunar = None if lacunar is None else \
            np.ascontiguousarray(lacunar, dtype=np.uint8)
        nleaf = int(np.prod(self.dim[1:], dtype=np.int64))
        if self.ptr.size != nleaf + 1:
            raise ValueError("ptr must have prod(dim[-1]) + 1 entries")
        if dimnames is None:
            dimnames = [None] * len(self.dim)
        self.dimnames = [None if d is None else list(d) for d in dimnames]
        self._robjs = None

    # -- construction -----------------------------------------------------
    @classmethod
    def from_dense(cls, a, type=None, dimnames=None, lacunar="auto"):
        """as(a, "SVT_SparseArray"): nonzero = `a != 0` (NA/NaN included).
        Leaves whose values are all 1 become lacunar (src/leaf_utils.c:
        115-122) unless lacunar=False."""
        a = np.asarray(a)
        if type is None:
            type = "double" if a.dtype.kind == "f" else \
                   "logical" if a.dtype.kind == "b" else "integer"
        a = a.astype(_NP[type], copy=False)
        if a.ndim < 1:
            raise ValueError("need at least 1 dimension")
        dim = a.shape
        nleaf = int(np.prod(dim[1:], dtype=np.int64))
        cols = a.reshape((dim[0], nleaf), order="F")
        ptr = np.zeros(nleaf + 1, dtype=np.int64)
        offs, vals, lac = [], [], np.zeros(nleaf, dtype=np.uint8)
        for l in range(nleaf):
            col = cols[:, l]
            nz = np.flatnonzero(col != 0)
            ptr[l + 1] = ptr[l] + nz.size
            offs.append(nz.astype(np.int32))
            v = col[nz]
            vals.append(v)
            if lacunar == "auto" and nz.size > 0 and np.all(v == 1):
                lac[l] = 1
        offs = np.concatenate(offs) if offs else np.zeros(0, np.int32)
        vals = np.concatenate(vals) if vals else np.zeros(0, _NP[type])
        nonempty = np.diff(ptr) > 0
        if lacunar == "auto" and nonempty.any() and lac[nonempty].all():
            return cls(dim, type, ptr, offs, None, None, dimnames)
        return cls(dim, type, ptr, offs, vals,
                   lac if lac.any() else None, dimnames)

    def to_dense(self):
        nleaf = self.ptr.size - 1
        out = np.zeros((self.dim[0], nleaf), dtype=_NP[self.type], order="F")
        for l in range(nleaf):
            a, b = self.ptr[l], self.ptr[l + 1]
            if a == b:
                continue
            lac = self.vals is None or \
                (self.lacunar is not None and self.lacunar[l])
            out[self.offs[a:b], l] = 1 if lac else self.vals[a:b]
        return out.reshape(self.dim, order="F")

    @property
    def nnz(self):
        return int(self.ptr[-1])

    def with_type(self, type):
        """`type(x) <- type` (R/SVT_SparseArray-class.R:133-146) for the
        lossless integer/logical -> double direction used before crossprod."""
        if type == self.type:
            return self
        if type != "double":
            raise ValueError("only coercion to \"double\" is supported")
        vals = None
        if self.vals is not None:
            vals = self.vals.astype(np.float64)
            vals[self.vals == NA_INTEGER] = NA_REAL
        return SVT_SparseArray(self.dim, type, self.ptr, self.offs, vals,
                               self.lacunar, self.dimnames)

    # -- R objects for .Call ---------------------------------------------
    def _leaf(self, l):
        a, b = int(self.ptr[l]), int(self.ptr[l + 1])
        if a == b:
            return None
        lac = self.vals is None or \
            (self.lacunar is not None and self.lacunar[l])
        nzvals = None if lac else rshim.wrap(self.vals[a:b], _RT[self.type])
        return rshim.rlist([nzvals, rshim.wrap(self.offs[a:b], rshim.INTSXP)])

    def _subtree(self, ndim, base, span):
        """SVT node covering leaves [base, base + span * dim[ndim-1])."""
        if ndim == 1:
            return self._leaf(base)
        n = self.dim[ndim - 1]
        sub = span // self.dim[ndim - 2] if ndim > 2 else 1
        if self.ptr[base + n * span] == self.ptr[base]:
            return None
        return rshim.rlist([self._subtree(ndim - 1, base + i * span, sub)
                            for i in range(n)])

    def _build_robjs(self):
        if self._robjs is not None:
            return self._robjs
        ndim = len(self.dim)
        nleaf = self.ptr.size - 1
        if self.nnz == 0 or nleaf == 0:
            svt = None
        elif ndim == 2:
            svt = rshim.svt_from_csc(nleaf, self.ptr, self.offs, self.vals,
                                     _RT[self.type], self.lacunar)
        elif ndim == 1:
            svt = self._leaf(0)
        else:
            span = 1
            for d in self.dim[1:-1]:
                span *= d
            svt = self._subtree(ndim, 0, span)
        if all(d is None for d in self.dimnames):
            dn = None
        else:
            dn = rshim.rlist([None if d is None else rshim.string(d)
                              for d in self.dimnames])
        self._robjs = {"dim": rshim.integer(list(self.dim)), "dimnames": dn,
                       "type": rshim.string(self.type), "SVT": svt}
        return self._robjs

    r_dim = property(lambda self: self._build_robjs()["dim"])
    r_dimnames = property(lambda self: self._build_robjs()["dimnames"])
    r_type = property(lambda self: self._build_robjs()["type"])
    r_SVT = property(lambda self: self._build_robjs()["SVT"])

    def release(self):
        if self._robjs is not None:
            for o in self._robjs.values():
                if o is not None:
                    o.release()
            self._robjs = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    # -- Arith with R's recycling (x op v, v op x); see Arith() ------------
    __array_ufunc__ = None   # `ndarray * x` defers to x instead of broadcasting

    def __mul__(self, other):
        return Arith(self, "*", other)

    def __rmul__(self, other):
        return Arith(other, "*", self)

    def __truediv__(self, other):
        return Arith(self, "/", other)

    def __rtruediv__(self, other):
        return Arith(other, "/", self)   # refused: v / x

    # `x + y`, `x - y` need two SVTs; `x + 1` reaches Arith()'s refusal
    def __add__(self, other):
        return Arith(self, "+", other)

    def __radd__(self, other):
        return Arith(other, "+", self)

    def __sub__(self, other):
        return Arith(self, "-", other)

    def __rsub__(self, other):
        return Arith(other, "-", self)

    # -- Logic between two SVTs; see Logic() --------------------------------
    def __and__(self, other):
        return Logic(self, "&", other)

    def __rand__(self, other):
        return Logic(other, "&", self)

    def __or__(self, other):
        return Logic(self, "|", other)

    def __ror__(self, other):
        return Logic(other, "|", self)

    # -- Compare (x op v; `v < x` reaches x.__gt__(v)); see Compare().  No
    # __eq__ / __ne__: SVT objects compare and hash by identity, so `==` and
    # `!=` go through Compare() ----------------------------------------------
    def __gt__(self, other):
        return Compare(self, ">", other)

    def __ge__(self, other):
        return Compare(self, ">=", other)

    def __lt__(self, other):
        return Compare(self, "<", other)

    def __le__(self, other):
        return Compare(self, "<=", other)

    # -- subsetting; see subset() ---------------------------------------------
    def __getitem__(self, key):
        """`x[key]` with numpy's conventions, served by subset(): one key
        per dimension (missing trailing ones mean all), each a 0-based int
        (negative counts from the end), a slice, a 1-D integer array or a
        boolean mask of exactly that extent.  Every dimension is kept, as
        with R's `drop = FALSE`: `x[3]` has one row."""
        if not isinstance(key, tuple):
            key = (key,)
        if len(key) > len(self.dim):
            raise IndexError("too many indices: the array has %d dimensions"
                             % len(self.dim))
        key = key + (slice(None),) * (len(self.dim) - len(key))
        return subset(self, [_numpy_key_to_subscript(k, n)
                             for k, n in zip(key, self.dim)])


class ResidentSVT(SVT_SparseArray):
    """An SVT_SparseArray whose SVT already lives in HBM: `r_SVT` is the
    external pointer made by C_svtgpu_resident_SVT, which every entry point
    of the GPU path accepts in place of the SVT list -- nothing is flattened
    or uploaded per call (SURVEY section 8f item 2).  Made by `to_device()`;
    `release()` (or garbage collection) frees the device memory."""


def to_device(x):
    """Flatten + upload `x` once; returns a ResidentSVT usable wherever an
    SVT_SparseArray is (colSums(), rowVars(), crossprod(), sum(), ...)."""
    if isinstance(x, ResidentSVT):
        return x
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    ans, _ = rcall.SparseArray_Call("C_svtgpu_resident_SVT", x.r_dim,
                                    x.r_type, x.r_SVT)
    r = ResidentSVT.__new__(ResidentSVT)
    r.dim, r.type = x.dim, x.type
    r.ptr, r.offs, r.vals, r.lacunar = x.ptr, x.offs, x.vals, x.lacunar
    r.dimnames = [None if d is None else list(d) for d in x.dimnames]
    if all(d is None for d in r.dimnames):
        dn = None
    else:
        dn = rshim.rlist([None if d is None else rshim.string(d)
                          for d in r.dimnames])
    r._robjs = {"dim": rshim.integer(list(r.dim)), "dimnames": dn,
                "type": rshim.string(r.type), "SVT": rshim.RObj(ans)}
    return r


def from_csc(dim, indptr, data, indices, indices_are_1based=False):
    """CSC arrays (a dgCMatrix's @p / @x / @i, a TENxMatrix group) straight
    into HBM: the reference builds an SVT from them with
    C_build_SVT_from_CSC() (R/SVT_SparseArray-class.R:261-275,
    src/SVT_SparseArray_class.c:833-861); here the extension entry point
    C_svtgpu_from_CSC makes a device-resident handle with the same
    conventions (zeros in `data` dropped, entries ordered by row) and no
    R list in between.  Returns a ResidentSVT."""
    data = np.asarray(data)
    type_ = "double" if data.dtype.kind == "f" else \
        "logical" if data.dtype.kind == "b" else "integer"
    data = np.ascontiguousarray(data, dtype=_NP[type_])
    indices = np.ascontiguousarray(indices, dtype=np.int32)
    indptr = np.asarray(indptr)
    if indptr.dtype.kind == "f" or (indptr.size and
                                    int(indptr[-1]) > 2**31 - 1):
        ip = rshim.wrap(np.ascontiguousarray(indptr, dtype=np.float64),
                        rshim.REALSXP)
    else:
        ip = rshim.wrap(np.ascontiguousarray(indptr, dtype=np.int32),
                        rshim.INTSXP)
    temps = [rshim.integer([int(d) for d in dim]), ip,
             rshim.wrap(data, _RT[type_]), rshim.wrap(indices, rshim.INTSXP),
             rshim.logical([int(indices_are_1based)])]
    try:
        ans, _ = rcall.SparseArray_Call("C_svtgpu_from_CSC", *temps)
    finally:
        for t in temps:
            t.release()
    r = ResidentSVT.__new__(ResidentSVT)
    r.dim, r.type = tuple(int(d) for d in dim), type_
    r.ptr = r.offs = r.vals = r.lacunar = None
    r.dimnames = [None] * len(r.dim)
    r._robjs = {"dim": rshim.integer(list(r.dim)), "dimnames": None,
                "type": rshim.string(r.type), "SVT": rshim.RObj(ans)}
    return r


def _resident_like(x, handle, type_):
    """A ResidentSVT around a new handle, with x's dim and dimnames (built
    the way from_csc() builds one)."""
    r = ResidentSVT.__new__(ResidentSVT)
    r.dim, r.type = tuple(x.dim), type_
    r.ptr = r.offs = r.vals = r.lacunar = None
    r.dimnames = [None if d is None else list(d) for d in x.dimnames]
    r._robjs = {"dim": rshim.integer(list(r.dim)),
                "dimnames": _dimnames_robj(_simplify_NULL_dimnames(
                    r.dimnames)),
                "type": rshim.string(r.type), "SVT": handle}
    return r


def _operand(v):
    """A numeric vector / scalar as an R vector: bool -> logical, integers ->
    integer (values outside the int range -> double), floats -> double."""
    a = np.asarray(v).reshape(-1)
    if a.dtype.kind == "b":
        return rshim.wrap(a.astype(np.int32), rshim.LGLSXP)
    if a.dtype.kind in "iu":
        if a.size == 0 or (a.min() >= -2**31 and a.max() <= 2**31 - 1):
            return rshim.wrap(a.astype(np.int32), rshim.INTSXP)
        return rshim.wrap(a.astype(np.float64), rshim.REALSXP)
    if a.dtype.kind == "f":
        return rshim.wrap(a.astype(np.float64), rshim.REALSXP)
    raise TypeError("non-numeric argument to binary operator")


def _ewise_result(ans, x):
    import ctypes
    elts = ctypes.cast(ans.contents.data, ctypes.POINTER(rshim.SEXP))
    type_ = rshim.strings(elts[1])[0]
    # a pointer of its own: elts[0] aliases the list slot cleared below
    handle = rshim.RObj(ctypes.cast(
        ctypes.c_void_p(ctypes.cast(elts[0], ctypes.c_void_p).value),
        rshim.SEXP))
    # detach the handle: releasing the list must not run its finalizer
    rshim.lib().SET_VECTOR_ELT(ans, 0, rshim.nil())
    rshim.lib().rshim_release_tree(ans)
    return _resident_like(x, handle, type_)


_COMPARE_OPS = (">", ">=", "<", "<=", "==", "!=")


def _arith_call(x, op, y, margin, y_on_left, entry="C_svtgpu_Arith_SVT"):
    if not isinstance(op, str):
        raise TypeError("'op' must be a single string")
    yv = _operand(y)
    temps = [yv, rshim.string(op), rshim.integer([margin]),
             rshim.logical([int(y_on_left)])]
    try:
        ans, warns = rcall.SparseArray_Call(
            entry, x.r_dim, x.r_type, x.r_SVT, temps[1], yv, temps[2],
            temps[3])
    finally:
        for t in temps:
            t.release()
    r = _ewise_result(ans, x)
    r.warnings = warns
    return r


def _ops2_call(e1, op, e2):
    """`e1 op e2` of two SVT_SparseArray objects through
    C_svtgpu_Ops_SVT_SVT; dimnames from e1, or from e2 when e1 has none."""
    if not isinstance(op, str):
        raise TypeError("'op' must be a single string")
    t = rshim.string(op)
    try:
        ans, warns = rcall.SparseArray_Call(
            "C_svtgpu_Ops_SVT_SVT", e1.r_dim, e1.r_type, e1.r_SVT, t,
            e2.r_dim, e2.r_type, e2.r_SVT)
    finally:
        t.release()
    like = e1 if any(d is not None for d in e1.dimnames) else e2
    r = _ewise_result(ans, like)
    r.warnings = warns
    return r


def _both_svt(e1, e2):
    return isinstance(e1, SVT_SparseArray) and isinstance(e2, SVT_SparseArray)


def Arith(e1, op, e2):
    """`e1 op e2` for op "*" or "/" where one side is an SVT_SparseArray and
    the other a numeric scalar or a vector of length nrow(x) (recycled along
    the first dimension, as R does).  Any other operand length is refused, as
    is `v / x` and every operation that would turn the implicit zeros into
    something else (`x * Inf`, `x * NA`, `x / 0`, "+", ...).  Served on the
    device: returns a new ResidentSVT (result type as in base R), with
    `.warnings` holding R's warnings.

    With two SVT_SparseArray operands of identical dimensions, op is "+",
    "-" or "*": `as.matrix(e1) op as.matrix(e2)` with zeros dropped, integer
    unless a side is double; "/", "^", "%%" and "%/%" are refused."""
    if _both_svt(e1, e2):
        return _ops2_call(e1, op, e2)
    if isinstance(e1, SVT_SparseArray):
        x, y, on_left = e1, e2, False
    elif isinstance(e2, SVT_SparseArray):
        x, y, on_left = e2, e1, True
    else:
        raise TypeError("one operand must be an SVT_SparseArray")
    n = np.asarray(y).size
    return _arith_call(x, op, y, 0 if n == 1 else 1, on_left)


def sweep(x, MARGIN, STATS, FUN="-"):
    """sweep(x, MARGIN, STATS, FUN) for FUN "*" or "/": STATS[i] applied to
    row i (MARGIN = 1) or STATS[j] to column j of a matrix (MARGIN = 2), as
    `t(t(x) / sf)`; a comparison FUN (">", ">=", "<", "<=", "==", "!=")
    goes to Compare().  FUN defaults to "-" as in R, which is refused (it
    would fill the implicit zeros)."""
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    if MARGIN not in (1, 2):
        _wmsg_stop("'MARGIN' must be 1 or 2")
    if FUN in _COMPARE_OPS:
        return _arith_call(x, FUN, STATS, int(MARGIN), False,
                           "C_svtgpu_Compare_SVT")
    return _arith_call(x, FUN, STATS, int(MARGIN), False)


def Compare(e1, op, e2):
    """`e1 op e2` for op ">", ">=", "<", "<=", "==" or "!=" where one side is
    an SVT_SparseArray and the other a numeric scalar or a vector of length
    nrow(x) (recycled along the first dimension, as in Arith()).  Admitted
    only when `0 op v` is FALSE for every element of the operand, so the
    implicit zeros stay FALSE (`x > 0`, `x >= 1`, `x == 3`, `x != 0`); any
    NA or NaN operand is refused.  Served on the device: returns a new
    ResidentSVT of type "logical" holding TRUE (and NA where x is NA or
    NaN).

    With two SVT_SparseArray operands of identical dimensions, op is ">",
    "<" or "!=" (`==`, `>=`, `<=` would make the implicit zeros TRUE and are
    refused); NA or NaN on either side gives NA."""
    if _both_svt(e1, e2):
        return _ops2_call(e1, op, e2)
    if isinstance(e1, SVT_SparseArray):
        x, y, on_left = e1, e2, False
    elif isinstance(e2, SVT_SparseArray):
        x, y, on_left = e2, e1, True
    else:
        raise TypeError("one operand must be an SVT_SparseArray")
    n = np.asarray(y).size
    return _arith_call(x, op, y, 0 if n == 1 else 1, on_left,
                       "C_svtgpu_Compare_SVT")


def Logic(e1, op, e2):
    """`e1 & e2` / `e1 | e2` of two SVT_SparseArray objects of identical
    dimensions: a new logical ResidentSVT, with base R's three-valued logic
    (a nonzero value is TRUE, NA and NaN are NA).  A scalar or vector
    operand is not supported."""
    if not _both_svt(e1, e2):
        raise TypeError("Logic on the GPU path needs two SVT_SparseArray "
                        "operands")
    return _ops2_call(e1, op, e2)


def _is_call(x, fun):
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    t = rshim.string(fun)
    try:
        ans, warns = rcall.SparseArray_Call("C_svtgpu_is_SVT", x.r_dim,
                                            x.r_type, x.r_SVT, t)
    finally:
        t.release()
    r = _ewise_result(ans, x)
    r.warnings = warns
    return r


def is_na(x):
    """is.na(x): a new logical ResidentSVT, TRUE where x holds NA or NaN."""
    return _is_call(x, "is.na")


def is_nan(x):
    """is.nan(x): TRUE where x holds a NaN that is not NA (never for integer
    or logical x)."""
    return _is_call(x, "is.nan")


def is_infinite(x):
    """is.infinite(x): TRUE where x holds Inf or -Inf."""
    return _is_call(x, "is.infinite")


def Math(x, op):
    """op(x) for the Math functions that map 0 to 0: abs, sign, sqrt, floor,
    ceiling, trunc, log1p, expm1 (any other name is refused).  Result type
    double, except abs() of integer / logical input; NA and NaN keep their
    kind; `.warnings` holds "NaNs produced" when one was made.  Returns a new
    ResidentSVT."""
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    t = rshim.string(op)
    try:
        ans, warns = rcall.SparseArray_Call("C_svtgpu_Math_SVT", x.r_dim,
                                            x.r_type, x.r_SVT, t)
    finally:
        t.release()
    r = _ewise_result(ans, x)
    r.warnings = warns
    return r


def to_csc(x, as_ngCMatrix=False):
    """(p, i, x) of a device-resident matrix, as
    C_from_SVT_SparseMatrix_to_CsparseMatrix() returns them
    (src/SVT_SparseArray_class.c:636-679); x is None for as_ngCMatrix."""
    if not isinstance(x, ResidentSVT):
        x = to_device(x)
    t = rshim.logical([int(as_ngCMatrix)])
    try:
        ans, _ = rcall.SparseArray_Call("C_svtgpu_to_CSC", x.r_SVT, t)
    finally:
        t.release()
    import ctypes
    elts = ctypes.cast(ans.contents.data, ctypes.POINTER(rshim.SEXP))
    out = []
    for k in range(3):
        out.append(None if rshim._is_nil(elts[k])
                   else np.array(rshim.to_numpy(elts[k])[0]))
    rshim.lib().rshim_release_tree(ans)
    return tuple(out)


def _numpy_key_to_subscript(k, n):
    """one numpy-style key along an extent n -> a 1-based int32 vector, or
    None for all of the dimension in order"""
    if isinstance(k, slice):
        idx = np.arange(*k.indices(n), dtype=np.int64)
        if idx.size == n and (n == 0 or (idx[0] == 0 and k.step in (None, 1))):
            return None
    elif isinstance(k, (bool, np.bool_)):
        raise IndexError("a boolean scalar is not a subscript")
    elif isinstance(k, (int, np.integer)):
        idx = np.array([int(k)], np.int64)
    else:
        a = np.asarray(k)
        if a.ndim != 1:
            raise IndexError("only 1-D index arrays are supported")
        if a.dtype.kind == "b":
            if a.size != n:
                raise IndexError("boolean index of length %d does not match "
                                 "the extent %d" % (a.size, n))
            idx = np.flatnonzero(a)
        elif a.dtype.kind in "iu" or a.size == 0:
            idx = a.astype(np.int64)
        else:
            raise IndexError("index arrays must hold integers or booleans")
    if idx.size and (idx.min() < -n or idx.max() >= n):
        raise IndexError("index out of bounds for an extent of %d" % n)
    return (np.where(idx < 0, idx + n, idx) + 1).astype(np.int32)


def subset(x, Nindex):
    """`x[i, j, ..., drop = FALSE]` after R's normalisation of the
    subscripts: Nindex has one element per dimension, None (all of it, in
    order) or a vector of 1-based integer positions in any order, with
    duplicates repeating the row / column and a zero-length vector giving an
    extent of 0.  Served on the device by C_svtgpu_subset_SVT: returns a new
    ResidentSVT of x's type, with dimension lengths(Nindex) and dimnames
    subset the same way; values are copied bit for bit.  NA in a subscript
    ("subscript contains NAs") and positions outside [1, dim(x)[k]]
    ("subscript contains out-of-bounds indices") are refused, as are
    non-integer subscripts and an Nindex of the wrong length."""
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    temps = []
    try:
        if isinstance(Nindex, (list, tuple)):
            elts = []
            for s in Nindex:
                if s is None:
                    elts.append(None)
                    continue
                a = np.asarray(s).reshape(-1)
                if a.dtype.kind in "iu" or a.size == 0:
                    r = rshim.wrap(a.astype(np.int32), rshim.INTSXP)
                elif a.dtype.kind == "b":
                    r = rshim.wrap(a.astype(np.int32), rshim.LGLSXP)
                else:
                    r = rshim.wrap(a.astype(np.float64), rshim.REALSXP)
                elts.append(r)
            nidx = rshim.rlist(elts)
        elif isinstance(Nindex, str):
            nidx = rshim.string(Nindex)
        else:
            nidx = _operand(Nindex)
        temps.append(nidx)
        ans, warns = rcall.SparseArray_Call("C_svtgpu_subset_SVT", x.r_dim,
                                            x.r_type, x.r_SVT, nidx)
    finally:
        for t in temps:
            t.release()
    dim, dimnames = [], []
    for k, s in enumerate(Nindex):
        names = x.dimnames[k]
        if s is None:
            dim.append(x.dim[k])
            dimnames.append(names)
        else:
            s = np.asarray(s).reshape(-1)
            dim.append(s.size)
            dimnames.append(None if names is None
                            else [names[i - 1] for i in s])
    like = SVT_SparseArray.__new__(SVT_SparseArray)
    like.dim, like.dimnames = tuple(dim), dimnames
    r = _ewise_result(ans, like)
    r.warnings = warns
    return r


SVT_SparseMatrix = SVT_SparseArray


# ---------------------------------------------------------------------------
# .Call plumbing

def _finish(ans, warns):
    value, names = rshim.to_numpy(ans)
    res = RArray(value, names=names, dimnames=rshim.dimnames(ans),
                 rtype=_TYPE_OF_SEXP.get(rshim.sexptype(ans)),
                 warnings=warns)
    rshim.release_result(ans)
    return res


def _call(name, args, temps):
    try:
        ans, warns = rcall.SparseArray_Call(name, *args)
        return _finish(ans, warns)
    finally:
        for t in temps:
            t.release()


def _normarg_dims(dims):
    if isinstance(dims, bool) or not isinstance(dims, (int, np.integer)):
        if isinstance(dims, float) and dims == int(dims):
            return int(dims)
        _wmsg_stop("'dims' must be a single integer")
    return int(dims)


def _normarg_useNames(useNames):
    if useNames is None or (isinstance(useNames, float) and
                            np.isnan(useNames)):
        return True
    if not isinstance(useNames, (bool, np.bool_)):
        _wmsg_stop("'useNames' must be TRUE or FALSE")
    return bool(useNames)


_DIMS_MSG = ("'dims' must be a single integer that is > 0 and <= "
             "length(dim(x)) for the col*() functions, and >= 0 and < "
             "length(dim(x)) for the row*() functions")


def _colStats(op, x, na_rm=False, center=None, dims=1, useNames=None):
    """.colStats_SparseArray(), R/SparseArray-matrixStats.R:68-107."""
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    dims = _normarg_dims(dims)
    if dims <= 0 or dims > len(x.dim):
        _wmsg_stop(_DIMS_MSG)
    if not isinstance(na_rm, (bool, np.bool_)):
        _wmsg_stop("'na.rm' must be TRUE or FALSE")
    if center is None:
        center = NA_REAL
    else:
        if not np.isscalar(center):
            _wmsg_stop("'center' must be NULL or a single number")
        center = float(center)
    useNames = _normarg_useNames(useNames)
    temps = [rshim.logical([0]), rshim.string(op),
             rshim.logical([int(na_rm)]), rshim.real([center]),
             rshim.integer([dims])]
    args = [x.r_dim, x.r_dimnames if useNames else None, x.r_type, x.r_SVT] \
        + temps
    return _call("C_colStats_SVT", args, temps)


_NATIVE_ROW_OPS = ("countNAs", "anyNA", "min", "max", "sum",
                   "centered_X2_sum")


def _rowStats(op, x, na_rm=False, center=None, dims=1, useNames=None):
    """.rowStats_SparseArray(), R/SparseArray-matrixStats.R:197-259."""
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    dims = _normarg_dims(dims)
    if dims < 0 or dims >= len(x.dim):
        _wmsg_stop(_DIMS_MSG)
    if dims == 0:
        return _colStats(op, x, na_rm=na_rm, center=center,
                         dims=len(x.dim), useNames=useNames)
    if op not in _NATIVE_ROW_OPS:
        # .OLD_rowStats_SparseArray() (:122-148): colStats(aperm(x)).  The
        # transposition happens on the device (extension entry point); only
        # matrices with dims=1 are served that way.
        if len(x.dim) != 2 or dims != 1:
            raise NotImplementedError(
                "row operation \"%s\" on arrays goes through aperm() in the "
                "reference and is not served by the GPU path" % op)
        if not isinstance(na_rm, (bool, np.bool_)):
            _wmsg_stop("'na.rm' must be TRUE or FALSE")
        if center is None:
            c = NA_REAL
        else:
            if not np.isscalar(center):
                _wmsg_stop("'center' must be NULL or a single number")
            c = float(center)
        useNames = _normarg_useNames(useNames)
        temps = [rshim.logical([0]), rshim.string(op),
                 rshim.logical([int(na_rm)]), rshim.real([c]),
                 rshim.integer([1])]
        args = [x.r_dim, x.r_dimnames if useNames else None, x.r_type,
                x.r_SVT] + temps
        return _call("C_rowStatsT_SVT", args, temps)
    if not isinstance(na_rm, (bool, np.bool_)):
        _wmsg_stop("'na.rm' must be TRUE or FALSE")
    temps = []
    cen = None
    if center is not None:
        c = np.asarray(center)
        if c.dtype.kind not in "fiu":
            _wmsg_stop("'center' must be NULL, a single number, or an "
                       "ordinary array")
        ans_dim = x.dim[:dims]
        n = int(np.prod(ans_dim, dtype=np.int64))
        if c.ndim >= 2:
            if tuple(c.shape) != tuple(ans_dim):
                _wmsg_stop("unexpected 'center' dimensions")
            c = c.reshape(-1, order="F")
        elif c.size in (1, n):
            c = np.broadcast_to(c.reshape(-1), (n,))
        else:
            _wmsg_stop("unexpected 'center' length")
        cen = rshim.real(np.array(c, dtype=np.float64))
        temps.append(cen)
    useNames = _normarg_useNames(useNames)
    t2 = [rshim.logical([0]), rshim.string(op), rshim.logical([int(na_rm)]),
          rshim.integer([dims])]
    temps += t2
    args = [x.r_dim, x.r_dimnames if useNames else None, x.r_type, x.r_SVT,
            t2[0], t2[1], t2[2], cen, t2[3]]
    return _call("C_rowStats_SVT", args, temps)


# ---------------------------------------------------------------------------
# matrixStats methods (R/SparseArray-matrixStats.R)

def colCountNAs(x, dims=1, useNames=None):
    return _colStats("countNAs", x, dims=dims, useNames=useNames)


def rowCountNAs(x, dims=1, useNames=None):
    return _rowStats("countNAs", x, dims=dims, useNames=useNames)


def _colCountVals(x, na_rm=False, dims=1):
    ans = float(np.prod(x.dim[:dims], dtype=np.float64))
    if na_rm:
        ans = ans - np.asarray(colCountNAs(x, dims=dims, useNames=False))
    return ans


def _rowCountVals(x, na_rm=False, dims=1):
    """:300-310"""
    ans = float(np.prod(x.dim[dims:], dtype=np.float64))
    if na_rm:
        ans = ans - np.asarray(rowCountNAs(x, dims=dims, useNames=False))
    return ans


def colAnyNAs(x, dims=1, useNames=None):
    return _colStats("anyNA", x, dims=dims, useNames=useNames)


def rowAnyNAs(x, dims=1, useNames=None):
    return _rowStats("anyNA", x, dims=dims, useNames=useNames)


def colAnys(x, na_rm=False, dims=1, useNames=None):
    return _colStats("any", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colAlls(x, na_rm=False, dims=1, useNames=None):
    return _colStats("all", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colMins(x, na_rm=False, dims=1, useNames=None):
    return _colStats("min", x, na_rm=na_rm, dims=dims, useNames=useNames)


def rowMins(x, na_rm=False, dims=1, useNames=None):
    return _rowStats("min", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colMaxs(x, na_rm=False, dims=1, useNames=None):
    return _colStats("max", x, na_rm=na_rm, dims=dims, useNames=useNames)


def rowMaxs(x, na_rm=False, dims=1, useNames=None):
    return _rowStats("max", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colRanges(x, na_rm=False, dims=1, useNames=None):
    """:439-453 (two passes, bound in R)."""
    mins = colMins(x, na_rm=na_rm, dims=dims, useNames=useNames)
    maxs = colMaxs(x, na_rm=na_rm, dims=dims, useNames=False)
    if dims == len(x.dim):
        return RArray(np.concatenate([mins.reshape(-1), maxs.reshape(-1)]),
                      rtype=mins.rtype, warnings=mins.warnings + maxs.warnings)
    return RArray(np.stack([np.asarray(mins), np.asarray(maxs)], axis=-1),
                  names=mins.names, rtype=mins.rtype,
                  warnings=mins.warnings + maxs.warnings)


def rowRanges(x, na_rm=False, dims=1, useNames=None):
    mins = rowMins(x, na_rm=na_rm, dims=dims, useNames=useNames)
    maxs = rowMaxs(x, na_rm=na_rm, dims=dims, useNames=False)
    return RArray(np.stack([np.asarray(mins), np.asarray(maxs)], axis=-1),
                  names=mins.names, rtype=mins.rtype,
                  warnings=mins.warnings + maxs.warnings)


def rowProds(x, na_rm=False, dims=1, useNames=None):
    return _rowStats("prod", x, na_rm=na_rm, dims=dims, useNames=useNames)


def rowMeans2(x, na_rm=False, dims=1, useNames=None):
    return _rowStats("mean", x, na_rm=na_rm, dims=dims, useNames=useNames)


def rowAnys(x, na_rm=False, dims=1, useNames=None):
    return _rowStats("any", x, na_rm=na_rm, dims=dims, useNames=useNames)


def rowAlls(x, na_rm=False, dims=1, useNames=None):
    return _rowStats("all", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colSums(x, na_rm=False, dims=1):
    return _colStats("sum", x, na_rm=na_rm, dims=dims)


def rowSums(x, na_rm=False, dims=1):
    return _rowStats("sum", x, na_rm=na_rm, dims=dims)


def colProds(x, na_rm=False, dims=1, useNames=None):
    return _colStats("prod", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colMeans(x, na_rm=False, dims=1):
    return _colStats("mean", x, na_rm=na_rm, dims=dims)


def rowMeans(x, na_rm=False, dims=1):
    """:511-517"""
    sums = rowSums(x, na_rm=na_rm, dims=dims)
    nvals = _rowCountVals(x, na_rm=na_rm, dims=dims)
    with np.errstate(all="ignore"):
        return _keep_na(sums, sums / nvals)


def colSums2(x, na_rm=False, dims=1, useNames=None):
    return _colStats("sum", x, na_rm=na_rm, dims=dims, useNames=useNames)


def rowSums2(x, na_rm=False, dims=1, useNames=None):
    return _rowStats("sum", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colMeans2(x, na_rm=False, dims=1, useNames=None):
    return _colStats("mean", x, na_rm=na_rm, dims=dims, useNames=useNames)


def colVars(x, na_rm=False, center=None, dims=1, useNames=None):
    return _colStats("var1", x, na_rm=na_rm, center=center, dims=dims,
                     useNames=useNames)


def colSds(x, na_rm=False, center=None, dims=1, useNames=None):
    return _colStats("sd1", x, na_rm=na_rm, center=center, dims=dims,
                     useNames=useNames)


def _keep_na(src, out):
    """numpy arithmetic may hand back either operand's NaN payload; R's
    arithmetic keeps NA_real_ when an operand is NA.  Restore that."""
    na = is_na_real(np.asarray(src)).reshape(np.shape(out))
    out = np.array(out, dtype=np.float64)
    out[na] = NA_REAL
    return RArray(out, names=getattr(src, "names", None),
                  dimnames=getattr(src, "dimnames", None), rtype="double",
                  warnings=getattr(src, "warnings", []))


def rowVars(x, na_rm=False, center=None, dims=1, useNames=None):
    """:645-661: nvals, center = sums / nvals, X2 / (nvals - 1)."""
    nvals = _rowCountVals(x, na_rm=na_rm, dims=dims)
    with np.errstate(all="ignore"):
        if center is None:
            sums = rowSums(x, na_rm=na_rm, dims=dims)
            center = _keep_na(sums, sums / nvals)
        x2 = _rowStats("centered_X2_sum", x, na_rm=na_rm,
                       center=np.asarray(center), dims=dims,
                       useNames=useNames)
        return _keep_na(x2, x2 / (nvals - 1))


def rowSds(x, na_rm=False, center=None, dims=1, useNames=None):
    v = rowVars(x, na_rm=na_rm, center=center, dims=dims, useNames=useNames)
    with np.errstate(all="ignore"):
        return _keep_na(v, np.sqrt(v))


def _medians(entry, x, na_rm, useNames):
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseArray")
    if not isinstance(na_rm, (bool, np.bool_)):
        _wmsg_stop("'na.rm' must be TRUE or FALSE")
    useNames = _normarg_useNames(useNames)
    temps = [rshim.logical([int(na_rm)])]
    args = [x.r_dim, x.r_dimnames if useNames else None, x.r_type, x.r_SVT,
            temps[0]]
    return _call(entry, args, temps)


def colMedians(x, na_rm=False, useNames=None):
    """Base R's median() of every column of a matrix, as doubles (the
    reference's colMedians() method, R/SparseArray-matrixStats.R:760-785)."""
    return _medians("C_colMedians_SVT", x, na_rm, useNames)


def rowMedians(x, na_rm=False, useNames=None):
    """Base R's median() of every row of a matrix, as doubles (:787-813);
    computed on the device transpose, which a resident handle keeps."""
    return _medians("C_rowMedians_SVT", x, na_rm, useNames)


def rowMoments(x, na_rm=False):
    """Extension: rowMeans + rowVars(center=NULL) in ONE pass over the SVT
    (the reference needs three C_rowStats_SVT passes).  Returns (mean, var)."""
    temps = [rshim.logical([int(na_rm)])]
    args = [x.r_dim, x.r_dimnames, x.r_type, x.r_SVT, temps[0]]
    try:
        ans, warns = rcall.SparseArray_Call("C_rowMoments_SVT", *args)
    finally:
        for t in temps:
            t.release()
    import ctypes
    elts = ctypes.cast(ans.contents.data, ctypes.POINTER(rshim.SEXP))
    mean = rshim.to_numpy(elts[0])[0]
    var = rshim.to_numpy(elts[1])[0]
    rshim.release_result(ans)
    return RArray(mean, rtype="double"), RArray(var, rtype="double")


# ---------------------------------------------------------------------------
# whole-array summaries (R/SparseArray-summarization.R)

def summarize_SVT(op, x, na_rm=False, center=None):
    """summarize_SVT(), R/SparseArray-summarization.R:19-46: the workhorse of
    sum(), prod(), mean(), var(), sd(), min(), max(), range(), any(), all()
    and anyNA() -- one .Call to C_summarize_SVT.  Returns a vector of length
    1 (2 for "range")."""
    if not isinstance(op, str) or not isinstance(x, SVT_SparseArray):
        raise TypeError("'op' must be a single string and 'x' an "
                        "SVT_SparseArray")
    if not isinstance(na_rm, (bool, np.bool_)):
        _wmsg_stop("'na.rm' must be TRUE or FALSE")
    if center is None:
        center = NA_REAL
    else:
        if not np.isscalar(center):
            _wmsg_stop("'center' must be NULL, or a single number")
        center = float(center)
    temps = [rshim.logical([0]), rshim.string(op),
             rshim.logical([int(na_rm)]), rshim.real([center])]
    args = [x.r_dim, x.r_type, x.r_SVT] + temps
    return _call("C_summarize_SVT", args, temps)


def anyNA(x):
    return summarize_SVT("anyNA", x)


def svt_any(x, na_rm=False):
    return summarize_SVT("any", x, na_rm=na_rm)


def svt_all(x, na_rm=False):
    return summarize_SVT("all", x, na_rm=na_rm)


def svt_min(x, na_rm=False):
    return summarize_SVT("min", x, na_rm=na_rm)


def svt_max(x, na_rm=False):
    return summarize_SVT("max", x, na_rm=na_rm)


def svt_range(x, na_rm=False, finite=False):
    """range.SVT_SparseArray(), R/SparseArray-summarization.R:181-192."""
    if finite is not False:
        _wmsg_stop("the range() method for SVT_SparseArray objects does not "
                   "support the 'finite' argument")
    return summarize_SVT("range", x, na_rm=na_rm)


def svt_sum(x, na_rm=False):
    return summarize_SVT("sum", x, na_rm=na_rm)


def svt_prod(x, na_rm=False):
    return summarize_SVT("prod", x, na_rm=na_rm)


def mean(x, na_rm=False):
    return summarize_SVT("mean", x, na_rm=na_rm)


def var(x, na_rm=False):
    return summarize_SVT("var1", x, na_rm=na_rm)


def sd(x, na_rm=False):
    return summarize_SVT("sd1", x, na_rm=na_rm)


# ---------------------------------------------------------------------------
# rowsum() / colsum() (R/rowsum-methods.R)

def _compute_ugroup(group, n, reorder):
    """S4Arrays:::compute_ugroup() as used by R/rowsum-methods.R:9,31: the
    distinct labels (None = NA), sorted with NA last when `reorder`."""
    group = list(group)
    if len(group) != n:
        _wmsg_stop("incorrect length for 'group'")
    if not isinstance(reorder, (bool, np.bool_)):
        _wmsg_stop("'reorder' must be TRUE or FALSE")
    seen, ugroup = set(), []
    for g in group:
        if g not in seen:
            seen.add(g)
            ugroup.append(g)
    if reorder:
        ugroup = sorted([g for g in ugroup if g is not None]) + \
            [g for g in ugroup if g is None]
    pos = {g: i + 1 for i, g in enumerate(ugroup)}
    return ugroup, [pos[g] for g in group]


def _groupsum(name, x, group, ngroup, na_rm):
    """.Call(name, x@dim, x@type, x@SVT, group, ngroup, na.rm); `group` =
    1-based labels (NA_INTEGER allowed)."""
    temps = [rshim.integer(group), rshim.integer([ngroup]),
             rshim.logical([int(na_rm)])]
    args = [x.r_dim, x.r_type, x.r_SVT] + temps
    return _call(name, args, temps)


def _groupsum_method(name, x, group, reorder, na_rm, by_row):
    if not isinstance(x, SVT_SparseArray) or len(x.dim) != 2:
        raise TypeError("'x' must be an SVT_SparseMatrix")
    ugroup, idx = _compute_ugroup(group, x.dim[0 if by_row else 1], reorder)
    if not isinstance(na_rm, (bool, np.bool_)):
        _wmsg_stop("'na.rm' must be TRUE or FALSE")
    ans = _groupsum(name, x, idx, len(ugroup), na_rm)
    labels = ["NA" if g is None else str(g) for g in ugroup]
    other = x.dimnames[1 if by_row else 0]
    ans.dimnames = [labels, other] if by_row else [other, labels]
    return ans


def rowsum(x, group, reorder=True, na_rm=False):
    """rowsum.SparseMatrix, R/rowsum-methods.R:7-27: sums of the rows of each
    group -> length(unique(group)) x ncol(x)."""
    return _groupsum_method("C_rowsum_SVT", x, group, reorder, na_rm, True)


def colsum(x, group, reorder=True, na_rm=False):
    """colsum() for SparseMatrix, R/rowsum-methods.R:29-49 -> nrow(x) x
    length(unique(group))."""
    return _groupsum_method("C_colsum_SVT", x, group, reorder, na_rm, False)


# ---------------------------------------------------------------------------
# crossprod / tcrossprod / %*% (R/SparseMatrix-mult.R)

def _dense_type(y):
    y = np.asarray(y)
    if y.dtype.kind == "f":
        return "double"
    if y.dtype.kind in "iu":
        return "integer"
    if y.dtype.kind == "b":
        return "logical"
    raise TypeError("unsupported matrix type")


def _common_type(tx, ty):
    """type(c(vector(type(x)), vector(type(y))))"""
    order = ["logical", "integer", "double"]
    return order[max(order.index(tx), order.index(ty))]


def _check_crossprod_input_type(type_):
    if type_ not in ("double", "integer"):
        _wmsg_stop("input objects must be of type() \"double\" or "
                   "\"integer\"")


def _simplify_NULL_dimnames(dn):
    return None if all(d is None for d in dn) else dn


def _as_matrix(y, type_):
    y = np.asarray(y)
    if y.ndim != 2:
        raise TypeError("'y' must be a matrix")
    if type_ == "double" and y.dtype.kind != "f":
        out = y.astype(np.float64)
        if y.dtype.kind in "iu":
            out[y == NA_INTEGER] = NA_REAL
        return out
    return y.astype(_NP[type_], copy=False)


def _dimnames_robj(dn):
    if dn is None:
        return None
    return rshim.rlist([None if d is None else rshim.string(list(d))
                        for d in dn])


def _crossprod2_SVT_SVT(x, y):
    """.crossprod2_SVT_SVT(), R/SparseMatrix-mult.R:88-118."""
    if len(x.dim) != 2 or len(y.dim) != 2:
        raise TypeError("'x' and 'y' must be SparseMatrix objects")
    if x.dim[0] != y.dim[0]:
        _wmsg_stop("non-conformable arguments")
    if x.type != y.type:
        xy_type = _common_type(x.type, y.type)
        _check_crossprod_input_type(xy_type)
        x, y = x.with_type(xy_type), y.with_type(xy_type)
    else:
        _check_crossprod_input_type(x.type)
    dn = _dimnames_robj(_simplify_NULL_dimnames([x.dimnames[1],
                                                 y.dimnames[1]]))
    temps = [rshim.string("double")]
    args = [x.r_dim, x.r_type, x.r_SVT, y.r_dim, y.r_type, y.r_SVT,
            temps[0], dn]
    if dn is not None:
        temps.append(dn)
    return _call("C_crossprod2_SVT_SVT", args, temps)


def _crossprod1_SVT(x):
    """.crossprod1_SVT(), R/SparseMatrix-mult.R:120-133."""
    if len(x.dim) != 2:
        raise TypeError("'x' must be a SparseMatrix")
    _check_crossprod_input_type(x.type)
    dn = _dimnames_robj(_simplify_NULL_dimnames([x.dimnames[1],
                                                 x.dimnames[1]]))
    temps = [rshim.string("double")]
    args = [x.r_dim, x.r_type, x.r_SVT, temps[0], dn]
    if dn is not None:
        temps.append(dn)
    return _call("C_crossprod1_SVT", args, temps)


def crossprod(x, y=None, transpose_y=False, y_dimnames=(None, None)):
    """crossprod(x, y) for (SVT_SparseMatrix, matrix), (matrix,
    SVT_SparseMatrix), two SVT_SparseMatrix objects, and crossprod(x):
    R/SparseMatrix-mult.R:22-133."""
    if y is None:
        return _crossprod1_SVT(x)
    if isinstance(x, SVT_SparseArray) and isinstance(y, SVT_SparseArray):
        return _crossprod2_SVT_SVT(x, y)
    if isinstance(x, SVT_SparseArray):
        return _crossprod2_SVT_mat(x, y, transpose_y, y_dimnames)
    if isinstance(y, SVT_SparseArray):
        return _crossprod2_mat_SVT(x, y, transpose_y, y_dimnames)
    raise TypeError("one operand must be an SVT_SparseMatrix")


def _crossprod2_SVT_mat(x, y, transpose_y=False, y_dimnames=(None, None)):
    if len(x.dim) != 2:
        raise TypeError("'x' must be a SparseMatrix")
    y = np.asarray(y)
    if y.ndim != 2:
        raise TypeError("'y' must be a matrix")
    if transpose_y:
        if x.dim[0] != y.shape[1]:
            _wmsg_stop("non-conformable arguments")
        ans_dimnames = [x.dimnames[1], y_dimnames[0]]
    else:
        if x.dim[0] != y.shape[0]:
            _wmsg_stop("non-conformable arguments")
        ans_dimnames = [x.dimnames[1], y_dimnames[1]]
    ty = _dense_type(y)
    if x.type == ty:
        _check_crossprod_input_type(x.type)
        xy_type = x.type
    else:
        xy_type = _common_type(x.type, ty)
        _check_crossprod_input_type(xy_type)
        x = x.with_type(xy_type)
    ym = rshim.matrix(_as_matrix(y, xy_type), _RT[xy_type])
    dn = _dimnames_robj(_simplify_NULL_dimnames(ans_dimnames))
    temps = [ym, rshim.logical([int(transpose_y)]), rshim.string("double")]
    args = [x.r_dim, x.r_type, x.r_SVT, temps[0], temps[1], temps[2], dn]
    if dn is not None:
        temps.append(dn)
    return _call("C_crossprod2_SVT_mat", args, temps)


def _crossprod2_mat_SVT(x, y, transpose_x=False, x_dimnames=(None, None)):
    if len(y.dim) != 2:
        raise TypeError("'y' must be a SparseMatrix")
    x = np.asarray(x)
    if x.ndim != 2:
        raise TypeError("'x' must be a matrix")
    if transpose_x:
        if x.shape[1] != y.dim[0]:
            _wmsg_stop("non-conformable arguments")
        ans_dimnames = [x_dimnames[0], y.dimnames[1]]
    else:
        if x.shape[0] != y.dim[0]:
            _wmsg_stop("non-conformable arguments")
        ans_dimnames = [x_dimnames[1], y.dimnames[1]]
    tx = _dense_type(x)
    if tx == y.type:
        _check_crossprod_input_type(y.type)
        xy_type = y.type
    else:
        xy_type = _common_type(tx, y.type)
        _check_crossprod_input_type(xy_type)
        y = y.with_type(xy_type)
    xm = rshim.matrix(_as_matrix(x, xy_type), _RT[xy_type])
    dn = _dimnames_robj(_simplify_NULL_dimnames(ans_dimnames))
    temps = [xm, rshim.logical([int(transpose_x)]), rshim.string("double")]
    args = [temps[0], y.r_dim, y.r_type, y.r_SVT, temps[1], temps[2], dn]
    if dn is not None:
        temps.append(dn)
    return _call("C_crossprod2_mat_SVT", args, temps)


def matmul(x, y, y_dimnames=(None, None)):
    """`x %*% y`.  (SVT_SparseMatrix, matrix): the reference computes
    crossprod(t(x), y) (:196-198), materialising t(x); here the extension
    entry point C_matmul_SVT_mat scatters without the transpose.
    (matrix, SVT_SparseMatrix): crossprod2(x, y, transpose.x=TRUE) :200-202."""
    if isinstance(x, SVT_SparseArray):
        if len(x.dim) != 2:
            raise TypeError("'x' must be a SparseMatrix")
        y = np.asarray(y)
        if y.ndim != 2:
            raise TypeError("'y' must be a matrix")
        if x.dim[1] != y.shape[0]:
            _wmsg_stop("non-conformable arguments")
        ty = _dense_type(y)
        xy_type = x.type if x.type == ty else _common_type(x.type, ty)
        _check_crossprod_input_type(xy_type)
        x = x.with_type(xy_type)
        ym = rshim.matrix(_as_matrix(y, xy_type), _RT[xy_type])
        dn = _dimnames_robj(_simplify_NULL_dimnames(
            [x.dimnames[0], y_dimnames[1]]))
        temps = [ym]
        args = [x.r_dim, x.r_type, x.r_SVT, ym, dn]
        if dn is not None:
            temps.append(dn)
        return _call("C_matmul_SVT_mat", args, temps)
    if isinstance(y, SVT_SparseArray):
        return _crossprod2_mat_SVT(x, y, transpose_x=True,
                                   x_dimnames=y_dimnames)
    raise TypeError("one operand must be an SVT_SparseMatrix")


def tcrossprod(x, y, y_dimnames=(None, None)):
    """tcrossprod(x, y) = x %*% t(y) for (SVT_SparseMatrix, matrix).  The
    reference computes crossprod(t(x), y, transpose.y=TRUE) on a materialised
    t(x) (R/SparseMatrix-mult.R:165-168); here the transpose of x happens on
    the device inside the `%*%` extension entry point."""
    if not isinstance(x, SVT_SparseArray):
        raise TypeError("'x' must be an SVT_SparseMatrix")
    y = np.asarray(y)
    if y.ndim != 2:
        raise TypeError("'y' must be a matrix")
    if x.dim[1] != y.shape[1]:
        _wmsg_stop("non-conformable arguments")
    return matmul(x, np.ascontiguousarray(y.T),
                  y_dimnames=(y_dimnames[1], y_dimnames[0]))
