"""Column-sharded use of the reference-facing API, one process per GPU.

Every rank holds the columns [l0, l1) of the matrix as its own host
SVT_SparseMatrix and calls the ordinary methods (`.Call` -> GPU) on it.
Column-shaped results are final per shard.  Row-shaped results compose across
shards exactly as the reference's R code composes them within one matrix
(R/SparseArray-matrixStats.R:300-310, 511-517, 645-661), with one allreduce of
a length-nrow vector where the R code has a whole-matrix value:

    nvals  = ncol_total - sum_over_shards(rowCountNAs)
    sums   = sum_over_shards(rowSums)
    X2     = sum_over_shards(centered_X2_sum(shard, center))   # each shard
             # starts from center^2 * ncol_shard, so the sum starts from
             # center^2 * ncol_total (src/SparseArray_matrixStats.c:1052-1058)
    rowVars = X2 / (nvals - 1)

The vectors are host arrays (they come out of `.Call`), so the reduction runs
on a CPU-capable process group (gloo) when one is given; nrow doubles only.
"""
import numpy as np

from . import svt as S


def _allreduce_sum(a, group):
    import torch
    import torch.distributed as dist
    if group is None or not dist.is_initialized() or \
            dist.get_world_size(group) == 1:
        return np.asarray(a, dtype=np.float64)
    t = torch.from_numpy(np.array(a, dtype=np.float64))
    # NA_real_ must survive the sum as NA: carry an NA count beside the data
    na = torch.from_numpy(S.is_na_real(np.asarray(a)).astype(np.float64))
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(na, op=dist.ReduceOp.SUM, group=group)
    out = t.numpy()
    out[na.numpy() > 0] = S.NA_REAL
    return out


def colSums(x, na_rm=False):
    return S.colSums(x, na_rm=na_rm)


def colMeans(x, na_rm=False):
    return S.colMeans(x, na_rm=na_rm)


def colVars(x, na_rm=False, center=None):
    return S.colVars(x, na_rm=na_rm, center=center)


def colMedians(x, na_rm=False):
    """Final per shard.  There is no sharded rowMedians(): a row median does
    not compose from the medians of column pieces."""
    return S.colMedians(x, na_rm=na_rm)


def rowSums(x, na_rm=False, group=None):
    return _allreduce_sum(S.rowSums(x, na_rm=na_rm), group)


def rowCountNAs(x, group=None):
    return _allreduce_sum(S.rowCountNAs(x, useNames=False), group)


def _ncol_total(x, group):
    import torch.distributed as dist
    if group is None or not dist.is_initialized() or \
            dist.get_world_size(group) == 1:
        return float(x.dim[1])
    return float(_allreduce_sum(np.array([x.dim[1]], dtype=np.float64),
                                group)[0])


def rowMeans(x, na_rm=False, group=None):
    nvals = _ncol_total(x, group)
    if na_rm:
        nvals = nvals - rowCountNAs(x, group)
    sums = rowSums(x, na_rm=na_rm, group=group)
    with np.errstate(all="ignore"):
        return np.asarray(S._keep_na(sums, sums / nvals))


def rowVars(x, na_rm=False, center=None, group=None):
    nvals = _ncol_total(x, group)
    if na_rm:
        nvals = nvals - rowCountNAs(x, group)
    with np.errstate(all="ignore"):
        if center is None:
            sums = rowSums(x, na_rm=na_rm, group=group)
            center = np.asarray(S._keep_na(sums, sums / nvals))
        x2 = _allreduce_sum(
            S._rowStats("centered_X2_sum", x, na_rm=na_rm,
                        center=np.asarray(center), useNames=False), group)
        return np.asarray(S._keep_na(x2, x2 / (nvals - 1)))


# ---------------------------------------------------------------------------
# whole-array summaries and grouped sums across column shards
#
# Every rank summarises its own shard through C_summarize_SVT / C_rowsum_SVT /
# C_colsum_SVT; the shard results combine the way the pieces of one vector do:
#
#   sum   = sum of shard sums                 (NA as soon as one shard says NA)
#   mean  = sum / (total length - #NA under na.rm)
#   var   = sum of centered_X2_sum(shard, center = global mean) / (n - 1)
#           (each shard adds center^2 for its own implicit zeros,
#            src/Rvector_summarization.c:1143-1147, so the pieces just add)
#   min / max / anyNA / countNAs: min / max / or / sum of the shard values
#   rowsum: column-shaped, final per shard;  colsum: one nrow x ngroup matrix
#           per shard (group labels are global), summed.

def _scalar(r):
    return float(np.asarray(r, dtype=np.float64).reshape(-1)[0])


def _length_total(x, group):
    return float(_allreduce_sum(np.array([float(np.prod(x.dim))]), group)[0])


def countNAs(x, group=None):
    n = _scalar(S.summarize_SVT("countNAs", x))
    return float(_allreduce_sum(np.array([n]), group)[0])


def anyNA(x, group=None):
    return countNAs(x, group) > 0


def _is_int(x):
    return x.type != "double"


def _shard_sum(x, na_rm):
    """this shard's sum as a double (NA_integer_ -> NA_real_)"""
    r = S.summarize_SVT("sum", x, na_rm=na_rm)
    a = np.asarray(r).reshape(-1)
    if a.dtype.kind == "i":
        return S.NA_REAL if a[0] == S.NA_INTEGER else float(a[0])
    return float(a[0])


def svt_sum(x, na_rm=False, group=None):
    """sum(svt) over all shards.  Integer input: an R integer when it fits,
    else a double (res2nakedSEXP(), src/Rvector_summarization.c:1284-1294);
    returned here as a float with NA_real_ standing for NA_integer_."""
    return float(_allreduce_sum(np.array([_shard_sum(x, na_rm)]), group)[0])


def mean(x, na_rm=False, group=None):
    n = _length_total(x, group)
    if na_rm:
        n -= countNAs(x, group)
    s = svt_sum(x, na_rm, group)
    if S.is_na_real(np.array([s]))[0]:
        return s
    with np.errstate(all="ignore"):
        return float(np.float64(s) / np.float64(n))


def var(x, na_rm=False, group=None):
    n = _length_total(x, group)
    if na_rm:
        n -= countNAs(x, group)
    center = mean(x, na_rm, group)
    if S.is_na_real(np.array([center]))[0]:
        return center          # an NA broke the sum: NA, as in the reference
    x2 = _scalar(S.summarize_SVT("centered_X2_sum", x, na_rm=na_rm,
                                 center=center)) \
        if not np.isnan(center) else float("nan")
    x2 = float(_allreduce_sum(np.array([x2]), group)[0])
    if n <= 1:
        return S.NA_REAL
    return x2 / (n - 1.0)


def sd(x, na_rm=False, group=None):
    v = var(x, na_rm, group)
    if S.is_na_real(np.array([v]))[0]:
        return v
    with np.errstate(all="ignore"):
        return float(np.sqrt(np.float64(v)))


def _extreme(x, op, na_rm, group):
    import torch
    import torch.distributed as dist
    r = np.asarray(S.summarize_SVT(op, x, na_rm=na_rm)).reshape(-1)
    if r.dtype.kind == "i":
        v = S.NA_REAL if r[0] == S.NA_INTEGER else float(r[0])
    else:
        v = float(r[0])
    if group is None or not dist.is_initialized() or \
            dist.get_world_size(group) == 1:
        return v
    # [value with NA/NaN neutralised, is NA, is NaN, shard is empty]
    na = bool(S.is_na_real(np.array([v]))[0])
    nan = bool(np.isnan(v)) and not na
    empty = float(np.prod(x.dim) == 0)
    neutral = np.inf if op == "min" else -np.inf
    val = torch.tensor([neutral if (na or nan) else v], dtype=torch.float64)
    flags = torch.tensor([float(na), float(nan), empty], dtype=torch.float64)
    dist.all_reduce(val, op=dist.ReduceOp.MIN if op == "min"
                    else dist.ReduceOp.MAX, group=group)
    dist.all_reduce(flags, op=dist.ReduceOp.SUM, group=group)
    if flags[0] > 0:
        return S.NA_REAL
    if flags[1] > 0:
        return float("nan")
    return float(val[0])


def svt_min(x, na_rm=False, group=None):
    """min over all shards (integer NA / empty-input NA come back as
    NA_real_); every shard must hold at least one column"""
    return _extreme(x, "min", na_rm, group)


def svt_max(x, na_rm=False, group=None):
    return _extreme(x, "max", na_rm, group)


def rowsum(x, row_group, ngroup, na_rm=False):
    """column-shaped: this shard's ngroup x ncol_shard block, no collective"""
    return S._groupsum("C_rowsum_SVT", x, row_group, ngroup, na_rm)


def colsum(x, col_group_of_shard, ngroup, na_rm=False, group=None):
    """nrow x ngroup sums over ALL shards: the labels of this shard's columns
    in the global numbering; integer overflow (a shard or the total leaving
    the int range) gives NA as in the reference.

    Deviation from the single-matrix reference, by construction of the
    sharding: add_sparse_vec_to_ints() (src/rowsum_methods.c:148-197) adds
    column by column and a cell stays NA once ANY prefix leaves the int range;
    here each shard applies that rule to its own columns and the shard totals
    are then added exactly -- a cell whose running sum overflows only across a
    shard boundary and comes back in range is a number here and NA there.
    (Counts near 2^31 per cell; not reachable with the BASELINE shapes.)
    Likewise NA_real_ vs NaN of a sharded double row sum follows "NA wins"
    in the host-side compositions of this module; the device-side
    DeviceSVT.rowstats() carries the reference's last-entry rule across
    shards (svt_row_sum_kind())."""
    r = S._groupsum("C_colsum_SVT", x, col_group_of_shard, ngroup, na_rm)
    a = np.asarray(r)
    if a.dtype.kind == "i":
        d = a.astype(np.float64)
        d[a == S.NA_INTEGER] = S.NA_REAL
        tot = _allreduce_sum(d, group)
        out = np.full(a.shape, S.NA_INTEGER, dtype=np.int32)
        ok = ~S.is_na_real(tot) & (np.abs(np.nan_to_num(tot)) <= 2147483647)
        out[ok] = tot[ok].astype(np.int32)
        return out
    return _allreduce_sum(a, group)
