"""Device-resident SVT column shards and the multi-GPU composition.

One process per GPU (torch.distributed): every rank owns a contiguous range of
columns (leaves) of the matrix as a device CSC.  Column-shaped results need no
collective; row-shaped results are reduced as per-row *states*
(include/svtgpu.h, svtgpu_rowstats_state_layout) that are summed / min-maxed
across ranks (NCCL allreduce over NVLink) before a tiny finalize kernel turns
them into R's answer (SURVEY.md section 8e).

torch provides device memory, streams and the process group only; all
arithmetic happens in the kernels of libsvtgpu.so, called through the C ABI.
"""
import ctypes

import numpy as np
import torch

from . import _native as N
from . import synth

_PAD = 64   # elements of slack behind offs/vals for 16-byte tail loads


def plan_column_shards(nleaf, world_size, leaf_ptr=None):
    """Contiguous leaf ranges [(l0, l1)] per rank: equal leaf counts, or
    balanced by nonzeros when the host leaf_ptr is given."""
    if world_size < 1:
        raise ValueError("world_size must be >= 1")
    if leaf_ptr is None:
        cuts = [(nleaf * r) // world_size for r in range(world_size + 1)]
    else:
        leaf_ptr = np.asarray(leaf_ptr, dtype=np.int64)
        nnz = int(leaf_ptr[-1])
        cuts = [0]
        for r in range(1, world_size):
            target = (nnz * r) // world_size
            c = int(np.searchsorted(leaf_ptr, target, side="left"))
            cuts.append(min(max(c, cuts[-1]), nleaf))
        cuts.append(nleaf)
    return [(cuts[r], cuts[r + 1]) for r in range(world_size)]


def combine_row_state(state, nrow, n_sum, n_ext, is_min, group=None):
    """Allreduce a per-row state in place: slots [0, n_sum) with SUM, slots
    [n_sum, n_sum + n_ext) with MIN or MAX.  Works on any backend (NCCL on the
    GPUs, gloo in the CPU tests).  group=None means "not sharded": nothing is
    exchanged (pass dist.group.WORLD to reduce over every rank)."""
    import torch.distributed as dist
    if group is None:          # no group given: this shard is the matrix
        return state
    if not (dist.is_available() and dist.is_initialized()):
        return state
    if dist.get_world_size(group) == 1:
        return state
    flat = state.view(-1)
    if n_sum > 0:
        dist.all_reduce(flat[: n_sum * nrow], op=dist.ReduceOp.SUM,
                        group=group)
    if n_ext > 0:
        dist.all_reduce(flat[n_sum * nrow: (n_sum + n_ext) * nrow],
                        op=dist.ReduceOp.MIN if is_min else dist.ReduceOp.MAX,
                        group=group)
    return state


def _stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class DeviceSVT:
    """A column shard [leaf0, leaf0 + nleaf) of an nrow x nleaf_total SVT in
    HBM.  val_type: "integer" / "logical" / "double"; vals None = lacunar."""

    def __init__(self, nrow, nleaf, nnz, val_type, leaf_ptr, offs, vals,
                 leaf0=0, nleaf_total=None, handle=None, owns_handle=False):
        self.nrow, self.nleaf, self.nnz = int(nrow), int(nleaf), int(nnz)
        self.val_type = val_type
        self.leaf_ptr, self.offs, self.vals = leaf_ptr, offs, vals
        self.leaf0 = int(leaf0)
        self.nleaf_total = int(nleaf if nleaf_total is None else nleaf_total)
        self._h = handle
        self._owns = owns_handle
        if self._h is None:
            h = ctypes.c_void_p()
            N.check(N.lib().svtgpu_matrix_wrap_device(
                ctypes.byref(h), self.nrow, self.nleaf, self.nnz,
                N.RTYPE[val_type], _ptr(leaf_ptr), _ptr(offs), _ptr(vals)))
            self._h = h
        if self.leaf0:
            N.check(N.lib().svtgpu_matrix_set_leaf_base(self._h, self.leaf0))

    # -- construction -------------------------------------------------
    @classmethod
    def from_host(cls, svt, leaf_range=None):
        """Upload (a column range of) a host SVT_SparseMatrix through the
        pinned staging path of the C ABI; the library owns the arrays."""
        if len(svt.dim) != 2:
            raise ValueError("DeviceSVT holds matrices")
        l0, l1 = (0, svt.dim[1]) if leaf_range is None else leaf_range
        ptr = svt.ptr[l0:l1 + 1]
        e0, e1 = int(ptr[0]), int(ptr[-1])
        ptr = np.ascontiguousarray(ptr - e0)
        offs = np.ascontiguousarray(svt.offs[e0:e1])
        vals = None
        if svt.vals is not None:
            vals = svt.vals[e0:e1]
            if svt.lacunar is not None:   # materialise ones for mixed SVTs
                vals = vals.copy()
                for l in np.flatnonzero(svt.lacunar[l0:l1]):
                    vals[ptr[l]:ptr[l + 1]] = 1
            vals = np.ascontiguousarray(vals)
        flags = N.HAS_OFFS | (N.HAS_VALS if vals is not None else 0)
        h = ctypes.c_void_p()
        L = N.lib()
        N.check(L.svtgpu_matrix_create(ctypes.byref(h), svt.dim[0], l1 - l0,
                                       e1 - e0, N.RTYPE[svt.type], flags))
        try:
            N.check(L.svtgpu_matrix_upload(
                h, ptr.ctypes.data_as(ctypes.c_void_p),
                offs.ctypes.data_as(ctypes.c_void_p),
                None if vals is None
                else vals.ctypes.data_as(ctypes.c_void_p)))
        except Exception:
            L.svtgpu_matrix_free(h)
            raise
        return cls(svt.dim[0], l1 - l0, e1 - e0, svt.type, None, None, None,
                   leaf0=l0, nleaf_total=svt.dim[1], handle=h,
                   owns_handle=True)

    @classmethod
    def generate_poisson(cls, nrow, nleaf, density, seed=0, na_rate=0.0,
                         val_type="integer", lacunar=False, leaf0=0,
                         nleaf_total=None, device=None):
        """poissonSparseArray-distributed shard generated directly in HBM
        (see sparsearray_b200/synth.py for the formula)."""
        dev = torch.device("cuda", torch.cuda.current_device()) \
            if device is None else torch.device(device)
        L = N.lib()
        nz_thr, vthr = synth.poisson_thresholds(density)
        na_thr = synth.na_threshold(na_rate)
        with torch.cuda.device(dev):
            s = _stream_ptr()
            counts = torch.empty(max(nleaf, 1), dtype=torch.int64, device=dev)
            N.check(L.svtgpu_gen_count(nrow, nleaf, leaf0, seed, nz_thr,
                                       _ptr(counts), s))
            leaf_ptr = torch.empty(nleaf + 1, dtype=torch.int64, device=dev)
            N.check(L.svtgpu_exclusive_scan(_ptr(counts), nleaf,
                                            _ptr(leaf_ptr), s))
            nnz = int(leaf_ptr[-1].item())
            offs = torch.zeros(nnz + _PAD, dtype=torch.int32, device=dev)
            vals = None
            code = 0
            if not lacunar:
                vals = torch.zeros(
                    nnz + _PAD, device=dev,
                    dtype=torch.float64 if val_type == "double"
                    else torch.int32)
                code = N.RTYPE[val_type]
            vt = (ctypes.c_uint32 * max(len(vthr), 1))(*[int(v) for v in vthr])
            N.check(L.svtgpu_gen_fill(nrow, nleaf, leaf0, seed, nz_thr,
                                      na_thr, vt, len(vthr), code,
                                      _ptr(leaf_ptr), _ptr(offs), _ptr(vals),
                                      s))
            torch.cuda.current_stream().synchronize()
        return cls(nrow, nleaf, nnz, val_type, leaf_ptr, offs, vals,
                   leaf0=leaf0, nleaf_total=nleaf_total)

    def free(self):
        if self._h is not None:
            N.lib().svtgpu_matrix_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # -- element-wise operations (new shard, no collective) ------------
    def ewise(self, op, operand=None, margin=0, operand_on_left=False):
        """x * v, v * x, x / v (op "*" / "/"), a Math function ("abs",
        "sign", "sqrt", "floor", "ceiling", "trunc", "log1p", "expm1"), a
        comparison (">", ">=", "<", "<=", "==", "!=") or "is.na", "is.nan",
        "is.infinite" as a new owning DeviceSVT with the same columns; see
        svtgpu_ewise() in include/svtgpu.h.  Comparisons and the is.*
        predicates give a "logical" result, without a value array when it
        holds no NA.  margin 2 takes the per-column vector of the whole
        matrix (length nleaf_total, sliced to this shard's columns) or this
        shard's slice.  The result's `warnings` lists R's warnings."""
        code = N.EW_OPCODES.get(op)
        if code is None:
            raise ValueError("unsupported element-wise operation %r" % (op,))
        vp, vt, vlen = None, 0, 0
        keep = None
        if op in ("*", "/") + N.EW_COMPARE:
            a = np.asarray(operand).reshape(-1)
            if margin == 2 and a.size == self.nleaf_total and \
                    self.nleaf != self.nleaf_total:
                a = a[self.leaf0:self.leaf0 + self.nleaf]
            if a.dtype.kind == "b":
                keep, vt = np.ascontiguousarray(a, dtype=np.int32), N.LGL
            elif a.dtype.kind in "iu":
                keep, vt = np.ascontiguousarray(a, dtype=np.int32), N.INT
            else:
                keep, vt = np.ascontiguousarray(a, dtype=np.float64), N.DOUBLE
            vp, vlen = keep.ctypes.data_as(ctypes.c_void_p), keep.size
        h = ctypes.c_void_p()
        warn = ctypes.c_int(0)
        N.check(N.lib().svtgpu_ewise(self._h, code, vp, vt, vlen, int(margin),
                                     int(operand_on_left), ctypes.byref(h),
                                     ctypes.byref(warn)))
        nnz, vtype = ctypes.c_int64(0), ctypes.c_int(0)
        N.check(N.lib().svtgpu_matrix_info(h, None, None, ctypes.byref(nnz),
                                           ctypes.byref(vtype), None))
        type_ = {N.LGL: "logical", N.INT: "integer",
                 N.DOUBLE: "double"}[vtype.value]
        out = DeviceSVT(self.nrow, self.nleaf, nnz.value, type_, None, None,
                        None, leaf0=self.leaf0, nleaf_total=self.nleaf_total,
                        handle=h, owns_handle=True)
        out.warnings = [msg for bit, msg in N.EW_WARNINGS if warn.value & bit]
        return out

    def download(self):
        """(leaf_ptr, offs, vals) of the shard on the host (vals None when
        the shard stores no values)."""
        L = N.lib()
        flags = ctypes.c_int(0)
        N.check(L.svtgpu_matrix_info(self._h, None, None, None, None,
                                     ctypes.byref(flags)))
        ptr = np.zeros(self.nleaf + 1, dtype=np.int64)
        offs = np.zeros(self.nnz, dtype=np.int32)
        vals = None
        if flags.value & N.HAS_VALS:
            vals = np.zeros(self.nnz, dtype=np.float64
                            if self.val_type == "double" else np.int32)
        N.check(L.svtgpu_matrix_download(
            self._h, ptr.ctypes.data_as(ctypes.c_void_p),
            offs.ctypes.data_as(ctypes.c_void_p),
            None if vals is None else vals.ctypes.data_as(ctypes.c_void_p)))
        return ptr, offs, vals

    # -- column statistics (no collective) ----------------------------
    def colstats(self, op, na_rm=False, center=None, out=None, warn=None):
        """One value per local column, left on the device."""
        code = N.OPCODES[op]
        is_int = N.lib().svtgpu_colstats_out_is_int(code,
                                                    N.RTYPE[self.val_type])
        if out is None:
            out = torch.empty(self.nleaf, device="cuda",
                              dtype=torch.int32 if is_int else torch.float64)
        if warn is None:
            warn = torch.zeros(4, dtype=torch.int32, device="cuda")
        c = synth.NA_REAL if center is None else float(center)
        N.check(N.lib().svtgpu_colstats_dev(
            self._h, code, int(na_rm), ctypes.c_double(c), 1, _ptr(out),
            _ptr(warn), _stream_ptr()))
        return out, warn

    def colmedians(self, na_rm=False, out=None):
        """colMedians() of the local columns as doubles, left on the
        device (svtgpu_colmedians_dev; no collective)."""
        if out is None:
            out = torch.empty(self.nleaf, device="cuda", dtype=torch.float64)
        N.check(N.lib().svtgpu_colmedians_dev(self._h, int(na_rm), _ptr(out),
                                              _stream_ptr()))
        return out

    def rowmedians(self, na_rm=False):
        """rowMedians() as doubles on the host, through the device transpose
        (cached in the handle).  Only for a shard that holds every column:
        a row median does not compose across column shards."""
        if self.nleaf != self.nleaf_total:
            raise ValueError("rowmedians() needs every column of the matrix "
                             "(this shard holds %d of %d): a row median does "
                             "not compose across column shards"
                             % (self.nleaf, self.nleaf_total))
        out = np.zeros(self.nrow, dtype=np.float64)
        N.check(N.lib().svtgpu_rowmedians(
            self._h, int(na_rm), out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def median_selected(self):
        """(columns or rows sent to exact selection, stored values its passes
        read) by the last host-result median call on this handle
        (svtgpu_colmedians_selected)."""
        n, r = ctypes.c_int64(0), ctypes.c_int64(0)
        N.check(N.lib().svtgpu_colmedians_selected(self._h, ctypes.byref(n),
                                                   ctypes.byref(r)))
        return n.value, r.value

    # -- whole-array summaries (host scalars; sum()/mean()/var()/range()) --
    def summarize(self, op, na_rm=False, center=None):
        """C_summarize_SVT over the local shard: (values, warn) on the host;
        values has length 1 (2 for "range")."""
        code = N.OPCODES[op]
        out = (ctypes.c_double * 2)(0.0, 0.0)
        warn = ctypes.c_int(0)
        c = synth.NA_REAL if center is None else float(center)
        N.check(N.lib().svtgpu_summarize(
            self._h, code, int(na_rm), ctypes.c_double(c), out,
            ctypes.byref(warn)))
        return [out[0], out[1]][:2 if op == "range" else 1], bool(warn.value)

    # -- grouped sums (host results; rowsum() / colsum()) -----------------
    def _groupsum(self, fn, group, ngroup, na_rm, shape):
        import numpy as np
        group = np.ascontiguousarray(group, dtype=np.int32)
        out = np.zeros(shape[0] * shape[1],
                       dtype=np.float64 if self.val_type == "double"
                       else np.int32)
        ov = ctypes.c_int(0)
        N.check(fn(self._h, group.ctypes.data_as(ctypes.c_void_p),
                   int(ngroup), int(na_rm),
                   out.ctypes.data_as(ctypes.c_void_p), ctypes.byref(ov)))
        t = N.Timings()
        N.check(N.lib().svtgpu_matrix_timings(self._h, ctypes.byref(t)))
        return out.reshape(shape, order="F"), bool(ov.value), t.kernel_ms

    def rowsum(self, group, ngroup, na_rm=False):
        """(ngroup x ncol matrix, overflow flag, kernel ms)"""
        return self._groupsum(N.lib().svtgpu_rowsum, group, ngroup, na_rm,
                              (ngroup, self.nleaf))

    def colsum(self, group, ngroup, na_rm=False):
        """(nrow x ngroup matrix, overflow flag, kernel ms)"""
        return self._groupsum(N.lib().svtgpu_colsum, group, ngroup, na_rm,
                              (self.nrow, ngroup))

    # -- row statistics (state + allreduce + finalize) ----------------
    def _ext_slots_matter(self, op, na_rm):
        """The MIN/MAX-combined slots of a row state hold the running extreme
        (min / max) or, for sums, the index of the last leaf that put an NA /
        a NaN into the row -- which only decides anything for double input
        without na.rm (svt_row_sum_kind(), csrc/svt_semantics.h: integer
        input has no NaN, na.rm ignores both).  Everything else needs ONE
        allreduce per row operation instead of two."""
        if op in ("min", "max"):
            return True
        return self.val_type == "double" and not na_rm

    def rowstats(self, op, na_rm=False, center=None, group=None, state=None):
        code = N.OPCODES[op]
        vt = N.RTYPE[self.val_type]
        n_sum, n_ext = ctypes.c_int(0), ctypes.c_int(0)
        N.check(N.lib().svtgpu_rowstats_state_layout(
            code, vt, ctypes.byref(n_sum), ctypes.byref(n_ext)))
        n_sum, n_ext = n_sum.value, n_ext.value
        if state is None:
            state = torch.empty((n_sum + n_ext) * self.nrow,
                                dtype=torch.float64, device="cuda")
        s = _stream_ptr()
        N.check(N.lib().svtgpu_rowstats_accumulate_dev(
            self._h, code, int(na_rm), _ptr(state), s))
        combine_row_state(state, self.nrow, n_sum,
                          n_ext if self._ext_slots_matter(op, na_rm) else 0,
                          op == "min", group)
        is_int = op == "anyNA" or (op in ("min", "max") and
                                   self.val_type != "double")
        out = torch.empty(self.nrow, device="cuda",
                          dtype=torch.int32 if is_int else torch.float64)
        warn = torch.zeros(4, dtype=torch.int32, device="cuda")
        N.check(N.lib().svtgpu_rowstats_finalize_dev(
            code, vt, int(na_rm), self.nrow, self.nleaf_total, _ptr(center),
            _ptr(state), _ptr(out), _ptr(warn), s))
        return out, warn

    def rowmoments(self, na_rm=False, group=None, state=None):
        """(rowMeans, rowVars) from one pass + one allreduce."""
        if state is None:
            state = torch.empty(6 * self.nrow, dtype=torch.float64,
                                device="cuda")
        s = _stream_ptr()
        N.check(N.lib().svtgpu_rowmoments_accumulate_dev(
            self._h, int(na_rm), _ptr(state), s))
        combine_row_state(state, self.nrow, 4,
                          2 if self._ext_slots_matter("sum", na_rm) else 0,
                          False, group)
        mean = torch.empty(self.nrow, dtype=torch.float64, device="cuda")
        var = torch.empty(self.nrow, dtype=torch.float64, device="cuda")
        N.check(N.lib().svtgpu_rowmoments_finalize_dev(
            N.RTYPE[self.val_type], int(na_rm), self.nrow, self.nleaf_total,
            _ptr(state), _ptr(mean), _ptr(var), s))
        return mean, var

    # -- products ------------------------------------------------------
    def crossprod(self, y_rowmajor, out=None):
        """crossprod(svt_shard, Y): Y is nrow x K row-major doubles
        (replicated on every rank); result is nleaf_local x K column-major
        (this rank's rows of the answer -- no collective)."""
        K = y_rowmajor.shape[1]
        if out is None:
            out = torch.empty(self.nleaf * K, dtype=torch.float64,
                              device="cuda")
        N.check(N.lib().svtgpu_crossprod_dev(
            self._h, _ptr(y_rowmajor), N.DOUBLE, K, _ptr(out), _stream_ptr()))
        return out

    def matmul(self, d_rowmajor, group=None, out=None):
        """svt %*% D: D is this shard's nleaf_local x K rows (row-major);
        result nrow x K row-major, summed over ranks."""
        import torch.distributed as dist
        K = d_rowmajor.shape[1]
        if out is None:
            out = torch.empty(self.nrow * K, dtype=torch.float64,
                              device="cuda")
        N.check(N.lib().svtgpu_matmul_dev(
            self._h, _ptr(d_rowmajor), N.DOUBLE, K, _ptr(out), _stream_ptr()))
        if group is not None and dist.is_available() and \
                dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
        return out
