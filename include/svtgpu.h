/* svtgpu.h -- thin C ABI between host code and the sm_100a CUDA kernels that
 * replace the tree-walk + per-leaf loops (layers L1/L0) of Bioconductor's
 * SparseArray for SVT_SparseMatrix column/row statistics and SVT x dense
 * products.  Plain C: pointers and sizes only, int status returns (0 = ok,
 * message via svtgpu_last_error()), no R types, no exceptions, no torch types.
 *
 * The library is libsvtgpu.so (sparsearray_b200/csrc/).  There is no CPU
 * fallback: every entry point fails with SVTGPU_ERR_NO_DEVICE when no CUDA
 * device is usable.
 *
 * Reference interfaces replaced (paths under Bioconductor/SparseArray):
 *   svtgpu_matrix_*      flattening of the SVT leaf list into a device CSC;
 *                        pattern: dump_SVT_to_CsparseMatrix_slots(),
 *                        src/SVT_SparseArray_class.c:598-679 (int64 offsets
 *                        here; the reference refuses nnz > INT_MAX, :643-647)
 *   svtgpu_colstats      REC_colStats_SVT() -> _summarize_SVT() ->
 *                        _postprocess_SummarizeResult():
 *                        src/SparseArray_matrixStats.c:200-231,
 *                        src/SparseArray_summarization.c:15-109,
 *                        src/Rvector_summarization.c:177-1177
 *   svtgpu_rowstats      SVT_row{Sums,CountNAs,AnyNAs,MinsMaxs,CenteredX2Sum}
 *                        + REC_rowStats_SVT() + update_out_for_row*():
 *                        src/SparseArray_matrixStats.c:303-1072
 *   svtgpu_rowmoments    one-pass replacement for the three passes of the R
 *                        method rowVars(): R/SparseArray-matrixStats.R:645-661
 *   svtgpu_crossprod     crossprod2_SVT_mat_{double,int}(),
 *                        crossprod2_mat_SVT_{double,int}() and the
 *                        _dotprod_*() leaf kernels:
 *                        src/SparseMatrix_mult.c:131-239,385-547,
 *                        src/SparseVec_dotprod.c:28-138
 *   svtgpu_matmul        `svt %*% dense` without materialising t(svt):
 *                        R/SparseMatrix-mult.R:196-198 +
 *                        src/SparseArray_aperm.c:348-423
 */
#ifndef SVTGPU_H
#define SVTGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ---- */
#define SVTGPU_OK               0
#define SVTGPU_ERR_NO_DEVICE    1  /* no usable CUDA device / driver */
#define SVTGPU_ERR_CUDA         2  /* a CUDA call failed */
#define SVTGPU_ERR_ARG          3  /* invalid argument */
#define SVTGPU_ERR_UNSUPPORTED  4  /* valid in the reference, not on this path */
#define SVTGPU_ERR_NOMEM        5

/* ---- value types: R's SEXPTYPE codes of the leaves' nzvals ---- */
#define SVTGPU_LGL     10  /* int32 payload, NA = INT_MIN */
#define SVTGPU_INT     13  /* int32 payload, NA = INT_MIN */
#define SVTGPU_DOUBLE  14  /* NA = NaN with low word 1954, other NaNs = NaN */

/* ---- opcodes: identical to src/Rvector_summarization.h:12-32 ---- */
#define SVTGPU_OP_ANYNA             1
#define SVTGPU_OP_COUNTNAS          2
#define SVTGPU_OP_ANY               3
#define SVTGPU_OP_ALL               4
#define SVTGPU_OP_MIN               5
#define SVTGPU_OP_MAX               6
#define SVTGPU_OP_RANGE             7  /* not reachable from the R methods */
#define SVTGPU_OP_SUM               8
#define SVTGPU_OP_PROD              9
#define SVTGPU_OP_MEAN             10
#define SVTGPU_OP_CENTERED_X2_SUM  11
#define SVTGPU_OP_SUM_X_X2         12  /* not reachable from the R methods */
#define SVTGPU_OP_VAR1             13
#define SVTGPU_OP_VAR2             14
#define SVTGPU_OP_SD1              15
#define SVTGPU_OP_SD2              16

/* ---- matrix flags ---- */
#define SVTGPU_HAS_OFFS  1  /* row offsets present (row ops, products) */
#define SVTGPU_HAS_VALS  2  /* values present; absent = all leaves lacunar */

/* A flattened SVT resident in device memory ("device CSC"):
 *   leaf_ptr  int64[nleaf+1]   leaf l owns nonzeros [leaf_ptr[l], leaf_ptr[l+1])
 *   offs      int32[nnz]       0-based offsets along dim 1, ascending per leaf
 *   vals      T[nnz]           int32 or double; absent for a lacunar matrix
 * nleaf = prod(dim[-1]) (= ncol for a matrix); empty (NULL) leaves have
 * leaf_ptr[l] == leaf_ptr[l+1]. */
typedef struct svtgpu_matrix svtgpu_matrix;

/* Phase timings of the most recent operation on a matrix, milliseconds.
 * flatten_ms is filled by the caller that does the flattening. */
typedef struct svtgpu_timings {
	double h2d_ms;      /* pinned async uploads, CUDA events */
	double kernel_ms;   /* kernels of the last op, CUDA events */
	double d2h_ms;      /* result download */
	double h2d_bytes;
	double d2h_bytes;
	int    launches;    /* kernels launched by the last op */
} svtgpu_timings;

/* ---- library / device ---- */
const char *svtgpu_last_error(void);          /* thread-local message */
int svtgpu_device_count(int *count);
/* One process drives one GPU from one thread at a time: the pinned staging
 * pool, the large-block cache and the launch counter are process-wide and not
 * thread-safe (only the error string is thread-local).  Call
 * svtgpu_set_device() before the first upload; switching devices later drops
 * the staging pool (its events belong to the old device) and must not happen
 * while an upload is in flight. */
int svtgpu_set_device(int device);
int svtgpu_get_device(int *device);
int svtgpu_device_info(char *name, int name_len, int *sm_count,
		       int64_t *total_mem_bytes);
/* Device arrays are served from CUDA's stream-ordered pool and stay cached in
 * it when a matrix is freed (the stateless .Call path would otherwise pay a
 * multi-GB cudaMalloc/cudaFree per call).  This returns the cached memory to
 * the driver (e.g. from an R finalizer or .onUnload). */
int svtgpu_release_cached_memory(void);
/* Total kernels launched by this library in this process (all matrices). */
int64_t svtgpu_launch_count(void);

/* ---- device CSC lifecycle ---- */

/* Allocate device storage for nnz nonzeros in nleaf leaves of length nrow. */
int svtgpu_matrix_create(svtgpu_matrix **m, int64_t nrow, int64_t nleaf,
			 int64_t nnz, int val_type, int flags);
/* Wrap device arrays owned by the caller (no copies, not freed by free()).
 * d_offs / d_vals must be 16-byte aligned and readable for 64 elements past
 * nnz (the optional bulk-copy kernels round their reads up to 16 bytes).
 * The arrays must not change while they are wrapped: the handle caches what
 * it learns from them (max |x|, the row-tile tables, a compact copy). */
int svtgpu_matrix_wrap_device(svtgpu_matrix **m, int64_t nrow, int64_t nleaf,
			      int64_t nnz, int val_type,
			      const int64_t *d_leaf_ptr, const int32_t *d_offs,
			      const void *d_vals);
int svtgpu_matrix_free(svtgpu_matrix *m);

/* Copy the leaf offsets array (nleaf+1 entries, leaf_ptr[0] == 0). */
int svtgpu_matrix_set_leaf_ptr(svtgpu_matrix *m, const int64_t *leaf_ptr);

/* Streaming upload used by the SVT flattener.  stage() hands out a pinned
 * staging slot able to hold `count` nonzeros (blocks until the slot's previous
 * copy has drained); the caller memcpy()s leaf payloads into it; commit()
 * enqueues the async H2D copy of that slot to nonzeros [dst, dst+count).
 * Slots rotate, so filling slot k overlaps the copy of slot k-1.
 * Either pointer may come back NULL when the matrix lacks that array. */
int svtgpu_matrix_stage_capacity(svtgpu_matrix *m, int64_t *max_count);
int svtgpu_matrix_stage(svtgpu_matrix *m, int64_t count,
			int32_t **offs_slot, void **vals_slot);
int svtgpu_matrix_commit(svtgpu_matrix *m, int64_t dst, int64_t count);
/* Same as commit() for a slot the caller filled with NARROWED payloads to save
 * host->device bytes: offsets as uint16 (offs_bytes = 2; needs nrow <= 65536)
 * and/or values as int8 (vals_bytes = 1; every value in [-127, 127], NA encoded
 * as -128; for a double matrix the values must be such integers).  The slot's
 * pinned buffers are simply reinterpreted.  The library copies the narrow
 * arrays to a device staging area and widens them in HBM into the device CSC,
 * so every kernel still sees int32 offsets and int32/double values.
 * offs_bytes = 4 and vals_bytes = the native width means "not narrowed".
 * offs_bytes = SVTGPU_OFFS_U16_WRAPPED (any nrow): the slot holds the LOW 16
 * bits of every offset; the caller guarantees that inside a leaf consecutive
 * offsets differ by less than 65536 and that a leaf's first offset is below
 * 65536, the library rebuilds the high halves per leaf (offsets ascend, so
 * the high half steps up exactly where the low half steps down).  Slots must
 * be committed in ascending `dst` order (a leaf may continue from the
 * previous slot), after svtgpu_matrix_set_leaf_ptr(). */
#define SVTGPU_OFFS_U16_WRAPPED 18
int svtgpu_matrix_commit_packed(svtgpu_matrix *m, int64_t dst, int64_t count,
				int offs_bytes, int vals_bytes);
/* Wait for all uploads; records h2d_ms. */
int svtgpu_matrix_finish_upload(svtgpu_matrix *m);

/* Convenience: upload whole host CSC arrays (offs/vals may be NULL according
 * to the flags the matrix was created with). */
int svtgpu_matrix_upload(svtgpu_matrix *m, const int64_t *leaf_ptr,
			 const int32_t *offs, const void *vals);

/* Copy the device CSC back to host arrays (any of them may be NULL). */
int svtgpu_matrix_download(svtgpu_matrix *m, int64_t *leaf_ptr, int32_t *offs,
			   void *vals);
/* t(m) as a device CSC (nrow and nleaf swapped; offsets ascend inside every
 * new leaf), built on the device by a stable counting sort -- the stand-in
 * for C_transpose_2D_SVT(), src/SparseArray_aperm.c:348-423 -- and cached in
 * (owned by) m: do not free *t.  *t = NULL with SVTGPU_OK when m has no
 * offsets / no nonzeros / a strip with >= 2^32 nonzeros. */
int svtgpu_matrix_transposed(svtgpu_matrix *m, svtgpu_matrix **t);

/* N-d row statistics (row*(x, dims = d), d >= 2): fold the dimensions
 * 2..d into the rows.  The matrix (nrow x nleaf) becomes (nrow * fold) x
 * (nleaf / fold): leaf l contributes its entries to new leaf l / fold at rows
 * off + nrow * (l % fold) -- exactly the strata geometry of C_rowStats_SVT
 * (reference src/SparseArray_matrixStats.c:1097-1118).  In place; only for
 * matrices the library uploaded itself. */
int svtgpu_matrix_fold_rows(svtgpu_matrix *m, int64_t fold);

/* For a column shard: the global index of its first leaf (default 0).  Row
 * sums of double data order NA / NaN entries by global leaf index. */
int svtgpu_matrix_set_leaf_base(svtgpu_matrix *m, int64_t leaf_base);

int svtgpu_matrix_info(const svtgpu_matrix *m, int64_t *nrow, int64_t *nleaf,
		       int64_t *nnz, int *val_type, int *flags);
int svtgpu_matrix_timings(const svtgpu_matrix *m, svtgpu_timings *t);
/* Device bytes held by the matrix's compact copy of its entries (0 = none).
 * Integer and logical matrices whose values lie in [-127, 127] get int8
 * values (and uint16 row offsets when nrow <= 65536) on the second column-sum
 * or row-sum / row-moment call on the handle; those statistics then read the
 * narrow arrays.  The copy is freed with the matrix and dropped when its
 * entries are rewritten (upload, svtgpu_matrix_fold_rows). */
int svtgpu_matrix_compact_bytes(const svtgpu_matrix *m, int64_t *bytes);

/* ---- column statistics ----
 * One result per group of `group` consecutive leaves (group = 1 for a matrix
 * with dims = 1; prod(dim[2..dims]) for colStats(dims > 1) on an array); the
 * virtual vector summarised has length nrow * group.
 * out: double[nleaf/group] for every opcode except
 *      int32 for ANYNA/ANY/ALL (logical) and for MIN/MAX of LGL/INT input.
 * center: NaN/NA = "use the mean" (CENTERED_X2_SUM/VAR1/SD1 only).
 * *warn is set to 1 when the reference would warn "NAs introduced by
 * coercion of infinite values to integers". */
int svtgpu_colstats(svtgpu_matrix *m, int opcode, int narm, double center,
		    int64_t group, void *out, int *warn);
/* Same, result left in device memory, enqueued on `stream` (a cudaStream_t;
 * NULL = default stream); d_warn: device int32, OR-ed into. No sync. */
int svtgpu_colstats_dev(svtgpu_matrix *m, int opcode, int narm, double center,
			int64_t group, void *d_out, int32_t *d_warn,
			void *stream);
int svtgpu_colstats_out_is_int(int opcode, int val_type);

/* ---- row statistics ----
 * Supported opcodes: ANYNA, COUNTNAS, MIN, MAX, SUM, CENTERED_X2_SUM -- the
 * set C_rowStats_SVT() implements natively (src/SparseArray_matrixStats.c:
 * 1163-1199).  Every leaf is a stratum over the same nrow rows (dims = 1).
 * center: NULL or double[nrow] (CENTERED_X2_SUM only).
 * out: double[nrow], or int32[nrow] for ANYNA and for MIN/MAX of LGL/INT. */
int svtgpu_rowstats(svtgpu_matrix *m, int opcode, int narm,
		    const double *center, void *out, int *warn);

/* Grouped sums of an integer or double matrix (2 dimensions).
 *   svtgpu_rowsum(): out[g, j] = sum of x[i, j] over the rows i of group g
 *                    -> ngroup x nleaf, column-major;
 *   svtgpu_colsum(): out[i, g] = sum of x[i, j] over the columns j of group g
 *                    -> nrow x ngroup, column-major.
 * `group` (host): the 1-based group of every row (rowsum: nrow entries) /
 * column (colsum: nleaf entries); NA_integer_ = the last group.  `out` (host)
 * is int32 for integer input, double for double input.  Replace C_rowsum_SVT /
 * C_colsum_SVT (reference src/rowsum_methods.c:281-326, :364-409, loops
 * :44-125 and :148-255): NA / NaN skipped under narm, integer sums become
 * NA_integer_ when a partial sum leaves [-INT_MAX, INT_MAX] with *overflow = 1
 * (the reference's "NAs produced by integer overflow" warning). */
int svtgpu_rowsum(svtgpu_matrix *m, const int32_t *group, int ngroup, int narm,
		  void *out, int *overflow);
int svtgpu_colsum(svtgpu_matrix *m, const int32_t *group, int ngroup, int narm,
		  void *out, int *overflow);

/* Whole-array summarisation: the matrix (nrow x nleaf, every leaf a column of
 * the N-D array's first dimension) as ONE vector of nrow * nleaf entries.
 * Replaces C_summarize_SVT / _summarize_SVT
 * (reference src/SparseArray_summarization.c:89-142) behind sum(), mean(),
 * var(), sd(), min(), max(), range(), prod(), any(), all(), anyNA() of an
 * SVT_SparseArray (R/SparseArray-summarization.R:19-46).  `center`: NA / NaN
 * = the mean (centered_X2_sum, var1, sd1).  out[0] (and out[1] for "range")
 * receive the result as doubles; integer / logical results are exact and
 * NA_integer_ / NA (logical) comes back as NA_real_.  *warn = 1 when the
 * reference would warn (integer min / max / range of nothing).
 * svtgpu_summarize_supported(): 1 if the operation is served for val_type. */
int svtgpu_summarize_supported(int opcode, int val_type);
int svtgpu_summarize(svtgpu_matrix *m, int opcode, int narm, double center,
		     double *out, int *warn);

/* Row statistics for the opcodes C_rowStats_SVT() does NOT implement natively
 * (PROD, MEAN, ANY, ALL, VAR1, SD1 ...): what the R methods obtain as
 * colStats(aperm(x)) (.OLD_rowStats_SparseArray(), R/SparseArray-matrixStats.R
 * :122-148), here as svtgpu_colstats() on the cached device transpose.
 * center: NaN/NA = "use the mean".  out: as svtgpu_colstats(), length nrow. */
int svtgpu_rowstats_via_transpose(svtgpu_matrix *m, int opcode, int narm,
				  double center, void *out, int *warn);

/* ---- medians ----
 * base R's median() of every dense column (svtgpu_colmedians; out[nleaf],
 * host) or row (svtgpu_rowmedians; out[nrow], host, computed as column
 * medians of the device transpose, which stays cached in m) as doubles,
 * replacing the R-level colMedians() / rowMedians() methods
 * (R/SparseArray-matrixStats.R:760-813).  A column holding NA or NaN gives
 * NA_real_ unless narm; with narm they are removed and an empty remainder
 * gives NA_real_.  Even counts give the correctly rounded midpoint of the
 * two middle values; -Inf and +Inf as the middles give NaN.  Every result
 * is exact (rules: svt_med_* in csrc/svt_semantics.h).  Logical input is
 * 0 / 1, lacunar leaves hold ones.
 * svtgpu_colmedians_dev(): result left in device memory (d_out[nleaf]),
 * enqueued on `stream`; no sync.
 * svtgpu_colmedians_selected(): how many leaves (rows) the last
 * svtgpu_colmedians / svtgpu_rowmedians on m sent to exact selection, i.e.
 * whose median the stored-value counts did not decide, and how many stored
 * values the selection passes read in all (either pointer may be NULL).
 * Only the host-result calls record these counts: svtgpu_colmedians_dev()
 * does not synchronise and leaves them unchanged. */
int svtgpu_colmedians(svtgpu_matrix *m, int narm, double *out);
int svtgpu_colmedians_dev(svtgpu_matrix *m, int narm, double *d_out,
			  void *stream);
int svtgpu_rowmedians(svtgpu_matrix *m, int narm, double *out);
int svtgpu_colmedians_selected(const svtgpu_matrix *m, int64_t *n_leaves,
			       int64_t *n_reads);

/* Two-stage form for column-sharded matrices (one shard per GPU/process):
 * accumulate() reduces this shard's leaves into a per-row state of
 * svtgpu_rowstats_state_len() doubles laid out as `nslots` arrays of nrow:
 *   slots [0, n_sum)       combine across shards with SUM
 *   slots [n_sum, nslots)  combine with MIN (op MIN) or MAX (op MAX)
 * finalize() turns a (combined) state into the result, given the total number
 * of strata (leaves) over all shards.  All pointers are device pointers. */
int svtgpu_rowstats_state_layout(int opcode, int val_type, int *n_sum_slots,
				 int *n_minmax_slots);
int svtgpu_rowstats_accumulate_dev(svtgpu_matrix *m, int opcode, int narm,
				   double *d_state, void *stream);
int svtgpu_rowstats_finalize_dev(int opcode, int val_type, int narm,
				 int64_t nrow, int64_t nstrata_total,
				 const double *d_center, const double *d_state,
				 void *d_out, int32_t *d_warn, void *stream);

/* State sizes: SUM and CENTERED_X2_SUM use 4 SUM-combined slots {sum x, #NA,
 * #NaN, sum x^2} followed by 2 MAX-combined slots (last leaf with an NA / a
 * NaN in the row); MIN / MAX use 3 + 1; COUNTNAS / ANYNA 3 + 0.
 * The row-moments state is the SUM layout (6 * nrow doubles). */

/* One-pass row moments: state slots {sum x, sum x^2, #NA/NaN} -> mean and
 * variance exactly as composed by the R methods rowMeans()/rowVars() with
 * center=NULL (R/SparseArray-matrixStats.R:511-517,645-661), without the
 * reference's three passes.  out_mean/out_var: double[nrow] (either may be
 * NULL). */
int svtgpu_rowmoments(svtgpu_matrix *m, int narm, double *out_mean,
		      double *out_var);
int svtgpu_rowmoments_accumulate_dev(svtgpu_matrix *m, int narm,
				     double *d_state /* 6 * nrow */,
				     void *stream);
int svtgpu_rowmoments_finalize_dev(int val_type, int narm, int64_t nrow,
				   int64_t nstrata_total,
				   const double *d_state, double *d_mean,
				   double *d_var, void *stream);

/* ---- SVT x dense products ----
 * crossprod: ans = t(svt) %*% y, ans is nleaf x K column-major (svt_on_left)
 *            or its transpose K x nleaf (svt on the right, mirror entry
 *            point).  y is a column-major R matrix of the SVT's type (int32
 *            or double), y_nrow x y_ncol; transpose_y = use t(y).
 *            K = transpose_y ? y_nrow : y_ncol; nrow(svt) must equal the
 *            other extent.  ans is always double. */
int svtgpu_crossprod(svtgpu_matrix *m, const void *y, int y_type,
		     int64_t y_nrow, int64_t y_ncol, int transpose_y,
		     int svt_on_left, double *ans);
/* Both operands sparse: ans = t(x) %*% y, nleaf(x) x nleaf(y) column-major
 * doubles (host).  x and y must have the same nrow and type; y may be x
 * (crossprod(x)).  Replaces C_crossprod2_SVT_SVT / C_crossprod1_SVT
 * (reference src/SparseMatrix_mult.c:1037-1140). */
int svtgpu_crossprod_svt(svtgpu_matrix *x, svtgpu_matrix *y, double *ans);
/* Device form: d_y is a row-major (K contiguous) double/int32 copy of the
 * dense operand, nrow x K; d_ans is nleaf x K column-major. No sync. */
int svtgpu_crossprod_dev(svtgpu_matrix *m, const void *d_y_rowmajor,
			 int y_type, int64_t K, double *d_ans, void *stream);

/* matmul: ans = svt %*% d, svt is nrow x nleaf, d is nleaf x K column-major
 * of the SVT's type; ans is nrow x K column-major double. */
int svtgpu_matmul(svtgpu_matrix *m, const void *d, int d_type, int64_t K,
		  double *ans);
/* Device form: d_d row-major nleaf x K; d_ans row-major nrow x K partial
 * product of this shard (sum shards' results for a column-sharded svt). */
int svtgpu_matmul_dev(svtgpu_matrix *m, const void *d_d_rowmajor, int d_type,
		      int64_t K, double *d_ans_rowmajor, void *stream);

/* ---- element-wise operations that keep the implicit zeros at zero ----
 * Arith `x * v`, `v * x`, `x / v`, the Math functions and the comparisons
 * and is.* predicates below, with base R's
 * dense semantics (result types, NA / NaN, integer overflow: the rules live
 * in csrc/svt_semantics.h).  *out is a NEW matrix (owned by the caller, free
 * it with svtgpu_matrix_free()) with x's geometry; computed values equal to 0
 * (-0 included) are dropped, NA and NaN kept; svtgpu_matrix_info(*out)
 * reports the result type.  The result starts with no cached knowledge
 * (value bounds, split tables, transpose).  x is not modified.
 *   operand: host memory, operand_type SVTGPU_LGL / INT / DOUBLE, ignored for
 *            Math ops (may be NULL);
 *   margin:  0 = scalar (operand_len 1), 1 = operand[row] (operand_len =
 *            nrow), 2 = operand[leaf] (operand_len = nleaf: a column shard
 *            passes its own slice of the per-column vector);
 *   operand_on_left: `v * x` / `v / x` (the latter is refused); for the
 *            comparisons `v op x`, served as the mirrored `x op' v`.
 * An operation that would turn the implicit zeros into something else
 * (`x * Inf`, `x * NA`, `x / 0`, `v / x`, other opcodes) fails with
 * SVTGPU_ERR_ARG and R's wording before any device work.
 * Comparisons (SVTGPU_EW_GT ... NE) and the is.* predicates
 * (SVTGPU_EW_IS_*) give a logical result (val_type SVTGPU_LGL): an entry is
 * stored where the value is TRUE or NA, and FALSE is dropped.  They are
 * admitted only when `0 op v` is FALSE for every operand element (NA / NaN
 * operands are refused).  A result with no NA has no value array (flags
 * without SVTGPU_HAS_VALS: every leaf lacunar); one with an NA stores 1 and
 * NA_integer_.  The is.* predicates take no operand and never hold NA.
 * *warn: SVTGPU_EW_WARN_* bits (never set by comparisons). */
#define SVTGPU_EW_MUL       1
#define SVTGPU_EW_DIV       2
#define SVTGPU_EW_ABS      11
#define SVTGPU_EW_SIGN     12
#define SVTGPU_EW_SQRT     13
#define SVTGPU_EW_FLOOR    14
#define SVTGPU_EW_CEILING  15
#define SVTGPU_EW_TRUNC    16
#define SVTGPU_EW_LOG1P    17
#define SVTGPU_EW_EXPM1    18
#define SVTGPU_EW_GT       21  /* x >  v */
#define SVTGPU_EW_GE       22  /* x >= v */
#define SVTGPU_EW_LT       23  /* x <  v */
#define SVTGPU_EW_LE       24  /* x <= v */
#define SVTGPU_EW_EQ       25  /* x == v */
#define SVTGPU_EW_NE       26  /* x != v */
#define SVTGPU_EW_IS_NA        31  /* is.na(x): NA or NaN */
#define SVTGPU_EW_IS_NAN       32  /* is.nan(x): NaN that is not NA */
#define SVTGPU_EW_IS_INFINITE  33  /* is.infinite(x) */
#define SVTGPU_EW_WARN_INT_OVERFLOW  1  /* "NAs produced by integer overflow" */
#define SVTGPU_EW_WARN_NAN           2  /* "NaNs produced" */
int svtgpu_ewise(svtgpu_matrix *x, int op, const void *operand,
		 int operand_type, int64_t operand_len, int margin,
		 int operand_on_left, svtgpu_matrix **out, int *warn);

/* ---- synthetic data (benchmark inputs, generated in HBM) ----
 * Counter-based, so any leaf can be regenerated anywhere: with
 *   h  = mix64(seed + (cell + 1) * 0x9E3779B97F4A7C15),  cell = leaf*nrow + i
 *   h2 = mix64(h ^ 0xD1B54A32D192ED03)
 * (mix64 = the splitmix64 finaliser) cell (i, leaf) is nonzero iff
 * (h >> 32) < nz_threshold; its value is 1 + #{j : (h2 >> 32) >=
 * value_thresholds[j]} (a zero-truncated Poisson when the thresholds are its
 * CDF scaled to 2^32), replaced by NA when (uint32) h2 < na_threshold.
 * This reproduces the distribution of the reference's poissonSparseArray()
 * (R/randomSparseArray.R:62-81, src/randomSparseArray.c:91-158); the
 * identical host formula lives in sparsearray_b200/synth.py.
 * leaf0 = global index of the first leaf generated (column shards).
 * val_type 0 generates offsets only (lacunar matrix). */
int svtgpu_gen_count(int64_t nrow, int64_t nleaf, int64_t leaf0,
		     uint64_t seed, uint32_t nz_threshold,
		     int64_t *d_leaf_nnz, void *stream);
int svtgpu_gen_fill(int64_t nrow, int64_t nleaf, int64_t leaf0, uint64_t seed,
		    uint32_t nz_threshold, uint32_t na_threshold,
		    const uint32_t *value_thresholds, int n_value_thresholds,
		    int val_type, const int64_t *d_leaf_ptr, int32_t *d_offs,
		    void *d_vals, void *stream);
/* Exclusive prefix sum of n int64 counts into n+1 offsets (device). */
int svtgpu_exclusive_scan(const int64_t *d_in, int64_t n, int64_t *d_out,
			  void *stream);

#ifdef __cplusplus
}
#endif

#endif  /* SVTGPU_H */
