/* .Call entry points C_colStats_SVT / C_rowStats_SVT served by the GPU path.
 *
 * Same signatures, argument checks, result types/shapes, dimnames propagation
 * and warnings as the reference's entry points
 * (src/SparseArray_matrixStats.c:234-284 and :1121-1205); the tree walk and
 * the per-leaf loops behind them (REC_colStats_SVT / REC_rowStats_SVT) are
 * replaced by: flatten the SVT -> upload -> one CUDA launch sequence ->
 * download into the R result.  No computation happens on the host.
 *
 * Not served (clean error instead of a wrong answer): NaArray input
 * (na_background = TRUE), types other than logical/integer/double,
 * and the opcodes no R method reaches
 * ("range", "sum_X_X2", "var2", "sd2").
 */
#include "rglue_common.h"

#include "../csrc/svt_semantics.h"

#include <string.h>

static const char *NA_COERCION_WARNING =
	"NAs introduced by coercion of infinite values to integers";

static int check_dims(SEXP dims, int min, int max)
{
	if (!IS_INTEGER(dims) || LENGTH(dims) != 1)
		error("'dims' must be a single integer");
	int d = INTEGER(dims)[0];
	if (d == NA_INTEGER || d < min || d > max)
		error("'dims' must be >= %d and <= %d", min, max);
	return d;
}

static void check_gpu_input(SEXPTYPE Rtype, int na_background,
			    const char *what)
{
	if (na_background)
		error("%s: NaArray objects (na_background=TRUE) are not "
		      "supported by the SparseArray GPU path", what);
	if (Rtype != LGLSXP && Rtype != INTSXP && Rtype != REALSXP)
		error("%s: SparseArray objects of type() \"%s\" are not "
		      "supported by the SparseArray GPU path", what,
		      type2char(Rtype));
}

/* allocate the result: a vector when it has <= 1 dimension, else an array
   (alloc_ans(), src/SparseArray_matrixStats.c:108-125) */
static SEXP alloc_ans(SEXPTYPE Rtype, const int *ans_dim, int ans_ndim)
{
	if (ans_ndim <= 1)
		return allocVector(Rtype, ans_ndim == 1 ? ans_dim[0] : 1);
	SEXP dim = PROTECT(NEW_INTEGER(ans_ndim));
	memcpy(INTEGER(dim), ans_dim, sizeof(int) * ans_ndim);
	SEXP ans = allocArray(Rtype, dim);
	UNPROTECT(1);
	return ans;
}

/* names / dimnames of the result = the kept dimnames [first, first + n)
   (propagate_{col,row}Stats_dimnames(), :127-172) */
static void propagate_dimnames(SEXP ans, SEXP x_dimnames, int first, int n)
{
	if (x_dimnames == R_NilValue || n == 0)
		return;
	if (n == 1) {
		SEXP names = VECTOR_ELT(x_dimnames, first);
		if (names != R_NilValue)
			SET_NAMES(ans, names);
		return;
	}
	int any_retained = 0;
	for (int along = 0; along < n; along++)
		if (VECTOR_ELT(x_dimnames, first + along) != R_NilValue)
			any_retained = 1;
	if (!any_retained)
		return;
	SEXP ans_dimnames = PROTECT(NEW_LIST(n));
	for (int along = 0; along < n; along++)
		SET_VECTOR_ELT(ans_dimnames, along,
			       VECTOR_ELT(x_dimnames, first + along));
	SET_DIMNAMES(ans, ans_dimnames);
	UNPROTECT(1);
}

/* --- .Call ENTRY POINT --- */
SEXP C_colStats_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type,
		    SEXP x_SVT, SEXP x_na_background,
		    SEXP op, SEXP na_rm, SEXP center, SEXP dims)
{
	SEXPTYPE x_Rtype = rglue_get_and_check_Rtype(x_type,
					"C_colStats_SVT", "x_type");
	int x_has_NAbg = rglue_get_and_check_na_background(x_na_background,
					"C_colStats_SVT", "x_na_background");
	int opcode = rglue_get_summarize_opcode(op, x_Rtype);

	if (!(IS_LOGICAL(na_rm) && LENGTH(na_rm) == 1))
		error("'na.rm' must be TRUE or FALSE");
	int narm = LOGICAL(na_rm)[0];

	if (!IS_NUMERIC(center) || LENGTH(center) != 1)
		error("SparseArray internal error in "
		      "C_colStats_SVT():\n"
		      "    'center' must be a single number");

	const int *dim = INTEGER(x_dim);
	int ndim = LENGTH(x_dim);
	int d = check_dims(dims, 1, ndim);
	check_gpu_input(x_Rtype, x_has_NAbg, "col*()");
	if (!svt_col_op_supported(opcode, (int) x_Rtype))
		error("col*(): operation \"%s\" is not supported by the "
		      "SparseArray GPU path", CHAR(STRING_ELT(op, 0)));

	SEXPTYPE ans_Rtype =
		(opcode == SVTGPU_OP_ANYNA || opcode == SVTGPU_OP_ANY ||
		 opcode == SVTGPU_OP_ALL) ? LGLSXP :
		svt_col_out_is_int(opcode, (int) x_Rtype) ? INTSXP : REALSXP;
	int ans_ndim = ndim - d;
	SEXP ans = PROTECT(alloc_ans(ans_Rtype, dim + d, ans_ndim));
	propagate_dimnames(ans, x_dimnames, d, ans_ndim);

	/* geometry: each result summarises 'group' consecutive leaves */
	int64_t group = 1, nout = 1;
	for (int along = 1; along < d; along++)
		group *= dim[along];
	for (int along = d; along < ndim; along++)
		nout *= dim[along];
	if (nout == 0) {
		UNPROTECT(1);
		return ans;
	}
	int warn = 0;
	if (group == 0) {
		/* every result summarises an empty vector: no data to move */
		SvtColPartial empty;
		svt_col_partial_init(&empty);
		SvtScalar r = svt_col_finalize(opcode, x_Rtype == REALSXP,
					narm, 0, REAL(center)[0], &empty);
		for (int64_t i = 0; i < nout; i++) {
			if (ans_Rtype == REALSXP) REAL(ans)[i] = r.d;
			else                      INTEGER(ans)[i] = r.i;
		}
		warn = r.warn;
	} else {
		/* column statistics never read the row offsets */
		rglue_input in;
		rglue_acquire(x_SVT, dim, ndim, x_Rtype, 0, 1, &in);
		int rc = svtgpu_colstats(in.m, opcode, narm, REAL(center)[0],
					 group, DATAPTR(ans), &warn);
		rglue_done(&in, "C_colStats_SVT");
		if (rc != SVTGPU_OK)
			rglue_fail(rc, "svtgpu_colstats");
	}
	if (warn)
		warning("%s", NA_COERCION_WARNING);
	UNPROTECT(1);
	return ans;
}

/* --- .Call ENTRY POINT --- */
SEXP C_rowStats_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type,
		    SEXP x_SVT, SEXP x_na_background,
		    SEXP op, SEXP na_rm, SEXP center, SEXP dims)
{
	SEXPTYPE x_Rtype = rglue_get_and_check_Rtype(x_type,
					"C_rowStats_SVT", "x_type");
	int x_has_NAbg = rglue_get_and_check_na_background(x_na_background,
					"C_colStats_SVT", "x_na_background");
	int opcode = rglue_get_summarize_opcode(op, x_Rtype);

	if (!(IS_LOGICAL(na_rm) && LENGTH(na_rm) == 1))
		error("'na.rm' must be TRUE or FALSE");
	int narm = LOGICAL(na_rm)[0];

	const int *dim = INTEGER(x_dim);
	int ndim = LENGTH(x_dim);
	int ans_ndim = check_dims(dims, 1, ndim - 1);

	/* check_rowStats_center(), :1079-1095 */
	const double *center_p = NULL;
	if (center != R_NilValue) {
		if (!IS_NUMERIC(center))
			error("SparseArray internal error in "
			      "check_rowStats_center():\n"
			      "    'center' must be NULL or a numeric array");
		R_xlen_t ans_len = 1;
		for (int along = 0; along < ans_ndim; along++)
			ans_len *= dim[along];
		if (LENGTH(center) != ans_len)
			error("SparseArray internal error in "
			      "check_rowStats_center():\n"
			      "    unexpected 'center' length");
		center_p = REAL(center);
	}

	if (!svt_row_op_supported(opcode))
		error("SparseArray internal error in C_rowStats_SVT():\n"
		      "    operation not supported");
	check_gpu_input(x_Rtype, x_has_NAbg, "row*()");
	/* dims >= 2: the strata are head(dim, dims)-shaped; fold dimensions
	   2..dims into the rows of the flattened matrix (:1097-1118) */
	int64_t fold = 1;
	for (int along = 1; along < ans_ndim; along++)
		fold *= dim[along];
	if (ans_ndim != 1 && TYPEOF(x_SVT) == EXTPTRSXP)
		error("row*(): 'dims' >= 2 is not supported on a "
		      "device-resident handle");

	SEXPTYPE ans_Rtype = opcode == SVTGPU_OP_ANYNA ? LGLSXP :
		((opcode == SVTGPU_OP_MIN || opcode == SVTGPU_OP_MAX) &&
		 x_Rtype != REALSXP) ? INTSXP : REALSXP;
	SEXP ans = PROTECT(alloc_ans(ans_Rtype, dim, ans_ndim));
	propagate_dimnames(ans, x_dimnames, 0, ans_ndim);
	if (LENGTH(ans) == 0) {
		UNPROTECT(1);
		return ans;
	}

	if ((opcode == SVTGPU_OP_COUNTNAS || opcode == SVTGPU_OP_ANYNA) &&
	    rglue_svt_stores_no_values(x_SVT, dim, ndim)) {
		/* lacunar leaves hold ones: no NA anywhere, nothing to upload */
		memset(DATAPTR(ans), 0, (size_t) XLENGTH(ans) *
		       (ans_Rtype == REALSXP ? sizeof(double) : sizeof(int)));
		UNPROTECT(1);
		return ans;
	}
	rglue_input in;
	rglue_acquire2(x_SVT, dim, ndim, x_Rtype, 1, 1, fold == 1, &in);
	int warn = 0;
	int rc = fold > 1 ? svtgpu_matrix_fold_rows(in.m, fold) : SVTGPU_OK;
	if (rc == SVTGPU_OK)
		rc = svtgpu_rowstats(in.m, opcode, narm, center_p, DATAPTR(ans),
				     &warn);
	rglue_done(&in, "C_rowStats_SVT");
	if (rc != SVTGPU_OK)
		rglue_fail(rc, "svtgpu_rowstats");
	if (warn)
		warning("%s", NA_COERCION_WARNING);
	UNPROTECT(1);
	return ans;
}

/* --- .Call ENTRY POINT (extension) ---
 * Row statistics for the operations C_rowStats_SVT does not implement
 * ("prod", "mean", "any", "all", "var1", "sd1", ...), which the R methods
 * compute as colStats(aperm(x)) (.OLD_rowStats_SparseArray(),
 * R/SparseArray-matrixStats.R:122-148): same arguments as C_colStats_SVT,
 * 2-D input, one result per row; the transpose happens on the device. */
SEXP C_rowStatsT_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type,
		     SEXP x_SVT, SEXP x_na_background,
		     SEXP op, SEXP na_rm, SEXP center, SEXP dims)
{
	SEXPTYPE x_Rtype = rglue_get_and_check_Rtype(x_type,
					"C_rowStatsT_SVT", "x_type");
	int x_has_NAbg = rglue_get_and_check_na_background(x_na_background,
					"C_rowStatsT_SVT", "x_na_background");
	int opcode = rglue_get_summarize_opcode(op, x_Rtype);
	if (!(IS_LOGICAL(na_rm) && LENGTH(na_rm) == 1))
		error("'na.rm' must be TRUE or FALSE");
	int narm = LOGICAL(na_rm)[0];
	if (!IS_NUMERIC(center) || LENGTH(center) != 1)
		error("SparseArray internal error in "
		      "C_rowStatsT_SVT():\n"
		      "    'center' must be a single number");
	const int *dim = INTEGER(x_dim);
	int ndim = LENGTH(x_dim);
	if (ndim != 2 || check_dims(dims, 1, 1) != 1)
		error("row*(): only 2-dimensional input with dims=1 is "
		      "supported by the SparseArray GPU path for this "
		      "operation");
	check_gpu_input(x_Rtype, x_has_NAbg, "row*()");
	if (!svt_col_op_supported(opcode, (int) x_Rtype))
		error("row*(): operation \"%s\" is not supported by the "
		      "SparseArray GPU path", CHAR(STRING_ELT(op, 0)));
	SEXPTYPE ans_Rtype =
		(opcode == SVTGPU_OP_ANYNA || opcode == SVTGPU_OP_ANY ||
		 opcode == SVTGPU_OP_ALL) ? LGLSXP :
		svt_col_out_is_int(opcode, (int) x_Rtype) ? INTSXP : REALSXP;
	SEXP ans = PROTECT(alloc_ans(ans_Rtype, dim, 1));
	propagate_dimnames(ans, x_dimnames, 0, 1);
	if (dim[0] == 0) {
		UNPROTECT(1);
		return ans;
	}
	rglue_input in;
	rglue_acquire(x_SVT, dim, ndim, x_Rtype, 1, 1, &in);
	int warn = 0;
	int rc = svtgpu_rowstats_via_transpose(in.m, opcode, narm,
					       REAL(center)[0], DATAPTR(ans),
					       &warn);
	rglue_done(&in, "C_rowStatsT_SVT");
	if (rc != SVTGPU_OK)
		rglue_fail(rc, "svtgpu_rowstats_via_transpose");
	if (warn)
		warning("%s", NA_COERCION_WARNING);
	UNPROTECT(1);
	return ans;
}

/* --- .Call ENTRY POINT (extension) ---
 * One pass over the matrix for what rowMeans()/rowVars(center=NULL) obtain
 * with up to three C_rowStats_SVT passes (R/SparseArray-matrixStats.R:
 * 511-517,645-661).  Returns list(mean=, var=) of length-nrow doubles. */
SEXP C_rowMoments_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		      SEXP na_rm)
{
	SEXPTYPE x_Rtype = rglue_get_and_check_Rtype(x_type,
					"C_rowMoments_SVT", "x_type");
	if (!(IS_LOGICAL(na_rm) && LENGTH(na_rm) == 1))
		error("'na.rm' must be TRUE or FALSE");
	int narm = LOGICAL(na_rm)[0];
	check_gpu_input(x_Rtype, 0, "rowMoments()");
	const int *dim = INTEGER(x_dim);
	int ndim = LENGTH(x_dim);
	if (ndim < 2)
		error("rowMoments(): input must have at least 2 dimensions");

	SEXP ans = PROTECT(NEW_LIST(2));
	SEXP mean = SET_VECTOR_ELT(ans, 0, NEW_NUMERIC(dim[0]));
	SEXP var = SET_VECTOR_ELT(ans, 1, NEW_NUMERIC(dim[0]));
	propagate_dimnames(mean, x_dimnames, 0, 1);
	propagate_dimnames(var, x_dimnames, 0, 1);
	SEXP names = PROTECT(NEW_CHARACTER(2));
	SET_STRING_ELT(names, 0, mkChar("mean"));
	SET_STRING_ELT(names, 1, mkChar("var"));
	SET_NAMES(ans, names);
	UNPROTECT(1);
	if (dim[0] == 0) {
		UNPROTECT(1);
		return ans;
	}
	rglue_input in;
	rglue_acquire(x_SVT, dim, ndim, x_Rtype, 1, 1, &in);
	int rc = svtgpu_rowmoments(in.m, narm, REAL(mean), REAL(var));
	rglue_done(&in, "C_rowMoments_SVT");
	if (rc != SVTGPU_OK)
		rglue_fail(rc, "svtgpu_rowmoments");
	UNPROTECT(1);
	return ans;
}

/* colMedians() / rowMedians() of a matrix: one double per column / row
   (svtgpu_colmedians / svtgpu_rowmedians) */
static SEXP medians_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
			SEXP na_rm, int rows, const char *fun)
{
	SEXPTYPE x_Rtype = rglue_get_and_check_Rtype(x_type, fun, "x_type");
	if (!(IS_LOGICAL(na_rm) && LENGTH(na_rm) == 1))
		error("'na.rm' must be TRUE or FALSE");
	int narm = LOGICAL(na_rm)[0];
	const char *what = rows ? "rowMedians()" : "colMedians()";
	check_gpu_input(x_Rtype, 0, what);
	const int *dim = INTEGER(x_dim);
	int ndim = LENGTH(x_dim);
	if (ndim != 2)
		error("%s: only matrices (2-dimensional objects) are supported; "
		      "'x' has %d dimensions", what, ndim);
	const int nout = dim[rows ? 0 : 1], nin = dim[rows ? 1 : 0];
	SEXP ans = PROTECT(NEW_NUMERIC(nout));
	propagate_dimnames(ans, x_dimnames, rows ? 0 : 1, 1);
	if (nout == 0) {
		UNPROTECT(1);
		return ans;
	}
	if (nin == 0) {
		/* every median is over an empty vector */
		SvtMedPlan p = svt_med_plan(0, 0, 0, 0, narm);
		for (int i = 0; i < nout; i++)
			REAL(ans)[i] = p.kind == SVT_MED_NA ? NA_REAL : 0.0;
		UNPROTECT(1);
		return ans;
	}
	rglue_input in;
	rglue_acquire(x_SVT, dim, ndim, x_Rtype, rows, 1, &in);
	int rc = rows ? svtgpu_rowmedians(in.m, narm, REAL(ans))
		      : svtgpu_colmedians(in.m, narm, REAL(ans));
	rglue_done(&in, fun);
	if (rc != SVTGPU_OK)
		rglue_fail(rc, rows ? "svtgpu_rowmedians" : "svtgpu_colmedians");
	UNPROTECT(1);
	return ans;
}

/* --- .Call ENTRY POINT (extension) ---
 * colMedians() of a 2-D SVT, which the reference computes in R
 * (R/SparseArray-matrixStats.R:760-813): base R's median() of every dense
 * column as a double vector, named by the column names. */
SEXP C_colMedians_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		      SEXP na_rm)
{
	return medians_SVT(x_dim, x_dimnames, x_type, x_SVT, na_rm, 0,
			   "C_colMedians_SVT");
}

/* --- .Call ENTRY POINT (extension) ---
 * rowMedians() of a 2-D SVT: the column medians of the device transpose,
 * which stays cached in a resident handle. */
SEXP C_rowMedians_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		      SEXP na_rm)
{
	return medians_SVT(x_dim, x_dimnames, x_type, x_SVT, na_rm, 1,
			   "C_rowMedians_SVT");
}
