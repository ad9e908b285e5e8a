/* Element-wise operations on device-resident SVTs (extension entry points):
 * the Arith, Math and Compare methods of SparseArray (and is.na(),
 * is.nan(), is.infinite()) for the operations that map the implicit zero to
 * zero (or to FALSE), with base R's dense semantics (the rules live in
 * csrc/svt_semantics.h, shared with the kernels).  The result is a NEW
 * device-resident handle, usable wherever x@SVT is:
 *
 *   C_svtgpu_Arith_SVT(x_dim, x_type, x_SVT, op, y, margin, y_on_left)
 *       op "*" or "/"; y a logical / integer / double vector; margin 0 (y a
 *       scalar), 1 (length(y) == nrow: `x op y` as R recycles it) or 2
 *       (length(y) == ncol, 2-D only: `sweep(x, 2, y, op)`); y_on_left for
 *       `y * x` (and `y / x`, which is refused)
 *   C_svtgpu_Math_SVT(x_dim, x_type, x_SVT, op)
 *       op one of abs, sign, sqrt, floor, ceiling, trunc, log1p, expm1
 *   C_svtgpu_Compare_SVT(x_dim, x_type, x_SVT, op, y, margin, y_on_left)
 *       op ">", ">=", "<", "<=", "==" or "!="; y, margin and y_on_left as
 *       for Arith (`y op x` is the mirrored `x op' y`); admitted only when
 *       `0 op y` is FALSE for every element of y
 *   C_svtgpu_is_SVT(x_dim, x_type, x_SVT, fun)
 *       fun "is.na", "is.nan" or "is.infinite"
 *   C_svtgpu_Ops_SVT_SVT(x_dim, x_type, x_SVT, op, y_dim, y_type, y_SVT)
 *       `x op y` of two SVTs (or handles) of identical dimensions, op "+",
 *       "-", "*", "&", "|", ">", "<" or "!="
 *
 * All return list(handle, type); Compare, Logic and is.* give type
 * "logical".  Every refusal (an operation that would
 * turn the implicit zeros into something else, a bad operand) is raised
 * before the device is touched; the input is never modified.  The warnings
 * carry R's wording.
 */
#include "rglue_common.h"

#include <string.h>

#include "../csrc/svt_semantics.h"

static const char *get_op(SEXP op)
{
	if (!(IS_CHARACTER(op) && LENGTH(op) == 1 &&
	      STRING_ELT(op, 0) != NA_STRING))
		error("'op' must be a single string");
	return CHAR(STRING_ELT(op, 0));
}

static SEXPTYPE get_x_type(SEXP x_type, SEXP x_dim, const char *fun,
			   const char *opname)
{
	SEXPTYPE Rtype = rglue_get_and_check_Rtype(x_type, fun, "x_type");
	if (Rtype != LGLSXP && Rtype != INTSXP && Rtype != REALSXP)
		error("\"%s\": SparseArray objects of type() \"%s\" are not "
		      "supported by the SparseArray GPU path", opname,
		      type2char(Rtype));
	if (!IS_INTEGER(x_dim) || LENGTH(x_dim) < 1)
		error("'x_dim' must be an integer vector of length >= 1");
	return Rtype;
}

static void refuse(int code, const char *opname, int kind, int op,
		   int v_type, const void *v, int64_t v_len, int margin,
		   int64_t nrow, int64_t nleaf, int64_t bad)
{
	char msg[512];
	svt_ew_refusal_message(code, opname, kind, op, v_type, v, v_len,
			       margin, nrow, nleaf, bad, msg, sizeof(msg));
	error("%s", msg);
}

static SEXP run(SEXP x_dim, SEXPTYPE Rtype, SEXP x_SVT, int op,
		const void *v, int v_type, int64_t v_len, int margin,
		int on_left, const char *fun)
{
	const int *dim = INTEGER(x_dim);
	const int ndim = LENGTH(x_dim);
	rglue_input in;
	rglue_acquire(x_SVT, dim, ndim, Rtype, 1, 1, &in);
	svtgpu_matrix *out = NULL;
	int warn = 0;
	const int rc = svtgpu_ewise(in.m, op, v, v_type, v_len, margin,
				    on_left, &out, &warn);
	/* the result is a new matrix: never the cached or the handle's one */
	rglue_done(&in, fun);
	if (rc != SVTGPU_OK)
		rglue_fail(rc, "svtgpu_ewise");
	rglue_record_timings(out, 0.0);
	int out_type = 0;
	svtgpu_matrix_info(out, NULL, NULL, NULL, &out_type, NULL);
	SEXP ans = PROTECT(NEW_LIST(2));
	SET_VECTOR_ELT(ans, 0, rglue_make_handle(out));
	SET_VECTOR_ELT(ans, 1, mkString(out_type == SVTGPU_DOUBLE ? "double"
					: out_type == SVTGPU_LGL ? "logical"
								  : "integer"));
	if (warn & SVTGPU_EW_WARN_INT_OVERFLOW)
		warning("NAs produced by integer overflow");
	if (warn & SVTGPU_EW_WARN_NAN)
		warning("NaNs produced");
	UNPROTECT(1);
	return ans;
}

static int64_t nleaf_of(SEXP x_dim)
{
	int64_t n = 1;
	for (int along = 1; along < LENGTH(x_dim); along++)
		n *= INTEGER(x_dim)[along];
	return n;
}

/* x op y for Arith (kind SVT_EW_KIND_ARITH) and Compare */
static SEXP binary(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op, SEXP y,
		   SEXP margin, SEXP y_on_left, int kind, const char *fun)
{
	const char *opname = get_op(op);
	const SEXPTYPE Rtype = get_x_type(x_type, x_dim, fun, opname);
	if (!(IS_INTEGER(margin) && LENGTH(margin) == 1))
		error("'margin' must be a single integer");
	if (!(IS_LOGICAL(y_on_left) && LENGTH(y_on_left) == 1 &&
	      LOGICAL(y_on_left)[0] != NA_LOGICAL))
		error("'y_on_left' must be TRUE or FALSE");
	const int code_op = kind == SVT_EW_KIND_COMPARE
		? svt_ew_compare_opcode(opname) : svt_ew_arith_opcode(opname);
	const int mg = INTEGER(margin)[0];
	const int on_left = LOGICAL(y_on_left)[0] != 0;
	const SEXPTYPE ytype = TYPEOF(y);
	const int64_t ylen = XLENGTH(y);
	const void *yv = (ytype == LGLSXP || ytype == INTSXP || ytype == REALSXP)
			 ? DATAPTR(y) : NULL;
	const int64_t nrow = INTEGER(x_dim)[0], nleaf = nleaf_of(x_dim);
	int64_t bad = -1;
	const int code = code_op == 0 ? SVT_EW_BAD_OPCODE :
		svt_ew_check(code_op, (int) Rtype, (int) ytype, ylen, mg, on_left,
			     LENGTH(x_dim), nrow, nleaf, yv, &bad);
	if (code != SVT_EW_OK)
		refuse(code, opname, kind, code_op, (int) ytype, yv, ylen, mg,
		       nrow, nleaf, bad);
	return run(x_dim, Rtype, x_SVT, code_op, yv, (int) ytype, ylen, mg,
		   on_left, fun);
}

/* --- .Call ENTRY POINT (extension) --- */
SEXP C_svtgpu_Arith_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op, SEXP y,
			SEXP margin, SEXP y_on_left)
{
	return binary(x_dim, x_type, x_SVT, op, y, margin, y_on_left,
		      SVT_EW_KIND_ARITH, "C_svtgpu_Arith_SVT");
}

/* --- .Call ENTRY POINT (extension) --- */
SEXP C_svtgpu_Compare_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op,
			  SEXP y, SEXP margin, SEXP y_on_left)
{
	return binary(x_dim, x_type, x_SVT, op, y, margin, y_on_left,
		      SVT_EW_KIND_COMPARE, "C_svtgpu_Compare_SVT");
}

/* --- .Call ENTRY POINT (extension) --- */
SEXP C_svtgpu_Math_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op)
{
	const char *opname = get_op(op);
	const SEXPTYPE Rtype = get_x_type(x_type, x_dim, "C_svtgpu_Math_SVT",
					  opname);
	const int code_op = svt_ew_math_opcode(opname);
	if (code_op == 0)
		refuse(SVT_EW_BAD_OPCODE, opname, SVT_EW_KIND_MATH, 0, 0, NULL, 0,
		       0, 0, 0, -1);
	return run(x_dim, Rtype, x_SVT, code_op, NULL, 0, 0, 0, 0,
		   "C_svtgpu_Math_SVT");
}

/* --- .Call ENTRY POINT (extension) --- */
SEXP C_svtgpu_is_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP fun)
{
	const char *name = get_op(fun);
	const SEXPTYPE Rtype = get_x_type(x_type, x_dim, "C_svtgpu_is_SVT",
					  name);
	const int code_op = svt_ew_is_opcode(name);
	if (code_op == 0)
		refuse(SVT_EW_BAD_OPCODE, name, SVT_EW_KIND_IS, 0, 0, NULL, 0, 0,
		       0, 0, -1);
	return run(x_dim, Rtype, x_SVT, code_op, NULL, 0, 0, 0, 0,
		   "C_svtgpu_is_SVT");
}

/* --- .Call ENTRY POINT (extension) ---
 * `x op y` between two SVT_SparseArray objects (the Arith, Logic and Compare
 * methods with two SparseArray operands).  Order matters, as in
 * C_crossprod2_SVT_SVT: every R error is raised while no per-call device
 * matrix is held; y is indexed (or taken as a handle) before x is acquired
 * and uploaded outside the device cache afterwards, so acquiring y can never
 * free the x just taken from the cache; the same SVT on both sides is
 * uploaded once. */
SEXP C_svtgpu_Ops_SVT_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op,
			  SEXP y_dim, SEXP y_type, SEXP y_SVT)
{
	const char *opname = get_op(op);
	const int code_op = svt_ew2_opcode(opname);
	if (code_op == 0) {
		char msg[512];
		svt_ew2_refusal_message(opname, msg, sizeof(msg));
		error("%s", msg);
	}
	const char *fun = "C_svtgpu_Ops_SVT_SVT";
	const SEXPTYPE x_Rtype = get_x_type(x_type, x_dim, fun, opname);
	const SEXPTYPE y_Rtype = get_x_type(y_type, y_dim, fun, opname);
	const int ndim = LENGTH(x_dim);
	if (LENGTH(y_dim) != ndim ||
	    memcmp(INTEGER(x_dim), INTEGER(y_dim), sizeof(int) * ndim) != 0)
		error("non-conformable arrays");
	const int *dim = INTEGER(x_dim);
	rglue_input inx, iny;
	const int same = y_SVT == x_SVT && y_Rtype == x_Rtype;
	const int y_is_handle = TYPEOF(y_SVT) == EXTPTRSXP;
	svt_leaf_index iy;
	if (!same && y_is_handle)
		rglue_acquire(y_SVT, dim, ndim, y_Rtype, 1, 1, &iny);
	else if (!same)
		svt_index_leaves(y_SVT, dim, ndim, y_Rtype, &iy);
	rglue_acquire(x_SVT, dim, ndim, x_Rtype, 1, 1, &inx);
	if (same) {
		iny = inx;
	} else if (!y_is_handle) {
		memset(&iny, 0, sizeof(iny));
		const int rcy = svt_upload_leaves(&iy, y_Rtype, 1, 1, &iny.m,
						  &iny.flatten_ms);
		iny.t_ready = rglue_now_ms();
		if (rcy != SVTGPU_OK) {
			rglue_done(&inx, fun);
			rglue_fail(rcy, "svt_upload_leaves");
		}
	}
	svtgpu_matrix *out = NULL;
	int warn = 0;
	const int rc = svtgpu_ewise2(inx.m, iny.m, code_op, &out, &warn);
	/* the result is a new matrix: never the cached or a handle's one */
	if (!same)
		rglue_done(&iny, "C_svtgpu_Ops_SVT_SVT (y)");
	rglue_done(&inx, fun);
	if (rc != SVTGPU_OK)
		rglue_fail(rc, "svtgpu_ewise2");
	rglue_record_timings(out, 0.0);
	int out_type = 0;
	svtgpu_matrix_info(out, NULL, NULL, NULL, &out_type, NULL);
	SEXP ans = PROTECT(NEW_LIST(2));
	SET_VECTOR_ELT(ans, 0, rglue_make_handle(out));
	SET_VECTOR_ELT(ans, 1, mkString(out_type == SVTGPU_DOUBLE ? "double"
					: out_type == SVTGPU_LGL ? "logical"
								  : "integer"));
	if (warn & SVTGPU_EW_WARN_INT_OVERFLOW)
		warning("NAs produced by integer overflow");
	UNPROTECT(1);
	return ans;
}
