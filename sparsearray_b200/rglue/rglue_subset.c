/* Subsetting of device-resident SVTs (extension entry point):
 *
 *   C_svtgpu_subset_SVT(x_dim, x_type, x_SVT, Nindex)
 *
 * x[i, j, ..., drop = FALSE] for an SVT_SparseArray (or a resident handle)
 * after R's `[` method has normalised the subscripts: Nindex is a list with
 * one element per dimension, each NULL (all of that dimension, in order) or
 * an integer vector of 1-based positions in any order, duplicates allowed.
 * Logical, negative and character subscripts are turned into such vectors in
 * R (S4Arrays / S4Vectors), as before this entry point existed.  The result
 * has dimension lengths(Nindex) (dim(x)[k] for a NULL element) and x's type;
 * it is returned as list(handle, type) like C_svtgpu_Arith_SVT, a NEW
 * device-resident handle that never is the cached matrix.  Every refusal is
 * raised before any device work.
 */
#include "rglue_common.h"

#include <string.h>

static const char *fun = "C_svtgpu_subset_SVT";

/* check subscript `along` (0-based) of Nindex; its length, or -1 for NULL */
static int64_t check_subscript(SEXP Nindex, int along, int extent)
{
	SEXP s = VECTOR_ELT(Nindex, along);
	if (s == R_NilValue)
		return -1;
	if (!IS_INTEGER(s))
		error("%s: subscript %d of 'Nindex' must be NULL or an integer "
		      "vector", fun, along + 1);
	const int *v = INTEGER(s);
	const int64_t n = XLENGTH(s);
	for (int64_t k = 0; k < n; k++)
		if (v[k] == NA_INTEGER)
			error("subscript contains NAs");
	for (int64_t k = 0; k < n; k++)
		if (v[k] < 1 || v[k] > extent)
			error("subscript contains out-of-bounds indices");
	return n;
}

/* --- .Call ENTRY POINT (extension) --- */
SEXP C_svtgpu_subset_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP Nindex)
{
	const SEXPTYPE Rtype = rglue_get_and_check_Rtype(x_type, fun, "x_type");
	if (Rtype != LGLSXP && Rtype != INTSXP && Rtype != REALSXP)
		error("%s: SparseArray objects of type() \"%s\" are not supported "
		      "by the SparseArray GPU path", fun, type2char(Rtype));
	if (!IS_INTEGER(x_dim) || LENGTH(x_dim) < 1)
		error("'x_dim' must be an integer vector of length >= 1");
	const int *dim = INTEGER(x_dim);
	const int ndim = LENGTH(x_dim);
	if (!IS_LIST(Nindex) || LENGTH(Nindex) != ndim)
		error("%s: 'Nindex' must be a list with one element per dimension "
		      "of 'x' (%d)", fun, ndim);
	int64_t len[ndim];
	for (int along = 0; along < ndim; along++)
		len[along] = check_subscript(Nindex, along, dim[along]);

	/* rows: 0-based int32; NULL = every row */
	int32_t *rows = NULL;
	if (len[0] >= 0) {
		const int *v = INTEGER(VECTOR_ELT(Nindex, 0));
		rows = (int32_t *) R_alloc((size_t) (len[0] > 0 ? len[0] : 1),
					   sizeof(int32_t));
		for (int64_t k = 0; k < len[0]; k++)
			rows[k] = v[k] - 1;
	}
	/* leaves: the Cartesian product of dims 2..N, column-major (the
	   subscript of dimension 2 varies fastest); NULL when all are NULL */
	int64_t *leaves = NULL, n_leaves = 1;
	int any = 0;
	for (int along = 1; along < ndim; along++) {
		const int64_t n = len[along] >= 0 ? len[along] : dim[along];
		any |= len[along] >= 0;
		if (n > 0 && n_leaves > INT32_MAX / n)
			error("%s: the result would have more than 2^31 - 2 "
			      "columns (leaves), which the GPU path does not "
			      "support", fun);
		n_leaves *= n;
	}
	if (any) {
		leaves = (int64_t *) R_alloc((size_t) (n_leaves > 0 ? n_leaves : 1),
					     sizeof(int64_t));
		int64_t stride = 1, span = 1;
		for (int64_t k = 0; k < n_leaves; k++)
			leaves[k] = 0;
		for (int along = 1; along < ndim; along++) {
			const int64_t n = len[along] >= 0 ? len[along] : dim[along];
			const int *v = len[along] >= 0
				? INTEGER(VECTOR_ELT(Nindex, along)) : NULL;
			/* leaf k of the result takes index (k / span) % n
			   along this dimension */
			for (int64_t k = 0; k < n_leaves; k++) {
				const int64_t i = (k / span) % n;
				leaves[k] += stride * (v != NULL ? v[i] - 1 : i);
			}
			span *= n;
			stride *= dim[along];
		}
	}

	rglue_input in;
	rglue_acquire(x_SVT, dim, ndim, Rtype, 1, 1, &in);
	svtgpu_matrix *out = NULL;
	const int rc = svtgpu_subset(in.m, rows, len[0], leaves, n_leaves, &out);
	/* the result is a new matrix: never the cached or the handle's one */
	rglue_done(&in, fun);
	if (rc != SVTGPU_OK)
		rglue_fail(rc, "svtgpu_subset");
	rglue_record_timings(out, 0.0);
	SEXP ans = PROTECT(NEW_LIST(2));
	SET_VECTOR_ELT(ans, 0, rglue_make_handle(out));
	SET_VECTOR_ELT(ans, 1, mkString(Rtype == REALSXP ? "double"
					: Rtype == LGLSXP ? "logical"
							  : "integer"));
	UNPROTECT(1);
	return ans;
}
