/* Helpers shared by the .Call entry points of the GPU glue. */
#ifndef RGLUE_COMMON_H
#define RGLUE_COMMON_H

#include <Rdefines.h>
#include <stdint.h>

#include "../../include/svtgpu.h"
#include "svt_flatten.h"

/* "logical"/"integer"/"double"/... -> SEXPTYPE, error like
 * _get_and_check_Rtype_from_Rstring() (src/argcheck_utils.c:11-19). */
SEXPTYPE rglue_get_and_check_Rtype(SEXP type, const char *fun,
				   const char *argname);
/* _get_and_check_na_background(), src/argcheck_utils.c:21-31 */
int rglue_get_and_check_na_background(SEXP na_background, const char *fun,
				      const char *argname);
/* _get_summarize_opcode(), src/Rvector_summarization.c:19-78 */
int rglue_get_summarize_opcode(SEXP op, SEXPTYPE Rtype);

/* Raise the R error for a failed svtgpu call (never returns). The caller has
 * already released every device/pinned resource it owned. */
void rglue_fail(int rc, const char *fun) __attribute__((noreturn));

/* wall clock in ms; phase trace to stderr when SVTGPU_TRACE is set */
double rglue_now_ms(void);
void rglue_trace(const char *fun, double t_index, double t_upload,
		 double t_op, double t_free);

/* last operation's phase timings, readable from R via C_svtgpu_last_timings */
void rglue_record_timings(const svtgpu_matrix *m, double flatten_ms);

/* The device matrix behind an 'x_SVT' argument.  Every entry point accepts,
 * in place of the SVT (a list tree or NULL), the external pointer made by
 * C_svtgpu_resident_SVT(): the matrix then already lives in HBM and nothing
 * is flattened or uploaded (SURVEY section 8f item 2: upload once, run many
 * statistics).  Otherwise the tree is indexed, flattened and uploaded for
 * this call only.  rglue_acquire() raises the R error itself on failure
 * (nothing is left allocated); rglue_done() records the timings, releases a
 * per-call matrix and prints the phase trace. */
typedef struct rglue_input {
	svtgpu_matrix *m;
	int resident;   /* nothing was uploaded for this call */
	int shared;     /* owned by a handle or by the cache: not freed here */
	double index_ms, upload_ms, flatten_ms, t_ready;
} rglue_input;
void rglue_acquire(SEXP x_SVT, const int *dim, int ndim, SEXPTYPE Rtype,
		   int want_offs, int want_vals, rglue_input *in);
/* may_share = 0: the caller is going to modify the device matrix (row
 * folding), so it must be this call's own and never come from / go into the
 * device cache (see rglue_common.c) */
/* no leaf stores values: countNAs / anyNA are all zero (see the definition) */
int rglue_svt_stores_no_values(SEXP x_SVT, const int *dim, int ndim);

void rglue_acquire2(SEXP x_SVT, const int *dim, int ndim, SEXPTYPE Rtype,
		    int want_offs, int want_vals, int may_share,
		    rglue_input *in);
void rglue_done(rglue_input *in, const char *fun);

SEXP C_colStats_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		    SEXP x_na_background, SEXP op, SEXP na_rm, SEXP center,
		    SEXP dims);
SEXP C_rowStats_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		    SEXP x_na_background, SEXP op, SEXP na_rm, SEXP center,
		    SEXP dims);
SEXP C_crossprod2_SVT_mat(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP y,
			  SEXP transpose_y, SEXP ans_type, SEXP ans_dimnames);
SEXP C_crossprod2_mat_SVT(SEXP x, SEXP y_dim, SEXP y_type, SEXP y_SVT,
			  SEXP transpose_x, SEXP ans_type, SEXP ans_dimnames);
SEXP C_crossprod2_SVT_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP y_dim,
			  SEXP y_type, SEXP y_SVT, SEXP ans_type,
			  SEXP ans_dimnames);
SEXP C_crossprod1_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP ans_type,
		      SEXP ans_dimnames);
SEXP C_summarize_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT,
		     SEXP x_na_background, SEXP op, SEXP na_rm, SEXP center);
SEXP C_rowsum_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP group,
		  SEXP ngroup, SEXP na_rm);
SEXP C_colsum_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP group,
		  SEXP ngroup, SEXP na_rm);
/* extensions (not in the reference): see INTEGRATION.md */
SEXP C_matmul_SVT_mat(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP y,
		      SEXP ans_dimnames);
SEXP C_rowMoments_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		      SEXP na_rm);
SEXP C_rowStatsT_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		     SEXP x_na_background, SEXP op, SEXP na_rm, SEXP center,
		     SEXP dims);
SEXP C_colMedians_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		      SEXP na_rm);
SEXP C_rowMedians_SVT(SEXP x_dim, SEXP x_dimnames, SEXP x_type, SEXP x_SVT,
		      SEXP na_rm);
SEXP C_svtgpu_last_timings(void);
SEXP C_svtgpu_resident_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT);
SEXP C_svtgpu_release(SEXP handle);
SEXP rglue_make_handle(svtgpu_matrix *m);
SEXP C_svtgpu_from_CSC(SEXP dim, SEXP indptr, SEXP data, SEXP indices,
		       SEXP indices_are_1based);
SEXP C_svtgpu_to_CSC(SEXP handle, SEXP as_ngCMatrix);
SEXP C_svtgpu_Arith_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op, SEXP y,
			SEXP margin, SEXP y_on_left);
SEXP C_svtgpu_Math_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op);
SEXP C_svtgpu_Compare_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op,
			  SEXP y, SEXP margin, SEXP y_on_left);
SEXP C_svtgpu_is_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP fun);
SEXP C_svtgpu_Ops_SVT_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP op,
			  SEXP y_dim, SEXP y_type, SEXP y_SVT);
SEXP C_svtgpu_subset_SVT(SEXP x_dim, SEXP x_type, SEXP x_SVT, SEXP Nindex);
SEXP C_svtgpu_set_cache(SEXP on);
SEXP C_svtgpu_cache_stats(void);
SEXP C_get_num_procs(void);
SEXP C_get_max_threads(void);
SEXP C_set_max_threads(SEXP nthread);

#endif  /* RGLUE_COMMON_H */
