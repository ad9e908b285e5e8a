/* Registration of the .Call entry points served by the GPU glue, plus the
 * thread-control routines SparseArray.Call() invokes around every call
 * (R/thread-control.R:87-92; src/thread_control.c:33-64).  Names and arities
 * are those of src/R_init_SparseArray.c:41-43,121-122,131-132 (and C_summarize_SVT,
 * the first widening beyond the four hot-path entry points). */
#include <R_ext/Rdynload.h>

#include "rglue_common.h"

#ifdef _OPENMP
#undef match
#include <omp.h>
#endif

SEXP C_get_num_procs(void)
{
#ifdef _OPENMP
	return ScalarInteger(omp_get_num_procs());
#else
	return ScalarInteger(0);
#endif
}

SEXP C_get_max_threads(void)
{
#ifdef _OPENMP
	return ScalarInteger(omp_get_max_threads());
#else
	return ScalarInteger(0);
#endif
}

/* The GPU kernels ignore nthread; it sizes the host-side flatten team. */
SEXP C_set_max_threads(SEXP nthread)
{
#ifdef _OPENMP
	int prev = omp_get_max_threads();
	omp_set_num_threads(INTEGER(nthread)[0]);
	return ScalarInteger(prev);
#else
	return ScalarInteger(0);
#endif
}

#define CALLMETHOD_DEF(fun, numArgs) {#fun, (DL_FUNC) &fun, numArgs}

static const R_CallMethodDef callMethods[] = {
	CALLMETHOD_DEF(C_get_num_procs, 0),
	CALLMETHOD_DEF(C_get_max_threads, 0),
	CALLMETHOD_DEF(C_set_max_threads, 1),
	CALLMETHOD_DEF(C_colStats_SVT, 9),
	CALLMETHOD_DEF(C_rowStats_SVT, 9),
	CALLMETHOD_DEF(C_crossprod2_SVT_mat, 7),
	CALLMETHOD_DEF(C_crossprod2_mat_SVT, 7),
	CALLMETHOD_DEF(C_crossprod2_SVT_SVT, 8),
	CALLMETHOD_DEF(C_crossprod1_SVT, 5),
	CALLMETHOD_DEF(C_summarize_SVT, 7),
	CALLMETHOD_DEF(C_rowsum_SVT, 6),
	CALLMETHOD_DEF(C_colsum_SVT, 6),
	/* extensions */
	CALLMETHOD_DEF(C_matmul_SVT_mat, 5),
	CALLMETHOD_DEF(C_rowMoments_SVT, 5),
	CALLMETHOD_DEF(C_rowStatsT_SVT, 9),
	CALLMETHOD_DEF(C_colMedians_SVT, 5),
	CALLMETHOD_DEF(C_rowMedians_SVT, 5),
	CALLMETHOD_DEF(C_svtgpu_last_timings, 0),
	CALLMETHOD_DEF(C_svtgpu_resident_SVT, 3),
	CALLMETHOD_DEF(C_svtgpu_release, 1),
	CALLMETHOD_DEF(C_svtgpu_from_CSC, 5),
	CALLMETHOD_DEF(C_svtgpu_to_CSC, 2),
	CALLMETHOD_DEF(C_svtgpu_Arith_SVT, 7),
	CALLMETHOD_DEF(C_svtgpu_Math_SVT, 4),
	CALLMETHOD_DEF(C_svtgpu_Compare_SVT, 7),
	CALLMETHOD_DEF(C_svtgpu_is_SVT, 4),
	CALLMETHOD_DEF(C_svtgpu_set_cache, 1),
	CALLMETHOD_DEF(C_svtgpu_cache_stats, 0),
	{NULL, NULL, 0}
};

void R_init_SparseArray(DllInfo *info)
{
	R_registerRoutines(info, NULL, callMethods, NULL, NULL);
	R_useDynamicSymbols(info, 0);
}
