/* svt_semantics.h -- result composition rules of the reference, shared by the
 * CUDA kernels (device) and by tests/semantics_host.cpp (host build of the
 * very same functions, so the NA/NaN/zero-background logic can be checked on
 * a machine without a GPU).  No loops over data here (except the check of an
 * element-wise operand, done once on the host): the kernels reduce a leaf (or
 * a row) to a small "partial" and these functions turn a partial into the
 * value the reference would have produced.
 *
 * Reference: src/Rvector_summarization.c (per-type loops :177-734, lacunar
 * :742-825, post-processing :1078-1177), src/SparseArray_summarization.c
 * :70-109 (two-pass variance), src/SparseArray_matrixStats.c (:303-430 row
 * update rules, :914-961 row min/max post-processing, :1044-1072 centered
 * X2 sums), src/SparseVec_dotprod.c:28-138 and src/SparseMatrix_mult.c
 * :193-239 (dot-product NA rules).
 */
#ifndef SVT_SEMANTICS_H
#define SVT_SEMANTICS_H

#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#ifndef __cplusplus
#include <stdbool.h>
#endif

#include "../../include/svtgpu.h"

#ifdef __CUDACC__
#define SVT_HD __host__ __device__ __forceinline__
#else
#define SVT_HD static inline
#endif

#define SVT_NA_INT INT32_MIN

SVT_HD uint64_t svt_d2u(double x)
{
#ifdef __CUDA_ARCH__
	return (uint64_t) __double_as_longlong(x);
#else
	uint64_t u;
	memcpy(&u, &x, sizeof(u));
	return u;
#endif
}

SVT_HD double svt_u2d(uint64_t u)
{
#ifdef __CUDA_ARCH__
	return __longlong_as_double((long long) u);
#else
	double x;
	memcpy(&x, &u, sizeof(x));
	return x;
#endif
}

/* R's NA_real_ (arithmetic.c: low word 1954) and the canonical quiet NaN. */
SVT_HD double svt_na_real(void) { return svt_u2d(0x7FF00000000007A2ULL); }
SVT_HD double svt_nan(void)     { return svt_u2d(0x7FF8000000000000ULL); }
SVT_HD double svt_posinf(void)  { return svt_u2d(0x7FF0000000000000ULL); }
SVT_HD double svt_neginf(void)  { return svt_u2d(0xFFF0000000000000ULL); }

SVT_HD bool svt_isnan(double x)
{
	return (svt_d2u(x) & 0x7FFFFFFFFFFFFFFFULL) > 0x7FF0000000000000ULL;
}

/* R_IsNA(): a NaN whose low word is 1954. */
SVT_HD bool svt_is_na_real(double x)
{
	return svt_isnan(x) && (uint32_t) svt_d2u(x) == 1954u;
}

SVT_HD bool svt_isfinite(double x)
{
	return (svt_d2u(x) & 0x7FF0000000000000ULL) != 0x7FF0000000000000ULL;
}

/* Never let an accidental payload decide between NA and NaN on output. */
SVT_HD double svt_clean_nan(double x)
{
	return svt_isnan(x) ? svt_nan() : x;
}

/* ------------------------------------------------------------------------
 * Column statistics
 */

/* What a kernel knows about one summarised segment (a leaf, or `group`
 * consecutive leaves) once its stored values have been reduced. */
typedef struct SvtColPartial {
	int64_t nz;      /* stored values (in_nzcount) */
	int64_t n_na;    /* int: == NA_INTEGER; double: R_IsNA() */
	int64_t n_nan;   /* double only: NaN that is not NA */
	int64_t n_zero;  /* stored values equal to 0 (ANY/ALL only) */
	double sum;      /* sum of regular (non-NA, non-NaN) values */
	double sum2;     /* sum of (x - center)^2 over regular values */
	double prod;     /* product of regular values */
	double vmin;     /* min / max over regular values, +Inf / -Inf if none */
	double vmax;
} SvtColPartial;

SVT_HD void svt_col_partial_init(SvtColPartial *p)
{
	p->nz = p->n_na = p->n_nan = p->n_zero = 0;
	p->sum = p->sum2 = 0.0;
	p->prod = 1.0;
	p->vmin = svt_posinf();
	p->vmax = svt_neginf();
}

/* Partial of a lacunar segment: nz implicit ones
 * (summarize_ones(), src/Rvector_summarization.c:742-825). */
SVT_HD void svt_col_partial_ones(SvtColPartial *p, int64_t nz, double center)
{
	svt_col_partial_init(p);
	p->nz = nz;
	if (nz == 0)
		return;
	p->sum = (double) nz;
	double delta = 1.0 - center;
	p->sum2 = delta * delta * (double) nz;
	p->vmin = p->vmax = 1.0;
}

SVT_HD int svt_col_out_is_int(int opcode, int val_type)
{
	if (opcode == SVTGPU_OP_ANYNA || opcode == SVTGPU_OP_ANY ||
	    opcode == SVTGPU_OP_ALL)
		return 1;
	if ((opcode == SVTGPU_OP_MIN || opcode == SVTGPU_OP_MAX) &&
	    val_type != SVTGPU_DOUBLE)
		return 1;
	return 0;
}

SVT_HD int svt_col_op_supported(int opcode, int val_type)
{
	switch (opcode) {
	    case SVTGPU_OP_ANYNA: case SVTGPU_OP_COUNTNAS:
	    case SVTGPU_OP_MIN: case SVTGPU_OP_MAX:
	    case SVTGPU_OP_SUM: case SVTGPU_OP_PROD: case SVTGPU_OP_MEAN:
	    case SVTGPU_OP_CENTERED_X2_SUM:
	    case SVTGPU_OP_VAR1: case SVTGPU_OP_SD1:
		return 1;
	    case SVTGPU_OP_ANY: case SVTGPU_OP_ALL:
		return val_type != SVTGPU_DOUBLE;
	}
	return 0;
}

SVT_HD int svt_col_op_needs_center(int opcode)
{
	return opcode == SVTGPU_OP_CENTERED_X2_SUM ||
	       opcode == SVTGPU_OP_VAR1 || opcode == SVTGPU_OP_SD1;
}

typedef struct SvtScalar {
	double d;   /* result when the output type is double */
	int32_t i;  /* result when the output type is int32/logical */
	int warn;
} SvtScalar;

/* mean of the segment as computed by replace_SummarizeOp_center_with_mean()
 * (src/SparseArray_summarization.c:70-87): MEAN_OPCODE with the same na.rm. */
SVT_HD double svt_col_mean(int is_double, int narm, int64_t in_length,
			   const SvtColPartial *p)
{
	if (!narm && p->n_na > 0)
		return svt_na_real();   /* breaking value, returned as is */
	double s = (!narm && p->n_nan > 0) ? svt_nan() : p->sum;
	int64_t nacount = narm ? p->n_na + p->n_nan : 0;
	(void) is_double;
	return s / (double) (in_length - nacount);
}

/* Turn the partial of a segment of virtual length `in_length` into the value
 * _summarize_SVT() + _postprocess_SummarizeResult() produce (na_background
 * FALSE).  For CENTERED_X2_SUM/VAR1/SD1 `center` must already be the mean when
 * the caller's center was NA/NaN, and p->sum2 must be relative to it. */
SVT_HD SvtScalar svt_col_finalize(int opcode, int is_double, int narm,
				  int64_t in_length, double center,
				  const SvtColPartial *p)
{
	SvtScalar r;
	r.d = 0.0; r.i = 0; r.warn = 0;
	const int64_t zerocount = in_length - p->nz;
	const int64_t n_nanish = p->n_na + p->n_nan;
	const int64_t n_reg = p->nz - n_nanish;

	if (opcode == SVTGPU_OP_ANYNA) {
		r.i = n_nanish > 0;
		return r;
	}
	if (opcode == SVTGPU_OP_COUNTNAS) {
		r.d = (double) n_nanish;
		return r;
	}
	if (opcode == SVTGPU_OP_ANY) {
		/* any_ints(), :261-286: a nonzero non-NA value wins, then NA. */
		if (n_reg - p->n_zero > 0)
			r.i = 1;
		else if (!narm && p->n_na > 0)
			r.i = SVT_NA_INT;
		else
			r.i = 0;
		return r;
	}
	if (opcode == SVTGPU_OP_ALL) {
		/* all_ints(), :291-316, then one background zero, :1100-1106 */
		if (p->n_zero > 0 || zerocount > 0)
			r.i = 0;
		else if (!narm && p->n_na > 0)
			r.i = SVT_NA_INT;
		else
			r.i = 1;
		return r;
	}

	/* Every remaining op bails out with NA on the first NA when !na.rm
	   (OUTBUF_IS_SET_WITH_BREAKING_VALUE: post-processing is skipped). */
	const int broke = !narm && p->n_na > 0;
	/* double input, !na.rm: a NaN sticks but does not break (:548-561). */
	const int stuck_nan = !narm && p->n_nan > 0;
	const int64_t nacount = narm ? n_nanish : 0;
	const int64_t effective_len = in_length - nacount;

	switch (opcode) {
	    case SVTGPU_OP_MIN: case SVTGPU_OP_MAX: {
		const int is_min = opcode == SVTGPU_OP_MIN;
		if (!is_double) {
			if (broke) {
				r.i = SVT_NA_INT;
				return r;
			}
			int have = n_reg > 0;
			double v = is_min ? p->vmin : p->vmax;
			if (zerocount > 0) {
				if (!have || (is_min ? 0.0 < v : 0.0 > v))
					v = 0.0;
				have = 1;
			}
			if (!have) {
				/* empty or all-NA with na.rm: :1108-1127 */
				r.i = SVT_NA_INT;
				r.warn = 1;
				return r;
			}
			r.i = (int32_t) v;
			return r;
		}
		if (broke) {
			r.d = svt_na_real();
			return r;
		}
		if (stuck_nan) {
			r.d = svt_nan();  /* the background zero cannot undo it */
			return r;
		}
		double v = is_min ? p->vmin : p->vmax;
		if (zerocount > 0 && (is_min ? 0.0 < v : 0.0 > v))
			v = 0.0;
		r.d = v;
		return r;
	    }
	    case SVTGPU_OP_SUM: case SVTGPU_OP_MEAN: {
		if (broke) {
			r.d = svt_na_real();
			return r;
		}
		double v = stuck_nan ? svt_nan() : p->sum;
		if (opcode == SVTGPU_OP_MEAN)
			v = v / (double) effective_len;
		r.d = svt_clean_nan(v);
		return r;
	    }
	    case SVTGPU_OP_PROD: {
		if (broke) {
			r.d = svt_na_real();
			return r;
		}
		double v = stuck_nan ? svt_nan() : p->prod;
		if (zerocount > 0)
			v = v * 0.0;  /* Inf * 0 -> NaN, as prod_*(&zero, 1) */
		r.d = svt_clean_nan(v);
		return r;
	    }
	    case SVTGPU_OP_CENTERED_X2_SUM:
	    case SVTGPU_OP_VAR1: case SVTGPU_OP_SD1: {
		if (broke) {
			r.d = svt_na_real();
			return r;
		}
		double v = stuck_nan ? svt_nan() : p->sum2;
		v += center * center * (double) zerocount;      /* :1145-1147 */
		if (opcode == SVTGPU_OP_CENTERED_X2_SUM) {
			r.d = svt_clean_nan(v);
			return r;
		}
		if (effective_len <= 1) {
			r.d = svt_na_real();
			return r;
		}
		v /= ((double) effective_len - 1.0);
		if (opcode == SVTGPU_OP_SD1)
			v = sqrt(v);
		r.d = svt_clean_nan(v);
		return r;
	    }
	}
	r.d = svt_nan();
	return r;
}

/* ------------------------------------------------------------------------
 * Row statistics: per-row state slots (arrays of nrow doubles)
 */

/* slot indices */
#define SVT_ROW_SLOT_SUM    0  /* sum of regular values */
#define SVT_ROW_SLOT_NA     1  /* # NA */
#define SVT_ROW_SLOT_NAN    2  /* # NaN (double input) */
#define SVT_ROW_SLOT_SUM2   3  /* sum of squares of regular values */
/* MIN/MAX use: 0 = coverage (# leaves with a stored value in the row),
   1 = #NA, 2 = #NaN, 3 = running min or max over regular values. */
#define SVT_ROW_SLOT_CVG    0
#define SVT_ROW_SLOT_EXT    3
/* SUM / CENTERED_X2_SUM also carry, MAX-combined, the (global) index of the
   LAST leaf that put an NA / a NaN into the row (-Inf = none, or not tracked
   by the kernel that built the state).  The reference adds the entries of a
   row in leaf order with a plain `*out += x`
   (src/SparseArray_matrixStats.c:409-430); when both operands of that
   addition are NaNs the hardware keeps the payload of the first operand, and
   the reference as compiled (gcc, x86-64: `addsd x, [out]`) has x first --
   so of several NA / NaN entries in one row the last one decides whether the
   row sum is NA_real_ or NaN.  (+Inf and -Inf in one row make a fresh NaN,
   which any NA / NaN entry, earlier or later, overrides the same way.) */
#define SVT_ROW_SLOT_LAST_NA     4
#define SVT_ROW_SLOT_LAST_NAN    5

SVT_HD int svt_row_op_supported(int opcode)
{
	return opcode == SVTGPU_OP_ANYNA || opcode == SVTGPU_OP_COUNTNAS ||
	       opcode == SVTGPU_OP_MIN || opcode == SVTGPU_OP_MAX ||
	       opcode == SVTGPU_OP_SUM ||
	       opcode == SVTGPU_OP_CENTERED_X2_SUM;
}

/* number of SUM-combined and MIN/MAX-combined slots of an op's state */
SVT_HD void svt_row_state_layout(int opcode, int *n_sum, int *n_ext)
{
	switch (opcode) {
	    case SVTGPU_OP_ANYNA: case SVTGPU_OP_COUNTNAS:
		*n_sum = 3; *n_ext = 0; return;
	    case SVTGPU_OP_SUM:
	    case SVTGPU_OP_CENTERED_X2_SUM:
		*n_sum = 4; *n_ext = 2; return;
	    case SVTGPU_OP_MIN: case SVTGPU_OP_MAX:
		*n_sum = 3; *n_ext = 1; return;
	}
	*n_sum = 0; *n_ext = 0;
}

/* Which NaN a row sum ends up with under the reference's sequential
 * `*out += x` (na.rm = FALSE): 0 = none (the sum of the regular values
 * stands), 1 = NA_real_, 2 = NaN: the kind of the last NA / NaN entry in leaf
 * order.  When the positions were not tracked (-Inf in the slot although the
 * count is positive) NA wins. */
SVT_HD int svt_row_sum_kind(const double *s, int64_t stride)
{
	const double ninf = svt_neginf();
	const double n_na = s[SVT_ROW_SLOT_NA * stride];
	const double n_nan = s[SVT_ROW_SLOT_NAN * stride];
	if (n_na <= 0.0 && n_nan <= 0.0)
		return 0;
	const double l_na = s[SVT_ROW_SLOT_LAST_NA * stride];
	const double l_nan = s[SVT_ROW_SLOT_LAST_NAN * stride];
	if ((n_na > 0.0 && !(l_na > ninf)) || (n_nan > 0.0 && !(l_nan > ninf)))
		return n_na > 0.0 ? 1 : 2;
	if (n_na <= 0.0)
		return 2;
	if (n_nan <= 0.0)
		return 1;
	return l_na > l_nan ? 1 : 2;
}

/* One row's result from its combined state.  `s` points at slot 0 of the row,
 * consecutive slots are `stride` doubles apart. */
SVT_HD SvtScalar svt_row_finalize(int opcode, int is_double, int narm,
				  int64_t nstrata, int have_center,
				  double center, const double *s,
				  int64_t stride)
{
	SvtScalar r;
	r.d = 0.0; r.i = 0; r.warn = 0;
	const double n_na = s[SVT_ROW_SLOT_NA * stride];
	const double n_nan = s[SVT_ROW_SLOT_NAN * stride];

	switch (opcode) {
	    case SVTGPU_OP_ANYNA:
		r.i = (n_na + n_nan) > 0.0;
		return r;
	    case SVTGPU_OP_COUNTNAS:
		r.d = n_na + n_nan;
		return r;
	    case SVTGPU_OP_SUM: {
		/* update_out_with_{int,double}_sum(), :409-430: a plain
		   running `out += x`, so NA/NaN survive unless na.rm. */
		const int kind = narm ? 0 : svt_row_sum_kind(s, stride);
		if (kind == 1)
			r.d = svt_na_real();
		else if (kind == 2)
			r.d = svt_nan();
		else
			r.d = svt_clean_nan(s[SVT_ROW_SLOT_SUM * stride]);
		return r;
	    }
	    case SVTGPU_OP_CENTERED_X2_SUM: {
		/* SVT_rowCenteredX2Sum(), :1044-1072, with the per-nonzero
		   term x*(x - 2c) (:693) summed as sum(x^2) - 2c*sum(x). */
		/* the running value starts at c^2 * ncol (:1052-1058) */
		if (have_center && svt_isnan(center)) {
			r.d = svt_is_na_real(center) ? svt_na_real() : svt_nan();
			return r;
		}
		const int kind = narm ? 0 : svt_row_sum_kind(s, stride);
		if (kind == 1) {
			r.d = svt_na_real();
			return r;
		}
		if (kind == 2) {
			r.d = svt_nan();
			return r;
		}
		double c = have_center ? center : 0.0;
		double sx = s[SVT_ROW_SLOT_SUM * stride];
		double sx2 = s[SVT_ROW_SLOT_SUM2 * stride];
		double v;
		if (!have_center) {
			v = sx2;        /* c == 0: no 0 * Inf from the cross term */
		} else if (sx2 == svt_posinf() && svt_isfinite(c)) {
			/* an infinite x contributes x * (x - 2c) = +Inf whatever
			   its sign; Inf - Inf in the expanded form must not
			   turn that into NaN */
			v = sx2;
		} else {
			v = c * c * (double) nstrata + (sx2 - 2.0 * c * sx);
		}
		if (narm)
			v -= (n_na + n_nan) * (c * c);   /* :665-669,681-684 */
		r.d = svt_clean_nan(v);
		return r;
	    }
	    case SVTGPU_OP_MIN: case SVTGPU_OP_MAX: {
		const int is_min = opcode == SVTGPU_OP_MIN;
		const double cvg = s[SVT_ROW_SLOT_CVG * stride];
		const double n_reg = cvg - n_na - n_nan;
		double v = s[SVT_ROW_SLOT_EXT * stride];
		int have = n_reg > 0.0;
		if (nstrata == 0) {             /* SVT_rowMinsMaxs(), :973-986 */
			if (is_double) {
				r.d = is_min ? svt_posinf() : svt_neginf();
			} else {
				r.i = SVT_NA_INT;
				r.warn = 1;
			}
			return r;
		}
		if (!narm && n_na > 0.0) {
			if (is_double) r.d = svt_na_real();
			else           r.i = SVT_NA_INT;
			return r;
		}
		if (!narm && n_nan > 0.0) {
			r.d = svt_nan();
			return r;
		}
		if (cvg < (double) nstrata) {   /* fold one background zero */
			if (!have || (is_min ? 0.0 < v : 0.0 > v))
				v = 0.0;
			have = 1;
		}
		if (!have) {
			/* na.rm and nothing but NAs: :931-933, :955-956 */
			if (is_double) {
				r.d = is_min ? svt_posinf() : svt_neginf();
			} else {
				r.i = SVT_NA_INT;
				r.warn = 1;
			}
			return r;
		}
		if (is_double) r.d = v;
		else           r.i = (int32_t) v;
		return r;
	    }
	}
	r.d = svt_nan();
	return r;
}

/* rowMeans()/rowVars(center=NULL) as composed in R
 * (R/SparseArray-matrixStats.R:300-310,511-517,645-661) from one state
 * {sum x, #NA, #NaN, sum x^2}. */
SVT_HD void svt_row_moments(int narm, int64_t nstrata, const double *s,
			    int64_t stride, double *mean, double *var)
{
	const double n_na = s[SVT_ROW_SLOT_NA * stride];
	const double n_nan = s[SVT_ROW_SLOT_NAN * stride];
	const double sx = s[SVT_ROW_SLOT_SUM * stride];
	const double sx2 = s[SVT_ROW_SLOT_SUM2 * stride];
	const double nvals = (double) nstrata - (narm ? n_na + n_nan : 0.0);
	double sums;
	const int kind = narm ? 0 : svt_row_sum_kind(s, stride);
	if (kind == 1)      sums = svt_na_real();
	else if (kind == 2) sums = svt_nan();
	else                sums = sx;
	const int is_na = svt_is_na_real(sums);
	double c = sums / nvals;
	*mean = is_na ? svt_na_real() : svt_clean_nan(c);
	double x2 = c * c * (double) nstrata + (sx2 - 2.0 * c * sx);
	if (narm)
		x2 -= (n_na + n_nan) * (c * c);
	double v = x2 / (nvals - 1.0);
	*var = is_na ? svt_na_real() : svt_clean_nan(v);
}

/* ------------------------------------------------------------------------
 * SVT x dense dot products
 */

/* What is known about one column of the dense operand. */
typedef struct SvtDenseColInfo {
	int32_t n_nonfinite;  /* double: !R_FINITE; int: == NA_INTEGER;
				 SVT_COL_FICTIVE_ZERO: the column belongs to a
				 fictive all-zero operand (a NULL SVT) */
	int32_t n_na;         /* double: R_IsNA;    int: == NA_INTEGER */
} SvtDenseColInfo;
#define SVT_COL_FICTIVE_ZERO (-1)

/* Result of dot(leaf, y[,k]) given the plain gathered sum `s`
 * (sum of v * y[off] over the leaf's stored values), what is known about the
 * leaf's NA / NaN entries, and how many of its nonzeros hit non-finite entries
 * of the column.
 *   leaf_flag bit 0: the leaf holds an NA
 *             bit 1: the first NA-or-NaN entry of the leaf is a NaN
 * int: _dotprod_intSV_noNA_ints()/_dotprod_intSV_ints()/_dotprod_ints_zero();
 * double: _dotprod_doubleSV_finite_doubles()/_dotprod_doubleSV_doubles()/
 * _dotprod_doubles_zero() (src/SparseVec_dotprod.c:28-138), selected per
 * dense column as in src/SparseMatrix_mult.c:193-239.  The finite-column loop
 * is `ans += v * y` on a register accumulator (:36-41): of several NaNs the
 * first one's payload survives, so NA_real_ comes out only when the NA is the
 * leaf's first NA/NaN entry; the dense walk (:52-63) returns NA_real_ as soon
 * as it meets any NA. */
#define SVT_LEAF_HAS_NA     1
#define SVT_LEAF_NAN_FIRST  2

SVT_HD double svt_dot_finalize(int is_double, double s, int leaf_flag,
			       int64_t hits_nonfinite, SvtDenseColInfo ci)
{
	const int leaf_has_na = leaf_flag & SVT_LEAF_HAS_NA;
	if (!is_double) {
		if (ci.n_na > 0 || leaf_has_na)
			return svt_na_real();
		return s;
	}
	if (ci.n_nonfinite == SVT_COL_FICTIVE_ZERO) {
		/* the other operand is a NULL SVT: _dotprod_doubleSV_zero() /
		   _dotprod_doubles_zero() (src/SparseVec_dotprod.c:116-147)
		   return NA as soon as ANY entry is NA, wherever it stands;
		   otherwise the sum of v * 0 (NaN when the leaf holds a NaN or
		   an infinity) */
		if (leaf_has_na)
			return svt_na_real();
		return svt_clean_nan(s);
	}
	if (ci.n_nonfinite == 0) {
		/* fast path: NA/NaN leaf values propagate arithmetically */
		if (leaf_has_na && !(leaf_flag & SVT_LEAF_NAN_FIRST))
			return svt_na_real();
		return svt_clean_nan(s);
	}
	/* dense walk over all rows: NA wins, then any 0 * non-finite is NaN */
	if (ci.n_na > 0 || leaf_has_na)
		return svt_na_real();
	if (hits_nonfinite < (int64_t) ci.n_nonfinite)
		return svt_nan();
	return svt_clean_nan(s);
}

/* ------------------------------------------------------------------------
 * Element-wise operations that map the implicit zero to zero (svtgpu_ewise)
 *
 * Base R's dense semantics (src/main/arithmetic.c: R_integer_times(),
 * real_binary(), math1(), do_abs()) restated for one stored value.  The glue
 * calls the checks on the host before any device work; the kernels call the
 * value rules; the result type is decided here once for both.
 */

/* refusal codes of svt_ew_check() */
#define SVT_EW_OK           0
#define SVT_EW_BAD_OPCODE   1  /* not an operation that keeps zeros at zero */
#define SVT_EW_LEFT_DIV     2  /* v / x */
#define SVT_EW_BAD_X_TYPE   3
#define SVT_EW_BAD_V_TYPE   4
#define SVT_EW_BAD_MARGIN   5
#define SVT_EW_BAD_LENGTH   6
#define SVT_EW_BAD_VALUE    7  /* *bad = 0-based index into the operand */

/* bits OR-ed by the value rules (the first two are svtgpu_ewise's *warn) */
#define SVT_EW_DROPPED      4  /* a computed value compares equal to 0 */
#define SVT_EW_NA_KEPT      8  /* a comparison kept an NA entry */

/* what svt_ew_cmp() makes of one stored value */
#define SVT_CMP_DROP        0  /* FALSE: the entry leaves the result */
#define SVT_CMP_TRUE        1
#define SVT_CMP_NA          2

/* what kind of name the caller was given (svt_ew_refusal_message()) */
#define SVT_EW_KIND_ARITH   0
#define SVT_EW_KIND_MATH    1
#define SVT_EW_KIND_COMPARE 2
#define SVT_EW_KIND_IS      3

SVT_HD int svt_ew_is_arith(int op)
{
	return op == SVTGPU_EW_MUL || op == SVTGPU_EW_DIV;
}

SVT_HD int svt_ew_is_math(int op)
{
	return op >= SVTGPU_EW_ABS && op <= SVTGPU_EW_EXPM1;
}

SVT_HD int svt_ew_is_compare(int op)
{
	return op >= SVTGPU_EW_GT && op <= SVTGPU_EW_NE;
}

/* is.na / is.nan / is.infinite */
SVT_HD int svt_ew_is_pred(int op)
{
	return op >= SVTGPU_EW_IS_NA && op <= SVTGPU_EW_IS_INFINITE;
}

/* operations that take no operand */
SVT_HD int svt_ew_is_unary(int op)
{
	return svt_ew_is_math(op) || svt_ew_is_pred(op);
}

/* `v op x` is `x op' v`: the order comparisons swap, == and != stay */
SVT_HD int svt_ew_mirror(int op)
{
	switch (op) {
	    case SVTGPU_EW_GT: return SVTGPU_EW_LT;
	    case SVTGPU_EW_GE: return SVTGPU_EW_LE;
	    case SVTGPU_EW_LT: return SVTGPU_EW_GT;
	    case SVTGPU_EW_LE: return SVTGPU_EW_GE;
	}
	return op;
}

SVT_HD int svt_ew_streq(const char *a, const char *b)
{
	while (*a != '\0' && *a == *b) {
		a++;
		b++;
	}
	return *a == *b;
}

/* "*" / "/" -> opcode; any other name (the rest of R's Arith group) -> 0 */
SVT_HD int svt_ew_arith_opcode(const char *name)
{
	if (svt_ew_streq(name, "*")) return SVTGPU_EW_MUL;
	if (svt_ew_streq(name, "/")) return SVTGPU_EW_DIV;
	return 0;
}

/* the Math-group functions with f(0) == 0 -> opcode; others -> 0 */
SVT_HD const char *svt_ew_opname(int op)
{
	switch (op) {
	    case SVTGPU_EW_MUL:     return "*";
	    case SVTGPU_EW_DIV:     return "/";
	    case SVTGPU_EW_ABS:     return "abs";
	    case SVTGPU_EW_SIGN:    return "sign";
	    case SVTGPU_EW_SQRT:    return "sqrt";
	    case SVTGPU_EW_FLOOR:   return "floor";
	    case SVTGPU_EW_CEILING: return "ceiling";
	    case SVTGPU_EW_TRUNC:   return "trunc";
	    case SVTGPU_EW_LOG1P:   return "log1p";
	    case SVTGPU_EW_EXPM1:   return "expm1";
	    case SVTGPU_EW_GT:      return ">";
	    case SVTGPU_EW_GE:      return ">=";
	    case SVTGPU_EW_LT:      return "<";
	    case SVTGPU_EW_LE:      return "<=";
	    case SVTGPU_EW_EQ:      return "==";
	    case SVTGPU_EW_NE:      return "!=";
	    case SVTGPU_EW_IS_NA:       return "is.na";
	    case SVTGPU_EW_IS_NAN:      return "is.nan";
	    case SVTGPU_EW_IS_INFINITE: return "is.infinite";
	}
	return "?";
}

SVT_HD int svt_ew_math_opcode(const char *name)
{
	for (int op = SVTGPU_EW_ABS; op <= SVTGPU_EW_EXPM1; op++)
		if (svt_ew_streq(name, svt_ew_opname(op)))
			return op;
	return 0;
}

/* R's Compare group (">", ">=", "<", "<=", "==", "!=") -> opcode; else 0 */
SVT_HD int svt_ew_compare_opcode(const char *name)
{
	for (int op = SVTGPU_EW_GT; op <= SVTGPU_EW_NE; op++)
		if (svt_ew_streq(name, svt_ew_opname(op)))
			return op;
	return 0;
}

/* "is.na", "is.nan", "is.infinite" -> opcode; any other name (is.finite
   would make the zeros TRUE) -> 0 */
SVT_HD int svt_ew_is_opcode(const char *name)
{
	for (int op = SVTGPU_EW_IS_NA; op <= SVTGPU_EW_IS_INFINITE; op++)
		if (svt_ew_streq(name, svt_ew_opname(op)))
			return op;
	return 0;
}

SVT_HD int svt_ew_type_ok(int t)
{
	return t == SVTGPU_LGL || t == SVTGPU_INT || t == SVTGPU_DOUBLE;
}

/* Type of the result (arithmetic.c): "/" is always double; "*" is integer
 * when neither side is double; Math is double except abs() of integer or
 * logical input (do_abs()). */
SVT_HD int svt_ew_result_type(int op, int x_type, int v_type)
{
	if (svt_ew_is_compare(op) || svt_ew_is_pred(op))
		return SVTGPU_LGL;
	if (op == SVTGPU_EW_MUL)
		return (x_type != SVTGPU_DOUBLE && v_type != SVTGPU_DOUBLE)
			? SVTGPU_INT : SVTGPU_DOUBLE;
	if (op == SVTGPU_EW_ABS && x_type != SVTGPU_DOUBLE)
		return SVTGPU_INT;
	return SVTGPU_DOUBLE;
}

/* Comparison or is.* predicate of one stored value (base R's relop.c and
 * do_isna() / do_isnan() / do_isinfinite()): SVT_CMP_TRUE, SVT_CMP_NA or
 * SVT_CMP_DROP (FALSE).  x: the value as a double (an int32 converts
 * exactly, so int op int compares as R does); x_na: the value is NA
 * (NA_integer_ or R_IsNA()).  v: the operand element as a double (never NA
 * or NaN once admitted), ignored by the predicates.  An NA or NaN value
 * compares to NA; is.na() is TRUE for both, is.nan() for a NaN that is not
 * NA. */
SVT_HD int svt_ew_cmp(int op, double x, int x_na, double v)
{
	switch (op) {
	    case SVTGPU_EW_IS_NA:
		return (x_na || svt_isnan(x)) ? SVT_CMP_TRUE : SVT_CMP_DROP;
	    case SVTGPU_EW_IS_NAN:
		return (!x_na && svt_isnan(x)) ? SVT_CMP_TRUE : SVT_CMP_DROP;
	    case SVTGPU_EW_IS_INFINITE:
		return (!x_na && (x == svt_posinf() || x == svt_neginf()))
			? SVT_CMP_TRUE : SVT_CMP_DROP;
	}
	if (x_na || svt_isnan(x) || svt_isnan(v))
		return SVT_CMP_NA;
	bool r;
	switch (op) {
	    case SVTGPU_EW_GT: r = x >  v; break;
	    case SVTGPU_EW_GE: r = x >= v; break;
	    case SVTGPU_EW_LT: r = x <  v; break;
	    case SVTGPU_EW_LE: r = x <= v; break;
	    case SVTGPU_EW_EQ: r = x == v; break;
	    case SVTGPU_EW_NE: r = x != v; break;
	    default:           return SVT_CMP_NA;
	}
	return r ? SVT_CMP_TRUE : SVT_CMP_DROP;
}

/* Would f(0) stay 0 for every element of the operand?  Arith ops only.
 *   margin 0: v is a scalar; 1: v[i] for row i (R's recycling of `x op v`
 *   with length(v) == nrow, any number of dimensions); 2: v[j] for column j
 *   (`sweep(x, 2, v, op)`, 2-D only; nleaf columns).
 * Comparisons (`v op x` mirrored first) need `0 op v` FALSE for every
 * element: v >= 0 for ">", v > 0 for ">=", v <= 0 for "<", v < 0 for "<=",
 * v != 0 for "==", v == 0 for "!="; NA and NaN never (0 op NA is NA).
 * Returns SVT_EW_OK or a refusal code; *bad receives the offending element
 * for SVT_EW_BAD_VALUE. */
SVT_HD int svt_ew_check(int op, int x_type, int v_type, int64_t v_len,
			int margin, int v_on_left, int ndim, int64_t nrow,
			int64_t nleaf, const void *v, int64_t *bad)
{
	*bad = -1;
	if (!svt_ew_type_ok(x_type))
		return SVT_EW_BAD_X_TYPE;
	if (svt_ew_is_unary(op))
		return SVT_EW_OK;
	const int cmp = svt_ew_is_compare(op);
	if (!svt_ew_is_arith(op) && !cmp)
		return SVT_EW_BAD_OPCODE;
	if (cmp && v_on_left)
		op = svt_ew_mirror(op);
	if (op == SVTGPU_EW_DIV && v_on_left)
		return SVT_EW_LEFT_DIV;
	if (!svt_ew_type_ok(v_type))
		return SVT_EW_BAD_V_TYPE;
	if (margin < 0 || margin > 2 || (margin == 2 && ndim != 2))
		return SVT_EW_BAD_MARGIN;
	const int64_t want = margin == 0 ? 1 : margin == 1 ? nrow : nleaf;
	if (v_len != want)
		return SVT_EW_BAD_LENGTH;
	for (int64_t i = 0; i < v_len; i++) {
		int ok;
		if (cmp) {
			const double d = v_type == SVTGPU_DOUBLE
				? ((const double *) v)[i]
				: (((const int32_t *) v)[i] == SVT_NA_INT ? svt_nan()
					: (double) ((const int32_t *) v)[i]);
			ok = svt_ew_cmp(op, 0.0, 0, d) == SVT_CMP_DROP;
		} else if (v_type == SVTGPU_DOUBLE) {
			const double d = ((const double *) v)[i];
			/* 0 * Inf is NaN, 0 * NA is NA; 0 / 0 is NaN, 0 / NA
			   is NA; 0 / Inf is 0 */
			ok = op == SVTGPU_EW_MUL ? svt_isfinite(d)
						 : !svt_isnan(d) && d != 0.0;
		} else {
			const int32_t k = ((const int32_t *) v)[i];
			ok = k != SVT_NA_INT && (op == SVTGPU_EW_MUL || k != 0);
		}
		if (!ok) {
			*bad = i;
			return SVT_EW_BAD_VALUE;
		}
	}
	return SVT_EW_OK;
}

/* operand element i as R prints it; `lgl_words`: logical as TRUE / FALSE */
static inline void svt_ew_value_name(int v_type, const void *v, int64_t i,
				     int lgl_words, char *buf, size_t len)
{
	if (v_type != SVTGPU_DOUBLE) {
		const int32_t k = ((const int32_t *) v)[i];
		if (k == SVT_NA_INT)
			snprintf(buf, len, "NA");
		else if (v_type == SVTGPU_LGL && lgl_words)
			snprintf(buf, len, "%s", k ? "TRUE" : "FALSE");
		else
			snprintf(buf, len, "%d", (int) k);
		return;
	}
	const double d = ((const double *) v)[i];
	if (svt_is_na_real(d))       snprintf(buf, len, "NA");
	else if (svt_isnan(d))       snprintf(buf, len, "NaN");
	else if (d == svt_posinf())  snprintf(buf, len, "Inf");
	else if (d == svt_neginf())  snprintf(buf, len, "-Inf");
	else                         snprintf(buf, len, "%.15g", d);
}

/* The R error message of a refusal (host only).  `opname` is the name the
 * caller was given (it may be an operator svt_ew_check() does not know);
 * `kind` (SVT_EW_KIND_*) the group it was given as. */
static inline void svt_ew_refusal_message(int code, const char *opname,
					  int kind, int op, int v_type, const void *v,
					  int64_t v_len, int margin,
					  int64_t nrow, int64_t nleaf,
					  int64_t bad, char *buf, size_t len)
{
	char vname[40];
	switch (code) {
	    case SVT_EW_BAD_OPCODE:
		if (kind == SVT_EW_KIND_COMPARE)
			snprintf(buf, len, "Compare operator \"%s\" is not "
				 "supported on a SparseArray on the GPU path "
				 "(supported: \">\", \">=\", \"<\", \"<=\", "
				 "\"==\", \"!=\")", opname);
		else if (kind == SVT_EW_KIND_IS)
			snprintf(buf, len, "\"%s\" is not supported on a "
				 "SparseArray on the GPU path: it would turn the "
				 "implicit zeros into TRUE or is not a predicate "
				 "(supported: is.na, is.nan, is.infinite)", opname);
		else if (kind == SVT_EW_KIND_MATH)
			snprintf(buf, len, "Math function \"%s\" is not supported "
				 "on a SparseArray on the GPU path: it does not "
				 "map zero to zero (supported: abs, sign, sqrt, "
				 "floor, ceiling, trunc, log1p, expm1)", opname);
		else
			snprintf(buf, len, "Arith operator \"%s\" is not "
				 "supported on a SparseArray on the GPU path: it "
				 "would turn the implicit zeros into nonzero "
				 "values (supported: \"*\" and \"/\")", opname);
		return;
	    case SVT_EW_LEFT_DIV:
		snprintf(buf, len, "operator \"/\" with the SparseArray on the "
			 "right is not supported: the implicit zeros would "
			 "become Inf, NA or NaN");
		return;
	    case SVT_EW_BAD_X_TYPE:
		snprintf(buf, len, "\"%s\": only logical, integer and double "
			 "SparseArray objects are supported on the GPU path",
			 opname);
		return;
	    case SVT_EW_BAD_V_TYPE:
		snprintf(buf, len, "operator \"%s\": the operand must be a "
			 "logical, integer or double vector", opname);
		return;
	    case SVT_EW_BAD_MARGIN:
		snprintf(buf, len, "operator \"%s\": MARGIN must be 0 (a scalar), "
			 "1 (along the rows) or 2 (along the columns of a "
			 "2-D object)", opname);
		return;
	    case SVT_EW_BAD_LENGTH:
		if (margin == 0)
			snprintf(buf, len, "operator \"%s\": the operand has "
				 "length %lld, a scalar operand must have length "
				 "1", opname, (long long) v_len);
		else
			snprintf(buf, len, "operator \"%s\": the operand has "
				 "length %lld, it must have length %s = %lld",
				 opname, (long long) v_len,
				 margin == 1 ? "nrow(x)" : "ncol(x)",
				 (long long) (margin == 1 ? nrow : nleaf));
		return;
	    case SVT_EW_BAD_VALUE: {
		const int cmp = svt_ew_is_compare(op);
		svt_ew_value_name(v_type, v, bad, cmp, vname, sizeof(vname));
		const char *zeros = op == SVTGPU_EW_MUL
			? "NaN or NA (0 * Inf, 0 * NA)" : "NaN or NA (0 / 0, 0 / NA)";
		if (cmp)
			zeros = (strcmp(vname, "NA") == 0 || strcmp(vname, "NaN") == 0)
				? "NA" : "TRUE";
		snprintf(buf, len, "operator \"%s\": element %lld of the operand "
			 "is %s, so the implicit zeros of the result would be "
			 "%s", opname, (long long) bad + 1, vname, zeros);
		return;
	    }
	}
	snprintf(buf, len, "operator \"%s\": refused (code %d)", opname, code);
}

/* Integer result: `x * v` of two integers (R_integer_times(): the product
 * in 64 bits, NA_integer_ with the overflow warning when it leaves the int
 * range or equals INT_MIN) and abs() of an integer.  v is never NA. */
SVT_HD int32_t svt_ew_int(int op, int32_t x, int32_t v, uint32_t *fl)
{
	if (x == SVT_NA_INT)
		return SVT_NA_INT;
	int64_t z = op == SVTGPU_EW_MUL ? (int64_t) x * (int64_t) v
					: (x < 0 ? -(int64_t) x : (int64_t) x);
	if (z > INT32_MAX || z <= INT32_MIN) {
		*fl |= SVTGPU_EW_WARN_INT_OVERFLOW;
		return SVT_NA_INT;
	}
	if (z == 0)
		*fl |= SVT_EW_DROPPED;
	return (int32_t) z;
}

/* Double result.  x_na: the input is NA (integer NA_integer_ or R_IsNA()).
 * NA stays NA_real_ and any other NaN keeps its own bits (math1(): "keep NA
 * vs NaN distinction"; for "*" and "/" the x86 FPU returns the NaN operand).
 * A NaN produced from a non-NaN value is the canonical quiet NaN; from a
 * Math function it sets the "NaNs produced" warning (math1()), from "*" or
 * "/" (Inf * 0, Inf / Inf) it does not (real_binary()). */
SVT_HD double svt_ew_dbl(int op, double x, int x_na, double v, uint32_t *fl)
{
	if (x_na)
		return svt_na_real();
	if (svt_isnan(x))
		return x;
	double r;
	switch (op) {
	    case SVTGPU_EW_MUL:     r = x * v; break;
	    case SVTGPU_EW_DIV:     r = x / v; break;
	    case SVTGPU_EW_ABS:     r = fabs(x); break;
	    case SVTGPU_EW_SIGN:    r = x > 0.0 ? 1.0 : (x < 0.0 ? -1.0 : 0.0);
				    break;
	    case SVTGPU_EW_SQRT:    r = sqrt(x); break;
	    case SVTGPU_EW_FLOOR:   r = floor(x); break;
	    case SVTGPU_EW_CEILING: r = ceil(x); break;
	    case SVTGPU_EW_TRUNC:   r = trunc(x); break;
	    case SVTGPU_EW_LOG1P:   r = log1p(x); break;
	    case SVTGPU_EW_EXPM1:   r = expm1(x); break;
	    default:                r = svt_nan(); break;
	}
	if (svt_isnan(r)) {
		if (svt_ew_is_math(op))
			*fl |= SVTGPU_EW_WARN_NAN;
		return svt_nan();
	}
	if (r == 0.0)
		*fl |= SVT_EW_DROPPED;
	return r;
}

/* ------------------------------------------------------------------------
 * Element-wise operations between two SVTs (svtgpu_ewise2)
 *
 * `x op y` of two arrays of the same dimensions, as base R computes
 * `as.matrix(x) op as.matrix(y)` (src/main/arithmetic.c: R_integer_plus(),
 * R_integer_minus(), R_integer_times(), real_binary(); relop.c; logic.c),
 * zeros dropped.  Only operators that map two zeros to 0 / FALSE are
 * admitted.  An entry stored on one side only meets an implicit zero on the
 * other (the value 0, never NA), so one rule per operator serves "x only",
 * "y only" and "both".  The svt_ew2_* opcodes are not opcodes of
 * svt_ew_check(): the scalar path keeps refusing them.
 */
SVT_HD int svt_ew2_is_arith(int op)
{
	return op == SVTGPU_EW_ADD || op == SVTGPU_EW_SUB || op == SVTGPU_EW_MUL;
}

SVT_HD int svt_ew2_is_logic(int op)
{
	return op == SVTGPU_EW_AND || op == SVTGPU_EW_OR;
}

SVT_HD int svt_ew2_is_compare(int op)
{
	return op == SVTGPU_EW_GT || op == SVTGPU_EW_LT || op == SVTGPU_EW_NE;
}

SVT_HD int svt_ew2_admitted(int op)
{
	return svt_ew2_is_arith(op) || svt_ew2_is_logic(op) ||
	       svt_ew2_is_compare(op);
}

SVT_HD const char *svt_ew2_opname(int op)
{
	switch (op) {
	    case SVTGPU_EW_ADD: return "+";
	    case SVTGPU_EW_SUB: return "-";
	    case SVTGPU_EW_MUL: return "*";
	    case SVTGPU_EW_AND: return "&";
	    case SVTGPU_EW_OR:  return "|";
	    case SVTGPU_EW_GT:  return ">";
	    case SVTGPU_EW_LT:  return "<";
	    case SVTGPU_EW_NE:  return "!=";
	}
	return "?";
}

/* "+", "-", "*", "&", "|", ">", "<", "!=" -> opcode; any other name -> 0 */
SVT_HD int svt_ew2_opcode(const char *name)
{
	const int ops[8] = { SVTGPU_EW_ADD, SVTGPU_EW_SUB, SVTGPU_EW_MUL,
			     SVTGPU_EW_AND, SVTGPU_EW_OR, SVTGPU_EW_GT,
			     SVTGPU_EW_LT, SVTGPU_EW_NE };
	for (int k = 0; k < 8; k++)
		if (svt_ew_streq(name, svt_ew2_opname(ops[k])))
			return ops[k];
	return 0;
}

/* Arith: integer unless a side is double (logical op logical is integer);
   Logic and Compare: logical */
SVT_HD int svt_ew2_result_type(int op, int x_type, int y_type)
{
	if (!svt_ew2_is_arith(op))
		return SVTGPU_LGL;
	return (x_type == SVTGPU_DOUBLE || y_type == SVTGPU_DOUBLE)
		? SVTGPU_DOUBLE : SVTGPU_INT;
}

/* The R error message for an operator svt_ew2_opcode() does not admit
 * (host only): what the implicit zeros would become, or the list of the
 * operators served. */
static inline void svt_ew2_refusal_message(const char *opname, char *buf,
					   size_t len)
{
	const char *zeros = NULL;
	char cmp[32];
	if (svt_ew_streq(opname, "/"))
		zeros = "NaN (0 / 0)";
	else if (svt_ew_streq(opname, "^"))
		zeros = "1 (0 ^ 0)";
	else if (svt_ew_streq(opname, "%%") || svt_ew_streq(opname, "%/%"))
		zeros = "NA (0 %% 0, 0 %/% 0)";
	else if (svt_ew_streq(opname, "==") || svt_ew_streq(opname, ">=") ||
		 svt_ew_streq(opname, "<="))
		zeros = (snprintf(cmp, sizeof(cmp), "TRUE (0 %s 0)", opname),
			 cmp);
	if (zeros != NULL)
		snprintf(buf, len, "operator \"%s\" between two SparseArray "
			 "objects is not supported on the GPU path: the implicit "
			 "zeros of the result would become %s", opname, zeros);
	else
		snprintf(buf, len, "operator \"%s\" between two SparseArray "
			 "objects is not supported on the GPU path (supported: "
			 "\"+\", \"-\", \"*\", \"&\", \"|\", \">\", \"<\", \"!=\")",
			 opname);
}

/* Integer result of "+", "-", "*": NA_integer_ on either side gives NA; the
 * result is computed in 64 bits and one outside (-2^31, 2^31) gives NA with
 * the overflow warning (R_integer_plus(), R_integer_minus(),
 * R_integer_times()). */
SVT_HD int32_t svt_ew2_int(int op, int32_t x, int32_t y, uint32_t *fl)
{
	if (x == SVT_NA_INT || y == SVT_NA_INT)
		return SVT_NA_INT;
	const int64_t a = x, b = y;
	const int64_t z = op == SVTGPU_EW_ADD ? a + b
			: op == SVTGPU_EW_SUB ? a - b : a * b;
	if (z > INT32_MAX || z <= INT32_MIN) {
		*fl |= SVTGPU_EW_WARN_INT_OVERFLOW;
		return SVT_NA_INT;
	}
	return (int32_t) z;
}

/* Double result of "+", "-", "*".  x_na / y_na: the operand is NA
 * (NA_integer_ or R_IsNA()).  Written out rather than left to the FPU,
 * whose choice among NaN operands differs between host and GPU: an NA or
 * NaN operand passes through with its own bits, x's before y's (an integer
 * NA as NA_real_; "-" does not negate a NaN); a NaN made from other values
 * (Inf - Inf, Inf * 0) is the canonical quiet NaN.  No contraction. */
SVT_HD double svt_ew2_dbl(int op, double x, int x_na, double y, int y_na)
{
	if (svt_isnan(x))
		return x;
	if (x_na)
		return svt_na_real();
	if (svt_isnan(y))
		return y;
	if (y_na)
		return svt_na_real();
	double r;
#ifdef __CUDA_ARCH__
	r = op == SVTGPU_EW_ADD ? __dadd_rn(x, y)
	  : op == SVTGPU_EW_SUB ? __dsub_rn(x, y) : __dmul_rn(x, y);
#else
	r = op == SVTGPU_EW_ADD ? x + y : op == SVTGPU_EW_SUB ? x - y : x * y;
#endif
	return svt_isnan(r) ? svt_nan() : r;
}

/* Logic and Compare: SVT_CMP_TRUE, SVT_CMP_NA or SVT_CMP_DROP (FALSE).
 * Logic: a nonzero value is TRUE, NA or NaN is NA; "&" is FALSE when a side
 * is FALSE, "|" TRUE when a side is TRUE, otherwise NA wins.  Compare: an
 * int32 is compared as a double (exact); NA or NaN on a side gives NA. */
SVT_HD int svt_ew2_lgl(int op, double x, int x_na, double y, int y_na)
{
	const int xn = x_na || svt_isnan(x), yn = y_na || svt_isnan(y);
	if (svt_ew2_is_logic(op)) {
		const int xt = xn ? SVT_CMP_NA
			: x != 0.0 ? SVT_CMP_TRUE : SVT_CMP_DROP;
		const int yt = yn ? SVT_CMP_NA
			: y != 0.0 ? SVT_CMP_TRUE : SVT_CMP_DROP;
		if (op == SVTGPU_EW_AND) {
			if (xt == SVT_CMP_DROP || yt == SVT_CMP_DROP)
				return SVT_CMP_DROP;
			return (xt == SVT_CMP_NA || yt == SVT_CMP_NA)
				? SVT_CMP_NA : SVT_CMP_TRUE;
		}
		if (xt == SVT_CMP_TRUE || yt == SVT_CMP_TRUE)
			return SVT_CMP_TRUE;
		return (xt == SVT_CMP_NA || yt == SVT_CMP_NA)
			? SVT_CMP_NA : SVT_CMP_DROP;
	}
	if (xn || yn)
		return SVT_CMP_NA;
	bool r;
	switch (op) {
	    case SVTGPU_EW_GT: r = x >  y; break;
	    case SVTGPU_EW_LT: r = x <  y; break;
	    case SVTGPU_EW_NE: r = x != y; break;
	    default:           return SVT_CMP_NA;
	}
	return r ? SVT_CMP_TRUE : SVT_CMP_DROP;
}

/* ------------------------------------------------------------------------
 * Medians (svtgpu_colmedians / svtgpu_rowmedians)
 *
 * Base R's median() of each dense column: NA_real_ when the column holds an
 * NA or NaN and na.rm is FALSE (median.default returns x[NA_integer_]); with
 * na.rm, NA and NaN are removed and nothing left gives NA_real_.  Otherwise
 * the value at 0-based rank (n-1)/2 of the sorted column, or for even n the
 * midpoint of the values at ranks n/2 - 1 and n/2.
 *
 * The implicit zeros (and stored zeros, +0 or -0) form one block in the
 * middle of the sorted order: [negatives | zeros | positives].  The counts of
 * stored negatives, positives and NA / NaN decide whether the middle ranks
 * fall inside the zero block; only when they do not does a kernel select a
 * stored value by rank, among the values of one sign ("side").
 */
#define SVT_MED_NA       0  /* the result is NA_real_ */
#define SVT_MED_ZERO     1  /* the result is +0 */
#define SVT_MED_SELECT   2  /* select the value at `rank` of `side` */

#define SVT_MED_NEG      0
#define SVT_MED_POS      1

#define SVT_MED_2ND_NONE 0  /* odd count: the selected value is the median */
#define SVT_MED_2ND_ZERO 1  /* midpoint of the selected value and 0 */
#define SVT_MED_2ND_NEXT 2  /* midpoint of the selected value and the next
			       larger stored nonzero value (either side) */

typedef struct SvtMedPlan {
	int kind;      /* SVT_MED_NA / _ZERO / _SELECT */
	int side;      /* SVT_MED_NEG / _POS (SELECT only) */
	int second;    /* SVT_MED_2ND_* (SELECT only) */
	int64_t rank;  /* 0-based rank among the side's values, ascending */
} SvtMedPlan;

/* nrow: length of the column; nneg / npos: stored values < 0 / > 0; nna:
   stored NA or NaN (stored zeros count in none of the three) */
SVT_HD SvtMedPlan svt_med_plan(int64_t nrow, int64_t nneg, int64_t npos,
			       int64_t nna, int narm)
{
	SvtMedPlan p;
	p.kind = SVT_MED_NA;
	p.side = SVT_MED_NEG;
	p.second = SVT_MED_2ND_NONE;
	p.rank = 0;
	if (nna > 0 && !narm)
		return p;
	const int64_t n = nrow - nna;
	if (n <= 0)
		return p;
	const int64_t z0 = nneg;                  /* first rank of the zeros */
	const int64_t p0 = n - npos;              /* first rank of positives */
	const int64_t lo = (n - 1) / 2, hi = n / 2;
	if (lo >= z0 && hi < p0) {
		p.kind = SVT_MED_ZERO;
		return p;
	}
	p.kind = SVT_MED_SELECT;
	if (lo < z0) {
		p.side = SVT_MED_NEG;
		p.rank = lo;
		p.second = hi == lo ? SVT_MED_2ND_NONE
			 : (hi < z0 || hi >= p0) ? SVT_MED_2ND_NEXT
			 : SVT_MED_2ND_ZERO;
	} else if (lo >= p0) {
		p.side = SVT_MED_POS;
		p.rank = lo - p0;
		p.second = hi == lo ? SVT_MED_2ND_NONE : SVT_MED_2ND_NEXT;
	} else {
		/* lo is the last zero, hi the first positive */
		p.side = SVT_MED_POS;
		p.rank = 0;
		p.second = SVT_MED_2ND_ZERO;
	}
	return p;
}

/* The midpoint of the two middle values, correctly rounded: (a + b) / 2
 * when a + b is finite (halving is exact), a/2 + b/2 when a + b overflows
 * for finite a and b (base R's mean() sums in long double and gets the
 * same).  -Inf and +Inf give NaN (never NA); a zero result is +0. */
SVT_HD double svt_med_mid(double a, double b)
{
	const double s = a + b;
	if (svt_isnan(s))
		return svt_nan();
	if (!svt_isfinite(s) && svt_isfinite(a) && svt_isfinite(b))
		return a / 2.0 + b / 2.0;
	return s / 2.0 + 0.0;
}

/* Order-preserving unsigned keys.  int32: NA_integer_ (INT_MIN) is not a
 * key (returns 0); every other value maps to x ^ 0x80000000, so keys of
 * non-NA values are >= 1.  double: NaN (NA included) is not a key; -x sorts
 * before +x, -0 before +0 (the kernels never select a zero). */
SVT_HD int svt_med_key_i32(int32_t x, uint32_t *key)
{
	*key = (uint32_t) x ^ 0x80000000u;
	return x != SVT_NA_INT;
}

SVT_HD int32_t svt_med_unkey_i32(uint32_t key)
{
	return (int32_t) (key ^ 0x80000000u);
}

SVT_HD int svt_med_key_f64(double x, uint64_t *key)
{
	const uint64_t u = svt_d2u(x);
	*key = (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
	return !svt_isnan(x);
}

SVT_HD double svt_med_unkey_f64(uint64_t key)
{
	return svt_u2d((key >> 63) ? (key & 0x7FFFFFFFFFFFFFFFULL) : ~key);
}

#endif  /* SVT_SEMANTICS_H */
