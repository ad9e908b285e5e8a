/* TEST INFRASTRUCTURE -- not part of the product.
 *
 * CPU restatement of the element-wise operations of svtgpu_ewise() on the
 * flat CSC view of an SVT (oracle/svt_oracle.h), written independently of
 * the product's rules in csrc/svt_semantics.h.  tests/test_ewise_host.py
 * holds it bit for bit to base R's dense definition computed with numpy;
 * tests/test_gpu_ewise.py and tools/bench_ewise.py hold the GPU to it.
 * Built on demand by tests/ewise_oracle.py.
 */
#include "../oracle/svt_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define INTSXP  13
#define REALSXP 14
#define NA_INT  INT_MIN

static double na_real(void)
{
	union { double d; uint64_t u; } x;
	x.u = 0x7FF00000000007A2ULL;  /* low word 1954 */
	return x.d;
}

/* Element-wise operations that keep zeros at zero, restated from base R's
 * dense semantics (src/main/arithmetic.c): R_integer_times(), real_binary()
 * (an integer NA operand becomes NA_real_), math1() (a NaN input keeps its
 * bits, a NaN made from a non-NaN value warns "NaNs produced"), do_abs()
 * (integer result for integer / logical input).  glibc's libm, as R uses on
 * Linux.  Results equal to 0 (-0 included) are dropped, NA / NaN kept; a NaN
 * made from a non-NaN value is written as the canonical quiet NaN and an NA
 * input as NA_real_.  Opcodes: 1 "*", 2 "/", 11-18 abs, sign, sqrt, floor,
 * ceiling, trunc, log1p, expm1.  margin 0: v[0]; 1: v[row]; 2: v[leaf].
 */
static int is_nan_bits(double x)
{
	uint64_t u;
	memcpy(&u, &x, 8);
	return (u & 0x7FFFFFFFFFFFFFFFULL) > 0x7FF0000000000000ULL;
}

static int is_na_bits(double x)
{
	uint64_t u;
	memcpy(&u, &x, 8);
	return is_nan_bits(x) && (uint32_t) u == 1954u;
}

static double canonical_nan(void)
{
	union { double d; uint64_t u; } x;
	x.u = 0x7FF8000000000000ULL;
	return x.d;
}

static double math_fun(int op, double x)
{
	switch (op) {
	    case 11: return fabs(x);
	    case 12: return x > 0 ? 1.0 : (x == 0 ? 0.0 : -1.0);
	    case 13: return sqrt(x);
	    case 14: return floor(x);
	    case 15: return ceil(x);
	    case 16: return trunc(x);
	    case 17: return log1p(x);
	    case 18: return expm1(x);
	}
	return canonical_nan();
}

/* op(x) / x op v: the result CSC is malloc()ed (the caller frees the three
 * arrays); *out_type is 13 or 14; *warn bit 0 = integer overflow, bit 1 =
 * NaNs produced.  Returns nonzero for an unknown op. */
int ewise_oracle(const svt_oracle_csc *x, int op, const void *v, int v_type,
		 int margin, int64_t **out_ptr, int32_t **out_offs,
		 void **out_vals, int *out_type, int *warn)
{
	const int is_math = op >= 11 && op <= 18;
	if (!is_math && op != 1 && op != 2)
		return 1;
	const int x_int = x->val_type != REALSXP;
	const int v_int = v_type != REALSXP;
	int otype;
	if (op == 1)
		otype = (x_int && v_int) ? INTSXP : REALSXP;
	else if (op == 11)
		otype = x_int ? INTSXP : REALSXP;
	else
		otype = REALSXP;
	*out_type = otype;
	*warn = 0;
	const int64_t nnz = x->leaf_ptr[x->nleaf];
	int64_t *ptr = (int64_t *) malloc(sizeof(int64_t) * (size_t) (x->nleaf + 1));
	int32_t *offs = (int32_t *) malloc(sizeof(int32_t) * (size_t) (nnz + 1));
	void *vals = malloc((otype == REALSXP ? 8 : 4) * (size_t) (nnz + 1));
	int64_t w = 0;
	ptr[0] = 0;
	for (int64_t l = 0; l < x->nleaf; l++) {
		const int lac = x->vals == NULL ||
				(x->lacunar != NULL && x->lacunar[l]);
		for (int64_t k = x->leaf_ptr[l]; k < x->leaf_ptr[l + 1]; k++) {
			const int32_t off = x->offs[k];
			const int64_t vi = margin == 0 ? 0 : margin == 1 ? off : l;
			int keep;
			if (otype == INTSXP) {
				/* R_integer_times() / do_abs() */
				const int xi = lac ? 1 : ((const int *) x->vals)[k];
				int r;
				if (xi == NA_INT) {
					r = NA_INT;
				} else {
					const long long z = op == 1
						? (long long) xi *
						  ((const int *) v)[vi]
						: llabs((long long) xi);
					if (z > INT_MAX || z <= INT_MIN) {
						*warn |= 1;
						r = NA_INT;
					} else {
						r = (int) z;
					}
				}
				keep = r != 0;
				((int *) vals)[w] = r;
			} else {
				double xd, r;
				int na;
				if (lac) {
					xd = 1.0;
					na = 0;
				} else if (x_int) {
					const int xi = ((const int *) x->vals)[k];
					na = xi == NA_INT;
					xd = (double) xi;
				} else {
					xd = ((const double *) x->vals)[k];
					na = is_na_bits(xd);
				}
				if (na) {
					r = na_real();
				} else if (is_nan_bits(xd)) {
					r = xd;
				} else {
					if (is_math) {
						r = math_fun(op, xd);
					} else {
						const double vd = v_int
							? (double) ((const int *) v)[vi]
							: ((const double *) v)[vi];
						r = op == 1 ? xd * vd : xd / vd;
					}
					if (is_nan_bits(r)) {
						if (is_math)
							*warn |= 2;
						r = canonical_nan();
					}
				}
				keep = !(r == 0.0);
				((double *) vals)[w] = r;
			}
			if (keep) {
				offs[w] = off;
				w++;
			}
		}
		ptr[l + 1] = w;
	}
	*out_ptr = ptr;
	*out_offs = offs;
	*out_vals = vals;
	return 0;
}
