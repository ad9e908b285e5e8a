/* TEST INFRASTRUCTURE -- not part of the product.
 *
 * CPU restatement of svtgpu_ewise2(): `x op y` of two flat CSCs of the same
 * geometry (oracle/svt_oracle.h), written independently of the product's
 * rules in csrc/svt_semantics.h.  A two-pointer merge of each leaf pair; a
 * row stored on one side only meets the value 0 on the other.
 * tests/test_ops2_host.py holds it to numpy's dense `a op b`;
 * tests/test_gpu_ops2.py and tools/bench_ops2.py hold the GPU to it.  Built
 * on demand by tests/ops2_oracle.py.
 *
 * Opcodes: 1 "*", 3 "+", 4 "-", 41 "&", 42 "|", 21 ">", 23 "<", 26 "!=".
 * Base R (src/main/arithmetic.c, relop.c, logic.c):
 *   integer Arith (no double side): NA if a side is NA; the exact result
 *     outside (-2^31, 2^31) is NA with "NAs produced by integer overflow";
 *   double Arith: an integer NA is NA_real_; the first NA / NaN operand
 *     (x before y) is returned with its bits; a NaN made from other values
 *     is the canonical quiet NaN;
 *   Logic: nonzero is TRUE, NA / NaN is NA (three-valued & and |);
 *   Compare: as doubles, NA / NaN on a side gives NA.
 * Zero, -0 and FALSE are dropped.  Logical results hold 1 / NA_integer_.
 */
#include "../oracle/svt_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define LGLSXP  10
#define INTSXP  13
#define REALSXP 14
#define NA_INT  INT_MIN

static uint64_t bits(double x)
{
	uint64_t u;
	memcpy(&u, &x, 8);
	return u;
}

static double from_bits(uint64_t u)
{
	double x;
	memcpy(&x, &u, 8);
	return x;
}

static int nan_bits(double x)
{
	return (bits(x) & 0x7FFFFFFFFFFFFFFFULL) > 0x7FF0000000000000ULL;
}

/* one operand value: lacunar -> 1; `present` 0 -> the implicit zero */
typedef struct {
	int is_int;
	int i;
	double d;
} val;

static val get(const svt_oracle_csc *m, int64_t l, int64_t k, int present)
{
	val v;
	v.is_int = m->val_type != REALSXP;
	v.i = 0;
	v.d = 0.0;
	if (!present)
		return v;
	if (m->vals == NULL || (m->lacunar != NULL && m->lacunar[l])) {
		v.i = 1;
		v.d = 1.0;
	} else if (v.is_int) {
		v.i = ((const int *) m->vals)[k];
	} else {
		v.d = ((const double *) m->vals)[k];
	}
	return v;
}

/* as a double: integer NA -> NA_real_ */
static double as_dbl(val v)
{
	if (!v.is_int)
		return v.d;
	return v.i == NA_INT ? from_bits(0x7FF00000000007A2ULL) : (double) v.i;
}

/* 0 FALSE, 1 TRUE, 2 NA */
static int truth(val v)
{
	if (v.is_int)
		return v.i == NA_INT ? 2 : v.i != 0;
	return nan_bits(v.d) ? 2 : v.d != 0.0;
}

/* returns nonzero when the entry is kept */
static int apply(int op, int otype, val a, val b, int *ri, double *rd,
		 int *warn)
{
	if (otype == INTSXP) {
		if (a.i == NA_INT || b.i == NA_INT) {
			*ri = NA_INT;
			return 1;
		}
		long long z = op == 3 ? (long long) a.i + b.i
			    : op == 4 ? (long long) a.i - b.i
			    : (long long) a.i * b.i;
		if (z > INT_MAX || z < -(long long) INT_MAX) {
			*warn |= 1;
			*ri = NA_INT;
			return 1;
		}
		*ri = (int) z;
		return z != 0;
	}
	if (otype == REALSXP) {
		const double x = as_dbl(a), y = as_dbl(b);
		double r;
		if (nan_bits(x))
			r = x;
		else if (nan_bits(y))
			r = y;
		else {
			volatile double t = op == 3 ? x + y : op == 4 ? x - y
							   : x * y;
			r = nan_bits(t) ? from_bits(0x7FF8000000000000ULL) : t;
		}
		*rd = r;
		return !(r == 0.0);
	}
	int t;
	if (op == 41 || op == 42) {
		const int p = truth(a), q = truth(b);
		if (op == 41)
			t = (p == 0 || q == 0) ? 0 : (p == 2 || q == 2) ? 2 : 1;
		else
			t = (p == 1 || q == 1) ? 1 : (p == 2 || q == 2) ? 2 : 0;
	} else {
		const double x = as_dbl(a), y = as_dbl(b);
		if (nan_bits(x) || nan_bits(y))
			t = 2;
		else
			t = op == 21 ? x > y : op == 23 ? x < y : x != y;
	}
	*ri = t == 2 ? NA_INT : 1;
	return t != 0;
}

/* x op y: the result CSC is malloc()ed (the caller frees the three arrays);
 * *out_type 10, 13 or 14; *warn bit 0 = integer overflow.  Returns nonzero
 * for an unknown op or different geometries. */
int ops2_oracle(const svt_oracle_csc *x, const svt_oracle_csc *y, int op,
		int64_t **out_ptr, int32_t **out_offs, void **out_vals,
		int *out_type, int *warn)
{
	if (x->nrow != y->nrow || x->nleaf != y->nleaf)
		return 1;
	int otype;
	if (op == 1 || op == 3 || op == 4)
		otype = (x->val_type == REALSXP || y->val_type == REALSXP)
			? REALSXP : INTSXP;
	else if (op == 41 || op == 42 || op == 21 || op == 23 || op == 26)
		otype = LGLSXP;
	else
		return 1;
	*out_type = otype;
	*warn = 0;
	const int64_t cap = x->leaf_ptr[x->nleaf] + y->leaf_ptr[y->nleaf] + 1;
	int64_t *ptr = (int64_t *) malloc(sizeof(int64_t) * (size_t) (x->nleaf + 1));
	int32_t *offs = (int32_t *) malloc(sizeof(int32_t) * (size_t) cap);
	void *vals = malloc((otype == REALSXP ? 8 : 4) * (size_t) cap);
	int64_t w = 0;
	ptr[0] = 0;
	for (int64_t l = 0; l < x->nleaf; l++) {
		int64_t i = x->leaf_ptr[l], j = y->leaf_ptr[l];
		const int64_t ie = x->leaf_ptr[l + 1], je = y->leaf_ptr[l + 1];
		while (i < ie || j < je) {
			const int32_t ox = i < ie ? x->offs[i] : INT_MAX;
			const int32_t oy = j < je ? y->offs[j] : INT_MAX;
			const int32_t off = ox < oy ? ox : oy;
			const int hx = ox == off, hy = oy == off;
			const val a = get(x, l, i, hx), b = get(y, l, j, hy);
			int ri = 0;
			double rd = 0.0;
			if (apply(op, otype, a, b, &ri, &rd, warn)) {
				offs[w] = off;
				if (otype == REALSXP)
					((double *) vals)[w] = rd;
				else
					((int *) vals)[w] = ri;
				w++;
			}
			i += hx;
			j += hy;
		}
		ptr[l + 1] = w;
	}
	*out_ptr = ptr;
	*out_offs = offs;
	*out_vals = vals;
	return 0;
}
