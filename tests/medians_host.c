/* TEST INFRASTRUCTURE -- not part of the product.
 *
 * Host build of the median rules of sparsearray_b200/csrc/svt_semantics.h
 * (the plan that the classify kernel applies to every leaf's counts, the
 * midpoint and the order-preserving keys of the selection kernel), so
 * tests/test_medians_host.py can hold them to numpy on a machine without a
 * GPU.  Built on demand into a temporary directory.
 */
#include "../sparsearray_b200/csrc/svt_semantics.h"

void plan_host(int64_t nrow, int64_t nneg, int64_t npos, int64_t nna,
	       int narm, int *kind, int *side, int *second, int64_t *rank)
{
	SvtMedPlan p = svt_med_plan(nrow, nneg, npos, nna, narm);
	*kind = p.kind;
	*side = p.side;
	*second = p.second;
	*rank = p.rank;
}

double mid_host(double a, double b)
{
	return svt_med_mid(a, b);
}

int key_i32_host(int32_t x, uint32_t *key)
{
	return svt_med_key_i32(x, key);
}

int32_t unkey_i32_host(uint32_t key)
{
	return svt_med_unkey_i32(key);
}

int key_f64_host(double x, uint64_t *key)
{
	return svt_med_key_f64(x, key);
}

double unkey_f64_host(uint64_t key)
{
	return svt_med_unkey_f64(key);
}
