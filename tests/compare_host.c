/* TEST INFRASTRUCTURE -- not part of the product.
 *
 * Host build of the comparison rules of sparsearray_b200/csrc/svt_semantics.h
 * (the value rule the CUDA kernels apply to every stored value, and the
 * admission check the glue and the C ABI run before any device work), so
 * tests/test_compare_host.py can hold them to numpy on a machine without a
 * GPU.  Built on demand into a temporary directory.
 */
#include "../sparsearray_b200/csrc/svt_semantics.h"

int cmp_host(int op, double x, int x_na, double v)
{
	return svt_ew_cmp(op, x, x_na, v);
}

int check_host(int op, int x_type, int v_type, int64_t v_len, int margin,
	       int v_on_left, int ndim, int64_t nrow, int64_t nleaf,
	       const void *v, int64_t *bad)
{
	return svt_ew_check(op, x_type, v_type, v_len, margin, v_on_left, ndim,
			    nrow, nleaf, v, bad);
}
