/* TEST INFRASTRUCTURE -- not part of the product.
 *
 * Host build of the rules of `x op y` between two SVTs in
 * sparsearray_b200/csrc/svt_semantics.h (svt_ew2_*: admission, result type,
 * the per-entry value rules the CUDA kernels apply, the refusal message), so
 * tests/test_ops2_host.py can hold them to numpy without a GPU.  Built on
 * demand into a temporary directory.
 */
#include "../sparsearray_b200/csrc/svt_semantics.h"

int e2_opcode(const char *name) { return svt_ew2_opcode(name); }

int e2_result_type(int op, int x_type, int y_type)
{
	return svt_ew2_result_type(op, x_type, y_type);
}

int e2_int(int op, int32_t x, int32_t y, uint32_t *fl)
{
	return svt_ew2_int(op, x, y, fl);
}

double e2_dbl(int op, double x, int x_na, double y, int y_na)
{
	return svt_ew2_dbl(op, x, x_na, y, y_na);
}

int e2_lgl(int op, double x, int x_na, double y, int y_na)
{
	return svt_ew2_lgl(op, x, x_na, y, y_na);
}

void e2_msg(const char *opname, char *buf, int len)
{
	svt_ew2_refusal_message(opname, buf, (size_t) len);
}
