/* Element-wise operations that keep the implicit zeros at zero: `x * v`,
 * `v * x`, `x / v` (scalar, per-row or per-column operand) and the Math
 * functions abs, sign, sqrt, floor, ceiling, trunc, log1p, expm1.  The value
 * rules (types, NA / NaN, integer overflow, what is dropped) and the
 * refusals are in svt_semantics.h; this file streams them over HBM.
 *
 * Reference: the dense semantics of base R (src/main/arithmetic.c); the
 * SparseArray package runs the same operations leaf by leaf on the host.
 *
 * Fast path, one pass: a map over [0, nnz) reads (offset, value) and writes
 * (offset, f(value)) at the same positions of a new device CSC; leaf_ptr is
 * copied.  The entry range is cut into tiles of 32,768 entries taken
 * cyclically (block b: tiles b, b + G, ...), so the GPU sweeps the arrays
 * front to back as row_hist does, with 16-byte loads and stores of four
 * entries per lane.  Per-column operands find the leaf of each tile's first
 * and last entry by binary search, as hist_tile_leaves does, then the leaf of
 * each group of four inside those bounds.  Warnings and "a value became 0"
 * are OR-ed into one device word.
 *
 * Compaction, only when a value became 0: a warp per leaf counts the kept
 * entries, svtgpu_exclusive_scan gives the new leaf_ptr and a second
 * warp-per-leaf pass copies the kept entries, in order, into arrays of the
 * exact size; the first pass's arrays are freed.
 *
 * Comparisons (x > v, ..., x != v) and is.na / is.nan / is.infinite are the
 * same compaction applied to x itself, a filter with a logical result: the
 * entries where the value is TRUE or NA survive, stored as 1 / NA_integer_
 * only when an NA survived (otherwise the result has no value array).
 */
#include "svtgpu_internal.h"

#include <stdlib.h>
#include <string.h>

#include <type_traits>

#define EW_TILE     32768                        /* entries per cyclic tile */
#define EW_THREADS  256
#define EW_QPT      (EW_TILE / 4 / EW_THREADS)   /* quads per lane and tile */
#define EW_BATCH    4                            /* quads in flight per lane */

enum { EW_IN_INT = 0, EW_IN_DBL = 1, EW_IN_ONES = 2 };

struct EwParams {
	const int64_t *leaf_ptr;
	const int32_t *offs;
	const void *vals;
	int32_t *out_offs;
	void *out_vals;
	const void *v;        /* int32 (integer result) or double operand */
	int64_t nnz, nleaf;
	int op;
	uint32_t *flags;
};

/* first leaf l in [lo, hi] whose range ends after entry e */
__device__ __forceinline__ int64_t ew_leaf_of(const int64_t *__restrict__ lp,
					      int64_t lo, int64_t hi, int64_t e)
{
	while (lo < hi) {
		const int64_t mid = lo + ((hi - lo) >> 1);
		if (__ldg(lp + mid + 1) <= e) lo = mid + 1;
		else                          hi = mid;
	}
	return lo;
}

template <int MARGIN, typename TV>
__device__ __forceinline__ TV ew_operand(const TV *__restrict__ v, TV v0,
					 int32_t off, int64_t leaf)
{
	if (MARGIN == 0) return v0;
	if (MARGIN == 1) return __ldg(v + off);
	return __ldg(v + leaf);
}

template <int IN, typename TOut, int MARGIN>
__global__ void __launch_bounds__(EW_THREADS)
ewise_map(EwParams P)
{
	typedef typename std::conditional<sizeof(TOut) == 4, int32_t,
					  double>::type TV;
	__shared__ int64_t s_leaf[2];
	const TV *vop = (const TV *) P.v;
	const bool arith = P.op == SVTGPU_EW_MUL || P.op == SVTGPU_EW_DIV;
	const TV v0 = arith ? vop[0] : (TV) 0;
	const int64_t ntiles = (P.nnz + EW_TILE - 1) / EW_TILE;
	uint32_t fl = 0;
	for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
		const int64_t e0 = t * EW_TILE;
		const int64_t e_end = e0 + EW_TILE < P.nnz ? e0 + EW_TILE : P.nnz;
		int64_t l_lo = 0, l_hi = 0;
		if (MARGIN == 2) {
			if (threadIdx.x < 2)
				s_leaf[threadIdx.x] = ew_leaf_of(P.leaf_ptr, 0,
					P.nleaf - 1, threadIdx.x == 0 ? e0 : e_end - 1);
			__syncthreads();
			l_lo = s_leaf[0];
			l_hi = s_leaf[1];
			__syncthreads();
		}
		#pragma unroll 1
		for (int b = 0; b < EW_QPT; b += EW_BATCH) {
			int64_t e[EW_BATCH];
			int4 o[EW_BATCH], xi[EW_BATCH];
			double2 xa[EW_BATCH], xb[EW_BATCH];
			#pragma unroll
			for (int k = 0; k < EW_BATCH; k++) {
				e[k] = e0 + 4 * ((int64_t) (b + k) * EW_THREADS +
						 threadIdx.x);
				if (e[k] < e_end) {
					o[k] = __ldcs((const int4 *) (P.offs + e[k]));
					if (IN == EW_IN_INT)
						xi[k] = __ldcs((const int4 *)
							((const int32_t *) P.vals + e[k]));
					if (IN == EW_IN_DBL) {
						const double2 *p = (const double2 *)
							((const double *) P.vals + e[k]);
						xa[k] = __ldcs(p);
						xb[k] = __ldcs(p + 1);
					}
				}
			}
			#pragma unroll
			for (int k = 0; k < EW_BATCH; k++) {
				if (e[k] >= e_end)
					continue;
				int64_t leaf = 0;
				if (MARGIN == 2)
					leaf = ew_leaf_of(P.leaf_ptr, l_lo, l_hi, e[k]);
				const int32_t oo[4] = { o[k].x, o[k].y, o[k].z,
							o[k].w };
				int32_t xs[4] = { 1, 1, 1, 1 };
				double xd[4] = { 1.0, 1.0, 1.0, 1.0 };
				if (IN == EW_IN_INT) {
					xs[0] = xi[k].x; xs[1] = xi[k].y;
					xs[2] = xi[k].z; xs[3] = xi[k].w;
				}
				if (IN == EW_IN_DBL) {
					xd[0] = xa[k].x; xd[1] = xa[k].y;
					xd[2] = xb[k].x; xd[3] = xb[k].y;
				}
				int32_t ro[4];
				TOut rv[4];
				#pragma unroll
				for (int j = 0; j < 4; j++) {
					const int64_t ej = e[k] + j;
					if (ej >= P.nnz) {      /* padding stays zero */
						ro[j] = 0;
						rv[j] = (TOut) 0;
						continue;
					}
					if (MARGIN == 2)
						while (__ldg(P.leaf_ptr + leaf + 1) <= ej)
							leaf++;
					const TV vv = arith ? ew_operand<MARGIN>(vop,
							v0, oo[j], leaf) : (TV) 0;
					ro[j] = oo[j];
					if (sizeof(TOut) == 4) {
						rv[j] = (TOut) svt_ew_int(P.op, xs[j],
							(int32_t) vv, &fl);
					} else if (IN == EW_IN_DBL) {
						rv[j] = (TOut) svt_ew_dbl(P.op, xd[j],
							svt_is_na_real(xd[j]),
							(double) vv, &fl);
					} else {
						rv[j] = (TOut) svt_ew_dbl(P.op,
							(double) xs[j],
							xs[j] == SVT_NA_INT,
							(double) vv, &fl);
					}
				}
				__stcs((int4 *) (P.out_offs + e[k]),
				       make_int4(ro[0], ro[1], ro[2], ro[3]));
				if (sizeof(TOut) == 4) {
					__stcs((int4 *) ((int32_t *) P.out_vals + e[k]),
					       make_int4((int32_t) rv[0], (int32_t) rv[1],
							 (int32_t) rv[2], (int32_t) rv[3]));
				} else {
					double2 *q = (double2 *)
						((double *) P.out_vals + e[k]);
					__stcs(q, make_double2((double) rv[0],
							       (double) rv[1]));
					__stcs(q + 1, make_double2((double) rv[2],
								   (double) rv[3]));
				}
			}
		}
	}
	fl = __reduce_or_sync(0xFFFFFFFFu, fl);
	if ((threadIdx.x & 31) == 0 && fl != 0)
		atomicOr(P.flags, fl);
}

/* ---- compaction: count -> scan -> stable copy ----
 * What is kept is a "keep rule" K:
 *   KeepNonzero<T>  a computed value array (Arith / Math): keep value != 0
 *                   (NaN and NA are not 0) and copy the value;
 *   KeepCmp<IN, M>  a comparison or is.* predicate of x's own values against
 *                   the operand (svt_ew_cmp()): keep TRUE and NA, write 1 or
 *                   NA_integer_ (only when the result stores values).
 * Every rule gives, per entry, SVT_CMP_DROP / SVT_CMP_TRUE / SVT_CMP_NA:
 *   leaf_operand(leaf)       the operand of a whole leaf (margin 0 / 2);
 *   cls1(e, off, vl)         one entry;
 *   load4(e, R) / cls4(R, vl, c)  four entries from 16-byte loads (e is a
 *                            multiple of 4, so the loads are aligned);
 *   out(e, c)                the value written for a kept entry. */
template <typename T>
struct KeepNonzero {
	typedef T TOut;
	struct Raw { T x[4]; };
	static constexpr int BATCH = 4;     /* quads in flight per lane */
	const T *vals;
	__device__ __forceinline__ double leaf_operand(int64_t) const { return 0.0; }
	__device__ __forceinline__ int cls1(int64_t e, int32_t, double) const
	{
		return vals[e] != (T) 0 ? SVT_CMP_TRUE : SVT_CMP_DROP;
	}
	__device__ __forceinline__ void load4(int64_t e, Raw &r) const
	{
		if (sizeof(T) == 4) {
			const int4 q = __ldcs((const int4 *) (vals + e));
			r.x[0] = (T) q.x; r.x[1] = (T) q.y;
			r.x[2] = (T) q.z; r.x[3] = (T) q.w;
		} else {
			const double2 *p = (const double2 *) (vals + e);
			const double2 a = __ldcs(p), b = __ldcs(p + 1);
			r.x[0] = (T) a.x; r.x[1] = (T) a.y;
			r.x[2] = (T) b.x; r.x[3] = (T) b.y;
		}
	}
	__device__ __forceinline__ void cls4(const Raw &r, double, int c[4]) const
	{
		#pragma unroll
		for (int j = 0; j < 4; j++)
			c[j] = r.x[j] != (T) 0 ? SVT_CMP_TRUE : SVT_CMP_DROP;
	}
	__device__ __forceinline__ T out(int64_t e, int) const { return vals[e]; }
	__device__ __forceinline__ int32_t off_at(int64_t) const { return 0; }
};

template <int IN, int MARGIN>
struct KeepCmp {
	typedef int32_t TOut;
	struct Raw { int4 o; int4 xi; double2 xa, xb; };
	/* offsets alone (a lacunar x) are light enough for 8; with 4, ptxas
	   spills 8 bytes in the margin-1 form */
	static constexpr int BATCH = IN == EW_IN_ONES ? 8 : 4;
	const int32_t *offs;
	const void *vals;
	const double *v;      /* operand as doubles (margin 1: nrow, 2: nleaf) */
	double v0;
	int op;
	__device__ __forceinline__ double leaf_operand(int64_t leaf) const
	{
		return MARGIN == 2 ? __ldg(v + leaf) : v0;
	}
	__device__ __forceinline__ int one(double x, int na, int32_t off,
					   double vl) const
	{
		return svt_ew_cmp(op, x, na, MARGIN == 1 ? __ldg(v + off) : vl);
	}
	__device__ __forceinline__ int cls_int(int32_t k, int32_t off,
					       double vl) const
	{
		return one((double) k, k == SVT_NA_INT, off, vl);
	}
	__device__ __forceinline__ int cls_dbl(double d, int32_t off,
					       double vl) const
	{
		return one(d, svt_is_na_real(d), off, vl);
	}
	__device__ __forceinline__ int cls1(int64_t e, int32_t off,
					    double vl) const
	{
		if (IN == EW_IN_INT)
			return cls_int(((const int32_t *) vals)[e], off, vl);
		if (IN == EW_IN_DBL)
			return cls_dbl(((const double *) vals)[e], off, vl);
		return one(1.0, 0, off, vl);
	}
	__device__ __forceinline__ void load4(int64_t e, Raw &r) const
	{
		r.o = MARGIN == 1 ? __ldcs((const int4 *) (offs + e))
				  : make_int4(0, 0, 0, 0);
		if (IN == EW_IN_INT)
			r.xi = __ldcs((const int4 *) ((const int32_t *) vals + e));
		if (IN == EW_IN_DBL) {
			const double2 *p = (const double2 *)
				((const double *) vals + e);
			r.xa = __ldcs(p);
			r.xb = __ldcs(p + 1);
		}
	}
	__device__ __forceinline__ void cls4(const Raw &r, double vl,
					     int c[4]) const
	{
		if (IN == EW_IN_INT) {
			c[0] = cls_int(r.xi.x, r.o.x, vl);
			c[1] = cls_int(r.xi.y, r.o.y, vl);
			c[2] = cls_int(r.xi.z, r.o.z, vl);
			c[3] = cls_int(r.xi.w, r.o.w, vl);
		} else if (IN == EW_IN_DBL) {
			c[0] = cls_dbl(r.xa.x, r.o.x, vl);
			c[1] = cls_dbl(r.xa.y, r.o.y, vl);
			c[2] = cls_dbl(r.xb.x, r.o.z, vl);
			c[3] = cls_dbl(r.xb.y, r.o.w, vl);
		} else {
			c[0] = one(1.0, 0, r.o.x, vl);
			c[1] = one(1.0, 0, r.o.y, vl);
			c[2] = one(1.0, 0, r.o.z, vl);
			c[3] = one(1.0, 0, r.o.w, vl);
		}
	}
	__device__ __forceinline__ int32_t out(int64_t, int c) const
	{
		return c == SVT_CMP_NA ? SVT_NA_INT : 1;
	}
	__device__ __forceinline__ int32_t off_at(int64_t e) const
	{
		return MARGIN == 1 ? offs[e] : 0;
	}
};

/* Count pass, a warp per leaf: the kept entries of every leaf; OR-s
 * SVT_EW_DROPPED (something was dropped) and SVT_EW_NA_KEPT into *flags.
 * The 4-aligned middle of a leaf is read as quads (16-byte loads,
 * K::BATCH of them in flight per lane), the at most 3 + 3 entries at its
 * ends by single lanes. */
template <class K>
__global__ void __launch_bounds__(256)
ewise_count_kept(const int64_t *__restrict__ leaf_ptr, int64_t nleaf, K k,
		 int64_t *__restrict__ counts, uint32_t *__restrict__ flags)
{
	const int lane = threadIdx.x & 31;
	const int64_t warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	uint32_t fl = 0;
	for (int64_t leaf = gw; leaf < nleaf; leaf += warps) {
		const int64_t a = leaf_ptr[leaf], b = leaf_ptr[leaf + 1];
		const int64_t a4r = (a + 3) & ~(int64_t) 3;
		const int64_t a4 = a4r < b ? a4r : b;
		const int64_t b4r = b & ~(int64_t) 3;
		const int64_t b4 = b4r > a4 ? b4r : a4;
		const double vl = k.leaf_operand(leaf);
		unsigned n = 0;
		int c;
		/* head [a, a4) and tail [b4, b) */
		if (lane < 8) {
			const int64_t e = lane < 4 ? a + lane : b4 + (lane - 4);
			if (e < (lane < 4 ? a4 : b)) {
				c = k.cls1(e, k.off_at(e), vl);
				n += c != SVT_CMP_DROP;
				fl |= c == SVT_CMP_NA ? SVT_EW_NA_KEPT
				    : c == SVT_CMP_DROP ? SVT_EW_DROPPED : 0u;
			}
		}
		const int64_t nq = (b4 - a4) >> 2;
		#pragma unroll 1
		for (int64_t q0 = lane; q0 < nq; q0 += 32 * K::BATCH) {
			typename K::Raw r[K::BATCH];
			#pragma unroll
			for (int j = 0; j < K::BATCH; j++)
				if (q0 + 32 * j < nq)
					k.load4(a4 + 4 * (q0 + 32 * j), r[j]);
			#pragma unroll
			for (int j = 0; j < K::BATCH; j++) {
				if (q0 + 32 * j >= nq)
					continue;
				int cc[4];
				k.cls4(r[j], vl, cc);
				#pragma unroll
				for (int t = 0; t < 4; t++) {
					n += cc[t] != SVT_CMP_DROP;
					fl |= cc[t] == SVT_CMP_NA ? SVT_EW_NA_KEPT
					    : cc[t] == SVT_CMP_DROP ? SVT_EW_DROPPED
					    : 0u;
				}
			}
		}
		n = __reduce_add_sync(0xFFFFFFFFu, n);
		if (lane == 0)
			counts[leaf] = (int64_t) n;
	}
	fl = __reduce_or_sync(0xFFFFFFFFu, fl);
	if (lane == 0 && fl != 0)
		atomicOr(flags, fl);
}

/* Write pass, a warp per leaf: stable copy of the kept entries of every
 * leaf to its new range (offsets, and values when out_vals is not NULL). */
template <class K>
__global__ void __launch_bounds__(256)
ewise_compact(const int64_t *__restrict__ old_ptr,
	      const int64_t *__restrict__ new_ptr,
	      const int32_t *__restrict__ offs, K k,
	      int32_t *__restrict__ out_offs,
	      typename K::TOut *__restrict__ out_vals, int64_t nleaf)
{
	const int lane = threadIdx.x & 31;
	const int64_t warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	for (int64_t leaf = gw; leaf < nleaf; leaf += warps) {
		const int64_t a = old_ptr[leaf], b = old_ptr[leaf + 1];
		const double vl = k.leaf_operand(leaf);
		int64_t w = new_ptr[leaf];
		for (int64_t e0 = a; e0 < b; e0 += 32) {
			const int64_t e = e0 + lane;
			const bool ok = e < b;
			const int32_t off = ok ? offs[e] : 0;
			const int c = ok ? k.cls1(e, off, vl) : SVT_CMP_DROP;
			const bool keep = c != SVT_CMP_DROP;
			const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
			if (keep) {
				const int64_t pos = w + __popc(m & ((1u << lane) - 1u));
				out_offs[pos] = off;
				if (out_vals != NULL)
					out_vals[pos] = k.out(e, c);
			}
			w += __popc(m);
		}
	}
}

/* as many blocks as are resident at once: the tiles are then taken in
   sweeps across the whole GPU */
template <typename K>
static unsigned ew_grid(K kernel, int64_t ntiles)
{
	int per_sm = 0;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel,
			EW_THREADS, 0) != cudaSuccess || per_sm < 1) {
		cudaGetLastError();
		per_sm = 1;
	}
	const int64_t g = (int64_t) svtgpu_sm_count() * per_sm;
	return (unsigned) (ntiles < g ? ntiles : g);
}

template <int IN, typename TOut>
static void launch_map(int margin, int64_t ntiles, cudaStream_t s,
		       const EwParams &P)
{
	if (margin == 0)
		ewise_map<IN, TOut, 0><<<ew_grid(ewise_map<IN, TOut, 0>, ntiles),
					 EW_THREADS, 0, s>>>(P);
	else if (margin == 1)
		ewise_map<IN, TOut, 1><<<ew_grid(ewise_map<IN, TOut, 1>, ntiles),
					 EW_THREADS, 0, s>>>(P);
	else
		ewise_map<IN, TOut, 2><<<ew_grid(ewise_map<IN, TOut, 2>, ntiles),
					 EW_THREADS, 0, s>>>(P);
}

/* the operand as the kernels read it: int32 for an integer result, else
   double (no NA: refused before); comparisons pass SVTGPU_DOUBLE */
static void *ew_host_operand(const void *operand, int operand_type,
			     int64_t len, int out_type, size_t *bytes)
{
	const size_t es = out_type == SVTGPU_DOUBLE ? 8 : 4;
	*bytes = es * (size_t) (len > 0 ? len : 1);
	void *h = calloc((size_t) (len > 0 ? len : 1), es);
	if (h == NULL || len == 0)
		return h;
	if (es == 4 || operand_type == SVTGPU_DOUBLE) {
		memcpy(h, operand, *bytes);
	} else {
		for (int64_t i = 0; i < len; i++)
			((double *) h)[i] = (double) ((const int32_t *) operand)[i];
	}
	return h;
}

struct EwWork {
	svtgpu_matrix *m1, *m2;
	void *d_aux;        /* flags word + operand */
	int64_t *d_counts;  /* nleaf counts + nleaf + 1 new leaf_ptr */
	void *h_op;
};

static int ewise_run(svtgpu_matrix *x, int op, const void *operand,
		     int operand_type, int64_t operand_len, int margin,
		     int out_type, EwWork *W, svtgpu_matrix **out, int *warn)
{
	cudaStream_t s = 0;
	const int64_t nnz = x->nnz;
	const int is_math = svt_ew_is_math(op);
	const bool dbl = out_type == SVTGPU_DOUBLE;
	SVT_CHECK(svtgpu_matrix_create(&W->m1, x->nrow, x->nleaf, nnz, out_type,
		nnz > 0 ? (SVTGPU_HAS_OFFS | SVTGPU_HAS_VALS) : 0));
	svtgpu_matrix *m1 = W->m1;
	/* the arrays were allocated (and the padding zeroed) on m1's upload
	   stream, which does not order against stream 0 */
	SVT_CUDA(cudaStreamSynchronize(m1->up_stream));
	SvtTimer tm;
	SVT_CHECK(svt_timer_begin(&tm, s));
	int launches = 0;
	SVT_CUDA(cudaMemcpyAsync(m1->d_leaf_ptr, x->d_leaf_ptr,
				 sizeof(int64_t) * (size_t) (x->nleaf + 1),
				 cudaMemcpyDeviceToDevice, s));
	uint32_t flags = 0;
	if (nnz > 0) {
		size_t op_bytes = 0;
		W->h_op = ew_host_operand(operand, operand_type,
					  is_math ? 0 : operand_len, out_type,
					  &op_bytes);
		if (W->h_op == NULL) {
			svtgpu_set_error("svtgpu_ewise: out of host memory");
			return SVTGPU_ERR_NOMEM;
		}
		SVT_CUDA(svt_malloc_async(&W->d_aux, 16 + op_bytes, s));
		uint32_t *d_flags = (uint32_t *) W->d_aux;
		void *d_v = (char *) W->d_aux + 16;
		SVT_CUDA(cudaMemsetAsync(d_flags, 0, 16, s));
		SVT_CUDA(cudaMemcpyAsync(d_v, W->h_op, op_bytes,
					 cudaMemcpyHostToDevice, s));
		EwParams P;
		P.leaf_ptr = x->d_leaf_ptr;
		P.offs = x->d_offs;
		P.vals = x->d_vals;
		P.out_offs = m1->d_offs;
		P.out_vals = m1->d_vals;
		P.v = d_v;
		P.nnz = nnz;
		P.nleaf = x->nleaf;
		P.op = op;
		P.flags = d_flags;
		const int in = ((x->flags & SVTGPU_HAS_VALS) && x->d_vals != NULL)
			? (svt_is_double(x->val_type) ? EW_IN_DBL : EW_IN_INT)
			: EW_IN_ONES;
		const int64_t ntiles = (nnz + EW_TILE - 1) / EW_TILE;
		if (in == EW_IN_DBL)
			launch_map<EW_IN_DBL, double>(margin, ntiles, s, P);
		else if (in == EW_IN_INT && dbl)
			launch_map<EW_IN_INT, double>(margin, ntiles, s, P);
		else if (in == EW_IN_INT)
			launch_map<EW_IN_INT, int32_t>(margin, ntiles, s, P);
		else if (dbl)
			launch_map<EW_IN_ONES, double>(margin, ntiles, s, P);
		else
			launch_map<EW_IN_ONES, int32_t>(margin, ntiles, s, P);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		launches++;
		SVT_CUDA(cudaMemcpyAsync(&flags, d_flags, sizeof(flags),
					 cudaMemcpyDeviceToHost, s));
		SVT_CUDA(cudaStreamSynchronize(s));
	}
	svtgpu_matrix *res = m1;
	if (flags & SVT_EW_DROPPED) {
		const int64_t nleaf = x->nleaf;
		const unsigned grid = (unsigned) (svtgpu_sm_count() * 8);
		SVT_CUDA(svt_malloc_async((void **) &W->d_counts,
					 sizeof(int64_t) * (size_t) (2 * nleaf + 1),
					 s));
		int64_t *d_counts = W->d_counts, *d_ptr = W->d_counts + nleaf;
		uint32_t *d_flags = (uint32_t *) W->d_aux;
		KeepNonzero<double> kd = { (const double *) m1->d_vals };
		KeepNonzero<int32_t> ki = { (const int32_t *) m1->d_vals };
		if (dbl)
			ewise_count_kept<<<grid, 256, 0, s>>>(m1->d_leaf_ptr,
				nleaf, kd, d_counts, d_flags);
		else
			ewise_count_kept<<<grid, 256, 0, s>>>(m1->d_leaf_ptr,
				nleaf, ki, d_counts, d_flags);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		SVT_CHECK(svtgpu_exclusive_scan(d_counts, nleaf, d_ptr, s));
		launches += 3;      /* the scan counts its own two */
		int64_t nnz_new = 0;
		SVT_CUDA(cudaMemcpyAsync(&nnz_new, d_ptr + nleaf, sizeof(int64_t),
					 cudaMemcpyDeviceToHost, s));
		SVT_CUDA(cudaStreamSynchronize(s));
		SVT_CHECK(svtgpu_matrix_create(&W->m2, x->nrow, nleaf, nnz_new,
			out_type, nnz_new > 0 ? (SVTGPU_HAS_OFFS | SVTGPU_HAS_VALS)
					      : 0));
		svtgpu_matrix *m2 = W->m2;
		SVT_CUDA(cudaStreamSynchronize(m2->up_stream));
		SVT_CUDA(cudaMemcpyAsync(m2->d_leaf_ptr, d_ptr,
					 sizeof(int64_t) * (size_t) (nleaf + 1),
					 cudaMemcpyDeviceToDevice, s));
		if (nnz_new > 0) {
			if (dbl)
				ewise_compact<<<grid, 256, 0, s>>>(
					m1->d_leaf_ptr, d_ptr, m1->d_offs, kd,
					m2->d_offs, (double *) m2->d_vals, nleaf);
			else
				ewise_compact<<<grid, 256, 0, s>>>(
					m1->d_leaf_ptr, d_ptr, m1->d_offs, ki,
					m2->d_offs, (int32_t *) m2->d_vals, nleaf);
			SVT_CUDA(cudaGetLastError());
			svtgpu_count_launch(1);
			launches++;
		}
		res = m2;
	}
	double ms = 0.0;
	SVT_CHECK(svt_timer_end(&tm, &ms));
	if (res == W->m2) {
		svtgpu_matrix_free(W->m1);
		W->m1 = NULL;
		W->m2 = NULL;
	} else {
		W->m1 = NULL;
	}
	res->leaf_base = x->leaf_base;
	res->tm.kernel_ms = ms;
	res->tm.launches = launches;
	*out = res;
	if (warn != NULL)
		*warn = (int) (flags & (SVTGPU_EW_WARN_INT_OVERFLOW |
					SVTGPU_EW_WARN_NAN));
	return SVTGPU_OK;
}

/* ---- comparisons and is.* predicates: a filter of x's entries ----
 * Count pass (rule KeepCmp) -> flags; then
 *   nothing dropped, no NA: leaf_ptr and offsets copied, no value array;
 *   otherwise scan + write pass, values (1 / NA) only when an NA was kept.
 * A lacunar x under a scalar operand (and is.nan / is.infinite of integer
 * values) needs no pass at all: the predicate is a constant. */
template <int IN, int MARGIN>
static void cmp_launch(const svtgpu_matrix *x, int op, const double *d_v,
		       double v0, bool write, const int64_t *d_ptr,
		       svtgpu_matrix *m, int64_t *d_counts, uint32_t *d_flags,
		       unsigned grid, cudaStream_t s)
{
	KeepCmp<IN, MARGIN> k;
	k.offs = x->d_offs;
	k.vals = x->d_vals;
	k.v = d_v;
	k.v0 = v0;
	k.op = op;
	if (!write)
		ewise_count_kept<<<grid, 256, 0, s>>>(x->d_leaf_ptr, x->nleaf, k,
						      d_counts, d_flags);
	else
		ewise_compact<<<grid, 256, 0, s>>>(x->d_leaf_ptr, d_ptr,
			x->d_offs, k, m->d_offs,
			(m->flags & SVTGPU_HAS_VALS) ? (int32_t *) m->d_vals : NULL,
			x->nleaf);
}

template <int IN>
static void cmp_launch_m(int margin, const svtgpu_matrix *x, int op,
			 const double *d_v, double v0, bool write,
			 const int64_t *d_ptr, svtgpu_matrix *m,
			 int64_t *d_counts, uint32_t *d_flags, unsigned grid,
			 cudaStream_t s)
{
	if (margin == 0)
		cmp_launch<IN, 0>(x, op, d_v, v0, write, d_ptr, m, d_counts,
				  d_flags, grid, s);
	else if (margin == 1)
		cmp_launch<IN, 1>(x, op, d_v, v0, write, d_ptr, m, d_counts,
				  d_flags, grid, s);
	else
		cmp_launch<IN, 2>(x, op, d_v, v0, write, d_ptr, m, d_counts,
				  d_flags, grid, s);
}

/* a logical result of x's geometry: leaf_ptr and offsets copied from x
   (everything kept), or nnz = 0 (nothing kept) */
static int cmp_result_copy(svtgpu_matrix *x, bool keep_all, EwWork *W,
			   cudaStream_t s)
{
	const int64_t nnz = keep_all ? x->nnz : 0;
	SVT_CHECK(svtgpu_matrix_create(&W->m2, x->nrow, x->nleaf, nnz,
				       SVTGPU_LGL, nnz > 0 ? SVTGPU_HAS_OFFS : 0));
	svtgpu_matrix *m = W->m2;
	SVT_CUDA(cudaStreamSynchronize(m->up_stream));
	const size_t lp_bytes = sizeof(int64_t) * (size_t) (x->nleaf + 1);
	if (keep_all)
		SVT_CUDA(cudaMemcpyAsync(m->d_leaf_ptr, x->d_leaf_ptr, lp_bytes,
					 cudaMemcpyDeviceToDevice, s));
	else
		SVT_CUDA(cudaMemsetAsync(m->d_leaf_ptr, 0, lp_bytes, s));
	if (nnz > 0)
		SVT_CUDA(cudaMemcpyAsync(m->d_offs, x->d_offs,
					 sizeof(int32_t) * (size_t) nnz,
					 cudaMemcpyDeviceToDevice, s));
	return SVTGPU_OK;
}

static int compare_run(svtgpu_matrix *x, int op, const void *operand,
		       int operand_type, int64_t operand_len, int margin,
		       EwWork *W, svtgpu_matrix **out)
{
	cudaStream_t s = 0;
	const int64_t nnz = x->nnz, nleaf = x->nleaf;
	const int in = ((x->flags & SVTGPU_HAS_VALS) && x->d_vals != NULL)
		? (svt_is_double(x->val_type) ? EW_IN_DBL : EW_IN_INT)
		: EW_IN_ONES;
	const int64_t vlen = svt_ew_is_pred(op) ? 0 : operand_len;
	size_t op_bytes = 0;
	W->h_op = ew_host_operand(operand, operand_type, vlen, SVTGPU_DOUBLE,
				  &op_bytes);
	if (W->h_op == NULL) {
		svtgpu_set_error("svtgpu_ewise: out of host memory");
		return SVTGPU_ERR_NOMEM;
	}
	const double v0 = ((const double *) W->h_op)[0];
	/* a constant predicate: every entry of x gives the same answer */
	int konst = -1;
	if (in == EW_IN_ONES && (margin == 0 || svt_ew_is_pred(op)))
		konst = svt_ew_cmp(op, 1.0, 0, v0);
	else if (in == EW_IN_INT && (op == SVTGPU_EW_IS_NAN ||
				     op == SVTGPU_EW_IS_INFINITE))
		konst = SVT_CMP_DROP;
	if (nnz == 0)
		konst = SVT_CMP_TRUE;
	SvtTimer tm;
	SVT_CHECK(svt_timer_begin(&tm, s));
	int launches = 0;
	if (konst >= 0) {
		SVT_CHECK(cmp_result_copy(x, konst != SVT_CMP_DROP, W, s));
	} else {
		const unsigned grid = (unsigned) (svtgpu_sm_count() * 8);
		SVT_CUDA(svt_malloc_async(&W->d_aux, 16 + op_bytes, s));
		uint32_t *d_flags = (uint32_t *) W->d_aux;
		double *d_v = (double *) ((char *) W->d_aux + 16);
		SVT_CUDA(cudaMemsetAsync(d_flags, 0, 16, s));
		SVT_CUDA(cudaMemcpyAsync(d_v, W->h_op, op_bytes,
					 cudaMemcpyHostToDevice, s));
		SVT_CUDA(svt_malloc_async((void **) &W->d_counts,
					 sizeof(int64_t) * (size_t) (2 * nleaf + 1),
					 s));
		int64_t *d_counts = W->d_counts, *d_ptr = W->d_counts + nleaf;
		if (in == EW_IN_DBL)
			cmp_launch_m<EW_IN_DBL>(margin, x, op, d_v, v0, false, NULL,
						NULL, d_counts, d_flags, grid, s);
		else if (in == EW_IN_INT)
			cmp_launch_m<EW_IN_INT>(margin, x, op, d_v, v0, false, NULL,
						NULL, d_counts, d_flags, grid, s);
		else
			cmp_launch_m<EW_IN_ONES>(margin, x, op, d_v, v0, false,
						 NULL, NULL, d_counts, d_flags,
						 grid, s);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		launches++;
		uint32_t flags = 0;
		SVT_CUDA(cudaMemcpyAsync(&flags, d_flags, sizeof(flags),
					 cudaMemcpyDeviceToHost, s));
		SVT_CUDA(cudaStreamSynchronize(s));
		if (!(flags & (SVT_EW_DROPPED | SVT_EW_NA_KEPT))) {
			SVT_CHECK(cmp_result_copy(x, true, W, s));
		} else {
			SVT_CHECK(svtgpu_exclusive_scan(d_counts, nleaf, d_ptr, s));
			launches += 2;
			int64_t nnz_new = 0;
			SVT_CUDA(cudaMemcpyAsync(&nnz_new, d_ptr + nleaf,
						 sizeof(int64_t),
						 cudaMemcpyDeviceToHost, s));
			SVT_CUDA(cudaStreamSynchronize(s));
			const int fl = nnz_new == 0 ? 0 : SVTGPU_HAS_OFFS |
				((flags & SVT_EW_NA_KEPT) ? SVTGPU_HAS_VALS : 0);
			SVT_CHECK(svtgpu_matrix_create(&W->m2, x->nrow, nleaf,
						       nnz_new, SVTGPU_LGL, fl));
			svtgpu_matrix *m = W->m2;
			SVT_CUDA(cudaStreamSynchronize(m->up_stream));
			SVT_CUDA(cudaMemcpyAsync(m->d_leaf_ptr, d_ptr,
						 sizeof(int64_t) * (size_t) (nleaf + 1),
						 cudaMemcpyDeviceToDevice, s));
			if (nnz_new > 0) {
				if (in == EW_IN_DBL)
					cmp_launch_m<EW_IN_DBL>(margin, x, op, d_v,
						v0, true, d_ptr, m, NULL, NULL, grid, s);
				else if (in == EW_IN_INT)
					cmp_launch_m<EW_IN_INT>(margin, x, op, d_v,
						v0, true, d_ptr, m, NULL, NULL, grid, s);
				else
					cmp_launch_m<EW_IN_ONES>(margin, x, op, d_v,
						v0, true, d_ptr, m, NULL, NULL, grid, s);
				SVT_CUDA(cudaGetLastError());
				svtgpu_count_launch(1);
				launches++;
			}
		}
	}
	double ms = 0.0;
	SVT_CHECK(svt_timer_end(&tm, &ms));
	svtgpu_matrix *res = W->m2;
	W->m2 = NULL;
	res->leaf_base = x->leaf_base;
	res->tm.kernel_ms = ms;
	res->tm.launches = launches;
	*out = res;
	return SVTGPU_OK;
}

extern "C" int svtgpu_ewise(svtgpu_matrix *x, int op, const void *operand,
			    int operand_type, int64_t operand_len, int margin,
			    int operand_on_left, svtgpu_matrix **out, int *warn)
{
	SVT_ARG(x != NULL && out != NULL, "svtgpu_ewise: NULL argument");
	*out = NULL;
	if (warn != NULL)
		*warn = 0;
	const int is_math = svt_ew_is_math(op);
	SVT_ARG(svt_ew_is_unary(op) || operand != NULL || operand_len == 0,
		"svtgpu_ewise: NULL operand");
	int64_t bad = -1;
	const int code = svt_ew_check(op, x->val_type, operand_type,
				      operand_len, margin, operand_on_left, 2,
				      x->nrow, x->nleaf, operand, &bad);
	if (code != SVT_EW_OK) {
		char msg[512];
		const int kind = is_math ? SVT_EW_KIND_MATH
			: svt_ew_is_compare(op) ? SVT_EW_KIND_COMPARE
			: svt_ew_is_pred(op) ? SVT_EW_KIND_IS : SVT_EW_KIND_ARITH;
		svt_ew_refusal_message(code, svt_ew_opname(op), kind, op,
				       operand_type, operand, operand_len,
				       margin, x->nrow, x->nleaf, bad, msg,
				       sizeof(msg));
		svtgpu_set_error("%s", msg);
		return SVTGPU_ERR_ARG;
	}
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(x->nnz == 0 || (x->flags & SVTGPU_HAS_OFFS),
		"svtgpu_ewise: the matrix was uploaded without row offsets");
	SVT_ARG(((uintptr_t) x->d_offs & 15) == 0 &&
		((uintptr_t) x->d_vals & 15) == 0,
		"svtgpu_ewise: the device arrays must be 16-byte aligned");
	SVT_CHECK(svtgpu_matrix_finish_upload(x));
	const int out_type = svt_ew_result_type(op, x->val_type, operand_type);
	EwWork W;
	memset(&W, 0, sizeof(W));
	const int rc = out_type == SVTGPU_LGL
		? compare_run(x, operand_on_left ? svt_ew_mirror(op) : op,
			      operand, operand_type, operand_len, margin, &W, out)
		: ewise_run(x, op, operand, operand_type, operand_len, margin,
			    out_type, &W, out, warn);
	if (W.d_aux != NULL)
		svt_free_async(W.d_aux, 0);
	if (W.d_counts != NULL)
		svt_free_async(W.d_counts, 0);
	free(W.h_op);
	if (rc != SVTGPU_OK) {
		cudaDeviceSynchronize();
		svtgpu_matrix_free(W.m1);
		svtgpu_matrix_free(W.m2);
		*out = NULL;
	}
	return rc;
}
