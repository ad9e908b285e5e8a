/* Column statistics of a device CSC: one result per segment (a leaf, or
 * `group` consecutive leaves) -- the replacement for REC_colStats_SVT() ->
 * _summarize_SVT() (src/SparseArray_matrixStats.c:200-231,
 * src/SparseArray_summarization.c:89-109) and the per-type loops of
 * src/Rvector_summarization.c.
 *
 * HBM-bound streaming reduction: each stored value is read exactly once
 * (row offsets are never read; lacunar matrices read only leaf_ptr).
 *
 *   colstats_tma      warp-specialised: every CTA holds NW producer/consumer
 *                     warp pairs.  A producer lane walks the leaves assigned
 *                     to its pair and streams each leaf (16-byte aligned
 *                     chunks of at most `stage_bytes`) into a 2-deep shared
 *                     memory ring with 1-D bulk async copies (TMA) that
 *                     complete on an mbarrier; the consumer warp reduces the
 *                     chunk out of shared memory with 16-byte loads and warp
 *                     shuffles.  The two-pass variance reads a leaf from HBM
 *                     once: when the leaf fits one stage, the second pass
 *                     runs over the copy already in shared memory.
 *   colstats_direct   warp per segment with plain coalesced loads; used for
 *                     value arrays that are not 16-byte aligned and as a
 *                     cross-check (SVTGPU_COLSTATS_IMPL=direct).
 *   colstats_lacunar  thread per segment: a lacunar leaf is summarised from
 *                     its length alone (summarize_ones(),
 *                     src/Rvector_summarization.c:742-825).
 *
 * Integer leaves are summed in int64 (exact), converted to double once; the
 * reference accumulates int -> double (sum_ints(), :518-537), which is
 * identical while partial sums stay below 2^53.
 */
#include "svtgpu_internal.h"
#include "svt_ptx.cuh"

#include <stdlib.h>
#include <string.h>

namespace {

enum ColClass { CC_COUNT = 0, CC_SUM, CC_MINMAX, CC_VAR, CC_ANYALL, CC_PROD };

__host__ __device__ inline int col_class_of(int opcode)
{
	switch (opcode) {
	    case SVTGPU_OP_ANYNA: case SVTGPU_OP_COUNTNAS: return CC_COUNT;
	    case SVTGPU_OP_SUM: case SVTGPU_OP_MEAN:       return CC_SUM;
	    case SVTGPU_OP_MIN: case SVTGPU_OP_MAX:        return CC_MINMAX;
	    case SVTGPU_OP_CENTERED_X2_SUM:
	    case SVTGPU_OP_VAR1: case SVTGPU_OP_SD1:       return CC_VAR;
	    case SVTGPU_OP_ANY: case SVTGPU_OP_ALL:        return CC_ANYALL;
	    case SVTGPU_OP_PROD:                           return CC_PROD;
	}
	return -1;
}

struct ColParams {
	const void *vals;
	const int64_t *leaf_ptr;
	int64_t nseg;
	int64_t group;
	int64_t seg_len;     /* nrow * group: length of the summarised vector */
	int opcode;
	int narm;
	int is_double;
	double center;
	void *out;
	int32_t *warn;
	int var_small;       /* int CC_VAR: 32-bit lane sums cannot overflow */
	int var_onepass;     /* double CC_VAR: sparse segments finish from S1, S2 */
};

/* Per-lane running state over the values a lane has seen (pass 1). */
template <int CC, typename T>
struct LaneAcc {
	long long isum;      /* int input: exact sum of non-NA values */
	double dsum;         /* double input: sum of regular values */
	double dsum2;        /* double input, CC_VAR: sum of their squares */
	double prod;
	double vmin, vmax;
	int imin, imax;      /* int input: min / max over non-NA values */
	unsigned long long isum2;   /* int input, CC_VAR: exact sum of squares */
	int n_na, n_nan, n_zero, n_reg;

	__device__ __forceinline__ void reset()
	{
		isum = 0; dsum = 0.0; dsum2 = 0.0; prod = 1.0;
		vmin = svt_posinf(); vmax = svt_neginf();
		imin = INT32_MAX; imax = INT32_MIN;
		isum2 = 0;
		n_na = n_nan = n_zero = n_reg = 0;
	}

	__device__ __forceinline__ void add(int32_t x)
	{
		const bool na = x == SVT_NA_INT;
		n_na += na;
		if (CC == CC_SUM || CC == CC_VAR)
			isum += na ? 0 : x;
		if (CC == CC_VAR) {
			/* |x| is tracked too: squares are exact in 64 bits
			   while |x| < 65536 (checked by the caller) */
			const int ax = na ? 0 : (x < 0 ? -x : x);
			imax = ax > imax ? ax : imax;
			isum2 += (unsigned long long) ((long long) ax * ax);
		}
		if (CC == CC_MINMAX) {
			/* NA = INT_MIN never raises the max; keep it out of
			   the min */
			imax = x > imax ? x : imax;
			const int xm = na ? INT32_MAX : x;
			imin = xm < imin ? xm : imin;
			n_reg += !na;
		}
		if (CC == CC_ANYALL)
			n_zero += x == 0;
		if (CC == CC_PROD && !na)
			prod *= (double) x;
	}

	__device__ __forceinline__ void add(double x)
	{
		if (svt_isnan(x)) {
			if ((uint32_t) svt_d2u(x) == 1954u) n_na++;
			else                                n_nan++;
			return;
		}
		if (CC == CC_SUM || CC == CC_VAR)
			dsum += x;
		if (CC == CC_VAR)
			dsum2 = fma(x, x, dsum2);
		if (CC == CC_MINMAX) {
			vmin = x < vmin ? x : vmin;
			vmax = x > vmax ? x : vmax;
		}
		if (CC == CC_PROD)
			prod *= x;
	}

	/* all lanes end up with the warp-wide partial */
	__device__ __forceinline__ void reduce_into(SvtColPartial *p,
						    int64_t nz) const
	{
		svt_col_partial_init(p);
		p->nz = nz;
		p->n_na = svt_warp_sum((long long) n_na);
		p->n_nan = svt_warp_sum((long long) n_nan);
		if (CC == CC_SUM || CC == CC_VAR) {
			if (sizeof(T) == 4)
				p->sum = (double) svt_warp_sum(isum);
			else
				p->sum = svt_warp_sum(dsum);
		}
		if (CC == CC_MINMAX) {
			if (sizeof(T) == 4) {
				int lo = imin, hi = imax;
				long long nr = n_reg;
#pragma unroll
				for (int m = 16; m > 0; m >>= 1) {
					const int ol = __shfl_xor_sync(
						SVT_FULL_MASK, lo, m);
					const int oh = __shfl_xor_sync(
						SVT_FULL_MASK, hi, m);
					lo = ol < lo ? ol : lo;
					hi = oh > hi ? oh : hi;
				}
				nr = svt_warp_sum(nr);
				p->vmin = nr > 0 ? (double) lo : svt_posinf();
				p->vmax = nr > 0 ? (double) hi : svt_neginf();
			} else {
				p->vmin = svt_warp_min(vmin);
				p->vmax = svt_warp_max(vmax);
			}
		}
		if (CC == CC_ANYALL)
			p->n_zero = svt_warp_sum((long long) n_zero);
		if (CC == CC_PROD)
			p->prod = svt_warp_prod(prod);
	}
};

/* pass 2 of the variance: (x - center)^2 over regular values */
__device__ __forceinline__ void add_sq(double &acc, int32_t x, double c)
{
	if (x != SVT_NA_INT) {
		double d = (double) x - c;
		acc += d * d;
	}
}

__device__ __forceinline__ void add_sq(double &acc, double x, double c)
{
	if (!svt_isnan(x)) {
		double d = x - c;
		acc += d * d;
	}
}

template <typename T> struct Vec16;
template <> struct Vec16<int32_t> {
	static constexpr int N = 4;
	int4 v;
	__device__ __forceinline__ int32_t get(int i) const
	{
		return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
	}
};
template <> struct Vec16<double> {
	static constexpr int N = 2;
	double2 v;
	__device__ __forceinline__ double get(int i) const
	{
		return i == 0 ? v.x : v.y;
	}
};

__device__ __forceinline__ void store_result(const ColParams &P, int64_t seg,
					     const SvtScalar &r)
{
	if (svt_col_out_is_int(P.opcode, P.is_double ? SVTGPU_DOUBLE
						     : SVTGPU_INT))
		((int32_t *) P.out)[seg] = r.i;
	else
		((double *) P.out)[seg] = r.d;
	if (r.warn && P.warn != NULL)
		atomicOr((int *) P.warn, 1);
}

/* centered_X2_sum / var1 / sd1 of an integer segment from its exact sums
 * (centre = the mean): the NA rules of svt_col_finalize(), the arithmetic in
 * 128-bit integers with a single rounding at the end. */
__host__ __device__ __forceinline__ SvtScalar var_from_int_sums(int opcode, int narm,
		int64_t in_length, const SvtColPartial *p,
		unsigned long long sum2)
{
	SvtScalar r;
	r.d = 0.0; r.i = 0; r.warn = 0;
	if (!narm && p->n_na > 0) {
		r.d = svt_na_real();
		return r;
	}
	const int64_t n = in_length - (narm ? p->n_na : 0);
	if (n <= 0) {
		/* mean = 0 / 0: NaN propagates as in the reference */
		r.d = opcode == SVTGPU_OP_CENTERED_X2_SUM ? svt_nan()
							  : svt_na_real();
		return r;
	}
	const __int128 s1 = (__int128) (long long) p->sum;   /* exact < 2^53 */
	const __int128 D = (__int128) n * (__int128) sum2 - s1 * s1;
	const double x2 = (double) D / (double) n;
	if (opcode == SVTGPU_OP_CENTERED_X2_SUM) {
		r.d = x2;
		return r;
	}
	if (n <= 1) {
		r.d = svt_na_real();
		return r;
	}
	double v = (double) D / ((double) n * (double) (n - 1));
	if (opcode == SVTGPU_OP_SD1)
		v = sqrt(v);
	r.d = v;
	return r;
}

#ifndef COL_INT_VEC
#define COL_INT_VEC 1
#endif

/* lane's share of [start, end): p[0], p[32], ... fed to the accumulator with
   eight loads in flight (immediate offsets, 32-bit trip count) */
template <int CC, typename T>
__device__ __forceinline__ void lane_accumulate(LaneAcc<CC, T> &acc,
		const T *__restrict__ vals, int64_t start, int64_t end, int lane)
{
	if (sizeof(T) == 4 && COL_INT_VEC && (((uintptr_t) vals) & 15) == 0) {
		/* 16-byte loads over the aligned middle of the segment, the
		   < 4 (< 2) entries at either end by single lanes: a read-only
		   stream of 4-byte loads tops out near 6.3 TB/s on B200, 8-
		   and 16-byte ones reach 7.2 (microbench/stream_width.cu);
		   colSums 1.51 -> 1.39 ms per 2.3e9 int32 values.  (Doubles:
		   16-byte loads measured SLOWER than the 8-byte loop below,
		   2.75 -> 3.3 ms; so did the packed integer variance.) */
		constexpr int VN = Vec16<T>::N;
		const int64_t a4 = (start + VN - 1) & ~(int64_t) (VN - 1);
		const int64_t b4 = end & ~(int64_t) (VN - 1);
		if (a4 < b4) {
			if (start + lane < a4)
				acc.add(vals[start + lane]);
			if (b4 + lane < end)
				acc.add(vals[b4 + lane]);
			const Vec16<T> *q = (const Vec16<T> *) (vals + a4) + lane;
			const int nv = (int) ((b4 - a4) / VN);   /* vectors */
			int i = lane;
			for (; i + 32 < nv; i += 64) {
				const Vec16<T> u = q[i - lane];
				const Vec16<T> w = q[i - lane + 32];
#pragma unroll
				for (int k = 0; k < VN; k++)
					acc.add(u.get(k));
#pragma unroll
				for (int k = 0; k < VN; k++)
					acc.add(w.get(k));
			}
			if (i < nv) {
				const Vec16<T> u = q[i - lane];
#pragma unroll
				for (int k = 0; k < VN; k++)
					acc.add(u.get(k));
			}
			return;
		}
	}
	const T *p = vals + start + lane;
	const int64_t left = end - start - lane;
	const int n = left > 0 ? (int) ((left + 31) >> 5) : 0;
	int i = 0;
	for (; i + 8 <= n; i += 8) {
		T x[8];
#pragma unroll
		for (int k = 0; k < 8; k++)
			x[k] = p[(i + k) * 32];
#pragma unroll
		for (int k = 0; k < 8; k++)
			acc.add(x[k]);
	}
	if (sizeof(T) == 4) {
		/* (int32: the 32-register kernel with 64 warps per SM hides
		   these round trips; the batched form below costs it registers
		   and 10-30 %, measured) */
		for (; i < n; i++)
			acc.add(p[i * 32]);
	} else if (i < n) {
		/* the last < 8 values: all loads in flight at once (one at a
		   time they cost the warp up to seven round trips per leaf) */
		T x[8];
#pragma unroll
		for (int k = 0; k < 8; k++)
			if (i + k < n)
				x[k] = p[(i + k) * 32];
#pragma unroll
		for (int k = 0; k < 8; k++)
			if (i + k < n)
				acc.add(x[k]);
	}
}

/* ------------------------------------------------------------------------
 * colstats_direct
 */
template <int CC, typename T>
__global__ void __launch_bounds__(256, sizeof(T) == 8 ? 4
		: (CC == CC_VAR || CC == CC_PROD) ? 5 : 8)
colstats_direct(ColParams P)
{
	const int lane = threadIdx.x & 31;
	const int64_t warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const T *vals = (const T *) P.vals;

	/* doubles: the bounds of a segment are requested one segment ahead
	   (int32 input: not worth the four registers, see lane_accumulate) */
	constexpr bool AHEAD = sizeof(T) == 8;
	int64_t nstart = 0, nend = 0;
	if (AHEAD && gw < P.nseg) {
		nstart = P.leaf_ptr[gw * P.group];
		nend = P.leaf_ptr[(gw + 1) * P.group];
	}
	for (int64_t seg = gw; seg < P.nseg; seg += warps) {
		const int64_t start = AHEAD ? nstart : P.leaf_ptr[seg * P.group];
		const int64_t end = AHEAD ? nend
					  : P.leaf_ptr[(seg + 1) * P.group];
		if (AHEAD && seg + warps < P.nseg) {
			nstart = P.leaf_ptr[(seg + warps) * P.group];
			nend = P.leaf_ptr[(seg + warps + 1) * P.group];
		}
		if (CC == CC_VAR && sizeof(T) == 4 && P.var_small) {
			/* integer input, centre = the mean, and the host knows
			   a bound of |x| under which a lane's sum and sum of
			   squares over one segment fit 32 bits: the exact
			   one-pass form below with a third of the integer
			   instructions */
			int s1 = 0, nna = 0;
			unsigned int s2 = 0;
			/* this lane's values: p[0], p[32], ... (n of them) */
			const T *p = vals + start + lane;
			const int64_t left = end - start - lane;
			const int n = left > 0 ? (int) ((left + 31) >> 5) : 0;
			int i = 0;
			if (P.var_small == 2) {
				/* no negative value in the matrix: NA = 0x80000000
				   is the only value with the top bit set.  Summed
				   as UNSIGNED 64-bit, the regular values stay
				   below 2^31 (the bound above), so the total is
				   #NA * 2^31 + sum; and NA * NA = 2^62 = 0 mod 2^32
				   leaves the sum of squares alone: three integer
				   instructions per value instead of five */
				unsigned long long w = 0;
				for (; i + 8 <= n; i += 8) {
					unsigned int x[8];
#pragma unroll
					for (int k = 0; k < 8; k++)
						x[k] = (unsigned int) p[(i + k) * 32];
#pragma unroll
					for (int k = 0; k < 8; k++) {
						w += x[k];
						s2 += x[k] * x[k];
					}
				}
				for (; i < n; i++) {
					const unsigned int x = (unsigned int) p[i * 32];
					w += x;
					s2 += x * x;
				}
				nna = (int) (w >> 31);
				s1 = (int) (w & 0x7FFFFFFFull);
			}
			for (; i + 8 <= n; i += 8) {
				int x[8];
#pragma unroll
				for (int k = 0; k < 8; k++)
					x[k] = (int) p[(i + k) * 32];
#pragma unroll
				for (int k = 0; k < 8; k++) {
					const bool na = x[k] == SVT_NA_INT;
					const int x0 = na ? 0 : x[k];
					nna += na;
					s1 += x0;
					s2 += (unsigned int) (x0 * x0);
				}
			}
			for (; i < n; i++) {
				const int x = (int) p[i * 32];
				const bool na = x == SVT_NA_INT;
				const int x0 = na ? 0 : x;
				nna += na;
				s1 += x0;
				s2 += (unsigned int) (x0 * x0);
			}
			SvtColPartial sp;
			svt_col_partial_init(&sp);
			sp.nz = end - start;
			sp.n_na = svt_warp_sum((long long) nna);
			sp.sum = (double) svt_warp_sum((long long) s1);
			unsigned long long t2 = s2;
#pragma unroll
			for (int m = 16; m > 0; m >>= 1)
				t2 += __shfl_xor_sync(SVT_FULL_MASK, t2, m);
			if (lane == 0)
				store_result(P, seg, var_from_int_sums(P.opcode,
						P.narm, P.seg_len, &sp, t2));
			continue;
		}
		LaneAcc<CC, T> acc;
		acc.reset();
		lane_accumulate<CC, T>(acc, vals, start, end, lane);
		SvtColPartial part;
		acc.reduce_into(&part, end - start);
		double center = P.center;
		if (CC == CC_VAR && sizeof(T) == 4 && svt_isnan(center)) {
			/* integer input, centre = the mean: one pass.  With the
			   exact integer sums S1 = sum x, S2 = sum x^2 over the
			   n_reg regular values and n = seg_len - #NA(na.rm),
			   sum (x - mean)^2 + mean^2 * #zeros = (n S2 - S1^2) / n
			   (src/SparseArray_summarization.c:70-102 computes the
			   left-hand side in two floating-point passes). */
			int amax = acc.imax;
			unsigned long long s2 = acc.isum2;
#pragma unroll
			for (int m = 16; m > 0; m >>= 1) {
				const int o = __shfl_xor_sync(SVT_FULL_MASK,
							      amax, m);
				amax = o > amax ? o : amax;
				s2 += __shfl_xor_sync(SVT_FULL_MASK, s2, m);
			}
			if (amax < 65536) {
				if (lane == 0)
					store_result(P, seg, var_from_int_sums(
						P.opcode, P.narm, P.seg_len,
						&part, s2));
				continue;
			}
			/* huge values: fall through to the two-pass form */
		}
		if (CC == CC_VAR) {
			const bool about_mean = svt_isnan(center);
			if (about_mean)
				center = svt_col_mean(P.is_double, P.narm,
						      P.seg_len, &part);
			bool one_pass = false;
			if (sizeof(T) == 8 && about_mean && P.var_onepass) {
				/* double input, centre = the mean, sparse segment:
				   sum (x - c)^2 = S2 - 2 c S1 + n_reg c^2 from the
				   sums of pass 1.  With rho = n_reg / n <= 1/4,
				   S1^2 <= n_reg S2 bounds every subtracted term by
				   rho S2, so what is left is >= (1 - rho)^2 S2 and
				   the cancellation costs a factor <= 2.1 on the
				   (tree-summed) rounding errors of S1, S2 -- no worse
				   than the sequential second pass of the reference
				   (src/SparseArray_summarization.c:89-102).  Dense
				   segments, and sums of squares near the ends of the
				   double range (Inf values, overflow, denormals), take
				   the second pass. */
				const double S2 = svt_warp_sum(acc.dsum2);
				const int64_t n_reg = part.nz - part.n_na - part.n_nan;
				const int64_t n = P.seg_len -
					(P.narm ? part.n_na + part.n_nan : 0);
				if (S2 >= 1e-200 && S2 <= 1e200 && n > 0 &&
				    4 * n_reg <= n && !svt_isnan(center)) {
					part.sum2 = S2 - 2.0 * center * part.sum +
						    (double) n_reg * center * center;
					one_pass = true;
				}
			}
			if (!one_pass) {
				double s2 = 0.0;
#pragma unroll 4
				for (int64_t e = start + lane; e < end; e += 32)
					add_sq(s2, vals[e], center);
				part.sum2 = svt_warp_sum(s2);
			}
		}
		if (lane == 0)
			store_result(P, seg, svt_col_finalize(P.opcode,
					P.is_double, P.narm, P.seg_len, center,
					&part));
	}
}

/* ------------------------------------------------------------------------
 * colstats_sum_i8: the integer SUM class (colSums, colMeans) over the compact
 * int8 values (svtgpu_internal.h).  A warp per segment, 16-byte loads over
 * the aligned middle with up to four per lane in flight, single bytes at the
 * ends.  Per 32-bit word __dp4a gives the signed byte sum, in which every NA
 * byte (-128) counts -128, and __vcmpeq4 marks the NA bytes (0xFF each), so
 * sum = dp4a + 128 #NA exactly: the partial equals the wide kernel's.
 */
__device__ __forceinline__ void sum_i8_word(uint32_t w, int &s, int &na_bits)
{
	s = __dp4a((int) w, 0x01010101, s);
	na_bits += __popc(__vcmpeq4(w, 0x80808080u));
}

#define SUM_I8_BLOCKS_PER_SM 6   /* 40 registers: four 16-byte loads in flight */
__global__ void __launch_bounds__(256, SUM_I8_BLOCKS_PER_SM)
colstats_sum_i8(ColParams P, const int8_t *__restrict__ v8)
{
	const int lane = threadIdx.x & 31;
	const int64_t warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	/* a C2 leaf is ~2.3 KB: its bounds are requested a segment ahead */
	int64_t nstart = 0, nend = 0;
	if (gw < P.nseg) {
		nstart = P.leaf_ptr[gw * P.group];
		nend = P.leaf_ptr[(gw + 1) * P.group];
	}
	for (int64_t seg = gw; seg < P.nseg; seg += warps) {
		const int64_t start = nstart, end = nend;
		if (seg + warps < P.nseg) {
			nstart = P.leaf_ptr[(seg + warps) * P.group];
			nend = P.leaf_ptr[(seg + warps + 1) * P.group];
		}
		long long sum = 0;
		int na_bits = 0;   /* 8 per NA */
		const int64_t a16 = (start + 15) & ~(int64_t) 15;
		const int64_t b16 = end & ~(int64_t) 15;
		int64_t lo = start, hi = end;   /* bytes left to single lanes */
		if (a16 < b16) {
			const uint4 *q = (const uint4 *) (v8 + a16);
			const int nv = (int) ((b16 - a16) >> 4);
			for (int i = lane; i < nv; i += 128) {
				uint4 u[4];
#pragma unroll
				for (int k = 0; k < 4; k++)
					u[k] = i + 32 * k < nv ? __ldcs(q + i + 32 * k)
							       : make_uint4(0, 0, 0, 0);
				int s = 0;
#pragma unroll
				for (int k = 0; k < 4; k++) {
					sum_i8_word(u[k].x, s, na_bits);
					sum_i8_word(u[k].y, s, na_bits);
					sum_i8_word(u[k].z, s, na_bits);
					sum_i8_word(u[k].w, s, na_bits);
				}
				sum += s;
			}
			/* < 16 bytes at either end */
			if (start + lane < a16) {
				const int x = v8[start + lane];
				sum += x;
				na_bits += x == SVT_COMPACT_NA_I8 ? 8 : 0;
			}
			lo = b16;
		}
		for (int64_t e = lo + lane; e < hi; e += 32) {
			const int x = v8[e];
			sum += x;
			na_bits += x == SVT_COMPACT_NA_I8 ? 8 : 0;
		}
		const long long n_na = svt_warp_sum((long long) na_bits) >> 3;
		sum = svt_warp_sum(sum) + 128 * n_na;
		if (lane == 0) {
			SvtColPartial part;
			svt_col_partial_init(&part);
			part.nz = end - start;
			part.n_na = n_na;
			part.sum = (double) sum;
			store_result(P, seg, svt_col_finalize(P.opcode, P.is_double,
					P.narm, P.seg_len, P.center, &part));
		}
	}
}

/* ------------------------------------------------------------------------
 * colstats_tma
 */

#define COL_NS 2   /* stages in each pair's ring */

enum {
	IT_FIRST = 1,    /* first item of its segment */
	IT_PASS_END = 2, /* last chunk of its pass */
	IT_PASS2 = 4,    /* chunk belongs to the second (centered) pass */
	IT_LAST = 8,     /* last item of its segment */
	IT_SINGLE = 16,  /* the segment is a single chunk: run pass 2 in place */
	IT_STOP = 32     /* no more work for this pair */
};

struct __align__(16) ItemMeta {
	int64_t seg;
	int64_t start, end;   /* element range of the segment */
	int64_t cbase;        /* element index held at byte 0 of the stage */
	int32_t celems;       /* elements held by the stage */
	int32_t flags;
};

template <int CC, typename T>
__device__ __forceinline__ void consume_pass1(LaneAcc<CC, T> &acc,
		const T *buf, int lo, int hi, int lane)
{
	constexpr int VN = Vec16<T>::N;
	const int lo_v = (lo + VN - 1) / VN * VN;
	const int hi_v = hi / VN * VN;
	if (lo_v >= hi_v) {
		for (int e = lo + lane; e < hi; e += 32)
			acc.add(buf[e]);
		return;
	}
	if (lo + lane < lo_v)
		acc.add(buf[lo + lane]);
	if (hi_v + lane < hi)
		acc.add(buf[hi_v + lane]);
	const Vec16<T> *vb = (const Vec16<T> *) buf;
#pragma unroll 2
	for (int v = lo_v / VN + lane; v < hi_v / VN; v += 32) {
		Vec16<T> x = vb[v];
#pragma unroll
		for (int i = 0; i < VN; i++)
			acc.add(x.get(i));
	}
}

template <typename T>
__device__ __forceinline__ void consume_pass2(double &s2, const T *buf,
		int lo, int hi, int lane, double c)
{
	constexpr int VN = Vec16<T>::N;
	const int lo_v = (lo + VN - 1) / VN * VN;
	const int hi_v = hi / VN * VN;
	if (lo_v >= hi_v) {
		for (int e = lo + lane; e < hi; e += 32)
			add_sq(s2, buf[e], c);
		return;
	}
	if (lo + lane < lo_v)
		add_sq(s2, buf[lo + lane], c);
	if (hi_v + lane < hi)
		add_sq(s2, buf[hi_v + lane], c);
	const Vec16<T> *vb = (const Vec16<T> *) buf;
#pragma unroll 2
	for (int v = lo_v / VN + lane; v < hi_v / VN; v += 32) {
		Vec16<T> x = vb[v];
#pragma unroll
		for (int i = 0; i < VN; i++)
			add_sq(s2, x.get(i), c);
	}
}

/* Shared memory: [pairs][COL_NS][stage_bytes] data, then ItemMeta
 * [pairs][COL_NS], then mbarriers full[pairs][COL_NS], empty[pairs][COL_NS]. */
template <int CC, typename T>
__global__ void __launch_bounds__(512, 1)
colstats_tma(ColParams P, int pairs, int stage_bytes)
{
	extern __shared__ __align__(128) unsigned char smem[];
	unsigned char *data = smem;
	ItemMeta *metas = (ItemMeta *) (smem + (size_t) pairs * COL_NS *
							 stage_bytes);
	uint64_t *bars = (uint64_t *) (metas + pairs * COL_NS);

	const int warp = threadIdx.x >> 5;
	const int lane = threadIdx.x & 31;
	const int pair = warp >> 1;
	const bool is_producer = (warp & 1) == 0;

	if (threadIdx.x == 0) {
		for (int i = 0; i < 2 * pairs * COL_NS; i++)
			svt_mbar_init(svt_smem_u32(&bars[i]), 1);
		svt_mbar_init_fence();
	}
	__syncthreads();

	unsigned char *ring = data + (size_t) pair * COL_NS * stage_bytes;
	ItemMeta *meta = metas + pair * COL_NS;
	const uint32_t full0 = svt_smem_u32(&bars[pair * COL_NS]);
	const uint32_t empty0 = svt_smem_u32(&bars[(pairs + pair) * COL_NS]);
	const int64_t npairs_total = (int64_t) gridDim.x * pairs;
	const int64_t gp = (int64_t) blockIdx.x * pairs + pair;
	constexpr int SZ = (int) sizeof(T);

	if (is_producer) {
		if (lane != 0)
			return;
		const char *vals = (const char *) P.vals;
		const uint64_t policy = svt_policy_evict_first();
		uint32_t it = 0;
		int64_t seg = gp;
		int64_t nstart = 0, nend = 0;
		if (seg < P.nseg) {
			nstart = P.leaf_ptr[seg * P.group];
			nend = P.leaf_ptr[(seg + 1) * P.group];
		}
		while (seg < P.nseg) {
			const int64_t start = nstart, end = nend;
			const int64_t next = seg + npairs_total;
			if (next < P.nseg) {   /* prefetch the next bounds */
				nstart = P.leaf_ptr[next * P.group];
				nend = P.leaf_ptr[(next + 1) * P.group];
			}
			const int64_t a0 = (start * SZ) & ~(int64_t) 15;
			const int64_t a1 = (end * SZ + 15) & ~(int64_t) 15;
			const int64_t nch = start == end ? 0
				: (a1 - a0 + stage_bytes - 1) / stage_bytes;
			const int npass = (CC == CC_VAR && nch > 1) ? 2 : 1;
			const int64_t nitems = nch == 0 ? 1 : nch * npass;
			int64_t k = 0;
			for (int pass = 0; pass < npass; pass++) {
			    for (int64_t ch = 0; ch < (nch == 0 ? 1 : nch);
				 ch++, k++) {
				const int st = it % COL_NS;
				svt_mbar_wait(empty0 + 8 * st,
					      ((it / COL_NS) & 1) ^ 1);
				const int64_t ca = a0 + ch * stage_bytes;
				int64_t cb = ca + stage_bytes;
				if (cb > a1) cb = a1;
				const uint32_t bytes = nch == 0 ? 0
						: (uint32_t) (cb - ca);
				ItemMeta md;
				md.seg = seg;
				md.start = start;
				md.end = end;
				md.cbase = ca / SZ;
				md.celems = (int32_t) (bytes / SZ);
				md.flags = (k == 0 ? IT_FIRST : 0) |
					(ch + 1 >= nch ? IT_PASS_END : 0) |
					(pass == 1 ? IT_PASS2 : 0) |
					(k + 1 == nitems ? IT_LAST : 0) |
					(nch <= 1 ? IT_SINGLE : 0);
				meta[st] = md;
				if (bytes == 0) {
					svt_mbar_arrive(full0 + 8 * st);
				} else {
					svt_mbar_arrive_expect_tx(
						full0 + 8 * st, bytes);
					svt_bulk_g2s_hint(svt_smem_u32(ring +
						(size_t) st * stage_bytes),
						vals + ca, bytes,
						full0 + 8 * st, policy);
				}
				it++;
			    }
			}
			seg = next;
		}
		/* tell the consumer to stop */
		const int st = it % COL_NS;
		svt_mbar_wait(empty0 + 8 * st, ((it / COL_NS) & 1) ^ 1);
		ItemMeta md;
		md.seg = -1; md.start = md.end = md.cbase = 0;
		md.celems = 0; md.flags = IT_STOP;
		meta[st] = md;
		svt_mbar_arrive(full0 + 8 * st);
		return;
	}

	/* consumer warp */
	LaneAcc<CC, T> acc;
	acc.reset();
	SvtColPartial part;
	svt_col_partial_init(&part);
	double center = P.center, s2 = 0.0;
	for (uint32_t it = 0; ; it++) {
		const int st = it % COL_NS;
		svt_mbar_wait(full0 + 8 * st, (it / COL_NS) & 1);
		const ItemMeta md = meta[st];
		if (md.flags & IT_STOP)
			break;
		const T *buf = (const T *) (ring + (size_t) st * stage_bytes);
		/* element window of the segment inside this stage */
		int64_t lo64 = md.start - md.cbase;
		int64_t hi64 = md.end - md.cbase;
		const int lo = lo64 < 0 ? 0 : (int) lo64;
		const int hi = hi64 > md.celems ? md.celems : (int) hi64;
		if (md.flags & IT_FIRST) {
			acc.reset();
			s2 = 0.0;
			center = P.center;
		}
		if (!(md.flags & IT_PASS2)) {
			consume_pass1<CC, T>(acc, buf, lo, hi, lane);
			if (md.flags & IT_PASS_END) {
				acc.reduce_into(&part, md.end - md.start);
				if (CC == CC_VAR) {
					if (svt_isnan(center))
						center = svt_col_mean(
							P.is_double, P.narm,
							P.seg_len, &part);
					if (md.flags & IT_SINGLE)
						consume_pass2<T>(s2, buf, lo,
							hi, lane, center);
				}
			}
		} else {
			consume_pass2<T>(s2, buf, lo, hi, lane, center);
		}
		if (md.flags & IT_LAST) {
			if (CC == CC_VAR)
				part.sum2 = svt_warp_sum(s2);
			if (lane == 0)
				store_result(P, md.seg, svt_col_finalize(
					P.opcode, P.is_double, P.narm,
					P.seg_len, center, &part));
		}
		__syncwarp();
		if (lane == 0)
			svt_mbar_arrive(empty0 + 8 * st);
	}
}

/* ------------------------------------------------------------------------
 * colstats_lacunar
 */
__global__ void __launch_bounds__(256)
colstats_lacunar(ColParams P)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t seg = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     seg < P.nseg; seg += stride) {
		const int64_t nz = P.leaf_ptr[(seg + 1) * P.group] -
				   P.leaf_ptr[seg * P.group];
		SvtColPartial part;
		svt_col_partial_ones(&part, nz, 0.0);
		double center = P.center;
		if (svt_col_op_needs_center(P.opcode)) {
			if (svt_isnan(center))
				center = svt_col_mean(P.is_double, P.narm,
						      P.seg_len, &part);
			svt_col_partial_ones(&part, nz, center);
		}
		store_result(P, seg, svt_col_finalize(P.opcode, P.is_double,
				P.narm, P.seg_len, center, &part));
	}
}

template <typename T>
int launch_typed(const ColParams &P, int cc, bool use_tma, int avg_seg_bytes,
		 cudaStream_t stream)
{
	const int sms = svtgpu_sm_count();
	if (!use_tma) {
		int64_t blocks = (P.nseg + 7) / 8;
		if (blocks > (int64_t) sms * 8) blocks = (int64_t) sms * 8;
		if (blocks < 1) blocks = 1;
#define DIRECT(CC) colstats_direct<CC, T><<<(unsigned) blocks, 256, 0, stream>>>(P)
		switch (cc) {
		    case CC_COUNT:  DIRECT(CC_COUNT); break;
		    case CC_SUM:    DIRECT(CC_SUM); break;
		    case CC_MINMAX: DIRECT(CC_MINMAX); break;
		    case CC_VAR:    DIRECT(CC_VAR); break;
		    case CC_ANYALL: DIRECT(CC_ANYALL); break;
		    case CC_PROD:   DIRECT(CC_PROD); break;
		}
#undef DIRECT
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		return SVTGPU_OK;
	}
	/* stage large enough for a typical segment (so the variance's second
	   pass stays on chip), as many pairs as 200 KB of shared memory hold */
	int stage_bytes = (avg_seg_bytes + avg_seg_bytes / 4 + 64 + 1023) /
			  1024 * 1024;
	const int stage_env = atoi(svtgpu_env("SVTGPU_COL_STAGE_KB", "0"));
	if (stage_env > 0) stage_bytes = stage_env * 1024;
	if (stage_bytes < 4096) stage_bytes = 4096;
	if (stage_bytes > 48 * 1024) stage_bytes = 48 * 1024;
	int pairs = (200 * 1024) / (COL_NS * stage_bytes);
	if (pairs > 8) pairs = 8;
	if (pairs < 1) pairs = 1;
	const int pairs_env = atoi(svtgpu_env("SVTGPU_COL_PAIRS", "0"));
	if (pairs_env > 0 && pairs_env <= 8) pairs = pairs_env;
	const size_t smem = (size_t) pairs * COL_NS * stage_bytes +
			    (size_t) pairs * COL_NS * sizeof(ItemMeta) +
			    (size_t) 2 * pairs * COL_NS * sizeof(uint64_t);
	int64_t blocks = (P.nseg + pairs - 1) / pairs;
	if (blocks > sms) blocks = sms;
	if (blocks < 1) blocks = 1;
#define TMA(CC) do { \
		SVT_CUDA(cudaFuncSetAttribute(colstats_tma<CC, T>, \
			cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem)); \
		colstats_tma<CC, T><<<(unsigned) blocks, pairs * 64, smem, stream>>>( \
			P, pairs, stage_bytes); \
	} while (0)
	switch (cc) {
	    case CC_COUNT:  TMA(CC_COUNT); break;
	    case CC_SUM:    TMA(CC_SUM); break;
	    case CC_MINMAX: TMA(CC_MINMAX); break;
	    case CC_VAR:    TMA(CC_VAR); break;
	    case CC_ANYALL: TMA(CC_ANYALL); break;
	    case CC_PROD:   TMA(CC_PROD); break;
	}
#undef TMA
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

}  /* namespace */

int svtgpu_launch_colstats(svtgpu_matrix *m, int opcode, int narm,
			   double center, int64_t group, void *d_out,
			   int32_t *d_warn, cudaStream_t stream)
{
	SVT_ARG(svt_col_op_supported(opcode, m->val_type),
		"colStats: operation %d is not supported on type %d by the "
		"GPU path", opcode, m->val_type);
	SVT_ARG(group >= 1 && (m->nleaf % group) == 0,
		"colStats: 'group' must divide the number of leaves");
	ColParams P;
	P.vals = m->d_vals;
	P.leaf_ptr = m->d_leaf_ptr;
	P.nseg = m->nleaf / group;
	P.group = group;
	P.seg_len = m->nrow * group;
	P.opcode = opcode;
	P.narm = narm != 0;
	P.is_double = svt_is_double(m->val_type);
	P.center = center;
	P.out = d_out;
	P.warn = d_warn;
	P.var_small = 0;
	P.var_onepass = strcmp(svtgpu_env("SVTGPU_COLVAR_DOUBLE", "auto"),
			       "twopass") != 0;
	if (!P.is_double && svt_isnan(center)) {
		/* a lane sees at most seg_len / 32 + 1 values of a segment */
		const int64_t B = svtgpu_value_bound(m);
		const int64_t per_lane = P.seg_len / 32 + 2;
		if (B >= 0 && B < 46340 &&
		    per_lane < (int64_t) 0x7FFFFFFF / (B * B + 1)) {
			P.var_small = 1;
			if (m->vmax_abs >= 0 && m->vmin >= 0 &&
			    strcmp(svtgpu_env("SVTGPU_COLVAR_NONNEG", "on"),
				   "on") == 0)
				P.var_small = 2;
		}
	}
	if (P.nseg == 0)
		return SVTGPU_OK;
	if (!(m->flags & SVTGPU_HAS_VALS)) {
		int64_t blocks = (P.nseg + 255) / 256;
		int64_t cap = (int64_t) svtgpu_sm_count() * 8;
		if (blocks > cap) blocks = cap;
		colstats_lacunar<<<(unsigned) blocks, 256, 0, stream>>>(P);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		return SVTGPU_OK;
	}
	const int cc = col_class_of(opcode);
	if (cc == CC_SUM && !P.is_double) {
		SVT_CHECK(svt_ensure_compact(m, stream));
		if (m->d_vals8 != NULL) {
			int64_t blocks = (P.nseg + 7) / 8;
			const int64_t cap = (int64_t) svtgpu_sm_count() *
					    SUM_I8_BLOCKS_PER_SM;
			if (blocks > cap)
				blocks = cap;
			colstats_sum_i8<<<(unsigned) blocks, 256, 0, stream>>>(
				P, m->d_vals8);
			SVT_CUDA(cudaGetLastError());
			svtgpu_count_launch(1);
			return SVTGPU_OK;
		}
	}
	const char *impl = svtgpu_env("SVTGPU_COLSTATS_IMPL", "direct");
	bool use_tma = strcmp(impl, "tma") == 0 &&
		       (((uintptr_t) m->d_vals) & 15) == 0;
	int64_t avg = m->nnz / P.nseg * (int64_t) svt_val_size(m->val_type);
	if (avg > (1 << 30)) avg = 1 << 30;
	if (P.is_double)
		return launch_typed<double>(P, cc, use_tma, (int) avg, stream);
	return launch_typed<int32_t>(P, cc, use_tma, (int) avg, stream);
}

extern "C" int svtgpu_colstats_out_is_int(int opcode, int val_type)
{
	return svt_col_out_is_int(opcode, val_type);
}

extern "C" int svtgpu_colstats_dev(svtgpu_matrix *m, int opcode, int narm,
				   double center, int64_t group, void *d_out,
				   int32_t *d_warn, void *stream)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && d_out != NULL, "svtgpu_colstats_dev: NULL argument");
	return svtgpu_launch_colstats(m, opcode, narm, center, group, d_out,
				      d_warn, (cudaStream_t) stream);
}

extern "C" int svtgpu_colstats(svtgpu_matrix *m, int opcode, int narm,
			       double center, int64_t group, void *out,
			       int *warn)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && out != NULL, "svtgpu_colstats: NULL argument");
	SVT_ARG(group >= 1 && (m->nleaf % group) == 0,
		"colStats: 'group' must divide the number of leaves");
	const int64_t nseg = m->nleaf / group;
	const size_t esz = svt_col_out_is_int(opcode, m->val_type) ? 4 : 8;
	if (warn != NULL)
		*warn = 0;
	m->tm.kernel_ms = m->tm.d2h_ms = 0.0;
	m->tm.d2h_bytes = 0.0;
	m->tm.launches = 0;
	if (nseg == 0)
		return SVTGPU_OK;
	void *scratch = NULL;
	SVT_CHECK(svtgpu_scratch(m, esz * (size_t) nseg + 16, &scratch));
	int32_t *d_warn = (int32_t *) scratch;
	void *d_out = (char *) scratch + 16;
	cudaStream_t s = 0;
	SVT_CUDA(cudaMemsetAsync(d_warn, 0, 16, s));
	SvtTimer t;
	SVT_CHECK(svt_timer_begin(&t, s));
	int64_t l0 = svtgpu_launch_count();
	int rc = svtgpu_launch_colstats(m, opcode, narm, center, group, d_out,
					d_warn, s);
	int rc2 = svt_timer_end(&t, &m->tm.kernel_ms);
	if (rc != SVTGPU_OK)
		return rc;
	SVT_CHECK(rc2);
	m->tm.launches = (int) (svtgpu_launch_count() - l0);
	SVT_CHECK(svt_timer_begin(&t, s));
	int32_t h_warn = 0;
	SVT_CUDA(cudaMemcpyAsync(out, d_out, esz * (size_t) nseg,
				 cudaMemcpyDeviceToHost, s));
	SVT_CUDA(cudaMemcpyAsync(&h_warn, d_warn, sizeof(int32_t),
				 cudaMemcpyDeviceToHost, s));
	SVT_CHECK(svt_timer_end(&t, &m->tm.d2h_ms));
	m->tm.d2h_bytes = (double) (esz * (size_t) nseg);
	if (warn != NULL)
		*warn = h_warn != 0;
	return SVTGPU_OK;
}

namespace {

/* ------------------------------------------------------------------------
 * Whole-array summarisation (C_summarize_SVT,
 * src/SparseArray_summarization.c:112-142): the matrix is ONE virtual vector
 * of nrow * nleaf entries.  The stored values are contiguous across leaves,
 * so every warp reduces one slice of [0, nnz) to an SvtColPartial and a
 * single warp combines the slices in a fixed order (deterministic results).
 */
template <int CC, typename T>
__global__ void __launch_bounds__(256)
summarize_slices(const T *__restrict__ vals, int64_t nnz, int64_t slice,
		 double center, int pass2, SvtColPartial *__restrict__ parts)
{
	const int lane = threadIdx.x & 31;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int64_t start = gw * slice;
	if (start >= nnz)
		return;
	const int64_t end = start + slice < nnz ? start + slice : nnz;
	SvtColPartial part;
	if (pass2) {
		double s2 = 0.0;
#pragma unroll 4
		for (int64_t e = start + lane; e < end; e += 32)
			add_sq(s2, vals[e], center);
		svt_col_partial_init(&part);
		part.sum2 = svt_warp_sum(s2);
	} else {
		LaneAcc<CC, T> acc;
		acc.reset();
		lane_accumulate<CC, T>(acc, vals, start, end, lane);
		acc.reduce_into(&part, end - start);
	}
	if (lane == 0)
		parts[gw] = part;
}

__device__ __forceinline__ void col_partial_merge(SvtColPartial *a,
						  const SvtColPartial *b)
{
	a->nz += b->nz;
	a->n_na += b->n_na;
	a->n_nan += b->n_nan;
	a->n_zero += b->n_zero;
	a->sum += b->sum;
	a->sum2 += b->sum2;
	a->prod *= b->prod;
	a->vmin = b->vmin < a->vmin ? b->vmin : a->vmin;
	a->vmax = b->vmax > a->vmax ? b->vmax : a->vmax;
}

__device__ __forceinline__ void col_partial_warp_merge(SvtColPartial *acc)
{
	acc->nz = svt_warp_sum((long long) acc->nz);
	acc->n_na = svt_warp_sum((long long) acc->n_na);
	acc->n_nan = svt_warp_sum((long long) acc->n_nan);
	acc->n_zero = svt_warp_sum((long long) acc->n_zero);
	acc->sum = svt_warp_sum(acc->sum);
	acc->sum2 = svt_warp_sum(acc->sum2);
	acc->prod = svt_warp_prod(acc->prod);
	acc->vmin = svt_warp_min(acc->vmin);
	acc->vmax = svt_warp_max(acc->vmax);
}

/* one block: thread t merges slices t, t + 1024, ... in order, the lanes of a
   warp merge in a butterfly, warp 0 merges the 32 warp results the same way:
   a fixed tree, deterministic */
__global__ void __launch_bounds__(1024)
summarize_combine(const SvtColPartial *__restrict__ parts, int64_t n,
		  SvtColPartial *__restrict__ out)
{
	__shared__ SvtColPartial warp_part[32];
	const int lane = threadIdx.x & 31;
	const int warp = threadIdx.x >> 5;
	SvtColPartial acc;
	svt_col_partial_init(&acc);
	for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
		const SvtColPartial p = parts[i];
		col_partial_merge(&acc, &p);
	}
	col_partial_warp_merge(&acc);
	if (lane == 0)
		warp_part[warp] = acc;
	__syncthreads();
	if (warp == 0) {
		acc = warp_part[lane];
		col_partial_warp_merge(&acc);
		if (lane == 0)
			*out = acc;
	}
}

template <typename T>
int launch_slices(int cc, const T *vals, int64_t nnz, int64_t slice,
		  int64_t nslices, double center, int pass2,
		  SvtColPartial *parts, cudaStream_t s)
{
	const unsigned blocks = (unsigned) ((nslices + 7) / 8);
#define SLICES(CC) summarize_slices<CC, T><<<blocks, 256, 0, s>>>( \
			vals, nnz, slice, center, pass2, parts)
	switch (cc) {
	    case CC_COUNT:  SLICES(CC_COUNT); break;
	    case CC_SUM: case CC_VAR: SLICES(CC_SUM); break;
	    case CC_MINMAX: SLICES(CC_MINMAX); break;
	    case CC_ANYALL: SLICES(CC_ANYALL); break;
	    case CC_PROD:   SLICES(CC_PROD); break;
	}
#undef SLICES
	SVT_CUDA(cudaGetLastError());
	summarize_combine<<<1, 1024, 0, s>>>(parts, nslices, parts + nslices);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(2);
	return SVTGPU_OK;
}

/* integer input, centre = the mean: exact sum and sum of squares of every
   slice in 64-bit integers -- one pass instead of the reference's two, merged
   on the host (a few thousand slices) and finished by var_from_int_sums() */
struct IntMoments { long long s1; unsigned long long s2; long long nna; };

__global__ void __launch_bounds__(256)
summarize_int_moments(const int32_t *__restrict__ vals, int64_t nnz,
		      int64_t slice, IntMoments *__restrict__ parts)
{
	const int lane = threadIdx.x & 31;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int64_t start = gw * slice;
	if (start >= nnz)
		return;
	const int64_t end = start + slice < nnz ? start + slice : nnz;
	long long s1 = 0, nna = 0;
	unsigned long long s2 = 0;
	const int32_t *p = vals + start + lane;
	const int64_t left = end - start - lane;
	const int n = left > 0 ? (int) ((left + 31) >> 5) : 0;
	int i = 0;
	for (; i + 8 <= n; i += 8) {
		int x[8];
#pragma unroll
		for (int k = 0; k < 8; k++)
			x[k] = p[(i + k) * 32];
#pragma unroll
		for (int k = 0; k < 8; k++) {
			const bool na = x[k] == SVT_NA_INT;
			const long long x0 = na ? 0 : x[k];
			nna += na;
			s1 += x0;
			s2 += (unsigned long long) (x0 * x0);
		}
	}
	for (; i < n; i++) {
		const int x = p[i * 32];
		const bool na = x == SVT_NA_INT;
		const long long x0 = na ? 0 : x;
		nna += na;
		s1 += x0;
		s2 += (unsigned long long) (x0 * x0);
	}
	s1 = svt_warp_sum(s1);
	nna = svt_warp_sum(nna);
#pragma unroll
	for (int m = 16; m > 0; m >>= 1)
		s2 += __shfl_xor_sync(SVT_FULL_MASK, s2, m);
	if (lane == 0) {
		IntMoments r;
		r.s1 = s1; r.s2 = s2; r.nna = nna;
		parts[gw] = r;
	}
}

/* 1 when the exact one-pass form applies (and *r is the answer), 0 when the
   caller must take the two-pass form, < 0 on error (status negated) */
int summarize_int_var(svtgpu_matrix *m, int opcode, int narm,
		      int64_t in_length, SvtScalar *r, cudaStream_t s)
{
	if (strcmp(svtgpu_env("SVTGPU_SUMMARIZE_VAR", "auto"), "twopass") == 0)
		return 0;
	const int64_t B = svtgpu_value_bound(m);
	/* sum < 2^53 (kept as a double later), sum of squares < 2^63 */
	if (B < 0 || B >= (1 << 20) ||
	    (B > 0 && m->nnz > ((int64_t) 1 << 52) / B) ||
	    (B > 0 && m->nnz > ((int64_t) 1 << 62) / (B * B)))
		return 0;
	const int64_t max_slices = (int64_t) svtgpu_sm_count() * 64;
	int64_t slice = (m->nnz + max_slices - 1) / max_slices;
	if (slice < 4096) slice = 4096;
	slice = (slice + 127) / 128 * 128;
	const int64_t nslices = (m->nnz + slice - 1) / slice;
	void *scratch = NULL;
	int rc = svtgpu_scratch(m, sizeof(IntMoments) * (size_t) nslices,
				&scratch);
	if (rc != SVTGPU_OK)
		return -rc;
	IntMoments *h = (IntMoments *) malloc(sizeof(IntMoments) *
					      (size_t) nslices);
	if (h == NULL) {
		svtgpu_set_error("out of host memory");
		return -SVTGPU_ERR_NOMEM;
	}
	summarize_int_moments<<<(unsigned) ((nslices + 7) / 8), 256, 0, s>>>(
		(const int32_t *) m->d_vals, m->nnz, slice,
		(IntMoments *) scratch);
	cudaError_t e = cudaGetLastError();
	svtgpu_count_launch(1);
	if (e == cudaSuccess)
		e = cudaMemcpyAsync(h, scratch, sizeof(IntMoments) *
				    (size_t) nslices, cudaMemcpyDeviceToHost, s);
	if (e == cudaSuccess)
		e = cudaStreamSynchronize(s);
	if (e != cudaSuccess) {
		free(h);
		return -svtgpu_cuda_fail(e, "summarize_int_moments", __FILE__,
					 __LINE__);
	}
	long long s1 = 0, nna = 0;
	unsigned long long s2 = 0;
	for (int64_t i = 0; i < nslices; i++) {
		s1 += h[i].s1;
		s2 += h[i].s2;
		nna += h[i].nna;
	}
	free(h);
	SvtColPartial part;
	svt_col_partial_init(&part);
	part.nz = m->nnz;
	part.n_na = nna;
	part.sum = (double) s1;
	*r = var_from_int_sums(opcode, narm, in_length, &part, s2);
	return 1;
}

/* one reduction of all stored values into *h_part (host) */
int summarize_pass(svtgpu_matrix *m, int cc, double center, int pass2,
		   SvtColPartial *h_part, cudaStream_t s)
{
	const int64_t max_slices = (int64_t) svtgpu_sm_count() * 64;
	/* slices of whole 128-element rounds, at least 4096 values each */
	int64_t slice = (m->nnz + max_slices - 1) / max_slices;
	if (slice < 4096) slice = 4096;
	slice = (slice + 127) / 128 * 128;
	const int64_t nslices = (m->nnz + slice - 1) / slice;
	void *scratch = NULL;
	SVT_CHECK(svtgpu_scratch(m, sizeof(SvtColPartial) *
				 (size_t) (nslices + 1), &scratch));
	SvtColPartial *parts = (SvtColPartial *) scratch;
	if (svt_is_double(m->val_type))
		SVT_CHECK(launch_slices<double>(cc, (const double *) m->d_vals,
				m->nnz, slice, nslices, center, pass2, parts, s));
	else
		SVT_CHECK(launch_slices<int32_t>(cc, (const int32_t *) m->d_vals,
				m->nnz, slice, nslices, center, pass2, parts, s));
	SVT_CUDA(cudaMemcpyAsync(h_part, parts + nslices, sizeof(SvtColPartial),
				 cudaMemcpyDeviceToHost, s));
	SVT_CUDA(cudaStreamSynchronize(s));
	return SVTGPU_OK;
}

}  /* namespace */

extern "C" int svtgpu_summarize_supported(int opcode, int val_type)
{
	return opcode == SVTGPU_OP_RANGE ||
	       svt_col_op_supported(opcode, val_type);
}

extern "C" int svtgpu_summarize(svtgpu_matrix *m, int opcode, int narm,
				double center, double *out, int *warn)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && out != NULL, "svtgpu_summarize: NULL argument");
	SVT_ARG(svtgpu_summarize_supported(opcode, m->val_type),
		"summarize: operation %d is not supported on type %d by the "
		"GPU path", opcode, m->val_type);
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	if (warn != NULL)
		*warn = 0;
	m->tm.kernel_ms = m->tm.d2h_ms = 0.0;
	m->tm.d2h_bytes = 0.0;
	m->tm.launches = 0;
	const int is_double = svt_is_double(m->val_type);
	const int64_t in_length = m->nrow * m->nleaf;
	const int needs_center = svt_col_op_needs_center(opcode);
	cudaStream_t s = 0;
	SvtColPartial part;
	svt_col_partial_init(&part);
	int exact = 0;
	SvtScalar exact_r;
	exact_r.d = 0.0; exact_r.i = 0; exact_r.warn = 0;
	SvtTimer t;
	SVT_CHECK(svt_timer_begin(&t, s));
	const int64_t l0 = svtgpu_launch_count();
	if (m->nnz > 0 && !(m->flags & SVTGPU_HAS_VALS)) {
		/* every stored value is 1 (summarize_ones(),
		   src/Rvector_summarization.c:742-825): O(1) */
		svt_col_partial_ones(&part, m->nnz, 0.0);
		if (needs_center) {
			if (svt_isnan(center))
				center = svt_col_mean(is_double, narm,
						      in_length, &part);
			svt_col_partial_ones(&part, m->nnz, center);
		}
	} else if (m->nnz > 0 && needs_center && !is_double &&
		   svt_isnan(center) &&
		   (exact = summarize_int_var(m, opcode, narm, in_length,
					      &exact_r, s)) != 0) {
		if (exact < 0) {
			double ms;
			svt_timer_end(&t, &ms);
			return -exact;
		}
	} else if (m->nnz > 0) {
		const int cc = opcode == SVTGPU_OP_RANGE ? (int) CC_MINMAX
							 : col_class_of(opcode);
		int rc = summarize_pass(m, cc, 0.0, 0, &part, s);
		if (rc == SVTGPU_OK && needs_center) {
			if (svt_isnan(center))
				center = svt_col_mean(is_double, narm,
						      in_length, &part);
			if (!svt_isnan(center)) {
				SvtColPartial p2;
				rc = summarize_pass(m, cc, center, 1, &p2, s);
				part.sum2 = p2.sum2;
			}
		}
		if (rc != SVTGPU_OK) {
			double ms;
			svt_timer_end(&t, &ms);
			return rc;
		}
	} else if (needs_center && svt_isnan(center)) {
		center = svt_col_mean(is_double, narm, in_length, &part);
	}
	SVT_CHECK(svt_timer_end(&t, &m->tm.kernel_ms));
	m->tm.launches = (int) (svtgpu_launch_count() - l0);
	const int nres = opcode == SVTGPU_OP_RANGE ? 2 : 1;
	for (int k = 0; k < nres; k++) {
		const int op = opcode != SVTGPU_OP_RANGE ? opcode
			     : k == 0 ? SVTGPU_OP_MIN : SVTGPU_OP_MAX;
		const SvtScalar r = exact > 0 ? exact_r
			: svt_col_finalize(op, is_double, narm, in_length,
					   center, &part);
		if (svt_col_out_is_int(op, m->val_type))
			out[k] = r.i == SVT_NA_INT ? svt_na_real()
						   : (double) r.i;
		else
			out[k] = r.d;
		if (r.warn && warn != NULL)
			*warn = 1;
	}
	return SVTGPU_OK;
}

extern "C" int svtgpu_rowstats_via_transpose(svtgpu_matrix *m, int opcode,
					     int narm, double center,
					     void *out, int *warn)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && out != NULL,
		"svtgpu_rowstats_via_transpose: NULL argument");
	SVT_ARG(svt_col_op_supported(opcode, m->val_type),
		"rowStats: operation %d is not supported on type %d by the "
		"GPU path", opcode, m->val_type);
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	if (warn != NULL)
		*warn = 0;
	if (m->nrow == 0)
		return SVTGPU_OK;
	svtgpu_matrix *t = NULL;
	if (m->nnz > 0 && (m->flags & SVTGPU_HAS_OFFS)) {
		SVT_CHECK(svtgpu_ensure_transpose(m, 0, &t));
		SVT_ARG(t != NULL, "rowStats: the device transpose could not "
			"be built for this matrix");
		int rc = svtgpu_colstats(t, opcode, narm, center, 1, out, warn);
		m->tm = t->tm;
		return rc;
	}
	/* no nonzeros: every row is nleaf implicit zeros -- an empty CSC with
	   the extents swapped */
	svtgpu_matrix *e = NULL;
	SVT_CHECK(svtgpu_matrix_create(&e, m->nleaf, m->nrow, 0, m->val_type,
				       SVTGPU_HAS_VALS));
	int64_t *zeros = (int64_t *) calloc((size_t) m->nrow + 1, 8);
	int rc = zeros == NULL ? SVTGPU_ERR_NOMEM
		: svtgpu_matrix_upload(e, zeros, NULL, NULL);
	free(zeros);
	if (rc == SVTGPU_OK)
		rc = svtgpu_colstats(e, opcode, narm, center, 1, out, warn);
	svtgpu_matrix_free(e);
	return rc;
}
