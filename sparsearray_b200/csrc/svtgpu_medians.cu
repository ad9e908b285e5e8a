/* Column medians of a device CSC (svtgpu_colmedians) and row medians through
 * the cached device transpose (svtgpu_rowmedians).  The reference computes
 * them in R, one column at a time (R/SparseArray-matrixStats.R:760-813).
 *
 *   median_classify  one streaming pass, a warp per leaf: counts the stored
 *                    negatives, positives and NA / NaN and the smallest and
 *                    largest key of either sign.  svt_med_plan() turns the
 *                    counts into the result (NA, 0) for most leaves; a leaf
 *                    whose middle ranks fall among its stored values is
 *                    finished here too when its middle values are extremes
 *                    of their side (or the side holds one distinct value),
 *                    and is otherwise appended to a device work list.
 *   median_select    a persistent grid, one CTA per listed leaf: radix select
 *                    over the keys of one side.  Every round histograms one
 *                    digit (<= 11 bits) of the keys that still match the
 *                    selected prefix, re-reading the leaf (from L2 at typical
 *                    column lengths); the first round starts at the highest
 *                    bit in which the side's smallest and largest keys
 *                    differ, and a round whose survivors all hold one key
 *                    ends the search.  The second middle value comes from the
 *                    final round's histogram or, failing that, from one
 *                    min-reduction pass over the keys above the first.
 *
 * No host synchronisation between the two kernels: the work-list length is
 * read on the device.
 */
#include "svtgpu_internal.h"
#include "svt_ptx.cuh"

namespace {

/* one leaf the counts could not decide */
struct MedItem {
	int64_t leaf;
	int64_t rank;        /* SvtMedPlan.rank */
	uint64_t kmin, kmax; /* smallest / largest key of the side */
	uint64_t kother;     /* smallest positive key (side NEG, NEXT) */
	int32_t side, second;
};

template <typename T> struct MedKey;
template <> struct MedKey<int32_t> { typedef uint32_t K; };
template <> struct MedKey<double> { typedef uint64_t K; };

/* key of x if x is a stored value of `side` (never NA / NaN / zero) */
__device__ __forceinline__ bool side_key(int32_t x, int side, uint32_t *k)
{
	svt_med_key_i32(x, k);
	return side == SVT_MED_NEG ? (x < 0 && x != SVT_NA_INT) : x > 0;
}

__device__ __forceinline__ bool side_key(double x, int side, uint64_t *k)
{
	svt_med_key_f64(x, k);
	return side == SVT_MED_NEG ? x < 0.0 : x > 0.0;   /* NaN: false */
}

__device__ __forceinline__ double key_value(uint32_t k)
{
	return (double) svt_med_unkey_i32(k);
}

__device__ __forceinline__ double key_value(uint64_t k)
{
	return svt_med_unkey_f64(k);
}

template <typename K>
__device__ __forceinline__ K warp_min(K v)
{
#pragma unroll
	for (int m = 16; m > 0; m >>= 1) {
		const K o = __shfl_xor_sync(SVT_FULL_MASK, v, m);
		v = o < v ? o : v;
	}
	return v;
}

template <typename K>
__device__ __forceinline__ K warp_max(K v)
{
#pragma unroll
	for (int m = 16; m > 0; m >>= 1) {
		const K o = __shfl_xor_sync(SVT_FULL_MASK, v, m);
		v = o > v ? o : v;
	}
	return v;
}

/* a lane's counts and key extremes over its share of one leaf */
template <typename T>
struct MedLane {
	typedef typename MedKey<T>::K K;
	int nneg, npos, nna;
	K nmin, nmax, pmin, pmax;

	__device__ __forceinline__ void reset()
	{
		nneg = npos = nna = 0;
		nmin = pmin = (K) ~(K) 0;
		nmax = pmax = 0;
	}

	__device__ __forceinline__ void add(int32_t x)
	{
		uint32_t k;
		const bool na = !svt_med_key_i32(x, &k);
		const bool neg = x < 0 && !na, pos = x > 0;
		nna += na;
		nneg += neg;
		npos += pos;
		nmin = neg && k < nmin ? k : nmin;
		nmax = neg && k > nmax ? k : nmax;
		pmin = pos && k < pmin ? k : pmin;
		pmax = pos && k > pmax ? k : pmax;
	}

	__device__ __forceinline__ void add(double x)
	{
		uint64_t k;
		const bool na = !svt_med_key_f64(x, &k);
		const bool neg = x < 0.0, pos = x > 0.0;
		nna += na;
		nneg += neg;
		npos += pos;
		nmin = neg && k < nmin ? k : nmin;
		nmax = neg && k > nmax ? k : nmax;
		pmin = pos && k < pmin ? k : pmin;
		pmax = pos && k > pmax ? k : pmax;
	}
};

/* lane's share of [start, end): 16-byte loads over the aligned middle of an
   int32 leaf (as colstats_direct), eight 8-byte loads in flight for doubles */
template <typename T>
__device__ __forceinline__ void med_accumulate(MedLane<T> &acc,
		const T *__restrict__ vals, int64_t start, int64_t end, int lane)
{
	if (sizeof(T) == 4 && (((uintptr_t) vals) & 15) == 0) {
		const int64_t a4 = (start + 3) & ~(int64_t) 3;
		const int64_t b4 = end & ~(int64_t) 3;
		if (a4 < b4) {
			if (start + lane < a4)
				acc.add(vals[start + lane]);
			if (b4 + lane < end)
				acc.add(vals[b4 + lane]);
			const int4 *q = (const int4 *) (vals + a4);
			const int nv = (int) ((b4 - a4) / 4);
			int i = lane;
			for (; i + 32 < nv; i += 64) {
				const int4 u = q[i];
				const int4 w = q[i + 32];
				acc.add((T) u.x); acc.add((T) u.y);
				acc.add((T) u.z); acc.add((T) u.w);
				acc.add((T) w.x); acc.add((T) w.y);
				acc.add((T) w.z); acc.add((T) w.w);
			}
			if (i < nv) {
				const int4 u = q[i];
				acc.add((T) u.x); acc.add((T) u.y);
				acc.add((T) u.z); acc.add((T) u.w);
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
	for (; i < n; i++)
		acc.add(p[i * 32]);
}

struct MedParams {
	const void *vals;          /* NULL: lacunar (every stored value is 1) */
	const int64_t *leaf_ptr;
	int64_t nleaf, nrow;
	int narm;
	double *out;
	MedItem *items;
	unsigned long long *nitems;
};

/* ------------------------------------------------------------------------
 * median_classify
 */
template <typename T>
__global__ void __launch_bounds__(256)
median_classify(MedParams P)
{
	typedef typename MedKey<T>::K K;
	const int lane = threadIdx.x & 31;
	const int64_t warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const T *vals = (const T *) P.vals;

	int64_t nstart = 0, nend = 0;
	if (gw < P.nleaf) {
		nstart = P.leaf_ptr[gw];
		nend = P.leaf_ptr[gw + 1];
	}
	for (int64_t leaf = gw; leaf < P.nleaf; leaf += warps) {
		const int64_t start = nstart, end = nend;
		if (leaf + warps < P.nleaf) {
			nstart = P.leaf_ptr[leaf + warps];
			nend = P.leaf_ptr[leaf + warps + 1];
		}
		int64_t nneg = 0, npos, nna = 0;
		K nmin = 0, nmax = 0, pmin, pmax;
		if (vals == NULL) {
			/* lacunar: the counts alone decide */
			npos = end - start;
			K one;
			if (sizeof(T) == 4) {
				uint32_t k;
				svt_med_key_i32(1, &k);
				one = (K) k;
			} else {
				uint64_t k;
				svt_med_key_f64(1.0, &k);
				one = (K) k;
			}
			pmin = pmax = one;
		} else {
			MedLane<T> acc;
			acc.reset();
			med_accumulate<T>(acc, vals, start, end, lane);
			nneg = svt_warp_sum((long long) acc.nneg);
			npos = svt_warp_sum((long long) acc.npos);
			nna = svt_warp_sum((long long) acc.nna);
			nmin = warp_min(acc.nmin);
			nmax = warp_max(acc.nmax);
			pmin = warp_min(acc.pmin);
			pmax = warp_max(acc.pmax);
		}
		if (lane != 0)
			continue;
		const SvtMedPlan pl = svt_med_plan(P.nrow, nneg, npos, nna,
						   P.narm);
		if (pl.kind != SVT_MED_SELECT) {
			P.out[leaf] = pl.kind == SVT_MED_NA ? svt_na_real() : 0.0;
			continue;
		}
		const bool neg = pl.side == SVT_MED_NEG;
		const int64_t ns = neg ? nneg : npos;
		const K kmin = neg ? nmin : pmin, kmax = neg ? nmax : pmax;
		/* the middle values when they are extremes of the side */
		bool have_a = true, have_b = true;
		K a = kmin, b = kmin;
		if (kmin == kmax || pl.rank == 0)
			a = kmin;
		else if (pl.rank == ns - 1)
			a = kmax;
		else
			have_a = false;
		if (pl.second == SVT_MED_2ND_NEXT) {
			if (pl.rank + 1 < ns && kmin == kmax)
				b = kmin;
			else if (pl.rank + 1 == ns - 1)
				b = kmax;
			else if (pl.rank == ns - 1)
				b = pmin;          /* side NEG, no zeros */
			else
				have_b = false;
		}
		if (have_a && have_b) {
			const double va = key_value(a);
			P.out[leaf] = pl.second == SVT_MED_2ND_NONE ? va
				: svt_med_mid(va, pl.second == SVT_MED_2ND_ZERO
						    ? 0.0 : key_value(b));
			continue;
		}
		const unsigned long long slot = atomicAdd(P.nitems, 1ull);
		MedItem it;
		it.leaf = leaf;
		it.rank = pl.rank;
		it.kmin = kmin;
		it.kmax = kmax;
		it.kother = pmin;
		it.side = pl.side;
		it.second = pl.second;
		P.items[slot] = it;
	}
}

/* ------------------------------------------------------------------------
 * median_select
 */
constexpr int SEL_THREADS = 512;
constexpr int SEL_WARPS = SEL_THREADS / 32;
constexpr int SEL_DIGIT = 11;
constexpr int SEL_BUCKETS = 1 << SEL_DIGIT;
constexpr int SEL_PER_THREAD = SEL_BUCKETS / SEL_THREADS;

struct SelShared {
	unsigned int hist[SEL_BUCKETS];
	unsigned long long red_min[SEL_WARPS], red_max[SEL_WARPS];
	unsigned int scan[SEL_WARPS];
	unsigned long long kmin, kmax;
	int bucket, next_bucket;
	long long below;
};

/* block-wide min and max (every thread gets them) */
template <typename K>
__device__ __forceinline__ void block_minmax(SelShared &S, K &lo, K &hi)
{
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	lo = warp_min(lo);
	hi = warp_max(hi);
	if (lane == 0) {
		S.red_min[w] = lo;
		S.red_max[w] = hi;
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		unsigned long long a = S.red_min[0], b = S.red_max[0];
		for (int i = 1; i < SEL_WARPS; i++) {
			a = S.red_min[i] < a ? S.red_min[i] : a;
			b = S.red_max[i] > b ? S.red_max[i] : b;
		}
		S.kmin = a;
		S.kmax = b;
	}
	__syncthreads();
	lo = (K) S.kmin;
	hi = (K) S.kmax;
}

template <typename T>
__global__ void __launch_bounds__(SEL_THREADS, 2)
median_select(const T *__restrict__ vals, const int64_t *__restrict__ leaf_ptr,
	      const MedItem *__restrict__ items,
	      unsigned long long *__restrict__ nitems,
	      double *__restrict__ out)
{
	typedef typename MedKey<T>::K K;
	constexpr int KBITS = 8 * sizeof(K);
	__shared__ SelShared S;
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	/* nitems[0]: list length; nitems[1]: values read by the passes */
	const unsigned long long n_items = nitems[0];
	for (unsigned long long it = blockIdx.x; it < n_items; it += gridDim.x) {
		const MedItem item = items[it];
		const int64_t start = leaf_ptr[item.leaf];
		const int64_t end = leaf_ptr[item.leaf + 1];
		const int side = item.side;
		int64_t r = item.rank;
		K prefix = (K) item.kmin;
		const K diff = (K) item.kmin ^ (K) item.kmax;
		/* bits below the side's common prefix (kmin != kmax here) */
		int nbits = diff == 0 ? 0
			  : KBITS - (sizeof(K) == 4 ? __clz((unsigned) diff)
						    : __clzll((long long) diff));
		prefix = nbits >= KBITS ? (K) 0 : (prefix >> nbits) << nbits;
		int64_t eq = 0;
		int last_shift = -1, next_bucket = -1;
		K last_mask = 0;
		bool done = nbits == 0;
		int passes = 0;
		while (!done) {
			passes++;
			const int d = nbits < SEL_DIGIT ? nbits : SEL_DIGIT;
			const int shift = nbits - d;
			const K dmask = (K) ((1u << d) - 1);
			for (int i = threadIdx.x; i < SEL_BUCKETS; i += SEL_THREADS)
				S.hist[i] = 0;
			__syncthreads();
			K lo = (K) ~(K) 0, hi = 0;
			for (int64_t base = start; base < end; base += SEL_THREADS) {
				const int64_t i = base + threadIdx.x;
				K k = 0;
				bool ok = false;
				if (i < end)
					ok = side_key(vals[i], side, &k) &&
					     (nbits >= KBITS || (k >> nbits) ==
							       (prefix >> nbits));
				const unsigned bk = ok ? (unsigned) ((k >> shift) & dmask)
						       : 0xFFFFFFFFu;
				lo = ok && k < lo ? k : lo;
				hi = ok && k > hi ? k : hi;
				/* ties are the rule (small counts): one shared
				   atomic per distinct bucket of the warp */
				const unsigned grp = __match_any_sync(SVT_FULL_MASK, bk);
				if (ok && lane == __ffs(grp) - 1)
					atomicAdd(&S.hist[bk], (unsigned) __popc(grp));
			}
			block_minmax<K>(S, lo, hi);
			if (lo == hi) {
				/* every survivor holds one key */
				prefix = lo;
				eq = S.hist[(unsigned) ((lo >> shift) & dmask)];
				last_shift = -1;
				break;
			}
			/* the bucket that holds rank r: thread t owns buckets
			   [t * SEL_PER_THREAD, (t + 1) * SEL_PER_THREAD) */
			unsigned int own = 0;
			const int b0 = threadIdx.x * SEL_PER_THREAD;
#pragma unroll
			for (int j = 0; j < SEL_PER_THREAD; j++)
				own += S.hist[b0 + j];
			unsigned int incl = own;
#pragma unroll
			for (int m = 1; m < 32; m <<= 1) {
				const unsigned int o = __shfl_up_sync(SVT_FULL_MASK, incl, m);
				if (lane >= m)
					incl += o;
			}
			if (lane == 31)
				S.scan[w] = incl;
			if (threadIdx.x == 0)
				S.next_bucket = 0x7FFFFFFF;
			__syncthreads();
			unsigned int wbase = 0;
			for (int i = 0; i < w; i++)
				wbase += S.scan[i];
			long long excl = (long long) wbase + incl - own;
			if (r >= excl && r < excl + own) {
				for (int j = 0; j < SEL_PER_THREAD; j++) {
					const unsigned int c = S.hist[b0 + j];
					if (r < excl + c) {
						S.bucket = b0 + j;
						S.below = excl;
						break;
					}
					excl += c;
				}
			}
			__syncthreads();
			const int b = S.bucket;
			for (int j = 0; j < SEL_PER_THREAD; j++)
				if (b0 + j > b && S.hist[b0 + j] != 0)
					atomicMin(&S.next_bucket, b0 + j);
			__syncthreads();
			r -= S.below;
			eq = S.hist[b];
			next_bucket = S.next_bucket;
			last_shift = shift;
			last_mask = dmask;
			prefix |= (K) b << shift;
			nbits = shift;
			done = nbits == 0;
			__syncthreads();   /* before the next round clears hist */
		}
		const double va = key_value(prefix);
		double res = va;
		if (item.second == SVT_MED_2ND_ZERO) {
			res = svt_med_mid(va, 0.0);
		} else if (item.second == SVT_MED_2ND_NEXT) {
			K kb;
			if (r + 1 < eq) {
				kb = prefix;
			} else if (last_shift == 0 && next_bucket < SEL_BUCKETS) {
				/* the final round resolved whole keys: its next
				   nonzero bucket is the next key */
				kb = (prefix & ~last_mask) | (K) next_bucket;
			} else {
				/* one min-reduction over the stored nonzero
				   values above the first */
				K lo = (K) ~(K) 0, hi = 0;
				for (int64_t i = start + threadIdx.x; i < end;
				     i += SEL_THREADS) {
					K k;
					if (side_key(vals[i], side, &k) && k > prefix &&
					    k < lo)
						lo = k;
				}
				block_minmax<K>(S, lo, hi);
				kb = lo != (K) ~(K) 0 ? lo : (K) item.kother;
				passes++;
			}
			res = svt_med_mid(va, key_value(kb));
		}
		if (threadIdx.x == 0) {
			out[item.leaf] = res;
			atomicAdd(&nitems[1], (unsigned long long) passes *
					      (unsigned long long) (end - start));
		}
		__syncthreads();   /* S is reused by the next item */
	}
}

template <typename T>
int launch_medians(svtgpu_matrix *m, int narm, double *d_out,
		   unsigned long long *h_selected, cudaStream_t s)
{
	MedParams P;
	P.vals = (m->flags & SVTGPU_HAS_VALS) ? m->d_vals : NULL;
	P.leaf_ptr = m->d_leaf_ptr;
	P.nleaf = m->nleaf;
	P.nrow = m->nrow;
	P.narm = narm != 0;
	P.out = d_out;
	P.items = NULL;
	P.nitems = NULL;
	/* room for every leaf on the work list (48 MB at 1e6 leaves): its
	   length is known only on the device, and learning it first would cost
	   a host synchronisation between the kernels.  The block comes from the
	   stream-ordered pool (svt_malloc_async), so an unused list costs no
	   cudaMalloc and no memory traffic. */
	const size_t item_bytes = sizeof(MedItem) * (size_t) m->nleaf;
	void *work = NULL;
	SVT_CUDA(svt_malloc_async(&work, 256 + item_bytes, s));
	P.nitems = (unsigned long long *) work;
	P.items = (MedItem *) ((char *) work + 256);
	cudaError_t e = cudaMemsetAsync(P.nitems, 0, 16, s);
	int64_t blocks = (m->nleaf + 7) / 8;
	const int64_t cap = (int64_t) svtgpu_sm_count() * 8;
	if (blocks > cap)
		blocks = cap;
	int launches = 0;
	if (e == cudaSuccess) {
		median_classify<T><<<(unsigned) blocks, 256, 0, s>>>(P);
		e = cudaGetLastError();
		launches++;
	}
	if (e == cudaSuccess && P.vals != NULL) {
		/* (lacunar leaves are all decided by classify) */
		median_select<T><<<(unsigned) svtgpu_sm_count() * 2, SEL_THREADS,
				   0, s>>>((const T *) P.vals, P.leaf_ptr, P.items,
					   P.nitems, d_out);
		e = cudaGetLastError();
		launches++;
	}
	if (e == cudaSuccess && h_selected != NULL)
		e = cudaMemcpyAsync(h_selected, P.nitems, 16,
				    cudaMemcpyDeviceToHost, s);
	svtgpu_count_launch(launches);
	cudaError_t e2 = svt_free_async(work, s);
	if (e != cudaSuccess)
		return svtgpu_cuda_fail(e, "median kernels", __FILE__, __LINE__);
	if (e2 != cudaSuccess)
		return svtgpu_cuda_fail(e2, "svt_free_async", __FILE__, __LINE__);
	return SVTGPU_OK;
}

int launch_colmedians(svtgpu_matrix *m, int narm, double *d_out,
		      unsigned long long *h_selected, cudaStream_t s)
{
	SVT_ARG(m->val_type == SVTGPU_LGL || m->val_type == SVTGPU_INT ||
		m->val_type == SVTGPU_DOUBLE,
		"colMedians: unsupported value type %d", m->val_type);
	if (h_selected != NULL)
		h_selected[0] = h_selected[1] = 0;
	if (m->nleaf == 0)
		return SVTGPU_OK;
	if (svt_is_double(m->val_type))
		return launch_medians<double>(m, narm, d_out, h_selected, s);
	return launch_medians<int32_t>(m, narm, d_out, h_selected, s);
}

/* host result: out[nleaf] */
int colmedians_host(svtgpu_matrix *m, int narm, double *out)
{
	m->tm.kernel_ms = m->tm.d2h_ms = 0.0;
	m->tm.d2h_bytes = 0.0;
	m->tm.launches = 0;
	m->med_selected = m->med_select_reads = 0;
	if (m->nleaf == 0)
		return SVTGPU_OK;
	cudaStream_t s = 0;
	double *d_out = NULL;
	SVT_CUDA(svt_malloc_async((void **) &d_out, 8 * (size_t) m->nleaf, s));
	unsigned long long sel[2] = {0, 0};
	SvtTimer t;
	int rc = svt_timer_begin(&t, s);
	const int64_t l0 = svtgpu_launch_count();
	if (rc == SVTGPU_OK)
		rc = launch_colmedians(m, narm, d_out, sel, s);
	const int rc2 = svt_timer_end(&t, &m->tm.kernel_ms);
	if (rc == SVTGPU_OK)
		rc = rc2;
	m->tm.launches = (int) (svtgpu_launch_count() - l0);
	if (rc == SVTGPU_OK) {
		rc = svt_timer_begin(&t, s);
		cudaError_t e = cudaMemcpyAsync(out, d_out, 8 * (size_t) m->nleaf,
						cudaMemcpyDeviceToHost, s);
		if (rc == SVTGPU_OK && e != cudaSuccess)
			rc = svtgpu_cuda_fail(e, "cudaMemcpyAsync", __FILE__,
					      __LINE__);
		const int rc3 = svt_timer_end(&t, &m->tm.d2h_ms);
		if (rc == SVTGPU_OK)
			rc = rc3;
		m->tm.d2h_bytes = 8.0 * (double) m->nleaf;
	}
	svt_free_async(d_out, s);
	m->med_selected = (int64_t) sel[0];
	m->med_select_reads = (int64_t) sel[1];
	return rc;
}

}  /* namespace */

extern "C" int svtgpu_colmedians(svtgpu_matrix *m, int narm, double *out)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && (out != NULL || m->nleaf == 0),
		"svtgpu_colmedians: NULL argument");
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	return colmedians_host(m, narm, out);
}

extern "C" int svtgpu_colmedians_dev(svtgpu_matrix *m, int narm,
				     double *d_out, void *stream)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && (d_out != NULL || m->nleaf == 0),
		"svtgpu_colmedians_dev: NULL argument");
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	return launch_colmedians(m, narm, d_out, NULL, (cudaStream_t) stream);
}

extern "C" int svtgpu_rowmedians(svtgpu_matrix *m, int narm, double *out)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && (out != NULL || m->nrow == 0),
		"svtgpu_rowmedians: NULL argument");
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	m->med_selected = m->med_select_reads = 0;
	if (m->nrow == 0)
		return SVTGPU_OK;
	svtgpu_matrix *t = NULL;
	if (m->nnz > 0 && (m->flags & SVTGPU_HAS_OFFS)) {
		SVT_CHECK(svtgpu_ensure_transpose(m, 0, &t));
		SVT_ARG(t != NULL, "rowMedians: the device transpose could not "
			"be built for this matrix");
		const int rc = svtgpu_colmedians(t, narm, out);
		m->tm = t->tm;
		m->med_selected = t->med_selected;
		m->med_select_reads = t->med_select_reads;
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
		rc = svtgpu_colmedians(e, narm, out);
	svtgpu_matrix_free(e);
	return rc;
}

extern "C" int svtgpu_colmedians_selected(const svtgpu_matrix *m,
					  int64_t *n_leaves, int64_t *n_reads)
{
	SVT_ARG(m != NULL, "svtgpu_colmedians_selected: NULL argument");
	if (n_leaves != NULL)
		*n_leaves = m->med_selected;
	if (n_reads != NULL)
		*n_reads = m->med_select_reads;
	return SVTGPU_OK;
}
