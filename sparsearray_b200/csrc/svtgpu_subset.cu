/* Subsetting: x[i, j, ..., drop = FALSE] of a device matrix as a NEW device
 * matrix, with the subscripts already normalised to 0-based positions (R's
 * `[` method turns logical, negative and character subscripts into positive
 * integers before the .Call).  The row subscript `rows` selects and orders
 * the entries inside every leaf; `leaves` gives the source leaf of every
 * result leaf (for an N-d array, the Cartesian product of the subscripts of
 * dimensions 2..N in column-major order, built by the caller).  Both may hold
 * duplicates; NULL means all, in order.  Values are copied bit for bit.
 *
 * Three routes:
 *   gather   (no row subscript, or 0..nrow-1): the gathered source leaves,
 *            laid end to end, form one sequence of entries whose positions
 *            are the scanned leaf lengths (= the result's leaf_ptr).  One
 *            copy pass, nothing counted.
 *   rowmap   (non-decreasing row subscript: which(mask), sorted gene lists,
 *            rep(each =) duplicates): old row r becomes the new rows
 *            [start[r], start[r] + cnt[r]) (cnt 0: dropped), which keeps the
 *            offsets ascending.  A count pass over the gathered sequence
 *            reads offsets and the map (never values), svtgpu_exclusive_scan
 *            of the per-CTA counts places every CTA's output, and a write
 *            pass emits the kept entries and the result's leaf_ptr.
 *   unsorted (any other row subscript): with u = sort(unique(rows)),
 *            x[rows, j] = t( t(x[u, j])[, match(rows, u)] ): the rowmap
 *            route, the device transpose, the gather route, the device
 *            transpose.  Both transposes act on matrices the size of the
 *            result, never on x.
 *
 * Every pass walks the gathered sequence in tiles of SS_TILE entries; lane t
 * of a CTA takes entries t, t + SS_THREADS, ... of the tile, so consecutive
 * lanes read and write consecutive entries of a leaf.  A CTA takes a
 * contiguous run of tiles: it finds its first leaf by one binary search over
 * the scanned lengths, and each lane then carries its leaf forward, galloping
 * over leaves (empty ones included) when it crosses a leaf end.  Every
 * position is int64.
 */
#include "svtgpu_internal.h"

#include <stdlib.h>
#include <string.h>

#include <type_traits>

#define SS_THREADS 256
#define SS_ITEMS   8
#define SS_TILE    (SS_THREADS * SS_ITEMS)
#define SS_WARPS   (SS_THREADS / 32)
#define SS_CTAS_PER_SM 8

struct SsParams {
	const int64_t *xp;        /* x's leaf_ptr */
	const int32_t *xo;        /* x's offsets */
	const void *xv;           /* x's values (NULL: none) */
	const int64_t *leaves;    /* source leaf of every result leaf; NULL: l */
	const int64_t *in_ptr;    /* n_out + 1 scanned gathered lengths */
	int64_t n_out, total;     /* result leaves, gathered entries */
	int64_t tiles_per_cta, ntiles;
	const int2 *map;          /* rowmap: {first new row, count} per old row */
	int64_t *cta_counts;      /* rowmap count pass */
	const int64_t *cta_base;  /* rowmap write pass */
	int64_t *out_ptr;         /* rowmap write pass */
	int32_t *out_offs;
	void *out_vals;           /* NULL: the result stores no values */
	int64_t out_nnz;
};

/* The leaf of gathered entry p as a lane walks forward: entry p is
   x's entry p + base, and the leaf's entries end at `next`. */
struct SsCursor {
	int64_t L, start, next, base;
};

/* first l in [lo, hi] with in_ptr[l + 1] > p */
__device__ __forceinline__ int64_t ss_search(const int64_t *__restrict__ ptr,
					     int64_t lo, int64_t hi, int64_t p)
{
	while (lo < hi) {
		const int64_t mid = lo + ((hi - lo) >> 1);
		if (__ldg(ptr + mid + 1) <= p) lo = mid + 1;
		else                           hi = mid;
	}
	return lo;
}

/* move c to the leaf of p, which lies after c.L: gallop, then bisect */
__device__ __forceinline__ void ss_seek(const SsParams &P, SsCursor &c,
					int64_t p)
{
	int64_t lo = c.L + 1, step = 1, hi;
	for (;;) {
		hi = lo + step - 1;
		if (hi >= P.n_out - 1) {
			hi = P.n_out - 1;
			break;
		}
		if (__ldg(P.in_ptr + hi + 1) > p)
			break;
		lo = hi + 1;
		step <<= 1;
	}
	c.L = ss_search(P.in_ptr, lo, hi, p);
	const int64_t src = P.leaves != NULL ? __ldg(P.leaves + c.L) : c.L;
	c.start = __ldg(P.in_ptr + c.L);
	c.next = __ldg(P.in_ptr + c.L + 1);
	c.base = __ldg(P.xp + src) - c.start;
}

/* this CTA's entries [*e0, *e1) and every lane's cursor just before them */
__device__ __forceinline__ bool ss_begin(const SsParams &P, int64_t *s_leaf,
					 int64_t &e0, int64_t &e1, SsCursor &c)
{
	const int64_t tile0 = (int64_t) blockIdx.x * P.tiles_per_cta;
	e0 = tile0 * SS_TILE;
	int64_t tile1 = tile0 + P.tiles_per_cta;
	if (tile1 > P.ntiles)
		tile1 = P.ntiles;
	e1 = tile1 * SS_TILE < P.total ? tile1 * SS_TILE : P.total;
	if (threadIdx.x == 0 && e0 < e1)
		*s_leaf = ss_search(P.in_ptr, 0, P.n_out - 1, e0);
	__syncthreads();
	if (e0 >= e1)
		return false;
	c.L = *s_leaf - 1;          /* in_ptr[c.L + 1] <= every p of this CTA */
	c.start = c.next = -1;
	c.base = 0;
	return true;
}

/* gather: the result's entry p is x's entry p + base of its leaf.  VS is
   the value size in bytes (0: no values). */
template <int VS>
__global__ void __launch_bounds__(SS_THREADS)
subset_gather(SsParams P)
{
	typedef typename std::conditional<VS == 8, unsigned long long,
					  unsigned>::type TV;
	__shared__ int64_t s_leaf;
	int64_t e0, e1;
	SsCursor c;
	if (!ss_begin(P, &s_leaf, e0, e1, c))
		return;
	const TV *__restrict__ xv = (const TV *) P.xv;
	TV *__restrict__ ov = (TV *) P.out_vals;
	for (int64_t t0 = e0; t0 < e1; t0 += SS_TILE) {
		int64_t src[SS_ITEMS];
		#pragma unroll
		for (int k = 0; k < SS_ITEMS; k++) {
			const int64_t p = t0 + k * SS_THREADS + threadIdx.x;
			src[k] = -1;
			if (p < e1) {
				if (p >= c.next)
					ss_seek(P, c, p);
				src[k] = p + c.base;
			}
		}
		int32_t o[SS_ITEMS];
		TV v[SS_ITEMS];
		#pragma unroll
		for (int k = 0; k < SS_ITEMS; k++) {
			if (src[k] >= 0) {
				o[k] = __ldg(P.xo + src[k]);
				if constexpr (VS != 0)
					v[k] = __ldg(xv + src[k]);
			}
		}
		#pragma unroll
		for (int k = 0; k < SS_ITEMS; k++) {
			if (src[k] >= 0) {
				const int64_t p = t0 + k * SS_THREADS + threadIdx.x;
				P.out_offs[p] = o[k];
				if constexpr (VS != 0)
					ov[p] = v[k];
			}
		}
	}
}

/* rowmap count pass: the entries every CTA keeps (offsets and map only) */
__global__ void __launch_bounds__(SS_THREADS)
subset_rows_count(SsParams P)
{
	__shared__ int64_t s_leaf;
	__shared__ unsigned long long s_warp[SS_WARPS];
	int64_t e0, e1;
	SsCursor c;
	unsigned long long n = 0;
	if (ss_begin(P, &s_leaf, e0, e1, c)) {
		for (int64_t t0 = e0; t0 < e1; t0 += SS_TILE) {
			int64_t src[SS_ITEMS];
			#pragma unroll
			for (int k = 0; k < SS_ITEMS; k++) {
				const int64_t p = t0 + k * SS_THREADS + threadIdx.x;
				src[k] = -1;
				if (p < e1) {
					if (p >= c.next)
						ss_seek(P, c, p);
					src[k] = p + c.base;
				}
			}
			int32_t o[SS_ITEMS];
			#pragma unroll
			for (int k = 0; k < SS_ITEMS; k++)
				if (src[k] >= 0)
					o[k] = __ldg(P.xo + src[k]);
			#pragma unroll
			for (int k = 0; k < SS_ITEMS; k++)
				if (src[k] >= 0)
					n += (unsigned) __ldg(&P.map[o[k]].y);
		}
	}
	#pragma unroll
	for (int s = 16; s > 0; s >>= 1)
		n += __shfl_down_sync(0xFFFFFFFFu, n, s);
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	if (lane == 0)
		s_warp[warp] = n;
	__syncthreads();
	if (threadIdx.x == 0) {
		unsigned long long t = 0;
		for (int w = 0; w < SS_WARPS; w++)
			t += s_warp[w];
		P.cta_counts[blockIdx.x] = (int64_t) t;
	}
}

/* rowmap write pass: the kept entries at their exact places, in the order
   of the gathered sequence, and the result's leaf_ptr.  VS as in gather. */
template <int VS>
__global__ void __launch_bounds__(SS_THREADS)
subset_rows_write(SsParams P)
{
	typedef typename std::conditional<VS == 8, unsigned long long,
					  unsigned>::type TV;
	__shared__ int64_t s_leaf;
	/* per (item k, warp): that warp's count, then its exclusive prefix in
	   the tile's entry order (k major) */
	__shared__ unsigned long long s_pre[SS_ITEMS * SS_WARPS];
	__shared__ unsigned long long s_tile;
	static_assert(SS_ITEMS * SS_WARPS == 64, "two prefix slots per lane");
	int64_t e0, e1;
	SsCursor c;
	if (!ss_begin(P, &s_leaf, e0, e1, c))
		return;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const TV *__restrict__ xv = (const TV *) P.xv;
	TV *__restrict__ ov = (TV *) P.out_vals;
	int64_t base = P.cta_base[blockIdx.x];
	for (int64_t t0 = e0; t0 < e1; t0 += SS_TILE) {
		int64_t src[SS_ITEMS];
		unsigned first = 0;     /* item k is the first entry of its leaf */
		int64_t lfirst[SS_ITEMS];
		#pragma unroll
		for (int k = 0; k < SS_ITEMS; k++) {
			const int64_t p = t0 + k * SS_THREADS + threadIdx.x;
			src[k] = -1;
			lfirst[k] = -1;
			if (p < e1) {
				if (p >= c.next)
					ss_seek(P, c, p);
				src[k] = p + c.base;
				if (p == c.start) {
					first |= 1u << k;
					lfirst[k] = c.L;
				}
			}
		}
		int2 mp[SS_ITEMS];
		#pragma unroll
		for (int k = 0; k < SS_ITEMS; k++) {
			mp[k] = make_int2(0, 0);
			if (src[k] >= 0)
				mp[k] = __ldg(P.map + __ldg(P.xo + src[k]));
		}
		/* warp-inclusive scans of the counts, one per item */
		unsigned long long incl[SS_ITEMS];
		#pragma unroll
		for (int k = 0; k < SS_ITEMS; k++) {
			incl[k] = (unsigned) mp[k].y;
			#pragma unroll
			for (int s = 1; s < 32; s <<= 1) {
				const unsigned long long t =
					__shfl_up_sync(0xFFFFFFFFu, incl[k], s);
				if (lane >= s)
					incl[k] += t;
			}
			if (lane == 31)
				s_pre[k * SS_WARPS + warp] = incl[k];
		}
		__syncthreads();
		if (warp == 0) {
			const unsigned long long a = s_pre[2 * lane];
			const unsigned long long b = s_pre[2 * lane + 1];
			unsigned long long x = a + b;
			#pragma unroll
			for (int s = 1; s < 32; s <<= 1) {
				const unsigned long long t =
					__shfl_up_sync(0xFFFFFFFFu, x, s);
				if (lane >= s)
					x += t;
			}
			s_pre[2 * lane] = x - a - b;
			s_pre[2 * lane + 1] = x - b;
			if (lane == 31)
				s_tile = x;
		}
		__syncthreads();
		#pragma unroll
		for (int k = 0; k < SS_ITEMS; k++) {
			if (src[k] < 0)
				continue;
			const unsigned cnt = (unsigned) mp[k].y;
			int64_t w = base + (int64_t) s_pre[k * SS_WARPS + warp] +
				    (int64_t) (incl[k] - cnt);
			const int64_t p = t0 + k * SS_THREADS + threadIdx.x;
			if ((first >> k) & 1u)  /* this leaf and the empty ones
						   right before it */
				for (int64_t l = lfirst[k];
				     l >= 0 && __ldg(P.in_ptr + l) == p; l--)
					P.out_ptr[l] = w;
			if (p == P.total - 1)   /* leaf_ptr[n_out], trailing empty
						   leaves */
				for (int64_t l = P.n_out;
				     l >= 0 && __ldg(P.in_ptr + l) == P.total; l--)
					P.out_ptr[l] = P.out_nnz;
			if (cnt == 0)
				continue;
			TV v = 0;
			if constexpr (VS != 0)
				v = __ldg(xv + src[k]);
			for (unsigned d = 0; d < cnt; d++, w++) {
				P.out_offs[w] = mp[k].x + (int32_t) d;
				if constexpr (VS != 0)
					ov[w] = v;
			}
		}
		base += (int64_t) s_tile;
		__syncthreads();        /* s_pre and s_tile are reused */
	}
}

__global__ void __launch_bounds__(256)
subset_lengths(const int64_t *__restrict__ xp,
	       const int64_t *__restrict__ leaves, int64_t n,
	       int64_t *__restrict__ len)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t k = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; k < n;
	     k += stride) {
		const int64_t l = leaves != NULL ? leaves[k] : k;
		len[k] = xp[l + 1] - xp[l];
	}
}

/* ---- host side ---- */

static int ss_vsize(const svtgpu_matrix *x)
{
	if (!(x->flags & SVTGPU_HAS_VALS) || x->d_vals == NULL)
		return 0;
	return (int) svt_val_size(x->val_type);
}

static unsigned ss_grid(int64_t n)
{
	const int64_t cap = (int64_t) svtgpu_sm_count() * 8;
	const int64_t g = (n + 255) / 256;
	return (unsigned) (g < 1 ? 1 : g < cap ? g : cap);
}

/* Everything a route allocates; released by ss_release.  The result is
   handed out (and cleared here) only on success. */
struct SsWork {
	svtgpu_matrix *m;       /* result under construction */
	void *d_leaves, *d_map, *d_in_ptr, *d_aux;
	svtgpu_matrix *tmp[2];  /* intermediates of the unsorted route */
};

static void ss_release(SsWork *W, int failed)
{
	if (W->d_leaves) svt_free_async(W->d_leaves, 0);
	if (W->d_map) svt_free_async(W->d_map, 0);
	if (W->d_in_ptr) svt_free_async(W->d_in_ptr, 0);
	if (W->d_aux) svt_free_async(W->d_aux, 0);
	W->d_leaves = W->d_map = W->d_in_ptr = W->d_aux = NULL;
	if (failed)
		cudaDeviceSynchronize();
	for (int i = 0; i < 2; i++) {
		svtgpu_matrix_free(W->tmp[i]);
		W->tmp[i] = NULL;
	}
	if (failed) {
		svtgpu_matrix_free(W->m);
		W->m = NULL;
	}
}

/* d_in_ptr = scanned lengths of the gathered leaves; returns their total */
static int ss_scan_lengths(const svtgpu_matrix *x, SsWork *W,
			   const int64_t *d_leaves, int64_t n_out,
			   cudaStream_t s, int64_t *total)
{
	SVT_CUDA(svt_malloc_async(&W->d_in_ptr,
				  sizeof(int64_t) * (size_t) (n_out + 1), s));
	int64_t *len = NULL;
	SVT_CUDA(svt_malloc_async((void **) &len,
				  sizeof(int64_t) * (size_t) (n_out + 1), s));
	if (n_out > 0) {
		subset_lengths<<<ss_grid(n_out), 256, 0, s>>>(x->d_leaf_ptr,
							      d_leaves, n_out,
							      len);
		svtgpu_count_launch(1);
	}
	cudaError_t e = cudaGetLastError();
	int rc = e == cudaSuccess ? svtgpu_exclusive_scan(len, n_out,
				      (int64_t *) W->d_in_ptr, s)
				  : svtgpu_cuda_fail(e, "subset_lengths",
						     __FILE__, __LINE__);
	svt_free_async(len, s);
	SVT_CHECK(rc);
	SVT_CUDA(cudaMemcpyAsync(total, (int64_t *) W->d_in_ptr + n_out,
				 sizeof(int64_t), cudaMemcpyDeviceToHost, s));
	SVT_CUDA(cudaStreamSynchronize(s));
	return SVTGPU_OK;
}

static void ss_tiles(SsParams &P, unsigned *grid)
{
	P.ntiles = (P.total + SS_TILE - 1) / SS_TILE;
	int64_t g = (int64_t) svtgpu_sm_count() * SS_CTAS_PER_SM;
	if (g > P.ntiles)
		g = P.ntiles;
	if (g < 1)
		g = 1;
	P.tiles_per_cta = (P.ntiles + g - 1) / g;
	*grid = (unsigned) ((P.ntiles + P.tiles_per_cta - 1) / P.tiles_per_cta);
}

static int ss_new_result(const svtgpu_matrix *x, int64_t nrow, int64_t nleaf,
			 int64_t nnz, SsWork *W)
{
	const int flags = nnz > 0 ? SVTGPU_HAS_OFFS |
		(ss_vsize(x) != 0 ? SVTGPU_HAS_VALS : 0) : 0;
	SVT_CHECK(svtgpu_matrix_create(&W->m, nrow, nleaf, nnz, x->val_type,
				       flags));
	/* allocated on the result's upload stream, not ordered against ours */
	SVT_CUDA(cudaStreamSynchronize(W->m->up_stream));
	return SVTGPU_OK;
}

#define SS_LAUNCH_VS(kern, vs, grid, s, P) do { \
		if ((vs) == 8)      kern<8><<<(grid), SS_THREADS, 0, (s)>>>(P); \
		else if ((vs) == 4) kern<4><<<(grid), SS_THREADS, 0, (s)>>>(P); \
		else                kern<0><<<(grid), SS_THREADS, 0, (s)>>>(P); \
	} while (0)

/* gather route: x[, leaves] (d_leaves on the device, NULL: every leaf) */
static int ss_gather(svtgpu_matrix *x, const int64_t *d_leaves, int64_t n_out,
		     SsWork *W, cudaStream_t s, int *launches)
{
	int64_t total = 0;
	SVT_CHECK(ss_scan_lengths(x, W, d_leaves, n_out, s, &total));
	*launches += (n_out > 0) + (n_out > 0 ? 2 : 0);
	SVT_CHECK(ss_new_result(x, x->nrow, n_out, total, W));
	svtgpu_matrix *m = W->m;
	SVT_CUDA(cudaMemcpyAsync(m->d_leaf_ptr, W->d_in_ptr,
				 sizeof(int64_t) * (size_t) (n_out + 1),
				 cudaMemcpyDeviceToDevice, s));
	if (total > 0) {
		SsParams P;
		memset(&P, 0, sizeof(P));
		P.xp = x->d_leaf_ptr;
		P.xo = x->d_offs;
		P.xv = x->d_vals;
		P.leaves = d_leaves;
		P.in_ptr = (const int64_t *) W->d_in_ptr;
		P.n_out = n_out;
		P.total = total;
		P.out_offs = m->d_offs;
		P.out_vals = m->d_vals;
		unsigned grid;
		ss_tiles(P, &grid);
		SS_LAUNCH_VS(subset_gather, ss_vsize(x), grid, s, P);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		(*launches)++;
	}
	return SVTGPU_OK;
}

/* rowmap route: x[rows, leaves] for a non-decreasing row subscript, given
   as its map (d_map: {first new row, count} per row of x) */
static int ss_rows(svtgpu_matrix *x, const int2 *d_map, int64_t new_nrow,
		   const int64_t *d_leaves, int64_t n_out, SsWork *W,
		   cudaStream_t s, int *launches)
{
	int64_t total = 0;
	SVT_CHECK(ss_scan_lengths(x, W, d_leaves, n_out, s, &total));
	*launches += (n_out > 0) + (n_out > 0 ? 2 : 0);
	SsParams P;
	memset(&P, 0, sizeof(P));
	P.xp = x->d_leaf_ptr;
	P.xo = x->d_offs;
	P.xv = x->d_vals;
	P.leaves = d_leaves;
	P.in_ptr = (const int64_t *) W->d_in_ptr;
	P.n_out = n_out;
	P.total = total;
	P.map = d_map;
	unsigned grid = 0;
	int64_t nnz = 0;
	if (total > 0) {
		ss_tiles(P, &grid);
		SVT_CUDA(svt_malloc_async(&W->d_aux, sizeof(int64_t) *
					  (size_t) (2 * grid + 1), s));
		P.cta_counts = (int64_t *) W->d_aux;
		P.cta_base = P.cta_counts + grid;
		subset_rows_count<<<grid, SS_THREADS, 0, s>>>(P);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		SVT_CHECK(svtgpu_exclusive_scan(P.cta_counts, grid,
						(int64_t *) P.cta_base, s));
		*launches += 3;
		SVT_CUDA(cudaMemcpyAsync(&nnz, P.cta_base + grid, sizeof(int64_t),
					 cudaMemcpyDeviceToHost, s));
		SVT_CUDA(cudaStreamSynchronize(s));
	}
	SVT_CHECK(ss_new_result(x, new_nrow, n_out, nnz, W));
	svtgpu_matrix *m = W->m;
	if (total == 0) {
		SVT_CUDA(cudaMemsetAsync(m->d_leaf_ptr, 0,
					 sizeof(int64_t) * (size_t) (n_out + 1),
					 s));
		return SVTGPU_OK;
	}
	P.out_ptr = m->d_leaf_ptr;
	P.out_offs = m->d_offs;   /* NULL when nothing is kept: never written */
	P.out_vals = m->d_vals;
	P.out_nnz = nnz;
	SS_LAUNCH_VS(subset_rows_write, ss_vsize(x), grid, s, P);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	(*launches)++;
	return SVTGPU_OK;
}

static int ss_upload(void **d, const void *h, size_t bytes, cudaStream_t s)
{
	SVT_CUDA(svt_malloc_async(d, bytes > 0 ? bytes : 8, s));
	if (bytes > 0)
		SVT_CUDA(cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, s));
	return SVTGPU_OK;
}

/* the row map of a non-decreasing subscript */
static int ss_upload_map(const int32_t *rows, int64_t n_rows, int64_t nrow,
			 SsWork *W, cudaStream_t s)
{
	int2 *map = (int2 *) calloc((size_t) (nrow > 0 ? nrow : 1),
				    sizeof(int2));
	if (map == NULL) {
		svtgpu_set_error("svtgpu_subset: out of host memory");
		return SVTGPU_ERR_NOMEM;
	}
	for (int64_t k = n_rows - 1; k >= 0; k--) {
		map[rows[k]].x = (int) k;
		map[rows[k]].y++;
	}
	const int rc = ss_upload(&W->d_map, map, sizeof(int2) * (size_t) nrow,
				 s);
	/* pageable source: the copy has been taken once the stream is idle */
	cudaStreamSynchronize(s);
	free(map);
	return rc;
}

/* t(m) as a new matrix the caller owns (built by the device transpose) */
static int ss_transpose(svtgpu_matrix *m, cudaStream_t s, svtgpu_matrix **t)
{
	SVT_CHECK(svtgpu_transpose_fresh(m, s, t));
	if (*t == NULL) {
		svtgpu_set_error("svtgpu_subset: an unsorted row subscript is "
				 "served through the device transpose, which "
				 "declined the %lld x %lld intermediate (a row "
				 "strip would hold 2^32 or more entries); sort "
				 "the row subscript or subset in parts",
				 (long long) m->nrow, (long long) m->nleaf);
		return SVTGPU_ERR_UNSUPPORTED;
	}
	return SVTGPU_OK;
}

static int cmp_i32(const void *a, const void *b)
{
	const int32_t x = *(const int32_t *) a, y = *(const int32_t *) b;
	return (x > y) - (x < y);
}

/* unsorted route: x[rows, leaves] = t( t(x[u, leaves])[, match(rows, u)] ) */
static int ss_unsorted(svtgpu_matrix *x, const int32_t *rows, int64_t n_rows,
		       const int64_t *d_leaves, int64_t n_out, SsWork *W,
		       cudaStream_t s, int *launches)
{
	int32_t *u = (int32_t *) malloc(sizeof(int32_t) * (size_t) n_rows);
	int64_t *pos = (int64_t *) malloc(sizeof(int64_t) * (size_t) n_rows);
	if (u == NULL || pos == NULL) {
		free(u);
		free(pos);
		svtgpu_set_error("svtgpu_subset: out of host memory");
		return SVTGPU_ERR_NOMEM;
	}
	memcpy(u, rows, sizeof(int32_t) * (size_t) n_rows);
	qsort(u, (size_t) n_rows, sizeof(int32_t), cmp_i32);
	int64_t n_u = 0;
	for (int64_t k = 0; k < n_rows; k++)
		if (n_u == 0 || u[n_u - 1] != u[k])
			u[n_u++] = u[k];
	for (int64_t k = 0; k < n_rows; k++) {
		const int32_t *hit = (const int32_t *) bsearch(
			rows + k, u, (size_t) n_u, sizeof(int32_t), cmp_i32);
		pos[k] = hit - u;
	}
	int rc = ss_upload_map(u, n_u, x->nrow, W, s);
	free(u);
	void *d_pos = NULL;
	if (rc == SVTGPU_OK)
		rc = ss_upload(&d_pos, pos, sizeof(int64_t) * (size_t) n_rows, s);
	if (rc == SVTGPU_OK)
		rc = cudaStreamSynchronize(s) == cudaSuccess ? SVTGPU_OK
			: svtgpu_cuda_fail(cudaGetLastError(), "upload",
					   __FILE__, __LINE__);
	free(pos);
	/* w = x[u, leaves] */
	if (rc == SVTGPU_OK)
		rc = ss_rows(x, (const int2 *) W->d_map, n_u, d_leaves, n_out, W,
			     s, launches);
	svtgpu_matrix *w = W->m;
	W->m = NULL;
	W->tmp[0] = w;
	if (rc == SVTGPU_OK && w->nnz == 0) {
		/* nothing kept: the result is empty, no transpose needed */
		rc = ss_new_result(x, n_rows, n_out, 0, W);
		if (rc == SVTGPU_OK && cudaMemsetAsync(W->m->d_leaf_ptr, 0,
				sizeof(int64_t) * (size_t) (n_out + 1), s) !=
				cudaSuccess)
			rc = svtgpu_cuda_fail(cudaGetLastError(), "memset",
					      __FILE__, __LINE__);
	} else if (rc == SVTGPU_OK) {
		svtgpu_matrix *tw = NULL, *v = NULL;
		rc = ss_transpose(w, s, &tw);          /* n_out x n_u */
		if (rc == SVTGPU_OK) {
			svtgpu_matrix_free(w);
			W->tmp[0] = tw;
			if (W->d_in_ptr) svt_free_async(W->d_in_ptr, s);
			W->d_in_ptr = NULL;
			rc = ss_gather(tw, (const int64_t *) d_pos, n_rows, W, s,
				       launches);   /* n_out x n_rows */
		}
		if (rc == SVTGPU_OK) {
			v = W->m;
			W->m = NULL;
			W->tmp[1] = v;
			svtgpu_matrix_free(tw);
			W->tmp[0] = NULL;
			svtgpu_matrix *r = NULL;
			rc = ss_transpose(v, s, &r);    /* n_rows x n_out */
			W->m = r;
		}
		*launches += 2 * 6;   /* the two transposes, roughly */
	}
	if (d_pos != NULL)
		svt_free_async(d_pos, s);
	return rc;
}

/* 0 = rows is NULL or 0 .. nrow-1, 1 = non-decreasing, 2 = other */
static int ss_row_kind(const int32_t *rows, int64_t n_rows, int64_t nrow)
{
	if (rows == NULL)
		return 0;
	int ident = n_rows == nrow, sorted = 1;
	for (int64_t k = 0; k < n_rows; k++) {
		if (rows[k] != k)
			ident = 0;
		if (k > 0 && rows[k] < rows[k - 1]) {
			sorted = 0;
			break;
		}
	}
	return ident ? 0 : sorted ? 1 : 2;
}

extern "C" int svtgpu_subset(svtgpu_matrix *x, const int32_t *rows,
			     int64_t n_rows, const int64_t *leaves,
			     int64_t n_leaves, svtgpu_matrix **out)
{
	SVT_ARG(x != NULL && out != NULL, "svtgpu_subset: NULL argument");
	*out = NULL;
	SVT_ARG(svt_ew_type_ok(x->val_type),
		"svtgpu_subset: only logical, integer and double matrices are "
		"supported");
	SVT_ARG(x->nrow >= 0 && x->nleaf >= 0 && x->nnz >= 0,
		"svtgpu_subset: bad matrix");
	if (rows == NULL)
		n_rows = x->nrow;
	if (leaves == NULL)
		n_leaves = x->nleaf;
	SVT_ARG(n_rows >= 0 && n_rows <= INT32_MAX,
		"svtgpu_subset: the row subscript must have between 0 and "
		"2^31 - 1 elements (got %lld)", (long long) n_rows);
	SVT_ARG(n_leaves >= 0, "svtgpu_subset: negative number of leaves");
	if (n_leaves >= INT32_MAX) {
		svtgpu_set_error("svtgpu_subset: at most 2^31 - 2 result leaves "
				 "are supported (got %lld)",
				 (long long) n_leaves);
		return SVTGPU_ERR_UNSUPPORTED;
	}
	if (rows != NULL)
		for (int64_t k = 0; k < n_rows; k++)
			SVT_ARG(rows[k] >= 0 && rows[k] < x->nrow,
				"svtgpu_subset: row subscript element %lld (%d) "
				"is outside [0, %lld)", (long long) k, rows[k],
				(long long) x->nrow);
	if (leaves != NULL)
		for (int64_t k = 0; k < n_leaves; k++)
			SVT_ARG(leaves[k] >= 0 && leaves[k] < x->nleaf,
				"svtgpu_subset: leaf subscript element %lld "
				"(%lld) is outside [0, %lld)", (long long) k,
				(long long) leaves[k], (long long) x->nleaf);
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(x->nnz == 0 || (x->flags & SVTGPU_HAS_OFFS),
		"svtgpu_subset: the matrix was uploaded without row offsets");
	SVT_CHECK(svtgpu_matrix_finish_upload(x));
	const int kind = ss_row_kind(rows, n_rows, x->nrow);
	cudaStream_t s = 0;
	SsWork W;
	memset(&W, 0, sizeof(W));
	SvtTimer tm;
	SVT_CHECK(svt_timer_begin(&tm, s));
	int launches = 0;
	int rc = SVTGPU_OK;
	if (leaves != NULL)
		rc = ss_upload(&W.d_leaves, leaves,
			       sizeof(int64_t) * (size_t) n_leaves, s);
	const int64_t *d_leaves = (const int64_t *) W.d_leaves;
	if (rc == SVTGPU_OK && kind == 0) {
		rc = ss_gather(x, d_leaves, n_leaves, &W, s, &launches);
	} else if (rc == SVTGPU_OK && kind == 1) {
		rc = ss_upload_map(rows, n_rows, x->nrow, &W, s);
		if (rc == SVTGPU_OK)
			rc = ss_rows(x, (const int2 *) W.d_map, n_rows, d_leaves,
				     n_leaves, &W, s, &launches);
	} else if (rc == SVTGPU_OK) {
		rc = ss_unsorted(x, rows, n_rows, d_leaves, n_leaves, &W, s,
				 &launches);
	}
	double ms = 0.0;
	const int rt = svt_timer_end(&tm, &ms);     /* frees its events */
	if (rc == SVTGPU_OK)
		rc = rt;
	ss_release(&W, rc != SVTGPU_OK);
	if (rc != SVTGPU_OK)
		return rc;
	svtgpu_matrix *m = W.m;
	m->tm.kernel_ms = ms;
	m->tm.launches = launches;
	*out = m;
	return SVTGPU_OK;
}
