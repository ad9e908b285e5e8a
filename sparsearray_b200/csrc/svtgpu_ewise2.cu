/* Element-wise operations between two matrices of the same geometry:
 * `x + y`, `x - y`, `x * y`, `x & y`, `x | y`, `x > y`, `x < y`, `x != y`.
 * The value rules (types, NA / NaN bits, integer overflow, what is dropped)
 * and the refusals are in svt_semantics.h (svt_ew2_*); this file merges the
 * two operands' leaves on the device.
 *
 * Reference: the dense semantics of base R (src/main/arithmetic.c, relop.c,
 * logic.c); the SparseArray package merges the two leaves on the host.
 *
 * Every leaf l of the result is the merge of x's and y's offset lists of
 * leaf l.  Laid end to end over all leaves, these merges form one sequence
 * of nnz(x) + nnz(y) "merge items" (an entry stored on both sides is two
 * items, x's first; the second produces nothing), and both operands are
 * consumed front to back along it.  The sequence is cut into tiles of
 * E2_TILE items, one CTA each, E2_ITEMS consecutive items per lane.  A lane
 * finds its leaf by binary search over leaf_ptr(x) + leaf_ptr(y) (inside the
 * tile's leaf range, which two lanes find first) and its place inside the
 * leaf by a merge-path search (the split of its first item between x and
 * y), then walks its items, crossing into the next leaf where one ends.  So
 * no lane walks a whole leaf, leaves of any length (and an empty side beside
 * a long one) cost the same per item, and every position is int64.
 *
 * Two passes over the items, the same walk:
 *   count  the kept entries of every tile (the rule applied, so exact) and
 *          the flags (integer overflow, an NA kept);
 *   scan   svtgpu_exclusive_scan of the tile counts: each tile's first
 *          output position and the result's nnz;
 *   write  each CTA scans its lanes' counts and writes the kept entries
 *          (offsets, and values unless the result is lacunar) at their
 *          positions; the lane holding the first item of a leaf writes that
 *          leaf's leaf_ptr (and the empty leaves just before it).
 * Each pass reads both operands' offsets and values (a lacunar side: its
 * offsets only); the result is written once, at its exact size, so nothing
 * is ever compacted.  Loads are 4 / 8-byte, so no array needs 16-byte
 * alignment.
 */
#include "svtgpu_internal.h"

#include <string.h>

#include <type_traits>

#define E2_THREADS 256
#define E2_ITEMS   8                          /* merge items per lane */
#define E2_TILE    (E2_THREADS * E2_ITEMS)    /* merge items per CTA */
#define E2_END     INT32_MAX                  /* past the last offset */

enum { E2_IN_INT = 0, E2_IN_DBL = 1, E2_IN_ONES = 2 };
enum { E2_RES_INT = 0, E2_RES_DBL = 1, E2_RES_LGL = 2 };

struct E2Params {
	const int64_t *xp, *yp;        /* leaf_ptr */
	const int32_t *xo, *yo;        /* offsets */
	const void *xv, *yv;           /* values (unused for a lacunar side) */
	int64_t nleaf, total;          /* total = nnz(x) + nnz(y) */
	int op;
	int64_t *tile_counts;          /* count pass */
	uint32_t *flags;               /* count pass */
	const int64_t *tile_base;      /* write pass */
	int64_t *out_ptr;
	int32_t *out_offs;
	void *out_vals;                /* NULL: lacunar result */
	int64_t out_nnz;
};

/* first merge item of leaf l */
__device__ __forceinline__ int64_t e2_cp(const E2Params &P, int64_t l)
{
	return __ldg(P.xp + l) + __ldg(P.yp + l);
}

/* the leaf of merge item p: first l in [lo, hi] whose items end after p */
__device__ __forceinline__ int64_t e2_leaf_of(const E2Params &P, int64_t lo,
					      int64_t hi, int64_t p)
{
	while (lo < hi) {
		const int64_t mid = lo + ((hi - lo) >> 1);
		if (e2_cp(P, mid + 1) <= p) lo = mid + 1;
		else                        hi = mid;
	}
	return lo;
}

/* merge path: how many of x's nx offsets are among the first d items of the
   merged order, x first on equal offsets */
__device__ __forceinline__ int64_t e2_split(const int32_t *__restrict__ xo,
					    int64_t nx,
					    const int32_t *__restrict__ yo,
					    int64_t ny, int64_t d)
{
	int64_t lo = d > ny ? d - ny : 0, hi = d < nx ? d : nx;
	while (lo < hi) {
		const int64_t mid = (lo + hi) >> 1;
		if (__ldg(xo + mid) <= __ldg(yo + d - 1 - mid)) lo = mid + 1;
		else                                          hi = mid;
	}
	return lo;
}

/* one stored value as the rules take it: int32, double, NA flag */
template <int IN>
__device__ __forceinline__ void e2_load(const void *vals, int64_t e,
					int32_t &i, double &d, int &na)
{
	if (IN == E2_IN_ONES) {
		i = 1;
		d = 1.0;
		na = 0;
	} else if (IN == E2_IN_INT) {
		i = __ldg((const int32_t *) vals + e);
		d = (double) i;
		na = i == SVT_NA_INT;
	} else {
		d = __ldg((const double *) vals + e);
		i = 0;
		na = svt_is_na_real(d);
	}
}

/* the rule for one result position; false: the value is 0 / FALSE */
template <int RES, typename TOut>
__device__ __forceinline__ bool e2_rule(int op, int32_t xi, double xd, int xna,
					int32_t yi, double yd, int yna,
					TOut &r, uint32_t &fl)
{
	if (RES == E2_RES_INT) {
		const int32_t v = svt_ew2_int(op, xi, yi, &fl);
		r = (TOut) v;
		return v != 0;
	}
	if (RES == E2_RES_DBL) {
		const double v = svt_ew2_dbl(op, xd, xna, yd, yna);
		r = (TOut) v;
		return !(v == 0.0);
	}
	const int c = svt_ew2_lgl(op, xd, xna, yd, yna);
	if (c == SVT_CMP_NA)
		fl |= SVT_EW_NA_KEPT;
	r = (TOut) (c == SVT_CMP_NA ? SVT_NA_INT : 1);
	return c != SVT_CMP_DROP;
}

template <int INX, int INY, int RES, bool WRITE>
__global__ void __launch_bounds__(E2_THREADS)
ewise2_merge(E2Params P)
{
	typedef typename std::conditional<RES == E2_RES_DBL, double,
					  int32_t>::type TOut;
	__shared__ int64_t s_leaf[2];
	__shared__ unsigned s_warp[E2_THREADS / 32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int64_t t0 = (int64_t) blockIdx.x * E2_TILE;
	const int64_t t1 = t0 + E2_TILE < P.total ? t0 + E2_TILE : P.total;
	if (threadIdx.x < 2)
		s_leaf[threadIdx.x] = e2_leaf_of(P, 0, P.nleaf - 1,
						 threadIdx.x == 0 ? t0 : t1 - 1);
	__syncthreads();
	const int64_t p0 = t0 + (int64_t) threadIdx.x * E2_ITEMS;
	const int64_t p1 = p0 + E2_ITEMS < t1 ? p0 + E2_ITEMS : t1;
	uint32_t fl = 0;
	unsigned keep = 0, lstart = 0;
	int64_t lfirst = -1;
	int32_t ro[E2_ITEMS];
	TOut rv[E2_ITEMS];
	if (p0 < p1) {
		int64_t L = e2_leaf_of(P, s_leaf[0], s_leaf[1], p0);
		int64_t xa = __ldg(P.xp + L), ya = __ldg(P.yp + L);
		int64_t nx = __ldg(P.xp + L + 1) - xa, ny = __ldg(P.yp + L + 1) - ya;
		int64_t i = e2_split(P.xo + xa, nx, P.yo + ya, ny,
				     p0 - (xa + ya));
		int64_t j = p0 - (xa + ya) - i;
		int32_t cx = i < nx ? __ldg(P.xo + xa + i) : E2_END;
		int32_t cy = j < ny ? __ldg(P.yo + ya + j) : E2_END;
		int32_t px = i > 0 ? __ldg(P.xo + xa + i - 1) : -1;
		#pragma unroll
		for (int k = 0; k < E2_ITEMS; k++) {
			if (p0 + k >= p1)
				continue;
			if (i == nx && j == ny) {        /* next nonempty leaf */
				do {
					L++;
					xa = __ldg(P.xp + L);
					ya = __ldg(P.yp + L);
					nx = __ldg(P.xp + L + 1) - xa;
					ny = __ldg(P.yp + L + 1) - ya;
				} while (nx + ny == 0);
				i = j = 0;
				cx = nx > 0 ? __ldg(P.xo + xa) : E2_END;
				cy = ny > 0 ? __ldg(P.yo + ya) : E2_END;
				px = -1;
			}
			if (i == 0 && j == 0) {
				lstart |= 1u << k;
				if (lfirst < 0)
					lfirst = L;
			}
			int32_t xi = 0, yi = 0, off;
			double xd = 0.0, yd = 0.0;
			int xna = 0, yna = 0;
			bool emit = true;
			if (cx <= cy) {                  /* x's entry, maybe both */
				off = cx;
				e2_load<INX>(P.xv, xa + i, xi, xd, xna);
				if (cy == cx)
					e2_load<INY>(P.yv, ya + j, yi, yd, yna);
				px = cx;
				i++;
				cx = i < nx ? __ldg(P.xo + xa + i) : E2_END;
			} else {                         /* y's entry */
				off = cy;
				emit = px != cy;         /* else served with x's */
				if (emit)
					e2_load<INY>(P.yv, ya + j, yi, yd, yna);
				j++;
				cy = j < ny ? __ldg(P.yo + ya + j) : E2_END;
			}
			if (emit && e2_rule<RES>(P.op, xi, xd, xna, yi, yd, yna,
						 rv[k], fl)) {
				keep |= 1u << k;
				ro[k] = off;
			}
		}
	}
	const unsigned n = __popc(keep);
	/* block scan of the lanes' counts */
	unsigned incl = n;
	#pragma unroll
	for (int s = 1; s < 32; s <<= 1) {
		const unsigned t = __shfl_up_sync(0xFFFFFFFFu, incl, s);
		if (lane >= s)
			incl += t;
	}
	if (lane == 31)
		s_warp[warp] = incl;
	__syncthreads();
	if (warp == 0) {
		const unsigned w = lane < E2_THREADS / 32 ? s_warp[lane] : 0u;
		unsigned wi = w;
		#pragma unroll
		for (int s = 1; s < E2_THREADS / 32; s <<= 1) {
			const unsigned t = __shfl_up_sync(0xFFFFFFFFu, wi, s);
			if (lane >= s)
				wi += t;
		}
		if (lane < E2_THREADS / 32)
			s_warp[lane] = wi - w;           /* exclusive */
		if (!WRITE && lane == E2_THREADS / 32 - 1)
			P.tile_counts[blockIdx.x] = (int64_t) wi;
	}
	if (!WRITE) {
		fl = __reduce_or_sync(0xFFFFFFFFu, fl);
		if (lane == 0 && fl != 0)
			atomicOr(P.flags, fl);
		return;
	}
	__syncthreads();
	if (p0 >= p1)
		return;
	int64_t w = P.tile_base[blockIdx.x] + s_warp[warp] + (incl - n);
	int64_t Lw = lfirst;
	bool first = true;
	#pragma unroll
	for (int k = 0; k < E2_ITEMS; k++) {
		if ((lstart >> k) & 1u) {
			if (!first) {                    /* next nonempty leaf */
				Lw++;
				while (e2_cp(P, Lw + 1) == e2_cp(P, Lw))
					Lw++;
			}
			first = false;
			/* this leaf and the empty leaves right before it */
			for (int64_t l = Lw; l >= 0 && e2_cp(P, l) == p0 + k; l--)
				P.out_ptr[l] = w;
		}
		if ((keep >> k) & 1u) {
			P.out_offs[w] = ro[k];
			if (P.out_vals != NULL)
				((TOut *) P.out_vals)[w] = rv[k];
			w++;
		}
	}
	if (p1 == P.total)      /* leaf_ptr[nleaf] and trailing empty leaves */
		for (int64_t l = P.nleaf; l >= 0 && e2_cp(P, l) == P.total; l--)
			P.out_ptr[l] = P.out_nnz;
}

template <int INX, int INY, int RES>
static void e2_launch3(bool write, unsigned grid, cudaStream_t s,
		       const E2Params &P)
{
	if (write)
		ewise2_merge<INX, INY, RES, true><<<grid, E2_THREADS, 0, s>>>(P);
	else
		ewise2_merge<INX, INY, RES, false><<<grid, E2_THREADS, 0, s>>>(P);
}

/* Dispatch on the result type, which follows the operands' types, not on
   how their values are stored: a double matrix without a value array (all
   leaves lacunar) reads as E2_IN_ONES yet gives a double Arith result.  An
   integer result never has a double side (ewise2_run checks), so it needs
   no E2_IN_DBL form. */
template <int INX, int INY>
static void e2_launch2(int res, bool write, unsigned grid, cudaStream_t s,
		       const E2Params &P)
{
	if (res == E2_RES_LGL) {
		e2_launch3<INX, INY, E2_RES_LGL>(write, grid, s, P);
	} else if (res == E2_RES_DBL) {
		e2_launch3<INX, INY, E2_RES_DBL>(write, grid, s, P);
	} else {
		if constexpr (INX != E2_IN_DBL && INY != E2_IN_DBL)
			e2_launch3<INX, INY, E2_RES_INT>(write, grid, s, P);
	}
}

template <int INX>
static void e2_launch1(int iny, int res, bool write, unsigned grid,
		       cudaStream_t s, const E2Params &P)
{
	if (iny == E2_IN_INT)
		e2_launch2<INX, E2_IN_INT>(res, write, grid, s, P);
	else if (iny == E2_IN_DBL)
		e2_launch2<INX, E2_IN_DBL>(res, write, grid, s, P);
	else
		e2_launch2<INX, E2_IN_ONES>(res, write, grid, s, P);
}

static void e2_launch(int inx, int iny, int res, bool write, unsigned grid,
		      cudaStream_t s, const E2Params &P)
{
	if (inx == E2_IN_INT)
		e2_launch1<E2_IN_INT>(iny, res, write, grid, s, P);
	else if (inx == E2_IN_DBL)
		e2_launch1<E2_IN_DBL>(iny, res, write, grid, s, P);
	else
		e2_launch1<E2_IN_ONES>(iny, res, write, grid, s, P);
}

static int e2_in_kind(const svtgpu_matrix *m)
{
	if (!(m->flags & SVTGPU_HAS_VALS) || m->d_vals == NULL)
		return E2_IN_ONES;
	return svt_is_double(m->val_type) ? E2_IN_DBL : E2_IN_INT;
}

struct E2Work {
	svtgpu_matrix *m;
	void *d_aux;        /* flags word, tile counts, tile bases */
};

static int ewise2_run(svtgpu_matrix *x, svtgpu_matrix *y, int op,
		      E2Work *W, svtgpu_matrix **out, int *warn)
{
	cudaStream_t s = 0;
	const int out_type = svt_ew2_result_type(op, x->val_type, y->val_type);
	const int res = out_type == SVTGPU_DOUBLE ? E2_RES_DBL
		      : out_type == SVTGPU_LGL ? E2_RES_LGL : E2_RES_INT;
	const int64_t nleaf = x->nleaf, total = x->nnz + y->nnz;
	const int64_t ntiles = (total + E2_TILE - 1) / E2_TILE;
	SVT_ARG(ntiles < INT32_MAX, "svtgpu_ewise2: too many entries");
	SVT_ARG(res != E2_RES_INT || (e2_in_kind(x) != E2_IN_DBL &&
				      e2_in_kind(y) != E2_IN_DBL),
		"svtgpu_ewise2: integer result from a double operand");
	SvtTimer tm;
	SVT_CHECK(svt_timer_begin(&tm, s));
	int launches = 0;
	uint32_t flags = 0;
	int64_t nnz = 0;
	E2Params P;
	memset(&P, 0, sizeof(P));
	if (total > 0) {
		SVT_CUDA(svt_malloc_async(&W->d_aux, 16 + sizeof(int64_t) *
					  (size_t) (2 * ntiles + 1), s));
		P.xp = x->d_leaf_ptr;
		P.yp = y->d_leaf_ptr;
		P.xo = x->d_offs;
		P.yo = y->d_offs;
		P.xv = x->d_vals;
		P.yv = y->d_vals;
		P.nleaf = nleaf;
		P.total = total;
		P.op = op;
		P.flags = (uint32_t *) W->d_aux;
		P.tile_counts = (int64_t *) ((char *) W->d_aux + 16);
		P.tile_base = P.tile_counts + ntiles;
		SVT_CUDA(cudaMemsetAsync(P.flags, 0, 16, s));
		e2_launch(e2_in_kind(x), e2_in_kind(y), res, false,
			  (unsigned) ntiles, s, P);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		SVT_CHECK(svtgpu_exclusive_scan(P.tile_counts, ntiles,
						(int64_t *) P.tile_base, s));
		launches += 3;      /* the scan counts its own two */
		SVT_CUDA(cudaMemcpyAsync(&nnz, P.tile_base + ntiles,
					 sizeof(int64_t), cudaMemcpyDeviceToHost,
					 s));
		SVT_CUDA(cudaMemcpyAsync(&flags, P.flags, sizeof(flags),
					 cudaMemcpyDeviceToHost, s));
		SVT_CUDA(cudaStreamSynchronize(s));
	}
	const int vals = res != E2_RES_LGL || (flags & SVT_EW_NA_KEPT);
	SVT_CHECK(svtgpu_matrix_create(&W->m, x->nrow, nleaf, nnz, out_type,
		nnz > 0 ? SVTGPU_HAS_OFFS | (vals ? SVTGPU_HAS_VALS : 0) : 0));
	svtgpu_matrix *m = W->m;
	/* allocated on m's upload stream, which does not order against s */
	SVT_CUDA(cudaStreamSynchronize(m->up_stream));
	if (nnz == 0) {
		SVT_CUDA(cudaMemsetAsync(m->d_leaf_ptr, 0,
					 sizeof(int64_t) * (size_t) (nleaf + 1),
					 s));
	} else {
		P.out_ptr = m->d_leaf_ptr;
		P.out_offs = m->d_offs;
		P.out_vals = vals ? m->d_vals : NULL;
		P.out_nnz = nnz;
		e2_launch(e2_in_kind(x), e2_in_kind(y), res, true,
			  (unsigned) ntiles, s, P);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		launches++;
	}
	double ms = 0.0;
	SVT_CHECK(svt_timer_end(&tm, &ms));
	W->m = NULL;
	m->leaf_base = x->leaf_base;
	m->tm.kernel_ms = ms;
	m->tm.launches = launches;
	*out = m;
	if (warn != NULL)
		*warn = (int) (flags & SVTGPU_EW_WARN_INT_OVERFLOW);
	return SVTGPU_OK;
}

extern "C" int svtgpu_ewise2(svtgpu_matrix *x, svtgpu_matrix *y, int op,
			     svtgpu_matrix **out, int *warn)
{
	SVT_ARG(x != NULL && y != NULL && out != NULL,
		"svtgpu_ewise2: NULL argument");
	*out = NULL;
	if (warn != NULL)
		*warn = 0;
	if (!svt_ew2_admitted(op)) {
		svtgpu_set_error("svtgpu_ewise2: opcode %d is not an operation "
				 "between two matrices that keeps the implicit "
				 "zeros at zero (supported: \"+\", \"-\", \"*\", "
				 "\"&\", \"|\", \">\", \"<\", \"!=\")", op);
		return SVTGPU_ERR_ARG;
	}
	SVT_ARG(svt_ew_type_ok(x->val_type) && svt_ew_type_ok(y->val_type),
		"svtgpu_ewise2: only logical, integer and double matrices are "
		"supported");
	SVT_ARG(x->nrow == y->nrow && x->nleaf == y->nleaf,
		"svtgpu_ewise2: non-conformable arrays (%lld x %lld and "
		"%lld x %lld)", (long long) x->nrow, (long long) x->nleaf,
		(long long) y->nrow, (long long) y->nleaf);
	SVT_ARG(x->nnz >= 0 && y->nnz >= 0 && x->nleaf >= 0,
		"svtgpu_ewise2: bad matrix");
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG((x->nnz == 0 || (x->flags & SVTGPU_HAS_OFFS)) &&
		(y->nnz == 0 || (y->flags & SVTGPU_HAS_OFFS)),
		"svtgpu_ewise2: a matrix was uploaded without row offsets");
	SVT_CHECK(svtgpu_matrix_finish_upload(x));
	if (y != x)
		SVT_CHECK(svtgpu_matrix_finish_upload(y));
	E2Work W;
	memset(&W, 0, sizeof(W));
	const int rc = ewise2_run(x, y, op, &W, out, warn);
	if (W.d_aux != NULL)
		svt_free_async(W.d_aux, 0);
	if (rc != SVTGPU_OK) {
		cudaDeviceSynchronize();
		svtgpu_matrix_free(W.m);
		*out = NULL;
	}
	return rc;
}
