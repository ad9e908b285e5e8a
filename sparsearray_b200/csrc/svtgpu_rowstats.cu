/* Row statistics of a device CSC -- the replacement for REC_rowStats_SVT() and
 * the update_out_for_row*() scatter loops, which the reference runs on a
 * single thread (src/SparseArray_matrixStats.c:498-829).
 *
 * Every stored value (offset, value) updates one of nrow per-row slots.  The
 * result is staged as a per-row "state" (see svt_semantics.h) which a tiny
 * kernel turns into R's answer; with a column-sharded matrix the states of the
 * shards are summed (NCCL allreduce) between the two steps.
 *
 *   row_hist (default for sums / moments of integer and lacunar input whose
 *       rows fit one SM)  shared-memory histogram: one CTA per SM streams its
 *       chunk of (offset, value) pairs and adds into one integer cell per row
 *       with shared-memory atomics; exact, so order-free.
 *   row_strips + row_combine (min / max, double input, SVTGPU_ROW_HIST=off)
 *       atomic-free two-pass scheme.  The grid is nchunks x ntiles CTAs.  A
 *       CTA owns the leaves of one chunk (balanced by nnz) and the rows of one
 *       tile, whose accumulators live in shared memory; every warp owns a
 *       strip of those rows.  Offsets ascend strictly inside a leaf
 *       (src/leaf_utils.h:14-15), so the part of a leaf that falls into a
 *       strip is one contiguous sub-run (found once per matrix by row_split)
 *       with distinct rows: plain shared-memory read-modify-writes, no
 *       atomics, no barrier.  Pass 2 (row_combine) sums the per-chunk partial
 *       vectors in a fixed order, so results do not depend on scheduling.
 *       NA/NaN are rare: they bypass the accumulators and bump per-row
 *       counters in the state with global atomics.
 *   row_tiles (SVTGPU_ROW_IMPL=tiles)  the first version of that scheme: a
 *       producer warp streams runs through a TMA ring, one named barrier per
 *       leaf.  Kept as a cross-check; slower (see DESIGN.md).
 *   row_flat             one thread per stored value, global atomics; used for
 *       countNAs/anyNA (which then only reads offsets of NA entries), for
 *       matrices with more rows than the tiled scheme covers, and as a
 *       cross-check (SVTGPU_ROW_IMPL=flat).
 */
#include "svtgpu_internal.h"
#include "svt_ptx.cuh"

#include <string.h>

namespace {

enum RowClass { RC_COUNT = 0, RC_SUM, RC_X2, RC_MINMAX };

inline int row_class_of(int opcode)
{
	switch (opcode) {
	    case SVTGPU_OP_ANYNA: case SVTGPU_OP_COUNTNAS: return RC_COUNT;
	    case SVTGPU_OP_SUM:                            return RC_SUM;
	    case SVTGPU_OP_CENTERED_X2_SUM:                return RC_X2;
	    case SVTGPU_OP_MIN: case SVTGPU_OP_MAX:        return RC_MINMAX;
	}
	return -1;
}

/* classification shared by every row kernel: returns 0 regular, 1 NA, 2 NaN
   and the value as a double */
__device__ __forceinline__ int classify(int32_t x, double &v)
{
	v = (double) x;
	return x == SVT_NA_INT ? 1 : 0;
}

__device__ __forceinline__ int classify(double x, double &v)
{
	v = x;
	if (!svt_isnan(x))
		return 0;
	return (uint32_t) svt_d2u(x) == 1954u ? 1 : 2;
}

/* last leaf that put an NA (kind 0) / NaN (1) into a row: see
   SVT_ROW_SLOT_LAST_* in svt_semantics.h */
__device__ __forceinline__ void atomic_max_double(double *addr, double v);
__device__ __forceinline__ void note_last(double *state, int64_t nrow,
					  int off, int kind, double pos)
{
	atomic_max_double(&state[(size_t) (SVT_ROW_SLOT_LAST_NA + kind) * nrow +
				 off], pos);
}

__device__ __forceinline__ void atomic_min_double(double *addr, double v)
{
	unsigned long long *a = (unsigned long long *) addr;
	unsigned long long old = *a;
	while (v < __longlong_as_double((long long) old)) {
		unsigned long long assumed = old;
		old = atomicCAS(a, assumed,
				(unsigned long long) __double_as_longlong(v));
		if (old == assumed)
			break;
	}
}

__device__ __forceinline__ void atomic_max_double(double *addr, double v)
{
	unsigned long long *a = (unsigned long long *) addr;
	unsigned long long old = *a;
	while (v > __longlong_as_double((long long) old)) {
		unsigned long long assumed = old;
		old = atomicCAS(a, assumed,
				(unsigned long long) __double_as_longlong(v));
		if (old == assumed)
			break;
	}
}

/* ------------------------------------------------------------------------
 * row_flat
 */
template <int RC, typename T, bool LACUNAR>
__global__ void __launch_bounds__(256)
row_flat(const int32_t *__restrict__ offs, const T *__restrict__ vals,
	 int64_t nnz, int64_t nrow, int is_min, double *state)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t e = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     e < nnz; e += stride) {
		double v = 1.0;
		int cls = 0;
		if (!LACUNAR)
			cls = classify(vals[e], v);
		if (RC == RC_COUNT) {
			if (cls != 0)
				atomicAdd(&state[(cls == 1 ? SVT_ROW_SLOT_NA
					: SVT_ROW_SLOT_NAN) * nrow + offs[e]],
					1.0);
			continue;
		}
		const int64_t r = offs[e];
		if (RC == RC_MINMAX)
			atomicAdd(&state[SVT_ROW_SLOT_CVG * nrow + r], 1.0);
		if (cls != 0) {
			atomicAdd(&state[(cls == 1 ? SVT_ROW_SLOT_NA
					: SVT_ROW_SLOT_NAN) * nrow + r], 1.0);
			continue;
		}
		if (RC == RC_SUM || RC == RC_X2)
			atomicAdd(&state[SVT_ROW_SLOT_SUM * nrow + r], v);
		if (RC == RC_X2)
			atomicAdd(&state[SVT_ROW_SLOT_SUM2 * nrow + r], v * v);
		if (RC == RC_MINMAX) {
			if (is_min)
				atomic_min_double(&state[SVT_ROW_SLOT_EXT *
							 nrow + r], v);
			else
				atomic_max_double(&state[SVT_ROW_SLOT_EXT *
							 nrow + r], v);
		}
	}
}

__global__ void fill_doubles(double *p, int64_t n, double v)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     i < n; i += stride)
		p[i] = v;
}

/* ------------------------------------------------------------------------
 * row_split: for every leaf and every interior tile boundary b*tile_rows, the
 * leaf-relative position of the first offset >= the boundary.
 */
__global__ void __launch_bounds__(256)
row_split(const int32_t *__restrict__ offs,
	  const int64_t *__restrict__ leaf_ptr, int64_t nleaf, int ntiles,
	  int tile_rows, int32_t *__restrict__ split)
{
	const int64_t total = nleaf * (ntiles - 1);
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     i < total; i += stride) {
		/* the searches of one leaf sit next to each other: its offsets
		   come from HBM once and serve every boundary out of L1 / L2
		   (boundary-major order read 74 GB for 9.4 GB of offsets) */
		const int64_t leaf = i / (ntiles - 1), b = i - leaf * (ntiles - 1);
		const int64_t start = leaf_ptr[leaf];
		const int32_t bound = (int32_t) ((b + 1) * tile_rows);
		int32_t lo = 0, hi = (int32_t) (leaf_ptr[leaf + 1] - start);
		while (lo < hi) {
			int32_t mid = lo + ((hi - lo) >> 1);
			if (offs[start + mid] < bound) lo = mid + 1;
			else                           hi = mid;
		}
		split[b * nleaf + leaf] = lo;
	}
}

/* ------------------------------------------------------------------------
 * row_tiles
 */

#define ROW_NS 4            /* ring depth */
#define ROW_CONSUMERS 256   /* consumer threads (8 warps) */
#define ROW_CWARPS (ROW_CONSUMERS / 32)
#define ROW_THREADS (ROW_CONSUMERS + 32)
#define ROW_UNROLL 4        /* independent read-modify-writes per thread */

struct RowTileParams {
	const int32_t *offs;
	const void *vals;          /* NULL: lacunar */
	const int64_t *leaf_ptr;
	const int32_t *split;      /* NULL when ntiles == 1 */
	int64_t nleaf, nnz, nrow;
	int ntiles, tile_rows, nchunks;
	int stage_elems;           /* SE */
	int is_min;
	int64_t flush_leaves;      /* int32 accumulators: flush every F leaves */
	double *part;              /* [nchunks][nacc][nrow] */
	double *state;             /* NA / NaN counters (global atomics) */
};

enum { RI_LEAF_END = 1, RI_FLUSH = 2, RI_STOP = 4 };

struct __align__(16) RowItem {
	int32_t n;           /* elements of the run held by the stage */
	int32_t odelta;      /* first element's index in the offs stage */
	int32_t vdelta;      /* first element's index in the vals stage */
	int32_t flags;
};

__device__ __forceinline__ void consumer_barrier(void)
{
	asm volatile("bar.sync 1, %0;" :: "n"(ROW_CONSUMERS) : "memory");
}

template <typename ACC> struct AccTraits;
template <> struct AccTraits<int32_t> {
	static __device__ __forceinline__ int32_t ext_init(int is_min)
	{
		return is_min ? INT32_MAX : INT32_MIN;
	}
};
template <> struct AccTraits<int16_t> {
	static __device__ __forceinline__ int16_t ext_init(int is_min)
	{
		return is_min ? INT16_MAX : INT16_MIN;
	}
};
template <> struct AccTraits<uint32_t> {
	static __device__ __forceinline__ uint32_t ext_init(int)
	{
		return 0;
	}
};
template <> struct AccTraits<double> {
	static __device__ __forceinline__ double ext_init(int is_min)
	{
		return is_min ? svt_posinf() : svt_neginf();
	}
};

/* Values of 4 consecutive stage slots.  NA / NaN entries are counted in the
 * global state (rare) and replaced by the neutral element of the reduction
 * (0 for sums, +-extreme for min / max); r* report which entries are regular. */
template <int RC, typename T, typename ACC>
__device__ __forceinline__ void load_group4(const T *p, int is_min,
		double *state, int64_t nrow, const int4 &o,
		ACC &v0, ACC &v1, ACC &v2, ACC &v3,
		bool &r0, bool &r1, bool &r2, bool &r3);

template <int RC>
__device__ __forceinline__ void note_special(double *state, int64_t nrow,
					     int off, int cls)
{
	atomicAdd(&state[(cls == 1 ? SVT_ROW_SLOT_NA : SVT_ROW_SLOT_NAN) *
			 nrow + off], 1.0);
}

template <int RC, typename ACC>
__device__ __forceinline__ ACC neutral_of(int is_min)
{
	if (RC == RC_MINMAX)
		return AccTraits<ACC>::ext_init(is_min);
	return (ACC) 0;
}

template <int RC, typename T, typename ACC>
__device__ __forceinline__ void load_group4_int(const int32_t *p, int is_min,
		double *state, int64_t nrow, const int4 &o,
		ACC &v0, ACC &v1, ACC &v2, ACC &v3,
		bool &r0, bool &r1, bool &r2, bool &r3)
{
	const int4 x = *(const int4 *) p;
	v0 = (ACC) x.x; v1 = (ACC) x.y; v2 = (ACC) x.z; v3 = (ACC) x.w;
	int m = x.x < x.y ? x.x : x.y;
	const int m2 = x.z < x.w ? x.z : x.w;
	m = m < m2 ? m : m2;
	if (m == SVT_NA_INT) {   /* rare */
		const ACC neutral = neutral_of<RC, ACC>(is_min);
		if (x.x == SVT_NA_INT) { r0 = false; v0 = neutral; note_special<RC>(state, nrow, o.x, 1); }
		if (x.y == SVT_NA_INT) { r1 = false; v1 = neutral; note_special<RC>(state, nrow, o.y, 1); }
		if (x.z == SVT_NA_INT) { r2 = false; v2 = neutral; note_special<RC>(state, nrow, o.z, 1); }
		if (x.w == SVT_NA_INT) { r3 = false; v3 = neutral; note_special<RC>(state, nrow, o.w, 1); }
	}
}

template <int RC, typename ACC>
__device__ __forceinline__ void load_group4_dbl(const double *p, int is_min,
		double *state, int64_t nrow, const int4 &o,
		ACC &v0, ACC &v1, ACC &v2, ACC &v3,
		bool &r0, bool &r1, bool &r2, bool &r3)
{
	const double2 xa = *(const double2 *) p;
	const double2 xb = *(const double2 *) (p + 2);
	v0 = (ACC) xa.x; v1 = (ACC) xa.y; v2 = (ACC) xb.x; v3 = (ACC) xb.y;
	/* x + x + ... is NaN iff some entry is NaN (or Inf - Inf: checked) */
	const double t = (xa.x + xa.y) + (xb.x + xb.y);
	if (svt_isnan(t)) {   /* rare */
		const ACC neutral = neutral_of<RC, ACC>(is_min);
		double dv;
		int c;
		if ((c = classify(xa.x, dv)) != 0) { r0 = false; v0 = neutral; note_special<RC>(state, nrow, o.x, c); }
		if ((c = classify(xa.y, dv)) != 0) { r1 = false; v1 = neutral; note_special<RC>(state, nrow, o.y, c); }
		if ((c = classify(xb.x, dv)) != 0) { r2 = false; v2 = neutral; note_special<RC>(state, nrow, o.z, c); }
		if ((c = classify(xb.y, dv)) != 0) { r3 = false; v3 = neutral; note_special<RC>(state, nrow, o.w, c); }
	}
}

template <int RC, typename T, typename ACC> struct GroupLoader;
template <int RC, typename ACC> struct GroupLoader<RC, int32_t, ACC> {
	static __device__ __forceinline__ void load(const int32_t *p,
		int is_min, double *state, int64_t nrow, const int4 &o,
		ACC &v0, ACC &v1, ACC &v2, ACC &v3,
		bool &r0, bool &r1, bool &r2, bool &r3)
	{
		load_group4_int<RC, int32_t, ACC>(p, is_min, state, nrow, o,
				v0, v1, v2, v3, r0, r1, r2, r3);
	}
};
template <int RC, typename ACC> struct GroupLoader<RC, double, ACC> {
	static __device__ __forceinline__ void load(const double *p,
		int is_min, double *state, int64_t nrow, const int4 &o,
		ACC &v0, ACC &v1, ACC &v2, ACC &v3,
		bool &r0, bool &r1, bool &r2, bool &r3)
	{
		load_group4_dbl<RC, ACC>(p, is_min, state, nrow, o,
				v0, v1, v2, v3, r0, r1, r2, r3);
	}
};

template <int RC, typename T, typename ACC>
__device__ __forceinline__ void load_group4(const T *p, int is_min,
		double *state, int64_t nrow, const int4 &o,
		ACC &v0, ACC &v1, ACC &v2, ACC &v3,
		bool &r0, bool &r1, bool &r2, bool &r3)
{
	GroupLoader<RC, T, ACC>::load(p, is_min, state, nrow, o, v0, v1, v2,
				      v3, r0, r1, r2, r3);
}

/* One CTA = one chunk of leaves x one tile of rows; tile accumulators of
 * type ACC in shared memory.  ACC = int32 for integer / lacunar input (exact:
 * the host bounds the leaves summed between two flushes so no accumulator can
 * overflow), double otherwise.
 * smem: acc[NACC][tile_rows] | ROW_NS x (offs stage | vals stage) |
 * RowItem[ROW_NS] | full[ROW_NS], empty[ROW_NS] */
template <int RC, typename T, bool LACUNAR, typename ACC>
__global__ void __launch_bounds__(ROW_THREADS)
row_tiles(RowTileParams P)
{
	constexpr int NACC = RC == RC_SUM ? 1 : 2;
	constexpr int VSZ = (int) sizeof(T);   /* T is int32_t when LACUNAR */
	extern __shared__ __align__(128) unsigned char smem[];
	ACC *acc = (ACC *) smem;
	const int offs_stage_bytes = P.stage_elems * 4 + 32;
	const int vals_stage_bytes = LACUNAR ? 0 : P.stage_elems * VSZ + 32;
	const int stage_bytes = offs_stage_bytes + vals_stage_bytes;
	const size_t acc_bytes = ((size_t) NACC * P.tile_rows * sizeof(ACC) +
				  127) & ~(size_t) 127;
	unsigned char *ring = smem + acc_bytes;
	RowItem *items = (RowItem *) (ring + (size_t) ROW_NS * stage_bytes);
	uint64_t *bars = (uint64_t *) (items + ROW_NS);
	const uint32_t full0 = svt_smem_u32(&bars[0]);
	const uint32_t empty0 = svt_smem_u32(&bars[ROW_NS]);

	const int chunk = blockIdx.x / P.ntiles;
	const int tile = blockIdx.x - chunk * P.ntiles;
	const int row0 = tile * P.tile_rows;
	int rows_here = (int) (P.nrow - row0 < P.tile_rows ? P.nrow - row0
							    : P.tile_rows);
	if (rows_here < 0) rows_here = 0;

	if (threadIdx.x == 0) {
		for (int i = 0; i < ROW_NS; i++) {
			svt_mbar_init(full0 + 8 * i, 1);
			svt_mbar_init(empty0 + 8 * i, ROW_CWARPS);
		}
		svt_mbar_init_fence();
	}
	__syncthreads();

	if (threadIdx.x >= ROW_CONSUMERS) {
		/* ---- producer warp ---- */
		const int lane = threadIdx.x & 31;
		/* leaves [l0, l1) of this chunk: boundaries are the first
		   leaves starting at or after c * nnz / nchunks */
		int64_t bounds[2];
		for (int k = 0; k < 2; k++) {
			const int c = chunk + k;
			if (c >= P.nchunks) { bounds[k] = P.nleaf; continue; }
			const int64_t target = (int64_t) ((double) P.nnz *
					((double) c / (double) P.nchunks));
			int64_t lo = 0, hi = P.nleaf;
			while (lo < hi) {
				int64_t mid = lo + ((hi - lo) >> 1);
				if (P.leaf_ptr[mid] < target) lo = mid + 1;
				else                          hi = mid;
			}
			bounds[k] = c == 0 ? 0 : lo;
		}
		const int64_t l0 = bounds[0], l1 = bounds[1];
		const uint64_t policy = svt_policy_evict_first();
		uint32_t st = 0, phase = 0;
		int64_t since_flush = 0;
		/* runs of the next 32 leaves, fetched one batch ahead */
		int64_t nx_lo = 0, nx_hi = 0;
		{
			const int64_t leaf = l0 + lane;
			if (leaf < l1) {
				const int64_t start = P.leaf_ptr[leaf];
				const int64_t nz = P.leaf_ptr[leaf + 1] - start;
				nx_lo = start + (tile == 0 ? 0
					: P.split[(int64_t) (tile - 1) *
						  P.nleaf + leaf]);
				nx_hi = start + (tile == P.ntiles - 1 ? nz
					: P.split[(int64_t) tile * P.nleaf +
						  leaf]);
			}
		}
		for (int64_t base = l0; base < l1; base += 32) {
			const int64_t my_lo = nx_lo, my_hi = nx_hi;
			{
				const int64_t leaf = base + 32 + lane;
				nx_lo = nx_hi = 0;
				if (leaf < l1) {
					const int64_t start = P.leaf_ptr[leaf];
					const int64_t nz = P.leaf_ptr[leaf + 1] -
							   start;
					nx_lo = start + (tile == 0 ? 0
						: P.split[(int64_t) (tile - 1) *
							  P.nleaf + leaf]);
					nx_hi = start + (tile == P.ntiles - 1
						? nz
						: P.split[(int64_t) tile *
							  P.nleaf + leaf]);
				}
			}
			const int n = (int) (l1 - base < 32 ? l1 - base : 32);
			for (int i = 0; i < n; i++) {
				const int64_t lo = __shfl_sync(SVT_FULL_MASK,
							       my_lo, i);
				const int64_t hi = __shfl_sync(SVT_FULL_MASK,
							       my_hi, i);
				if (lane != 0 || lo >= hi)
					continue;
				since_flush++;
				for (int64_t c0 = lo; c0 < hi;
				     c0 += P.stage_elems) {
					int64_t c1 = c0 + P.stage_elems;
					if (c1 > hi) c1 = hi;
					svt_mbar_wait(empty0 + 8 * st, phase ^ 1);
					unsigned char *sb = ring +
						(size_t) st * stage_bytes;
					const int64_t oa0 = (c0 * 4) &
							    ~(int64_t) 15;
					const int64_t oa1 = (c1 * 4 + 15) &
							    ~(int64_t) 15;
					uint32_t bytes = (uint32_t) (oa1 - oa0);
					int64_t va0 = 0, va1 = 0;
					if (!LACUNAR) {
						va0 = (c0 * VSZ) & ~(int64_t) 15;
						va1 = (c1 * VSZ + 15) &
						      ~(int64_t) 15;
						bytes += (uint32_t) (va1 - va0);
					}
					RowItem ri;
					ri.n = (int32_t) (c1 - c0);
					ri.odelta = (int32_t) (c0 - oa0 / 4);
					ri.vdelta = LACUNAR ? 0
						: (int32_t) (c0 - va0 / VSZ);
					ri.flags = 0;
					if (c1 == hi) {
						ri.flags = RI_LEAF_END;
						if (since_flush >=
						    P.flush_leaves) {
							ri.flags |= RI_FLUSH;
							since_flush = 0;
						}
					}
					items[st] = ri;
					svt_mbar_arrive_expect_tx(
						full0 + 8 * st, bytes);
					svt_bulk_g2s_hint(svt_smem_u32(sb),
						(const char *) P.offs + oa0,
						(uint32_t) (oa1 - oa0),
						full0 + 8 * st, policy);
					if (!LACUNAR)
						svt_bulk_g2s_hint(
						    svt_smem_u32(sb +
							offs_stage_bytes),
						    (const char *) P.vals + va0,
						    (uint32_t) (va1 - va0),
						    full0 + 8 * st, policy);
					if (++st == ROW_NS) { st = 0; phase ^= 1; }
				}
			}
			__syncwarp();
		}
		if (lane == 0) {
			svt_mbar_wait(empty0 + 8 * st, phase ^ 1);
			RowItem ri;
			ri.n = ri.odelta = ri.vdelta = 0;
			ri.flags = RI_STOP;
			items[st] = ri;
			svt_mbar_arrive(full0 + 8 * st);
		}
		return;
	}

	/* ---- consumer warps ---- */
	const int ctid = threadIdx.x;
	const int lane = threadIdx.x & 31;
	ACC *acc0 = acc;                    /* sum | coverage */
	ACC *acc1 = acc + P.tile_rows;      /* sum2 | extreme */
	const ACC ext_init = AccTraits<ACC>::ext_init(P.is_min);
	for (int r = ctid; r < P.tile_rows; r += ROW_CONSUMERS) {
		acc0[r] = 0;
		if (NACC == 2)
			acc1[r] = RC == RC_MINMAX ? ext_init : (ACC) 0;
	}
	consumer_barrier();

	double *part = P.part + (size_t) chunk * NACC * P.nrow;
	bool first_flush = true;
	uint32_t st = 0, phase = 0;
	/* accumulators addressed by absolute row offset */
	ACC *const A0 = acc0 - row0;
	ACC *const A1 = acc1 - row0;
	for (;;) {
		svt_mbar_wait(full0 + 8 * st, phase);
		const RowItem ri = items[st];
		if (ri.flags & RI_STOP)
			break;
		const unsigned char *sb = ring + (size_t) st * stage_bytes;
		const int32_t *so = (const int32_t *) sb;     /* 16-B aligned */
		const T *sv = (const T *) (sb + offs_stage_bytes) +
			      (ri.vdelta - ri.odelta);   /* sv[s] pairs so[s] */
		/* stage slots [s_lo, s_hi) hold the run; whole groups of 4
		   slots [v_lo, v_hi) take the vector path, the <= 6 slots at
		   the two ragged ends the scalar path */
		const int s_lo = ri.odelta, s_hi = ri.odelta + ri.n;
		const int v_lo = (s_lo + 3) & ~3;
		int v_hi = s_hi & ~3;
		if (v_hi < v_lo) v_hi = v_lo;
		for (int g = (v_lo >> 2) + ctid; g < (v_hi >> 2);
		     g += ROW_CONSUMERS) {
			const int4 o = ((const int4 *) so)[g];
			ACC v0 = (ACC) 1, v1 = (ACC) 1, v2 = (ACC) 1,
			    v3 = (ACC) 1;
			bool r0 = true, r1 = true, r2 = true, r3 = true;
			if (!LACUNAR)
				load_group4<RC, T, ACC>(sv + 4 * g, P.is_min,
					P.state, P.nrow, o, v0, v1, v2, v3,
					r0, r1, r2, r3);
			/* rows are distinct inside a run: four independent
			   read-modify-writes */
			const ACC a0 = A0[o.x], a1 = A0[o.y], a2 = A0[o.z],
				  a3 = A0[o.w];
			if (RC == RC_SUM) {
				A0[o.x] = a0 + v0; A0[o.y] = a1 + v1;
				A0[o.z] = a2 + v2; A0[o.w] = a3 + v3;
			} else if (RC == RC_X2) {
				const ACC b0 = A1[o.x], b1 = A1[o.y],
					  b2 = A1[o.z], b3 = A1[o.w];
				A0[o.x] = a0 + v0; A0[o.y] = a1 + v1;
				A0[o.z] = a2 + v2; A0[o.w] = a3 + v3;
				A1[o.x] = b0 + v0 * v0; A1[o.y] = b1 + v1 * v1;
				A1[o.z] = b2 + v2 * v2; A1[o.w] = b3 + v3 * v3;
			} else {
				const ACC b0 = A1[o.x], b1 = A1[o.y],
					  b2 = A1[o.z], b3 = A1[o.w];
				A0[o.x] = a0 + (ACC) 1; A0[o.y] = a1 + (ACC) 1;
				A0[o.z] = a2 + (ACC) 1; A0[o.w] = a3 + (ACC) 1;
				/* NA/NaN were replaced by the neutral element */
				if (P.is_min) {
					A1[o.x] = v0 < b0 ? v0 : b0;
					A1[o.y] = v1 < b1 ? v1 : b1;
					A1[o.z] = v2 < b2 ? v2 : b2;
					A1[o.w] = v3 < b3 ? v3 : b3;
				} else {
					A1[o.x] = v0 > b0 ? v0 : b0;
					A1[o.y] = v1 > b1 ? v1 : b1;
					A1[o.z] = v2 > b2 ? v2 : b2;
					A1[o.w] = v3 > b3 ? v3 : b3;
				}
			}
		}
		if (ctid < 8) {
			/* ragged ends: head [s_lo, min(v_lo, s_hi)),
			   tail [v_hi, s_hi) */
			const int head_end = v_lo < s_hi ? v_lo : s_hi;
			const int head_n = head_end - s_lo;
			const int tail_lo = v_hi > head_end ? v_hi : head_end;
			const int slot = ctid < head_n ? s_lo + ctid
						: tail_lo + (ctid - head_n);
			if (slot < s_hi) {
				const int off = so[slot];
				ACC v = (ACC) 1;
				bool reg = true;
				if (!LACUNAR) {
					double dv;
					const T x = sv[slot];
					const int cls = classify(x, dv);
					v = (ACC) x;
					if (cls != 0) {
						reg = false;
						atomicAdd(&P.state[(cls == 1
							? SVT_ROW_SLOT_NA
							: SVT_ROW_SLOT_NAN) *
							P.nrow + off], 1.0);
					}
				}
				if (RC == RC_MINMAX) {
					A0[off] += (ACC) 1;
					if (reg && (P.is_min ? v < A1[off]
							     : v > A1[off]))
						A1[off] = v;
				} else if (reg) {
					A0[off] += v;
					if (RC == RC_X2)
						A1[off] += v * v;
				}
			}
		}
		/* this warp is done with the stage */
		__syncwarp();
		if (lane == 0)
			svt_mbar_arrive(empty0 + 8 * st);
		if (++st == ROW_NS) { st = 0; phase ^= 1; }
		if (ri.flags & RI_LEAF_END) {
			/* the next run may hit the same rows */
			consumer_barrier();
			if (ri.flags & RI_FLUSH) {
				for (int r = ctid; r < rows_here;
				     r += ROW_CONSUMERS) {
					const double s0 = (double) acc0[r];
					part[row0 + r] = first_flush ? s0
						: part[row0 + r] + s0;
					acc0[r] = 0;
					if (RC == RC_X2) {
						const double s1 =
							(double) acc1[r];
						part[P.nrow + row0 + r] =
						    first_flush ? s1
						    : part[P.nrow + row0 + r] + s1;
						acc1[r] = 0;
					}
				}
				first_flush = false;
				consumer_barrier();
			}
		}
	}

	/* flush this CTA's partial rows (every thread has passed the barrier
	   that follows the last run) */
	for (int r = ctid; r < rows_here; r += ROW_CONSUMERS) {
		const double s0 = (double) acc0[r];
		part[row0 + r] = first_flush ? s0 : part[row0 + r] + s0;
		if (RC == RC_X2) {
			const double s1 = (double) acc1[r];
			part[P.nrow + row0 + r] = first_flush ? s1
				: part[P.nrow + row0 + r] + s1;
		}
		if (RC == RC_MINMAX)
			part[P.nrow + row0 + r] = (double) acc1[r];
	}
}

/* ------------------------------------------------------------------------
 * row_strips: every warp owns a strip of rows.
 *
 * The grid is nchunks x ntiles CTAs of W warps.  A CTA keeps the accumulators
 * of its row tile in shared memory; warp w owns the rows [w, w+1) * strip_rows
 * of the tile and nobody else ever touches them.  Offsets ascend inside a
 * leaf, so the nonzeros of a leaf that fall into a strip are one contiguous
 * sub-run (found once per matrix by row_split, one int32 per leaf and strip
 * boundary), and their rows are distinct: the warp applies a sub-run with
 * plain shared-memory read-modify-writes -- no atomics, no block barrier, no
 * coupling between warps.  Each warp streams its sub-runs straight from
 * global memory into registers, ST_D leaves ahead of the one it is applying
 * (ST_D x ST_U x 8 bytes in flight per lane), so the memory system always has
 * plenty of requests from every warp.
 */
/* ST_D = leaves prefetched ahead per warp, ST_U = 32-wide slots held per leaf
 * (sub-runs up to 32 * ST_U nonzeros come out of the ring; longer ones finish
 * on a scalar path); both are template parameters picked from the expected
 * sub-run length.
 * PACKED (RC_X2, uint32 accumulators, non-negative small integers): one
 * accumulator per row holds sum(x) in its low and sum(x^2) in its high 16
 * bits, so the two moments of rowVars cost one read-modify-write. */

struct RowStripParams {
	const int32_t *offs;
	const void *vals;          /* NULL: lacunar */
	const int64_t *leaf_ptr;
	const int32_t *split;      /* [nstrips - 1][nleaf]; NULL if 1 strip */
	int64_t nleaf, nnz, nrow;
	int ntiles, nchunks, nstrips, strip_rows;
	int is_min;
	int flush_leaves;
	double *part;              /* [nchunks][nacc][nrow] */
	double *state;
};

template <typename T>
__device__ __forceinline__ T ldg_stream(const T *p);
template <>
__device__ __forceinline__ int32_t ldg_stream<int32_t>(const int32_t *p)
{
	int32_t r;
	asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];"
		     : "=r"(r) : "l"(p));
	return r;
}
template <>
__device__ __forceinline__ double ldg_stream<double>(const double *p)
{
	double r;
	asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];"
		     : "=d"(r) : "l"(p));
	return r;
}

__device__ __forceinline__ int4 ldg_stream_v4(const int4 *p)
{
	int4 r;
	asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];"
		     : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
	return r;
}

__device__ __forceinline__ uint2 ldg_stream_v2(const uint2 *p)
{
	uint2 r;
	asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];"
		     : "=r"(r.x), "=r"(r.y) : "l"(p));
	return r;
}

/* PACKED row min / max (non-negative integers < 65535): coverage count in
 * the high, running extreme in the low 16 bits of one accumulator.  A minimum
 * is kept as the maximum of the complemented values (x ^ 0xFFFF), so both
 * directions are one unsigned max: with the count already bumped, the
 * candidate shares the accumulator's high half and the comparison is decided
 * by the low halves. */
__device__ __forceinline__ uint32_t packed_max(uint32_t a, uint32_t vc)
{
	const uint32_t t = a + 0x10000u;
	const uint32_t c = (t & 0xFFFF0000u) | vc;
	return t > c ? t : c;
}

/* Accumulators are addressed by 32-bit shared-memory address (one LEA per
 * element instead of a generic-pointer computation) and updated in a full
 * register whatever their stored width (no sub-word moves). */
template <typename ACC> struct SmemAcc;
template <> struct SmemAcc<int16_t> {
	typedef int32_t reg;
	static __device__ __forceinline__ reg ld(uint32_t a)
	{
		int32_t r;
		asm volatile("ld.shared.s16 %0, [%1];" : "=r"(r) : "r"(a));
		return r;
	}
	static __device__ __forceinline__ void st(uint32_t a, reg v)
	{
		asm volatile("st.shared.u16 [%0], %1;" :: "r"(a), "r"(v)
			     : "memory");
	}
};
template <> struct SmemAcc<int32_t> {
	typedef int32_t reg;
	static __device__ __forceinline__ reg ld(uint32_t a)
	{
		int32_t r;
		asm volatile("ld.shared.s32 %0, [%1];" : "=r"(r) : "r"(a));
		return r;
	}
	static __device__ __forceinline__ void st(uint32_t a, reg v)
	{
		asm volatile("st.shared.s32 [%0], %1;" :: "r"(a), "r"(v)
			     : "memory");
	}
};
template <> struct SmemAcc<uint32_t> {
	typedef uint32_t reg;
	static __device__ __forceinline__ reg ld(uint32_t a)
	{
		uint32_t r;
		asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(a));
		return r;
	}
	static __device__ __forceinline__ void st(uint32_t a, reg v)
	{
		asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v)
			     : "memory");
	}
};
template <> struct SmemAcc<double> {
	typedef double reg;
	static __device__ __forceinline__ reg ld(uint32_t a)
	{
		double r;
		asm volatile("ld.shared.f64 %0, [%1];" : "=d"(r) : "r"(a));
		return r;
	}
	static __device__ __forceinline__ void st(uint32_t a, reg v)
	{
		asm volatile("st.shared.f64 [%0], %1;" :: "r"(a), "d"(v)
			     : "memory");
	}
};

/* true if any of the ring values of a leaf may be NA / NaN (slots the
 * sub-run does not fill hold older values: a false positive only takes the
 * exact path, which looks at the filled slots alone) */
template <int U>
__device__ __forceinline__ bool any_special(const int32_t (&x)[U])
{
	int32_t m = x[0];
#pragma unroll
	for (int k = 1; k < U; k++)
		m = x[k] < m ? x[k] : m;
	return m == SVT_NA_INT;
}
template <int U>
__device__ __forceinline__ bool any_special(const double (&x)[U])
{
	bool sp = false;
#pragma unroll
	for (int k = 0; k < U; k++)
		sp |= svt_isnan(x[k]);
	return sp;
}

template <int RC, typename T, bool LACUNAR, typename ACC, bool PACKED,
	  int ST_D, int ST_U>
__global__ void __launch_bounds__(512, 1)
row_strips(RowStripParams P)
{
	constexpr int PT_NACC = RC == RC_SUM ? 1 : 2;   /* partial arrays */
	constexpr int NACC = PACKED ? 1 : PT_NACC;       /* smem arrays */
	/* two double accumulators per row (row moments of doubles): one
	   16-byte cell {sum, sum of squares} per row -- one 16-byte load and
	   one 16-byte store per nonzero instead of two 8-byte ones each; on
	   random rows that is 10 instead of 12.3 shared-memory wavefronts per
	   pair of accesses, and the kernel is bound by them */
	constexpr bool IL = NACC == 2 && RC == RC_X2 && sizeof(ACC) == 8;
	constexpr int RS = IL ? 2 : 1;                   /* cells per row */
	extern __shared__ __align__(128) unsigned char smem[];
	int lane;
	/* read the lane id once (volatile: not re-materialised in the loop) */
	asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
	const int warp = threadIdx.x >> 5;
	const int W = blockDim.x >> 5;
	const int chunk = blockIdx.x / P.ntiles;
	const int tile = blockIdx.x - chunk * P.ntiles;
	const int gs = tile * W + warp;               /* global strip index */
	const int row0 = gs * P.strip_rows;
	int rows_here = (int) (P.nrow - row0 < P.strip_rows ? P.nrow - row0
							     : P.strip_rows);
	if (rows_here < 0) rows_here = 0;
	const T *vals = (const T *) P.vals;

	/* this warp's accumulators; A0/A1 are addressed by absolute row */
	ACC *A0, *A1;
	uint32_t a0s, a10;
	/* packed min / max: a minimum runs on complemented values */
	const uint32_t mm_mask = (PACKED && RC == RC_MINMAX && P.is_min)
				 ? 0xFFFFu : 0u;
	{
	ACC *acc0 = (ACC *) smem + (size_t) warp * NACC * P.strip_rows;
	ACC *acc1 = IL ? acc0 + 1 : acc0 + P.strip_rows;
	const ACC ext_init = AccTraits<ACC>::ext_init(P.is_min);
	/* packed min / max: the low half starts at the neutral extreme */
	const ACC acc0_init = (ACC) 0;
	for (int r = lane; r < P.strip_rows; r += 32) {
		acc0[r * RS] = acc0_init;
		if (NACC == 2)
			acc1[r * RS] = RC == RC_MINMAX ? ext_init : (ACC) 0;
	}
	__syncwarp();
	A0 = acc0 - (size_t) row0 * RS;
	A1 = acc1 - (size_t) row0 * RS;
	/* the same bases as 32-bit shared-memory addresses (a10: from the
	   first to the second accumulator of a row) */
	a0s = (uint32_t) __cvta_generic_to_shared(acc0) -
	      (uint32_t) row0 * (uint32_t) (sizeof(ACC) * RS);
	a10 = IL ? (uint32_t) sizeof(ACC)
		 : (uint32_t) P.strip_rows * (uint32_t) sizeof(ACC);
	}

	/* leaves [l0, l1) of this chunk (balanced by nonzeros) */
	int64_t l0, l1;
	{
		int64_t bounds[2];
		for (int k = 0; k < 2; k++) {
			const int c = chunk + k;
			if (c >= P.nchunks) { bounds[k] = P.nleaf; continue; }
			const int64_t target = (int64_t) ((double) P.nnz *
					((double) c / (double) P.nchunks));
			int64_t lo = 0, hi = P.nleaf;
			while (lo < hi) {
				int64_t mid = lo + ((hi - lo) >> 1);
				if (P.leaf_ptr[mid] < target) lo = mid + 1;
				else                          hi = mid;
			}
			bounds[k] = c == 0 ? 0 : lo;
		}
		l0 = bounds[0];
		l1 = bounds[1];
	}

	/* element positions are kept relative to the chunk's first nonzero
	   (a chunk holds far fewer than 2^31): 32-bit bounds in the ring */
	const int64_t cbase = l0 < P.nleaf ? P.leaf_ptr[l0] : 0;
	const int32_t *const offs_c = P.offs + cbase + lane;
	const T *const vals_c = vals + cbase + lane;

	/* sub-run of leaf `leaf` in this strip: first element and length */
	auto subrun = [&](int64_t leaf, int32_t &lo, int &n) {
		lo = 0; n = 0;
		if (leaf < l1) {
			const int64_t start = P.leaf_ptr[leaf];
			const int nz = (int) (P.leaf_ptr[leaf + 1] - start);
			const int a = gs == 0 ? 0
				: P.split[(int64_t) (gs - 1) * P.nleaf + leaf];
			const int b = gs == P.nstrips - 1 ? nz
				: P.split[(int64_t) gs * P.nleaf + leaf];
			lo = (int32_t) (start - cbase) + a;
			n = b - a;
		}
	};

	bool first_flush = true;
	int since_flush = 0;
	auto flush = [&](bool final) {
		__syncwarp();
		double *const part = P.part + (size_t) chunk * PT_NACC * P.nrow;
		ACC *const acc0 = A0 + (size_t) row0 * RS;
		ACC *const acc1 = A1 + (size_t) row0 * RS;
		for (int r0 = lane; r0 < rows_here; r0 += 32) {
			const int r = r0 * RS;        /* cell of the row */
			double s0 = (double) acc0[r];
			if (PACKED && RC == RC_X2)
				s0 = (double) ((uint32_t) acc0[r] & 0xFFFFu);
			if (PACKED && RC == RC_MINMAX)
				s0 = (double) ((uint32_t) acc0[r] >> 16);
			part[row0 + r0] = first_flush ? s0 : part[row0 + r0] + s0;
			if (PACKED && RC == RC_MINMAX) {
				/* keep the running extreme, drop the count */
				if (final)
					part[P.nrow + row0 + r0] = (double)
						(((uint32_t) acc0[r] & 0xFFFFu)
						 ^ mm_mask);
				acc0[r] = (ACC) ((uint32_t) acc0[r] & 0xFFFFu);
				continue;
			}
			if (RC == RC_X2) {
				const double s1 = PACKED
					? (double) ((uint32_t) acc0[r] >> 16)
					: (double) acc1[NACC == 2 ? r : 0];
				part[P.nrow + row0 + r0] = first_flush ? s1
					: part[P.nrow + row0 + r0] + s1;
				if (NACC == 2)
					acc1[r] = 0;
			}
			acc0[r] = 0;
			if (RC == RC_MINMAX && final)
				part[P.nrow + row0 + r0] = (double) acc1[r];
		}
		first_flush = false;
		since_flush = 0;
		__syncwarp();
	};

	/* register ring: ST_D leaves x ST_U slots per lane */
	int32_t boff[ST_D][ST_U];
	T bval[ST_D][ST_U];
#pragma unroll
	for (int d = 0; d < ST_D; d++) {
#pragma unroll
		for (int k = 0; k < ST_U; k++) {
			boff[d][k] = 0;
			bval[d][k] = (T) 0;
		}
	}

	int bn[ST_D];

	/* bounds of 32 leaves per batch, one leaf per lane, fetched one batch
	   ahead of their use */
	int32_t cur_lo, nxt_lo;
	int cur_n, nxt_n;
	subrun(l0 + lane, cur_lo, cur_n);
	subrun(l0 + 32 + lane, nxt_lo, nxt_n);

	auto fetch = [&](int d, int32_t lo, int n) {
		bn[d] = n;
		/* lane's elements: lo + lane + 32 k, valid while 32 k < n - lane */
		const int32_t *po;
		const T *pv;
		asm volatile("mad.wide.u32 %0, %1, 4, %2;" : "=l"(po)
			     : "r"(lo), "l"(offs_c));
		asm volatile("mad.wide.u32 %0, %1, %2, %3;" : "=l"(pv)
			     : "r"(lo), "n"((int) sizeof(T)), "l"(vals_c));
		const int rem = n - lane;
#pragma unroll
		for (int k = 0; k < ST_U; k++) {
			if (k * 32 < rem) {
				boff[d][k] = ldg_stream<int32_t>(po + k * 32);
				if (!LACUNAR)
					bval[d][k] = ldg_stream<T>(pv + k * 32);
			}
		}
	};

	/* one element into the accumulators (scalar path: long sub-runs) */
	auto apply1 = [&](int off, T x) {
		ACC v = (ACC) 1;
		bool reg = true;
		if (!LACUNAR) {
			double dv;
			const int cls = classify(x, dv);
			v = (ACC) x;
			if (cls != 0) {
				reg = false;
				atomicAdd(&P.state[(cls == 1 ? SVT_ROW_SLOT_NA
					: SVT_ROW_SLOT_NAN) * P.nrow + off], 1.0);
			}
		}
		const size_t c = (size_t) off * RS;     /* the row's cell */
		if (RC == RC_MINMAX && PACKED) {
			A0[c] = (ACC) packed_max((uint32_t) A0[c],
					reg ? ((uint32_t) v ^ mm_mask) : 0u);
		} else if (RC == RC_MINMAX) {
			A0[c] += (ACC) 1;
			if (reg && (P.is_min ? v < A1[c] : v > A1[c]))
				A1[c] = v;
		} else if (reg) {
			if (PACKED)
				v = (ACC) ((uint32_t) v +
					   (((uint32_t) v * (uint32_t) v) << 16));
			A0[c] += v;
			if (RC == RC_X2 && !PACKED)
				A1[c] += v * v;
		}
	};

	typedef typename SmemAcc<ACC>::reg REG;

	auto apply = [&](int d, int32_t cur_lo_i) {
		const int n = bn[d];
		if (n == 0)
			return;
		since_flush++;
		const int rem = n - lane;
		if (!LACUNAR && any_special<ST_U>(bval[d])) {
			/* NA / NaN among this lane's elements (rare): the
			   exact element-wise path */
#pragma unroll
			for (int k = 0; k < ST_U; k++)
				if (k * 32 < rem)
					apply1(boff[d][k], bval[d][k]);
		} else {
			/* rows are distinct inside a sub-run: all loads, then
			   all stores */
			uint32_t sa[ST_U];
			REG a[ST_U], b[ST_U];
#pragma unroll
			for (int k = 0; k < ST_U; k++) {
				sa[k] = a0s + (uint32_t) boff[d][k] *
					      (uint32_t) (sizeof(ACC) * RS);
				if (k * 32 < rem) {
					if constexpr (IL) {
						asm volatile(
						    "ld.shared.v2.f64 {%0, %1}, [%2];"
						    : "=d"(a[k]), "=d"(b[k])
						    : "r"(sa[k]));
					} else {
						a[k] = SmemAcc<ACC>::ld(sa[k]);
						if (NACC == 2)
							b[k] = SmemAcc<ACC>::ld(
								sa[k] + a10);
					}
				}
			}
#pragma unroll
			for (int k = 0; k < ST_U; k++) {
				const REG v = LACUNAR ? (REG) 1
						      : (REG) bval[d][k];
				if (k * 32 < rem) {
					if (RC == RC_MINMAX && PACKED) {
						SmemAcc<ACC>::st(sa[k],
							(REG) packed_max(
							(uint32_t) a[k],
							(uint32_t) v ^ mm_mask));
					} else if (RC == RC_MINMAX) {
						SmemAcc<ACC>::st(sa[k],
							a[k] + (REG) 1);
						SmemAcc<ACC>::st(sa[k] + a10,
							P.is_min
							? (v < b[k] ? v : b[k])
							: (v > b[k] ? v : b[k]));
					} else if (PACKED) {
						/* x + (x^2 << 16) = x (1 + (x << 16)) */
						SmemAcc<ACC>::st(sa[k], (REG)
						    ((uint32_t) a[k] +
						     (uint32_t) v *
						     (((uint32_t) v << 16) + 1u)));
					} else if constexpr (IL) {
						asm volatile(
						    "st.shared.v2.f64 [%0], {%1, %2};"
						    :: "r"(sa[k]), "d"(a[k] + v),
						       "d"(b[k] + v * v) : "memory");
					} else {
						SmemAcc<ACC>::st(sa[k],
								 a[k] + v);
						if (RC == RC_X2)
							SmemAcc<ACC>::st(
								sa[k] + a10,
								b[k] + v * v);
					}
				}
			}
		}
		/* the part of a long sub-run the ring does not hold */
		if (n > ST_U * 32) {
			/* rare: fetch the sub-run's start again instead of
			   keeping it in a register per ring slot */
			const int32_t lo = cur_lo_i;
			for (int e = ST_U * 32; e < n - lane; e += 32)
				apply1(offs_c[lo + e],
				       LACUNAR ? (T) 1 : vals_c[lo + e]);
		}
		__syncwarp();
		if (since_flush >= P.flush_leaves) {
			if constexpr (PACKED && RC == RC_X2) {
				/* flush_leaves is the number of leaves that
				   cannot add 2^15 to either half: as long as no
				   half has reached 2^15 nothing can overflow
				   before the next look, and the accumulators
				   stay on chip (sparse rows: practically
				   always) */
				bool risky = false;
				for (int r = lane; r < rows_here; r += 32)
					risky |= (SmemAcc<ACC>::ld(a0s +
						(uint32_t) (row0 + r) *
						(uint32_t) sizeof(ACC)) &
						0x80008000u) != 0;
				if (__any_sync(SVT_FULL_MASK, risky))
					flush(false);
				else
					since_flush = 0;
			} else {
				flush(false);
			}
		}
	};

	/* prologue: leaves l0 .. l0 + ST_D - 1 */
#pragma unroll
	for (int d = 0; d < ST_D; d++) {
		const int32_t lo = __shfl_sync(SVT_FULL_MASK, cur_lo, d);
		const int n = __shfl_sync(SVT_FULL_MASK, cur_n, d);
		fetch(d, lo, n);
	}
	for (int64_t base = l0; base < l1; base += 32) {
		/* leaves base + i, i = 0..31; prefetch reaches ST_D further */
		for (int i0 = 0; i0 < 32; i0 += ST_D) {
			if (base + i0 >= l1)
				break;
#pragma unroll
			for (int d = 0; d < ST_D; d++) {
				const int i = i0 + d;
				apply(d, bn[d] > ST_U * 32
					? __shfl_sync(SVT_FULL_MASK, cur_lo, i)
					: 0);
				/* refill the slot with leaf base + i + ST_D */
				const int j = i + ST_D;
				int32_t lo;
				int n;
				if (j < 32) {
					lo = __shfl_sync(SVT_FULL_MASK, cur_lo, j);
					n = __shfl_sync(SVT_FULL_MASK, cur_n, j);
				} else {
					lo = __shfl_sync(SVT_FULL_MASK, nxt_lo,
							 j - 32);
					n = __shfl_sync(SVT_FULL_MASK, nxt_n,
							j - 32);
				}
				fetch(d, lo, n);
			}
		}
		cur_lo = nxt_lo;
		cur_n = nxt_n;
		subrun(base + 64 + lane, nxt_lo, nxt_n);
	}
	flush(true);
}

/* max |x| over the non-NA values of an integer matrix (bounds the int32
 * accumulators of row_tiles) */
__global__ void __launch_bounds__(256)
absmax_int(const int32_t *__restrict__ vals, int64_t nnz,
	   unsigned long long *out /* [0] max |x|, [1] #negative */)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	long long m = 0, neg = 0;
	for (int64_t e = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     e < nnz; e += stride) {
		const long long x = vals[e];
		if (x != (long long) SVT_NA_INT) {
			const long long a = x < 0 ? -x : x;
			m = a > m ? a : m;
			neg += x < 0;
		}
	}
#pragma unroll
	for (int k = 16; k > 0; k >>= 1) {
		const long long o = __shfl_xor_sync(SVT_FULL_MASK, m, k);
		m = o > m ? o : m;
		neg += __shfl_xor_sync(SVT_FULL_MASK, neg, k);
	}
	if ((threadIdx.x & 31) == 0) {
		if (m > 0)
			atomicMax(out, (unsigned long long) m);
		if (neg > 0)
			atomicAdd(out + 1, (unsigned long long) neg);
	}
}

/* pass 2: fixed-order sum (or min/max) of the per-chunk partial vectors into
 * the state slots */
template <int RC>
__global__ void __launch_bounds__(256)
row_combine(const double *__restrict__ part, int nchunks, int64_t nrow,
	    int is_min, double *__restrict__ state)
{
	constexpr int NACC = RC == RC_SUM ? 1 : 2;
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     r < nrow; r += stride) {
		double a0 = 0.0;
		double a1 = RC == RC_MINMAX
			? (is_min ? svt_posinf() : svt_neginf()) : 0.0;
		for (int c = 0; c < nchunks; c++) {
			const double *p = part + (size_t) c * NACC * nrow;
			a0 += p[r];
			if (NACC == 2) {
				const double x = p[nrow + r];
				if (RC == RC_MINMAX)
					a1 = (is_min ? x < a1 : x > a1) ? x : a1;
				else
					a1 += x;
			}
		}
		if (RC == RC_SUM) {
			state[SVT_ROW_SLOT_SUM * nrow + r] = a0;
		} else if (RC == RC_X2) {
			state[SVT_ROW_SLOT_SUM * nrow + r] = a0;
			state[SVT_ROW_SLOT_SUM2 * nrow + r] = a1;
		} else {
			state[SVT_ROW_SLOT_CVG * nrow + r] = a0;
			state[SVT_ROW_SLOT_EXT * nrow + r] = a1;
		}
	}
}

/* state -> R's answer */
__global__ void __launch_bounds__(256)
row_finalize(int opcode, int is_double, int narm, int64_t nrow,
	     int64_t nstrata, const double *__restrict__ center,
	     const double *__restrict__ state, void *out, int32_t *warn)
{
	const int out_is_int = opcode == SVTGPU_OP_ANYNA ||
		((opcode == SVTGPU_OP_MIN || opcode == SVTGPU_OP_MAX) &&
		 !is_double);
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     r < nrow; r += stride) {
		SvtScalar s = svt_row_finalize(opcode, is_double, narm,
				nstrata, center != NULL,
				center != NULL ? center[r] : 0.0,
				state + r, nrow);
		if (out_is_int) ((int32_t *) out)[r] = s.i;
		else            ((double *) out)[r] = s.d;
		if (s.warn && warn != NULL)
			atomicOr((int *) warn, 1);
	}
}

__global__ void __launch_bounds__(256)
row_moments_finalize(int narm, int64_t nrow, int64_t nstrata,
		     const double *__restrict__ state, double *mean,
		     double *var)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     r < nrow; r += stride) {
		double mu, v;
		svt_row_moments(narm, nstrata, state + r, nrow, &mu, &v);
		if (mean != NULL) mean[r] = mu;
		if (var != NULL)  var[r] = v;
	}
}

/* Which NA / NaN entry of a row came last (SVT_ROW_SLOT_LAST_*, see
 * svt_semantics.h) matters only for rows that hold both kinds, so the hot
 * kernels just count.  row_last_plan gives rows with a single kind the
 * position "somewhere in this shard" (enough to order them against other
 * shards) and raises *mixed when a row of this shard holds both kinds;
 * row_last_exact then scans the values once for the exact leaf indices and
 * returns immediately otherwise. */
__global__ void __launch_bounds__(256)
row_last_plan(double *__restrict__ state, int64_t nrow, double shard_pos,
	      int *mixed)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     r < nrow; r += stride) {
		const bool na = state[SVT_ROW_SLOT_NA * nrow + r] > 0.0;
		const bool nan = state[SVT_ROW_SLOT_NAN * nrow + r] > 0.0;
		if (na && nan)
			*mixed = 1;
		else if (na)
			state[SVT_ROW_SLOT_LAST_NA * nrow + r] = shard_pos;
		else if (nan)
			state[SVT_ROW_SLOT_LAST_NAN * nrow + r] = shard_pos;
	}
}

__global__ void __launch_bounds__(256)
row_last_exact(const int32_t *__restrict__ offs,
	       const double *__restrict__ vals,
	       const int64_t *__restrict__ leaf_ptr, int64_t nleaf, int64_t nnz,
	       int64_t nrow, int64_t leaf_base, double *state, const int *mixed)
{
	if (*mixed == 0)
		return;
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t e = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     e < nnz; e += stride) {
		double v;
		const int cls = classify(vals[e], v);
		if (cls == 0)
			continue;
		/* leaf holding element e: last l with leaf_ptr[l] <= e */
		int64_t lo = 0, hi = nleaf;
		while (lo < hi) {
			const int64_t mid = lo + ((hi - lo) >> 1);
			if (leaf_ptr[mid + 1] <= e) lo = mid + 1;
			else                        hi = mid;
		}
		note_last(state, nrow, offs[e], cls - 1,
			  (double) (leaf_base + lo));
	}
}

inline unsigned grid_for(int64_t n, int per_block)
{
	int64_t b = (n + per_block - 1) / per_block;
	int64_t cap = (int64_t) svtgpu_sm_count() * 16;
	if (b > cap) b = cap;
	if (b < 1) b = 1;
	return (unsigned) b;
}

struct TileConfig {
	int ok;
	int ntiles, tile_rows, nchunks, stage_elems;
	int ctas_per_sm;
	size_t smem;
};

size_t tile_smem_bytes(int64_t tile_rows, int nacc, int acc_size, int se,
		       int vsz)
{
	size_t acc = ((size_t) nacc * tile_rows * acc_size + 127) & ~(size_t) 127;
	return acc + (size_t) ROW_NS * ((size_t) se * 4 + 32 +
			(vsz ? (size_t) se * vsz + 32 : 0)) +
	       ROW_NS * sizeof(RowItem) + 2 * ROW_NS * 8 + 128;
}

/* Smallest number of row tiles whose accumulators + staging ring let two CTAs
 * share an SM (their barrier / mbarrier bubbles then overlap); one CTA per SM
 * when even 64 tiles cannot do that. */
TileConfig choose_tiles(int64_t nrow, int64_t nleaf, int64_t nnz, int nacc,
			int acc_size, int vsz)
{
	TileConfig c;
	memset(&c, 0, sizeof(c));
	const int sms = svtgpu_sm_count();
	const double avg_leaf = nleaf > 0 ? (double) nnz / (double) nleaf : 0.0;
	const int force = atoi(svtgpu_env("SVTGPU_ROW_NTILES", "0"));
	const int force_se = atoi(svtgpu_env("SVTGPU_ROW_STAGE_ELEMS", "0"));
	int per_sm = atoi(svtgpu_env("SVTGPU_ROW_CTAS_PER_SM", "2"));
	if (per_sm < 1) per_sm = 1;
	if (per_sm > 4) per_sm = 4;
	for (; per_sm >= 1; per_sm--) {
		/* 227 KB per SM, 1 KB reserved per resident CTA */
		const size_t budget = (size_t) (227 * 1024) / per_sm - 1024 - 512;
		for (int nt = force > 0 ? force : 1; nt <= 64; nt++) {
			int64_t tr = (nrow + nt - 1) / nt;
			tr = (tr + 31) / 32 * 32;
			if (tr < 32) tr = 32;
			int se = (int) (avg_leaf / nt * 1.15) + 32;
			se = (se + 127) / 128 * 128;
			if (se < 256) se = 256;
			if (se > 2048) se = 2048;
			if (force_se > 0) se = (force_se + 3) / 4 * 4;
			size_t smem = tile_smem_bytes(tr, nacc, acc_size, se, vsz);
			/* a tight fit may still work with shorter stages */
			while (smem > budget && se > 512 && force_se == 0) {
				se -= 128;
				smem = tile_smem_bytes(tr, nacc, acc_size, se,
						       vsz);
			}
			if (smem <= budget) {
				c.ok = 1;
				c.ntiles = nt;
				c.tile_rows = (int) tr;
				c.stage_elems = se;
				c.smem = smem;
				c.ctas_per_sm = per_sm;
				c.nchunks = sms * per_sm / nt;
				if (c.nchunks < 1) c.nchunks = 1;
				if ((int64_t) c.nchunks > nleaf)
					c.nchunks = nleaf > 0 ? (int) nleaf : 1;
				return c;
			}
			if (force > 0)
				break;
		}
	}
	return c;
}

/* split points are cached per (ntiles, tile_rows): rowSums and rowVars use
 * different tilings of the same matrix */
int ensure_split(svtgpu_matrix *m, const TileConfig &c, cudaStream_t s,
		 const int32_t **split)
{
	*split = NULL;
	if (c.ntiles <= 1)
		return SVTGPU_OK;
	int slot = -1;
	for (int i = 0; i < SVTGPU_NSPLIT; i++) {
		if (m->d_split[i] != NULL &&
		    m->split_tile_rows[i] == c.tile_rows &&
		    m->split_ntiles[i] == c.ntiles) {
			*split = m->d_split[i];
			return SVTGPU_OK;
		}
		if (slot < 0 && m->d_split[i] == NULL)
			slot = i;
	}
	if (slot < 0) {   /* evict round-robin */
		slot = m->split_next;
		m->split_next = (m->split_next + 1) % SVTGPU_NSPLIT;
		SVT_CUDA(svt_free_async(m->d_split[slot], s));
		m->d_split[slot] = NULL;
	}
	const int64_t n = m->nleaf * (c.ntiles - 1);
	SVT_CUDA(svt_malloc_async((void **) &m->d_split[slot],
				 sizeof(int32_t) * (size_t) (n > 0 ? n : 1), s));
	row_split<<<grid_for(n, 256), 256, 0, s>>>(m->d_offs, m->d_leaf_ptr,
			m->nleaf, c.ntiles, c.tile_rows, m->d_split[slot]);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	m->split_tile_rows[slot] = c.tile_rows;
	m->split_ntiles[slot] = c.ntiles;
	*split = m->d_split[slot];
	return SVTGPU_OK;
}

/* max |x| of an integer matrix, computed once and cached in the handle */
/* ------------------------------------------------------------------------
 * row_hist: row sums of integer / lacunar input as a shared-memory histogram.
 *
 * A row sum does not care which leaf a nonzero comes from, so the kernel
 * streams its chunk of (offset, value) pairs -- no split tables, no sub-runs --
 * and adds into one cell per row with native shared-memory atomics.  Cells
 * are int32 (values) or 16-bit halves of a 32-bit word (lacunar: counts), so
 * 100,000 rows fit one SM.  A row meets at most one nonzero per leaf: the
 * chunk is cut (at leaf boundaries) into pieces of at most `piece_leaves`
 * leaves, the host's bound for "cannot overflow a cell", and the cells are
 * added to the global state (exact integer-valued doubles, any order) after
 * every piece.  NA values bump the per-row NA counter instead.
 */
struct RowHistParams {
	const int32_t *offs;
	const int32_t *vals;       /* NULL: lacunar */
	const uint16_t *offs16;    /* compact copy (row_hist<MODE, true>) */
	const int8_t *vals8;
	const int64_t *leaf_ptr;
	int64_t nleaf, nnz, nrow;
	int nchunks;
	int piece_leaves;
	int back_first;
	int lacunar_vec;
	const int64_t *tile_leaf;  /* cyclic form: [ntiles + 1], else NULL */
	int64_t tile, ntiles;
	double *state;
};

enum { HIST_COUNT16 = 0, HIST_SUM32 = 1, HIST_MOMENTS = 2, HIST_MAX32 = 3 };
#define HIST_THREADS 1024

__device__ __forceinline__ void hist_red(uint32_t saddr, uint32_t v)
{
	asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(saddr), "r"(v)
		     : "memory");
}

__device__ __forceinline__ void hist_red_max(uint32_t saddr, uint32_t v)
{
	asm volatile("red.shared.max.u32 [%0], %1;" :: "r"(saddr), "r"(v)
		     : "memory");
}

/* MODE: HIST_COUNT16 lacunar counts in 16-bit halves; HIST_SUM32 integer sums
   in int32 cells; HIST_MOMENTS small non-negative integers, sum(x) in the low
   and sum(x^2) in the high 16 bits of one cell -- piece_leaves is then what
   cannot add 2^15 to a half, and the cells are only flushed when a guard bit
   (2^15 of a half) shows, as in row_strips. */
template <int MODE, bool NARROW>
__global__ void __launch_bounds__(HIST_THREADS, 1)
row_hist(RowHistParams P)
{
	extern __shared__ __align__(128) unsigned char smem[];
	unsigned int *cell = (unsigned int *) smem;
	const uint32_t cell_s = (uint32_t) __cvta_generic_to_shared(cell);
	constexpr bool LACUNAR = MODE == HIST_COUNT16;
	const int64_t ncell = LACUNAR ? (P.nrow + 1) / 2 : P.nrow;
	/* loads per thread and batch (64 KB per SM); the value modes keep two
	   batches in flight */
	constexpr int U = LACUNAR ? 16 : 8;

	/* entries [start, end) into the cells */
	auto stream = [&](const int64_t start, const int64_t end) {
	/* full batches of HIST_THREADS x U entries: no bounds,
	   one pointer + immediate offsets, 32-bit shared
	   addresses (ncu: the predicated 64-bit form below cost
	   23 warp instructions per 32 entries and made the
	   lacunar kernel issue-bound at 0.60 of HBM) */
	/* (lacunar counts stay on the predicated loop: with one
	   atomic per 4 bytes they are bound by the bank
	   conflicts of the atomics -- 3.5 wavefronts per warp
	   instruction, tools/microbench/atoms_patterns.cu --
	   and measured 2.03 ms that way against 2.2-2.4 ms
	   with the leaner loop) */
	int64_t lac_done = 0;
	if (LACUNAR && P.lacunar_vec) {
		/* lacunar counts: 16-byte loads -- four load
		   instructions per 16 entries instead of sixteen.
		   With one atomic per 4 bytes this kernel waits on
		   the MIO queue (ncu: 52 % of the stall samples,
		   the shared-memory pipe 35 % busy), and the load
		   instructions are what filled it: 2.07 -> 1.65 ms
		   at 2e9 entries (double-buffering on top: no
		   change).  The value modes, which are HBM-bound,
		   got slower with 16-byte loads and keep 4-byte
		   ones. */
		int64_t head = (4 - (start & 3)) & 3;
		if (head > end - start) head = end - start;
		if ((int64_t) threadIdx.x < head) {
			const int o = P.offs[start + threadIdx.x];
			atomicAdd(&cell[o >> 1], 1u << ((o & 1) * 16));
		}
		const int64_t vstart = start + head;
		const int64_t nb = (end - vstart) /
				   ((int64_t) HIST_THREADS * 16);
		const int4 *pq = (const int4 *) (P.offs + vstart) +
				 threadIdx.x;
		for (int64_t b = 0; b < nb; b++) {
			int4 v[4];
#pragma unroll
			for (int k = 0; k < 4; k++)
				v[k] = ldg_stream_v4(pq + k * HIST_THREADS);
			pq += 4 * HIST_THREADS;
#pragma unroll
			for (int k = 0; k < 4; k++) {
				const uint32_t e[4] = {
					(uint32_t) v[k].x, (uint32_t) v[k].y,
					(uint32_t) v[k].z, (uint32_t) v[k].w };
#pragma unroll
				for (int j = 0; j < 4; j++)
					hist_red(cell_s + ((e[j] << 1) & ~3u),
						 (e[j] & 1u) * 0xFFFFu + 1u);
			}
		}
		lac_done = head + nb * HIST_THREADS * 16;
	}
	const int64_t nfull = LACUNAR ? 0 : (end - start) /
			      ((int64_t) HIST_THREADS * U);
	const int32_t *po = P.offs + start + threadIdx.x;
	const int32_t *pv = LACUNAR ? NULL
			  : P.vals + start + threadIdx.x;
	/* double-buffered: the next batch is requested before
	   this one is added, so loads stay in flight while the
	   shared-memory pipe works through the atomics */
	int o_nx[U], x_nx[U];
	auto request = [&]() {
#pragma unroll
		for (int k = 0; k < U; k++) {
			o_nx[k] = ldg_stream<int32_t>(
				po + k * HIST_THREADS);
			if (!LACUNAR)
				x_nx[k] = ldg_stream<int32_t>(
					pv + k * HIST_THREADS);
		}
		po += HIST_THREADS * U;
		if (!LACUNAR)
			pv += HIST_THREADS * U;
	};
	if (nfull > 0)
		request();
	for (int64_t b = 0; b < nfull; b++) {
		int o[U], x[U];
#pragma unroll
		for (int k = 0; k < U; k++) {
			o[k] = o_nx[k];
			if (!LACUNAR)
				x[k] = x_nx[k];
		}
		if (b + 1 < nfull)
			request();
#pragma unroll
		for (int k = 0; k < U; k++) {
			if (MODE == HIST_COUNT16) {
				const uint32_t ou = (uint32_t) o[k];
				hist_red(cell_s + ((ou << 1) & ~3u),
					 (ou & 1u) * 0xFFFFu + 1u);
			} else if (x[k] == SVT_NA_INT) {
				atomicAdd(&P.state[SVT_ROW_SLOT_NA *
					P.nrow + o[k]], 1.0);
			} else if (MODE == HIST_MOMENTS) {
				const unsigned int v =
					(unsigned int) x[k];
				hist_red(cell_s + ((uint32_t) o[k] << 2),
					 v * ((v << 16) + 1u));
			} else if (MODE == HIST_MAX32) {
				hist_red_max(cell_s +
					((uint32_t) o[k] << 2),
					(unsigned int) x[k] + 1u);
			} else {
				hist_red(cell_s + ((uint32_t) o[k] << 2),
					 (unsigned int) x[k]);
			}
		}
	}
	for (int64_t base = start + lac_done +
			    nfull * HIST_THREADS * U +
			    threadIdx.x; base < end;
	     base += (int64_t) HIST_THREADS * U) {
		int o[U], x[U];
#pragma unroll
		for (int k = 0; k < U; k++) {
			const int64_t e = base +
				(int64_t) k * HIST_THREADS;
			const bool ok = e < end;
			o[k] = ok ? P.offs[e] : -1;
			x[k] = (ok && !LACUNAR) ? P.vals[e] : 1;
		}
#pragma unroll
		for (int k = 0; k < U; k++) {
			if (o[k] < 0)
				continue;
			if (MODE == HIST_COUNT16) {
				atomicAdd(&cell[o[k] >> 1],
					  1u << ((o[k] & 1) * 16));
			} else if (x[k] == SVT_NA_INT) {
				atomicAdd(&P.state[SVT_ROW_SLOT_NA *
					P.nrow + o[k]], 1.0);
			} else if (MODE == HIST_MOMENTS) {
				const unsigned int v =
					(unsigned int) x[k];
				atomicAdd(&cell[o[k]],
					  v * ((v << 16) + 1u));
			} else if (MODE == HIST_MAX32) {
				atomicMax(&cell[o[k]],
					  (unsigned int) x[k] + 1u);
			} else {
				atomicAdd(&cell[o[k]],
					  (unsigned int) x[k]);
			}
		}
	}
	};
	/* NARROW (HIST_SUM32 / HIST_MOMENTS only): the same entries from the
	   compact copy (svtgpu_internal.h), 3 bytes each instead of 8 */
	auto add8 = [&](const uint32_t o, const int x) {
		if (x == SVT_COMPACT_NA_I8) {
			atomicAdd(&P.state[SVT_ROW_SLOT_NA * P.nrow + o], 1.0);
		} else if (MODE == HIST_MOMENTS) {
			const unsigned int v = (unsigned int) x;
			hist_red(cell_s + (o << 2), v * ((v << 16) + 1u));
		} else {
			hist_red(cell_s + (o << 2), (unsigned int) x);
		}
	};
	auto stream8 = [&](const int64_t start, const int64_t end) {
	/* single entries up to a multiple of 8, then batches in which every
	   thread takes K groups of 8 entries (one 16-byte load of offsets and
	   one 8-byte load of values each), double-buffered as above */
	constexpr int K = 2;
	int64_t head = (8 - (start & 7)) & 7;
	if (head > end - start)
		head = end - start;
	if ((int64_t) threadIdx.x < head)
		add8(P.offs16[start + threadIdx.x], P.vals8[start + threadIdx.x]);
	const int64_t vstart = start + head;
	const int64_t nfull = (end - vstart) / ((int64_t) HIST_THREADS * 8 * K);
	const int4 *po = (const int4 *) (P.offs16 + vstart) + threadIdx.x;
	const uint2 *pv = (const uint2 *) (P.vals8 + vstart) + threadIdx.x;
	int4 o_nx[K];
	uint2 v_nx[K];
	auto request = [&]() {
#pragma unroll
		for (int k = 0; k < K; k++) {
			o_nx[k] = ldg_stream_v4(po + k * HIST_THREADS);
			v_nx[k] = ldg_stream_v2(pv + k * HIST_THREADS);
		}
		po += K * HIST_THREADS;
		pv += K * HIST_THREADS;
	};
	if (nfull > 0)
		request();
	for (int64_t b = 0; b < nfull; b++) {
		int4 o[K];
		uint2 v[K];
#pragma unroll
		for (int k = 0; k < K; k++) {
			o[k] = o_nx[k];
			v[k] = v_nx[k];
		}
		if (b + 1 < nfull)
			request();
#pragma unroll
		for (int k = 0; k < K; k++) {
			const uint32_t ow[4] = { (uint32_t) o[k].x, (uint32_t) o[k].y,
						 (uint32_t) o[k].z, (uint32_t) o[k].w };
			const uint32_t vw[2] = { v[k].x, v[k].y };
#pragma unroll
			for (int j = 0; j < 8; j++)
				add8((ow[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu,
				     (int) (int8_t) (vw[j >> 2] >> ((j & 3) * 8)));
		}
	}
	for (int64_t e = vstart + nfull * HIST_THREADS * 8 * K + threadIdx.x;
	     e < end; e += HIST_THREADS)
		add8(P.offs16[e], P.vals8[e]);
	};
	auto feed = [&](const int64_t start, const int64_t end) {
		if (NARROW)
			stream8(start, end);
		else
			stream(start, end);
	};
	/* after a piece: MOMENTS keeps accumulating on chip while no guard bit
	   shows; everything else (and the last piece) goes to the row state */
	auto checkpoint = [&](const bool last) {
	__syncthreads();
	if (MODE == HIST_MOMENTS && !last) {
		/* keep accumulating on chip while no half has
		   reached 2^15 */
		int risky = 0;
		for (int64_t r = threadIdx.x; r < P.nrow;
		     r += blockDim.x)
			risky |= (cell[r] & 0x80008000u) != 0;
		if (!__syncthreads_or(risky))
			return;
	}
	for (int64_t r = threadIdx.x; r < P.nrow;
	     r += blockDim.x) {
		if (MODE == HIST_MAX32) {
			/* the extreme, and "the row holds a
			   regular value" in the coverage slot
			   (see launch_class) */
			const unsigned int c = cell[r];
			if (c != 0) {
				atomic_max_double(&P.state[
					SVT_ROW_SLOT_EXT * P.nrow + r],
					(double) (c - 1u));
				atomicAdd(&P.state[SVT_ROW_SLOT_CVG *
					P.nrow + r], 1.0);
			}
			continue;
		}
		if (MODE == HIST_MOMENTS) {
			const unsigned int c = cell[r];
			if (c != 0) {
				atomicAdd(&P.state[SVT_ROW_SLOT_SUM *
					P.nrow + r],
					(double) (c & 0xFFFFu));
				atomicAdd(&P.state[SVT_ROW_SLOT_SUM2 *
					P.nrow + r],
					(double) (c >> 16));
			}
			continue;
		}
		const int v = LACUNAR
			? (int) ((cell[r >> 1] >> ((r & 1) * 16))
				 & 0xFFFFu)
			: (int) cell[r];
		if (v != 0)
			atomicAdd(&P.state[SVT_ROW_SLOT_SUM *
				P.nrow + r], (double) v);
	}
	__syncthreads();
	if (!last) {
		for (int64_t i = threadIdx.x; i < ncell;
		     i += blockDim.x)
			cell[i] = 0;
		__syncthreads();
	}

	};

	if (P.tile_leaf != NULL) {
		/* CYCLIC: the entry range is cut into tiles of P.tile entries
		   and CTA b takes tiles b, b + grid, ... -- the whole GPU sweeps
		   the arrays front to back, as the column kernels do, instead of
		   148 streams far apart.  Measured on 2.3e9 entries: 2.74 ms
		   against 2.87 ms back to back, and 2.74 against 3.03-3.27 ms
		   right after a column reduction (the first 1.4 ms of the
		   chunked kernel ran 10-30 % slower after any other kernel).
		   tile_leaf[t] = the leaf that holds the tile's first entry: a
		   tile touches tile_leaf[t + 1] - tile_leaf[t] + 1 leaves (the
		   host has checked that this never exceeds piece_leaves), and
		   the cells are looked at before that count can pass
		   piece_leaves. */
		for (int64_t i = threadIdx.x; i < ncell; i += blockDim.x)
			cell[i] = 0;
		__syncthreads();
		int64_t used = 0;
		int64_t t = blockIdx.x;
		int64_t la = 0, lb = 0;
		if (t < P.ntiles) {
			la = P.tile_leaf[t];
			lb = P.tile_leaf[t + 1];
		}
		while (t < P.ntiles) {
			const int64_t L = lb - la + 1;
			const int64_t tn = t + gridDim.x;
			int64_t na = 0, nb = 0;
			if (tn < P.ntiles) {          /* the next tile's leaves */
				na = P.tile_leaf[tn];
				nb = P.tile_leaf[tn + 1];
			}
			if (used + L > P.piece_leaves) {
				checkpoint(false);
				used = 0;
			}
			used += L;
			const int64_t start = t * P.tile;
			feed(start, start + P.tile < P.nnz ? start + P.tile
							   : P.nnz);
			t = tn;
			la = na;
			lb = nb;
		}
		checkpoint(true);
		return;
	}

	for (int chunk_i = blockIdx.x; chunk_i < P.nchunks; chunk_i += gridDim.x) {
		/* (chunked form: the second half of the arrays first, which
		   halves the slow start described above) */
		int chunk = chunk_i;
		if (P.back_first && P.nchunks == 2 * (int) gridDim.x)
			chunk = chunk_i < (int) gridDim.x ? chunk_i + (int) gridDim.x
							  : chunk_i - (int) gridDim.x;
		/* leaves [l0, l1) of this chunk, balanced by nonzeros */
		int64_t bounds[2];
		for (int k = 0; k < 2; k++) {
			const int c = chunk + k;
			if (c >= P.nchunks) { bounds[k] = P.nleaf; continue; }
			const int64_t target = (int64_t) ((double) P.nnz *
					((double) c / (double) P.nchunks));
			int64_t lo = 0, hi = P.nleaf;
			while (lo < hi) {
				const int64_t mid = lo + ((hi - lo) >> 1);
				if (P.leaf_ptr[mid] < target) lo = mid + 1;
				else                          hi = mid;
			}
			bounds[k] = c == 0 ? 0 : lo;
		}
		for (int64_t i = threadIdx.x; i < ncell; i += blockDim.x)
			cell[i] = 0;
		__syncthreads();
		for (int64_t p0 = bounds[0]; p0 < bounds[1];
		     p0 += P.piece_leaves) {
			const int64_t p1 = p0 + P.piece_leaves < bounds[1]
					   ? p0 + P.piece_leaves : bounds[1];
			feed(P.leaf_ptr[p0], P.leaf_ptr[p1]);
			checkpoint(p1 == bounds[1]);
		}
	}
}

/* tile_leaf[t] = the leaf that holds entry t * tile (t = ntiles: the last
   leaf); *max_leaves = the most leaves any tile touches */
__global__ void __launch_bounds__(256)
hist_tile_leaves(const int64_t *__restrict__ leaf_ptr, int64_t nleaf,
		 int64_t nnz, int64_t tile, int64_t ntiles,
		 int64_t *__restrict__ tile_leaf, int *max_leaves, int pass)
{
	const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (t > ntiles)
		return;
	if (pass == 0) {
		int64_t e = t * tile;
		if (e > nnz - 1) e = nnz - 1;
		/* first leaf whose range ends after entry e */
		int64_t lo = 0, hi = nleaf;
		while (lo < hi) {
			const int64_t mid = lo + ((hi - lo) >> 1);
			if (leaf_ptr[mid + 1] <= e) lo = mid + 1;
			else                        hi = mid;
		}
		tile_leaf[t] = lo;
	} else if (t < ntiles) {
		const int64_t L = tile_leaf[t + 1] - tile_leaf[t] + 1;
		atomicMax(max_leaves, L > INT32_MAX ? INT32_MAX : (int) L);
	}
}

int launch_row_hist(svtgpu_matrix *m, int mode, int64_t max_abs,
		    double *d_state, cudaStream_t s)
{
	const bool lac = mode == HIST_COUNT16;
	RowHistParams P;
	memset(&P, 0, sizeof(P));
	P.offs = m->d_offs;
	P.vals = lac ? NULL : (const int32_t *) m->d_vals;
	P.leaf_ptr = m->d_leaf_ptr;
	P.nleaf = m->nleaf;
	P.nnz = m->nnz;
	P.nrow = m->nrow;
	bool narrow = false;
	if (mode == HIST_SUM32 || mode == HIST_MOMENTS) {
		SVT_CHECK(svt_ensure_compact(m, s));
		narrow = m->d_offs16 != NULL && m->d_vals8 != NULL;
		P.offs16 = m->d_offs16;
		P.vals8 = m->d_vals8;
	}
	const int sms = svtgpu_sm_count();
	P.nchunks = (int64_t) sms * 2 < m->nleaf ? sms * 2
						 : (m->nleaf > 0 ? (int) m->nleaf : 1);
	/* a row meets at most one nonzero per leaf */
	const int64_t M = max_abs > 0 ? max_abs : 1;
	const int64_t lim = mode == HIST_COUNT16 ? 65535
			  : mode == HIST_MAX32 ? ((int64_t) 1 << 30)
			  : mode == HIST_MOMENTS ? 32767 / (M * M)
			  : (int64_t) INT32_MAX / M;
	P.piece_leaves = (int) (lim < 1 ? 1 : lim > (1 << 30) ? (1 << 30) : lim);
	/* test hook: shorter pieces exercise the flush / guard paths on small
	   inputs (never longer than the safe bound) */
	const int forced = atoi(svtgpu_env("SVTGPU_ROW_HIST_PIECE", "0"));
	if (forced > 0 && forced < P.piece_leaves)
		P.piece_leaves = forced;
	P.state = d_state;
	P.back_first = strcmp(svtgpu_env("SVTGPU_ROW_HIST_ORDER", "back"),
			      "back") == 0;
	P.lacunar_vec = atoi(svtgpu_env("SVTGPU_ROW_HIST_LACUNAR_VEC", "1")) &&
			(((uintptr_t) m->d_offs) & 15) == 0;
	const size_t smem = lac ? 4 * (size_t) ((m->nrow + 1) / 2)
				: 4 * (size_t) m->nrow;
	int grid = P.nchunks < sms ? P.nchunks : sms;
	/* the cyclic form (tiles of 4 batches, round-robin over the SMs) when
	   there are at least 4 tiles per SM and no tile touches more leaves
	   than a cell can take; the tile table is built once per matrix */
	const int64_t tile = (int64_t) HIST_THREADS * (lac ? 16 : 8) * 4;
	const int64_t ntiles = (m->nnz + tile - 1) / tile;
	if (ntiles >= (int64_t) sms * 4 &&
	    strcmp(svtgpu_env("SVTGPU_ROW_HIST_TILES", "cyclic"), "cyclic") == 0) {
		if (m->d_hist_tiles == NULL || m->hist_tile != tile) {
			if (m->d_hist_tiles != NULL)
				svt_free_async(m->d_hist_tiles, s);
			m->d_hist_tiles = NULL;
			int *d_max = NULL;
			SVT_CUDA(svt_malloc_async((void **) &m->d_hist_tiles,
					8 * (size_t) (ntiles + 1) + 64, s));
			d_max = (int *) (m->d_hist_tiles + ntiles + 1);
			SVT_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int), s));
			const unsigned g = (unsigned) ((ntiles + 1 + 255) / 256);
			hist_tile_leaves<<<g, 256, 0, s>>>(m->d_leaf_ptr, m->nleaf,
				m->nnz, tile, ntiles, m->d_hist_tiles, d_max, 0);
			hist_tile_leaves<<<g, 256, 0, s>>>(m->d_leaf_ptr, m->nleaf,
				m->nnz, tile, ntiles, m->d_hist_tiles, d_max, 1);
			SVT_CUDA(cudaGetLastError());
			svtgpu_count_launch(2);
			int h_max = 0;
			SVT_CUDA(cudaMemcpyAsync(&h_max, d_max, sizeof(int),
					cudaMemcpyDeviceToHost, s));
			SVT_CUDA(cudaStreamSynchronize(s));
			m->hist_tile = tile;
			m->hist_ntiles = ntiles;
			m->hist_max_leaves = h_max;
		}
		if (m->hist_max_leaves <= P.piece_leaves) {
			P.tile_leaf = m->d_hist_tiles;
			P.tile = tile;
			P.ntiles = ntiles;
			grid = sms;
		}
	}
#define HIST_LAUNCH(MODE, NARROW) do { \
		SVT_CUDA(cudaFuncSetAttribute(row_hist<MODE, NARROW>, \
			cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem)); \
		row_hist<MODE, NARROW><<<grid, HIST_THREADS, smem, s>>>(P); \
	} while (0)
	if (mode == HIST_COUNT16)      HIST_LAUNCH(HIST_COUNT16, false);
	else if (mode == HIST_MOMENTS && narrow) HIST_LAUNCH(HIST_MOMENTS, true);
	else if (mode == HIST_MOMENTS) HIST_LAUNCH(HIST_MOMENTS, false);
	else if (mode == HIST_MAX32)   HIST_LAUNCH(HIST_MAX32, false);
	else if (narrow)               HIST_LAUNCH(HIST_SUM32, true);
	else                           HIST_LAUNCH(HIST_SUM32, false);
#undef HIST_LAUNCH
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

/* lacunar input after the counting pass: slot 0 holds the number of stored
   entries of the row (= sum = coverage) */
__global__ void __launch_bounds__(256)
row_lacunar_derive(double *state, int64_t nrow, int want_sum2)
{
	const int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= nrow)
		return;
	const double n = state[SVT_ROW_SLOT_SUM * nrow + r];
	if (want_sum2)
		state[SVT_ROW_SLOT_SUM2 * nrow + r] = n;
	else if (n > 0.0)
		state[SVT_ROW_SLOT_EXT * nrow + r] = 1.0;
}

/* row_hist<HIST_MAX32>: coverage slot += #NA, so that the number of regular
   values of svt_row_finalize() (coverage - #NA) is positive exactly when the
   row holds one */
__global__ void __launch_bounds__(256)
row_max_hist_coverage(double *state, int64_t nrow)
{
	const int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (r < nrow)
		state[SVT_ROW_SLOT_CVG * nrow + r] +=
			state[SVT_ROW_SLOT_NA * nrow + r];
}

int ensure_absmax(svtgpu_matrix *m, cudaStream_t s)
{
	if (m->vmax_abs >= 0)
		return SVTGPU_OK;
	if (!(m->flags & SVTGPU_HAS_VALS) || m->nnz == 0) {
		m->vmax_abs = 1;
		m->vmin = 0;
		return SVTGPU_OK;
	}
	unsigned long long *d_max = NULL, h_max[2] = { 0, 0 };
	SVT_CUDA(svt_malloc_async((void **) &d_max, 2 * sizeof(*d_max), s));
	cudaError_t e = cudaMemsetAsync(d_max, 0, 2 * sizeof(*d_max), s);
	if (e == cudaSuccess) {
		absmax_int<<<grid_for(m->nnz, 256 * 16), 256, 0, s>>>(
			(const int32_t *) m->d_vals, m->nnz, d_max);
		e = cudaGetLastError();
		svtgpu_count_launch(1);
	}
	if (e == cudaSuccess)
		e = cudaMemcpyAsync(h_max, d_max, sizeof(h_max),
				    cudaMemcpyDeviceToHost, s);
	if (e == cudaSuccess)
		e = cudaStreamSynchronize(s);
	svt_free_async(d_max, s);
	SVT_CUDA(e);
	m->vmax_abs = (int64_t) h_max[0];
	m->vmin = h_max[1] > 0 ? -1 : 0;   /* only the sign matters */
	return SVTGPU_OK;
}

template <int RC, typename T, bool LAC>
int launch_flat(const svtgpu_matrix *m, int is_min, double *d_state,
		cudaStream_t s)
{
	row_flat<RC, T, LAC><<<grid_for(m->nnz, 256 * 8), 256, 0, s>>>(
		m->d_offs, (const T *) m->d_vals, m->nnz, m->nrow, is_min,
		d_state);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

template <int RC, typename T, bool LAC, typename ACC>
int launch_tiles(svtgpu_matrix *m, const TileConfig &c, int is_min,
		 int64_t flush_leaves, double *d_state, cudaStream_t s)
{
	constexpr int NACC = RC == RC_SUM ? 1 : 2;
	const int32_t *split = NULL;
	SVT_CHECK(ensure_split(m, c, s, &split));
	void *part = NULL;
	SVT_CHECK(svtgpu_scratch(m, sizeof(double) * (size_t) c.nchunks *
				 NACC * (size_t) m->nrow + 64, &part));
	RowTileParams P;
	P.offs = m->d_offs;
	P.vals = LAC ? NULL : m->d_vals;
	P.leaf_ptr = m->d_leaf_ptr;
	P.split = split;
	P.nleaf = m->nleaf;
	P.nnz = m->nnz;
	P.nrow = m->nrow;
	P.ntiles = c.ntiles;
	P.tile_rows = c.tile_rows;
	P.nchunks = c.nchunks;
	P.stage_elems = c.stage_elems;
	P.is_min = is_min;
	P.flush_leaves = flush_leaves;
	P.part = (double *) part;
	P.state = d_state;
	SVT_CUDA(cudaFuncSetAttribute(row_tiles<RC, T, LAC, ACC>,
		cudaFuncAttributeMaxDynamicSharedMemorySize, (int) c.smem));
	row_tiles<RC, T, LAC, ACC><<<(unsigned) (c.nchunks * c.ntiles),
				     ROW_THREADS, c.smem, s>>>(P);
	SVT_CUDA(cudaGetLastError());
	row_combine<RC><<<grid_for(m->nrow, 256), 256, 0, s>>>(
		(const double *) part, c.nchunks, m->nrow, is_min, d_state);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(2);
	return SVTGPU_OK;
}

struct StripConfig {
	int ok;
	int ntiles, nchunks, nstrips, strip_rows, warps;
	int slots;           /* ST_U: 2, 3, 4 or 6 */
	size_t smem;
};

/* One CTA per SM holding as many rows as fit; W warps each owning
 * strip_rows of them.  W is picked so a typical sub-run fills the register
 * ring's slots well. */
StripConfig choose_strips(int64_t nrow, int64_t nleaf, int64_t nnz, int nacc,
			  int acc_size)
{
	StripConfig c;
	memset(&c, 0, sizeof(c));
	const int sms = svtgpu_sm_count();
	const size_t budget = (size_t) 227 * 1024 - 1024 - 256;
	const double avg_leaf = nleaf > 0 ? (double) nnz / (double) nleaf : 0.0;
	int force_w = atoi(svtgpu_env("SVTGPU_ROW_WARPS", "0"));
	int force_t = atoi(svtgpu_env("SVTGPU_ROW_NTILES", "0"));
	for (int nt = force_t > 0 ? force_t : 1; nt <= 64; nt++) {
		int W = force_w;
		if (W <= 0) {
			/* as many warps as give sub-runs of >= ~60 nonzeros:
			   memory-level parallelism comes from warps (measured:
			   16 warps x 62 beats 8 warps x 125 by 19 %) */
			double per_tile = avg_leaf / nt;
			W = (int) (per_tile / 60.0 + 0.5);
			if (W < 4) W = 4;
			if (W > 16) W = 16;
			/* two double accumulators per row (row moments of
			   doubles): measured on 33,538 rows at d = 0.07, 16
			   warps x 3 tiles with a 2-slot ring (the ~20 % of
			   sub-runs beyond 64 entries take the scalar tail) runs
			   at 8.4 ms per 2.3e9 nonzeros against 12.5 ms for 13
			   warps and 3 slots (tools/sweep_rows.sh) */
			if (nacc == 2 && acc_size == 8 && per_tile >= 16 * 24.0)
				W = 16;
		}
		if (W > 16) W = 16;   /* __launch_bounds__(512): 128 registers */
		const int S = nt * W;
		int64_t sr = (nrow + S - 1) / S;
		sr = (sr + 31) / 32 * 32;
		if (sr < 32) sr = 32;
		const size_t smem = (size_t) W * nacc * sr * acc_size + 128;
		if (smem <= budget) {
			/* slots for mean + 3 sigma of a sub-run's length */
			const double L = avg_leaf / S;
			const double need = (L + 3.0 * sqrt(L > 0 ? L : 0.0)) /
					    32.0;
			c.slots = need <= 2.0 ? 2 : need <= 3.0 ? 3
				: need <= 4.0 ? 4 : 6;
			if (nacc == 2 && acc_size == 8 && need <= 3.0)
				c.slots = 2;
			const int fu = atoi(svtgpu_env("SVTGPU_ROW_SLOTS", "0"));
			if (fu == 2 || fu == 3 || fu == 4 || fu == 6)
				c.slots = fu;
			c.ok = 1;
			c.ntiles = nt;
			c.warps = W;
			c.nstrips = S;
			c.strip_rows = (int) sr;
			c.smem = smem;
			c.nchunks = sms / nt;
			if (c.nchunks < 1) c.nchunks = 1;
			const int mult = atoi(svtgpu_env("SVTGPU_ROW_CHUNK_MULT",
							 "1"));
			if (mult > 1) c.nchunks *= mult;
			/* the kernel keeps 32-bit positions relative to its
			   chunk: a chunk is < nnz / nchunks + nrow nonzeros */
			const int64_t minc = nnz / ((int64_t) 1 << 30) + 1;
			if ((int64_t) c.nchunks < minc) c.nchunks = (int) minc;
			if ((int64_t) c.nchunks > nleaf)
				c.nchunks = nleaf > 0 ? (int) nleaf : 1;
			return c;
		}
		if (force_t > 0)
			break;
	}
	return c;
}

template <int RC, typename T, bool LAC, typename ACC, bool PACKED>
int launch_strips(svtgpu_matrix *m, const StripConfig &c, int is_min,
		  int64_t flush_leaves, double *d_state, cudaStream_t s)
{
	constexpr int NACC = RC == RC_SUM ? 1 : 2;
	TileConfig tc;
	memset(&tc, 0, sizeof(tc));
	tc.ntiles = c.nstrips;
	tc.tile_rows = c.strip_rows;
	const int32_t *split = NULL;
	SVT_CHECK(ensure_split(m, tc, s, &split));
	void *part = NULL;
	SVT_CHECK(svtgpu_scratch(m, sizeof(double) * (size_t) c.nchunks *
				 NACC * (size_t) m->nrow + 64, &part));
	RowStripParams P;
	P.offs = m->d_offs;
	P.vals = LAC ? NULL : m->d_vals;
	P.leaf_ptr = m->d_leaf_ptr;
	P.split = split;
	P.nleaf = m->nleaf;
	P.nnz = m->nnz;
	P.nrow = m->nrow;
	P.ntiles = c.ntiles;
	P.nchunks = c.nchunks;
	P.nstrips = c.nstrips;
	P.strip_rows = c.strip_rows;
	P.is_min = is_min;
	P.flush_leaves = flush_leaves > INT32_MAX ? INT32_MAX
						   : (int) flush_leaves;
	P.part = (double *) part;
	P.state = d_state;
#define STRIP_LAUNCH(D, U) do { \
		SVT_CUDA(cudaFuncSetAttribute( \
			row_strips<RC, T, LAC, ACC, PACKED, D, U>, \
			cudaFuncAttributeMaxDynamicSharedMemorySize, \
			(int) c.smem)); \
		row_strips<RC, T, LAC, ACC, PACKED, D, U><<<(unsigned) \
			(c.nchunks * c.ntiles), c.warps * 32, c.smem, s>>>(P); \
	} while (0)
	switch (c.slots) {
	    case 2: STRIP_LAUNCH(8, 2); break;
	    case 3: STRIP_LAUNCH(8, 3); break;
	    case 4: STRIP_LAUNCH(4, 4); break;
	    default: STRIP_LAUNCH(4, 6); break;
	}
#undef STRIP_LAUNCH
	SVT_CUDA(cudaGetLastError());
	row_combine<RC><<<grid_for(m->nrow, 256), 256, 0, s>>>(
		(const double *) part, c.nchunks, m->nrow, is_min, d_state);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(2);
	return SVTGPU_OK;
}

template <int RC>
int launch_class(svtgpu_matrix *m, const char *impl, int is_min,
		 double *d_state, cudaStream_t s)
{
	constexpr int NACC = RC == RC_SUM ? 1 : 2;
	const bool lac = !(m->flags & SVTGPU_HAS_VALS);
	const bool dbl = svt_is_double(m->val_type);
	const bool aligned = (((uintptr_t) m->d_offs) & 15) == 0 &&
			     (((uintptr_t) m->d_vals) & 15) == 0;
	bool tiles = aligned && strcmp(impl, "flat") != 0;
	/* integer / lacunar input: int32 accumulators when the values allow a
	   useful number of leaves between flushes */
	bool int_acc = false;
	int64_t flush_leaves = INT64_MAX;
	if (tiles && (lac || !dbl) && strcmp(impl, "f64acc") != 0) {
		SVT_CHECK(ensure_absmax(m, s));
		const int64_t M = m->vmax_abs > 0 ? m->vmax_abs : 1;
		const int64_t lim = INT32_MAX;
		int64_t F = lim / M;                       /* sums, coverage */
		if (RC == RC_X2)
			F = M > 46340 ? 0 : lim / (M * M);  /* sums of squares */
		if (RC == RC_MINMAX)
			F = lim;
		if (F >= 64) {
			int_acc = true;
			flush_leaves = F;
		}
	}
	/* row sums (and packed row moments) of integer / lacunar input whose
	   cells fit one SM: the shared-memory histogram -- the default;
	   SVTGPU_ROW_HIST=off goes back to the strip kernels */
	if ((RC == RC_SUM || RC == RC_X2) && (lac || !dbl) && int_acc &&
	    (strcmp(impl, "strips") == 0 || strcmp(impl, "hist") == 0) &&
	    strcmp(svtgpu_env("SVTGPU_ROW_HIST", "auto"), "off") != 0) {
		const int64_t M = m->vmax_abs > 0 ? m->vmax_abs : 1;
		const bool fits32 = 4 * (size_t) m->nrow <= (size_t) 200 * 1024;
		if (RC == RC_SUM && lac &&
		    2 * (size_t) (m->nrow + 1) <= (size_t) 200 * 1024)
			return launch_row_hist(m, HIST_COUNT16, 1, d_state, s);
		if (RC == RC_SUM && !lac && fits32)
			return launch_row_hist(m, HIST_SUM32, M, d_state, s);
		if (RC == RC_X2 && !lac && fits32 && m->vmin >= 0 &&
		    M * M * 64 <= 32767)
			return launch_row_hist(m, HIST_MOMENTS, M, d_state, s);
	}
	/* row maxima of NON-NEGATIVE integers: one shared-memory atomic max
	   per nonzero.  The background zero never beats a regular value >= 0,
	   so the exact coverage count is not needed: svt_row_finalize() only
	   has to know whether the row holds any regular value (else the row is
	   all NA and its coverage is the NA count, which is exact).  The
	   coverage slot therefore receives #NA (row_max_hist_coverage) + one
	   per chunk that saw a regular value.  Row minima need the true
	   coverage and stay on row_strips. */
	if (RC == RC_MINMAX && !is_min && !lac && !dbl && int_acc &&
	    m->vmin >= 0 && m->vmax_abs < INT32_MAX - 1 &&
	    4 * (size_t) m->nrow <= (size_t) 200 * 1024 &&
	    (strcmp(impl, "strips") == 0 || strcmp(impl, "hist") == 0) &&
	    strcmp(svtgpu_env("SVTGPU_ROW_HIST", "auto"), "off") != 0) {
		SVT_CHECK(launch_row_hist(m, HIST_MAX32, 1, d_state, s));
		row_max_hist_coverage<<<grid_for(m->nrow, 256), 256, 0, s>>>(
			d_state, m->nrow);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		return SVTGPU_OK;
	}
	if (tiles && strcmp(impl, "tiles") != 0) {   /* default: strips */
		const int64_t M = m->vmax_abs > 0 ? m->vmax_abs : 1;
		const bool nonneg = lac || m->vmin >= 0;
		const bool small_ok = strcmp(impl, "acc32") != 0;
		/* rowVars of small non-negative integers: one packed
		   accumulator, flushed before either half can overflow */
		if (RC == RC_X2 && int_acc && nonneg && small_ok &&
		    M * M * 64 <= 32767) {
			StripConfig sc = choose_strips(m->nrow, m->nleaf,
						       m->nnz, 1, 4);
			if (sc.ok) {
				/* leaves that cannot add 2^15 to a half: the
				   kernel looks at its accumulators that often
				   and only flushes when one got that far */
				const int64_t F = 32767 / (M * M);
				if (lac)
					return launch_strips<RC, int32_t, true,
						uint32_t, true>(m, sc, is_min, F,
								d_state, s);
				return launch_strips<RC, int32_t, false,
					uint32_t, true>(m, sc, is_min, F,
							d_state, s);
			}
		}
		/* row min / max of non-negative integers < 65535: coverage
		   count and extreme share one accumulator */
		if (RC == RC_MINMAX && int_acc && nonneg && small_ok &&
		    M < 65535) {
			StripConfig sc = choose_strips(m->nrow, m->nleaf,
						       m->nnz, 1, 4);
			if (sc.ok) {
				const int64_t F = 65535;
				if (lac)
					return launch_strips<RC, int32_t, true,
						uint32_t, true>(m, sc, is_min, F,
								d_state, s);
				return launch_strips<RC, int32_t, false,
					uint32_t, true>(m, sc, is_min, F,
							d_state, s);
			}
		}
		/* sums of small integers whose int32 accumulators would not
		   fit one SM: int16 accumulators */
		if (RC == RC_SUM && int_acc && small_ok && M * 64 <= 32767) {
			StripConfig s32 = choose_strips(m->nrow, m->nleaf,
							m->nnz, 1, 4);
			StripConfig s16 = choose_strips(m->nrow, m->nleaf,
							m->nnz, 1, 2);
			if (s16.ok && (!s32.ok || s16.ntiles < s32.ntiles)) {
				const int64_t F = 32767 / M;
				if (lac)
					return launch_strips<RC, int32_t, true,
						int16_t, false>(m, s16, is_min, F,
								d_state, s);
				return launch_strips<RC, int32_t, false,
					int16_t, false>(m, s16, is_min, F,
							d_state, s);
			}
		}
		StripConfig sc = choose_strips(m->nrow, m->nleaf, m->nnz, NACC,
					       int_acc ? 4 : 8);
		if (sc.ok) {
			if (lac && int_acc)
				return launch_strips<RC, int32_t, true, int32_t,
					false>(m, sc, is_min, flush_leaves,
					       d_state, s);
			if (lac)
				return launch_strips<RC, int32_t, true, double,
					false>(m, sc, is_min, flush_leaves,
					       d_state, s);
			if (dbl)
				return launch_strips<RC, double, false, double,
					false>(m, sc, is_min, flush_leaves,
					       d_state, s);
			if (int_acc)
				return launch_strips<RC, int32_t, false, int32_t,
					false>(m, sc, is_min, flush_leaves,
					       d_state, s);
			return launch_strips<RC, int32_t, false, double, false>(
				m, sc, is_min, flush_leaves, d_state, s);
		}
	}
	TileConfig c;
	memset(&c, 0, sizeof(c));
	if (tiles) {
		const int vsz = lac ? 0 : (int) svt_val_size(m->val_type);
		c = choose_tiles(m->nrow, m->nleaf, m->nnz, NACC,
				 int_acc ? 4 : 8, vsz);
		tiles = c.ok != 0;
	}
	if (tiles) {
		if (lac && int_acc)
			return launch_tiles<RC, int32_t, true, int32_t>(m, c,
					is_min, flush_leaves, d_state, s);
		if (lac)
			return launch_tiles<RC, int32_t, true, double>(m, c,
					is_min, flush_leaves, d_state, s);
		if (dbl)
			return launch_tiles<RC, double, false, double>(m, c,
					is_min, flush_leaves, d_state, s);
		if (int_acc)
			return launch_tiles<RC, int32_t, false, int32_t>(m, c,
					is_min, flush_leaves, d_state, s);
		return launch_tiles<RC, int32_t, false, double>(m, c, is_min,
					flush_leaves, d_state, s);
	}
	if (lac) return launch_flat<RC, int32_t, true>(m, is_min, d_state, s);
	if (dbl) return launch_flat<RC, double, false>(m, is_min, d_state, s);
	return launch_flat<RC, int32_t, false>(m, is_min, d_state, s);
}

}  /* namespace */

/* max |x| of an integer matrix (one pass, cached in the handle) */
int svtgpu_ensure_absmax(svtgpu_matrix *m, cudaStream_t s)
{
	if (svt_is_double(m->val_type))
		return SVTGPU_OK;
	return ensure_absmax(m, s);
}


/* split points of every leaf at the row boundaries b * strip_rows,
 * b = 1 .. nstrips - 1 (cached in the matrix handle); shared with the
 * strip-tiled products */
int svtgpu_ensure_split(svtgpu_matrix *m, int nstrips, int strip_rows,
			cudaStream_t s, const int32_t **split)
{
	TileConfig tc;
	memset(&tc, 0, sizeof(tc));
	tc.ntiles = nstrips;
	tc.tile_rows = strip_rows;
	return ensure_split(m, tc, s, split);
}

/* Reduce the leaves of `m` into a state of (n_sum + n_ext) x nrow doubles.
 * want_sum2 upgrades SUM to the {sum, sum2} accumulation used by rowVars. */
int svtgpu_launch_row_accumulate(svtgpu_matrix *m, int opcode, int narm,
				 int want_sum2, double *d_state,
				 cudaStream_t s)
{
	(void) narm;   /* NA handling is decided when the state is finalised */
	SVT_ARG(svt_row_op_supported(opcode),
		"rowStats: operation %d is not supported natively (the "
		"reference only implements countNAs, anyNA, min, max, sum and "
		"centered_X2_sum in C_rowStats_SVT)", opcode);
	SVT_ARG((m->flags & SVTGPU_HAS_OFFS) || m->nnz == 0,
		"rowStats: the matrix was uploaded without row offsets");
	int rc_class = row_class_of(opcode);
	if (rc_class == RC_SUM && want_sum2)
		rc_class = RC_X2;
	const int is_min = opcode == SVTGPU_OP_MIN;
	int n_sum = 0, n_ext = 0;
	svt_row_state_layout(rc_class == RC_X2 ? SVTGPU_OP_CENTERED_X2_SUM
					       : opcode, &n_sum, &n_ext);
	const int64_t nrow = m->nrow;
	if (nrow == 0)
		return SVTGPU_OK;
	SVT_CUDA(cudaMemsetAsync(d_state, 0,
				 sizeof(double) * (size_t) (n_sum * nrow), s));
	if (n_ext > 0) {
		/* running min starts at +Inf; running max and the "last
		   leaf" slots of the sums start at -Inf */
		const bool neg = !(rc_class == RC_MINMAX && is_min);
		fill_doubles<<<grid_for((int64_t) n_ext * nrow, 256), 256, 0,
			       s>>>(d_state + (size_t) n_sum * nrow,
				    (int64_t) n_ext * nrow,
				    neg ? svt_neginf() : svt_posinf());
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
	}
	if (m->nnz == 0)
		return SVTGPU_OK;
	const char *impl = svtgpu_env("SVTGPU_ROW_IMPL", "strips");
	if (rc_class == RC_COUNT) {
		/* lacunar leaves hold no NA: nothing to scan */
		if (!(m->flags & SVTGPU_HAS_VALS))
			return SVTGPU_OK;
		if (svt_is_double(m->val_type))
			return launch_flat<RC_COUNT, double, false>(m, 0,
								    d_state, s);
		return launch_flat<RC_COUNT, int32_t, false>(m, 0, d_state, s);
	}
	int rc;
	if (!(m->flags & SVTGPU_HAS_VALS) && rc_class != RC_SUM &&
	    strcmp(svtgpu_env("SVTGPU_ROW_LACUNAR", "count"), "full") != 0) {
		/* every stored value is 1: sum = sum of squares = coverage =
		   the number of stored entries of the row, and the extreme is
		   1 where there is one -- a single counting pass serves all
		   the row statistics of a lacunar matrix */
		SVT_CHECK(launch_class<RC_SUM>(m, impl, 0, d_state, s));
		row_lacunar_derive<<<grid_for(nrow, 256), 256, 0, s>>>(
			d_state, nrow, rc_class == RC_X2);
		SVT_CUDA(cudaGetLastError());
		svtgpu_count_launch(1);
		return SVTGPU_OK;
	}
	switch (rc_class) {
	    case RC_SUM:
		rc = launch_class<RC_SUM>(m, impl, is_min, d_state, s);
		break;
	    case RC_X2:
		rc = launch_class<RC_X2>(m, impl, is_min, d_state, s);
		break;
	    case RC_MINMAX:
		return launch_class<RC_MINMAX>(m, impl, is_min, d_state, s);
	    default:
		svtgpu_set_error("rowStats: internal error (row class)");
		return SVTGPU_ERR_ARG;
	}
	SVT_CHECK(rc);
	/* double sums: order the NA / NaN entries of rows that hold both */
	if (svt_is_double(m->val_type) && (m->flags & SVTGPU_HAS_VALS)) {
		int *d_mixed = NULL;
		SVT_CUDA(svt_malloc_async((void **) &d_mixed, sizeof(int), s));
		cudaError_t e = cudaMemsetAsync(d_mixed, 0, sizeof(int), s);
		if (e == cudaSuccess) {
			row_last_plan<<<grid_for(nrow, 256), 256, 0, s>>>(
				d_state, nrow, (double) m->leaf_base, d_mixed);
			row_last_exact<<<grid_for(m->nnz, 256 * 8), 256, 0, s>>>(
				m->d_offs, (const double *) m->d_vals,
				m->d_leaf_ptr, m->nleaf, m->nnz, nrow,
				m->leaf_base, d_state, d_mixed);
			e = cudaGetLastError();
			svtgpu_count_launch(2);
		}
		svt_free_async(d_mixed, s);
		SVT_CUDA(e);
	}
	return SVTGPU_OK;
}

int svtgpu_launch_row_finalize(int opcode, int val_type, int narm,
			       int64_t nrow, int64_t nstrata,
			       const double *d_center, const double *d_state,
			       void *d_out, int32_t *d_warn, cudaStream_t s)
{
	if (nrow == 0)
		return SVTGPU_OK;
	row_finalize<<<grid_for(nrow, 256), 256, 0, s>>>(opcode,
		svt_is_double(val_type), narm != 0, nrow, nstrata, d_center,
		d_state, d_out, d_warn);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

int svtgpu_launch_row_moments_finalize(int val_type, int narm, int64_t nrow,
				       int64_t nstrata, const double *d_state,
				       double *d_mean, double *d_var,
				       cudaStream_t s)
{
	(void) val_type;
	if (nrow == 0)
		return SVTGPU_OK;
	row_moments_finalize<<<grid_for(nrow, 256), 256, 0, s>>>(narm != 0,
		nrow, nstrata, d_state, d_mean, d_var);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

/* ---- C ABI ---- */

extern "C" int svtgpu_rowstats_state_layout(int opcode, int val_type,
					    int *n_sum_slots,
					    int *n_minmax_slots)
{
	(void) val_type;
	SVT_ARG(svt_row_op_supported(opcode),
		"rowStats: unsupported operation %d", opcode);
	svt_row_state_layout(opcode, n_sum_slots, n_minmax_slots);
	return SVTGPU_OK;
}

extern "C" int svtgpu_rowstats_accumulate_dev(svtgpu_matrix *m, int opcode,
					      int narm, double *d_state,
					      void *stream)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && d_state != NULL,
		"svtgpu_rowstats_accumulate_dev: NULL argument");
	return svtgpu_launch_row_accumulate(m, opcode, narm, 0, d_state,
					    (cudaStream_t) stream);
}

extern "C" int svtgpu_rowstats_finalize_dev(int opcode, int val_type,
		int narm, int64_t nrow, int64_t nstrata_total,
		const double *d_center, const double *d_state, void *d_out,
		int32_t *d_warn, void *stream)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(svt_row_op_supported(opcode),
		"rowStats: unsupported operation %d", opcode);
	return svtgpu_launch_row_finalize(opcode, val_type, narm, nrow,
			nstrata_total, d_center, d_state, d_out, d_warn,
			(cudaStream_t) stream);
}

extern "C" int svtgpu_rowmoments_accumulate_dev(svtgpu_matrix *m, int narm,
						double *d_state, void *stream)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && d_state != NULL,
		"svtgpu_rowmoments_accumulate_dev: NULL argument");
	return svtgpu_launch_row_accumulate(m, SVTGPU_OP_SUM, narm, 1, d_state,
					    (cudaStream_t) stream);
}

extern "C" int svtgpu_rowmoments_finalize_dev(int val_type, int narm,
		int64_t nrow, int64_t nstrata_total, const double *d_state,
		double *d_mean, double *d_var, void *stream)
{
	SVT_CHECK(svtgpu_require_device());
	return svtgpu_launch_row_moments_finalize(val_type, narm, nrow,
			nstrata_total, d_state, d_mean, d_var,
			(cudaStream_t) stream);
}

extern "C" int svtgpu_rowstats(svtgpu_matrix *m, int opcode, int narm,
			       const double *center, void *out, int *warn)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && out != NULL, "svtgpu_rowstats: NULL argument");
	SVT_ARG(svt_row_op_supported(opcode),
		"rowStats: operation %d is not supported natively (the "
		"reference only implements countNAs, anyNA, min, max, sum and "
		"centered_X2_sum in C_rowStats_SVT)", opcode);
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	if (warn != NULL)
		*warn = 0;
	m->tm.kernel_ms = m->tm.d2h_ms = 0.0;
	m->tm.d2h_bytes = 0.0;
	m->tm.launches = 0;
	const int64_t nrow = m->nrow;
	if (nrow == 0)
		return SVTGPU_OK;
	const int out_is_int = opcode == SVTGPU_OP_ANYNA ||
		((opcode == SVTGPU_OP_MIN || opcode == SVTGPU_OP_MAX) &&
		 !svt_is_double(m->val_type));
	const size_t esz = out_is_int ? 4 : 8;
	cudaStream_t s = 0;
	/* state (4 slots) | out | center | warn in one side allocation: the
	   matrix scratch is used by the accumulate step for partials */
	double *d_buf = NULL;
	SVT_CUDA(svt_malloc_async((void **) &d_buf,
				 sizeof(double) * (size_t) (10 * nrow) + 64, s));
	double *d_state = d_buf;                  /* up to 8 slots */
	void *d_out = d_buf + 8 * nrow;
	double *d_center = d_buf + 9 * nrow;
	int32_t *d_warn = (int32_t *) (d_buf + 10 * nrow);
	int rc = SVTGPU_OK;
	const bool use_center = center != NULL &&
				opcode == SVTGPU_OP_CENTERED_X2_SUM;
	cudaError_t e = cudaMemsetAsync(d_warn, 0, 64, s);
	if (!use_center)
		d_center = NULL;
	else if (e == cudaSuccess)
		e = cudaMemcpyAsync(d_center, center, sizeof(double) * nrow,
				    cudaMemcpyHostToDevice, s);
	if (e != cudaSuccess) {
		rc = svtgpu_cuda_fail(e, "svtgpu_rowstats setup", __FILE__,
				      __LINE__);
		svt_free_async(d_buf, s);
		return rc;
	}
	SvtTimer t;
	int64_t l0 = svtgpu_launch_count();
	rc = svt_timer_begin(&t, s);
	if (rc == SVTGPU_OK)
		rc = svtgpu_launch_row_accumulate(m, opcode, narm, 0, d_state,
						  s);
	if (rc == SVTGPU_OK)
		rc = svtgpu_launch_row_finalize(opcode, m->val_type, narm,
				nrow, m->nleaf, d_center, d_state, d_out,
				d_warn, s);
	int rc2 = svt_timer_end(&t, &m->tm.kernel_ms);
	if (rc == SVTGPU_OK)
		rc = rc2;
	m->tm.launches = (int) (svtgpu_launch_count() - l0);
	int32_t h_warn = 0;
	if (rc == SVTGPU_OK) {
		rc = svt_timer_begin(&t, s);
		e = cudaMemcpyAsync(out, d_out, esz * (size_t) nrow,
				    cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess)
			e = cudaMemcpyAsync(&h_warn, d_warn, sizeof(int32_t),
					    cudaMemcpyDeviceToHost, s);
		rc2 = svt_timer_end(&t, &m->tm.d2h_ms);
		if (e != cudaSuccess)
			rc = svtgpu_cuda_fail(e, "svtgpu_rowstats D2H",
					      __FILE__, __LINE__);
		else if (rc == SVTGPU_OK)
			rc = rc2;
		m->tm.d2h_bytes = (double) (esz * (size_t) nrow);
	}
	svt_free_async(d_buf, s);
	if (rc == SVTGPU_OK && warn != NULL)
		*warn = h_warn != 0;
	return rc;
}

extern "C" int svtgpu_rowmoments(svtgpu_matrix *m, int narm, double *out_mean,
				 double *out_var)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL, "svtgpu_rowmoments: NULL matrix");
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	m->tm.kernel_ms = m->tm.d2h_ms = 0.0;
	m->tm.d2h_bytes = 0.0;
	m->tm.launches = 0;
	const int64_t nrow = m->nrow;
	if (nrow == 0)
		return SVTGPU_OK;
	cudaStream_t s = 0;
	double *d_buf = NULL;
	SVT_CUDA(svt_malloc_async((void **) &d_buf,
				 sizeof(double) * (size_t) (10 * nrow), s));
	double *d_state = d_buf, *d_mean = d_buf + 8 * nrow,
	       *d_var = d_buf + 9 * nrow;
	SvtTimer t;
	int64_t l0 = svtgpu_launch_count();
	int rc = svt_timer_begin(&t, s);
	if (rc == SVTGPU_OK)
		rc = svtgpu_launch_row_accumulate(m, SVTGPU_OP_SUM, narm, 1,
						  d_state, s);
	if (rc == SVTGPU_OK)
		rc = svtgpu_launch_row_moments_finalize(m->val_type, narm,
				nrow, m->nleaf, d_state, d_mean, d_var, s);
	int rc2 = svt_timer_end(&t, &m->tm.kernel_ms);
	if (rc == SVTGPU_OK)
		rc = rc2;
	m->tm.launches = (int) (svtgpu_launch_count() - l0);
	if (rc == SVTGPU_OK) {
		rc = svt_timer_begin(&t, s);
		cudaError_t e = cudaSuccess;
		if (out_mean != NULL)
			e = cudaMemcpyAsync(out_mean, d_mean,
					    sizeof(double) * nrow,
					    cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess && out_var != NULL)
			e = cudaMemcpyAsync(out_var, d_var,
					    sizeof(double) * nrow,
					    cudaMemcpyDeviceToHost, s);
		rc2 = svt_timer_end(&t, &m->tm.d2h_ms);
		if (e != cudaSuccess)
			rc = svtgpu_cuda_fail(e, "svtgpu_rowmoments D2H",
					      __FILE__, __LINE__);
		else if (rc == SVTGPU_OK)
			rc = rc2;
		m->tm.d2h_bytes = 8.0 * (double) nrow *
			((out_mean != NULL) + (out_var != NULL));
	}
	svt_free_async(d_buf, s);
	return rc;
}
