/* Device transpose of a device CSC (CSC of x -> CSC of t(x)), cached in the
 * matrix handle.  It stands in for C_transpose_2D_SVT()
 * (src/SparseArray_aperm.c:348-423: count, allocate, fill -- three serial
 * passes over all nonzeros), which the reference runs before every
 * `svt %*% dense` and tcrossprod (R/SparseMatrix-mult.R:165-168,196-198).
 *
 * Stable counting sort by row with the ownership scheme of row_strips
 * (svtgpu_rowstats.cu): the grid is chunks of leaves (balanced by nonzeros) x
 * row tiles, every warp owns a strip of rows, and the nonzeros of a leaf that
 * fall into a strip are one contiguous sub-run with distinct rows.
 *   pass 1  transpose_walk<.., FILL=false>: per (chunk, row) counts in shared
 *           memory -> cnt[chunk][row]
 *   plan    row totals -> exclusive scan = t_ptr; cnt[chunk][row] becomes the
 *           first output position of (chunk, row) relative to its strip
 *   pass 2  transpose_walk<.., FILL=true>: the same walk; a per-row cursor in
 *           shared memory (plain read-modify-write: rows are distinct inside
 *           a sub-run, and only the owning warp touches a row) gives every
 *           nonzero its position; leaves are visited in ascending order, so
 *           the new offsets ascend inside every new leaf.
 * No atomics, deterministic.
 *
 * The fill pass used to store every element straight to HBM: 4- and 8-byte
 * stores into nchunks x nrow output streams whose 32-byte sectors fill up over
 * many leaves -- partially written sectors were evicted from L2 and came back
 * as DRAM read-modify-writes (ncu: 6x write amplification, 150 ms at 2.3e9
 * nonzeros).  Now every row of a strip has an 8-element staging line in shared
 * memory (offsets + values); the lane that completes a line writes it out as
 * whole 32-byte sectors (16-byte vector stores).  Only the first and the last
 * sector of a (chunk, row) stream are partial.
 */
#include "svtgpu_internal.h"
#include "svt_ptx.cuh"

#include <string.h>

namespace {


struct TrParams {
	const int32_t *offs;
	const void *vals;
	const int64_t *leaf_ptr;
	const int32_t *split;
	int64_t nleaf, nnz, nrow;
	int ntiles, nchunks, nstrips, strip_rows;
	int hints;                /* L2 policies: stream the input, keep the
				     partially written output sectors */
	uint32_t *cnt;            /* [nchunks][nrow]: counts, then positions */
	const int64_t *t_ptr;     /* FILL */
	int32_t *t_offs;          /* FILL */
	void *t_vals;             /* FILL */
};

/* TR_U: 32-wide slots of a sub-run held in registers; TR_D: leaves fetched
   ahead per warp (32 % TR_D == 0).  The walk is latency-bound -- few warps,
   sub-runs of a few dozen elements -- so short sub-runs are fetched far ahead */
template <typename T, bool LACUNAR, bool FILL, int TR_U, int TR_D, int LN>
__global__ void __launch_bounds__(512, 1)
transpose_walk(TrParams P)
{
	extern __shared__ __align__(128) unsigned char smem[];
	int lane;
	asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
	const int warp = threadIdx.x >> 5;
	const int W = blockDim.x >> 5;
	const int chunk = blockIdx.x / P.ntiles;
	const int tile = blockIdx.x - chunk * P.ntiles;
	const int gs = tile * W + warp;
	const int64_t row0 = (int64_t) gs * P.strip_rows;
	int rows_here = (int) (P.nrow - row0 < P.strip_rows ? P.nrow - row0
							     : P.strip_rows);
	if (rows_here < 0) rows_here = 0;
	const T *vals = (const T *) P.vals;
	T *t_vals = (T *) P.t_vals;

	/* per warp: cursors [strip_rows]; FILL: first position of the stream
	   [strip_rows], staged offsets [strip_rows][LN], staged values
	   [strip_rows][LN].  LN = elements of a row's staging line: the line
	   leaves for HBM when it is full, as ONE coalesced store of LN * 4 B of
	   offsets and LN * sizeof(T) B of values -- the fill pass is bound by
	   the number of DRAM transactions (random rows), not by bytes. */
	const size_t per_warp = (size_t) P.strip_rows *
		(FILL ? 8 + LN * 4 + (LACUNAR ? 0 : LN * sizeof(T)) : 4);
	unsigned char *wbase = smem + (size_t) warp * per_warp;
	uint32_t *cur = (uint32_t *) wbase;
	uint32_t *first = cur + P.strip_rows;
	int32_t *soff = (int32_t *) (first + P.strip_rows);
	T *sval = (T *) (soff + (size_t) P.strip_rows * LN);
	uint32_t *gcnt = P.cnt + (size_t) chunk * P.nrow + row0;
	for (int r = lane; r < P.strip_rows; r += 32) {
		const uint32_t c0 = FILL && r < rows_here ? gcnt[r] : 0u;
		cur[r] = c0;
		if (FILL)
			first[r] = c0;
	}
	__syncwarp();
	uint32_t *const C0 = cur - row0;
	const int64_t strip_base = FILL && rows_here > 0 ? P.t_ptr[row0] : 0;
	/* element `at` (global position) of local row r is staged in slot
	   at % LN of the row's line.  A line whose last slot has been written
	   is complete unless the stream started inside it (the first line of a
	   (chunk, row) stream begins wherever the previous chunk's stream
	   ended): that one, and the unfinished line at the end, go out element
	   by element. */
	auto flush_partial = [&](int r, int64_t at_last) {
		const int64_t sec = at_last & ~(int64_t) (LN - 1);
		const int64_t lo = strip_base + first[r];
		const int f0 = lo > sec ? (int) (lo - sec) : 0;
		const int f1 = (int) (at_last - sec);          /* inclusive */
		for (int k = f0; k <= f1; k++) {
			P.t_offs[sec + k] = soff[(size_t) r * LN + k];
			if (!LACUNAR)
				t_vals[sec + k] = sval[(size_t) r * LN + k];
		}
	};
	/* the whole warp writes the complete lines of the lanes in `mask`:
	   lanes 0 .. LN/4-1 the offsets, the next LN*sizeof(T)/16 the values,
	   16 bytes each */
	auto flush_full = [&](unsigned mask, int r_mine, int64_t at_mine) {
		constexpr int NO = LN / 4;
		constexpr int NV = LACUNAR ? 0 : (int) (LN * sizeof(T) / 16);
		while (mask) {
			const int src = __ffs(mask) - 1;
			mask &= mask - 1;
			const int r = __shfl_sync(SVT_FULL_MASK, r_mine, src);
			const int64_t at = __shfl_sync(SVT_FULL_MASK, at_mine, src);
			const int64_t sec = at & ~(int64_t) (LN - 1);
			if (NO + NV <= 32) {
				if (lane < NO) {
					((int4 *) (P.t_offs + sec))[lane] =
						((const int4 *) (soff + (size_t) r * LN))[lane];
				} else if (lane < NO + NV) {
					((int4 *) (t_vals + sec))[lane - NO] =
						((const int4 *) (sval + (size_t) r * LN))[lane - NO];
				}
			} else {
				for (int k = lane; k < NO + NV; k += 32) {
					if (k < NO)
						((int4 *) (P.t_offs + sec))[k] =
							((const int4 *) (soff + (size_t) r * LN))[k];
					else
						((int4 *) (t_vals + sec))[k - NO] =
							((const int4 *) (sval + (size_t) r * LN))[k - NO];
				}
			}
		}
	};
	/* stage one element; returns true when its line is now complete */
	auto stage = [&](int r, int64_t at, int32_t leaf_id, T v) -> bool {
		const int slot = (int) (at & (LN - 1));
		soff[(size_t) r * LN + slot] = leaf_id;
		if (!LACUNAR)
			sval[(size_t) r * LN + slot] = v;
		if (slot != LN - 1)
			return false;
		const int64_t sec = at - (LN - 1);
		if (strip_base + (int64_t) first[r] > sec) {   /* stream began inside */
			flush_partial(r, at);
			return false;
		}
		if (LN == 8) {
			/* short lines: the lane writes its own (measured: 122 ms
			   against 185 ms for the warp-cooperative copy, which
			   serialises the ~2.5 complete lines of a slot) */
			const int4 *so = (const int4 *) (soff + (size_t) r * LN);
			int4 *dst = (int4 *) (P.t_offs + sec);
			dst[0] = so[0];
			dst[1] = so[1];
			if (!LACUNAR) {
				const int4 *sv = (const int4 *) (sval + (size_t) r * LN);
				int4 *dv = (int4 *) (t_vals + sec);
#pragma unroll
				for (int k = 0; k < (int) (LN * sizeof(T) / 16); k++)
					dv[k] = sv[k];
			}
			return false;
		}
		return true;
	};

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
	auto subrun = [&](int64_t leaf, int64_t &lo, int &n) {
		lo = 0; n = 0;
		if (leaf < l1) {
			const int64_t start = P.leaf_ptr[leaf];
			const int nz = (int) (P.leaf_ptr[leaf + 1] - start);
			const int a = gs == 0 ? 0
				: P.split[(int64_t) (gs - 1) * P.nleaf + leaf];
			const int b = gs == P.nstrips - 1 ? nz
				: P.split[(int64_t) gs * P.nleaf + leaf];
			lo = start + a;
			n = b - a;
		}
	};

	int32_t boff[TR_D][TR_U];
	T bval[TR_D][TR_U];
	int64_t blo[TR_D];
	int bn[TR_D];
	/* the input is read once: let it leave L2 first; the output sectors are
	   completed one element at a time over many leaves: keep them */
	const bool hints = FILL && (P.hints & 1);
	const uint64_t pol_in = svt_policy_evict_first();
	auto fetch = [&](int d, int64_t lo, int n) {
		blo[d] = lo;
		bn[d] = n;
		const int32_t *po = P.offs + lo + lane;
		const T *pv = vals + lo + lane;
		const int rem = n - lane;
#pragma unroll
		for (int k = 0; k < TR_U; k++) {
			if (k * 32 < rem) {
				if (hints) {
					boff[d][k] = svt_ldg_hint(po + k * 32, pol_in);
					if (!LACUNAR)
						bval[d][k] = svt_ldg_hint(pv + k * 32,
									  pol_in);
				} else {
					boff[d][k] = __ldg(po + k * 32);
					if (FILL && !LACUNAR)
						bval[d][k] = __ldg(pv + k * 32);
				}
			}
		}
	};
	auto apply = [&](int d, int64_t leaf) {
		const int n = bn[d];
		if (n == 0)
			return;
		const int rem = n - lane;
		uint32_t p[TR_U];
#pragma unroll
		for (int k = 0; k < TR_U; k++)
			if (k * 32 < rem)
				p[k] = C0[boff[d][k]];
#pragma unroll
		for (int k = 0; k < TR_U; k++)
			if (k * 32 < rem)
				C0[boff[d][k]] = p[k] + 1u;
		if (FILL) {
#pragma unroll
			for (int k = 0; k < TR_U; k++) {
				/* (warp-uniform: some lane has an element in slot k) */
				if (k * 32 < n) {
					bool full = false;
					int r = 0;
					int64_t at = 0;
					if (k * 32 < rem) {
						at = strip_base + p[k];
						r = boff[d][k] - (int) row0;
						full = stage(r, at, (int32_t) leaf,
							     LACUNAR ? (T) 0 : bval[d][k]);
					}
					__syncwarp();
					const unsigned mask = __ballot_sync(SVT_FULL_MASK, full);
					if (mask)
						flush_full(mask, r, at);
				}
			}
		}
		/* the part of a long sub-run the ring does not hold */
		for (int e0 = TR_U * 32; e0 < n; e0 += 32) {
			const int e = e0 + lane;
			bool full = false;
			int r = 0;
			int64_t at = 0;
			if (e < n) {
				const int off = P.offs[blo[d] + e];
				const uint32_t q = C0[off];
				C0[off] = q + 1u;
				if (FILL) {
					at = strip_base + q;
					r = off - (int) row0;
					full = stage(r, at, (int32_t) leaf,
						     LACUNAR ? (T) 0 : vals[blo[d] + e]);
				}
			}
			if (FILL) {
				__syncwarp();
				const unsigned mask = __ballot_sync(SVT_FULL_MASK, full);
				if (mask)
					flush_full(mask, r, at);
			}
		}
		__syncwarp();
	};

	int64_t cur_lo, nxt_lo;
	int cur_n, nxt_n;
	subrun(l0 + lane, cur_lo, cur_n);
	subrun(l0 + 32 + lane, nxt_lo, nxt_n);
#pragma unroll
	for (int d = 0; d < TR_D; d++) {
		const int64_t lo = __shfl_sync(SVT_FULL_MASK, cur_lo, d);
		const int n = __shfl_sync(SVT_FULL_MASK, cur_n, d);
		fetch(d, lo, n);
	}
	for (int64_t base = l0; base < l1; base += 32) {
		for (int i0 = 0; i0 < 32; i0 += TR_D) {
			if (base + i0 >= l1)
				break;
#pragma unroll
			for (int d = 0; d < TR_D; d++) {
				const int i = i0 + d;
				apply(d, base + i);
				const int j = i + TR_D;
				int64_t lo;
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
	__syncwarp();
	if (!FILL) {
		for (int r = lane; r < rows_here; r += 32)
			gcnt[r] = cur[r];
	} else {
		/* lines that did not reach the end of their sector */
		for (int r = lane; r < rows_here; r += 32) {
			const uint32_t c1 = cur[r];
			if (c1 == first[r])
				continue;                 /* empty stream */
			const int64_t at_last = strip_base + c1 - 1;
			if ((at_last & (LN - 1)) != LN - 1)
				flush_partial(r, at_last);
		}
	}
}

/* ------------------------------------------------------------------------
 * transpose_batch: the same counting sort, element-parallel.
 *
 * transpose_walk gives every warp a strip of rows and lets it walk ALL leaves
 * of its chunk alone: nleaf x nstrips visits of ~20 elements and ~130
 * instructions each, one dependent chain per warp -- 100 ms for the fill at
 * 2.3e9 nonzeros whatever the number of warps, with or without the stores
 * (measured).  Here a CTA = (chunk of leaves, tile of rows) takes its leaves
 * 8 at a time and all 512 threads work on the ~500 elements of such a batch:
 *
 *   phase 1  every element sets bit j (its leaf's place in the batch) in
 *            mask[row]                                  (shared-memory atomic)
 *   phase 2  every element finds its place: cursor[row] + number of lower
 *            bits set in mask[row] -- leaves in ascending order, as the
 *            reference fills its leaves (src/SparseArray_aperm.c:384-392) --
 *            and goes into slot (position % 16) of the row's staging ring
 *   phase 3  one thread per row advances cursor[row] by popc(mask[row]) and,
 *            when that completed a 32-byte sector of offsets (8 elements),
 *            writes the sector (and its 64 bytes of values) to HBM with
 *            16-byte stores.  A row gets at most 8 elements per batch, so a
 *            16-slot ring never wraps onto unsent elements.
 *
 * The loads of a batch are issued three batches ahead.  The counting pass is
 * phase 1 with a counter instead of the mask and no barrier at all.
 */
#define TB_B 8
#define TB_RING 16

template <typename T, bool LACUNAR, bool FILL>
__global__ void __launch_bounds__(512, 1)
transpose_batch(TrParams P)
{
	extern __shared__ __align__(128) unsigned char smem[];
	const int tid = threadIdx.x;
	const int lane = tid & 31;
	const int warp = tid >> 5;
	const int j = warp >> 1;                    /* leaf of the batch */
	const int sl = ((warp & 1) << 5) | lane;    /* place among its 64 lanes */
	const int chunk = blockIdx.x / P.ntiles;
	const int tile = blockIdx.x - chunk * P.ntiles;
	const int R = P.strip_rows;
	const int64_t row0 = (int64_t) tile * R;
	int rows_here = (int) (P.nrow - row0 < R ? P.nrow - row0 : R);
	if (rows_here < 0) rows_here = 0;
	const T *vals = (const T *) P.vals;
	T *t_vals = (T *) P.t_vals;

	uint32_t *cursor = (uint32_t *) smem;
	uint32_t *first = cursor + R;
	uint32_t *mask = first + R;
	int32_t *soff = (int32_t *) (mask + R);
	T *sval = (T *) (soff + (size_t) R * TB_RING);
	uint32_t *gcnt = P.cnt + (size_t) chunk * P.nrow + row0;
	for (int r = tid; r < R; r += blockDim.x) {
		const uint32_t c0 = FILL && r < rows_here ? gcnt[r] : 0u;
		cursor[r] = c0;
		if (FILL) {
			first[r] = c0;
			mask[r] = 0u;
		}
	}
	const int64_t base = FILL && rows_here > 0 ? P.t_ptr[row0] : 0;

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
	__syncthreads();

	/* the part of leaf lf that falls into this tile */
	auto bounds_of = [&](int64_t lf, int64_t &lo, int &n) {
		lo = 0; n = 0;
		if (lf < l1) {
			const int64_t start = __ldg(P.leaf_ptr + lf);
			const int nz = (int) (__ldg(P.leaf_ptr + lf + 1) - start);
			const int a = tile == 0 ? 0
				: __ldg(P.split + (int64_t) (tile - 1) * P.nleaf + lf);
			const int b = tile == P.ntiles - 1 ? nz
				: __ldg(P.split + (int64_t) tile * P.nleaf + lf);
			lo = start + a;
			n = b - a;
		}
	};
	auto load = [&](int64_t lo, int n, int32_t &o, T &v) {
		o = 0;
		v = (T) 0;
		if (sl < n) {
			o = __ldg(P.offs + lo + sl);
			if (FILL && !LACUNAR)
				v = __ldg(vals + lo + sl);
		}
	};
	/* write positions [from, to] (inclusive, global) of local row r */
	auto flush = [&](int r, int64_t from, int64_t to) {
		if (to - from == 7 && (from & 7) == 0) {
			const int ro = (int) (from & (TB_RING - 1));
			const int4 *so = (const int4 *) (soff + (size_t) r * TB_RING + ro);
			int4 *dst = (int4 *) (P.t_offs + from);
			dst[0] = so[0];
			dst[1] = so[1];
			if (!LACUNAR) {
				const int4 *sv = (const int4 *)
					(sval + (size_t) r * TB_RING + ro);
				int4 *dv = (int4 *) (t_vals + from);
#pragma unroll
				for (int k = 0; k < (int) (8 * sizeof(T) / 16); k++)
					dv[k] = sv[k];
			}
		} else {
			for (int64_t at = from; at <= to; at++) {
				const int ro = (int) (at & (TB_RING - 1));
				P.t_offs[at] = soff[(size_t) r * TB_RING + ro];
				if (!LACUNAR)
					t_vals[at] = sval[(size_t) r * TB_RING + ro];
			}
		}
	};

	int64_t lo0, lo1, lo2, lo3;
	int n0, n1, n2, n3;
	int32_t o0, o1, o2;
	T v0, v1, v2;
	bounds_of(l0 + j, lo0, n0);
	bounds_of(l0 + TB_B + j, lo1, n1);
	bounds_of(l0 + 2 * TB_B + j, lo2, n2);
	bounds_of(l0 + 3 * TB_B + j, lo3, n3);
	load(lo0, n0, o0, v0);
	load(lo1, n1, o1, v1);
	load(lo2, n2, o2, v2);
	const uint32_t bit = 1u << j;

	for (int64_t lb = l0; lb < l1; lb += TB_B) {
		const int32_t leaf = (int32_t) (lb + j);
		/* phase 1 */
		if (sl < n0) {
			if (FILL) atomicOr(mask + (o0 - (int) row0), bit);
			else      atomicAdd(cursor + (o0 - (int) row0), 1u);
		}
		for (int e = sl + 64; e < n0; e += 64) {
			const int o = P.offs[lo0 + e];
			if (FILL) atomicOr(mask + (o - (int) row0), bit);
			else      atomicAdd(cursor + (o - (int) row0), 1u);
		}
		if (FILL) {
			__syncthreads();
			/* phase 2 */
			if (sl < n0) {
				const int r = o0 - (int) row0;
				const uint32_t p = cursor[r] +
					(uint32_t) __popc(mask[r] & (bit - 1u));
				const int ro = (int) ((base + p) & (TB_RING - 1));
				soff[(size_t) r * TB_RING + ro] = leaf;
				if (!LACUNAR)
					sval[(size_t) r * TB_RING + ro] = v0;
			}
			for (int e = sl + 64; e < n0; e += 64) {
				const int r = P.offs[lo0 + e] - (int) row0;
				const uint32_t p = cursor[r] +
					(uint32_t) __popc(mask[r] & (bit - 1u));
				const int ro = (int) ((base + p) & (TB_RING - 1));
				soff[(size_t) r * TB_RING + ro] = leaf;
				if (!LACUNAR)
					sval[(size_t) r * TB_RING + ro] = vals[lo0 + e];
			}
			__syncthreads();
			/* phase 3 */
			for (int r = tid; r < rows_here; r += blockDim.x) {
				const uint32_t m = mask[r];
				if (m == 0u)
					continue;
				mask[r] = 0u;
				const uint32_t c0 = cursor[r];
				const uint32_t c1 = c0 + (uint32_t) __popc(m);
				cursor[r] = c1;
				const int64_t at0 = base + c0, at1 = base + c1;
				if ((at1 >> 3) != (at0 >> 3)) {
					/* the sector that holds at0 is complete */
					const int64_t sec = at0 & ~(int64_t) 7;
					const int64_t lo = base + first[r];
					flush(r, lo > sec ? lo : sec, sec + 7);
				}
			}
			__syncthreads();
		}
		lo0 = lo1; n0 = n1; o0 = o1; v0 = v1;
		lo1 = lo2; n1 = n2; o1 = o2; v1 = v2;
		lo2 = lo3; n2 = n3;
		load(lo2, n2, o2, v2);
		bounds_of(lb + 4 * TB_B + j, lo3, n3);
	}
	__syncthreads();
	if (!FILL) {
		for (int r = tid; r < rows_here; r += blockDim.x)
			gcnt[r] = cursor[r];
	} else {
		/* the unfinished last sector of every stream */
		for (int r = tid; r < rows_here; r += blockDim.x) {
			const uint32_t c1 = cursor[r];
			if (c1 == first[r])
				continue;
			const int64_t at1 = base + c1;
			if ((at1 & 7) == 0)
				continue;
			const int64_t sec = at1 & ~(int64_t) 7;
			const int64_t lo = base + first[r];
			flush(r, lo > sec ? lo : sec, at1 - 1);
		}
	}
}

/* ------------------------------------------------------------------------
 * transpose_blocks: the fill pass as a sequence of in-shared-memory sorts.
 *
 * A CTA = (chunk of leaves, tile of R rows) takes its leaves in batches of up
 * to 32 * MW (their elements inside the tile must fit the staging area) and
 * sorts each batch by (row, leaf) in shared memory:
 *
 *   P0  bounds of the next 32 * MW leaves inside the tile, their running
 *       total, and how many of them fit the staging area
 *   P1  every element sets bit j (its leaf's place in the batch) of
 *       mask[row] -- MW words per row                (shared-memory atomics)
 *   P2  rowstart = exclusive scan of popc(mask[row]) over the rows
 *   P3  every element goes to staging[rowstart[row] + number of lower bits
 *       set in mask[row]]: rows in order, leaves in order inside a row, as
 *       the reference fills its leaves (src/SparseArray_aperm.c:384-392)
 *   P4  one thread per staged element writes it behind what earlier batches
 *       wrote to its row (runs of ~13-18 contiguous elements), then the
 *       rows' cursors advance and their masks are cleared
 *
 * ~12,000 elements per batch and 5 barriers: every thread handles ~25
 * elements per phase, against ~1 in transpose_batch (whose per-batch fixed
 * cost of ~260 warp instructions made it no faster than the serial walk:
 * 89 ms vs 100 ms for the fill at 2.3e9 nonzeros, measured).
 */
#define TBK_THREADS 1024

template <typename T, bool LACUNAR, int MW>
__global__ void __launch_bounds__(TBK_THREADS, 1)
transpose_blocks(TrParams P, int cap)
{
	constexpr int LB = 32 * MW;
	constexpr int LPW = LB / (TBK_THREADS / 32) < 4 ? 4
			  : LB / (TBK_THREADS / 32);   /* leaves per warp */
	extern __shared__ __align__(128) unsigned char smem[];
	const int tid = threadIdx.x;
	const int lane = tid & 31;
	const int warp = tid >> 5;
	constexpr int W = TBK_THREADS / 32;
	const int chunk = blockIdx.x / P.ntiles;
	const int tile = blockIdx.x - chunk * P.ntiles;
	const int R = P.strip_rows;
	const int64_t row0 = (int64_t) tile * R;
	int rows_here = (int) (P.nrow - row0 < R ? P.nrow - row0 : R);
	if (rows_here < 0) rows_here = 0;
	const T *vals = (const T *) P.vals;
	T *t_vals = (T *) P.t_vals;

	uint32_t *cursor = (uint32_t *) smem;                /* [R] */
	uint32_t *rowstart = cursor + R;                     /* [R + 8] */
	uint32_t *mask = rowstart + R + 8;                   /* [R][MW] */
	int64_t *blo = (int64_t *) (mask + (size_t) R * MW); /* [LB] */
	int *bn = (int *) (blo + LB);                        /* [LB] */
	uint32_t *wsum = (uint32_t *) (bn + LB);             /* [32] */
	uint16_t *pos16 = (uint16_t *) (wsum + 32);          /* [R][MW] */
	int32_t *soff = (int32_t *) (pos16 + (size_t) R * MW); /* [cap] */
	T *sval = (T *) (soff + cap);                        /* [cap] */
	const uint32_t *gcnt = P.cnt + (size_t) chunk * P.nrow + row0;
	for (int r = tid; r < R; r += TBK_THREADS) {
		cursor[r] = r < rows_here ? gcnt[r] : 0u;
#pragma unroll
		for (int w = 0; w < MW; w++)
			mask[(size_t) r * MW + w] = 0u;
	}
	const int64_t base = rows_here > 0 ? P.t_ptr[row0] : 0;

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
	__syncthreads();

	int64_t lb = l0;
	while (lb < l1) {
		/* ---- P0: the batch ---- */
		int64_t lo = 0;
		int n = 0;
		if (tid < LB && lb + tid < l1) {
			const int64_t lf = lb + tid;
			const int64_t start = __ldg(P.leaf_ptr + lf);
			const int nz = (int) (__ldg(P.leaf_ptr + lf + 1) - start);
			const int a = tile == 0 ? 0
				: __ldg(P.split + (int64_t) (tile - 1) * P.nleaf + lf);
			const int b = tile == P.ntiles - 1 ? nz
				: __ldg(P.split + (int64_t) tile * P.nleaf + lf);
			lo = start + a;
			n = b - a;
		}
		/* inclusive scan of n over the block's first LB threads */
		int cum = n;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const int t = __shfl_up_sync(SVT_FULL_MASK, cum, d);
			if (lane >= d) cum += t;
		}
		if (lane == 31)
			wsum[warp] = (uint32_t) cum;
		__syncthreads();
		{
			int add = 0;
			for (int w = 0; w < warp; w++)
				add += (int) wsum[w];
			cum += add;
		}
		int nb = __syncthreads_count(tid < LB && lb + tid < l1 &&
					     cum <= cap);
		if (nb < 1) nb = 1;          /* (a leaf never exceeds cap >= R) */
		if (tid < LB) {
			blo[tid] = lo;
			bn[tid] = n;
		}
		__syncthreads();

		/* ---- P1: mask bits ----
		   All of the warp's loads of the batch are issued before the
		   first atomic (leaf by leaf, every leaf cost one round trip
		   to HBM with 16 warps to hide it: ncu, 46 % of the stall
		   samples on the first use of the offset).  The offsets of the
		   first 64 entries of each part stay in registers for P3. */
		int32_t ro[LPW][2];
#pragma unroll
		for (int u = 0; u < LPW; u++) {
			const int jj = warp + u * W;
			ro[u][0] = ro[u][1] = -1;
			if (jj < nb) {
				const int64_t jlo = blo[jj];
				const int jn = bn[jj];
				if (lane < jn)
					ro[u][0] = __ldg(P.offs + jlo + lane);
				if (lane + 32 < jn)
					ro[u][1] = __ldg(P.offs + jlo + lane + 32);
			}
		}
#pragma unroll
		for (int u = 0; u < LPW; u++) {
			const int jj = warp + u * W;
			if (jj >= nb)
				break;
			const uint32_t bit = 1u << (jj & 31);
#pragma unroll
			for (int k = 0; k < 2; k++) {
				if (ro[u][k] >= 0) {
					ro[u][k] -= (int) row0;
					atomicOr(mask + (size_t) ro[u][k] * MW +
						 (jj >> 5), bit);
				}
			}
			const int jn = bn[jj];
			if (jn > 64) {
				const int64_t jlo = blo[jj];
				for (int e = lane + 64; e < jn; e += 32) {
					const int r = __ldg(P.offs + jlo + e) -
						      (int) row0;
					atomicOr(mask + (size_t) r * MW +
						 (jj >> 5), bit);
				}
			}
		}
		__syncthreads();

		/* ---- P2: rowstart = exclusive scan of the rows' counts ---- */
		{
			/* two rows per thread (R <= 2 * TBK_THREADS) */
			const int r0 = 2 * tid, r1 = 2 * tid + 1;
			int c0 = 0, c1 = 0;
			if (r0 < R) {
#pragma unroll
				for (int w = 0; w < MW; w++)
					c0 += __popc(mask[(size_t) r0 * MW + w]);
			}
			if (r1 < R) {
#pragma unroll
				for (int w = 0; w < MW; w++)
					c1 += __popc(mask[(size_t) r1 * MW + w]);
			}
			int incl = c0 + c1;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				const int t = __shfl_up_sync(SVT_FULL_MASK, incl, d);
				if (lane >= d) incl += t;
			}
			if (lane == 31)
				wsum[warp] = (uint32_t) incl;
			__syncthreads();
			int add = 0;
			for (int w = 0; w < warp; w++)
				add += (int) wsum[w];
			const int excl = incl + add - (c0 + c1);
			if (r0 < R) rowstart[r0] = (uint32_t) excl;
			if (r1 < R) rowstart[r1] = (uint32_t) (excl + c0);
			if (r1 == R - 1 || r0 == R - 1)
				rowstart[R] = (uint32_t) (excl + c0 + c1);
			/* first staging slot of (row, mask word): P3 then needs
			   one mask word and one of these per element */
			if (r0 < R) {
				int at = excl;
#pragma unroll
				for (int w = 0; w < MW; w++) {
					pos16[(size_t) r0 * MW + w] = (uint16_t) at;
					at += __popc(mask[(size_t) r0 * MW + w]);
				}
			}
			if (r1 < R) {
				int at = excl + c0;
#pragma unroll
				for (int w = 0; w < MW; w++) {
					pos16[(size_t) r1 * MW + w] = (uint16_t) at;
					at += __popc(mask[(size_t) r1 * MW + w]);
				}
			}
		}
		__syncthreads();

		/* ---- P3: scatter into the staging area (values: four leaves'
		   loads in flight per lane) ---- */
		auto place = [&](int jj, int r, T v) {
			const int wj = jj >> 5;
			const uint32_t below = (1u << (jj & 31)) - 1u;
			const uint32_t slot = (uint32_t) pos16[(size_t) r * MW + wj] +
				(uint32_t) __popc(mask[(size_t) r * MW + wj] & below);
			/* (row, place of the leaf in the batch): P4 finds the
			   element's row without a search */
			soff[slot] = (int32_t) (((uint32_t) r << 8) | (uint32_t) jj);
			if (!LACUNAR)
				sval[slot] = v;
		};
#pragma unroll
		for (int u0 = 0; u0 < LPW; u0 += 4) {
			T v[4][2];
#pragma unroll
			for (int u = 0; u < 4; u++) {
				const int jj = warp + (u0 + u) * W;
				v[u][0] = v[u][1] = (T) 0;
				if (!LACUNAR && jj < nb) {
					const int64_t jlo = blo[jj];
					if (ro[u0 + u][0] >= 0)
						v[u][0] = __ldg(vals + jlo + lane);
					if (ro[u0 + u][1] >= 0)
						v[u][1] = __ldg(vals + jlo + lane + 32);
				}
			}
#pragma unroll
			for (int u = 0; u < 4; u++) {
				const int jj = warp + (u0 + u) * W;
				if (jj >= nb)
					break;
#pragma unroll
				for (int k = 0; k < 2; k++)
					if (ro[u0 + u][k] >= 0)
						place(jj, ro[u0 + u][k], v[u][k]);
				const int jn = bn[jj];
				if (jn > 64) {
					const int64_t jlo = blo[jj];
					for (int e = lane + 64; e < jn; e += 32)
						place(jj, __ldg(P.offs + jlo + e) -
							  (int) row0,
						      LACUNAR ? (T) 0
							: __ldg(vals + jlo + e));
				}
			}
		}
		__syncthreads();

		/* ---- P4: the sorted batch goes out, one element per thread:
		   consecutive slots of a row are consecutive positions of its
		   stream (the per-row loop this replaces spent 44 % of the
		   kernel's instructions on ~18-element runs: ncu) ---- */
		{
			const uint32_t total = rowstart[R];
			for (uint32_t k = tid; k < total; k += TBK_THREADS) {
				const uint32_t pk = (uint32_t) soff[k];
				const uint32_t r = pk >> 8;
				const int64_t dst = base + cursor[r] +
						    (k - rowstart[r]);
				P.t_offs[dst] = (int32_t) (lb + (pk & 255u));
				if (!LACUNAR)
					t_vals[dst] = sval[k];
			}
		}
		__syncthreads();
		for (int r = tid; r < rows_here; r += TBK_THREADS) {
			const uint32_t n = rowstart[r + 1] - rowstart[r];
			if (n != 0u) {
				cursor[r] += n;
#pragma unroll
				for (int w = 0; w < MW; w++)
					mask[(size_t) r * MW + w] = 0u;
			}
		}
		__syncthreads();
		lb += nb;
	}
}

/* row totals over the chunks */
__global__ void __launch_bounds__(256)
transpose_row_totals(const uint32_t *__restrict__ cnt, int nchunks,
		     int64_t nrow, int64_t *__restrict__ total)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     r < nrow; r += stride) {
		int64_t t = 0;
		for (int c = 0; c < nchunks; c++)
			t += cnt[(size_t) c * nrow + r];
		total[r] = t;
	}
}

/* cnt[c][r] := first position of (chunk c, row r) relative to the first
 * position of the strip that owns row r; *overflow is set when a strip holds
 * 2^32 nonzeros or more */
__global__ void __launch_bounds__(256)
transpose_positions(uint32_t *__restrict__ cnt, int nchunks, int64_t nrow,
		    int strip_rows, const int64_t *__restrict__ t_ptr,
		    int *overflow)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t r = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     r < nrow; r += stride) {
		const int64_t s0 = r / strip_rows * strip_rows;
		int64_t pos = t_ptr[r] - t_ptr[s0];
		for (int c = 0; c < nchunks; c++) {
			const uint32_t n = cnt[(size_t) c * nrow + r];
			cnt[(size_t) c * nrow + r] = (uint32_t) pos;
			pos += n;
		}
		if (pos > (int64_t) UINT32_MAX)
			*overflow = 1;
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

struct TrConfig {
	int ok, ntiles, nchunks, nstrips, strip_rows, warps, slots;
	int line;            /* elements of a row's staging line: 8, 16 or 32 */
	size_t smem;
};

/* Rows per CTA are bounded by the staging lines (8 + 32 + 8 * sizeof(value)
 * bytes of shared memory per row); a CTA's rows are cut into one strip per
 * warp; chunks of leaves fill the remaining SMs. */
TrConfig choose(const svtgpu_matrix *m)
{
	TrConfig c;
	memset(&c, 0, sizeof(c));
	const size_t budget = (size_t) 227 * 1024 - 1024 - 256;
	const int sms = svtgpu_sm_count();
	const bool lac = !(m->flags & SVTGPU_HAS_VALS);
	c.line = atoi(svtgpu_env("SVTGPU_TR_LINE", "8"));
	if (c.line != 8 && c.line != 16 && c.line != 32)
		c.line = 8;
	const size_t bpr = 8 + (size_t) c.line *
		(4 + (lac ? 0 : svt_val_size(m->val_type)));
	const double avg_leaf = m->nleaf > 0
		? (double) m->nnz / (double) m->nleaf : 0.0;
	const double density = m->nrow > 0 ? avg_leaf / (double) m->nrow : 0.0;
	int W = atoi(svtgpu_env("SVTGPU_TR_WARPS", "8"));
	if (W < 1 || W > 16) W = 8;
	int64_t max_rows = (int64_t) (budget / bpr);          /* per CTA */
	int64_t nt = (m->nrow + max_rows - 1) / max_rows;
	const int force_t = atoi(svtgpu_env("SVTGPU_TR_NTILES", "0"));
	if (force_t > 0 && force_t > nt) nt = force_t;
	if (nt < 1) nt = 1;
	/* strips shorter than ~24 expected nonzeros waste lanes: fewer warps */
	for (;;) {
		int64_t sr = (m->nrow + nt * W - 1) / (nt * W);
		if (W > 2 && density * (double) sr < 24.0 &&
		    atoi(svtgpu_env("SVTGPU_TR_WARPS", "0")) == 0) {
			W--;
			continue;
		}
		sr = (sr + 7) / 8 * 8;
		if ((size_t) sr * W * bpr > budget) {     /* rounding overflowed */
			nt++;
			continue;
		}
		c.strip_rows = (int) sr;
		break;
	}
	if (nt > INT32_MAX / 16)
		return c;
	c.ntiles = (int) nt;
	c.warps = W;
	c.nstrips = c.ntiles * W;
	c.smem = (size_t) c.strip_rows * W * bpr + 128;
	const double L = density * (double) c.strip_rows;
	const double need = (L + 3.0 * sqrt(L > 0 ? L : 0.0)) / 32.0;
	c.slots = need <= 1.0 ? 1 : need <= 2.0 ? 2 : need <= 3.0 ? 3 : 6;
	const int force_u = atoi(svtgpu_env("SVTGPU_TR_SLOTS", "0"));
	if (force_u == 1 || force_u == 2 || force_u == 3 || force_u == 6)
		c.slots = force_u;
	c.nchunks = sms / c.ntiles;
	if (c.nchunks < 1) c.nchunks = 1;
	if ((int64_t) c.nchunks > m->nleaf)
		c.nchunks = m->nleaf > 0 ? (int) m->nleaf : 1;
	c.ok = 1;
	return c;
}

/* transpose_batch: rows per CTA bounded by cursor + first + mask + the
 * 16-slot staging ring; as many tiles as needed, then as many chunks of
 * leaves as keep every SM busy (tiles x chunks close to a multiple of the SM
 * count). */
TrConfig choose_batch(const svtgpu_matrix *m)
{
	TrConfig c;
	memset(&c, 0, sizeof(c));
	const size_t budget = (size_t) 227 * 1024 - 1024;
	const int sms = svtgpu_sm_count();
	const bool lac = !(m->flags & SVTGPU_HAS_VALS);
	const size_t bpr = 12 + (size_t) TB_RING *
		(4 + (lac ? 0 : svt_val_size(m->val_type)));
	const int64_t max_rows = (int64_t) (budget / bpr) / 8 * 8;
	int64_t nt = (m->nrow + max_rows - 1) / max_rows;
	if (nt < 1) nt = 1;
	if (nt < sms) {
		/* a few more tiles can fill the last wave: maximise
		   floor(sms / tiles) * tiles */
		int64_t best = nt, best_cov = (sms / nt) * nt;
		for (int64_t t = nt + 1; t <= 2 * nt && t <= sms; t++) {
			const int64_t cov = (sms / t) * t;
			if (cov > best_cov) { best = t; best_cov = cov; }
		}
		nt = best;
	}
	const int force_t = atoi(svtgpu_env("SVTGPU_TR_NTILES", "0"));
	if (force_t > nt) nt = force_t;
	if (nt > INT32_MAX / 16)
		return c;
	int64_t R = (m->nrow + nt - 1) / nt;
	R = (R + 7) / 8 * 8;
	c.ntiles = (int) nt;
	c.nstrips = (int) nt;
	c.strip_rows = (int) R;
	c.warps = 16;
	c.smem = (size_t) R * bpr + 128;
	c.nchunks = (int) (nt < sms ? sms / nt : 1);
	if ((int64_t) c.nchunks > m->nleaf)
		c.nchunks = m->nleaf > 0 ? (int) m->nleaf : 1;
	c.ok = 1;
	return c;
}

/* transpose_blocks: R rows per CTA (<= 1024: two per thread in the scan),
 * MW mask words per row, and whatever is left of shared memory as staging for
 * the sorted batch; chosen so that 32 * MW leaves of average length roughly
 * fill the staging area. */
struct TbkConfig {
	int ok, MW, cap;
	TrConfig t;
};

TbkConfig choose_blocks(const svtgpu_matrix *m)
{
	TbkConfig k;
	memset(&k, 0, sizeof(k));
	const size_t budget = (size_t) 227 * 1024 - 1024;
	const int sms = svtgpu_sm_count();
	const bool lac = !(m->flags & SVTGPU_HAS_VALS);
	const size_t esz = 4 + (lac ? 0 : svt_val_size(m->val_type));
	const double density = m->nrow > 0 && m->nleaf > 0
		? (double) m->nnz / ((double) m->nrow * (double) m->nleaf) : 0.0;
	/* tiles: at most 1024 rows, and a few more tiles when that fills the
	   last wave (floor(sms / tiles) * tiles as large as possible) */
	int64_t nt = (m->nrow + 1023) / 1024;
	if (nt < 1) nt = 1;
	if (nt < sms) {
		int64_t best = nt, best_cov = (sms / nt) * nt;
		for (int64_t t = nt + 1; t <= 2 * nt + 8 && t <= sms; t++) {
			const int64_t cov = (sms / t) * t;
			if (cov > best_cov) { best = t; best_cov = cov; }
		}
		nt = best;
	}
	const int force_t = atoi(svtgpu_env("SVTGPU_TR_NTILES", "0"));
	if (force_t > nt) nt = force_t;
	if (nt > INT32_MAX / 16)
		return k;
	int64_t R = (m->nrow + nt - 1) / nt;
	R = (R + 7) / 8 * 8;
	if (R > 1024)
		return k;
	for (int MW = 8; MW >= 1; MW >>= 1) {
		const size_t fixed = (size_t) R * 4 + (size_t) (R + 8) * 4 +
			(size_t) R * MW * 4 + (size_t) 32 * MW * 12 + 128 + 256 +
			(size_t) R * MW * 2;
		if (fixed + (size_t) R * esz > budget)
			continue;
		int64_t cap = (int64_t) ((budget - fixed) / esz) / 8 * 8;
		if (cap > 65528) cap = 65528;   /* 16-bit staging positions */
		/* fewer mask words when the leaves of a batch would not fill
		   the staging area anyway */
		if (MW > 1 && density * (double) R * 32.0 * (MW / 2) >=
		    (double) cap)
			continue;
		k.MW = MW;
		k.cap = (int) cap;
		k.t.smem = fixed + (size_t) cap * esz;
		break;
	}
	if (k.MW == 0)
		return k;
	k.t.ntiles = (int) nt;
	k.t.nstrips = (int) nt;
	k.t.strip_rows = (int) R;
	k.t.warps = 16;
	k.t.nchunks = (int) (nt < sms ? sms / nt : 1);
	if ((int64_t) k.t.nchunks > m->nleaf)
		k.t.nchunks = m->nleaf > 0 ? (int) m->nleaf : 1;
	k.t.ok = k.ok = 1;
	return k;
}

template <typename T, bool LAC>
int launch_blocks(const TbkConfig &k, const TrParams &P, cudaStream_t s)
{
#define TBK_LAUNCH(MWV) do { \
		SVT_CUDA(cudaFuncSetAttribute(transpose_blocks<T, LAC, MWV>, \
			cudaFuncAttributeMaxDynamicSharedMemorySize, \
			(int) k.t.smem)); \
		transpose_blocks<T, LAC, MWV><<<(unsigned) (k.t.nchunks * \
			k.t.ntiles), TBK_THREADS, k.t.smem, s>>>(P, k.cap); \
	} while (0)
	if (k.MW == 8)      TBK_LAUNCH(8);
	else if (k.MW == 4) TBK_LAUNCH(4);
	else if (k.MW == 2) TBK_LAUNCH(2);
	else                TBK_LAUNCH(1);
#undef TBK_LAUNCH
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

/* per (chunk, row) counts: every nonzero of the (chunk, tile) bumps its row's
   counter in shared memory (order does not matter for counting) */
/* The counting pass as a shared-memory histogram: how many entries of every
 * row fall into each chunk of leaves does not depend on where a leaf starts
 * or on the row tiles of the fill, so a CTA streams one contiguous piece of
 * its chunk's offsets (16-byte loads; no leaf_ptr, no split tables) into one
 * int32 cell per row and adds its cells to cnt[chunk][row] at the end.  A row
 * has at most one entry per leaf: no cell can overflow.  (The warp-per-leaf
 * form below waited on four dependent loads per 64-entry part of a leaf:
 * 8.5 ms per 2.3e9 entries.) */
__global__ void __launch_bounds__(1024, 1)
transpose_count_flat(TrParams P, int per_chunk)
{
	extern __shared__ __align__(128) unsigned char smem[];
	uint32_t *cell = (uint32_t *) smem;
	const uint32_t cell_s = (uint32_t) __cvta_generic_to_shared(cell);
	const int chunk = blockIdx.x / per_chunk;
	const int part = blockIdx.x - chunk * per_chunk;
	for (int64_t r = threadIdx.x; r < P.nrow; r += blockDim.x)
		cell[r] = 0u;
	/* entries [e0, e1) of the chunk (same leaf bounds as the fill) */
	int64_t e0, e1;
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
		const int64_t c0 = P.leaf_ptr[bounds[0]], c1 = P.leaf_ptr[bounds[1]];
		const int64_t n = c1 - c0;
		/* pieces of whole 16-byte vectors (relative to the array) */
		e0 = c0 + (n * part / per_chunk);
		e1 = c0 + (n * (part + 1) / per_chunk);
		if (part > 0) e0 = (e0 + 3) & ~(int64_t) 3;
		if (part + 1 < per_chunk) e1 = (e1 + 3) & ~(int64_t) 3;
		if (e0 < c0) e0 = c0;
		if (e1 > c1) e1 = c1;
		if (e0 > e1) e0 = e1;
	}
	__syncthreads();
	auto bump = [&](int o) {
		asm volatile("red.shared.add.u32 [%0], %1;"
			     :: "r"(cell_s + ((uint32_t) o << 2)), "r"(1u) : "memory");
	};
	int64_t head = (4 - (e0 & 3)) & 3;
	if (head > e1 - e0) head = e1 - e0;
	if ((int64_t) threadIdx.x < head)
		bump(P.offs[e0 + threadIdx.x]);
	const int64_t v0 = e0 + head;
	const int64_t nvec = (e1 - v0) >> 2;
	const int4 *q = (const int4 *) (P.offs + v0);
	for (int64_t i = threadIdx.x; i < nvec; i += 4 * 1024) {
		int4 v[4];
#pragma unroll
		for (int k = 0; k < 4; k++)
			if (i + k * 1024 < nvec)
				v[k] = q[i + k * 1024];
#pragma unroll
		for (int k = 0; k < 4; k++) {
			if (i + k * 1024 < nvec) {
				bump(v[k].x); bump(v[k].y);
				bump(v[k].z); bump(v[k].w);
			}
		}
	}
	const int64_t t0 = v0 + 4 * nvec;
	if (t0 + threadIdx.x < e1)
		bump(P.offs[t0 + threadIdx.x]);
	__syncthreads();
	uint32_t *gcnt = P.cnt + (size_t) chunk * P.nrow;
	for (int64_t r = threadIdx.x; r < P.nrow; r += blockDim.x)
		if (cell[r] != 0u)
			atomicAdd(gcnt + r, cell[r]);
}

__global__ void __launch_bounds__(1024, 1)
transpose_count(TrParams P)
{
	extern __shared__ __align__(128) unsigned char smem[];
	uint32_t *cnt = (uint32_t *) smem;
	const int chunk = blockIdx.x / P.ntiles;
	const int tile = blockIdx.x - chunk * P.ntiles;
	const int R = P.strip_rows;
	const int64_t row0 = (int64_t) tile * R;
	int rows_here = (int) (P.nrow - row0 < R ? P.nrow - row0 : R);
	if (rows_here < 0) rows_here = 0;
	for (int r = threadIdx.x; r < R; r += blockDim.x)
		cnt[r] = 0u;
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
	__syncthreads();
	/* a warp per leaf, lanes over the part of the leaf inside the tile */
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int W = blockDim.x >> 5;
	for (int64_t lf = l0 + warp; lf < l1; lf += W) {
		const int64_t start = __ldg(P.leaf_ptr + lf);
		const int nz = (int) (__ldg(P.leaf_ptr + lf + 1) - start);
		const int a = tile == 0 ? 0
			: __ldg(P.split + (int64_t) (tile - 1) * P.nleaf + lf);
		const int b = tile == P.ntiles - 1 ? nz
			: __ldg(P.split + (int64_t) tile * P.nleaf + lf);
		for (int e = a + lane; e < b; e += 32)
			atomicAdd(cnt + (__ldg(P.offs + start + e) - (int) row0), 1u);
	}
	__syncthreads();
	uint32_t *gcnt = P.cnt + (size_t) chunk * P.nrow + row0;
	for (int r = threadIdx.x; r < rows_here; r += blockDim.x)
		gcnt[r] = cnt[r];
}

template <typename T, bool LAC, bool FILL>
int launch_batch(const TrConfig &c, const TrParams &P, cudaStream_t s)
{
	SVT_CUDA(cudaFuncSetAttribute(transpose_batch<T, LAC, FILL>,
		cudaFuncAttributeMaxDynamicSharedMemorySize, (int) c.smem));
	transpose_batch<T, LAC, FILL><<<(unsigned) (c.nchunks * c.ntiles), 512,
		c.smem, s>>>(P);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

template <typename T, bool LAC, bool FILL>
int launch_walk(const TrConfig &c, const TrParams &P, cudaStream_t s)
{
#define TR_LAUNCH2(U, D, LNV) do { \
		SVT_CUDA(cudaFuncSetAttribute( \
			transpose_walk<T, LAC, FILL, U, D, LNV>, \
			cudaFuncAttributeMaxDynamicSharedMemorySize, \
			(int) c.smem)); \
		transpose_walk<T, LAC, FILL, U, D, LNV><<<(unsigned) (c.nchunks * \
			c.ntiles), c.warps * 32, c.smem, s>>>(P); \
	} while (0)
#define TR_LAUNCH(U, D) do { \
		if (!FILL || c.line == 8) TR_LAUNCH2(U, D, 8); \
		else if (c.line == 16)    TR_LAUNCH2(U, D, 16); \
		else                      TR_LAUNCH2(U, D, 32); \
	} while (0)
	if (c.slots == 1)      TR_LAUNCH(1, 8);
	else if (c.slots == 2) TR_LAUNCH(2, 8);
	else if (c.slots == 3) TR_LAUNCH(3, 8);
	else                   TR_LAUNCH(6, 4);
#undef TR_LAUNCH2
#undef TR_LAUNCH
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	return SVTGPU_OK;
}

}  /* namespace */

/* t(m) as a device CSC owned by (and cached in) m; NULL + SVTGPU_OK when the
 * transpose cannot be built this way (the caller falls back) */
int svtgpu_ensure_transpose(svtgpu_matrix *m, cudaStream_t s,
			    svtgpu_matrix **out)
{
	*out = NULL;
	if (m->transposed != NULL) {
		*out = m->transposed;
		return SVTGPU_OK;
	}
	if (m->transpose_failed || !(m->flags & SVTGPU_HAS_OFFS) ||
	    m->nnz == 0 || m->nrow == 0 || m->nleaf > INT32_MAX)
		return SVTGPU_OK;
	const char *impl = svtgpu_env("SVTGPU_TR_IMPL", "blocks");
	TbkConfig kb;
	memset(&kb, 0, sizeof(kb));
	if (strcmp(impl, "blocks") == 0)
		kb = choose_blocks(m);
	const bool blocks = kb.ok != 0;
	const bool batch = !blocks && strcmp(impl, "walk") != 0;
	const TrConfig c = blocks ? kb.t : batch ? choose_batch(m) : choose(m);
	if (!c.ok)
		return SVTGPU_OK;
	const bool lac = !(m->flags & SVTGPU_HAS_VALS);
	const bool dbl = svt_is_double(m->val_type);
	const int32_t *split = NULL;
	SVT_CHECK(svtgpu_ensure_split(m, c.nstrips, c.strip_rows, s, &split));

	uint32_t *cnt = NULL;
	int64_t *total = NULL, *t_ptr = NULL;
	int32_t *t_offs = NULL;
	void *t_vals = NULL;
	int *d_over = NULL, h_over = 0;
	const size_t vs = svt_val_size(m->val_type);
	cudaError_t e = svt_malloc_async((void **) &cnt,
			4 * (size_t) c.nchunks * (size_t) m->nrow + 64, s);
	if (e == cudaSuccess)
		e = svt_malloc_async((void **) &total, 8 * (size_t) m->nrow + 64, s);
	if (e == cudaSuccess)
		e = svt_malloc_async((void **) &t_ptr,
				    8 * (size_t) (m->nrow + 1), s);
	if (e == cudaSuccess)
		e = svt_malloc_async((void **) &t_offs,
				    4 * ((size_t) m->nnz + 64), s);
	if (e == cudaSuccess && !lac)
		e = svt_malloc_async(&t_vals, vs * ((size_t) m->nnz + 64), s);
	if (e == cudaSuccess)
		e = svt_malloc_async((void **) &d_over, sizeof(int), s);
	if (e == cudaSuccess)
		e = cudaMemsetAsync(d_over, 0, sizeof(int), s);
	if (e == cudaSuccess)
		e = cudaMemsetAsync(t_offs + m->nnz, 0, 4 * 64, s);
	if (e == cudaSuccess && !lac)
		e = cudaMemsetAsync((char *) t_vals + vs * (size_t) m->nnz, 0,
				    vs * 64, s);
	int rc = SVTGPU_OK;
	if (e != cudaSuccess)
		rc = svtgpu_cuda_fail(e, "transpose alloc", __FILE__, __LINE__);

	TrParams P;
	memset(&P, 0, sizeof(P));
	P.offs = m->d_offs;
	P.vals = lac ? NULL : m->d_vals;
	P.leaf_ptr = m->d_leaf_ptr;
	P.split = split;
	P.nleaf = m->nleaf;
	P.nnz = m->nnz;
	P.nrow = m->nrow;
	P.ntiles = c.ntiles;
	P.nchunks = c.nchunks;
	P.nstrips = c.nstrips;
	P.strip_rows = c.strip_rows;
	P.cnt = cnt;
	P.hints = strcmp(svtgpu_env("SVTGPU_TR_HINTS", "on"), "on") == 0;
	P.t_ptr = t_ptr;
	P.t_offs = t_offs;
	P.t_vals = t_vals;
	const bool flat_count = blocks &&
		4 * (size_t) m->nrow <= (size_t) 200 * 1024 &&
		(((uintptr_t) m->d_offs) & 15) == 0 &&
		strcmp(svtgpu_env("SVTGPU_TR_COUNT", "flat"), "flat") == 0;
	if (rc == SVTGPU_OK && flat_count) {
		int per_chunk = svtgpu_sm_count() / c.nchunks;
		if (per_chunk < 1) per_chunk = 1;
		cudaError_t ec = cudaMemsetAsync(cnt, 0,
			4 * (size_t) c.nchunks * (size_t) m->nrow, s);
		if (ec == cudaSuccess)
			ec = cudaFuncSetAttribute(transpose_count_flat,
				cudaFuncAttributeMaxDynamicSharedMemorySize,
				(int) (4 * (size_t) m->nrow));
		if (ec == cudaSuccess) {
			transpose_count_flat<<<(unsigned) (c.nchunks * per_chunk),
				1024, 4 * (size_t) m->nrow, s>>>(P, per_chunk);
			ec = cudaGetLastError();
		}
		if (ec != cudaSuccess)
			rc = svtgpu_cuda_fail(ec, "transpose_count_flat", __FILE__,
					      __LINE__);
		svtgpu_count_launch(1);
	} else if (rc == SVTGPU_OK && blocks) {
		transpose_count<<<(unsigned) (c.nchunks * c.ntiles), 1024,
			(size_t) c.strip_rows * 4, s>>>(P);
		cudaError_t ec = cudaGetLastError();
		if (ec != cudaSuccess)
			rc = svtgpu_cuda_fail(ec, "transpose_count", __FILE__,
					      __LINE__);
		svtgpu_count_launch(1);
	} else if (rc == SVTGPU_OK) {   /* counting never looks at the values */
		rc = batch ? launch_batch<int32_t, true, false>(c, P, s)
			   : launch_walk<int32_t, true, false>(c, P, s);
	}
	if (rc == SVTGPU_OK) {
		transpose_row_totals<<<grid_for(m->nrow, 256), 256, 0, s>>>(
			cnt, c.nchunks, m->nrow, total);
		svtgpu_count_launch(1);
		rc = svtgpu_exclusive_scan(total, m->nrow, t_ptr, s);
	}
	if (rc == SVTGPU_OK) {
		transpose_positions<<<grid_for(m->nrow, 256), 256, 0, s>>>(cnt,
			c.nchunks, m->nrow, c.strip_rows, t_ptr, d_over);
		svtgpu_count_launch(1);
		e = cudaMemcpyAsync(&h_over, d_over, sizeof(int),
				    cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess)
			e = cudaStreamSynchronize(s);
		if (e != cudaSuccess)
			rc = svtgpu_cuda_fail(e, "transpose plan", __FILE__,
					      __LINE__);
	}
	if (rc == SVTGPU_OK && !h_over && blocks) {
		if (lac)
			rc = launch_blocks<int32_t, true>(kb, P, s);
		else if (dbl)
			rc = launch_blocks<double, false>(kb, P, s);
		else
			rc = launch_blocks<int32_t, false>(kb, P, s);
	} else if (rc == SVTGPU_OK && !h_over && batch) {
		if (lac)
			rc = launch_batch<int32_t, true, true>(c, P, s);
		else if (dbl)
			rc = launch_batch<double, false, true>(c, P, s);
		else
			rc = launch_batch<int32_t, false, true>(c, P, s);
	} else if (rc == SVTGPU_OK && !h_over) {
		if (lac)
			rc = launch_walk<int32_t, true, true>(c, P, s);
		else if (dbl)
			rc = launch_walk<double, false, true>(c, P, s);
		else
			rc = launch_walk<int32_t, false, true>(c, P, s);
	}
	if (cnt) svt_free_async(cnt, s);
	if (total) svt_free_async(total, s);
	if (d_over) svt_free_async(d_over, s);
	if (rc != SVTGPU_OK || h_over) {
		if (t_ptr) svt_free_async(t_ptr, s);
		if (t_offs) svt_free_async(t_offs, s);
		if (t_vals) svt_free_async(t_vals, s);
		m->transpose_failed = 1;
		return rc;
	}
	svtgpu_matrix *t = (svtgpu_matrix *) calloc(1, sizeof(svtgpu_matrix));
	if (t == NULL) {
		svt_free_async(t_ptr, s);
		svt_free_async(t_offs, s);
		if (t_vals) svt_free_async(t_vals, s);
		svtgpu_set_error("transpose: out of host memory");
		return SVTGPU_ERR_NOMEM;
	}
	t->nrow = m->nleaf;
	t->nleaf = m->nrow;
	t->nnz = m->nnz;
	t->val_type = m->val_type;
	t->flags = m->flags;
	t->owns = 1;
	t->device = m->device;
	t->d_leaf_ptr = t_ptr;
	t->d_offs = t_offs;
	t->d_vals = t_vals;
	t->stage_cur = -1;
	t->vmax_abs = m->vmax_abs;
	t->vmin = m->vmin;
	m->transposed = t;
	*out = t;
	return SVTGPU_OK;
}

/* t(m) for a matrix m that the caller built and is about to free: the
 * transpose is handed to the caller (free it with svtgpu_matrix_free) instead
 * of staying cached in m.  NULL + SVTGPU_OK as for svtgpu_ensure_transpose. */
int svtgpu_transpose_fresh(svtgpu_matrix *m, cudaStream_t s,
			   svtgpu_matrix **out)
{
	SVT_CHECK(svtgpu_ensure_transpose(m, s, out));
	m->transposed = NULL;
	return SVTGPU_OK;
}
