/* Internal declarations shared by the translation units of libsvtgpu.so. */
#ifndef SVTGPU_INTERNAL_H
#define SVTGPU_INTERNAL_H

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/svtgpu.h"
#include "svt_semantics.h"

#define SVTGPU_NSTAGE 3   /* pinned staging slots that rotate during upload */
#define SVTGPU_NSPLIT 4   /* cached row-tile split arrays per matrix */

struct svtgpu_matrix {
	int64_t nrow, nleaf, nnz;
	int val_type;        /* SVTGPU_LGL / SVTGPU_INT / SVTGPU_DOUBLE */
	int flags;           /* SVTGPU_HAS_OFFS | SVTGPU_HAS_VALS */
	int owns;            /* device arrays allocated by us */
	int device;

	int64_t *d_leaf_ptr; /* nleaf + 1 */
	int32_t *d_offs;     /* nnz (+ padding) */
	void *d_vals;        /* nnz (+ padding) */

	/* upload machinery */
	cudaStream_t up_stream;
	int64_t stage_cap;   /* nonzeros per staging slot */
	int32_t *h_offs_stage[SVTGPU_NSTAGE];
	void *h_vals_stage[SVTGPU_NSTAGE];
	cudaEvent_t stage_done[SVTGPU_NSTAGE];
	int stage_busy[SVTGPU_NSTAGE];
	int stage_cur;       /* slot handed out by the last stage() */
	cudaEvent_t up_begin, up_end;
	int up_begun;
	/* device staging for narrowed uploads (uint16 offsets, int8 values) */
	void *d_narrow[SVTGPU_NSTAGE];
	size_t narrow_bytes;

	/* lazily allocated scratch (row partials, tile splits, dense operand) */
	void *d_scratch;
	size_t scratch_bytes;
	/* (ntiles-1) x nleaf leaf-relative split points, per row tiling */
	int32_t *d_split[SVTGPU_NSPLIT];
	int split_tile_rows[SVTGPU_NSPLIT];
	int split_ntiles[SVTGPU_NSPLIT];
	int split_next;
	/* tile table (svt_ensure_tile_table): the leaf that holds the first
	   entry of every tile of tile_entries entries, and the most leaves a
	   tile touches */
	int64_t *d_tile_leaf;
	int64_t tile_entries, tile_count;
	int tile_max_leaves;
	int64_t vmax_abs;    /* max |x| of an integer matrix, -1 = not computed */
	/* value payloads committed as int8 / at native width: a matrix that
	   only ever saw int8 payloads has |x| <= 127 without looking */
	int64_t n_i8_commits, n_wide_commits;
	int64_t vmin;        /* < 0 when the matrix holds a negative value */
	int64_t leaf_base;   /* global index of leaf 0 when m is a column shard */
	struct svtgpu_matrix *transposed;   /* cached t(m), owned by m */
	int transpose_failed;
	/* compact copy of the entries, owned by m (see svt_ensure_compact) */
	uint16_t *d_offs16;  /* nnz + SVT_COMPACT_PAD, or NULL */
	int8_t *d_vals8;     /* nnz + SVT_COMPACT_PAD, or NULL */
	int compact_state;   /* SVT_COMPACT_NONE / _BUILT / _INELIGIBLE */
	int compact_uses;    /* eligible statistic calls seen while NONE */
	int64_t med_selected;  /* leaves sent to selection by the last
				  svtgpu_colmedians / svtgpu_rowmedians */
	int64_t med_select_reads;  /* values its selection passes read */

	svtgpu_timings tm;
};

/* ---- compact copy ----
 * The hot statistics of small-count integer matrices are bound by the bytes
 * they read, and 4-byte offsets and values mostly carry padding.  A matrix may
 * hold a second, narrow copy of its entries beside the wide arrays:
 *   d_vals8   int8 values; NA is SVT_COMPACT_NA_I8 (-128).  Built for integer
 *             and logical matrices whose non-NA values all lie in [-127, 127]
 *             (vmax_abs <= 127, so no stored value is -128).
 *   d_offs16  uint16 row offsets.  Built for nrow <= 65536, and only beside
 *             d_vals8: no kernel reads the offsets alone.
 * Both are padded by SVT_COMPACT_PAD zeroed entries so that 16-byte loads
 * past the last entry stay inside the allocation.  The copy is built on the
 * second eligible statistic call on a handle (a handle used once never pays
 * for it), dropped wherever the wide arrays are rewritten, and not inherited
 * by derived matrices. */
#define SVT_COMPACT_NA_I8 (-128)
#define SVT_COMPACT_PAD 64
#define SVT_COMPACT_NONE 0
#define SVT_COMPACT_BUILT 1
#define SVT_COMPACT_INELIGIBLE 2
#define SVT_COMPACT_MAX_ABS 127
#define SVT_COMPACT_MAX_NROW 65536

/* Count one eligible statistic call on m and build the compact copy on the
   second (synchronises s once).  Never fails for lack of memory: the matrix
   is then marked ineligible and the wide arrays serve. */
int svt_ensure_compact(svtgpu_matrix *m, cudaStream_t s);
/* Free the compact copy (stream-ordered on s) and forget that it was decided. */
void svt_drop_compact(svtgpu_matrix *m, cudaStream_t s);

/* ---- tile table ----
 * The cyclic form of row_hist cuts the entries into tiles of `tile` entries
 * and lets the CTAs take them round-robin, so that the whole GPU sweeps the
 * arrays front to back.  m->d_tile_leaf[t] (t <= ntiles) is the leaf that
 * holds entry min(t * tile, nnz - 1): tile t touches leaves d_tile_leaf[t] ..
 * d_tile_leaf[t + 1], and m->tile_max_leaves is the most leaves any tile
 * touches.  Built once per matrix and tile size (synchronises s once).
 * SVT_TILE_ENTRIES is the tile of the value modes.  Requires nnz > 0. */
#define SVT_TILE_ENTRIES 32768
int svt_ensure_tile_table(svtgpu_matrix *m, int64_t tile, cudaStream_t s);

/* upper bound of |x| over the non-NA values of an integer matrix when one is
   known without a pass over the data, else -1 */
int64_t svtgpu_value_bound(const svtgpu_matrix *m);

/* error plumbing */
void svtgpu_set_error(const char *fmt, ...);
int svtgpu_cuda_fail(cudaError_t e, const char *what, const char *file,
		     int line);

#define SVT_CUDA(call) \
	do { \
		cudaError_t e__ = (call); \
		if (e__ != cudaSuccess) \
			return svtgpu_cuda_fail(e__, #call, __FILE__, __LINE__); \
	} while (0)

#define SVT_CHECK(call) \
	do { \
		int rc__ = (call); \
		if (rc__ != SVTGPU_OK) \
			return rc__; \
	} while (0)

#define SVT_ARG(cond, ...) \
	do { \
		if (!(cond)) { \
			svtgpu_set_error(__VA_ARGS__); \
			return SVTGPU_ERR_ARG; \
		} \
	} while (0)

/* device memory: large blocks bypass the stream-ordered pool (see
   svtgpu_matrix.cu) */
cudaError_t svt_malloc_async(void **out, size_t bytes, cudaStream_t s);
cudaError_t svt_free_async(void *p, cudaStream_t s);

int svtgpu_require_device(void);
void svtgpu_count_launch(int n);
int svtgpu_scratch(svtgpu_matrix *m, size_t bytes, void **ptr);
int svtgpu_sm_count(void);
const char *svtgpu_env(const char *name, const char *dflt);

static inline int svt_is_double(int val_type)
{
	return val_type == SVTGPU_DOUBLE;
}

static inline size_t svt_val_size(int val_type)
{
	return val_type == SVTGPU_DOUBLE ? sizeof(double) : sizeof(int32_t);
}

/* launchers implemented in the kernel files */
int svtgpu_ensure_absmax(svtgpu_matrix *m, cudaStream_t s);
int svtgpu_ensure_split(svtgpu_matrix *m, int nstrips, int strip_rows,
			cudaStream_t s, const int32_t **split);
int svtgpu_ensure_transpose(svtgpu_matrix *m, cudaStream_t s,
			    svtgpu_matrix **out);
/* the same, t(m) owned by the caller rather than cached in m */
int svtgpu_transpose_fresh(svtgpu_matrix *m, cudaStream_t s,
			   svtgpu_matrix **out);
int svtgpu_launch_colstats(svtgpu_matrix *m, int opcode, int narm,
			   double center, int64_t group, void *d_out,
			   int32_t *d_warn, cudaStream_t stream);
int svtgpu_launch_row_accumulate(svtgpu_matrix *m, int opcode, int narm,
				 int want_sum2, double *d_state,
				 cudaStream_t stream);
int svtgpu_launch_row_finalize(int opcode, int val_type, int narm,
			       int64_t nrow, int64_t nstrata,
			       const double *d_center, const double *d_state,
			       void *d_out, int32_t *d_warn,
			       cudaStream_t stream);
int svtgpu_launch_row_moments_finalize(int val_type, int narm, int64_t nrow,
				       int64_t nstrata, const double *d_state,
				       double *d_mean, double *d_var,
				       cudaStream_t stream);

/* event-timed region helpers */
struct SvtTimer {
	cudaEvent_t a, b;
	cudaStream_t s;
	int ok;
};
int svt_timer_begin(SvtTimer *t, cudaStream_t s);
int svt_timer_end(SvtTimer *t, double *ms);   /* synchronises the stream */

#endif  /* SVTGPU_INTERNAL_H */
