/* Device CSC lifecycle: allocation, pinned-staging upload, scratch, errors.
 *
 * The flattened SVT ("device CSC") is three arrays in HBM: int64 leaf_ptr
 * [nleaf+1], int32 offs[nnz], T vals[nnz] (absent when every leaf is lacunar).
 * offs/vals are over-allocated by 64 elements so 16-byte vector and bulk loads
 * that run past the last nonzero stay inside the allocation.
 *
 * Upload path (reference analogue: none -- the reference computes in place on
 * R vectors; the host-side pattern is dump_SVT_to_CsparseMatrix_slots(),
 * src/SVT_SparseArray_class.c:598-679): a process-wide pool of SVTGPU_NSTAGE
 * pinned staging slots rotates; the flattener fills slot k while slot k-1 is
 * in flight on the copy engine.
 */
#include "svtgpu_internal.h"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <cub/device/device_scan.cuh>

/* ---- errors ---- */

static thread_local char g_err[1024] = "";

void svtgpu_set_error(const char *fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
}

extern "C" const char *svtgpu_last_error(void)
{
	return g_err;
}

int svtgpu_cuda_fail(cudaError_t e, const char *what, const char *file,
		     int line)
{
	svtgpu_set_error("CUDA error %d (%s) in %s at %s:%d", (int) e,
			 cudaGetErrorString(e), what, file, line);
	if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver)
		return SVTGPU_ERR_NO_DEVICE;
	if (e == cudaErrorMemoryAllocation)
		return SVTGPU_ERR_NOMEM;
	return SVTGPU_ERR_CUDA;
}

const char *svtgpu_env(const char *name, const char *dflt)
{
	const char *v = getenv(name);
	return (v != NULL && v[0] != '\0') ? v : dflt;
}

/* ---- device ---- */

static int g_device_checked = 0;
static int g_sm_count = 0;

int svtgpu_require_device(void)
{
	if (g_device_checked)
		return SVTGPU_OK;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0) {
		svtgpu_set_error("no usable CUDA device (%s); libsvtgpu has no "
				 "CPU fallback",
				 e != cudaSuccess ? cudaGetErrorString(e)
						  : "device count is 0");
		return SVTGPU_ERR_NO_DEVICE;
	}
	int dev = 0;
	SVT_CUDA(cudaGetDevice(&dev));
	cudaDeviceProp prop;
	SVT_CUDA(cudaGetDeviceProperties(&prop, dev));
	if (prop.major < 10) {
		svtgpu_set_error("device '%s' is sm_%d%d; libsvtgpu is built "
				 "for sm_100a only", prop.name, prop.major,
				 prop.minor);
		return SVTGPU_ERR_NO_DEVICE;
	}
	g_sm_count = prop.multiProcessorCount;
	/* device arrays come from the stream-ordered pool and stay cached in
	   it between calls: cudaMalloc/cudaFree of multi-GB arrays cost
	   hundreds of ms, which the stateless .Call path would pay per call */
	cudaMemPool_t pool;
	if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
		uint64_t keep = UINT64_MAX;
		cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold,
					&keep);
	}
	cudaGetLastError();
	g_device_checked = 1;
	return SVTGPU_OK;
}

int svtgpu_sm_count(void)
{
	return g_sm_count > 0 ? g_sm_count : 148;
}

extern "C" int svtgpu_device_count(int *count)
{
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess) {
		*count = 0;
		return svtgpu_cuda_fail(e, "cudaGetDeviceCount", __FILE__,
					__LINE__);
	}
	*count = n;
	return SVTGPU_OK;
}

static void pool_teardown(void);

extern "C" int svtgpu_set_device(int device)
{
	int cur = -1;
	cudaGetDevice(&cur);
	/* the pinned staging pool's events belong to the device that was
	   current when they were made: recording them on another device's
	   stream fails (cudaErrorInvalidResourceHandle) */
	if (cur != device)
		pool_teardown();
	SVT_CUDA(cudaSetDevice(device));
	g_device_checked = 0;
	return svtgpu_require_device();
}

extern "C" int svtgpu_get_device(int *device)
{
	SVT_CUDA(cudaGetDevice(device));
	return SVTGPU_OK;
}

extern "C" int svtgpu_device_info(char *name, int name_len, int *sm_count,
				  int64_t *total_mem_bytes)
{
	SVT_CHECK(svtgpu_require_device());
	int dev = 0;
	SVT_CUDA(cudaGetDevice(&dev));
	cudaDeviceProp prop;
	SVT_CUDA(cudaGetDeviceProperties(&prop, dev));
	if (name != NULL && name_len > 0) {
		strncpy(name, prop.name, (size_t) name_len - 1);
		name[name_len - 1] = '\0';
	}
	if (sm_count != NULL)
		*sm_count = prop.multiProcessorCount;
	if (total_mem_bytes != NULL)
		*total_mem_bytes = (int64_t) prop.totalGlobalMem;
	return SVTGPU_OK;
}

static void big_release_all(void);

extern "C" int svtgpu_release_cached_memory(void)
{
	SVT_CHECK(svtgpu_require_device());
	int dev = 0;
	SVT_CUDA(cudaGetDevice(&dev));
	SVT_CUDA(cudaDeviceSynchronize());
	big_release_all();
	cudaMemPool_t pool;
	SVT_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
	SVT_CUDA(cudaMemPoolTrimTo(pool, 0));
	return SVTGPU_OK;
}

/* ---- device memory ----
 * Small arrays come from CUDA's stream-ordered pool.  Large ones do NOT: the
 * first time the pool has to grow by a multi-GB block, svt_malloc_async() takes
 * 0.6 - 4.6 s (measured on B200, tools/microbench/alloc_time.cu: 29 GB in
 * 632 ms / 3115 ms, against 2 - 3 ms for plain cudaMalloc() of the same
 * arrays) -- that was the erratic first `svt %*% D`.  Blocks of 32 MB and more
 * are cudaMalloc()ed and, when released, parked in a small cache (cudaFree()
 * synchronises the device: 11 ms for 29 GB) together with an event that marks
 * the end of their last use; svtgpu_release_cached_memory() frees them. */
#define SVT_BIG_BYTES ((size_t) 32 << 20)
#define SVT_NBIG 64

struct BigBlock {
	void *ptr;
	size_t bytes;
	int device;
	int in_use;
	cudaEvent_t done;   /* last use, valid while parked */
	int has_event;
};
static BigBlock g_big[SVT_NBIG];

cudaError_t svt_malloc_async(void **out, size_t bytes, cudaStream_t s)
{
	if (bytes < SVT_BIG_BYTES)
		return cudaMallocAsync(out, bytes, s);
	int dev = 0;
	cudaGetDevice(&dev);
	/* best fit among the parked blocks: at most 12.5 % larger */
	int best = -1;
	for (int i = 0; i < SVT_NBIG; i++) {
		BigBlock *b = &g_big[i];
		if (b->ptr == NULL || b->in_use || b->device != dev ||
		    b->bytes < bytes || b->bytes - bytes > bytes / 8)
			continue;
		if (best < 0 || b->bytes < g_big[best].bytes)
			best = i;
	}
	if (best >= 0) {
		BigBlock *b = &g_big[best];
		if (b->has_event) {
			cudaError_t e = cudaStreamWaitEvent(s, b->done, 0);
			if (e != cudaSuccess)
				return e;
		}
		b->in_use = 1;
		*out = b->ptr;
		return cudaSuccess;
	}
	int slot = -1;
	for (int i = 0; i < SVT_NBIG && slot < 0; i++)
		if (g_big[i].ptr == NULL)
			slot = i;
	if (slot < 0) {
		/* table full: evict the smallest parked block */
		for (int i = 0; i < SVT_NBIG; i++)
			if (!g_big[i].in_use && (slot < 0 ||
			    g_big[i].bytes < g_big[slot].bytes))
				slot = i;
		if (slot < 0)
			return cudaMallocAsync(out, bytes, s);
		cudaFree(g_big[slot].ptr);
		g_big[slot].ptr = NULL;
	}
	void *p = NULL;
	cudaError_t e = cudaMalloc(&p, bytes);
	if (e == cudaErrorMemoryAllocation) {
		/* give the parked blocks back and try once more */
		cudaGetLastError();
		for (int i = 0; i < SVT_NBIG; i++)
			if (g_big[i].ptr != NULL && !g_big[i].in_use) {
				cudaFree(g_big[i].ptr);
				g_big[i].ptr = NULL;
			}
		e = cudaMalloc(&p, bytes);
	}
	if (e != cudaSuccess)
		return e;
	BigBlock *b = &g_big[slot];
	b->ptr = p;
	b->bytes = bytes;
	b->device = dev;
	b->in_use = 1;
	*out = p;
	return cudaSuccess;
}

cudaError_t svt_free_async(void *p, cudaStream_t s)
{
	if (p == NULL)
		return cudaSuccess;
	for (int i = 0; i < SVT_NBIG; i++) {
		BigBlock *b = &g_big[i];
		if (b->ptr != p || !b->in_use)
			continue;
		if (!b->has_event) {
			if (cudaEventCreateWithFlags(&b->done,
					cudaEventDisableTiming) == cudaSuccess)
				b->has_event = 1;
		}
		if (b->has_event)
			cudaEventRecord(b->done, s);
		else
			cudaStreamSynchronize(s);
		b->in_use = 0;
		return cudaSuccess;
	}
	return cudaFreeAsync(p, s);
}

static void big_release_all(void)
{
	for (int i = 0; i < SVT_NBIG; i++) {
		BigBlock *b = &g_big[i];
		if (b->ptr != NULL && !b->in_use) {
			cudaFree(b->ptr);
			b->ptr = NULL;
			if (b->has_event) {
				cudaEventDestroy(b->done);
				b->has_event = 0;
			}
		}
	}
}

static long long g_launches = 0;

void svtgpu_count_launch(int n)
{
	__atomic_add_fetch(&g_launches, (long long) n, __ATOMIC_RELAXED);
}

extern "C" int64_t svtgpu_launch_count(void)
{
	return (int64_t) __atomic_load_n(&g_launches, __ATOMIC_RELAXED);
}

/* ---- timers ---- */

int svt_timer_begin(SvtTimer *t, cudaStream_t s)
{
	t->ok = 0;
	t->s = s;
	SVT_CUDA(cudaEventCreate(&t->a));
	SVT_CUDA(cudaEventCreate(&t->b));
	SVT_CUDA(cudaEventRecord(t->a, s));
	t->ok = 1;
	return SVTGPU_OK;
}

int svt_timer_end(SvtTimer *t, double *ms)
{
	if (!t->ok)
		return SVTGPU_OK;
	float f = 0.f;
	cudaError_t e = cudaEventRecord(t->b, t->s);
	if (e == cudaSuccess)
		e = cudaEventSynchronize(t->b);
	if (e == cudaSuccess)
		e = cudaEventElapsedTime(&f, t->a, t->b);
	cudaEventDestroy(t->a);
	cudaEventDestroy(t->b);
	t->ok = 0;
	if (e != cudaSuccess)
		return svtgpu_cuda_fail(e, "timer", __FILE__, __LINE__);
	if (ms != NULL)
		*ms = (double) f;
	return SVTGPU_OK;
}

/* ---- process-wide pinned staging pool ---- */

struct StagePool {
	int64_t cap;   /* nonzeros per slot */
	int32_t *offs[SVTGPU_NSTAGE];
	double *vals[SVTGPU_NSTAGE];   /* sized for doubles */
	cudaEvent_t done[SVTGPU_NSTAGE];
	int busy[SVTGPU_NSTAGE];
	int inited;
	int next;
};
static StagePool g_pool;

static void pool_teardown(void)
{
	if (!g_pool.inited)
		return;
	for (int i = 0; i < SVTGPU_NSTAGE; i++) {
		if (g_pool.busy[i])
			cudaEventSynchronize(g_pool.done[i]);
		cudaEventDestroy(g_pool.done[i]);
		if (g_pool.offs[i]) cudaFreeHost(g_pool.offs[i]);
		if (g_pool.vals[i]) cudaFreeHost(g_pool.vals[i]);
	}
	memset(&g_pool, 0, sizeof(g_pool));
}

static int64_t stage_cap_limit(void)
{
	long mb = atol(svtgpu_env("SVTGPU_STAGE_MB", "128"));
	if (mb < 1)
		mb = 1;
	return (int64_t) mb * 1024 * 1024 / 8;
}

static int pool_reserve(int64_t want)
{
	int64_t limit = stage_cap_limit();
	if (want > limit)
		want = limit;
	if (want < 1024)
		want = 1024;
	if (!g_pool.inited) {
		memset(&g_pool, 0, sizeof(g_pool));
		for (int i = 0; i < SVTGPU_NSTAGE; i++)
			SVT_CUDA(cudaEventCreateWithFlags(&g_pool.done[i],
						cudaEventDisableTiming));
		g_pool.inited = 1;
	}
	if (g_pool.cap >= want)
		return SVTGPU_OK;
	for (int i = 0; i < SVTGPU_NSTAGE; i++) {
		if (g_pool.busy[i]) {
			SVT_CUDA(cudaEventSynchronize(g_pool.done[i]));
			g_pool.busy[i] = 0;
		}
		if (g_pool.offs[i]) cudaFreeHost(g_pool.offs[i]);
		if (g_pool.vals[i]) cudaFreeHost(g_pool.vals[i]);
		g_pool.offs[i] = NULL;
		g_pool.vals[i] = NULL;
	}
	g_pool.cap = 0;
	for (int i = 0; i < SVTGPU_NSTAGE; i++) {
		SVT_CUDA(cudaHostAlloc((void **) &g_pool.offs[i],
				       sizeof(int32_t) * (size_t) want,
				       cudaHostAllocDefault));
		SVT_CUDA(cudaHostAlloc((void **) &g_pool.vals[i],
				       sizeof(double) * (size_t) want,
				       cudaHostAllocDefault));
	}
	g_pool.cap = want;
	return SVTGPU_OK;
}

/* ---- matrix ---- */

static int matrix_new(svtgpu_matrix **out, int64_t nrow, int64_t nleaf,
		      int64_t nnz, int val_type, int flags)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(out != NULL, "svtgpu_matrix: NULL output pointer");
	SVT_ARG(nrow >= 0 && nrow <= INT32_MAX,
		"svtgpu_matrix: nrow must be in [0, 2^31-1]");
	SVT_ARG(nleaf >= 0 && nnz >= 0, "svtgpu_matrix: negative extent");
	SVT_ARG(val_type == SVTGPU_LGL || val_type == SVTGPU_INT ||
		val_type == SVTGPU_DOUBLE,
		"svtgpu_matrix: unsupported value type %d (only logical, "
		"integer and double SVTs are supported on the GPU path)",
		val_type);
	svtgpu_matrix *m = (svtgpu_matrix *) calloc(1, sizeof(svtgpu_matrix));
	if (m == NULL) {
		svtgpu_set_error("svtgpu_matrix: out of host memory");
		return SVTGPU_ERR_NOMEM;
	}
	m->nrow = nrow;
	m->nleaf = nleaf;
	m->nnz = nnz;
	m->val_type = val_type;
	m->flags = flags;
	m->stage_cur = -1;
	m->vmax_abs = -1;
	m->n_i8_commits = m->n_wide_commits = 0;
	cudaGetDevice(&m->device);
	*out = m;
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_create(svtgpu_matrix **out, int64_t nrow,
				    int64_t nleaf, int64_t nnz, int val_type,
				    int flags)
{
	svtgpu_matrix *m = NULL;
	SVT_CHECK(matrix_new(&m, nrow, nleaf, nnz, val_type, flags));
	m->owns = 1;
	const size_t pad = 64;
	cudaError_t e = cudaStreamCreateWithFlags(&m->up_stream,
						  cudaStreamNonBlocking);
	if (e == cudaSuccess)
		e = svt_malloc_async((void **) &m->d_leaf_ptr,
				    sizeof(int64_t) * (size_t) (nleaf + 1),
				    m->up_stream);
	if (e == cudaSuccess && (flags & SVTGPU_HAS_OFFS))
		e = svt_malloc_async((void **) &m->d_offs,
				    sizeof(int32_t) * ((size_t) nnz + pad),
				    m->up_stream);
	if (e == cudaSuccess && (flags & SVTGPU_HAS_VALS))
		e = svt_malloc_async(&m->d_vals,
				    svt_val_size(val_type) * ((size_t) nnz + pad),
				    m->up_stream);
	if (e == cudaSuccess)
		e = cudaEventCreate(&m->up_begin);
	if (e == cudaSuccess)
		e = cudaEventCreate(&m->up_end);
	/* zero the padding so over-reads see defined bytes */
	if (e == cudaSuccess && m->d_offs != NULL)
		e = cudaMemsetAsync(m->d_offs + nnz, 0, sizeof(int32_t) * pad,
				    m->up_stream);
	if (e == cudaSuccess && m->d_vals != NULL)
		e = cudaMemsetAsync((char *) m->d_vals +
				    svt_val_size(val_type) * (size_t) nnz, 0,
				    svt_val_size(val_type) * pad, m->up_stream);
	if (e != cudaSuccess) {
		int rc = svtgpu_cuda_fail(e, "svtgpu_matrix_create", __FILE__,
					  __LINE__);
		svtgpu_matrix_free(m);
		return rc;
	}
	*out = m;
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_wrap_device(svtgpu_matrix **out, int64_t nrow,
					 int64_t nleaf, int64_t nnz,
					 int val_type,
					 const int64_t *d_leaf_ptr,
					 const int32_t *d_offs,
					 const void *d_vals)
{
	svtgpu_matrix *m = NULL;
	int flags = (d_offs != NULL ? SVTGPU_HAS_OFFS : 0) |
		    (d_vals != NULL ? SVTGPU_HAS_VALS : 0);
	SVT_ARG(d_leaf_ptr != NULL, "svtgpu_matrix_wrap_device: NULL leaf_ptr");
	SVT_CHECK(matrix_new(&m, nrow, nleaf, nnz, val_type, flags));
	m->owns = 0;
	m->d_leaf_ptr = (int64_t *) d_leaf_ptr;
	m->d_offs = (int32_t *) d_offs;
	m->d_vals = (void *) d_vals;
	*out = m;
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_free(svtgpu_matrix *m)
{
	if (m == NULL)
		return SVTGPU_OK;
	/* kernels of the device-form entry points may still be running */
	cudaDeviceSynchronize();
	if (m->transposed != NULL) {
		svtgpu_matrix_free(m->transposed);
		m->transposed = NULL;
	}
	if (m->up_stream != NULL) {
		for (int i = 0; i < SVTGPU_NSTAGE; i++)
			if (m->stage_busy[i])
				g_pool.busy[i] = 0;
	}
	if (m->owns) {
		if (m->d_leaf_ptr) svt_free_async(m->d_leaf_ptr, m->up_stream);
		if (m->d_offs) svt_free_async(m->d_offs, m->up_stream);
		if (m->d_vals) svt_free_async(m->d_vals, m->up_stream);
	}
	for (int i = 0; i < SVTGPU_NSTAGE; i++)
		if (m->d_narrow[i]) svt_free_async(m->d_narrow[i], 0);
	if (m->d_scratch) svt_free_async(m->d_scratch, 0);
	for (int i = 0; i < SVTGPU_NSPLIT; i++)
		if (m->d_split[i]) svt_free_async(m->d_split[i], 0);
	if (m->d_tile_leaf) svt_free_async(m->d_tile_leaf, 0);
	svt_drop_compact(m, 0);
	cudaDeviceSynchronize();
	if (m->up_begin) cudaEventDestroy(m->up_begin);
	if (m->up_end) cudaEventDestroy(m->up_end);
	if (m->up_stream) cudaStreamDestroy(m->up_stream);
	free(m);
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_info(const svtgpu_matrix *m, int64_t *nrow,
				  int64_t *nleaf, int64_t *nnz, int *val_type,
				  int *flags)
{
	SVT_ARG(m != NULL, "svtgpu_matrix_info: NULL matrix");
	if (nrow) *nrow = m->nrow;
	if (nleaf) *nleaf = m->nleaf;
	if (nnz) *nnz = m->nnz;
	if (val_type) *val_type = m->val_type;
	if (flags) *flags = m->flags;
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_set_leaf_base(svtgpu_matrix *m, int64_t leaf_base)
{
	SVT_ARG(m != NULL && leaf_base >= 0,
		"svtgpu_matrix_set_leaf_base: bad argument");
	m->leaf_base = leaf_base;
	return SVTGPU_OK;
}

/* ---- N-d row statistics: fold leading dimensions into the rows ---- */

__global__ void __launch_bounds__(256)
fold_offsets(const int64_t *__restrict__ leaf_ptr, int32_t *__restrict__ offs,
	     int64_t nleaf, int64_t fold, int32_t nrow)
{
	const int lane = threadIdx.x & 31;
	const int64_t warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	for (int64_t leaf = gw; leaf < nleaf; leaf += warps) {
		const int32_t shift = nrow * (int32_t) (leaf % fold);
		if (shift == 0)
			continue;
		const int64_t end = leaf_ptr[leaf + 1];
		for (int64_t e = leaf_ptr[leaf] + lane; e < end; e += 32)
			offs[e] += shift;
	}
}

__global__ void __launch_bounds__(256)
fold_leaf_ptr(const int64_t *__restrict__ leaf_ptr, int64_t *__restrict__ out,
	      int64_t nleaf_new, int64_t fold)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t k = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     k <= nleaf_new; k += stride)
		out[k] = leaf_ptr[k * fold];
}

extern "C" int svtgpu_matrix_fold_rows(svtgpu_matrix *m, int64_t fold)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && fold >= 1, "svtgpu_matrix_fold_rows: bad argument");
	SVT_ARG(m->owns, "svtgpu_matrix_fold_rows: the matrix wraps caller-"
		"owned device arrays");
	if (fold == 1)
		return SVTGPU_OK;
	SVT_ARG(m->nleaf % fold == 0, "svtgpu_matrix_fold_rows: 'fold' must "
		"divide the number of leaves");
	SVT_ARG((double) m->nrow * (double) fold <= 2147483647.0,
		"svtgpu_matrix_fold_rows: more than 2^31 - 1 folded rows");
	SVT_ARG((m->flags & SVTGPU_HAS_OFFS) || m->nnz == 0,
		"svtgpu_matrix_fold_rows: the matrix was uploaded without row "
		"offsets");
	SVT_ARG(m->transposed == NULL, "svtgpu_matrix_fold_rows: the matrix "
		"already has a cached transpose");
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	cudaStream_t s = 0;
	const int64_t nleaf_new = m->nleaf / fold;
	const unsigned grid = (unsigned) (svtgpu_sm_count() * 8);
	if (m->nnz > 0) {
		fold_offsets<<<grid, 256, 0, s>>>(m->d_leaf_ptr, m->d_offs,
						  m->nleaf, fold,
						  (int32_t) m->nrow);
		SVT_CUDA(cudaGetLastError());
	}
	int64_t *tmp = NULL;
	SVT_CUDA(svt_malloc_async((void **) &tmp,
				 sizeof(int64_t) * (size_t) (nleaf_new + 1), s));
	fold_leaf_ptr<<<grid, 256, 0, s>>>(m->d_leaf_ptr, tmp, nleaf_new, fold);
	cudaError_t e = cudaGetLastError();
	if (e == cudaSuccess)
		e = cudaMemcpyAsync(m->d_leaf_ptr, tmp,
				    sizeof(int64_t) * (size_t) (nleaf_new + 1),
				    cudaMemcpyDeviceToDevice, s);
	svt_free_async(tmp, s);
	SVT_CUDA(e);
	svtgpu_count_launch(2);
	m->nrow *= fold;
	m->nleaf = nleaf_new;
	/* per-tiling split tables describe the old geometry */
	for (int i = 0; i < SVTGPU_NSPLIT; i++) {
		if (m->d_split[i] != NULL)
			svt_free_async(m->d_split[i], s);
		m->d_split[i] = NULL;
	}
	if (m->d_tile_leaf != NULL)
		svt_free_async(m->d_tile_leaf, s);
	m->d_tile_leaf = NULL;
	m->tile_entries = 0;
	/* the compact offsets hold the old rows (and nrow may now exceed
	   what 16 bits can hold) */
	svt_drop_compact(m, s);
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_download(svtgpu_matrix *m, int64_t *leaf_ptr,
				      int32_t *offs, void *vals)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL, "svtgpu_matrix_download: NULL matrix");
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	SVT_CUDA(cudaDeviceSynchronize());
	if (leaf_ptr != NULL)
		SVT_CUDA(cudaMemcpy(leaf_ptr, m->d_leaf_ptr,
				    8 * (size_t) (m->nleaf + 1),
				    cudaMemcpyDeviceToHost));
	if (offs != NULL && m->d_offs != NULL && m->nnz > 0)
		SVT_CUDA(cudaMemcpy(offs, m->d_offs, 4 * (size_t) m->nnz,
				    cudaMemcpyDeviceToHost));
	if (vals != NULL && m->d_vals != NULL && m->nnz > 0)
		SVT_CUDA(cudaMemcpy(vals, m->d_vals,
				    svt_val_size(m->val_type) * (size_t) m->nnz,
				    cudaMemcpyDeviceToHost));
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_transposed(svtgpu_matrix *m, svtgpu_matrix **t)
{
	SVT_CHECK(svtgpu_require_device());
	SVT_ARG(m != NULL && t != NULL, "svtgpu_matrix_transposed: NULL argument");
	SVT_CHECK(svtgpu_matrix_finish_upload(m));
	SVT_CHECK(svtgpu_ensure_transpose(m, 0, t));
	SVT_CUDA(cudaStreamSynchronize(0));
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_timings(const svtgpu_matrix *m, svtgpu_timings *t)
{
	SVT_ARG(m != NULL && t != NULL, "svtgpu_matrix_timings: NULL argument");
	*t = m->tm;
	return SVTGPU_OK;
}

static int upload_begin(svtgpu_matrix *m)
{
	/* the entries are about to be rewritten */
	svt_drop_compact(m, m->up_stream);
	if (!m->up_begun) {
		SVT_CUDA(cudaEventRecord(m->up_begin, m->up_stream));
		m->up_begun = 1;
		m->tm.h2d_bytes = 0;
	}
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_set_leaf_ptr(svtgpu_matrix *m,
					  const int64_t *leaf_ptr)
{
	SVT_ARG(m != NULL && m->owns, "svtgpu_matrix_set_leaf_ptr: matrix does "
		"not own its storage");
	SVT_ARG(leaf_ptr[0] == 0 && leaf_ptr[m->nleaf] == m->nnz,
		"svtgpu_matrix_set_leaf_ptr: leaf_ptr does not span [0, nnz]");
	SVT_CHECK(upload_begin(m));
	/* pageable source: the runtime stages it, which is fine for 8 B/leaf */
	SVT_CUDA(cudaMemcpyAsync(m->d_leaf_ptr, leaf_ptr,
				 sizeof(int64_t) * (size_t) (m->nleaf + 1),
				 cudaMemcpyHostToDevice, m->up_stream));
	m->tm.h2d_bytes += 8.0 * (double) (m->nleaf + 1);
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_stage_capacity(svtgpu_matrix *m,
					    int64_t *max_count)
{
	SVT_ARG(m != NULL && m->owns, "svtgpu_matrix_stage_capacity: matrix "
		"does not own its storage");
	SVT_CHECK(pool_reserve(m->nnz));
	*max_count = g_pool.cap;
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_stage(svtgpu_matrix *m, int64_t count,
				   int32_t **offs_slot, void **vals_slot)
{
	SVT_ARG(m != NULL && m->owns, "svtgpu_matrix_stage: matrix does not "
		"own its storage");
	SVT_CHECK(pool_reserve(m->nnz));
	SVT_ARG(count >= 0 && count <= g_pool.cap,
		"svtgpu_matrix_stage: count exceeds the staging capacity");
	int s = g_pool.next;
	g_pool.next = (g_pool.next + 1) % SVTGPU_NSTAGE;
	if (g_pool.busy[s]) {
		SVT_CUDA(cudaEventSynchronize(g_pool.done[s]));
		g_pool.busy[s] = 0;
	}
	m->stage_busy[s] = 0;
	m->stage_cur = s;
	if (offs_slot)
		*offs_slot = (m->flags & SVTGPU_HAS_OFFS) ? g_pool.offs[s]
							  : NULL;
	if (vals_slot)
		*vals_slot = (m->flags & SVTGPU_HAS_VALS)
				? (void *) g_pool.vals[s] : NULL;
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_commit(svtgpu_matrix *m, int64_t dst,
				    int64_t count)
{
	SVT_ARG(m != NULL && m->stage_cur >= 0,
		"svtgpu_matrix_commit: no staged slot");
	SVT_ARG(dst >= 0 && count >= 0 && dst + count <= m->nnz,
		"svtgpu_matrix_commit: range outside [0, nnz]");
	int s = m->stage_cur;
	SVT_CHECK(upload_begin(m));
	if (count > 0 && (m->flags & SVTGPU_HAS_OFFS)) {
		SVT_CUDA(cudaMemcpyAsync(m->d_offs + dst, g_pool.offs[s],
					 sizeof(int32_t) * (size_t) count,
					 cudaMemcpyHostToDevice,
					 m->up_stream));
		m->tm.h2d_bytes += 4.0 * (double) count;
	}
	if (count > 0 && (m->flags & SVTGPU_HAS_VALS)) {
		size_t vs = svt_val_size(m->val_type);
		m->n_wide_commits++;
		SVT_CUDA(cudaMemcpyAsync((char *) m->d_vals + vs * (size_t) dst,
					 g_pool.vals[s], vs * (size_t) count,
					 cudaMemcpyHostToDevice,
					 m->up_stream));
		m->tm.h2d_bytes += (double) vs * (double) count;
	}
	SVT_CUDA(cudaEventRecord(g_pool.done[s], m->up_stream));
	g_pool.busy[s] = 1;
	m->stage_busy[s] = 1;
	m->stage_cur = -1;
	return SVTGPU_OK;
}

int64_t svtgpu_value_bound(const svtgpu_matrix *m)
{
	if (svt_is_double(m->val_type))
		return -1;
	if (m->vmax_abs >= 0)
		return m->vmax_abs;
	if (m->owns && m->n_i8_commits > 0 && m->n_wide_commits == 0)
		return 127;
	return -1;
}

/* ---- narrowed uploads: widen in HBM ---- */

__global__ void __launch_bounds__(256)
widen_u16_i32(const uint16_t *__restrict__ src, int32_t *__restrict__ dst,
	      int64_t n)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     i < n; i += stride)
		dst[i] = (int32_t) src[i];
}

template <typename T>
__global__ void __launch_bounds__(256)
widen_i8(const int8_t *__restrict__ src, T *__restrict__ dst, int64_t n)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	     i < n; i += stride) {
		const int x = src[i];
		if (sizeof(T) == 4)
			dst[i] = (T) (x == -128 ? SVT_NA_INT : x);
		else
			dst[i] = x == -128 ? (T) svt_na_real() : (T) x;
	}
}

/* 16-bit offsets of a matrix with more than 65536 rows: the LOW halves only.
 * Offsets ascend strictly inside a leaf and the sender guarantees gaps below
 * 65536 (and a first entry below 65536), so the high half goes up by exactly
 * one wherever the low half goes down: a warp per leaf rebuilds it with a
 * ballot / popcount prefix.  A leaf that began in an earlier slot continues
 * from its last widened entry (same stream: already written). */
__global__ void __launch_bounds__(256)
widen_u16_wrapped(const uint16_t *__restrict__ src, int32_t *offs,
		  const int64_t *__restrict__ leaf_ptr, int64_t nleaf,
		  int64_t dst, int64_t count)
{
	const int lane = threadIdx.x & 31;
	const int64_t warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
	const int64_t gw = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int64_t end = dst + count;
	/* first leaf whose range ends after entry dst */
	int64_t lo_l = 0, hi_l = nleaf;
	while (lo_l < hi_l) {
		const int64_t mid = lo_l + ((hi_l - lo_l) >> 1);
		if (leaf_ptr[mid + 1] <= dst) lo_l = mid + 1;
		else                          hi_l = mid;
	}
	for (int64_t leaf = lo_l + gw; leaf < nleaf; leaf += warps) {
		const int64_t a = leaf_ptr[leaf];
		if (a >= end)
			break;
		const int64_t b = leaf_ptr[leaf + 1];
		const int64_t from = a > dst ? a : dst;
		const int64_t to = b < end ? b : end;
		int hi = 0, prev_lo = -1;
		if (from > a && from < to) {
			const int32_t p = offs[from - 1];
			hi = p >> 16;
			prev_lo = p & 0xFFFF;
		}
		for (int64_t e0 = from; e0 < to; e0 += 32) {
			const int64_t e = e0 + lane;
			const bool ok = e < to;
			const int lo = ok ? (int) src[e - dst] : 0x10000;
			int before = __shfl_up_sync(0xFFFFFFFFu, lo, 1);
			if (lane == 0)
				before = prev_lo;
			const unsigned wraps = __ballot_sync(0xFFFFFFFFu,
							     ok && lo < before);
			if (ok)
				offs[e] = ((hi + __popc(wraps &
					(0xFFFFFFFFu >> (31 - lane)))) << 16) | lo;
			hi += __popc(wraps);
			prev_lo = __shfl_sync(0xFFFFFFFFu, lo, 31);
		}
	}
}

extern "C" int svtgpu_matrix_commit_packed(svtgpu_matrix *m, int64_t dst,
					   int64_t count, int offs_bytes,
					   int vals_bytes)
{
	SVT_ARG(m != NULL && m->stage_cur >= 0,
		"svtgpu_matrix_commit_packed: no staged slot");
	const int vs = (int) svt_val_size(m->val_type);
	if (offs_bytes == 4 && vals_bytes == vs)
		return svtgpu_matrix_commit(m, dst, count);
	SVT_ARG(offs_bytes == 4 || (offs_bytes == 2 && m->nrow <= 65536) ||
		offs_bytes == SVTGPU_OFFS_U16_WRAPPED,
		"svtgpu_matrix_commit_packed: offsets can be 2 or 4 bytes (2 "
		"needs nrow <= 65536) or SVTGPU_OFFS_U16_WRAPPED");
	SVT_ARG(vals_bytes == vs || vals_bytes == 1,
		"svtgpu_matrix_commit_packed: values can be 1 byte or native");
	SVT_ARG(dst >= 0 && count >= 0 && dst + count <= m->nnz,
		"svtgpu_matrix_commit_packed: range outside [0, nnz]");
	const int s = m->stage_cur;
	SVT_CHECK(upload_begin(m));
	/* staging: [cap x 2 bytes offsets | cap x 1 byte values] per slot */
	const size_t need = (size_t) g_pool.cap * 3 + 256;
	if (m->narrow_bytes < need) {
		for (int i = 0; i < SVTGPU_NSTAGE; i++) {
			if (m->d_narrow[i] != NULL)
				SVT_CUDA(svt_free_async(m->d_narrow[i],
						       m->up_stream));
			m->d_narrow[i] = NULL;
			SVT_CUDA(svt_malloc_async(&m->d_narrow[i], need,
						 m->up_stream));
		}
		m->narrow_bytes = need;
	}
	char *stg = (char *) m->d_narrow[s];
	const size_t voff = ((size_t) g_pool.cap * 2 + 255) & ~(size_t) 255;
	const unsigned grid = (unsigned) (svtgpu_sm_count() * 8);
	if (count > 0 && (m->flags & SVTGPU_HAS_OFFS)) {
		if (offs_bytes == 2) {
			SVT_CUDA(cudaMemcpyAsync(stg, g_pool.offs[s],
					2 * (size_t) count,
					cudaMemcpyHostToDevice, m->up_stream));
			widen_u16_i32<<<grid, 256, 0, m->up_stream>>>(
				(const uint16_t *) stg, m->d_offs + dst, count);
			svtgpu_count_launch(1);
		} else if (offs_bytes == SVTGPU_OFFS_U16_WRAPPED) {
			SVT_CUDA(cudaMemcpyAsync(stg, g_pool.offs[s],
					2 * (size_t) count,
					cudaMemcpyHostToDevice, m->up_stream));
			widen_u16_wrapped<<<grid, 256, 0, m->up_stream>>>(
				(const uint16_t *) stg, m->d_offs,
				m->d_leaf_ptr, m->nleaf, dst, count);
			svtgpu_count_launch(1);
		} else {
			SVT_CUDA(cudaMemcpyAsync(m->d_offs + dst, g_pool.offs[s],
					4 * (size_t) count,
					cudaMemcpyHostToDevice, m->up_stream));
		}
		m->tm.h2d_bytes += (double) (offs_bytes ==
			SVTGPU_OFFS_U16_WRAPPED ? 2 : offs_bytes) * (double) count;
	}
	if (count > 0 && (m->flags & SVTGPU_HAS_VALS)) {
		if (vals_bytes == 1) {
			m->n_i8_commits++;
			SVT_CUDA(cudaMemcpyAsync(stg + voff, g_pool.vals[s],
					(size_t) count, cudaMemcpyHostToDevice,
					m->up_stream));
			if (vs == 4)
				widen_i8<int32_t><<<grid, 256, 0, m->up_stream>>>(
					(const int8_t *) (stg + voff),
					(int32_t *) m->d_vals + dst, count);
			else
				widen_i8<double><<<grid, 256, 0, m->up_stream>>>(
					(const int8_t *) (stg + voff),
					(double *) m->d_vals + dst, count);
			svtgpu_count_launch(1);
		} else {
			m->n_wide_commits++;
			SVT_CUDA(cudaMemcpyAsync((char *) m->d_vals +
					(size_t) vs * (size_t) dst,
					g_pool.vals[s], (size_t) vs * (size_t) count,
					cudaMemcpyHostToDevice, m->up_stream));
		}
		m->tm.h2d_bytes += (double) vals_bytes * (double) count;
	}
	SVT_CUDA(cudaGetLastError());
	/* the slot (host and device side) is free once the widening is done */
	SVT_CUDA(cudaEventRecord(g_pool.done[s], m->up_stream));
	g_pool.busy[s] = 1;
	m->stage_busy[s] = 1;
	m->stage_cur = -1;
	return SVTGPU_OK;
}

/* ---- compact copy: narrow the wide arrays in HBM (the mirror of widen_*) ----
 * Groups of 16 entries, cyclic over the grid: four 16-byte loads of values ->
 * one 16-byte store, four of offsets -> two.  Unaligned wide arrays (a caller
 * may wrap any pointer) take the scalar loop for everything. */
__device__ __forceinline__ uint32_t narrow_byte(int32_t x)
{
	return x == SVT_NA_INT ? (uint32_t) (uint8_t) SVT_COMPACT_NA_I8
			       : (uint32_t) (uint8_t) x;
}

__global__ void __launch_bounds__(256)
narrow_compact(const int32_t *__restrict__ offs,
	       const int32_t *__restrict__ vals, uint16_t *__restrict__ o16,
	       int8_t *__restrict__ v8, int64_t n, int vec)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	const int64_t t0 = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	const int64_t ng = vec ? n / 16 : 0;
	for (int64_t g = t0; g < ng; g += stride) {
		const int4 *qv = (const int4 *) vals + 4 * g;
		uint32_t w[4];
#pragma unroll
		for (int k = 0; k < 4; k++) {
			const int4 a = __ldcs(qv + k);
			w[k] = narrow_byte(a.x) | (narrow_byte(a.y) << 8) |
			       (narrow_byte(a.z) << 16) | (narrow_byte(a.w) << 24);
		}
		((uint4 *) v8)[g] = make_uint4(w[0], w[1], w[2], w[3]);
		if (o16 == NULL)
			continue;
		const int4 *qo = (const int4 *) offs + 4 * g;
		uint32_t h[8];
#pragma unroll
		for (int k = 0; k < 4; k++) {
			const int4 a = __ldcs(qo + k);
			h[2 * k] = ((uint32_t) a.x & 0xFFFFu) | ((uint32_t) a.y << 16);
			h[2 * k + 1] = ((uint32_t) a.z & 0xFFFFu) |
				       ((uint32_t) a.w << 16);
		}
		((uint4 *) o16)[2 * g] = make_uint4(h[0], h[1], h[2], h[3]);
		((uint4 *) o16)[2 * g + 1] = make_uint4(h[4], h[5], h[6], h[7]);
	}
	for (int64_t i = ng * 16 + t0; i < n; i += stride) {
		v8[i] = (int8_t) narrow_byte(vals[i]);
		if (o16 != NULL)
			o16[i] = (uint16_t) offs[i];
	}
}

void svt_drop_compact(svtgpu_matrix *m, cudaStream_t s)
{
	if (m->d_offs16 != NULL)
		svt_free_async(m->d_offs16, s);
	if (m->d_vals8 != NULL)
		svt_free_async(m->d_vals8, s);
	m->d_offs16 = NULL;
	m->d_vals8 = NULL;
	m->compact_state = SVT_COMPACT_NONE;
	m->compact_uses = 0;
}

int svt_ensure_compact(svtgpu_matrix *m, cudaStream_t s)
{
	if (m->compact_state != SVT_COMPACT_NONE)
		return SVTGPU_OK;
	if (svt_is_double(m->val_type) || !(m->flags & SVTGPU_HAS_VALS) ||
	    m->nnz == 0) {
		m->compact_state = SVT_COMPACT_INELIGIBLE;
		return SVTGPU_OK;
	}
	if (++m->compact_uses < 2)
		return SVTGPU_OK;
	SVT_CHECK(svtgpu_ensure_absmax(m, s));
	if (m->vmax_abs > SVT_COMPACT_MAX_ABS) {
		m->compact_state = SVT_COMPACT_INELIGIBLE;
		return SVTGPU_OK;
	}
	const bool want_offs = (m->flags & SVTGPU_HAS_OFFS) &&
			       m->nrow <= SVT_COMPACT_MAX_NROW;
	const size_t n = (size_t) m->nnz + SVT_COMPACT_PAD;
	cudaError_t e = svt_malloc_async((void **) &m->d_vals8, n, s);
	if (e == cudaSuccess && want_offs)
		e = svt_malloc_async((void **) &m->d_offs16, 2 * n, s);
	if (e == cudaErrorMemoryAllocation) {
		/* the wide arrays serve as before */
		cudaGetLastError();
		svt_drop_compact(m, s);
		m->compact_state = SVT_COMPACT_INELIGIBLE;
		return SVTGPU_OK;
	}
	SVT_CUDA(e);
	SVT_CUDA(cudaMemsetAsync(m->d_vals8 + m->nnz, 0, SVT_COMPACT_PAD, s));
	if (m->d_offs16 != NULL)
		SVT_CUDA(cudaMemsetAsync(m->d_offs16 + m->nnz, 0,
					 2 * SVT_COMPACT_PAD, s));
	const int vec = (((uintptr_t) m->d_vals) & 15) == 0 &&
			(m->d_offs16 == NULL || (((uintptr_t) m->d_offs) & 15) == 0);
	narrow_compact<<<(unsigned) (svtgpu_sm_count() * 8), 256, 0, s>>>(
		m->d_offs, (const int32_t *) m->d_vals, m->d_offs16, m->d_vals8,
		m->nnz, vec);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(1);
	/* later calls may come on other streams */
	SVT_CUDA(cudaStreamSynchronize(s));
	m->compact_state = SVT_COMPACT_BUILT;
	return SVTGPU_OK;
}

/* ---- tile table (svtgpu_internal.h) ---- */
__global__ void __launch_bounds__(256)
tile_leaves(const int64_t *__restrict__ leaf_ptr, int64_t nleaf, int64_t nnz,
	    int64_t tile, int64_t ntiles, int64_t *__restrict__ tile_leaf,
	    int *max_leaves, int pass)
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

int svt_ensure_tile_table(svtgpu_matrix *m, int64_t tile, cudaStream_t s)
{
	if (m->d_tile_leaf != NULL && m->tile_entries == tile)
		return SVTGPU_OK;
	if (m->d_tile_leaf != NULL)
		svt_free_async(m->d_tile_leaf, s);
	m->d_tile_leaf = NULL;
	m->tile_entries = 0;
	const int64_t ntiles = (m->nnz + tile - 1) / tile;
	SVT_CUDA(svt_malloc_async((void **) &m->d_tile_leaf,
				  8 * (size_t) (ntiles + 1) + 64, s));
	int *d_max = (int *) (m->d_tile_leaf + ntiles + 1);
	SVT_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int), s));
	const unsigned g = (unsigned) ((ntiles + 1 + 255) / 256);
	tile_leaves<<<g, 256, 0, s>>>(m->d_leaf_ptr, m->nleaf, m->nnz, tile,
				      ntiles, m->d_tile_leaf, d_max, 0);
	tile_leaves<<<g, 256, 0, s>>>(m->d_leaf_ptr, m->nleaf, m->nnz, tile,
				      ntiles, m->d_tile_leaf, d_max, 1);
	SVT_CUDA(cudaGetLastError());
	svtgpu_count_launch(2);
	int h_max = 0;
	SVT_CUDA(cudaMemcpyAsync(&h_max, d_max, sizeof(int),
				 cudaMemcpyDeviceToHost, s));
	SVT_CUDA(cudaStreamSynchronize(s));
	m->tile_entries = tile;
	m->tile_count = ntiles;
	m->tile_max_leaves = h_max;
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_compact_bytes(const svtgpu_matrix *m,
					   int64_t *bytes)
{
	SVT_ARG(m != NULL && bytes != NULL,
		"svtgpu_matrix_compact_bytes: NULL argument");
	const int64_t n = m->nnz + SVT_COMPACT_PAD;
	*bytes = (m->d_vals8 != NULL ? n : 0) + (m->d_offs16 != NULL ? 2 * n : 0);
	return SVTGPU_OK;
}

extern "C" int svtgpu_matrix_finish_upload(svtgpu_matrix *m)
{
	SVT_ARG(m != NULL, "svtgpu_matrix_finish_upload: NULL matrix");
	if (!m->owns || !m->up_begun)
		return SVTGPU_OK;
	SVT_CUDA(cudaEventRecord(m->up_end, m->up_stream));
	SVT_CUDA(cudaStreamSynchronize(m->up_stream));
	float ms = 0.f;
	SVT_CUDA(cudaEventElapsedTime(&ms, m->up_begin, m->up_end));
	m->tm.h2d_ms = (double) ms;
	m->up_begun = 0;
	for (int i = 0; i < SVTGPU_NSTAGE; i++) {
		if (m->stage_busy[i]) {
			g_pool.busy[i] = 0;
			m->stage_busy[i] = 0;
		}
	}
	return SVTGPU_OK;
}

static int is_pinned_host(const void *p)
{
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return a.type == cudaMemoryTypeHost;
}

extern "C" int svtgpu_matrix_upload(svtgpu_matrix *m, const int64_t *leaf_ptr,
				    const int32_t *offs, const void *vals)
{
	SVT_ARG(m != NULL && m->owns, "svtgpu_matrix_upload: matrix does not "
		"own its storage");
	SVT_ARG(leaf_ptr != NULL, "svtgpu_matrix_upload: NULL leaf_ptr");
	SVT_ARG(!(m->flags & SVTGPU_HAS_OFFS) || offs != NULL || m->nnz == 0,
		"svtgpu_matrix_upload: offs required");
	SVT_ARG(!(m->flags & SVTGPU_HAS_VALS) || vals != NULL || m->nnz == 0,
		"svtgpu_matrix_upload: vals required");
	SVT_CHECK(svtgpu_matrix_set_leaf_ptr(m, leaf_ptr));
	const size_t vs = svt_val_size(m->val_type);
	const int want_offs = (m->flags & SVTGPU_HAS_OFFS) != 0;
	const int want_vals = (m->flags & SVTGPU_HAS_VALS) != 0;
	/* caller-pinned arrays go straight to the copy engine */
	const int direct = m->nnz > 0 &&
		(!want_offs || is_pinned_host(offs)) &&
		(!want_vals || is_pinned_host(vals));
	if (direct) {
		if (want_offs) {
			SVT_CUDA(cudaMemcpyAsync(m->d_offs, offs,
					sizeof(int32_t) * (size_t) m->nnz,
					cudaMemcpyHostToDevice, m->up_stream));
			m->tm.h2d_bytes += 4.0 * (double) m->nnz;
		}
		if (want_vals) {
			SVT_CUDA(cudaMemcpyAsync(m->d_vals, vals,
					vs * (size_t) m->nnz,
					cudaMemcpyHostToDevice, m->up_stream));
			m->tm.h2d_bytes += (double) vs * (double) m->nnz;
		}
		return svtgpu_matrix_finish_upload(m);
	}
	int64_t cap = 0;
	if (m->nnz > 0)
		SVT_CHECK(svtgpu_matrix_stage_capacity(m, &cap));
	for (int64_t e0 = 0; e0 < m->nnz; e0 += cap) {
		int64_t n = m->nnz - e0 < cap ? m->nnz - e0 : cap;
		int32_t *so = NULL;
		void *sv = NULL;
		SVT_CHECK(svtgpu_matrix_stage(m, n, &so, &sv));
		if (want_offs)
			memcpy(so, offs + e0, sizeof(int32_t) * (size_t) n);
		if (want_vals)
			memcpy(sv, (const char *) vals + vs * (size_t) e0,
			       vs * (size_t) n);
		SVT_CHECK(svtgpu_matrix_commit(m, e0, n));
	}
	return svtgpu_matrix_finish_upload(m);
}

/* ---- scratch ---- */

int svtgpu_scratch(svtgpu_matrix *m, size_t bytes, void **ptr)
{
	if (bytes > m->scratch_bytes) {
		/* stream 0 is ordered against every blocking stream */
		if (m->d_scratch != NULL)
			SVT_CUDA(svt_free_async(m->d_scratch, 0));
		m->d_scratch = NULL;
		m->scratch_bytes = 0;
		SVT_CUDA(svt_malloc_async(&m->d_scratch, bytes, 0));
		m->scratch_bytes = bytes;
	}
	*ptr = m->d_scratch;
	return SVTGPU_OK;
}

/* ---- exclusive scan (leaf counts -> leaf_ptr), used by the generators ---- */

extern "C" int svtgpu_exclusive_scan(const int64_t *d_in, int64_t n,
				     int64_t *d_out, void *stream)
{
	SVT_CHECK(svtgpu_require_device());
	cudaStream_t s = (cudaStream_t) stream;
	SVT_ARG(n >= 0 && n < INT32_MAX, "svtgpu_exclusive_scan: n too large");
	/* d_out has n+1 entries: scan n+1 items whose last input is ignored by
	   using an inclusive scan shifted by one. */
	SVT_CUDA(cudaMemsetAsync(d_out, 0, sizeof(int64_t), s));
	if (n == 0)
		return SVTGPU_OK;
	void *tmp = NULL;
	size_t tmp_bytes = 0;
	SVT_CUDA(cub::DeviceScan::InclusiveSum(NULL, tmp_bytes, d_in, d_out + 1,
					       (int) n, s));
	SVT_CUDA(svt_malloc_async(&tmp, tmp_bytes, s));
	SVT_CUDA(cub::DeviceScan::InclusiveSum(tmp, tmp_bytes, d_in, d_out + 1,
					       (int) n, s));
	SVT_CUDA(svt_free_async(tmp, s));
	svtgpu_count_launch(2);
	return SVTGPU_OK;
}
