// Ceiling of the compact column sums: a read-only stream of 2.35 GB of int8
// (the C2 compact values) in 32 KB tiles that the CTAs take round-robin
// (CTA b takes tiles b, b + grid, ...), each 16-byte word summed with
// __dp4a.  Three ways to bring a tile in:
//   ring   1-D bulk async copies into a ring of NS shared-memory stages fed by
//          one producer lane, drained by W consumer warps (mbarriers full /
//          empty per stage), CPS CTAs per SM;
//   reg    16-byte register loads of the tile, every load of a thread in
//          flight before the first add (256 threads, 8 words each);
//   int4   the plain grid-stride int4 loop of stream_width.cu.
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tile_ring tile_ring.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "../../sparsearray_b200/csrc/svt_ptx.cuh"

#define TILE 32768

__device__ __forceinline__ int sum16(uint4 u, int s)
{
	s = __dp4a((int) u.x, 0x01010101, s);
	s = __dp4a((int) u.y, 0x01010101, s);
	s = __dp4a((int) u.z, 0x01010101, s);
	return __dp4a((int) u.w, 0x01010101, s);
}

template <int NS, int W>
__global__ void __launch_bounds__((W + 1) * 32)
ring(const int8_t *v, int64_t n, int *sink)
{
	extern __shared__ __align__(128) unsigned char smem[];
	uint64_t *bars = (uint64_t *) (smem + (size_t) NS * TILE);
	const uint32_t full0 = svt_smem_u32(bars), empty0 = full0 + 8 * NS;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	if (threadIdx.x == 0) {
		for (int i = 0; i < NS; i++) {
			svt_mbar_init(full0 + 8 * i, 1);
			svt_mbar_init(empty0 + 8 * i, W);
		}
		svt_mbar_init_fence();
	}
	__syncthreads();
	const int64_t ntiles = (n + TILE - 1) / TILE;
	if (warp == W) {
		if (lane != 0)
			return;
		const uint64_t pol = svt_policy_evict_first();
		uint32_t j = 0;
		for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, j++) {
			const int st = j % NS;
			svt_mbar_wait(empty0 + 8 * st, ((j / NS) & 1) ^ 1);
			int64_t bytes = n - t * TILE;
			bytes = bytes > TILE ? TILE : (bytes + 15) & ~15;
			svt_mbar_arrive_expect_tx(full0 + 8 * st, (uint32_t) bytes);
			svt_bulk_g2s_hint(svt_smem_u32(smem + (size_t) st * TILE),
					  v + t * TILE, (uint32_t) bytes,
					  full0 + 8 * st, pol);
		}
		return;
	}
	int s = 0;
	uint32_t j = 0;
	for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, j++) {
		const int st = j % NS;
		svt_mbar_wait(full0 + 8 * st, (j / NS) & 1);
		const uint4 *q = (const uint4 *) (smem + (size_t) st * TILE);
#pragma unroll 4
		for (int i = threadIdx.x; i < TILE / 16; i += W * 32)
			s = sum16(q[i], s);
		__syncwarp();
		if (lane == 0)
			svt_mbar_arrive(empty0 + 8 * st);
	}
	if (s == 0x12345678) *sink = s;
}

__global__ void __launch_bounds__(256)
reg(const int8_t *v, int64_t n, int *sink)
{
	const int64_t ntiles = n / TILE;
	int s = 0;
	for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
		const uint4 *q = (const uint4 *) (v + t * TILE) + threadIdx.x;
		uint4 u[8];
#pragma unroll
		for (int k = 0; k < 8; k++) u[k] = __ldcs(q + 256 * k);
#pragma unroll
		for (int k = 0; k < 8; k++) s = sum16(u[k], s);
	}
	if (s == 0x12345678) *sink = s;
}

__global__ void __launch_bounds__(256)
plain(const uint4 *p, int64_t n, int *sink)
{
	int s = 0;
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	for (; i + 3 * stride < n; i += 4 * stride) {
		uint4 u[4];
#pragma unroll
		for (int k = 0; k < 4; k++) u[k] = p[i + k * stride];
#pragma unroll
		for (int k = 0; k < 4; k++) s = sum16(u[k], s);
	}
	if (s == 0x12345678) *sink = s;
}

static float best_of(void (*launch)(const int8_t *, int64_t, int *, int),
		     const int8_t *v, int64_t n, int *sink, int arg)
{
	cudaEvent_t a, b;
	cudaEventCreate(&a);
	cudaEventCreate(&b);
	launch(v, n, sink, arg);   /* warm-up */
	float best = 1e9f;
	for (int rep = 0; rep < 7; rep++) {
		cudaEventRecord(a);
		launch(v, n, sink, arg);
		cudaEventRecord(b);
		cudaEventSynchronize(b);
		float ms;
		cudaEventElapsedTime(&ms, a, b);
		if (ms < best) best = ms;
	}
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) {
		printf("error: %s\n", cudaGetErrorString(e));
		return -1.0f;
	}
	return best;
}

static int sms;

template <int NS, int W>
static void launch_ring(const int8_t *v, int64_t n, int *sink, int cps)
{
	const size_t smem = (size_t) NS * TILE + 16 * NS;
	cudaFuncSetAttribute(ring<NS, W>,
			     cudaFuncAttributeMaxDynamicSharedMemorySize,
			     (int) smem);
	ring<NS, W><<<sms * cps, (W + 1) * 32, smem>>>(v, n, sink);
}

template <int NS, int W>
static void report_ring(const int8_t *v, int64_t n, int *sink, int cps)
{
	if ((size_t) cps * (NS * TILE + 16 * NS) > 227 * 1024)
		return;
	const float ms = best_of(launch_ring<NS, W>, v, n, sink, cps);
	printf("ring  stages %d  consumer warps %2d  CTAs/SM %d   %.3f ms  %5.0f GB/s\n",
	       NS, W, cps, ms, n / ms / 1e6);
}

static void launch_reg(const int8_t *v, int64_t n, int *sink, int cps)
{
	reg<<<sms * cps, 256>>>(v, n, sink);
}

static void launch_plain(const int8_t *v, int64_t n, int *sink, int bps)
{
	plain<<<sms * bps, 256>>>((const uint4 *) v, n / 16, sink);
}

template <int W>
static void sweep_stages(const int8_t *v, int64_t n, int *sink)
{
	for (int cps = 1; cps <= 2; cps++) {
		report_ring<2, W>(v, n, sink, cps);
		report_ring<3, W>(v, n, sink, cps);
		report_ring<4, W>(v, n, sink, cps);
		report_ring<6, W>(v, n, sink, cps);
	}
}

int main()
{
	const int64_t n = 2348000000LL / TILE * TILE;   /* C2: nnz = 2.348e9 */
	int8_t *v;
	int *sink;
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
	cudaMalloc(&v, n + 64);
	cudaMalloc(&sink, 4);
	cudaMemset(v, 1, n + 64);
	cudaDeviceProp p;
	cudaGetDeviceProperties(&p, 0);
	printf("%s, %d SMs, %.3f GB of int8\n", p.name, sms, n / 1e9);
	for (int bps = 4; bps <= 8; bps += 4) {
		const float ms = best_of(launch_plain, v, n, sink, bps);
		printf("int4  x4  %d CTAs/SM of 256                  %.3f ms  %5.0f GB/s\n",
		       bps, ms, n / ms / 1e6);
	}
	for (int cps = 4; cps <= 8; cps += 4) {
		const float ms = best_of(launch_reg, v, n, sink, cps);
		printf("reg   8 x 16 B per thread, %d CTAs/SM of 256   %.3f ms  %5.0f GB/s\n",
		       cps, ms, n / ms / 1e6);
	}
	sweep_stages<4>(v, n, sink);
	sweep_stages<8>(v, n, sink);
	sweep_stages<16>(v, n, sink);
	cudaFree(v);
	cudaFree(sink);
	return 0;
}
