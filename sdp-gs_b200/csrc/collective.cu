// b200gs -- two-shot SUM all-reduce over NVLink peer memory (include/b200gs_collective.h).
//
// Algorithmic bytes per rank: reads world * n/world * 4 (own slice from every rank) + writes world * n/world * 4
// = 8n bytes over NVLink/NVSwitch for n floats, against 2 * (world-1)/world * 4n for a ring: the same wire traffic,
// but one kernel, two block-level barriers and no intermediate buffers.  With an NVLS multicast mapping the switch
// performs the reduction (multimem.ld_reduce) and the broadcast (multimem.st): 4n/world read + 4n/world written per rank.
#include <type_traits>
#include "common.cuh"
#include "../../include/b200gs_collective.h"

int train_fail(int code, const char* msg);  // api.cu

namespace {

constexpr int AR_BLOCKS = 256;   // maximum grid (sizes the flag array); the launch uses AR_GRID
constexpr int AR_GRID = 64;      // measured flat between 16 and 128 blocks (the wire is the bound), slower at 256
// float4 per thread and step = 16 / world: ~16 NVLink requests per thread in flight cover the remote-load latency
constexpr int AR_THREADS = 512;
constexpr int AR_MAX_WORLD = 8;

// One-way epoch flags: a rank announces itself by STORING the launch's epoch into its slot of every peer's flag array
// (a posted NVLink write -- no round trip, unlike the compare-and-swap handshake this replaced) and waits, spinning on
// its own memory, until every peer's slot shows the same epoch.  The epoch is a per-block launch counter kept in the
// rank's own flag array (every rank launches the same sequence of collectives with the same grid, so the counters
// agree); it lives in device memory, so a captured CUDA graph replays correctly.  A peer is never more than one
// barrier ahead (it needs this rank's store to get any further), and the two barriers of a launch use separate slots.
__device__ __forceinline__ void st_flag(uint32_t* addr, uint32_t v) {
	asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(addr), "r"(v) : "memory");  // ordered by the system fence before it
}
__device__ __forceinline__ uint32_t ld_flag(const uint32_t* addr) {
	uint32_t v;
	asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(addr) : "memory");  // the system fence after the spin orders what follows
	return v;
}
__device__ __forceinline__ uint32_t* epoch_word(void* const* flags, int rank) {
	return reinterpret_cast<uint32_t*>(flags[rank]) + (size_t)2 * AR_BLOCKS * AR_MAX_WORLD + blockIdx.x;
}

// Block b of every rank meets block b of every other rank.  Slot layout of a rank's flag array: [phase][block][source rank],
// then one launch counter per block.
__device__ __forceinline__ void block_barrier(void* const* flags, int rank, int world, int phase, uint32_t epoch) {
	__syncthreads();
	if ((int)threadIdx.x < world) {
		const int peer = threadIdx.x;
		__threadfence_system();  // everything this block wrote (observed through the barrier above) is ordered before the flag
		uint32_t* theirs = reinterpret_cast<uint32_t*>(flags[peer]) + ((size_t)phase * AR_BLOCKS + blockIdx.x) * AR_MAX_WORLD + rank;
		const uint32_t* mine = reinterpret_cast<uint32_t*>(flags[rank]) + ((size_t)phase * AR_BLOCKS + blockIdx.x) * AR_MAX_WORLD + peer;
		st_flag(theirs, epoch);
		while (ld_flag(mine) != epoch) {}
		__threadfence_system();
	}
	__syncthreads();
}

template <int WORLD>
__global__ void __launch_bounds__(AR_THREADS) allreduce_p2p_kernel(void* const* __restrict__ bufs, void* const* __restrict__ flags,
                                                                    int64_t off4, int64_t n4, int rank)
{
	__shared__ void* s_flags[AR_MAX_WORLD];
	float4* p[WORLD];
#pragma unroll
	for (int r = 0; r < WORLD; r++) p[r] = reinterpret_cast<float4*>(bufs[r]) + off4;
	if ((int)threadIdx.x < WORLD) s_flags[threadIdx.x] = flags[threadIdx.x];
	__syncthreads();
	const uint32_t epoch = *epoch_word(s_flags, rank) + 1u;
	block_barrier(s_flags, rank, WORLD, 0, epoch);  // every rank's producer kernels have finished (stream order) before its flags go up
	const int64_t per = (n4 + WORLD - 1) / WORLD;
	const int64_t lo = per * rank, hi = min(n4, lo + per);
	constexpr int AR_UNROLL = WORLD <= 2 ? 8 : (WORLD <= 4 ? 4 : 2);
	const int64_t stride = (int64_t)gridDim.x * AR_THREADS;
	for (int64_t i0 = lo + (int64_t)blockIdx.x * AR_THREADS + threadIdx.x; i0 < hi; i0 += stride * AR_UNROLL) {
		float4 v[AR_UNROLL][WORLD];
#pragma unroll
		for (int u = 0; u < AR_UNROLL; u++) {
			const int64_t i = i0 + u * stride;
#pragma unroll
			for (int r = 0; r < WORLD; r++) v[u][r] = i < hi ? __ldcg(p[r] + i) : make_float4(0.f, 0.f, 0.f, 0.f);  // all loads in flight first
		}
#pragma unroll
		for (int u = 0; u < AR_UNROLL; u++) {
			const int64_t i = i0 + u * stride;
			float4 a = v[u][0];  // fixed-order sum: identical on every rank
#pragma unroll
			for (int r = 1; r < WORLD; r++) { a.x += v[u][r].x; a.y += v[u][r].y; a.z += v[u][r].z; a.w += v[u][r].w; }
			if (i < hi) {
#pragma unroll
				for (int r = 0; r < WORLD; r++) __stcg(p[r] + i, a);
			}
		}
	}
	block_barrier(s_flags, rank, WORLD, 1, epoch);  // every slice has landed everywhere
	if (threadIdx.x == 0) *epoch_word(s_flags, rank) = epoch;
}

__global__ void __launch_bounds__(AR_THREADS) allreduce_multimem_kernel(void* const* __restrict__ flags, float4* mc, int64_t off4, int64_t n4,
                                                                         int rank, int world)
{
	__shared__ void* s_flags[AR_MAX_WORLD];
	if ((int)threadIdx.x < world) s_flags[threadIdx.x] = flags[threadIdx.x];
	__syncthreads();
	const uint32_t epoch = *epoch_word(s_flags, rank) + 1u;
	block_barrier(s_flags, rank, world, 0, epoch);
	const int64_t per = (n4 + world - 1) / world;
	const int64_t lo = per * rank, hi = min(n4, lo + per);
	for (int64_t i = lo + (int64_t)blockIdx.x * AR_THREADS + threadIdx.x; i < hi; i += (int64_t)gridDim.x * AR_THREADS) {
		float4 a;
		float4* addr = mc + off4 + i;
		asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
		             : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "l"(addr) : "memory");
		asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(addr), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w) : "memory");
	}
	block_barrier(s_flags, rank, world, 1, epoch);
	if (threadIdx.x == 0) *epoch_word(s_flags, rank) = epoch;
}

// Gather half of the fused gradient exchange (include/b200gs_collective.h: b200gs_gather_reduce_f32).
template <int WORLD>
__global__ void __launch_bounds__(AR_THREADS) gather_reduce_kernel(void* const* __restrict__ staging, void* const* __restrict__ outs,
                                                                    void* const* __restrict__ flags, int64_t Ps, int rank)
{
	__shared__ void* s_flags[AR_MAX_WORLD];
	float4* out[WORLD];
#pragma unroll
	for (int r = 0; r < WORLD; r++) out[r] = reinterpret_cast<float4*>(outs[r]);
	const float4* st = reinterpret_cast<const float4*>(staging[rank]);
	if ((int)threadIdx.x < WORLD) s_flags[threadIdx.x] = flags[threadIdx.x];
	pdl_trigger();
	pdl_wait();  // this rank's own pushes (the backward kernel just before) are complete
	__syncthreads();
	const uint32_t epoch = *epoch_word(s_flags, rank) + 1u;
	block_barrier(s_flags, rank, WORLD, 0, epoch);  // ... and so are everybody else's
	const int64_t Pp4 = Ps * WORLD / 4, Ps4 = Ps / 4;  // Ps % 128 == 0
	const int64_t n4 = Ps4 * 62, src_stride4 = Ps4 * 64;
	constexpr int UNROLL = WORLD <= 2 ? 4 : 2;
	const int64_t stride = (int64_t)gridDim.x * AR_THREADS;
	for (int64_t i0 = (int64_t)blockIdx.x * AR_THREADS + threadIdx.x; i0 < n4; i0 += stride * UNROLL) {
		float4 v[UNROLL][WORLD];
#pragma unroll
		for (int u = 0; u < UNROLL; u++) {
			const int64_t i = i0 + u * stride;
#pragma unroll
			for (int r = 0; r < WORLD; r++) v[u][r] = i < n4 ? __ldcg(st + r * src_stride4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
		}
#pragma unroll
		for (int u = 0; u < UNROLL; u++) {
			const int64_t i = i0 + u * stride;
			if (i >= n4) continue;
			float4 a = v[u][0];  // fixed-order sum: identical on every rank
#pragma unroll
			for (int r = 1; r < WORLD; r++) { a.x += v[u][r].x; a.y += v[u][r].y; a.z += v[u][r].z; a.w += v[u][r].w; }
			// segment of staging index i (float4 units of one shard): c * Ps4 <= i < (c + w) * Ps4
			const int64_t q = i / Ps4;  // == floats-per-Gaussian offset the index falls into
			const int c = q < 3 ? 0 : (q < 51 ? 3 : (q < 52 ? 51 : (q < 55 ? 52 : (q < 59 ? 55 : 59))));
			const int w = q < 3 ? 3 : (q < 51 ? 48 : (q < 52 ? 1 : (q < 55 ? 3 : (q < 59 ? 4 : 3))));
			const int64_t o = (int64_t)c * Pp4 + (int64_t)rank * Ps4 * w + (i - (int64_t)c * Ps4);
#pragma unroll
			for (int r = 0; r < WORLD; r++) __stcg(out[r] + o, a);
		}
	}
	block_barrier(s_flags, rank, WORLD, 1, epoch);  // every shard has landed everywhere
	if (threadIdx.x == 0) *epoch_word(s_flags, rank) = epoch;
}

// Launches f(std::integral_constant<int, WORLD>) for WORLD = world, 2 <= world <= AR_MAX_WORLD.
template <int WORLD = 2, typename F>
cudaError_t launch_for_world(int world, F&& f) {
	if constexpr (WORLD < AR_MAX_WORLD) {
		if (world > WORLD) return launch_for_world<WORLD + 1>(world, f);
	}
	return f(std::integral_constant<int, WORLD>{});
}

}  // namespace

extern "C" {

size_t b200gs_allreduce_flag_words(int32_t world) { (void)world; return (size_t)2 * AR_BLOCKS * AR_MAX_WORLD + AR_BLOCKS; }

int b200gs_allreduce_sum_f32(void* const* buffers_dev, void* const* flags_dev, void* multicast_ptr, int64_t offset_floats,
                             int64_t n_floats, int32_t rank, int32_t world, void* stream_) {
	if (!buffers_dev || !flags_dev || world < 1 || world > AR_MAX_WORLD || rank < 0 || rank >= world || n_floats < 0 ||
	    (n_floats & 3) || (offset_floats & 3))
		return train_fail(B200GS_E_ARG, "allreduce_sum_f32: bad arguments (world <= 8, offset and n multiples of 4)");
	if (world == 1 || n_floats == 0) return 0;
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	const int64_t n4 = n_floats / 4, off4 = offset_floats / 4;
	if (multicast_ptr)
		return launch_status(launch(0u, allreduce_multimem_kernel, dim3(AR_GRID), dim3(AR_THREADS), 0, stream, flags_dev,
		                            reinterpret_cast<float4*>(multicast_ptr), off4, n4, rank, world));
	return launch_status(launch_for_world(world, [&](auto w) {
		return launch(0u, allreduce_p2p_kernel<decltype(w)::value>, dim3(AR_GRID), dim3(AR_THREADS), 0, stream, buffers_dev, flags_dev, off4, n4, rank);
	}));
}

int b200gs_gather_reduce_f32(void* const* staging_dev, void* const* out_dev, void* const* flags_dev, int64_t shard_rows,
                             int32_t rank, int32_t world, int32_t chained, void* stream_) {
	if (!staging_dev || !out_dev || !flags_dev || world < 2 || world > AR_MAX_WORLD || rank < 0 || rank >= world || shard_rows <= 0 ||
	    (shard_rows & 127))
		return train_fail(B200GS_E_ARG, "gather_reduce_f32: bad arguments (2 <= world <= 8, shard_rows a positive multiple of 128)");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	return launch_status(launch_for_world(world, [&](auto w) {
		return launch(chained ? PDL_TRAIN : 0u, gather_reduce_kernel<decltype(w)::value>, dim3(AR_GRID), dim3(AR_THREADS), 0, stream, staging_dev,
		              out_dev, flags_dev, shard_rows, rank);
	}));
}

}  // extern "C"
