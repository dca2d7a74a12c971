// b200gs -- shared declarations for the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/b200gs.h"

#define TILE_X 16  // tile geometry of the reference (DGR/cuda_rasterizer/config.h:16-17); part of the
#define TILE_Y 16  // bit-exact contract (tile rects, sort keys, tile ranges)
#define TILE_PIX (TILE_X * TILE_Y)

// Per-Gaussian "splat record": everything the blend kernels need, packed into 64 bytes so that a
// tile's gather touches exactly two fully-used 32-B sectors per Gaussian.
//   g0 = {x, y, conic.a, conic.b}
//   g1 = {conic.c, opacity, cull_thr (= 2 ln(255 o)), -b/c}      g0+g1: all a cull test and `power` need (one sector)
//   g2 = {r, g, b, z_view}                                       payload, only touched by Gaussians that survive the cull
//   g3 = {f0, f1, f2, 0}                                         (SDP-GS feature head)
#define REC_FLOATS 16
// Per-Gaussian gradient record accumulated by the blend backward (64 bytes):
//   {dmean2D.x, dmean2D.y, dconic.a, dconic.b | dconic.c, dopacity, -, - | dr, dg, db, dz | df0, df1, df2, -}
// (first half: pixel moments of G*dL/dG, second half: channel sums of alpha*T -- written by different half-warps)
#define GREC_FLOATS 16

struct GeomHeader {  // first 256 bytes of the geom workspace
	unsigned long long num_rendered;  // inclusive-scan total of tiles touched: ASSIGNED by scan_emit's last tile (never needs zeroing)
	unsigned int overflow;            // bit 0: num_rendered > binning capacity, bit 1: prefilter violation; assigned with num_rendered
	unsigned int scan_ticket;         // dynamic tile id allocator for the look-back scan
	unsigned int sort_ticket[8];      // one per radix pass (4 depth passes + up to 4 tile passes)
	unsigned int ranges_done;         // CTAs of the tile-ranges kernel that have finished (last one builds the blend schedule)
	unsigned int emit_done;           // CTAs of scan_emit that have finished (last one turns tile counts into ranges + schedule)
	unsigned int blend_ticket[2];     // next blend unit to hand out (forward, backward): persistent warps draw from it
	unsigned int blend_exit[2];       // warps that have run dry; the last one re-arms ticket and counter
	unsigned long long num_acc;       // instance count accumulated by the preprocess kernel (num_rendered is assigned from the scan)
	unsigned int prefilter_violation; // 2 when a Gaussian was culled although `prefiltered` was set
	unsigned int sort_barrier[2];     // grid barriers of the fused multi-pass sorts (depth, tile)
	unsigned int pad[41];
};
static_assert(sizeof(GeomHeader) == 256, "header size");

struct GeomState {
	GeomHeader* hdr;
	float* depths;           // f32[P]
	ushort4* rect;           // (x0,y0,x1,y1) tile rect per Gaussian; all-zero when culled
	float4* rec;             // [P][4] float4 records
	uint8_t* clamped;        // u8[P]
	uint32_t* order;         // u32[P]  depth-sorted Gaussian ids (final sort output)
	uint32_t* key_a;         // depth-sort ping-pong
	uint32_t* key_b;
	uint32_t* val_b;         // (val_a aliases `order`)
	uint32_t* hist;          // [8][256] global digit histograms (4 depth passes, up to 4 tile passes)
	uint32_t* lookback;      // [tiles_P][256] onesweep look-back words, reused by every depth pass
	unsigned long long* scan_state;  // [scan_tiles] look-back words of the offsets scan
	size_t clean_bytes;      // [hdr .. scan_state]: zero at the start of every forward
	size_t bytes;
};

struct ImageState {
	float* final_T;        // f32[N]
	uint32_t* n_contrib;   // u32[N]
	uint2* ranges;         // [tiles]
	uint32_t* tile_order;  // [tiles] tile ids, heaviest (longest range) first: launch order of the blend units
	uint32_t* tile_count;  // [tiles] instances per tile, counted while they are emitted (zeroed by the preprocess kernel)
	// Persistent workspaces only (a session renders the same view again and again): what the blend units of each tile cost the
	// last time -- [0][t] forward, [1][t] backward, in units of (rounds walked, survivors blended) -- accumulated by the blend
	// kernels and consumed (and zeroed) by the next call's schedule builder, which then orders the tiles by measured cost
	// instead of list length (the two correlate poorly: long lists saturate early).  Zero = no history.
	uint32_t* tile_cost;       // [2][tiles]
	uint32_t* tile_order_bwd;  // [tiles] launch order of the backward's units
	size_t bytes;
};
// Tile grids of at most COUNT_TILES_MAX tiles take scan_emit's TILE_COUNTS path (binning.cu): its last CTA builds the tile
// ranges and blend orders from ImageState::tile_count, which holds one counter every COUNT_STRIDE words.
constexpr int COUNT_TILES_MAX = 2048;
constexpr int COUNT_STRIDE = 32;  // words between two tiles' global counters

struct BinningState {
	uint32_t* key_a;  // tile ids, ping
	uint32_t* key_b;  // pong
	uint32_t* val_a;  // Gaussian ids, ping
	uint32_t* val_b;  // pong
	uint32_t* lookback;  // [tiles_L][256]
	uint32_t* sorted_vals;  // == point_list after the tile sort (val_a or val_b depending on pass parity)
	uint32_t* sorted_keys;
	// Survivor bitmap, [8 sub-blocks][surv_words]: bit (i & 31) of word (range.x >> 5) + tile + (i >> 5) of plane s says whether
	// list entry i of the tile survived the conservative cull of 8x4 pixel block s.  Written by the blend forward (the ballot of
	// every round it stages), read by the blend backward instead of fetching and culling the entry again.  The words of two
	// tiles never collide: ranges are ordered by tile id and (x' >> 5) + t' >= (x >> 5) + floor(n / 32) + t + 1.
	uint32_t* surv_bits;
	size_t surv_words;
	size_t bytes;
};

// Radix sort tiling: 256 threads x ITEMS items per CTA tile.
#define SORT_THREADS 256
#ifndef SORT_ITEMS_SMALL
#define SORT_ITEMS_SMALL 4
#endif
#define SORT_ITEMS_LARGE 16
static inline int sort_items_for(int64_t n) { return n <= (1 << 20) ? SORT_ITEMS_SMALL : SORT_ITEMS_LARGE; }
static inline int64_t sort_tiles_for(int64_t n) {
	int64_t per = (int64_t)SORT_THREADS * sort_items_for(n);
	return (n + per - 1) / per;
}
#define SCAN_THREADS 1024       // Gaussians per CTA of scan_emit_kernel (one per thread) ...
#define SCAN_THREADS_SMALL 256  // ... and for small Gaussian counts (more CTAs to spread the emission over)
#define SCAN_SMALL_MAX 32768
#define SCAN_ITEMS 1
static inline int scan_threads_for(int64_t n) { return n <= SCAN_SMALL_MAX ? SCAN_THREADS_SMALL : SCAN_THREADS; }
static inline int64_t scan_tiles_for(int64_t n) { const int t = scan_threads_for(n); return (n + t - 1) / t; }

// The 16x16 tile grid of one view and everything the stages derive from it.
struct TileGrid {
	int W, H;
	uint32_t gx, gy, units;  // units: 8 blend units per tile
	size_t tiles;
	int tile_bits, tile_passes;  // key bits of the tile sort (getHigherMsb(tiles), rasterizer_impl.cu:35-50) and its radix passes
	bool ranges_from_emit;       // tiles <= COUNT_TILES_MAX: scan_emit's last CTA builds the ranges and blend orders
	bool list_in_b;              // odd pass count: the sorted list ends in BinningState::key_b / val_b
};
TileGrid tile_grid(int W, int H);

GeomState geom_from_chunk(char* base, int P);
ImageState image_from_chunk(char* base, const TileGrid& t);
BinningState binning_from_chunk(char* base, const TileGrid& t, int64_t capacity);  // sorted_keys / sorted_vals per t.list_in_b

// What one rasterizer call works on, derived once from its arguments and handed to every stage launcher.
struct RasterPlan {
	const b200gs_view_t* v;
	TileGrid grid;
	int P;
	int64_t capacity;
	bool persistent;  // the workspaces persist across calls: blend units ordered by (and recording) ImageState::tile_cost
	GeomState gs;
	ImageState is;
	BinningState bs;
};

// ---- stage launchers (each enqueues on `stream`) ----
void launch_preprocess_forward(const RasterPlan& pl, const b200gs_gaussians_t& g, int32_t* radii, cudaStream_t stream);
// cam != NULL: also the camera gradients (a second, small kernel reduces the per-CTA partials in cam->scratch)
void launch_preprocess_backward(const RasterPlan& pl, const b200gs_gaussians_t& g, const int32_t* radii, float* grec,
                                const b200gs_grads_t& gr, const b200gs_camera_grads_t* cam, cudaStream_t stream);
size_t camera_scratch_bytes(int P);
void launch_mark_visible(int P, const float* means3D, const float* viewmatrix, uint8_t* present, cudaStream_t stream);

void launch_depth_order(const RasterPlan& pl, cudaStream_t stream);  // stable sort of Gaussian ids by depth bits
void launch_scan_emit(const RasterPlan& pl, cudaStream_t stream, bool chained /* the previous kernel in the stream is our depth sort */);
void launch_tile_sort(const RasterPlan& pl, cudaStream_t stream);
void launch_tile_ranges(const RasterPlan& pl, int64_t n_max /* 0: nothing was emitted */, cudaStream_t stream);
void launch_finalize_header(const RasterPlan& pl, cudaStream_t stream);
void launch_debug_keys(const RasterPlan& pl, uint64_t* keys_out, int64_t L, cudaStream_t stream);
// Stable LSD radix sort of (u32 key, u32 value) pairs on key bits [0, end_bit) (binning.cu); n is read from *n_dev (clamped to
// n_max) when n_dev != nullptr, else n = n_max.  The result is in (key_a, val_a) after an even number of passes, else in
// (key_b, val_b).  hist[p][256]: the digit counts of pass p, produced by the kernel that wrote the keys.  lookback
// ([passes][sort_tiles_for(n_max)][256] words), tickets[passes] and *barrier must be zero on entry.
void launch_radix_sort(uint32_t* key_a, uint32_t* key_b, uint32_t* val_a, uint32_t* val_b, int64_t n_max,
                       const unsigned long long* n_dev, int end_bit, uint32_t* hist, uint32_t* lookback,
                       unsigned int* tickets, unsigned int* barrier, cudaStream_t stream);

void launch_blend_forward(const RasterPlan& pl, const b200gs_outputs_t& out, cudaStream_t stream);  // also writes bs.surv_bits
void launch_blend_backward(const RasterPlan& pl, const b200gs_grad_outputs_t& gout, float* grec, cudaStream_t stream);

// Environment knobs, each read once, when first asked for: the value, or nullptr / `unset` when the variable is not set.
enum Knob { KNOB_PDL, KNOB_BLEND_WIDE, KNOB_BLEND_CTAS, KNOB_SCATTER_TMA, KNOB_COUNT };
const char* knob(Knob k);
int knob_int(Knob k, int unset);

// 0 after a successful launch (`e`, then cudaGetLastError), else B200GS_E_CUDA with the error's name as the last error
int launch_status(cudaError_t e);
void count_launch();

// ---- device helpers ----
#ifdef __CUDACC__
// Programmatic dependent launch (sm_90+): every kernel of the chain is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization (launch() below).  pdl_trigger() lets the NEXT kernel's CTAs
// become resident while this one is still running; pdl_wait() blocks until every earlier kernel in the stream
// has completed and its writes are visible.  Rule used throughout: trigger first, touch only shared memory
// and registers, then wait before the first global access.  Without the launch attribute both are no-ops.
// Data produced by an earlier kernel of the chain must NOT be read through the non-coherent path (__ldg /
// `const __restrict__` -> LDG.E.CONSTANT): a programmatically launched grid is already alive while its producer
// writes, so "read-only for the lifetime of the kernel" does not hold and stale lines were observed (wrong sort
// output).  Such loads use __ldcg (streamed once) or __ldca (re-used within an SM) explicitly.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

unsigned pdl_mask();  // B200GS_PDL=<bitmask of launch sites> (0 turns programmatic launches off; A/B measurements)
enum PdlSite { PDL_SORT = 1, PDL_EMIT = 2, PDL_RANGES = 4, PDL_BLEND_FWD = 8, PDL_PRE_BWD = 16, PDL_TRAIN = 32 };

// Every kernel is launched here, and counted (b200gs_launch_count).  A site enabled in pdl_mask() makes it a programmatic
// launch: its predecessor in the stream must be one of OUR kernels, all of which execute pdl_wait.  Site 0 gives full stream
// ordering, for the first kernel of a chain, whose predecessor is a memset / copy / foreign kernel (measured: a programmatic
// launch behind cudaMemsetAsync may start before the memset has landed).
template <typename... KArgs, typename... Args>
inline cudaError_t launch(unsigned site, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
	count_launch();
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = grid;
	cfg.blockDim = block;
	cfg.dynamicSmemBytes = smem;
	cfg.stream = stream;
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	attr[0].val.programmaticStreamSerializationAllowed = 1;
	cfg.attrs = attr;
	cfg.numAttrs = (site & pdl_mask()) ? 1 : 0;
	return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// CTAs of KERNEL resident on the device at once (occupancy x SM count, at most per_sm_limit per SM when > 0), computed once
// per kernel.  Dynamic shared memory above 48 KB is opted into first.
template <auto KERNEL>
unsigned resident_ctas(int block, size_t smem, int per_sm_limit = 0) {
	static unsigned ctas = 0;
	if (!ctas) {
		int dev = 0, sms = 0, per_sm = 0;
		cudaGetDevice(&dev);
		cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
		if (smem > 48 * 1024) cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, KERNEL, block, smem);
		if (per_sm < 1) per_sm = 1;
		if (sms < 1) sms = 148;
		if (per_sm_limit > 0 && per_sm > per_sm_limit) per_sm = per_sm_limit;
		ctas = (unsigned)(per_sm * sms);
	}
	return ctas;
}
// a0*b0 + a1*b1 + a2*b2 with the rounding sequence the reference's sm_100a build executes
// (FMUL, FFMA, FFMA); pinned with .rn intrinsics so neither cicc nor ptxas may re-associate.
__device__ __forceinline__ float dot3_pinned(float a0, float b0, float a1, float b1, float a2, float b2) {
	return __fmaf_rn(a2, b2, __fmaf_rn(a0, b0, __fmul_rn(a1, b1)));
}
// row r of transformPoint4x3/4x4 (DGR/cuda_rasterizer/auxiliary.h:58-77)
__device__ __forceinline__ float xform_row(const float* __restrict__ m, int r, float x, float y, float z) {
	return __fadd_rn(dot3_pinned(x, m[r], y, m[4 + r], z, m[8 + r]), m[12 + r]);
}
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
#endif
