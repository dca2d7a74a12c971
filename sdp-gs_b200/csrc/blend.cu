// b200gs -- alpha blending, forward (K6) and backward (K7).
//
// Semantics: DGR/cuda_rasterizer/forward.cu:261-374 and backward.cu:399-557, generalised from 3 colour
// channels to the 8 blended channels SDP-GS reads, [r,g,b | z | 1 | f0,f1,f2] (SURVEY.md Appendix D;
// background only under r,g,b).  Per-pair arithmetic is the reference's, operation for operation (power =
// fma(q, -0.5, -(dy*(dx*b))), CUDA expf, fma(T, alpha*c, C)), so the image is bit-identical; the decomposition
// is not the reference's:
//   * unit of work = one warp = one 8x4 pixel block of a 16x16 tile.  Warps are autonomous (no CTA barrier
//     anywhere): a persistent grid of 4-warp CTAs draws units from a global ticket, heaviest tile first -- by
//     what the tile's units cost the last time the workspace rendered (ImageState::tile_cost, persistent
//     workspaces; the kernels record 4 x rounds + survivors per unit), else by list length;
//   * a round = 32 consecutive entries of the tile's sorted list, one per lane.  Ids are loaded three rounds
//     ahead, the 32-byte geometry half of the splat record two rounds ahead (registers), the lane then runs the
//     conservative ellipse-vs-block cull (blend_common.cuh) and only survivors (39 % on the LLFF shape) are
//     appended, in list order, to a 64-slot ring in the warp's shared memory; their payload half (colour, depth,
//     feature) is fetched by cp.async straight into the ring, up to K_INFLIGHT rounds of copies in flight;
//   * per-pixel work runs on dense, 16-aligned batches of survivors read from shared memory as broadcasts with
//     immediate offsets, the pair evaluation on packed f32x2 instructions (two survivors per FADD2/FMUL2/FFMA2,
//     blend_common.cuh); the loops carry no index arithmetic, bounds checks or per-survivor bookkeeping loads;
//   * at the LLFF / DTU image sizes a kernel lasts as long as its deepest unit, and a unit is one warp running a
//     chain of dependent FP32 operations (tools/blend_trace.py, DESIGN.md section 4): the WIDE instantiations
//     put more independent work in front of every serial stretch (all 16 alphas of a batch before its recurrence /
//     the T-independent half of the backward's phase 1 for 8 survivors at a time) at 150-166 registers and 3 CTAs
//     per SM; with many units per warp slot (1297x840 and up) the narrow instantiations at 6 / 5 CTAs per SM win;
//   * backward: phase 1 (lane = pixel) replays the recurrence back to front and leaves two weights per
//     (pixel, Gaussian) pair in shared memory; phase 2 (lane = (half, Gaussian)) turns them into the 13
//     per-Gaussian sums -- six pixel moments of wg = G*dL/dG (-> dL/dmean2D, dL/dconic, dL/dopacity) on the
//     lower half-warp, seven channel sums of wc = alpha*T on the upper one, the same instruction stream for
//     both: sum_p w[p] * basis[p][0..6] with a per-warp basis table.  Two red.global.add.v4.f32 per lane
//     replace the reference's 9 float atomics per blended pair (backward.cu:523,545-554).
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include "common.cuh"
#include "blend_common.cuh"

namespace {

// tuning constants (overridable with -D for A/B builds, tools/build_variants.sh)
#ifndef B200GS_BLEND_WARPS
#define B200GS_BLEND_WARPS 4
#endif
#ifndef B200GS_K_INFLIGHT
#define B200GS_K_INFLIGHT 2
#endif
#ifndef B200GS_FWD_CTAS
#define B200GS_FWD_CTAS 0  // CTAs per SM of the persistent forward grid (0: as many as fit)
#endif
#ifndef B200GS_BWD_CTAS
#define B200GS_BWD_CTAS 0
#endif
constexpr int BLEND_WARPS = B200GS_BLEND_WARPS;  // warps per CTA (each with a private shared-memory slice)
constexpr int RING = 64;                         // survivor slots per warp
constexpr int K_INFLIGHT = B200GS_K_INFLIGHT;    // commit groups (= rounds) of payload copies allowed in flight
constexpr int BATCH = 16;                        // survivors per batch; ring positions of a batch never wrap
constexpr int WSTRIDE = BATCH + 2;               // row stride of the pair-weight matrices: even, so phase 1 stores two weights at once; 18 l mod 32 is
                                                 // conflict-free over a half-warp of 64-bit stores and over phase 2's 16 consecutive columns
#define NOID 0xFFFFFFFFu

__device__ __forceinline__ uint32_t sptr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
	asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(sptr(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

#ifdef B200GS_BLEND_TRACE
// developer builds only (tools/build_variants.sh ... "-DB200GS_BLEND_TRACE"): one record per blend unit, read back by tools/blend_trace.py
__device__ uint32_t g_trace[2][1 << 16][8];
__device__ uint32_t g_trace2[1 << 16][4];
__device__ uint32_t g_unit_lo = 0;  // B200GS_BLEND_UNIT_RANGE=lo,hi: only these units are processed (profiling a slice of the schedule)
__device__ __forceinline__ uint32_t trace_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return (uint32_t)t; }
__device__ __forceinline__ uint32_t trace_smid() { uint32_t v; asm("mov.u32 %0, %%smid;" : "=r"(v)); return v; }
__device__ __forceinline__ void trace_put(int dir, uint32_t unit, uint32_t t0, uint32_t c0, int n, int rounds, int surv) {
	if ((threadIdx.x & 31) == 0 && unit < (1u << 16)) {
		uint32_t* r = g_trace[dir][unit];
		r[0] = unit; r[1] = trace_smid(); r[2] = t0; r[3] = trace_ns(); r[4] = (uint32_t)n; r[5] = (uint32_t)rounds; r[6] = (uint32_t)surv;
		r[7] = (uint32_t)clock64() - c0;
	}
}
#endif

struct Unit {
	uint32_t tile, sub;
	unsigned px, py;
	bool inside;
	float pxf, pyf;
	PixelBlock pb;
	uint2 range;
};

__device__ __forceinline__ Unit make_unit(uint32_t unit, const uint32_t* order, const uint2* ranges, int W, int H, int grid_x) {
	Unit u;
	const unsigned lane = threadIdx.x & 31;
	const uint32_t tile = u.tile = __ldcg(order + (unit >> 3));
	const unsigned sub = u.sub = unit & 7;
	const unsigned tx = tile % grid_x, ty = tile / grid_x;
	const unsigned bx = tx * TILE_X + (sub & 1) * 8, by = ty * TILE_Y + (sub >> 1) * 4;
	u.px = bx + (lane & 7);
	u.py = by + (lane >> 3);
	u.inside = u.px < (unsigned)W && u.py < (unsigned)H;
	u.pxf = (float)u.px;
	u.pyf = (float)u.py;
	u.pb.X0 = (float)bx; u.pb.X1 = u.pb.X0 + 7.f;
	u.pb.Y0 = (float)by; u.pb.Y1 = u.pb.Y0 + 3.f;
	u.range = __ldcg(ranges + tile);
	return u;
}

// Per-warp shared memory.
// Geometry of the staged survivors, two per entry so that one packed f32x2 instruction evaluates both:
//   geo[j] = {x0, x1, y0, y1 | a0, a1, b0, b1 | c0, c1, o0, o1} for ring slots 2j (index 0) and 2j+1 (index 1).
struct GeoPair {
	float4 xy, ab, co;
};
__device__ __forceinline__ void geo_store(GeoPair* geo, int slot, const float4 g0, const float4 g1) {
	float* p = reinterpret_cast<float*>(geo + (slot >> 1)) + (slot & 1);
	p[0] = g0.x; p[2] = g0.y; p[4] = g0.z; p[6] = g0.w; p[8] = g1.x; p[10] = g1.y;
}
template <bool EXT>
struct FwdSmem {
	GeoPair geo[RING / 2];
	float4 g2[RING];
	float4 g3[EXT ? RING : 1];
	uint32_t pos[RING];  // 1-based position of the survivor in its tile's list
};
template <bool EXT>
struct BwdSmem {
	float4 g0[RING], g1[RING];
	float4 g2[RING];
	float4 g3[EXT ? RING : 1];
	uint32_t pos[RING];
	uint32_t id[RING];
	float4 basis[32][2][2];          // [pixel][half]: {1, cx, cy, cx^2 | cx*cy, cy^2, 0, 0} / {dL/d(r,g,b,z) | dL/d(f0,f1,f2), 0}
	float w[2][32 * WSTRIDE + 16];   // [0]: wg = G*dL/dG, [1]: wc = alpha*T; the +16 puts the two planes 16 banks apart
};

// The list walk shared by both directions.  Walk entry i is list position pos(i): forward i, backward top - i
// (deepest contributor first).  Lane l handles entry 32 r + l of round r.
template <bool FWD>
struct Walk {
	const uint32_t* list;   // point_list + range.x
	const float4* rec;
	int n, top;
	unsigned lane;
	__device__ __forceinline__ int pos(int i) const { return FWD ? i : top - i; }
	__device__ __forceinline__ uint32_t load_id(int r) const {
		const int i = 32 * r + (int)lane;
		return i < n ? __ldcg(list + pos(i)) : NOID;
	}
	__device__ __forceinline__ void load_geo(uint32_t id, float4& g0, float4& g1) const {
		if (id != NOID) { const float4* p = rec + 4 * (size_t)id; g0 = __ldca(p); g1 = __ldca(p + 1); }
	}
	// cull round r; survivors go to ring slots head.. in walk order, their payload copies are issued.  The round's survivor
	// mask is left in `bits[r]` for the backward (BinningState::surv_bits).
	template <bool EXT, typename S>
	__device__ __forceinline__ int stage(S& s, int r, uint32_t id, const float4 g0, const float4 g1, const PixelBlock& pb, int head,
	                                     uint32_t* bits) const {
		const bool keep = id != NOID && !cull_block(g0, g1, pb);
		const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
		if (lane == 0) bits[r] = m;
		if (m == 0u) return 0;
		if (keep) {
			const int slot = (head + __popc(m & ((1u << lane) - 1u))) & (RING - 1);
			const float4* src = rec + 4 * (size_t)id + 2;
			cp_async16(&s.g2[slot], src);
			if (EXT) cp_async16(&s.g3[slot], src + 1);
			geo_store(s.geo, slot, g0, g1);
			s.pos[slot] = (uint32_t)(pos(32 * r + (int)lane) + 1);
		}
		return __popc(m);
	}
};

// Persistent unit loop: lane 0 draws the next unit from the ticket; the last warp to run dry re-arms both
// counters, so the kernel can be launched again on the same workspace without a memset.
struct Ticket {
	unsigned int* ticket;
	unsigned int* exits;
	__device__ __forceinline__ uint32_t next(unsigned lane) const {
		uint32_t u = 0;
		if (lane == 0) u = atomicAdd(ticket, 1u);
		return __shfl_sync(0xFFFFFFFFu, u, 0);
	}
	__device__ __forceinline__ void leave(unsigned lane, unsigned total_warps) const {
		if (lane == 0) {
			__threadfence();
			if (atomicAdd(exits, 1u) == total_warps - 1u) { atomicExch(ticket, 0u); atomicExch(exits, 0u); }
		}
	}
};

// Two instantiations of each kernel.  WIDE: the alphas of a whole batch of 16 are evaluated before its recurrence (forward) /
// phase 1 is straight-line code over 8 survivors at a time (backward), ~150-170 registers, 3 CTAs per SM: each warp has several
// independent chains in flight, which is what a kernel needs whose critical path is its deepest unit -- one warp -- as long as
// there are only a few units per warp slot (the LLFF shape: 6144 units).  !WIDE: groups of 4 / a loop over survivor pairs, 78-96
// registers, 6 / 5 CTAs per SM: more warps hide more latency once there are many units per slot (measured at 35k and 65k
// units: 3-7 % faster than WIDE; at 6144 units WIDE is 14 % / 11 % faster).
constexpr unsigned WIDE_MAX_UNITS = 16384;
#ifndef B200GS_FWD_NARROW_CTAS
#define B200GS_FWD_NARROW_CTAS 6
#endif
template <bool EXT, bool WIDE>
__global__ void __launch_bounds__(BLEND_WARPS * 32, WIDE ? 3 : B200GS_FWD_NARROW_CTAS) blend_forward_kernel(
	const uint2* ranges, const uint32_t* order, const uint32_t* point_list, const float4* rec,
	int W, int H, int grid_x, uint32_t units, GeomHeader* hdr, uint4* clean_words, size_t clean_count,
	uint32_t* surv_bits, size_t surv_words, uint32_t* tile_cost,
	const float* __restrict__ bg, float* __restrict__ final_T, uint32_t* __restrict__ n_contrib,
	float* __restrict__ out_color, float* __restrict__ out_depth, float* __restrict__ out_alpha, float* __restrict__ out_feat)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	FwdSmem<EXT>& S = reinterpret_cast<FwdSmem<EXT>*>(smem_raw)[threadIdx.x >> 5];
	const unsigned lane = threadIdx.x & 31;
	pdl_trigger();
	pdl_wait();
	const float bg0 = __ldg(bg), bg1 = __ldg(bg + 1), bg2 = __ldg(bg + 2);
	const Ticket tk{&hdr->blend_ticket[0], &hdr->blend_exit[0]};
	// Every kernel that used the geom workspace's counters, histograms and look-back words has completed (pdl_wait): leave
	// them zeroed for the next forward on this workspace, so that a persistent workspace never needs a memset
	// (b200gs_workspace_t.persistent).  num_rendered / overflow stay: they are assigned, not accumulated.
	for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < clean_count; i += (size_t)gridDim.x * blockDim.x)
		clean_words[i] = make_uint4(0u, 0u, 0u, 0u);
	if (blockIdx.x == 0 && threadIdx.x < 8) hdr->sort_ticket[threadIdx.x] = 0u;
	if (blockIdx.x == 0 && threadIdx.x == 8) {
		hdr->scan_ticket = 0u; hdr->ranges_done = 0u; hdr->emit_done = 0u; hdr->num_acc = 0ull; hdr->prefilter_violation = 0u;
		hdr->sort_barrier[0] = 0u; hdr->sort_barrier[1] = 0u;
	}

#ifdef B200GS_BLEND_TRACE
#define TK_NEXT (tk.next(lane) + g_unit_lo)
#else
#define TK_NEXT tk.next(lane)
#endif
	for (uint32_t unit = TK_NEXT; unit < units; unit = TK_NEXT) {
		const Unit u = make_unit(unit, order, ranges, W, H, grid_x);
#ifdef B200GS_BLEND_TRACE
		const uint32_t tr_t0 = trace_ns(), tr_c0 = (uint32_t)clock64();
		int tr_rounds = 0, tr_surv = 0;
		uint32_t tr_proc = 0, tr_wait = 0, tr_nb = 0;  // (B200GS_BLEND_TRACE=2: exposed latency of the id and geometry loads)
#endif
		Walk<true> wk;
		wk.list = point_list + u.range.x; wk.rec = rec; wk.n = (int)(u.range.y - u.range.x); wk.top = 0; wk.lane = lane;
		const int R = (wk.n + 31) >> 5;
		uint32_t* bits = surv_bits + (size_t)u.sub * surv_words + (u.range.x >> 5) + u.tile;  // this unit's survivor-bitmap words

		uint32_t unit_cost = 8;  // what this unit costs, in the schedule builder's units: 4 per round walked + 1 per survivor staged
		bool done = !u.inside;
		float T = 1.0f;
		int lc = -1;                    // ring-absolute index of the last survivor blended into this pixel
		uint32_t last_contributor = 0;  // ... and its 1-based list position (looked up once per batch)
		float2 C01 = make_float2(0.f, 0.f), C56 = C01;  // channel accumulators, (r,g) and (f0,f1) as packed pairs
		float C2 = 0.f, C3 = 0.f, C4 = 0.f, C7 = 0.f;
		const float2 npx = splat2(-u.pxf), npy = splat2(-u.pyf);

		// Blend four staged survivors at ring slots base..base+3 (base % 4 == 0, front to back).  First the four alphas
		// (independent), then the recurrence, branch-free: a pair that is skipped or comes after the pixel is saturated
		// accumulates with weight 0 (exact for finite payloads).  T >= 1e-4 holds while the pixel is live, so a skipped
		// pair (alpha = 0, test_T == T) can never trip the saturation test.
		// N (4 or 16) staged survivors at ring slots base.. (front to back, base % N == 0).  First all N alphas -- packed pairs,
		// independent of each other, so a warp on its own still fills the pipes -- then the N-step recurrence.  Evaluating a
		// whole batch of 16 before its recurrence is what shortens the deepest units (the kernel's critical path: one warp each,
		// latency bound): with groups of 4 in a loop every group paid the shared-memory loads, the alpha chain and the
		// recurrence back to back.
		auto group = [&](auto NCONST, int base, int abs0) {
			constexpr int N = decltype(NCONST)::value;
			constexpr bool EARLY = N <= 4;  // small groups fetch their payload with the geometry (fewer registers are live across the recurrence)
			float al[N];
			float4 pc[EARLY ? N : 1], pf[EARLY ? N : 1];
#pragma unroll
			for (int h = 0; h < N / 2; h++) {  // survivors (base + 2h, base + 2h + 1): one packed evaluation
				const GeoPair& gp = S.geo[(base >> 1) + h];
				const float4 xy = gp.xy, ab = gp.ab, co = gp.co;
				if (EARLY) {
					pc[2 * h] = S.g2[base + 2 * h]; pc[2 * h + 1] = S.g2[base + 2 * h + 1];
					if (EXT) { pf[2 * h] = S.g3[base + 2 * h]; pf[2 * h + 1] = S.g3[base + 2 * h + 1]; }
				}
				const float2 dx = add2(make_float2(xy.x, xy.y), npx), dy = add2(make_float2(xy.z, xy.w), npy);
				const float2 power = pair_power2(dx, dy, make_float2(ab.x, ab.y), make_float2(ab.z, ab.w), make_float2(co.x, co.y));
				const float2 oe = mul2(make_float2(co.z, co.w), expf2(power));
				const float a0 = fminf(0.99f, oe.x), a1 = fminf(0.99f, oe.y);
				al[2 * h] = (power.x > 0.0f || a0 < 1.0f / 255.0f) ? 0.f : a0;  // 0 <=> skipped pair (forward.cu:336-345)
				al[2 * h + 1] = (power.y > 0.0f || a1 < 1.0f / 255.0f) ? 0.f : a1;
			}
			int lc_rel = -1;
#pragma unroll
			for (int k = 0; k < N; k++) {
				const float4 cc = EARLY ? pc[k] : S.g2[base + k];
				const float alpha = al[k];
				const float test_T = __fmul_rn(T, __fsub_rn(1.0f, alpha));
				const bool pdone = done || test_T < 0.0001f;
				const float Tb = pdone ? 0.f : T;
				// rgb: the reference's exact sequence fma(T, alpha*c, C) (forward.cu:355), images are bit-identical
				C01 = fma2(splat2(Tb), mul2(splat2(alpha), make_float2(cc.x, cc.y)), C01);
				C2 = __fmaf_rn(Tb, __fmul_rn(alpha, cc.z), C2);
				if (EXT) {
					const float4 ff = EARLY ? pf[k] : S.g3[base + k];
					const float wt = __fmul_rn(alpha, Tb);
					C3 = __fmaf_rn(wt, cc.w, C3);
					C4 = __fadd_rn(C4, wt);
					C56 = fma2(splat2(wt), make_float2(ff.x, ff.y), C56);
					C7 = __fmaf_rn(wt, ff.z, C7);
				}
				lc_rel = (!pdone && alpha != 0.f) ? k : lc_rel;
				T = pdone ? T : test_T;
				done = pdone;
			}
			lc = lc_rel >= 0 ? abs0 + lc_rel : lc;
		};
		// a full batch [tail, tail + 16) (tail % 16 == 0) / the final flush's groups of 4 [tail, tail + 4 * ngroups)
		constexpr int GROUP = WIDE ? BATCH : 4;
		auto process_batch = [&](int tail) {
#pragma unroll 1
			for (int j = 0; j < BATCH; j += GROUP)  // (one pass when WIDE; the narrow variant must not unroll: registers)
				group(std::integral_constant<int, GROUP>{}, (tail & (RING - 1)) + j, tail + j);
			if (lc >= tail) last_contributor = S.pos[lc & (RING - 1)];  // before the slot can be recycled
		};
		auto process = [&](int tail, int ngroups) {
			const int base0 = tail & (RING - 1);
			for (int j = 0; j < ngroups; j++) group(std::integral_constant<int, 4>{}, base0 + 4 * j, tail + 4 * j);
			if (lc >= tail) last_contributor = S.pos[lc & (RING - 1)];
		};

		if (R > 0) {
			float4 ga0, ga1, gb0, gb1;
			ga0 = ga1 = gb0 = gb1 = make_float4(0.f, 0.f, 0.f, 0.f);
			uint32_t ida = wk.load_id(0), idb = wk.load_id(1), idc = wk.load_id(2);
			wk.load_geo(ida, ga0, ga1);
			wk.load_geo(idb, gb0, gb1);
			int head = 0, tail = 0;
			int hist[K_INFLIGHT + 1];  // hist[j] = head after round r-1-j: what has landed is hist[K_INFLIGHT]
#pragma unroll
			for (int j = 0; j <= K_INFLIGHT; j++) hist[j] = 0;
			bool all_done = false;
			for (int r = 0; r < R; r++) {
#if defined(B200GS_BLEND_TRACE) && B200GS_BLEND_TRACE == 2
				const uint32_t lt0 = (uint32_t)clock64();
#endif
				const uint32_t idd = wk.load_id(r + 3);            // ids, round r+3
#if defined(B200GS_BLEND_TRACE) && B200GS_BLEND_TRACE == 2
				asm volatile("" ::"r"(idd) : "memory");
				const uint32_t lt1 = (uint32_t)clock64();
#endif
				float4 gc0 = make_float4(0.f, 0.f, 0.f, 0.f), gc1 = gc0;
				wk.load_geo(idc, gc0, gc1);                        // geometry, round r+2
#if defined(B200GS_BLEND_TRACE) && B200GS_BLEND_TRACE == 2
				asm volatile("" ::"f"(gc0.x), "f"(gc1.x) : "memory");
				{ const uint32_t lt2 = (uint32_t)clock64(); tr_proc += lt1 - lt0; tr_wait += lt2 - lt1; tr_nb++; }
#endif
				cp_wait<K_INFLIGHT>();  // every group but the latest K has landed: survivors of rounds <= r-1-K are complete
				if (hist[K_INFLIGHT] - tail >= BATCH || head - tail > RING - 32) {
					if (head - tail > RING - 32) { cp_wait<0>(); hist[K_INFLIGHT] = head; }  // a dense stretch: make room for a full round
					__syncwarp();
					do { process_batch(tail); tail += BATCH; } while (hist[K_INFLIGHT] - tail >= BATCH);
					__syncwarp();
					all_done = __all_sync(0xFFFFFFFFu, done);
					if (all_done) break;
				}
				head += wk.template stage<EXT>(S, r, ida, ga0, ga1, u.pb, head, bits);
				unit_cost = 8u + 4u * (uint32_t)(r + 1) + (uint32_t)head;
#ifdef B200GS_BLEND_TRACE
				tr_rounds = r + 1; tr_surv = head;
#endif
				cp_commit();
#pragma unroll
				for (int j = K_INFLIGHT; j > 0; j--) hist[j] = hist[j - 1];
				hist[0] = head;
				ga0 = gb0; ga1 = gb1; gb0 = gc0; gb1 = gc1;
				ida = idb; idb = idc; idc = idd;
			}
			cp_wait<0>();
			if (!all_done && head > tail) {
				// final flush: pad with inert survivors (opacity 0, finite payload) up to a multiple of 4
				const int pad = (tail - head) & 3;
				if ((int)lane < pad) {
					const int slot = (head + (int)lane) & (RING - 1);
					const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
					geo_store(S.geo, slot, z, z);
					S.g2[slot] = z;
					if (EXT) S.g3[slot] = z;
				}
				head += pad;
				__syncwarp();
				while (head > tail) {
					const int g = min(BATCH, head - tail) / 4;
					process(tail, g);
					tail += 4 * g;
					if (__all_sync(0xFFFFFFFFu, done)) break;
				}
			}
			__syncwarp();  // the ring is reused by the next unit
		}
		if (tile_cost && lane == 0) atomicAdd(tile_cost + u.tile, unit_cost);
#ifdef B200GS_BLEND_TRACE
		trace_put(0, unit, tr_t0, tr_c0, wk.n, tr_rounds, tr_surv);
		if (lane == 0 && unit < (1u << 16)) { g_trace2[unit][0] = tr_proc; g_trace2[unit][1] = tr_wait; g_trace2[unit][2] = 0; g_trace2[unit][3] = tr_nb; }
#endif
		if (u.inside) {
			const size_t pix = (size_t)u.py * W + u.px, HW = (size_t)H * W;
			final_T[pix] = T;
			n_contrib[pix] = last_contributor;
			out_color[pix] = __fmaf_rn(bg0, T, C01.x);
			out_color[HW + pix] = __fmaf_rn(bg1, T, C01.y);
			out_color[2 * HW + pix] = __fmaf_rn(bg2, T, C2);
			if (EXT) {
				out_depth[pix] = C3;
				out_alpha[pix] = C4;
				out_feat[pix] = C56.x;
				out_feat[HW + pix] = C56.y;
				out_feat[2 * HW + pix] = C7;
			}
		}
	}
	tk.leave(lane, gridDim.x * BLEND_WARPS);
}

template <bool EXT, bool WIDE>
__global__ void __launch_bounds__(BLEND_WARPS * 32, WIDE ? 3 : 5) blend_backward_kernel(
	const uint2* ranges, const uint32_t* order, const uint32_t* point_list, const float4* rec,
	int W, int H, int grid_x, uint32_t units, unsigned int* ticket, unsigned int* exits,
	const uint32_t* surv_bits, size_t surv_words, uint32_t* tile_cost,
	const float* __restrict__ bg, const float* final_T, const uint32_t* n_contrib, const float* __restrict__ dL_dcolor,
	const float* __restrict__ dL_ddepth, const float* __restrict__ dL_dalpha_map, const float* __restrict__ dL_dfeat,
	float* __restrict__ grec)
{
	constexpr int NC = EXT ? 8 : 3;
	constexpr int NACC = EXT ? 7 : 6;  // accumulators per phase-2 lane (6 moments / 7 or 3 channel sums)
	extern __shared__ __align__(16) unsigned char smem_raw[];
	BwdSmem<EXT>& S = reinterpret_cast<BwdSmem<EXT>*>(smem_raw)[threadIdx.x >> 5];
	const unsigned lane = threadIdx.x & 31;
	pdl_trigger();
	pdl_wait();
	const float bg0 = __ldg(bg), bg1 = __ldg(bg + 1), bg2 = __ldg(bg + 2);
	const float ddelx_dx = 0.5f * W, ddely_dy = 0.5f * H;
	const Ticket tk{ticket, exits};
	const uint32_t gridDim_tiles = units >> 3;  // tiles of the image: the backward's costs are the second plane of tile_cost
	{  // pixel-moment half of the basis table: the same for every unit
		const float cx = (float)(lane & 7), cy = (float)(lane >> 3);
		S.basis[lane][0][0] = make_float4(1.f, cx, cy, cx * cx);
		S.basis[lane][0][1] = make_float4(cx * cy, cy * cy, 0.f, 0.f);
	}

	for (uint32_t unit = tk.next(lane); unit < units; unit = tk.next(lane)) {
		const Unit u = make_unit(unit, order, ranges, W, H, grid_x);
		const size_t pix = (size_t)u.py * W + u.px, HW = (size_t)H * W;
#ifdef B200GS_BLEND_TRACE
		const uint32_t tr_t0 = trace_ns(), tr_c0 = (uint32_t)clock64();
#endif

		// everything the unit needs from the image planes is requested at once, ahead of the wmax == 0 test
		const float T_final = u.inside ? __ldcg(final_T + pix) : 0.f;
		float T = T_final;
		const uint32_t last_contributor = u.inside ? __ldcg(n_contrib + pix) : 0u;
		float dpix[NC];
#pragma unroll
		for (int ch = 0; ch < NC; ch++) dpix[ch] = 0.f;
		if (u.inside) {
			if (dL_dcolor) { dpix[0] = __ldcg(dL_dcolor + pix); dpix[1] = __ldcg(dL_dcolor + HW + pix); dpix[2] = __ldcg(dL_dcolor + 2 * HW + pix); }
			if (EXT) {
				if (dL_ddepth) dpix[3] = __ldcg(dL_ddepth + pix);
				if (dL_dalpha_map) dpix[4] = __ldcg(dL_dalpha_map + pix);
				if (dL_dfeat) { dpix[5] = __ldcg(dL_dfeat + pix); dpix[6] = __ldcg(dL_dfeat + HW + pix); dpix[7] = __ldcg(dL_dfeat + 2 * HW + pix); }
			}
		}
		uint32_t wmax = last_contributor;
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) wmax = max(wmax, __shfl_xor_sync(0xFFFFFFFFu, wmax, o));
		if (wmax == 0) continue;  // nothing was blended into this block

		// cotangents of the channels that own a per-Gaussian gradient: r,g,b,z | f0,f1,f2
		S.basis[lane][1][0] = make_float4(dpix[0], dpix[1], dpix[2], EXT ? dpix[3] : 0.f);
		S.basis[lane][1][1] = EXT ? make_float4(dpix[5], dpix[6], dpix[7], 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
		const float bg_dot_dpixel = bg0 * dpix[0] + bg1 * dpix[1] + bg2 * dpix[2];
		float A = 0.f, lastD = 0.f, last_alpha = 0.f;
		const float2 d01 = make_float2(dpix[0], dpix[1]), d23 = make_float2(dpix[2], EXT ? dpix[3] : 0.f), d56 = make_float2(EXT ? dpix[5] : 0.f, EXT ? dpix[6] : 0.f);

		Walk<false> wk;
		wk.list = point_list + u.range.x; wk.rec = rec; wk.n = (int)wmax; wk.top = (int)wmax - 1; wk.lane = lane;
		const int R = (wk.n + 31) >> 5;

		// One batch: `count` staged survivors at ring slots base.. (base % 16 == 0), deepest first; `cpad` = count rounded
		// up to even (an odd tail is padded with an inert survivor).
		auto process = [&](auto FULLC, int base, int count, int cpad) {
			constexpr bool FULL = decltype(FULLC)::value && WIDE;  // a whole batch of 16: phase 1 is straight-line code
			// ---- phase 1: lane = pixel.  The reference's per-channel accum_rec recurrence (backward.cu:509-516) is
			// carried as one scalar, A = sum_ch accum_rec[ch] * dL/dpixel[ch].
			float* wrow = &S.w[0][lane * WSTRIDE];
			if (FULL) {
				// Everything that does not depend on the running T and A -- G, alpha, 1/(1-alpha), the channel dot product D -- is
				// evaluated for eight survivors at a time (independent chains: a warp on its own still fills the pipes), then the
				// eight recurrence steps follow branch-free.  The deepest units are the kernel's critical path and each is one warp.
#pragma unroll
				for (int half = 0; half < 2; half++) {
					float al[8], inv[8], Dk[8], og[8];
					bool act[8];
#pragma unroll
					for (int k = 0; k < 8; k++) {
						const int sl = base + 8 * half + k;
						const float4 a = S.g0[sl];
						const float4 b = S.g1[sl];
						const float dx = __fsub_rn(a.x, u.pxf), dy = __fsub_rn(a.y, u.pyf);
						const float pw = pair_power(dx, dy, a.z, a.w, b.x);
						const float G = exp_fast(pw);
						al[k] = fminf(0.99f, __fmul_rn(b.y, G));
						act[k] = (S.pos[sl] <= last_contributor) && !(pw > 0.0f) && !(al[k] < 1.0f / 255.0f);
						inv[k] = rcp_approx(1.0f - al[k]);
						og[k] = G * b.y;
						const float4 c = S.g2[sl];
						if (EXT) {
							const float4 f = S.g3[sl];
							float2 Dp = mul2(make_float2(c.x, c.y), d01);
							Dp = fma2(make_float2(c.z, c.w), d23, Dp);
							Dp = fma2(make_float2(f.x, f.y), d56, Dp);
							Dk[k] = (Dp.x + Dp.y) + fmaf(f.z, dpix[7], dpix[4]);
						} else {
							Dk[k] = c.x * dpix[0] + c.y * dpix[1] + c.z * dpix[2];
						}
					}
#pragma unroll
					for (int k = 0; k < 8; k += 2) {
						float wgs[2], wcs[2];
#pragma unroll
						for (int q = 0; q < 2; q++) {
							const int i = k + q;
							const float Tn = T * inv[i];
							const float An = fmaf(1.f - last_alpha, A, last_alpha * lastD);
							const float dL_dalpha = (Dk[i] - An) * Tn - (T_final * inv[i]) * bg_dot_dpixel;
							wgs[q] = act[i] ? og[i] * dL_dalpha : 0.f;  // G * dL/dG; clamp ignored as in backward.cu:538
							wcs[q] = act[i] ? al[i] * Tn : 0.f;
							T = act[i] ? Tn : T;
							A = act[i] ? An : A;
							lastD = act[i] ? Dk[i] : lastD;
							last_alpha = act[i] ? al[i] : last_alpha;
						}
						*reinterpret_cast<float2*>(wrow + 8 * half + k) = make_float2(wgs[0], wgs[1]);
						*reinterpret_cast<float2*>(wrow + 32 * WSTRIDE + 16 + 8 * half + k) = make_float2(wcs[0], wcs[1]);  // S.w[1]
					}
				}
			} else
			for (int k0 = 0; k0 < cpad; k0 += 2) {
				float Gk[2], op[2], pw[2], al[2];
#pragma unroll
				for (int k = 0; k < 2; k++) {
					const float4 a = S.g0[base + k0 + k];
					const float4 b = S.g1[base + k0 + k];
					const float dx = __fsub_rn(a.x, u.pxf), dy = __fsub_rn(a.y, u.pyf);
					pw[k] = pair_power(dx, dy, a.z, a.w, b.x);
					op[k] = b.y;
					Gk[k] = exp_fast(pw[k]);
					al[k] = fminf(0.99f, __fmul_rn(b.y, Gk[k]));
				}
				bool act[2];
				float wgs[2], wcs[2];
#pragma unroll
				for (int k = 0; k < 2; k++)
					act[k] = (S.pos[base + k0 + k] <= last_contributor) && !(pw[k] > 0.0f) && !(al[k] < 1.0f / 255.0f);
#pragma unroll
				for (int k = 0; k < 2; k++) {
					float wg = 0.f, wc = 0.f;
					if (act[k]) {
						const float alpha = al[k];
						const float inv = rcp_approx(1.0f - alpha);
						T *= inv;
						const float4 c = S.g2[base + k0 + k];
						float D;
						if (EXT) {
							const float4 f = S.g3[base + k0 + k];
							float2 Dp = mul2(make_float2(c.x, c.y), d01);
							Dp = fma2(make_float2(c.z, c.w), d23, Dp);
							Dp = fma2(make_float2(f.x, f.y), d56, Dp);
							D = (Dp.x + Dp.y) + fmaf(f.z, dpix[7], dpix[4]);
						} else {
							D = c.x * dpix[0] + c.y * dpix[1] + c.z * dpix[2];
						}
						A = last_alpha * lastD + (1.f - last_alpha) * A;
						lastD = D;
						last_alpha = alpha;
						const float dL_dalpha = (D - A) * T - (T_final * inv) * bg_dot_dpixel;
						wg = Gk[k] * (op[k] * dL_dalpha);  // G * dL/dG; clamp ignored as in backward.cu:538
						wc = alpha * T;
					}
					wgs[k] = wg; wcs[k] = wc;
				}
				*reinterpret_cast<float2*>(wrow + k0) = make_float2(wgs[0], wgs[1]);
				*reinterpret_cast<float2*>(wrow + 32 * WSTRIDE + 16 + k0) = make_float2(wcs[0], wcs[1]);  // S.w[1]
			}
			__syncwarp();
			// ---- phase 2: lane = (half h, Gaussian g).  h = 0: pixel moments of wg; h = 1: channel sums of wc.
			const int g = (int)(lane & 15u), h = (int)(lane >> 4);
			if (g < count) {
				// packed sums: (acc0, acc1), (acc2, acc3), (acc4, acc5) advance with one FFMA2 each
				float2 a01 = make_float2(0.f, 0.f), a23 = a01, a45 = a01;
				float a6 = 0.f;
				const float* wcol = S.w[h] + g;
#pragma unroll
				for (int p = 0; p < 32; p++) {
					const float2 wv = splat2(wcol[p * WSTRIDE]);
					const float4 b0 = S.basis[p][h][0];
					a01 = fma2(wv, make_float2(b0.x, b0.y), a01);
					a23 = fma2(wv, make_float2(b0.z, b0.w), a23);
					const float4 b1 = S.basis[p][h][1];
					a45 = fma2(wv, make_float2(b1.x, b1.y), a45);
					if (EXT) a6 = fmaf(wv.x, b1.z, a6);
				}
				const float acc[7] = {a01.x, a01.y, a23.x, a23.y, a45.x, a45.y, a6};
				bool any = false;
#pragma unroll
				for (int k = 0; k < NACC; k++) any = any || (acc[k] != 0.f);
				if (any) {
					float* dst = grec + (size_t)S.id[base + g] * GREC_FLOATS + 8 * h;
					if (h == 0) {
						const float4 a = S.g0[base + g];
						const float4 b = S.g1[base + g];
						const float S0 = acc[0], Cx = acc[1], Cy = acc[2], Cxx = acc[3], Cxy = acc[4], Cyy = acc[5];
						const float ex = a.x - u.pb.X0, ey = a.y - u.pb.Y0;  // d = mean - pixel = (ex - cx, ey - cy)
						const float Sx = ex * S0 - Cx, Sy = ey * S0 - Cy;
						const float Sxx = ex * (ex * S0 - 2.f * Cx) + Cxx;
						const float Syy = ey * (ey * S0 - 2.f * Cy) + Cyy;
						const float Sxy = ex * (ey * S0 - Cy) - ey * Cx + Cxy;
						red_add_v4(dst, -(a.z * Sx + a.w * Sy) * ddelx_dx, -(b.x * Sy + a.w * Sx) * ddely_dy, -0.5f * Sxx, -0.5f * Sxy);
						red_add_v4(dst + 4, -0.5f * Syy, S0 / b.y, 0.f, 0.f);
					} else {
						red_add_v4(dst, acc[0], acc[1], acc[2], acc[3]);
						if (EXT) red_add_v4(dst + 4, acc[4], acc[5], acc[6], 0.f);
					}
				}
			}
			__syncwarp();
		};

		// The walk: the forward left, for every round it staged, the ballot of its cull (survivor bitmap), so an entry is neither
		// fetched nor culled again here: lanes read their bit and their id two rounds ahead, and survivors have their whole
		// 64-byte record copied into the ring by cp.async.
		const uint32_t* bits = surv_bits + (size_t)u.sub * surv_words + (u.range.x >> 5) + u.tile;
		// Register pipeline, as in the forward: the survivor word of round r+3 and the id of round r+2 (fetched only when its bit
		// is set in the word requested a round earlier) are requested at the end of round r, after the rotation.
		auto load_word = [&](int r) -> uint32_t {  // survivor-bitmap word that holds the bit of walk entry 32 r + lane
			const int i = 32 * r + (int)lane;
			return i < wk.n ? __ldcg(bits + ((wk.top - i) >> 5)) : 0u;
		};
		auto load_entry = [&](int r, uint32_t word) -> uint32_t {  // id of walk entry 32 r + lane, NOID when it did not survive (or is past the end)
			const int i = 32 * r + (int)lane;
			if (i < wk.n) {
				const int p = wk.top - i;
				if ((word >> (p & 31)) & 1u) return __ldcg(wk.list + p);
			}
			return NOID;
		};
		auto stage = [&](int r, uint32_t id, int hd) -> int {
			const unsigned m = __ballot_sync(0xFFFFFFFFu, id != NOID);
			if (m == 0u) return 0;
			if (id != NOID) {
				const int slot = (hd + __popc(m & ((1u << lane) - 1u))) & (RING - 1);
				const float4* src = rec + 4 * (size_t)id;
				cp_async16(&S.g0[slot], src);
				cp_async16(&S.g1[slot], src + 1);
				cp_async16(&S.g2[slot], src + 2);
				if (EXT) cp_async16(&S.g3[slot], src + 3);
				S.pos[slot] = (uint32_t)(wk.top - (32 * r + (int)lane) + 1);
				S.id[slot] = id;
			}
			return __popc(m);
		};
		uint32_t ida = load_entry(0, load_word(0)), idb = load_entry(1, load_word(1)), idc = load_entry(2, load_word(2));
		uint32_t wd = load_word(3);
		int head = 0, tail = 0;
		int hist[K_INFLIGHT + 1];
#pragma unroll
		for (int j = 0; j <= K_INFLIGHT; j++) hist[j] = 0;
		__syncwarp();  // basis visible
		for (int r = 0; r < R; r++) {
			cp_wait<K_INFLIGHT>();
			if (hist[K_INFLIGHT] - tail >= BATCH || head - tail > RING - 32) {
				if (head - tail > RING - 32) { cp_wait<0>(); hist[K_INFLIGHT] = head; }
				__syncwarp();
				do { process(std::true_type{}, tail & (RING - 1), BATCH, BATCH); tail += BATCH; } while (hist[K_INFLIGHT] - tail >= BATCH);
			}
			head += stage(r, ida, head);
			cp_commit();
#pragma unroll
			for (int j = K_INFLIGHT; j > 0; j--) hist[j] = hist[j - 1];
			hist[0] = head;
			ida = idb; idb = idc;
			idc = load_entry(r + 3, wd);
			wd = load_word(r + 4);
		}
		cp_wait<0>();
		if (head > tail) {
			if ((head & 1) && lane == 0) {  // inert survivor after an odd tail: never active (position beyond every n_contrib)
				const int slot = head & (RING - 1);
				const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
				S.g0[slot] = z; S.g1[slot] = z;
				S.pos[slot] = 0xFFFFFFFFu;
			}
			__syncwarp();
			while (head > tail) {
				const int c = min(BATCH, head - tail);
				process(std::false_type{}, tail & (RING - 1), c, (c + 1) & ~1);
				tail += c;
			}
		}
		if (tile_cost && lane == 0) atomicAdd(tile_cost + (size_t)gridDim_tiles + u.tile, 16u + (uint32_t)R + (uint32_t)head);
#ifdef B200GS_BLEND_TRACE
		trace_put(1, unit, tr_t0, tr_c0, wk.n, R, head);
#endif
	}
	tk.leave(lane, gridDim.x * BLEND_WARPS);
}

// CTAs per SM of the persistent grids (forward, backward).  Fewer resident warps than units lets the ticket balance the
// SMs; more warps hide more latency.  Defaults measured on B200 (DESIGN.md); B200GS_BLEND_CTAS=f,b overrides for A/B runs.
int ctas_per_sm(int dir) {
	int a = 0, b = 0;
	if (const char* e = knob(KNOB_BLEND_CTAS))
		if (sscanf(e, "%d,%d", &a, &b) == 2) return dir ? b : a;
	return dir ? B200GS_BWD_CTAS : B200GS_FWD_CTAS;
}

}  // namespace

#ifdef B200GS_BLEND_TRACE
extern "C" int b200gs_debug_blend_trace2(uint32_t* host_out) {
	return (int)cudaMemcpyFromSymbol(host_out, g_trace2, sizeof(uint32_t) * (1 << 16) * 4, 0);
}
extern "C" int b200gs_debug_blend_trace(uint32_t* host_out, int dir) {
	return (int)cudaMemcpyFromSymbol(host_out, g_trace, sizeof(uint32_t) * (1 << 16) * 8, (size_t)dir * sizeof(uint32_t) * (1 << 16) * 8);
}
#endif

namespace {
bool use_wide(unsigned units) {
	const int forced = knob_int(KNOB_BLEND_WIDE, -1);  // 0 / 1: A/B runs
	return forced >= 0 ? forced != 0 : units <= WIDE_MAX_UNITS;
}
// One persistent wave: as many CTAs as fit on the device, never more than there are units.
template <bool EXT, bool WIDE>
void forward_variant(const RasterPlan& pl, const b200gs_outputs_t& out, cudaStream_t stream, unsigned units) {
	const b200gs_view_t& v = *pl.v;
	const GeomState& gs = pl.gs;
	const ImageState& is = pl.is;
	constexpr size_t smem = BLEND_WARPS * sizeof(FwdSmem<EXT>);
	const unsigned cap = resident_ctas<blend_forward_kernel<EXT, WIDE>>(BLEND_WARPS * 32, smem, ctas_per_sm(0));
	const unsigned want = (units + BLEND_WARPS - 1) / BLEND_WARPS;
	uint4* clean_words = reinterpret_cast<uint4*>(gs.hdr + 1);  // the geom clean region past the header
	const size_t clean_count = (gs.clean_bytes - sizeof(GeomHeader)) / sizeof(uint4);
	launch(PDL_BLEND_FWD, blend_forward_kernel<EXT, WIDE>, dim3(want < cap ? want : cap), dim3(BLEND_WARPS * 32), smem, stream,
		(const uint2*)is.ranges, (const uint32_t*)is.tile_order, (const uint32_t*)pl.bs.sorted_vals, (const float4*)gs.rec,
		v.width, v.height, (int)pl.grid.gx, units, gs.hdr, clean_words, clean_count, pl.bs.surv_bits, pl.bs.surv_words,
		pl.persistent ? is.tile_cost : (uint32_t*)nullptr, v.background, is.final_T, is.n_contrib,
		out.color, EXT ? out.depth : (float*)nullptr, EXT ? out.alpha : (float*)nullptr, EXT ? out.feature : (float*)nullptr);
}
template <bool EXT, bool WIDE>
void backward_variant(const RasterPlan& pl, const b200gs_grad_outputs_t& gout, float* grec, cudaStream_t stream) {
	const b200gs_view_t& v = *pl.v;
	const GeomState& gs = pl.gs;
	const ImageState& is = pl.is;
	const unsigned units = pl.grid.units;
	constexpr size_t smem = BLEND_WARPS * sizeof(BwdSmem<EXT>);
	const unsigned cap = resident_ctas<blend_backward_kernel<EXT, WIDE>>(BLEND_WARPS * 32, smem, ctas_per_sm(1));
	const unsigned want = (units + BLEND_WARPS - 1) / BLEND_WARPS;
	// first kernel of the backward chain: its predecessor is a memset / the caller's loss kernels, so no programmatic launch
	launch(0u, blend_backward_kernel<EXT, WIDE>, dim3(want < cap ? want : cap), dim3(BLEND_WARPS * 32), smem, stream,
		(const uint2*)is.ranges, (const uint32_t*)is.tile_order_bwd, (const uint32_t*)pl.bs.sorted_vals, (const float4*)gs.rec,
		v.width, v.height, (int)pl.grid.gx, units, &gs.hdr->blend_ticket[1], &gs.hdr->blend_exit[1], (const uint32_t*)pl.bs.surv_bits,
		pl.bs.surv_words, pl.persistent ? is.tile_cost : (uint32_t*)nullptr, v.background, (const float*)is.final_T,
		(const uint32_t*)is.n_contrib, gout.dL_dcolor, EXT ? gout.dL_ddepth : (const float*)nullptr,
		EXT ? gout.dL_dalpha : (const float*)nullptr, EXT ? gout.dL_dfeature : (const float*)nullptr, grec);
}
}  // namespace

void launch_blend_forward(const RasterPlan& pl, const b200gs_outputs_t& out, cudaStream_t stream) {
	unsigned units = pl.grid.units;
	const bool wide = use_wide(units);
#ifdef B200GS_BLEND_TRACE
	if (const char* e = getenv("B200GS_BLEND_UNIT_RANGE")) {
		unsigned lo = 0, hi = units;
		if (sscanf(e, "%u,%u", &lo, &hi) == 2) { cudaMemcpyToSymbol(g_unit_lo, &lo, 4); if (hi < units) units = hi; }
	}
#endif
	if (pl.v->extended) {
		if (wide) forward_variant<true, true>(pl, out, stream, units);
		else forward_variant<true, false>(pl, out, stream, units);
	} else {
		if (wide) forward_variant<false, true>(pl, out, stream, units);
		else forward_variant<false, false>(pl, out, stream, units);
	}
}

void launch_blend_backward(const RasterPlan& pl, const b200gs_grad_outputs_t& gout, float* grec, cudaStream_t stream) {
	const bool wide = use_wide(pl.grid.units);
	if (pl.v->extended) {
		if (wide) backward_variant<true, true>(pl, gout, grec, stream);
		else backward_variant<true, false>(pl, gout, grec, stream);
	} else {
		if (wide) backward_variant<false, true>(pl, gout, grec, stream);
		else backward_variant<false, false>(pl, gout, grec, stream);
	}
}
