// b200gs -- ordering stages: depth order of the Gaussians, instance offsets + duplicate-with-keys,
// tile sort, tile ranges + blend schedule.
//
// The reference sorts all L (Gaussian, tile) instances by a 64-bit key (tile << 32 | depth bits)
// with a stable LSD radix sort over 32 + getHigherMsb(tiles) bits (DGR/cuda_rasterizer/
// rasterizer_impl.cu:70-111, 277-318): about six 8-bit passes over 12-byte pairs.  An LSD sort
// on (tile, depth) IS a stable sort by depth followed by a stable sort by tile, so the same
// permutation is produced here in two cheaper steps:
//   1. stable radix sort of the P Gaussians by their depth bits (4 passes over P, not L, items);
//   2. instances emitted in that order (y-major, x-minor tiles per Gaussian, as the reference
//      does), then a stable radix sort by tile id only (ceil(bit/8) = 2 passes over 8-byte pairs).
// point_list, tile ranges and (reconstructed) 64-bit keys are bit-identical to the reference.
//
// The radix pass is a single-read "onesweep" pass: per-tile digit counts are chained between
// CTAs with decoupled look-back (one 32-bit status word per (tile, digit)), tile ids are handed
// out by an atomic ticket so a CTA only ever waits on CTAs that already started.  The digit
// histograms of ALL passes are produced by the kernel that writes the keys (preprocess for the
// depth keys, scan_emit for the tile keys), not by a separate read of the keys or inside the passes.
#include "common.cuh"

namespace {

constexpr uint32_t FLAG_LOCAL = 1u << 30;   // word holds this tile's own count
constexpr uint32_t FLAG_INCL = 2u << 30;    // word holds the inclusive count over tiles [0..t]
constexpr uint32_t FLAG_MASK = 3u << 30;
constexpr uint32_t VALUE_MASK = ~FLAG_MASK;
#ifndef B200GS_LOOKBACK_WINDOW
#define B200GS_LOOKBACK_WINDOW 8
#endif
constexpr int LOOKBACK_WINDOW = B200GS_LOOKBACK_WINDOW;  // predecessors inspected per step (independent loads in flight): the
                                                         // INCLUSIVE frontier advances this many tiles per L2 round trip

__device__ __forceinline__ uint32_t ld_volatile(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
__device__ __forceinline__ void st_volatile(uint32_t* p, uint32_t v) { *reinterpret_cast<volatile uint32_t*>(p) = v; }

__device__ __forceinline__ int64_t load_count(const unsigned long long* n_dev, int64_t n_max) {
	if (n_dev == nullptr) return n_max;
	unsigned long long n = __ldcg(n_dev);
	return n < (unsigned long long)n_max ? (int64_t)n : n_max;
}

// Exclusive prefix of `mine` over tiles [0, tile) for one status column (stride words apart), publishing this
// tile's LOCAL then INCLUSIVE word.  Predecessors are inspected LOOKBACK_WINDOW at a time so the walk is a few
// independent load batches instead of one dependent L2 round trip per predecessor.
__device__ __forceinline__ uint32_t lookback_exclusive(uint32_t* __restrict__ column, size_t stride, uint32_t tile, uint32_t mine) {
	uint32_t* my = column + (size_t)tile * stride;
	if (tile == 0) {
		st_volatile(my, mine | FLAG_INCL);
		return 0;
	}
	st_volatile(my, mine | FLAG_LOCAL);
	uint32_t excl = 0;
	int64_t t = (int64_t)tile - 1;
	while (true) {
		uint32_t w[LOOKBACK_WINDOW];
#pragma unroll
		for (int i = 0; i < LOOKBACK_WINDOW; i++) w[i] = (t - i >= 0) ? ld_volatile(column + (size_t)(t - i) * stride) : FLAG_INCL;
		bool found = false;
#pragma unroll
		for (int i = 0; i < LOOKBACK_WINDOW; i++) {
			if (!found) {
				while ((w[i] & FLAG_MASK) == 0) w[i] = ld_volatile(column + (size_t)(t - i) * stride);
				excl += w[i] & VALUE_MASK;
				found = (w[i] & FLAG_INCL) != 0;
			}
		}
		if (found) break;
		t -= LOOKBACK_WINDOW;
	}
	st_volatile(my, (excl + mine) | FLAG_INCL);
	return excl;
}

// Same contract, executed by one full warp on a stride-1 column: the 32 lanes inspect 32 consecutive predecessors
// with one coalesced request, so the INCLUSIVE frontier moves 32 tiles per L2 round trip.  Result valid in all lanes.
__device__ __forceinline__ uint32_t lookback_exclusive_warp(uint32_t* __restrict__ column, uint32_t tile, uint32_t mine) {
	const unsigned lane = threadIdx.x & 31;
	if (tile == 0) {
		if (lane == 0) st_volatile(column, mine | FLAG_INCL);
		return 0;
	}
	if (lane == 0) st_volatile(column + tile, mine | FLAG_LOCAL);
	uint32_t excl = 0;
	int64_t t = (int64_t)tile - 1;
	while (true) {
		const int64_t mine_t = t - lane;
		uint32_t w = mine_t >= 0 ? ld_volatile(column + mine_t) : FLAG_INCL;
		unsigned first, need;
		while (true) {
			const unsigned incl = __ballot_sync(0xFFFFFFFFu, (w & FLAG_INCL) != 0);
			const unsigned ready = __ballot_sync(0xFFFFFFFFu, (w & FLAG_MASK) != 0);
			first = incl ? (unsigned)(__ffs(incl) - 1) : 32u;
			need = first >= 31u ? 0xFFFFFFFFu : ((2u << first) - 1u);
			if ((ready & need) == need) break;
			if ((w & FLAG_MASK) == 0) w = ld_volatile(column + mine_t);
		}
		uint32_t v = ((need >> lane) & 1u) ? (w & VALUE_MASK) : 0u;
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
		excl += v;
		if (first < 32u) break;
		t -= 32;
	}
	if (lane == 0) st_volatile(column + tile, (excl + mine) | FLAG_INCL);
	return excl;
}

// One tile of one radix pass.  `ticket` != nullptr: the tile id is drawn from it (a CTA only ever waits on CTAs that already
// started); nullptr: tile = blockIdx.x (all CTAs of the grid are co-resident, fused multi-pass kernel below).
template <int ITEMS>
__device__ __forceinline__ void onesweep_tile(
	const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, uint32_t* __restrict__ keys_out,
	uint32_t* __restrict__ vals_out, int64_t n, int shift, int bits,
	const uint32_t* __restrict__ hist /*[256] this pass: produced by the kernel that wrote the keys*/,
	uint32_t* __restrict__ lookback /*[tiles][256]*/, unsigned int* __restrict__ ticket)
{
	constexpr int TILE = SORT_THREADS * ITEMS;
	constexpr int WARPS = SORT_THREADS / 32;
	__shared__ uint32_t s_warp_hist[WARPS][256];
	__shared__ uint32_t s_local_off[256];
	__shared__ uint32_t s_digit_base[256];
	__shared__ uint32_t s_keys[TILE];
	__shared__ uint32_t s_vals[TILE];
	__shared__ uint32_t s_g[WARPS], s_l[WARPS];
	__shared__ uint32_t s_tile;
	__shared__ int s_trivial;

	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	for (int i = tid; i < WARPS * 256; i += SORT_THREADS) (&s_warp_hist[0][0])[i] = 0;
	if (tid == 0) { s_tile = ticket ? atomicAdd(ticket, 1u) : blockIdx.x; s_trivial = 0; }
	__syncthreads();
	if ((int64_t)__ldcg(hist + tid) == n && n > 0) s_trivial = 1;  // every key has the same digit: the pass is the identity permutation
	const uint32_t tile = s_tile;
	const int64_t tile_base = (int64_t)tile * TILE;
	if (tile_base >= n) return;
	const int tile_n = (int)min((int64_t)TILE, n - tile_base);
	const uint32_t dmask = (1u << bits) - 1;

	// 1. load (warp-striped: warp w owns a contiguous 32*ITEMS chunk) and rank within the warp
	uint32_t key[ITEMS], val[ITEMS], rnk[ITEMS];
	const int warp_base = warp * 32 * ITEMS;
#pragma unroll
	for (int j = 0; j < ITEMS; j++) {
		const int li = warp_base + j * 32 + lane;
		const bool valid = li < tile_n;
		key[j] = valid ? __ldcg(keys_in + tile_base + li) : 0xFFFFFFFFu;  // .cg, never .nc: see the note on pdl_wait() in common.cuh
		val[j] = valid ? __ldcg(vals_in + tile_base + li) : 0u;
	}
	__syncthreads();  // s_trivial settled
	if (s_trivial) {
#pragma unroll
		for (int j = 0; j < ITEMS; j++) {
			const int li = warp_base + j * 32 + lane;
			if (li < tile_n) { keys_out[tile_base + li] = key[j]; vals_out[tile_base + li] = val[j]; }
		}
		return;
	}
#pragma unroll
	for (int j = 0; j < ITEMS; j++) {
		const int li = warp_base + j * 32 + lane;
		const bool valid = li < tile_n;
		const uint32_t d = (key[j] >> shift) & dmask;
		const uint32_t peers = __match_any_sync(0xFFFFFFFFu, valid ? d : (0x80000000u | lane));
		const uint32_t before = __popc(peers & ((1u << lane) - 1));
		uint32_t pre = 0;
		if (valid) pre = s_warp_hist[warp][d];
		__syncwarp();
		if (valid && before == 0) s_warp_hist[warp][d] = pre + __popc(peers);
		__syncwarp();
		rnk[j] = pre + before;
	}
	__syncthreads();

	// 2. per digit (thread d): exclusive scan over warps, tile total, decoupled look-back
	{
		const int d = tid;
		uint32_t tile_count = 0;
#pragma unroll
		for (int w = 0; w < WARPS; w++) {
			const uint32_t t = s_warp_hist[w][d];
			s_warp_hist[w][d] = tile_count;
			tile_count += t;
		}
		const uint32_t excl = lookback_exclusive(lookback + d, 256, tile, tile_count);
		// exclusive scan of the global digit histogram and of the tile counts across the 256 digits
		const uint32_t g = __ldcg(hist + d), l = tile_count;
		uint32_t gi = g, li = l;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, gi, o), b = __shfl_up_sync(0xFFFFFFFFu, li, o);
			if (lane >= o) { gi += a; li += b; }
		}
		if (lane == 31) { s_g[warp] = gi; s_l[warp] = li; }
		__syncthreads();
		uint32_t gw = 0, lw = 0;
		for (int w = 0; w < warp; w++) { gw += s_g[w]; lw += s_l[w]; }
		const uint32_t g_excl = gw + gi - g, l_excl = lw + li - l;
		s_local_off[d] = l_excl;
		s_digit_base[d] = g_excl + excl - l_excl;  // global position = s_digit_base[d] + local position (mod 2^32)
	}
	__syncthreads();

	// 3. reorder inside the tile so each digit's run leaves the CTA as one contiguous write
#pragma unroll
	for (int j = 0; j < ITEMS; j++) {
		const int li = warp_base + j * 32 + lane;
		if (li < tile_n) {
			const uint32_t d = (key[j] >> shift) & dmask;
			const uint32_t pos = s_local_off[d] + s_warp_hist[warp][d] + rnk[j];
			s_keys[pos] = key[j];
			s_vals[pos] = val[j];
		}
	}
	__syncthreads();
	for (int i = tid; i < tile_n; i += SORT_THREADS) {
		const uint32_t k = s_keys[i];
		const uint32_t d = (k >> shift) & dmask;
		const uint32_t dst = s_digit_base[d] + (uint32_t)i;
		keys_out[dst] = k;
		vals_out[dst] = s_vals[i];
	}
}

template <int ITEMS>
__global__ void __launch_bounds__(SORT_THREADS, ITEMS == SORT_ITEMS_LARGE ? 3 : 6) onesweep_pass_kernel(
	const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, uint32_t* __restrict__ keys_out,
	uint32_t* __restrict__ vals_out, int64_t n_max, const unsigned long long* __restrict__ n_dev, int shift, int bits,
	const uint32_t* __restrict__ hist, uint32_t* __restrict__ lookback, unsigned int* __restrict__ ticket)
{
	pdl_trigger();
	pdl_wait();
	onesweep_tile<ITEMS>(keys_in, vals_in, keys_out, vals_out, load_count(n_dev, n_max), shift, bits, hist, lookback, ticket);
}

// All passes of a sort in ONE launch, for grids that are co-resident (one CTA per tile, grid barrier between passes).  At
// P = 100 k a radix pass is 98 CTAs and ~4 us of SM work inside ~9 us of launch, ramp and drain (ncu: SMs active 40 % of the
// kernel's duration): four launches paid that four times.
template <int ITEMS>
__global__ void __launch_bounds__(SORT_THREADS, ITEMS == SORT_ITEMS_LARGE ? 3 : 6) onesweep_fused_kernel(
	uint32_t* key_a, uint32_t* key_b, uint32_t* val_a, uint32_t* val_b, int64_t n_max, const unsigned long long* __restrict__ n_dev,
	int end_bit, const uint32_t* __restrict__ hist /*[passes][256]*/, uint32_t* __restrict__ lookback /*[passes][tiles][256]*/,
	unsigned int* __restrict__ barrier /*zero on entry*/)
{
	pdl_trigger();
	pdl_wait();
	const int64_t n = load_count(n_dev, n_max);
	const int passes = (end_bit + 7) / 8;
	uint32_t *ki = key_a, *ko = key_b, *vi = val_a, *vo = val_b;
	for (int p = 0; p < passes; p++) {
		const int bits = end_bit - 8 * p < 8 ? end_bit - 8 * p : 8;
		onesweep_tile<ITEMS>(ki, vi, ko, vo, n, 8 * p, bits, hist + 256 * p, lookback + (size_t)p * gridDim.x * 256, nullptr);
		if (p + 1 < passes) {  // grid barrier: every tile of pass p has been scattered before pass p+1 reads
			__syncthreads();
			if (threadIdx.x == 0) {
				__threadfence();
				atomicAdd(barrier, 1u);
				const unsigned target = (unsigned)(p + 1) * gridDim.x;
				while (ld_volatile(barrier) < target) {}
				__threadfence();
			}
			__syncthreads();
		}
		uint32_t* t = ki; ki = ko; ko = t;
		t = vi; vi = vo; vo = t;
	}
}

// K2 + K3 fused: inclusive scan of tiles-touched in depth order (rasterizer_impl.cu:277) with decoupled
// look-back, and duplicateWithKeys (rasterizer_impl.cu:70-111) straight from the scanned offsets.  The depth
// half of the reference's key is implied by the emission order, so only the tile id is written as sort key.
// Also: digit histograms of the tile ids for the tile sort, and the zeroing of its look-back words.
constexpr int EMIT_ITEMS = SCAN_ITEMS;

// TILE_COUNTS (images of at most COUNT_TILES_MAX tiles): every emitted instance is also counted into its tile, in
// shared memory, and each CTA adds its non-zero counters to a global per-tile array (one counter per 128-byte
// line: L2 atomics on neighbouring words serialise).  The last CTA to finish turns the totals into the tile
// ranges, the digit histograms of the tile sort and the blend schedule, so no kernel has to re-read the sorted
// keys.  Larger tile grids keep the separate ranges kernel (a per-instance global RED costs more than it saves).

// Launch orders of the blend units (forward, backward): tile ids, heaviest first.  Weight of a tile = what its units cost the
// last time this workspace rendered (ImageState::tile_cost, persistent workspaces) or, without history, the length of its
// list.  Counting sort on a 7-bit key (position of the leading one + the next two bits), descending; the order inside a
// bucket is arbitrary (blend units are independent of each other).  Called by every thread of one CTA; s_cnt is zero on entry.
// The cost words are consumed: left zero for the blend kernels of this call to accumulate into.
__device__ __forceinline__ uint32_t order_key(uint32_t w) {
	if (w == 0) return 0u;
	const int msb = 31 - __clz(w);
	const uint32_t frac = msb >= 2 ? (w >> (msb - 2)) & 3u : (w << (2 - msb)) & 3u;
	return min(127u, (uint32_t)(msb + 1) * 4u + frac - 3u);
}
template <typename LenFn>
__device__ __forceinline__ void build_blend_orders(int tid, int nthreads, int tiles, LenFn len_of, uint32_t* cost, uint32_t* order_fwd,
                                                   uint32_t* order_bwd, uint32_t (*s_cnt)[128], uint32_t (*s_off)[128]) {
	for (int t = tid; t < tiles; t += nthreads) {
		uint32_t kf = order_key(len_of(t)), kb = kf;
		if (cost) {
			const uint32_t cf = __ldcg(cost + t), cb = __ldcg(cost + tiles + t);
			if (cf) kf = order_key(cf);
			if (cb) kb = order_key(cb);
			cost[t] = kf | (kb << 8);  // kept for the second pass (same thread)
		}
		atomicAdd(&s_cnt[0][kf], 1u);
		atomicAdd(&s_cnt[1][kb], 1u);
	}
	__syncthreads();
	if (tid < 2) {
		uint32_t run = 0;
		for (int k = 127; k >= 0; k--) { s_off[tid][k] = run; run += s_cnt[tid][k]; }
	}
	__syncthreads();
	for (int t = tid; t < tiles; t += nthreads) {
		uint32_t kf, kb;
		if (cost) {
			const uint32_t pk = cost[t];
			kf = pk & 255u; kb = pk >> 8;
			cost[t] = 0u; cost[tiles + t] = 0u;
		} else {
			kf = kb = order_key(len_of(t));
		}
		order_fwd[atomicAdd(&s_off[0][kf], 1u)] = (uint32_t)t;
		order_bwd[atomicAdd(&s_off[1][kb], 1u)] = (uint32_t)t;
	}
}

// EMIT_THREADS Gaussians per CTA: 1024, or 256 for small counts -- at 10 k Gaussians ten CTAs emitted 270 k instances in 40 us,
// forty do it in half the time; at 100 k the shorter look-back chain of the 1024-thread CTAs wins.
template <bool TILE_COUNTS, int EMIT_THREADS>
__global__ void __launch_bounds__(EMIT_THREADS) scan_emit_kernel(
	const uint32_t* __restrict__ order, const ushort4* __restrict__ rect, int P, uint32_t grid_x, int64_t capacity,
	int tile_bits, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals, uint32_t* __restrict__ scan_state,
	uint32_t* __restrict__ tile_hist /*[4][256]*/, uint32_t* __restrict__ zero_words, size_t zero_count,
	GeomHeader* __restrict__ hdr, uint32_t* __restrict__ tile_count, int tiles, uint2* __restrict__ ranges,
	uint32_t* __restrict__ tile_order, uint32_t* __restrict__ tile_order_bwd, uint32_t* tile_cost /* nullptr: no history */)
{
	constexpr int TILE = EMIT_THREADS * EMIT_ITEMS;
	__shared__ uint32_t s_warp[EMIT_THREADS / 32];
	__shared__ uint32_t s_prefix;
	__shared__ uint32_t s_tile;
	__shared__ bool s_last;
	__shared__ uint32_t s_ph[4][256];  // digit histograms of the tile-sort passes (TILE_COUNTS: built by the last CTA from the tile counts)
	__shared__ uint32_t s_cnt[2][128], s_off[2][128];
	__shared__ uint32_t s_tc[TILE_COUNTS ? COUNT_TILES_MAX : 1];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	pdl_trigger();
	for (int i = tid; i < 4 * 256; i += EMIT_THREADS) (&s_ph[0][0])[i] = 0;
	if (tid < 256) (&s_cnt[0][0])[tid] = 0;
	if (TILE_COUNTS) for (int i = tid; i < tiles; i += EMIT_THREADS) s_tc[i] = 0;
	pdl_wait();
	if (tid == 0) s_tile = atomicAdd(&hdr->scan_ticket, 1u);
	// zero the tile sort's look-back words (they are first read by the next kernel)
	for (size_t i = (size_t)blockIdx.x * EMIT_THREADS + tid; i < zero_count; i += (size_t)gridDim.x * EMIT_THREADS) zero_words[i] = 0;
	__syncthreads();
	const uint32_t tile = s_tile;
	const int base = tile * TILE + tid * EMIT_ITEMS;

	uint32_t g[EMIT_ITEMS], n[EMIT_ITEMS];
	ushort4 r[EMIT_ITEMS];
	uint32_t sum = 0;
#pragma unroll
	for (int k = 0; k < EMIT_ITEMS; k++) {
		g[k] = 0; n[k] = 0; r[k] = make_ushort4(0, 0, 0, 0);
		if (base + k < P) {
			g[k] = __ldcg(order + base + k);
			r[k] = __ldcg(rect + g[k]);
			n[k] = (uint32_t)(r[k].z - r[k].x) * (uint32_t)(r[k].w - r[k].y);
		}
		sum += n[k];
	}
	uint32_t inc = sum;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, inc, o);
		if (lane >= o) inc += a;
	}
	if (lane == 31) s_warp[warp] = inc;
	__syncthreads();
	uint32_t wpre = 0, total = 0;
	for (int w = 0; w < EMIT_THREADS / 32; w++) {
		if (w < warp) wpre += s_warp[w];
		total += s_warp[w];
	}
	if (warp == 0) {
		const uint32_t excl = lookback_exclusive_warp(scan_state, tile, total);
		if (lane == 0) s_prefix = excl;
		if (lane == 0 && (int64_t)(tile + 1) * TILE >= P) {  // last tile: instance count, overflow flag
			// the scan's grand total IS the instance count (what the reference reads back, rasterizer_impl.cu:281): assigned here,
			// together with the status word, so neither ever needs zeroing (preprocess accumulates its own copy in num_acc)
			const unsigned long long L = (unsigned long long)excl + total;
			hdr->num_rendered = L;
			hdr->overflow = (L > (unsigned long long)capacity ? 1u : 0u) | __ldcg(&hdr->prefilter_violation);
		}
	}
	__syncthreads();
	uint32_t start = s_prefix + wpre + inc - sum;  // exclusive offset of this thread's first item

	const uint32_t m0 = (1u << min(8, tile_bits)) - 1u;
	auto put = [&](uint32_t pos, uint32_t key, uint32_t val) {
		if ((int64_t)pos < capacity) {
			keys[pos] = key;
			vals[pos] = val;
			if (TILE_COUNTS) atomicAdd(&s_tc[key], 1u);
			else {
				atomicAdd(&s_ph[0][key & m0], 1u);
				if (tile_bits > 8) atomicAdd(&s_ph[1][(key >> 8) & 255u], 1u);
				if (tile_bits > 16) { atomicAdd(&s_ph[2][(key >> 16) & 255u], 1u); if (tile_bits > 24) atomicAdd(&s_ph[3][key >> 24], 1u); }
			}
		}
	};
	// Slot-major emission: lane l of a warp writes output slots wbase + l, wbase + 32 + l, ... and finds the Gaussian that
	// owns a slot by a binary search over the warp's 32 exclusive offsets (shuffles, no shared memory).  Every store
	// instruction covers 32 consecutive slots (4 sectors) whatever the footprints are; the per-thread version wrote one
	// Gaussian's run per lane and touched ~12 sectors per request (ncu at L = 48 M: 6x write amplification, 500 us).
	static_assert(EMIT_ITEMS == 1, "slot-major emission assumes one Gaussian per thread");
	{
		const uint32_t wbase = __shfl_sync(0xFFFFFFFFu, start, 0);
		const uint32_t rel = start - wbase;  // non-decreasing over the lanes
		const uint32_t T = __shfl_sync(0xFFFFFFFFu, rel + n[0], 31);
		const uint32_t rw = (uint32_t)(r[0].z - r[0].x);
		for (uint32_t j0 = 0; j0 < T; j0 += 32) {
			const uint32_t j = j0 + lane;
			int lo = 0, hi = 32;  // the last lane whose offset is <= j owns slot j (empty lanes share the offset of their successor)
#pragma unroll
			for (int it = 0; it < 5; it++) {
				const int mid = (lo + hi) >> 1;
				const uint32_t v = __shfl_sync(0xFFFFFFFFu, rel, mid);
				if (v <= j) lo = mid; else hi = mid;
			}
			const uint32_t og = __shfl_sync(0xFFFFFFFFu, g[0], lo);
			const uint32_t ox = __shfl_sync(0xFFFFFFFFu, (uint32_t)r[0].x, lo), oy = __shfl_sync(0xFFFFFFFFu, (uint32_t)r[0].y, lo);
			const uint32_t ow = __shfl_sync(0xFFFFFFFFu, rw, lo);
			const uint32_t local = j - __shfl_sync(0xFFFFFFFFu, rel, lo);
			if (j < T) put(wbase + j, (oy + local / ow) * grid_x + (ox + local % ow), og);
		}
	}
	__syncthreads();
	if (!TILE_COUNTS) {
		for (int i = tid; i < 256 * ((tile_bits + 7) / 8); i += EMIT_THREADS) {
			const uint32_t c = (&s_ph[0][0])[i];
			if (c) atomicAdd(tile_hist + i, c);
		}
		return;
	}
	// ---- the last CTA to get here turns the tile counts into: tile ranges (identifyTileRanges,
	// rasterizer_impl.cu:116-138: [start,end) per tile, (0,0) for untouched tiles), the digit histograms of the
	// tile-sort passes, and the launch order of the blend units (tile ids, longest range first; 7-bit key =
	// position of the leading one + the next two bits of the length; order inside a bucket is arbitrary).
	for (int i = tid; i < tiles; i += EMIT_THREADS) {
		const uint32_t c = s_tc[i];
		if (c) atomicAdd(tile_count + (size_t)i * COUNT_STRIDE, c);
	}
	__syncthreads();
	if (tid == 0) {
		__threadfence();  // cumulative: the CTA's REDs (observed through the barrier) are ordered before the ticket
		s_last = atomicAdd(&hdr->emit_done, 1u) == gridDim.x - 1;
	}
	__syncthreads();
	if (!s_last) return;
	__threadfence();
	const int passes = (tile_bits + 7) / 8;
	uint32_t running = 0;
	for (int t0 = 0; t0 < tiles; t0 += EMIT_THREADS) {
		const int t = t0 + tid;
		const uint32_t c = t < tiles ? __ldcg(tile_count + (size_t)t * COUNT_STRIDE) : 0u;
		uint32_t incl = c;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, incl, o);
			if (lane >= o) incl += a;
		}
		__syncthreads();  // s_warp / s_prefix reuse
		if (lane == 31) s_warp[warp] = incl;
		__syncthreads();
		uint32_t wp = 0, tot = 0;
		for (int w = 0; w < EMIT_THREADS / 32; w++) {
			if (w < warp) wp += s_warp[w];
			tot += s_warp[w];
		}
		if (t < tiles) {
			const uint32_t b = running + wp + incl - c;
			ranges[t] = c ? make_uint2(b, b + c) : make_uint2(0u, 0u);
			if (c) {
				for (int p = 0; p < passes; p++) atomicAdd(&s_ph[p][((uint32_t)t >> (8 * p)) & 255u], c);
			}
		}
		running += tot;
	}
	__syncthreads();
	for (int i = tid; i < passes * 256; i += EMIT_THREADS) tile_hist[i] = (&s_ph[0][0])[i];
	build_blend_orders(tid, EMIT_THREADS, tiles, [&](int t) { return __ldcg(tile_count + (size_t)t * COUNT_STRIDE); }, tile_cost, tile_order,
	                   tile_order_bwd, s_cnt, s_off);
}

// K5: identifyTileRanges (rasterizer_impl.cu:116-138; `ranges` zero-initialised by the preprocess kernel, :310),
// and -- by the last CTA to finish -- the launch order of the blend units: tile ids, heaviest (longest range)
// first.  key = 7 bits (position of the leading one and the next two bits of the range length); counting sort
// by descending key; order inside a bucket is arbitrary (blend units are independent of each other).
__global__ void __launch_bounds__(256) tile_ranges_schedule_kernel(
	const uint32_t* __restrict__ tile_keys, int64_t n_max, const unsigned long long* __restrict__ n_dev,
	uint2* __restrict__ ranges, int tiles, uint32_t* __restrict__ order, uint32_t* __restrict__ order_bwd, uint32_t* tile_cost /* nullptr: no history */,
	unsigned int* __restrict__ done_counter)
{
	pdl_trigger();
	pdl_wait();
	const int64_t n = load_count(n_dev, n_max);
	// four consecutive keys per thread and step (one 128-bit load + the key before them): ncu showed the one-key version
	// latency bound (long_scoreboard 50 stalls per issue, 12 % of DRAM peak at L = 48 M)
	const int64_t n4 = (n + 3) / 4;
	for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += (int64_t)gridDim.x * blockDim.x) {
		const int64_t i0 = 4 * q;
		uint32_t k[4];
		if (i0 + 3 < n) {
			const uint4 v = __ldcg(reinterpret_cast<const uint4*>(tile_keys) + q);
			k[0] = v.x; k[1] = v.y; k[2] = v.z; k[3] = v.w;
		} else {
#pragma unroll
			for (int j = 0; j < 4; j++) k[j] = i0 + j < n ? __ldcg(tile_keys + i0 + j) : 0u;
		}
		uint32_t prev = i0 > 0 ? __ldcg(tile_keys + i0 - 1) : 0u;
#pragma unroll
		for (int j = 0; j < 4; j++) {
			const int64_t idx = i0 + j;
			if (idx < n) {
				const uint32_t cur = k[j];
				if (idx == 0) ranges[cur].x = 0;
				else if (cur != prev) { ranges[prev].y = (uint32_t)idx; ranges[cur].x = (uint32_t)idx; }
				if (idx == n - 1) ranges[cur].y = (uint32_t)n;
				prev = cur;
			}
		}
	}
	__shared__ bool s_last;
	__shared__ uint32_t s_cnt[2][128], s_off[2][128];
	__syncthreads();
	const int tid = threadIdx.x;
	if (tid == 0) {
		__threadfence();  // cumulative: orders the whole CTA's range writes (observed through the barrier) before the ticket
		s_last = atomicAdd(done_counter, 1u) == gridDim.x - 1;
	}
	(&s_cnt[0][0])[tid] = 0;  // 256 threads
	__syncthreads();
	if (!s_last) return;
	__threadfence();
	build_blend_orders(tid, (int)blockDim.x, tiles, [&](int t) { const uint2 r = __ldcg(ranges + t); return r.y - r.x; }, tile_cost, order, order_bwd,
	                   s_cnt, s_off);
}

__global__ void __launch_bounds__(256) debug_keys_kernel(const uint32_t* __restrict__ tile_keys, const uint32_t* __restrict__ point_list,
                                                         const float* __restrict__ depths, uint64_t* __restrict__ out, int64_t L) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= L) return;
	out[i] = ((uint64_t)tile_keys[i] << 32) | (uint64_t)__float_as_uint(depths[point_list[i]]);
}

}  // namespace

// No instance was emitted (capacity 0): the status words scan_emit would have assigned
__global__ void finalize_header_kernel(GeomHeader* hdr, long long capacity) {
	pdl_trigger();
	pdl_wait();
	const unsigned long long L = __ldcg(&hdr->num_acc);
	hdr->num_rendered = L;
	hdr->overflow = (L > (unsigned long long)capacity ? 1u : 0u) | __ldcg(&hdr->prefilter_violation);
}

void launch_finalize_header(const RasterPlan& pl, cudaStream_t stream) {
	launch(PDL_EMIT, finalize_header_kernel, dim3(1), dim3(1), 0, stream, pl.gs.hdr, (long long)pl.capacity);
}

// (declared in common.cuh)
void launch_radix_sort(uint32_t* key_a, uint32_t* key_b, uint32_t* val_a, uint32_t* val_b, int64_t n_max,
                       const unsigned long long* n_dev, int end_bit, uint32_t* hist /*[passes][256]*/, uint32_t* lookback,
                       unsigned int* tickets, unsigned int* barrier /*zero on entry*/, cudaStream_t stream) {
	if (n_max <= 0 || end_bit <= 0) return;
	const int passes = (end_bit + 7) / 8;
	const int items = sort_items_for(n_max);
	const int64_t tiles = sort_tiles_for(n_max);
	const bool small = items == SORT_ITEMS_SMALL;
	const dim3 grid((unsigned)tiles), block(SORT_THREADS);
	if (passes > 1 && tiles <= (int64_t)(small ? resident_ctas<onesweep_fused_kernel<SORT_ITEMS_SMALL>>(SORT_THREADS, 0)
	                                          : resident_ctas<onesweep_fused_kernel<SORT_ITEMS_LARGE>>(SORT_THREADS, 0))) {
		// every tile's CTA fits on the device at once: all passes in one launch
		auto fused = small ? onesweep_fused_kernel<SORT_ITEMS_SMALL> : onesweep_fused_kernel<SORT_ITEMS_LARGE>;
		launch(PDL_SORT, fused, grid, block, 0, stream, key_a, key_b, val_a, val_b, n_max, n_dev, end_bit, (const uint32_t*)hist, lookback, barrier);
		return;
	}
	auto pass = small ? onesweep_pass_kernel<SORT_ITEMS_SMALL> : onesweep_pass_kernel<SORT_ITEMS_LARGE>;
	uint32_t *ki = key_a, *ko = key_b, *vi = val_a, *vo = val_b;
	for (int p = 0; p < passes; p++) {
		const int bits = end_bit - 8 * p < 8 ? end_bit - 8 * p : 8;
		uint32_t* lb = lookback + (size_t)p * tiles * 256;
		launch(PDL_SORT, pass, grid, block, 0, stream, ki, vi, ko, vo, n_max, n_dev, 8 * p, bits, hist + 256 * p, lb, tickets + p);
		uint32_t* t = ki; ki = ko; ko = t;
		t = vi; vi = vo; vo = t;
	}
}

// Depth order of the P Gaussians.  After this: gs.order = ids by (depth bits, id).
void launch_depth_order(const RasterPlan& pl, cudaStream_t stream) {
	const GeomState& gs = pl.gs;
	// keys: key_a, values: order (identity), digit histograms gs.hist[0..3]: all written by preprocess; 4 passes -> result in (key_a, order)
	launch_radix_sort(gs.key_a, gs.key_b, gs.order, gs.val_b, pl.P, nullptr, 32, gs.hist, gs.lookback, gs.hdr->sort_ticket,
	                  &gs.hdr->sort_barrier[0], stream);
}

void launch_scan_emit(const RasterPlan& pl, cudaStream_t stream, bool chained) {
	const GeomState& gs = pl.gs;
	const TileGrid& t = pl.grid;
	const int threads = scan_threads_for(pl.P);
	const dim3 grid((unsigned)scan_tiles_for(pl.P));
	const size_t lookback_words = (size_t)t.tile_passes * sort_tiles_for(pl.capacity) * 256;
	auto go = [&](auto kernel) {
		launch(chained ? PDL_EMIT : 0u, kernel, grid, dim3(threads), 0, stream, (const uint32_t*)gs.order, (const ushort4*)gs.rect, pl.P, t.gx,
			pl.capacity, t.tile_bits, pl.bs.key_a, pl.bs.val_a, reinterpret_cast<uint32_t*>(gs.scan_state), gs.hist + 4 * 256, pl.bs.lookback,
			lookback_words, gs.hdr, pl.is.tile_count, (int)t.tiles, pl.is.ranges, pl.is.tile_order, pl.is.tile_order_bwd,
			pl.persistent ? pl.is.tile_cost : (uint32_t*)nullptr);
	};
	const bool counts = t.ranges_from_emit;
	if (threads == SCAN_THREADS_SMALL) { if (counts) go(scan_emit_kernel<true, SCAN_THREADS_SMALL>); else go(scan_emit_kernel<false, SCAN_THREADS_SMALL>); }
	else { if (counts) go(scan_emit_kernel<true, SCAN_THREADS>); else go(scan_emit_kernel<false, SCAN_THREADS>); }
}

void launch_tile_sort(const RasterPlan& pl, cudaStream_t stream) {
	const GeomState& gs = pl.gs;
	const BinningState& bs = pl.bs;
	launch_radix_sort(bs.key_a, bs.key_b, bs.val_a, bs.val_b, pl.capacity, &gs.hdr->num_rendered, pl.grid.tile_bits, gs.hist + 4 * 256,
	                  bs.lookback, gs.hdr->sort_ticket + 4, &gs.hdr->sort_barrier[1], stream);
}

void launch_tile_ranges(const RasterPlan& pl, int64_t n_max, cudaStream_t stream) {
	// few CTAs (grid-stride): every CTA ends with one atomic on the same counter
	const int64_t chunks = (n_max + 1023) / 1024;  // 256 threads x 4 keys
	const unsigned grid = (unsigned)(n_max > 0 ? (chunks < 148 * 8 ? chunks : 148 * 8) : 1);
	const ImageState& is = pl.is;
	launch(PDL_RANGES, tile_ranges_schedule_kernel, dim3(grid), dim3(256), 0, stream, (const uint32_t*)pl.bs.sorted_keys, n_max,
	       &pl.gs.hdr->num_rendered, is.ranges, (int)pl.grid.tiles, is.tile_order, is.tile_order_bwd,
	       pl.persistent ? is.tile_cost : (uint32_t*)nullptr, &pl.gs.hdr->ranges_done);
}

void launch_debug_keys(const RasterPlan& pl, uint64_t* keys_out, int64_t L, cudaStream_t stream) {
	if (L <= 0) return;
	launch(0u, debug_keys_kernel, dim3((unsigned)((L + 255) / 256)), dim3(256), 0, stream, pl.bs.sorted_keys, pl.bs.sorted_vals, pl.gs.depths,
	       keys_out, L);
}
