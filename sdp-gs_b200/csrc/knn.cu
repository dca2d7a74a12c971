// b200gs -- exact 3 nearest neighbours over a Morton-ordered implicit box hierarchy (b200gs_knn3_tree).
//
// Same outputs, bit for bit, as the exhaustive b200gs_knn3 (train_ops.cu), in O(P log P) work:
//   1. bounds of the finite points (device reduction), one cubic extent, 21-bit-per-axis quantisation interleaved into a
//      63-bit Morton code; the same kernel writes the digit histograms of all eight radix passes;
//   2. stable sort of (code, index): onesweep sort of the low word, then of the high word gathered through the first
//      permutation (an LSD sort on (hi, lo) is a stable sort by lo followed by a stable sort by hi);
//   3. implicit tree: leaves are 32 consecutive sorted points, each upper level groups 32 consecutive nodes; every node
//      stores the AABB of the finite points below it (empty: lo = +inf, hi = -inf);
//   4. one warp per leaf (one lane per query) walks the tree with a shared-memory stack.
// Why the result is the exhaustive kernel's:
//   * distances use its rounding sequence (dx = cand - query, fl(fl(dx^2 + dy^2) + dz^2)), mean (d0 + d1 + d2) / 3;
//   * the exhaustive kernel sees candidates in index order and lets ties not displace, i.e. it keeps the three smallest
//     (d, index) pairs with d < 3e38 (its sentinel), padded with (3e38, -1).  Candidates arrive here in Morton order, so
//     they are ranked by (d, index) lexicographically; a candidate with d >= 3e38, inf or NaN never enters, and self is
//     excluded by index (duplicates at distance 0 are each other's neighbours);
//   * a node is skipped only when its lower bound is STRICTLY greater than the third distance of every lane it is tested
//     for (an equal bound may hide a tie with a lower index).  The bound applies the same rounded sequence to the axis gaps
//     fl(node_lo - query_hi) / fl(query_lo - node_hi), clamped at 0: rounding is monotone, so it never exceeds the
//     computed distance of a pair it covers;
//   * nothing depends on visiting order (no float atomics touch the results), so every call gives the same bits.
// No host synchronisation: the call can be captured in a CUDA graph.
#include <cmath>
#include "common.cuh"
#include "../../include/b200gs_train.h"

int train_fail(int code, const char* msg);  // api.cu

namespace {

constexpr int KNN_MAX_LEVELS = 6;              // P < 2^30: at most 2^25 leaves -> levels of 2^25, 2^20, ..., 2^5, 1 nodes
constexpr int KNN_STACK = 32 * KNN_MAX_LEVELS;  // at most 32 entries pending per level below the root
constexpr int KNN_WARPS = 8;                    // warps (leaves) per CTA of the query kernel
constexpr int KNN_KEY_CTAS = 148 * 2;           // grid of the reduction kernels: few CTAs, few global atomics
constexpr float KNN_SENTINEL = 3.0e38f;         // b200gs_knn3's initial distance

struct Levels {
	int n;                           // number of levels; level n-1 is the root (a single node)
	int count[KNN_MAX_LEVELS];       // nodes per level (level 0 = leaves)
	int offset[KNN_MAX_LEVELS];      // first node of each level in the box arrays
};

struct Layout {
	size_t hdr, hist, lookback, zero_end;  // [0, zero_end): zeroed by every call
	size_t key_a, key_b, val_a, val_b, hi, pts, box_lo, box_hi, bytes;
	int64_t tiles;
	Levels lv;
};

// words of the header: ordered bounds (min as ~ordered, so that zero is the identity of both), sort tickets, sort barriers
enum { HDR_BOUNDS = 0, HDR_TICKETS = 6, HDR_BARRIER = 14, HDR_WORDS = 16 };

Layout layout_for(int P) {
	Layout L{};
	size_t off = 0;
	auto take = [&](size_t bytes) { const size_t at = off; off += (bytes + 255) & ~(size_t)255; return at; };
	L.tiles = sort_tiles_for(P);
	L.hdr = take(HDR_WORDS * 4);
	L.hist = take(8 * 256 * 4);
	L.lookback = take((size_t)2 * 4 * L.tiles * 256 * 4);  // two sorts of four passes
	L.zero_end = off;
	L.key_a = take((size_t)P * 4); L.key_b = take((size_t)P * 4);
	L.val_a = take((size_t)P * 4); L.val_b = take((size_t)P * 4);
	L.hi = take((size_t)P * 4);
	L.pts = take((size_t)P * 16);
	int n = 0, nodes = 0, c = (P + 31) / 32;
	while (true) {
		L.lv.count[n] = c; L.lv.offset[n] = nodes; nodes += c; n++;
		if (c == 1) break;
		c = (c + 31) / 32;
	}
	L.lv.n = n;
	L.box_lo = take((size_t)nodes * 16);
	L.box_hi = take((size_t)nodes * 16);
	L.bytes = off;
	return L;
}

// float <-> unsigned with the same order (NaN excluded)
__device__ __forceinline__ uint32_t f2ord(float f) { const uint32_t b = __float_as_uint(f); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float ord2f(uint32_t u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u); }
__device__ __forceinline__ bool finite3(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z); }

__device__ __forceinline__ float dist2(float dx, float dy, float dz) {  // b200gs_knn3's rounding sequence
	return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}
// lower bound of dist2(cand - query) over cand in [lo, hi] and query in [qlo, qhi] (a point query: qlo == qhi)
__device__ __forceinline__ float box_bound(float4 lo, float4 hi, float3 qlo, float3 qhi) {
	const float gx = fmaxf(fmaxf(lo.x - qhi.x, qlo.x - hi.x), 0.f);
	const float gy = fmaxf(fmaxf(lo.y - qhi.y, qlo.y - hi.y), 0.f);
	const float gz = fmaxf(fmaxf(lo.z - qhi.z, qlo.z - hi.z), 0.f);
	return dist2(gx, gy, gz);
}

__global__ void __launch_bounds__(256) knn_bounds_kernel(int P, const float* __restrict__ xyz, uint32_t* __restrict__ hdr) {
	uint32_t mn[3] = {0u, 0u, 0u}, mx[3] = {0u, 0u, 0u};  // both as maxima: mn holds ~ordered(min)
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x) {
		const float x = xyz[3 * (size_t)i], y = xyz[3 * (size_t)i + 1], z = xyz[3 * (size_t)i + 2];
		if (!finite3(x, y, z)) continue;
		const float v[3] = {x, y, z};
#pragma unroll
		for (int a = 0; a < 3; a++) { mn[a] = max(mn[a], ~f2ord(v[a])); mx[a] = max(mx[a], f2ord(v[a])); }
	}
#pragma unroll
	for (int a = 0; a < 3; a++) {
		mn[a] = __reduce_max_sync(0xFFFFFFFFu, mn[a]);
		mx[a] = __reduce_max_sync(0xFFFFFFFFu, mx[a]);
	}
	if ((threadIdx.x & 31) == 0) {
#pragma unroll
		for (int a = 0; a < 3; a++) {
			if (mn[a]) atomicMax(hdr + HDR_BOUNDS + a, mn[a]);
			if (mx[a]) atomicMax(hdr + HDR_BOUNDS + 3 + a, mx[a]);
		}
	}
}

__device__ __forceinline__ uint64_t spread3(uint32_t v) {  // 21 bits -> every third bit of 63
	uint64_t x = v & 0x1FFFFFu;
	x = (x | (x << 32)) & 0x1F00000000FFFFull;
	x = (x | (x << 16)) & 0x1F0000FF0000FFull;
	x = (x | (x << 8)) & 0x100F00F00F00F00Full;
	x = (x | (x << 4)) & 0x10C30C30C30C30C3ull;
	x = (x | (x << 2)) & 0x1249249249249249ull;
	return x;
}

// Morton code of every point (low word -> key_a, high word -> hi, index -> val_a) and the digit histograms of the eight
// radix passes (four over each word).
__global__ void __launch_bounds__(256) knn_keys_kernel(int P, const float* __restrict__ xyz, const uint32_t* __restrict__ hdr,
                                                       uint32_t* __restrict__ key_lo, uint32_t* __restrict__ key_hi,
                                                       uint32_t* __restrict__ vals, uint32_t* __restrict__ hist) {
	__shared__ uint32_t s_h[8][256];
	for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) (&s_h[0][0])[i] = 0;
	float lo[3], scale = 0.f;
	bool any = true;
	float extent = 0.f;
#pragma unroll
	for (int a = 0; a < 3; a++) {
		const uint32_t wmin = __ldcg(hdr + HDR_BOUNDS + a), wmax = __ldcg(hdr + HDR_BOUNDS + 3 + a);
		any = any && wmin != 0u;
		lo[a] = ord2f(~wmin);
		extent = fmaxf(extent, ord2f(wmax) - lo[a]);
	}
	// one cubic extent (the largest side): flat clouds do not divide by zero; all points identical -> every code 0
	if (any && extent > 0.f && isfinite(extent)) scale = fminf(2097151.f / extent, 3.0e38f);
	if (!any) lo[0] = lo[1] = lo[2] = 0.f;
	__syncthreads();
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x) {
		uint64_t code = 0;
#pragma unroll
		for (int a = 0; a < 3; a++) {
			// NaN -> 0 (fmaxf returns the number), +-inf and overflow -> the ends of the range
			const float t = fminf(fmaxf((xyz[3 * (size_t)i + a] - lo[a]) * scale, 0.f), 2097151.f);
			code |= spread3(__float2uint_rz(t)) << a;
		}
		const uint32_t l = (uint32_t)code, h = (uint32_t)(code >> 32);
		key_lo[i] = l; key_hi[i] = h; vals[i] = (uint32_t)i;
#pragma unroll
		for (int p = 0; p < 4; p++) {
			atomicAdd(&s_h[p][(l >> (8 * p)) & 255u], 1u);
			atomicAdd(&s_h[4 + p][(h >> (8 * p)) & 255u], 1u);
		}
	}
	__syncthreads();
	for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) {
		const uint32_t c = (&s_h[0][0])[i];
		if (c) atomicAdd(hist + i, c);
	}
}

__global__ void __launch_bounds__(256) knn_gather_hi_kernel(int P, const uint32_t* __restrict__ perm, const uint32_t* __restrict__ hi,
                                                            uint32_t* __restrict__ out) {
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < P) out[i] = __ldcg(hi + __ldcg(perm + i));
}

// warp-wide AABB of the lanes with `live`; (+inf, -inf) when there are none
__device__ __forceinline__ void warp_box(bool live, float x, float y, float z, float4& lo, float4& hi) {
	if (!__any_sync(0xFFFFFFFFu, live)) {
		lo = make_float4(INFINITY, INFINITY, INFINITY, 0.f);
		hi = make_float4(-INFINITY, -INFINITY, -INFINITY, 0.f);
		return;
	}
	const unsigned F = 0xFFFFFFFFu;
	lo = make_float4(ord2f(__reduce_min_sync(F, live ? f2ord(x) : 0xFFFFFFFFu)), ord2f(__reduce_min_sync(F, live ? f2ord(y) : 0xFFFFFFFFu)),
	                 ord2f(__reduce_min_sync(F, live ? f2ord(z) : 0xFFFFFFFFu)), 0.f);
	hi = make_float4(ord2f(__reduce_max_sync(F, live ? f2ord(x) : 0u)), ord2f(__reduce_max_sync(F, live ? f2ord(y) : 0u)),
	                 ord2f(__reduce_max_sync(F, live ? f2ord(z) : 0u)), 0.f);
}

// One warp per leaf: the sorted points as (x, y, z, original index) and the leaf's AABB over its finite points.
__global__ void __launch_bounds__(256) knn_leaves_kernel(int P, const float* __restrict__ xyz, const uint32_t* __restrict__ order,
                                                         float4* __restrict__ pts, float4* __restrict__ box_lo, float4* __restrict__ box_hi,
                                                         int leaves) {
	const int leaf = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
	if (leaf >= leaves) return;  // whole warps
	const int k = leaf * 32 + (int)lane_id();
	float x = 0.f, y = 0.f, z = 0.f;
	bool fin = false;
	if (k < P) {
		const uint32_t o = __ldcg(order + k);
		x = xyz[3 * (size_t)o]; y = xyz[3 * (size_t)o + 1]; z = xyz[3 * (size_t)o + 2];
		pts[k] = make_float4(x, y, z, __int_as_float((int)o));
		fin = finite3(x, y, z);
	}
	float4 lo, hi;
	warp_box(fin, x, y, z, lo, hi);
	if (lane_id() == 0) { box_lo[leaf] = lo; box_hi[leaf] = hi; }
}

// One warp per node of an upper level: the union of its (up to) 32 children's boxes.
__global__ void __launch_bounds__(256) knn_level_kernel(const float4* __restrict__ child_lo, const float4* __restrict__ child_hi, int children,
                                                        float4* __restrict__ box_lo, float4* __restrict__ box_hi, int nodes) {
	const int node = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
	if (node >= nodes) return;
	const int c = node * 32 + (int)lane_id();
	const bool has = c < children;
	const float4 l = has ? __ldcg(child_lo + c) : make_float4(0.f, 0.f, 0.f, 0.f), h = has ? __ldcg(child_hi + c) : l;
	const unsigned F = 0xFFFFFFFFu;  // empty children (+inf, -inf) are the identities of min / max
	const float4 lo = make_float4(ord2f(__reduce_min_sync(F, has ? f2ord(l.x) : 0xFFFFFFFFu)), ord2f(__reduce_min_sync(F, has ? f2ord(l.y) : 0xFFFFFFFFu)),
	                              ord2f(__reduce_min_sync(F, has ? f2ord(l.z) : 0xFFFFFFFFu)), 0.f);
	const float4 hi = make_float4(ord2f(__reduce_max_sync(F, has ? f2ord(h.x) : 0u)), ord2f(__reduce_max_sync(F, has ? f2ord(h.y) : 0u)),
	                              ord2f(__reduce_max_sync(F, has ? f2ord(h.z) : 0u)), 0.f);
	if (lane_id() == 0) { box_lo[node] = lo; box_hi[node] = hi; }
}

struct Top3 {
	float d0 = KNN_SENTINEL, d1 = KNN_SENTINEL, d2 = KNN_SENTINEL;
	int i0 = -1, i1 = -1, i2 = -1;
	// keep the three smallest (d, j); the sentinel (3e38, -1) admits only d < 3e38, never inf or NaN
	__device__ __forceinline__ void insert(float d, int j) {
		if (d < d2 || (d == d2 && j < i2)) {
			if (d < d1 || (d == d1 && j < i1)) {
				d2 = d1; i2 = i1;
				if (d < d0 || (d == d0 && j < i0)) { d1 = d0; i1 = i0; d0 = d; i0 = j; }
				else { d1 = d; i1 = j; }
			} else { d2 = d; i2 = j; }
		}
	}
};

// every lane tests its query against the (up to) 32 points of one leaf
__device__ __forceinline__ void scan_leaf(const float4* __restrict__ pts, int P, int leaf, float4 q, int qi, Top3& t) {
	const int base = leaf * 32, cnt = min(32, P - base);
	const int lane = (int)lane_id();
	const float4 c = lane < cnt ? __ldcg(pts + base + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
	for (int s = 0; s < cnt; s++) {
		const float cx = __shfl_sync(0xFFFFFFFFu, c.x, s), cy = __shfl_sync(0xFFFFFFFFu, c.y, s), cz = __shfl_sync(0xFFFFFFFFu, c.z, s);
		const int ci = __shfl_sync(0xFFFFFFFFu, __float_as_int(c.w), s);
		const float d = dist2(cx - q.x, cy - q.y, cz - q.z);
		if (ci != qi) t.insert(d, ci);
	}
}

// largest third distance over the lanes with a finite query (distances are >= +0, so their bits order like unsigned)
__device__ __forceinline__ float warp_worst(bool fin, const Top3& t) {
	return __uint_as_float(__reduce_max_sync(0xFFFFFFFFu, fin ? __float_as_uint(t.d2) : 0u));
}

__global__ void __launch_bounds__(KNN_WARPS * 32) knn_query_kernel(int P, const float4* __restrict__ pts, const float4* __restrict__ box_lo,
                                                                   const float4* __restrict__ box_hi, Levels lv, float* __restrict__ mean_d2,
                                                                   int32_t* __restrict__ idx3) {
	__shared__ uint32_t s_node[KNN_WARPS][KNN_STACK];  // (level << 27) | index within the level
	__shared__ float s_bound[KNN_WARPS][KNN_STACK];    // box-to-box bound when pushed
	const int w = threadIdx.x >> 5, lane = (int)lane_id();
	const int leaf = blockIdx.x * KNN_WARPS + w;
	if (leaf >= lv.count[0]) return;  // whole warps
	const int k = leaf * 32 + lane;
	const bool live = k < P;
	const float4 q = live ? __ldcg(pts + k) : make_float4(0.f, 0.f, 0.f, 0.f);
	const int qi = live ? __float_as_int(q.w) : -2;
	const bool fin = live && finite3(q.x, q.y, q.z);
	Top3 t;
	// a lane with a non-finite query has no candidate (every distance is inf or NaN) and takes no part in the walk
	if (__any_sync(0xFFFFFFFFu, fin)) {
		const float3 qp = make_float3(q.x, q.y, q.z);
		scan_leaf(pts, P, leaf, q, qi, t);  // the own leaf first: a tight initial third distance
		float worst = warp_worst(fin, t);
		uint32_t* stk = s_node[w];
		float* stb = s_bound[w];
		int top = 0;
		if (lv.n > 1) {
			if (lane == 0) { stk[0] = (uint32_t)(lv.n - 1) << 27; stb[0] = 0.f; }
			top = 1;
		}
		__syncwarp();
		while (top > 0) {
			top--;
			const uint32_t node = stk[top];
			const float pushed = stb[top];
			__syncwarp();  // read before any lane overwrites the slot
			if (pushed > worst) continue;
			const int level = (int)(node >> 27), id = (int)(node & ((1u << 27) - 1));
			if (level == 0 && id == leaf) continue;
			// each lane's own point against the node: skip unless some lane could still take a candidate from it
			const int g = lv.offset[level] + id;
			const float4 nlo = __ldcg(box_lo + g), nhi = __ldcg(box_hi + g);
			const bool need = fin && !(box_bound(nlo, nhi, qp, qp) > t.d2);
			if (!__any_sync(0xFFFFFFFFu, need)) continue;
			if (level == 0) {
				scan_leaf(pts, P, id, q, qi, t);
				worst = warp_worst(fin, t);
				continue;
			}
			// Children, one per lane, against the box of the lanes that need this node (a lane that does not need it cannot
			// need a child inside it): push those whose bound does not exceed the largest third distance of those lanes,
			// nearest on top.  When one far lane (an outlier) is all that needs a node, this is its own point's bound, so its
			// walk stays nearest-first although the warp's whole query box covers the scene.
			float4 blo, bhi;
			warp_box(need, q.x, q.y, q.z, blo, bhi);
			const float need_worst = warp_worst(need, t);
			const int c = id * 32 + lane;
			const bool has = c < lv.count[level - 1];
			float cb = INFINITY;
			if (has) {
				const int gc = lv.offset[level - 1] + c;
				cb = box_bound(__ldcg(box_lo + gc), __ldcg(box_hi + gc), make_float3(blo.x, blo.y, blo.z), make_float3(bhi.x, bhi.y, bhi.z));
			}
			const bool keep = has && !(cb > need_worst);
			const uint32_t m = __ballot_sync(0xFFFFFFFFu, keep);
			const int n = __popc(m);
			int rank = 0;
			for (uint32_t mm = m; mm; mm &= mm - 1) {
				const int o = __ffs(mm) - 1;
				const float bo = __shfl_sync(0xFFFFFFFFu, cb, o);
				rank += (bo < cb || (bo == cb && o < lane)) ? 1 : 0;
			}
			if (keep) { stk[top + n - 1 - rank] = ((uint32_t)(level - 1) << 27) | (uint32_t)c; stb[top + n - 1 - rank] = cb; }
			top += n;
			__syncwarp();
		}
	}
	if (live) {
		mean_d2[qi] = (t.d0 + t.d1 + t.d2) / 3.0f;  // b200gs_knn3's expression
		idx3[3 * (size_t)qi] = t.i0; idx3[3 * (size_t)qi + 1] = t.i1; idx3[3 * (size_t)qi + 2] = t.i2;
	}
}

bool knn_tree_p_ok(int32_t P) { return P >= 4 && P < (1 << 30); }

}  // namespace

extern "C" {

size_t b200gs_knn3_scratch_bytes(int32_t P) { return knn_tree_p_ok(P) ? layout_for(P).bytes : 0; }

int b200gs_knn3_tree(int32_t P, const float* xyz, float* mean_dist2, int32_t* indices, void* scratch, size_t scratch_bytes, void* stream_) {
	if (!knn_tree_p_ok(P)) return train_fail(B200GS_E_ARG, "knn3_tree: P must be in [4, 2^30)");
	if (!xyz || !mean_dist2 || !indices || !scratch) return train_fail(B200GS_E_ARG, "knn3_tree: null pointer");
	const Layout L = layout_for(P);
	if (scratch_bytes < L.bytes) return train_fail(B200GS_E_ARG, "knn3_tree: scratch too small (b200gs_knn3_scratch_bytes)");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	char* base = static_cast<char*>(scratch);
	auto u32 = [&](size_t off) { return reinterpret_cast<uint32_t*>(base + off); };
	auto f4 = [&](size_t off) { return reinterpret_cast<float4*>(base + off); };
	uint32_t* hdr = u32(L.hdr);
	uint32_t* hist = u32(L.hist);
	uint32_t* lookback = u32(L.lookback);
	cudaError_t e = cudaMemsetAsync(base, 0, L.zero_end, stream);
	if (e != cudaSuccess) return launch_status(e);
	const unsigned red_grid = (unsigned)min((P + 255) / 256, KNN_KEY_CTAS);
	launch(0u, knn_bounds_kernel, dim3(red_grid), dim3(256), 0, stream, (int)P, xyz, hdr);
	launch(0u, knn_keys_kernel, dim3(red_grid), dim3(256), 0, stream, (int)P, xyz, (const uint32_t*)hdr, u32(L.key_a), u32(L.hi),
	       u32(L.val_a), hist);
	// low word, then the high word in the low word's order: four passes each, results back in (key_a, val_a)
	const size_t lb_sort = (size_t)4 * L.tiles * 256;
	unsigned int* tickets = hdr + HDR_TICKETS;
	launch_radix_sort(u32(L.key_a), u32(L.key_b), u32(L.val_a), u32(L.val_b), P, nullptr, 32, hist, lookback, tickets,
	                  hdr + HDR_BARRIER, stream);
	launch(0u, knn_gather_hi_kernel, dim3((P + 255) / 256), dim3(256), 0, stream, (int)P, (const uint32_t*)u32(L.val_a),
	       (const uint32_t*)u32(L.hi), u32(L.key_a));
	launch_radix_sort(u32(L.key_a), u32(L.key_b), u32(L.val_a), u32(L.val_b), P, nullptr, 31, hist + 4 * 256, lookback + lb_sort,
	                  tickets + 4, hdr + HDR_BARRIER + 1, stream);
	float4 *lo = f4(L.box_lo), *hi = f4(L.box_hi);
	const int leaves = L.lv.count[0];
	launch(0u, knn_leaves_kernel, dim3((leaves + 7) / 8), dim3(256), 0, stream, (int)P, xyz, (const uint32_t*)u32(L.val_a), f4(L.pts), lo, hi,
	       leaves);
	for (int l = 1; l < L.lv.n; l++) {
		const int nodes = L.lv.count[l];
		launch(0u, knn_level_kernel, dim3((nodes + 7) / 8), dim3(256), 0, stream, (const float4*)(lo + L.lv.offset[l - 1]),
		       (const float4*)(hi + L.lv.offset[l - 1]), L.lv.count[l - 1], lo + L.lv.offset[l], hi + L.lv.offset[l], nodes);
	}
	return launch_status(launch(0u, knn_query_kernel, dim3((leaves + KNN_WARPS - 1) / KNN_WARPS), dim3(KNN_WARPS * 32), 0, stream, (int)P,
	                            (const float4*)f4(L.pts), (const float4*)lo, (const float4*)hi, L.lv, mean_dist2, indices));
}

}  // extern "C"
