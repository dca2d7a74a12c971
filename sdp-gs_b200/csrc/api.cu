// b200gs -- C-ABI entry points, workspace layout and stage orchestration (see include/b200gs.h).
//
// Stage order mirrors CudaRasterizer::Rasterizer::forward/backward
// (DGR/cuda_rasterizer/rasterizer_impl.cu:198-336, 340-434); what differs is documented in
// binning.cu / blend.cu.  Nothing here allocates device memory or touches the legacy default
// stream: the caller owns the three byte workspaces and passes the stream.
#include <atomic>
#include <mutex>
#include <string>
#include <vector>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include "common.cuh"

namespace {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
	return code;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- optional per-stage timing (CUDA events on the launch stream), used by bench.py for the roofline ----
enum Stage { ST_MEMSET = 0, ST_PREPROCESS, ST_DEPTH_SORT, ST_SCAN, ST_EMIT, ST_TILE_SORT, ST_RANGES, ST_BLEND_FWD,
             ST_BLEND_BWD, ST_PREPROCESS_BWD, ST_COUNT };
bool g_profile = false;
struct Pending { int stage; cudaEvent_t a, b; };
std::vector<Pending> g_pending;
std::vector<cudaEvent_t> g_free_events;
std::mutex g_prof_mu;
double g_stage_ms[ST_COUNT] = {0};
long long g_stage_n[ST_COUNT] = {0};

cudaEvent_t get_event() {
	if (!g_free_events.empty()) { cudaEvent_t e = g_free_events.back(); g_free_events.pop_back(); return e; }
	cudaEvent_t e;
	cudaEventCreate(&e);
	return e;
}
struct StageScope {
	cudaStream_t s; int stage; cudaEvent_t a;
	StageScope(cudaStream_t s_, int st) : s(s_), stage(st), a(nullptr) {
		if (g_profile) { std::lock_guard<std::mutex> l(g_prof_mu); a = get_event(); cudaEventRecord(a, s); }
	}
	~StageScope() {
		if (a) { std::lock_guard<std::mutex> l(g_prof_mu); cudaEvent_t b = get_event(); cudaEventRecord(b, s); g_pending.push_back({stage, a, b}); }
	}
};

template <typename T>
void carve(char*& p, T*& out, size_t count) {
	p = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(p), 256));
	out = reinterpret_cast<T*>(p);
	p += count * sizeof(T);
}

int check_stage(const b200gs_view_t* v, cudaStream_t s, const char* what) {
	cudaError_t e = cudaGetLastError();
	if (e == cudaSuccess && v->debug) e = cudaStreamSynchronize(s);  // CHECK_CUDA, auxiliary.h:166-173
	if (e != cudaSuccess) return fail(B200GS_E_CUDA, "[CUDA ERROR] in stage %s: %s", what, cudaGetErrorString(e));
	return 0;
}

}  // namespace

int train_fail(int code, const char* msg) { return fail(code, "%s", msg); }

int launch_status(cudaError_t e) {
	if (e == cudaSuccess) e = cudaGetLastError();
	return e == cudaSuccess ? 0 : fail(B200GS_E_CUDA, "%s", cudaGetErrorString(e));
}

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

const char* knob(Knob k) {
	static const char* const names[KNOB_COUNT] = {"B200GS_PDL", "B200GS_BLEND_WIDE", "B200GS_BLEND_CTAS", "B200GS_SCATTER_TMA"};
	static std::once_flag once[KNOB_COUNT];
	static std::string value[KNOB_COUNT];
	static bool set[KNOB_COUNT];
	std::call_once(once[k], [k] {
		if (const char* e = getenv(names[k])) { value[k] = e; set[k] = true; }
	});
	return set[k] ? value[k].c_str() : nullptr;
}

int knob_int(Knob k, int unset) {
	const char* e = knob(k);
	return e ? (int)strtol(e, nullptr, 0) : unset;
}

unsigned pdl_mask() { return (unsigned)knob_int(KNOB_PDL, 0xFF) & 0xFFu; }

static uint32_t higher_msb(uint32_t n) {  // getHigherMsb, DGR/cuda_rasterizer/rasterizer_impl.cu:35-50
	uint32_t msb = sizeof(n) * 4, step = msb;
	while (step > 1) {
		step /= 2;
		if (n >> msb) msb += step; else msb -= step;
	}
	if (n >> msb) msb++;
	return msb;
}

TileGrid tile_grid(int W, int H) {
	TileGrid t;
	t.W = W;
	t.H = H;
	t.gx = (W + TILE_X - 1) / TILE_X;
	t.gy = (H + TILE_Y - 1) / TILE_Y;
	t.tiles = (size_t)t.gx * t.gy;
	t.units = (uint32_t)(t.tiles * 8);
	t.tile_bits = (int)higher_msb((uint32_t)t.tiles);
	t.tile_passes = (t.tile_bits + 7) / 8;
	t.ranges_from_emit = t.tiles <= (size_t)COUNT_TILES_MAX;
	t.list_in_b = (t.tile_passes & 1) != 0;
	return t;
}

// geom layout: [hdr | hist | depth look-back (4 passes) | scan state] (zeroed per forward) then the arrays
GeomState geom_from_chunk(char* base, int P) {
	GeomState g;
	char* p = base;
	const size_t n = (size_t)(P > 0 ? P : 1);
	carve(p, g.hdr, 1);
	carve(p, g.hist, 8 * 256);
	carve(p, g.lookback, (size_t)4 * sort_tiles_for(P) * 256);
	carve(p, g.scan_state, (size_t)scan_tiles_for(P) + 1);
	g.clean_bytes = align_up((size_t)(p - base), 256);
	carve(p, g.depths, n);
	carve(p, g.rect, n);
	carve(p, g.rec, 4 * n);
	carve(p, g.clamped, n);
	carve(p, g.order, n);
	carve(p, g.key_a, n);
	carve(p, g.key_b, n);
	carve(p, g.val_b, n);
	g.bytes = align_up((size_t)(p - base), 256) + 256;
	return g;
}

ImageState image_from_chunk(char* base, const TileGrid& t) {
	ImageState s;
	char* p = base;
	const size_t N = (size_t)t.W * t.H, tiles = t.tiles;
	carve(p, s.ranges, tiles ? tiles : 1);
	carve(p, s.tile_order, tiles ? tiles : 1);
	carve(p, s.final_T, N ? N : 1);
	carve(p, s.n_contrib, N ? N : 1);
	carve(p, s.tile_count, (tiles ? tiles : 1) * (size_t)COUNT_STRIDE);
	carve(p, s.tile_cost, 2 * (tiles ? tiles : 1));
	carve(p, s.tile_order_bwd, tiles ? tiles : 1);
	s.bytes = align_up((size_t)(p - base), 256) + 256;
	return s;
}

BinningState binning_from_chunk(char* base, const TileGrid& t, int64_t capacity) {
	BinningState b;
	char* p = base;
	const size_t n = (size_t)(capacity > 0 ? capacity : 1);
	b.surv_words = n / 32 + t.tiles + 2;
	carve(p, b.lookback, (size_t)4 * sort_tiles_for(capacity) * 256);  // up to 4 tile passes (bit <= 32)
	carve(p, b.surv_bits, 8 * b.surv_words);
	carve(p, b.key_a, n);
	carve(p, b.key_b, n);
	carve(p, b.val_a, n);
	carve(p, b.val_b, n);
	b.sorted_keys = t.list_in_b ? b.key_b : b.key_a;  // where the tile sort's last pass leaves the list
	b.sorted_vals = t.list_in_b ? b.val_b : b.val_a;
	b.bytes = align_up((size_t)(p - base), 256) + 256;
	return b;
}

static RasterPlan plan_call(const b200gs_view_t* v, int P, const b200gs_workspace_t* ws, int64_t capacity) {
	RasterPlan pl;
	pl.v = v;
	pl.grid = tile_grid(v->width, v->height);
	pl.P = P;
	pl.capacity = capacity;
	pl.persistent = ws->persistent != 0;
	pl.gs = geom_from_chunk(reinterpret_cast<char*>(ws->geom), P);
	pl.is = image_from_chunk(reinterpret_cast<char*>(ws->image), pl.grid);
	pl.bs = binning_from_chunk(reinterpret_cast<char*>(ws->binning), pl.grid, capacity);
	return pl;
}

// Checks the arguments every rasterizer call shares and plans the call (`capacity` is checked by the callers that use it).
static int validate(RasterPlan& pl, const b200gs_view_t* v, const b200gs_gaussians_t* g, const b200gs_workspace_t* ws, int64_t capacity) {
	if (!v || !g || !ws) return fail(B200GS_E_ARG, "null argument");
	if (g->P < 0 || v->width <= 0 || v->height <= 0) return fail(B200GS_E_ARG, "bad sizes P=%d W=%d H=%d", g->P, v->width, v->height);
	pl = plan_call(v, g->P, ws, capacity);
	if (pl.grid.gx > 65535 || pl.grid.gy > 65535) return fail(B200GS_E_ARG, "image too large for 16-bit tile rects");
	if (g->P > 0) {
		if (!g->means3D || !g->opacities) return fail(B200GS_E_ARG, "means3D and opacities are required");
		if ((g->shs == nullptr) == (g->colors_precomp == nullptr))
			return fail(B200GS_E_ARG, "Please provide excatly one of either SHs or precomputed colors!");
		const bool sr = g->scales != nullptr && g->rotations != nullptr;
		if (sr == (g->cov3D_precomp != nullptr) || ((g->scales != nullptr) != (g->rotations != nullptr)))
			return fail(B200GS_E_ARG, "Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
		if (g->shs && v->sh_coeffs < (v->sh_degree + 1) * (v->sh_degree + 1))
			return fail(B200GS_E_ARG, "sh_coeffs=%d too small for sh_degree=%d", v->sh_coeffs, v->sh_degree);
		if (v->sh_degree < 0 || v->sh_degree > 3) return fail(B200GS_E_ARG, "sh_degree must be 0..3");
	}
	if (!v->background || !v->viewmatrix || !v->projmatrix || !v->campos) return fail(B200GS_E_ARG, "view pointers are required");
	if (!ws->geom || ws->geom_bytes < pl.gs.bytes) return fail(B200GS_E_ARG, "geom workspace too small");
	if (!ws->image || ws->image_bytes < pl.is.bytes) return fail(B200GS_E_ARG, "image workspace too small");
	return 0;
}

static int check_binning(const RasterPlan& pl, const b200gs_workspace_t* ws) {
	if (!ws->binning || ws->binning_bytes < pl.bs.bytes) return fail(B200GS_E_ARG, "binning workspace too small");
	return 0;
}

static int check_preprocess_args(const RasterPlan& pl, const b200gs_outputs_t* out) {
	if (!out || (pl.P > 0 && !out->radii)) return fail(B200GS_E_ARG, "radii output is required");
	return 0;
}

static int check_render_args(const RasterPlan& pl, const b200gs_outputs_t* out, const b200gs_workspace_t* ws) {
	if (!out || !out->color) return fail(B200GS_E_ARG, "color output is required");
	if (pl.v->extended && (!out->depth || !out->alpha || !out->feature)) return fail(B200GS_E_ARG, "extended outputs are required");
	if (pl.capacity < 0) return fail(B200GS_E_ARG, "negative capacity");
	if (pl.capacity >= (1ll << 30)) return fail(B200GS_E_ARG, "capacity exceeds 2^30 instances (30-bit look-back counters)");
	return check_binning(pl, ws);
}

static int forward_preprocess(const RasterPlan& pl, const b200gs_outputs_t* out, const b200gs_gaussians_t* g, cudaStream_t stream) {
	if (!pl.persistent || pl.P == 0) {  // persistent workspaces are left clean by the previous forward's blend kernel
		StageScope t(stream, ST_MEMSET);
		cudaMemsetAsync(pl.gs.hdr, 0, pl.gs.clean_bytes, stream);
		if (pl.P == 0) cudaMemsetAsync(pl.is.ranges, 0, pl.grid.tiles * sizeof(uint2), stream);  // otherwise zeroed by the preprocess kernel (rasterizer_impl.cu:310)
	}
	if (pl.P == 0) return 0;
	{ StageScope t(stream, ST_PREPROCESS); launch_preprocess_forward(pl, *g, out->radii, stream); }
	if (int e = check_stage(pl.v, stream, "preprocess")) return e;
	{ StageScope t(stream, ST_DEPTH_SORT); launch_depth_order(pl, stream); }
	return check_stage(pl.v, stream, "depth order");
}

// chained: the previous kernel in the stream is our depth sort
static int forward_render(const RasterPlan& pl, const b200gs_outputs_t* out, cudaStream_t stream, bool chained) {
	const bool emitted = pl.P > 0 && pl.capacity > 0;
	if (emitted) {
		{ StageScope t(stream, ST_EMIT); launch_scan_emit(pl, stream, chained); }
		if (int e = check_stage(pl.v, stream, "instance offsets / duplicate-with-keys")) return e;
		{ StageScope t(stream, ST_TILE_SORT); launch_tile_sort(pl, stream); }
		if (int e = check_stage(pl.v, stream, "tile sort")) return e;
	}
	if (pl.P > 0 && !emitted) launch_finalize_header(pl, stream);  // the status words scan_emit assigns
	if (!emitted || !pl.grid.ranges_from_emit) {  // small tile grids: scan_emit's last CTA already built ranges + schedule
		{ StageScope t(stream, ST_RANGES); launch_tile_ranges(pl, emitted ? pl.capacity : 0, stream); }
		if (int e = check_stage(pl.v, stream, "tile ranges / schedule")) return e;
	}
	{ StageScope t(stream, ST_BLEND_FWD); launch_blend_forward(pl, *out, stream); }
	return check_stage(pl.v, stream, "blend forward");
}

extern "C" {

int b200gs_version(void) { return B200GS_VERSION; }
const char* b200gs_last_error(void) { return g_err; }
int64_t b200gs_launch_count(void) { return g_launches.load(); }
void b200gs_profile_enable(int32_t on) { std::lock_guard<std::mutex> l(g_prof_mu); g_profile = on != 0; }
int b200gs_profile_read(double* ms_out, int64_t* n_out, int32_t reset) {
	std::lock_guard<std::mutex> l(g_prof_mu);
	for (auto& p : g_pending) {
		if (cudaEventSynchronize(p.b) != cudaSuccess) return fail(B200GS_E_CUDA, "profile event sync failed");
		float ms = 0.f;
		cudaEventElapsedTime(&ms, p.a, p.b);
		g_stage_ms[p.stage] += ms;
		g_stage_n[p.stage] += 1;
		g_free_events.push_back(p.a);
		g_free_events.push_back(p.b);
	}
	g_pending.clear();
	for (int i = 0; i < ST_COUNT; i++) {
		if (ms_out) ms_out[i] = g_stage_ms[i];
		if (n_out) n_out[i] = g_stage_n[i];
		if (reset) { g_stage_ms[i] = 0; g_stage_n[i] = 0; }
	}
	return 0;
}
void b200gs_abi_sizes(int64_t* out6) {
	out6[0] = sizeof(b200gs_view_t); out6[1] = sizeof(b200gs_gaussians_t); out6[2] = sizeof(b200gs_outputs_t);
	out6[3] = sizeof(b200gs_workspace_t); out6[4] = sizeof(b200gs_grad_outputs_t); out6[5] = sizeof(b200gs_grads_t);
}

size_t b200gs_geom_bytes(int32_t P) { return geom_from_chunk(nullptr, P).bytes; }
size_t b200gs_image_bytes(int32_t width, int32_t height) { return image_from_chunk(nullptr, tile_grid(width, height)).bytes; }
size_t b200gs_binning_bytes(int64_t capacity, int32_t width, int32_t height) {
	return binning_from_chunk(nullptr, tile_grid(width, height), capacity).bytes;
}
size_t b200gs_scratch_bytes(int32_t P) { return (size_t)(P > 0 ? P : 1) * GREC_FLOATS * sizeof(float); }

void b200gs_geom_layout(int32_t P, int64_t* off) {
	GeomState g = geom_from_chunk(nullptr, P);
	off[0] = (int64_t)reinterpret_cast<size_t>(g.hdr);
	off[1] = (int64_t)reinterpret_cast<size_t>(g.depths);
	off[2] = (int64_t)reinterpret_cast<size_t>(g.rect);
	off[3] = (int64_t)reinterpret_cast<size_t>(g.rec);
	off[4] = (int64_t)reinterpret_cast<size_t>(g.clamped);
	off[5] = (int64_t)reinterpret_cast<size_t>(g.order);
	off[6] = (int64_t)reinterpret_cast<size_t>(g.key_a);
}
void b200gs_image_layout(int32_t width, int32_t height, int64_t* off) {
	ImageState s = image_from_chunk(nullptr, tile_grid(width, height));
	off[0] = (int64_t)reinterpret_cast<size_t>(s.final_T);
	off[1] = (int64_t)reinterpret_cast<size_t>(s.n_contrib);
	off[2] = (int64_t)reinterpret_cast<size_t>(s.ranges);
}
void b200gs_binning_layout(int32_t width, int32_t height, int64_t capacity, int64_t* off) {
	BinningState b = binning_from_chunk(nullptr, tile_grid(width, height), capacity);
	off[0] = (int64_t)reinterpret_cast<size_t>(b.sorted_vals);
	off[1] = (int64_t)reinterpret_cast<size_t>(b.sorted_keys);
}

int b200gs_workspace_init(const b200gs_workspace_t* ws, int32_t P, void* scratch, void* stream_) {
	if (!ws || !ws->geom || P < 0 || ws->geom_bytes < b200gs_geom_bytes(P)) return fail(B200GS_E_ARG, "workspace_init: bad arguments");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	cudaError_t e = cudaMemsetAsync(ws->geom, 0, geom_from_chunk(nullptr, P).clean_bytes, stream);
	if (e == cudaSuccess && scratch) e = cudaMemsetAsync(scratch, 0, b200gs_scratch_bytes(P), stream);
	if (e == cudaSuccess && ws->image && ws->image_bytes) e = cudaMemsetAsync(ws->image, 0, ws->image_bytes, stream);  // no cost history yet
	if (e != cudaSuccess) return fail(B200GS_E_CUDA, "[CUDA ERROR] workspace_init: %s", cudaGetErrorString(e));
	return 0;
}

int b200gs_forward_preprocess(const b200gs_view_t* v, const b200gs_gaussians_t* g, const b200gs_outputs_t* out,
                              const b200gs_workspace_t* ws, void* stream_, int64_t* num_rendered_host) {
	RasterPlan pl;
	if (int e = validate(pl, v, g, ws, 0)) return e;
	if (int e = check_preprocess_args(pl, out)) return e;
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	if (int e = forward_preprocess(pl, out, g, stream)) return e;
	if (num_rendered_host) {
		unsigned long long n = 0;
		cudaError_t e = cudaMemcpyAsync(&n, &pl.gs.hdr->num_acc, sizeof(n), cudaMemcpyDeviceToHost, stream);
		if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
		if (e != cudaSuccess) return fail(B200GS_E_CUDA, "[CUDA ERROR] reading num_rendered: %s", cudaGetErrorString(e));
		*num_rendered_host = (int64_t)n;
	}
	return 0;
}

int b200gs_forward_render(const b200gs_view_t* v, const b200gs_gaussians_t* g, const b200gs_outputs_t* out,
                          const b200gs_workspace_t* ws, int64_t capacity, void* stream) {
	RasterPlan pl;
	if (int e = validate(pl, v, g, ws, capacity)) return e;
	if (int e = check_render_args(pl, out, ws)) return e;
	return forward_render(pl, out, reinterpret_cast<cudaStream_t>(stream), false);
}

int b200gs_forward(const b200gs_view_t* v, const b200gs_gaussians_t* g, const b200gs_outputs_t* out,
                   const b200gs_workspace_t* ws, int64_t capacity, void* stream_) {
	RasterPlan pl;
	if (int e = validate(pl, v, g, ws, capacity)) return e;
	if (int e = check_preprocess_args(pl, out)) return e;
	if (int e = check_render_args(pl, out, ws)) return e;
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	if (int e = forward_preprocess(pl, out, g, stream)) return e;
	return forward_render(pl, out, stream, pl.P > 0);
}

int b200gs_forward_status(const b200gs_workspace_t* ws, void* stream_, int64_t* num_rendered, int32_t* overflow) {
	if (!ws || !ws->geom) return fail(B200GS_E_ARG, "null workspace");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	GeomHeader h;
	cudaError_t e = cudaMemcpyAsync(&h, ws->geom, sizeof(h), cudaMemcpyDeviceToHost, stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
	if (e != cudaSuccess) return fail(B200GS_E_CUDA, "[CUDA ERROR] reading status: %s", cudaGetErrorString(e));
	if (num_rendered) *num_rendered = (int64_t)h.num_rendered;
	if (overflow) *overflow = (int32_t)h.overflow;
	if (h.overflow & 2u) return fail(B200GS_E_ARG, "Point is filtered although prefiltered is set. This shouldn't happen!");
	if (h.overflow & 1u) return fail(B200GS_E_OVERFLOW, "num_rendered=%lld exceeds the binning capacity", (long long)h.num_rendered);
	return 0;
}

size_t b200gs_camera_scratch_bytes(int32_t P) { return camera_scratch_bytes(P); }
int64_t b200gs_camera_grads_abi_size(void) { return (int64_t)sizeof(b200gs_camera_grads_t); }

int b200gs_backward(const b200gs_view_t* v, const b200gs_gaussians_t* g, const int32_t* radii,
                    const b200gs_workspace_t* ws, int64_t capacity, const b200gs_grad_outputs_t* gout,
                    const b200gs_grads_t* grads, void* stream) {
	return b200gs_backward_camera(v, g, radii, ws, capacity, gout, grads, nullptr, stream);
}

int b200gs_backward_camera(const b200gs_view_t* v, const b200gs_gaussians_t* g, const int32_t* radii,
                           const b200gs_workspace_t* ws, int64_t capacity, const b200gs_grad_outputs_t* gout,
                           const b200gs_grads_t* grads, const b200gs_camera_grads_t* cam, void* stream_) {
	RasterPlan pl;
	if (int e = validate(pl, v, g, ws, capacity)) return e;
	if (!gout || !grads) return fail(B200GS_E_ARG, "null gradient structs");
	if (cam) {
		if (!cam->dL_dviewmatrix || !cam->dL_dprojmatrix || !cam->dL_dcampos || !cam->scratch)
			return fail(B200GS_E_ARG, "camera gradients: dL_dviewmatrix, dL_dprojmatrix, dL_dcampos and scratch are required");
		if (grads->scatter_bases)
			return fail(B200GS_E_ARG, "camera gradients are not supported together with the gradient scatter (scatter_bases)");
	}
	const int P = g->P;
	if (P == 0) {  // rasterize_points.cu:161; the camera gradients of an empty scene are zero
		if (!cam) return 0;
		cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
		cudaError_t e = cudaMemsetAsync(cam->dL_dviewmatrix, 0, 16 * sizeof(float), stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(cam->dL_dprojmatrix, 0, 16 * sizeof(float), stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(cam->dL_dcampos, 0, 3 * sizeof(float), stream);
		if (e != cudaSuccess) return fail(B200GS_E_CUDA, "[CUDA ERROR] zeroing camera gradients: %s", cudaGetErrorString(e));
		return 0;
	}
	if (!radii || !grads->scratch) return fail(B200GS_E_ARG, "radii and scratch are required");
	if (grads->scatter_bases) {
		if (grads->scatter_world < 2 || grads->scatter_rank < 0 || grads->scatter_rank >= grads->scatter_world || grads->scatter_shard_rows <= 0 ||
		    (grads->scatter_shard_rows & 127) || grads->scatter_shard_rows * grads->scatter_world < P)
			return fail(B200GS_E_ARG, "bad gradient scatter descriptor (shard_rows must be a multiple of 128 and cover P)");
		if (!g->shs || v->sh_coeffs != 16 || !g->scales || !g->rotations)
			return fail(B200GS_E_ARG, "gradient scatter needs shs with 16 coefficients and the scales/rotations path");
	}
	if (int e = check_binning(pl, ws)) return e;
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	float* grec = reinterpret_cast<float*>(grads->scratch);
	if (!pl.persistent) { StageScope t(stream, ST_MEMSET); cudaMemsetAsync(grec, 0, b200gs_scratch_bytes(P), stream); }
	{ StageScope t(stream, ST_BLEND_BWD); launch_blend_backward(pl, *gout, grec, stream); }
	if (int e = check_stage(v, stream, "blend backward")) return e;
	{ StageScope t(stream, ST_PREPROCESS_BWD); launch_preprocess_backward(pl, *g, radii, grec, *grads, cam, stream); }
	return check_stage(v, stream, "preprocess backward");
}

int b200gs_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                        uint8_t* present, void* stream_) {
	(void)projmatrix;  // the reference computes p_proj but its frustum test only uses p_view.z (auxiliary.h:154)
	if (P < 0 || (P > 0 && (!means3D || !viewmatrix || !present))) return fail(B200GS_E_ARG, "bad arguments");
	if (P == 0) return 0;
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	launch_mark_visible(P, means3D, viewmatrix, present, stream);
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return fail(B200GS_E_CUDA, "[CUDA ERROR] mark_visible: %s", cudaGetErrorString(e));
	return 0;
}

int b200gs_debug_sorted_keys(const b200gs_view_t* v, int32_t P, const b200gs_workspace_t* ws, int64_t capacity,
                             uint64_t* keys_out, int64_t L, void* stream_) {
	if (!v || !ws || !keys_out || !ws->geom || !ws->binning) return fail(B200GS_E_ARG, "null argument");
	if (L > capacity) return fail(B200GS_E_ARG, "L exceeds capacity");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	launch_debug_keys(plan_call(v, P, ws, capacity), keys_out, L, stream);
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return fail(B200GS_E_CUDA, "[CUDA ERROR] debug keys: %s", cudaGetErrorString(e));
	return 0;
}

}  // extern "C"
