// b200gs -- per-Gaussian stages: preprocess forward (K1), preprocess backward (K8+K9 fused), markVisible.
//
// Forward semantics follow DGR/cuda_rasterizer/forward.cu:155-256 (preprocessCUDA), :74-113
// (computeCov2D), :118-152 (computeCov3D), :20-71 (computeColorFromSH == utils/sh_utils.py:57-112)
// and auxiliary.h:41-56,139-164 (ndc2Pix, getRect, in_frustum).  radii, depth bits and tile rects
// are part of the bit-exact contract, so every operation that feeds them is written with
// round-to-nearest intrinsics in the order the reference's sm_100a build executes them (read off
// its SASS: cicc *and* ptxas contract mul+add into fma there, e.g. det = fma(a, c, -(b*b))).
#include "common.cuh"
#include "tma.cuh"

namespace {

__constant__ float kSH_C0 = 0.28209479177387814f;
__constant__ float kSH_C1 = 0.4886025119029199f;
__constant__ float kSH_C2[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f,
                                -1.0925484305920792f, 0.5462742152960396f};
__constant__ float kSH_C3[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f, 0.3731763325901154f,
                                -0.4570457994644658f, 1.445305721320277f, -0.5900435899266435f};

struct ViewConsts {
	float view[16];
	float proj[16];
	float campos[3];
};

__device__ __forceinline__ void load_view(ViewConsts& vc, const float* __restrict__ view, const float* __restrict__ proj,
                                          const float* __restrict__ campos) {
#pragma unroll
	for (int i = 0; i < 16; i++) { vc.view[i] = __ldg(view + i); vc.proj[i] = __ldg(proj + i); }
	vc.campos[0] = __ldg(campos); vc.campos[1] = __ldg(campos + 1); vc.campos[2] = __ldg(campos + 2);
}

// computeCov3D forward with the reference build's rounding sequence.
__device__ __forceinline__ void cov3d_pinned(float s0, float s1, float s2, float mod, float4 q, float* cov) {
	const float sx = __fmul_rn(mod, s0), sy = __fmul_rn(mod, s1), sz = __fmul_rn(mod, s2);
	const float r = q.x, x = q.y, y = q.z, z = q.w;
	const float xz = __fmul_rn(x, z), rx = __fmul_rn(r, x), rz = __fmul_rn(r, z);
	const float yy = __fmul_rn(y, y), zz = __fmul_rn(z, z);
	const float xz_p_ry = __fmaf_rn(r, y, xz), xz_m_ry = __fmaf_rn(-r, y, xz);
	const float yz_m_rx = __fmaf_rn(y, z, -rx), yz_p_rx = __fmaf_rn(y, z, rx);
	const float xy_m_rz = __fmaf_rn(x, y, -rz), xy_p_rz = __fmaf_rn(x, y, rz);
	const float xx_yy = __fmaf_rn(x, x, yy), yy_zz = __fadd_rn(yy, zz), xx_zz = __fmaf_rn(x, x, zz);
	const float M00 = __fmul_rn(sx, __fsub_rn(1.0f, __fadd_rn(yy_zz, yy_zz)));
	const float M01 = __fmul_rn(sy, __fadd_rn(xy_m_rz, xy_m_rz));
	const float M02 = __fmul_rn(sz, __fadd_rn(xz_p_ry, xz_p_ry));
	const float M10 = __fmul_rn(sx, __fadd_rn(xy_p_rz, xy_p_rz));
	const float M11 = __fmul_rn(sy, __fsub_rn(1.0f, __fadd_rn(xx_zz, xx_zz)));
	const float M12 = __fmul_rn(sz, __fadd_rn(yz_m_rx, yz_m_rx));
	const float M20 = __fmul_rn(sx, __fadd_rn(xz_m_ry, xz_m_ry));
	const float M21 = __fmul_rn(sy, __fadd_rn(yz_p_rx, yz_p_rx));
	const float M22 = __fmul_rn(sz, __fsub_rn(1.0f, __fadd_rn(xx_yy, xx_yy)));
	cov[0] = dot3_pinned(M00, M00, M01, M01, M02, M02);
	cov[1] = dot3_pinned(M00, M10, M01, M11, M02, M12);
	cov[2] = dot3_pinned(M00, M20, M01, M21, M02, M22);
	cov[3] = dot3_pinned(M10, M10, M11, M11, M12, M12);
	cov[4] = dot3_pinned(M10, M20, M11, M21, M12, M22);
	cov[5] = dot3_pinned(M20, M20, M21, M21, M22, M22);
}

__device__ __forceinline__ float ndc2pix_pinned(float v, int S) {
	double t = __dadd_rn((double)v, 1.0);
	t = __fma_rn(t, (double)S, -1.0);
	return __double2float_rn(__dmul_rn(t, 0.5));
}

// SH -> RGB (+0.5, clamp at 0, remember which channels clamped)
__device__ __forceinline__ void sh_to_rgb(int deg, const float* __restrict__ sh, float dx, float dy, float dz,
                                          float* rgb, unsigned& clamp_bits) {
	const float len = __fsqrt_rn(dot3_pinned(dx, dx, dy, dy, dz, dz));
	const float x = __fdiv_rn(dx, len), y = __fdiv_rn(dy, len), z = __fdiv_rn(dz, len);
	float res[3];
#pragma unroll
	for (int c = 0; c < 3; c++) res[c] = kSH_C0 * sh[c];
	if (deg > 0) {
		const float c1y = y * kSH_C1, c1z = z * kSH_C1, c1x = x * kSH_C1;
#pragma unroll
		for (int c = 0; c < 3; c++) {
			res[c] = res[c] - c1y * sh[3 + c];
			res[c] = fmaf(c1z, sh[6 + c], res[c]);
			res[c] = res[c] - c1x * sh[9 + c];
		}
		if (deg > 1) {
			const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
			const float k4 = xy * kSH_C2[0], k5 = yz * kSH_C2[1], k6 = ((zz + zz) - xx - yy) * kSH_C2[2];
			const float k7 = xz * kSH_C2[3], k8 = (xx - yy) * kSH_C2[4];
#pragma unroll
			for (int c = 0; c < 3; c++) {
				res[c] = fmaf(k4, sh[12 + c], res[c]);
				res[c] = fmaf(k5, sh[15 + c], res[c]);
				res[c] = fmaf(k6, sh[18 + c], res[c]);
				res[c] = fmaf(k7, sh[21 + c], res[c]);
				res[c] = fmaf(k8, sh[24 + c], res[c]);
			}
			if (deg > 2) {
				const float k9 = (y * kSH_C3[0]) * (xx * 3.0f - yy);
				const float k10 = z * (xy * kSH_C3[1]);
				const float k11 = (y * kSH_C3[2]) * (zz * 4.0f - xx - yy);
				const float k12 = (z * kSH_C3[3]) * ((zz + zz) - xx * 3.0f - yy * 3.0f);
				const float k13 = (x * kSH_C3[4]) * (zz * 4.0f - xx - yy);
				const float k14 = (z * kSH_C3[5]) * (xx - yy);
				const float k15 = (x * kSH_C3[6]) * (xx - yy * 3.0f);
#pragma unroll
				for (int c = 0; c < 3; c++) {
					res[c] = fmaf(k9, sh[27 + c], res[c]);
					res[c] = fmaf(k10, sh[30 + c], res[c]);
					res[c] = fmaf(k11, sh[33 + c], res[c]);
					res[c] = fmaf(k12, sh[36 + c], res[c]);
					res[c] = fmaf(k13, sh[39 + c], res[c]);
					res[c] = fmaf(k14, sh[42 + c], res[c]);
					res[c] = fmaf(k15, sh[45 + c], res[c]);
				}
			}
		}
	}
	clamp_bits = 0;
#pragma unroll
	for (int c = 0; c < 3; c++) {
		res[c] += 0.5f;
		if (res[c] < 0.0f) clamp_bits |= 1u << c;
		rgb[c] = fmaxf(res[c], 0.0f);
	}
}

// One CTA handles PRE_THREADS consecutive Gaussians.  Their attribute arrays are array-of-structs with odd strides
// (12, 16, 24, 12*M bytes), which makes per-thread global loads touch ~20 sectors per request (ncu, round 1).  The
// CTA's slice of every array is contiguous in memory, so it is brought into shared memory whole: by the TMA bulk-copy
// engine (cp.async.bulk + mbarrier) when the slice is a full, 16-byte aligned tile, by coalesced loads otherwise.
constexpr int PRE_THREADS = 128;

struct Stage {
	uint64_t* bar;
	uint32_t tx;
	bool tma;
	int cnt;
	int tid;
	__device__ __forceinline__ void load(float* dst, const float* src, int floats_per_item, size_t base) {
		if (src == nullptr) return;
		const float* g = src + base * floats_per_item;
		if (tma) {
			if (tid == 0) { const uint32_t bytes = (uint32_t)(PRE_THREADS * floats_per_item * 4); tma_load_1d(dst, g, bytes, bar); }
		} else {
			for (int i = tid; i < cnt * floats_per_item; i += PRE_THREADS) dst[i] = g[i];
		}
	}
};

__global__ void __launch_bounds__(PRE_THREADS) preprocess_forward_kernel(
	int P, int D, int M, const float* __restrict__ means3D, const float* __restrict__ scales, float scale_modifier,
	const float* __restrict__ rotations, const float* __restrict__ opacities, const float* __restrict__ shs,
	const float* __restrict__ cov3D_precomp, const float* __restrict__ colors_precomp,
	const float* __restrict__ feat_precomp, const float* __restrict__ shs_language, const float* __restrict__ confidence,
	const float* __restrict__ viewmatrix, const float* __restrict__ projmatrix, const float* __restrict__ campos,
	int W, int H, float tan_fovx, float tan_fovy, float focal_x, float focal_y, int extended, int prefiltered,
	int32_t* __restrict__ radii, float* __restrict__ depths, ushort4* __restrict__ rects, float4* __restrict__ rec,
	uint8_t* __restrict__ clamped, uint32_t* __restrict__ sort_keys, uint32_t* __restrict__ sort_vals,
	uint32_t* __restrict__ depth_hist /*[4][256]: digit histograms of all four depth-sort passes*/, uint2* __restrict__ ranges, uint32_t* __restrict__ tile_count, int count_stride, int tiles, GeomHeader* __restrict__ hdr,
	int tma_ok, const uint32_t* live_count)
{
	// digit histograms of the depth-sort keys for all four radix passes that follow (taken here, where the key is
	// produced: one conflict-bounded shared-memory atomic per digit per Gaussian; taking them inside the passes cost
	// 16 same-address atomics per thread on the skewed exponent byte -- ncu: 110 us instead of 45 us per pass at P = 6 M)
	__shared__ uint32_t s_hist[4][256];
	__shared__ unsigned long long s_instances;
	__shared__ __align__(128) float s_sh[PRE_THREADS * 48];     // SH coefficients (M <= 16) or precomputed colours
	__shared__ __align__(16) float s_means[PRE_THREADS * 3];
	__shared__ __align__(16) float s_geo[PRE_THREADS * 7];      // scales [0,3T) + rotations [3T,7T), or cov3D_precomp [0,6T)
	__shared__ __align__(16) float s_opac[PRE_THREADS];
	__shared__ __align__(16) float s_conf[PRE_THREADS];
	__shared__ __align__(16) float s_feat[PRE_THREADS * 3];     // language_feature_precomp or shs_language
	// outgoing splat records: staged in the SH buffer once every thread is done with its coefficients (8 KB less shared
	// memory = 6 instead of 5 CTAs per SM: the 782 CTAs of the 100 k-Gaussian shape then fit ONE wave of 888 slots instead of
	// one and a 6 % tail wave, which had doubled the kernel's latency-bound duration)
	float4* s_rec = reinterpret_cast<float4*>(s_sh);
	__shared__ __align__(8) uint64_t s_bar;
	const int li = threadIdx.x;
	pdl_trigger();
	const size_t base = (size_t)blockIdx.x * PRE_THREADS;
	const int cnt = (int)min((size_t)PRE_THREADS, (size_t)P - base);
	const bool sh_staged = shs != nullptr && M <= 16;
	Stage st;
	st.bar = &s_bar; st.tma = tma_ok && cnt == PRE_THREADS; st.cnt = cnt; st.tid = li;
	if (li == 0 && st.tma) mbar_init(&s_bar, 1);
	for (int i = threadIdx.x; i < 4 * 256; i += blockDim.x) (&s_hist[0][0])[i] = 0;
	if (threadIdx.x == 0) s_instances = 0ull;
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	pdl_wait();  // the parameters may have been written by the kernel just before this one (optimizer step)
	// tile ranges start at (0,0) for every tile (cudaMemset in the reference, rasterizer_impl.cu:310); per-tile instance counters at 0
	for (int t = idx; t < tiles; t += gridDim.x * blockDim.x) { ranges[t] = make_uint2(0u, 0u); tile_count[(size_t)t * count_stride] = 0u; }
	__syncthreads();
	if (li == 0 && st.tma) {
		uint32_t tx = PRE_THREADS * 4 * (3 + 1);
		tx += (cov3D_precomp != nullptr) ? PRE_THREADS * 4 * 6 : PRE_THREADS * 4 * 7;
		if (sh_staged) tx += PRE_THREADS * 4 * 3 * M;
		if (colors_precomp != nullptr) tx += PRE_THREADS * 4 * 3;
		if (confidence != nullptr) tx += PRE_THREADS * 4;
		if (extended && (feat_precomp != nullptr || shs_language != nullptr)) tx += PRE_THREADS * 4 * 3;
		mbar_arrive_expect_tx(&s_bar, tx);
	}
	st.load(s_means, means3D, 3, base);
	st.load(s_opac, opacities, 1, base);
	if (cov3D_precomp != nullptr) st.load(s_geo, cov3D_precomp, 6, base);
	else { st.load(s_geo, scales, 3, base); st.load(s_geo + 3 * PRE_THREADS, rotations, 4, base); }
	if (sh_staged) st.load(s_sh, shs, 3 * M, base);
	if (colors_precomp != nullptr) st.load(s_sh, colors_precomp, 3, base);
	if (confidence != nullptr) st.load(s_conf, confidence, 1, base);
	if (extended) st.load(s_feat, feat_precomp != nullptr ? feat_precomp : shs_language, 3, base);
	if (st.tma) mbar_wait(&s_bar, 0);
	else __syncthreads();
	float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0, r2 = r0, r3 = r0;
	uint32_t touched = 0;
	if (idx < P) {
	ViewConsts vc;
	load_view(vc, viewmatrix, projmatrix, campos);
	const float* v = vc.view;

	// defaults for a culled Gaussian: radius 0, empty rect, sorts last (no instances are emitted for it)
	int32_t out_radius = 0;
	ushort4 out_rect = make_ushort4(0, 0, 0, 0);
	uint32_t out_key = 0xFFFFFFFFu;

	const float x = s_means[3 * li], y = s_means[3 * li + 1], z = s_means[3 * li + 2];
	const float pz = xform_row(v, 2, x, y, z);
	bool alive = !(pz <= 0.2f);  // in_frustum, auxiliary.h:154
	if (!alive && prefiltered) atomicOr(&hdr->prefilter_violation, 2u);  // reference: printf + __trap (auxiliary.h:156-160)
	if (live_count != nullptr && (uint32_t)idx >= __ldcg(live_count)) alive = false;  // a spare row of a capacity-sized buffer (b200gs_gaussians_t.live_count)

	if (alive) {
		const float hx = xform_row(vc.proj, 0, x, y, z), hy = xform_row(vc.proj, 1, x, y, z);
		const float hw = xform_row(vc.proj, 3, x, y, z);
		const float p_w = __frcp_rn(__fadd_rn(hw, 0.0000001f));
		const float projx = __fmul_rn(hx, p_w), projy = __fmul_rn(hy, p_w);

		float c3[6];
		if (cov3D_precomp != nullptr) {
#pragma unroll
			for (int i = 0; i < 6; i++) c3[i] = s_geo[6 * li + i];
		} else {
			const float4 q = reinterpret_cast<const float4*>(s_geo + 3 * PRE_THREADS)[li];
			cov3d_pinned(s_geo[3 * li], s_geo[3 * li + 1], s_geo[3 * li + 2], scale_modifier, q, c3);
		}
		// computeCov2D
		const float tx = xform_row(v, 0, x, y, z), ty = xform_row(v, 1, x, y, z), tz = pz;
		const float limx = __fmul_rn(tan_fovx, 1.3f), limy = __fmul_rn(tan_fovy, 1.3f);
		const float cx = fminf(limx, fmaxf(-limx, __fdiv_rn(tx, tz)));
		const float cy = fminf(limy, fmaxf(-limy, __fdiv_rn(ty, tz)));
		const float tz2 = __fmul_rn(tz, tz);
		const float J00 = __fdiv_rn(focal_x, tz), J02 = __fdiv_rn(__fmul_rn(__fmul_rn(tz, -cx), focal_x), tz2);
		const float J11 = __fdiv_rn(focal_y, tz), J12 = __fdiv_rn(__fmul_rn(__fmul_rn(tz, -cy), focal_y), tz2);
		const float T00 = __fmaf_rn(v[2], J02, __fmul_rn(v[0], J00));
		const float T01 = __fmaf_rn(v[6], J02, __fmul_rn(v[4], J00));
		const float T02 = __fmaf_rn(v[10], J02, __fmul_rn(v[8], J00));
		const float T10 = __fmaf_rn(v[2], J12, __fmul_rn(v[1], J11));
		const float T11 = __fmaf_rn(v[6], J12, __fmul_rn(v[5], J11));
		const float T12 = __fmaf_rn(v[10], J12, __fmul_rn(v[9], J11));
		const float A00 = dot3_pinned(T00, c3[0], T01, c3[1], T02, c3[2]);
		const float A01 = dot3_pinned(T10, c3[0], T11, c3[1], T12, c3[2]);
		const float A10 = dot3_pinned(T00, c3[1], T01, c3[3], T02, c3[4]);
		const float A11 = dot3_pinned(T10, c3[1], T11, c3[3], T12, c3[4]);
		const float A20 = dot3_pinned(T00, c3[2], T01, c3[4], T02, c3[5]);
		const float A21 = dot3_pinned(T10, c3[2], T11, c3[4], T12, c3[5]);
		const float a = __fadd_rn(dot3_pinned(T00, A00, T01, A10, T02, A20), 0.3f);
		const float b = dot3_pinned(T00, A01, T01, A11, T02, A21);
		const float c = __fadd_rn(dot3_pinned(T10, A01, T11, A11, T12, A21), 0.3f);
		const float det = __fmaf_rn(a, c, -__fmul_rn(b, b));
		if (det == 0.0f) alive = false;
		if (alive) {
			const float det_inv = __frcp_rn(det);
			const float mid = __fmul_rn(__fadd_rn(a, c), 0.5f);
			const float sq = __fsqrt_rn(fmaxf(__fmaf_rn(mid, mid, -det), 0.1f));
			const float lam = fmaxf(__fadd_rn(mid, sq), __fsub_rn(mid, sq));
			const int irad = (int)ceilf(__fmul_rn(__fsqrt_rn(lam), 3.0f));
			const float pxi = ndc2pix_pinned(projx, W), pyi = ndc2pix_pinned(projy, H);
			// getRect (auxiliary.h:46-56)
			const unsigned gx = (W + TILE_X - 1) / TILE_X, gy = (H + TILE_Y - 1) / TILE_Y;
			const float r = (float)irad;
			const unsigned x0 = min(gx, (unsigned)max(0, (int)__fmul_rn(__fsub_rn(pxi, r), 0.0625f)));
			const unsigned y0 = min(gy, (unsigned)max(0, (int)__fmul_rn(__fsub_rn(pyi, r), 0.0625f)));
			const unsigned x1 = min(gx, (unsigned)max(0, (int)__fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(pxi, r), 16.0f), -1.0f), 0.0625f)));
			const unsigned y1 = min(gy, (unsigned)max(0, (int)__fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(pyi, r), 16.0f), -1.0f), 0.0625f)));
			if ((x1 - x0) * (y1 - y0) != 0) {
				float rgb[3];
				unsigned clamp_bits = 0;
				if (colors_precomp != nullptr) {
					rgb[0] = s_sh[3 * li]; rgb[1] = s_sh[3 * li + 1]; rgb[2] = s_sh[3 * li + 2];
				} else {
					if (sh_staged && M == 16) {
						// 12 x LDS.128 (row stride 192 B: 4-way bank conflict) instead of 48 scalar loads (16-way)
						float shr[48];
						const float4* row = reinterpret_cast<const float4*>(s_sh + li * 48);
#pragma unroll
						for (int j = 0; j < 12; j++) { const float4 t4 = row[j]; shr[4 * j] = t4.x; shr[4 * j + 1] = t4.y; shr[4 * j + 2] = t4.z; shr[4 * j + 3] = t4.w; }
						sh_to_rgb(D, shr, __fsub_rn(x, vc.campos[0]), __fsub_rn(y, vc.campos[1]), __fsub_rn(z, vc.campos[2]), rgb, clamp_bits);
					} else {
						sh_to_rgb(D, sh_staged ? s_sh + li * M * 3 : shs + (size_t)idx * M * 3, __fsub_rn(x, vc.campos[0]), __fsub_rn(y, vc.campos[1]),
						          __fsub_rn(z, vc.campos[2]), rgb, clamp_bits);
					}
				}
				float f[3] = {rgb[0], rgb[1], rgb[2]};  // include_feature=False: feature aliases colour
				if (extended) {
					if (feat_precomp != nullptr) {
						f[0] = s_feat[3 * li]; f[1] = s_feat[3 * li + 1]; f[2] = s_feat[3 * li + 2];
					} else if (shs_language != nullptr) {  // gaussian_renderer/__init__.py:283-287
						const float v0 = kSH_C0 * s_feat[3 * li], v1 = kSH_C0 * s_feat[3 * li + 1];
						const float v2 = kSH_C0 * s_feat[3 * li + 2];
						const float inv = 1.0f / (sqrtf(v0 * v0 + v1 * v1 + v2 * v2) + 1e-9f);
						f[0] = v0 * inv; f[1] = v1 * inv; f[2] = v2 * inv;
					}
				}
				float o = s_opac[li];
				if (confidence != nullptr) o *= s_conf[li];
				const float ca = __fmul_rn(c, det_inv), cb = __fmul_rn(b, -det_inv), cc = __fmul_rn(a, det_inv);
				// warp-level cull helpers for the blend kernels (conservative, see blend.cu)
				const float thr = 2.0f * logf(255.0f * o);
				r0 = make_float4(pxi, pyi, ca, cb);
				r1 = make_float4(cc, o, thr, -cb / cc);
				r2 = make_float4(rgb[0], rgb[1], rgb[2], pz);
				r3 = make_float4(f[0], f[1], f[2], 0.f);
				clamped[idx] = (uint8_t)clamp_bits;
				depths[idx] = pz;
				out_radius = irad;
				out_rect = make_ushort4((unsigned short)x0, (unsigned short)y0, (unsigned short)x1, (unsigned short)y1);
				out_key = __float_as_uint(pz);
			}
		}
	}
	radii[idx] = out_radius;
	rects[idx] = out_rect;
	sort_keys[idx] = out_key;
	sort_vals[idx] = (uint32_t)idx;
	atomicAdd(&s_hist[0][out_key & 255u], 1u);
	atomicAdd(&s_hist[1][(out_key >> 8) & 255u], 1u);
	atomicAdd(&s_hist[2][(out_key >> 16) & 255u], 1u);
	atomicAdd(&s_hist[3][out_key >> 24], 1u);
	touched = (uint32_t)(out_rect.z - out_rect.x) * (uint32_t)(out_rect.w - out_rect.y);
	}
	{
		const uint32_t wsum = __reduce_add_sync(0xFFFFFFFFu, touched);  // < 2^32 per warp: 32 x 65535^2 cannot be reached by 16-bit x 16-bit tile grids in practice
		if ((li & 31) == 0 && wsum) atomicAdd(&s_instances, (unsigned long long)wsum);
	}
	// splat records leave the CTA as one contiguous bulk store
	__syncthreads();  // every thread has read its SH row / colour: the buffer is free for the records
	s_rec[4 * li] = r0; s_rec[4 * li + 1] = r1; s_rec[4 * li + 2] = r2; s_rec[4 * li + 3] = r3;
	tma_store_fence();
	__syncthreads();
	if (li == 0) {
		tma_store_1d(rec + 4 * base, s_rec, (uint32_t)cnt * 64u);
		tma_store_commit();
		tma_store_wait_read();
	}
	// num_rendered = total number of (Gaussian, tile) instances (what the reference reads back after its scan, rasterizer_impl.cu:281)
	if (threadIdx.x == 0 && s_instances) atomicAdd(&hdr->num_acc, s_instances);
	for (int i = threadIdx.x; i < 4 * 256; i += blockDim.x) {
		const uint32_t c = (&s_hist[0][0])[i];
		if (c) atomicAdd(depth_hist + i, c);
	}
}

__global__ void __launch_bounds__(256) mark_visible_kernel(int P, const float* __restrict__ means3D,
                                                           const float* __restrict__ viewmatrix, uint8_t* __restrict__ present) {
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= P) return;
	float v[16];
#pragma unroll
	for (int i = 0; i < 16; i++) v[i] = __ldg(viewmatrix + i);
	const float pz = xform_row(v, 2, __ldg(means3D + 3 * idx), __ldg(means3D + 3 * idx + 1), __ldg(means3D + 3 * idx + 2));
	present[idx] = !(pz <= 0.2f);  // checkFrustum, rasterizer_impl.cu:54-66
}

// ---------------------------------------------------------------------------------------------
// Backward: computeCov2DCUDA (backward.cu:144-274) + preprocessCUDA (:346-396) + SH backward
// (:20-139) + computeCov3D backward (:278-341), fused into one pass that also writes the zeros
// the reference gets from nine torch::zeros fills (rasterize_points.cu:151-159).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void store3(float* p, size_t i, float a, float b, float c) {
	if (p) { p[3 * i] = a; p[3 * i + 1] = b; p[3 * i + 2] = c; }
}

// Camera gradients (CAM = true): the 27 entries of viewmatrix / projmatrix / campos the forward reads, per row
//   [3c + r]       viewmatrix (r, c), r = 0..2, c = 0..3   (storage 4c + r)
//   [12 + 3c + k]  projmatrix (r, c), r = 0, 1, 3 for k = 0, 1, 2
//   [24 + k]       campos k
// Each CTA assigns its sums to a column-major [CAM_TERMS][gridDim.x] scratch, which camera_grad_reduce_kernel reduces.
// Shared memory allows 5 CTAs per SM; left alone, ptxas gives CAM = true 122 registers (4 CTAs), so it is held to 5
// (96 registers, 100 bytes of spill stores).  CAM = false keeps no minimum (0): its code is the same as without CAM.
constexpr int CAM_TERMS = 27;

template <bool CAM>
__global__ void __launch_bounds__(PRE_THREADS, CAM ? 5 : 0) preprocess_backward_kernel(
	int P, int D, int M, const float* __restrict__ means3D, const int32_t* __restrict__ radii,
	const float* __restrict__ shs, const uint8_t* __restrict__ clamped, const float* __restrict__ scales,
	const float* __restrict__ rotations, float scale_modifier, const float* __restrict__ cov3D_precomp,
	const float* __restrict__ feat_precomp, const float* __restrict__ shs_language, const float* __restrict__ confidence,
	const float* __restrict__ viewmatrix, const float* __restrict__ projmatrix, const float* __restrict__ campos,
	float focal_x, float focal_y, float tan_fovx, float tan_fovy, int extended,
	float4* grec, int rezero_grec,
	float* __restrict__ dL_dmeans3D, float* __restrict__ dL_dmeans2D, float* __restrict__ dL_dshs,
	float* __restrict__ dL_dcolors, float* __restrict__ dL_dopac, float* __restrict__ dL_dscales,
	float* __restrict__ dL_drots, float* __restrict__ dL_dcov3D, float* __restrict__ dL_dfeat,
	float* __restrict__ dL_dshs_lang, int tma_ok, void* const* __restrict__ scatter_bases, long long scatter_Ps, int scatter_rank,
	int accumulate, int scatter_tma, float* __restrict__ cam_part)
{
	// inputs staged as in the forward; the same buffers are reused for the outgoing gradients (a thread only ever
	// touches its own row), which leave as contiguous bulk stores instead of 12/24/192-byte strided scalar stores
	__shared__ __align__(128) float s_sh[PRE_THREADS * 48];     // SH in -> dL/dSH out
	__shared__ __align__(128) float4 s_grec[PRE_THREADS * 4];   // (read straight from global it cost +35 % at 6 M Gaussians: 16-byte loads of 64-byte rows)
	__shared__ __align__(16) float s_means[PRE_THREADS * 3];    // means in -> dL/dmeans3D out
	__shared__ __align__(16) float s_geo[PRE_THREADS * 7];      // scales+rotations / cov3D in -> dL/dscales / dL/dcov3D out
	__shared__ __align__(16) float s_feat[PRE_THREADS * 3];     // feature / language SH in -> their gradient out
	__shared__ __align__(16) float s_conf[PRE_THREADS];
	__shared__ __align__(16) float s_o2[PRE_THREADS * 3];       // dL/dmeans2D out
	__shared__ __align__(16) float s_oc[PRE_THREADS * 3];       // dL/dcolors out
	__shared__ __align__(8) uint64_t s_bar;
	const int li = threadIdx.x;
	pdl_trigger();
	const size_t base = (size_t)blockIdx.x * PRE_THREADS;
	const int cnt = (int)min((size_t)PRE_THREADS, (size_t)P - base);
	const bool sh_staged = shs != nullptr && M <= 16;
	const bool full = tma_ok && cnt == PRE_THREADS;
	Stage st;
	st.bar = &s_bar; st.tma = full; st.cnt = cnt; st.tid = li;
	if (li == 0 && full) mbar_init(&s_bar, 1);
	pdl_wait();
	__syncthreads();
	if (li == 0 && full) {
		uint32_t tx = PRE_THREADS * 4 * (16 + 3);
		tx += (cov3D_precomp != nullptr) ? PRE_THREADS * 4 * 6 : PRE_THREADS * 4 * 7;
		if (sh_staged) tx += PRE_THREADS * 4 * 3 * M;
		if (confidence != nullptr) tx += PRE_THREADS * 4;
		if (extended && shs_language != nullptr && feat_precomp == nullptr) tx += PRE_THREADS * 4 * 3;
		mbar_arrive_expect_tx(&s_bar, tx);
	}
	st.load(reinterpret_cast<float*>(s_grec), reinterpret_cast<const float*>(grec), 16, base);
	st.load(s_means, means3D, 3, base);
	if (cov3D_precomp != nullptr) st.load(s_geo, cov3D_precomp, 6, base);
	else { st.load(s_geo, scales, 3, base); st.load(s_geo + 3 * PRE_THREADS, rotations, 4, base); }
	if (sh_staged) st.load(s_sh, shs, 3 * M, base);
	if (confidence != nullptr) st.load(s_conf, confidence, 1, base);
	if (extended && shs_language != nullptr && feat_precomp == nullptr) st.load(s_feat, shs_language, 3, base);
	if (full) mbar_wait(&s_bar, 0);
	else __syncthreads();

	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	// per-Gaussian results (zeros for Gaussians that were not rendered: the reference's torch::zeros)
	float o_mean[3] = {0.f, 0.f, 0.f}, o_m2[2] = {0.f, 0.f}, o_col[3] = {0.f, 0.f, 0.f}, o_sc[3] = {0.f, 0.f, 0.f};
	float o_feat[3] = {0.f, 0.f, 0.f}, o_shl[3] = {0.f, 0.f, 0.f}, o_cov[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
	float o_op = 0.f;
	float4 o_rot = make_float4(0.f, 0.f, 0.f, 0.f);
	float shw[16];  // dL/dSH[k][c] = shw[k] * dRGB[c]
#pragma unroll
	for (int k = 0; k < 16; k++) shw[k] = 0.f;
	float dRGB[3] = {0.f, 0.f, 0.f};
	float cg[CAM_TERMS];  // this row's camera terms (zero unless rendered)
	if constexpr (CAM) {
#pragma unroll
		for (int i = 0; i < CAM_TERMS; i++) cg[i] = 0.f;
	}
	if (idx < P && __ldcg(radii + idx) > 0) {
	ViewConsts vc;
	load_view(vc, viewmatrix, projmatrix, campos);
	const float* vm = vc.view;
	const float* proj = vc.proj;

	const float4 g0 = s_grec[4 * li], g1 = s_grec[4 * li + 1], g2 = s_grec[4 * li + 2], g3 = s_grec[4 * li + 3];
	const float dm2x = g0.x, dm2y = g0.y, dca = g0.z, dcb = g0.w, dcc = g1.x;
	float dop = g1.y;
	dRGB[0] = g2.x; dRGB[1] = g2.y; dRGB[2] = g2.z;
	const float dz = g2.w;
	const float df[3] = {g3.x, g3.y, g3.z};

	const float mx = s_means[3 * li], my = s_means[3 * li + 1], mz = s_means[3 * li + 2];

	// cov3D (recomputed; the reference stores it in geomState.cov3D)
	float c3[6];
	float4 q = make_float4(1.f, 0.f, 0.f, 0.f);
	float s3[3] = {0.f, 0.f, 0.f};
	if (cov3D_precomp != nullptr) {
		for (int i = 0; i < 6; i++) c3[i] = s_geo[6 * li + i];
	} else {
		q = reinterpret_cast<const float4*>(s_geo + 3 * PRE_THREADS)[li];
		s3[0] = s_geo[3 * li]; s3[1] = s_geo[3 * li + 1]; s3[2] = s_geo[3 * li + 2];
		cov3d_pinned(s3[0], s3[1], s3[2], scale_modifier, q, c3);
	}

	// ---- computeCov2DCUDA ----
	float tx = vm[0] * mx + vm[4] * my + vm[8] * mz + vm[12];
	float ty = vm[1] * mx + vm[5] * my + vm[9] * mz + vm[13];
	const float tz = vm[2] * mx + vm[6] * my + vm[10] * mz + vm[14];
	const float limx = 1.3f * tan_fovx, limy = 1.3f * tan_fovy;
	const float txtz = tx / tz, tytz = ty / tz;
	tx = fminf(limx, fmaxf(-limx, txtz)) * tz;
	ty = fminf(limy, fmaxf(-limy, tytz)) * tz;
	const float x_grad_mul = (txtz < -limx || txtz > limx) ? 0.f : 1.f;
	const float y_grad_mul = (tytz < -limy || tytz > limy) ? 0.f : 1.f;
	const float itz = 1.f / tz, itz2 = itz * itz, itz3 = itz2 * itz;
	const float J00 = focal_x * itz, J02 = -(focal_x * tx) * itz2, J11 = focal_y * itz, J12 = -(focal_y * ty) * itz2;
	// T = W * J (GLM column-major); Tc[j][i]
	const float T00 = vm[0] * J00 + vm[2] * J02, T01 = vm[4] * J00 + vm[6] * J02, T02 = vm[8] * J00 + vm[10] * J02;
	const float T10 = vm[1] * J11 + vm[2] * J12, T11 = vm[5] * J11 + vm[6] * J12, T12 = vm[9] * J11 + vm[10] * J12;
	// V * T0, V * T1 with V the symmetric cov3D
	const float VT00 = c3[0] * T00 + c3[1] * T01 + c3[2] * T02;
	const float VT01 = c3[1] * T00 + c3[3] * T01 + c3[4] * T02;
	const float VT02 = c3[2] * T00 + c3[4] * T01 + c3[5] * T02;
	const float VT10 = c3[0] * T10 + c3[1] * T11 + c3[2] * T12;
	const float VT11 = c3[1] * T10 + c3[3] * T11 + c3[4] * T12;
	const float VT12 = c3[2] * T10 + c3[4] * T11 + c3[5] * T12;
	const float a = T00 * VT00 + T01 * VT01 + T02 * VT02 + 0.3f;
	const float b = T00 * VT10 + T01 * VT11 + T02 * VT12;
	const float c = T10 * VT10 + T11 * VT11 + T12 * VT12 + 0.3f;
	const float denom = a * c - b * b;
	const float denom2inv = 1.0f / ((denom * denom) + 0.0000001f);
	float dL_da = 0.f, dL_db = 0.f, dL_dc = 0.f;
	float dcov[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
	if (denom2inv != 0.f) {
		dL_da = denom2inv * (-c * c * dca + 2 * b * c * dcb + (denom - a * c) * dcc);
		dL_dc = denom2inv * (-a * a * dcc + 2 * a * b * dcb + (denom - a * c) * dca);
		dL_db = denom2inv * 2 * (b * c * dca - (denom + 2 * b * b) * dcb + a * b * dcc);
		dcov[0] = T00 * T00 * dL_da + T00 * T10 * dL_db + T10 * T10 * dL_dc;
		dcov[3] = T01 * T01 * dL_da + T01 * T11 * dL_db + T11 * T11 * dL_dc;
		dcov[5] = T02 * T02 * dL_da + T02 * T12 * dL_db + T12 * T12 * dL_dc;
		dcov[1] = 2 * T00 * T01 * dL_da + (T00 * T11 + T01 * T10) * dL_db + 2 * T10 * T11 * dL_dc;
		dcov[2] = 2 * T00 * T02 * dL_da + (T00 * T12 + T02 * T10) * dL_db + 2 * T10 * T12 * dL_dc;
		dcov[4] = 2 * T02 * T01 * dL_da + (T01 * T12 + T02 * T11) * dL_db + 2 * T11 * T12 * dL_dc;
	}
	const float dT00 = 2 * VT00 * dL_da + VT10 * dL_db, dT01 = 2 * VT01 * dL_da + VT11 * dL_db, dT02 = 2 * VT02 * dL_da + VT12 * dL_db;
	const float dT10 = 2 * VT10 * dL_dc + VT00 * dL_db, dT11 = 2 * VT11 * dL_dc + VT01 * dL_db, dT12 = 2 * VT12 * dL_dc + VT02 * dL_db;
	const float dJ00 = vm[0] * dT00 + vm[4] * dT01 + vm[8] * dT02;
	const float dJ02 = vm[2] * dT00 + vm[6] * dT01 + vm[10] * dT02;
	const float dJ11 = vm[1] * dT10 + vm[5] * dT11 + vm[9] * dT12;
	const float dJ12 = vm[2] * dT10 + vm[6] * dT11 + vm[10] * dT12;
	const float dtx = x_grad_mul * -focal_x * itz2 * dJ02;
	const float dty = y_grad_mul * -focal_y * itz2 * dJ12;
	const float dtz = -focal_x * itz2 * dJ00 - focal_y * itz2 * dJ11 + (2 * focal_x * tx) * itz3 * dJ02 + (2 * focal_y * ty) * itz3 * dJ12;
	float dmean[3] = {vm[0] * dtx + vm[1] * dty + vm[2] * dtz, vm[4] * dtx + vm[5] * dty + vm[6] * dtz,
	                  vm[8] * dtx + vm[9] * dty + vm[10] * dtz};

	// ---- preprocessCUDA backward: mean2D -> mean3D through the projection ----
	const float hw = proj[3] * mx + proj[7] * my + proj[11] * mz + proj[15];
	const float m_w = 1.0f / (hw + 0.0000001f);
	const float mul1 = (proj[0] * mx + proj[4] * my + proj[8] * mz + proj[12]) * m_w * m_w;
	const float mul2 = (proj[1] * mx + proj[5] * my + proj[9] * mz + proj[13]) * m_w * m_w;
	dmean[0] += (proj[0] * m_w - proj[3] * mul1) * dm2x + (proj[1] * m_w - proj[3] * mul2) * dm2y;
	dmean[1] += (proj[4] * m_w - proj[7] * mul1) * dm2x + (proj[5] * m_w - proj[7] * mul2) * dm2y;
	dmean[2] += (proj[8] * m_w - proj[11] * mul1) * dm2x + (proj[9] * m_w - proj[11] * mul2) * dm2y;
	if (extended) {  // depth head: z_i = view row 2 . mean  (SURVEY.md Appendix D)
		dmean[0] += vm[2] * dz; dmean[1] += vm[6] * dz; dmean[2] += vm[10] * dz;
	}

	// ---- feature head ----
	if (extended) {
		if (feat_precomp != nullptr) {
			o_feat[0] = df[0]; o_feat[1] = df[1]; o_feat[2] = df[2];
		} else if (shs_language != nullptr) {
			const float v0 = kSH_C0 * s_feat[3 * li], v1 = kSH_C0 * s_feat[3 * li + 1], v2 = kSH_C0 * s_feat[3 * li + 2];
			const float n = sqrtf(v0 * v0 + v1 * v1 + v2 * v2), ne = n + 1e-9f;
			const float vd = v0 * df[0] + v1 * df[1] + v2 * df[2];
			const float k = (n > 0.f) ? vd / (n * ne * ne) : 0.f;
			o_shl[0] = kSH_C0 * (df[0] / ne - v0 * k); o_shl[1] = kSH_C0 * (df[1] / ne - v1 * k); o_shl[2] = kSH_C0 * (df[2] / ne - v2 * k);
		} else {  // feature channels alias the colours
			dRGB[0] += df[0]; dRGB[1] += df[1]; dRGB[2] += df[2];
		}
	}

	// ---- colours: either straight out, or SH backward ----
	if (shs == nullptr) {
		o_col[0] = dRGB[0]; o_col[1] = dRGB[1]; o_col[2] = dRGB[2];
	} else {
		const unsigned cl = __ldcg(clamped + idx);
		dRGB[0] *= (cl & 1u) ? 0.f : 1.f; dRGB[1] *= (cl & 2u) ? 0.f : 1.f; dRGB[2] *= (cl & 4u) ? 0.f : 1.f;
		const float dox = mx - vc.campos[0], doy = my - vc.campos[1], doz = mz - vc.campos[2];
		// The squares below have several uses; the default build rounds each once and fuses none of them into an add.  The
		// CAM build would fuse some (its extra code changes the compiler's choices), so there they are pinned to that
		// rounding: the parameter gradients of both builds stay bit-identical.
		auto sq = [](float a) { if constexpr (CAM) return __fmul_rn(a, a); else return a * a; };
		auto add = [](float a, float b) { if constexpr (CAM) return __fadd_rn(a, b); else return a + b; };
		const float ilen = 1.0f / sqrtf(add(add(sq(dox), sq(doy)), sq(doz)));
		const float x = dox * ilen, y = doy * ilen, z = doz * ilen;
		const float* sh = sh_staged ? s_sh + li * M * 3 : shs + (size_t)idx * M * 3;
		float ddir[3] = {0.f, 0.f, 0.f};  // dL/ddir
		auto wr = [&](int k, float w) { shw[k] = w; };  // the row is written after every read of `sh` (same buffer)
		float sd[16];  // sd[k] = sh[k] . dRGB
		if (sh_staged && M == 16) {
			const float4* row = reinterpret_cast<const float4*>(s_sh + li * 48);
#pragma unroll
			for (int j = 0; j < 4; j++) {  // 4 coefficients = 12 floats = 3 x LDS.128 per step
				const float4 a4 = row[3 * j], b4 = row[3 * j + 1], c4 = row[3 * j + 2];
				sd[4 * j] = a4.x * dRGB[0] + a4.y * dRGB[1] + a4.z * dRGB[2];
				sd[4 * j + 1] = a4.w * dRGB[0] + b4.x * dRGB[1] + b4.y * dRGB[2];
				sd[4 * j + 2] = b4.z * dRGB[0] + b4.w * dRGB[1] + c4.x * dRGB[2];
				sd[4 * j + 3] = c4.y * dRGB[0] + c4.z * dRGB[1] + c4.w * dRGB[2];
			}
		} else {
#pragma unroll
			for (int k = 0; k < 16; k++) sd[k] = (k < (D + 1) * (D + 1)) ? sh[3 * k] * dRGB[0] + sh[3 * k + 1] * dRGB[1] + sh[3 * k + 2] * dRGB[2] : 0.f;
		}
		auto shdot = [&](int k) { return sd[k]; };
		wr(0, kSH_C0);
		int written = 1;
		if (D > 0) {
			wr(1, -kSH_C1 * y); wr(2, kSH_C1 * z); wr(3, -kSH_C1 * x);
			written = 4;
			const float s1 = shdot(1), s2 = shdot(2), s3d = shdot(3);
			ddir[0] = -kSH_C1 * s3d; ddir[1] = -kSH_C1 * s1; ddir[2] = kSH_C1 * s2;
			if (D > 1) {
				const float xx = sq(x), yy = sq(y), zz = sq(z), xy = x * y, yz = y * z, xz = x * z;
				wr(4, kSH_C2[0] * xy); wr(5, kSH_C2[1] * yz); wr(6, kSH_C2[2] * (2.f * zz - xx - yy));
				wr(7, kSH_C2[3] * xz); wr(8, kSH_C2[4] * (xx - yy));
				written = 9;
				const float s4 = shdot(4), s5 = shdot(5), s6 = shdot(6), s7 = shdot(7), s8 = shdot(8);
				ddir[0] += kSH_C2[0] * y * s4 + kSH_C2[2] * 2.f * -x * s6 + kSH_C2[3] * z * s7 + kSH_C2[4] * 2.f * x * s8;
				ddir[1] += kSH_C2[0] * x * s4 + kSH_C2[1] * z * s5 + kSH_C2[2] * 2.f * -y * s6 + kSH_C2[4] * 2.f * -y * s8;
				ddir[2] += kSH_C2[1] * y * s5 + kSH_C2[2] * 2.f * 2.f * z * s6 + kSH_C2[3] * x * s7;
				if (D > 2) {
					wr(9, kSH_C3[0] * y * (3.f * xx - yy)); wr(10, kSH_C3[1] * xy * z);
					wr(11, kSH_C3[2] * y * (4.f * zz - xx - yy)); wr(12, kSH_C3[3] * z * (2.f * zz - 3.f * xx - 3.f * yy));
					wr(13, kSH_C3[4] * x * (4.f * zz - xx - yy)); wr(14, kSH_C3[5] * z * (xx - yy));
					wr(15, kSH_C3[6] * x * (xx - 3.f * yy));
					written = 16;
					const float s9 = shdot(9), s10 = shdot(10), s11 = shdot(11), s12 = shdot(12), s13 = shdot(13),
					            s14 = shdot(14), s15 = shdot(15);
					ddir[0] += kSH_C3[0] * s9 * 3.f * 2.f * xy + kSH_C3[1] * s10 * yz + kSH_C3[2] * s11 * -2.f * xy +
					           kSH_C3[3] * s12 * -3.f * 2.f * xz + kSH_C3[4] * s13 * (-3.f * xx + 4.f * zz - yy) +
					           kSH_C3[5] * s14 * 2.f * xz + kSH_C3[6] * s15 * 3.f * (xx - yy);
					ddir[1] += kSH_C3[0] * s9 * 3.f * (xx - yy) + kSH_C3[1] * s10 * xz + kSH_C3[2] * s11 * (-3.f * yy + 4.f * zz - xx) +
					           kSH_C3[3] * s12 * -3.f * 2.f * yz + kSH_C3[4] * s13 * -2.f * xy + kSH_C3[5] * s14 * -2.f * yz +
					           kSH_C3[6] * s15 * -3.f * 2.f * xy;
					ddir[2] += kSH_C3[1] * s10 * xy + kSH_C3[2] * s11 * 4.f * 2.f * yz + kSH_C3[3] * s12 * 3.f * (2.f * zz - xx - yy) +
					           kSH_C3[4] * s13 * 4.f * 2.f * xz + kSH_C3[5] * s14 * (xx - yy);
				}
			}
		}
		(void)written;
		// dnormvdv (auxiliary.h:107-117)
		const float sum2 = add(add(sq(dox), sq(doy)), sq(doz));
		const float invsum32 = 1.0f / sqrtf(sum2 * sum2 * sum2);
		const float nx = (+sum2 - sq(dox)) * ddir[0] - doy * dox * ddir[1] - doz * dox * ddir[2];
		const float ny = -dox * doy * ddir[0] + (sum2 - sq(doy)) * ddir[1] - doz * doy * ddir[2];
		const float nz = -dox * doz * ddir[0] - doy * doz * ddir[1] + (sum2 - sq(doz)) * ddir[2];
		if constexpr (CAM) {
			// dir = mean - campos.  Here the product n * invsum32 has a second use, so the compiler would round it before
			// the add; the FMA it contracts to in the default build is pinned, keeping dL/dmean bit-identical to it
			dmean[0] = __fmaf_rn(nx, invsum32, dmean[0]); dmean[1] = __fmaf_rn(ny, invsum32, dmean[1]);
			dmean[2] = __fmaf_rn(nz, invsum32, dmean[2]);
			cg[24] = -(nx * invsum32); cg[25] = -(ny * invsum32); cg[26] = -(nz * invsum32);
		} else {
			dmean[0] += nx * invsum32; dmean[1] += ny * invsum32; dmean[2] += nz * invsum32;
		}
	}

	o_mean[0] = dmean[0]; o_mean[1] = dmean[1]; o_mean[2] = dmean[2];
	o_m2[0] = dm2x; o_m2[1] = dm2y;
	if (confidence != nullptr) dop *= s_conf[li];
	o_op = dop;

	// ---- cov3D -> scale / rotation (computeCov3D backward) ----
	if (cov3D_precomp != nullptr) {
#pragma unroll
		for (int i = 0; i < 6; i++) o_cov[i] = dcov[i];
	} else {
		const float r = q.x, x = q.y, y = q.z, z = q.w;
		// GLM column-major R[col][row]
		const float R[3][3] = {{1.f - 2.f * (y * y + z * z), 2.f * (x * y - r * z), 2.f * (x * z + r * y)},
		                       {2.f * (x * y + r * z), 1.f - 2.f * (x * x + z * z), 2.f * (y * z - r * x)},
		                       {2.f * (x * z - r * y), 2.f * (y * z + r * x), 1.f - 2.f * (x * x + y * y)}};
		const float s[3] = {scale_modifier * s3[0], scale_modifier * s3[1], scale_modifier * s3[2]};
		const float dS[3][3] = {{dcov[0], 0.5f * dcov[1], 0.5f * dcov[2]}, {0.5f * dcov[1], dcov[3], 0.5f * dcov[4]},
		                        {0.5f * dcov[2], 0.5f * dcov[4], dcov[5]}};
		float dMt[3][3];  // dMt[k][i] = dM[i][k],  dM[j][i] = sum_m 2*M[m][i]*dS[j][m],  M[m][i] = s_i R[m][i]
#pragma unroll
		for (int k = 0; k < 3; k++)
#pragma unroll
			for (int i = 0; i < 3; i++)
				dMt[k][i] = 2.0f * s[k] * (R[0][k] * dS[i][0] + R[1][k] * dS[i][1] + R[2][k] * dS[i][2]);
		float dsc[3];
#pragma unroll
		for (int k = 0; k < 3; k++) dsc[k] = R[0][k] * dMt[k][0] + R[1][k] * dMt[k][1] + R[2][k] * dMt[k][2];
		o_sc[0] = dsc[0]; o_sc[1] = dsc[1]; o_sc[2] = dsc[2];
#pragma unroll
		for (int k = 0; k < 3; k++)
#pragma unroll
			for (int i = 0; i < 3; i++) dMt[k][i] *= s[k];
		float4 dq;
		dq.x = 2 * z * (dMt[0][1] - dMt[1][0]) + 2 * y * (dMt[2][0] - dMt[0][2]) + 2 * x * (dMt[1][2] - dMt[2][1]);
		dq.y = 2 * y * (dMt[1][0] + dMt[0][1]) + 2 * z * (dMt[2][0] + dMt[0][2]) + 2 * r * (dMt[1][2] - dMt[2][1]) - 4 * x * (dMt[2][2] + dMt[1][1]);
		dq.z = 2 * x * (dMt[1][0] + dMt[0][1]) + 2 * r * (dMt[2][0] - dMt[0][2]) + 2 * z * (dMt[1][2] + dMt[2][1]) - 4 * y * (dMt[2][2] + dMt[0][0]);
		dq.w = 2 * r * (dMt[0][1] - dMt[1][0]) + 2 * x * (dMt[2][0] + dMt[0][2]) + 2 * y * (dMt[1][2] + dMt[2][1]) - 4 * z * (dMt[1][1] + dMt[0][0]);
		o_rot = dq;
	}
	if constexpr (CAM) {
		// t = A mh (mh = (mean, 1)): dA(r, c) += dt_r mh_c, the depth head's cotangent joining dt_z
		const float mh[4] = {mx, my, mz, 1.f};
		const float dt[3] = {dtx, dty, extended ? dtz + dz : dtz};
		// h = Pm mh, projected as h_r / (h_3 + 1e-7): dPm(r, c) += dh_r mh_c for r = 0, 1, 3
		const float dh[3] = {dm2x * m_w, dm2y * m_w, -(dm2x * mul1 + dm2y * mul2)};
#pragma unroll
		for (int c = 0; c < 4; c++)
#pragma unroll
			for (int r = 0; r < 3; r++) { cg[3 * c + r] = dt[r] * mh[c]; cg[12 + 3 * c + r] = dh[r] * mh[c]; }
		// T = J W with W = A[0:3, 0:3]: T0j = J00 W0j + J02 W2j, T1j = J11 W1j + J12 W2j
		const float dT0[3] = {dT00, dT01, dT02}, dT1[3] = {dT10, dT11, dT12};
#pragma unroll
		for (int j = 0; j < 3; j++) {
			cg[3 * j] += dT0[j] * J00;
			cg[3 * j + 1] += dT1[j] * J11;
			cg[3 * j + 2] += dT0[j] * J02 + dT1[j] * J12;
		}
	}
	}  // rendered Gaussian

	// ---- write out: rows into the staging buffers, then one bulk store per array (or coalesced copies) ----
	const bool valid = idx < P;
	__syncwarp();
	s_means[3 * li] = o_mean[0]; s_means[3 * li + 1] = o_mean[1]; s_means[3 * li + 2] = o_mean[2];
	s_o2[3 * li] = o_m2[0]; s_o2[3 * li + 1] = o_m2[1]; s_o2[3 * li + 2] = 0.f;
	s_oc[3 * li] = o_col[0]; s_oc[3 * li + 1] = o_col[1]; s_oc[3 * li + 2] = o_col[2];
	const bool feat_out = dL_dfeat != nullptr;  // at most one of dL_dfeat / dL_dshs_lang is requested per call
	s_feat[3 * li] = feat_out ? o_feat[0] : o_shl[0]; s_feat[3 * li + 1] = feat_out ? o_feat[1] : o_shl[1];
	s_feat[3 * li + 2] = feat_out ? o_feat[2] : o_shl[2];
	__syncthreads();  // all reads of s_geo (quaternions live past the scales) are done before it is overwritten
	if (cov3D_precomp != nullptr) {
#pragma unroll
		for (int i = 0; i < 6; i++) s_geo[6 * li + i] = o_cov[i];
	} else {
		s_geo[3 * li] = o_sc[0]; s_geo[3 * li + 1] = o_sc[1]; s_geo[3 * li + 2] = o_sc[2];
	}
	if (dL_dshs != nullptr) {
		if (sh_staged) {
			if (M == 16) {
				float4* row = reinterpret_cast<float4*>(s_sh + li * 48);
#pragma unroll
				for (int j = 0; j < 4; j++) {
					const float w0 = shw[4 * j], w1 = shw[4 * j + 1], w2 = shw[4 * j + 2], w3 = shw[4 * j + 3];
					row[3 * j] = make_float4(w0 * dRGB[0], w0 * dRGB[1], w0 * dRGB[2], w1 * dRGB[0]);
					row[3 * j + 1] = make_float4(w1 * dRGB[1], w1 * dRGB[2], w2 * dRGB[0], w2 * dRGB[1]);
					row[3 * j + 2] = make_float4(w2 * dRGB[2], w3 * dRGB[0], w3 * dRGB[1], w3 * dRGB[2]);
				}
			} else {
				float* row = s_sh + li * M * 3;
#pragma unroll
				for (int k = 0; k < 16; k++) {
					if (k < M) { row[3 * k] = shw[k] * dRGB[0]; row[3 * k + 1] = shw[k] * dRGB[1]; row[3 * k + 2] = shw[k] * dRGB[2]; }
				}
			}
		} else if (valid) {  // unstaged rows are written in place; with accumulate, coefficients 16.. (no gradient) keep their sums
			float* row = dL_dshs + (size_t)idx * M * 3;
#pragma unroll
			for (int k = 0; k < 16; k++) {
				if (k < M) {
					const float g0 = shw[k] * dRGB[0], g1 = shw[k] * dRGB[1], g2 = shw[k] * dRGB[2];
					row[3 * k] = accumulate ? __fadd_rn(row[3 * k], g0) : g0;  // fl(previous + this view), as add_local
					row[3 * k + 1] = accumulate ? __fadd_rn(row[3 * k + 1], g1) : g1;
					row[3 * k + 2] = accumulate ? __fadd_rn(row[3 * k + 2], g2) : g2;
				}
			}
			if (!accumulate)
				for (int i = 48; i < 3 * M; i++) row[i] = 0.f;
		}
	}
	// Image-parallel training: the parameter gradients of this 128-Gaussian tile go straight into the staging buffer of
	// the rank that owns the tile (plain 16-byte stores over NVLink; layout in include/b200gs_collective.h), so the
	// reduce-scatter half of the gradient exchange costs no kernel of its own.
	float* fb = nullptr;    // owner's staging block for this source rank
	size_t li0 = 0;         // first row of the tile inside the owner's shard
	if (scatter_bases != nullptr) {
		const size_t Ps = (size_t)scatter_Ps;
		const size_t o = base / Ps;
		li0 = base - o * Ps;
		fb = reinterpret_cast<float*>(scatter_bases[o]) + (size_t)scatter_rank * Ps * 64;
	}
	// the caller's rotation-gradient array need not be 16-byte aligned (a float4 access there faults): scalar accesses then
	const bool rots16 = (reinterpret_cast<uintptr_t>(dL_drots) & 15u) == 0;
	if (valid && accumulate) {  // several views per optimizer step: add what the earlier views left in the local arrays
		if (dL_dopac) o_op += dL_dopac[idx];
		if (dL_drots) {
			const float4 t = rots16 ? reinterpret_cast<const float4*>(dL_drots)[idx]
			                        : make_float4(dL_drots[4 * idx], dL_drots[4 * idx + 1], dL_drots[4 * idx + 2], dL_drots[4 * idx + 3]);
			o_rot.x += t.x; o_rot.y += t.y; o_rot.z += t.z; o_rot.w += t.w;
		}
	}
	if (valid) {
		if (fb) {
			fb[51 * (size_t)scatter_Ps + li0 + li] = o_op;
			reinterpret_cast<float4*>(fb + 55 * (size_t)scatter_Ps)[li0 + li] = o_rot;
		} else {
			if (dL_dopac) dL_dopac[idx] = o_op;
			if (dL_drots && rots16) reinterpret_cast<float4*>(dL_drots)[idx] = o_rot;
			else if (dL_drots) { float* r = dL_drots + 4 * (size_t)idx; r[0] = o_rot.x; r[1] = o_rot.y; r[2] = o_rot.z; r[3] = o_rot.w; }
		}
	}
	if constexpr (CAM) {
		float* s_cam = reinterpret_cast<float*>(s_grec);  // [warp][32] warp sums (every row of s_grec was read before the last barrier)
		// transposing butterfly: at each step a lane keeps half of its values and adds its partner's copy of that half,
		// so 32 values (27 terms, zero-padded) need 16 + 8 + 4 + 2 + 1 shuffles and lane l ends with the warp's sum of value l
		float v[32];
#pragma unroll
		for (int i = 0; i < 32; i++) v[i] = i < CAM_TERMS ? cg[i] : 0.f;
#pragma unroll
		for (int s = 16; s >= 1; s >>= 1) {
			const bool hi = (li & s) != 0;
#pragma unroll
			for (int i = 0; i < s; i++) {
				const float send = hi ? v[i] : v[i + s], keep = hi ? v[i + s] : v[i];
				v[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, s);
			}
		}
		s_cam[li] = v[0];
	}
	tma_store_fence();
	__syncthreads();
	if constexpr (CAM) {  // the CTA's sums, warps added in a fixed order: assigned, so the scratch needs no zeroing
		const float* s_cam = reinterpret_cast<const float*>(s_grec);
		if (li < CAM_TERMS)
			cam_part[(size_t)li * gridDim.x + blockIdx.x] = (s_cam[li] + s_cam[32 + li]) + (s_cam[64 + li] + s_cam[96 + li]);
	}
	auto put = [&](float* dst, const float* src, int floats_per_item) {
		if (dst == nullptr) return;
		float* g = dst + base * floats_per_item;
		if (full) {
			if (li == 0) tma_store_1d(g, src, (uint32_t)(PRE_THREADS * floats_per_item * 4));
		} else {
			for (int i = li; i < cnt * floats_per_item; i += PRE_THREADS) g[i] = src[i];
		}
	};
	auto push = [&](int seg, const float* src, int floats_per_item) {  // rows li0.. of segment `seg` in the owner's staging block
		float* g = fb + (size_t)seg * (size_t)scatter_Ps + li0 * floats_per_item;  // 16-byte aligned: Ps and li0 are multiples of 128
		if (full && scatter_tma) {  // one bulk copy per array through the TMA engine instead of 16-byte LSU stores
			if (li == 0) tma_store_1d(g, src, (uint32_t)(PRE_THREADS * floats_per_item * 4));
			return;
		}
		const int n = cnt * floats_per_item;
		for (int i = li; i < n / 4; i += PRE_THREADS) reinterpret_cast<float4*>(g)[i] = reinterpret_cast<const float4*>(src)[i];
		for (int i = (n & ~3) + li; i < n; i += PRE_THREADS) g[i] = src[i];
	};
	if (rezero_grec && valid) {  // persistent workspaces: the scratch rows this thread consumed are zero again for the next backward
		const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
		float4* row = grec + 4 * (size_t)idx;
		row[0] = z; row[1] = z; row[2] = z; row[3] = z;
	}
	if (accumulate) {
		auto add_local = [&](const float* local, float* stage, int floats_per_item) {
			if (local == nullptr) return;
			const float* g = local + base * floats_per_item;
			for (int i = li; i < cnt * floats_per_item; i += PRE_THREADS) stage[i] += g[i];
		};
		add_local(dL_dmeans3D, s_means, 3);
		add_local(dL_dfeat, s_feat, 3);
		add_local(dL_dshs_lang, s_feat, 3);
		if (cov3D_precomp == nullptr) add_local(dL_dscales, s_geo, 3);
		if (sh_staged) add_local(dL_dshs, s_sh, 3 * M);
		tma_store_fence();
		__syncthreads();
	}
	put(dL_dmeans2D, s_o2, 3);
	put(dL_dcolors, s_oc, 3);
	if (cov3D_precomp != nullptr) put(dL_dcov3D, s_geo, 6);
	if (fb) {
		push(0, s_means, 3);
		if (sh_staged && M == 16) push(3, s_sh, 48);
		if (cov3D_precomp == nullptr) push(52, s_geo, 3);
		if (dL_dfeat != nullptr || dL_dshs_lang != nullptr) push(59, s_feat, 3);
	} else {
		put(dL_dmeans3D, s_means, 3);
		put(dL_dfeat, s_feat, 3);
		put(dL_dshs_lang, s_feat, 3);
		if (cov3D_precomp == nullptr) put(dL_dscales, s_geo, 3);
		if (sh_staged) put(dL_dshs, s_sh, 3 * M);
	}
	if (full && li == 0) { tma_store_commit(); tma_store_wait_read(); }
}

// One CTA per output float of b200gs_camera_grads_t (16 viewmatrix, 16 projmatrix, 3 campos, in storage order): the CTA
// partials of its term summed in float64 in a fixed order; entries the forward never reads are written as zeros.  Each
// thread keeps CAM_REDUCE_UNROLL loads in flight (46 875 partials per term at 6 M Gaussians: one dependent load per step
// would make this latency-bound kernel cost more than the per-row arithmetic).
constexpr int CAM_REDUCE_THREADS = 1024, CAM_REDUCE_UNROLL = 8;
__global__ void __launch_bounds__(CAM_REDUCE_THREADS) camera_grad_reduce_kernel(
	const float* cam_part, int nblk, float* __restrict__ dL_dview, float* __restrict__ dL_dproj, float* __restrict__ dL_dcampos)
{
	__shared__ double s_sum[CAM_REDUCE_THREADS];
	pdl_trigger();
	const int e = blockIdx.x, tid = threadIdx.x;
	int term = -1;
	if (e < 16) {
		const int r = e & 3, c = e >> 2;
		if (r != 3) term = 3 * c + r;
	} else if (e < 32) {
		const int r = (e - 16) & 3, c = (e - 16) >> 2;
		if (r != 2) term = 12 + 3 * c + (r == 3 ? 2 : r);
	} else {
		term = 24 + (e - 32);
	}
	pdl_wait();  // the partials are written by the preprocess backward just before
	double acc = 0.0;
	if (term >= 0) {
		const float* p = cam_part + (size_t)term * nblk;
		for (int i0 = tid; i0 < nblk; i0 += CAM_REDUCE_THREADS * CAM_REDUCE_UNROLL) {
			float x[CAM_REDUCE_UNROLL];
#pragma unroll
			for (int u = 0; u < CAM_REDUCE_UNROLL; u++) {
				const int i = i0 + u * CAM_REDUCE_THREADS;
				x[u] = i < nblk ? __ldcg(p + i) : 0.f;
			}
#pragma unroll
			for (int u = 0; u < CAM_REDUCE_UNROLL; u++) acc += (double)x[u];
		}
	}
	s_sum[tid] = acc;
	__syncthreads();
#pragma unroll
	for (int w = CAM_REDUCE_THREADS / 2; w > 0; w >>= 1) {
		if (tid < w) s_sum[tid] += s_sum[tid + w];
		__syncthreads();
	}
	if (tid == 0) {
		float* out = e < 16 ? dL_dview + e : e < 32 ? dL_dproj + (e - 16) : dL_dcampos + (e - 32);
		*out = (float)s_sum[0];
	}
}

}  // namespace

size_t camera_scratch_bytes(int P) {
	const size_t nblk = P > 0 ? ((size_t)P + PRE_THREADS - 1) / PRE_THREADS : 1;
	return nblk * CAM_TERMS * sizeof(float);
}

void launch_preprocess_forward(const RasterPlan& pl, const b200gs_gaussians_t& g, int32_t* radii, cudaStream_t stream) {
	const b200gs_view_t& v = *pl.v;
	const GeomState& gs = pl.gs;
	const int P = g.P;
	const float focal_y = v.height / (2.0f * v.tan_fovy);  // rasterizer_impl.cu:222-223
	const float focal_x = v.width / (2.0f * v.tan_fovx);
	const auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
	const int tma_ok = al16(g.means3D) && al16(g.scales) && al16(g.rotations) && al16(g.opacities) && al16(g.shs) &&
	                   al16(g.cov3D_precomp) && al16(g.colors_precomp) && al16(g.language_feature_precomp) &&
	                   al16(g.shs_language) && al16(g.confidence);
	launch(0u, preprocess_forward_kernel, dim3((P + PRE_THREADS - 1) / PRE_THREADS), dim3(PRE_THREADS), 0, stream,
		P, v.sh_degree, v.sh_coeffs, g.means3D, g.scales, v.scale_modifier, g.rotations, g.opacities, g.shs,
		g.cov3D_precomp, g.colors_precomp, g.language_feature_precomp, g.shs_language, g.confidence,
		v.viewmatrix, v.projmatrix, v.campos, v.width, v.height, v.tan_fovx, v.tan_fovy, focal_x, focal_y,
		v.extended, v.prefiltered, radii, gs.depths, gs.rect, gs.rec, gs.clamped, gs.key_a, gs.order, gs.hist, pl.is.ranges, pl.is.tile_count,
		COUNT_STRIDE, (int)pl.grid.tiles, gs.hdr, tma_ok, g.live_count);
}

void launch_preprocess_backward(const RasterPlan& pl, const b200gs_gaussians_t& g, const int32_t* radii, float* grec,
                                const b200gs_grads_t& gr, const b200gs_camera_grads_t* cam, cudaStream_t stream) {
	const b200gs_view_t& v = *pl.v;
	const int P = g.P;
	const unsigned nblk = (P + PRE_THREADS - 1) / PRE_THREADS;
	const float focal_y = v.height / (2.0f * v.tan_fovy);
	const float focal_x = v.width / (2.0f * v.tan_fovx);
	const auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
	const int tma_ok = al16(g.means3D) && al16(g.scales) && al16(g.rotations) && al16(g.shs) && al16(g.cov3D_precomp) &&
	                   al16(g.shs_language) && al16(g.confidence) && al16(grec) && al16(gr.dL_dmeans3D) && al16(gr.dL_dmeans2D) &&
	                   al16(gr.dL_dshs) && al16(gr.dL_dcolors) && al16(gr.dL_dscales) && al16(gr.dL_dcov3D) && al16(gr.dL_dfeatures) &&
	                   al16(gr.dL_dshs_language);
	const int scatter_tma = knob_int(KNOB_SCATTER_TMA, 1);  // 0: plain stores to the peer staging blocks (A/B)
	float* cam_part = cam ? reinterpret_cast<float*>(cam->scratch) : nullptr;
	launch(PDL_PRE_BWD, cam ? preprocess_backward_kernel<true> : preprocess_backward_kernel<false>, dim3(nblk), dim3(PRE_THREADS), 0, stream,
		P, v.sh_degree, v.sh_coeffs, g.means3D, radii, g.shs, pl.gs.clamped, g.scales, g.rotations, v.scale_modifier,
		g.cov3D_precomp, g.language_feature_precomp, g.shs_language, g.confidence, v.viewmatrix, v.projmatrix,
		v.campos, focal_x, focal_y, v.tan_fovx, v.tan_fovy, v.extended, reinterpret_cast<float4*>(grec), pl.persistent ? 1 : 0,
		gr.dL_dmeans3D, gr.dL_dmeans2D, gr.dL_dshs, gr.dL_dcolors, gr.dL_dopacities, gr.dL_dscales,
		gr.dL_drotations, gr.dL_dcov3D, gr.dL_dfeatures, gr.dL_dshs_language, tma_ok, gr.scatter_bases,
		(long long)gr.scatter_shard_rows, (int)gr.scatter_rank, (int)gr.accumulate, scatter_tma, cam_part);
	if (cam)
		launch(PDL_PRE_BWD, camera_grad_reduce_kernel, dim3(35), dim3(CAM_REDUCE_THREADS), 0, stream, (const float*)cam_part, (int)nblk,
		       cam->dL_dviewmatrix, cam->dL_dprojmatrix, cam->dL_dcampos);
}

void launch_mark_visible(int P, const float* means3D, const float* viewmatrix, uint8_t* present, cudaStream_t stream) {
	launch(0u, mark_visible_kernel, dim3((P + 255) / 256), dim3(256), 0, stream, P, means3D, viewmatrix, present);
}
