// b200gs -- the kernels of one training iteration that sit around the rasterizer (include/b200gs_train.h;
// SURVEY.md section 8(f) rows 1 and 3): fused photometric loss (L1 + SSIM, value and gradient), Pearson depth
// loss (value and gradient), and the fused parameter step (activation backward + Adam + re-activation +
// densification statistics).  All of it is streaming / stencil work bounded by HBM bandwidth.
#include <cmath>
#include <cstdio>
#include "common.cuh"
#include "../../include/b200gs_train.h"

int train_fail(int code, const char* msg);  // api.cu

namespace {

// ------------------------------------------------------------------------------------------------------------
// Photometric loss.  ssim() of utils/loss_utils.py:129-163: depthwise 11x11 Gaussian window (sigma 1.5), zero
// padding 5, mean over C*H*W.  Forward kernel: per 16x16 pixel tile and channel, separable convolution of
// (x, y, x^2, y^2, xy) in shared memory -> SSIM value + the three derivative maps the backward needs.
// With f = a1*a2 / (b1*b2), a1 = 2 mu1 mu2 + C1, a2 = 2 s12 + C2, b1 = mu1^2 + mu2^2 + C1, b2 = s1 + s2 + C2:
//   mA = df/dmu1 - 2 mu1 df/ds1 - mu2 df/ds12,  mB = df/ds1,  mC = df/ds12
//   dSSIM_sum/dx_q = (W*mA)_q + 2 x_q (W*mB)_q + y_q (W*mC)_q          (W symmetric; maps are 0 outside the image)
// Backward kernel: the same separable convolution over the three maps, plus the L1 term.
constexpr int LT = 16;        // tile edge
constexpr int HALO = 5;
constexpr int LW = LT + 2 * HALO;  // 26
constexpr int ACC_SLOTS = 64;      // partial sums are spread over this many L2 lines: same-address f64 atomics from
                                   // thousands of blocks serialise in L2 (ncu: 24 us for a 504x378 image before the spread)

struct Window { float w[11]; };

__global__ void __launch_bounds__(LT * LT) ssim_l1_forward_kernel(
	const float* __restrict__ img, const float* __restrict__ gt, int W, int H, Window win,
	float* __restrict__ mapA, float* __restrict__ mapB, float* __restrict__ mapC,
	double* __restrict__ accum /*[ACC_SLOTS][2] = {sum|x-y|, sum ssim}, then the block counter*/, const b200gs_hparams_t* __restrict__ hp,
	double* __restrict__ loss_out)
{
	__shared__ float sx[LW][LW + 1], sy[LW][LW + 1];
	__shared__ float hsum[5][LW][LT + 1];
	__shared__ double red[2][LT * LT / 32];
	const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * LT + tx;
	const int ch = blockIdx.z;
	const int x0 = blockIdx.x * LT, y0 = blockIdx.y * LT;
	const size_t plane = (size_t)ch * W * H;
	for (int i = tid; i < LW * LW; i += LT * LT) {
		const int ly = i / LW, lx = i % LW;
		const int gx = x0 + lx - HALO, gy = y0 + ly - HALO;
		const bool in = gx >= 0 && gx < W && gy >= 0 && gy < H;
		sx[ly][lx] = in ? img[plane + (size_t)gy * W + gx] : 0.f;
		sy[ly][lx] = in ? gt[plane + (size_t)gy * W + gx] : 0.f;
	}
	__syncthreads();
	for (int i = tid; i < LW * LT; i += LT * LT) {  // horizontal pass: 26 rows x 16 columns
		const int ly = i / LT, lx = i % LT;
		float a = 0.f, b = 0.f, aa = 0.f, bb = 0.f, ab = 0.f;
#pragma unroll
		for (int k = 0; k < 11; k++) {
			const float xv = sx[ly][lx + k], yv = sy[ly][lx + k], wk = win.w[k];
			a = fmaf(wk, xv, a); b = fmaf(wk, yv, b);
			aa = fmaf(wk, xv * xv, aa); bb = fmaf(wk, yv * yv, bb); ab = fmaf(wk, xv * yv, ab);
		}
		hsum[0][ly][lx] = a; hsum[1][ly][lx] = b; hsum[2][ly][lx] = aa; hsum[3][ly][lx] = bb; hsum[4][ly][lx] = ab;
	}
	__syncthreads();
	float mu1 = 0.f, mu2 = 0.f, e11 = 0.f, e22 = 0.f, e12 = 0.f;
#pragma unroll
	for (int k = 0; k < 11; k++) {
		const float wk = win.w[k];
		mu1 = fmaf(wk, hsum[0][ty + k][tx], mu1); mu2 = fmaf(wk, hsum[1][ty + k][tx], mu2);
		e11 = fmaf(wk, hsum[2][ty + k][tx], e11); e22 = fmaf(wk, hsum[3][ty + k][tx], e22);
		e12 = fmaf(wk, hsum[4][ty + k][tx], e12);
	}
	const int gx = x0 + tx, gy = y0 + ty;
	const bool in = gx < W && gy < H;
	double l1 = 0.0, ss = 0.0;
	if (in) {
		const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
		const float s1 = e11 - mu1 * mu1, s2 = e22 - mu2 * mu2, s12 = e12 - mu1 * mu2;
		const float a1 = 2.f * mu1 * mu2 + C1, a2 = 2.f * s12 + C2;
		const float b1 = mu1 * mu1 + mu2 * mu2 + C1, b2 = s1 + s2 + C2;
		const float inv = 1.f / (b1 * b2);
		const float f = a1 * a2 * inv;
		const float df_dmu1 = 2.f * mu2 * a2 * inv - f * 2.f * mu1 / b1;
		const float df_ds1 = -f / b2;
		const float df_ds12 = 2.f * a1 * inv;
		const size_t o = plane + (size_t)gy * W + gx;
		mapA[o] = df_dmu1 - 2.f * mu1 * df_ds1 - mu2 * df_ds12;
		mapB[o] = df_ds1;
		mapC[o] = df_ds12;
		ss = (double)f;
		l1 = (double)fabsf(sx[ty + HALO][tx + HALO] - sy[ty + HALO][tx + HALO]);
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) { l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, o); ss += __shfl_xor_sync(0xFFFFFFFFu, ss, o); }
	if ((tid & 31) == 0) { red[0][tid >> 5] = l1; red[1][tid >> 5] = ss; }
	__syncthreads();
	__shared__ bool s_last;
	if (tid == 0) {
		double a = 0.0, b = 0.0;
		for (int i = 0; i < LT * LT / 32; i++) { a += red[0][i]; b += red[1][i]; }
		const unsigned lin = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
		double* slot = accum + 16 * (lin % ACC_SLOTS);  // one 128-byte line per slot
		atomicAdd(slot, a);
		atomicAdd(slot + 1, b);
		__threadfence();
		unsigned long long* counter = reinterpret_cast<unsigned long long*>(accum + 16 * ACC_SLOTS);
		const unsigned long long total = (unsigned long long)gridDim.x * gridDim.y * gridDim.z;
		s_last = atomicAdd(counter, 1ull) == total - 1;
	}
	__syncthreads();
	if (!s_last) return;
	// last block: the 64 slots are gathered by 64 threads (one L2 round trip, not 64), the accumulators are left zero
	__threadfence();
	double sa = 0.0, sb = 0.0;
	if (tid < ACC_SLOTS) {
		sa = __ldcg(accum + 16 * tid); sb = __ldcg(accum + 16 * tid + 1);
		accum[16 * tid] = 0.0; accum[16 * tid + 1] = 0.0;
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) { sa += __shfl_xor_sync(0xFFFFFFFFu, sa, o); sb += __shfl_xor_sync(0xFFFFFFFFu, sb, o); }
	if ((tid & 31) == 0) { red[0][tid >> 5] = sa; red[1][tid >> 5] = sb; }
	__syncthreads();
	if (tid == 0) {
		sa = red[0][0] + red[0][1]; sb = red[1][0] + red[1][1];  // ACC_SLOTS = 64 = two warps
		const double n = 3.0 * (double)W * (double)H;
		const double L1 = sa / n, S = sb / n;
		const double lam = (double)hp->lambda_dssim;
		loss_out[0] = (1.0 - lam) * L1 + lam * (1.0 - S);
		loss_out[1] = L1;
		loss_out[2] = S;
		*reinterpret_cast<unsigned long long*>(accum + 16 * ACC_SLOTS) = 0ull;
	}
}

__global__ void __launch_bounds__(LT * LT) ssim_l1_backward_kernel(
	const float* __restrict__ img, const float* __restrict__ gt, int W, int H, Window win,
	const float* mapA, const float* mapB, const float* mapC, const b200gs_hparams_t* __restrict__ hp,
	float* __restrict__ dL_dimg)
{
	__shared__ float sm[3][LW][LW + 1];
	__shared__ float hsum[3][LW][LT + 1];
	pdl_trigger();
	const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * LT + tx;
	const int ch = blockIdx.z;
	const int x0 = blockIdx.x * LT, y0 = blockIdx.y * LT;
	const size_t plane = (size_t)ch * W * H;
	pdl_wait();
	for (int i = tid; i < LW * LW; i += LT * LT) {
		const int ly = i / LW, lx = i % LW;
		const int gx = x0 + lx - HALO, gy = y0 + ly - HALO;
		const bool in = gx >= 0 && gx < W && gy >= 0 && gy < H;
		const size_t o = plane + (size_t)gy * W + gx;
		sm[0][ly][lx] = in ? __ldcg(mapA + o) : 0.f;  // produced by the kernel just before this one: never through the .nc path
		sm[1][ly][lx] = in ? __ldcg(mapB + o) : 0.f;
		sm[2][ly][lx] = in ? __ldcg(mapC + o) : 0.f;
	}
	__syncthreads();
	for (int i = tid; i < LW * LT; i += LT * LT) {
		const int ly = i / LT, lx = i % LT;
		float a = 0.f, b = 0.f, c = 0.f;
#pragma unroll
		for (int k = 0; k < 11; k++) {
			const float wk = win.w[k];
			a = fmaf(wk, sm[0][ly][lx + k], a); b = fmaf(wk, sm[1][ly][lx + k], b); c = fmaf(wk, sm[2][ly][lx + k], c);
		}
		hsum[0][ly][lx] = a; hsum[1][ly][lx] = b; hsum[2][ly][lx] = c;
	}
	__syncthreads();
	float cA = 0.f, cB = 0.f, cC = 0.f;
#pragma unroll
	for (int k = 0; k < 11; k++) {
		const float wk = win.w[k];
		cA = fmaf(wk, hsum[0][ty + k][tx], cA); cB = fmaf(wk, hsum[1][ty + k][tx], cB); cC = fmaf(wk, hsum[2][ty + k][tx], cC);
	}
	const int gx = x0 + tx, gy = y0 + ty;
	if (gx < W && gy < H) {
		const size_t o = plane + (size_t)gy * W + gx;
		const float x = img[o], y = gt[o];
		const float n = 3.f * (float)W * (float)H;
		const float lam = hp->lambda_dssim;
		const float d = x - y;
		const float sgn = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
		dL_dimg[o] = (-lam / n) * (cA + 2.f * x * cB + y * cC) + ((1.f - lam) / n) * sgn;
	}
}

// ------------------------------------------------------------------------------------------------------------
// Pearson depth loss (train.py:115-131).  x1 = depth_mono, x2 = 1 / (200 - depth_mono), y = rendered depth.
// r = Sxy / sqrt(Sxx Syy) over centred sums; loss = w * min(1 - r1, 1 - r2);
// dL/dy_i = w * ( -(x_i - mx) / sqrt(Sxx Syy) + r (y_i - my) / Syy ) for the selected branch = A x_i + B y_i + C0.
__global__ void __launch_bounds__(256) pearson_reduce_kernel(
	const float* __restrict__ depth, const float* __restrict__ mono, int n,
	double* __restrict__ accum /*[ACC_SLOTS][16] partial sums (8 used), then counter, then 4 coefficients*/,
	const b200gs_hparams_t* __restrict__ hp, double* __restrict__ loss_out, const float* __restrict__ weight_override, int single_branch)
{
	__shared__ double red[8][8];
	pdl_trigger();
	pdl_wait();
	double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // y, yy, x1, x1x1, x1y, x2, x2x2, x2y
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const float yf = __ldcg(depth + i), x1f = mono[i];
		const float x2f = 1.0f / (-x1f + 200.0f);
		const double y = yf, x1 = x1f, x2 = x2f;
		s[0] += y; s[1] += y * y; s[2] += x1; s[3] += x1 * x1; s[4] += x1 * y; s[5] += x2; s[6] += x2 * x2; s[7] += x2 * y;
	}
#pragma unroll
	for (int k = 0; k < 8; k++) {
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xFFFFFFFFu, s[k], o);
	}
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	if (lane == 0) {
#pragma unroll
		for (int k = 0; k < 8; k++) red[k][warp] = s[k];
	}
	__syncthreads();
	if (threadIdx.x < 8) {
		double t = 0.0;
		for (int w = 0; w < 8; w++) t += red[threadIdx.x][w];
		atomicAdd(accum + 16 * (blockIdx.x % ACC_SLOTS) + threadIdx.x, t);
	}
	__syncthreads();
	__shared__ bool s_last;
	if (threadIdx.x == 0) {
		__threadfence();
		unsigned long long* counter = reinterpret_cast<unsigned long long*>(accum + 16 * ACC_SLOTS);
		s_last = atomicAdd(counter, 1ull) == (unsigned long long)gridDim.x - 1;
	}
	__syncthreads();
	if (!s_last) return;
	__threadfence();
	{   // last block: thread (slot, k) gathers one partial sum; 8 x 64 values reduced over the slots through shared memory
		__shared__ double part[ACC_SLOTS][8];
		for (int i = threadIdx.x; i < ACC_SLOTS * 8; i += blockDim.x) {
			const int sl = i >> 3, k = i & 7;
			part[sl][k] = __ldcg(accum + 16 * sl + k);
			accum[16 * sl + k] = 0.0;
		}
		__syncthreads();
		if (threadIdx.x < 8) {
			double t = 0.0;
			for (int sl = 0; sl < ACC_SLOTS; sl++) t += part[sl][threadIdx.x];
			red[threadIdx.x][0] = t;
		}
		__syncthreads();
	}
	if (threadIdx.x == 0) {
		{
			double t[8];
			for (int k = 0; k < 8; k++) t[k] = red[k][0];
			*reinterpret_cast<unsigned long long*>(accum + 16 * ACC_SLOTS) = 0ull;
			const double N = (double)n;
			const double my = t[0] / N, Syy = t[1] - t[0] * t[0] / N;
			const double m1 = t[2] / N, S11 = t[3] - t[2] * t[2] / N, S1y = t[4] - t[2] * t[0] / N;
			const double m2 = t[5] / N, S22 = t[6] - t[5] * t[5] / N, S2y = t[7] - t[5] * t[0] / N;
			const double D1 = sqrt(S11 * Syy), D2 = sqrt(S22 * Syy);
			double r1 = S1y / D1, r2 = S2y / D2;
			r1 = fmin(1.0, fmax(-1.0, r1)); r2 = fmin(1.0, fmax(-1.0, r2));
			// pseudo views (train.py:143-153): weight = loss_scale * depth_pseudo_weight from its own device word, and the single
			// correlation 1 - pearson(depth, -midas) instead of the min over the two forms
			const double w = weight_override ? (double)__ldcg(weight_override) : (double)hp->depth_weight;
			const bool first = single_branch || (1.0 - r1) <= (1.0 - r2);  // python min(a, b) returns a on ties
			const double r = first ? r1 : r2, D = first ? D1 : D2, mx = first ? m1 : m2;
			double* coef = accum + 16 * ACC_SLOTS + 2;
			coef[0] = -w / D;                               // A
			coef[1] = w * r / Syy;                          // B
			coef[2] = w * (mx / D - r * my / Syy);          // C0
			coef[3] = first ? 0.0 : 1.0;                    // which x
			const double dl = w * (1.0 - r);
			loss_out[3] = dl;
			loss_out[0] += dl;
		}
	}
}

__global__ void __launch_bounds__(256) pearson_grad_kernel(const float* __restrict__ depth, const float* __restrict__ mono, int n,
                                                           const double* coef, float* __restrict__ dL_ddepth)
{
	pdl_trigger();
	pdl_wait();
	const double A = __ldcg(coef), B = __ldcg(coef + 1), C0 = __ldcg(coef + 2);
	const bool second = __ldcg(coef + 3) != 0.0;
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const float x1 = mono[i];
		const float x = second ? 1.0f / (-x1 + 200.0f) : x1;
		dL_ddepth[i] = (float)(A * (double)x + B * (double)__ldcg(depth + i) + C0);
	}
}

// ------------------------------------------------------------------------------------------------------------
// Parameter step.  One launch walks the six groups with 128-bit accesses.  For every element:
//   g_raw = g_act * d act / d raw     (identity | sigmoid: o(1-o) | exp: s | normalize: (g - q^ (q^.g)) / |q|)
//   m = b1 m + (1-b1) g_raw;  v = b2 v + (1-b2) g_raw^2
//   p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)           (torch.optim.Adam, no amsgrad / weight decay)
// then the activated copy is rewritten from the new raw value.
struct AdamC { float b1, b2, eps, step_scale /* 1/(1-b1^t) */, inv_sqrt_bc2; };

__device__ __forceinline__ float adam1(float& p, float& m, float& v, float g, float lr, const AdamC& c) {
	m = fmaf(c.b1, m, (1.f - c.b1) * g);
	v = fmaf(c.b2, v, (1.f - c.b2) * g * g);
	const float denom = sqrtf(v) * c.inv_sqrt_bc2 + c.eps;
	p -= (lr * c.step_scale) * (m / denom);
	return p;
}

__global__ void __launch_bounds__(256) param_step_kernel(b200gs_param_state_t s, const b200gs_hparams_t* __restrict__ hp, int mode)
{
	const bool update = mode == 1;   // Adam update + statistics; mode 2: statistics only (the reference's densify iterations, where the
	                                 // freshly re-created parameters have no gradient and optimizer.step() changes nothing)

	pdl_trigger();
	pdl_wait();
	const b200gs_hparams_t h = *hp;
	AdamC c;
	c.b1 = h.beta1; c.b2 = h.beta2; c.eps = h.eps;
	c.step_scale = (float)(1.0 / (1.0 - pow((double)h.beta1, (double)h.step)));   // torch evaluates the bias corrections in double
	c.inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow((double)h.beta2, (double)h.step)));
	const size_t P = (size_t)s.P;
	const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;

	auto flat4 = [&](float* p, float* m, float* v, const float* g, size_t count, auto lr_of) {  // identity activation, count % 4 == 0 handled below
		const size_t n4 = count / 4;
		for (size_t i = tid; i < n4; i += nth) {
			float4 pp = reinterpret_cast<float4*>(p)[i], mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
			const float4 gg = __ldcg(reinterpret_cast<const float4*>(g) + i);
			const uint32_t e = (uint32_t)(4 * i);  // < 2^32 elements per group
			adam1(pp.x, mm.x, vv.x, gg.x, lr_of(e), c); adam1(pp.y, mm.y, vv.y, gg.y, lr_of(e + 1), c);
			adam1(pp.z, mm.z, vv.z, gg.z, lr_of(e + 2), c); adam1(pp.w, mm.w, vv.w, gg.w, lr_of(e + 3), c);
			reinterpret_cast<float4*>(p)[i] = pp; reinterpret_cast<float4*>(m)[i] = mm; reinterpret_cast<float4*>(v)[i] = vv;
		}
		for (size_t i = n4 * 4 + tid; i < count; i += nth) adam1(p[i], m[i], v[i], __ldcg(g + i), lr_of((uint32_t)i), c);
	};
	if (update) {
		flat4(s.xyz, s.m_xyz, s.v_xyz, s.g_xyz, 3 * P, [&](uint32_t) { return h.lr_xyz; });
		flat4(s.shs, s.m_shs, s.v_shs, s.g_shs, 48 * P, [&](uint32_t i) { return (i % 48u) < 3u ? h.lr_f_dc : h.lr_f_rest; });
		if (s.feature) flat4(s.feature, s.m_feature, s.v_feature, s.g_feature, 3 * P, [&](uint32_t) { return h.lr_feature; });
	}
	// opacity: sigmoid
	for (size_t i = tid; i < P; i += nth) {
		float raw = s.opacity[i];
		if (update) {
			const float o = 1.f / (1.f + expf(-raw));
			const float g = __ldcg(s.g_opacity + i) * o * (1.f - o);
			adam1(raw, s.m_opacity[i], s.v_opacity[i], g, h.lr_opacity, c);
			s.opacity[i] = raw;
		}
		s.opacity_act[i] = 1.f / (1.f + expf(-raw));
	}
	// scaling: exp
	for (size_t i = tid; i < 3 * P; i += nth) {
		float raw = s.scaling[i];
		if (update) {
			const float g = __ldcg(s.g_scaling + i) * expf(raw);
			adam1(raw, s.m_scaling[i], s.v_scaling[i], g, h.lr_scaling, c);
			s.scaling[i] = raw;
		}
		s.scaling_act[i] = expf(raw);
	}
	// rotation: normalize (torch.nn.functional.normalize, eps 1e-12)
	for (size_t i = tid; i < P; i += nth) {
		float4 q = reinterpret_cast<float4*>(s.rotation)[i];
		if (update) {
			const float nrm = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
			const float inv = 1.f / nrm;
			const float4 u = make_float4(q.x * inv, q.y * inv, q.z * inv, q.w * inv);
			const float4 ga = __ldcg(reinterpret_cast<const float4*>(s.g_rotation) + i);
			const float d = u.x * ga.x + u.y * ga.y + u.z * ga.z + u.w * ga.w;
			const float4 g = make_float4((ga.x - u.x * d) * inv, (ga.y - u.y * d) * inv, (ga.z - u.z * d) * inv, (ga.w - u.w * d) * inv);
			float4 mm = reinterpret_cast<float4*>(s.m_rotation)[i], vv = reinterpret_cast<float4*>(s.v_rotation)[i];
			adam1(q.x, mm.x, vv.x, g.x, h.lr_rotation, c); adam1(q.y, mm.y, vv.y, g.y, h.lr_rotation, c);
			adam1(q.z, mm.z, vv.z, g.z, h.lr_rotation, c); adam1(q.w, mm.w, vv.w, g.w, h.lr_rotation, c);
			reinterpret_cast<float4*>(s.rotation)[i] = q;
			reinterpret_cast<float4*>(s.m_rotation)[i] = mm; reinterpret_cast<float4*>(s.v_rotation)[i] = vv;
		}
		const float inv2 = 1.f / fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
		reinterpret_cast<float4*>(s.rotation_act)[i] = make_float4(q.x * inv2, q.y * inv2, q.z * inv2, q.w * inv2);
	}
	// densification statistics of this step's view (train.py:218-221, scene/gaussian_model.py:610-612)
	if (mode != 0 && s.xyz_gradient_accum) {
		for (size_t i = tid; i < P; i += nth) {
			const int r = __ldcg(s.radii + i);
			if (r > 0) {
				const float gx = __ldcg(s.g_means2D + 3 * i), gy = __ldcg(s.g_means2D + 3 * i + 1);
				s.xyz_gradient_accum[i] += sqrtf(gx * gx + gy * gy);
				s.denom[i] += 1.f;
				s.max_radii2D[i] = max(s.max_radii2D[i], r);
			}
		}
	}
}

__global__ void hparams_advance_kernel(b200gs_hparams_t* hp, float lr_init, float lr_final, float delay_mult, float max_steps) {
	pdl_trigger();
	pdl_wait();
	if (threadIdx.x != 0 || blockIdx.x != 0) return;
	// The reference calls update_learning_rate(iteration) AFTER optimizer.step() (train.py:230-233): Adam step t runs with
	// the learning rate of iteration t-1 (position_lr_init for the first one).  The block is advanced after step `done`,
	// so the rate it leaves for step done+1 is expon_lr(done).
	const float done = hp->step;
	hp->step = done + 1.f;
	if (lr_init == 0.f && lr_final == 0.f) { hp->lr_xyz = 0.f; return; }
	// lr_delay_steps == 0 in scene/gaussian_model.py:268-271, so delay_rate == 1 (delay_mult only matters with delay steps)
	(void)delay_mult;
	const double t = fmin(fmax((double)done / (double)max_steps, 0.0), 1.0);
	hp->lr_xyz = (float)exp(log((double)lr_init) * (1.0 - t) + log((double)lr_final) * t);
}

// Exact 3-NN, brute force over shared-memory tiles of candidates (b200gs_knn3).
constexpr int KNN_THREADS = 256;
constexpr int KNN_TILE = 2048;
__global__ void __launch_bounds__(KNN_THREADS) knn3_kernel(int P, const float* __restrict__ xyz, float* __restrict__ mean_d2, int32_t* __restrict__ idx3) {
	__shared__ float s_x[KNN_TILE], s_y[KNN_TILE], s_z[KNN_TILE];
	const int i = blockIdx.x * KNN_THREADS + threadIdx.x;
	const bool live = i < P;
	const float qx = live ? xyz[3 * (size_t)i] : 0.f, qy = live ? xyz[3 * (size_t)i + 1] : 0.f, qz = live ? xyz[3 * (size_t)i + 2] : 0.f;
	float d0 = 3.0e38f, d1 = 3.0e38f, d2 = 3.0e38f;
	int i0 = -1, i1 = -1, i2 = -1;
	for (int base = 0; base < P; base += KNN_TILE) {
		const int cnt = min(KNN_TILE, P - base);
		__syncthreads();
		for (int j = threadIdx.x; j < cnt; j += KNN_THREADS) {
			s_x[j] = xyz[3 * (size_t)(base + j)]; s_y[j] = xyz[3 * (size_t)(base + j) + 1]; s_z[j] = xyz[3 * (size_t)(base + j) + 2];
		}
		__syncthreads();
		if (!live) continue;
#pragma unroll 4
		for (int j = 0; j < cnt; j++) {
			const float dx = s_x[j] - qx, dy = s_y[j] - qy, dz = s_z[j] - qz;
			const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));  // simple_knn: d.x*d.x + d.y*d.y + d.z*d.z, left to right
			if (d < d2 && base + j != i) {  // candidates arrive in index order and ties do not displace: lower index first
				if (d < d1) {
					d2 = d1; i2 = i1;
					if (d < d0) { d1 = d0; i1 = i0; d0 = d; i0 = base + j; }
					else { d1 = d; i1 = base + j; }
				} else { d2 = d; i2 = base + j; }
			}
		}
	}
	if (live) {
		mean_d2[i] = (d0 + d1 + d2) / 3.0f;
		idx3[3 * (size_t)i] = i0; idx3[3 * (size_t)i + 1] = i1; idx3[3 * (size_t)i + 2] = i2;
	}
}

Window make_window() {
	Window w;
	double g[11], sum = 0.0;
	for (int i = 0; i < 11; i++) { g[i] = exp(-(double)((i - 5) * (i - 5)) / (2.0 * 1.5 * 1.5)); sum += g[i]; }
	for (int i = 0; i < 11; i++) w.w[i] = (float)(g[i] / sum);
	return w;
}

}  // namespace

extern "C" {

size_t b200gs_photometric_scratch_bytes(int32_t width, int32_t height) { return (size_t)9 * width * height * sizeof(float); }
size_t b200gs_loss_accum_doubles(void) { return (size_t)16 * ACC_SLOTS + 8; }

int b200gs_photometric_loss(const float* image, const float* gt, int32_t width, int32_t height,
                            const b200gs_hparams_t* hp, float* scratch, double* accum, double* loss_out,
                            float* dL_dimage, void* stream_) {
	if (!image || !gt || !hp || !scratch || !accum || !loss_out || !dL_dimage || width <= 0 || height <= 0)
		return train_fail(B200GS_E_ARG, "photometric_loss: bad arguments");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	const Window win = make_window();
	const size_t n = (size_t)3 * width * height;
	float *mA = scratch, *mB = scratch + n, *mC = scratch + 2 * n;
	const dim3 grid((width + LT - 1) / LT, (height + LT - 1) / LT, 3), block(LT, LT);
	// its predecessor is the rasterizer's blend kernel (ours, executes pdl_wait), but the forward kernel starts the chain plainly
	launch(0u, ssim_l1_forward_kernel, grid, block, 0, stream, image, gt, (int)width, (int)height, win, mA, mB, mC, accum, hp, loss_out);
	return launch_status(launch(PDL_TRAIN, ssim_l1_backward_kernel, grid, block, 0, stream, image, gt, (int)width, (int)height, win,
	                            (const float*)mA, (const float*)mB, (const float*)mC, hp, dL_dimage));
}

int b200gs_depth_pearson_loss(const float* depth, const float* depth_mono, int32_t n, const b200gs_hparams_t* hp,
                              double* accum, double* loss_out, float* dL_ddepth, void* stream_) {
	return b200gs_depth_pearson_loss_pseudo(depth, depth_mono, n, hp, nullptr, 0, accum, loss_out, dL_ddepth, stream_);
}

int b200gs_depth_pearson_loss_pseudo(const float* depth, const float* depth_ref, int32_t n, const b200gs_hparams_t* hp,
                                     const float* weight_device, int32_t single_branch, double* accum, double* loss_out,
                                     float* dL_ddepth, void* stream_) {
	if (!depth || !depth_ref || !hp || !accum || !loss_out || !dL_ddepth || n <= 0)
		return train_fail(B200GS_E_ARG, "depth_pearson_loss: bad arguments");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	const unsigned grid = (unsigned)min((n + 255) / 256, 148 * 4);
	launch(PDL_TRAIN, pearson_reduce_kernel, dim3(grid), dim3(256), 0, stream, depth, depth_ref, (int)n, accum, hp, loss_out, weight_device,
	       (int)single_branch);
	return launch_status(launch(PDL_TRAIN, pearson_grad_kernel, dim3(grid), dim3(256), 0, stream, depth, depth_ref, (int)n,
	                            (const double*)(accum + 16 * ACC_SLOTS + 2), dL_ddepth));
}

int b200gs_knn3(int32_t P, const float* xyz, float* mean_dist2, int32_t* indices, void* stream_) {
	if (P < 0 || (P > 0 && (!xyz || !mean_dist2 || !indices))) return train_fail(B200GS_E_ARG, "knn3: bad arguments");
	if (P < 4) return train_fail(B200GS_E_ARG, "knn3: at least 4 points are needed for 3 neighbours");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	return launch_status(launch(0u, knn3_kernel, dim3((P + KNN_THREADS - 1) / KNN_THREADS), dim3(KNN_THREADS), 0, stream, P, xyz, mean_dist2, indices));
}

int b200gs_hparams_advance(b200gs_hparams_t* hp, float lr_init, float lr_final, float lr_delay_mult, float max_steps, void* stream_) {
	if (!hp || max_steps <= 0.f) return train_fail(B200GS_E_ARG, "hparams_advance: bad arguments");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	return launch_status(launch(PDL_TRAIN, hparams_advance_kernel, dim3(1), dim3(32), 0, stream, hp, lr_init, lr_final, lr_delay_mult, max_steps));
}

void b200gs_train_abi_sizes(int64_t* out2) { out2[0] = sizeof(b200gs_param_state_t); out2[1] = sizeof(b200gs_hparams_t); }

int b200gs_param_step(const b200gs_param_state_t* s, const b200gs_hparams_t* hp, int32_t update, void* stream_) {
	const bool foreign = (update & B200GS_STEP_AFTER_FOREIGN) != 0;
	update &= 3;
	if (!s || !hp || s->P < 0) return train_fail(B200GS_E_ARG, "param_step: bad arguments");
	if (s->P == 0) return 0;
	if (!s->xyz || !s->shs || !s->opacity || !s->scaling || !s->rotation || !s->opacity_act || !s->scaling_act || !s->rotation_act)
		return train_fail(B200GS_E_ARG, "param_step: parameter pointers are required");
	if (update == 1 && (!s->g_xyz || !s->g_shs || !s->g_opacity || !s->g_scaling || !s->g_rotation || !s->m_xyz || !s->v_xyz ||
	               !s->m_shs || !s->v_shs || !s->m_opacity || !s->v_opacity || !s->m_scaling || !s->v_scaling || !s->m_rotation ||
	               !s->v_rotation || (s->feature && (!s->g_feature || !s->m_feature || !s->v_feature))))
		return train_fail(B200GS_E_ARG, "param_step: gradients and Adam moments are required for an update");
	if (update && s->xyz_gradient_accum && (!s->denom || !s->max_radii2D || !s->g_means2D || !s->radii))
		return train_fail(B200GS_E_ARG, "param_step: densification statistics need denom, max_radii2D, g_means2D and radii");
	cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
	// its predecessor is the preprocess backward or the gather kernel (ours: both execute griddepcontrol.wait) in a training step;
	// launched with full stream ordering when used stand-alone or behind a foreign kernel (B200GS_STEP_AFTER_FOREIGN)
	return launch_status(launch((update && !foreign) ? PDL_TRAIN : 0u, param_step_kernel, dim3(148 * 8), dim3(256), 0, stream, *s, hp, (int)update));
}

}  // extern "C"
