// Direct checks of the blend kernels' device helpers (sdp-gs_b200/csrc/blend_common.cuh), built by
// tests/test_blend_edges_gpu.py with the library's own flags (no fast-math) and called through ctypes.
//
//   check_cull:   cull_block is sound -- a block it culls has no pixel centre at which the forward keeps the pair;
//   check_expf2:  expf2 is bit-identical to expf, per half, over every float with the sign bit set (and +0);
//   check_packed: add2 / mul2 / fma2 / pair_power2 are bit-identical to their scalar forms, per half.
//
// Every launcher takes device pointers to unsigned long long counters (zeroed by the caller), synchronises and returns
// the CUDA error code.  Inputs are generated on the device from a counter-based hash, so a run is reproducible.
#include <cstdint>
#include <cuda_runtime.h>
#include "../../sdp-gs_b200/csrc/blend_common.cuh"

namespace {

__device__ __forceinline__ uint64_t mix64(uint64_t z) {  // splitmix64 finaliser
	z += 0x9E3779B97F4A7C15ull;
	z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
	z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
	return z ^ (z >> 31);
}
struct Rng {
	uint64_t s;
	__device__ uint64_t next() { s = mix64(s); return s; }
	__device__ double uni() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }  // [0, 1)
	__device__ uint32_t u32() { return (uint32_t)(next() >> 32); }
};

// The forward's decision for one (pair, pixel): blend.cu computes dx = mx + (-px), power = pair_power, alpha =
// min(0.99, o * expf(power)) and skips the pair when power > 0 or alpha < 1/255.
__device__ __forceinline__ bool forward_keeps(float mx, float my, float ca, float cb, float cc, float o, float px, float py) {
	const float dx = __fadd_rn(mx, -px), dy = __fadd_rn(my, -py);
	const float power = pair_power(dx, dy, ca, cb, cc);
	const float alpha = fminf(0.99f, __fmul_rn(o, expf(power)));
	return !(power > 0.0f || alpha < 1.0f / 255.0f);
}

// counters: [0] cases, [1] culled, [2] unsound culls (culled although a pixel keeps the pair), [3] kept although no pixel
// keeps it (not tight), [4] degenerate conics (non-PD, zero, inf, NaN) [5] degenerate conics culled (must be 0)
__global__ void cull_kernel(uint64_t n, uint64_t seed, unsigned long long* cnt) {
	unsigned long long culled = 0, unsound = 0, loose = 0, degen = 0, degen_culled = 0, cases = 0;
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
		Rng r{mix64(seed ^ (i * 0xD1B54A32D192ED03ull))};
		// the block: an 8x4 pixel block of a 16x16 tile somewhere in a large image
		const float bx = (float)(16 * (r.u32() % 256) + 8 * (r.u32() & 1)), by = (float)(16 * (r.u32() % 256) + 4 * (r.u32() & 3));
		PixelBlock pb;
		pb.X0 = bx; pb.X1 = bx + 7.f; pb.Y0 = by; pb.Y1 = by + 3.f;
		// opacity in [1/255 (1 + 1e-6), 1], log-uniform; the record as preprocess.cu builds it
		const double omin = (1.0 / 255.0) * (1.0 + 1e-6);
		float o = (float)(omin * exp(r.uni() * log(1.0 / omin)));
		if (o < (float)omin) o = nextafterf((float)omin, 1.f);
		// conic: eigenvalues 1/sigma^2 with sigma in [0.25, 3e3] px and condition number 1 .. 1e8, any rotation
		const double emax = exp(log(16.0) - r.uni() * log(16.0 * 9e6 / 1.0));
		const double kappa = exp(r.uni() * log(1e8));
		const double emin = emax / kappa;
		const double th = r.uni() * 6.283185307179586;
		const double cs = cos(th), sn = sin(th);
		double A = emax * cs * cs + emin * sn * sn, B = (emax - emin) * cs * sn, Cc = emax * sn * sn + emin * cs * cs;
		float ca = (float)A, cb = (float)B, cc = (float)Cc;
		const uint32_t kind = r.u32() % 64;
		bool degenerate = false;
		if (kind == 0) { cb = sqrtf(ca * cc) * (1.0f + 0.5f * (float)r.uni()) + 1e-30f; degenerate = true; }  // not PD
		else if (kind == 1) { ca = cb = cc = 0.f; degenerate = true; }
		else if (kind == 2) { const float v = __int_as_float(0x7F800000); if (r.u32() & 1) ca = v; else cc = v; degenerate = true; }
		else if (kind == 3) { const float v = __int_as_float(0x7FC00000); const uint32_t w = r.u32() % 3; if (w == 0) ca = v; else if (w == 1) cb = v; else cc = v; degenerate = true; }
		else if (kind == 4) { ca = -ca; degenerate = true; }
		const float thr = 2.0f * logf(255.0f * o);
		const float nbc = -cb / cc;
		// the mean: the exact (float64) q = thr contour passes within +-[1e-4, 1] px of a pixel centre, an edge point or a corner
		// of the block (most cases), or the mean lies inside the block, or far away
		double mx, my;
		const uint32_t where = r.u32() % 16;
		if (where == 0) {
			mx = bx - 0.5 + 8.0 * r.uni(); my = by - 0.5 + 4.0 * r.uni();
		} else if (where == 1) {
			const double a = r.uni() * 6.283185307179586, d = exp(log(10.0) + r.uni() * log(1e3));
			mx = bx + 3.5 + d * cos(a); my = by + 1.5 + d * sin(a);
		} else {
			double tx, ty;
			const uint32_t w = where % 3;
			if (w == 0) { tx = bx + (double)(r.u32() & 7); ty = by + (double)(r.u32() & 3); }          // pixel centre
			else if (w == 1) {                                                                        // edge point
				const double t = r.uni();
				switch (r.u32() & 3) { case 0: tx = bx + 7 * t; ty = by; break; case 1: tx = bx + 7 * t; ty = by + 3; break;
				                       case 2: tx = bx; ty = by + 3 * t; break; default: tx = bx + 7; ty = by + 3 * t; }
			} else { tx = bx + 7.0 * (r.u32() & 1); ty = by + 3.0 * (r.u32() & 1); }                 // corner
			// contour point in direction phi from the mean: d = u * sqrt(thr / (u^T Q u)) (Q from the rounded conic)
			const double phi = r.uni() * 6.283185307179586, ux = cos(phi), uy = sin(phi);
			const double quu = (double)ca * ux * ux + 2.0 * (double)cb * ux * uy + (double)cc * uy * uy;
			const double s = (quu > 0.0 && thr > 0.f) ? sqrt((double)thr / quu) : 0.0;
			const double delta = ((r.u32() & 1) ? 1.0 : -1.0) * exp(log(1e-4) + r.uni() * log(1e4));
			const double psi = r.uni() * 6.283185307179586;
			mx = tx - ux * s + delta * cos(psi);
			my = ty - uy * s + delta * sin(psi);
		}
		const float4 g0 = make_float4((float)mx, (float)my, ca, cb), g1 = make_float4(cc, o, thr, nbc);
		const bool cull = cull_block(g0, g1, pb);
		bool any = false;
		for (int p = 0; p < 32; p++)
			any |= forward_keeps(g0.x, g0.y, ca, cb, cc, o, bx + (float)(p & 7), by + (float)(p >> 3));
		cases++;
		culled += cull;
		unsound += (cull && any);
		loose += (!cull && !any);
		degen += degenerate;
		degen_culled += (degenerate && cull);
	}
	atomicAdd(cnt + 0, cases); atomicAdd(cnt + 1, culled); atomicAdd(cnt + 2, unsound); atomicAdd(cnt + 3, loose);
	atomicAdd(cnt + 4, degen); atomicAdd(cnt + 5, degen_culled);
}

__device__ __forceinline__ bool same(float a, float b) {
	return (__float_as_uint(a) == __float_as_uint(b)) || (a != a && b != b);  // bits, NaN matches any NaN
}

// counters: [0] inputs checked, [1] mismatches.  Inputs: 0x80000000 | i for i < 2^31 (every float with the sign bit set:
// -0, negative denormals, normals, -inf and NaNs), plus +0 on thread 0.  Each half gets a different input.
__global__ void expf2_kernel(unsigned long long* cnt, unsigned int* first_bad) {
	unsigned long long checked = 0, bad = 0;
	const uint32_t half = 1u << 30;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < half; i += gridDim.x * blockDim.x) {
		const float x = __uint_as_float(0x80000000u | i), y = __uint_as_float(0x80000000u | (i + half));
		const float2 e = expf2(make_float2(x, y));
		const bool bx = !same(e.x, expf(x)), by = !same(e.y, expf(y));
		if (bx) atomicCAS(first_bad, 0u, __float_as_uint(x));
		if (by) atomicCAS(first_bad, 0u, __float_as_uint(y));
		checked += 2;
		bad += bx + by;
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) {
		const float2 e = expf2(make_float2(0.f, 0.f));
		checked += 1;
		bad += !same(e.x, expf(0.f)) || !same(e.y, expf(0.f));
	}
	atomicAdd(cnt + 0, checked); atomicAdd(cnt + 1, bad);
}

// random float bit patterns with the special values mixed in
__device__ __forceinline__ float rand_float(Rng& r) {
	const uint32_t k = r.u32();
	const uint32_t sign = (k & 1u) << 31;
	switch ((k >> 1) % 16) {
	case 0: return __uint_as_float(sign);                                  // signed zero
	case 1: return __uint_as_float(sign | 0x7F800000u);                    // infinity
	case 2: return __uint_as_float(sign | (r.u32() & 0x007FFFFFu));        // denormal
	case 3: return __uint_as_float(sign | 0x7F800000u | (r.u32() | 1u));   // NaN
	case 4: case 5: case 6: {                                              // moderate magnitudes: finite sums, products and fmas
		const uint32_t e = 100u + r.u32() % 56u;
		return __uint_as_float(sign | (e << 23) | (r.u32() & 0x007FFFFFu));
	}
	default: return __uint_as_float(r.u32());                              // any bit pattern
	}
}

// counters: [0] add2, [1] mul2, [2] fma2, [3] pair_power2 mismatches, [4] cases per operation
__global__ void packed_kernel(uint64_t n, uint64_t seed, unsigned long long* cnt) {
	unsigned long long bad[4] = {0, 0, 0, 0}, cases = 0;
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
		Rng r{mix64(seed ^ (i * 0xA0761D6478BD642Full))};
		float v[10];
		for (int k = 0; k < 10; k++) v[k] = rand_float(r);
		const float2 a = make_float2(v[0], v[1]), b = make_float2(v[2], v[3]), c = make_float2(v[4], v[5]);
		const float2 s = add2(a, b), m = mul2(a, b), f = fma2(a, b, c);
		bad[0] += !same(s.x, __fadd_rn(a.x, b.x)) || !same(s.y, __fadd_rn(a.y, b.y));
		bad[1] += !same(m.x, __fmul_rn(a.x, b.x)) || !same(m.y, __fmul_rn(a.y, b.y));
		bad[2] += !same(f.x, __fmaf_rn(a.x, b.x, c.x)) || !same(f.y, __fmaf_rn(a.y, b.y, c.y));
		const float2 d = make_float2(v[6], v[7]), e = make_float2(v[8], v[9]);
		const float2 p = pair_power2(a, b, c, d, e);
		bad[3] += !same(p.x, pair_power(a.x, b.x, c.x, d.x, e.x)) || !same(p.y, pair_power(a.y, b.y, c.y, d.y, e.y));
		cases++;
	}
	for (int k = 0; k < 4; k++) atomicAdd(cnt + k, bad[k]);
	atomicAdd(cnt + 4, cases);
}

}  // namespace

extern "C" int check_cull(unsigned long long n, unsigned long long seed, unsigned long long* cnt) {
	cull_kernel<<<148 * 8, 256>>>(n, seed, cnt);
	return (int)cudaDeviceSynchronize();
}
extern "C" int check_expf2(unsigned long long* cnt, unsigned int* first_bad) {
	expf2_kernel<<<148 * 16, 256>>>(cnt, first_bad);
	return (int)cudaDeviceSynchronize();
}
extern "C" int check_packed(unsigned long long n, unsigned long long seed, unsigned long long* cnt) {
	packed_kernel<<<148 * 8, 256>>>(n, seed, cnt);
	return (int)cudaDeviceSynchronize();
}
