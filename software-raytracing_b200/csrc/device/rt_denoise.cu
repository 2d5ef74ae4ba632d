// rt_denoise.cu -- the denoiser behind RaylibB200_Denoise* and RaylibB200_AccumulatorDenoise (rt_denoise.h, DESIGN.md
// section 14): spatial SVGF (Schied et al. 2017, without the temporal part) on the edge-avoiding a-trous wavelet filter
// (Dammertz et al. 2010).
//
//   k_denoise_prepare  demodulate (irradiance = colour / albedo), classify (surface / miss), decode the normal, estimate
//                      the luminance variance: over the 7 x 7 window (images) or from the accumulator's sums
//   k_denoise_atrous   one a-trous iteration of step 1, 2, 4, 8 or 16 over the {irradiance, variance} records; the last
//                      one remodulates into the output image
//
// The output must equal tests/native/denoise_restatement.cc bit for bit: fixed summation orders, no atomics, IEEE division
// and square root, --fmad=false (Makefile), and the exponential of include/rt_libm.h.  Constants are fixed, not options.
#include "rt_denoise.h"
#include "rt_math.cuh"
#include "rt_libm.h"

#include <cuda_runtime.h>
#include <stdio.h>
#include <string>

static thread_local std::string g_denoiseError;
extern "C" const char* rt_denoise_last_error(void) { return g_denoiseError.c_str(); }

#define RT_DN_CUDA(expr)                                                                   \
	do {                                                                                   \
		cudaError_t _e = (expr);                                                           \
		if (_e != cudaSuccess) {                                                           \
			char _buf[512];                                                                \
			snprintf(_buf, sizeof(_buf), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
			g_denoiseError = _buf;                                                         \
			cudaGetLastError();                                                            \
			return (int)_e;                                                                \
		}                                                                                  \
	} while (0)

#define RT_DN_BX 32
#define RT_DN_BY 8
#define RT_DN_VAR_R 3                                   // the variance window is (2 R + 1)^2 = 7 x 7
#define RT_DN_TILE_W (RT_DN_BX + 2 * RT_DN_VAR_R)
#define RT_DN_TILE_H (RT_DN_BY + 2 * RT_DN_VAR_R)
#define RT_DN_ALBEDO_MIN 1e-3f                          // albedo channels at or below this demodulate by 1

// luminance3 of rt_device.cu (Rec. 709, the weights of k_max_luminance), in its order of operations
RT_DEV float dn_luminance(float x, float y, float z) { return x * 0.2126f + y * 0.7152f + z * 0.0722f; }

RT_DEV float3 dn_albedo(const float4* albedo, uint32_t i)
{
	if (!albedo) return v3(1.0f);
	const float4 a = __ldg(albedo + i);
	return v3(a.x > RT_DN_ALBEDO_MIN ? a.x : 1.0f, a.y > RT_DN_ALBEDO_MIN ? a.y : 1.0f, a.z > RT_DN_ALBEDO_MIN ? a.z : 1.0f);
}

// {n.xyz, class}: class 1 = surface, 0 = miss (an encoded normal of exactly (0,0,0))
RT_DEV float4 dn_guide(const float4* normal, uint32_t i)
{
	if (!normal) return make_float4(0.0f, 0.0f, 1.0f, 1.0f);
	const float4 e = __ldg(normal + i);
	if (e.x == 0.0f && e.y == 0.0f && e.z == 0.0f) return make_float4(0.0f, 0.0f, 0.0f, 0.0f);
	const float x = 2.0f * e.x - 1.0f, y = 2.0f * e.y - 1.0f, z = 2.0f * e.z - 1.0f;
	const float len = sqrtf(x * x + y * y + z * z);
	if (len > 0.0f) return make_float4(x / len, y / len, z / len, 1.0f);
	return make_float4(0.0f, 0.0f, 0.0f, 1.0f);
}

RT_DEV float3 dn_irradiance(float3 c, float3 a) { return v3(c.x / a.x, c.y / a.y, c.z / a.z); }

// kSums: `color` is the accumulator's running sums of n samples; otherwise a colour image and the spatial variance
template <bool kSums>
__global__ void __launch_bounds__(RT_DN_BX * RT_DN_BY) k_denoise_prepare(const float4* color, float n, const float4* albedo,
                                                                        const float4* normal, int width, int height,
                                                                        float4* rec, float4* guide)
{
	const int x = blockIdx.x * RT_DN_BX + threadIdx.x, y = blockIdx.y * RT_DN_BY + threadIdx.y;
	__shared__ float2 tile[RT_DN_TILE_W * RT_DN_TILE_H];     // {luminance of the irradiance, class}, -1 = outside
	if (!kSums)
	{
		const int x0 = blockIdx.x * RT_DN_BX - RT_DN_VAR_R, y0 = blockIdx.y * RT_DN_BY - RT_DN_VAR_R;
		for (int t = threadIdx.y * RT_DN_BX + threadIdx.x; t < RT_DN_TILE_W * RT_DN_TILE_H; t += RT_DN_BX * RT_DN_BY)
		{
			const int gx = x0 + t % RT_DN_TILE_W, gy = y0 + t / RT_DN_TILE_W;
			float2 v = make_float2(0.0f, -1.0f);
			if (gx >= 0 && gx < width && gy >= 0 && gy < height)
			{
				const uint32_t q = (uint32_t)gy * (uint32_t)width + (uint32_t)gx;
				const float3 irr = dn_irradiance(xyz(__ldg(color + q)), dn_albedo(albedo, q));
				v = make_float2(dn_luminance(irr.x, irr.y, irr.z), dn_guide(normal, q).w);
			}
			tile[t] = v;
		}
		__syncthreads();
	}
	if (x >= width || y >= height) return;
	const uint32_t i = (uint32_t)y * (uint32_t)width + (uint32_t)x;
	const float3 a = dn_albedo(albedo, i);
	const float4 g = dn_guide(normal, i);
	float3 irr;
	float var;
	if (kSums)
	{
		// the resolve of k_resolve, and its variance of one sample's luminance, divided by n: the variance of the mean
		const float4 s = __ldg(color + i);
		irr = dn_irradiance(div_assign3(xyz(s), n), a);
		const float m = dn_luminance(s.x, s.y, s.z) / n;
		const float sampleVar = fmaxf(0.0f, (s.w - n * m * m) / (n - 1.0f));
		const float ya = dn_luminance(a.x, a.y, a.z);
		var = sampleVar / n / (ya * ya);
	}
	else
	{
		irr = dn_irradiance(xyz(__ldg(color + i)), a);
		float sy = 0.0f, sy2 = 0.0f, k = 0.0f;
		for (int dy = -RT_DN_VAR_R; dy <= RT_DN_VAR_R; ++dy)
			for (int dx = -RT_DN_VAR_R; dx <= RT_DN_VAR_R; ++dx)
			{
				const float2 v = tile[(threadIdx.y + RT_DN_VAR_R + dy) * RT_DN_TILE_W + threadIdx.x + RT_DN_VAR_R + dx];
				if (v.y == g.w) { sy += v.x; sy2 += v.x * v.x; k += 1.0f; }
			}
		const float m1 = sy / k, m2 = sy2 / k;
		var = fmaxf(0.0f, m2 - m1 * m1);
	}
	rec[i] = make_float4(irr.x, irr.y, irr.z, var);
	guide[i] = g;
}

// out == NULL: writes the next {irradiance, variance} records; otherwise the remodulated colour (alpha 1)
__global__ void __launch_bounds__(RT_DN_BX * RT_DN_BY) k_denoise_atrous(const float4* rec, const float4* guide, int width,
                                                                       int height, int step, float4* recOut,
                                                                       const float4* albedo, float4* out)
{
	const int x = blockIdx.x * RT_DN_BX + threadIdx.x, y = blockIdx.y * RT_DN_BY + threadIdx.y;
	if (x >= width || y >= height) return;
	const uint32_t i = (uint32_t)y * (uint32_t)width + (uint32_t)x;
	const float4 rp = __ldg(rec + i), gp = __ldg(guide + i);
	const float yp = dn_luminance(rp.x, rp.y, rp.z);

	// 3 x 3 (1/4, 1/2, 1/4) blur of the variance over the in-image neighbours, renormalised
	float bs = 0.0f, bw = 0.0f;
	for (int dy = -1; dy <= 1; ++dy)
	{
		const int qy = y + dy;
		if (qy < 0 || qy >= height) continue;
		for (int dx = -1; dx <= 1; ++dx)
		{
			const int qx = x + dx;
			if (qx < 0 || qx >= width) continue;
			const float w = (dx == 0 ? 0.5f : 0.25f) * (dy == 0 ? 0.5f : 0.25f);
			bs += w * __ldg(rec + (uint32_t)qy * (uint32_t)width + (uint32_t)qx).w;
			bw += w;
		}
	}
	const float denom = 4.0f * sqrtf(bs / bw) + 1e-10f;

	float sw = 0.0f, sv = 0.0f;
	float3 sc = v3(0.0f);
	for (int dy = -2; dy <= 2; ++dy)
	{
		const int qy = y + dy * step;
		if (qy < 0 || qy >= height) continue;
		const float hy = dy == 0 ? 0.375f : (dy == 1 || dy == -1) ? 0.25f : 0.0625f;
		for (int dx = -2; dx <= 2; ++dx)
		{
			const int qx = x + dx * step;
			if (qx < 0 || qx >= width) continue;
			const uint32_t q = (uint32_t)qy * (uint32_t)width + (uint32_t)qx;
			const float4 rq = __ldg(rec + q), gq = __ldg(guide + q);
			float w;
			if (dx == 0 && dy == 0) w = 0.140625f;             // h(0)^2 = 9/64: the centre always counts
			else
			{
				const float hx = dx == 0 ? 0.375f : (dx == 1 || dx == -1) ? 0.25f : 0.0625f;
				float wn;
				if (gp.w != 0.0f && gq.w != 0.0f)
				{
					wn = fmaxf(0.0f, gp.x * gq.x + gp.y * gq.y + gp.z * gq.z);
					for (int k = 0; k < 7; ++k) wn = wn * wn;     // ^128
				}
				else wn = gp.w == gq.w ? 1.0f : 0.0f;
				const float wl = rt_expf(-fabsf(yp - dn_luminance(rq.x, rq.y, rq.z)) / denom);
				w = hx * hy * wn * wl;
			}
			sw += w;
			sc = v3(sc.x + w * rq.x, sc.y + w * rq.y, sc.z + w * rq.z);
			sv += w * w * rq.w;
		}
	}
	const float3 f = v3(sc.x / sw, sc.y / sw, sc.z / sw);
	if (out)
	{
		const float3 a = dn_albedo(albedo, i);
		out[i] = make_float4(f.x * a.x, f.y * a.y, f.z * a.z, 1.0f);
	}
	else recOut[i] = make_float4(f.x, f.y, f.z, sv / (sw * sw));
}

extern "C" uint64_t rt_denoise_scratch_bytes(uint32_t width, uint32_t height) { return (uint64_t)width * height * 48ull; }

static int denoise(int device, const void* color, uint32_t n, const void* albedo, const void* normal, uint32_t width,
                   uint32_t height, void* scratch, void* out, void* streamPtr, double* deviceMs)
{
	if (!color || !scratch || !out || width == 0 || height == 0) { g_denoiseError = "rt_denoise: null or empty image"; return -1; }
	const dim3 block(RT_DN_BX, RT_DN_BY), grid((width + RT_DN_BX - 1) / RT_DN_BX, (height + RT_DN_BY - 1) / RT_DN_BY);
	if ((uint64_t)width * height >= (1ull << 31) || grid.y > 65535u) { g_denoiseError = "rt_denoise: image too large"; return -1; }
	RT_DN_CUDA(cudaSetDevice(device));
	cudaStream_t stream = (cudaStream_t)streamPtr;
	const uint64_t count = (uint64_t)width * height;
	float4* recA = reinterpret_cast<float4*>(scratch);
	float4* recB = recA + count;
	float4* guide = recB + count;
	const float4* alb = reinterpret_cast<const float4*>(albedo);
	const float4* nrm = reinterpret_cast<const float4*>(normal);
	struct Events { cudaEvent_t e[2] = { nullptr, nullptr }; ~Events() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); } } ev;
	if (deviceMs)
	{
		RT_DN_CUDA(cudaEventCreate(&ev.e[0]));
		RT_DN_CUDA(cudaEventCreate(&ev.e[1]));
		RT_DN_CUDA(cudaEventRecord(ev.e[0], stream));
	}
	if (n) k_denoise_prepare<true><<<grid, block, 0, stream>>>(reinterpret_cast<const float4*>(color), (float)n, alb, nrm,
	                                                            (int)width, (int)height, recA, guide);
	else k_denoise_prepare<false><<<grid, block, 0, stream>>>(reinterpret_cast<const float4*>(color), 0.0f, alb, nrm,
	                                                           (int)width, (int)height, recA, guide);
	for (int step = 1; step <= 16; step *= 2)
	{
		const bool last = step == 16;
		k_denoise_atrous<<<grid, block, 0, stream>>>(recA, guide, (int)width, (int)height, step, recB, alb,
		                                             last ? reinterpret_cast<float4*>(out) : nullptr);
		float4* t = recA; recA = recB; recB = t;
	}
	RT_DN_CUDA(cudaGetLastError());
	if (deviceMs)
	{
		RT_DN_CUDA(cudaEventRecord(ev.e[1], stream));
		RT_DN_CUDA(cudaEventSynchronize(ev.e[1]));
		float ms = 0.0f;
		RT_DN_CUDA(cudaEventElapsedTime(&ms, ev.e[0], ev.e[1]));
		*deviceMs = ms;
	}
	RT_DN_CUDA(cudaStreamSynchronize(stream));
	return 0;
}

extern "C" int rt_denoise(int device, const void* color, const void* albedo, const void* normal, uint32_t width, uint32_t height,
                          void* scratch, void* out, void* stream, double* deviceMs)
{
	return denoise(device, color, 0, albedo, normal, width, height, scratch, out, stream, deviceMs);
}

extern "C" int rt_denoise_sums(int device, const void* sums, uint32_t n, const void* albedo, const void* normal, uint32_t width,
                               uint32_t height, void* scratch, void* out, void* stream, double* deviceMs)
{
	if (n < 2) { g_denoiseError = "rt_denoise_sums: the variance needs at least 2 samples"; return -1; }
	return denoise(device, sums, n, albedo, normal, width, height, scratch, out, stream, deviceMs);
}
