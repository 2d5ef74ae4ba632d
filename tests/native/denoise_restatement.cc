// denoise_restatement.cc -- the denoiser of csrc/device/rt_denoise.cu (DESIGN.md section 14) restated in plain C++, the
// reference its output is held to bit for bit.  Built by tests/test_denoise.py with g++ -O2 -ffp-contract=off (no FMA
// contraction, like nvcc --fmad=false); the exponential is include/rt_libm.h's, as on the device.
//
// Images are row-major W x H RGBA float32 arrays; albedo and normal may be NULL.
#include "rt_libm.h"

#include <math.h>
#include <stdint.h>
#include <vector>

namespace
{
	struct F4 { float x, y, z, w; };

	float Luminance(float x, float y, float z) { return x * 0.2126f + y * 0.7152f + z * 0.0722f; }

	// a' = a > 1e-3 ? a : 1 per channel; a null albedo is 1
	void Albedo(const float* albedo, size_t i, float a[3])
	{
		for (int c = 0; c < 3; ++c) a[c] = (!albedo || !(albedo[4 * i + c] > 1e-3f)) ? 1.0f : albedo[4 * i + c];
	}

	// {n.xyz, class}: 1 = surface, 0 = miss (encoded (0,0,0)); a null normal image is a surface facing +z everywhere
	F4 Guide(const float* normal, size_t i)
	{
		if (!normal) return { 0.0f, 0.0f, 1.0f, 1.0f };
		const float* e = normal + 4 * i;
		if (e[0] == 0.0f && e[1] == 0.0f && e[2] == 0.0f) return { 0.0f, 0.0f, 0.0f, 0.0f };
		const float x = 2.0f * e[0] - 1.0f, y = 2.0f * e[1] - 1.0f, z = 2.0f * e[2] - 1.0f;
		const float len = sqrtf(x * x + y * y + z * z);
		if (len > 0.0f) return { x / len, y / len, z / len, 1.0f };
		return { 0.0f, 0.0f, 0.0f, 1.0f };
	}

	// B3-spline taps h(-2..2)
	float H(int d) { return d == 0 ? 0.375f : (d == 1 || d == -1) ? 0.25f : 0.0625f; }

	void Filter(std::vector<F4>& rec, const std::vector<F4>& guide, const float* albedo, int W, int H_, float* out)
	{
		std::vector<F4> next(rec.size());
		for (int step = 1; step <= 16; step *= 2)
		{
			const bool last = step == 16;
			for (int y = 0; y < H_; ++y)
				for (int x = 0; x < W; ++x)
				{
					const size_t i = (size_t)y * W + x;
					const F4 rp = rec[i], gp = guide[i];
					const float yp = Luminance(rp.x, rp.y, rp.z);
					float bs = 0.0f, bw = 0.0f;
					for (int dy = -1; dy <= 1; ++dy)
						for (int dx = -1; dx <= 1; ++dx)
						{
							const int qx = x + dx, qy = y + dy;
							if (qx < 0 || qx >= W || qy < 0 || qy >= H_) continue;
							const float w = (dx == 0 ? 0.5f : 0.25f) * (dy == 0 ? 0.5f : 0.25f);
							bs += w * rec[(size_t)qy * W + qx].w;
							bw += w;
						}
					const float denom = 4.0f * sqrtf(bs / bw) + 1e-10f;
					float sw = 0.0f, sx = 0.0f, sy = 0.0f, sz = 0.0f, sv = 0.0f;
					for (int dy = -2; dy <= 2; ++dy)
						for (int dx = -2; dx <= 2; ++dx)
						{
							const int qx = x + dx * step, qy = y + dy * step;
							if (qx < 0 || qx >= W || qy < 0 || qy >= H_) continue;
							const size_t q = (size_t)qy * W + qx;
							const F4 rq = rec[q], gq = guide[q];
							float w;
							if (dx == 0 && dy == 0) w = 9.0f / 64.0f;
							else
							{
								float wn;
								if (gp.w != 0.0f && gq.w != 0.0f)
								{
									wn = fmaxf(0.0f, gp.x * gq.x + gp.y * gq.y + gp.z * gq.z);
									for (int k = 0; k < 7; ++k) wn = wn * wn;
								}
								else wn = gp.w == gq.w ? 1.0f : 0.0f;
								const float wl = rt_expf(-fabsf(yp - Luminance(rq.x, rq.y, rq.z)) / denom);
								w = H(dx) * H(dy) * wn * wl;
							}
							sw += w;
							sx += w * rq.x; sy += w * rq.y; sz += w * rq.z;
							sv += w * w * rq.w;
						}
					const float fx = sx / sw, fy = sy / sw, fz = sz / sw;
					if (last)
					{
						float a[3];
						Albedo(albedo, i, a);
						out[4 * i + 0] = fx * a[0]; out[4 * i + 1] = fy * a[1]; out[4 * i + 2] = fz * a[2]; out[4 * i + 3] = 1.0f;
					}
					else next[i] = { fx, fy, fz, sv / (sw * sw) };
				}
			rec.swap(next);
		}
	}
}

extern "C" {

// Colour image: the variance is the spatial one of the demodulated luminance over the same-class in-image pixels of the
// 7 x 7 window, max(0, E[Y^2] - E[Y]^2), summed row by row.
void denoise_restated(const float* color, const float* albedo, const float* normal, int W, int H_, float* out)
{
	const size_t n = (size_t)W * H_;
	std::vector<F4> guide(n), rec(n);
	std::vector<float> lum(n);
	for (size_t i = 0; i < n; ++i)
	{
		float a[3];
		Albedo(albedo, i, a);
		guide[i] = Guide(normal, i);
		rec[i] = { color[4 * i] / a[0], color[4 * i + 1] / a[1], color[4 * i + 2] / a[2], 0.0f };
		lum[i] = Luminance(rec[i].x, rec[i].y, rec[i].z);
	}
	for (int y = 0; y < H_; ++y)
		for (int x = 0; x < W; ++x)
		{
			const size_t i = (size_t)y * W + x;
			float s = 0.0f, s2 = 0.0f, k = 0.0f;
			for (int dy = -3; dy <= 3; ++dy)
				for (int dx = -3; dx <= 3; ++dx)
				{
					const int qx = x + dx, qy = y + dy;
					if (qx < 0 || qx >= W || qy < 0 || qy >= H_) continue;
					const size_t q = (size_t)qy * W + qx;
					if (guide[q].w != guide[i].w) continue;
					s += lum[q]; s2 += lum[q] * lum[q]; k += 1.0f;
				}
			const float m1 = s / k, m2 = s2 / k;
			rec[i].w = fmaxf(0.0f, m2 - m1 * m1);
		}
	Filter(rec, guide, albedo, W, H_, out);
}

// Running sums {sum R, sum G, sum B, sum Y^2} of n samples: colour = sum * (1 / n) (the resolve), variance = that of the
// mean luminance, var / n / luminance(albedo)^2 with var = max(0, (sum Y^2 - n m^2) / (n - 1)), m = luminance(sum) / n.
void denoise_sums_restated(const float* sums, uint32_t samples, const float* albedo, const float* normal, int W, int H_, float* out)
{
	const size_t count = (size_t)W * H_;
	const float n = (float)samples, inv = 1.0f / n;
	std::vector<F4> guide(count), rec(count);
	for (size_t i = 0; i < count; ++i)
	{
		float a[3];
		Albedo(albedo, i, a);
		guide[i] = Guide(normal, i);
		const float* s = sums + 4 * i;
		const float m = Luminance(s[0], s[1], s[2]) / n;
		const float var = fmaxf(0.0f, (s[3] - n * m * m) / (n - 1.0f));
		const float ya = Luminance(a[0], a[1], a[2]);
		rec[i] = { s[0] * inv / a[0], s[1] * inv / a[1], s[2] * inv / a[2], var / n / (ya * ya) };
	}
	Filter(rec, guide, albedo, W, H_, out);
}

}
