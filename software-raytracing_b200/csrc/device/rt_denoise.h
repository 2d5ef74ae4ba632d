// rt_denoise.h -- device entry points of the denoiser (RaylibB200_Denoise* and RaylibB200_AccumulatorDenoise of
// include/raylib_b200.h).  Internal to libraylib_b200: hidden, unlike the thin device ABI of rt_device_abi.h.
//
// The filter (DESIGN.md section 14): spatial SVGF without its temporal part -- a prepare kernel that demodulates the colour
// by the albedo and estimates each pixel's luminance variance, then five edge-avoiding a-trous iterations (steps 1, 2, 4,
// 8, 16) weighted by normals and by luminance distance over the filtered standard deviation; the last one remodulates.
// Every sum runs in a fixed order without atomics, so the output is a pure function of the inputs, and
// tests/native/denoise_restatement.cc reproduces it bit for bit.
#pragma once
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

// Bytes of the scratch buffer the two entry points need: two {irradiance, variance} records and one guide record per pixel.
uint64_t rt_denoise_scratch_bytes(uint32_t width, uint32_t height);

// color, albedo (nullable: 1), normal (nullable: every pixel a surface facing +z, encoded 0.5 + 0.5 N, (0,0,0) = miss) and
// out are row-major W x H RGBA float4 images on `device`; out receives the filtered colour with alpha 1.  The variance is
// the spatial one of the demodulated luminance over the same-class pixels of the 7 x 7 window.  Synchronous; deviceMs
// (nullable) receives the CUDA-event time of the launches.  Returns 0 or a CUDA error code (rt_denoise_last_error).
int rt_denoise(int device, const void* color, const void* albedo, const void* normal, uint32_t width, uint32_t height,
               void* scratch, void* out, void* stream, double* deviceMs);

// The same on an accumulator's running sums {sum R, sum G, sum B, sum luminance^2} of n >= 2 samples: the colour is their
// resolve (sum * (1 / n)), the variance the sample variance of the mean luminance divided by luminance(albedo)^2.
int rt_denoise_sums(int device, const void* sums, uint32_t n, const void* albedo, const void* normal, uint32_t width,
                    uint32_t height, void* scratch, void* out, void* stream, double* deviceMs);

// Kernel launches of one call of either entry point.
#define RT_DENOISE_LAUNCHES 6u

const char* rt_denoise_last_error(void);

#ifdef __cplusplus
}
#endif
