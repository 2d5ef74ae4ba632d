// rt_progressive.h -- device entry points of progressive rendering (RaylibB200_RenderAccumulate and the accumulator
// calls of include/raylib_b200.h).  Internal to libraylib_b200: hidden, unlike the thin device ABI of rt_device_abi.h.
#pragma once
#include <stdint.h>
#include "rt_device_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

// Renders samples [sampleBegin, sampleEnd) of this shard's pixels; passes are sized by the window's length as a frame of that
// many samples would be.  runningSum == NULL: the window must start at 0 and this is rt_render_shard with sampleEnd samples.
// Otherwise (path tracing only) runningSum is the row-major W x H float4 buffer {sum R, sum G, sum B, sum luminance^2} of
// samples [0, sampleBegin) -- local or a peer GPU's memory -- and receives the sums of [0, sampleEnd): the same float
// additions, in the same order, as one frame of sampleEnd samples.
int rt_render_window(RtRenderContext* ctx, const RtDeviceScene* scene, const RtCamera* camera, const RtRenderParams* params,
                     uint32_t sampleBegin, uint32_t sampleEnd, void* runningSum, void* deviceShardOut, void* stream,
                     RtRenderStats* stats);

// From `count` running sums of n samples each: deviceImageOut (nullable) = sum / n with alpha 1, the division of the last
// pass of a one-shot frame; deviceNoiseOut (nullable) = relative standard error of the mean luminance per pixel (n >= 2);
// hostNoiseSum (nullable, n >= 2) = the sum of that figure over the pixels, reduced in a fixed order.  Synchronous.
int rt_resolve(int device, const void* sums, uint32_t count, uint32_t n, void* deviceImageOut, float* deviceNoiseOut,
               double* hostNoiseSum, void* stream);

// 64-bit fingerprint of what an upload holds (tree, primitive records, materials, textures, texels, scene scalars; not the
// sun, which a frame may override, nor the reference topology of statistics frames).  Equal arrays give equal values.
int rt_scene_fingerprint(const RtDeviceScene* scene, uint64_t* out);

int rt_device_zero(int device, void* ptr, uint64_t bytes);

#ifdef __cplusplus
}
#endif
