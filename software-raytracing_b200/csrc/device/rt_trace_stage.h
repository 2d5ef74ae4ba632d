// rt_trace_stage.h -- the traversal stage kernels of a render on caller rays (RaylibB200_TraceRaysStaged of
// include/raylib_b200.h, for the parity tests).  Internal to libraylib_b200: hidden, unlike the thin device ABI of
// rt_device_abi.h.
//
// rt_trace_closest runs k_trace_rays (one ray per thread); a frame's rays go through k_extend / k_extend_pool (lane refill,
// warp scheduling, hit records written as hits are accepted, material queues) and k_shadow (the only any-hit walk).
// rt_trace_stage runs ONE launch of one of those kernels at bounce 0 of pipe 0's arena: the rays go to the path records
// (layout of rt_trace_closest: o.xyz, time, d.xyz, unused), hostOrder (a permutation of 0..numRays-1) becomes the queue the
// kernel drains, and the scheduling is the caller's.
//   closest-hit modes: hostOutQueue[i] = the queue slot i was pushed to (RtMaterialType 0..5 of the hit, RT_STAGE_QUEUE_MISS),
//     -1 if it was pushed nowhere, -2 if more than once; hostOutHit[4i..4i+3] = the slot's hit record {t, bu, bv, ref bits}
//     (bu = face 0..5 of a cube, 0 for a sphere; a miss leaves the all-ones sentinel); hostOutQueueCounts[0..6] (nullable)
//     = the queues' counters.
//   RT_STAGE_SHADOW: every slot is a sun-visibility ray along -sunDirection (the scene's sun convention) with the scene's
//     sun replaced by illuminance (1, 1, 1) from sunDirection and no sky term: hostOutQueue[i] = 0 (the sun is visible, the
//     path's radiance is (1, 1, 1)), 1 (occluded, radiance 0) or -1 (anything else); hostOutHit[4i..] = that radiance.
// Synchronous.  Returns 0 or an error code (rt_last_error).
#pragma once
#include "rt_device_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

#define RT_STAGE_EXTEND        0     // k_extend<false>
#define RT_STAGE_EXTEND_STATS  1     // k_extend<true>: also fills the statistics counters
#define RT_STAGE_EXTEND_POOL   2     // k_extend_pool
#define RT_STAGE_SHADOW        3     // k_shadow (any hit)
#define RT_STAGE_QUEUE_MISS    6     // queue of the rays that hit nothing (after the six material queues)

typedef struct RtStageSchedule
{
	uint32_t refillThreshold;     // k_extend / k_shadow: a warp refills below this many live rays, 1..32 (0 = 20, as a render)
	uint32_t walkThreshold;       // 1..32 (0 = 20)
	uint32_t poolNodeThreshold;   // k_extend_pool: node step while this many rays can step, 1..32 (0 = 24)
	uint32_t poolRefill;          // k_extend_pool: refill once this many ray slots are free, 1..64 (0 = 24)
	uint32_t gridCtas;            // CTAs of the launch (0 = the persistent grid a render launches)
} RtStageSchedule;

int rt_trace_stage(RtRenderContext* ctx, const RtDeviceScene* scene, int mode, const float* hostRays, const uint32_t* hostOrder,
                   int64_t numRays, float tMin, const float* sunDirection, const RtStageSchedule* schedule, int32_t* hostOutQueue,
                   float* hostOutHit, uint32_t* hostOutQueueCounts, RtRenderStats* stats);

#ifdef __cplusplus
}
#endif
