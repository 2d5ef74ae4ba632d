// raylib_b200.h -- C-ABI additions of the B200 build.  Nothing here is needed by a client that
// only uses the reference API in raylib.h; these calls expose what a GPU deployment adds:
// deterministic seeding, device-resident output, tile-sharded rendering for one-process-per-GPU
// launches (the frame is partitioned by interleaved 16x16 tiles, scene replicated per GPU, and
// the only exchange is one gather of the shard buffers), timing/ray statistics, and a closest-hit
// query used by the parity tests.
//
// Reference interfaces they extend:
//   RaylibB200_RenderShard / _RenderShardToFrame / _AssembleShards / _RenderToDevice  -> Raylib_Render (raylib/raylib.h:106-110)
//   RaylibB200_TraceRays / _PrimaryHits / _TraceRaysStaged      -> BVHNode::Hit  (raylib/geom/bvh.cc:82-107)
//   RaylibB200_SetFrameSeed / _SetBvhBuildKey                   -> std::random_device seeding (raylib/core/random.h:17-29, geom/bvh.cc:43)
//   RaylibB200_RenderAccumulate / _Accumulator*                 -> Raylib_Render in installments (progressive rendering)
#pragma once
#include "raylib_types.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct RaylibB200Stats
{
	uint64_t rayQueries;        // scene-level ray queries (camera + scattered + sun-shadow + debug second rays)
	uint64_t pixelSamples;      // pixels * samples rendered
	uint64_t boxTests, triTests, sphereTests, nodeVisits;   // work done by the device traversal (RaylibB200_SetCollectStats)
	uint64_t refBoxTests, refTriTests, refSphereTests;      // work the reference's exhaustive traversal does for the same
	uint64_t statRays;                                      //   statRays closest-hit rays (roofline accounting)
	double   deviceMs;          // CUDA-event time of the kernels of the last render on this rank
	double   extendMs;          // sum of the traversal (k_extend) launch durations (RaylibB200_SetTimeStages)
	uint32_t extendLaunches;
	uint32_t pad0;
	double   totalMs;           // wall time of the whole call (upload of per-frame data, kernels, readback)
	uint64_t h2dBytes, d2hBytes;
	uint32_t kernelLaunches;
	uint32_t passes;
	uint32_t device;
	uint32_t devicesUsed;       // GPUs the frame was spread over (Raylib_Render uses every active device for large frames)
	// RaylibB200_SetCollectStats: SIMD occupancy of the traversal loop, in lane-iterations (lanes per instruction of a phase
	// = 32 * busy / iterations): node phase all / stepping / owning a ray, leaf phase all / testing a leaf
	uint64_t nodeIters, nodeStep, nodeAlive, leafIters, leafBusy;
	uint64_t gateTests, cubeTests;   // RaylibB200_SetCollectStats: exact gate-box tests of accepted hits, cube tests
} RaylibB200Stats;

// Number of usable CUDA devices (0 = none; Raylib_Render then fails loudly, there is no CPU path).
RAYLIB_API int32_t RaylibB200_DeviceCount(void);
// Device used by this process (default: $RAYLIB_B200_DEVICE, else $LOCAL_RANK, else 0).
RAYLIB_API int32_t RaylibB200_SetDevice(int32_t device);
RAYLIB_API int32_t RaylibB200_GetDevice(void);
// Raylib_Render spreads a frame over several GPUs of the box inside ONE process, like the reference spreads it over every
// core (raylib/render/renderer.cc:286,302-334): interleaved 16x16 tiles, scene replicated per GPU (cloned device to device
// over NVLink), final pixels stored straight into the frame on the first device through peer mappings, one read-back.
// Default: every visible device, unless the process is pinned to one (RaylibB200_SetDevice, $RAYLIB_B200_DEVICE, $LOCAL_RANK
// of a one-process-per-GPU launch) or $RAYLIB_B200_DEVICES = all | k | a,b,c says otherwise.  SetDevices(k) selects the
// first k devices (0 = all) and returns how many are in use.  The image does not depend on the device count.
// Frames below $RAYLIB_B200_MULTI_MIN_SAMPLES pixel-samples (default 2 Mi) stay on the first device.
RAYLIB_API int32_t RaylibB200_SetDevices(int32_t count);
RAYLIB_API int32_t RaylibB200_GetDeviceCountInUse(void);
// Re-reads the RAYLIB_B200_* tuning variables (DESIGN.md section 9); they are otherwise read once per process.
RAYLIB_API void RaylibB200_ReloadTuning(void);

// Frame seed of the per-(pixel, sample) random streams (default 1337) and key of the BVH split-axis stream (default 0xB7).
RAYLIB_API void RaylibB200_SetFrameSeed(uint64_t seed);
RAYLIB_API void RaylibB200_SetBvhBuildKey(uint64_t key);
// 1 = count box/triangle/sphere tests in the traversal kernels (slower).
RAYLIB_API void RaylibB200_SetCollectStats(int32_t enable);
// 1 = bracket every traversal launch with CUDA events and report their sum in RaylibB200Stats.extendMs.
RAYLIB_API void RaylibB200_SetTimeStages(int32_t enable);
// Passes in flight at once (1..4, 0 = default 2): each pass runs on its own stream and path-state arena, so the
// memory-bound stage kernels of one pass overlap the traversal kernels of another.  The image does not depend on it.
RAYLIB_API void RaylibB200_SetPipes(uint32_t pipes);
// Samples kept in flight per pixel per pass (0 = automatic).
RAYLIB_API void RaylibB200_SetSamplesPerPass(uint32_t samples);
// Small frames render as ONE cooperative launch per frame (grid-wide barriers between the stages instead of kernel
// boundaries).  0 = automatic (frames of at most 1 Mi paths, $RAYLIB_B200_FUSED_PATHS_K), 1 = never, 2 = whenever the
// frame's samples fit in flight at once.  The image does not depend on it.
RAYLIB_API void RaylibB200_SetFusedPass(uint32_t mode);

// Statistics of the last Raylib_Render / RaylibB200_Render* call made by this thread. Returns 1 if available.
RAYLIB_API int32_t RaylibB200_GetLastStats(RaylibB200Stats* outStats);
// Human-readable reason of the last failure on this thread ("" if none).
RAYLIB_API const char* RaylibB200_GetLastError(void);

// Bytes the flattened scene occupies on the device (0 if not uploaded). Uploads lazily.
RAYLIB_API uint64_t RaylibB200_SceneDeviceBytes(SceneHandle scene);
// Counts of the flattened scene: out[0]=nodes, [1]=triangles, [2]=spheres, [3]=cubes, [4]=materials, [5]=textures, [6]=max node depth, [7]=leaves
RAYLIB_API int32_t RaylibB200_SceneCounts(SceneHandle scene, uint64_t* out8);

// ---- tile-sharded rendering ------------------------------------------------------------------
// A shard buffer holds RaylibB200_ShardPixelCapacity(...) RGBA float4 pixels (tile-major).
RAYLIB_API uint64_t RaylibB200_ShardPixelCapacity(uint32_t width, uint32_t height, uint32_t shardCount);
// Renders the tiles t with t % shardCount == shardRank into deviceShardOut (device memory on this
// process' device).  cudaStream may be NULL (default stream).  Synchronous: returns when the shard is complete.
RAYLIB_API int32_t RaylibB200_RenderShard(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	uint32_t shardRank, uint32_t shardCount, void* deviceShardOut, void* cudaStream);
// De-interleaves shardCount gathered shard buffers (rank-major, contiguous) into a row-major W x H RGBA float4 device image.
RAYLIB_API int32_t RaylibB200_AssembleShards(const void* deviceShards, uint32_t shardCount,
	uint32_t width, uint32_t height, void* deviceImageOut, void* cudaStream);
// ---- shared frame: the gather fused into the render ------------------------------------------------
// One process per GPU, all on one NVLink/NVSwitch box: one rank creates the row-major W x H RGBA float4 frame and
// exports a 64-byte CUDA IPC handle, the others map it; every rank then renders the final pixels of its tiles
// STRAIGHT into that frame (the last k_accumulate stores through the peer mapping), so no shard buffer, no
// collective and no de-interleave pass exist.  The launcher only has to order "all ranks returned" before reading
// the frame (a barrier).  Output is bit-identical to RenderShard + gather + AssembleShards.
// RenderShardToFrame is synchronous like RenderShard.  deviceFrame may also be plain local device memory
// (shardCount 1 = RaylibB200_RenderToDevice).
RAYLIB_API int32_t RaylibB200_RenderShardToFrame(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	uint32_t shardRank, uint32_t shardCount, void* deviceFrame, void* cudaStream);
// Allocates the frame on this process' device; outIpcHandle64 (nullable) receives the handle to pass to the other ranks.
RAYLIB_API void*   RaylibB200_FrameCreate(uint32_t width, uint32_t height, unsigned char* outIpcHandle64);
RAYLIB_API void    RaylibB200_FrameDestroy(void* deviceFrame);
// Maps a frame created by another process (peer access over NVLink is enabled lazily).  NULL on failure.
RAYLIB_API void*   RaylibB200_FrameOpen(const unsigned char* ipcHandle64);
RAYLIB_API int32_t RaylibB200_FrameClose(void* mappedFrame);
// Device -> host copy of a frame (hostRgbaOut: W*H*4 floats, ideally pinned).
RAYLIB_API int32_t RaylibB200_FrameRead(const void* deviceFrame, uint32_t width, uint32_t height, float* hostRgbaOut, void* cudaStream);

// Host-side helpers for launchers that move shard buffers through host memory (MPI / gloo) and for tests:
// outPixelIndex[slot] = y*width+x of the image pixel stored in that shard slot, or -1 for padding.
RAYLIB_API int32_t RaylibB200_ShardPixelMap(uint32_t width, uint32_t height, uint32_t shardRank, uint32_t shardCount, int64_t* outPixelIndex);
RAYLIB_API int32_t RaylibB200_AssembleShardsHost(const float* hostShards, uint32_t shardCount,
	uint32_t width, uint32_t height, float* hostImageOut);
// Whole frame on one device into device memory (W x H RGBA float4, row-major); no host copy of the image.
RAYLIB_API int32_t RaylibB200_RenderToDevice(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	void* deviceImageOut, void* cudaStream);

// ---- the steps around the path: denoiser inputs and post-processing ------------------------------------
// Albedo and MicrosurfaceNormal views (ERenderMode 1 and 3) from ONE primary-hit pass instead of two more
// Raylib_Render calls (reference callers: src/main.cc:464-476, gui-app MainForm.cs:191-198).  Pixel values are
// identical to the two separate renders.  Images are resized to the settings' viewport.
RAYLIB_API int32_t RaylibB200_RenderAux(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	ImageHandle outAlbedoImage, ImageHandle outNormalImage);
// Image2D::PostProcess (raylib/render/image.cc:44-103: max-luminance, extended Reinhard, clamp, gamma 2.2) as CUDA
// kernels.  Device form: W x H RGBA float4 image in place; outArgb8 (nullable, W*H uint32) receives Pixel::ToUint32
// of the result; outMaxWhite (nullable) the reduced maximum luminance.  Host form: same on an Image2D (H2D + D2H).
RAYLIB_API int32_t RaylibB200_PostProcessDevice(void* deviceImage, uint32_t width, uint32_t height, void* deviceOutArgb8,
	float* outMaxWhite, void* cudaStream);
RAYLIB_API int32_t RaylibB200_PostProcessGPU(ImageHandle image);

// Raw RGBA access to an image handle (the reference ABI only reads RGB back, Raylib_DumpImageData): W*H*4 floats, row 0 on top.
// SetRGBA resizes the image.  Both return 1 on success.
RAYLIB_API int32_t RaylibB200_ImageSetRGBA(ImageHandle image, uint32_t width, uint32_t height, const float* rgba);
RAYLIB_API int32_t RaylibB200_ImageGetRGBA(ImageHandle image, float* outRgba);

// ---- progressive rendering: a frame in installments -----------------------------------------------
// An accumulator holds, for every pixel of a W x H frame, the float sums {sum R, sum G, sum B, sum luminance^2} of the
// samples rendered so far, on the device that was current when it was created, and their count n.  RenderAccumulate
// renders samples [n, n + samples) of every pixel and adds them to the sums in sample order -- the float additions of
// one Raylib_Render of n + samples samples -- so that a resolve after any installment is BIT-IDENTICAL to Raylib_Render
// with samplesPerPixel = n at the same frame seed, whatever the installment sizes, pipes, passes or device count were.
// The first installment binds the accumulator to what decides the image: viewport (= the accumulator's size),
// maxPathLength, rayTMin, frame seed, camera, the sun the frame is rendered with, and the uploaded scene (a fingerprint of
// its arrays: a scene and its RaylibB200_LoadFlattenedScene reload are the same scene, a swapped sky is not).  A later
// installment that differs in any of them is refused (0; GetLastError names every differing field) and changes nothing: start a new
// image with Reset.  Installments spread over the active GPUs like Raylib_Render (the sums live on the first one, which
// must be the accumulator's device; without peer access they render there alone).  Functions returning int32_t return
// 1 on success and 0 on failure (GetLastError).
typedef struct RaylibB200Accumulator RaylibB200Accumulator;
// NULL without a CUDA device.  Create: n = 0, unbound.  Reset zeroes the sums and drops the binding.
RAYLIB_API RaylibB200Accumulator* RaylibB200_AccumulatorCreate(uint32_t width, uint32_t height);
RAYLIB_API void    RaylibB200_AccumulatorDestroy(RaylibB200Accumulator* acc);
RAYLIB_API int32_t RaylibB200_AccumulatorReset(RaylibB200Accumulator* acc);
RAYLIB_API uint32_t RaylibB200_AccumulatorSamples(const RaylibB200Accumulator* acc);      // n
// settings->samplesPerPixel is ignored; renderMode must be 0 (path tracing); n + samples <= 2^24 (the divisor stays exact).
// GetLastStats reports this installment (its pixel-samples, ray queries, passes).
RAYLIB_API int32_t RaylibB200_RenderAccumulate(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	RaylibB200Accumulator* acc, uint32_t samples);
// The average of the n samples (alpha 1) into an Image2D (resized like Raylib_Render resizes it) or into a W x H RGBA float4
// device image on the accumulator's device (cudaStream may be NULL; synchronous).
RAYLIB_API int32_t RaylibB200_AccumulatorResolve(RaylibB200Accumulator* acc, ImageHandle outImage);
RAYLIB_API int32_t RaylibB200_AccumulatorResolveDevice(RaylibB200Accumulator* acc, void* deviceImageOut, void* cudaStream);
// The raw sums, W*H*4 floats {sum R, sum G, sum B, sum luminance^2}, row 0 on top.
RAYLIB_API int32_t RaylibB200_AccumulatorRead(RaylibB200Accumulator* acc, float* outRgba);
// Relative standard error of each pixel's mean luminance: with m = luminance(sum) / n and var = max(0, (sumY2 - n m^2) / (n - 1)),
// sqrt(var / n) / max(m, 1e-4).  perPixel (nullable) receives W*H floats, mean (nullable) their average, summed in a fixed
// order (the same sums give the same double).  Needs n >= 2.
RAYLIB_API int32_t RaylibB200_AccumulatorNoise(RaylibB200Accumulator* acc, float* perPixel, double* mean);
// Checkpoint file: header, binding, n, sums and a checksum.  Load validates the whole file before it touches a device (a
// foreign, truncated or damaged file is refused even without a GPU) and creates the accumulator on the current device.
RAYLIB_API int32_t RaylibB200_AccumulatorSave(const RaylibB200Accumulator* acc, const char* path);
RAYLIB_API RaylibB200Accumulator* RaylibB200_AccumulatorLoad(const char* path);

// ---- denoising: the step between RenderAux and post-processing ------------------------------------------
// An edge-avoiding a-trous filter guided by the albedo and normal views RaylibB200_RenderAux writes (spatial SVGF without
// its temporal part; DESIGN.md section 14): the colour is divided by the albedo, filtered in five iterations weighted by
// normal agreement and by luminance distance over the estimated noise, and multiplied back.  A null albedo image counts as
// 1 everywhere; a null normal image makes every pixel a surface facing +z.  Normals are encoded 0.5 + 0.5 N, (0,0,0)
// marking a miss.  The output (alpha 1) is a pure function of the inputs: the same inputs give the same bits on every
// call.  All three calls are synchronous and return 1 on success or 0 (GetLastError); their arguments are checked before
// a device is used.  GetLastStats reports the call (device and wall time, launches, copies; no rays).
// Noise estimate: the image and device forms only have the image, so they estimate each pixel's variance spatially, over
// its 7 x 7 neighbourhood.  That counts real high-frequency detail (fine geometry, texture, shadow edges) as noise and can
// blur it, making such scenes worse than the raw frame (measured: scatter10M and the textured room, DESIGN.md section 14).
// When the frame comes from an accumulator, prefer RaylibB200_AccumulatorDenoise: it uses each pixel's exact sample
// variance and keeps that detail.
// Raylib_Denoise's image arguments (raylib/raylib.h) without the HDR flag: the filter does not depend on the range.
// outImage is resized to the main image's size; albedo and normal must have that size.  Raylib_Denoise keeps returning 0.
RAYLIB_API int32_t RaylibB200_Denoise(ImageHandle mainImage, ImageHandle albedoImage, ImageHandle normalImage, ImageHandle outImage);
// W x H RGBA float4 images in device memory of the current device (albedo and normal nullable), each 16-byte aligned
// (a misaligned pointer is refused); cudaStream may be NULL.
RAYLIB_API int32_t RaylibB200_DenoiseDevice(const void* deviceColor, const void* deviceAlbedo, const void* deviceNormal,
	uint32_t width, uint32_t height, void* deviceOut, void* cudaStream);
// The accumulator's resolved image, filtered with the exact per-pixel variance of its mean from the sums (divided by the
// squared luminance of the albedo: exact for grey albedo, an approximation for coloured).  Reads the sums in place and
// leaves them and n untouched.  Needs n >= 2; guides must have the accumulator's size.
RAYLIB_API int32_t RaylibB200_AccumulatorDenoise(RaylibB200Accumulator* acc, ImageHandle albedoImage, ImageHandle normalImage,
	ImageHandle outImage);

// ---- queries used by parity tests ---------------------------------------------------------------
// Closest hit of caller-supplied rays (8 floats each: o.xyz, time, d.xyz, unused).  outRank = global
// in-order leaf rank of the hit primitive or -1; outT = hit distance or 0.
RAYLIB_API int32_t RaylibB200_TraceRays(SceneHandle scene, const float* rays, int64_t numRays, float tMin,
	int32_t* outRank, float* outT);
// Primary visibility through the device ray generator: one unjittered camera ray per pixel.
RAYLIB_API int32_t RaylibB200_PrimaryHits(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	int32_t* outRank, float* outT);
// The same rays through the traversal kernels a render runs (TraceRays uses a plain one-ray-per-thread kernel): one launch
// of the closest-hit stage (mode 0: k_extend, 1: k_extend with statistics, 2: the pooled k_extend_pool) or of the
// sun-visibility any-hit stage (mode 3: k_shadow), with `order` (a permutation of 0..numRays-1) as the queue it drains and
// explicit scheduling: refill / walk thresholds (1..32, 0 = 20), the pooled kernel's node and refill thresholds (1..32 and
// 1..64, 0 = 24) and the grid in CTAs (1..4096, 0 = the persistent grid of a render).
//   Closest hit: outQueue[i] = the queue ray i was pushed to (material type 0..5 of the hit primitive, 6 = miss; -1 none,
//   -2 more than one), outHit[4i..4i+3] = its hit record {t, bu, bv, primitive reference bits} (bu/bv: triangle
//   barycentrics, bu = face 0..5 of a cube; a miss leaves all-ones bits), outQueueCounts[0..6] (nullable) = the counters.
//   Any hit: every ray is a sun-visibility ray from its origin at its shutter time along -sunDirection (the scene's sun
//   convention; the rays' own directions are not read): outQueue[i] = 0 visible, 1 occluded, -1 neither; outHit[4i..] =
//   the path's radiance with a sun of illuminance (1, 1, 1) and no sky.  sunDirection must be finite and non-zero.
// rays: 8 floats each (o.xyz, time, d.xyz, unused).  Arguments are checked before a device is used; GetLastStats reports the
// call (mode 1 fills the work counters, as TraceRays does with RaylibB200_SetCollectStats).  Returns 1 on success.
RAYLIB_API int32_t RaylibB200_TraceRaysStaged(SceneHandle scene, int32_t mode, const float* rays, const uint32_t* order,
	int64_t numRays, float tMin, const float* sunDirection, uint32_t refillThreshold, uint32_t walkThreshold,
	uint32_t poolNodeThreshold, uint32_t poolRefill, uint32_t gridCtas, int32_t* outQueue, float* outHit, uint32_t* outQueueCounts);

// The device's own sinf / cosf / tanf / asinf / acosf / atanf / expf / logf / powf / atan2f (fn 0..9; include/rt_libm.h:
// glibc's algorithms restated so that the GPU consumes the same bits as the reference's host build) evaluated on `count`
// arguments.  y may be NULL for the one-argument functions.  Returns 1 on success.
RAYLIB_API int32_t RaylibB200_LibmEval(int32_t fn, const float* x, const float* y, float* out, uint64_t count);

// ---- flattened-scene cache ------------------------------------------------------------------------------
// Writes the flattened form of a finalized scene (the arrays Raylib_Render uploads: traversal tree, triangle / sphere /
// cube records, materials, textures, sky, sun) to `path`, and reads such a file back as a scene handle that renders
// without the client object graph, the reference BVH build or the SAH pipeline -- what re-loading a San-Miguel-scale
// OBJ costs in the reference every time (raylib/loader/obj_loader.cc:128-245, geom/static_mesh.cc:80-95).  The file
// carries record sizes and a checksum; a file from another build or a damaged one is refused (GetLastError).
// The loaded handle works with Raylib_Render / RaylibB200_Render* / _TraceRays and is destroyed by Raylib_DestroyScene;
// it cannot be edited (no elements, sky and sun are the stored ones).  Both calls work without a GPU.
RAYLIB_API int32_t RaylibB200_SaveFlattenedScene(SceneHandle scene, const char* path);
RAYLIB_API SceneHandle RaylibB200_LoadFlattenedScene(const char* path);

// ---- host-only inspection of the flattened scene (works without a GPU) -----------------------------
// Returns the RtSceneDesc (include/rt_scene_format.h) that Raylib_Render would upload; owned by the
// library until RaylibB200_ReleaseInspection / scene destruction.  NULL on failure (see GetLastError).
struct RtSceneDesc;
struct RtCamera;
RAYLIB_API const struct RtSceneDesc* RaylibB200_FlattenForInspection(SceneHandle scene);
RAYLIB_API void RaylibB200_ReleaseInspection(SceneHandle scene);
RAYLIB_API int32_t RaylibB200_CameraBlock(CameraHandle camera, struct RtCamera* outCamera);

#ifdef __cplusplus
}
#endif
