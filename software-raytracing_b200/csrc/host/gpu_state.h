// gpu_state.h -- per-process GPU bookkeeping of libraylib: the device in use, its render context
// (path-state arenas) and the uploaded copy of every finalized scene.
#pragma once
#include "rt_device_abi.h"
#include "raylib_b200.h"
#include <memory>
#include <string>

struct RtFlatScene;
class Scene;
class Camera;
class Image2D;
struct RendererSettings;

namespace RtGpu
{
	int  DeviceCount();
	int  CurrentDevice();
	bool SetDevice(int device);
	// Devices a Raylib_Render frame is spread over: the first `count` visible devices (0 = all).  Returns how many.
	int  SetDevices(int count);
	int  ActiveDeviceCount();
	// Tuning knobs (RtTuning): read from the environment once per process, again on ReloadTuning().
	void ReloadTuning();
	const RtTuning& Tuning();
	// Drops the page-lock of an Image2D's storage before the storage goes away (Raylib_DestroyImage, Image2D::Reallocate).
	void ForgetHostImage(const Image2D* image);

	void SetFrameSeed(uint64_t seed);
	uint64_t FrameSeed();
	void SetCollectStats(bool enable);
	void SetTimeStages(bool enable);
	void SetSamplesPerPass(uint32_t samples);
	void SetPipes(uint32_t pipes);
	void SetFusedPass(uint32_t mode);

	void SetLastError(const std::string& message);
	const char* LastError();
	void SetLastStats(const RaylibB200Stats& stats);
	bool GetLastStats(RaylibB200Stats* out);

	// Flatten + upload (once per scene and device). nullptr on failure (LastError says why).
	const RtDeviceScene* AcquireScene(const Scene* scene, uint64_t* outCounts8 = nullptr);
	RtRenderContext* AcquireContext();
	// A scene whose flattened form was read from disk (RaylibB200_LoadFlattenedScene): AcquireScene uploads it as is.
	void AdoptPrebuilt(const Scene* scene, std::shared_ptr<RtFlatScene> flat);
	std::shared_ptr<RtFlatScene> Prebuilt(const Scene* scene);
	void ReleaseAll();

	// Samples [begin, end) of a whole frame added to the running sums of an accumulator (row-major W x H float4 on the
	// primary device): rt_render_window of rt_progressive.h.
	struct SampleWindow { uint32_t begin, end; void* sums; };

	// Shared implementation of every render entry point.  Exactly one of hostImage / deviceImage /
	// deviceShard / window is non-null.
	bool Render(const RendererSettings* settings, const Scene* scene, const Camera* camera,
	            Image2D* hostImage, void* deviceImage, void* deviceShard,
	            uint32_t shardRank, uint32_t shardCount, uint32_t renderModeOverride, void* stream, bool pinHostImage = false,
	            const SampleWindow* window = nullptr);

	// Progressive rendering (RaylibB200_Accumulator*, include/raylib_b200.h)
	RaylibB200Accumulator* AccumulatorCreate(uint32_t width, uint32_t height);
	void AccumulatorDestroy(RaylibB200Accumulator* acc);
	bool AccumulatorReset(RaylibB200Accumulator* acc);
	uint32_t AccumulatorSamples(const RaylibB200Accumulator* acc);
	bool RenderAccumulate(const RendererSettings* settings, const Scene* scene, const Camera* camera, RaylibB200Accumulator* acc, uint32_t samples);
	bool AccumulatorResolve(RaylibB200Accumulator* acc, Image2D* hostImage, void* deviceImage, void* stream);
	// The denoiser (rt_denoise_sums of rt_denoise.h) on the sums, which it leaves as they are; n >= 2, guides nullable.
	bool AccumulatorDenoise(RaylibB200Accumulator* acc, const Image2D* albedo, const Image2D* normal, Image2D* out);
	bool AccumulatorRead(RaylibB200Accumulator* acc, float* rgba);
	bool AccumulatorNoise(RaylibB200Accumulator* acc, float* perPixel, double* mean);
	bool AccumulatorSave(const RaylibB200Accumulator* acc, const char* path);
	RaylibB200Accumulator* AccumulatorLoad(const char* path);

	// Denoiser inputs in one primary-hit pass (reference: the Albedo and MicrosurfaceNormal debug renders of
	// src/main.cc:464-476, two extra Raylib_Render calls).  Host images are resized to the viewport.
	bool RenderAux(const RendererSettings* settings, const Scene* scene, const Camera* camera, Image2D* albedoImage, Image2D* normalImage);

	// Image2D::PostProcess on the GPU: device-resident RGBA float4 image in place, optional packed ARGB8 copy.
	bool PostProcessDevice(void* deviceImage, uint32_t width, uint32_t height, void* deviceOutArgb8, float* outMaxWhite, void* stream);
	// Same for a host Image2D (H2D, kernels, D2H); used for large frames.
	bool PostProcessHostImage(Image2D* image);

	// The denoiser (rt_denoise of rt_denoise.h) on host images (H2D, kernels, D2H; out is resized to the colour image) or on
	// W x H RGBA float4 images on the current device.  Guides are nullable.  Arguments are checked before a device is used.
	bool Denoise(const Image2D* color, const Image2D* albedo, const Image2D* normal, Image2D* out);
	bool DenoiseDevice(const void* color, const void* albedo, const void* normal, uint32_t width, uint32_t height, void* out, void* stream);
}
