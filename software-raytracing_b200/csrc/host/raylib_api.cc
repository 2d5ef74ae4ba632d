// raylib_api.cc -- the exported C ABI: the reference's 33 entry points (raylib/raylib.cc:25-331)
// with the same handle conventions (handles are raw object pointers, Destroy* returns 1 only for
// handles this library created), plus the RaylibB200_* additions of include/raylib_b200.h.
#include "raylib.h"
#include "raylib_b200.h"
#include "gpu_state.h"
#include "loader/obj_loader.h"
#include "host_internal.h"
#include "flatten.h"
#include "geom/scene.h"
#include "geom/primitives.h"
#include "render/camera.h"
#include "render/image.h"
#include "render/renderer.h"

#include <algorithm>
#include <cstring>
#include <iostream>
#include <map>
#include <string>
#include <mutex>
#include <vector>

namespace
{
	// Registry of library-created objects; guards Destroy* against foreign or stale handles.
	template<typename T>
	class HandleTable
	{
	public:
		void Add(T* object) { std::lock_guard<std::mutex> lock(mutex); items.push_back(object); }
		bool Remove(T* object)
		{
			std::lock_guard<std::mutex> lock(mutex);
			auto it = std::find(items.begin(), items.end(), object);
			if (it == items.end()) return false;
			items.erase(it);
			return true;
		}
		bool Contains(const T* object)
		{
			std::lock_guard<std::mutex> lock(mutex);
			return std::find(items.begin(), items.end(), object) != items.end();
		}
	private:
		std::mutex mutex;
		std::vector<T*> items;
	};


	HandleTable<OBJModel> g_objModels;
	HandleTable<Camera> g_cameras;
	HandleTable<Image2D> g_images;
	HandleTable<Scene> g_scenes;
}

bool RtIsLibraryImage(const Image2D* image) { return image && g_images.Contains(image); }

extern "C" {

// ---- lifetime -----------------------------------------------------------------------------------

int32_t Raylib_Initialize()
{
	std::cout << "Initialize raylib (B200 build, " << RtGpu::DeviceCount() << " CUDA device(s) visible)" << std::endl;
	Logger::StartLogThread();
	return 1;
}

int32_t Raylib_Terminate()
{
	std::cout << "Terminate raylib" << std::endl;
	RtGpu::ReleaseAll();
	Logger::KillAndWaitForLogThread();
	return 0;      // the reference returns 0 here as well (raylib.cc:43-51)
}

// ---- media ----------------------------------------------------------------------------------------

// raylib.cc:61-73: a failed load returns NULL and registers nothing
OBJModelHandle Raylib_LoadOBJModel(const char* objPath)
{
	OBJModel* model = new OBJModel;
	bool loaded = false;
	try { loaded = OBJLoader::LoadModelFromFile(objPath, model); }
	catch (const std::exception& e) { RtGpu::SetLastError(std::string("Raylib_LoadOBJModel: ") + e.what()); }
	if (!loaded)
	{
		delete model;
		return 0;
	}
	g_objModels.Add(model);
	return (OBJModelHandle)model;
}

void Raylib_TransformOBJModel(OBJModelHandle objModel,
	float translationX, float translationY, float translationZ,
	float yaw, float pitch, float roll, float scaleX, float scaleY, float scaleZ)
{
	OBJModel* model = (OBJModel*)objModel;
	if (!model) return;
	Transform transform;
	transform.Init(vec3(translationX, translationY, translationZ), Rotator(yaw, pitch, roll), vec3(scaleX, scaleY, scaleZ));
	for (StaticMesh* mesh : model->staticMeshes) mesh->ApplyTransform(transform);
}

void Raylib_FinalizeOBJModel(OBJModelHandle objModel)
{
	OBJModel* model = (OBJModel*)objModel;
	if (!model) return;
	model->FinalizeAllMeshes();
}

int32_t Raylib_UnloadOBJModel(OBJModelHandle objHandle)
{
	OBJModel* model = (OBJModel*)objHandle;
	if (!g_objModels.Remove(model)) return 0;
	delete model;
	return 1;
}

ImageHandle Raylib_LoadImage(const char* filepath)
{
	Image2D* image = nullptr;
	// nothing may unwind through the C boundary: a damaged file that asks for more memory than there is comes back as NULL
	try { image = ImageIO::LoadImage2DFromFile(filepath); }
	catch (const std::exception& e) { RtGpu::SetLastError(std::string("Raylib_LoadImage: ") + e.what()); image = nullptr; }
	if (image) g_images.Add(image);
	return (ImageHandle)image;
}

// ---- scene ----------------------------------------------------------------------------------------

SceneHandle Raylib_CreateScene()
{
	Scene* scene = new Scene;
	g_scenes.Add(scene);
	return (SceneHandle)scene;
}

void Raylib_AddSceneElement(SceneHandle scene, SceneElementHandle element)
{
	if (!scene || !element) return;
	((Scene*)scene)->AddSceneElement((Hitable*)element);
}

void Raylib_AddOBJModelToScene(SceneHandle scene, OBJModelHandle objModel)
{
	if (!scene || !objModel) return;
	((Scene*)scene)->AddSceneElement(((OBJModel*)objModel)->rootObject);
}

void Raylib_SetSkyPanorama(SceneHandle scene, ImageHandle skyImage) { if (scene) ((Scene*)scene)->SetSkyPanorama(skyImage); }
void Raylib_SetSunIlluminance(SceneHandle scene, float r, float g, float b) { if (scene) ((Scene*)scene)->SetSunIlluminance(vec3(r, g, b)); }
void Raylib_SetSunDirection(SceneHandle scene, float x, float y, float z) { if (scene) ((Scene*)scene)->SetSunDirection(vec3(x, y, z)); }

void Raylib_FinalizeScene(SceneHandle scene)
{
	if (!scene) return;
	((Scene*)scene)->Finalize();
	// The GPU copy is created on first use (sky/sun may still be set after Finalize in client code,
	// src/main.cc:438-442 sets them before; either order works here).
}

int32_t Raylib_DestroyScene(SceneHandle sceneHandle)
{
	Scene* scene = (Scene*)sceneHandle;
	if (!g_scenes.Remove(scene)) return 0;
	RaylibB200_ReleaseInspection(sceneHandle);   // handles are addresses and get reused
	delete scene;                                // ~Scene drops the GPU copy (RtForgetScene)
	return 1;
}

// ---- camera ---------------------------------------------------------------------------------------

CameraHandle Raylib_CreateCamera()
{
	Camera* camera = new Camera;
	g_cameras.Add(camera);
	return (CameraHandle)camera;
}

void Raylib_CameraSetPosition(CameraHandle handle, float x, float y, float z)
{
	Camera* camera = (Camera*)handle; if (!camera) return;
	camera->origin = vec3(x, y, z);
	camera->UpdateInternal();
}

void Raylib_CameraSetLookAt(CameraHandle handle, float tx, float ty, float tz)
{
	Camera* camera = (Camera*)handle; if (!camera) return;
	camera->lookAt = vec3(tx, ty, tz);
	camera->UpdateInternal();
}

void Raylib_CameraSetPerspective(CameraHandle handle, float fovY_degrees, float aspectWH)
{
	Camera* camera = (Camera*)handle; if (!camera) return;
	camera->fovY_degrees = fovY_degrees;
	camera->aspectWH = aspectWH;
	camera->UpdateInternal();
}

void Raylib_CameraSetLens(CameraHandle handle, float aperture, float focalDistance)
{
	Camera* camera = (Camera*)handle; if (!camera) return;
	camera->aperture = aperture;
	camera->focalDistance = focalDistance;
	camera->UpdateInternal();
}

void Raylib_CameraSetMotion(CameraHandle handle, float beginTime, float endTime)
{
	Camera* camera = (Camera*)handle; if (!camera) return;
	camera->beginTime = beginTime;
	camera->endTime = endTime;
	camera->UpdateInternal();
}

void Raylib_CameraCopy(CameraHandle srcCamera, CameraHandle dstCamera)
{
	if (!srcCamera || !dstCamera) return;
	*(Camera*)dstCamera = *(Camera*)srcCamera;
}

int32_t Raylib_DestroyCamera(CameraHandle handle)
{
	Camera* camera = (Camera*)handle;
	if (!g_cameras.Remove(camera)) return 0;
	delete camera;
	return 1;
}

// ---- images ---------------------------------------------------------------------------------------

ImageHandle Raylib_CreateImage(uint32_t width, uint32_t height)
{
	Image2D* image = new Image2D(width, height, 0x0);
	g_images.Add(image);
	return (ImageHandle)image;
}

void Raylib_DumpImageData(ImageHandle imageHandle, float* outDest)
{
	if (!imageHandle || !outDest) return;
	((Image2D*)imageHandle)->DumpFloatRGBs(outDest);
}

int32_t Raylib_DestroyImage(ImageHandle imageHandle)
{
	Image2D* image = (Image2D*)imageHandle;
	if (!g_images.Remove(image)) return 0;
	RtGpu::ForgetHostImage(image);      // its storage may be page-locked for read-backs
	delete image;
	return 1;
}

// ---- rendering ------------------------------------------------------------------------------------

void Raylib_Render(const RendererSettings* settings, SceneHandle scene, CameraHandle camera, ImageHandle outMainImage)
{
	Renderer renderer;
	renderer.RenderScene(settings, (Scene*)scene, (Camera*)camera, (Image2D*)outMainImage);
}

int32_t Raylib_Denoise(ImageHandle inMainImage, int32_t bMainImageHDR,
	ImageHandle inAlbedoImage, ImageHandle inNormalImage, ImageHandle outDenoisedImage)
{
	if (!inMainImage || !outDenoisedImage) return 0;
	Renderer renderer;
	return renderer.DenoiseScene((Image2D*)inMainImage, bMainImageHDR != 0,
		(Image2D*)inAlbedoImage, (Image2D*)inNormalImage, (Image2D*)outDenoisedImage) ? 1 : 0;
}

void Raylib_PostProcess(ImageHandle image) { if (image) ((Image2D*)image)->PostProcess(); }

int32_t Raylib_IsDenoiserSupported() { return Renderer::IsDenoiserSupported() ? 1 : 0; }

// ---- utilities --------------------------------------------------------------------------------------

const char* Raylib_GetRenderModeString(uint32_t auxMode)
{
	static const char* const names[RAYLIB_RENDERMODE_MAX] = {
		"Default", "Albedo", "SurfaceNormal", "MicrosurfaceNormal", "Texcoord", "Emission", "Reflectance",
	};
	return auxMode < RAYLIB_RENDERMODE_MAX ? names[auxMode] : nullptr;
}

int32_t Raylib_WriteImageToDisk(ImageHandle imageHandle, const char* filepath, uint32_t fileTypeRaw)
{
	if (!imageHandle || !filepath || fileTypeRaw >= RAYLIB_IMAGEFILETYPE_MAX) return 0;
	return ImageIO::WriteImage2DToDisk((Image2D*)imageHandle, filepath, (EImageFileType)fileTypeRaw) ? 1 : 0;
}

void Raylib_FlushLogThread() { Logger::FlushLogThread(); }

// ---- B200 additions -----------------------------------------------------------------------------------

int32_t RaylibB200_DeviceCount(void) { return RtGpu::DeviceCount(); }
int32_t RaylibB200_SetDevice(int32_t device) { return RtGpu::SetDevice(device) ? 1 : 0; }
int32_t RaylibB200_GetDevice(void) { return RtGpu::CurrentDevice(); }
int32_t RaylibB200_SetDevices(int32_t count) { return RtGpu::SetDevices(count); }
int32_t RaylibB200_GetDeviceCountInUse(void) { return RtGpu::ActiveDeviceCount(); }
void RaylibB200_ReloadTuning(void) { RtGpu::ReloadTuning(); }
void RaylibB200_SetFrameSeed(uint64_t seed) { RtGpu::SetFrameSeed(seed); }
void RaylibB200_SetBvhBuildKey(uint64_t key) { RtSetBvhBuildKey(key); }
void RaylibB200_SetCollectStats(int32_t enable) { RtGpu::SetCollectStats(enable != 0); }
void RaylibB200_SetTimeStages(int32_t enable) { RtGpu::SetTimeStages(enable != 0); }
void RaylibB200_SetSamplesPerPass(uint32_t samples) { RtGpu::SetSamplesPerPass(samples); }
void RaylibB200_SetPipes(uint32_t pipes) { RtGpu::SetPipes(pipes); }
void RaylibB200_SetFusedPass(uint32_t mode) { RtGpu::SetFusedPass(mode); }
int32_t RaylibB200_GetLastStats(RaylibB200Stats* outStats) { return RtGpu::GetLastStats(outStats) ? 1 : 0; }
const char* RaylibB200_GetLastError(void) { return RtGpu::LastError(); }

uint64_t RaylibB200_SceneDeviceBytes(SceneHandle scene)
{
	const RtDeviceScene* ds = RtGpu::AcquireScene((const Scene*)scene);
	return ds ? rt_scene_device_bytes(ds) : 0;
}

int32_t RaylibB200_SceneCounts(SceneHandle scene, uint64_t* out8)
{
	return RtGpu::AcquireScene((const Scene*)scene, out8) ? 1 : 0;
}

// Host-only view of the flattened scene (no device needed): lets tools and the CPU-side tests
// inspect exactly what would be uploaded.
namespace
{
	std::mutex g_inspectMutex;
	std::map<SceneHandle, RtFlatScene*> g_inspect;
}

const RtSceneDesc* RaylibB200_FlattenForInspection(SceneHandle scene)
{
	std::lock_guard<std::mutex> lock(g_inspectMutex);
	if (auto pre = RtGpu::Prebuilt((const Scene*)scene)) return &pre->desc;       // loaded from disk: owned by the scene
	auto it = g_inspect.find(scene);
	if (it != g_inspect.end()) return &it->second->desc;
	RtFlatScene* flat = new RtFlatScene;
	std::string why;
	if (!RtFlattenScene((const Scene*)scene, *flat, why))
	{
		RtGpu::SetLastError("cannot flatten scene: " + why);
		delete flat;
		return nullptr;
	}
	g_inspect[scene] = flat;
	return &flat->desc;
}

void RaylibB200_ReleaseInspection(SceneHandle scene)
{
	std::lock_guard<std::mutex> lock(g_inspectMutex);
	auto it = g_inspect.find(scene);
	if (it != g_inspect.end()) { delete it->second; g_inspect.erase(it); }
}

// ---- flattened-scene cache (SURVEY 8f row 4) ------------------------------------------------------------
int32_t RaylibB200_SaveFlattenedScene(SceneHandle scene, const char* path)
{
	const RtSceneDesc* desc = RaylibB200_FlattenForInspection(scene);
	if (!desc) return 0;
	std::string why;
	bool ok;
	if (auto pre = RtGpu::Prebuilt((const Scene*)scene)) ok = RtSaveFlatScene(*pre, path, why);
	else
	{
		std::lock_guard<std::mutex> lock(g_inspectMutex);
		auto it = g_inspect.find(scene);
		ok = it != g_inspect.end() && RtSaveFlatScene(*it->second, path, why);
	}
	if (!ok) RtGpu::SetLastError("RaylibB200_SaveFlattenedScene: " + (why.empty() ? std::string("scene not flattened") : why));
	return ok ? 1 : 0;
}

SceneHandle RaylibB200_LoadFlattenedScene(const char* path)
{
	auto flat = std::make_shared<RtFlatScene>();
	std::string why;
	if (!RtLoadFlatScene(path, *flat, why))
	{
		RtGpu::SetLastError("RaylibB200_LoadFlattenedScene: " + why);
		return (SceneHandle)0;
	}
	Scene* scene = new Scene;             // no object graph behind it: rendering uses the arrays read from disk
	g_scenes.Add(scene);
	RtGpu::AdoptPrebuilt(scene, flat);
	return (SceneHandle)scene;
}

RaylibB200Accumulator* RaylibB200_AccumulatorCreate(uint32_t width, uint32_t height) { return RtGpu::AccumulatorCreate(width, height); }
void RaylibB200_AccumulatorDestroy(RaylibB200Accumulator* acc) { RtGpu::AccumulatorDestroy(acc); }
int32_t RaylibB200_AccumulatorReset(RaylibB200Accumulator* acc) { return RtGpu::AccumulatorReset(acc) ? 1 : 0; }
uint32_t RaylibB200_AccumulatorSamples(const RaylibB200Accumulator* acc) { return RtGpu::AccumulatorSamples(acc); }
int32_t RaylibB200_RenderAccumulate(const RendererSettings* settings, SceneHandle scene, CameraHandle camera, RaylibB200Accumulator* acc, uint32_t samples)
{
	return RtGpu::RenderAccumulate(settings, (const Scene*)scene, (const Camera*)camera, acc, samples) ? 1 : 0;
}
int32_t RaylibB200_AccumulatorResolve(RaylibB200Accumulator* acc, ImageHandle outImage)
{
	if (!outImage) { RtGpu::SetLastError("RaylibB200_AccumulatorResolve: null image"); return 0; }
	return RtGpu::AccumulatorResolve(acc, (Image2D*)outImage, nullptr, nullptr) ? 1 : 0;
}
int32_t RaylibB200_AccumulatorResolveDevice(RaylibB200Accumulator* acc, void* deviceImageOut, void* cudaStream)
{
	if (!deviceImageOut) { RtGpu::SetLastError("RaylibB200_AccumulatorResolveDevice: null image"); return 0; }
	return RtGpu::AccumulatorResolve(acc, nullptr, deviceImageOut, cudaStream) ? 1 : 0;
}
int32_t RaylibB200_AccumulatorDenoise(RaylibB200Accumulator* acc, ImageHandle albedoImage, ImageHandle normalImage, ImageHandle outImage)
{
	return RtGpu::AccumulatorDenoise(acc, (const Image2D*)albedoImage, (const Image2D*)normalImage, (Image2D*)outImage) ? 1 : 0;
}
int32_t RaylibB200_AccumulatorRead(RaylibB200Accumulator* acc, float* outRgba) { return RtGpu::AccumulatorRead(acc, outRgba) ? 1 : 0; }
int32_t RaylibB200_AccumulatorNoise(RaylibB200Accumulator* acc, float* perPixel, double* mean) { return RtGpu::AccumulatorNoise(acc, perPixel, mean) ? 1 : 0; }
int32_t RaylibB200_AccumulatorSave(const RaylibB200Accumulator* acc, const char* path) { return RtGpu::AccumulatorSave(acc, path) ? 1 : 0; }
RaylibB200Accumulator* RaylibB200_AccumulatorLoad(const char* path) { return RtGpu::AccumulatorLoad(path); }

int32_t RaylibB200_CameraBlock(CameraHandle camera, RtCamera* out)
{
	if (!camera || !out) return 0;
	RtFlattenCamera((const Camera*)camera, *out);
	return 1;
}

uint64_t RaylibB200_ShardPixelCapacity(uint32_t width, uint32_t height, uint32_t shardCount)
{
	return (uint64_t)rt_shard_tile_capacity(width, height, shardCount) * RT_TILE_PIXELS;
}

// Host mirror of the device's slot -> pixel mapping (csrc/device/rt_device.cu: slot_to_pixel): tiles of
// RT_TILE_W x RT_TILE_H pixels are dealt round-robin to the shards, and inside a tile pixels are stored as
// eight 8x4 sub-blocks so that one warp covers a compact screen patch.
static inline bool ShardSlotToPixel(uint32_t width, uint32_t height, uint32_t shardRank, uint32_t shardCount,
	uint64_t slot, uint32_t& x, uint32_t& y)
{
	const uint32_t tilesX = (width + RT_TILE_W - 1) / RT_TILE_W, tilesY = (height + RT_TILE_H - 1) / RT_TILE_H;
	const uint64_t localTile = slot / RT_TILE_PIXELS;
	const uint32_t within = (uint32_t)(slot % RT_TILE_PIXELS);
	const uint64_t tile = localTile * shardCount + shardRank;
	if (tile >= (uint64_t)tilesX * tilesY) return false;
	const uint32_t tx = (uint32_t)(tile % tilesX), ty = (uint32_t)(tile / tilesX);
	const uint32_t sub = within >> 5, lane = within & 31u;
	x = tx * RT_TILE_W + (sub & 1u) * 8u + (lane & 7u);
	y = ty * RT_TILE_H + (sub >> 1) * 4u + (lane >> 3);
	return x < width && y < height;
}

int32_t RaylibB200_ShardPixelMap(uint32_t width, uint32_t height, uint32_t shardRank, uint32_t shardCount, int64_t* outPixelIndex)
{
	if (!outPixelIndex || shardCount == 0 || shardRank >= shardCount) return 0;
	const uint64_t cap = RaylibB200_ShardPixelCapacity(width, height, shardCount);
	for (uint64_t slot = 0; slot < cap; ++slot)
	{
		uint32_t x, y;
		outPixelIndex[slot] = ShardSlotToPixel(width, height, shardRank, shardCount, slot, x, y) ? (int64_t)y * width + x : -1;
	}
	return 1;
}

int32_t RaylibB200_AssembleShardsHost(const float* hostShards, uint32_t shardCount, uint32_t width, uint32_t height, float* hostImageOut)
{
	if (!hostShards || !hostImageOut || shardCount == 0) return 0;
	const uint64_t cap = RaylibB200_ShardPixelCapacity(width, height, shardCount);
	for (uint32_t r = 0; r < shardCount; ++r)
		for (uint64_t slot = 0; slot < cap; ++slot)
		{
			uint32_t x, y;
			if (!ShardSlotToPixel(width, height, r, shardCount, slot, x, y)) continue;
			memcpy(hostImageOut + 4 * ((uint64_t)y * width + x), hostShards + 4 * ((uint64_t)r * cap + slot), 16);
		}
	return 1;
}

int32_t RaylibB200_RenderShard(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	uint32_t shardRank, uint32_t shardCount, void* deviceShardOut, void* cudaStream)
{
	if (!deviceShardOut || shardCount == 0 || shardRank >= shardCount) { RtGpu::SetLastError("RaylibB200_RenderShard: bad shard arguments"); return 0; }
	return RtGpu::Render(settings, (const Scene*)scene, (const Camera*)camera, nullptr, nullptr, deviceShardOut,
		shardRank, shardCount, 0, cudaStream) ? 1 : 0;
}

// ---- shared frame: every rank renders its tiles straight into one row-major image (no shard buffers, no gather) ----
int32_t RaylibB200_RenderShardToFrame(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	uint32_t shardRank, uint32_t shardCount, void* deviceFrame, void* cudaStream)
{
	if (!deviceFrame || shardCount == 0 || shardRank >= shardCount) { RtGpu::SetLastError("RaylibB200_RenderShardToFrame: bad shard arguments"); return 0; }
	return RtGpu::Render(settings, (const Scene*)scene, (const Camera*)camera, nullptr, deviceFrame, nullptr,
		shardRank, shardCount, 0, cudaStream) ? 1 : 0;
}

void* RaylibB200_FrameCreate(uint32_t width, uint32_t height, unsigned char* outIpcHandle64)
{
	void* frame = nullptr;
	const int device = RtGpu::CurrentDevice();
	if (width == 0 || height == 0) { RtGpu::SetLastError("RaylibB200_FrameCreate: empty frame"); return nullptr; }
	if (rt_device_alloc(device, (uint64_t)width * height * 16ull, &frame) != 0)
	{
		RtGpu::SetLastError(std::string("RaylibB200_FrameCreate: ") + rt_last_error());
		return nullptr;
	}
	if (outIpcHandle64 && rt_ipc_export(device, frame, outIpcHandle64) != 0)
	{
		RtGpu::SetLastError(std::string("RaylibB200_FrameCreate: cannot export the frame: ") + rt_last_error());
		rt_device_free(device, frame);
		return nullptr;
	}
	return frame;
}

void RaylibB200_FrameDestroy(void* deviceFrame)
{
	if (deviceFrame) rt_device_free(RtGpu::CurrentDevice(), deviceFrame);
}

void* RaylibB200_FrameOpen(const unsigned char* ipcHandle64)
{
	void* frame = nullptr;
	if (!ipcHandle64) { RtGpu::SetLastError("RaylibB200_FrameOpen: null handle"); return nullptr; }
	if (rt_ipc_open(RtGpu::CurrentDevice(), ipcHandle64, &frame) != 0)
	{
		RtGpu::SetLastError(std::string("RaylibB200_FrameOpen: ") + rt_last_error());
		return nullptr;
	}
	return frame;
}

int32_t RaylibB200_FrameClose(void* mappedFrame)
{
	if (!mappedFrame) return 0;
	if (rt_ipc_close(RtGpu::CurrentDevice(), mappedFrame) != 0)
	{
		RtGpu::SetLastError(std::string("RaylibB200_FrameClose: ") + rt_last_error());
		return 0;
	}
	return 1;
}

int32_t RaylibB200_FrameRead(const void* deviceFrame, uint32_t width, uint32_t height, float* hostRgbaOut, void* cudaStream)
{
	if (!deviceFrame || !hostRgbaOut) { RtGpu::SetLastError("RaylibB200_FrameRead: null argument"); return 0; }
	if (rt_copy_to_host(RtGpu::CurrentDevice(), hostRgbaOut, deviceFrame, (uint64_t)width * height * 16ull, cudaStream) != 0)
	{
		RtGpu::SetLastError(std::string("RaylibB200_FrameRead: ") + rt_last_error());
		return 0;
	}
	return 1;
}

int32_t RaylibB200_AssembleShards(const void* deviceShards, uint32_t shardCount, uint32_t width, uint32_t height,
	void* deviceImageOut, void* cudaStream)
{
	if (!deviceShards || !deviceImageOut || shardCount == 0) { RtGpu::SetLastError("RaylibB200_AssembleShards: bad arguments"); return 0; }
	const int device = RtGpu::CurrentDevice();
	if (rt_assemble(device, deviceShards, shardCount, width, height, deviceImageOut, cudaStream) != 0 || rt_stream_sync(device, cudaStream) != 0)
	{
		RtGpu::SetLastError(std::string("rt_assemble: ") + rt_last_error());
		return 0;
	}
	return 1;
}

int32_t RaylibB200_RenderToDevice(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	void* deviceImageOut, void* cudaStream)
{
	if (!deviceImageOut) { RtGpu::SetLastError("RaylibB200_RenderToDevice: null output"); return 0; }
	return RtGpu::Render(settings, (const Scene*)scene, (const Camera*)camera, nullptr, deviceImageOut, nullptr, 0, 1, 0, cudaStream) ? 1 : 0;
}

int32_t RaylibB200_RenderAux(const RendererSettings* settings, SceneHandle scene, CameraHandle camera,
	ImageHandle outAlbedoImage, ImageHandle outNormalImage)
{
	return RtGpu::RenderAux(settings, (const Scene*)scene, (const Camera*)camera, (Image2D*)outAlbedoImage, (Image2D*)outNormalImage) ? 1 : 0;
}

int32_t RaylibB200_PostProcessDevice(void* deviceImage, uint32_t width, uint32_t height, void* deviceOutArgb8, float* outMaxWhite, void* cudaStream)
{
	if (!deviceImage) { RtGpu::SetLastError("RaylibB200_PostProcessDevice: null image"); return 0; }
	return RtGpu::PostProcessDevice(deviceImage, width, height, deviceOutArgb8, outMaxWhite, cudaStream) ? 1 : 0;
}

int32_t RaylibB200_ImageSetRGBA(ImageHandle imageHandle, uint32_t width, uint32_t height, const float* rgba)
{
	Image2D* image = (Image2D*)imageHandle;
	if (!image || !rgba) return 0;
	if (image->GetWidth() != width || image->GetHeight() != height) image->Reallocate(width, height);
	memcpy((void*)image->MutablePixels(), rgba, (size_t)width * height * sizeof(Pixel));      // Pixel is four packed floats
	return 1;
}

int32_t RaylibB200_ImageGetRGBA(ImageHandle imageHandle, float* outRgba)
{
	Image2D* image = (Image2D*)imageHandle;
	if (!image || !outRgba) return 0;
	memcpy(outRgba, image->MutablePixels(), (size_t)image->GetWidth() * image->GetHeight() * sizeof(Pixel));
	return 1;
}

int32_t RaylibB200_LibmEval(int32_t fn, const float* x, const float* y, float* out, uint64_t count)
{
	if (!x || !out || fn < 0 || fn > 9) { RtGpu::SetLastError("RaylibB200_LibmEval: bad arguments"); return 0; }
	if (RtGpu::DeviceCount() <= 0) { RtGpu::SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)"); return 0; }
	if (rt_libm_eval(RtGpu::CurrentDevice(), fn, x, y, out, count) != 0) { RtGpu::SetLastError(std::string("rt_libm_eval: ") + rt_last_error()); return 0; }
	return 1;
}

int32_t RaylibB200_PostProcessGPU(ImageHandle image) { return RtGpu::PostProcessHostImage((Image2D*)image) ? 1 : 0; }

int32_t RaylibB200_Denoise(ImageHandle mainImage, ImageHandle albedoImage, ImageHandle normalImage, ImageHandle outImage)
{
	return RtGpu::Denoise((const Image2D*)mainImage, (const Image2D*)albedoImage, (const Image2D*)normalImage, (Image2D*)outImage) ? 1 : 0;
}

int32_t RaylibB200_DenoiseDevice(const void* color, const void* albedo, const void* normal, uint32_t width, uint32_t height, void* out, void* cudaStream)
{
	return RtGpu::DenoiseDevice(color, albedo, normal, width, height, out, cudaStream) ? 1 : 0;
}

int32_t RaylibB200_TraceRays(SceneHandle scene, const float* rays, int64_t numRays, float tMin, int32_t* outRank, float* outT)
{
	const RtDeviceScene* ds = RtGpu::AcquireScene((const Scene*)scene);
	RtRenderContext* ctx = ds ? RtGpu::AcquireContext() : nullptr;
	if (!ds || !ctx) return 0;
	RtRenderStats rs;
	if (rt_trace_closest(ctx, ds, rays, numRays, tMin, outRank, outT, &rs) != 0)
	{
		RtGpu::SetLastError(std::string("rt_trace_closest: ") + rt_last_error());
		return 0;
	}
	RaylibB200Stats st;
	memset(&st, 0, sizeof(st));
	st.rayQueries = rs.rayQueries; st.boxTests = rs.boxTests; st.triTests = rs.triTests; st.sphereTests = rs.sphereTests;
	st.nodeVisits = rs.nodeVisits; st.deviceMs = rs.deviceMs; st.kernelLaunches = 1;
	st.gateTests = rs.gateTests; st.cubeTests = rs.cubeTests;
	st.refBoxTests = rs.refBoxTests; st.refTriTests = rs.refTriTests; st.refSphereTests = rs.refSphereTests; st.statRays = rs.statRays;
	RtGpu::SetLastStats(st);
	return 1;
}

int32_t RaylibB200_TraceRaysStaged(SceneHandle scene, int32_t mode, const float* rays, const uint32_t* order, int64_t numRays,
	float tMin, const float* sunDirection, uint32_t refillThreshold, uint32_t walkThreshold, uint32_t poolNodeThreshold,
	uint32_t poolRefill, uint32_t gridCtas, int32_t* outQueue, float* outHit, uint32_t* outQueueCounts)
{
	const RtStageSchedule schedule = { refillThreshold, walkThreshold, poolNodeThreshold, poolRefill, gridCtas };
	return RtGpu::TraceRaysStaged((const Scene*)scene, mode, rays, order, numRays, tMin, sunDirection, schedule, outQueue, outHit,
		outQueueCounts) ? 1 : 0;
}

int32_t RaylibB200_PrimaryHits(const RendererSettings* settings, SceneHandle scene, CameraHandle camera, int32_t* outRank, float* outT)
{
	if (!settings || !outRank || !outT) { RtGpu::SetLastError("RaylibB200_PrimaryHits: null argument"); return 0; }
	const size_t n = (size_t)settings->viewportWidth * settings->viewportHeight;
	Image2D scratch(settings->viewportWidth, settings->viewportHeight, 0x0);
	// internal render mode 100: pixel = (t, bit pattern of the leaf rank, bu, bv)
	if (!RtGpu::Render(settings, (const Scene*)scene, (const Camera*)camera, &scratch, nullptr, nullptr, 0, 1, 100u, nullptr)) return 0;
	const std::vector<Pixel>& px = scratch.GetPixelArray();
	for (size_t i = 0; i < n; ++i)
	{
		outT[i] = px[i].r;
		memcpy(&outRank[i], &px[i].g, 4);
	}
	return 1;
}

} // extern "C"
