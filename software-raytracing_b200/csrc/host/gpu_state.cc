// gpu_state.cc -- see gpu_state.h.  Also implements Renderer (reference: raylib/render/renderer.cc:273-356):
// where the reference builds 8x8 work cells, spins up a thread pool and polls it, this library hands the
// frame to the CUDA wavefront path tracer and copies the finished pixels back.
#include "gpu_state.h"
#include "flatten.h"
#include "host_internal.h"
#include "rt_checksum.h"
#include "rt_progressive.h"
#include "rt_denoise.h"
#include "geom/scene.h"
#include "render/camera.h"
#include "render/image.h"
#include "render/renderer.h"
#include "core/logger.h"
#include "core/assertion.h"
#include "rt_rng.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <condition_variable>
#include <functional>
#include <memory>
#include <thread>
#include <vector>

namespace
{
	struct SceneEntry
	{
		RtDeviceScene* device = nullptr;
		bool referenceTree = false;      // uploaded with the reference topology (statistics frames only)
		uint64_t counts[8] = { 0 };
		// distant lighting the upload was made with: the sky panorama lives in the uploaded texture arrays, so a scene whose
		// sky changed is flattened again; the sun is passed per frame (RtRenderParams.lightingOverride)
		ImageHandle skyHandle = 0;
		uint64_t skySignature = 0;
		uint64_t fingerprint = 0;        // rt_scene_fingerprint of this upload, computed when an accumulator first binds to it
		bool fingerprinted = false;
	};

	std::recursive_mutex g_mutex;
	std::vector<int> g_devices;      // devices a Raylib_Render frame is spread over; [0] is the primary (frame + device-only calls)
	bool g_devicesResolved = false;
	uint64_t g_frameSeed = RT_RNG_DEFAULT_FRAME_SEED;
	bool g_collectStats = false;
	bool g_timeStages = false;
	uint32_t g_samplesPerPass = 0;
	uint32_t g_pipes = 0;
	uint32_t g_fusedPass = 0;       // RaylibB200_SetFusedPass: 0 = the environment's / automatic
	RtTuning g_tuning;
	bool g_tuningLoaded = false;
	uint64_t g_multiDeviceMinSamples = 2ull << 20;   // frames with fewer pixel-samples stay on the primary device
	std::map<int, RtRenderContext*> g_contexts;                      // per device
	std::map<std::pair<const Scene*, int>, SceneEntry> g_scenes;     // (scene, device)
	std::map<const Scene*, std::shared_ptr<RtFlatScene>> g_prebuilt; // scenes that came from RaylibB200_LoadFlattenedScene
	struct Scratch { void* ptr = nullptr; uint64_t bytes = 0; };
	std::map<std::pair<int, int>, Scratch> g_scratch;                // (device, slot)
	std::map<std::pair<int, int>, bool> g_peerOk;                    // (device, peer) -> device can store into peer's memory
	std::map<const Image2D*, std::pair<void*, uint64_t>> g_pinnedImages;   // library-created images whose storage is page-locked

	// One persistent host thread per additional device: it keeps its CUDA thread state (a fresh thread pays ~10 ms for its
	// first runtime call on a device, every frame) and issues that device's launches while the caller's thread drives the
	// primary device.
	class DeviceWorker
	{
	public:
		DeviceWorker() : thread([this]() { Loop(); }) {}
		~DeviceWorker()
		{
			{ std::lock_guard<std::mutex> lock(mutex); quit = true; }
			wake.notify_all();
			thread.join();
		}
		void Submit(std::function<void()> job)
		{
			{ std::lock_guard<std::mutex> lock(mutex); task = std::move(job); busy = true; }
			wake.notify_all();
		}
		void Wait()
		{
			std::unique_lock<std::mutex> lock(mutex);
			done.wait(lock, [this]() { return !busy; });
		}
	private:
		void Loop()
		{
			for (;;)
			{
				std::function<void()> job;
				{
					std::unique_lock<std::mutex> lock(mutex);
					wake.wait(lock, [this]() { return quit || (busy && task); });
					if (quit) return;
					job = std::move(task);
					task = nullptr;
				}
				job();
				{ std::lock_guard<std::mutex> lock(mutex); busy = false; }
				done.notify_all();
			}
		}
		std::mutex mutex;
		std::condition_variable wake, done;
		std::function<void()> task;
		bool busy = false, quit = false;
		std::thread thread;
	};
	std::map<int, std::unique_ptr<DeviceWorker>> g_workers;         // per device

	thread_local std::string t_lastError;
	thread_local RaylibB200Stats t_lastStats;
	thread_local bool t_haveStats = false;

	const char* Env(const char* name) { const char* v = getenv(name); return (v && *v) ? v : nullptr; }

	// The knobs of DESIGN.md section 9, read from the environment once per process (and again on RaylibB200_ReloadTuning).
	void LoadTuning()
	{
		memset(&g_tuning, 0, sizeof(g_tuning));
		auto u32 = [](const char* name, uint32_t lo, uint32_t hi) -> uint32_t
		{
			const char* v = Env(name);
			return v ? (uint32_t)std::max<long>(lo, std::min<long>(hi, atol(v))) : 0u;
		};
		g_tuning.refillThreshold = u32("RAYLIB_B200_REFILL", 1, 32);
		g_tuning.walkThreshold = u32("RAYLIB_B200_WALK", 1, 32);
		g_tuning.traversalCtas = u32("RAYLIB_B200_TRAVERSAL_CTAS", 1, 16);
		g_tuning.pathsM = u32("RAYLIB_B200_PATHS_M", 1, 4096);
		g_tuning.binOriginBits = Env("RAYLIB_B200_BIN_OBITS") ? (int32_t)u32("RAYLIB_B200_BIN_OBITS", 0, 18) : -1;
		g_tuning.binDirBits = Env("RAYLIB_B200_BIN_DBITS") ? (int32_t)u32("RAYLIB_B200_BIN_DBITS", 0, 4) : -1;
		g_tuning.pipes = u32("RAYLIB_B200_PIPES", 1, 4);
		g_tuning.extendRing = u32("RAYLIB_B200_RING", 0, 1);
		g_tuning.dumpBounces = Env("RAYLIB_B200_DUMP_BOUNCES") ? 1u : 0u;
		g_tuning.dumpTimeline = Env("RAYLIB_B200_DUMP_TIMELINE") ? 1u : 0u;
		g_tuning.fusedPass = u32("RAYLIB_B200_FUSED", 0, 2);
		g_tuning.fusedPathsK = u32("RAYLIB_B200_FUSED_PATHS_K", 1, 1u << 20);
		g_tuning.pooledTraversal = u32("RAYLIB_B200_POOL", 0, 1);
		g_tuning.poolNodeThreshold = u32("RAYLIB_B200_POOL_NODE", 1, 32);
		g_tuning.poolRefill = u32("RAYLIB_B200_POOL_REFILL", 1, 64);
		g_tuning.poolCtas = u32("RAYLIB_B200_POOL_CTAS", 1, 16);
		if (const char* v = Env("RAYLIB_B200_MULTI_MIN_SAMPLES")) g_multiDeviceMinSamples = (uint64_t)std::max<long long>(0, atoll(v));
		g_tuningLoaded = true;
	}

	// Which devices a frame is spread over.  An explicit single device -- RaylibB200_SetDevice, $RAYLIB_B200_DEVICE, or
	// $LOCAL_RANK of a one-process-per-GPU launch -- pins the process to it; otherwise $RAYLIB_B200_DEVICES = all | k |
	// a,b,c; otherwise every visible device, like the reference's Raylib_Render uses every core (renderer.cc:286).
	void ResolveDevices()
	{
		if (g_devicesResolved) return;
		g_devicesResolved = true;
		g_devices.clear();
		const int n = rt_device_count();
		if (n <= 0) return;
		for (const char* name : { "RAYLIB_B200_DEVICE", "LOCAL_RANK" })
			if (const char* v = Env(name))
			{
				const int d = atoi(v);
				if (d < 0 || d >= n)
					fprintf(stderr, "raylib-b200: %s=%s names no CUDA device (%d visible); using device %d\n", name, v, n, ((d % n) + n) % n);
				g_devices.push_back(((d % n) + n) % n);
				return;
			}
		if (const char* v = Env("RAYLIB_B200_DEVICES"))
		{
			if (strchr(v, ','))
			{
				for (const char* c = v; *c;)
				{
					const int d = atoi(c);
					if (d >= 0 && d < n && std::find(g_devices.begin(), g_devices.end(), d) == g_devices.end()) g_devices.push_back(d);
					c = strchr(c, ',');
					if (!c) break;
					++c;
				}
			}
			else if (strcmp(v, "all") != 0)
			{
				const int k = std::max(1, std::min(n, atoi(v)));
				for (int d = 0; d < k; ++d) g_devices.push_back(d);
			}
		}
		if (g_devices.empty()) for (int d = 0; d < n; ++d) g_devices.push_back(d);
	}

	void* ScratchBuffer(int device, int slot, uint64_t bytes)
	{
		Scratch& s = g_scratch[{device, slot}];
		if (s.bytes >= bytes && s.ptr) return s.ptr;
		if (s.ptr) rt_device_free(device, s.ptr);
		s.ptr = nullptr; s.bytes = 0;
		if (rt_device_alloc(device, bytes, &s.ptr) != 0) return nullptr;
		s.bytes = bytes;
		return s.ptr;
	}

	// Cheap fingerprint of the sky panorama: the reference reads the image live on every miss (renderer.cc:170-180), so a
	// client may swap or repaint it between frames; the uploaded copy is refreshed when this changes.
	uint64_t SkySignature(ImageHandle sky)
	{
		const Image2D* img = (const Image2D*)sky;
		if (!img) return 0;
		const uint64_t w = img->GetWidth(), h = img->GetHeight(), n = w * h;
		uint64_t sig = 0x9E3779B97F4A7C15ull ^ (w << 32) ^ h;
		const std::vector<Pixel>& px = img->GetPixelArray();
		if (n == 0 || px.size() < n) return sig;
		const uint64_t step = std::max<uint64_t>(1, n / 4096);
		for (uint64_t i = 0; i < n; i += step)
		{
			uint32_t bits[4];
			memcpy(bits, &px[i], 16);
			for (uint32_t b : bits) { sig ^= b; sig *= 0x100000001B3ull; }
		}
		return sig;
	}

	RtRenderContext* ContextOn(int device)
	{
		auto it = g_contexts.find(device);
		if (it != g_contexts.end()) return it->second;
		RtRenderContext* ctx = nullptr;
		if (rt_context_create(device, &ctx) != 0) { RtGpu::SetLastError(std::string("rt_context_create: ") + rt_last_error()); return nullptr; }
		g_contexts[device] = ctx;
		return ctx;
	}

	bool PeerOk(int device, int peer)
	{
		if (device == peer) return true;
		auto it = g_peerOk.find({ device, peer });
		if (it != g_peerOk.end()) return it->second;
		const bool ok = rt_peer_enable(device, peer) == 0;
		g_peerOk[{ device, peer }] = ok;
		return ok;
	}

	// The scene's copy on `device`: flattened + uploaded the first time any device needs it, cloned device-to-device
	// (NVLink peer copy) for every further device -- the host flattens ONCE whatever the number of GPUs.
	const SceneEntry* SceneOn(const Scene* scene, int device)
	{
		auto key = std::make_pair(scene, device);
		auto it = g_scenes.find(key);
		const auto pre = g_prebuilt.find(scene);
		if (it != g_scenes.end() && pre == g_prebuilt.end())
		{
			// lighting that lives in the upload: a changed sky invalidates every device's copy
			const ImageHandle sky = scene->GetSkyPanorama();
			if (sky != it->second.skyHandle || SkySignature(sky) != it->second.skySignature)
			{
				const bool prebuiltScene = false;
				(void)prebuiltScene;
				for (auto e = g_scenes.begin(); e != g_scenes.end();)
				{
					if (e->first.first == scene) { rt_scene_free(e->second.device); e = g_scenes.erase(e); }
					else ++e;
				}
				it = g_scenes.end();
			}
		}
		// a statistics frame walks the reference topology, which plain uploads leave on the host: upload again with it
		if (it != g_scenes.end() && g_collectStats && !it->second.referenceTree)
		{
			for (auto e = g_scenes.begin(); e != g_scenes.end();)
			{
				if (e->first.first == scene) { rt_scene_free(e->second.device); e = g_scenes.erase(e); }
				else ++e;
			}
			it = g_scenes.end();
		}
		if (it != g_scenes.end()) return &it->second;

		// another device already holds it: clone over the fabric
		for (auto& kv : g_scenes)
		{
			if (kv.first.first != scene) continue;
			SceneEntry entry = kv.second;
			entry.device = nullptr;
			const auto t0 = std::chrono::steady_clock::now();
			PeerOk(device, kv.first.second);      // lets cudaMemcpyPeer go straight over NVLink; a staged copy works without it
			if (rt_scene_clone(kv.second.device, device, &entry.device) != 0)
			{
				RtGpu::SetLastError(std::string("rt_scene_clone: ") + rt_last_error());
				return nullptr;
			}
			LOG("[STAT] scene -> GPU %d: cloned from GPU %d in %.1f ms", device, kv.first.second,
				std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
			return &g_scenes.emplace(key, entry).first->second;
		}

		RtFlatScene fresh;
		std::string why;
		const auto t0 = std::chrono::steady_clock::now();
		if (pre == g_prebuilt.end() && !RtFlattenScene(scene, fresh, why)) { RtGpu::SetLastError("cannot flatten scene: " + why); return nullptr; }
		const RtFlatScene& flat = pre != g_prebuilt.end() ? *pre->second : fresh;
		const auto t1 = std::chrono::steady_clock::now();
		SceneEntry entry;
		entry.referenceTree = g_collectStats;
		if (rt_scene_upload(device, &flat.desc, entry.referenceTree ? RT_UPLOAD_REFERENCE_TREE : 0u, &entry.device) != 0)
		{
			RtGpu::SetLastError(std::string("rt_scene_upload: ") + rt_last_error());
			return nullptr;
		}
		const auto t2 = std::chrono::steady_clock::now();
		entry.counts[0] = flat.nodes.empty() ? flat.quantNodes.size() : flat.nodes.size(); entry.counts[1] = flat.triHot.size(); entry.counts[2] = flat.spheres.size();
		entry.counts[3] = flat.cubes.size(); entry.counts[4] = flat.materials.size(); entry.counts[5] = flat.textures.size();
		entry.counts[6] = flat.desc.maxStackDepth; entry.counts[7] = flat.desc.numLeaves;
		if (pre == g_prebuilt.end()) { entry.skyHandle = scene->GetSkyPanorama(); entry.skySignature = SkySignature(entry.skyHandle); }
		LOG("[STAT] scene -> GPU %d: %llu nodes, %llu triangles, %llu spheres, %.1f MB, flatten %.1f ms, upload %.1f ms",
			device, (unsigned long long)entry.counts[0], (unsigned long long)entry.counts[1], (unsigned long long)entry.counts[2],
			(double)flat.HostBytes() / 1.0e6,
			std::chrono::duration<double, std::milli>(t1 - t0).count(), std::chrono::duration<double, std::milli>(t2 - t1).count());
		return &g_scenes.emplace(key, entry).first->second;
	}

	void AddStats(RaylibB200Stats& st, const RtRenderStats& rs)
	{
		st.rayQueries += rs.rayQueries; st.pixelSamples += rs.pixelSamples;
		st.boxTests += rs.boxTests; st.triTests += rs.triTests; st.sphereTests += rs.sphereTests; st.nodeVisits += rs.nodeVisits;
		st.refBoxTests += rs.refBoxTests; st.refTriTests += rs.refTriTests; st.refSphereTests += rs.refSphereTests; st.statRays += rs.statRays;
		st.deviceMs = std::max(st.deviceMs, rs.deviceMs);      // the devices run side by side
		st.extendMs += rs.extendMs; st.extendLaunches += rs.extendLaunches;
		st.nodeIters += rs.nodeIters; st.nodeStep += rs.nodeStep; st.nodeAlive += rs.nodeAlive; st.leafIters += rs.leafIters; st.leafBusy += rs.leafBusy;
		st.gateTests += rs.gateTests; st.cubeTests += rs.cubeTests;
		st.kernelLaunches += rs.kernelLaunches;
		st.passes = std::max(st.passes, rs.passes);
	}
}

namespace RtGpu
{
	int DeviceCount() { return rt_device_count(); }

	int CurrentDevice()
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		ResolveDevices();
		return g_devices.empty() ? 0 : g_devices[0];
	}

	bool SetDevice(int device)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		if (device < 0 || device >= DeviceCount()) { SetLastError("RaylibB200_SetDevice: no such CUDA device"); return false; }
		g_devices.assign(1, device);
		g_devicesResolved = true;
		return true;
	}

	int SetDevices(int count)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		const int n = DeviceCount();
		if (n <= 0) { SetLastError("RaylibB200_SetDevices: no CUDA device is available"); return 0; }
		const int k = count <= 0 ? n : std::min(count, n);
		g_devices.clear();
		for (int d = 0; d < k; ++d) g_devices.push_back(d);
		g_devicesResolved = true;
		return k;
	}

	int ActiveDeviceCount()
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		ResolveDevices();
		return (int)g_devices.size();
	}

	void ReloadTuning() { std::lock_guard<std::recursive_mutex> lock(g_mutex); LoadTuning(); }
	const RtTuning& Tuning()
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		if (!g_tuningLoaded) LoadTuning();
		return g_tuning;
	}

	void SetFrameSeed(uint64_t seed) { g_frameSeed = seed; }
	uint64_t FrameSeed() { return g_frameSeed; }
	void SetCollectStats(bool enable) { g_collectStats = enable; }
	void SetTimeStages(bool enable) { g_timeStages = enable; }
	void SetSamplesPerPass(uint32_t samples) { g_samplesPerPass = samples; }
	void SetPipes(uint32_t pipes) { g_pipes = pipes; }
	void SetFusedPass(uint32_t mode) { g_fusedPass = std::min(mode, 2u); }

	void SetLastError(const std::string& message)
	{
		t_lastError = message;
		if (!message.empty()) fprintf(stderr, "raylib-b200: %s\n", message.c_str());
	}
	const char* LastError() { return t_lastError.c_str(); }
	void SetLastStats(const RaylibB200Stats& stats) { t_lastStats = stats; t_haveStats = true; }
	bool GetLastStats(RaylibB200Stats* out)
	{
		if (!t_haveStats || !out) return false;
		*out = t_lastStats;
		return true;
	}

	RtRenderContext* AcquireContext()
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		if (DeviceCount() <= 0)
		{
			SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)");
			return nullptr;
		}
		return ContextOn(CurrentDevice());
	}

	const RtDeviceScene* AcquireScene(const Scene* scene, uint64_t* outCounts8)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		if (!scene) { SetLastError("null scene handle"); return nullptr; }
		if (DeviceCount() <= 0)
		{
			SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)");
			return nullptr;
		}
		const SceneEntry* entry = SceneOn(scene, CurrentDevice());
		if (!entry) return nullptr;
		if (outCounts8) memcpy(outCounts8, entry->counts, sizeof(entry->counts));
		return entry->device;
	}

	void ForgetHostImage(const Image2D* image)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		auto it = g_pinnedImages.find(image);
		if (it == g_pinnedImages.end()) return;
		if (it->second.first) rt_host_unregister(it->second.first);
		g_pinnedImages.erase(it);
	}

	void ReleaseAll()
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		for (auto& kv : g_pinnedImages) if (kv.second.first) rt_host_unregister(kv.second.first);
		g_pinnedImages.clear();
		for (auto& kv : g_scenes) rt_scene_free(kv.second.device);
		g_scenes.clear();
		g_prebuilt.clear();
		for (auto& kv : g_scratch) rt_device_free(kv.first.first, kv.second.ptr);
		g_scratch.clear();
		g_workers.clear();      // joins the per-device threads
		for (auto& kv : g_contexts) rt_context_destroy(kv.second);
		g_contexts.clear();
		g_peerOk.clear();
	}

	// Page-locks the storage of a library-created Image2D once, so that the read-back of every later frame is one
	// full-speed DMA instead of a staged pageable copy (a third of the time of millisecond frames otherwise).
	static void PinHostImage(Image2D* image, uint64_t bytes)
	{
		void* ptr = image->MutablePixels();
		auto it = g_pinnedImages.find(image);
		if (it != g_pinnedImages.end())
		{
			if ((it->second.first == ptr || it->second.first == nullptr) && it->second.second == bytes) return;
			if (it->second.first) rt_host_unregister(it->second.first);
			g_pinnedImages.erase(it);
		}
		if (rt_host_register(ptr, bytes) == 0) g_pinnedImages[image] = { ptr, bytes };
		else
		{
			// remember the refusal (an entry with no registration) so that the attempt is not repeated on every frame
			g_pinnedImages[image] = { nullptr, bytes };
			fprintf(stderr, "raylib-b200: could not page-lock a %llu-byte image (%s); read-backs into it use pageable copies\n", (unsigned long long)bytes, rt_last_error());
		}
	}

	bool Render(const RendererSettings* settings, const Scene* scene, const Camera* camera,
	            Image2D* hostImage, void* deviceImage, void* deviceShard,
	            uint32_t shardRank, uint32_t shardCount, uint32_t renderModeOverride, void* stream, bool pinHostImage,
	            const SampleWindow* window)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		const auto wall0 = std::chrono::steady_clock::now();
		t_lastError.clear();
		if (!settings || !scene || !camera) { SetLastError("Raylib_Render: null settings/scene/camera"); return false; }
		if (settings->viewportWidth == 0 || settings->viewportHeight == 0) { SetLastError("Raylib_Render: empty viewport"); return false; }
		if (settings->renderMode >= RAYLIB_RENDERMODE_MAX && renderModeOverride == 0) { SetLastError("Raylib_Render: invalid renderMode"); return false; }
		if (DeviceCount() <= 0)
		{
			SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)");
			return false;
		}
		ResolveDevices();
		const int primary = CurrentDevice();

		RtCamera cam;
		RtFlattenCamera(camera, cam);

		RtRenderParams params;
		memset(&params, 0, sizeof(params));
		params.width = settings->viewportWidth;
		params.height = settings->viewportHeight;
		params.samplesPerPixel = settings->samplesPerPixel;
		params.maxPathLength = settings->maxPathLength;
		params.rayTMin = settings->rayTMin;
		params.renderMode = renderModeOverride ? renderModeOverride : settings->renderMode;
		params.frameSeed = g_frameSeed;
		params.samplesPerPass = g_samplesPerPass;
		params.pipes = g_pipes;
		params.collectStats = g_collectStats ? 1u : 0u;
		params.timeStages = g_timeStages ? 1u : 0u;
		params.tuning = Tuning();
		if (g_fusedPass) params.tuning.fusedPass = g_fusedPass;
		if (g_prebuilt.find(scene) == g_prebuilt.end())
		{
			// the sun as the Scene object holds it NOW (the reference reads it on every miss, renderer.cc:160-191)
			vec3 illuminance, direction;
			scene->GetSun(illuminance, direction);
			params.lightingOverride = 1;
			params.sunIlluminance[0] = illuminance.x; params.sunIlluminance[1] = illuminance.y; params.sunIlluminance[2] = illuminance.z;
			params.sunDirection[0] = direction.x; params.sunDirection[1] = direction.y; params.sunDirection[2] = direction.z;
		}

		// ---- which devices render this frame -------------------------------------------------------------
		// A whole frame (read back into a host image, or left in a row-major device image on the primary device) is spread over the
		// active devices by interleaved 16x16 tiles (SURVEY 8e); shards, debug views and statistics frames stay on the primary device.
		const uint64_t samples = window ? (uint64_t)(window->end - window->begin) : (uint64_t)std::max(1, params.samplesPerPixel);
		const uint64_t pixelSamples = (uint64_t)params.width * params.height * samples;
		std::vector<int> devices(1, primary);
		const bool wholeFrame = window || hostImage || (deviceImage && !deviceShard && shardCount <= 1);
		if (wholeFrame && params.renderMode == 0u && !g_collectStats && !g_timeStages && g_devices.size() > 1 &&
		    pixelSamples >= g_multiDeviceMinSamples)
			devices = g_devices;
		// the running sums of an installment live on the primary device: a device that cannot address them sits it out
		if (window && devices.size() > 1)
			for (size_t i = 1; i < devices.size(); ++i)
				if (!PeerOk(devices[i], primary)) { devices.assign(1, primary); break; }
		const uint32_t n = (uint32_t)devices.size();

		// hostImage: always the whole frame; deviceShard / deviceImage: the tiles of (shardRank, shardCount)
		if (hostImage) { shardRank = 0; shardCount = 1; }
		if (shardCount == 0) shardCount = 1;
		if (shardRank >= shardCount) { SetLastError("Raylib_Render: shardRank >= shardCount"); return false; }

		struct PerDevice
		{
			int device = 0;
			RtRenderContext* ctx = nullptr;
			const RtDeviceScene* scene = nullptr;
			void* shard = nullptr;         // tile-major shard buffer (gather fall-back only)
			RtRenderParams params;
			RtRenderStats stats;
			int rc = 0;
			std::string error;
		};
		std::vector<PerDevice> work(n);
		for (uint32_t i = 0; i < n; ++i)
		{
			PerDevice& w = work[i];
			w.device = devices[i];
			const SceneEntry* entry = SceneOn(scene, w.device);
			if (!entry) return false;
			w.scene = entry->device;
			w.ctx = ContextOn(w.device);
			if (!w.ctx) return false;
		}

		// Final pixels go straight into the row-major frame on the primary device -- its own kernels store locally, the
		// other devices store through peer mappings over NVLink: the last accumulate IS the gather -- unless the caller
		// asked for a tile-major shard buffer, or some device cannot address the primary's memory (then: shard buffers +
		// peer copies + one de-interleave pass on the primary).
		const uint64_t imageBytes = (uint64_t)params.width * params.height * 16ull;
		void* imageBuffer = nullptr;
		bool direct = true;
		for (uint32_t i = 1; i < n; ++i) direct = direct && PeerOk(work[i].device, primary);
		if (!deviceShard)
		{
			imageBuffer = window ? window->sums : deviceImage ? deviceImage : ScratchBuffer(primary, 1, imageBytes);
			if (!imageBuffer) { SetLastError(std::string("device allocation failed: ") + rt_last_error()); return false; }
		}
		const uint64_t shardBytes = (uint64_t)rt_shard_tile_capacity(params.width, params.height, n) * RT_TILE_PIXELS * 16ull;
		for (uint32_t i = 0; i < n; ++i)
		{
			PerDevice& w = work[i];
			w.params = params;
			w.params.shardRank = n > 1 ? i : shardRank;
			w.params.shardCount = n > 1 ? n : shardCount;
			if (deviceShard) w.shard = deviceShard;
			else if (direct) w.params.imageOut = imageBuffer;
			else
			{
				w.shard = ScratchBuffer(w.device, 0, shardBytes);
				if (!w.shard) { SetLastError(std::string("device allocation failed: ") + rt_last_error()); return false; }
			}
		}

		// one host thread per device issues that device's launches (about ten thousand per 4K frame) and waits for it;
		// they share nothing but the read-only camera block
		auto renderOn = [&cam, window](PerDevice& w, void* onStream)
		{
			w.rc = window ? rt_render_window(w.ctx, w.scene, &cam, &w.params, window->begin, window->end, window->sums, w.shard, onStream, &w.stats)
			              : rt_render_shard(w.ctx, w.scene, &cam, &w.params, w.shard, onStream, &w.stats);
			if (w.rc != 0) w.error = rt_last_error();
		};
		{
			std::vector<DeviceWorker*> helpers;
			for (uint32_t i = 1; i < n; ++i)
			{
				std::unique_ptr<DeviceWorker>& worker = g_workers[work[i].device];
				if (!worker) worker.reset(new DeviceWorker);
				PerDevice* w = &work[i];
				worker->Submit([renderOn, w]() { renderOn(*w, nullptr); });
				helpers.push_back(worker.get());
			}
			renderOn(work[0], n > 1 ? nullptr : stream);
			for (DeviceWorker* h : helpers) h->Wait();
		}
		for (const PerDevice& w : work)
			if (w.rc != 0) { SetLastError("rt_render_shard (GPU " + std::to_string(w.device) + "): " + w.error); return false; }

		if (n > 1 && !direct)
		{
			void* gathered = ScratchBuffer(primary, 3, shardBytes * n);
			if (!gathered) { SetLastError(std::string("device allocation failed: ") + rt_last_error()); return false; }
			for (uint32_t i = 0; i < n; ++i)
				if (rt_copy_peer(primary, (char*)gathered + shardBytes * i, work[i].device, work[i].shard, shardBytes) != 0)
				{
					SetLastError(std::string("peer copy of a shard failed: ") + rt_last_error());
					return false;
				}
			if (rt_assemble(primary, gathered, n, params.width, params.height, imageBuffer, nullptr) != 0 || rt_stream_sync(primary, nullptr) != 0)
			{
				SetLastError(std::string("rt_assemble: ") + rt_last_error());
				return false;
			}
		}

		uint64_t d2h = 0;
		if (hostImage)
		{
			if (pinHostImage) PinHostImage(hostImage, imageBytes);
			// Pixel is four packed floats, same as the device float4 image
			if (rt_copy_to_host(primary, hostImage->MutablePixels(), imageBuffer, imageBytes, n > 1 ? nullptr : stream) != 0)
			{
				SetLastError(std::string("device -> host copy failed: ") + rt_last_error());
				return false;
			}
			d2h = imageBytes;
		}

		RaylibB200Stats st;
		memset(&st, 0, sizeof(st));
		for (const PerDevice& w : work) AddStats(st, w.stats);
		st.totalMs = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
		st.h2dBytes = (sizeof(RtCamera) + sizeof(RtRenderParams)) * n;
		st.d2hBytes = d2h;
		st.device = (uint32_t)primary;
		st.devicesUsed = n;
		SetLastStats(st);
		return true;
	}
}

namespace RtGpu
{
	bool RenderAux(const RendererSettings* settings, const Scene* scene, const Camera* camera, Image2D* albedoImage, Image2D* normalImage)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		const auto wall0 = std::chrono::steady_clock::now();
		t_lastError.clear();
		if (!settings || !scene || !camera || !albedoImage || !normalImage) { SetLastError("RaylibB200_RenderAux: null argument"); return false; }
		if (settings->viewportWidth == 0 || settings->viewportHeight == 0) { SetLastError("RaylibB200_RenderAux: empty viewport"); return false; }
		const RtDeviceScene* deviceScene = AcquireScene(scene);
		if (!deviceScene) return false;
		RtRenderContext* ctx = AcquireContext();
		if (!ctx) return false;
		const int device = CurrentDevice();
		const uint32_t W = settings->viewportWidth, H = settings->viewportHeight;
		for (Image2D* img : { albedoImage, normalImage })
			if (img->GetWidth() != W || img->GetHeight() != H) img->Reallocate(W, H);

		RtCamera cam;
		RtFlattenCamera(camera, cam);
		const uint64_t shardBytes = (uint64_t)rt_shard_tile_capacity(W, H, 1) * RT_TILE_PIXELS * 16ull;
		const uint64_t imageBytes = (uint64_t)W * H * 16ull;
		void* shardA = ScratchBuffer(device, 0, shardBytes);
		void* shardB = ScratchBuffer(device, 2, shardBytes);
		void* image = ScratchBuffer(device, 1, imageBytes);
		if (!shardA || !shardB || !image) { SetLastError(std::string("device allocation failed: ") + rt_last_error()); return false; }

		RtRenderParams params;
		memset(&params, 0, sizeof(params));
		params.width = W; params.height = H;
		params.samplesPerPixel = 1; params.maxPathLength = settings->maxPathLength;
		params.rayTMin = settings->rayTMin;
		params.renderMode = RT_RENDERMODE_AUX;
		params.frameSeed = g_frameSeed;
		params.shardRank = 0; params.shardCount = 1;
		params.auxShardOut = shardB;
		RtRenderStats rs;
		if (rt_render_shard(ctx, deviceScene, &cam, &params, shardA, nullptr, &rs) != 0)
		{
			SetLastError(std::string("rt_render_shard: ") + rt_last_error());
			return false;
		}
		Image2D* targets[2] = { albedoImage, normalImage };
		void* shards[2] = { shardA, shardB };
		for (int i = 0; i < 2; ++i)
		{
			if (rt_assemble(device, shards[i], 1, W, H, image, nullptr) != 0 ||
			    rt_copy_to_host(device, targets[i]->MutablePixels(), image, imageBytes, nullptr) != 0)
			{
				SetLastError(std::string("aux readback failed: ") + rt_last_error());
				return false;
			}
		}
		RaylibB200Stats st;
		memset(&st, 0, sizeof(st));
		st.rayQueries = rs.rayQueries; st.pixelSamples = rs.pixelSamples; st.deviceMs = rs.deviceMs;
		st.totalMs = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
		st.h2dBytes = sizeof(RtCamera) + sizeof(RtRenderParams); st.d2hBytes = 2 * imageBytes;
		st.kernelLaunches = rs.kernelLaunches + 2; st.device = (uint32_t)device;
		SetLastStats(st);
		return true;
	}

	bool PostProcessDevice(void* deviceImage, uint32_t width, uint32_t height, void* deviceOutArgb8, float* outMaxWhite, void* stream)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		if (DeviceCount() <= 0) { SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)"); return false; }
		if (rt_postprocess(CurrentDevice(), deviceImage, width, height, (uint32_t*)deviceOutArgb8, outMaxWhite, stream) != 0)
		{
			SetLastError(std::string("rt_postprocess: ") + rt_last_error());
			return false;
		}
		return rt_stream_sync(CurrentDevice(), stream) == 0;
	}

	bool PostProcessHostImage(Image2D* hostImage)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		if (!hostImage || hostImage->GetWidth() == 0 || hostImage->GetHeight() == 0) { SetLastError("RaylibB200_PostProcessGPU: empty image"); return false; }
		if (DeviceCount() <= 0) { SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)"); return false; }
		const int device = CurrentDevice();
		const uint64_t bytes = (uint64_t)hostImage->GetWidth() * hostImage->GetHeight() * 16ull;
		void* image = ScratchBuffer(device, 1, bytes);
		if (!image) { SetLastError(std::string("device allocation failed: ") + rt_last_error()); return false; }
		float maxWhite = 1.0f;
		if (rt_copy_to_device(device, image, hostImage->MutablePixels(), bytes, nullptr) != 0 ||
		    rt_postprocess(device, image, hostImage->GetWidth(), hostImage->GetHeight(), nullptr, &maxWhite, nullptr) != 0 ||
		    rt_copy_to_host(device, hostImage->MutablePixels(), image, bytes, nullptr) != 0)
		{
			SetLastError(std::string("GPU post-process failed: ") + rt_last_error());
			return false;
		}
		LOG("Max white luminance: %f", maxWhite);
		return true;
	}
}

// ---------------------------------------------------------------------------------------------
// Denoising (DESIGN.md section 14): the filter of rt_denoise.h over device images, host images or an accumulator's sums

namespace
{
	const int kDenoiseScratchSlot = 5;      // the filter's records (rt_denoise_scratch_bytes)
	const int kDenoiseImageSlot = 6;        // device copies of a host call's images: colour, albedo, normal, output

	// "" or why a guide image cannot go with a W x H colour image
	std::string GuideSizeError(const Image2D* guide, const char* name, uint32_t width, uint32_t height, const char* against)
	{
		if (!guide || (guide->GetWidth() == width && guide->GetHeight() == height)) return "";
		return std::string("the ") + name + " image is " + std::to_string(guide->GetWidth()) + "x" + std::to_string(guide->GetHeight()) +
		       ", " + against + " is " + std::to_string(width) + "x" + std::to_string(height);
	}

	// Uploads the non-null host images of `images` into consecutive W x H float4 images of the slot buffer (which also
	// holds the output, returned in *out); NULL stays NULL.
	bool UploadDenoiseImages(const std::string& fn, int device, const Image2D* const images[3], uint64_t bytes, void* dev[3],
	                         void** out, RaylibB200Stats& st)
	{
		char* base = (char*)ScratchBuffer(device, kDenoiseImageSlot, 4 * bytes);
		if (!base) { RtGpu::SetLastError(fn + "device allocation failed: " + rt_last_error()); return false; }
		for (int k = 0; k < 3; ++k)
		{
			dev[k] = nullptr;
			if (!images[k]) continue;
			dev[k] = base + k * bytes;
			if (rt_copy_to_device(device, dev[k], images[k]->GetPixelArray().data(), bytes, nullptr) != 0)
			{
				RtGpu::SetLastError(fn + rt_last_error());
				return false;
			}
			st.h2dBytes += bytes;
		}
		*out = base + 3 * bytes;
		return true;
	}

	// rt_denoise (n == 0) or rt_denoise_sums on device images of `device`; fills the device part of the statistics
	bool RunDenoise(const std::string& fn, int device, const void* color, uint32_t n, const void* albedo, const void* normal,
	                uint32_t width, uint32_t height, void* out, void* stream, RaylibB200Stats& st)
	{
		void* scratch = ScratchBuffer(device, kDenoiseScratchSlot, rt_denoise_scratch_bytes(width, height));
		if (!scratch) { RtGpu::SetLastError(fn + "device allocation failed: " + rt_last_error()); return false; }
		const int rc = n ? rt_denoise_sums(device, color, n, albedo, normal, width, height, scratch, out, stream, &st.deviceMs)
		                 : rt_denoise(device, color, albedo, normal, width, height, scratch, out, stream, &st.deviceMs);
		if (rc != 0) { RtGpu::SetLastError(fn + rt_denoise_last_error()); return false; }
		st.kernelLaunches = RT_DENOISE_LAUNCHES;
		st.device = (uint32_t)device;
		st.devicesUsed = 1;
		return true;
	}

	// The result of a host call: read back into `out`, resized to W x H only now that the filter has run
	bool ReadDenoised(const std::string& fn, int device, const void* image, uint32_t width, uint32_t height, Image2D* out, RaylibB200Stats& st)
	{
		if (out->GetWidth() != width || out->GetHeight() != height) out->Reallocate(width, height);
		const uint64_t bytes = (uint64_t)width * height * 16ull;
		if (rt_copy_to_host(device, out->MutablePixels(), image, bytes, nullptr) != 0) { RtGpu::SetLastError(fn + rt_last_error()); return false; }
		st.d2hBytes += bytes;
		return true;
	}

	double MsSince(std::chrono::steady_clock::time_point t0)
	{
		return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
	}
}

namespace RtGpu
{
	bool Denoise(const Image2D* color, const Image2D* albedo, const Image2D* normal, Image2D* out)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		const auto wall0 = std::chrono::steady_clock::now();
		t_lastError.clear();
		const std::string fn = "RaylibB200_Denoise: ";
		if (!color || !out) { SetLastError(fn + "null main or output image"); return false; }
		const uint32_t W = color->GetWidth(), H = color->GetHeight();
		if (W == 0 || H == 0 || (uint64_t)W * H >= (1ull << 31)) { SetLastError(fn + "the main image must be non-empty and below 2^31 pixels"); return false; }
		for (const std::string& why : { GuideSizeError(albedo, "albedo", W, H, "the main image"), GuideSizeError(normal, "normal", W, H, "the main image") })
			if (!why.empty()) { SetLastError(fn + why); return false; }
		if (DeviceCount() <= 0) { SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)"); return false; }
		const int device = CurrentDevice();
		RaylibB200Stats st;
		memset(&st, 0, sizeof(st));
		const Image2D* images[3] = { color, albedo, normal };
		void* dev[3];
		void* image = nullptr;
		if (!UploadDenoiseImages(fn, device, images, (uint64_t)W * H * 16ull, dev, &image, st) ||
		    !RunDenoise(fn, device, dev[0], 0, dev[1], dev[2], W, H, image, nullptr, st) ||
		    !ReadDenoised(fn, device, image, W, H, out, st))
			return false;
		st.totalMs = MsSince(wall0);
		SetLastStats(st);
		return true;
	}

	bool DenoiseDevice(const void* color, const void* albedo, const void* normal, uint32_t width, uint32_t height, void* out, void* stream)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		const auto wall0 = std::chrono::steady_clock::now();
		t_lastError.clear();
		const std::string fn = "RaylibB200_DenoiseDevice: ";
		if (!color || !out) { SetLastError(fn + "null colour or output image"); return false; }
		if (width == 0 || height == 0 || (uint64_t)width * height >= (1ull << 31)) { SetLastError(fn + "the image must be non-empty and below 2^31 pixels"); return false; }
		// the kernels read and write whole float4 pixels: a misaligned view (a sliced tensor) is refused here, not faulted on
		for (const void* p : { color, albedo, normal, (const void*)out })
			if ((uintptr_t)p % 16u != 0) { SetLastError(fn + "device images must be 16-byte aligned (RGBA float4 pixels)"); return false; }
		if (DeviceCount() <= 0) { SetLastError("no CUDA device is available; this library renders on the GPU only (no CPU path)"); return false; }
		RaylibB200Stats st;
		memset(&st, 0, sizeof(st));
		if (!RunDenoise(fn, CurrentDevice(), color, 0, albedo, normal, width, height, out, stream, st)) return false;
		st.totalMs = MsSince(wall0);
		SetLastStats(st);
		return true;
	}
}

// ---------------------------------------------------------------------------------------------
// The traversal stage kernels on caller rays (RaylibB200_TraceRaysStaged, rt_trace_stage of rt_trace_stage.h)

namespace RtGpu
{
	bool TraceRaysStaged(const Scene* scene, int mode, const float* rays, const uint32_t* order, int64_t numRays, float tMin,
	                     const float* sunDirection, const RtStageSchedule& schedule, int32_t* outQueue, float* outHit,
	                     uint32_t* outQueueCounts)
	{
		const auto wall0 = std::chrono::steady_clock::now();
		t_lastError.clear();
		const std::string fn = "RaylibB200_TraceRaysStaged: ";
		if (!scene) { SetLastError(fn + "null scene"); return false; }
		if (!rays || !order || !outQueue || !outHit) { SetLastError(fn + "null ray, order or output buffer"); return false; }
		if (mode < RT_STAGE_EXTEND || mode > RT_STAGE_SHADOW) { SetLastError(fn + "unknown mode " + std::to_string(mode) + " (0..3)"); return false; }
		if (numRays <= 0 || numRays >= ((int64_t)1 << 31)) { SetLastError(fn + "the ray count must be in [1, 2^31)"); return false; }
		if (mode == RT_STAGE_SHADOW)
		{
			if (!sunDirection) { SetLastError(fn + "the any-hit mode needs a sun direction"); return false; }
			bool finite = true, zero = true;
			for (int i = 0; i < 3; ++i) { finite = finite && std::isfinite(sunDirection[i]); zero = zero && sunDirection[i] == 0.0f; }
			if (!finite || zero) { SetLastError(fn + "the sun direction must be finite and non-zero"); return false; }
		}
		if (schedule.refillThreshold > 32u || schedule.walkThreshold > 32u || schedule.poolNodeThreshold > 32u ||
		    schedule.poolRefill > 64u || schedule.gridCtas > 4096u)
		{
			SetLastError(fn + "scheduling out of range (refill, walk, pool node: 0..32; pool refill: 0..64; grid: 0..4096 CTAs)");
			return false;
		}
		{
			std::vector<uint8_t> seen((size_t)numRays, 0);
			for (int64_t i = 0; i < numRays; ++i)
			{
				if ((int64_t)order[i] >= numRays || seen[order[i]]) { SetLastError(fn + "the order is not a permutation of 0..numRays-1"); return false; }
				seen[order[i]] = 1;
			}
		}
		const RtDeviceScene* ds = AcquireScene(scene);
		RtRenderContext* ctx = ds ? AcquireContext() : nullptr;
		if (!ds || !ctx) return false;
		RtRenderStats rs;
		if (rt_trace_stage(ctx, ds, mode, rays, order, numRays, tMin, sunDirection, &schedule, outQueue, outHit, outQueueCounts, &rs) != 0)
		{
			SetLastError(fn + rt_last_error());
			return false;
		}
		RaylibB200Stats st;
		memset(&st, 0, sizeof(st));
		AddStats(st, rs);
		st.totalMs = MsSince(wall0);
		st.device = (uint32_t)CurrentDevice();
		st.devicesUsed = 1;
		st.h2dBytes = (uint64_t)numRays * 36u;                                   // rays + order
		st.d2hBytes = (uint64_t)numRays * (mode == RT_STAGE_SHADOW ? 16u : 36u);   // records or radiance (+ queues)
		SetLastStats(st);
		return true;
	}
}

namespace RtGpu
{
	void AdoptPrebuilt(const Scene* scene, std::shared_ptr<RtFlatScene> flat)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		g_prebuilt[scene] = std::move(flat);
	}
	std::shared_ptr<RtFlatScene> Prebuilt(const Scene* scene)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		auto it = g_prebuilt.find(scene);
		return it == g_prebuilt.end() ? nullptr : it->second;
	}
}

// ---------------------------------------------------------------------------------------------
// Progressive rendering: an accumulator is the running sum of a frame rendered in installments (DESIGN.md section 13)

// What decides the image of an accumulated frame; recorded by the first installment, compared by every later one, and
// stored in checkpoint files as is.
struct RtAccumBinding
{
	uint32_t width, height;
	int32_t  maxPathLength;
	float    rayTMin;
	uint64_t frameSeed;
	RtCamera camera;
	float    sunIlluminance[3], sunDirection[3];
	uint64_t sceneFingerprint;
};
static_assert(sizeof(RtAccumBinding) == 152, "the binding record has no padding (it is compared and stored bytewise)");

struct RaylibB200Accumulator
{
	int device = 0;
	uint32_t width = 0, height = 0;
	void* sums = nullptr;             // row-major W x H float4 {sum R, sum G, sum B, sum luminance^2}
	uint32_t samples = 0;             // n
	bool bound = false;
	RtAccumBinding binding;
};

namespace
{
	const uint32_t kMaxAccumSamples = 1u << 24;       // every count up to here is exact as the float divisor
	const char* kNoDevice = "no CUDA device is available; this library renders on the GPU only (no CPU path)";

	struct AccumFileHeader
	{
		char     magic[8];            // "RTACCUM1"
		uint32_t headerBytes;         // sizeof(AccumFileHeader)
		uint32_t bindingBytes;        // sizeof(RtAccumBinding)
		uint32_t width, height;
		uint32_t samples;             // n
		uint32_t bound;
		uint64_t checksum;            // RtChecksum of this header (checksum = 0), the binding and the sums
	};
	static_assert(sizeof(AccumFileHeader) == 40, "accumulator file header is 40 bytes");

	uint64_t AccumFileChecksum(const AccumFileHeader& h, const RtAccumBinding& b, const float* sums, uint64_t sumBytes)
	{
		AccumFileHeader zeroed = h;
		zeroed.checksum = 0;
		RtChecksum sum;
		sum.Add(&zeroed, sizeof(zeroed));
		sum.Add(&b, sizeof(b));
		sum.Add(sums, (size_t)sumBytes);
		return sum.h;
	}

	// the sun a frame of `scene` is rendered with: the Scene object's as it is now, or the stored one of a flattened-scene file
	void FrameSun(const Scene* scene, float illuminance[3], float direction[3])
	{
		const auto pre = g_prebuilt.find(scene);
		if (pre != g_prebuilt.end())
		{
			memcpy(illuminance, pre->second->desc.sunIlluminance, 12);
			memcpy(direction, pre->second->desc.sunDirection, 12);
			return;
		}
		vec3 i, d;
		scene->GetSun(i, d);
		illuminance[0] = i.x; illuminance[1] = i.y; illuminance[2] = i.z;
		direction[0] = d.x; direction[1] = d.y; direction[2] = d.z;
	}

	bool SceneFingerprint(const Scene* scene, int device, uint64_t* out)
	{
		if (!SceneOn(scene, device)) return false;
		SceneEntry& entry = g_scenes[{ scene, device }];
		if (!entry.fingerprinted)
		{
			if (rt_scene_fingerprint(entry.device, &entry.fingerprint) != 0)
			{
				RtGpu::SetLastError(std::string("rt_scene_fingerprint: ") + rt_last_error());
				return false;
			}
			entry.fingerprinted = true;
		}
		*out = entry.fingerprint;
		return true;
	}

	// every field in which two bindings differ ("" = none): an installment for another scene usually has another sun, too
	std::string BindingDifference(const RtAccumBinding& a, const RtAccumBinding& b)
	{
		std::string fields;
		auto differs = [&fields](bool different, const char* field) { if (different) fields += (fields.empty() ? "" : ", ") + std::string(field); };
		differs(a.width != b.width || a.height != b.height, "viewport");
		differs(a.maxPathLength != b.maxPathLength, "maxPathLength");
		differs(memcmp(&a.rayTMin, &b.rayTMin, 4) != 0, "rayTMin");
		differs(a.frameSeed != b.frameSeed, "frame seed");
		differs(memcmp(&a.camera, &b.camera, sizeof(a.camera)) != 0, "camera");
		differs(memcmp(a.sunIlluminance, b.sunIlluminance, 12) != 0 || memcmp(a.sunDirection, b.sunDirection, 12) != 0, "sun");
		differs(a.sceneFingerprint != b.sceneFingerprint, "scene");
		return fields;
	}

	RaylibB200Accumulator* NewAccumulator(uint32_t width, uint32_t height, const char* fn)
	{
		if (rt_device_count() <= 0) { RtGpu::SetLastError(kNoDevice); return nullptr; }
		ResolveDevices();
		std::unique_ptr<RaylibB200Accumulator> acc(new RaylibB200Accumulator);
		memset(&acc->binding, 0, sizeof(acc->binding));
		acc->device = g_devices[0];
		acc->width = width; acc->height = height;
		const uint64_t bytes = (uint64_t)width * height * 16ull;
		if (rt_device_alloc(acc->device, bytes, &acc->sums) != 0 || rt_device_zero(acc->device, acc->sums, bytes) != 0)
		{
			RtGpu::SetLastError(std::string(fn) + "device allocation failed: " + rt_last_error());
			if (acc->sums) rt_device_free(acc->device, acc->sums);
			return nullptr;
		}
		return acc.release();
	}
}

namespace RtGpu
{
	RaylibB200Accumulator* AccumulatorCreate(uint32_t width, uint32_t height)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		if (width == 0 || height == 0 || (uint64_t)width * height >= (1ull << 31))
		{
			SetLastError("RaylibB200_AccumulatorCreate: size must be non-empty and below 2^31 pixels");
			return nullptr;
		}
		return NewAccumulator(width, height, "RaylibB200_AccumulatorCreate: ");
	}

	void AccumulatorDestroy(RaylibB200Accumulator* acc)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		if (!acc) return;
		rt_device_free(acc->device, acc->sums);
		delete acc;
	}

	bool AccumulatorReset(RaylibB200Accumulator* acc)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		if (!acc) { SetLastError("RaylibB200_AccumulatorReset: null accumulator"); return false; }
		if (rt_device_zero(acc->device, acc->sums, (uint64_t)acc->width * acc->height * 16ull) != 0)
		{
			SetLastError(std::string("RaylibB200_AccumulatorReset: ") + rt_last_error());
			return false;
		}
		acc->samples = 0;
		acc->bound = false;
		memset(&acc->binding, 0, sizeof(acc->binding));
		return true;
	}

	uint32_t AccumulatorSamples(const RaylibB200Accumulator* acc) { return acc ? acc->samples : 0u; }

	bool RenderAccumulate(const RendererSettings* settings, const Scene* scene, const Camera* camera, RaylibB200Accumulator* acc, uint32_t samples)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		const std::string fn = "RaylibB200_RenderAccumulate: ";
		if (!settings || !scene || !camera || !acc) { SetLastError(fn + "null argument"); return false; }
		if (samples == 0) { SetLastError(fn + "an installment renders at least one sample"); return false; }
		if (settings->renderMode != 0u) { SetLastError(fn + "only renderMode 0 (path tracing) accumulates"); return false; }
		if ((uint64_t)acc->samples + samples > kMaxAccumSamples) { SetLastError(fn + "more than 2^24 samples per pixel"); return false; }
		if (DeviceCount() <= 0) { SetLastError(kNoDevice); return false; }
		ResolveDevices();
		const int primary = g_devices[0];
		if (primary != acc->device)
		{
			SetLastError(fn + "the accumulator lives on GPU " + std::to_string(acc->device) + ", the first active device is GPU " + std::to_string(primary));
			return false;
		}

		RtAccumBinding b;
		memset(&b, 0, sizeof(b));
		b.width = settings->viewportWidth; b.height = settings->viewportHeight;
		b.maxPathLength = settings->maxPathLength;
		b.rayTMin = settings->rayTMin;
		b.frameSeed = g_frameSeed;
		RtFlattenCamera(camera, b.camera);
		FrameSun(scene, b.sunIlluminance, b.sunDirection);
		if (b.width != acc->width || b.height != acc->height)
		{
			SetLastError(fn + "viewport " + std::to_string(b.width) + "x" + std::to_string(b.height) + " differs from the accumulator's " +
			             std::to_string(acc->width) + "x" + std::to_string(acc->height));
			return false;
		}
		if (!SceneFingerprint(scene, primary, &b.sceneFingerprint)) return false;
		if (acc->bound)
		{
			const std::string fields = BindingDifference(acc->binding, b);
			if (!fields.empty())
			{
				SetLastError(fn + "the accumulated image's " + fields + (fields.find(',') == std::string::npos ? " differs" : " differ") +
				             " from this installment's; Reset the accumulator to start a new image");
				return false;
			}
		}

		const SampleWindow window = { acc->samples, acc->samples + samples, acc->sums };
		if (!Render(settings, scene, camera, nullptr, nullptr, nullptr, 0, 1, 0, nullptr, false, &window)) return false;
		acc->binding = b;
		acc->bound = true;
		acc->samples += samples;
		return true;
	}

	bool AccumulatorResolve(RaylibB200Accumulator* acc, Image2D* hostImage, void* deviceImage, void* stream)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		const std::string fn = "RaylibB200_AccumulatorResolve: ";
		if (!acc || (!hostImage && !deviceImage)) { SetLastError(fn + "null argument"); return false; }
		if (acc->samples == 0) { SetLastError(fn + "the accumulator holds no samples"); return false; }
		const uint64_t count = (uint64_t)acc->width * acc->height, bytes = count * 16ull;
		if (deviceImage)
		{
			if (rt_resolve(acc->device, acc->sums, (uint32_t)count, acc->samples, deviceImage, nullptr, nullptr, stream) != 0)
			{
				SetLastError(fn + rt_last_error());
				return false;
			}
			return true;
		}
		if (hostImage->GetWidth() != acc->width || hostImage->GetHeight() != acc->height) hostImage->Reallocate(acc->width, acc->height);
		void* image = ScratchBuffer(acc->device, 1, bytes);
		if (!image) { SetLastError(fn + "device allocation failed: " + rt_last_error()); return false; }
		if (rt_resolve(acc->device, acc->sums, (uint32_t)count, acc->samples, image, nullptr, nullptr, nullptr) != 0 ||
		    rt_copy_to_host(acc->device, hostImage->MutablePixels(), image, bytes, nullptr) != 0)
		{
			SetLastError(fn + rt_last_error());
			return false;
		}
		return true;
	}

	bool AccumulatorDenoise(RaylibB200Accumulator* acc, const Image2D* albedo, const Image2D* normal, Image2D* out)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		const auto wall0 = std::chrono::steady_clock::now();
		t_lastError.clear();
		const std::string fn = "RaylibB200_AccumulatorDenoise: ";
		if (!acc || !out) { SetLastError(fn + "null accumulator or output image"); return false; }
		if (acc->samples < 2) { SetLastError(fn + "the variance needs at least 2 samples per pixel"); return false; }
		const uint32_t W = acc->width, H = acc->height;
		for (const std::string& why : { GuideSizeError(albedo, "albedo", W, H, "the accumulator"), GuideSizeError(normal, "normal", W, H, "the accumulator") })
			if (!why.empty()) { SetLastError(fn + why); return false; }
		RaylibB200Stats st;
		memset(&st, 0, sizeof(st));
		const Image2D* images[3] = { nullptr, albedo, normal };
		void* dev[3];
		void* image = nullptr;
		if (!UploadDenoiseImages(fn, acc->device, images, (uint64_t)W * H * 16ull, dev, &image, st) ||
		    !RunDenoise(fn, acc->device, acc->sums, acc->samples, dev[1], dev[2], W, H, image, nullptr, st) ||
		    !ReadDenoised(fn, acc->device, image, W, H, out, st))
			return false;
		st.totalMs = MsSince(wall0);
		SetLastStats(st);
		return true;
	}

	bool AccumulatorRead(RaylibB200Accumulator* acc, float* rgba)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		if (!acc || !rgba) { SetLastError("RaylibB200_AccumulatorRead: null argument"); return false; }
		if (rt_copy_to_host(acc->device, rgba, acc->sums, (uint64_t)acc->width * acc->height * 16ull, nullptr) != 0)
		{
			SetLastError(std::string("RaylibB200_AccumulatorRead: ") + rt_last_error());
			return false;
		}
		return true;
	}

	bool AccumulatorNoise(RaylibB200Accumulator* acc, float* perPixel, double* mean)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		const std::string fn = "RaylibB200_AccumulatorNoise: ";
		if (!acc) { SetLastError(fn + "null accumulator"); return false; }
		if (acc->samples < 2) { SetLastError(fn + "the noise figure needs at least 2 samples per pixel"); return false; }
		const uint64_t count = (uint64_t)acc->width * acc->height;
		float* noise = nullptr;
		if (perPixel && !(noise = (float*)ScratchBuffer(acc->device, 4, count * 4ull))) { SetLastError(fn + "device allocation failed: " + rt_last_error()); return false; }
		double total = 0.0;
		if (rt_resolve(acc->device, acc->sums, (uint32_t)count, acc->samples, nullptr, noise, mean ? &total : nullptr, nullptr) != 0 ||
		    (perPixel && rt_copy_to_host(acc->device, perPixel, noise, count * 4ull, nullptr) != 0))
		{
			SetLastError(fn + rt_last_error());
			return false;
		}
		if (mean) *mean = total / (double)count;
		return true;
	}

	bool AccumulatorSave(const RaylibB200Accumulator* acc, const char* path)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		const std::string fn = "RaylibB200_AccumulatorSave: ";
		if (!acc || !path || !*path) { SetLastError(fn + "null accumulator or empty path"); return false; }
		const uint64_t sumBytes = (uint64_t)acc->width * acc->height * 16ull;
		std::vector<float> sums((size_t)(sumBytes / 4));
		if (rt_copy_to_host(acc->device, sums.data(), acc->sums, sumBytes, nullptr) != 0) { SetLastError(fn + rt_last_error()); return false; }
		AccumFileHeader h;
		memset(&h, 0, sizeof(h));
		memcpy(h.magic, "RTACCUM1", 8);
		h.headerBytes = sizeof(h); h.bindingBytes = sizeof(RtAccumBinding);
		h.width = acc->width; h.height = acc->height; h.samples = acc->samples; h.bound = acc->bound ? 1u : 0u;
		h.checksum = AccumFileChecksum(h, acc->binding, sums.data(), sumBytes);
		const std::string tmp = std::string(path) + ".tmp";
		FILE* f = fopen(tmp.c_str(), "wb");
		if (!f) { SetLastError(fn + "cannot create " + tmp); return false; }
		bool ok = fwrite(&h, 1, sizeof(h), f) == sizeof(h) && fwrite(&acc->binding, 1, sizeof(acc->binding), f) == sizeof(acc->binding) &&
		          fwrite(sums.data(), 1, (size_t)sumBytes, f) == (size_t)sumBytes;
		ok = (fclose(f) == 0) && ok;
		if (!ok || rename(tmp.c_str(), path) != 0) { remove(tmp.c_str()); SetLastError(fn + "write failed: " + path); return false; }
		return true;
	}

	RaylibB200Accumulator* AccumulatorLoad(const char* path)
	{
		std::lock_guard<std::recursive_mutex> lock(g_mutex);
		t_lastError.clear();
		const std::string fn = std::string("RaylibB200_AccumulatorLoad: ") + (path ? path : "(null)") + ": ";
		FILE* f = path ? fopen(path, "rb") : nullptr;
		if (!f) { SetLastError(fn + "cannot open"); return nullptr; }
		AccumFileHeader h;
		RtAccumBinding b;
		std::vector<float> sums;
		std::string why;
		if (fread(&h, 1, sizeof(h), f) != sizeof(h) || memcmp(h.magic, "RTACCUM1", 8) != 0) why = "not an accumulator checkpoint file";
		else if (h.headerBytes != sizeof(h) || h.bindingBytes != sizeof(b)) why = "checkpoint written by a build with a different format";
		else if (h.width == 0 || h.height == 0 || (uint64_t)h.width * h.height >= (1ull << 31) || h.bound > 1u ||
		         h.samples > kMaxAccumSamples || (h.samples > 0u) != (h.bound != 0u))
			why = "checkpoint header is inconsistent";
		else
		{
			const uint64_t sumBytes = (uint64_t)h.width * h.height * 16ull;
			const uint64_t expect = sizeof(h) + sizeof(b) + sumBytes;
			long size = -1;
			if (fseek(f, 0, SEEK_END) == 0) size = ftell(f);
			if (size < 0 || fseek(f, (long)sizeof(h), SEEK_SET) != 0) why = "cannot read";
			else if ((uint64_t)size < expect) why = "checkpoint is truncated";
			else if ((uint64_t)size > expect) why = "checkpoint has trailing bytes";
			else
			{
				sums.resize((size_t)(sumBytes / 4));
				if (fread(&b, 1, sizeof(b), f) != sizeof(b) || fread(sums.data(), 1, (size_t)sumBytes, f) != (size_t)sumBytes) why = "checkpoint is truncated";
				else if (AccumFileChecksum(h, b, sums.data(), sumBytes) != h.checksum) why = "checkpoint is corrupt (checksum mismatch)";
				else if (h.bound && (b.width != h.width || b.height != h.height)) why = "checkpoint header is inconsistent";
			}
		}
		fclose(f);
		if (!why.empty()) { SetLastError(fn + why); return nullptr; }
		RaylibB200Accumulator* acc = NewAccumulator(h.width, h.height, fn.c_str());
		if (!acc) return nullptr;
		if (rt_copy_to_device(acc->device, acc->sums, sums.data(), (uint64_t)sums.size() * 4ull, nullptr) != 0)
		{
			SetLastError(fn + rt_last_error());
			AccumulatorDestroy(acc);
			return nullptr;
		}
		acc->samples = h.samples;
		acc->bound = h.bound != 0u;
		acc->binding = b;
		return acc;
	}
}

void RtForgetScene(const Scene* scene)
{
	std::lock_guard<std::recursive_mutex> lock(g_mutex);
	g_prebuilt.erase(scene);
	for (auto it = g_scenes.begin(); it != g_scenes.end();)
	{
		if (it->first.first == scene) { rt_scene_free(it->second.device); it = g_scenes.erase(it); }
		else ++it;
	}
}

// ---------------------------------------------------------------------------------------------
// Renderer

bool Renderer::IsDenoiserSupported() { return false; }    // OIDN is a Windows-only prebuilt in the reference (renderer.cc:28-33)

void Renderer::RenderScene(const RendererSettings* settings, const Scene* world, const Camera* camera, Image2D* outImage)
{
	CHECK(settings != nullptr && world != nullptr && camera != nullptr && outImage != nullptr);
	if (!settings || !world || !camera || !outImage) return;
	CHECK(world->GetAccelStruct() != nullptr || RtGpu::Prebuilt(world) != nullptr);      // scenes read from the flattened-scene cache have no object graph

	if (settings->viewportWidth != outImage->GetWidth() || settings->viewportHeight != outImage->GetHeight())
		outImage->Reallocate(settings->viewportWidth, settings->viewportHeight);

	if (!RtGpu::Render(settings, world, camera, outImage, nullptr, nullptr, 0, 1, 0, nullptr, RtIsLibraryImage(outImage)))
	{
		LOG("Raylib_Render FAILED: %s", RtGpu::LastError());
		return;
	}
	RaylibB200Stats st;
	if (RtGpu::GetLastStats(&st))
	{
		LOG("[STAT] GPU render: %.3f ms device, %.3f ms total, %.2f Mrays/s, %.2f M pixel-samples/s",
			st.deviceMs, st.totalMs,
			st.deviceMs > 0.0 ? (double)st.rayQueries / st.deviceMs * 1.0e-3 : 0.0,
			st.deviceMs > 0.0 ? (double)st.pixelSamples / st.deviceMs * 1.0e-3 : 0.0);
	}
}

bool Renderer::DenoiseScene(Image2D* mainImage, bool, Image2D*, Image2D*, Image2D* outDenoisedImage)
{
	CHECKF(mainImage != nullptr, "mainImage should not be null");
	CHECKF(outDenoisedImage != nullptr, "outDenoisedImage should not be null");
	return false;
}
