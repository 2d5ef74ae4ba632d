// rt_device.cu -- the sm_100a wavefront path tracer behind Raylib_Render, and the implementation
// of the thin C ABI in include/rt_device_abi.h.
//
// Stage kernels (one launch each per bounce; all persistent: a fixed grid of CTAs whose warps fetch
// 32 work items at a time from a device-side queue with one atomic per warp, and append to the
// next queues with ballot/popc (match_any) compaction):
//   k_raygen      GenerateCell's jitter + Camera::GetCameraRay      render/renderer.cc:232-239, camera.h:44-53
//   k_extend      BVHNode::Hit closest hit                           geom/bvh.cc:82-107 (+ aabb/triangle/sphere/cube)
//   k_shade<M>    Material::Scatter/ScatteringPdf/Emitted, one launch per material type ("material-sorted")
//                                                                    render/renderer.cc:131-153, material.cc
//   k_miss        sky lookup, spawns the sun visibility ray          render/renderer.cc:156-193
//   k_shadow      any-hit query toward the sun                       render/renderer.cc:194-198
//   k_accumulate  accum += Li (sample order), /= SPP, SetPixel       render/renderer.cc:244-248
//                 (or: continue and store back a running sum, rt_progressive.h)
//   k_debug_view  TraceSceneDebugMode                                render/renderer.cc:62-111
// Recursion is unrolled into a per-path bounce stack {reflectance, scatPdf, emitted, pdf} that is
// folded tail-first when the path ends, reproducing the nested arithmetic of TraceScene exactly.
//
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a --fmad=false -lineinfo (see Makefile).
#include "rt_device_abi.h"
#include "rt_progressive.h"
#include "rt_trace_stage.h"
#include "rt_checksum.h"
#include "rt_shade.cuh"

#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>
#include <algorithm>

#ifndef RT_PACKED_STATE
#define RT_PACKED_STATE 1      // path state as 32-byte records (one sector per access); 0 = separate float4 arrays
#endif

// ------------------------------------------------------------------------------------------------
// error plumbing

static thread_local std::string g_lastError;
extern "C" const char* rt_last_error(void) { return g_lastError.c_str(); }

#define RT_CUDA(expr)                                                                      \
	do {                                                                                   \
		cudaError_t _e = (expr);                                                           \
		if (_e != cudaSuccess) {                                                           \
			char _buf[512];                                                                \
			snprintf(_buf, sizeof(_buf), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
			g_lastError = _buf;                                                            \
			cudaGetLastError();     /* the runtime keeps the code for the next call otherwise */ \
			return (int)_e;                                                                \
		}                                                                                  \
	} while (0)

// The traversal stack of a thread: RT_MAX_STACK {ref, entry t} entries in thread-local memory (rt_traverse.cuh).
#if RT_STACK_SMEM_LEVELS > 0
#define RT_DECLARE_STACK(name) uint2 localStack_[RT_MAX_STACK]; __shared__ uint2 sharedStack_[RT_STACK_SMEM_LEVELS * 128]; \
	RtStack name; name.base = localStack_; name.stride = 1; name.sm = sharedStack_ + threadIdx.x
#else
#define RT_DECLARE_STACK(name) uint2 localStack_[RT_MAX_STACK]; RtStack name; name.base = localStack_; name.stride = 1
#endif

// ------------------------------------------------------------------------------------------------
// device-side control block and launch descriptor

#define RT_Q_MISS RT_MAT_NUM_TYPES
#define RT_MAX_BOUNCE_STATS 16
#define RT_NUM_HIT_QUEUES (RT_MAT_NUM_TYPES + 1)

// Queue counters of ONE bounce (128 B, so that consecutive bounces do not share a line).  A pass zeroes the whole array
// once (cudaMemsetAsync) instead of resetting shared counters between bounces with a one-thread kernel.
struct RtBounceCtl
{
	uint32_t extCount, extCursor;              // rays entering k_extend of this bounce
	uint32_t matCount[RT_NUM_HIT_QUEUES];      // [0..5] one per material type, [RT_Q_MISS] rays that hit nothing
	uint32_t matCursor[RT_NUM_HIT_QUEUES];
	uint32_t shadowCount, shadowCursor;        // sun-visibility rays spawned by this bounce's misses
	uint32_t pad[32 - 4 - 2 * RT_NUM_HIT_QUEUES];
};
static_assert(sizeof(RtBounceCtl) == 128, "RtBounceCtl is one 128-byte line");

// Frame-wide counters (zeroed at the start of a frame), followed in memory by RtBounceCtl[depth capacity + 1].
struct RtQueueCtl
{
	unsigned long long rayQueries;
	unsigned long long boxTests, triTests, sphereTests, nodeVisits;
	unsigned long long refBoxTests, refTriTests, refSphereTests, statRays;
	unsigned long long gateTests, cubeTests;
	unsigned long long nodeIters, nodeStep, nodeAlive, leafIters, leafBusy;   // lane-iterations of k_extend's traversal loop (statistics build)
	unsigned long long bounceRays[RT_MAX_BOUNCE_STATS];     // closest-hit rays per bounce, summed over the passes of a frame
};

struct RtLaunch
{
	RtSceneView S;
	RtCamera cam;
	// path-state arena (SoA, indexed by path slot)
	// Path state is read and written through queue indices, i.e. as per-slot gathers: every record a stage kernel touches
	// is ONE 32-byte sector moved by one 256-bit load / store (RT_PACKED_STATE 0 keeps the round-1 layout of separate
	// float4 arrays, where each access used half a sector: the stage kernels ran at ~50 % sector efficiency).
#if RT_PACKED_STATE
	RtF8*   ray;           // {o.xyz, time | d.xyz, -}
	RtF8*   hitCtl;        // {t, bu, bv, ref bits | rngCtr, slotKey (bin of the ray a shade kernel wrote into this slot), -, -}
	RtF8*   stack;         // [bounce][slot] {reflectance.xyz, scatPdf | emitted.xyz, pdf}
#else
	float4* rayO;          // o.xyz, time
	float4* rayD;          // d.xyz, -
	float4* hit;           // t, bu, bv, ref bits
	float4* stackA;        // [bounce][slot] reflectance.xyz, scatPdf
	float4* stackB;        // [bounce][slot] emitted.xyz, pdf
#endif
	float4* Li;            // per path result
	float4* missPartial;   // sky term while the sun ray is in flight
	float4* accum;         // [shard pixel] running sample sum
	float4* out;           // [shard pixel] final Pixel
	float4* image;         // optional: row-major W x H frame the final pixels go to DIRECTLY (may be another GPU's memory,
	                       // mapped over NVLink): fuses the tile gather into the last accumulate; `out` is then unused
	float4* out2;          // [shard pixel] second output of the fused denoiser-input pass (RT_RENDERMODE_AUX)
#if !RT_PACKED_STATE
	uint32_t* rngCtr;
#endif
	uint32_t* extQ[2];
	uint32_t* matQ[RT_NUM_HIT_QUEUES];   // extend's output queues: material-sorted hits + misses
	uint32_t* shadowQ;
	// ray binning (counting sort of the next bounce's rays by origin cell + direction octant, see k_bin_*)
#if !RT_PACKED_STATE
	uint32_t* slotKey;     // [slot] bin of the ray a shade kernel wrote into this slot
#endif
	uint32_t* extKey;      // [queue position] bin of the ray at that position of the coming bounce's extend queue: written next
	                       // to the queue entry (coalesced), so that the scatter pass streams instead of gathering per slot
	uint32_t* extSorted;   // the extend queue of the coming bounce in bin order
	uint32_t* binCount;    // [numBins] histogram, filled by the shade kernels, zeroed again by k_bin_scan
	uint32_t* binCursor;   // [numBins] exclusive prefix = next free position of every bin
	uint32_t  binBits;     // origin bits + direction bits of the key (0 = binning off)
	uint32_t  binAxisBits[3];      // origin cells per axis = 2^binAxisBits
	uint32_t  binDirBits;  // the octahedral direction map has 2^binDirBits cells per side
	uint32_t  numBins;
	float     binOrigin[3], binScale[3], binTop[3];
	RtQueueCtl* ctl;       // frame-wide counters
	RtBounceCtl* bounceCtl; // [maxDepth + 2] queue counters of the pass in flight ([maxDepth + 1]: arrival counter of k_pass_fused's barrier)
	// frame
	uint64_t seed;
	uint32_t width, height, tilesX, numTiles;
	uint32_t npix;         // pixel slots of this shard (tile capacity * RT_TILE_PIXELS)
	uint32_t K;            // samples in flight per pixel in this pass
	uint32_t passBase;     // first sample index of this pass
	uint32_t spp;          // max(1, samplesPerPixel)
	int32_t  maxDepth;
	uint32_t renderMode;
	uint32_t shardRank, shardCount;
	uint32_t capacity;     // path slots allocated
	uint2*   poolStack;        // k_extend_pool: [warp of the grid][level][RT_POOL_RAYS] traversal stacks in global memory
	uint32_t poolNodeThreshold, poolRefill;
	uint32_t refillThreshold;  // a warp refills its idle lanes once fewer than this many lanes are traversing
	uint32_t walkThreshold;    // the node phase yields to the leaf phase once fewer than this many lanes can step
	float    tMin;
	uint32_t runningSum;       // 1 = `image` holds the undivided per-pixel sums {sum RGB, sum luminance^2} of earlier samples:
	                           //   the first pass continues them, the last pass stores them back (progressive rendering)
};

// ---- path-state accessors (one definition per layout) ------------------------------------------------------------
RT_DEV RtF8 ld8_state(const RtF8* p)
{
	RtF8 r;
	asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
		: "=f"(r.lo.x), "=f"(r.lo.y), "=f"(r.lo.z), "=f"(r.lo.w), "=f"(r.hi.x), "=f"(r.hi.y), "=f"(r.hi.z), "=f"(r.hi.w) : "l"(p) : "memory");
	return r;
}
RT_DEV void st8_state(RtF8* p, float4 lo, float4 hi)
{
	asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
		:: "l"(p), "f"(lo.x), "f"(lo.y), "f"(lo.z), "f"(lo.w), "f"(hi.x), "f"(hi.y), "f"(hi.z), "f"(hi.w) : "memory");
}
#if RT_PACKED_STATE
RT_DEV void load_ray(const RtLaunch& L, uint32_t slot, float4& o, float4& d) { const RtF8 v = ld8_state(L.ray + slot); o = v.lo; d = v.hi; }
RT_DEV float4 load_ray_origin(const RtLaunch& L, uint32_t slot) { return reinterpret_cast<const float4*>(L.ray + slot)[0]; }
RT_DEV float4 load_ray_dir(const RtLaunch& L, uint32_t slot) { return reinterpret_cast<const float4*>(L.ray + slot)[1]; }
RT_DEV void store_ray(const RtLaunch& L, uint32_t slot, float4 o, float4 d) { st8_state(L.ray + slot, o, d); }
RT_DEV void store_hit(const RtLaunch& L, uint32_t slot, float4 h) { reinterpret_cast<float4*>(L.hitCtl + slot)[0] = h; }
RT_DEV void load_hit_and_counter(const RtLaunch& L, uint32_t slot, float4& h, uint32_t& ctr)
{
	const RtF8 v = ld8_state(L.hitCtl + slot);
	h = v.lo; ctr = __float_as_uint(v.hi.x);
}
RT_DEV void store_counter(const RtLaunch& L, uint32_t slot, uint32_t ctr) { reinterpret_cast<uint32_t*>(L.hitCtl + slot)[4] = ctr; }
RT_DEV void store_counter_and_key(const RtLaunch& L, uint32_t slot, uint32_t ctr, uint32_t key)
{
	reinterpret_cast<uint2*>(L.hitCtl + slot)[2] = make_uint2(ctr, key);
}
RT_DEV uint32_t load_slot_key(const RtLaunch& L, uint32_t slot) { return reinterpret_cast<const uint32_t*>(L.hitCtl + slot)[5]; }
RT_DEV void load_bounce(const RtLaunch& L, int bounce, uint32_t slot, float4& a, float4& b)
{
	const RtF8 v = ld8_state(L.stack + (size_t)bounce * L.capacity + slot);
	a = v.lo; b = v.hi;
}
RT_DEV void store_bounce(const RtLaunch& L, int bounce, uint32_t slot, float4 a, float4 b) { st8_state(L.stack + (size_t)bounce * L.capacity + slot, a, b); }
#else
RT_DEV void load_ray(const RtLaunch& L, uint32_t slot, float4& o, float4& d) { o = L.rayO[slot]; d = L.rayD[slot]; }
RT_DEV float4 load_ray_origin(const RtLaunch& L, uint32_t slot) { return L.rayO[slot]; }
RT_DEV float4 load_ray_dir(const RtLaunch& L, uint32_t slot) { return L.rayD[slot]; }
RT_DEV void store_ray(const RtLaunch& L, uint32_t slot, float4 o, float4 d) { L.rayO[slot] = o; L.rayD[slot] = d; }
RT_DEV void store_hit(const RtLaunch& L, uint32_t slot, float4 h) { L.hit[slot] = h; }
RT_DEV void load_hit_and_counter(const RtLaunch& L, uint32_t slot, float4& h, uint32_t& ctr) { h = L.hit[slot]; ctr = L.rngCtr[slot]; }
RT_DEV void store_counter(const RtLaunch& L, uint32_t slot, uint32_t ctr) { L.rngCtr[slot] = ctr; }
RT_DEV void store_counter_and_key(const RtLaunch& L, uint32_t slot, uint32_t ctr, uint32_t key) { L.rngCtr[slot] = ctr; L.slotKey[slot] = key; }
RT_DEV uint32_t load_slot_key(const RtLaunch& L, uint32_t slot) { return L.slotKey[slot]; }
RT_DEV void load_bounce(const RtLaunch& L, int bounce, uint32_t slot, float4& a, float4& b)
{
	a = L.stackA[(size_t)bounce * L.capacity + slot]; b = L.stackB[(size_t)bounce * L.capacity + slot];
}
RT_DEV void store_bounce(const RtLaunch& L, int bounce, uint32_t slot, float4 a, float4 b)
{
	L.stackA[(size_t)bounce * L.capacity + slot] = a; L.stackB[(size_t)bounce * L.capacity + slot] = b;
}
#endif

// shard pixel slot -> image pixel (tiles interleaved across shards, 8x4 sub-blocks per warp)
RT_DEV bool slot_to_pixel(const RtLaunch& L, uint32_t lp, uint32_t& x, uint32_t& y)
{
	const uint32_t localTile = lp / RT_TILE_PIXELS, within = lp % RT_TILE_PIXELS;
	const uint32_t tile = localTile * L.shardCount + L.shardRank;
	if (tile >= L.numTiles) return false;
	const uint32_t tx = tile % L.tilesX, ty = tile / L.tilesX;
	const uint32_t sub = within >> 5, lane = within & 31u;
	x = tx * RT_TILE_W + (sub & 1u) * 8u + (lane & 7u);
	y = ty * RT_TILE_H + (sub >> 1) * 4u + (lane >> 3);
	return x < L.width && y < L.height;
}

// Final pixel of shard slot lp = image pixel (x, y): into the shard buffer, or straight into the (possibly remote) frame.
RT_DEV void store_pixel(const RtLaunch& L, uint32_t lp, uint32_t x, uint32_t y, float4 value)
{
	if (L.image) L.image[(size_t)y * L.width + x] = value;
	else L.out[lp] = value;
}

// Bin of a ray for the coherence sort: cell of the origin in the scene box (binAxisBits per axis, chosen by the host so
// that cells come out roughly cubic) above the direction's cell on the octahedral map (2^binDirBits squared).  Rays of
// one warp then start in the same corner of the tree and leave it the same way.
RT_DEV uint32_t bin_key(const RtLaunch& L, float3 o, float3 d)
{
	const uint32_t cx = (uint32_t)fminf(fmaxf((o.x - L.binOrigin[0]) * L.binScale[0], 0.0f), L.binTop[0]);
	const uint32_t cy = (uint32_t)fminf(fmaxf((o.y - L.binOrigin[1]) * L.binScale[1], 0.0f), L.binTop[1]);
	const uint32_t cz = (uint32_t)fminf(fmaxf((o.z - L.binOrigin[2]) * L.binScale[2], 0.0f), L.binTop[2]);
	uint32_t key = (((cx << L.binAxisBits[1]) | cy) << L.binAxisBits[2]) | cz;
	if (L.binDirBits)
	{
		const float inv = 1.0f / (fabsf(d.x) + fabsf(d.y) + fabsf(d.z));
		float u = d.x * inv, v = d.y * inv;
		if (d.z < 0.0f)
		{
			const float fu = (1.0f - fabsf(v)) * (u < 0.0f ? -1.0f : 1.0f), fv = (1.0f - fabsf(u)) * (v < 0.0f ? -1.0f : 1.0f);
			u = fu; v = fv;
		}
		const float cells = (float)(1u << L.binDirBits), top = cells - 1.0f;
		const uint32_t du = (uint32_t)fminf(fmaxf((u * 0.5f + 0.5f) * cells, 0.0f), top);
		const uint32_t dv = (uint32_t)fminf(fmaxf((v * 0.5f + 0.5f) * cells, 0.0f), top);
		key = (((key << L.binDirBits) | du) << L.binDirBits) | dv;
	}
	return min(key, L.numBins - 1u);
}

// ------------------------------------------------------------------------------------------------
// warp-level queue primitives

RT_DEV uint32_t lane_id() { return threadIdx.x & 31u; }

// One atomic per warp: reserve 32 consecutive work items.
RT_DEV uint32_t warp_fetch32(uint32_t* cursor)
{
	uint32_t base = 0;
	if (lane_id() == 0) base = atomicAdd(cursor, 32u);
	return __shfl_sync(0xFFFFFFFFu, base, 0);
}

// Append `value` to the queue selected by `target` (< 0: none).  Lanes with the same target are
// grouped with match_any; the group leader reserves popc(group) slots with one atomic.
RT_DEV void warp_push(uint32_t* const* queues, uint32_t* counts, int target, uint32_t value)
{
	const uint32_t active = __ballot_sync(0xFFFFFFFFu, target >= 0);
	if (target < 0) return;
	const uint32_t group = __match_any_sync(active, target);
	const uint32_t leader = __ffs(group) - 1u;
	uint32_t base = 0;
	if (lane_id() == leader) base = atomicAdd(counts + target, __popc(group));
	base = __shfl_sync(group, base, leader);
	queues[target][base + __popc(group & ((1u << lane_id()) - 1u))] = value;
}

// Returns the queue position the value went to (undefined for lanes with pred == false).
RT_DEV uint32_t warp_push_one(uint32_t* queue, uint32_t* count, bool pred, uint32_t value)
{
	const uint32_t mask = __ballot_sync(0xFFFFFFFFu, pred);
	if (!pred) return 0u;
	const uint32_t leader = __ffs(mask) - 1u;
	uint32_t base = 0;
	if (lane_id() == leader) base = atomicAdd(count, __popc(mask));
	base = __shfl_sync(mask, base, leader);
	const uint32_t pos = base + __popc(mask & ((1u << lane_id()) - 1u));
	queue[pos] = value;
	return pos;
}

// ------------------------------------------------------------------------------------------------
// path termination: unwind the bounce stack (TraceScene's recursion, renderer.cc:133-153)

RT_DEV void finish_path(const RtLaunch& L, uint32_t slot, int lastBounce, float3 Lterm)
{
	float3 Lr = Lterm;
	for (int k = lastBounce; k >= 0; --k)
	{
		float4 a, b;
		load_bounce(L, k, slot, a, b);
		Lr = fold_bounce(xyz(a), a.w, b.w, xyz(b), Lr);
	}
	L.Li[slot] = make_float4(Lr.x, Lr.y, Lr.z, 0.0f);
}

// ------------------------------------------------------------------------------------------------
// kernels

// Every stage is a device function (`*_stage`) with a thin kernel around it, so that the one-launch-per-pass kernel of small
// frames (k_pass_fused below) runs the very same code between grid-wide barriers.
RT_DEV void raygen_stage(const RtLaunch& L)
{
	const uint32_t total = L.K * L.npix;
	for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < ((total + 31u) & ~31u); slot += gridDim.x * blockDim.x)
	{
		bool valid = slot < total;
		uint32_t x = 0, y = 0, s = 0;
		if (valid)
		{
			const uint32_t k = slot / L.npix, lp = slot - k * L.npix;
			s = L.passBase + k;
			valid = (s < L.spp) && slot_to_pixel(L, lp, x, y);
		}
		if (valid)
		{
			RtRng rng; rng.key = rt_sample_key(L.seed, y * L.width + x, s); rng.ctr = 0;
			float u = (float)x / (float)L.width;
			float v = (float)y / (float)L.height;
			if (s != 0)
			{
				u += (rng.next() - 0.5f) * 2.0f / (float)L.width;
				v += (rng.next() - 0.5f) * 2.0f / (float)L.height;
			}
			const RtRay r = camera_ray(L.cam, u, v, rng);
			store_ray(L, slot, make_float4(r.o.x, r.o.y, r.o.z, r.time), make_float4(r.d.x, r.d.y, r.d.z, 0.0f));
			store_counter(L, slot, rng.ctr);
			L.Li[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
		}
		warp_push_one(L.extQ[0], &L.bounceCtl[0].extCount, valid && L.maxDepth > 0, slot);
	}
}
__global__ void __launch_bounds__(256) k_raygen(const __grid_constant__ RtLaunch L) { raygen_stage(L); }

// ---- traversal kernels --------------------------------------------------------------------------------
// Persistent warps with PER-LANE work replacement: a lane whose ray has finished parks its result; as soon as
// fewer than `refill` lanes of the warp are still traversing, the warp flushes the parked results (one
// ballot/match-compacted append per target queue) and hands fresh rays to the idle lanes (one atomic for the
// whole warp).  This removes the tail where a few long rays keep a mostly idle warp alive.
enum { LANE_EMPTY = 0, LANE_ACTIVE = 1, LANE_DONE = 2 };
#ifndef RT_DEFAULT_PIPES
#define RT_DEFAULT_PIPES 2
#endif
#ifndef RT_DEFAULT_EXTEND_RING
#define RT_DEFAULT_EXTEND_RING 0      // measured: serialising the extends (ring) loses 4 % -- co-running stage kernels slow the traversal by as much as they hide
#endif
#ifndef RT_DUAL_PIPE_TRAVERSAL_CTAS
#define RT_DUAL_PIPE_TRAVERSAL_CTAS 7
#endif
#ifndef RT_DEFAULT_BIN_OBITS
#define RT_DEFAULT_BIN_OBITS 12     // origin bits of the ray-binning key (0 = no binning)
#endif
#ifndef RT_BIN_MIN_LEAVES
#define RT_BIN_MIN_LEAVES 65536u    // scenes with fewer leaves stay in L1/L2 anyway: binning only costs there (measured: Cornell -30 %)
#endif
#ifndef RT_DEFAULT_BIN_DBITS
#define RT_DEFAULT_BIN_DBITS 2      // bits per side of the octahedral direction map
#endif
#ifndef RT_HIT_TO_MEMORY
#define RT_HIT_TO_MEMORY 1          // k_extend writes an accepted hit to the path's hit record at once instead of carrying bu / bv (needs RT_PACKED_STATE)
#endif
#if !RT_PACKED_STATE
#undef RT_HIT_TO_MEMORY
#define RT_HIT_TO_MEMORY 0          // the separate-arrays layout keeps the round-1 flush
#endif
#ifndef RT_PARK_DIRECTION
#define RT_PARK_DIRECTION 0         // k_extend keeps {d, time} of its rays in shared memory while they walk inner nodes (see trav_run)
#endif
#ifndef RT_EXTEND_MIN_BLOCKS
#define RT_EXTEND_MIN_BLOCKS 9      // CTAs of 128 threads per SM the traversal kernels are compiled for (register cap = 65536 / (128 * N));
                                    // 9 = 56 registers: 42 bytes of spills, all outside the node/leaf loops (8: 64 registers, 10: spills in the loops)
#endif

template<bool STATS>
RT_DEV void extend_stage(const RtLaunch& L, int bounce, RtStack stack)
{
#if RT_PARK_DIRECTION
	__shared__ float4 parkedDir[128];     // {d.xyz, time} of every lane's ray while it walks inner nodes (trav_run)
#endif
	const uint32_t cur = bounce & 1;
	RtBounceCtl& bc = L.bounceCtl[bounce];
	const uint32_t count = bc.extCount;
	const uint32_t* queue = (L.binBits && bounce > 0) ? L.extSorted : L.extQ[cur];     // bounced rays arrive in bin order
	RtTravStats st = {};

	int state = LANE_EMPTY;
	uint32_t slot = 0;
	RtRay r;
	RtTrav ts;
	bool exhausted = false;            // warp-uniform: the queue has no more rays for this warp

	for (;;)
	{
		// ---- flush parked results (warp-synchronous) ----
		int target = -1;
		if (state == LANE_DONE)
		{
		#if !RT_HIT_TO_MEMORY
			store_hit(L, slot, make_float4(ts.best.t, ts.best.bu, ts.best.bv, __uint_as_float(ts.best.ref)));
		#endif      // else: every accepted hit went to the record when it was accepted (trav_leaf); nobody reads the record of a miss
			if (ts.found()) target = ts.hitType;        // recorded when the hit was accepted: no dependent loads here
			else target = RT_Q_MISS;
			state = LANE_EMPTY;
		}
		warp_push(L.matQ, bc.matCount, target, slot);

		// ---- hand fresh rays to idle lanes ----
		if (!exhausted)
		{
			const uint32_t idle = __ballot_sync(0xFFFFFFFFu, state == LANE_EMPTY);
			const uint32_t n = __popc(idle);
			const uint32_t leader = idle ? (uint32_t)(__ffs(idle) - 1) : 0u;
			uint32_t base = 0;
			if (n && lane_id() == leader) base = atomicAdd(&bc.extCursor, n);
			base = __shfl_sync(0xFFFFFFFFu, base, leader);
			if (state == LANE_EMPTY)
			{
				const uint32_t i = base + __popc(idle & ((1u << lane_id()) - 1u));
				if (i < count)
				{
					slot = queue[i];
					float4 o, d;
					load_ray(L, slot, o, d);
					r = make_ray(xyz(o), xyz(d), o.w);
				#if RT_PARK_DIRECTION
					parkedDir[threadIdx.x] = make_float4(d.x, d.y, d.z, o.w);
				#endif
					if (STATS) count_reference_work(L.S, r, L.tMin, stack, st);
					state = trav_begin<STATS>(L.S, r, L.tMin, ts, st) ? LANE_ACTIVE : LANE_DONE;
				}
			}
			if (n && base + n >= count) exhausted = true;
		}

		const uint32_t active = __ballot_sync(0xFFFFFFFFu, state == LANE_ACTIVE);
		if (active == 0)
		{
			if (__ballot_sync(0xFFFFFFFFu, state == LANE_DONE) == 0) break;     // nothing in flight, nothing parked
			continue;                                                           // only parked results: flush them
		}

		// ---- traverse until too few lanes are busy ----
		bool alive = state == LANE_ACTIVE;
	#if RT_HIT_TO_MEMORY
		trav_run<false, STATS>(L.S, r, L.tMin, stack, ts, alive, exhausted ? 1u : L.refillThreshold, L.walkThreshold, st, nullptr,
		                       reinterpret_cast<float4*>(L.hitCtl), slot);
	#elif RT_PARK_DIRECTION
		trav_run<false, STATS>(L.S, r, L.tMin, stack, ts, alive, exhausted ? 1u : L.refillThreshold, L.walkThreshold, st, parkedDir + threadIdx.x);
	#else
		trav_run<false, STATS>(L.S, r, L.tMin, stack, ts, alive, exhausted ? 1u : L.refillThreshold, L.walkThreshold, st);
	#endif
		if (state == LANE_ACTIVE && !alive) state = LANE_DONE;
	}
	if (STATS)
	{
		atomicAdd(&L.ctl->boxTests, (unsigned long long)st.box);
		atomicAdd(&L.ctl->triTests, (unsigned long long)st.tri);
		atomicAdd(&L.ctl->sphereTests, (unsigned long long)st.sphere);
		atomicAdd(&L.ctl->nodeVisits, (unsigned long long)st.nodes);
		atomicAdd(&L.ctl->gateTests, (unsigned long long)st.gate); atomicAdd(&L.ctl->cubeTests, (unsigned long long)st.cube);
		atomicAdd(&L.ctl->refBoxTests, (unsigned long long)st.refBox);
		atomicAdd(&L.ctl->refTriTests, (unsigned long long)st.refTri);
		atomicAdd(&L.ctl->refSphereTests, (unsigned long long)st.refSphere);
		atomicAdd(&L.ctl->nodeIters, (unsigned long long)st.nodeIters); atomicAdd(&L.ctl->nodeStep, (unsigned long long)st.nodeStep);
		atomicAdd(&L.ctl->nodeAlive, (unsigned long long)st.nodeAlive);
		atomicAdd(&L.ctl->leafIters, (unsigned long long)st.leafIters); atomicAdd(&L.ctl->leafBusy, (unsigned long long)st.leafBusy);
		if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&L.ctl->statRays, (unsigned long long)count);
	}
}
template<bool STATS>
__global__ void __launch_bounds__(128, RT_EXTEND_MIN_BLOCKS) k_extend(const __grid_constant__ RtLaunch L, int bounce)
{
	RT_DECLARE_STACK(stack);
	extend_stage<STATS>(L, bounce, stack);
}

// ---- pooled traversal (opt-in, RAYLIB_B200_POOL=1) --------------------------------------------------------------------
// k_extend gives every lane ONE ray for that ray's whole walk, so a node step runs at ~21 of 32 lanes (the others are
// blocked on leaves or wait for the next refill) and a leaf step at ~16.  Here a warp owns a POOL of RT_POOL_RAYS rays
// whose traversal state lives in shared memory; at every step the warp compacts the rays that can take that kind of step
// and hands one to each lane, so that node steps and leaf steps both run (nearly) full.  The step functions are the very
// ones k_extend uses (trav_step, trav_pending_leaf): results are identical.  Stacks move to global memory, laid out
// [level][ray of the pool] like thread-local memory lays them out [level][lane].
#ifndef RT_POOL_RAYS
#define RT_POOL_RAYS 64
#endif
#ifndef RT_POOL_MIN_BLOCKS
#define RT_POOL_MIN_BLOCKS 8
#endif
struct RtWarpPool
{
	float4   A[RT_POOL_RAYS];      // o.xyz, best t
	float4   B[RT_POOL_RAYS];      // clamped 1/d, prune limit
	uint4    C[RT_POOL_RAYS];      // cur, pending leaf, stack entries, path slot
	uint4    D[RT_POOL_RAYS];      // bu bits, bv bits, best ref, material type of the best hit (-1: none)
	uint32_t list[RT_POOL_RAYS];   // rays chosen for the step in flight, compacted
};

// lane i of the warp gets the i-th set bit of `mask` (a ray of the pool), for the first min(32, popc) bits
RT_DEV uint32_t pool_select(RtWarpPool& P, uint64_t mask, uint32_t& outCount)
{
	const uint32_t lane = lane_id();
	#pragma unroll
	for (uint32_t half = 0; half < RT_POOL_RAYS / 32u; ++half)
	{
		const uint32_t r = lane + 32u * half;
		if ((mask >> r) & 1ull)
		{
			const uint32_t pos = (uint32_t)__popcll(mask & ((1ull << r) - 1ull));
			if (pos < 32u) P.list[pos] = r;
		}
	}
	__syncwarp();
	outCount = min(32u, (uint32_t)__popcll(mask));
	const uint32_t r = P.list[lane];
	__syncwarp();
	return r;
}
RT_DEV uint64_t pool_or64(uint64_t v)
{
	const uint32_t lo = __reduce_or_sync(0xFFFFFFFFu, (uint32_t)v), hi = __reduce_or_sync(0xFFFFFFFFu, (uint32_t)(v >> 32));
	return ((uint64_t)hi << 32) | lo;
}

__global__ void __launch_bounds__(128, RT_POOL_MIN_BLOCKS) k_extend_pool(const __grid_constant__ RtLaunch L, int bounce)
{
	__shared__ RtWarpPool pools[4];
	RtWarpPool& P = pools[threadIdx.x >> 5];
	const uint32_t lane = lane_id();
	uint2* const warpStack = L.poolStack + (size_t)(blockIdx.x * 4u + (threadIdx.x >> 5)) * RT_MAX_STACK * RT_POOL_RAYS;
	RtBounceCtl& bc = L.bounceCtl[bounce];
	const uint32_t count = bc.extCount;
	const uint32_t* queue = (L.binBits && bounce > 0) ? L.extSorted : L.extQ[bounce & 1];
	const uint64_t all = RT_POOL_RAYS == 64 ? ~0ull : ((1ull << RT_POOL_RAYS) - 1ull);
	RtTravStats st = {};

	// warp-uniform status of the pool's rays, one bit each
	uint64_t emptyMask = all, stepMask = 0, leafMask = 0, doneMask = 0;
	bool exhausted = false;
	for (;;)
	{
		const uint32_t nStep = (uint32_t)__popcll(stepMask), nFree = (uint32_t)__popcll(emptyMask | doneMask);
		const uint64_t blockedMask = leafMask & ~stepMask;
		const uint32_t nBlocked = (uint32_t)__popcll(blockedMask);
		if ((nFree >= L.poolRefill && !exhausted) || (nStep == 0 && leafMask == 0))
		{
			if (nFree == RT_POOL_RAYS && exhausted && doneMask == 0) break;
			// ---- flush finished rays, hand fresh rays to the free slots ----
			uint32_t freeBefore = 0;
			uint32_t base = 0;
			const uint64_t freeMask = emptyMask | doneMask;
			if (!exhausted)
			{
				if (lane == 0) base = atomicAdd(&bc.extCursor, nFree);
				base = __shfl_sync(0xFFFFFFFFu, base, 0);
			}
			uint64_t newStep = 0, newDone = 0, newEmpty = 0;
			#pragma unroll
			for (uint32_t half = 0; half < RT_POOL_RAYS / 32u; ++half)
			{
				const uint32_t r = lane + 32u * half;
				const uint64_t bit = 1ull << r;
				int target = -1;
				uint32_t slot = 0;
				if (doneMask & bit)
				{
					const float4 a = P.A[r]; const uint4 c = P.C[r], d = P.D[r];
					slot = c.w;
					store_hit(L, slot, make_float4(a.w, __uint_as_float(d.x), __uint_as_float(d.y), __uint_as_float(d.z)));
					target = ((int32_t)d.w >= 0) ? (int32_t)d.w : RT_Q_MISS;
				}
				warp_push(L.matQ, bc.matCount, target, slot);
				if (freeMask & bit)
				{
					const uint32_t i = base + freeBefore + (uint32_t)__popc((uint32_t)(freeMask >> (32u * half)) & ((1u << lane) - 1u));
					if (!exhausted && i < count)
					{
						const uint32_t s = queue[i];
						float4 o, d;
						load_ray(L, s, o, d);
						const RtRay ray = make_ray(xyz(o), xyz(d), o.w);
						RtTrav ts;
						const bool inside = trav_begin<false>(L.S, ray, L.tMin, ts, st);
						P.A[r] = make_float4(ray.o.x, ray.o.y, ray.o.z, ts.best.t);
						P.B[r] = make_float4(ray.idc.x, ray.idc.y, ray.idc.z, ts.limit);
						P.C[r] = make_uint4(inside ? ts.cur : RT_REF_DONE, RT_REF_DONE, 0u, s);
						P.D[r] = make_uint4(0u, 0u, RT_MISS_REF, 0xFFFFFFFFu);
						if (inside) newStep |= bit; else newDone |= bit;
					}
					else newEmpty |= bit;
				}
				freeBefore += (uint32_t)__popc((uint32_t)(freeMask >> (32u * half)));
			}
			if (!exhausted && base + nFree >= count) exhausted = true;
			newStep = pool_or64(newStep); newDone = pool_or64(newDone); newEmpty = pool_or64(newEmpty);
			stepMask |= newStep;
			doneMask = newDone;
			emptyMask = newEmpty;
			__syncwarp();
			continue;
		}

		const bool nodeStep = nStep >= 32u || (nStep >= L.poolNodeThreshold) || (nStep > 0u && leafMask == 0) || (nStep > 0u && nBlocked == 0u && nStep >= 8u);
		if (nodeStep)
		{
			uint32_t n;
			const uint32_t r = pool_select(P, stepMask, n);
			uint64_t bit = 0, nowStep = 0, nowLeaf = 0, nowDone = 0;
			if (lane < n)
			{
				bit = 1ull << r;
				const float4 a = P.A[r], b = P.B[r];
				const uint4 c = P.C[r];
				RtRay ray;
				ray.o = xyz(a); ray.idc = xyz(b); ray.d = v3(0.0f); ray.time = 0.0f;
				RtTrav ts;
				ts.best.t = a.w; ts.best.bu = 0.0f; ts.best.bv = 0.0f; ts.best.ref = RT_MISS_REF;
				ts.limit = b.w; ts.cur = c.x; ts.leaf = c.y; ts.sp = c.z; ts.hitType = -1;
				RtStack stack; stack.base = warpStack + r; stack.stride = RT_POOL_RAYS;
				trav_step<false, false>(L.S, ray, L.tMin, stack, ts, st);
				P.C[r] = make_uint4(ts.cur, ts.leaf, ts.sp, c.w);
				if (trav_finished(ts)) nowDone = bit;
				else
				{
					if (trav_can_step(ts)) nowStep = bit;
					if (ts.leaf != RT_REF_DONE) nowLeaf = bit;
				}
			}
			const uint64_t processed = pool_or64(bit);
			stepMask = (stepMask & ~processed) | pool_or64(nowStep);
			leafMask = (leafMask & ~processed) | pool_or64(nowLeaf);
			doneMask |= pool_or64(nowDone);
			continue;
		}

		// ---- leaf step: rays blocked on two leaves first, then rays carrying a postponed leaf ----
		{
			uint32_t n;
			const uint64_t pick = nBlocked >= 32u ? blockedMask : leafMask;
			const uint32_t r = pool_select(P, pick, n);
			uint64_t bit = 0, nowStep = 0, nowLeaf = 0, nowDone = 0;
			if (lane < n)
			{
				bit = 1ull << r;
				const float4 a = P.A[r], b = P.B[r];
				const uint4 c = P.C[r], d = P.D[r];
				float4 o, dir;
				load_ray(L, c.w, o, dir);       // the direction (and shutter time) come back from the path's record
				RtRay ray;
				ray.o = xyz(a); ray.d = xyz(dir); ray.idc = xyz(b); ray.time = o.w;
				RtTrav ts;
				ts.best.t = a.w; ts.best.bu = __uint_as_float(d.x); ts.best.bv = __uint_as_float(d.y); ts.best.ref = d.z;
				ts.limit = b.w; ts.cur = c.x; ts.leaf = c.y; ts.sp = c.z; ts.hitType = (int32_t)d.w;
				trav_pending_leaf<false, false>(L.S, ray, L.tMin, ts, st);
				P.A[r] = make_float4(a.x, a.y, a.z, ts.best.t);
				P.B[r] = make_float4(b.x, b.y, b.z, ts.limit);
				P.C[r] = make_uint4(ts.cur, ts.leaf, ts.sp, c.w);
				P.D[r] = make_uint4(__float_as_uint(ts.best.bu), __float_as_uint(ts.best.bv), ts.best.ref, (uint32_t)ts.hitType);
				if (trav_finished(ts)) nowDone = bit;
				else
				{
					if (trav_can_step(ts)) nowStep = bit;
					if (ts.leaf != RT_REF_DONE) nowLeaf = bit;
				}
			}
			const uint64_t processed = pool_or64(bit);
			stepMask = (stepMask & ~processed) | pool_or64(nowStep);
			leafMask = (leafMask & ~processed) | pool_or64(nowLeaf);
			doneMask |= pool_or64(nowDone);
		}
	}
}

template<int MT>
RT_DEV void shade_stage(const RtLaunch& L, int bounce)
{
	RtBounceCtl& bc = L.bounceCtl[bounce];
	const uint32_t count = bc.matCount[MT];
	if (count == 0u) return;        // no atomics on the cursor for a material nobody hit this bounce
	const uint32_t* queue = L.matQ[MT];
	const uint32_t nxt = (bounce & 1) ^ 1;
	for (;;)
	{
		const uint32_t base = warp_fetch32(&bc.matCursor[MT]);
		if (base >= count) break;
		const uint32_t i = base + lane_id();
		bool cont = false;
		uint32_t slot = 0, binKey = 0;
		if (i < count)
		{
			slot = queue[i];
			float4 o, d, hq;
			uint32_t rngCounter;
			load_ray(L, slot, o, d);
			load_hit_and_counter(L, slot, hq, rngCounter);
			RtRay r; r.o = xyz(o); r.d = xyz(d); r.time = o.w; r.idc = v3(0.0f);
			RtHit h; h.t = hq.x; h.bu = hq.y; h.bv = hq.z; h.ref = __float_as_uint(hq.w);
			RtSurface sf;
			reconstruct_surface(L.S, r, h, sf);
			const RtMaterial m = L.S.materials[sf.material];

			// pixel/sample of this slot -> RNG stream
			const uint32_t k = slot / L.npix, lp = slot - k * L.npix;
			uint32_t x, y; slot_to_pixel(L, lp, x, y);
			RtRng rng; rng.key = rt_sample_key(L.seed, y * L.width + x, L.passBase + k); rng.ctr = rngCounter;

			RtBounce b;
			if (MT == RT_MAT_MICROFACET) build_basis(sf);       // hitResult.BuildOrthonormalBasis(), renderer.cc:131
			scatter<MT>(L.S, m, r, sf, rng, b);
			store_bounce(L, bounce, slot, make_float4(b.reflectance.x, b.reflectance.y, b.reflectance.z, b.scatPdf),
			             make_float4(b.emitted.x, b.emitted.y, b.emitted.z, b.pdf));

			cont = (b.pdf > 0.0f) && (bounce + 1 < L.maxDepth);
			if (cont)
			{
				store_ray(L, slot, make_float4(sf.p.x, sf.p.y, sf.p.z, r.time), make_float4(b.nextDir.x, b.nextDir.y, b.nextDir.z, 0.0f));
				if (L.binBits)
				{
					binKey = bin_key(L, sf.p, b.nextDir);
					atomicAdd(L.binCount + binKey, 1u);
				}
				store_counter(L, slot, rng.ctr);
			}
			else
			{
				// either no recursive term, or the recursive call returns 0 at the depth limit (renderer.cc:120-123)
				finish_path(L, slot, bounce, v3(0.0f));
			}
		}
		const uint32_t pos = warp_push_one(L.extQ[nxt], &L.bounceCtl[bounce + 1].extCount, cont, slot);
		if (cont && L.binBits) L.extKey[pos] = binKey;
	}
}
// The microfacet shader is the only heavy one (72 registers uncapped: 7 CTAs per SM); RT_MICROFACET_MIN_BLOCKS caps it.
#ifndef RT_MICROFACET_MIN_BLOCKS
#define RT_MICROFACET_MIN_BLOCKS 1
#endif
template<int MT>
__global__ void __launch_bounds__(128, MT == RT_MAT_MICROFACET ? RT_MICROFACET_MIN_BLOCKS : 1) k_shade(const __grid_constant__ RtLaunch L, int bounce) { shade_stage<MT>(L, bounce); }

// ---- ray binning: counting sort of the coming bounce's extend queue -----------------------------------------
// The shade kernels left a histogram of bin keys (binCount) and the key of every continuing slot (slotKey).
// k_bin_scan turns the histogram into start positions (one CTA: numBins <= 2^18) and clears it for the next bounce;
// k_bin_scatter moves every queue entry to its bin.  Order inside a bin is arbitrary -- paths are independent, the
// image does not depend on queue order.
__global__ void __launch_bounds__(1024) k_bin_scan(uint32_t* binCount, uint32_t* binCursor, uint32_t numBins)
{
	__shared__ uint32_t warpSum[32];
	__shared__ uint32_t carry;
	if (threadIdx.x == 0) carry = 0;
	__syncthreads();
	// chunks of 4 bins per thread, 4096 bins per sweep of the CTA
	for (uint32_t base = 0; base < numBins; base += 4096u)
	{
		const uint32_t i = base + threadIdx.x * 4u;
		uint4 c = make_uint4(0, 0, 0, 0);
		if (i + 3u < numBins) c = *reinterpret_cast<const uint4*>(binCount + i);
		else { if (i < numBins) c.x = binCount[i]; if (i + 1u < numBins) c.y = binCount[i + 1u]; if (i + 2u < numBins) c.z = binCount[i + 2u]; }
		const uint32_t mine = c.x + c.y + c.z + c.w;
		uint32_t incl = mine;
		#pragma unroll
		for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if ((threadIdx.x & 31u) >= (uint32_t)d) incl += v; }
		if ((threadIdx.x & 31u) == 31u) warpSum[threadIdx.x >> 5] = incl;
		__syncthreads();
		if (threadIdx.x < 32u)
		{
			uint32_t w = warpSum[threadIdx.x], wi = w;
			#pragma unroll
			for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, wi, d); if (threadIdx.x >= (uint32_t)d) wi += v; }
			warpSum[threadIdx.x] = wi - w;       // exclusive prefix of the warp totals
		}
		__syncthreads();
		const uint32_t start = carry + warpSum[threadIdx.x >> 5] + incl - mine;
		const uint4 o = make_uint4(start, start + c.x, start + c.x + c.y, start + c.x + c.y + c.z);
		if (i + 3u < numBins)
		{
			*reinterpret_cast<uint4*>(binCursor + i) = o;
			*reinterpret_cast<uint4*>(binCount + i) = make_uint4(0, 0, 0, 0);
		}
		else
		{
			if (i < numBins) { binCursor[i] = o.x; binCount[i] = 0; }
			if (i + 1u < numBins) { binCursor[i + 1u] = o.y; binCount[i + 1u] = 0; }
			if (i + 2u < numBins) { binCursor[i + 2u] = o.z; binCount[i + 2u] = 0; }
		}
		__syncthreads();
		if (threadIdx.x == 1023u) carry = start + mine;
		__syncthreads();
	}
}

__global__ void __launch_bounds__(256) k_bin_scatter(const __grid_constant__ RtLaunch L, int bounce)
{
	const uint32_t nxt = (bounce & 1) ^ 1;
	const uint32_t count = L.bounceCtl[bounce + 1].extCount;
	const uint32_t* queue = L.extQ[nxt];
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x)
	{
		const uint32_t slot = queue[i];
		const uint32_t pos = atomicAdd(L.binCursor + L.extKey[i], 1u);
		L.extSorted[pos] = slot;
	}
}

RT_DEV void miss_stage(const RtLaunch& L, int bounce)
{
	RtBounceCtl& bc = L.bounceCtl[bounce];
	const uint32_t count = bc.matCount[RT_Q_MISS];
	if (count == 0u) return;
	for (;;)
	{
		const uint32_t base = warp_fetch32(&bc.matCursor[RT_Q_MISS]);
		if (base >= count) break;
		const uint32_t i = base + lane_id();
		bool toSun = false;
		uint32_t slot = 0;
		if (i < count)
		{
			slot = L.matQ[RT_Q_MISS][i];
			const float4 d = load_ray_dir(L, slot);
			const float3 sky = sky_radiance(L.S, xyz(d));
			if (L.S.hasSun)
			{
				L.missPartial[slot] = make_float4(sky.x, sky.y, sky.z, 0.0f);
				toSun = true;
			}
			else finish_path(L, slot, bounce - 1, sky);
		}
		warp_push_one(L.shadowQ, &bc.shadowCount, toSun, slot);
	}
}
__global__ void __launch_bounds__(128) k_miss(const __grid_constant__ RtLaunch L, int bounce) { miss_stage(L, bounce); }

RT_DEV void shadow_stage(const RtLaunch& L, int bounce, RtStack stack)
{
	RtBounceCtl& bc = L.bounceCtl[bounce];
	const uint32_t count = bc.shadowCount;
	if (count == 0u) return;
	RtTravStats st = {};

	int state = LANE_EMPTY;
	uint32_t slot = 0;
	RtRay r;
	RtTrav ts;
	bool exhausted = false;
	for (;;)
	{
		if (state == LANE_DONE)
		{
			// the sun contributes unless ANY primitive is hit (renderer.cc:194-197)
			float3 miss = xyz(L.missPartial[slot]);
			if (!ts.found()) miss = miss + v3(L.S.sunIlluminance);
			finish_path(L, slot, bounce - 1, miss);
			state = LANE_EMPTY;
		}
		if (!exhausted)
		{
			const uint32_t idle = __ballot_sync(0xFFFFFFFFu, state == LANE_EMPTY);
			const uint32_t n = __popc(idle);
			const uint32_t leader = idle ? (uint32_t)(__ffs(idle) - 1) : 0u;
			uint32_t base = 0;
			if (n && lane_id() == leader) base = atomicAdd(&bc.shadowCursor, n);
			base = __shfl_sync(0xFFFFFFFFu, base, leader);
			if (state == LANE_EMPTY)
			{
				const uint32_t i = base + __popc(idle & ((1u << lane_id()) - 1u));
				if (i < count)
				{
					slot = L.shadowQ[i];
					const float4 o = load_ray_origin(L, slot);
					// the visibility ray starts at the missing ray's ORIGIN (renderer.cc:193)
					r = make_ray(xyz(o), -v3(L.S.sunDirection), o.w);
					state = trav_begin<false>(L.S, r, L.tMin, ts, st) ? LANE_ACTIVE : LANE_DONE;
				}
			}
			if (n && base + n >= count) exhausted = true;
		}
		const uint32_t active = __ballot_sync(0xFFFFFFFFu, state == LANE_ACTIVE);
		if (active == 0)
		{
			if (__ballot_sync(0xFFFFFFFFu, state == LANE_DONE) == 0) break;
			continue;
		}
		bool alive = state == LANE_ACTIVE;
		trav_run<true, false>(L.S, r, L.tMin, stack, ts, alive, exhausted ? 1u : L.refillThreshold, L.walkThreshold, st);
		if (state == LANE_ACTIVE && !alive) state = LANE_DONE;
	}
}
__global__ void __launch_bounds__(128, RT_EXTEND_MIN_BLOCKS) k_shadow(const __grid_constant__ RtLaunch L, int bounce)
{
	RT_DECLARE_STACK(stack);
	shadow_stage(L, bounce, stack);
}

// Rec. 709 weights, as Image2D::PostProcess uses them (render/image.cc:44-103)
RT_DEV float luminance3(float3 v) { return dot3(v, v3(0.2126f, 0.7152f, 0.0722f)); }

// Grid-stride over the shard's pixel slots: every pixel sums its K samples in sample order (renderer.cc:244-246).
// Running-sum mode continues the sums held in the row-major `image` and stores them back undivided, so that samples [a, b)
// added to the stored sum of [0, a) take exactly the float additions of one frame of b samples; .w sums the squared
// luminance of the samples (the noise estimate of RaylibB200_AccumulatorNoise).
RT_DEV void accumulate_stage(const RtLaunch& L, int firstPass, int lastPass)
{
	if (blockIdx.x == 0 && threadIdx.x == 0)
	{
		// ray queries of the pass that just finished: closest-hit rays of every bounce + the sun-visibility rays
		unsigned long long rays = 0;
		for (int b = 0; b < L.maxDepth; ++b)
		{
			rays += L.bounceCtl[b].extCount + L.bounceCtl[b].shadowCount;
			L.ctl->bounceRays[min(b, RT_MAX_BOUNCE_STATS - 1)] += L.bounceCtl[b].extCount;
		}
		L.ctl->rayQueries += rays;
	}
	for (uint32_t lp = blockIdx.x * blockDim.x + threadIdx.x; lp < L.npix; lp += gridDim.x * blockDim.x)
	{
		uint32_t x, y;
		if (!slot_to_pixel(L, lp, x, y))
		{
			if (lastPass && !L.image) L.out[lp] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);      // padding slot of the shard buffer
			continue;
		}
		const size_t pixel = (size_t)y * L.width + x;
		const float4 start = !firstPass ? L.accum[lp] : L.runningSum ? L.image[pixel] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
		float3 a = xyz(start);
		float y2 = start.w;
		const uint32_t kValid = min(L.K, L.spp - L.passBase);
		for (uint32_t k = 0; k < kValid; ++k)
		{
			const float3 li = xyz(L.Li[(size_t)k * L.npix + lp]);
			a = a + li;
			if (L.runningSum) { const float lum = luminance3(li); y2 += lum * lum; }
		}
		if (lastPass && L.runningSum) L.image[pixel] = make_float4(a.x, a.y, a.z, y2);
		else if (lastPass)
		{
			a = div_assign3(a, (float)L.spp);
			store_pixel(L, lp, x, y, make_float4(a.x, a.y, a.z, 1.0f));
		}
		else L.accum[lp] = make_float4(a.x, a.y, a.z, y2);
	}
}
__global__ void __launch_bounds__(256) k_accumulate(const __grid_constant__ RtLaunch L, int firstPass, int lastPass) { accumulate_stage(L, firstPass, lastPass); }

// ---- one launch per pass (small frames) ------------------------------------------------------------------------------
// A frame of a few hundred thousand paths spends its time between kernels, not in them: ~11 launches per bounce, each a
// persistent grid that starts, finds a short queue and drains (the 320x180x8 smoke frame: 112 launches for 2.9 ms).  Here the
// whole pass -- camera rays, every bounce's extend / shade / miss / sun-visibility stage, the per-pixel sums -- is ONE
// cooperative launch; stages are separated by a grid-wide barrier instead of a kernel boundary.  The stages are the very
// device functions the separate kernels wrap, so the image is bit-identical (test_fused_pass_is_the_same_image).
//   * barrier: one arrival counter per pass (zeroed with the bounce counters), thread 0 of every CTA fences, arrives, spins
//     with acquire loads and fences again -- the gpu-scope fence also invalidates the SM's L1 (CCTL.IVALL), which a kernel
//     boundary did implicitly: path state written by other SMs in the previous stage must not be served from a stale line;
//   * the sun-visibility stage of bounce b and the extend stage of bounce b+1 touch disjoint paths (a path that missed is
//     over), so they share one phase: two barriers per bounce;
//   * a pass whose paths have all ended leaves the bounce loop early (the counter is uniform after the barrier).
RT_DEV void grid_barrier(uint32_t* arrivals, uint32_t& target)
{
	__syncthreads();
	if (threadIdx.x == 0)
	{
		target += gridDim.x;
		__threadfence();
		atomicAdd(arrivals, 1u);
		uint32_t seen;
		do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(arrivals) : "memory"); } while (seen < target);
		__threadfence();
	}
	__syncthreads();
}

RT_DEV uint32_t load_counter(const uint32_t* p)
{
	uint32_t v;
	asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}

#ifndef RT_DEFAULT_PATHS_M
#define RT_DEFAULT_PATHS_M 64u               // Mi paths in flight over all pipes (16 / 32 / 64 / 128: 2495 / 2600 / 2674 / 2679 Mrays/s on scatter10M)
#endif
#ifndef RT_DEFAULT_FUSED_PATHS_K
#define RT_DEFAULT_FUSED_PATHS_K 1024u      // frames of up to this many Ki paths (width x height x samples) render as one launch
#endif
#ifndef RT_FUSED_MIN_BLOCKS
#define RT_FUSED_MIN_BLOCKS 4
#endif
__global__ void __launch_bounds__(128, RT_FUSED_MIN_BLOCKS) k_pass_fused(const __grid_constant__ RtLaunch L, uint32_t materialMask, int firstPass, int lastPass)
{
	RT_DECLARE_STACK(stack);
	uint32_t* arrivals = &L.bounceCtl[L.maxDepth + 1].extCount;      // the spare control block behind the last bounce's
	uint32_t target = 0;
	raygen_stage(L);
	grid_barrier(arrivals, target);
	for (int b = 0; b < L.maxDepth; ++b)
	{
		// the previous bounce's sun-visibility rays ride along with this bounce's closest-hit rays
		if (b > 0 && L.S.hasSun) shadow_stage(L, b - 1, stack);
		if (load_counter(&L.bounceCtl[b].extCount) == 0u) break;
		extend_stage<false>(L, b, stack);
		grid_barrier(arrivals, target);
		if (materialMask & (1u << RT_MAT_LAMBERTIAN)) shade_stage<RT_MAT_LAMBERTIAN>(L, b);
		if (materialMask & (1u << RT_MAT_METAL))      shade_stage<RT_MAT_METAL>(L, b);
		if (materialMask & (1u << RT_MAT_DIELECTRIC)) shade_stage<RT_MAT_DIELECTRIC>(L, b);
		if (materialMask & (1u << RT_MAT_MIRROR))     shade_stage<RT_MAT_MIRROR>(L, b);
		if (materialMask & (1u << RT_MAT_LIGHT))      shade_stage<RT_MAT_LIGHT>(L, b);
		if (materialMask & (1u << RT_MAT_MICROFACET)) shade_stage<RT_MAT_MICROFACET>(L, b);
		miss_stage(L, b);
		grid_barrier(arrivals, target);
		if (b + 1 == L.maxDepth && L.S.hasSun) shadow_stage(L, b, stack);
	}
	grid_barrier(arrivals, target);
	accumulate_stage(L, firstPass, lastPass);
}

// ---- debug views (render modes 1..6): one unjittered camera ray per pixel ---------------------------
RT_DEV float3 debug_albedo(const RtSceneView& S, const RtMaterial& m, float u, float v)
{
	switch (m.type)
	{
	case RT_MAT_LAMBERTIAN: case RT_MAT_METAL: return v3(m.color);
	case RT_MAT_MICROFACET: return microfacet_albedo(S, m, u, v);
	default: return v3(0.0f);          // Material::GetAlbedo base (material.h:44)
	}
}
RT_DEV bool debug_mirror_like(const RtSceneView& S, const RtMaterial& m, float u, float v)
{
	if (m.type == RT_MAT_DIELECTRIC || m.type == RT_MAT_MIRROR) return true;
	if (m.type == RT_MAT_MICROFACET) return microfacet_roughness(S, m, u, v) < 0.1f;
	return false;
}

__global__ void __launch_bounds__(128) k_debug_view(const __grid_constant__ RtLaunch L)
{
	RT_DECLARE_STACK(stack);
	RtTravStats st = {};
	unsigned long long rays = 0;
	const bool aux = L.renderMode == RT_RENDERMODE_AUX;
	// every warp walks its pixels 32 at a time so that the lanes can traverse together (traverse_warp)
	const uint32_t rounded = (L.npix + 31u) & ~31u;
	for (uint32_t lp = blockIdx.x * blockDim.x + threadIdx.x; lp < rounded; lp += gridDim.x * blockDim.x)
	{
		uint32_t x = 0, y = 0;
		const bool slotExists = lp < L.npix;
		const bool inside = slotExists && slot_to_pixel(L, lp, x, y);
		RtRng rng; rng.key = rt_sample_key(L.seed, y * L.width + x, 0u); rng.ctr = 0;
		const RtRay r = camera_ray(L.cam, (float)x / (float)L.width, (float)y / (float)L.height, rng);
		float3 value = v3(0.0f), value2 = v3(0.0f);
		RtHit h;
		if (inside) rays++;
		const bool hit = traverse_warp<false>(L.S, r, L.tMin, stack, inside, L.walkThreshold, h, st);

		// per-lane shading of the primary hit; Albedo may ask for a second ray (one mirror bounce, renderer.cc:70-84)
		bool needSecond = false;
		RtRay r2 = r;
		if (hit && L.renderMode != RT_RENDERMODE_PRIMARY_EXPORT)
		{
			RtSurface sf;
			reconstruct_surface(L.S, r, h, sf);
			const RtMaterial m = L.S.materials[sf.material];
			if (L.renderMode == 1u || aux)
			{
				value = debug_albedo(L.S, m, sf.u, sf.v);
				if (debug_mirror_like(L.S, m, sf.u, sf.v))
				{
					needSecond = true;
					r2 = make_ray(sf.p, reflect3(r.d, sf.n), r.time);
					rays++;
				}
			}
			else if (L.renderMode == 2u) value = v3(0.5f) + 0.5f * sf.n;
			if (L.renderMode == 3u || aux)
			{
				// the debug views never call BuildOrthonormalBasis: LocalToWorld runs on the zero tangent / bitangent of a
				// default-constructed HitResult (vec3() is (0,0,0), core/vec3.h:16), i.e. the view shows N.z * n
				sf.tangent = v3(0.0f); sf.bitangent = v3(0.0f);
				float3 N = (m.type == RT_MAT_MICROFACET) ? microfacet_normal(L.S, m, sf.u, sf.v) : v3(0.0f, 0.0f, 1.0f);
				N = local_to_world(sf, N);
				if (aux) value2 = 0.5f + 0.5f * N;
				else value = 0.5f + 0.5f * N;
			}
			else if (L.renderMode == 4u) value = v3(sf.u, sf.v, 0.0f);
			else if (L.renderMode == 5u)
			{
				value = (m.type == RT_MAT_LIGHT) ? v3(m.color) : (m.type == RT_MAT_MICROFACET) ? microfacet_emitted(L.S, m, sf.u) : v3(0.0f);
			}
			else if (L.renderMode == 6u)
			{
				RtBounce b;
				value = v3(1.0f, 0.75f, 0.8f);
				sf.tangent = v3(0.0f); sf.bitangent = v3(0.0f);     // Scatter on the unbuilt (zero) frame, as in renderer.cc:103-107
				switch (m.type)
				{
				case RT_MAT_LAMBERTIAN: scatter<RT_MAT_LAMBERTIAN>(L.S, m, r, sf, rng, b); value = b.reflectance; break;
				case RT_MAT_METAL:      scatter<RT_MAT_METAL>(L.S, m, r, sf, rng, b); value = b.reflectance; break;
				case RT_MAT_DIELECTRIC: scatter<RT_MAT_DIELECTRIC>(L.S, m, r, sf, rng, b); value = b.reflectance; break;
				case RT_MAT_MIRROR:     scatter<RT_MAT_MIRROR>(L.S, m, r, sf, rng, b); value = b.reflectance; break;
				case RT_MAT_MICROFACET: scatter<RT_MAT_MICROFACET>(L.S, m, r, sf, rng, b); value = b.reflectance; break;
				default: break;
				}
			}
		}
		if (L.renderMode == 1u || aux)
		{
			RtHit h2;
			if (traverse_warp<false>(L.S, r2, L.tMin, stack, needSecond, L.walkThreshold, h2, st))
			{
				RtSurface sf2;
				reconstruct_surface(L.S, r2, h2, sf2);
				value = debug_albedo(L.S, L.S.materials[sf2.material], sf2.u, sf2.v);
			}
		}

		if (!slotExists) continue;
		if (!inside)
		{
			if (!L.image) L.out[lp] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
			if (aux) L.out2[lp] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
		}
		else if (L.renderMode == RT_RENDERMODE_PRIMARY_EXPORT)
		{
			// primary-visibility export for the parity tests: (t, leaf rank bits, barycentrics)
			store_pixel(L, lp, x, y, hit ? make_float4(h.t, __int_as_float((int)rank_of(L.S, h.ref)), h.bu, h.bv)
			                             : make_float4(0.0f, __int_as_float(-1), 0.0f, 0.0f));
		}
		else
		{
			store_pixel(L, lp, x, y, make_float4(value.x, value.y, value.z, 1.0f));
			if (aux) L.out2[lp] = make_float4(value2.x, value2.y, value2.z, 1.0f);
		}
	}
	atomicAdd(&L.ctl->rayQueries, rays);
}

// ---- arbitrary-ray closest hit (parity tests, primary-visibility export) ---------------------------
template<bool STATS>
__global__ void __launch_bounds__(128) k_trace_rays(const __grid_constant__ RtSceneView S, const float4* rays, int64_t numRays,
                                                     float tMin, int32_t* outRank, float* outT, RtQueueCtl* ctl)
{
	RT_DECLARE_STACK(stack);
	RtTravStats st = {};
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < numRays; i += (int64_t)gridDim.x * blockDim.x)
	{
		const float4 o = rays[2 * i], d = rays[2 * i + 1];
		const RtRay r = make_ray(xyz(o), xyz(d), o.w);
		RtHit h;
		const bool found = traverse<false, STATS>(S, r, tMin, stack, h, st);
		if (STATS) count_reference_work(S, r, tMin, stack, st);
		outRank[i] = found ? (int32_t)rank_of(S, h.ref) : -1;
		outT[i] = found ? h.t : 0.0f;
	}
	if (STATS)
	{
		atomicAdd(&ctl->boxTests, (unsigned long long)st.box);
		atomicAdd(&ctl->triTests, (unsigned long long)st.tri);
		atomicAdd(&ctl->sphereTests, (unsigned long long)st.sphere);
		atomicAdd(&ctl->nodeVisits, (unsigned long long)st.nodes);
		atomicAdd(&ctl->gateTests, (unsigned long long)st.gate); atomicAdd(&ctl->cubeTests, (unsigned long long)st.cube);
		atomicAdd(&ctl->refBoxTests, (unsigned long long)st.refBox);
		atomicAdd(&ctl->refTriTests, (unsigned long long)st.refTri);
		atomicAdd(&ctl->refSphereTests, (unsigned long long)st.refSphere);
	}
}

// ---- gather epilogue: tile-major shard slabs -> row-major image ---------------------------------------
__global__ void __launch_bounds__(256) k_assemble(const float4* shards, uint32_t shardCount, uint32_t capTiles,
                                                   uint32_t width, uint32_t height, float4* image)
{
	const uint32_t tilesX = (width + RT_TILE_W - 1) / RT_TILE_W;
	const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
	if (pixel >= width * height) return;
	const uint32_t x = pixel % width, y = pixel / width;
	const uint32_t tile = (y / RT_TILE_H) * tilesX + (x / RT_TILE_W);
	const uint32_t rank = tile % shardCount, localTile = tile / shardCount;
	const uint32_t ix = x % RT_TILE_W, iy = y % RT_TILE_H;
	const uint32_t sub = (iy / 4u) * 2u + (ix / 8u), lane = (iy % 4u) * 8u + (ix % 8u);
	image[pixel] = shards[((size_t)rank * capTiles + localTile) * RT_TILE_PIXELS + sub * 32u + lane];
}

// ------------------------------------------------------------------------------------------------
// host side

struct RtDeviceScene
{
	int device = 0;
	RtSceneView view;
	std::vector<void*> allocations;
	std::vector<size_t> allocationBytes;
	std::vector<size_t> contentBytes;     // bytes of each allocation that hold uploaded data (an empty array still allocates)
	uint32_t maxStackDepth = 0;
	uint32_t materialTypeMask = 0;
	uint32_t numLeaves = 0;
	uint64_t bytes = 0;
};

// One pipe = one set of path-state arenas + queue control block + stream.  Passes alternate between two pipes so that
// the memory-latency-bound stage kernels of one pass (shade, miss, raygen) overlap the issue-bound traversal of the other.
#define RT_MAX_PIPES 4
struct RtPipe
{
	RtLaunch L;                  // arena pointers live here
	RtQueueCtl* ctl = nullptr;           // frame-wide counters (allocated with the context)
	std::vector<void*> allocations;
	uint32_t capacity = 0;       // path slots
	int32_t  depthCapacity = 0;  // bounce-stack levels
	uint2* poolStack = nullptr;          // k_extend_pool: traversal stacks of every warp of its grid
	size_t poolStackEntries = 0;
	cudaStream_t stream = nullptr;      // used only when two pipes are active (a single pipe runs on the caller's stream)
	cudaEvent_t evAccum = nullptr;      // "this pipe's latest k_accumulate is done": orders the per-pixel sums across pipes
	cudaEvent_t evExtend = nullptr;     // "this pipe's latest k_extend is done": the extend ring (rt_render_shard)
	std::vector<cudaEvent_t> stageEvents;   // pairs bracketing k_extend launches when stage timing is on
};

struct RtRenderContext
{
	int device = 0;
	int numSMs = 0;
	bool cooperative = false;    // the device launches cooperative kernels (k_pass_fused)
	RtPipe pipe[RT_MAX_PIPES];
	float4* accum = nullptr;     // [shard pixel] running sample sum, shared by the pipes
	uint32_t pixCapacity = 0;
	cudaEvent_t evStart = nullptr, evStop = nullptr, evFork = nullptr;
	std::map<const void*, int> gridCache;      // persistent_grid results
};

extern "C" int rt_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n;
}

template<typename T>
static int upload_array(RtDeviceScene* sc, const T* host, size_t count, const T** outDev)
{
	*outDev = nullptr;
	const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
	void* dev = nullptr;
	RT_CUDA(cudaMalloc(&dev, bytes));
	sc->allocations.push_back(dev);
	sc->allocationBytes.push_back(bytes);
	sc->contentBytes.push_back(count * sizeof(T));
	sc->bytes += bytes;
	if (count) RT_CUDA(cudaMemcpy(dev, host, count * sizeof(T), cudaMemcpyHostToDevice));
	*outDev = reinterpret_cast<const T*>(dev);
	return 0;
}

// sRGB textures are decoded ONCE, when the scene is uploaded: the reference applies pow(x, 2.2) to all four channels of every
// texel it fetches (render/texture.cc:45-51 -> image.h:79-83), a pure function of the texel, so running the very same rt_m_powf
// over the uploaded copy gives the bits a fetch-time decode would -- and takes four double-precision pow evaluations out
// of every microfacet texture fetch and one out of every cut-out test inside the traversal loop.  Every (image, sRGB flag)
// pair owns its texel range (RtSceneFlattener::AddTexture), so the in-place rewrite cannot touch a linear view of the image.
__global__ void __launch_bounds__(256) k_linearize_texels(float4* texels, uint64_t count)
{
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x)
	{
		float4 px = texels[i];
		px.x = rt_m_powf(px.x, 2.2f); px.y = rt_m_powf(px.y, 2.2f); px.z = rt_m_powf(px.z, 2.2f); px.w = rt_m_powf(px.w, 2.2f);
		texels[i] = px;
	}
}

extern "C" int rt_scene_has_reference_tree(const RtDeviceScene* sc) { return (sc && sc->view.refNodes) ? 1 : 0; }

extern "C" int rt_scene_upload(int device, const RtSceneDesc* d, uint32_t flags, RtDeviceScene** outScene)
{
	*outScene = nullptr;
	RT_CUDA(cudaSetDevice(device));
	RtDeviceScene* sc = new RtDeviceScene;
	sc->device = device;
	RtSceneView& v = sc->view;
	memset(&v, 0, sizeof(v));
	int rc = 0;
	const RtNodeQ4* nodes = nullptr; const RtNode* refNodes = nullptr; const RtTriHot* hot = nullptr; const RtSphere* sph = nullptr;
	const float* texels = nullptr; const float* gates = nullptr;
	// the kernels walk the 4-wide tree; the reference topology is only read by the statistics build
	if ((rc = upload_array(sc, d->quantNodes, d->numWideNodes, &nodes))) goto fail;
	if (flags & RT_UPLOAD_REFERENCE_TREE) { if ((rc = upload_array(sc, d->refNodes, d->numRefNodes, &refNodes))) goto fail; }
	if ((rc = upload_array(sc, d->triHot, d->numTris, &hot))) goto fail;
	if ((rc = upload_array(sc, d->triCold, d->numTris, &v.triCold))) goto fail;
	v.triRank = nullptr; v.triGate = nullptr;       // rank and gate index of a triangle are words of its hot record
	if ((rc = upload_array(sc, d->gateBoxes, (size_t)d->numGates * 8, &gates))) goto fail;
	if ((rc = upload_array(sc, d->spheres, d->numSpheres, &sph))) goto fail;
	if ((rc = upload_array(sc, d->sphereMaterial, d->numSpheres, &v.sphereMaterial))) goto fail;
	if ((rc = upload_array(sc, d->sphereRank, d->numSpheres, &v.sphereRank))) goto fail;
	if ((rc = upload_array(sc, d->sphereGate, d->numSpheres, &v.sphereGate))) goto fail;
	if ((rc = upload_array(sc, d->cubes, d->numCubes, &v.cubes))) goto fail;
	if ((rc = upload_array(sc, d->cubeRank, d->numCubes, &v.cubeRank))) goto fail;
	if ((rc = upload_array(sc, d->cubeGate, d->numCubes, &v.cubeGate))) goto fail;
	if ((rc = upload_array(sc, d->materials, d->numMaterials, &v.materials))) goto fail;
	if ((rc = upload_array(sc, d->texels, (size_t)d->numTexels * 4, &texels))) goto fail;
	{
		// the device's texture table says "linear" for the textures decoded here
		std::vector<RtTexture> table(d->textures, d->textures + d->numTextures);
		for (RtTexture& tx : table)
		{
			if (!tx.srgb) continue;
			const uint64_t count = (uint64_t)tx.width * tx.height;
			if (count)
			{
				float4* first = reinterpret_cast<float4*>(const_cast<float*>(texels)) + tx.texelOffset;
				k_linearize_texels<<<(unsigned)std::min<uint64_t>((count + 255) / 256, 148u * 16u), 256>>>(first, count);
			}
			tx.srgb = 0u;
		}
		if ((rc = upload_array(sc, table.data(), table.size(), &v.textures))) goto fail;
		if (cudaError_t e = cudaDeviceSynchronize()) { g_lastError = std::string("rt_scene_upload: texture decode: ") + cudaGetErrorString(e); cudaGetLastError(); rc = (int)e; goto fail; }
	}
	v.nodes = reinterpret_cast<const float4*>(nodes);
	v.refNodes = reinterpret_cast<const float4*>(refNodes);
	v.triHot = reinterpret_cast<const float4*>(hot);
	v.spheres = reinterpret_cast<const float4*>(sph);
	v.texels = reinterpret_cast<const float4*>(texels);
	v.gateBoxes = reinterpret_cast<const float4*>(gates);
	for (int i = 0; i < 3; ++i) { v.rootMin[i] = d->rootMin[i]; v.rootMax[i] = d->rootMax[i]; }
	v.rootRef = d->wideRootRef;
	for (int i = 0; i < 3; ++i) { v.refRootMin[i] = d->refRootMin[i]; v.refRootMax[i] = d->refRootMax[i]; }
	v.refRootRef = d->refRootRef;
	v.refRootBoxTests = d->refRootBoxTests;
	v.flags = d->flags;
	v.q4magic = 0x3F000000u;
	v.skyTexture = d->skyTexture;
	for (int i = 0; i < 9; ++i) v.skyRotation[i] = d->skyRotation[i];
	for (int i = 0; i < 3; ++i) { v.sunIlluminance[i] = d->sunIlluminance[i]; v.sunDirection[i] = d->sunDirection[i]; }
	// renderer.cc:191: if (sunIlluminance != vec3(0.0f))
	v.hasSun = (d->sunIlluminance[0] != 0.0f || d->sunIlluminance[1] != 0.0f || d->sunIlluminance[2] != 0.0f) ? 1u : 0u;
	sc->maxStackDepth = std::max(d->wideMaxStack, d->refMaxDepth);
	sc->materialTypeMask = d->materialTypeMask;
	sc->numLeaves = d->numLeaves;
	*outScene = sc;
	return 0;
fail:
	rt_scene_free(sc);
	return rc;
}

// A second device's copy of an uploaded scene, made over NVLink (cudaMemcpyPeer) instead of a second pass through host
// memory: Raylib_Render spreads a frame over all visible GPUs with the scene replicated on each (SURVEY 8e).
extern "C" int rt_scene_clone(const RtDeviceScene* src, int device, RtDeviceScene** outScene)
{
	*outScene = nullptr;
	if (!src) { g_lastError = "rt_scene_clone: null scene"; return -1; }
	RT_CUDA(cudaSetDevice(device));
	RtDeviceScene* sc = new RtDeviceScene(*src);
	sc->device = device;
	sc->allocations.clear();
	for (size_t i = 0; i < src->allocations.size(); ++i)
	{
		void* dev = nullptr;
		cudaError_t e = cudaMalloc(&dev, src->allocationBytes[i]);
		if (e == cudaSuccess) { sc->allocations.push_back(dev); e = cudaMemcpyPeer(dev, device, src->allocations[i], src->device, src->allocationBytes[i]); }
		if (e != cudaSuccess)
		{
			g_lastError = std::string("rt_scene_clone: ") + cudaGetErrorString(e);
			cudaGetLastError();
			rt_scene_free(sc);
			return (int)e;
		}
	}
	// every pointer of the view is the base address of one allocation: point it at the copy
	auto remap = [&](const void* p) -> const void*
	{
		for (size_t i = 0; i < src->allocations.size(); ++i) if (src->allocations[i] == p) return sc->allocations[i];
		return p;
	};
	RtSceneView& v = sc->view;
	#define RT_REMAP(field) v.field = reinterpret_cast<decltype(v.field)>(remap(v.field))
	RT_REMAP(nodes); RT_REMAP(refNodes); RT_REMAP(triHot); RT_REMAP(triCold); RT_REMAP(triRank); RT_REMAP(triGate); RT_REMAP(gateBoxes);
	RT_REMAP(spheres); RT_REMAP(sphereMaterial); RT_REMAP(sphereRank); RT_REMAP(sphereGate);
	RT_REMAP(cubes); RT_REMAP(cubeRank); RT_REMAP(cubeGate); RT_REMAP(materials); RT_REMAP(textures); RT_REMAP(texels);
	#undef RT_REMAP
	*outScene = sc;
	return 0;
}

extern "C" void rt_scene_free(RtDeviceScene* sc)
{
	if (!sc) return;
	cudaSetDevice(sc->device);
	for (void* p : sc->allocations) cudaFree(p);
	delete sc;
}

extern "C" uint64_t rt_scene_device_bytes(const RtDeviceScene* sc) { return sc ? sc->bytes : 0; }

extern "C" uint32_t rt_shard_tile_capacity(uint32_t width, uint32_t height, uint32_t shardCount)
{
	const uint32_t tilesX = (width + RT_TILE_W - 1) / RT_TILE_W, tilesY = (height + RT_TILE_H - 1) / RT_TILE_H;
	const uint32_t numTiles = tilesX * tilesY;
	shardCount = std::max(1u, shardCount);
	return (numTiles + shardCount - 1) / shardCount;
}

extern "C" int rt_context_create(int device, RtRenderContext** outCtx)
{
	*outCtx = nullptr;
	RT_CUDA(cudaSetDevice(device));
	RtRenderContext* ctx = new RtRenderContext;
	ctx->device = device;
	cudaDeviceProp prop;
	RT_CUDA(cudaGetDeviceProperties(&prop, device));
	ctx->numSMs = prop.multiProcessorCount;
	ctx->cooperative = prop.cooperativeLaunch != 0;
	for (RtPipe& pipe : ctx->pipe)
	{
		memset(&pipe.L, 0, sizeof(pipe.L));
		RT_CUDA(cudaMalloc((void**)&pipe.ctl, sizeof(RtQueueCtl)));
		RT_CUDA(cudaMemset(pipe.ctl, 0, sizeof(RtQueueCtl)));
		RT_CUDA(cudaStreamCreateWithFlags(&pipe.stream, cudaStreamNonBlocking));
		RT_CUDA(cudaEventCreateWithFlags(&pipe.evAccum, cudaEventDisableTiming));
		RT_CUDA(cudaEventCreateWithFlags(&pipe.evExtend, cudaEventDisableTiming));
	}
	RT_CUDA(cudaEventCreate(&ctx->evStart));
	RT_CUDA(cudaEventCreate(&ctx->evStop));
	RT_CUDA(cudaEventCreateWithFlags(&ctx->evFork, cudaEventDisableTiming));
	*outCtx = ctx;
	return 0;
}

static void free_arena(RtPipe& pipe)
{
	for (void* p : pipe.allocations) cudaFree(p);
	pipe.allocations.clear();
	pipe.capacity = 0; pipe.depthCapacity = 0;
}

extern "C" void rt_context_destroy(RtRenderContext* ctx)
{
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	for (RtPipe& pipe : ctx->pipe)
	{
		free_arena(pipe);
		if (pipe.ctl) cudaFree(pipe.ctl);
		if (pipe.poolStack) cudaFree(pipe.poolStack);
		if (pipe.stream) cudaStreamDestroy(pipe.stream);
		if (pipe.evAccum) cudaEventDestroy(pipe.evAccum);
		if (pipe.evExtend) cudaEventDestroy(pipe.evExtend);
		for (cudaEvent_t e : pipe.stageEvents) cudaEventDestroy(e);
	}
	if (ctx->accum) cudaFree(ctx->accum);
	if (ctx->evStart) cudaEventDestroy(ctx->evStart);
	if (ctx->evStop) cudaEventDestroy(ctx->evStop);
	if (ctx->evFork) cudaEventDestroy(ctx->evFork);
	delete ctx;
}

template<typename T>
static int arena_alloc(RtPipe& pipe, T** out, size_t count)
{
	void* p = nullptr;
	RT_CUDA(cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)));
	pipe.allocations.push_back(p);
	*out = reinterpret_cast<T*>(p);
	return 0;
}

#define RT_MAX_BINS (1u << 18)
// bytes of path state per slot at a given bounce-stack depth (everything ensure_arena allocates per slot)
static uint64_t arena_slot_bytes(int32_t depth)
{
#if RT_PACKED_STATE
	return 32ull * 2 /* ray hitCtl */ + 16ull * 2 /* Li missPartial */ + 32ull * (uint64_t)std::max(1, depth) /* stack */
	     + 4ull * (2 + RT_NUM_HIT_QUEUES + 1 + 2) /* extQ[2] matQ[] shadowQ extSorted extKey */;
#else
	return 16ull * 5 /* rayO rayD hit Li missPartial */ + 32ull * (uint64_t)std::max(1, depth) /* stackA stackB */
	     + 4ull * (1 + 2 + RT_NUM_HIT_QUEUES + 1 + 3) /* rngCtr extQ[2] matQ[] shadowQ slotKey extSorted extKey */;
#endif
}
static int ensure_arena(RtPipe& pipe, uint32_t slots, int32_t depth)
{
	if (slots <= pipe.capacity && depth <= pipe.depthCapacity) return 0;
	slots = std::max(slots, pipe.capacity); depth = std::max(std::max(depth, pipe.depthCapacity), 1);
	free_arena(pipe);
	RtLaunch& L = pipe.L;
	int rc;
#if RT_PACKED_STATE
	if ((rc = arena_alloc(pipe, &L.ray, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.hitCtl, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.stack, (size_t)slots * depth))) return rc;
#else
	if ((rc = arena_alloc(pipe, &L.rayO, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.rayD, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.hit, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.stackA, (size_t)slots * depth))) return rc;
	if ((rc = arena_alloc(pipe, &L.stackB, (size_t)slots * depth))) return rc;
#endif
	if ((rc = arena_alloc(pipe, &L.Li, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.missPartial, slots))) return rc;
#if !RT_PACKED_STATE
	if ((rc = arena_alloc(pipe, &L.rngCtr, slots))) return rc;
#endif
	for (int i = 0; i < 2; ++i) if ((rc = arena_alloc(pipe, &L.extQ[i], slots))) return rc;
	for (int i = 0; i < RT_NUM_HIT_QUEUES; ++i) if ((rc = arena_alloc(pipe, &L.matQ[i], slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.shadowQ, slots))) return rc;
#if !RT_PACKED_STATE
	if ((rc = arena_alloc(pipe, &L.slotKey, slots))) return rc;
#endif
	if ((rc = arena_alloc(pipe, &L.extSorted, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.extKey, slots))) return rc;
	if ((rc = arena_alloc(pipe, &L.binCount, RT_MAX_BINS))) return rc;
	if ((rc = arena_alloc(pipe, &L.binCursor, RT_MAX_BINS))) return rc;
	if ((rc = arena_alloc(pipe, &L.bounceCtl, (size_t)depth + 2))) return rc;      // + the next bounce's counter of the last shade stage + the fused pass's barrier
	RT_CUDA(cudaMemset(L.binCount, 0, RT_MAX_BINS * sizeof(uint32_t)));
	pipe.capacity = slots; pipe.depthCapacity = depth;
	return 0;
}

static int ensure_accum(RtRenderContext* ctx, uint32_t pixels)
{
	if (pixels <= ctx->pixCapacity && ctx->accum) return 0;
	if (ctx->accum) cudaFree(ctx->accum);
	ctx->accum = nullptr; ctx->pixCapacity = 0;
	RT_CUDA(cudaMalloc((void**)&ctx->accum, std::max<size_t>(pixels, 1) * sizeof(float4)));
	ctx->pixCapacity = pixels;
	return 0;
}

static uint32_t stack_levels(const RtDeviceScene* sc) { return std::max(8u, (sc->maxStackDepth + 2u + 3u) & ~3u); }
static bool stack_fits(uint32_t levels) { return levels <= RT_MAX_STACK; }

// Grid of a persistent kernel: resident CTAs per SM x SMs.  The occupancy query is made once per (context, kernel) -- a
// dozen of them per render call were a measurable part of millisecond frames.
template<typename Kernel>
static int persistent_grid(RtRenderContext* ctx, Kernel kernel, int blockSize, size_t smem, int* outGrid)
{
	const void* key = reinterpret_cast<const void*>(kernel);
	auto it = ctx->gridCache.find(key);
	if (it != ctx->gridCache.end()) { *outGrid = it->second; return 0; }
	int perSM = 0;
	if (smem > 48 * 1024) RT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	RT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kernel, blockSize, smem));
	*outGrid = ctx->numSMs * std::max(1, perSM);
	ctx->gridCache[key] = *outGrid;
	return 0;
}

static void fill_scene(RtLaunch& L, const RtDeviceScene* sc, const RtCamera* cam, const RtRenderParams* p, uint32_t stackLevels)
{
	L.S = sc->view;
	L.cam = *cam;
	L.seed = p->frameSeed;
	L.width = p->width; L.height = p->height;
	L.tilesX = (p->width + RT_TILE_W - 1) / RT_TILE_W;
	L.numTiles = L.tilesX * ((p->height + RT_TILE_H - 1) / RT_TILE_H);
	L.shardCount = std::max(1u, p->shardCount);
	L.shardRank = p->shardRank;
	L.npix = rt_shard_tile_capacity(p->width, p->height, L.shardCount) * RT_TILE_PIXELS;
	L.spp = (uint32_t)std::max(1, p->samplesPerPixel);
	L.maxDepth = p->maxPathLength;
	L.renderMode = p->renderMode;
	L.tMin = p->rayTMin;
	const RtTuning& tune = p->tuning;
	L.refillThreshold = tune.refillThreshold ? std::min(32u, tune.refillThreshold) : 20u;
	L.walkThreshold = tune.walkThreshold ? std::min(32u, tune.walkThreshold) : 20u;      // re-tuned after the hit record left the registers: 16 -> 20 is +1-2 % on scatter10M, neutral elsewhere (profiles/r02x)
	if (p->lightingOverride)
	{
		// the Scene's sun as it is NOW (renderer.cc:160-191 reads it on every miss); hasSun as in renderer.cc:191
		for (int i = 0; i < 3; ++i) { L.S.sunIlluminance[i] = p->sunIlluminance[i]; L.S.sunDirection[i] = p->sunDirection[i]; }
		L.S.hasSun = (p->sunIlluminance[0] != 0.0f || p->sunIlluminance[1] != 0.0f || p->sunIlluminance[2] != 0.0f) ? 1u : 0u;
	}
	// ray binning: RAYLIB_B200_BIN_OBITS origin bits, handed out one at a time to the axis whose cells are longest, and
	// RAYLIB_B200_BIN_DBITS bits per side of the octahedral direction map (numBins <= RT_MAX_BINS)
	uint32_t originBits = tune.binOriginBits >= 0 ? (uint32_t)std::min(18, tune.binOriginBits) : (sc->numLeaves >= RT_BIN_MIN_LEAVES ? RT_DEFAULT_BIN_OBITS : 0u);
	L.binDirBits = tune.binDirBits >= 0 ? (uint32_t)std::min(4, tune.binDirBits) : RT_DEFAULT_BIN_DBITS;
	if (originBits == 0u) L.binDirBits = 0u;
	while (originBits + 2u * L.binDirBits > 18u) { if (L.binDirBits > 1u) L.binDirBits--; else originBits--; }
	float cell[3];
	for (int i = 0; i < 3; ++i)
	{
		const float extent = sc->view.rootMax[i] - sc->view.rootMin[i];
		cell[i] = (extent > 0.0f && std::isfinite(extent)) ? extent : 0.0f;
		L.binAxisBits[i] = 0u;
		L.binOrigin[i] = sc->view.rootMin[i];
	}
	for (uint32_t b = 0; b < originBits; ++b)
	{
		const int axis = (cell[0] >= cell[1] && cell[0] >= cell[2]) ? 0 : (cell[1] >= cell[2] ? 1 : 2);
		L.binAxisBits[axis]++;
		cell[axis] *= 0.5f;
	}
	for (int i = 0; i < 3; ++i)
	{
		const float extent = sc->view.rootMax[i] - sc->view.rootMin[i];
		const float cells = (float)(1u << L.binAxisBits[i]);
		L.binScale[i] = (extent > 0.0f && std::isfinite(extent)) ? cells / extent : 0.0f;
		L.binTop[i] = cells - 1.0f;
	}
	L.binBits = originBits + 2u * L.binDirBits;
	L.numBins = L.binBits ? (1u << L.binBits) : 0u;
}

extern "C" int rt_render_shard(RtRenderContext* ctx, const RtDeviceScene* sc, const RtCamera* cam,
                               const RtRenderParams* p, void* deviceShardOut, void* streamPtr, RtRenderStats* stats)
{
	if (!p) { g_lastError = "rt_render_shard: null argument"; return -1; }
	return rt_render_window(ctx, sc, cam, p, 0u, (uint32_t)std::max(1, p->samplesPerPixel), nullptr, deviceShardOut, streamPtr, stats);
}

extern "C" int rt_render_window(RtRenderContext* ctx, const RtDeviceScene* sc, const RtCamera* cam, const RtRenderParams* params,
                                uint32_t sampleBegin, uint32_t sampleEnd, void* runningSum, void* deviceShardOut, void* streamPtr,
                                RtRenderStats* stats)
{
	if (!ctx || !sc || !cam || !params || (!deviceShardOut && !params->imageOut && !runningSum)) { g_lastError = "rt_render_shard: null argument"; return -1; }
	if (sampleBegin >= sampleEnd || sampleEnd > (uint32_t)INT32_MAX) { g_lastError = "rt_render_window: empty sample window"; return -1; }
	if (runningSum ? params->renderMode != 0u : sampleBegin != 0u)
	{
		g_lastError = "rt_render_window: a running sum needs path tracing, a window not starting at sample 0 a running sum";
		return -1;
	}
	// the window's end is the frame's sample count of the kernels (raygen skips samples >= spp); its length sizes the passes
	RtRenderParams windowParams = *params;
	windowParams.samplesPerPixel = (int32_t)sampleEnd;
	const RtRenderParams* p = &windowParams;
	if (p->imageOut && p->renderMode == RT_RENDERMODE_AUX) { g_lastError = "rt_render_shard: the fused denoiser-input pass writes shard buffers only"; return -1; }
	if (sc->device != ctx->device) { g_lastError = "rt_render_shard: scene and context live on different devices"; return -1; }
	if (p->width == 0 || p->height == 0) { g_lastError = "rt_render_shard: empty viewport"; return -1; }
	RT_CUDA(cudaSetDevice(ctx->device));
	cudaStream_t stream = (cudaStream_t)streamPtr;

	const uint32_t levels = stack_levels(sc);
	const size_t smem = 0;      // no dynamic shared memory: the traversal stack is thread-local
	if (!stack_fits(levels)) { g_lastError = "rt_render_shard: BVH too deep for the traversal stack"; return -1; }

	RtLaunch probe;
	memset(&probe, 0, sizeof(probe));
	fill_scene(probe, sc, cam, p, levels);
	const uint32_t npix = probe.npix, spp = probe.spp;
	const uint32_t win = spp - sampleBegin;      // samples per pixel this call renders
	const bool pathTrace = p->renderMode == 0u;
	if (p->renderMode == RT_RENDERMODE_AUX && !p->auxShardOut) { g_lastError = "rt_render_shard: RT_RENDERMODE_AUX needs auxShardOut"; return -1; }

	// Two pipes when there is more than one pass worth of samples: pass i runs on pipe i % 2, each pipe on its own stream.
	int pipes = p->pipes ? (int)std::min<uint32_t>(p->pipes, RT_MAX_PIPES) : p->tuning.pipes ? (int)std::min<uint32_t>(p->tuning.pipes, RT_MAX_PIPES) : RT_DEFAULT_PIPES;
	if (!pathTrace || p->collectStats) pipes = 1;

	// Small frames: the whole pass as one cooperative launch (k_pass_fused).  All samples of the frame are in flight at once,
	// one pipe, no ray binning (a few hundred thousand rays fit the L2 whatever their order).
	bool fused = false;
	if (pathTrace && !p->collectStats && !p->timeStages && !p->samplesPerPass && p->tuning.fusedPass != 1u && !p->tuning.pooledTraversal && ctx->cooperative)
	{
		const uint64_t limit = (uint64_t)(p->tuning.fusedPathsK ? p->tuning.fusedPathsK : RT_DEFAULT_FUSED_PATHS_K) << 10;
		const uint64_t paths = (uint64_t)win * npix;
		fused = p->tuning.fusedPass == 2u ? paths <= (32ull << 20) : paths <= limit;
	}
	if (fused) pipes = 1;

	// samples in flight per pixel and pass: enough paths to fill the machine, bounded by memory
	uint32_t K = 1;
	if (pathTrace)
	{
		// ~330 B of path state per slot at depth 8: 64 Mi paths = 21 GB of the 180 GB.  More paths in flight = fewer, fuller
		// launches (measured: +5 % on scatter10M, +10 % on grid1M going from 4 M to 32 M).
		const uint64_t targetPaths = (uint64_t)(p->tuning.pathsM ? p->tuning.pathsM : RT_DEFAULT_PATHS_M) << 20;
		const uint64_t perPass = std::max<uint64_t>(1, targetPaths / std::max(1u, npix));
		if (fused) K = win;
		else if (p->samplesPerPass) { K = std::min<uint32_t>(p->samplesPerPass, win); if (K >= win) pipes = 1; }
		else if (pipes > 1 && win >= 2u)
		{
			K = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, perPass / pipes), (win + pipes - 1) / pipes);
			// few samples per pixel: prefer two passes per pipe (more overlap) while a pass still fills the machine
			const uint32_t finer = (win + 2u * pipes - 1u) / (2u * pipes);
			if (finer < K && (uint64_t)finer * npix >= (4ull << 20)) K = finer;
		}
		else { K = (uint32_t)std::min<uint64_t>(perPass, win); pipes = 1; }
	}
	// path slots are 32-bit indices: never more than 2^31 paths in one pass, whatever the caller asks for
	if (pathTrace) K = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(K, (1ull << 31) / std::max(1u, npix)));
	// Never more path state than the device can hold next to the scene: a slot costs arena_slot_bytes(depth), so a frame with
	// a very long maxPathLength runs with fewer samples in flight instead of failing.  Asked only when an arena has to grow
	// (cudaMemGetInfo costs a fraction of a millisecond -- a third of a small frame).
	if (pathTrace)
	{
		bool grows = false;
		for (int q = 0; q < pipes; ++q)
			grows = grows || (uint64_t)K * npix > ctx->pipe[q].capacity || std::max(1, p->maxPathLength) > ctx->pipe[q].depthCapacity;
		size_t freeBytes = 0, totalBytes = 0;
		if (grows && cudaMemGetInfo(&freeBytes, &totalBytes) == cudaSuccess)
		{
			uint64_t held = 0;      // what the arenas hold now is released before they grow
			for (const RtPipe& pipe : ctx->pipe) held += (uint64_t)pipe.capacity * arena_slot_bytes(pipe.depthCapacity);
			const uint64_t budget = (uint64_t)((freeBytes + held) * 0.8);
			const uint64_t slotsPerPipe = budget / arena_slot_bytes(std::max(1, p->maxPathLength)) / (uint64_t)pipes;
			if ((uint64_t)K * npix > slotsPerPipe) K = (uint32_t)std::max<uint64_t>(1, slotsPerPipe / std::max(1u, npix));
		}
		else if (grows) cudaGetLastError();
	}
	uint32_t numPasses = pathTrace ? (win + K - 1) / K : 1u;
	if (numPasses < 2u) pipes = 1;

	int rc;
	if ((rc = ensure_accum(ctx, npix))) return rc;
	// path-state arenas; if the device cannot hold them after all (memory taken by another process since the estimate
	// above), halve the samples in flight and try again instead of failing the frame
	for (;;)
	{
		bool outOfMemory = false;
		for (int q = 0; q < pipes && !outOfMemory; ++q)
		{
			rc = ensure_arena(ctx->pipe[q], pathTrace ? K * npix : 32u, pathTrace ? std::max(1, p->maxPathLength) : 1);
			if (rc == (int)cudaErrorMemoryAllocation && pathTrace && K > 1u) outOfMemory = true;
			else if (rc) return rc;
		}
		if (!outOfMemory) break;
		for (RtPipe& pipe : ctx->pipe) free_arena(pipe);
		K = std::max(1u, K / 2u);
		numPasses = (win + K - 1) / K;
	}
	for (int q = 0; q < pipes; ++q)
	{
		RtPipe& pipe = ctx->pipe[q];
		RtLaunch& L = pipe.L;
		fill_scene(L, sc, cam, p, levels);
		L.capacity = pipe.capacity;
		L.K = K;
		L.accum = ctx->accum;
		L.out = reinterpret_cast<float4*>(deviceShardOut);
		L.image = reinterpret_cast<float4*>(runningSum ? runningSum : p->imageOut);
		L.runningSum = runningSum ? 1u : 0u;
		L.out2 = reinterpret_cast<float4*>(p->auxShardOut);
		L.ctl = pipe.ctl;
		if (fused) { L.binBits = 0; L.numBins = 0; }
	}
	// memory pressure may have cut the samples in flight: the fused pass wants them all at once
	if (fused && (K < win || numPasses != 1u)) fused = false;

	uint32_t launches = 0, passes = 0, extendLaunches[RT_MAX_PIPES] = { 0 };
	const bool timeStages = p->timeStages != 0 && stats != nullptr;
	for (int q = 0; q < pipes; ++q)
	{
		RT_CUDA(cudaMemsetAsync(ctx->pipe[q].ctl, 0, sizeof(RtQueueCtl), stream));
		// k_bin_scan leaves the histogram zeroed; clear it anyway so that a frame that died half-way cannot skew the next one
		if (pathTrace && ctx->pipe[q].L.numBins) RT_CUDA(cudaMemsetAsync(ctx->pipe[q].L.binCount, 0, ctx->pipe[q].L.numBins * sizeof(uint32_t), stream));
	}
	RT_CUDA(cudaEventRecord(ctx->evStart, stream));

	if (!pathTrace)
	{
		int grid = 0;
		if ((rc = persistent_grid(ctx, k_debug_view, 128, smem, &grid))) return rc;
		k_debug_view<<<grid, 128, smem, stream>>>(ctx->pipe[0].L);
		launches++;
	}
	if (pathTrace && fused)
	{
		RtPipe& pipe = ctx->pipe[0];
		RtLaunch& L = pipe.L;
		L.passBase = sampleBegin;
		int grid = 0;
		if ((rc = persistent_grid(ctx, k_pass_fused, 128, smem, &grid))) return rc;
		RT_CUDA(cudaMemsetAsync(L.bounceCtl, 0, ((size_t)std::max(0, p->maxPathLength) + 2) * sizeof(RtBounceCtl), stream));
		uint32_t materialMask = sc->materialTypeMask;
		int firstPass = 1, lastPass = 1;
		void* args[] = { (void*)&L, (void*)&materialMask, (void*)&firstPass, (void*)&lastPass };
		const cudaError_t e = cudaLaunchCooperativeKernel((const void*)k_pass_fused, dim3((unsigned)grid), dim3(128), args, smem, stream);
		if (e == cudaSuccess) { launches++; passes++; }
		else
		{
			// a device or a partition that will not co-schedule the grid (MIG slices, MPS limits): remember it and render this
			// frame -- one pass on one pipe, as sized above -- with the kernel-per-stage path below
			cudaGetLastError();
			ctx->cooperative = false;
			fused = false;
		}
	}
	if (pathTrace && !fused)
	{
		int gridExtend = 0, gridShadow = 0, gridMiss = 0, gridShade[RT_MAT_NUM_TYPES];
		const bool st = p->collectStats != 0;
		if (st) { if ((rc = persistent_grid(ctx, k_extend<true>, 128, smem, &gridExtend))) return rc; }
		else    { if ((rc = persistent_grid(ctx, k_extend<false>, 128, smem, &gridExtend))) return rc; }
		if ((rc = persistent_grid(ctx, k_shadow, 128, smem, &gridShadow))) return rc;
		if ((rc = persistent_grid(ctx, k_miss, 128, 0, &gridMiss))) return rc;
		if ((rc = persistent_grid(ctx, k_shade<RT_MAT_LAMBERTIAN>, 128, 0, &gridShade[RT_MAT_LAMBERTIAN]))) return rc;
		if ((rc = persistent_grid(ctx, k_shade<RT_MAT_METAL>, 128, 0, &gridShade[RT_MAT_METAL]))) return rc;
		if ((rc = persistent_grid(ctx, k_shade<RT_MAT_DIELECTRIC>, 128, 0, &gridShade[RT_MAT_DIELECTRIC]))) return rc;
		if ((rc = persistent_grid(ctx, k_shade<RT_MAT_MIRROR>, 128, 0, &gridShade[RT_MAT_MIRROR]))) return rc;
		if ((rc = persistent_grid(ctx, k_shade<RT_MAT_LIGHT>, 128, 0, &gridShade[RT_MAT_LIGHT]))) return rc;
		if ((rc = persistent_grid(ctx, k_shade<RT_MAT_MICROFACET>, 128, 0, &gridShade[RT_MAT_MICROFACET]))) return rc;
		// opt-in: the pooled traversal kernel (a warp regroups its rays at every step) instead of k_extend
		const bool pooled = p->tuning.pooledTraversal != 0 && !st;
		int gridPool = 0;
		if (pooled)
		{
			if ((rc = persistent_grid(ctx, k_extend_pool, 128, 0, &gridPool))) return rc;
			if (p->tuning.poolCtas) gridPool = std::min(gridPool, ctx->numSMs * (int)p->tuning.poolCtas);
			else if (pipes > 1) gridPool = std::min(gridPool, ctx->numSMs * (p->tuning.traversalCtas ? (int)p->tuning.traversalCtas : RT_DUAL_PIPE_TRAVERSAL_CTAS));
			const size_t entries = (size_t)gridPool * 4u * RT_MAX_STACK * RT_POOL_RAYS;
			for (int q = 0; q < pipes; ++q)
			{
				RtPipe& pipe = ctx->pipe[q];
				if (pipe.poolStackEntries < entries)
				{
					if (pipe.poolStack) cudaFree(pipe.poolStack);
					pipe.poolStack = nullptr; pipe.poolStackEntries = 0;
					RT_CUDA(cudaMalloc((void**)&pipe.poolStack, entries * sizeof(uint2)));
					pipe.poolStackEntries = entries;
				}
				pipe.L.poolStack = pipe.poolStack;
				pipe.L.poolNodeThreshold = p->tuning.poolNodeThreshold ? p->tuning.poolNodeThreshold : 24u;
				pipe.L.poolRefill = p->tuning.poolRefill ? p->tuning.poolRefill : 24u;
			}
		}
		if (pipes > 1)
		{
			// leave room on every SM for the other pipe's stage kernels while a traversal kernel is resident
			const int perSM = p->tuning.traversalCtas ? (int)p->tuning.traversalCtas : RT_DUAL_PIPE_TRAVERSAL_CTAS;
			gridExtend = std::min(gridExtend, ctx->numSMs * perSM);
			gridShadow = std::min(gridShadow, ctx->numSMs * perSM);
			RT_CUDA(cudaEventRecord(ctx->evFork, stream));
			for (int q = 0; q < pipes; ++q) RT_CUDA(cudaStreamWaitEvent(ctx->pipe[q].stream, ctx->evFork, 0));
		}

		// Passes are issued in groups of `pipes`, bounce by bounce across the group, so that cross-stream events can order
		// kernels of different pipes.  Extend ring (two or more pipes): the k_extend launches of the group run one after
		// the other -- each waits for the previous one in issue order -- instead of drifting into lock-step and sharing
		// the SMs with each other; what runs next to a traversal is then always the OTHER pipe's stage kernels (shade,
		// miss, shadow, binning), which is the overlap the pipes exist for.
		const bool ring = pipes > 1 && (p->tuning.extendRing != 0 || RT_DEFAULT_EXTEND_RING != 0);
		cudaEvent_t lastExtend = nullptr;
		for (uint32_t group = 0; group < numPasses; group += (uint32_t)pipes)
		{
			const int inGroup = (int)std::min<uint32_t>((uint32_t)pipes, numPasses - group);
			for (int q = 0; q < inGroup; ++q)
			{
				RtPipe& pipe = ctx->pipe[q];
				RtLaunch& L = pipe.L;
				cudaStream_t ps = pipes > 1 ? pipe.stream : stream;
				L.passBase = sampleBegin + (group + (uint32_t)q) * K;
				RT_CUDA(cudaMemsetAsync(L.bounceCtl, 0, ((size_t)std::max(0, p->maxPathLength) + 2) * sizeof(RtBounceCtl), ps));
				const uint32_t total = K * npix;
				k_raygen<<<std::min<uint32_t>((total + 255) / 256, (uint32_t)ctx->numSMs * 8u), 256, 0, ps>>>(L);
				launches++;
			}
			for (int b = 0; b < std::max(0, p->maxPathLength); ++b)
			for (int q = 0; q < inGroup; ++q)
			{
				RtPipe& pipe = ctx->pipe[q];
				RtLaunch& L = pipe.L;
				cudaStream_t ps = pipes > 1 ? pipe.stream : stream;
				uint32_t& ext = extendLaunches[q];
				if (ring && lastExtend) RT_CUDA(cudaStreamWaitEvent(ps, lastExtend, 0));
				if (timeStages)
				{
					while (pipe.stageEvents.size() < (size_t)(2 * (ext + 1)))
					{
						cudaEvent_t e; RT_CUDA(cudaEventCreate(&e)); pipe.stageEvents.push_back(e);
					}
					RT_CUDA(cudaEventRecord(pipe.stageEvents[2 * ext], ps));
				}
				if (st) k_extend<true><<<gridExtend, 128, smem, ps>>>(L, b);
				else if (pooled) k_extend_pool<<<gridPool, 128, 0, ps>>>(L, b);
				else    k_extend<false><<<gridExtend, 128, smem, ps>>>(L, b);
				if (timeStages) RT_CUDA(cudaEventRecord(pipe.stageEvents[2 * ext + 1], ps));
				if (ring) { RT_CUDA(cudaEventRecord(pipe.evExtend, ps)); lastExtend = pipe.evExtend; }
				ext++;
				launches++;
				const uint32_t mask = sc->materialTypeMask;
				if (mask & (1u << RT_MAT_LAMBERTIAN)) { k_shade<RT_MAT_LAMBERTIAN><<<gridShade[RT_MAT_LAMBERTIAN], 128, 0, ps>>>(L, b); launches++; }
				if (mask & (1u << RT_MAT_METAL))      { k_shade<RT_MAT_METAL><<<gridShade[RT_MAT_METAL], 128, 0, ps>>>(L, b); launches++; }
				if (mask & (1u << RT_MAT_DIELECTRIC)) { k_shade<RT_MAT_DIELECTRIC><<<gridShade[RT_MAT_DIELECTRIC], 128, 0, ps>>>(L, b); launches++; }
				if (mask & (1u << RT_MAT_MIRROR))     { k_shade<RT_MAT_MIRROR><<<gridShade[RT_MAT_MIRROR], 128, 0, ps>>>(L, b); launches++; }
				if (mask & (1u << RT_MAT_LIGHT))      { k_shade<RT_MAT_LIGHT><<<gridShade[RT_MAT_LIGHT], 128, 0, ps>>>(L, b); launches++; }
				if (mask & (1u << RT_MAT_MICROFACET)) { k_shade<RT_MAT_MICROFACET><<<gridShade[RT_MAT_MICROFACET], 128, 0, ps>>>(L, b); launches++; }
				k_miss<<<gridMiss, 128, 0, ps>>>(L, b);
				launches++;
				if (sc->view.hasSun) { k_shadow<<<gridShadow, 128, smem, ps>>>(L, b); launches++; }
				if (L.binBits && b + 1 < L.maxDepth)
				{
					k_bin_scan<<<1, 1024, 0, ps>>>(L.binCount, L.binCursor, L.numBins);
					k_bin_scatter<<<ctx->numSMs * 8, 256, 0, ps>>>(L, b);
					launches += 2;
				}
			}
			for (int q = 0; q < inGroup; ++q)
			{
				const uint32_t pass = group + (uint32_t)q;
				RtPipe& pipe = ctx->pipe[q];
				cudaStream_t ps = pipes > 1 ? pipe.stream : stream;
				// the per-pixel sums are taken in sample order (renderer.cc:244-246): pass i's accumulate waits for pass i-1's
				if (pipes > 1 && pass > 0) RT_CUDA(cudaStreamWaitEvent(ps, ctx->pipe[(pass - 1) % (uint32_t)pipes].evAccum, 0));
				k_accumulate<<<(npix + 255) / 256, 256, 0, ps>>>(pipe.L, pass == 0, pass + 1 == numPasses);
				if (pipes > 1) RT_CUDA(cudaEventRecord(pipe.evAccum, ps));
				launches++;
				passes++;
			}
		}
		// join: the last accumulate is ordered after every earlier one, and each pipe's kernels precede its accumulates
		if (pipes > 1) RT_CUDA(cudaStreamWaitEvent(stream, ctx->pipe[(numPasses - 1) % (uint32_t)pipes].evAccum, 0));
	}
	RT_CUDA(cudaEventRecord(ctx->evStop, stream));
	RT_CUDA(cudaGetLastError());

	if (stats)
	{
		RT_CUDA(cudaStreamSynchronize(stream));
		memset(stats, 0, sizeof(*stats));
		for (int q = 0; q < pipes; ++q)
		{
			RtQueueCtl h;
			RT_CUDA(cudaMemcpy(&h, ctx->pipe[q].ctl, sizeof(h), cudaMemcpyDeviceToHost));
			stats->rayQueries += h.rayQueries;
			stats->boxTests += h.boxTests; stats->triTests += h.triTests; stats->sphereTests += h.sphereTests; stats->nodeVisits += h.nodeVisits;
			stats->gateTests += h.gateTests; stats->cubeTests += h.cubeTests;
			stats->refBoxTests += h.refBoxTests; stats->refTriTests += h.refTriTests; stats->refSphereTests += h.refSphereTests;
			stats->statRays += h.statRays;
			stats->nodeIters += h.nodeIters; stats->nodeStep += h.nodeStep; stats->nodeAlive += h.nodeAlive;
			stats->leafIters += h.leafIters; stats->leafBusy += h.leafBusy;
			stats->extendLaunches += extendLaunches[q];
			if (timeStages)
			{
				// sum of the launch durations; with two pipes launches of different passes overlap in time
				double perBounce[RT_MAX_BOUNCE_STATS] = { 0.0 };
				const uint32_t depth = (uint32_t)std::max(1, p->maxPathLength);
				for (uint32_t i = 0; i < extendLaunches[q]; ++i)
				{
					float e = 0.0f;
					RT_CUDA(cudaEventElapsedTime(&e, ctx->pipe[q].stageEvents[2 * i], ctx->pipe[q].stageEvents[2 * i + 1]));
					stats->extendMs += e;
					perBounce[std::min<uint32_t>(i % depth, RT_MAX_BOUNCE_STATS - 1)] += e;
				}
				if (p->tuning.dumpTimeline)     // development: when every k_extend launch ran, relative to the frame start
					for (uint32_t i = 0; i < extendLaunches[q]; ++i)
					{
						float t0 = 0.0f, t1 = 0.0f;
						RT_CUDA(cudaEventElapsedTime(&t0, ctx->evStart, ctx->pipe[q].stageEvents[2 * i]));
						RT_CUDA(cudaEventElapsedTime(&t1, ctx->evStart, ctx->pipe[q].stageEvents[2 * i + 1]));
						fprintf(stderr, "[timeline] pipe %d launch %u bounce %u: %.3f .. %.3f ms\n", q, i, i % depth, t0, t1);
					}
				if (p->tuning.dumpBounces)      // development: k_extend time and rays per bounce
					for (uint32_t b = 0; b < std::min<uint32_t>(depth, RT_MAX_BOUNCE_STATS); ++b)
						fprintf(stderr, "[bounce] pipe %d bounce %u: %llu rays, k_extend %.3f ms, %.1f Mrays/s\n", q, b,
						        (unsigned long long)h.bounceRays[b], perBounce[b], perBounce[b] > 0.0 ? h.bounceRays[b] / perBounce[b] / 1e3 : 0.0);
			}
		}
		float ms = 0.0f;
		RT_CUDA(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evStop));
		stats->deviceMs = ms;
		stats->kernelLaunches = launches;
		stats->passes = passes;
		// pixels of this shard that lie inside the image
		uint64_t px = 0;
		const uint32_t tilesX = probe.tilesX;
		for (uint32_t t = probe.shardRank; t < probe.numTiles; t += probe.shardCount)
		{
			const uint32_t tx = t % tilesX, ty = t / tilesX;
			const uint32_t w = std::min<uint32_t>(RT_TILE_W, p->width - tx * RT_TILE_W), hgt = std::min<uint32_t>(RT_TILE_H, p->height - ty * RT_TILE_H);
			px += (uint64_t)w * hgt;
			stats->tilesRendered++;
		}
		stats->pixelSamples = px * (pathTrace ? win : 1u);
	}
	return 0;
}

extern "C" int rt_assemble(int device, const void* deviceShards, uint32_t shardCount, uint32_t width, uint32_t height,
                           void* deviceImageOut, void* streamPtr)
{
	RT_CUDA(cudaSetDevice(device));
	const uint32_t cap = rt_shard_tile_capacity(width, height, shardCount);
	const uint32_t n = width * height;
	k_assemble<<<(n + 255) / 256, 256, 0, (cudaStream_t)streamPtr>>>(reinterpret_cast<const float4*>(deviceShards), std::max(1u, shardCount), cap,
		width, height, reinterpret_cast<float4*>(deviceImageOut));
	RT_CUDA(cudaGetLastError());
	return 0;
}

extern "C" int rt_trace_closest(RtRenderContext* ctx, const RtDeviceScene* sc, const float* hostRays, int64_t numRays,
                                float tMin, int32_t* hostOutRank, float* hostOutT, RtRenderStats* stats)
{
	if (!ctx || !sc) { g_lastError = "rt_trace_closest: null argument"; return -1; }
	RT_CUDA(cudaSetDevice(ctx->device));
	if (numRays <= 0) return 0;
	float4* dRays = nullptr; int32_t* dRank = nullptr; float* dT = nullptr;
	struct Scratch      // frees the three buffers on every return path (RT_CUDA returns early on errors)
	{
		float4*& rays; int32_t*& rank; float*& t;
		~Scratch() { cudaFree(rays); cudaFree(rank); cudaFree(t); }
	} scratch{ dRays, dRank, dT };
	RT_CUDA(cudaMalloc((void**)&dRays, (size_t)numRays * 32));
	RT_CUDA(cudaMalloc((void**)&dRank, (size_t)numRays * 4));
	RT_CUDA(cudaMalloc((void**)&dT, (size_t)numRays * 4));
	RT_CUDA(cudaMemcpy(dRays, hostRays, (size_t)numRays * 32, cudaMemcpyHostToDevice));
	RtQueueCtl* ctl = ctx->pipe[0].ctl;
	RT_CUDA(cudaMemset(ctl, 0, sizeof(RtQueueCtl)));
	const uint32_t levels = stack_levels(sc);
	const size_t smem = 0;      // no dynamic shared memory: the traversal stack is thread-local
	if (!stack_fits(levels)) { g_lastError = "rt_trace_closest: BVH too deep for the traversal stack"; return -1; }
	int grid = 0, rc;
	const bool st = stats != nullptr;
	if (st) { if ((rc = persistent_grid(ctx, k_trace_rays<true>, 128, smem, &grid))) return rc; }
	else    { if ((rc = persistent_grid(ctx, k_trace_rays<false>, 128, smem, &grid))) return rc; }
	grid = (int)std::min<int64_t>(grid, (numRays + 127) / 128);
	RT_CUDA(cudaEventRecord(ctx->evStart, 0));
	if (st) k_trace_rays<true><<<grid, 128, smem>>>(sc->view, dRays, numRays, tMin, dRank, dT, ctl);
	else    k_trace_rays<false><<<grid, 128, smem>>>(sc->view, dRays, numRays, tMin, dRank, dT, ctl);
	RT_CUDA(cudaEventRecord(ctx->evStop, 0));
	RT_CUDA(cudaGetLastError());
	RT_CUDA(cudaMemcpy(hostOutRank, dRank, (size_t)numRays * 4, cudaMemcpyDeviceToHost));
	RT_CUDA(cudaMemcpy(hostOutT, dT, (size_t)numRays * 4, cudaMemcpyDeviceToHost));
	if (stats)
	{
		RtQueueCtl h;
		RT_CUDA(cudaMemcpy(&h, ctl, sizeof(h), cudaMemcpyDeviceToHost));
		float ms = 0.0f;
		RT_CUDA(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evStop));
		memset(stats, 0, sizeof(*stats));
		stats->rayQueries = (uint64_t)numRays;
		stats->boxTests = h.boxTests; stats->triTests = h.triTests; stats->sphereTests = h.sphereTests; stats->nodeVisits = h.nodeVisits;
		stats->gateTests = h.gateTests; stats->cubeTests = h.cubeTests;
		stats->refBoxTests = h.refBoxTests; stats->refTriTests = h.refTriTests; stats->refSphereTests = h.refSphereTests;
		stats->statRays = (uint64_t)numRays;
		stats->deviceMs = ms;
		stats->kernelLaunches = 1;
	}
	return 0;
}

// ---- the traversal stage kernels of a render on caller rays (parity tests, rt_trace_stage.h) --------------------------
// One of k_extend / k_extend_pool / k_shadow at bounce 0 on an arena prepared by hand: the caller's rays in the path
// records, the caller's order as the queue.
extern "C" int rt_trace_stage(RtRenderContext* ctx, const RtDeviceScene* sc, int mode, const float* hostRays, const uint32_t* hostOrder,
                              int64_t numRays, float tMin, const float* sunDirection, const RtStageSchedule* schedule,
                              int32_t* hostOutQueue, float* hostOutHit, uint32_t* hostOutQueueCounts, RtRenderStats* stats)
{
	if (!ctx || !sc || !hostRays || !hostOrder || !schedule || !hostOutQueue || !hostOutHit) { g_lastError = "rt_trace_stage: null argument"; return -1; }
	if (mode < RT_STAGE_EXTEND || mode > RT_STAGE_SHADOW) { g_lastError = "rt_trace_stage: unknown mode"; return -1; }
	if (mode == RT_STAGE_SHADOW && !sunDirection) { g_lastError = "rt_trace_stage: the any-hit mode needs a sun direction"; return -1; }
	if (numRays <= 0 || numRays >= ((int64_t)1 << 31)) { g_lastError = "rt_trace_stage: the ray count must be in [1, 2^31)"; return -1; }
	if (sc->device != ctx->device) { g_lastError = "rt_trace_stage: scene and context live on different devices"; return -1; }
	const uint32_t n = (uint32_t)numRays;
	{
		// the kernels index the path records with the queue's entries: anything but a permutation would address outside them
		std::vector<uint8_t> seen(n, 0);
		for (uint32_t i = 0; i < n; ++i)
		{
			if (hostOrder[i] >= n || seen[hostOrder[i]]) { g_lastError = "rt_trace_stage: the order is not a permutation of the rays"; return -1; }
			seen[hostOrder[i]] = 1;
		}
	}
#if !RT_PACKED_STATE
	g_lastError = "rt_trace_stage: needs the packed path-state layout (RT_PACKED_STATE 1)";
	return -1;
#else
	RT_CUDA(cudaSetDevice(ctx->device));
	const uint32_t levels = stack_levels(sc);
	if (!stack_fits(levels)) { g_lastError = "rt_trace_stage: BVH too deep for the traversal stack"; return -1; }
	RtPipe& pipe = ctx->pipe[0];
	int rc;
	if ((rc = ensure_arena(pipe, n, 1))) return rc;

	// one bounce of a 1 x 1 frame: no pixels are touched, only the scene, tMin and the scheduling thresholds matter
	RtRenderParams p;
	memset(&p, 0, sizeof(p));
	p.width = 1; p.height = 1; p.samplesPerPixel = 1; p.maxPathLength = 1; p.rayTMin = tMin; p.shardCount = 1;
	p.tuning.refillThreshold = schedule->refillThreshold;
	p.tuning.walkThreshold = schedule->walkThreshold;
	p.tuning.binOriginBits = 0; p.tuning.binDirBits = 0;      // no ray binning (bounce 0 reads extQ[0] either way)
	RtCamera cam;
	memset(&cam, 0, sizeof(cam));
	RtLaunch L = pipe.L;         // the arena's pointers
	fill_scene(L, sc, &cam, &p, levels);
	L.capacity = pipe.capacity;
	L.K = 1;
	L.ctl = pipe.ctl;
	L.accum = nullptr; L.out = nullptr; L.image = nullptr; L.out2 = nullptr; L.runningSum = 0u;
	if (mode == RT_STAGE_SHADOW)
	{
		// a sun of illuminance 1 and no sky term: a path's radiance is (1, 1, 1) if its sun ray is unoccluded, 0 otherwise
		for (int i = 0; i < 3; ++i) { L.S.sunDirection[i] = sunDirection[i]; L.S.sunIlluminance[i] = 1.0f; }
		L.S.hasSun = 1u;
	}

	int grid = 0;
	const size_t smem = 0;
	if (mode == RT_STAGE_EXTEND) rc = persistent_grid(ctx, k_extend<false>, 128, smem, &grid);
	else if (mode == RT_STAGE_EXTEND_STATS) rc = persistent_grid(ctx, k_extend<true>, 128, smem, &grid);
	else if (mode == RT_STAGE_EXTEND_POOL) rc = persistent_grid(ctx, k_extend_pool, 128, 0, &grid);
	else rc = persistent_grid(ctx, k_shadow, 128, smem, &grid);
	if (rc) return rc;
	if (schedule->gridCtas) grid = (int)schedule->gridCtas;
	if (mode == RT_STAGE_EXTEND_POOL)
	{
		const size_t entries = (size_t)grid * 4u * RT_MAX_STACK * RT_POOL_RAYS;
		if (pipe.poolStackEntries < entries)
		{
			if (pipe.poolStack) cudaFree(pipe.poolStack);
			pipe.poolStack = nullptr; pipe.poolStackEntries = 0;
			RT_CUDA(cudaMalloc((void**)&pipe.poolStack, entries * sizeof(uint2)));
			pipe.poolStackEntries = entries;
		}
		pipe.L.poolStack = pipe.poolStack;
		L.poolStack = pipe.poolStack;
		L.poolNodeThreshold = schedule->poolNodeThreshold ? schedule->poolNodeThreshold : 24u;
		L.poolRefill = schedule->poolRefill ? schedule->poolRefill : 24u;
	}

	// the rays into the path records ({o.xyz, time | d.xyz, -}, the caller's layout), the order into the queue the kernel
	// drains, its counter set and every other counter of the bounce block zeroed; hit records, radiance and the output
	// queues start as all-ones sentinels, so that a slot the kernel never wrote is seen as such
	uint32_t* const queueIn = mode == RT_STAGE_SHADOW ? L.shadowQ : L.extQ[0];
	RT_CUDA(cudaMemcpy(L.ray, hostRays, (size_t)n * sizeof(RtF8), cudaMemcpyHostToDevice));
	RT_CUDA(cudaMemcpy(queueIn, hostOrder, (size_t)n * 4, cudaMemcpyHostToDevice));
	RT_CUDA(cudaMemset(L.bounceCtl, 0, ((size_t)pipe.depthCapacity + 2) * sizeof(RtBounceCtl)));
	RtBounceCtl bc;
	memset(&bc, 0, sizeof(bc));
	if (mode == RT_STAGE_SHADOW) bc.shadowCount = n; else bc.extCount = n;
	RT_CUDA(cudaMemcpy(L.bounceCtl, &bc, sizeof(bc), cudaMemcpyHostToDevice));
	RT_CUDA(cudaMemset(L.hitCtl, 0xFF, (size_t)n * sizeof(RtF8)));
	RT_CUDA(cudaMemset(L.Li, 0xFF, (size_t)n * sizeof(float4)));
	RT_CUDA(cudaMemset(L.missPartial, 0, (size_t)n * sizeof(float4)));
	for (int k = 0; k < RT_NUM_HIT_QUEUES; ++k) RT_CUDA(cudaMemset(L.matQ[k], 0xFF, (size_t)n * 4));
	RT_CUDA(cudaMemset(pipe.ctl, 0, sizeof(RtQueueCtl)));

	RT_CUDA(cudaEventRecord(ctx->evStart, 0));
	if (mode == RT_STAGE_EXTEND) k_extend<false><<<grid, 128, smem>>>(L, 0);
	else if (mode == RT_STAGE_EXTEND_STATS) k_extend<true><<<grid, 128, smem>>>(L, 0);
	else if (mode == RT_STAGE_EXTEND_POOL) k_extend_pool<<<grid, 128, 0>>>(L, 0);
	else k_shadow<<<grid, 128, smem>>>(L, 0);
	RT_CUDA(cudaEventRecord(ctx->evStop, 0));
	RT_CUDA(cudaGetLastError());
	RT_CUDA(cudaDeviceSynchronize());

	if (hostOutQueueCounts) memset(hostOutQueueCounts, 0, RT_NUM_HIT_QUEUES * sizeof(uint32_t));
	if (mode == RT_STAGE_SHADOW)
	{
		std::vector<float4> li(n);
		RT_CUDA(cudaMemcpy(li.data(), L.Li, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost));
		for (uint32_t i = 0; i < n; ++i)
		{
			const float4 v = li[i];
			memcpy(hostOutHit + 4 * (size_t)i, &v, sizeof(v));
			const bool visible = v.x == 1.0f && v.y == 1.0f && v.z == 1.0f && v.w == 0.0f;
			const bool occluded = v.x == 0.0f && v.y == 0.0f && v.z == 0.0f && v.w == 0.0f;
			hostOutQueue[i] = visible ? 0 : occluded ? 1 : -1;
		}
	}
	else
	{
		RtBounceCtl done;
		RT_CUDA(cudaMemcpy(&done, L.bounceCtl, sizeof(done), cudaMemcpyDeviceToHost));
		std::vector<RtF8> rec(n);
		RT_CUDA(cudaMemcpy(rec.data(), L.hitCtl, (size_t)n * sizeof(RtF8), cudaMemcpyDeviceToHost));
		for (uint32_t i = 0; i < n; ++i)
		{
			memcpy(hostOutHit + 4 * (size_t)i, &rec[i].lo, sizeof(float4));
			hostOutQueue[i] = -1;
		}
		std::vector<uint32_t> q;
		for (int k = 0; k < RT_NUM_HIT_QUEUES; ++k)
		{
			if (hostOutQueueCounts) hostOutQueueCounts[k] = done.matCount[k];
			q.resize(std::min(done.matCount[k], n));        // a counter above n fails the caller's sum check on its own
			if (!q.empty()) RT_CUDA(cudaMemcpy(q.data(), L.matQ[k], q.size() * 4, cudaMemcpyDeviceToHost));
			for (uint32_t s : q)
				if (s < n) hostOutQueue[s] = hostOutQueue[s] == -1 ? k : -2;
		}
	}
	if (stats)
	{
		RtQueueCtl h;
		RT_CUDA(cudaMemcpy(&h, pipe.ctl, sizeof(h), cudaMemcpyDeviceToHost));
		float ms = 0.0f;
		RT_CUDA(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evStop));
		memset(stats, 0, sizeof(*stats));
		stats->rayQueries = n;
		stats->boxTests = h.boxTests; stats->triTests = h.triTests; stats->sphereTests = h.sphereTests; stats->nodeVisits = h.nodeVisits;
		stats->gateTests = h.gateTests; stats->cubeTests = h.cubeTests;
		stats->refBoxTests = h.refBoxTests; stats->refTriTests = h.refTriTests; stats->refSphereTests = h.refSphereTests;
		stats->statRays = h.statRays;
		stats->nodeIters = h.nodeIters; stats->nodeStep = h.nodeStep; stats->nodeAlive = h.nodeAlive;
		stats->leafIters = h.leafIters; stats->leafBusy = h.leafBusy;
		stats->deviceMs = ms;
		stats->kernelLaunches = 1;
		stats->extendLaunches = mode == RT_STAGE_SHADOW ? 0u : 1u;
	}
	return 0;
#endif
}

// ---- Image2D::PostProcess on the device (render/image.cc:44-103) -----------------------------------------

// Luminance is never negative where it matters (the maximum starts at 1.0), so the float order equals the order of
// the bit patterns and one atomicMax per block on the raw bits is exact.
__global__ void __launch_bounds__(256) k_max_luminance(const float4* image, uint32_t count, uint32_t* maxBits)
{
	float m = 1.0f;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x)
	{
		const float lum = luminance3(xyz(image[i]));
		if (m < lum) m = lum;
	}
	for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
	__shared__ float warpMax[8];
	if ((threadIdx.x & 31u) == 0) warpMax[threadIdx.x >> 5] = m;
	__syncthreads();
	if (threadIdx.x < 8)
	{
		m = warpMax[threadIdx.x];
		for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFu, m, o));
		if (threadIdx.x == 0) atomicMax(maxBits, __float_as_uint(m));
	}
}

__global__ void __launch_bounds__(256) k_tonemap(float4* image, uint32_t count, const uint32_t* maxBits, uint32_t* outArgb8)
{
	const float maxWhite = __uint_as_float(*maxBits);
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x)
	{
		float4 px = image[i];
		float3 rgb = xyz(px);
		const float lumOld = luminance3(rgb);
		if (lumOld <= 0.0001f) rgb = v3(0.0f);
		else
		{
			const float numerator = lumOld * (1.0f + (lumOld / (maxWhite * maxWhite)));
			const float lumNew = numerator / (1.0f + lumOld);
			rgb = rgb * (lumNew / lumOld);
		}
		rgb = v3(fminf(1.0f, rgb.x), fminf(1.0f, rgb.y), fminf(1.0f, rgb.z));
		const float g = 1.0f / 2.2f;
		rgb = v3(rt_m_powf(rgb.x, g), rt_m_powf(rgb.y, g), rt_m_powf(rgb.z, g));
		px.x = rgb.x; px.y = rgb.y; px.z = rgb.z;
		image[i] = px;
		if (outArgb8)
		{
			const uint32_t A = (uint32_t)(px.w * 255.0f) & 0xffu, R = (uint32_t)(px.x * 255.0f) & 0xffu;
			const uint32_t G = (uint32_t)(px.y * 255.0f) & 0xffu, B = (uint32_t)(px.z * 255.0f) & 0xffu;
			outArgb8[i] = (A << 24) | (R << 16) | (G << 8) | B;
		}
	}
}

extern "C" int rt_postprocess(int device, void* deviceImage, uint32_t width, uint32_t height, uint32_t* deviceOutArgb8,
                              float* hostOutMaxWhite, void* streamPtr)
{
	if (!deviceImage || width == 0 || height == 0) { g_lastError = "rt_postprocess: empty image"; return -1; }
	RT_CUDA(cudaSetDevice(device));
	cudaStream_t stream = (cudaStream_t)streamPtr;
	cudaDeviceProp prop;
	RT_CUDA(cudaGetDeviceProperties(&prop, device));
	uint32_t* maxBits = nullptr;
	RT_CUDA(cudaMallocAsync((void**)&maxBits, 4, stream));
	const float one = 1.0f;
	RT_CUDA(cudaMemcpyAsync(maxBits, &one, 4, cudaMemcpyHostToDevice, stream));
	const uint32_t count = width * height;
	const int grid = (int)std::min<uint32_t>((count + 255u) / 256u, (uint32_t)prop.multiProcessorCount * 8u);
	k_max_luminance<<<grid, 256, 0, stream>>>(reinterpret_cast<const float4*>(deviceImage), count, maxBits);
	k_tonemap<<<grid, 256, 0, stream>>>(reinterpret_cast<float4*>(deviceImage), count, maxBits, deviceOutArgb8);
	RT_CUDA(cudaGetLastError());
	if (hostOutMaxWhite)
	{
		RT_CUDA(cudaMemcpyAsync(hostOutMaxWhite, maxBits, 4, cudaMemcpyDeviceToHost, stream));
		RT_CUDA(cudaStreamSynchronize(stream));
	}
	RT_CUDA(cudaFreeAsync(maxBits, stream));
	return 0;
}

// ---- progressive rendering: resolve of a running sum, scene fingerprint (rt_progressive.h) ------------------------------
// One pixel per thread; the noise figure's sum is reduced by a fixed tree in each block and the blocks are added in index
// order on the host, so the same sums give the same double every time.
__global__ void __launch_bounds__(256) k_resolve(const float4* sums, uint32_t count, float n, float4* image, float* noise, double* blockSums)
{
	__shared__ double part[256];
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	double rel = 0.0;
	if (i < count)
	{
		const float4 s = sums[i];
		if (image)
		{
			const float3 a = div_assign3(xyz(s), n);      // the last pass of a one-shot frame of n samples
			image[i] = make_float4(a.x, a.y, a.z, 1.0f);
		}
		if (noise || blockSums)
		{
			// relative standard error of the mean luminance: sqrt(var / n) / mean, var the unbiased sample variance
			const float m = luminance3(xyz(s)) / n;
			const float var = fmaxf(0.0f, (s.w - n * m * m) / (n - 1.0f));
			const float r = sqrtf(var / n) / fmaxf(m, 1e-4f);
			if (noise) noise[i] = r;
			rel = r;
		}
	}
	if (!blockSums) return;
	part[threadIdx.x] = rel;
	__syncthreads();
	for (uint32_t half = blockDim.x / 2u; half > 0u; half >>= 1)
	{
		if (threadIdx.x < half) part[threadIdx.x] += part[threadIdx.x + half];
		__syncthreads();
	}
	if (threadIdx.x == 0) blockSums[blockIdx.x] = part[0];
}

extern "C" int rt_resolve(int device, const void* sums, uint32_t count, uint32_t n, void* deviceImageOut, float* deviceNoiseOut,
                          double* hostNoiseSum, void* streamPtr)
{
	if (!sums || count == 0 || n == 0) { g_lastError = "rt_resolve: empty accumulator"; return -1; }
	if ((deviceNoiseOut || hostNoiseSum) && n < 2) { g_lastError = "rt_resolve: the noise figure needs at least 2 samples"; return -1; }
	RT_CUDA(cudaSetDevice(device));
	cudaStream_t stream = (cudaStream_t)streamPtr;
	const uint32_t blocks = (count + 255u) / 256u;
	double* blockSums = nullptr;
	if (hostNoiseSum) RT_CUDA(cudaMallocAsync((void**)&blockSums, blocks * sizeof(double), stream));
	k_resolve<<<blocks, 256, 0, stream>>>(reinterpret_cast<const float4*>(sums), count, (float)n,
	                                      reinterpret_cast<float4*>(deviceImageOut), deviceNoiseOut, blockSums);
	RT_CUDA(cudaGetLastError());
	if (hostNoiseSum)
	{
		std::vector<double> host(blocks);
		RT_CUDA(cudaMemcpyAsync(host.data(), blockSums, blocks * sizeof(double), cudaMemcpyDeviceToHost, stream));
		RT_CUDA(cudaFreeAsync(blockSums, stream));
		RT_CUDA(cudaStreamSynchronize(stream));
		double total = 0.0;
		for (double b : host) total += b;
		*hostNoiseSum = total;
	}
	else RT_CUDA(cudaStreamSynchronize(stream));
	return 0;
}

// Each thread hashes one RT_HASH_CHUNK-byte chunk with RtChecksum (allocations are 256-byte aligned, so the words are
// aligned 8-byte loads); the host combines the chunk values in order.
#define RT_HASH_CHUNK 4096u
__global__ void __launch_bounds__(256) k_hash_chunks(const unsigned char* data, uint64_t bytes, uint64_t* chunkHash)
{
	const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint64_t begin = c * RT_HASH_CHUNK;
	if (begin >= bytes) return;
	const uint64_t len = bytes - begin < RT_HASH_CHUNK ? bytes - begin : RT_HASH_CHUNK;
	const uint64_t* words = reinterpret_cast<const uint64_t*>(data + begin);
	RtChecksum sum;
	uint64_t i = 0;
	for (; i + 8u <= len; i += 8u) sum.Mix(words[i / 8u]);
	if (i < len)
	{
		uint64_t w = 0;
		for (uint64_t b = i; b < len; ++b) w |= (uint64_t)data[begin + b] << (8u * (b - i));
		sum.Mix(w);
	}
	sum.Mix(len);
	chunkHash[c] = sum.h;
}

extern "C" int rt_scene_fingerprint(const RtDeviceScene* sc, uint64_t* out)
{
	if (!sc || !out) { g_lastError = "rt_scene_fingerprint: null argument"; return -1; }
	RT_CUDA(cudaSetDevice(sc->device));
	RtChecksum sum;
	uint64_t* chunkHash = nullptr;
	size_t capacity = 0;
	std::vector<uint64_t> host;
	int rc = 0;
	for (size_t a = 0; a < sc->allocations.size() && rc == 0; ++a)
	{
		if (sc->allocations[a] == (const void*)sc->view.refNodes) continue;      // statistics frames only
		const uint64_t bytes = sc->contentBytes[a];
		const uint64_t chunks = (bytes + RT_HASH_CHUNK - 1u) / RT_HASH_CHUNK;
		sum.Mix(bytes);
		if (!chunks) continue;
		if (chunks > capacity)
		{
			if (chunkHash) cudaFree(chunkHash);
			chunkHash = nullptr; capacity = 0;
			cudaError_t e = cudaMalloc((void**)&chunkHash, chunks * sizeof(uint64_t));
			if (e != cudaSuccess) { g_lastError = std::string("rt_scene_fingerprint: ") + cudaGetErrorString(e); cudaGetLastError(); rc = (int)e; break; }
			capacity = chunks;
		}
		k_hash_chunks<<<(unsigned)((chunks + 255u) / 256u), 256>>>(reinterpret_cast<const unsigned char*>(sc->allocations[a]), bytes, chunkHash);
		host.resize(chunks);
		cudaError_t e = cudaMemcpy(host.data(), chunkHash, chunks * sizeof(uint64_t), cudaMemcpyDeviceToHost);
		if (e != cudaSuccess) { g_lastError = std::string("rt_scene_fingerprint: ") + cudaGetErrorString(e); cudaGetLastError(); rc = (int)e; break; }
		for (uint64_t h : host) sum.Mix(h);
	}
	if (chunkHash) cudaFree(chunkHash);
	if (rc) return rc;
	// the scalars of the view that decide the image (pointers differ per upload; the sun is a per-frame value)
	const RtSceneView& v = sc->view;
	sum.Add(v.rootMin, sizeof(v.rootMin)); sum.Add(v.rootMax, sizeof(v.rootMax)); sum.Mix(v.rootRef);
	sum.Add(v.refRootMin, sizeof(v.refRootMin)); sum.Add(v.refRootMax, sizeof(v.refRootMax)); sum.Mix(v.refRootRef); sum.Mix(v.refRootBoxTests);
	sum.Mix(v.flags); sum.Mix((uint32_t)v.skyTexture); sum.Add(v.skyRotation, sizeof(v.skyRotation));
	sum.Mix(sc->maxStackDepth); sum.Mix(sc->materialTypeMask); sum.Mix(sc->numLeaves);
	*out = sum.h;
	return 0;
}

extern "C" int rt_device_zero(int device, void* ptr, uint64_t bytes)
{
	RT_CUDA(cudaSetDevice(device));
	RT_CUDA(cudaMemset(ptr, 0, bytes));
	return 0;
}

extern "C" int rt_copy_to_device(int device, void* deviceDst, const void* hostSrc, uint64_t bytes, void* stream)
{
	RT_CUDA(cudaSetDevice(device));
	RT_CUDA(cudaMemcpyAsync(deviceDst, hostSrc, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
	RT_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
	return 0;
}

// ---- CUDA IPC: one process per GPU, every rank writes its tiles into rank 0's frame over NVLink ----------------
extern "C" int rt_ipc_export(int device, void* devicePtr, unsigned char* outHandle64)
{
	RT_CUDA(cudaSetDevice(device));
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
	cudaIpcMemHandle_t h;
	RT_CUDA(cudaIpcGetMemHandle(&h, devicePtr));
	memcpy(outHandle64, &h, 64);
	return 0;
}
extern "C" int rt_ipc_open(int device, const unsigned char* handle64, void** outPtr)
{
	*outPtr = nullptr;
	RT_CUDA(cudaSetDevice(device));
	cudaIpcMemHandle_t h;
	memcpy(&h, handle64, 64);
	RT_CUDA(cudaIpcOpenMemHandle(outPtr, h, cudaIpcMemLazyEnablePeerAccess));
	return 0;
}
extern "C" int rt_ipc_close(int device, void* ptr)
{
	RT_CUDA(cudaSetDevice(device));
	RT_CUDA(cudaIpcCloseMemHandle(ptr));
	return 0;
}

extern "C" int rt_device_alloc(int device, uint64_t bytes, void** outPtr)
{
	*outPtr = nullptr;
	RT_CUDA(cudaSetDevice(device));
	RT_CUDA(cudaMalloc(outPtr, std::max<uint64_t>(bytes, 16)));
	return 0;
}
extern "C" void rt_device_free(int device, void* ptr) { if (ptr) { cudaSetDevice(device); cudaFree(ptr); } }
extern "C" int rt_copy_to_host(int device, void* hostDst, const void* deviceSrc, uint64_t bytes, void* stream)
{
	RT_CUDA(cudaSetDevice(device));
	RT_CUDA(cudaMemcpyAsync(hostDst, deviceSrc, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
	RT_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
	return 0;
}
extern "C" int rt_stream_sync(int device, void* stream)
{
	RT_CUDA(cudaSetDevice(device));
	RT_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
	return 0;
}

// ---- several devices in one process ----------------------------------------------------------------------------
extern "C" int rt_peer_enable(int device, int peer)
{
	if (device == peer) return 0;
	RT_CUDA(cudaSetDevice(device));
	int can = 0;
	RT_CUDA(cudaDeviceCanAccessPeer(&can, device, peer));
	if (!can) { g_lastError = "rt_peer_enable: no peer access between the two devices"; return -1; }
	const cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
	if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return 0; }
	RT_CUDA(e);
	return 0;
}
extern "C" int rt_copy_peer(int dstDevice, void* dst, int srcDevice, const void* src, uint64_t bytes)
{
	RT_CUDA(cudaMemcpyPeer(dst, dstDevice, src, srcDevice, bytes));
	return 0;
}
extern "C" int rt_host_register(void* ptr, uint64_t bytes)
{
	RT_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
	return 0;
}
extern "C" int rt_host_unregister(void* ptr)
{
	RT_CUDA(cudaHostUnregister(ptr));
	return 0;
}
extern "C" int rt_device_free_bytes(int device, uint64_t* outFree, uint64_t* outTotal)
{
	RT_CUDA(cudaSetDevice(device));
	size_t f = 0, t = 0;
	RT_CUDA(cudaMemGetInfo(&f, &t));
	if (outFree) *outFree = f;
	if (outTotal) *outTotal = t;
	return 0;
}

// ---- transcendentals on the device, for the parity tests (include/rt_libm.h against the host C library) -------------
__global__ void __launch_bounds__(256) k_libm_eval(int fn, const float* x, const float* y, float* out, uint64_t n)
{
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
	{
		const float a = x[i], b = y ? y[i] : 0.0f;
		float r;
		switch (fn)
		{
		case 0: r = rt_m_sinf(a); break;
		case 1: r = rt_m_cosf(a); break;
		case 2: r = rt_m_tanf(a); break;
		case 3: r = rt_m_asinf(a); break;
		case 4: r = rt_m_acosf(a); break;
		case 5: r = rt_m_atanf(a); break;
		case 6: r = rt_m_expf(a); break;
		case 7: r = rt_m_logf(a); break;
		case 8: r = rt_m_powf(a, b); break;
		default: r = rt_m_atan2f(a, b); break;
		}
		out[i] = r;
	}
}

extern "C" int rt_libm_eval(int device, int fn, const float* hostX, const float* hostY, float* hostOut, uint64_t n)
{
	if (n == 0) return 0;
	RT_CUDA(cudaSetDevice(device));
	float *dx = nullptr, *dy = nullptr, *dout = nullptr;
	struct Scratch { float*& a; float*& b; float*& c; ~Scratch() { cudaFree(a); cudaFree(b); cudaFree(c); } } scratch{ dx, dy, dout };
	RT_CUDA(cudaMalloc((void**)&dx, n * 4));
	RT_CUDA(cudaMalloc((void**)&dout, n * 4));
	RT_CUDA(cudaMemcpy(dx, hostX, n * 4, cudaMemcpyHostToDevice));
	if (hostY) { RT_CUDA(cudaMalloc((void**)&dy, n * 4)); RT_CUDA(cudaMemcpy(dy, hostY, n * 4, cudaMemcpyHostToDevice)); }
	k_libm_eval<<<148 * 8, 256>>>(fn, dx, dy, dout, n);
	RT_CUDA(cudaGetLastError());
	RT_CUDA(cudaMemcpy(hostOut, dout, n * 4, cudaMemcpyDeviceToHost));
	return 0;
}
