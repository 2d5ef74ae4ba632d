// rt_traverse.cuh -- ray / box / triangle / sphere / cube tests and the stack
// traversal of the flattened reference BVH (include/rt_scene_format.h).
//
// Reference semantics being reproduced (all file:line under raylib/):
//   box      geom/aabb.h:41-53    slab test, swap on negative 1/d, reject on tMax <  tMin
//   triangle geom/triangle.cc:18-58  plane t, inclusive range, barycentrics by two divisions
//   sphere   geom/sphere.cc:3-45  near root then far root, strict range
//   cube     geom/cube.cc:3-43    moving slab box
//   BVH      geom/bvh.cc:82-107   EXHAUSTIVE: both children get the caller's tMax (FLT_MAX), the
//                                 closer result wins, ties go to the RIGHT child.
// Closed form of the last rule: winner = minimum t, ties -> highest in-order leaf rank.  A
// near-first traversal that shrinks its search interval yields the same winner as long as it
// (a) uses the reference's pass/fail box test against [tMin, FLT_MAX] and (b) only skips a box
// whose entry distance lies beyond the current best t.  (b) relies on "a primitive's hit t is
// not smaller than the entry t of every box around it", which floating-point rounding can
// violate: by a few ulps for grazing rays on triangles, and by up to ~sqrt(2^-23) = 3.5e-4 RELATIVE for a sphere
// seen from more than ~4000 radii away, where b*b - a*c of geom/sphere.cc:11 cancels catastrophically and the
// reference's own t is that inexact.  RT_PRUNE_SLACK (2e-3 relative) widens the skip threshold beyond both, so the
// device finds whatever the reference finds; tests/test_gpu_parity.py reports the mismatch rate.
#pragma once
#include "rt_math.cuh"
#include "rt_scene_format.h"
#include <float.h>

#define RT_PRUNE_SLACK 2.0e-3f
// stack-pop attempts per traversal step (an entry beyond the best hit is dropped; with one attempt the lane retries in its
// next step, which the warp runs anyway for its other lanes)
// RT_POP_HOISTED 1: the two stack entries a step may pop are loaded at the START of the step, next to the node fetch, instead
// of after the pushes: a step that pushes never needs them (what it pops is the entry it has just pushed, still in
// registers), so the loads never depend on the step's own stores and their latency hides behind the node's.
#ifndef RT_POP_HOISTED
#define RT_POP_HOISTED 0
#endif
#ifndef RT_POP_ATTEMPTS
#define RT_POP_ATTEMPTS 2
#endif
#define RT_MISS_REF 0xFFFFFFFFu

// prmt.b32 with an immediate selector: `b` must stay in a register (the SASS form has one immediate slot)
RT_DEV uint32_t rt_prmt(uint32_t a, uint32_t b, uint32_t selector) { return __byte_perm(a, b, selector); }

struct RtSceneView
{
	const float4*     nodes;        // traversal tree, 4 x float4 per RtNodeQ4
	const float4*     refNodes;     // reference topology (statistics only)
	const float4*     triHot;       // 4 x float4 (64 B) per triangle
	const RtTriCold*  triCold;
	const uint32_t*   triRank;      // not uploaded: rank and gate index live in the hot record (RT_TRI_RANK, RT_TRI_GATE)
	const uint32_t*   triGate;
	const float4*     gateBoxes;    // 2 x float4 per gate
	const float4*     spheres;
	const uint32_t*   sphereMaterial;
	const uint32_t*   sphereRank;
	const uint32_t*   sphereGate;
	const RtCube*     cubes;
	const uint32_t*   cubeRank;
	const uint32_t*   cubeGate;
	const RtMaterial* materials;
	const RtTexture*  textures;
	const float4*     texels;
	float    rootMin[3], rootMax[3];
	uint32_t rootRef;
	float    refRootMin[3], refRootMax[3];
	uint32_t refRootRef;
	uint32_t refRootBoxTests;
	uint32_t flags;
	uint32_t q4magic;     // 0x3F000000, kept in a register-resident field so PRMT can take its selector as the immediate
	int32_t  skyTexture;
	uint32_t hasSun;
	float    skyRotation[9];
	float    sunIlluminance[3];
	float    sunDirection[3];
};

struct RtRay
{
	float3 o, d;
	float3 idc;     // 1/d clamped to +-RT_IDC_LIMIT: used only by the conservative culling test of inner nodes
	float  time;
};
#define RT_IDC_LIMIT 1.0e18f

RT_DEV float3 exact_inv_dir(const RtRay& r) { return v3(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z); }

RT_DEV RtRay make_ray(float3 o, float3 d, float time)
{
	RtRay r;
	r.o = o; r.d = d; r.time = time;
	const float3 inv = exact_inv_dir(r);
	r.idc = v3(fminf(fmaxf(inv.x, -RT_IDC_LIMIT), RT_IDC_LIMIT), fminf(fmaxf(inv.y, -RT_IDC_LIMIT), RT_IDC_LIMIT), fminf(fmaxf(inv.z, -RT_IDC_LIMIT), RT_IDC_LIMIT));
	return r;
}

struct RtHit
{
	float    t;
	float    bu, bv;     // triangle barycentrics (paramU/paramV of triangle.cc:42-43 before the UV blend)
	uint32_t ref;        // RT_MAKE_REF(RT_REF_TRI|SPHERE|CUBE, index) or RT_MISS_REF
};

// box/tri/sphere/nodes: work the pruned device traversal actually did.
// refBox/refTri/refSphere: work the REFERENCE's exhaustive traversal does for the same ray
// (count_reference_work below) -- the "algorithmic" counts of the roofline model.
struct RtTravStats
{
	uint32_t box, tri, sphere, nodes, refBox, refTri, refSphere;
	uint32_t gate, cube;    // exact gate-box tests of accepted hits, cube tests
	// SIMD occupancy of the traversal loop: node-phase iterations this lane was in, ... could step in, ... owned a ray in;
	// leaf-phase iterations it was in and ... tested a leaf in (summed over lanes: lanes per iteration = x / iterations / 32 * 32)
	uint32_t nodeIters, nodeStep, nodeAlive, leafIters, leafBusy;
};

// ---- texture fetch (render/texture.cc:30-53) -------------------------------------------------
template<bool ALPHA_ONLY>
RT_DEV float4 sample_texture_impl(const RtSceneView& S, int32_t texIndex, float u, float v)
{
	const RtTexture tx = S.textures[texIndex];
	u = fmodf(u, 1.0f); if (u < 0.0f) u += 1.0f;
	v = fmodf(v, 1.0f); if (v < 0.0f) v += 1.0f; v = 1.0f - v;
	if (isnan(u) || isinf(u)) u = 0.0f;
	if (isnan(v) || isinf(v)) v = 0.0f;
	int32_t x = (int32_t)((float)(tx.width - 1u) * u);
	int32_t y = (int32_t)((float)(tx.height - 1u) * v);
	x = max(0, min((int32_t)tx.width - 1, x));
	y = max(0, min((int32_t)tx.height - 1, y));
	float4 px = __ldg(S.texels + tx.texelOffset + (uint64_t)y * tx.width + (uint64_t)x);
	if (tx.srgb)
	{
		// SRGBToLinear decodes all four channels, alpha included (render/image.h:79-83); the cut-out test of the traversal
		// loop only looks at alpha, so it skips the three powf it would throw away
		if (!ALPHA_ONLY) { px.x = rt_powf(px.x, 2.2f); px.y = rt_powf(px.y, 2.2f); px.z = rt_powf(px.z, 2.2f); }
		px.w = rt_powf(px.w, 2.2f);
	}
	return px;
}
RT_DEV float4 sample_texture(const RtSceneView& S, int32_t texIndex, float u, float v) { return sample_texture_impl<false>(S, texIndex, u, v); }
RT_DEV float sample_texture_alpha(const RtSceneView& S, int32_t texIndex, float u, float v) { return sample_texture_impl<true>(S, texIndex, u, v).w; }

// ---- in-order rank of a primitive reference (only consulted on exact t ties) -----------------
RT_DEV uint32_t rank_of(const RtSceneView& S, uint32_t ref)
{
	const uint32_t kind = RT_REF_KIND(ref), idx = RT_REF_INDEX(ref);
	if (kind == RT_REF_TRI) return __float_as_uint(__ldg(reinterpret_cast<const float*>(S.triHot + 4u * (size_t)idx) + RT_TRI_RANK));
	if (kind == RT_REF_SPHERE) return S.sphereRank[idx];
	return S.cubeRank[idx];
}

RT_DEV bool wins_tie(const RtSceneView& S, uint32_t candidate, uint32_t incumbent)
{
	return rank_of(S, candidate) > rank_of(S, incumbent);
}

// ---- slab test: returns the reference's verdict against [tMin, FLT_MAX]; entry = clipped near t
RT_DEV bool box_test(float3 bmin, float3 bmax, float3 o, float3 invD, float tMin, float& entry)
{
	float ax = (bmin.x - o.x) * invD.x, bx = (bmax.x - o.x) * invD.x;
	float ay = (bmin.y - o.y) * invD.y, by = (bmax.y - o.y) * invD.y;
	float az = (bmin.z - o.z) * invD.z, bz = (bmax.z - o.z) * invD.z;
	const float nx = invD.x < 0.0f ? bx : ax, fx = invD.x < 0.0f ? ax : bx;
	const float ny = invD.y < 0.0f ? by : ay, fy = invD.y < 0.0f ? ay : by;
	const float nz = invD.z < 0.0f ? bz : az, fz = invD.z < 0.0f ? az : bz;
	// "t0 > tMin ? t0 : tMin" keeps tMin when t0 is NaN, exactly like fmaxf(tMin, t0)
	const float lo = fmaxf(fmaxf(fmaxf(tMin, nx), ny), nz);
	const float hi = fminf(fminf(fminf(FLT_MAX, fx), fy), fz);
	entry = lo;
	return !(hi < lo);
}
// Same test with 1/d computed on the spot (IEEE division, as AABB::Hit does): for the few exact tests per ray
// -- the root box and the gate of an accepted hit.
RT_DEV bool box_test(float3 bmin, float3 bmax, const RtRay& r, float tMin, float& entry)
{
	return box_test(bmin, bmax, r.o, exact_inv_dir(r), tMin, entry);
}

// The reference only calls a primitive's Hit() if the box of the BVHNode holding it passed AABB::Hit (geom/bvh.cc:84).
// The traversal tree culls with supersets of that box, so an accepted hit is confirmed against the exact gate here.
RT_DEV bool gate_passes(const RtSceneView& S, uint32_t gate, const RtRay& r, float tMin)
{
	if (gate == RT_NO_GATE) return true;
	const RtF8 g = ldg8(S.gateBoxes + 2u * (size_t)gate);
	float unused;
	return box_test(xyz(g.lo), xyz(g.hi), r, tMin, unused);
}

// ---- primitive tests ----------------------------------------------------------------------------
// Each returns true when the reference's Hit() would return true for [tMin, FLT_MAX].

RT_DEV bool triangle_test(const RtSceneView& S, uint32_t idx, const RtRay& r, float tMin, float tLimit,
                          float& outT, float& outBu, float& outBv, int32_t& outMatType, uint32_t& gateTests)
{
	const RtF8 ta = ldg8(S.triHot + 4u * (size_t)idx), tb = ldg8(S.triHot + 4u * (size_t)idx + 2);
	const float4 q0 = ta.lo, q1 = ta.hi, q2 = tb.lo;
	const float3 v0 = v3(q0.x, q0.y, q0.z);
	const float3 n  = v3(q0.w, q1.x, q1.y);
	const float t = dot3(v0 - r.o, n) / dot3(r.d, n);
	if (t < tMin || t > FLT_MAX) return false;     // triangle.cc:25 (a NaN t falls through, as there)
	if (t > tLimit) return false;                  // cannot beat the current best
	const float3 p = r.o + t * r.d;
	const float3 u = v3(q1.z, q1.w, q2.x);
	const float3 v = v3(q2.y, q2.z, q2.w);
	const float3 w = p - v0;
	const float uv = dot3(u, v), wv = dot3(w, v), uu = dot3(u, u), vv = dot3(v, v), wu = dot3(w, u);
	const float uvuv = uv * uv, uuvv = uu * vv;
	const float pu = (uv * wv - vv * wu) / (uvuv - uuvv);
	const float pv = (uv * wu - uu * wv) / (uvuv - uuvv);
	if (0.0f <= pu && 0.0f <= pv && pu + pv <= 1.0f)
	{
		if (S.flags & RT_SCENE_FLAG_ALPHA_TEST)
		{
			// Triangle::Hit ends with material->AlphaTest(u, v) (triangle.cc:54, material.cc:397-404)
			// material index and type ride in the hot record: no dependent load through the cold record to find them
			const int32_t albedoTex = (__float_as_uint(tb.hi.w) == (uint32_t)RT_MAT_MICROFACET)
				? S.materials[__float_as_uint(tb.hi.y)].tex[RT_TEX_ALBEDO] : -1;
			if (albedoTex >= 0)
			{
				const RtTriCold* c = S.triCold + idx;
				const float k = 1.0f - pu - pv;
				const float s = k * c->st[0] + pu * c->st[2] + pv * c->st[4];
				const float tt = k * c->st[1] + pu * c->st[3] + pv * c->st[5];
				if (!(sample_texture_alpha(S, albedoTex, s, tt) >= 0.5f)) return false;
			}
		}
		// the reference only reaches this triangle if the box of the BVHNode holding it passed (geom/bvh.cc:84);
		// with the SAH tree that box is not on our path, so it is checked here, on the (rare) accepted hits
		gateTests++;
		if (!gate_passes(S, __float_as_uint(tb.hi.x), r, tMin)) return false;
		outT = t; outBu = pu; outBv = pv;
		outMatType = (int32_t)__float_as_uint(tb.hi.w);
		return true;
	}
	return false;
}

RT_DEV bool sphere_test(const RtSceneView& S, uint32_t idx, const RtRay& r, float tMin, float& outT)
{
	const float4 s = ldg4(S.spheres + idx);
	const float3 oc = r.o - v3(s.x, s.y, s.z);
	const float a = dot3(r.d, r.d);
	const float b = dot3(oc, r.d);
	const float c = dot3(oc, oc) - s.w * s.w;
	const float D = b * b - a * c;
	if (D > 0.0f)
	{
		const float root = sqrtf(D);
		float t = (-b - root) / a;
		if (tMin < t && t < FLT_MAX) { outT = t; return true; }
		t = (-b + root) / a;
		if (tMin < t && t < FLT_MAX) { outT = t; return true; }
	}
	return false;
}

RT_DEV bool cube_test(const RtSceneView& S, uint32_t idx, const RtRay& r, float tMin, float& outT, int& outFace)
{
	const RtCube cb = S.cubes[idx];
	const float3 move = v3(cb.velocity) * fmaxf(0.0f, r.time - cb.timeStartMove);
	const float3 lo = v3(cb.minBounds) + move, hi = v3(cb.maxBounds) + move;
	const float t1 = (lo.x - r.o.x) / r.d.x, t2 = (hi.x - r.o.x) / r.d.x;
	const float t3 = (lo.y - r.o.y) / r.d.y, t4 = (hi.y - r.o.y) / r.d.y;
	const float t5 = (lo.z - r.o.z) / r.d.z, t6 = (hi.z - r.o.z) / r.d.z;
	// std::max(a,b) = (a < b) ? b : a ; std::min(a,b) = (b < a) ? b : a  (NaN-order sensitive, so spelled out)
	#define RT_SMAX(a, b) (((a) < (b)) ? (b) : (a))
	#define RT_SMIN(a, b) (((b) < (a)) ? (b) : (a))
	const float m12 = RT_SMIN(t1, t2), m34 = RT_SMIN(t3, t4), m56 = RT_SMIN(t5, t6);
	const float M12 = RT_SMAX(t1, t2), M34 = RT_SMAX(t3, t4), M56 = RT_SMAX(t5, t6);
	const float m1234 = RT_SMAX(m12, m34);
	const float t7 = RT_SMAX(m1234, m56);
	const float M1234 = RT_SMIN(M12, M34);
	const float t8 = RT_SMIN(M1234, M56);
	#undef RT_SMAX
	#undef RT_SMIN
	if (t8 < 0.0f || t7 > t8) return false;
	if (tMin <= t7 && t7 <= FLT_MAX)
	{
		outT = t7;
		outFace = (t7 == t1) ? 0 : (t7 == t2) ? 1 : (t7 == t3) ? 2 : (t7 == t4) ? 3 : (t7 == t5) ? 4 : (t7 == t6) ? 5 : 6;
		return true;
	}
	return false;
}

// ---- traversal --------------------------------------------------------------------------------------
// Traversal stack: {ref, entry-t bits} per level, in thread-local memory (L1-cached, interleaved per lane by the
// hardware): leaves the whole 228 KB of the SM to L1 and lets the register file alone bound occupancy.  Measured
// alternatives that lost (profiles/README.md): all of it in shared memory, a shared-memory window for the newest
// entries, the newest entry in registers.
#define RT_MAX_STACK 96
struct RtStack
{
	uint2*   base;
	uint32_t stride;
	RT_DEV void push(uint32_t level, uint32_t ref, float entry) { base[level * stride] = make_uint2(ref, __float_as_uint(entry)); }
	RT_DEV uint2 at(uint32_t level) const { return base[level * stride]; }
};

// Resumable traversal state of one ray, so that a warp can swap finished rays for fresh ones while the
// other lanes keep going (k_extend / k_shadow).
#define RT_REF_DONE 0xFFFFFFFFu      // == RT_MAKE_REF(RT_REF_NONE, RT_REF_INDEX_MASK): nothing left / no pending leaf
#define RT_REF_POP  0xF0000000u      // == RT_MAKE_REF(RT_REF_NONE, 0): take the next entry from the stack

struct RtTrav
{
	RtHit    best;
	float    limit;     // boxes entering beyond this are skipped (best t plus slack)
	uint32_t cur;       // next reference to process: inner node, leaf, RT_REF_POP, or RT_REF_DONE when the stack ran dry
	uint32_t leaf;      // postponed leaf, RT_REF_DONE if none
	uint32_t sp;        // stack entries in use
	int32_t  hitType;   // RtMaterialType of the best hit's material, -1 while nothing has been hit
	RT_DEV bool found() const { return hitType >= 0; }
};

RT_DEV bool is_leaf_ref(uint32_t ref) { const uint32_t k = RT_REF_KIND(ref); return k != RT_REF_NODE && k != RT_REF_NONE; }

// A ray can take a traversal step unless its walk is over or it holds two leaves (one postponed, one current).
RT_DEV bool trav_can_step(const RtTrav& ts) { return ts.cur != RT_REF_DONE && !(ts.leaf != RT_REF_DONE && is_leaf_ref(ts.cur)); }
RT_DEV bool trav_finished(const RtTrav& ts) { return ts.cur == RT_REF_DONE && ts.leaf == RT_REF_DONE; }

// Returns false when the ray misses the root box (nothing to traverse).
template<bool STATS>
RT_DEV bool trav_begin(const RtSceneView& S, const RtRay& r, float tMin, RtTrav& ts, RtTravStats& st)
{
	ts.best.t = FLT_MAX; ts.best.bu = 0.0f; ts.best.bv = 0.0f; ts.best.ref = RT_MISS_REF;
	ts.limit = FLT_MAX;
	ts.hitType = -1;
	ts.sp = 0;
	ts.cur = S.rootRef;
	ts.leaf = RT_REF_DONE;
	float entry;
	if (STATS) st.box++;
	return box_test(v3(S.rootMin), v3(S.rootMax), r, tMin, entry);
}

// Tests the one or two primitives of a leaf reference against the ray and updates the best hit with the
// reference's rule: minimum t, ties to the highest in-order rank.  Returns true if an any-hit query is done.
// `hitRecords` (optional): when given, an accepted hit is written straight to record `hitSlot` there ({t, bu, bv, ref}: the first
// half of the path's 32-byte hit record) instead of being carried in ts.best.bu / .bv until the ray is done: two registers
// less across the node loop of k_extend (+1-2.5 %, profiles/README.md); a ray accepts one or two hits in its life.
template<bool ANY_HIT, bool STATS>
RT_DEV bool trav_leaf(const RtSceneView& S, const RtRay& r, float tMin, uint32_t leaf, RtTrav& ts, RtTravStats& st,
                      float4* hitRecords = nullptr, uint32_t hitSlot = 0u)
{
	const uint32_t kind = RT_REF_KIND(leaf), first = RT_REF_INDEX(leaf);
	const uint32_t count = (kind == RT_REF_TRI2 || kind == RT_REF_SPHERE2 || kind == RT_REF_CUBE2) ? 2u : 1u;
	for (uint32_t i = 0; i < count; ++i)
	{
		const uint32_t idx = first + i;
		float t, bu = 0.0f, bv = 0.0f;
		uint32_t ref;
		int32_t matType = 0;
		bool hit;
		if (kind == RT_REF_TRI || kind == RT_REF_TRI2)
		{
			if (STATS) st.tri++;
			uint32_t gates = 0;
			hit = triangle_test(S, idx, r, tMin, ANY_HIT ? FLT_MAX : ts.best.t, t, bu, bv, matType, gates);
			if (STATS) st.gate += gates;
			ref = RT_MAKE_REF(RT_REF_TRI, idx);
		}
		else if (kind == RT_REF_SPHERE || kind == RT_REF_SPHERE2)
		{
			if (STATS) st.sphere++;
			hit = sphere_test(S, idx, r, tMin, t);
			if (STATS && hit) st.gate++;
			hit = hit && gate_passes(S, S.sphereGate[idx], r, tMin);
			if (hit && !ANY_HIT) matType = (int32_t)S.materials[S.sphereMaterial[idx]].type;
			ref = RT_MAKE_REF(RT_REF_SPHERE, idx);
		}
		else
		{
			int face;
			if (STATS) st.cube++;
			hit = cube_test(S, idx, r, tMin, t, face);
			if (STATS && hit) st.gate++;
			hit = hit && gate_passes(S, S.cubeGate[idx], r, tMin);
			if (hit && !ANY_HIT) matType = (int32_t)S.materials[S.cubes[idx].material].type;
			ref = RT_MAKE_REF(RT_REF_CUBE, idx);
			bu = (float)face;
		}
		if (hit)
		{
			if (ANY_HIT) { ts.best.t = t; ts.best.ref = ref; ts.hitType = 0; return true; }
			if (!ts.found() || t < ts.best.t || (t == ts.best.t && wins_tie(S, ref, ts.best.ref)))
			{
				ts.best.t = t; ts.best.ref = ref;
				if (hitRecords) hitRecords[2u * (size_t)hitSlot] = make_float4(t, bu, bv, __uint_as_float(ref));
				else { ts.best.bu = bu; ts.best.bv = bv; }
				ts.limit = t + fabsf(t) * RT_PRUNE_SLACK;
				ts.hitType = matType;
			}
		}
	}
	return false;
}

// One traversal step, written as three short predicated regions instead of nested branches so that the
// lanes of a warp stay together (profiles/README.md: the branchy form ran the stack code at 2-3 lanes per
// instruction):
//   1. inner node: test the four child boxes, continue with the nearest one, stack the others farthest-first
//      (occlusion queries use the same order: skipping the sort there measured +0.4 %, not worth a second path);
//   2. a leaf reached while no leaf is pending is POSTPONED (ts.leaf), so that the warp tests primitives
//      together instead of one lane at a time;
//   3. RT_REF_POP: up to two attempts to take a stack entry that can still matter (entries beyond the
//      current best hit are dropped; a third culled entry simply costs this lane another step).
// Precondition: trav_can_step(ts).
template<bool ANY_HIT, bool STATS>
RT_DEV void trav_step(const RtSceneView& S, const RtRay& r, float tMin, RtStack stack, RtTrav& ts, RtTravStats& st)
{
	uint32_t cur = ts.cur;
#if RT_POP_HOISTED
	const uint32_t sp0 = ts.sp;
	const uint2 top1 = stack.at(sp0 - (sp0 >= 1u ? 1u : 0u));      // slot 0 when the stack is shorter: never used then
	const uint2 top2 = stack.at(sp0 - (sp0 >= 2u ? 2u : 0u));
	uint32_t pushedRef = 0u;        // the entry this step pushed last (the nearest of the stacked children)
#endif
	if (RT_REF_KIND(cur) == RT_REF_NODE)
	{
		// 64-byte RtNodeQ4 in two 256-bit loads: {base.xyz Sx qlo.xyz qhi.x} {qhi.yz ref[4] Sy Sz}
		const float4* np = S.nodes + 4u * (size_t)RT_REF_INDEX(cur);
		const RtF8 A = ldg8(np), B = ldg8(np + 2);
		if (STATS) { st.nodes++; }
		uint32_t r0 = __float_as_uint(B.lo.z), r1 = __float_as_uint(B.lo.w), r2 = __float_as_uint(B.hi.x), r3 = __float_as_uint(B.hi.y);
		// Conservative slab test in ray space.  A child plane is p = m*S + base (m in [0.5, 2) from the stored byte), so
		// its ray parameter is t = m*(S/d) + (base - o)/d: one PRMT + one FMA per plane.  Compared with what AABB::Hit
		// computes on any box inside this one, rounding moves t by at most ~2^-23 * (|(base-o)/d| + |t|) on that axis
		// (S is not a power of two: the rounding of S/d adds 2^-24 * |m*S/d| <= 2^-24 * (|(base-o)/d| + |t|), inside the same bound);
		// the first term is folded into the per-axis addends (near planes pulled in, far planes pushed out), the second
		// is applied to the final interval, 4x over-estimated, plus tMin on the far side for rays lying in a face plane.
		// Inner nodes only have to be supersets: the exact verdict is the gate test of the accepted hit.
		const float kSlack = 3.81469727e-6f;     // 2^-18: 32x the rounding bound -- rays from 1e5..1e6 scene sizes away keep every hit the reference finds (tools/soak_parity.py)
		const float ax = __fmul_rn(A.lo.w, r.idc.x), ay = __fmul_rn(B.hi.z, r.idc.y), az = __fmul_rn(B.hi.w, r.idc.z);
		const float bx = __fmul_rn(A.lo.x - r.o.x, r.idc.x), by = __fmul_rn(A.lo.y - r.o.y, r.idc.y), bz = __fmul_rn(A.lo.z - r.o.z, r.idc.z);
		const float bnx = __fmaf_rn(-kSlack, fabsf(bx), bx), bny = __fmaf_rn(-kSlack, fabsf(by), by), bnz = __fmaf_rn(-kSlack, fabsf(bz), bz);
		const float bfx = __fmaf_rn(kSlack, fabsf(bx), bx), bfy = __fmaf_rn(kSlack, fabsf(by), by), bfz = __fmaf_rn(kSlack, fabsf(bz), bz);
		// per axis: the word holding the near planes and the one holding the far planes for this ray's direction
		const bool nx = r.idc.x < 0.0f, ny = r.idc.y < 0.0f, nz = r.idc.z < 0.0f;
		const uint32_t wlx = __float_as_uint(A.hi.x), wly = __float_as_uint(A.hi.y), wlz = __float_as_uint(A.hi.z);
		const uint32_t whx = __float_as_uint(A.hi.w), why = __float_as_uint(B.lo.x), whz = __float_as_uint(B.lo.y);
		const uint32_t nwx = nx ? whx : wlx, fwx = nx ? wlx : whx;
		const uint32_t nwy = ny ? why : wly, fwy = ny ? wly : why;
		const uint32_t nwz = nz ? whz : wlz, fwz = nz ? wlz : whz;
		float e0, e1, e2, e3;
		#define RT_Q4_M(word, k) __uint_as_float(rt_prmt(word, S.q4magic, 0x7044u | ((k) << 8)))
		// the near and the far plane of a child on one axis in ONE packed fma.rn.f32x2 (FFMA2): 12 instead of 24 FFMA per
		// inner node, same roundings (+0.3-0.5 %, profiles/README.md)
		#define RT_Q4_CHILD(k, e, p) { \
			const float2 tx = fma2_rn(make_float2(RT_Q4_M(nwx, k), RT_Q4_M(fwx, k)), make_float2(ax, ax), make_float2(bnx, bfx)); \
			const float2 ty = fma2_rn(make_float2(RT_Q4_M(nwy, k), RT_Q4_M(fwy, k)), make_float2(ay, ay), make_float2(bny, bfy)); \
			const float2 tz = fma2_rn(make_float2(RT_Q4_M(nwz, k), RT_Q4_M(fwz, k)), make_float2(az, az), make_float2(bnz, bfz)); \
			const float tn = fmaxf(fmaxf(tx.x, ty.x), tz.x); \
			const float tf = fminf(fminf(tx.y, ty.y), tz.y); \
			e = fmaxf(__fmaf_rn(-kSlack, fabsf(tn), tn), tMin); \
			p = e <= fminf(__fmaf_rn(kSlack, fabsf(tf), tf) + tMin, ts.limit); }
		bool p0, p1, p2, p3;
		RT_Q4_CHILD(0, e0, p0); RT_Q4_CHILD(1, e1, p1); RT_Q4_CHILD(2, e2, p2); RT_Q4_CHILD(3, e3, p3);
		#undef RT_Q4_CHILD
		#undef RT_Q4_M
		// absent children carry an inverted box (lo at the top of the grid, hi at the bottom); the slack could let a
		// ray through it, so they are masked explicitly
		p2 = p2 && r2 != RT_REF_ABSENT;
		p3 = p3 && r3 != RT_REF_ABSENT;
		if (STATS) { st.box += 2u + (r2 != RT_REF_ABSENT ? 1u : 0u) + (r3 != RT_REF_ABSENT ? 1u : 0u); }
		{
			const float inf = __int_as_float(0x7f800000);
			e0 = p0 ? e0 : inf; e1 = p1 ? e1 : inf; e2 = p2 ? e2 : inf; e3 = p3 ? e3 : inf;
			// order the four (entry, ref) pairs by entry distance: misses (+inf) sink to the end
			#define RT_CSWAP(ea, ra, eb, rb) { const bool sw = eb < ea; const float te = sw ? eb : ea; const uint32_t tr = sw ? rb : ra; \
			                                   eb = sw ? ea : eb; rb = sw ? ra : rb; ea = te; ra = tr; }
			RT_CSWAP(e0, r0, e1, r1); RT_CSWAP(e2, r2, e3, r3); RT_CSWAP(e0, r0, e2, r2); RT_CSWAP(e1, r1, e3, r3); RT_CSWAP(e1, r1, e2, r2);
			#undef RT_CSWAP
			// continue with the nearest, stack the other hits farthest-first
			if (e3 < inf) stack.push(ts.sp++, r3, e3);
			if (e2 < inf) stack.push(ts.sp++, r2, e2);
			if (e1 < inf) stack.push(ts.sp++, r1, e1);
		#if RT_POP_HOISTED
			pushedRef = r1;
		#endif
			cur = (e0 < inf) ? r0 : RT_REF_POP;
		}
	}
	if (ts.leaf == RT_REF_DONE && is_leaf_ref(cur)) { ts.leaf = cur; cur = RT_REF_POP; }
#if RT_POP_HOISTED
	{
		// first attempt: the entry pushed by this very step if there is one (it passed the cull test a moment ago), else the old top
		const bool pushed = ts.sp != sp0;
		const bool pop = cur == RT_REF_POP;
		const bool has = ts.sp != 0u;
		const uint32_t fromOld = !has ? RT_REF_DONE : ((__uint_as_float(top1.y) > ts.limit) ? RT_REF_POP : top1.x);
		const uint32_t next = pushed ? pushedRef : fromOld;
		cur = pop ? next : cur;
		ts.sp = pop ? ts.sp - (has ? 1u : 0u) : ts.sp;
		// second attempt: only after the old top was dropped, i.e. nothing was pushed and ts.sp == sp0 - 1
		const bool pop2 = cur == RT_REF_POP;
		const bool has2 = ts.sp != 0u;
		const uint32_t next2 = !has2 ? RT_REF_DONE : ((__uint_as_float(top2.y) > ts.limit) ? RT_REF_POP : top2.x);
		cur = pop2 ? next2 : cur;
		ts.sp = pop2 ? ts.sp - (has2 ? 1u : 0u) : ts.sp;
	}
#else
	// two pop attempts as straight-line code: the top entry is read whether or not this lane pops (slot 0 when the
	// stack is empty: never used), the selects do the rest -- no divergent regions, ~16 instructions fewer per step
	#pragma unroll
	for (int attempt = 0; attempt < RT_POP_ATTEMPTS; ++attempt)
	{
		const bool pop = cur == RT_REF_POP;
		const bool has = ts.sp != 0u;
		const uint32_t idx = ts.sp - (has ? 1u : 0u);
		const uint2 e = stack.at(idx);
		const uint32_t next = !has ? RT_REF_DONE : ((__uint_as_float(e.y) > ts.limit) ? RT_REF_POP : e.x);
		cur = pop ? next : cur;
		ts.sp = pop ? idx : ts.sp;
	}
#endif
	ts.cur = cur;
}

// The pending leaf of a ray (one per call): test its primitives, then promote a second leaf the walk stopped at.
// Returns true when an any-hit query has its answer.
template<bool ANY_HIT, bool STATS>
RT_DEV bool trav_pending_leaf(const RtSceneView& S, const RtRay& r, float tMin, RtTrav& ts, RtTravStats& st,
                              float4* hitRecords = nullptr, uint32_t hitSlot = 0u)
{
	const uint32_t leaf = ts.leaf;
	ts.leaf = RT_REF_DONE;
	if (trav_leaf<ANY_HIT, STATS>(S, r, tMin, leaf, ts, st, hitRecords, hitSlot)) return true;
	if (is_leaf_ref(ts.cur)) { ts.leaf = ts.cur; ts.cur = RT_REF_POP; }
	return false;
}

// Runs the traversal for the lanes with alive == true until fewer than `keepGoing` lanes of the warp are still
// busy.  Must be called by all 32 lanes.  A lane that finishes clears `alive`; its result is in ts.best / ts.found().
//
// Node phase: all lanes that can step do so together.  It ends when nobody can step, or when fewer than
// `walkThreshold` lanes can and at least one lane is blocked on leaves -- waiting for the slowest lane to
// collect its leaves left 2/3 of the SIMD lanes idle (ncu: 9.8 active threads per warp).
// Leaf phase: every lane with a pending leaf tests it (lanes blocked on two leaves become steppable again).
template<bool ANY_HIT, bool STATS>
RT_DEV void trav_run(const RtSceneView& S, const RtRay& r, float tMin, RtStack stack, RtTrav& ts, bool& alive,
                     uint32_t keepGoing, uint32_t walkThreshold, RtTravStats& st,
                     float4* hitRecords = nullptr, uint32_t hitSlot = 0u)
{
	for (;;)
	{
		for (;;)
		{
			const bool step = alive && trav_can_step(ts);
			const uint32_t nStep = __popc(__ballot_sync(0xFFFFFFFFu, step));
			if (nStep == 0) break;
			if (nStep < walkThreshold && __any_sync(0xFFFFFFFFu, alive && !step)) break;
			if (STATS) { st.nodeIters++; st.nodeStep += step ? 1u : 0u; st.nodeAlive += alive ? 1u : 0u; }
			if (step)
			{
				trav_step<ANY_HIT, STATS>(S, r, tMin, stack, ts, st);
				if (trav_finished(ts)) alive = false;
			}
		}
		if (STATS) { st.leafIters++; st.leafBusy += (alive && ts.leaf != RT_REF_DONE) ? 1u : 0u; }
		if (alive && ts.leaf != RT_REF_DONE)
		{
			if (trav_pending_leaf<ANY_HIT, STATS>(S, r, tMin, ts, st, hitRecords, hitSlot)) alive = false;
			else if (trav_finished(ts)) alive = false;
		}
		if ((uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, alive)) < keepGoing) return;
	}
}

template<bool ANY_HIT, bool STATS>
RT_DEV bool traverse(const RtSceneView& S, const RtRay& r, float tMin, RtStack stack, RtHit& best, RtTravStats& st)
{
	// single-ray form (debug views, ray queries): same steps, no warp cooperation
	RtTrav ts;
	if (trav_begin<STATS>(S, r, tMin, ts, st))
	{
		for (;;)
		{
			while (trav_can_step(ts)) trav_step<ANY_HIT, STATS>(S, r, tMin, stack, ts, st);
			if (ts.leaf == RT_REF_DONE) break;
			if (trav_pending_leaf<ANY_HIT, STATS>(S, r, tMin, ts, st)) break;
		}
	}
	best = ts.best;
	return ts.found();
}

// Closest hit for one ray per lane with the warp cooperating (node phase / leaf phase as in k_extend, no refill):
// must be called by all 32 lanes; lanes with valid == false ride along.
template<bool STATS>
RT_DEV bool traverse_warp(const RtSceneView& S, const RtRay& r, float tMin, RtStack stack, bool valid, uint32_t walkThreshold,
                          RtHit& best, RtTravStats& st)
{
	RtTrav ts;
	bool alive = trav_begin<STATS>(S, r, tMin, ts, st) && valid;
	if (!alive) { ts.cur = RT_REF_DONE; ts.leaf = RT_REF_DONE; }
	trav_run<false, STATS>(S, r, tMin, stack, ts, alive, 1u, walkThreshold, st);
	best = ts.best;
	return valid && ts.found();
}

// Statistics build only: replays the reference's traversal (geom/bvh.cc:82-107 -- every child whose
// box passes is visited, nothing is pruned) and counts the box / triangle / sphere tests it performs.
RT_DEV void count_reference_work(const RtSceneView& S, const RtRay& r, float tMin, RtStack stack, RtTravStats& st)
{
	if (!S.refNodes) return;        // the scene was uploaded without the reference topology (rt_scene_upload flags)
	float entry;
	const float3 invD = exact_inv_dir(r);
	const bool rootPass = box_test(v3(S.refRootMin), v3(S.refRootMax), r.o, invD, tMin, entry);
	st.refBox += rootPass ? S.refRootBoxTests : min(1u, S.refRootBoxTests);
	if (!rootPass) return;
	uint32_t sp = 0;
	uint32_t cur = S.refRootRef;
	for (;;)
	{
		const uint32_t kind = RT_REF_KIND(cur);
		if (kind == RT_REF_NODE)
		{
			const float4* np = S.refNodes + 4u * (size_t)RT_REF_INDEX(cur);
			const float4 n0 = ldg4(np + 0), n1 = ldg4(np + 1), n2 = ldg4(np + 2), n3 = ldg4(np + 3);
			const uint32_t lref = __float_as_uint(n0.w), rref = __float_as_uint(n1.w);
			const uint32_t lTests = __float_as_uint(n2.w), rTests = __float_as_uint(n3.w);
			const bool pl = box_test(xyz(n0), xyz(n1), r.o, invD, tMin, entry);
			const bool hasR = RT_REF_KIND(rref) != RT_REF_NONE;
			const bool pr = hasR && box_test(xyz(n2), xyz(n3), r.o, invD, tMin, entry);
			st.refBox += pl ? lTests : min(1u, lTests);
			if (hasR) st.refBox += pr ? rTests : min(1u, rTests);
			if (pl && pr) { stack.push(sp++, rref, 0.0f); cur = lref; continue; }
			if (pl) { cur = lref; continue; }
			if (pr) { cur = rref; continue; }
		}
		else if (kind == RT_REF_TRI) st.refTri += 1;
		else if (kind == RT_REF_TRI2) st.refTri += 2;
		else if (kind == RT_REF_SPHERE) st.refSphere += 1;
		else if (kind == RT_REF_SPHERE2) st.refSphere += 2;
		if (sp == 0) return;
		cur = stack.at(--sp).x;
	}
}
