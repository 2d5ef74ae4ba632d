/* oracle/rt_oracle.c -- TEST INFRASTRUCTURE (not product code).
 *
 * Plain-C restatement of the reference's closest-hit query and camera-ray generation, evaluated on the
 * flattened scene arrays of include/rt_scene_format.h.  It follows the reference literally -- recursive,
 * EXHAUSTIVE traversal (both children always get tMax = FLT_MAX), no pruning, no reordering:
 *     BVHNode::Hit          raylib/geom/bvh.cc:82-107      (left.t < right.t ? left : right; ties -> right)
 *     AABB::Hit             raylib/geom/aabb.h:41-53
 *     Triangle::Hit         raylib/geom/triangle.cc:18-58
 *     Sphere::Hit           raylib/geom/sphere.cc:3-45
 *     Cube::Hit             raylib/geom/cube.cc:3-43
 *     Camera::GetCameraRay  raylib/render/camera.h:44-53
 *     Texture2D::Sample     raylib/render/texture.cc:30-53  (alpha cut-out, material.cc:397-404)
 * Pinned against the compiled reference itself (oracle/_ref/libraylib_ref.so: oracle_primary_hits,
 * oracle_trace_rays) by tests/test_oracle_cpu.py on every procedural scene -- the reference has no golden
 * vectors of its own (SURVEY.md section 4).  It exists so that the flattener and the traversal semantics
 * can be checked on hosts without /root/reference and without a GPU.
 *
 * Build: gcc -O2 -ffp-contract=off (no FMA contraction, baseline x86-64), see oracle/Makefile.restate.
 */
#include "../include/rt_scene_format.h"
#include "../include/rt_rng.h"
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

typedef struct { float x, y, z; } V3;
static V3 v3(float x, float y, float z) { V3 r = { x, y, z }; return r; }
static V3 v3p(const float* p) { V3 r = { p[0], p[1], p[2] }; return r; }
static V3 add(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
static V3 sub(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
static V3 muls(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
static float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static V3 normalize(V3 a) { float k = 1.0f / sqrtf(a.x * a.x + a.y * a.y + a.z * a.z); return v3(a.x * k, a.y * k, a.z * k); }

static int g_useTraversalTree = 0;

typedef struct { V3 o, d; float time; } Ray;
/* u, v: paramU / paramV of a triangle hit (triangle.cc:42-43); face: 0..5 of a cube hit, in the device's order (t1..t6 of
 * cube.cc, csrc/device/rt_traverse.cuh cube_test); mat: RtMaterialType of the hit primitive's material */
typedef struct { int hit; float t; uint32_t rank; float u, v; int32_t face, mat; } Hit;
typedef struct { uint64_t box, tri, sphere, cube; } Counts;

/* aabb.h:41-53 */
static int box_hit(const float* lo, const float* hi, const Ray* r, float tMin, float tMax)
{
	const float o[3] = { r->o.x, r->o.y, r->o.z }, d[3] = { r->d.x, r->d.y, r->d.z };
	for (int a = 0; a < 3; ++a)
	{
		float invD = 1.0f / d[a];
		float t0 = (lo[a] - o[a]) * invD;
		float t1 = (hi[a] - o[a]) * invD;
		if (invD < 0.0f) { float s = t0; t0 = t1; t1 = s; }
		tMin = t0 > tMin ? t0 : tMin;
		tMax = t1 < tMax ? t1 : tMax;
		if (tMax < tMin) return 0;
	}
	return 1;
}

/* texture.cc:30-53 */
static void sample_texture(const RtSceneDesc* S, int32_t tex, float u, float v, float out[4])
{
	const RtTexture* tx = &S->textures[tex];
	u = fmodf(u, 1.0f); if (u < 0.0f) u += 1.0f;
	v = fmodf(v, 1.0f); if (v < 0.0f) v += 1.0f; v = 1.0f - v;
	if (isnan(u) || isinf(u)) u = 0.0f;
	if (isnan(v) || isinf(v)) v = 0.0f;
	int32_t x = (int32_t)((float)(tx->width - 1u) * u);
	int32_t y = (int32_t)((float)(tx->height - 1u) * v);
	const float* px = S->texels + 4 * (tx->texelOffset + (uint64_t)y * tx->width + (uint64_t)x);
	for (int i = 0; i < 4; ++i) out[i] = tx->srgb ? powf(px[i], 2.2f) : px[i];
}

/* triangle.cc:18-58 */
/* Device traversal trees only (modes 1-3): a primitive is a candidate iff the box of the reference BVHNode that
 * holds it -- its gate -- passes AABB::Hit; the trees above cull with supersets of that box (rt_scene_format.h). */
static int gate_ok(const RtSceneDesc* S, uint32_t gate, const Ray* r, float t_min)
{
	if (!g_useTraversalTree || gate == RT_NO_GATE) return 1;
	const float* g = S->gateBoxes + 8 * (size_t)gate;
	return box_hit(g, g + 4, r, t_min, FLT_MAX);
}

static int triangle_hit(const RtSceneDesc* S, uint32_t idx, const Ray* r, float t_min, float t_max, float* outT, float* outU, float* outV)
{
	const float* q = S->triHot[idx].q;
	const V3 v0 = v3p(q), n = v3p(q + 3), u = v3p(q + 6), v = v3p(q + 9);
	float t = dot(sub(v0, r->o), n) / dot(r->d, n);
	V3 p = add(r->o, muls(r->d, t));
	if (t < t_min || t > t_max) return 0;
	V3 w = sub(p, v0);
	float uv = dot(u, v), wv = dot(w, v), uu = dot(u, u), vv = dot(v, v), wu = dot(w, u);
	float uvuv = uv * uv, uuvv = uu * vv;
	float paramU = (uv * wv - vv * wu) / (uvuv - uuvv);
	float paramV = (uv * wu - uu * wv) / (uvuv - uuvv);
	if (0.0f <= paramU && 0.0f <= paramV && paramU + paramV <= 1.0f)
	{
		const RtTriCold* c = &S->triCold[idx];
		const RtMaterial* m = &S->materials[c->material];
		if (m->type == RT_MAT_MICROFACET && m->tex[RT_TEX_ALBEDO] >= 0)
		{
			float k = 1 - paramU - paramV;
			float s = k * c->st[0] + paramU * c->st[2] + paramV * c->st[4];
			float tt = k * c->st[1] + paramU * c->st[3] + paramV * c->st[5];
			float px[4];
			sample_texture(S, m->tex[RT_TEX_ALBEDO], s, tt, px);
			if (!(px[3] >= 0.5f)) return 0;
		}
		/* device traversal tree only: the triangle's reference gate box (see rt_scene_format.h) must pass */
		if (!gate_ok(S, S->triGate[idx], r, t_min)) return 0;
		*outT = t; *outU = paramU; *outV = paramV;
		return 1;
	}
	return 0;
}

/* sphere.cc:3-45 */
static int sphere_hit(const RtSceneDesc* S, uint32_t idx, const Ray* r, float t_min, float t_max, float* outT)
{
	const RtSphere* s = &S->spheres[idx];
	V3 oc = sub(r->o, v3p(s->center));
	float a = dot(r->d, r->d);
	float b = dot(oc, r->d);
	float c = dot(oc, oc) - s->radius * s->radius;
	float D = b * b - a * c;
	if (D > 0.0f)
	{
		float temp = (-b - sqrtf(b * b - a * c)) / a;
		if (t_min < temp && temp < t_max) { *outT = temp; return gate_ok(S, S->sphereGate[idx], r, t_min); }
		temp = (-b + sqrtf(b * b - a * c)) / a;
		if (t_min < temp && temp < t_max) { *outT = temp; return gate_ok(S, S->sphereGate[idx], r, t_min); }
	}
	return 0;
}

static float fmax_std(float a, float b) { return (a < b) ? b : a; }   /* std::max */
static float fmin_std(float a, float b) { return (b < a) ? b : a; }   /* std::min */

/* cube.cc:3-43 */
static int cube_hit(const RtSceneDesc* S, uint32_t idx, const Ray* r, float t_min, float t_max, float* outT, int32_t* outFace)
{
	const RtCube* cb = &S->cubes[idx];
	V3 move = muls(v3p(cb->velocity), fmax_std(0.0f, r->time - cb->timeStartMove));
	V3 lo = add(v3p(cb->minBounds), move), hi = add(v3p(cb->maxBounds), move);
	float t[9];
	t[1] = (lo.x - r->o.x) / r->d.x; t[2] = (hi.x - r->o.x) / r->d.x;
	t[3] = (lo.y - r->o.y) / r->d.y; t[4] = (hi.y - r->o.y) / r->d.y;
	t[5] = (lo.z - r->o.z) / r->d.z; t[6] = (hi.z - r->o.z) / r->d.z;
	t[7] = fmax_std(fmax_std(fmin_std(t[1], t[2]), fmin_std(t[3], t[4])), fmin_std(t[5], t[6]));
	t[8] = fmin_std(fmin_std(fmax_std(t[1], t[2]), fmax_std(t[3], t[4])), fmax_std(t[5], t[6]));
	if (t[8] < 0 || t[7] > t[8]) return 0;
	if (t_min <= t[7] && t[7] <= t_max)
	{
		*outT = t[7];
		*outFace = 6;
		for (int k = 6; k >= 1; --k) if (t[7] == t[k]) *outFace = k - 1;       /* the first of t1..t6 equal to the entry */
		return gate_ok(S, S->cubeGate[idx], r, t_min);
	}
	return 0;
}

static Hit miss(void) { Hit h = { 0, 0.0f, 0, 0.0f, 0.0f, -1, -1 }; return h; }

static Hit prim_hit(const RtSceneDesc* S, uint32_t kind, uint32_t idx, const Ray* r, float tMin, float tMax, Counts* c)
{
	Hit h = miss();
	float t, u = 0.0f, v = 0.0f;
	int32_t face = -1;
	if (kind == RT_REF_TRI)
	{
		c->tri++;
		if (triangle_hit(S, idx, r, tMin, tMax, &t, &u, &v)) { h.hit = 1; h.t = t; h.rank = S->triRank[idx]; h.u = u; h.v = v; h.mat = (int32_t)S->materials[S->triCold[idx].material].type; }
	}
	else if (kind == RT_REF_SPHERE)
	{
		c->sphere++;
		if (sphere_hit(S, idx, r, tMin, tMax, &t)) { h.hit = 1; h.t = t; h.rank = S->sphereRank[idx]; h.mat = (int32_t)S->materials[S->sphereMaterial[idx]].type; }
	}
	else
	{
		c->cube++;
		if (cube_hit(S, idx, r, tMin, tMax, &t, &face)) { h.hit = 1; h.t = t; h.rank = S->cubeRank[idx]; h.face = face; h.mat = (int32_t)S->materials[S->cubes[idx].material].type; }
	}
	return h;
}

/* bvh.cc:90-104: the closer hit wins, ties go to the RIGHT child.  In the reference topology "right" is the
 * same as "higher in-order rank"; on the device's own tree the structural order means nothing, so the rule is
 * applied in its closed form (minimum t, ties -> highest rank). */
static Hit combine(Hit l, Hit r)
{
	if (l.hit && r.hit)
	{
		if (!g_useTraversalTree) return (l.t < r.t) ? l : r;
		if (l.t < r.t) return l;
		if (r.t < l.t) return r;
		return (l.rank > r.rank) ? l : r;
	}
	if (l.hit) return l;
	return r;
}

/* `ref` with its box already accepted by the caller (the reference tests a node's own box on entry).
 * `nodes` is the reference topology (S->refNodes) -- or, for the equivalence tests, the device traversal
 * tree (S->nodes), visited exhaustively in the same way. */
static Hit visit(const RtSceneDesc* S, const RtNode* nodes, uint32_t ref, const Ray* r, float tMin, float tMax, Counts* c)
{
	const uint32_t kind = RT_REF_KIND(ref), idx = RT_REF_INDEX(ref);
	switch (kind)
	{
	case RT_REF_NODE: {
		const RtNode* n = &nodes[idx];
		Hit l = miss(), rr = miss();
		/* children that are bare primitives carry an infinite box: the reference does not box-test them */
		if (isinf(n->lmin[0]) || (c->box++, box_hit(n->lmin, n->lmax, r, tMin, tMax))) l = visit(S, nodes, n->lref, r, tMin, tMax, c);
		if (RT_REF_KIND(n->rref) != RT_REF_NONE)
			if (isinf(n->rmin[0]) || (c->box++, box_hit(n->rmin, n->rmax, r, tMin, tMax))) rr = visit(S, nodes, n->rref, r, tMin, tMax, c);
		return combine(l, rr);
	}
	case RT_REF_TRI: case RT_REF_SPHERE: case RT_REF_CUBE:
		return prim_hit(S, kind, idx, r, tMin, tMax, c);
	case RT_REF_TRI2:    return combine(prim_hit(S, RT_REF_TRI, idx, r, tMin, tMax, c), prim_hit(S, RT_REF_TRI, idx + 1, r, tMin, tMax, c));
	case RT_REF_SPHERE2: return combine(prim_hit(S, RT_REF_SPHERE, idx, r, tMin, tMax, c), prim_hit(S, RT_REF_SPHERE, idx + 1, r, tMin, tMax, c));
	case RT_REF_CUBE2:   return combine(prim_hit(S, RT_REF_CUBE, idx, r, tMin, tMax, c), prim_hit(S, RT_REF_CUBE, idx + 1, r, tMin, tMax, c));
	default: return miss();
	}
}

/* The 4-wide tree the device walks (RtNode4, csrc/host/bvh_sah.cc: RtCollapseToWide), visited exhaustively. */
static Hit visit_wide(const RtSceneDesc* S, uint32_t ref, const Ray* r, float tMin, float tMax, Counts* c)
{
	if (RT_REF_KIND(ref) != RT_REF_NODE) return visit(S, S->nodes, ref, r, tMin, tMax, c);
	const RtNode4* n = &S->wideNodes[RT_REF_INDEX(ref)];
	Hit best = miss();
	for (int i = 0; i < 4; ++i)
	{
		if (n->ref[i] == RT_REF_ABSENT) continue;
		const float lo[3] = { n->lox[i], n->loy[i], n->loz[i] }, hi[3] = { n->hix[i], n->hiy[i], n->hiz[i] };
		c->box++;
		if (!box_hit(lo, hi, r, tMin, tMax)) continue;
		best = combine(best, visit_wide(S, n->ref[i], r, tMin, tMax, c));
	}
	return best;
}

/* The quantized 64-byte nodes the kernels actually fetch (RtNodeQ4): boxes decoded with rt_q4_plane, then tested
 * with the reference's slab test (the device uses a conservative ray-space form of the same decoded boxes). */
static Hit visit_quant(const RtSceneDesc* S, uint32_t ref, const Ray* r, float tMin, float tMax, Counts* c)
{
	if (RT_REF_KIND(ref) != RT_REF_NODE) return visit(S, S->nodes, ref, r, tMin, tMax, c);
	const RtNodeQ4* n = &S->quantNodes[RT_REF_INDEX(ref)];
	const float sc[3] = { n->scaleX, n->scaleY, n->scaleZ };
	Hit best = miss();
	for (int i = 0; i < 4; ++i)
	{
		if (n->ref[i] == RT_REF_ABSENT) continue;
		float lo[3], hi[3];
		for (int a = 0; a < 3; ++a)
		{
			lo[a] = rt_q4_plane((n->qlo[a] >> (8 * i)) & 255u, sc[a], n->base[a]);
			hi[a] = rt_q4_plane((n->qhi[a] >> (8 * i)) & 255u, sc[a], n->base[a]);
		}
		c->box++;
		if (!box_hit(lo, hi, r, tMin, tMax)) continue;
		best = combine(best, visit_quant(S, n->ref[i], r, tMin, tMax, c));
	}
	return best;
}

/* Mode 4: the quantized nodes tested the way the KERNELS test them (csrc/device/rt_traverse.cuh trav_step): planes are never
 * decoded to coordinates; the ray parameter of a plane is t = m * (S * idc) + (base - o) * idc with idc = 1/d clamped to
 * +-1e18, one rounding per operation exactly as the device's __fmul_rn / __fmaf_rn produce them, near planes pulled in and
 * far planes pushed out by kSlack * |(base - o) * idc|, the final interval widened by kSlack * |t| (+ tMin on the far side).
 * Visited exhaustively (limit = FLT_MAX).  A test that lets fewer rays through than AABB::Hit on the exact boxes would lose
 * hits: tests/test_cpu_host.py compares this mode with the reference topology on adversarial rays, without a GPU. */
static int device_child_test(const RtNodeQ4* n, int k, const Ray* r, float tMin, float limit)
{
	const float kSlack = 3.81469727e-6f, lim = 1.0e18f;
	const float o[3] = { r->o.x, r->o.y, r->o.z }, d[3] = { r->d.x, r->d.y, r->d.z };
	const float sc[3] = { n->scaleX, n->scaleY, n->scaleZ };
	float tn = 0.0f, tf = 0.0f;
	for (int a = 0; a < 3; ++a)
	{
		float idc = 1.0f / d[a];
		idc = fminf(fmaxf(idc, -lim), lim);
		const float av = sc[a] * idc;
		const float diff = n->base[a] - o[a];
		const float b = diff * idc;
		const float bn = fmaf(-kSlack, fabsf(b), b), bf = fmaf(kSlack, fabsf(b), b);
		const int neg = idc < 0.0f;
		const uint32_t nearByte = ((neg ? n->qhi[a] : n->qlo[a]) >> (8 * k)) & 255u, farByte = ((neg ? n->qlo[a] : n->qhi[a]) >> (8 * k)) & 255u;
		union { uint32_t u; float f; } mn, mf;
		mn.u = 0x3F000000u | (nearByte << 16); mf.u = 0x3F000000u | (farByte << 16);
		const float t0 = fmaf(mn.f, av, bn), t1 = fmaf(mf.f, av, bf);
		tn = a == 0 ? t0 : fmaxf(tn, t0);
		tf = a == 0 ? t1 : fminf(tf, t1);
	}
	const float e = fmaxf(fmaf(-kSlack, fabsf(tn), tn), tMin);
	return e <= fminf(fmaf(kSlack, fabsf(tf), tf) + tMin, limit);
}

static Hit visit_quant_device(const RtSceneDesc* S, uint32_t ref, const Ray* r, float tMin, float tMax, Counts* c)
{
	if (RT_REF_KIND(ref) != RT_REF_NODE) return visit(S, S->nodes, ref, r, tMin, tMax, c);
	const RtNodeQ4* n = &S->quantNodes[RT_REF_INDEX(ref)];
	Hit best = miss();
	for (int i = 0; i < 4; ++i)
	{
		if (n->ref[i] == RT_REF_ABSENT) continue;
		c->box++;
		if (!device_child_test(n, i, r, tMin, tMax)) continue;
		best = combine(best, visit_quant_device(S, n->ref[i], r, tMin, tMax, c));
	}
	return best;
}

/* Host-side check used by the tests: every decoded box must contain the exact box of the same child (clamped to
 * +-RT_Q4_COORD_LIMIT).  Returns the number of violations (0 expected). */
uint64_t rt_oracle_check_quantization(const RtSceneDesc* S)
{
	uint64_t bad = 0;
	for (uint32_t i = 0; i < S->numWideNodes; ++i)
	{
		const RtNode4* w = &S->wideNodes[i];
		const RtNodeQ4* n = &S->quantNodes[i];
		const float sc[3] = { n->scaleX, n->scaleY, n->scaleZ };
		for (int k = 0; k < 4; ++k)
		{
			if (w->ref[k] != n->ref[k]) { bad++; continue; }
			if (w->ref[k] == RT_REF_ABSENT) continue;
			const float wl[3] = { w->lox[k], w->loy[k], w->loz[k] }, wh[3] = { w->hix[k], w->hiy[k], w->hiz[k] };
			for (int a = 0; a < 3; ++a)
			{
				const float lo = rt_q4_plane((n->qlo[a] >> (8 * k)) & 255u, sc[a], n->base[a]);
				const float hi = rt_q4_plane((n->qhi[a] >> (8 * k)) & 255u, sc[a], n->base[a]);
				const float el = wl[a] < -RT_Q4_COORD_LIMIT ? -RT_Q4_COORD_LIMIT : wl[a], eh = wh[a] > RT_Q4_COORD_LIMIT ? RT_Q4_COORD_LIMIT : wh[a];
				if (!(lo <= el) || !(hi >= eh)) bad++;
			}
		}
	}
	return bad;
}

/* 0 (default): the reference topology.  1: the binary SAH tree over the reference's leaf groups.
 * 2: that tree collapsed to 4-wide nodes (exact boxes).  3: the quantized 4-wide nodes the kernels traverse, decoded to
 * boxes.  4: the same nodes with the kernels' own ray-space test. */
void rt_oracle_select_tree(int useTraversalTree) { g_useTraversalTree = useTraversalTree; }

static Hit closest(const RtSceneDesc* S, const Ray* r, float tMin, Counts* c)
{
	c->box++;
	if (g_useTraversalTree)
	{
		if (!box_hit(S->rootMin, S->rootMax, r, tMin, FLT_MAX)) return miss();
		if (g_useTraversalTree == 2) return visit_wide(S, S->wideRootRef, r, tMin, FLT_MAX, c);
		if (g_useTraversalTree == 3) return visit_quant(S, S->wideRootRef, r, tMin, FLT_MAX, c);
		if (g_useTraversalTree == 4) return visit_quant_device(S, S->wideRootRef, r, tMin, FLT_MAX, c);
		return visit(S, S->nodes, S->rootRef, r, tMin, FLT_MAX, c);
	}
	if (!box_hit(S->refRootMin, S->refRootMax, r, tMin, FLT_MAX)) return miss();
	return visit(S, S->refNodes, S->refRootRef, r, tMin, FLT_MAX, c);
}

/* ---- exported ------------------------------------------------------------------------------------ */

/* rays: 8 floats each (o.xyz, time, d.xyz, unused); counts4 (nullable): box, tri, sphere, cube tests */
void rt_oracle_trace(const RtSceneDesc* S, const float* rays, int64_t numRays, float tMin,
                     int32_t* outRank, float* outT, uint64_t* counts4)
{
	Counts c = { 0, 0, 0, 0 };
	for (int64_t i = 0; i < numRays; ++i)
	{
		const float* q = rays + 8 * i;
		Ray r; r.o = v3(q[0], q[1], q[2]); r.time = q[3]; r.d = v3(q[4], q[5], q[6]);
		Hit h = closest(S, &r, tMin, &c);
		outRank[i] = h.hit ? (int32_t)h.rank : -1;
		outT[i] = h.hit ? h.t : 0.0f;
	}
	if (counts4) { counts4[0] = c.box; counts4[1] = c.tri; counts4[2] = c.sphere; counts4[3] = c.cube; }
}

/* rt_oracle_trace plus what the hit record of a device path holds and where the path goes next (nullable outputs, n each):
 * outUV (2 floats per ray) = paramU, paramV of a triangle hit, else 0; outFace = 0..5 of a cube hit (device order), else -1;
 * outMat = RtMaterialType of the hit primitive's material, -1 on a miss. */
void rt_oracle_trace_hits(const RtSceneDesc* S, const float* rays, int64_t numRays, float tMin,
                          int32_t* outRank, float* outT, float* outUV, int32_t* outFace, int32_t* outMat, uint64_t* counts4)
{
	Counts c = { 0, 0, 0, 0 };
	for (int64_t i = 0; i < numRays; ++i)
	{
		const float* q = rays + 8 * i;
		Ray r; r.o = v3(q[0], q[1], q[2]); r.time = q[3]; r.d = v3(q[4], q[5], q[6]);
		Hit h = closest(S, &r, tMin, &c);
		outRank[i] = h.hit ? (int32_t)h.rank : -1;
		outT[i] = h.hit ? h.t : 0.0f;
		if (outUV) { outUV[2 * i] = h.hit ? h.u : 0.0f; outUV[2 * i + 1] = h.hit ? h.v : 0.0f; }
		if (outFace) outFace[i] = h.hit ? h.face : -1;
		if (outMat) outMat[i] = h.hit ? h.mat : -1;
	}
	if (counts4) { counts4[0] = c.box; counts4[1] = c.tri; counts4[2] = c.sphere; counts4[3] = c.cube; }
}

/* camera.h:44-53 with core/random.cc:44-50 (disk) and the shared counter stream */
static Ray camera_ray(const RtCamera* cam, float s, float t, uint64_t key, uint32_t* ctr)
{
	float u1 = rt_uniform(key, ++*ctr);
	float u2 = rt_uniform(key, ++*ctr);
	float rr = sqrtf(u1);
	float theta = 2.0f * (float)M_PI * u2;
	V3 rd = muls(v3(rr * cosf(theta), rr * sinf(theta), 0.0f), cam->lensRadius);
	V3 offset = add(muls(v3p(cam->u), rd.x), muls(v3p(cam->v), rd.y));
	float captureTime = cam->beginTime + cam->timePeriod * rt_uniform(key, ++*ctr);
	Ray r;
	r.o = add(v3p(cam->origin), offset);
	r.d = normalize(sub(sub(add(add(v3p(cam->topLeft), muls(v3p(cam->horizontal), s)), muls(v3p(cam->vertical), 1.0f - t)), v3p(cam->origin)), offset));
	r.time = captureTime;
	return r;
}

/* One unjittered camera ray per pixel (renderer.cc:256-260), rows [y0, y1). rayDump nullable (8 floats/pixel). */
void rt_oracle_primary(const RtSceneDesc* S, const RtCamera* cam, uint32_t width, uint32_t height,
                       uint32_t y0, uint32_t y1, float tMin, uint64_t frameSeed,
                       int32_t* outRank, float* outT, float* rayDump, uint64_t* counts4)
{
	Counts c = { 0, 0, 0, 0 };
	for (uint32_t y = y0; y < y1 && y < height; ++y)
		for (uint32_t x = 0; x < width; ++x)
		{
			const uint32_t pixel = y * width + x;
			uint32_t ctr = 0;
			Ray r = camera_ray(cam, (float)x / (float)width, (float)y / (float)height, rt_sample_key(frameSeed, pixel, 0u), &ctr);
			Hit h = closest(S, &r, tMin, &c);
			outRank[pixel] = h.hit ? (int32_t)h.rank : -1;
			outT[pixel] = h.hit ? h.t : 0.0f;
			if (rayDump)
			{
				float* q = rayDump + 8 * (size_t)pixel;
				q[0] = r.o.x; q[1] = r.o.y; q[2] = r.o.z; q[3] = r.time; q[4] = r.d.x; q[5] = r.d.y; q[6] = r.d.z; q[7] = 0.0f;
			}
		}
	if (counts4) { counts4[0] = c.box; counts4[1] = c.tri; counts4[2] = c.sphere; counts4[3] = c.cube; }
}
