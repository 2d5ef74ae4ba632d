// flatten.cc -- see flatten.h and include/rt_scene_format.h for the layout and the reference
// semantics it preserves.
#include "flatten.h"
#include "bvh_sah.h"
#include "compact_mesh.h"
#include "geom/scene.h"
#include "geom/primitives.h"
#include "render/material.h"
#include "render/camera.h"
#include "render/image.h"
#include "rt_checksum.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <memory>
#include <mutex>
#include <thread>
#include <typeinfo>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <unordered_map>

uint64_t RtFlatScene::HostBytes() const
{
	return (nodes.size() + refNodes.size()) * sizeof(RtNode) + wideNodes.size() * sizeof(RtNode4) + quantNodes.size() * sizeof(RtNodeQ4) + triHot.size() * sizeof(RtTriHot) + triCold.size() * sizeof(RtTriCold)
		+ triRank.size() * 4 + triGate.size() * 4 + gateBoxes.size() * 4 + spheres.size() * sizeof(RtSphere) + sphereMaterial.size() * 4 + sphereRank.size() * 4 + sphereGate.size() * 4 + cubeGate.size() * 4
		+ cubes.size() * sizeof(RtCube) + cubeRank.size() * 4 + materials.size() * sizeof(RtMaterial)
		+ textures.size() * sizeof(RtTexture) + texels.size() * 4;
}

static void Store3(float* dst, const vec3& v) { dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; }

struct RtSceneFlattener
{
	RtFlatScene& out;
	std::string& error;
	std::unordered_map<const Material*, uint32_t> materialIndex;
	const Material* lastMaterial = nullptr;
	uint32_t lastMaterialIndex = 0;
	std::map<std::pair<const Image2D*, bool>, int32_t> textureIndex;
	RtLeafGroups groups;                 // SAH build items: one per triangle (tight box), one per sphere/cube leaf group (gate box)
	std::vector<std::pair<uint32_t, uint32_t>> meshRanges;   // [begin, end) into groups: the triangles of one StaticMesh (two-level SAH build)
	std::vector<AABB> triBounds;         // per emitted triangle: exact vertex bounds
	uint32_t nextRank = 0;
	uint32_t maxNodeDepth = 0;
	uint32_t flags = 0;
	uint32_t materialTypeMask = 0;
	bool failed = false;

	struct Child { uint32_t ref; float lo[3], hi[3]; uint32_t refBoxTests; };

	// Parallel graph walk.  The serial walk of the scene's upper levels only PLACES a StaticMesh: the index ranges its
	// subtree will occupy follow from its triangle count alone (the reference build is a median split down to leaves of one
	// or two, geom/bvh.cc:57-71), its materials are merged into the table in walk order, and the subtree itself is written
	// afterwards by a worker thread -- a flattener in `direct` mode that stores at its own cursors into the scene's arrays,
	// which were sized once without being touched (RtArray).  The result is bit-identical to the serial walk.
	bool direct = false;                       // worker: write at the cursors below instead of appending
	uint32_t cTri = 0, cGate = 0, cNode = 0, cGroup = 0;
	uint32_t triBoundsBase = 0;                // direct: triBounds is local to the mesh, indexed by (triangle - this)
	RtLeafGroups* groupsOut = nullptr;
	const std::unordered_map<const Material*, uint32_t>* sharedMaterials = nullptr;
	struct Placement
	{
		const StaticMesh* mesh; uint32_t triBase, rankBase, gateBase, nodeBase, groupBase, tris, gates, nodes, depth; Child* result;
		const RtCompactMesh* fragment = nullptr;       // OBJ fast path: the mesh's records exist already, copy + re-base them
		std::vector<uint32_t> materialRemap;           // fragment: local material index -> scene material index
	};
	std::vector<Placement> placements;
	bool parallelWalk = false;
	std::vector<std::unique_ptr<Child>> placedChildren;
	std::unordered_map<uint32_t, std::pair<uint32_t, uint32_t>> shapeMemo;     // triangles -> (leaf nodes, inner nodes)

	RtSceneFlattener(RtFlatScene& inOut, std::string& inError) : out(inOut), error(inError) {}

	void Fail(const std::string& why) { if (!failed) { failed = true; error = why; } }

	// ---- textures & materials ----------------------------------------------------------------
	int32_t AddTexture(const Image2D* image, bool srgb)
	{
		if (!image || image->GetWidth() == 0 || image->GetHeight() == 0) return -1;
		auto key = std::make_pair(image, srgb);
		auto it = textureIndex.find(key);
		if (it != textureIndex.end()) return it->second;
		RtTexture tx;
		memset(&tx, 0, sizeof(tx));
		tx.texelOffset = out.texels.size() / 4;
		tx.width = image->GetWidth();
		tx.height = image->GetHeight();
		tx.srgb = srgb ? 1u : 0u;
		const std::vector<Pixel>& px = image->GetPixelArray();
		const size_t base = out.texels.size();
		out.texels.resize(base + px.size() * 4);
		memcpy(out.texels.data() + base, px.data(), px.size() * sizeof(Pixel));
		const int32_t index = (int32_t)out.textures.size();
		out.textures.push_back(tx);
		textureIndex[key] = index;
		return index;
	}

	int32_t AddTexture(const Texture2D* texture)
	{
		if (!texture || texture->mipmaps.empty() || !texture->mipmaps[0]) return -1;
		return AddTexture(texture->mipmaps[0].get(), texture->sampler.bSRGB);
	}

	uint32_t AddMaterial(const Material* material)
	{
		if (!material) { Fail("a primitive has a null material"); return 0; }
		if (material == lastMaterial) return lastMaterialIndex;          // neighbouring triangles share materials
		if (direct)
		{
			// worker thread: the table was completed by the placement; only look up
			auto shared = sharedMaterials->find(material);
			if (shared == sharedMaterials->end()) { Fail("internal: a mesh material was not registered by the placement"); return 0; }
			lastMaterial = material; lastMaterialIndex = shared->second;
			return shared->second;
		}
		auto it = materialIndex.find(material);
		if (it != materialIndex.end()) { lastMaterial = material; lastMaterialIndex = it->second; return it->second; }
		RtMaterial m;
		memset(&m, 0, sizeof(m));
		for (int i = 0; i < 5; ++i) m.tex[i] = -1;
		if (const Lambertian* lam = dynamic_cast<const Lambertian*>(material))
		{
			m.type = RT_MAT_LAMBERTIAN; Store3(m.color, lam->albedo);
		}
		else if (const Metal* metal = dynamic_cast<const Metal*>(material))
		{
			m.type = RT_MAT_METAL; Store3(m.color, metal->albedo); m.param0 = metal->fuzziness;
		}
		else if (const Dielectric* glass = dynamic_cast<const Dielectric*>(material))
		{
			m.type = RT_MAT_DIELECTRIC; Store3(m.color, glass->transmissionFilter); m.param0 = glass->ref_idx;
		}
		else if (const Mirror* mirror = dynamic_cast<const Mirror*>(material))
		{
			m.type = RT_MAT_MIRROR; Store3(m.color, mirror->baseColor);
		}
		else if (const DiffuseLight* light = dynamic_cast<const DiffuseLight*>(material))
		{
			m.type = RT_MAT_LIGHT; Store3(m.color, light->intensity);
		}
		else if (const MicrofacetMaterial* mf = dynamic_cast<const MicrofacetMaterial*>(material))
		{
			m.type = RT_MAT_MICROFACET;
			Store3(m.color, mf->albedoFallback);
			m.param0 = mf->roughnessFallback;
			m.param1 = mf->metallicFallback;
			Store3(m.emissive, mf->emissiveFallback);
			m.tex[RT_TEX_ALBEDO] = AddTexture(mf->albedoTexture);
			m.tex[RT_TEX_NORMAL] = AddTexture(mf->normalmapTexture);
			m.tex[RT_TEX_ROUGHNESS] = AddTexture(mf->roughnessTexture);
			m.tex[RT_TEX_METALLIC] = AddTexture(mf->metallicTexture);
			m.tex[RT_TEX_EMISSIVE] = AddTexture(mf->emissiveTexture);
			if (m.tex[RT_TEX_ALBEDO] >= 0) flags |= RT_SCENE_FLAG_ALPHA_TEST;
		}
		else
		{
			Fail("a primitive uses a Material subclass the GPU path does not know (only the six raylib materials are supported)");
			return 0;
		}
		materialTypeMask |= 1u << m.type;
		const uint32_t index = (uint32_t)out.materials.size();
		out.materials.push_back(m);
		materialIndex[material] = index;
		lastMaterial = material; lastMaterialIndex = index;
		return index;
	}

	// ---- primitives ---------------------------------------------------------------------------
	enum PrimKind { PK_NONE, PK_TRI, PK_SPHERE, PK_CUBE };

	static PrimKind Classify(const Hitable* h)
	{
		// exact type match (a typeid compare, no hierarchy walk: this runs once per primitive): a client subclass that
		// overrides Hit() is NOT the primitive the device implements and is reported as unsupported
		const std::type_info& type = typeid(*h);
		if (type == typeid(Triangle)) return PK_TRI;
		if (type == typeid(Sphere)) return PK_SPHERE;
		if (type == typeid(Cube)) return PK_CUBE;
		return PK_NONE;
	}

	uint32_t EmitPrimitive(const Hitable* h, PrimKind kind)
	{
		const uint32_t rank = nextRank++;
		if (kind == PK_TRI)
		{
			const Triangle* t = static_cast<const Triangle*>(h);
			RtTriHot hot;
			const vec3 e1 = t->v1 - t->v0, e2 = t->v2 - t->v0;
			hot.q[0] = t->v0.x; hot.q[1] = t->v0.y; hot.q[2] = t->v0.z;
			hot.q[3] = t->n.x;  hot.q[4] = t->n.y;  hot.q[5] = t->n.z;
			hot.q[6] = e1.x; hot.q[7] = e1.y; hot.q[8] = e1.z;
			hot.q[9] = e2.x; hot.q[10] = e2.y; hot.q[11] = e2.z;
			const uint32_t words[4] = { RT_NO_GATE, 0u, rank, 0u };      // gate + material are patched below
			memcpy(&hot.q[RT_TRI_GATE], words, 16);
			RtTriCold cold;
			Store3(cold.n0, t->n0); Store3(cold.n1, t->n1); Store3(cold.n2, t->n2);
			cold.st[0] = t->s0; cold.st[1] = t->t0; cold.st[2] = t->s1; cold.st[3] = t->t1; cold.st[4] = t->s2; cold.st[5] = t->t2;
			cold.material = AddMaterial(t->material);
			memcpy(&hot.q[RT_TRI_MATERIAL], &cold.material, 4);
			memcpy(&hot.q[RT_TRI_MATTYPE], &out.materials[cold.material].type, 4);
			triBounds.push_back(t->bounds);
			if (direct)
			{
				const uint32_t index = cTri++;
				out.triHot[index] = hot; out.triCold[index] = cold; out.triRank[index] = rank; out.triGate[index] = RT_NO_GATE;
				return index;
			}
			out.triHot.push_back(hot); out.triCold.push_back(cold); out.triRank.push_back(rank);
			out.triGate.push_back(RT_NO_GATE);
			return (uint32_t)out.triHot.size() - 1;
		}
		if (kind == PK_SPHERE)
		{
			const Sphere* s = static_cast<const Sphere*>(h);
			RtSphere rec;
			Store3(rec.center, s->center); rec.radius = s->radius;
			out.spheres.push_back(rec); out.sphereMaterial.push_back(AddMaterial(s->material)); out.sphereRank.push_back(rank);
			out.sphereGate.push_back(RT_NO_GATE);
			return (uint32_t)out.spheres.size() - 1;
		}
		const Cube* c = static_cast<const Cube*>(h);
		RtCube rec;
		memset(&rec, 0, sizeof(rec));
		Store3(rec.minBounds, c->minBounds); Store3(rec.maxBounds, c->maxBounds); Store3(rec.velocity, c->velocity);
		rec.timeStartMove = c->timeStartMove;
		rec.material = AddMaterial(c->material);
		out.cubes.push_back(rec); out.cubeRank.push_back(rank); out.cubeGate.push_back(RT_NO_GATE);
		return (uint32_t)out.cubes.size() - 1;
	}

	static uint32_t RefKind(PrimKind kind, bool pair)
	{
		switch (kind)
		{
		case PK_TRI: return pair ? RT_REF_TRI2 : RT_REF_TRI;
		case PK_SPHERE: return pair ? RT_REF_SPHERE2 : RT_REF_SPHERE;
		default: return pair ? RT_REF_CUBE2 : RT_REF_CUBE;
		}
	}

	static void InfiniteBox(Child& c)
	{
		const float inf = std::numeric_limits<float>::infinity();
		for (int i = 0; i < 3; ++i) { c.lo[i] = -inf; c.hi[i] = inf; }
	}

	// ---- graph walk -----------------------------------------------------------------------------
	// Returns how `h` appears as a child slot of its parent: the box the reference tests before
	// descending into it (none for bare primitives) and the reference to follow.
	// Registers the leaf group `ref` (one or two primitives of one kind) whose reference gate is `gate`.
	void AddGroup(const AABB& gate, uint32_t ref)
	{
		const uint32_t kind = RT_REF_KIND(ref), first = RT_REF_INDEX(ref);
		if (kind == RT_REF_TRI || kind == RT_REF_TRI2)
		{
			// triangles: one SAH item each (box filled in once the scene extent is known), shared gate
			const float g8[8] = { gate.minBounds.x, gate.minBounds.y, gate.minBounds.z, 0.0f, gate.maxBounds.x, gate.maxBounds.y, gate.maxBounds.z, 0.0f };
			uint32_t gateIndex;
			if (direct) { gateIndex = cGate++; memcpy(out.gateBoxes.data() + (size_t)gateIndex * 8, g8, sizeof(g8)); }
			else { gateIndex = (uint32_t)(out.gateBoxes.size() / 8); out.gateBoxes.insert(out.gateBoxes.end(), g8, g8 + 8); }
			const uint32_t n = (kind == RT_REF_TRI2) ? 2u : 1u;
			for (uint32_t i = 0; i < n; ++i)
			{
				out.triGate[first + i] = gateIndex;
				memcpy(&out.triHot[first + i].q[RT_TRI_GATE], &gateIndex, 4);
				RtLeafGroup item;
				const AABB& tb = triBounds[first + i - triBoundsBase];
				Store3(item.lo, tb.minBounds); Store3(item.hi, tb.maxBounds);
				item.ref = RT_MAKE_REF(RT_REF_TRI, first + i);
				if (direct) (*groupsOut)[cGroup++] = item;
				else groups.push_back(item);
			}
			return;
		}
		// spheres / cubes: the group keeps its gate as its box (their own tests are not tight enough to cull by) and
		// the accepted hit is checked against the exact gate, like a triangle's
		{
			const uint32_t gateIndex = (uint32_t)(out.gateBoxes.size() / 8);
			const float g8[8] = { gate.minBounds.x, gate.minBounds.y, gate.minBounds.z, 0.0f, gate.maxBounds.x, gate.maxBounds.y, gate.maxBounds.z, 0.0f };
			out.gateBoxes.insert(out.gateBoxes.end(), g8, g8 + 8);
			const uint32_t n = (kind == RT_REF_SPHERE2 || kind == RT_REF_CUBE2) ? 2u : 1u;
			for (uint32_t i = 0; i < n; ++i)
			{
				if (kind == RT_REF_SPHERE || kind == RT_REF_SPHERE2) out.sphereGate[first + i] = gateIndex;
				else out.cubeGate[first + i] = gateIndex;
			}
		}
		RtLeafGroup g;
		Store3(g.lo, gate.minBounds); Store3(g.hi, gate.maxBounds);
		g.ref = ref;
		groups.push_back(g);
	}

	// Widens the per-triangle boxes so that every ray the reference's triangle test can accept also passes the
	// box: that test leaves the plane by <= ~5 ulp of the ray-origin distance and the triangle outline by a few
	// ulp of its size (more for slivers), DESIGN.md "Traversal tree".
	void InflateTriangleItems(const float* sceneLo, const float* sceneHi)
	{
		float scale = 0.0f;
		for (int a = 0; a < 3; ++a)
		{
			const float lo = std::max(sceneLo[a], -1.0e18f), hi = std::min(sceneHi[a], 1.0e18f);
			scale = std::max(scale, std::max(std::abs(lo), std::abs(hi)));
			scale = std::max(scale, hi - lo);
		}
		const float absPad = scale * (1.0f / 65536.0f);
		for (RtLeafGroup& g : groups)
		{
			if (RT_REF_KIND(g.ref) != RT_REF_TRI) continue;
			const float dx = g.hi[0] - g.lo[0], dy = g.hi[1] - g.lo[1], dz = g.hi[2] - g.lo[2];
			const float pad = absPad + (dx + dy + dz) * (1.0f / 1024.0f);
			for (int a = 0; a < 3; ++a) { g.lo[a] -= pad; g.hi[a] += pad; }
		}
	}

	static size_t CountTriangles(const Hitable* h)
	{
		if (!h) return 0;
		if (typeid(*h) == typeid(BVHNode))
		{
			const BVHNode* node = static_cast<const BVHNode*>(h);
			return CountTriangles(node->left) + (node->right != node->left ? CountTriangles(node->right) : 0);
		}
		if (typeid(*h) == typeid(StaticMesh))
		{
			const StaticMesh* mesh = static_cast<const StaticMesh*>(h);
			const RtCompactMesh* compact = RtFindCompactMesh(mesh);
			return compact ? compact->NumTriangles() : mesh->triangles.size();
		}
		if (typeid(*h) == typeid(HitableList))
		{
			size_t n = 0;
			for (const Hitable* m : static_cast<const HitableList*>(h)->hitables) n += CountTriangles(m);
			return n;
		}
		return typeid(*h) == typeid(Triangle) ? 1 : 0;
	}

	// `gate`: box of the BVHNode that holds `h` directly (what the reference tested last before calling h->Hit)
	Child Emit(const Hitable* h, uint32_t nodeDepth, const AABB* gate)
	{
		Child me;
		me.ref = RT_MAKE_REF(RT_REF_NONE, RT_REF_INDEX_MASK);
		me.refBoxTests = 0;
		InfiniteBox(me);
		if (failed || !h) { if (!h) Fail("null scene element"); return me; }

		if (typeid(*h) == typeid(BVHNode))
		{
			const BVHNode* node = static_cast<const BVHNode*>(h);
			Store3(me.lo, node->box.minBounds); Store3(me.hi, node->box.maxBounds);
			const Hitable* l = node->left;
			const Hitable* r = (node->right == node->left) ? nullptr : node->right;
			if (!l) { Fail("empty BVH node (scene finalized with no elements?)"); return me; }
			const PrimKind lk = Classify(l), rk = r ? Classify(r) : PK_NONE;
			if (lk != PK_NONE && (!r || rk == lk))
			{
				// leaf BVHNode over one or two primitives of one kind: no record, the parent points at them
				const uint32_t first = EmitPrimitive(l, lk);
				if (r) EmitPrimitive(r, lk);
				me.ref = RT_MAKE_REF(RefKind(lk, r != nullptr), first);
				me.refBoxTests = 1;
				AddGroup(node->box, me.ref);
				return me;
			}
			uint32_t index;
			if (direct) index = cNode++;
			else { index = (uint32_t)out.refNodes.size(); out.refNodes.push_back(RtNode()); }
			if (nodeDepth + 1 > maxNodeDepth) maxNodeDepth = nodeDepth + 1;
			const Child cl = Emit(l, nodeDepth + 1, &node->box);
			Child cr; cr.ref = RT_MAKE_REF(RT_REF_NONE, RT_REF_INDEX_MASK); cr.refBoxTests = 0; InfiniteBox(cr);
			if (r) cr = Emit(r, nodeDepth + 1, &node->box);
			RtNode& rec = out.refNodes[index];
			memcpy(rec.lmin, cl.lo, 12); memcpy(rec.lmax, cl.hi, 12); rec.lref = cl.ref; rec.lRefBoxTests = cl.refBoxTests;
			memcpy(rec.rmin, cr.lo, 12); memcpy(rec.rmax, cr.hi, 12); rec.rref = cr.ref; rec.rRefBoxTests = cr.refBoxTests;
			me.ref = RT_MAKE_REF(RT_REF_NODE, index);
			me.refBoxTests = 1;
			return me;
		}
		if (typeid(*h) == typeid(StaticMesh))
		{
			const StaticMesh* mesh = static_cast<const StaticMesh*>(h);
			if (const RtCompactMesh* compact = RtFindCompactMesh(mesh))
			{
				// OBJ fast path (compact_mesh.h): the mesh finalized straight into flattened records
				if (!compact->finalized || !mesh->boundsValid) { Fail("a StaticMesh was added to the scene before Finalize()"); return me; }
				if (compact->NumTriangles() == 0) { Fail("empty BVH node (scene finalized with no elements?)"); return me; }
				return PlaceFragment(mesh, *compact, nodeDepth);
			}
			if (!mesh->bvh || !mesh->boundsValid) { Fail("a StaticMesh was added to the scene before Finalize()"); return me; }
			// StaticMesh::Hit = bounds test, then the mesh BVH (root box test again), static_mesh.cc:97-109
			// the mesh's materials enter the table in the order of its triangle list, before its subtree is walked: the same
			// rule for the serial walk and for the parallel one, which walks the subtree later on another thread
			for (const Triangle& tri : mesh->triangles) AddMaterial(tri.material);
			if (failed) return me;
			if (parallelWalk && !mesh->triangles.empty()) return Place(mesh, nodeDepth);
			const uint32_t firstGroup = (uint32_t)groups.size();
			Child inner = Emit(mesh->bvh, nodeDepth, gate);
			if (groups.size() > firstGroup) meshRanges.push_back({ firstGroup, (uint32_t)groups.size() });
			const bool sameBox = mesh->bounds.minBounds == mesh->bvh->box.minBounds && mesh->bounds.maxBounds == mesh->bvh->box.maxBounds;
			if (sameBox) { inner.refBoxTests += 1; return inner; }      // the two tests are the same test
			// different boxes: Finalize always recomputes the bounds, so this cannot happen through the API
			Fail("a StaticMesh's bounds differ from the root box of its BVH (mesh modified after Finalize?)");
			return me;
		}
		const PrimKind kind = Classify(h);
		if (kind != PK_NONE)
		{
			// bare primitive under an inner node: the reference calls its Hit() without a box test
			me.ref = RT_MAKE_REF(RefKind(kind, false), EmitPrimitive(h, kind));
			me.refBoxTests = 0;
			if (gate) AddGroup(*gate, me.ref);
			else Fail("internal: primitive without an enclosing BVH node");
			return me;
		}
		if (typeid(*h) == typeid(HitableList)) return EmitList(static_cast<const HitableList*>(h), nodeDepth, gate);
		Fail("a scene element is a Hitable subclass the GPU path does not know");
		return me;
	}

	// A raw HitableList as a scene element (geom/hit.cc:34-50): a linear closest-hit scan with a SHRINKING upper bound --
	// member i is asked Hit(r, tMin, closest) -- reached whenever the box of the BVHNode holding the list passes (the list
	// has no box test of its own).  In closed form the winner is the member with minimum t; on EQUAL t a later member
	// replaces the incumbent iff its own range test is inclusive (Triangle: t > tMax rejects, triangle.cc:25; Cube:
	// t7 <= tMax, cube.cc:20) and does not iff it is strict (Sphere: t < tMax, sphere.cc:16,27).  So among equal-t members
	// the last non-sphere wins, and if there are only spheres the FIRST one does.  Ordering the members "spheres in reverse
	// list order, then the others in list order" turns that into the rule the traversal already implements -- minimum t,
	// ties to the highest in-order rank -- so a list becomes a run of consecutive ranks under virtual inner nodes whose
	// boxes are infinite (no test) and every member's gate is the holder's box.
	// One difference is documented rather than reproduced: a member the reference's scan reaches with closest already
	// below its own t by rounding only (a few ulp) -- the same epsilon ties as everywhere else (DESIGN.md section 3).
	Child EmitList(const HitableList* list, uint32_t nodeDepth, const AABB* gate)
	{
		Child me;
		me.ref = RT_MAKE_REF(RT_REF_NONE, RT_REF_INDEX_MASK);
		me.refBoxTests = 0;
		InfiniteBox(me);
		if (!gate) { Fail("internal: HitableList without an enclosing BVH node"); return me; }
		if (list->hitables.empty()) { Fail("an empty HitableList was added as a scene element"); return me; }
		std::vector<const Hitable*> ordered;
		for (size_t i = list->hitables.size(); i-- > 0;)
		{
			const Hitable* m = list->hitables[i];
			if (!m || Classify(m) == PK_NONE)
			{
				Fail("a HitableList scene element may hold Sphere, Cube and Triangle members only (wrap meshes and nested lists in a BVHNode, as loader/obj_loader.cc:237 does)");
				return me;
			}
			if (Classify(m) == PK_SPHERE) ordered.push_back(m);
		}
		for (const Hitable* m : list->hitables) if (Classify(m) != PK_SPHERE) ordered.push_back(m);
		return EmitListRange(ordered, 0, ordered.size(), nodeDepth, *gate);
	}

	Child EmitListRange(const std::vector<const Hitable*>& members, size_t lo, size_t hi, uint32_t nodeDepth, const AABB& gate)
	{
		Child me;
		me.refBoxTests = 0;
		InfiniteBox(me);
		if (hi - lo == 1)
		{
			const PrimKind kind = Classify(members[lo]);
			me.ref = RT_MAKE_REF(RefKind(kind, false), EmitPrimitive(members[lo], kind));
			AddGroup(gate, me.ref);
			return me;
		}
		const uint32_t index = (uint32_t)out.refNodes.size();
		out.refNodes.push_back(RtNode());
		if (nodeDepth + 1 > maxNodeDepth) maxNodeDepth = nodeDepth + 1;
		const size_t mid = lo + (hi - lo) / 2;
		const Child cl = EmitListRange(members, lo, mid, nodeDepth + 1, gate);
		const Child cr = EmitListRange(members, mid, hi, nodeDepth + 1, gate);
		RtNode& rec = out.refNodes[index];
		memcpy(rec.lmin, cl.lo, 12); memcpy(rec.lmax, cl.hi, 12); rec.lref = cl.ref; rec.lRefBoxTests = 0;
		memcpy(rec.rmin, cr.lo, 12); memcpy(rec.rmax, cr.hi, 12); rec.rref = cr.ref; rec.rRefBoxTests = 0;
		me.ref = RT_MAKE_REF(RT_REF_NODE, index);
		return me;
	}

	// ---- parallel walk ---------------------------------------------------------------------------
	static void CollectMeshes(const Hitable* h, size_t& meshes, size_t& tris)
	{
		if (!h) return;
		if (typeid(*h) == typeid(BVHNode))
		{
			const BVHNode* node = static_cast<const BVHNode*>(h);
			CollectMeshes(node->left, meshes, tris);
			if (node->right != node->left) CollectMeshes(node->right, meshes, tris);
		}
		else if (typeid(*h) == typeid(StaticMesh))
		{
			const StaticMesh* mesh = static_cast<const StaticMesh*>(h);
			const RtCompactMesh* compact = RtFindCompactMesh(mesh);
			meshes++; tris += compact ? compact->NumTriangles() : mesh->triangles.size();
		}
	}

	// (leaf BVHNodes, inner BVHNodes) of the reference build over n triangles: n <= 2 is one leaf node, otherwise the list is
	// halved (geom/bvh.cc:57-71)
	std::pair<uint32_t, uint32_t> MeshShape(uint32_t n)
	{
		if (n <= 2) return { 1u, 0u };
		auto it = shapeMemo.find(n);
		if (it != shapeMemo.end()) return it->second;
		const auto l = MeshShape(n / 2), r = MeshShape(n - n / 2);
		const std::pair<uint32_t, uint32_t> s{ l.first + r.first, 1u + l.second + r.second };
		shapeMemo[n] = s;
		return s;
	}

	// The serial walk reached a finalized mesh: reserve the ranges its subtree will fill and hand it to the workers.
	Child Place(const StaticMesh* mesh, uint32_t nodeDepth)
	{
		placedChildren.emplace_back(new Child);
		Child& me = *placedChildren.back();
		me.ref = RT_MAKE_REF(RT_REF_NONE, RT_REF_INDEX_MASK);
		me.refBoxTests = 0;
		InfiniteBox(me);
		const uint32_t n = (uint32_t)mesh->triangles.size();
		const auto shape = MeshShape(n);
		Placement p;
		p.mesh = mesh;
		p.triBase = (uint32_t)out.triHot.size(); p.rankBase = nextRank; p.gateBase = (uint32_t)(out.gateBoxes.size() / 8);
		p.nodeBase = (uint32_t)out.refNodes.size(); p.groupBase = (uint32_t)groups.size();
		p.tris = n; p.gates = shape.first; p.nodes = shape.second; p.depth = nodeDepth;
		p.result = &me;
		// reserve the ranges: the arrays do not initialise new elements (RtArray), the pages are first touched by the worker
		out.triHot.resize(out.triHot.size() + n); out.triCold.resize(out.triCold.size() + n);
		out.triRank.resize(out.triRank.size() + n); out.triGate.resize(out.triGate.size() + n);
		out.gateBoxes.resize(out.gateBoxes.size() + (size_t)shape.first * 8);
		out.refNodes.resize(out.refNodes.size() + shape.second);
		groups.resize(groups.size() + n);
		nextRank += n;
		meshRanges.push_back({ p.groupBase, p.groupBase + n });
		placements.push_back(p);
		// what the parent records for this child is known without walking the subtree: StaticMesh::Hit tests the mesh bounds,
		// then the identical root box of the mesh BVH (static_mesh.cc:97-109): two box tests, one box
		const bool sameBox = mesh->bounds.minBounds == mesh->bvh->box.minBounds && mesh->bounds.maxBounds == mesh->bvh->box.maxBounds;
		if (!sameBox) { Fail("a StaticMesh's bounds differ from the root box of its BVH (mesh modified after Finalize?)"); return me; }
		Store3(me.lo, mesh->bvh->box.minBounds); Store3(me.hi, mesh->bvh->box.maxBounds);
		me.refBoxTests = 2;
		// the root of the subtree: its first inner record, or the leaf group itself for a mesh of one or two triangles
		me.ref = shape.second ? RT_MAKE_REF(RT_REF_NODE, p.nodeBase) : RT_MAKE_REF(n == 2 ? RT_REF_TRI2 : RT_REF_TRI, p.triBase);
		return me;
	}

	// A mesh from the OBJ fast path: its records were produced by StaticMesh::Finalize (RtCompactFinalize); reserve their
	// ranges, map its materials (in the order of its triangle list, like every mesh) and leave the copy to the workers.
	Child PlaceFragment(const StaticMesh* mesh, const RtCompactMesh& fragment, uint32_t nodeDepth)
	{
		placedChildren.emplace_back(new Child);
		Child& me = *placedChildren.back();
		InfiniteBox(me);
		Placement p;
		p.mesh = mesh; p.fragment = &fragment;
		p.materialRemap.reserve(fragment.distinctMaterials.size());
		for (const Material* m : fragment.distinctMaterials) p.materialRemap.push_back(AddMaterial(m));
		const uint32_t n = (uint32_t)fragment.triHot.size();
		p.triBase = (uint32_t)out.triHot.size(); p.rankBase = nextRank; p.gateBase = (uint32_t)(out.gateBoxes.size() / 8);
		p.nodeBase = (uint32_t)out.refNodes.size(); p.groupBase = (uint32_t)groups.size();
		p.tris = n; p.gates = (uint32_t)(fragment.gateBoxes.size() / 8); p.nodes = (uint32_t)fragment.refNodes.size(); p.depth = nodeDepth;
		p.result = &me;
		out.triHot.resize(out.triHot.size() + n); out.triCold.resize(out.triCold.size() + n);
		out.triRank.resize(out.triRank.size() + n); out.triGate.resize(out.triGate.size() + n);
		out.gateBoxes.resize(out.gateBoxes.size() + fragment.gateBoxes.size());
		out.refNodes.resize(out.refNodes.size() + fragment.refNodes.size());
		groups.resize(groups.size() + n);
		nextRank += n;
		maxNodeDepth = std::max(maxNodeDepth, nodeDepth + fragment.maxNodeDepth);
		meshRanges.push_back({ p.groupBase, p.groupBase + n });
		memcpy(me.lo, fragment.topLo, 12); memcpy(me.hi, fragment.topHi, 12);
		me.refBoxTests = 2;      // the mesh bounds, then the identical root box of its tree (static_mesh.cc:97-109)
		me.ref = RelocateRef(fragment.topRef, p);
		placements.push_back(std::move(p));
		return me;
	}

	static uint32_t RelocateRef(uint32_t ref, const Placement& p)
	{
		const uint32_t kind = RT_REF_KIND(ref);
		if (kind == RT_REF_NODE) return RT_MAKE_REF(kind, RT_REF_INDEX(ref) + p.nodeBase);
		if (kind == RT_REF_TRI || kind == RT_REF_TRI2) return RT_MAKE_REF(kind, RT_REF_INDEX(ref) + p.triBase);
		return ref;
	}

	void CopyFragment(const Placement& p)
	{
		const RtCompactMesh& f = *p.fragment;
		for (size_t t = 0; t < f.triHot.size(); ++t)
		{
			RtTriHot hot = f.triHot[t];
			RtTriCold cold = f.triCold[t];
			uint32_t words[4];
			memcpy(words, &hot.q[RT_TRI_GATE], 16);
			if (words[0] != RT_NO_GATE) words[0] += p.gateBase;
			words[1] = p.materialRemap[words[1]];
			words[2] += p.rankBase;
			words[3] = out.materials[words[1]].type;
			memcpy(&hot.q[RT_TRI_GATE], words, 16);
			cold.material = words[1];
			out.triHot[p.triBase + t] = hot;
			out.triCold[p.triBase + t] = cold;
			out.triRank[p.triBase + t] = words[2];
			out.triGate[p.triBase + t] = words[0];
			RtLeafGroup item = f.groups[t];
			item.ref = RelocateRef(item.ref, p);
			groups[p.groupBase + t] = item;
		}
		if (!f.gateBoxes.empty()) memcpy(out.gateBoxes.data() + (size_t)p.gateBase * 8, f.gateBoxes.data(), f.gateBoxes.size() * sizeof(float));
		for (size_t k = 0; k < f.refNodes.size(); ++k)
		{
			RtNode rec = f.refNodes[k];
			rec.lref = RelocateRef(rec.lref, p); rec.rref = RelocateRef(rec.rref, p);
			out.refNodes[p.nodeBase + k] = rec;
		}
	}

	void WalkPlacedMeshes()
	{
		if (placements.empty()) return;
		std::atomic<size_t> next(0);
		std::atomic<uint32_t> deepest(maxNodeDepth);
		std::mutex failMutex;
		auto worker = [&]()
		{
			for (;;)
			{
				const size_t i = next.fetch_add(1);
				if (i >= placements.size()) break;
				const Placement& p = placements[i];
				if (p.fragment) { CopyFragment(p); continue; }
				std::string subError;
				RtSceneFlattener sub(out, subError);
				sub.direct = true;
				sub.cTri = p.triBase; sub.cGate = p.gateBase; sub.cNode = p.nodeBase; sub.cGroup = p.groupBase;
				sub.nextRank = p.rankBase;
				sub.triBoundsBase = p.triBase;
				sub.triBounds.reserve(p.tris);
				sub.groupsOut = &groups;
				sub.sharedMaterials = &materialIndex;
				const Child top = sub.Emit(p.mesh->bvh, p.depth, nullptr);
				bool bad = sub.failed;
				if (!bad && (sub.cTri != p.triBase + p.tris || sub.cGate != p.gateBase + p.gates || sub.cNode != p.nodeBase + p.nodes ||
				             sub.cGroup != p.groupBase + p.tris || top.ref != p.result->ref))
				{
					bad = true;
					subError = "internal: a StaticMesh's BVH does not have the shape of the reference build (was it built by this library?)";
				}
				if (bad) { std::lock_guard<std::mutex> lock(failMutex); Fail(subError); }
				uint32_t seen = deepest.load();
				while (sub.maxNodeDepth > seen && !deepest.compare_exchange_weak(seen, sub.maxNodeDepth)) {}
			}
		};
		const unsigned threads = std::max(1u, std::min<unsigned>(std::thread::hardware_concurrency(), (unsigned)placements.size()));
		std::vector<std::thread> pool;
		for (unsigned t = 1; t < threads; ++t) pool.emplace_back(worker);
		worker();
		for (std::thread& th : pool) th.join();
		maxNodeDepth = deepest.load();
		placements.clear();
	}

	bool Run(const Scene* scene)
	{
		const BVHNode* root = scene->accelStruct;
		if (!root) { Fail("scene is not finalized (call Raylib_FinalizeScene)"); return false; }
		if (!root->left) { Fail("scene has no elements"); return false; }

		const auto tStart = std::chrono::steady_clock::now();
		{
			size_t meshCount = 0, meshTris = 0;
			CollectMeshes(root, meshCount, meshTris);
			const char* env = getenv("RAYLIB_B200_PARALLEL_WALK");
			parallelWalk = env ? atoi(env) != 0 : (meshCount >= 16 && meshTris >= (1u << 17));
			// size the per-triangle arrays once (growth by doubling would copy gigabytes on a 10 M-triangle scene)
			const size_t tris = CountTriangles(root);
			out.triHot.reserve(tris); out.triCold.reserve(tris); out.triRank.reserve(tris); out.triGate.reserve(tris);
			groups.reserve(tris); out.gateBoxes.reserve(tris * 8 + 64); out.refNodes.reserve(tris + 64);
			if (!parallelWalk) triBounds.reserve(tris);
		}
		auto msSince = [](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count(); };
		const Child top = Emit(root, 0, nullptr);
		const double msUpper = msSince(tStart);
		if (!failed) WalkPlacedMeshes();
		const double msWalk = msSince(tStart);
		if (failed) return false;
		if (out.triHot.size() > RT_REF_INDEX_MASK || out.refNodes.size() > RT_REF_INDEX_MASK)
		{
			Fail("scene exceeds 2^28 primitives or nodes");
			return false;
		}

		RtSceneDesc& d = out.desc;
		memset(&d, 0, sizeof(d));
		memcpy(d.refRootMin, top.lo, 12); memcpy(d.refRootMax, top.hi, 12);
		d.refRootRef = top.ref;
		d.refRootBoxTests = top.refBoxTests;
		d.refMaxDepth = maxNodeDepth;
		d.numLeaves = nextRank;
		{
			InflateTriangleItems(top.lo, top.hi);
			auto t0 = std::chrono::steady_clock::now();
			RtSahResult tree;
			// many meshes of comparable size (an OBJ with thousands of shapes, an instance scatter): one subtree per mesh, built
			// in parallel, under a small top tree; one huge mesh or a handful of elements: the one-level build
			const char* twoLevelEnv = getenv("RAYLIB_B200_SAH_TWO_LEVEL");
			const bool twoLevel = twoLevelEnv ? atoi(twoLevelEnv) != 0 : (meshRanges.size() >= 64 && groups.size() >= (1u << 18));
			if (twoLevel) RtBuildTwoLevelSahTree(groups, meshRanges, tree);
			else RtBuildBestSahTree(groups, tree);
			const double msSah = msSince(t0); t0 = std::chrono::steady_clock::now();
			RtWideResult wide;
			RtCollapseToWide(tree, wide);
			out.nodes.swap(tree.nodes);
			out.wideNodes.swap(wide.nodes);
			const double msWide = msSince(t0); t0 = std::chrono::steady_clock::now();
			RtQuantizeWide(out.wideNodes, out.quantNodes);
			if (getenv("RAYLIB_B200_VERBOSE"))
				fprintf(stderr, "raylib-b200: flatten: graph walk %.0f ms (upper levels %.0f ms), SAH build %.0f ms, 4-wide collapse %.0f ms, quantize %.0f ms\n", msWalk, msUpper, msSah, msWide, msSince(t0));
			memcpy(d.rootMin, tree.rootMin, 12); memcpy(d.rootMax, tree.rootMax, 12);
			d.rootRef = tree.rootRef;
			d.maxStackDepth = tree.maxDepth;
			d.treeKind = RT_TREE_SAH;
			d.wideRootRef = wide.rootRef;
			d.wideMaxStack = wide.maxStack;
		}
		RtLeafGroups().swap(groups);
		std::vector<AABB>().swap(triBounds);

		// sky panorama: addressed directly by texel (renderer.cc:176-180), never gamma-decoded
		d.skyTexture = AddTexture((const Image2D*)scene->skyPanorama, false);
		Rotator skyYaw; skyYaw.yaw = 90.0f;
		const vec3 cx = skyYaw.rotate(vec3(1.0f, 0.0f, 0.0f)), cy = skyYaw.rotate(vec3(0.0f, 1.0f, 0.0f)), cz = skyYaw.rotate(vec3(0.0f, 0.0f, 1.0f));
		d.skyRotation[0] = cx.x; d.skyRotation[1] = cy.x; d.skyRotation[2] = cz.x;
		d.skyRotation[3] = cx.y; d.skyRotation[4] = cy.y; d.skyRotation[5] = cz.y;
		d.skyRotation[6] = cx.z; d.skyRotation[7] = cy.z; d.skyRotation[8] = cz.z;
		Store3(d.sunIlluminance, scene->sunIlluminance);
		Store3(d.sunDirection, scene->sunDirection);
		d.flags = flags;
		d.materialTypeMask = materialTypeMask;

		RtBindFlatScene(out);
		return true;
	}

	static void FlattenCamera(const Camera* c, RtCamera& o)
	{
		memset(&o, 0, sizeof(o));
		Store3(o.origin, c->origin); o.lensRadius = c->lensRadius;
		Store3(o.topLeft, c->top_left); o.beginTime = c->beginTime;
		Store3(o.horizontal, c->horizontal); o.timePeriod = c->timePeriod;
		Store3(o.vertical, c->vertical);
		Store3(o.u, c->u);
		Store3(o.v, c->v);
	}
};

void RtBindFlatScene(RtFlatScene& out)
{
	RtSceneDesc& d = out.desc;
	d.nodes = out.nodes.data(); d.numNodes = (uint32_t)out.nodes.size();
	d.wideNodes = out.wideNodes.data(); d.numWideNodes = (uint32_t)std::max(out.wideNodes.size(), out.quantNodes.size());
	d.quantNodes = out.quantNodes.data();
	d.refNodes = out.refNodes.data(); d.numRefNodes = (uint32_t)out.refNodes.size();
	d.triHot = out.triHot.data(); d.triCold = out.triCold.data(); d.triRank = out.triRank.data(); d.numTris = (uint32_t)out.triHot.size();
	d.triGate = out.triGate.data(); d.gateBoxes = out.gateBoxes.data(); d.numGates = (uint32_t)(out.gateBoxes.size() / 8);
	d.spheres = out.spheres.data(); d.sphereMaterial = out.sphereMaterial.data(); d.sphereRank = out.sphereRank.data(); d.sphereGate = out.sphereGate.data(); d.numSpheres = (uint32_t)out.spheres.size();
	d.cubes = out.cubes.data(); d.cubeRank = out.cubeRank.data(); d.cubeGate = out.cubeGate.data(); d.numCubes = (uint32_t)out.cubes.size();
	d.materials = out.materials.data(); d.numMaterials = (uint32_t)out.materials.size();
	d.textures = out.textures.data(); d.numTextures = (uint32_t)out.textures.size();
	d.texels = out.texels.data(); d.numTexels = out.texels.size() / 4;
}

// ---- on-disk cache ---------------------------------------------------------------------------------------
namespace
{
	struct FlatFileHeader
	{
		char     magic[8];            // "RTFLAT01"
		uint32_t headerBytes;         // sizeof(FlatFileHeader)
		uint32_t descBytes;           // sizeof(RtSceneDesc): guards against a changed scene format
		uint32_t recordBytes[8];      // RtNodeQ4, RtNode, RtTriHot, RtTriCold, RtSphere, RtCube, RtMaterial, RtTexture
		uint64_t checksum;            // of everything after the header
		uint64_t payloadBytes;
	};
	static_assert(sizeof(FlatFileHeader) == 64, "flat-scene file header is 64 bytes");

	void FillRecordSizes(uint32_t* r)
	{
		r[0] = sizeof(RtNodeQ4); r[1] = sizeof(RtNode); r[2] = sizeof(RtTriHot); r[3] = sizeof(RtTriCold);
		r[4] = sizeof(RtSphere); r[5] = sizeof(RtCube); r[6] = sizeof(RtMaterial); r[7] = sizeof(RtTexture);
	}

	struct FlatWriter
	{
		FILE* f; RtChecksum sum; uint64_t bytes = 0; bool ok = true;
		void Raw(const void* data, size_t n) { if (n && fwrite(data, 1, n, f) != n) ok = false; sum.Add(data, n); bytes += n; }
		template<typename T, typename A> void Array(const std::vector<T, A>& v) { const uint64_t n = v.size(); Raw(&n, 8); Raw(v.data(), v.size() * sizeof(T)); }
	};
	struct FlatReader
	{
		FILE* f; RtChecksum sum; bool ok = true;
		void Raw(void* data, size_t n) { if (n && fread(data, 1, n, f) != n) ok = false; else sum.Add(data, n); }
		template<typename T, typename A> void Array(std::vector<T, A>& v, uint64_t limitBytes)
		{
			uint64_t n = 0; Raw(&n, 8);
			if (!ok || n > limitBytes / sizeof(T)) { ok = false; return; }       // a division: n * sizeof(T) could wrap
			v.resize((size_t)n);
			Raw(v.data(), (size_t)n * sizeof(T));
		}
	};

	template<typename IO> void FlatArrays(IO& io, RtFlatScene& s, uint64_t limit);
	template<> void FlatArrays<FlatWriter>(FlatWriter& io, RtFlatScene& s, uint64_t)
	{
		io.Array(s.quantNodes); io.Array(s.refNodes); io.Array(s.triHot); io.Array(s.triCold); io.Array(s.triRank); io.Array(s.triGate);
		io.Array(s.gateBoxes); io.Array(s.spheres); io.Array(s.sphereMaterial); io.Array(s.sphereRank); io.Array(s.sphereGate);
		io.Array(s.cubes); io.Array(s.cubeRank); io.Array(s.cubeGate); io.Array(s.materials); io.Array(s.textures); io.Array(s.texels);
	}
	template<> void FlatArrays<FlatReader>(FlatReader& io, RtFlatScene& s, uint64_t limit)
	{
		io.Array(s.quantNodes, limit); io.Array(s.refNodes, limit); io.Array(s.triHot, limit); io.Array(s.triCold, limit); io.Array(s.triRank, limit);
		io.Array(s.triGate, limit); io.Array(s.gateBoxes, limit); io.Array(s.spheres, limit); io.Array(s.sphereMaterial, limit);
		io.Array(s.sphereRank, limit); io.Array(s.sphereGate, limit); io.Array(s.cubes, limit); io.Array(s.cubeRank, limit); io.Array(s.cubeGate, limit);
		io.Array(s.materials, limit); io.Array(s.textures, limit); io.Array(s.texels, limit);
	}
}

bool RtSaveFlatScene(const RtFlatScene& flat, const char* path, std::string& error)
{
	if (!path || !*path) { error = "empty path"; return false; }
	const std::string tmp = std::string(path) + ".tmp";
	FILE* f = fopen(tmp.c_str(), "wb");
	if (!f) { error = std::string("cannot create ") + tmp; return false; }
	FlatFileHeader h;
	memset(&h, 0, sizeof(h));
	memcpy(h.magic, "RTFLAT01", 8);
	h.headerBytes = sizeof(h); h.descBytes = sizeof(RtSceneDesc);
	FillRecordSizes(h.recordBytes);
	bool ok = fwrite(&h, 1, sizeof(h), f) == sizeof(h);
	FlatWriter w{ f };
	RtSceneDesc scalars = flat.desc;       // pointers are meaningless on disk: RtBindFlatScene restores them
	scalars.numNodes = 0;                  // the binary SAH tree and the exact 4-wide nodes stay on the host that built them
	scalars.nodes = nullptr; scalars.wideNodes = nullptr; scalars.quantNodes = nullptr; scalars.refNodes = nullptr;
	scalars.triHot = nullptr; scalars.triCold = nullptr; scalars.triRank = nullptr; scalars.triGate = nullptr; scalars.gateBoxes = nullptr;
	scalars.spheres = nullptr; scalars.sphereMaterial = nullptr; scalars.sphereRank = nullptr; scalars.sphereGate = nullptr;
	scalars.cubes = nullptr; scalars.cubeRank = nullptr; scalars.cubeGate = nullptr; scalars.materials = nullptr; scalars.textures = nullptr; scalars.texels = nullptr;
	w.Raw(&scalars, sizeof(scalars));
	FlatArrays(w, const_cast<RtFlatScene&>(flat), 0);
	h.checksum = w.sum.h; h.payloadBytes = w.bytes;
	ok = ok && w.ok && fseek(f, 0, SEEK_SET) == 0 && fwrite(&h, 1, sizeof(h), f) == sizeof(h);
	ok = (fclose(f) == 0) && ok;
	if (!ok || rename(tmp.c_str(), path) != 0) { remove(tmp.c_str()); error = std::string("write failed: ") + path; return false; }
	return true;
}

bool RtLoadFlatScene(const char* path, RtFlatScene& out, std::string& error)
{
	out = RtFlatScene();
	FILE* f = path ? fopen(path, "rb") : nullptr;
	if (!f) { error = std::string("cannot open ") + (path ? path : "(null)"); return false; }
	FlatFileHeader h, expect;
	memset(&expect, 0, sizeof(expect));
	FillRecordSizes(expect.recordBytes);
	bool ok = fread(&h, 1, sizeof(h), f) == sizeof(h);
	if (!ok || memcmp(h.magic, "RTFLAT01", 8) != 0) { fclose(f); error = "not a flattened-scene file"; return false; }
	if (h.headerBytes != sizeof(h) || h.descBytes != sizeof(RtSceneDesc) || memcmp(h.recordBytes, expect.recordBytes, sizeof(h.recordBytes)) != 0)
	{
		fclose(f); error = "flattened-scene file was written by a build with a different scene format"; return false;
	}
	FlatReader r{ f };
	r.Raw(&out.desc, sizeof(out.desc));
	FlatArrays(r, out, h.payloadBytes);
	char extra;
	const bool atEnd = fread(&extra, 1, 1, f) == 0;
	fclose(f);
	if (!r.ok || !atEnd || r.sum.h != h.checksum) { out = RtFlatScene(); error = "flattened-scene file is truncated or corrupt"; return false; }
	// structural checks the kernels rely on
	const RtSceneDesc& d = out.desc;
	const bool sizesOk = out.triCold.size() == out.triHot.size() && out.triRank.size() == out.triHot.size() && out.triGate.size() == out.triHot.size()
		&& out.sphereMaterial.size() == out.spheres.size() && out.sphereRank.size() == out.spheres.size() && out.sphereGate.size() == out.spheres.size()
		&& out.cubeRank.size() == out.cubes.size() && out.cubeGate.size() == out.cubes.size() && out.gateBoxes.size() % 8 == 0 && out.texels.size() % 4 == 0
		&& d.numWideNodes == out.quantNodes.size() && d.numRefNodes == out.refNodes.size();
	if (!sizesOk) { out = RtFlatScene(); error = "flattened-scene file is inconsistent"; return false; }
	RtBindFlatScene(out);
	return true;
}

bool RtFlattenScene(const Scene* scene, RtFlatScene& out, std::string& error)
{
	out = RtFlatScene();
	RtSceneFlattener flattener(out, error);
	return flattener.Run(scene);
}

void RtFlattenCamera(const Camera* camera, RtCamera& out) { RtSceneFlattener::FlattenCamera(camera, out); }
