// rt_shade.cuh -- surface reconstruction, material scattering and miss shading.
// Device restatement of (all under raylib/):
//   HitResult fill-in      geom/triangle.cc:47-52, geom/sphere.cc:18-41, geom/cube.cc:25-39
//   tangent frame          geom/hit.cc:6-29
//   sampling helpers       core/random.cc:3-50
//   Lambertian/Metal/Dielectric/Mirror/DiffuseLight/Microfacet
//                          render/material.cc:195-431, render/material.h:50-169, render/brdf.h:14-115
//   sky + sun              render/renderer.cc:156-199
// Draw order per bounce (SURVEY N1): Lambertian 2, Metal 2, Dielectric 1, Microfacet 2, Mirror/Light 0.
#pragma once
#include "rt_traverse.cuh"
#include "rt_rng.h"

#define RT_BRDF_PI 3.14159265359f

struct RtRng
{
	uint64_t key;
	uint32_t ctr;
	RT_DEV float next() { return rt_uniform(key, ++ctr); }
};

struct RtSurface
{
	float3 p, n;
	float  u, v;             // HitResult::paramU / paramV
	float3 tangent, bitangent;
	uint32_t material;
};

// core/random.cc:3-24
RT_DEV float3 random_on_sphere(RtRng& rng)
{
	const float u1 = rng.next();
	const float u2 = rng.next();
	const float z = 1.0f - 2.0f * u1;
	const float r = sqrtf(fmaxf(0.0f, 1.0f - z * z));
	const float phi = 2.0f * 3.141592f * u2;
	return v3(r * rt_cosf(phi), r * rt_sinf(phi), z);
}

// core/random.cc:44-50
RT_DEV float3 random_in_disk(RtRng& rng)
{
	const float u1 = rng.next();
	const float u2 = rng.next();
	const float r = sqrtf(u1);
	const float theta = 2.0f * 3.14159265358979323846f * u2;
	return v3(r * rt_cosf(theta), r * rt_sinf(theta), 0.0f);
}

// render/camera.h:44-53 (the derived block is computed on the host, camera.h:55-78)
RT_DEV RtRay camera_ray(const RtCamera& cam, float s, float t, RtRng& rng)
{
	const float3 rd = cam.lensRadius * random_in_disk(rng);
	const float3 offset = (v3(cam.u) * rd.x) + (v3(cam.v) * rd.y);
	const float captureTime = cam.beginTime + cam.timePeriod * rng.next();
	const float3 o = v3(cam.origin) + offset;
	const float3 d = normalize3(v3(cam.topLeft) + s * v3(cam.horizontal) + (1.0f - t) * v3(cam.vertical) - v3(cam.origin) - offset);
	return make_ray(o, d, captureTime);
}

RT_DEV void build_basis(RtSurface& sf)
{
	float3 T = (fabsf(sf.n.x) > 0.9f) ? v3(0.0f, 1.0f, 0.0f) : v3(1.0f, 0.0f, 0.0f);
	sf.bitangent = normalize3(cross3(T, sf.n));
	sf.tangent = normalize3(cross3(sf.n, sf.bitangent));
}
RT_DEV float3 world_to_local(const RtSurface& sf, float3 v) { return v3(dot3(v, sf.tangent), dot3(v, sf.bitangent), dot3(v, sf.n)); }
RT_DEV float3 local_to_world(const RtSurface& sf, float3 v)
{
	return v3(dot3(v3(sf.tangent.x, sf.bitangent.x, sf.n.x), v),
	          dot3(v3(sf.tangent.y, sf.bitangent.y, sf.n.y), v),
	          dot3(v3(sf.tangent.z, sf.bitangent.z, sf.n.z), v));
}

// Rebuild the HitResult fields the shaders need from (ray, t, barycentrics, primitive).
RT_DEV void reconstruct_surface(const RtSceneView& S, const RtRay& r, const RtHit& h, RtSurface& sf)
{
	const uint32_t kind = RT_REF_KIND(h.ref), idx = RT_REF_INDEX(h.ref);
	sf.p = r.o + h.t * r.d;
	if (kind == RT_REF_TRI)
	{
		const RtTriCold* c = S.triCold + idx;
		const float4* cq = reinterpret_cast<const float4*>(c);
		const float4 c0 = ldg4(cq + 0), c1 = ldg4(cq + 1), c2 = ldg4(cq + 2), c3 = ldg4(cq + 3);
		const float3 n0 = v3(c0.x, c0.y, c0.z), n1 = v3(c0.w, c1.x, c1.y), n2 = v3(c1.z, c1.w, c2.x);
		const float k = 1.0f - h.bu - h.bv;
		sf.n = normalize3(k * n0 + h.bu * n1 + h.bv * n2);
		sf.u = k * c2.y + h.bu * c2.w + h.bv * c3.y;
		sf.v = k * c2.z + h.bu * c3.x + h.bv * c3.z;
		sf.material = __float_as_uint(c3.w);
	}
	else if (kind == RT_REF_SPHERE)
	{
		const float4 s = ldg4(S.spheres + idx);
		const float3 op = sf.p - v3(s.x, s.y, s.z);
		sf.n = op / s.w;
		sf.u = rt_atanf(op.y / op.x);
		sf.v = rt_acosf(op.z / s.w);
		sf.material = S.sphereMaterial[idx];
	}
	else
	{
		const int face = (int)h.bu;
		sf.n = face == 0 ? v3(-1.0f, 0.0f, 0.0f) : face == 1 ? v3(1.0f, 0.0f, 0.0f)
		     : face == 2 ? v3(0.0f, -1.0f, 0.0f) : face == 3 ? v3(0.0f, 1.0f, 0.0f)
		     : face == 4 ? v3(0.0f, 0.0f, -1.0f) : face == 5 ? v3(0.0f, 0.0f, 1.0f) : v3(0.0f);
		sf.u = 0.0f; sf.v = 0.0f;      // Cube::Hit leaves paramU/V unset in the reference
		sf.material = S.cubes[idx].material;
	}
}

// ------------------------------------------------------------------------------------------------
// Microfacet helpers (material.cc:16-190, brdf.h)

RT_DEV float clampf(float v, float lo, float hi) { return fmaxf(lo, fminf(hi, v)); }

RT_DEV float erf_inv(float x)
{
	float w, p;
	x = clampf(x, -.99999f, .99999f);
	w = -rt_logf((1.0f - x) * (1.0f + x));
	if (w < 5.0f)
	{
		w = w - 2.5f;
		p = 2.81022636e-08f;
		p = 3.43273939e-07f + p * w;
		p = -3.5233877e-06f + p * w;
		p = -4.39150654e-06f + p * w;
		p = 0.00021858087f + p * w;
		p = -0.00125372503f + p * w;
		p = -0.00417768164f + p * w;
		p = 0.246640727f + p * w;
		p = 1.50140941f + p * w;
	}
	else
	{
		w = sqrtf(w) - 3.0f;
		p = -0.000200214257f;
		p = 0.000100950558f + p * w;
		p = 0.00134934322f + p * w;
		p = -0.00367342844f + p * w;
		p = 0.00573950773f + p * w;
		p = -0.0076224613f + p * w;
		p = 0.00943887047f + p * w;
		p = 1.00167406f + p * w;
		p = 2.83297682f + p * w;
	}
	return p * x;
}

RT_DEV float erf_as(float x)
{
	const float a1 = 0.254829592f, a2 = -0.284496736f, a3 = 1.421413741f, a4 = -1.453152027f, a5 = 1.061405429f;
	const float pp = 0.3275911f;
	const int sign = (x < 0.0f) ? -1 : 1;
	x = fabsf(x);
	const float t = 1.0f / (1.0f + pp * x);
	const float y = 1.0f - (((((a5 * t + a4) * t) + a3) * t + a2) * t + a1) * t * rt_expf(-x * x);
	return (float)sign * y;
}

RT_DEV float sin_theta(float3 w) { return sqrtf(fmaxf(0.0f, 1.0f - w.z * w.z)); }
RT_DEV float cos_phi(float3 w) { const float s = sin_theta(w); return (s == 0.0f) ? 1.0f : clampf(w.x / s, -1.0f, 1.0f); }
RT_DEV float sin_phi(float3 w) { const float s = sin_theta(w); return (s == 0.0f) ? 0.0f : clampf(w.y / s, -1.0f, 1.0f); }

RT_DEV void beckmann_sample11(float cosThetaI, float U1, float U2, float* slope_x, float* slope_y)
{
	const float Pi = RT_BRDF_PI;
	if ((double)cosThetaI > .9999)
	{
		const float r = sqrtf(-rt_logf(1.0f - U1));
		const float sinPhi = rt_sinf(2.0f * Pi * U2);
		const float cosPhi = rt_cosf(2.0f * Pi * U2);
		*slope_x = r * cosPhi;
		*slope_y = r * sinPhi;
		return;
	}
	const float sinThetaI = sqrtf(fmaxf(0.0f, 1.0f - cosThetaI * cosThetaI));
	const float tanThetaI = sinThetaI / cosThetaI;
	const float cotThetaI = 1.0f / tanThetaI;

	float a = -1.0f, c = erf_as(cotThetaI);
	const float sample_x = fmaxf(U1, 1e-6f);

	const float thetaI = rt_acosf(cosThetaI);
	const float fit = 1.0f + thetaI * (-0.876f + thetaI * (0.4265f - 0.0594f * thetaI));
	float b = c - (1.0f + c) * rt_powf(1.0f - sample_x, fit);

	const float SQRT_PI_INV = 1.f / sqrtf(Pi);
	const float normalization = 1.0f / (1.0f + c + SQRT_PI_INV * tanThetaI * rt_expf(-cotThetaI * cotThetaI));

	int it = 0;
	while (++it < 10)
	{
		if (!(b >= a && b <= c)) b = 0.5f * (a + c);
		const float invErf = erf_inv(b);
		const float value = normalization * (1.0f + b + SQRT_PI_INV * tanThetaI * rt_expf(-invErf * invErf)) - sample_x;
		const float derivative = normalization * (1.0f - invErf * tanThetaI);
		if (fabsf(value) < 1e-5f) break;
		if (value > 0.0f) c = b; else a = b;
		b -= value / derivative;
	}
	*slope_x = erf_inv(b);
	*slope_y = erf_inv(2.0f * fmaxf(U2, 1e-6f) - 1.0f);
}

RT_DEV float3 beckmann_sample(float3 wi, float alpha_x, float alpha_y, float U1, float U2)
{
	const float3 wiStretched = normalize3(v3(alpha_x * wi.x, alpha_y * wi.y, wi.z));
	float slope_x, slope_y;
	beckmann_sample11(wiStretched.z, U1, U2, &slope_x, &slope_y);
	const float tmp = cos_phi(wiStretched) * slope_x - sin_phi(wiStretched) * slope_y;
	slope_y = sin_phi(wiStretched) * slope_x + cos_phi(wiStretched) * slope_y;
	slope_x = tmp;
	slope_x = alpha_x * slope_x;
	slope_y = alpha_y * slope_y;
	return normalize3(v3(-slope_x, -slope_y, 1.f));
}

RT_DEV float3 fresnel_schlick(float cosTheta, float3 F0) { return F0 + (1.0f - F0) * rt_powf(1.0f - cosTheta, 5.0f); }

RT_DEV float distribution_beckmann(float3 N, float3 H, float roughness)
{
	float cosH = dot3(N, H);
	if (roughness == 0.0f) return 1.0f;
	if (H.z < 0.0f) cosH = -cosH;
	const float cosH2 = cosH * cosH;
	const float rr = roughness * roughness;
	const float exp_x = (1.0f - cosH2) / (rr * cosH);
	const float num = (cosH > 0.0f ? 1.0f : 0.0f) * rt_expf(-exp_x);
	const float denom = RT_BRDF_PI * rr * cosH2 * cosH2;
	return num / denom;
}

RT_DEV float geometry_beckmann(float3 N, float3 H, float3 V, float roughness)
{
	const float thetaV = rt_acosf(dot3(N, V));
	const float tanThetaV = rt_tanf(thetaV);
	const float a = 1.0f / (roughness * tanThetaV);
	const float aa = a * a;
	if (dot3(V, H) / dot3(V, N) <= 0.0f) return 0.0f;
	if (a < 1.6f)
	{
		const float num = 3.535f * a + 2.181f * aa;
		const float denom = 1.0f + 2.276f * a + 2.577f * aa;
		return num / denom;
	}
	return 1.0f;
}

RT_DEV float geometry_smith_beckmann(float3 N, float3 H, float3 V, float3 L, float roughness)
{
	const float g2 = geometry_beckmann(N, H, V, roughness);
	const float g1 = geometry_beckmann(N, H, L, roughness);
	return 1.0f / (1.0f + g1 * g2);
}

// material.cc:387-395, :406-415, :342-350
RT_DEV float3 microfacet_albedo(const RtSceneView& S, const RtMaterial& m, float u, float v)
{
	if (m.tex[RT_TEX_ALBEDO] >= 0)
	{
		const float4 px = sample_texture(S, m.tex[RT_TEX_ALBEDO], u, v);
		return v3(px.x, px.y, px.z) * px.w;
	}
	return v3(m.color);
}
RT_DEV float3 microfacet_normal(const RtSceneView& S, const RtMaterial& m, float u, float v)
{
	if (m.tex[RT_TEX_NORMAL] >= 0)
	{
		const float4 px = sample_texture(S, m.tex[RT_TEX_NORMAL], u, v);
		return normalize3(2.0f * v3(px.x, px.y, px.z) - 1.0f);
	}
	return v3(0.0f, 0.0f, 1.0f);
}
RT_DEV float microfacet_roughness(const RtSceneView& S, const RtMaterial& m, float u, float v)
{
	return (m.tex[RT_TEX_ROUGHNESS] >= 0) ? sample_texture(S, m.tex[RT_TEX_ROUGHNESS], u, v).x : m.param0;
}
RT_DEV float3 microfacet_emitted(const RtSceneView& S, const RtMaterial& m, float u)
{
	// reference quirk: sampled at (u,u) and the comma expression keeps only the blue channel
	if (m.tex[RT_TEX_EMISSIVE] >= 0) return v3(sample_texture(S, m.tex[RT_TEX_EMISSIVE], u, u).z);
	return v3(m.emissive);
}
RT_DEV float microfacet_scattering_pdf(const RtSceneView& S, const RtMaterial& m, const RtSurface& sf, float3 WoWorld, float3 WiWorld)
{
	const float3 wo = world_to_local(sf, WoWorld);
	const float3 wi = world_to_local(sf, WiWorld);
	float3 wh = normalize3(wo + wi);
	if (wh.z < 0.0f) wh.z = -wh.z;
	const float3 n = microfacet_normal(S, m, sf.u, sf.v);
	const float roughness = microfacet_roughness(S, m, sf.u, sf.v);
	const float D = distribution_beckmann(n, wh, roughness);
	return D * absdot3(wh, n);
}

// ------------------------------------------------------------------------------------------------
// One bounce: the outcome of Material::Scatter + ScatteringPdf + Emitted for TraceScene's fold.
struct RtBounce
{
	float3 reflectance;   // outReflectance
	float  scatPdf;       // material->ScatteringPdf(hit, -d, scattered.d)
	float3 emitted;       // material->Emitted(hit, d)
	float  pdf;           // outPdf, forced to 0 when Scatter() returned false (no recursive term)
	float3 nextDir;       // scattered ray direction (origin is the hit point)
};

template<int MAT_TYPE>
RT_DEV void scatter(const RtSceneView& S, const RtMaterial& m, const RtRay& r, const RtSurface& sf, RtRng& rng, RtBounce& out)
{
	out.emitted = v3(0.0f);
	out.scatPdf = 1.0f / RT_BRDF_PI;      // Material::ScatteringPdf default (material.h:35-41)
	out.pdf = 0.0f;
	out.reflectance = v3(0.0f);
	out.nextDir = v3(0.0f);

	if (MAT_TYPE == RT_MAT_LAMBERTIAN)
	{
		float3 dir = random_on_sphere(rng);
		if ((double)dot3(dir, sf.n) < 0.0) dir = -dir;
		const float3 Wi = normalize3(dir);
		out.nextDir = Wi;
		out.reflectance = v3(m.color);
		out.pdf = absdot3(sf.n, Wi) / RT_BRDF_PI;
		out.scatPdf = fmaxf(0.0f, dot3(sf.n, Wi)) / RT_BRDF_PI;
	}
	else if (MAT_TYPE == RT_MAT_METAL)
	{
		const float3 ud = normalize3(r.d);
		const float3 reflected = reflect3(ud, sf.n);
		out.nextDir = reflected + m.param0 * random_on_sphere(rng);
		out.reflectance = v3(m.color);
		out.pdf = (dot3(out.nextDir, sf.n) > 0.0f) ? 1.0f : 0.0f;
	}
	else if (MAT_TYPE == RT_MAT_DIELECTRIC)
	{
		const float ref_idx = m.param0;
		float3 outward_normal;
		const float3 reflected = reflect3(r.d, sf.n);
		float ni_over_nt, reflect_prob, cosine;
		out.reflectance = v3(m.color);
		if (dot3(r.d, sf.n) > 0.0f)
		{
			outward_normal = -sf.n;
			ni_over_nt = ref_idx;
			cosine = ref_idx * dot3(r.d, sf.n) / length3(r.d);
		}
		else
		{
			outward_normal = sf.n;
			ni_over_nt = 1.0f / ref_idx;
			cosine = -dot3(r.d, sf.n) / length3(r.d);
		}
		// refract (vec3.h:131-140)
		float3 refracted = v3(0.0f);
		const float3 unit = normalize3(r.d);
		const float dt = dot3(unit, outward_normal);
		const float disc = 1.0f - ni_over_nt * ni_over_nt * (1.0f - dt * dt);
		if (disc > 0.0f)
		{
			refracted = ni_over_nt * (unit - outward_normal * dt) - outward_normal * sqrtf(disc);
			float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
			r0 = r0 * r0;
			reflect_prob = r0 + (1.0f - r0) * rt_powf(1.0f - cosine, 5.0f);
		}
		else
		{
			reflect_prob = 1.0f;
		}
		out.nextDir = (rng.next() < reflect_prob) ? reflected : refracted;
		out.pdf = 1.0f;
	}
	else if (MAT_TYPE == RT_MAT_MIRROR)
	{
		out.reflectance = v3(m.color);
		out.nextDir = reflect3(r.d, sf.n);
		out.pdf = 1.0f;
		out.scatPdf = 1.0f;
	}
	else if (MAT_TYPE == RT_MAT_LIGHT)
	{
		out.emitted = v3(m.color);      // Scatter() returns false: pdf stays 0
	}
	else if (MAT_TYPE == RT_MAT_MICROFACET)
	{
		// the tangent frame is the caller's business: TraceScene builds it before Scatter (renderer.cc:131), the debug
		// views never do and run on the zero frame of a default-constructed HitResult (geom/hit.h:16-36)
		const float3 baseColor = microfacet_albedo(S, m, sf.u, sf.v);
		const float roughness = microfacet_roughness(S, m, sf.u, sf.v);
		const float metallic = (m.tex[RT_TEX_METALLIC] >= 0) ? sample_texture(S, m.tex[RT_TEX_METALLIC], sf.u, sf.v).x : m.param1;

		const float3 N = microfacet_normal(S, m, sf.u, sf.v);
		const float3 Wo = world_to_local(sf, -r.d);
		// Sample_wh (material.cc:417-431)
		const float u0 = rng.next();
		const float u1 = rng.next();
		const bool flip = Wo.z < 0.0f;
		float3 Wh = beckmann_sample(flip ? -Wo : Wo, roughness, roughness, u0, u1);
		if (flip) Wh = -Wh;
		float3 Wi = reflect3(-Wo, Wh);
		const float NdotWi = absdot3(N, Wi);

		float3 F0 = v3(0.04f);
		F0 = mix3(F0, baseColor, metallic);
		const float3 F = fresnel_schlick(absdot3(Wh, Wo), F0);
		const float G = geometry_smith_beckmann(N, Wh, Wo, Wi, roughness);
		const float NDF = distribution_beckmann(N, Wh, roughness);

		const float3 kS = F;
		const float3 kD = 1.0f - kS;
		const float3 diffuse = baseColor * (1.0f - metallic);
		const float3 specular = (F * G * NDF) / (4.0f * NdotWi * absdot3(N, Wo) + 0.001f);

		Wi = local_to_world(sf, Wi);
		out.nextDir = Wi;
		out.reflectance = (kD * diffuse + kS * specular) * NdotWi;
		const float sp = microfacet_scattering_pdf(S, m, sf, -r.d, Wi);
		out.pdf = sp / (4.0f * dot3(Wo, Wh));
		out.scatPdf = sp;
		out.emitted = microfacet_emitted(S, m, sf.u);
	}
}

// Miss shading, sky part (renderer.cc:157-181).  Returns 0 + sky texel.
RT_DEV float3 sky_radiance(const RtSceneView& S, float3 d)
{
	float3 miss = v3(0.0f);
	if (S.skyTexture >= 0)
	{
		const float3 dir = normalize3(d);
		const float3 D = v3(dot3(v3(S.skyRotation + 0), dir), dot3(v3(S.skyRotation + 3), dir), dot3(v3(S.skyRotation + 6), dir));
		float u = rt_atan2f(D.z, D.x), v = rt_asinf(D.y);
		u *= 0.1591f; v *= 0.3183f;
		u += 0.5f; v += 0.5f;
		const RtTexture tx = S.textures[S.skyTexture];
		int32_t x = (int32_t)(u * (float)(tx.width - 1u));
		int32_t y = (int32_t)(v * (float)(tx.height - 1u));
		x = max(0, min((int32_t)tx.width - 1, x));
		y = max(0, min((int32_t)tx.height - 1, y));
		const float4 px = __ldg(S.texels + tx.texelOffset + (uint64_t)y * tx.width + (uint64_t)x);
		miss = miss + v3(px.x, px.y, px.z);
	}
	return miss;
}

// One step of TraceScene's recursion unwinding (renderer.cc:133-153):
//   radiance = 0; if (scattered && pdf > 0) radiance += reflectance * Li * scatPdf / pdf; radiance += emitted
RT_DEV float3 fold_bounce(float3 reflectance, float scatPdf, float pdf, float3 emitted, float3 Li)
{
	float3 radiance = v3(0.0f);
	if (pdf > 0.0f) radiance = radiance + ((reflectance * Li) * scatPdf) / pdf;
	radiance = radiance + emitted;
	return radiance;
}
