// rt_math.cuh -- float3 helpers whose operation ORDER mirrors the reference's vec3
// (raylib/core/vec3.h:10-229).  This translation unit is compiled with --fmad=false,
// IEEE division and square root, so every expression below rounds exactly like the
// reference built with g++ -O2 -ffp-contract=off on x86-64.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define RT_DEV __device__ __forceinline__

// Transcendentals: include/rt_libm.h, glibc's float algorithms restated operation for operation (double-precision
// polynomials, the library's own tables), so the shaders consume the SAME BITS as the reference's host build; CUDA's
// libdevice functions are 1-2 ulp away from glibc, enough to change images (profiles/r02c_exact_libm_variants.jsonl).
#include "rt_libm.h"

RT_DEV float3 v3(float x, float y, float z) { return make_float3(x, y, z); }
RT_DEV float3 v3(float s) { return make_float3(s, s, s); }
RT_DEV float3 v3(const float* p) { return make_float3(p[0], p[1], p[2]); }

RT_DEV float3 operator+(float3 a, float3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
RT_DEV float3 operator-(float3 a, float3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
RT_DEV float3 operator*(float3 a, float3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
RT_DEV float3 operator-(float3 a) { return v3(-a.x, -a.y, -a.z); }
RT_DEV float3 operator*(float3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
RT_DEV float3 operator*(float s, float3 a) { return v3(a.x * s, a.y * s, a.z * s); }
RT_DEV float3 operator/(float3 a, float s) { return v3(a.x / s, a.y / s, a.z / s); }     // true division (vec3.h:92-94)
RT_DEV float3 operator+(float3 a, float s) { return v3(a.x + s, a.y + s, a.z + s); }
RT_DEV float3 operator+(float s, float3 a) { return v3(a.x + s, a.y + s, a.z + s); }
RT_DEV float3 operator-(float s, float3 a) { return v3(s - a.x, s - a.y, s - a.z); }
RT_DEV float3 operator-(float3 a, float s) { return v3(a.x - s, a.y - s, a.z - s); }

RT_DEV float dot3(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
RT_DEV float absdot3(float3 a, float3 b) { return fabsf(a.x * b.x + a.y * b.y + a.z * b.z); }
RT_DEV float length3(float3 a) { return sqrtf(a.x * a.x + a.y * a.y + a.z * a.z); }
RT_DEV float3 cross3(float3 a, float3 b)
{
	return v3(a.y * b.z - a.z * b.y, -(a.x * b.z - a.z * b.x), a.x * b.y - a.y * b.x);
}
// vec3::Normalize: k = 1/len, three multiplies (vec3.h:49-54)
RT_DEV float3 normalize3(float3 a) { const float k = 1.0f / length3(a); return v3(a.x * k, a.y * k, a.z * k); }
// vec3::operator/=(float): multiply by the reciprocal (vec3.h:214-220)
RT_DEV float3 div_assign3(float3 a, float s) { const float k = 1.0f / s; return v3(a.x * k, a.y * k, a.z * k); }
RT_DEV float3 reflect3(float3 v, float3 n) { return v - 2.0f * dot3(v, n) * n; }
RT_DEV float3 mix3(float3 a, float3 b, float t) { return (1.0f - t) * a + t * b; }
RT_DEV float3 xyz(float4 q) { return v3(q.x, q.y, q.z); }

// 128-bit read-only loads of scene records (ld.global.nc.v4)
RT_DEV float4 ldg4(const float4* p) { return __ldg(p); }

// 256-bit read-only load (sm_100a: LDG.E.ENL2.256.CONSTANT).  Scene records are 64 B: two of these per node or
// triangle put half as many wavefronts through L1TEX as four 128-bit loads -- the traversal kernels are bound
// by that pipe, not by DRAM or issue slots (profiles/README.md).  `p` must be 32-byte aligned.
struct __align__(32) RtF8 { float4 lo, hi; };
// No L1 eviction policy: hints on the node and triangle loads measured within +-0.5 % (profiles/README.md).
RT_DEV RtF8 ldg8(const void* p)
{
	RtF8 r;
	asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
		: "=f"(r.lo.x), "=f"(r.lo.y), "=f"(r.lo.z), "=f"(r.lo.w), "=f"(r.hi.x), "=f"(r.hi.y), "=f"(r.hi.z), "=f"(r.hi.w) : "l"(p));
	return r;
}
// Two IEEE fused multiply-adds in one instruction (sm_100a: FFMA2, fma.rn.f32x2): {a.x*b.x+c.x, a.y*b.y+c.y}, each half
// rounded exactly like __fmaf_rn.  Used by the conservative slab test of the inner nodes (rt_traverse.cuh).
RT_DEV float2 fma2_rn(float2 a, float2 b, float2 c)
{
	float2 d;
	asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\t"
	    "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
	    "fma.rn.f32x2 rd, ra, rb, rc;\n\t"
	    "mov.b64 {%0, %1}, rd;\n\t}"
	    : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
	return d;
}
