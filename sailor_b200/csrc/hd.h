// hd.h — scalar/vector helpers shared by every kernel body.
//
// Every arithmetic helper here restates the exact operation ORDER of the glm / std / SSE call the reference uses,
// because hit IDs, barycentrics, BVH topology and flattened triangles must be bit-identical to the reference
// (north_star: "bit-exact primary hits").  The CUDA translation units are compiled with -fmad=false (no FMA
// contraction), -prec-div=true, -prec-sqrt=true, -ftz=false, i.e. IEEE-754 single like the g++ -ffp-contract=off
// reference build.  min/max are written as the reference's ternaries: CUDA's fminf/fmaxf drop NaNs, glm/std/SSE
// do not, and the slab test depends on that (SURVEY H2).
#pragma once
#include <stdint.h>
#include <math.h>
#include <float.h>
#include <string.h>

#if defined(__CUDACC__)
#define SPT_HD __host__ __device__ __forceinline__
#define SPT_HD_NOINLINE __host__ __device__
#else
#define SPT_HD inline
#define SPT_HD_NOINLINE inline
#endif

namespace spt
{
	struct V2 { float x, y; };
	struct V3 { float x, y, z; };
	struct alignas(16) V4 { float x, y, z, w; };

	SPT_HD V3 v3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
	SPT_HD V3 v3(float s) { return v3(s, s, s); }
	SPT_HD V2 v2(float x, float y) { V2 r; r.x = x; r.y = y; return r; }
	SPT_HD V4 v4(float x, float y, float z, float w) { V4 r; r.x = x; r.y = y; r.z = z; r.w = w; return r; }

	SPT_HD V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
	SPT_HD V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
	SPT_HD V3 operator*(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
	SPT_HD V3 operator/(V3 a, V3 b) { return v3(a.x / b.x, a.y / b.y, a.z / b.z); }
	SPT_HD V3 operator*(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
	SPT_HD V3 operator*(float s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
	SPT_HD V3 operator/(V3 a, float s) { return v3(a.x / s, a.y / s, a.z / s); }
	SPT_HD V3 operator-(V3 a) { return v3(-a.x, -a.y, -a.z); }
	SPT_HD V3 operator+(V3 a, float s) { return v3(a.x + s, a.y + s, a.z + s); }
	SPT_HD V3 operator-(V3 a, float s) { return v3(a.x - s, a.y - s, a.z - s); }
	SPT_HD V3 operator-(float s, V3 a) { return v3(s - a.x, s - a.y, s - a.z); }
	SPT_HD V2 operator+(V2 a, V2 b) { return v2(a.x + b.x, a.y + b.y); }
	SPT_HD V2 operator-(V2 a, V2 b) { return v2(a.x - b.x, a.y - b.y); }
	SPT_HD V2 operator*(float s, V2 a) { return v2(s * a.x, s * a.y); }
	SPT_HD bool eq0(V3 a) { return a.x == 0.0f && a.y == 0.0f && a.z == 0.0f; } // glm: v == vec3(0)

	// glm::dot(vec3): tmp = a*b; tmp.x + tmp.y + tmp.z (glm/detail/func_geometric.inl:48-56)
	SPT_HD float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
	SPT_HD float dot(V2 a, V2 b) { return a.x * b.x + a.y * b.y; }
	// glm::cross (func_geometric.inl:80-90)
	SPT_HD V3 cross(V3 x, V3 y) { return v3(x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y); }
	SPT_HD float length(V3 v) { return sqrtf(dot(v, v)); }
	// glm::normalize = v * inversesqrt(dot(v,v)), inversesqrt(x) = 1/sqrt(x)
	SPT_HD V3 normalize(V3 v) { const float s = 1.0f / sqrtf(dot(v, v)); return v * s; }

	// std::min / std::max / glm::min / glm::max as comparisons (NaN-order preserving)
	SPT_HD float std_min(float a, float b) { return (b < a) ? b : a; }
	SPT_HD float std_max(float a, float b) { return (a < b) ? b : a; }
	SPT_HD float glm_min(float x, float y) { return (y < x) ? y : x; }
	SPT_HD float glm_max(float x, float y) { return (x < y) ? y : x; }
	SPT_HD float sse_min(float a, float b) { return (a < b) ? a : b; } // _mm_min_ps: second operand on NaN / equal
	SPT_HD float sse_max(float a, float b) { return (a > b) ? a : b; } // _mm_max_ps
	SPT_HD float glm_clamp(float x, float lo, float hi) { return glm_min(glm_max(x, lo), hi); }
	SPT_HD V3 glm_clamp(V3 v, float lo, float hi) { return v3(glm_clamp(v.x, lo, hi), glm_clamp(v.y, lo, hi), glm_clamp(v.z, lo, hi)); }
	SPT_HD float std_clamp(float v, float lo, float hi) { return (v < lo) ? lo : ((hi < v) ? hi : v); }
	SPT_HD V3 glm_min(V3 a, V3 b) { return v3(glm_min(a.x, b.x), glm_min(a.y, b.y), glm_min(a.z, b.z)); }
	SPT_HD V3 glm_max(V3 a, V3 b) { return v3(glm_max(a.x, b.x), glm_max(a.y, b.y), glm_max(a.z, b.z)); }
	// glm::mix(x, y, a) with float a: x*(1-a) + y*a
	SPT_HD float glm_mix(float x, float y, float a) { return x * (1.0f - a) + y * a; }
	SPT_HD V3 glm_mix(V3 x, V3 y, float a) { return v3(glm_mix(x.x, y.x, a), glm_mix(x.y, y.y, a), glm_mix(x.z, y.z, a)); }

	SPT_HD float comp(V3 v, int a) { return a == 0 ? v.x : (a == 1 ? v.y : v.z); }

	SPT_HD uint32_t f2u(float f) { union { float f; uint32_t u; } c; c.f = f; return c.u; }
	SPT_HD float u2f(uint32_t u) { union { float f; uint32_t u; } c; c.u = u; return c.f; }

	// Order-preserving float <-> uint key, so min/max over a set (order independent) can use integer atomics.
	SPT_HD uint32_t float_key(float f) { const uint32_t u = f2u(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
	SPT_HD float key_float(uint32_t k) { return u2f((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k); }

	// 128-bit read-only load (LDG.E.128 through the non-coherent path on the device)
#if defined(__CUDA_ARCH__)
	__device__ __forceinline__ V4 ld4(const V4* p) { const float4 f = __ldg(reinterpret_cast<const float4*>(p)); V4 r; r.x = f.x; r.y = f.y; r.z = f.z; r.w = f.w; return r; }
	__device__ __forceinline__ uint4 ld4u(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
	__device__ __forceinline__ float ldf(const float* p) { return __ldg(p); }
	// start fetching a line whose address is known long before the (conditional, sequential) code that reads it gets there
	__device__ __forceinline__ void prefetch(const void* p) { asm volatile("prefetch.global.L1 [%0];" :: "l"(p)); }
	__device__ __forceinline__ uint32_t ldu(const uint32_t* p) { return __ldg(p); }
#else
	inline V4 ld4(const V4* p) { return *p; }
	inline void prefetch(const void*) {}
	inline float ldf(const float* p) { return *p; }
	inline uint32_t ldu(const uint32_t* p) { return *p; }
	struct U4 { uint32_t x, y, z, w; };
	inline U4 ld4u(const void* p) { return *reinterpret_cast<const U4*>(p); }
#endif

	// A scalar of a glTF buffer: an aligned load on the device (staged streams start at multiples of 4 bytes), memcpy on the host
	// (an accessor inside a file need not be aligned)
	template<class T> SPT_HD T load_as(const uint8_t* p)
	{
#if defined(__CUDA_ARCH__)
		return *reinterpret_cast<const T*>(p);
#else
		T v; memcpy(&v, p, sizeof(T)); return v;
#endif
	}

	// Component c of a stored vertex-attribute element as float (glTF 2.0 accessors, KHR_mesh_quantization): u8 v/255, u16 v/65535,
	// i8 max(v/127, -1), i16 max(v/32767, -1) when normalized, (float)v otherwise; u32 and unknown component types read 0.  The
	// loader (instance TRS) and DecodeStreamKernel (vertex streams) both decode through here, so both give the same bits.
	SPT_HD float DecodeComponent(const uint8_t* e, uint32_t componentType, bool normalized, uint32_t c)
	{
		switch (componentType)
		{
		case 5126: return load_as<float>(e + 4 * c);
		case 5121: { const float v = (float)e[c]; return normalized ? v / 255.0f : v; }
		case 5120: { const float v = (float)load_as<int8_t>(e + c); return normalized ? std_max(v / 127.0f, -1.0f) : v; }
		case 5123: { const float v = (float)load_as<uint16_t>(e + 2 * c); return normalized ? v / 65535.0f : v; }
		case 5122: { const float v = (float)load_as<int16_t>(e + 2 * c); return normalized ? std_max(v / 32767.0f, -1.0f) : v; }
		default: return 0.0f;
		}
	}

	// Entry i of a stored index list (u8 / u16 / u32; any other component type reads 0)
	SPT_HD uint32_t IndexAt(const uint8_t* p, uint32_t componentType, uint64_t i)
	{
		switch (componentType)
		{
		case 5121: return p[i];
		case 5123: return load_as<uint16_t>(p + 2 * i);
		case 5125: return load_as<uint32_t>(p + 4 * i);
		default: return 0u;
		}
	}

	// Reference constants
	constexpr float kPiSailor = 3.1415926f;            // Math::Pi (Runtime/Math/Math.h:14)
	constexpr float kPiGlm = 3.14159265358979323846264338327950288f; // glm::pi<float>()
	constexpr float kFltMax = 3.402823466e+38f;
}
