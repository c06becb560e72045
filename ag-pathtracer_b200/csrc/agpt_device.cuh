// agpt_device.cuh -- device-side scene tables, strict-fp math and ray/primitive tests.
//
// Every function states the reference lines it realises.  This translation unit is built
// with --fmad=false: a*b+c stays FMUL+FADD, `/` and sqrtf are IEEE (correctly rounded), so
// +,-,*,/,sqrt sequences written in the reference's operation order give the same bits as
// the g++ -O2 oracle on x86 (SURVEY 7 "hard parts").  min/max follow the template's
// re-definitions `a<b?a:b` / `a>b?a:b` (template/precomp.h:364-365) and std::min/std::max
// where the reference calls those -- they differ in which operand a NaN selects.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>

#include "agpt.h"

#define AGPT_PI      3.14159265358979323846264f
#define AGPT_INVPI   0.31830988618379067153777f
#define AGPT_INV2PI  0.15915494309189533576888f
#define AGPT_TWOPI   6.28318530717958647692528f
#define AGPT_EPSILON 0.0001f
#define AGPT_ONE_MINUS_EPS 0x1.fffffep-1f

// -DAGPT_DEBUG build (make debug -> libagpt_debug.so): in-kernel checks on stack depth, node / triangle
// indices, queue slots and the adaptive pixel lists.  A failed check records its code and value in g_agptDebug (no trap: the
// context stays usable) and agpt_debug_status() reports it.  compute-sanitizer is closed on the GPU
// pool this was developed on, so the small GPU tests are run once per round against this build.
enum { AGPT_DBG_STACK = 1, AGPT_DBG_NODE = 2, AGPT_DBG_TRI = 3, AGPT_DBG_QUEUE = 4, AGPT_DBG_PATH = 5, AGPT_DBG_PRIM = 6, AGPT_DBG_MATERIAL = 7,
       AGPT_DBG_LIST = 8 /* adaptive pixel list entry or pixel index */, AGPT_DBG_SAMPLE = 9 /* a pixel's samples past max_samples */,
       AGPT_DBG_GUIDE = 10 /* k_guides: path slot */, AGPT_DBG_TAP = 11 /* denoise, reprojection: filter or history tap outside the film */,
       AGPT_DBG_TEXTURE = 12 /* texture index of a material */, AGPT_DBG_TEXEL = 13 /* texel index of a lookup */,
       AGPT_DBG_MAPS = 14 /* material index into the map binding table */, AGPT_DBG_MASK = 15 /* material index into the mask table */,
       AGPT_DBG_EMIT = 16 /* material index into the emission table */ };
#ifdef AGPT_DEBUG
__device__ unsigned long long g_agptDebug[4];     // [0] failures, [1] first code, [2] first value, [3] checks executed
#define AGPT_CHECK(cond, code, value) do { atomicAdd(&g_agptDebug[3], 1ull); if (!(cond)) { \
	if (atomicAdd(&g_agptDebug[0], 1ull) == 0ull) { g_agptDebug[1] = (unsigned long long)(code); g_agptDebug[2] = (unsigned long long)(long long)(value); } } } while (0)
#else
#define AGPT_CHECK(cond, code, value) ((void)0)
#endif

struct DMesh {
	const float4* nodes;     // 2 x float4 per BVHNode; nullptr for a plain TriangleMesh
	const float4* tris;      // 3 x float4 per triangle, leaf order; tris[3j].w != 0 marks a triangle upstream rejects as degenerate
	const int* ids;          // original triangle number per slot
	const float4* normals;   // 3 x float4 per triangle or nullptr
	const float2* uvs;       // 3 x float2 per triangle or nullptr
	int n_nodes, n_tris;
};

// EXTENSION: sampling table of a plane or mesh area light with AGPT_LIGHT_SAMPLE_SHAPE (agpt.h), one per light.
struct DShapeLight {
	int cdfOff;              // meshes: Distribution1D::cdf over the triangle areas in slot order at shapeCdf[cdfOff .. cdfOff + n]
	int n;                   // triangles
	float area;              // total area; 0: never sampled (not a sampled shape light, or nothing to sample)
	float pad;
};
struct DShapeTables {        // passed beside DScene, to the kernels that sample shapes only
	const DShapeLight* lights;       // n_lights entries, or nullptr when no light samples its shape
	const float* cdf;
};

// EXTENSION: image textures on the base colour of Disney materials (agpt.h agpt_upload_textures), passed beside DScene to the
// textured instantiations only.
struct DTexture {
	int width, height;
	long long off;               // first texel in DTexTables::texels
};
// one material's bindings (agpt_material_textures): two 128-bit loads
struct __align__(16) DMatMaps {
	int base, roughnessMetallic, normal;   // texture indices or -1
	float normalScale;
	float color[3];                        // base colour when base < 0 and roughnessMetallic >= 0
	float pad;
};
struct DTexTables {
	const float4* texels;        // every texture's texels, row-major, .w unused: one bilinear lookup = four 128-bit loads
	const DTexture* textures;
	const int* matTex;           // per material: its base-colour texture, or -1
	int nTextures;
	long long nTexels;
	const DMatMaps* matMaps;     // per material: its map bindings (agpt_upload_material_textures); read by the TEX == 2 kernels only
	int nMatMaps;
};
// EXTENSION: alpha masks (agpt.h agpt_upload_alpha_masks), passed beside DScene to the MASK trace instantiations only; DScene's
// layout, which every other kernel shares, stays as it is.
struct DMaskTables {
	DTexTables tt;                   // the resident texels and textures (the bindings are not read)
	const agpt_alpha_mask* masks;    // per material: {texture or -1, channel, cutoff}
	int nMasks;
};
// EXTENSION: emissive materials (agpt.h agpt_upload_emission), passed to k_shade_a_emit only, beside DScene.
struct DEmitTables {
	DTexTables tt;                   // the resident texels and textures (the bindings are not read)
	const agpt_emission* rows;       // per material: {texture or -1, factor}
	int nRows;
};

struct DScene {
	const agpt_prim* prims;
	const int* sphereRun;            // per primitive: length of the run of sphere primitives with consecutive payloads starting here (0: not a sphere)
	const float4* sphereRunBox;      // per primitive, 3 x float4 for run starts: grown box min.xyz,max.x | max.yz,-,- | centre.xyz, max |O-centre|^2 for the cull to be safe
	const agpt_sphere* spheres;
	const agpt_plane* planes;
	const DMesh* meshes;
	const agpt_instance* instances;  // extension: placed meshes (rows of AGPT_PRIM_INSTANCE)
	const agpt_material* mats;
	const agpt_light* lights;
	int n_prims, n_lights;
	int width, height;
	// InfiniteAreaLight tables (agpt_envmap); envW == 0: none
	const float* envRgb;
	const float* envFunc;
	const float* envCdf;
	float envFuncInt;
	int envW, envH;
	float cellLo[3], cellScale[3];   // ray-bucket grid over the bounded geometry: cell = (p - lo) * scale
	const float4* keyBoxes;          // ray-bucket key: root boxes of the meshes that do NOT cover the scene (2 x float4: min.xyz,max.x | max.yz,-,-)
	int n_keyBoxes;
	agpt_camera cam;
};

// ---------------------------------------------------------------------------------------
// float3 helpers in the reference's operation order (template/precomp.h:427-768)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 f3(float s) { return make_float3(s, s, s); }
__device__ __forceinline__ float3 f3(const float* p) { return make_float3(p[0], p[1], p[2]); }
__device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float3 operator*(float s, float3 a) { return f3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float3 operator/(float3 a, float s) { return f3(a.x / s, a.y / s, a.z / s); }
__device__ __forceinline__ void operator+=(float3& a, float3 b) { a.x += b.x; a.y += b.y; a.z += b.z; }
__device__ __forceinline__ void operator*=(float3& a, float3 b) { a.x *= b.x; a.y *= b.y; a.z *= b.z; }
__device__ __forceinline__ void operator*=(float3& a, float s) { a.x *= s; a.y *= s; a.z *= s; }
__device__ __forceinline__ void operator/=(float3& a, float s) { a.x /= s; a.y /= s; a.z /= s; }
__device__ __forceinline__ float dot(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ float sqrLength(float3 v) { return dot(v, v); }
__device__ __forceinline__ float length(float3 v) { return sqrtf(dot(v, v)); }
__device__ __forceinline__ float absdot(float3 a, float3 b) { return fabsf(dot(a, b)); }
// normalize = v * (1/sqrtf(dot)), precomp.h:366,735
__device__ __forceinline__ float3 normalize(float3 v) { float inv = 1.0f / sqrtf(dot(v, v)); return v * inv; }
__device__ __forceinline__ float3 cross(float3 a, float3 b) {
	return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ bool IsBlack(float3 v) { return v.x == 0 && v.y == 0 && v.z == 0; }
__device__ __forceinline__ float3 Faceforward(float3 v, float3 v2) { return (dot(v, v2) < 0.f) ? -v : v; }   // precomp.h:712
__device__ __forceinline__ float3 Lerp(float t, float3 a, float3 b) { return (1 - t) * a + t * b; }          // precomp.h:676
__device__ __forceinline__ float3 Reflect(float3 wo, float3 n) { return -wo + 2.0f * dot(wo, n) * n; }        // precomp.h:762

// EXTENSION: instances (agpt.h agpt_instance; CPU statement: oracle/agpt_oracle.cpp XformPoint / XformVector).
__device__ __forceinline__ float3 XformPoint(const float* m, float3 p) {
	return f3(m[0] * p.x + m[1] * p.y + m[2] * p.z + m[3], m[4] * p.x + m[5] * p.y + m[6] * p.z + m[7], m[8] * p.x + m[9] * p.y + m[10] * p.z + m[11]);
}
__device__ __forceinline__ float3 XformVector(const float* m, float3 v) {
	return f3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[4] * v.x + m[5] * v.y + m[6] * v.z, m[8] * v.x + m[9] * v.y + m[10] * v.z);
}
__device__ __forceinline__ float3 XformNormal(const float* w2o, float3 n) {        // transpose(W2O)
	return f3(w2o[0] * n.x + w2o[4] * n.y + w2o[8] * n.z, w2o[1] * n.x + w2o[5] * n.y + w2o[9] * n.z, w2o[2] * n.x + w2o[6] * n.y + w2o[10] * n.z);
}

// template fminf/fmaxf (precomp.h:364-365) and clamp (precomp.h:678)
__device__ __forceinline__ float rmin(float a, float b) { return a < b ? a : b; }
__device__ __forceinline__ float rmax(float a, float b) { return a > b ? a : b; }
__device__ __forceinline__ float rclamp(float f, float a, float b) { return rmax(a, rmin(f, b)); }
// std::max / std::min as libstdc++ defines them
__device__ __forceinline__ float smax(float a, float b) { return (a < b) ? b : a; }
__device__ __forceinline__ float smin(float a, float b) { return (b < a) ? b : a; }

// sinf / cosf / acosf with the oracle's bits.  The reference calls libm; CUDA's sinf/cosf/
// acosf are different 1-2 ulp routines, and even a correctly rounded result differs from
// glibc's in ~0.8 % (sin/cos) and ~7.7 % (acos) of calls -- each such ulp is then amplified by
// every later bounce off a curved surface.  So the device evaluates the SAME published
// algorithms glibc 2.39 uses (the oracle's libm), which makes secondary rays bit-identical too:
//   * sinf/cosf: ARM optimized-routines "sincosf" (glibc sysdeps/ieee754/flt-32/s_sinf.c,
//     s_cosf.c, sincosf.h): reduction by pi/2 and odd/even minimax polynomials, all in double;
//   * acosf: Sun fdlibm e_acosf.c rational approximation in float (glibc e_acosf.c).
// Checked on the host against libm: 0 mismatches in 4e7 (sin, cos) and 2e7 (acos) arguments.
// Arguments on this path lie in [-pi/4, 2 pi]; beyond |x| >= 120 (never reached) the slow
// reduction is replaced by the double routine.  Kept out of line (called from many sites).
__device__ __forceinline__ float SinCosPoly(double x, double x2, bool negate, int n) {
	const double sg = negate ? -1.0 : 1.0;     // glibc's __sincosf_table[1] is table[0] with the cosine coefficients negated
	if ((n & 1) == 0) {
		double x3 = x * x2;
		double s1 = 0x1.1107605230bc4p-7 + x2 * -0x1.994eb3774cf24p-13;
		double x7 = x3 * x2;
		double s = x + x3 * -0x1.555545995a603p-3;
		return (float)(s + x7 * s1);
	}
	double x4 = x2 * x2;
	double c2 = sg * -0x1.6c087e89a359dp-10 + x2 * (sg * 0x1.99343027bf8c3p-16);
	double c1 = sg * -0x1.ffffffd0c621cp-2 + x2 * (sg * 0x1.55553e1068f19p-5);
	double x6 = x4 * x2;
	double c = sg * 0x1p0 + x2 * c1;
	return (float)(c + x6 * c2);
}
__device__ __forceinline__ uint32_t AbsTop12(float x) { return (__float_as_uint(x) >> 20) & 0x7ffu; }
// returns sin (cosine == false) or cos (cosine == true) of y
__device__ __forceinline__ float GlibcSinCos(float y, bool cosine) {
	double x = (double)y;
	if (AbsTop12(y) < AbsTop12(0x1.921FB6p-1f)) {             // |y| < pi/4
		double x2 = x * x;
		if (AbsTop12(y) < AbsTop12(0x1p-12f)) return cosine ? 1.0f : y;
		return SinCosPoly(x, x2, false, cosine ? 1 : 0);
	}
	if (AbsTop12(y) < AbsTop12(120.0f)) {
		double r = x * 0x1.45F306DC9C883p+23;                 // 2/pi * 2^24
		int n = (__double2int_rz(r) + 0x800000) >> 24;
		x = x - n * 0x1.921FB54442D18p0;
		double sgn = ((n & 3) == 1 || (n & 3) == 2) ? -1.0 : 1.0;   // sign[4] = { 1, -1, -1, 1 }
		return SinCosPoly(x * sgn, x * x, (n & 2) != 0, cosine ? (n ^ 1) : n);
	}
	return cosine ? (float)cos(x) : (float)sin(x);
}
__device__ __noinline__ float rsin(float x) { return GlibcSinCos(x, false); }
__device__ __noinline__ float rcos(float x) { return GlibcSinCos(x, true); }
// (returned by value: out-pointers of an out-of-line function live in local memory)
__device__ __noinline__ float2 rsincos2(float x) { return make_float2(GlibcSinCos(x, false), GlibcSinCos(x, true)); }
__device__ __forceinline__ void rsincos(float x, float* s, float* c) { float2 sc = rsincos2(x); *s = sc.x; *c = sc.y; }
__device__ __noinline__ float racos(float x) {
	const float one = 1.0000000000e+00f, pi = 3.1415925026e+00f, pio2_hi = 1.5707962513e+00f, pio2_lo = 7.5497894159e-08f,
		pS0 = 1.6666667163e-01f, pS1 = -3.2556581497e-01f, pS2 = 2.0121252537e-01f, pS3 = -4.0055535734e-02f,
		pS4 = 7.9153501429e-04f, pS5 = 3.4793309169e-05f,
		qS1 = -2.4033949375e+00f, qS2 = 2.0209457874e+00f, qS3 = -6.8828397989e-01f, qS4 = 7.7038154006e-02f;
	float z, p, q, r, w, s, c, df;
	int hx = __float_as_int(x), ix = hx & 0x7fffffff;
	if (ix == 0x3f800000) return hx > 0 ? 0.0f : pi + 2.0f * pio2_lo;
	if (ix > 0x3f800000) return (x - x) / (x - x);
	if (ix < 0x3f000000) {                                    // |x| < 0.5
		if (ix <= 0x23000000) return pio2_hi + pio2_lo;
		z = x * x;
		p = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
		q = one + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
		r = p / q;
		return pio2_hi - (x - (pio2_lo - x * r));
	}
	if (hx < 0) {                                             // x < -0.5
		z = (one + x) * 0.5f;
		p = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
		q = one + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
		s = sqrtf(z);
		r = p / q;
		w = r * s - pio2_lo;
		return pi - 2.0f * (s + w);
	}
	z = (one - x) * 0.5f;                                     // x > 0.5
	s = sqrtf(z);
	df = __int_as_float(__float_as_int(s) & 0xfffff000);
	c = (z - df * df) / (s + df);
	p = z * (pS0 + z * (pS1 + z * (pS2 + z * (pS3 + z * (pS4 + z * pS5)))));
	q = one + z * (qS1 + z * (qS2 + z * (qS3 + z * qS4)));
	r = p / q;
	w = r * s + c;
	return 2.0f * (df + w);
}

// atan2f: Sun fdlibm e_atan2f.c / s_atanf.c in float (the lineage of glibc's).  On this path it
// only feeds SphericalPhi -> a texel column of the environment map (lights.cpp:84-90,100-111),
// a discrete index, so the last ulp is immaterial; measured against glibc 2.39 on the host it
// differs in 31 of 3e7 arguments, all with |y/x| > 2^24.  The sphere uv of textured materials (extension) states this
// algorithm, not glibc's (statements/agpt_texture_oracle.cpp ports it).  COPY: the textured kernels call copy 1, so the call
// graph of the kernels that ran before textures existed, and with it their code, stays as it was.
template <int COPY>
__device__ __noinline__ float ratanfT(float x) {
	const float atanhi[4] = { 4.6364760399e-01f, 7.8539812565e-01f, 9.8279368877e-01f, 1.5707962513e+00f };
	const float atanlo[4] = { 5.0121582440e-09f, 3.7748947079e-08f, 3.4473217170e-08f, 7.5497894159e-08f };
	const float aT[11] = { 3.3333334327e-01f, -2.0000000298e-01f, 1.4285714924e-01f, -1.1111110449e-01f, 9.0908870101e-02f,
		-7.6918758452e-02f, 6.6610731184e-02f, -5.8335702866e-02f, 4.9768779427e-02f, -3.6531571299e-02f, 1.6285819933e-02f };
	int hx = __float_as_int(x), ix = hx & 0x7fffffff, id;
	if (ix >= 0x4c800000) {
		if (ix > 0x7f800000) return x + x;
		return hx > 0 ? atanhi[3] + atanlo[3] : -atanhi[3] - atanlo[3];
	}
	if (ix < 0x3ee00000) {
		if (ix < 0x31000000) return x;
		id = -1;
	}
	else {
		x = fabsf(x);
		if (ix < 0x3f980000) {
			if (ix < 0x3f300000) { id = 0; x = (2.0f * x - 1.0f) / (2.0f + x); }
			else { id = 1; x = (x - 1.0f) / (x + 1.0f); }
		}
		else {
			if (ix < 0x401c0000) { id = 2; x = (x - 1.5f) / (1.0f + 1.5f * x); }
			else { id = 3; x = -1.0f / x; }
		}
	}
	float z = x * x, w = z * z;
	float s1 = z * (aT[0] + w * (aT[2] + w * (aT[4] + w * (aT[6] + w * (aT[8] + w * aT[10])))));
	float s2 = w * (aT[1] + w * (aT[3] + w * (aT[5] + w * (aT[7] + w * aT[9]))));
	if (id < 0) return x - x * (s1 + s2);
	z = atanhi[id] - ((x * (s1 + s2) - atanlo[id]) - x);
	return hx < 0 ? -z : z;
}
template <int COPY>
__device__ __noinline__ float ratan2T(float y, float x) {
	const float tiny = 1.0e-30f, pi_o_4 = 7.8539818525e-01f, pi_o_2 = 1.5707963705e+00f, pi = 3.1415927410e+00f, pi_lo = -8.7422776573e-08f;
	int hx = __float_as_int(x), ix = hx & 0x7fffffff, hy = __float_as_int(y), iy = hy & 0x7fffffff;
	if (ix > 0x7f800000 || iy > 0x7f800000) return x + y;
	if (hx == 0x3f800000) return ratanfT<COPY>(y);
	int m = ((hy >> 31) & 1) | ((hx >> 30) & 2);
	if (iy == 0) return m < 2 ? y : (m == 2 ? pi + tiny : -pi - tiny);
	if (ix == 0) return hy < 0 ? -pi_o_2 - tiny : pi_o_2 + tiny;
	if (ix == 0x7f800000) {
		if (iy == 0x7f800000) return m == 0 ? pi_o_4 + tiny : m == 1 ? -pi_o_4 - tiny : m == 2 ? 3.0f * pi_o_4 + tiny : -3.0f * pi_o_4 - tiny;
		return m == 0 ? 0.0f : m == 1 ? -0.0f : m == 2 ? pi + tiny : -pi - tiny;
	}
	if (iy == 0x7f800000) return hy < 0 ? -pi_o_2 - tiny : pi_o_2 + tiny;
	int k = (iy - ix) >> 23;
	float z;
	if (k > 24) z = pi_o_2 + 0.5f * pi_lo;
	else if (hx < 0 && k < -24) z = 0.0f;
	else z = ratanfT<COPY>(fabsf(y / x));
	switch (m) {
	case 0: return z;
	case 1: return -z;
	case 2: return pi - (z - pi_lo);
	default: return (z - pi_lo) - pi;
	}
}
__device__ __forceinline__ float ratan2(float y, float x) { return ratan2T<0>(y, x); }

// powf with the oracle's bits, for Accumulator::CopyToSurface's gamma (common.h:41-44: pow(c, 1/2.2f)
// on floats = powf).  glibc 2.39's powf is the ARM optimized-routines algorithm
// (sysdeps/ieee754/flt-32/e_powf.c, e_powf_log2_data.c, e_exp2f_data.c): log2(x) from a 16-entry
// table + degree-5 polynomial, exp2 from a 32-entry table + cubic, all in double.  On x86-64 hosts
// with FMA, glibc dispatches to the same source compiled with -mfma (__powf_fma), in which every
// a*b+c below is one fused operation; the explicit fma() calls restate that build (--fmad=false
// leaves explicit fma alone).  Checked on the host against libm for ALL 2,139,095,041 non-negative
// float bit patterns with y = 1/2.2f: 0 mismatches.  Only what this path needs: y finite, > 0 and
// not an integer (the special cases of e_powf.c:155-196 for such y).
// (tables in global memory, read through L1: per-thread local copies would be rebuilt on every call)
__device__ const double kPowfLog2[16][2] = {
	{ 0x1.661ec79f8f3bep+0, -0x1.efec65b963019p-2 }, { 0x1.571ed4aaf883dp+0, -0x1.b0b6832d4fca4p-2 },
	{ 0x1.49539f0f010b0p+0, -0x1.7418b0a1fb77bp-2 }, { 0x1.3c995b0b80385p+0, -0x1.39de91a6dcf7bp-2 },
	{ 0x1.30d190c8864a5p+0, -0x1.01d9bf3f2b631p-2 }, { 0x1.25e227b0b8ea0p+0, -0x1.97c1d1b3b7af0p-3 },
	{ 0x1.1bb4a4a1a343fp+0, -0x1.2f9e393af3c9fp-3 }, { 0x1.12358f08ae5bap+0, -0x1.960cbbf788d5cp-4 },
	{ 0x1.0953f419900a7p+0, -0x1.a6f9db6475fcep-5 }, { 0x1.0000000000000p+0, 0x0.0p+0 },
	{ 0x1.e608cfd9a47acp-1, 0x1.338ca9f24f53dp-4 }, { 0x1.ca4b31f026aa0p-1, 0x1.476a9543891bap-3 },
	{ 0x1.b2036576afce6p-1, 0x1.e840b4ac4e4d2p-3 }, { 0x1.9c2d163a1aa2dp-1, 0x1.40645f0c6651cp-2 },
	{ 0x1.886e6037841edp-1, 0x1.88e9c2c1b9ff8p-2 }, { 0x1.767dcf5534862p-1, 0x1.ce0a44eb17bccp-2 } };
__device__ const unsigned long long kExp2f[32] = {
	0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull, 0x3fef72b83c7d517bull, 0x3fef54873168b9aaull,
	0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull, 0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
	0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull, 0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull,
	0x3feea11473eb0187ull, 0x3feea589994cce13ull, 0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
	0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull, 0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full,
	0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull };
__device__ __noinline__ float rpowf(float x, float y) {
	const double A0 = 0x1.27616c9496e0bp-2, A1 = -0x1.71969a075c67ap-2, A2 = 0x1.ec70a6ca7baddp-2, A3 = -0x1.7154748bef6c8p-1, A4 = 0x1.71547652ab82bp+0;
	const double C0 = 0x1.c6af84b912394p-5, C1 = 0x1.ebfce50fac4f3p-3, C2 = 0x1.62e42ff0c52d6p-1, SHIFT = 0x1.8p+47;
	uint32_t ix = __float_as_uint(x);
	if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u) {
		// x is zero, subnormal, negative, inf or nan
		if (2u * ix == 0u) return 0.0f;                                   // (+-0)^y = +0 for y > 0 not an odd integer
		if ((ix & 0x7fffffffu) > 0x7f800000u) return x + y;               // nan
		if (ix == 0x7f800000u || ix == 0xff800000u) return __uint_as_float(0x7f800000u);   // (+-inf)^y = +inf
		if (ix & 0x80000000u) return __uint_as_float(0xffc00000u);       // negative finite base, non-integer y: invalid -> the x86 default nan of (x-x)/(x-x)
		ix = __float_as_uint(x * 0x1p23f);                                // subnormal: normalise
		ix &= 0x7fffffffu;
		ix -= 23u << 23;
	}
	// log2_inline (e_powf.c:44-77)
	uint32_t tmp = ix - 0x3f330000u;
	int i = (int)((tmp >> (23 - 4)) % 16u);
	uint32_t top = tmp & 0xff800000u;
	uint32_t iz = ix - top;
	int k = (int)top >> 23;
	double invc = kPowfLog2[i][0], logc = kPowfLog2[i][1];
	double z = (double)__uint_as_float(iz);
	double r = fma(z, invc, -1.0);
	double y0 = logc + (double)k;
	double r2 = r * r;
	double yy = fma(A0, r, A1);
	double p = fma(A2, r, A3);
	double r4 = r2 * r2;
	double q = fma(A4, r, y0);
	q = fma(p, r2, q);
	yy = fma(yy, r4, q);
	double ylogx = (double)y * yy;
	if (((unsigned long long)__double_as_longlong(ylogx) >> 47 & 0xffffull) >= ((unsigned long long)__double_as_longlong(126.0) >> 47)) {
		if (ylogx > 0x1.fffffffd1d571p+6) return __uint_as_float(0x7f800000u);      // overflow
		if (ylogx <= -150.0) return 0.0f;                                            // underflow
	}
	// exp2_inline (e_powf.c:96-127)
	double kd = ylogx + SHIFT;
	unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
	kd -= SHIFT;
	double rr = ylogx - kd;
	unsigned long long t = kExp2f[ki % 32ull];
	t += ki << (52 - 5);
	double s = __longlong_as_double((long long)t);
	double zz = fma(C0, rr, C1);
	double rr2 = rr * rr;
	double y2 = fma(C2, rr, 1.0);
	y2 = fma(zz, rr2, y2);
	y2 = y2 * s;
	return (float)y2;
}

// common.h:145-151
__device__ __forceinline__ void CoordinateSystem(float3 v1, float3* v2, float3* v3) {
	if (fabsf(v1.x) > fabsf(v1.y)) *v2 = f3(-v1.z, 0, v1.x) / sqrtf(v1.x * v1.x + v1.z * v1.z);
	else *v2 = f3(0, v1.z, -v1.y) / sqrtf(v1.y * v1.y + v1.z * v1.z);
	*v3 = cross(v1, *v2);
}

// ---------------------------------------------------------------------------------------
// RNG: Marsaglia xorshift32 of the template (template/template.cpp:666-685) on a per-path
// state; stream start = WangHash(WangHash((pixel+1)*17) + sample), 0 -> 1 (cl/tools.cl:1-2,
// SURVEY 8a row 3).
// ---------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t WangHash(uint32_t s) {
	s = (s ^ 61u) ^ (s >> 16);
	s *= 9u;
	s = s ^ (s >> 4);
	s *= 0x27d4eb2du;
	s = s ^ (s >> 15);
	return s;
}
__host__ __device__ __forceinline__ uint32_t StreamSeed(uint32_t pixel, uint32_t sample) {
	uint32_t s = WangHash(WangHash((pixel + 1u) * 17u) + sample);
	return s ? s : 1u;
}
__device__ __forceinline__ float RandomFloat(uint32_t& s) {
	s ^= s << 13;
	s ^= s >> 17;
	s ^= s << 5;
	return __uint2float_rn(s) * 2.3283064365387e-10f;
}

// ---------------------------------------------------------------------------------------
// Ray: O, D = normalize(d), t (camera.h:3-15)
// ---------------------------------------------------------------------------------------
struct DRay {
	float3 O, D;
	float t;
};
__device__ __forceinline__ DRay MakeRay(float3 o, float3 d, float t = FLT_MAX) {
	DRay r;
	r.O = o; r.D = normalize(d); r.t = t;
	return r;
}

// Bounds::Intersect (bvhtrimesh.h:18-36).  The per-axis early-outs of the reference are
// folded into one test after the third axis: tmin never decreases, tmax never increases and
// rounding of tmax*1.00000024f is monotonic, so "some axis failed" == "the last axis fails".
// NaNs from 0/0 are dropped by the select order exactly as upstream drops them.
__device__ __forceinline__ bool BoundsIntersect(float3 bmin, float3 bmax, float3 O, float3 D, float rayT, float& tEntry) {
	float tmin = 0.0f, tmax = rayT;
	{
		float a = (bmin.x - O.x) / D.x, b = (bmax.x - O.x) / D.x;
		float t0 = rmin(a, b), t1 = rmax(a, b);
		tmin = rmax(t0, tmin); tmax = rmin(t1, tmax);
	}
	{
		float a = (bmin.y - O.y) / D.y, b = (bmax.y - O.y) / D.y;
		float t0 = rmin(a, b), t1 = rmax(a, b);
		tmin = rmax(t0, tmin); tmax = rmin(t1, tmax);
	}
	{
		float a = (bmin.z - O.z) / D.z, b = (bmax.z - O.z) / D.z;
		float t0 = rmin(a, b), t1 = rmax(a, b);
		tmin = rmax(t0, tmin); tmax = rmin(t1, tmax);
	}
	tEntry = tmin;
	return !((tmax * 1.00000024f) < tmin);
}

// ---------------------------------------------------------------------------------------
// Exact-filtered slab test.  Bounds::Intersect costs six IEEE divisions per box.  What the
// walk needs from it are DECISIONS -- box hit or not, and which child is nearer -- not the
// distances themselves.  q~ = (b - O) * fl(1/D) differs from the reference's fl((b - O)/D) by
// at most 3 * 2^-24 relative (same numerator, two roundings against one), signs and exact
// zeros are preserved, and min/max keep that bound.  So each decision is first taken on the
// cheap values with a guard band of 2^-19 relative -- 8x the worst case incl. the rounding of
// tmax*1.00000024f -- and only when a comparison falls inside the band is the pair re-done
// with the reference arithmetic (BoundsIntersect above).  Decisions, hence traversal order,
// visit counts and hits, are identical to the strict walk; tests assert exactly that.
// Rays with a direction component below 1e-18 in magnitude (or zero) always take the
// reference arithmetic, as do non-finite inputs.
// ---------------------------------------------------------------------------------------
#define AGPT_GUARD 1.9073486328125e-06f      // 2^-19

__device__ __forceinline__ void SlabApprox(float3 bmin, float3 bmax, float3 O, float3 rD, float rayT, float& tmin, float& tmax) {
	float ax = (bmin.x - O.x) * rD.x, bx = (bmax.x - O.x) * rD.x;
	float ay = (bmin.y - O.y) * rD.y, by = (bmax.y - O.y) * rD.y;
	float az = (bmin.z - O.z) * rD.z, bz = (bmax.z - O.z) * rD.z;
	tmin = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), 0.0f));
	tmax = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), rayT));
}
// 1 = certainly hit, 0 = certainly missed, -1 = inside the guard band (ask the reference arithmetic)
__device__ __forceinline__ int SlabDecision(float tmin, float tmax) {
	float T = tmax * 1.00000024f;
	if (T < tmin * (1.0f - AGPT_GUARD)) return 0;
	if (T > tmin * (1.0f + AGPT_GUARD)) return 1;
	return -1;
}
// 1 = right child certainly nearer (swap), 0 = certainly not, -1 = inside the guard band
__device__ __forceinline__ int NearerDecision(float dl, float dr) {
	if (dl == 0.0f && dr == 0.0f) return 0;          // origin inside both boxes: exact zeros on both sides
	if (dr < dl * (1.0f - AGPT_GUARD)) return 1;
	if (dr > dl * (1.0f + AGPT_GUARD)) return 0;
	return -1;
}

// Moller-Trumbore of TriangleMesh::TriangleIntersect(P) (trianglemesh.cpp:7-43,117-155):
// no culling, no epsilon; reject det==0, b1<0||b1>1, b2<0||b1+b2>1, t<=0||t>=ray.t.
__device__ __forceinline__ bool TriangleTest(float3 v0, float3 v1, float3 v2, float3 O, float3 D, float rayT,
		float& tOut, float& b1Out, float& b2Out) {
	float3 e1 = v1 - v0;
	float3 e2 = v2 - v0;
	float3 pvec = cross(D, e2);
	float det = dot(e1, pvec);
	if (det == 0.0f) return false;
	float inv_det = 1.0f / det;
	float3 tvec = O - v0;
	float b1 = dot(tvec, pvec) * inv_det;
	if (b1 < 0.0f || b1 > 1.0f) return false;
	float3 qvec = cross(tvec, e1);
	float b2 = dot(D, qvec) * inv_det;
	if (b2 < 0.0f || b1 + b2 > 1.0f) return false;
	float t = dot(e2, qvec) * inv_det;
	if (t <= 0.0f || t >= rayT) return false;
	tOut = t; b1Out = b1; b2Out = b2;
	return true;
}

// Triangle partial derivatives (trianglemesh.cpp:59-80).  Returns false when upstream
// declares the triangle degenerate and drops the hit (:74-77).
__device__ __forceinline__ bool TriangleDerivatives(float3 v0, float3 v1, float3 v2, float2 uv0, float2 uv1, float2 uv2,
		float3& dpdu, float3& dpdv) {
	float2 duv02 = make_float2(uv0.x - uv2.x, uv0.y - uv2.y), duv12 = make_float2(uv1.x - uv2.x, uv1.y - uv2.y);
	float3 dp02 = v0 - v2, dp12 = v1 - v2;
	float determinant = duv02.x * duv12.y - duv02.y * duv12.x;
	bool degenerateUV = (double)fabsf(determinant) < 1e-8;
	dpdu = f3(0.f); dpdv = f3(0.f);   // upstream leaves them uninitialised here; only read when !degenerateUV
	if (!degenerateUV) {
		float invdet = 1 / determinant;
		dpdu = (duv12.y * dp02 - duv02.y * dp12) * invdet;
		dpdv = (-duv12.x * dp02 + duv02.x * dp12) * invdet;
	}
	if (degenerateUV || sqrLength(cross(dpdu, dpdv)) == 0) {
		float3 ng = cross(v2 - v0, v1 - v0);
		if (sqrLength(ng) == 0) return false;
		CoordinateSystem(normalize(ng), &dpdu, &dpdv);
	}
	return true;
}

// Sphere::Intersect / IntersectP root selection (intersectable.h:164-181,207-226); assumes |D|=1.
__device__ __forceinline__ bool SphereTest(const agpt_sphere& s, float3 O, float3 D, float rayT, float& tOut) {
	float3 oc = O - f3(s.center);
	float half_b = dot(oc, D);
	float c = sqrLength(oc) - s.r2;
	float discriminant = half_b * half_b - c;
	if (discriminant < 0) return false;
	float sqrtd = sqrtf(discriminant);
	float root = -half_b - sqrtd;
	if (root < 0 || rayT < root) {
		root = -half_b + sqrtd;
		if (root < 0 || rayT < root) return false;
	}
	tOut = root;
	return true;
}

// Plane::Intersect / IntersectP (intersectable.h:123-150).
__device__ __forceinline__ bool PlaneTest(const agpt_plane& p, float3 O, float3 D, float rayT, float& tOut) {
	if (D.y == 0) return false;
	float t = (p.o[1] - O.y) / D.y;
	if (t <= 0 || t >= rayT) return false;
	float3 P = O + t * D;
	float u = (P.x - p.o[0]) / p.half_x;
	float v = (P.z - p.o[2]) / p.half_z;
	if (fabsf(u) <= 1 && fabsf(v) <= 1) { tOut = t; return true; }
	return false;
}

// ---------------------------------------------------------------------------------------
// EXTENSION: Sample_Li of a plane or mesh area light with AGPT_LIGHT_SAMPLE_SHAPE (agpt.h; CPU statement:
// oracle/agpt_shape_oracle.cpp ShapeSample).  PBRT-v3's Shape::Sample(ref, u) in solid angle: SampleDiscrete over the area cdf
// (FindInterval as sampling.h:4-18), UniformSampleTriangle on the remapped u.x and u.y; a plane samples its rectangle.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float ShapeSolidAnglePdf(float d2, float3 n, float3 wi, float area) {
	float c = absdot(n, wi);
	if (c == 0) return 0.f;
	float pdf = d2 / (c * area);
	return isinf(pdf) ? 0.f : pdf;
}
__device__ __forceinline__ float3 TriangleGeomNormal(const float4* tri) {
	float4 a = tri[0], b = tri[1], c = tri[2];
	float3 v0 = f3(a.x, a.y, a.z);
	return normalize(cross(f3(b.x, b.y, b.z) - v0, f3(c.x, c.y, c.z) - v0));
}
__device__ __forceinline__ void ShapeSampleFrom(const DScene& sc, const DShapeTables& st, int light, const agpt_prim& pr, float3 refP, float2 u, float3* pOut, float3* nOut, float* pdf) {
	const DShapeLight sl = st.lights[light];
	*pdf = 0.f; *pOut = f3(0.f); *nOut = f3(0.f);
	if (!(sl.area > 0)) return;
	float3 p, n;
	if (pr.type == AGPT_PRIM_PLANE) {
		const agpt_plane& pl = sc.planes[pr.payload];
		p = f3(pl.o[0] + (2 * u.x - 1) * pl.half_x, pl.o[1], pl.o[2] + (2 * u.y - 1) * pl.half_z);
		n = f3(0.f, 1.f, 0.f);
	}
	else {
		const float* cdf = st.cdf + sl.cdfOff;
		const int size = sl.n + 1;
		int first = 0, len = size;
		while (len > 0) {
			int half = len >> 1, middle = first + half;
			if (cdf[middle] <= u.x) { first = middle + 1; len -= half + 1; }
			else len = half;
		}
		const int offset = min(max(first - 1, 0), size - 2);
		const float width = cdf[offset + 1] - cdf[offset];
		if (!(width > 0)) return;                          // a zero-area triangle (u.x == 1 can land on one at the end)
		const float ur = (u.x - cdf[offset]) / width;
		const float4* tri = sc.meshes[pr.payload].tris + 3 * offset;
		float4 a = tri[0], b = tri[1], c = tri[2];
		float3 v0 = f3(a.x, a.y, a.z), v1 = f3(b.x, b.y, b.z), v2 = f3(c.x, c.y, c.z);
		float su0 = sqrtf(ur);
		float b0 = 1 - su0, b1 = u.y * su0;
		p = b0 * v0 + b1 * v1 + (1 - b0 - b1) * v2;
		n = normalize(cross(v1 - v0, v2 - v0));
	}
	*pOut = p; *nOut = n;
	float3 wi = p - refP;
	float d2 = sqrLength(wi);
	if (d2 == 0) return;
	wi /= sqrtf(d2);
	*pdf = ShapeSolidAnglePdf(d2, n, wi, sl.area);
}
