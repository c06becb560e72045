// agpt_bsdf.cuh -- surface interaction, BSDF (Disney diffuse/retro + Trowbridge-Reitz
// microfacet, mirror) and light sampling on the device, restated from the reference in its
// operation order.  No virtual dispatch: a material is a 64-byte record whose lobe set is a
// bit mask in BSDF::bxdfs[] order (diffuse, retro, microfacet | specular), material.h:51-58.
#pragma once

#include "agpt_device.cuh"

// ---------------------------------------------------------------------------------------
// shading-space helpers (microfacet.h:3-32)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float CosTheta(float3 w) { return w.z; }
__device__ __forceinline__ float Cos2Theta(float3 w) { return w.z * w.z; }
__device__ __forceinline__ float AbsCosTheta(float3 w) { return fabsf(w.z); }
__device__ __forceinline__ float Sin2Theta(float3 w) { return smax(0.f, 1.f - Cos2Theta(w)); }
__device__ __forceinline__ float SinTheta(float3 w) { return sqrtf(Sin2Theta(w)); }
__device__ __forceinline__ float TanTheta(float3 w) { return SinTheta(w) / CosTheta(w); }
__device__ __forceinline__ float Tan2Theta(float3 w) { return Sin2Theta(w) / Cos2Theta(w); }
__device__ __forceinline__ float CosPhi(float3 w) { float s = SinTheta(w); return (s == 0) ? 1 : rclamp(w.x / s, -1.f, 1.f); }
__device__ __forceinline__ float SinPhi(float3 w) { float s = SinTheta(w); return (s == 0) ? 0 : rclamp(w.y / s, -1.f, 1.f); }
__device__ __forceinline__ float Cos2Phi(float3 w) { return CosPhi(w) * CosPhi(w); }
__device__ __forceinline__ float Sin2Phi(float3 w) { return SinPhi(w) * SinPhi(w); }
__device__ __forceinline__ bool SameHemisphere(float3 w, float3 wp) { return w.z * wp.z > 0; }   // precomp.h:713

// ---------------------------------------------------------------------------------------
// sampling helpers (common.h:84-89,118-143,153-169)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float2 ConcentricSampleDisk(float2 u) {
	float2 o = make_float2(2.f * u.x - 1, 2.f * u.y - 1);
	if (o.x == 0 && o.y == 0) return make_float2(0, 0);
	float theta, r;
	if (fabsf(o.x) > fabsf(o.y)) { r = o.x; theta = (AGPT_PI / 4) * (o.y / o.x); }
	else { r = o.y; theta = (AGPT_PI / 2) - (AGPT_PI / 4) * (o.x / o.y); }
	float st, ct;
	rsincos(theta, &st, &ct);
	return make_float2(r * ct, r * st);
}
__device__ __forceinline__ float3 CosineSampleHemisphere(float2 u) {
	float2 d = ConcentricSampleDisk(u);
	float z = sqrtf(smax(0.f, 1 - d.x * d.x - d.y * d.y));
	return f3(d.x, d.y, z);
}
__device__ __forceinline__ float3 SphericalDirection(float sinTheta, float cosTheta, float phi, float3 x, float3 y, float3 z) {
	float sp, cp;
	rsincos(phi, &sp, &cp);
	return sinTheta * cp * x + sinTheta * sp * y + cosTheta * z;
}
__device__ __forceinline__ float3 RandomInSphereU(float2 u) {   // common.h:84-89
	float a = 1 - 2 * u.x;
	float b = sqrtf(1 - a * a);
	float phi = 2 * AGPT_PI * u.y;
	float sp, cp;
	rsincos(phi, &sp, &cp);
	return f3(b * cp, b * sp, a);
}
__device__ __forceinline__ float UniformConePdf(float cosThetaMax) { return 1 / (2 * AGPT_PI * (1 - cosThetaMax)); }

// ---------------------------------------------------------------------------------------
// Fresnel / Disney terms (microfacet.h:180-201, disney.h:12-22,62-71)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float FrDielectric(float cosThetaI, float etaI, float etaT) {
	cosThetaI = rclamp(cosThetaI, -1.f, 1.f);
	bool entering = cosThetaI > 0.f;
	if (!entering) { float t = etaI; etaI = etaT; etaT = t; cosThetaI = fabsf(cosThetaI); }
	float sinThetaI = sqrtf(smax(0.f, 1.f - cosThetaI * cosThetaI));
	float sinThetaT = etaI / etaT * sinThetaI;
	if (sinThetaT >= 1) return 1;
	float cosThetaT = sqrtf(smax(0.f, 1.f - sinThetaT * sinThetaT));
	float Rparl = ((etaT * cosThetaI) - (etaI * cosThetaT)) / ((etaT * cosThetaI) + (etaI * cosThetaT));
	float Rperp = ((etaI * cosThetaI) - (etaT * cosThetaT)) / ((etaI * cosThetaI) + (etaT * cosThetaT));
	return (Rparl * Rparl + Rperp * Rperp) / 2;
}
__device__ __forceinline__ float SchlickWeight(float cosTheta) {
	float m = rclamp(1 - cosTheta, 0.f, 1.f);
	return (m * m) * (m * m) * m;
}
__device__ __forceinline__ float3 FrSchlick(float3 R0, float cosTheta) { return Lerp(SchlickWeight(cosTheta), R0, f3(1.f)); }
__device__ __forceinline__ float3 DisneyFresnel(const agpt_material& m, float cosI) {
	return Lerp(m.metallic, f3(FrDielectric(cosI, 1, m.eta)), FrSchlick(f3(m.spec_r0), cosI));
}
// the same with a per-hit R0 (extension: textured base colour)
__device__ __forceinline__ float3 DisneyFresnel(const agpt_material& m, float3 R0, float cosI) {
	return Lerp(m.metallic, f3(FrDielectric(cosI, 1, m.eta)), FrSchlick(R0, cosI));
}

// ---------------------------------------------------------------------------------------
// Trowbridge-Reitz distribution (microfacet.h:34-153) with Disney's separable G (disney.h:73-82)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float TR_D(float ax, float ay, float3 wh) {
	float tan2Theta = Tan2Theta(wh);
	if (isinf(tan2Theta)) return 0.;
	const float cos4Theta = Cos2Theta(wh) * Cos2Theta(wh);
	float e = (Cos2Phi(wh) / (ax * ax) + Sin2Phi(wh) / (ay * ay)) * tan2Theta;
	return 1 / (AGPT_PI * ax * ay * cos4Theta * (1 + e) * (1 + e));
}
__device__ __forceinline__ float TR_Lambda(float ax, float ay, float3 w) {
	float absTanTheta = fabsf(TanTheta(w));
	if (isinf(absTanTheta)) return 0.f;
	float alpha = sqrtf(Cos2Phi(w) * ax * ax + Sin2Phi(w) * ay * ay);
	float alpha2Tan2Theta = (alpha * absTanTheta) * (alpha * absTanTheta);
	return (-1 + sqrtf(1.f + alpha2Tan2Theta)) / 2;
}
__device__ __forceinline__ float TR_G1(float ax, float ay, float3 w) { return 1 / (1 + TR_Lambda(ax, ay, w)); }
__device__ __forceinline__ void TrowbridgeReitzSample11(float cosTheta, float U1, float U2, float* slope_x, float* slope_y) {
	if (cosTheta > .9999f) {
		float r = sqrtf(U1 / (1 - U1));
		float phi = 6.28318530718f * U2;
		float sp, cp;
		rsincos(phi, &sp, &cp);
		*slope_x = r * cp;
		*slope_y = r * sp;
		return;
	}
	float sinTheta = sqrtf(smax(0.f, 1.f - cosTheta * cosTheta));
	float tanTheta = sinTheta / cosTheta;
	float a = 1 / tanTheta;
	float G1 = 2 / (1 + sqrtf(1.f + 1.f / (a * a)));
	float A = 2 * U1 / G1 - 1;
	float tmp = 1.f / (A * A - 1.f);
	if ((double)tmp > 1e10) tmp = 1e10f;
	float B = tanTheta;
	float D = sqrtf(smax(B * B * tmp * tmp - (A * A - B * B) * tmp, 0.f));
	float slope_x_1 = B * tmp - D;
	float slope_x_2 = B * tmp + D;
	*slope_x = (A < 0 || slope_x_2 > 1.f / tanTheta) ? slope_x_1 : slope_x_2;
	float S;
	if (U2 > 0.5f) { S = 1.f; U2 = 2.f * (U2 - .5f); }
	else { S = -1.f; U2 = 2.f * (.5f - U2); }
	float z = (U2 * (U2 * (U2 * 0.27385f - 0.73369f) + 0.46341f)) /
		(U2 * (U2 * (U2 * 0.093073f + 0.309420f) - 1.000000f) + 0.597999f);
	*slope_y = S * z * sqrtf(1.f + *slope_x * *slope_x);
}
__device__ __forceinline__ float3 TrowbridgeReitzSample(float3 wi, float ax, float ay, float U1, float U2) {
	float3 wiS = normalize(f3(ax * wi.x, ay * wi.y, wi.z));
	float sx, sy;
	TrowbridgeReitzSample11(CosTheta(wiS), U1, U2, &sx, &sy);
	float tmp = CosPhi(wiS) * sx - SinPhi(wiS) * sy;
	sy = SinPhi(wiS) * sx + CosPhi(wiS) * sy;
	sx = tmp;
	sx = ax * sx;
	sy = ay * sy;
	return normalize(f3(-sx, -sy, 1.f));
}
__device__ __forceinline__ float3 TR_Sample_wh(float ax, float ay, float3 wo, float2 u) {
	bool flip = wo.z < 0;
	float3 wh = TrowbridgeReitzSample(flip ? -wo : wo, ax, ay, u.x, u.y);
	if (flip) wh = -wh;
	return wh;
}

// BxDF::Pdf of a cosine-sampled lobe (reflection.h:16-18); the lobes' f / Pdf live in EvalLobes below
__device__ __forceinline__ float Cosine_Pdf(float3 wo, float3 wi) { return SameHemisphere(wo, wi) ? AbsCosTheta(wi) * AGPT_INVPI : 0; }

// lobe order of BSDF::bxdfs[] for a material (material.h:51-58,79-81)
__device__ __forceinline__ int LobeList(const agpt_material& m, bool skipSpecular, int* lobes) {
	int n = 0;
	if (m.lobes & AGPT_LOBE_DIFFUSE) lobes[n++] = AGPT_LOBE_DIFFUSE;
	if (m.lobes & AGPT_LOBE_RETRO) lobes[n++] = AGPT_LOBE_RETRO;
	if (m.lobes & AGPT_LOBE_MICROFACET) lobes[n++] = AGPT_LOBE_MICROFACET;
	if ((m.lobes & AGPT_LOBE_SPECULAR) && !skipSpecular) lobes[n++] = AGPT_LOBE_SPECULAR;
	if (m.lobes & AGPT_LOBE_GLASS_REFLECT) lobes[n++] = AGPT_LOBE_GLASS_REFLECT;       // extension (agpt.h)
	if (m.lobes & AGPT_LOBE_GLASS_TRANSMIT) lobes[n++] = AGPT_LOBE_GLASS_TRANSMIT;
	return n;
}

// ---------------------------------------------------------------------------------------
// EXTENSION: rough dielectric (agpt.h AGPT_LOBE_GLASS_*; CPU statement: oracle/agpt_oracle.cpp GlassT_f / GlassT_Pdf / Refract).
// The reflection half is the reference's MicrofacetReflection over its plain TrowbridgeReitzDistribution and
// FresnelDielectric; the transmission half follows PBRT-v3's MicrofacetTransmission (radiance transport).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ bool Refract(float3 wi, float3 n, float eta, float3* wt) {
	float cosThetaI = dot(n, wi);
	float sin2ThetaI = smax(0.f, 1.f - cosThetaI * cosThetaI);
	float sin2ThetaT = eta * eta * sin2ThetaI;
	if (sin2ThetaT >= 1) return false;
	float cosThetaT = sqrtf(1 - sin2ThetaT);
	*wt = eta * -wi + (eta * cosThetaI - cosThetaT) * n;
	return true;
}
// lambdaO = Lambda(wo), G1o = G1(wo): hoisted per vertex
__device__ __forceinline__ float GlassT_Pdf(const agpt_material& m, float3 wo, float3 wi, float G1o, float absCosO) {
	if (SameHemisphere(wo, wi)) return 0;
	float eta = CosTheta(wo) > 0 ? (m.eta / 1.f) : (1.f / m.eta);
	float3 wh = normalize(wo + wi * eta);
	if (dot(wo, wh) * dot(wi, wh) > 0) return 0;
	float sqrtDenom = dot(wo, wh) + eta * dot(wi, wh);
	float dwh_dwi = fabsf((eta * eta * dot(wi, wh)) / (sqrtDenom * sqrtDenom));
	return TR_D(m.alpha_x, m.alpha_y, wh) * G1o * absdot(wo, wh) / absCosO * dwh_dwi;
}
__device__ __forceinline__ float3 GlassT_f(const agpt_material& m, float3 wo, float3 wi, float lambdaO, float lambdaI) {
	if (SameHemisphere(wo, wi)) return f3(0.f);
	float cosThetaO = CosTheta(wo), cosThetaI = CosTheta(wi);
	if (cosThetaI == 0 || cosThetaO == 0) return f3(0.f);
	float eta = CosTheta(wo) > 0 ? (m.eta / 1.f) : (1.f / m.eta);
	float3 wh = normalize(wo + wi * eta);
	if (wh.z < 0) wh = -wh;
	if (dot(wo, wh) * dot(wi, wh) > 0) return f3(0.f);
	float F = FrDielectric(dot(wo, wh), 1.f, m.eta);
	float sqrtDenom = dot(wo, wh) + eta * dot(wi, wh);
	float factor = 1 / eta;
	float G = 1 / (1 + lambdaO + lambdaI);
	return (f3(1.f) - f3(F)) * f3(m.diffuse_r) *
		fabsf(TR_D(m.alpha_x, m.alpha_y, wh) * G * eta * eta * absdot(wi, wh) * absdot(wo, wh) * factor * factor / (cosThetaI * cosThetaO * sqrtDenom * sqrtDenom));
}

// ---------------------------------------------------------------------------------------
// BSDF (reflection.h:83-201, reflection.cpp:6-11): frame and transforms.  BSDF::f / Pdf /
// Sample_f themselves are realised by the fused per-vertex evaluator further down.
// ---------------------------------------------------------------------------------------
struct DBSDF {
	float3 ng, ns, ss, ts;
	const agpt_material* mat;
};
__device__ __forceinline__ float3 WorldToLocal(const DBSDF& b, float3 v) { return f3(dot(v, b.ss), dot(v, b.ts), dot(v, b.ns)); }
__device__ __forceinline__ float3 LocalToWorld(const DBSDF& b, float3 v) {
	return f3(b.ss.x * v.x + b.ts.x * v.y + b.ns.x * v.z,
		b.ss.y * v.x + b.ts.y * v.y + b.ns.y * v.z,
		b.ss.z * v.x + b.ts.z * v.y + b.ns.z * v.z);
}
__device__ __forceinline__ bool BSDF_IsPerfectlySpecular(const DBSDF& b) { return (b.mat->lobes & ~AGPT_LOBE_SPECULAR) == 0; }

// ---------------------------------------------------------------------------------------
// SurfaceInteraction (intersectable.h:63-115) rebuilt once for the closest hit
// ---------------------------------------------------------------------------------------
struct DSurface {
	float3 p, n;          // point, geometric normal (after Faceforward by SetShadingGeometry)
	float3 sn;            // shading.n
	float3 sdpdu;         // shading.dpdu (== the geometric dpdu the interaction was built with, :76,:87)
};
__device__ __forceinline__ void SurfaceInit(DSurface& s, float3 p, float3 dpdu, float3 dpdv) {
	s.p = p;
	s.n = normalize(cross(dpdu, dpdv));
	s.sn = s.n;
	s.sdpdu = dpdu;
}
__device__ __forceinline__ DBSDF MakeBSDF(const DSurface& s, const agpt_material* m) {   // reflection.cpp:6-11
	DBSDF b;
	b.ng = s.n; b.ns = s.sn;
	b.ss = normalize(s.sdpdu);
	b.ts = cross(b.ns, b.ss);
	b.mat = m;
	return b;
}

// Sphere hit -> interaction (intersectable.h:183-204); dpdu/dpdv are passed swapped upstream.
// uv (extension, textured instantiations only; agpt.h agpt_upload_textures): the sphere's surface uv, or nullptr.  dpduOut,
// dpdvOut (extension, normal maps; agpt.h agpt_upload_material_textures): dp/du and dp/dv of that uv (before the swap), or nullptr.
__device__ __forceinline__ void SphereSurface(const agpt_sphere& sp, float3 O, float3 D, float root, DSurface& s, float2* uv = nullptr,
		float3* dpduOut = nullptr, float3* dpdvOut = nullptr) {
	float3 p = O + root * D;
	float3 pHit = p - f3(sp.center);
	if (pHit.x == 0 && pHit.y == 0) pHit.x = AGPT_EPSILON * sp.r;
	float theta = racos(rclamp(pHit.z / sp.r, -1.f, 1.f));
	float zRadius = sqrtf(pHit.x * pHit.x + pHit.y * pHit.y);
	float invZRadius = 1 / zRadius;
	float cosPhi = pHit.x * invZRadius;
	float sinPhi = pHit.y * invZRadius;
	float3 dpdu = f3(-AGPT_TWOPI * pHit.y, AGPT_TWOPI * pHit.x, 0);
	float3 dpdv = AGPT_PI * f3(pHit.z * cosPhi, pHit.z * sinPhi, -sp.r * rsin(theta));
	SurfaceInit(s, p, dpdv, dpdu);
	if (dpduOut) { *dpduOut = dpdu; *dpdvOut = dpdv; }
	if (uv) {
		float phi = ratan2T<1>(pHit.y, pHit.x);
		if (phi < 0) phi = phi + AGPT_TWOPI;
		*uv = make_float2(phi / AGPT_TWOPI, theta / AGPT_PI);
	}
}
__device__ __forceinline__ void PlaneSurface(float3 O, float3 D, float t, DSurface& s) {   // intersectable.h:128-133
	SurfaceInit(s, O + t * D, f3(0, 0, 1), f3(1, 0, 0));
}
// a triangle's uvs (the mesh's, or the default (0,0), (1,0), (1,1), trianglemesh.cpp:52-56) and the uv of barycentrics b1, b2, for
// shared by TriangleSurface and the alpha-mask test of the trace walk (agpt_upload_textures step 1).
__device__ __forceinline__ void TriangleUVs(const DMesh& mesh, int slot, float2& uv0, float2& uv1, float2& uv2) {
	uv0 = make_float2(0, 0); uv1 = make_float2(1, 0); uv2 = make_float2(1, 1);
	if (mesh.uvs) { uv0 = __ldg(mesh.uvs + 3 * slot); uv1 = __ldg(mesh.uvs + 3 * slot + 1); uv2 = __ldg(mesh.uvs + 3 * slot + 2); }
}
__device__ __forceinline__ float2 BaryUV(float b1, float b2, float2 uv0, float2 uv1, float2 uv2) {
	const float b0 = 1.f - b1 - b2;
	return make_float2((b0 * uv0.x + b1 * uv1.x) + b2 * uv2.x, (b0 * uv0.y + b1 * uv1.y) + b2 * uv2.y);
}
// Triangle hit -> interaction + shading frame (trianglemesh.cpp:45-113, intersectable.h:80-89)
// `in` (extension, agpt.h agpt_instance): the mesh is a placed one -- vertices go to world space first, the shading
// normal through transpose(W2O); nullptr for the reference's own meshes.  uvOut (extension, textured instantiations only): the
// interpolated uv, or nullptr.  dpduOut, dpdvOut (extension, normal maps): TriangleDerivatives' dpdu, dpdv, or nullptr.
__device__ __forceinline__ void TriangleSurface(const DMesh& mesh, int slot, float3 O, float3 D, float t, float b1, float b2, DSurface& s, const agpt_instance* in,
		float2* uvOut = nullptr, float3* dpduOut = nullptr, float3* dpdvOut = nullptr) {
	float4 a = __ldg(mesh.tris + 3 * slot), b = __ldg(mesh.tris + 3 * slot + 1), c = __ldg(mesh.tris + 3 * slot + 2);
	float3 v0 = f3(a.x, a.y, a.z), v1 = f3(b.x, b.y, b.z), v2 = f3(c.x, c.y, c.z);
	if (in) { v0 = XformPoint(in->object_to_world, v0); v1 = XformPoint(in->object_to_world, v1); v2 = XformPoint(in->object_to_world, v2); }
	float b0 = 1.f - b1 - b2;
	float2 uv0, uv1, uv2;
	TriangleUVs(mesh, slot, uv0, uv1, uv2);
	if (uvOut) *uvOut = BaryUV(b1, b2, uv0, uv1, uv2);
	float3 dpdu, dpdv;
	TriangleDerivatives(v0, v1, v2, uv0, uv1, uv2, dpdu, dpdv);
	SurfaceInit(s, O + t * D, dpdu, dpdv);
	if (dpduOut) { *dpduOut = dpdu; *dpdvOut = dpdv; }
	if (mesh.normals) {
		float4 na = __ldg(mesh.normals + 3 * slot), nb = __ldg(mesh.normals + 3 * slot + 1), nc = __ldg(mesh.normals + 3 * slot + 2);
		float3 ns = f3(na.x, na.y, na.z) * b0 + f3(nb.x, nb.y, nb.z) * b1 + f3(nc.x, nc.y, nc.z) * b2;
		if (in) ns = XformNormal(in->world_to_object, ns);
		if (sqrLength(ns) > 0.f) ns = normalize(ns);
		else ns = s.n;
		float3 ss = normalize(dpdu);
		float3 ts = cross(ss, ns);
		if (sqrLength(ts) > 0.f) { ts = normalize(ts); ss = cross(ts, ns); }
		else CoordinateSystem(ns, &ss, &ts);
		// SetShadingGeometry(ss, ts, true): shading.n from the shading tangents, geometric n
		// flipped toward it; shading.dpdu keeps the geometric dpdu (quirk, SURVEY 8a row 17)
		s.sn = normalize(cross(ss, ts));
		s.n = Faceforward(s.n, s.sn);
	}
}

// ---------------------------------------------------------------------------------------
// EXTENSION: image textures on the base colour of Disney materials, stated in agpt.h (agpt_upload_textures) and on the
// CPU in statements/agpt_texture_oracle.cpp.  Plain loads: the texture unit's filtering weights are 8-bit fractions.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float2 PlaneUV(const agpt_plane& pl, float3 p) {
	return make_float2(((p.x - pl.o[0]) / pl.half_x + 1) * 0.5f, ((p.z - pl.o[2]) / pl.half_z + 1) * 0.5f);
}
__device__ __forceinline__ int TexWrap(int x, int n) { return x < 0 ? x + n : x >= n ? x - n : x; }
__device__ __forceinline__ float3 TexelAt(const DTexTables& tt, const DTexture& d, int x, int y) {
	const long long i = d.off + (long long)y * d.width + x;
	AGPT_CHECK(i >= d.off && i < d.off + (long long)d.width * d.height && i < tt.nTexels, AGPT_DBG_TEXEL, i);
	const float4 t = __ldg(tt.texels + i);
	return f3(t.x, t.y, t.z);
}
// bilinear, repeat-wrapped, texel centres at (i + 0.5) / W
__device__ __forceinline__ float3 TexLookup(const DTexTables& tt, int tex, float2 uv) {
	AGPT_CHECK(tex >= 0 && tex < tt.nTextures, AGPT_DBG_TEXTURE, tex);
	const DTexture d = tt.textures[tex];
	const float u = isfinite(uv.x) ? uv.x - floorf(uv.x) : 0.f, v = isfinite(uv.y) ? uv.y - floorf(uv.y) : 0.f;
	const float s = u * (float)d.width - 0.5f, t = v * (float)d.height - 0.5f;
	const float fs = floorf(s), ft = floorf(t);
	const int x0 = TexWrap((int)fs, d.width), x1 = TexWrap((int)fs + 1, d.width);
	const int y0 = TexWrap((int)ft, d.height), y1 = TexWrap((int)ft + 1, d.height);
	const float fx = s - fs, fy = t - ft;
	const float3 t00 = TexelAt(tt, d, x0, y0), t10 = TexelAt(tt, d, x1, y0), t01 = TexelAt(tt, d, x0, y1), t11 = TexelAt(tt, d, x1, y1);
	const float3 a = t00 + fx * (t10 - t00), b = t01 + fx * (t11 - t01);
	return a + fy * (b - a);
}
// channel k (0, 1, 2) of the same lookup: the alpha of a mask (the three channels' arithmetic is independent, so this is the
// one-channel lookup bit for bit)
__device__ __forceinline__ float TexLookupChannel(const DTexTables& tt, int tex, int k, float2 uv) {
	const float3 c = TexLookup(tt, tex, uv);
	return k == 0 ? c.x : k == 1 ? c.y : c.z;
}
// The two colours a Disney material derives from its base colour (host/material.h DisneyMaterial), for one hit.
struct TexColors {
	float3 diffuse;   // agpt_material.diffuse_r
	float3 spec0;     // agpt_material.spec_r0
};
// DisneyMaterial's colour arithmetic (host/material.h) for base colour c: the one statement of it on the device
__device__ __forceinline__ TexColors DisneyColors(float3 c, float metallic, float eta) {
	TexColors tc;
	const float dw = (1 - metallic) * (1 - 0.f);
	tc.diffuse = dw > 0 ? dw * c : f3(0.f);
	const float r0 = ((eta - 1) * (eta - 1)) / ((eta + 1) * (eta + 1));
	tc.spec0 = Lerp(metallic, f3(r0), c);
	return tc;
}
__device__ __forceinline__ TexColors HitColors(const DTexTables& tt, int material, const agpt_material& m, float2 uv) {
	TexColors tc;
	const int tex = tt.matTex[material];
	if (tex < 0) { tc.diffuse = f3(m.diffuse_r); tc.spec0 = f3(m.spec_r0); return tc; }
	return DisneyColors(TexLookup(tt, tex, uv), m.metallic, m.eta);
}

// ---------------------------------------------------------------------------------------
// EXTENSION: roughness-metallic and normal maps on Disney materials, stated in agpt.h (agpt_upload_material_textures) and on
// the CPU in statements/agpt_material_maps_oracle.cpp.  The TEX == 2 instantiations shade with the record this builds.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float MapClamp01(float x) { return x < 0.f ? 0.f : x > 1.f ? 1.f : x; }
// step 1: the hit's material record
__device__ __forceinline__ agpt_material MapsMaterial(const DTexTables& tt, const DMatMaps& mm, const agpt_material& rec, float2 uv) {
	agpt_material m = rec;
	if (mm.roughnessMetallic < 0 && mm.base < 0) return m;
	float r = rec.roughness, k = rec.metallic;
	float3 C;
	if (mm.roughnessMetallic < 0) C = TexLookup(tt, mm.base, uv);          // agpt_upload_textures step 3
	else {
		const float3 rm = TexLookup(tt, mm.roughnessMetallic, uv);
		C = mm.base >= 0 ? TexLookup(tt, mm.base, uv) : f3(mm.color[0], mm.color[1], mm.color[2]);
		r = rec.roughness * MapClamp01(rm.y); k = rec.metallic * MapClamp01(rm.z);
		const float a = smax(.001f, smax(.001f, r * r));         // std::max, as the constructor
		m.lobes = ((1 - k) * (1 - 0.f) > 0 ? (uint32_t)(AGPT_LOBE_DIFFUSE | AGPT_LOBE_RETRO) : 0u) | (uint32_t)AGPT_LOBE_MICROFACET;
		m.roughness = r; m.metallic = k;
		m.alpha_x = a; m.alpha_y = a;
	}
	const TexColors tc = DisneyColors(C, k, rec.eta);
	m.diffuse_r[0] = tc.diffuse.x; m.diffuse_r[1] = tc.diffuse.y; m.diffuse_r[2] = tc.diffuse.z;
	m.spec_r0[0] = tc.spec0.x; m.spec_r0[1] = tc.spec0.y; m.spec_r0[2] = tc.spec0.z;
	return m;
}
// step 2: the normal map's shading frame; T, B = dp/du, dp/dv of the texture's uv.  Leaves s as it is in the three cases agpt.h
// names, so a flat map reproduces the unmapped surface bit for bit.
__device__ __forceinline__ void ApplyNormalMap(const DTexTables& tt, int tex, float scale, float2 uv, float3 T, float3 B, DSurface& s) {
	const float3 c = TexLookup(tt, tex, uv);
	const float3 nts = f3(scale * (2 * c.x - 1), scale * (2 * c.y - 1), 2 * c.z - 1);
	if (nts.x == 0 && nts.y == 0 && nts.z > 0) return;
	const float3 N = s.sn;
	float3 Tp = T - N * dot(N, T);
	if (dot(Tp, Tp) == 0) return;
	Tp = normalize(Tp);
	float3 Bp = cross(N, Tp);
	if (dot(Bp, B) < 0) Bp = -Bp;
	float3 n = (nts.x * Tp + nts.y * Bp) + nts.z * N;
	if (!(dot(n, N) > 0)) return;
	n = normalize(n);
	s.sn = n;
	s.sdpdu = Tp - n * dot(n, Tp);
}
// steps 1 and 2 for a hit on material `material` (a Disney record: the render-time check binds maps to nothing else)
__device__ __forceinline__ agpt_material HitMaps(const DTexTables& tt, int material, const agpt_material& rec, float2 uv, float3 T, float3 B, DSurface& s) {
	AGPT_CHECK(material >= 0 && material < tt.nMatMaps, AGPT_DBG_MAPS, material);
	const DMatMaps mm = tt.matMaps[material];
	if (mm.normal >= 0) ApplyNormalMap(tt, mm.normal, mm.normalScale, uv, T, B, s);
	return MapsMaterial(tt, mm, rec, uv);
}

// ---------------------------------------------------------------------------------------
// Sphere light sampling (intersectable.h:230-317)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void SphereSampleFrom(const agpt_sphere& sp, float3 refP, float2 u, float3* pOut, float3* nOut, float* pdf) {
	float3 pCenter = f3(sp.center);
	if (sqrLength(refP - pCenter) <= sp.r2) {
		// uniform area sampling (:230-237) converted to solid angle (:245-256)
		float3 pObj = pCenter + sp.r * RandomInSphereU(u);
		float3 n = normalize(pObj);      // upstream normalises the world position (kept)
		*pdf = 1 / (4.f * AGPT_PI * sp.r2);
		float3 wi = pObj - refP;
		if (sqrLength(wi) == 0) *pdf = 0;
		else {
			wi = normalize(wi);
			*pdf *= sqrLength(refP - pObj) / absdot(n, -wi);
		}
		if (isinf(*pdf)) *pdf = 0;
		*pOut = pObj; *nOut = n;
		return;
	}
	float dc = length(refP - pCenter);
	float invDc = 1 / dc;
	float3 wc = (pCenter - refP) * invDc;
	float3 wcX, wcY;
	CoordinateSystem(wc, &wcX, &wcY);
	float sinThetaMax = sp.r * invDc;
	float sinThetaMax2 = sinThetaMax * sinThetaMax;
	float invSinThetaMax = 1 / sinThetaMax;
	float cosThetaMax = sqrtf(smax(0.f, 1 - sinThetaMax2));
	float cosTheta = (cosThetaMax - 1) * u.x + 1;
	float sinTheta2 = 1 - cosTheta * cosTheta;
	if (sinThetaMax2 < 0.00068523f) {
		sinTheta2 = sinThetaMax2 * u.x;
		cosTheta = sqrtf(1 - sinTheta2);
	}
	float cosAlpha = sinTheta2 * invSinThetaMax + cosTheta * sqrtf(smax(0.f, 1.f - sinTheta2 * invSinThetaMax * invSinThetaMax));
	float sinAlpha = sqrtf(smax(0.f, 1.f - cosAlpha * cosAlpha));
	float phi = u.y * 2 * AGPT_PI;
	float3 nWorld = SphericalDirection(sinAlpha, cosAlpha, phi, -wcX, -wcY, -wc);
	*pOut = pCenter + sp.r * f3(nWorld.x, nWorld.y, nWorld.z);
	*nOut = nWorld;
	*pdf = 1 / (2 * AGPT_PI * (1 - cosThetaMax));
}
__device__ __forceinline__ float SpherePdfFrom(const agpt_sphere& sp, float3 refP) {
	float3 pCenter = f3(sp.center);
	if (sqrLength(refP - pCenter) <= sp.r2) return 1 / (4 * AGPT_PI);
	float sinThetaMax2 = sp.r2 / sqrLength(refP - pCenter);
	float cosThetaMax = sqrtf(smax(0.f, 1 - sinThetaMax2));
	return UniformConePdf(cosThetaMax);
}

// ---------------------------------------------------------------------------------------
// InfiniteAreaLight (lights.cpp:31-112, built with ILS), HDRTexture::value (texture.h:59-67),
// Distribution1D::SampleContinuous / DiscretePDF (sampling.h:4-18,38-64)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float SphericalTheta(float3 v) { return racos(rclamp(v.z, -1.f, 1.f)); }                 // common.h:158-160
__device__ __forceinline__ float SphericalPhi(float3 v) { float p = ratan2(v.y, v.x); return (p < 0) ? (p + AGPT_TWOPI) : p; }   // common.h:162-165
__device__ __forceinline__ int EnvMod(int a, int b) { int r = a - (a / b) * b; return r < 0 ? r + b : r; }           // texture.h:78-81
__device__ __forceinline__ float3 EnvTexel(const DScene& sc, int x, int y) {
	const float* p = sc.envRgb + 3 * ((size_t)y * sc.envW + x);
	return f3(__ldg(p), __ldg(p + 1), __ldg(p + 2));
}
// InfiniteAreaLight::Le(ray): direction -> lat-long texel, nearest lookup with wrap (lights.cpp:108-112)
__device__ __noinline__ float3 EnvLe(const DScene& sc, float3 rayD) {
	float3 w = normalize(rayD);
	w = f3(w.x, w.z, w.y);
	float u = SphericalPhi(w) * AGPT_INV2PI, v = SphericalTheta(w) * AGPT_INVPI;
	int s = (int)floorf(u * sc.envW - .5f);
	int t = (int)floorf(v * sc.envH - .5f);
	return EnvTexel(sc, EnvMod(s, sc.envW), EnvMod(t, sc.envH));
}
// InfiniteAreaLight::Pdf_Li (lights.cpp:92-106)
__device__ __noinline__ float EnvPdfLi(const DScene& sc, float3 wi) {
	float3 w = normalize(wi);
	w = f3(w.x, w.z, w.y);
	float theta = SphericalTheta(w), phi = SphericalPhi(w);
	float sinTheta = rsin(theta);
	if (sinTheta == 0) return 0;
	int x = min(max((int)(phi * AGPT_INV2PI * sc.envW), 0), sc.envW - 1);
	int y = min(max((int)(theta * AGPT_INVPI * sc.envH), 0), sc.envH - 1);
	int count = sc.envW * sc.envH;
	float discrete = __ldg(sc.envFunc + (y * sc.envW + x)) / (sc.envFuncInt * count);
	return count * discrete / (2 * AGPT_PI * AGPT_PI * sinTheta);
}
// InfiniteAreaLight::Sample_Li (lights.cpp:50-90): u01 is the one extra draw it makes.
// Returns false where upstream returns black before writing *pdf (mapPdf == 0).
__device__ __noinline__ bool EnvSampleLi(const DScene& sc, float u01, float3* wi, float* pdf) {
	const int n = sc.envW * sc.envH;
	// FindInterval(cdf.size(), cdf[index] <= u) (sampling.h:4-18)
	int first = 0, len = n + 1;
	while (len > 0) {
		int half = len >> 1, middle = first + half;
		if (__ldg(sc.envCdf + middle) <= u01) { first = middle + 1; len -= half + 1; }
		else len = half;
	}
	int offset = min(max(first - 1, 0), n + 1 - 2);
	float c0 = __ldg(sc.envCdf + offset), c1 = __ldg(sc.envCdf + offset + 1);
	float du = u01 - c0;
	if ((c1 - c0) > 0) du /= c1 - c0;
	float mapPdf = (sc.envFuncInt > 0) ? __ldg(sc.envFunc + offset) / sc.envFuncInt : 0;
	float sample = (offset + du) / n;
	if (mapPdf == 0) return false;
	int idx = (int)(sample * n);
	float uvx = ((idx % sc.envW) + .5f) / sc.envW, uvy = ((idx / sc.envW) + .5f) / sc.envH;
	float theta = uvy * AGPT_PI, phi = uvx * AGPT_TWOPI;
	float cosTheta = rcos(theta), sinTheta = rsin(theta);
	float sinPhi = rsin(phi), cosPhi = rcos(phi);
	*wi = f3(sinTheta * cosPhi, cosTheta, sinTheta * sinPhi);
	*pdf = mapPdf / (2 * AGPT_PI * AGPT_PI * sinTheta);
	if (sinTheta == 0) *pdf = 0;
	return true;
}

__device__ __forceinline__ float PowerHeuristic(int nf, float fPdf, int ng, float gPdf) {   // integrator.h:33-36
	float f = nf * fPdf, g = ng * gPdf;
	return (f * f) / (f * f + g * g);
}

// ---------------------------------------------------------------------------------------
// Fused per-vertex evaluation used by the shade kernel.
//
// One path vertex needs the BSDF at three directions: the light sample (BSDF::f + BSDF::Pdf,
// integrator.h:46-47), the MIS sample and the continuation sample (BSDF::Sample_f twice,
// integrator.h:66,174 -- each re-evaluates every lobe's f and Pdf at the sampled direction,
// reflection.h:156-171).  Evaluated through BSDF_f / BSDF_Pdf / BSDF_Sample_f above that is
// four copies of the microfacet code and ~28 K SASS instructions in k_shade, which made the
// kernel instruction-fetch bound (ncu: stall_no_instruction dominant).  Here the terms that
// depend on wo only (local wo, Schlick weight, G1(wo)) are computed once per vertex and ONE
// out-of-line evaluator returns, for a direction, the summed lobe values and the two distinct
// lobe pdfs.  Every value is produced by the same operations in the same order as the
// reference's per-function code (reflection.h:114-188); the probe kernel runs exactly these
// functions against golden vectors of the reference's BSDF::f / Pdf / Sample_f.
// ---------------------------------------------------------------------------------------
struct VertexBsdf {
	DBSDF b;
	float3 woW, wo;          // outgoing direction, world and shading space
	float absCosO, Fo, G1o;  // |cos theta_o|, SchlickWeight(|cos theta_o|), G1(wo)
	float lambdaO;           // Lambda(wo) (GLASS only: the non-separable G of the plain Trowbridge-Reitz distribution)
	bool woOk;               // wo.z != 0 (BSDF::f / Pdf / Sample_f return 0 otherwise)
	int nLobes;              // non-specular lobes: diffuse, retro, microfacet, glass reflection, glass transmission
};
// GLASS: the scene has a rough-dielectric material (extension); the instantiation without it carries none of that code.
template <bool GLASS>
__device__ __forceinline__ void VertexBsdfInit(VertexBsdf& v, const DSurface& si, const agpt_material* m, float3 woW) {
	v.b = MakeBSDF(si, m);
	v.woW = woW;
	v.wo = WorldToLocal(v.b, woW);
	v.woOk = v.wo.z != 0;
	v.absCosO = AbsCosTheta(v.wo);
	v.Fo = SchlickWeight(v.absCosO);
	v.lambdaO = 0.f;
	if (GLASS && (m->lobes & (AGPT_LOBE_GLASS_REFLECT | AGPT_LOBE_GLASS_TRANSMIT))) {
		v.lambdaO = TR_Lambda(m->alpha_x, m->alpha_y, v.wo);
		v.G1o = 1 / (1 + v.lambdaO);
	}
	else v.G1o = (m->lobes & AGPT_LOBE_MICROFACET) ? TR_G1(m->alpha_x, m->alpha_y, v.wo) : 0.f;
	v.nLobes = ((m->lobes & AGPT_LOBE_DIFFUSE) ? 1 : 0) + ((m->lobes & AGPT_LOBE_RETRO) ? 1 : 0) + ((m->lobes & AGPT_LOBE_MICROFACET) ? 1 : 0);
	if (GLASS) v.nLobes += ((m->lobes & AGPT_LOBE_GLASS_REFLECT) ? 1 : 0) + ((m->lobes & AGPT_LOBE_GLASS_TRANSMIT) ? 1 : 0);
}

struct LobeEval {
	float3 f;          // sum of the non-specular lobes' f(wo, wi) in bxdfs[] order (caller applies `reflect`)
	float pdfCos;      // BxDF::Pdf of a cosine-sampled lobe (reflection.h:16-18)
	float pdfMicro;    // MicrofacetReflection::Pdf (reflection.h:67-71): the Disney microfacet lobe or the glass reflection lobe
	float3 fT;         // GLASS: f of the transmission lobe (contributes when wi, wo lie on opposite sides of the geometric normal)
	float pdfT;        // GLASS: MicrofacetTransmission::Pdf
};
// TEX (extension): the diffuse reflectance and Schlick R0 come from tc (the hit's textured colours), not from the record.
template <bool GLASS, bool TEX = false>
__device__ __forceinline__ void EvalLobes(const VertexBsdf& v, float3 wi, LobeEval& out, TexColors tc = TexColors()) {
	const agpt_material& m = *v.b.mat;
	const float absCosI = AbsCosTheta(wi);
	const bool same = SameHemisphere(v.wo, wi);
	out.pdfCos = same ? absCosI * AGPT_INVPI : 0;
	out.pdfMicro = 0;
	float3 f = f3(0.f);
	float3 wh = wi + v.wo;
	const bool whZero = wh.x == 0 && wh.y == 0 && wh.z == 0;
	wh = normalize(wh);
	const float Fi = SchlickWeight(absCosI);
	const float3 R = TEX ? tc.diffuse : f3(m.diffuse_r);
	if (m.lobes & AGPT_LOBE_DIFFUSE) f += R * AGPT_INVPI * (1 - v.Fo / 2) * (1 - Fi / 2);                 // disney.h:27-34
	if (m.lobes & AGPT_LOBE_RETRO) {                                                                    // disney.h:42-54
		float3 fr = f3(0.f);
		if (!whZero) {
			float cosThetaD = dot(wi, wh);
			float Rr = 2 * m.roughness * cosThetaD * cosThetaD;
			fr = R * AGPT_INVPI * Rr * (v.Fo + Fi + v.Fo * Fi * (Rr - 1));
		}
		f += fr;
	}
	if (m.lobes & AGPT_LOBE_MICROFACET) {                                                               // reflection.h:42-54,67-71
		float3 fm = f3(0.f);
		if (!(absCosI == 0 || v.absCosO == 0) && !whZero) {
			float3 F = TEX ? DisneyFresnel(m, tc.spec0, dot(wi, Faceforward(wh, f3(0, 0, 1)))) : DisneyFresnel(m, dot(wi, Faceforward(wh, f3(0, 0, 1))));
			float D = TR_D(m.alpha_x, m.alpha_y, wh);
			float G = v.G1o * TR_G1(m.alpha_x, m.alpha_y, wi);
			fm = f3(1.f) * D * G * F / (4 * absCosI * v.absCosO);
			if (same) out.pdfMicro = D * v.G1o * absdot(v.wo, wh) / v.absCosO / (4 * dot(v.wo, wh));
		}
		f += fm;
	}
	out.fT = f3(0.f); out.pdfT = 0.f;
	if (GLASS && (m.lobes & (AGPT_LOBE_GLASS_REFLECT | AGPT_LOBE_GLASS_TRANSMIT))) {
		const float lambdaI = TR_Lambda(m.alpha_x, m.alpha_y, wi);
		if (m.lobes & AGPT_LOBE_GLASS_REFLECT) {                                                        // reflection.h:42-54,67-71 + microfacet.h:103-105,220-228
			float3 fr = f3(0.f);
			if (!(absCosI == 0 || v.absCosO == 0) && !whZero) {
				float3 F = f3(FrDielectric(dot(wi, Faceforward(wh, f3(0, 0, 1))), 1.f, m.eta));
				float D = TR_D(m.alpha_x, m.alpha_y, wh);
				float G = 1 / (1 + v.lambdaO + lambdaI);
				fr = f3(m.mirror_r) * D * G * F / (4 * absCosI * v.absCosO);
			}
			// (MicrofacetReflection::Pdf has no zero-vector check: wh = normalize(wo + wi) as is)
			if (same) out.pdfMicro = TR_D(m.alpha_x, m.alpha_y, wh) * v.G1o * absdot(v.wo, wh) / v.absCosO / (4 * dot(v.wo, wh));
			f += fr;
		}
		if (m.lobes & AGPT_LOBE_GLASS_TRANSMIT) {
			out.fT = GlassT_f(m, v.wo, wi, v.lambdaO, lambdaI);
			out.pdfT = GlassT_Pdf(m, v.wo, wi, v.G1o, v.absCosO);
		}
	}
	out.f = f;
}

// BSDF::f and BSDF::Pdf of a given world direction from one EvalLobes result (reflection.h:114-123,
// 174-188; specular lobes contribute nothing to either).  The caller checks v.woOk.
template <bool GLASS>
__device__ __forceinline__ float3 FinishEval(const VertexBsdf& v, const LobeEval& e, float3 wiW, float* pdfOut) {
	const agpt_material& m = *v.b.mat;
	bool reflect = dot(wiW, v.b.ng) * dot(v.woW, v.b.ng) > 0;
	float p = 0.f;
	if (m.lobes & AGPT_LOBE_DIFFUSE) p += e.pdfCos;
	if (m.lobes & AGPT_LOBE_RETRO) p += e.pdfCos;
	if (m.lobes & AGPT_LOBE_MICROFACET) p += e.pdfMicro;
	if (GLASS && (m.lobes & AGPT_LOBE_GLASS_REFLECT)) p += e.pdfMicro;
	if (GLASS && (m.lobes & AGPT_LOBE_GLASS_TRANSMIT)) p += e.pdfT;
	*pdfOut = v.nLobes > 0 ? p / v.nLobes : 0.f;
	return reflect ? e.f : (GLASS ? e.fT : f3(0.f));
}

struct DirSample {
	float3 wi;        // sampled direction, shading space
	float3 fSpec;     // value of a specular lobe (reflection.cpp:13-17)
	float pdf;        // pdf of the chosen lobe alone
	int lobe;         // AGPT_LOBE_* that was sampled
	int matching;     // lobes that took part in the choice
	bool ok;          // false where BSDF::Sample_f returns black (reflection.h:130-157)
};
// First half of BSDF::Sample_f: choose the lobe, remap u, sample its direction (reflection.h:126-157).
template <bool GLASS>
__device__ __forceinline__ void SampleLobeDir(const VertexBsdf& v, float2 u, bool skipSpecular, DirSample& s) {
	const agpt_material& m = *v.b.mat;
	int lobes[6];
	int matching = LobeList(m, skipSpecular, lobes);
	s.ok = false; s.pdf = 0; s.lobe = 0; s.matching = matching; s.wi = f3(0.f); s.fSpec = f3(0.f);
	if (matching == 0) return;
	int comp = min((int)floorf(u.x * matching), matching - 1);
	int lobe = lobes[comp];
	float2 uR = make_float2(smin(u.x * matching - comp, AGPT_ONE_MINUS_EPS), u.y);
	s.lobe = lobe;
	if (!v.woOk) return;
	float3 wo = v.wo, wi = f3(0.f);
	float pdf = 0;
	if (lobe == AGPT_LOBE_SPECULAR) {
		wi = f3(-wo.x, -wo.y, wo.z);
		pdf = 1;
		s.fSpec = f3(1.f) * f3(m.mirror_r) / AbsCosTheta(wi);
	}
	else if (lobe == AGPT_LOBE_MICROFACET || (GLASS && lobe == AGPT_LOBE_GLASS_REFLECT)) {
		float3 wh = TR_Sample_wh(m.alpha_x, m.alpha_y, wo, uR);
		if (!(dot(wo, wh) < 0)) {
			wi = Reflect(wo, wh);
			if (SameHemisphere(wo, wi))
				pdf = TR_D(m.alpha_x, m.alpha_y, wh) * v.G1o * absdot(wo, wh) / v.absCosO / (4 * dot(wo, wh));
		}
	}
	else if (GLASS && lobe == AGPT_LOBE_GLASS_TRANSMIT) {                          // MicrofacetTransmission::Sample_f
		float3 wh = TR_Sample_wh(m.alpha_x, m.alpha_y, wo, uR);
		if (!(dot(wo, wh) < 0)) {
			float eta = CosTheta(wo) > 0 ? (1.f / m.eta) : (m.eta / 1.f);
			if (Refract(wo, wh, eta, &wi)) pdf = GlassT_Pdf(m, wo, wi, v.G1o, v.absCosO);
		}
	}
	else {
		wi = CosineSampleHemisphere(uR);
		if (wo.z < 0) wi.z *= -1;
		pdf = Cosine_Pdf(wo, wi);
	}
	if (pdf == 0) return;
	s.wi = wi; s.pdf = pdf; s.ok = true;
}
// Second half of BSDF::Sample_f: overall pdf over the matching lobes and the BSDF value (reflection.h:158-171).
template <bool GLASS>
__device__ __forceinline__ float3 FinishSample(const VertexBsdf& v, const DirSample& s, const LobeEval& e, float3 wiW, float* pdfOut) {
	const agpt_material& m = *v.b.mat;
	const bool specular = s.lobe == AGPT_LOBE_SPECULAR;
	float pdf = s.pdf;
	if (!specular && s.matching > 1) {
		if ((m.lobes & AGPT_LOBE_DIFFUSE) && s.lobe != AGPT_LOBE_DIFFUSE) pdf += e.pdfCos;
		if ((m.lobes & AGPT_LOBE_RETRO) && s.lobe != AGPT_LOBE_RETRO) pdf += e.pdfCos;
		if ((m.lobes & AGPT_LOBE_MICROFACET) && s.lobe != AGPT_LOBE_MICROFACET) pdf += e.pdfMicro;
		if (GLASS && (m.lobes & AGPT_LOBE_GLASS_REFLECT) && s.lobe != AGPT_LOBE_GLASS_REFLECT) pdf += e.pdfMicro;
		if (GLASS && (m.lobes & AGPT_LOBE_GLASS_TRANSMIT) && s.lobe != AGPT_LOBE_GLASS_TRANSMIT) pdf += e.pdfT;
	}
	if (s.matching > 1) pdf /= s.matching;
	*pdfOut = pdf;
	if (specular) return s.fSpec;
	bool reflect = dot(wiW, v.b.ng) * dot(v.woW, v.b.ng) > 0;
	return reflect ? e.f : (GLASS ? e.fT : f3(0.f));
}

