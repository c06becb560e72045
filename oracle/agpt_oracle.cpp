// oracle/agpt_oracle.cpp -- TEST INFRASTRUCTURE, not product code.
//
// Plain C++ restatement of the reference's per-pixel path-tracing hot path, working on the
// flattened scene tables of include/agpt.h (the same tables the GPU gets).  Every function
// cites the /root/reference lines it follows.  It is a checker: only tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline leg may load the library built from it.
//
// Pinned: tests/test_oracle_port.py compares it BIT FOR BIT with oracle/_ref (the reference's
// own sources compiled from /root/reference) on every configuration, and with the golden
// fixtures under tests/golden/ (generated from oracle/_ref by tests/golden/make_golden.py), so
// the restatement is anchored on the reference itself.  Same compiler, same flags (-O2, no
// FMA contraction, no fast-math), same glibc libm => identical bits are expected, not a tolerance.
//
// Unlike the GPU wavefront this follows the reference's own control flow: recursive BVH
// descent (bvhtrimesh.h:332-413) and the sequential bounce loop of PathTracer::Li
// (integrator.h:124-191) with one RNG stream per (pixel, sample).
#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include "agpt.h"

namespace {

// ---- math in the reference's operation order (template/precomp.h:363-768) ---------------
struct V3 { float x, y, z; };
inline V3 v3(float x, float y, float z) { return { x, y, z }; }
inline V3 v3(float s) { return { s, s, s }; }
inline V3 v3(const float* p) { return { p[0], p[1], p[2] }; }
inline V3 operator-(V3 a) { return { -a.x, -a.y, -a.z }; }
inline V3 operator+(V3 a, V3 b) { return { a.x + b.x, a.y + b.y, a.z + b.z }; }
inline V3 operator-(V3 a, V3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
inline V3 operator*(V3 a, V3 b) { return { a.x * b.x, a.y * b.y, a.z * b.z }; }
inline V3 operator*(V3 a, float s) { return { a.x * s, a.y * s, a.z * s }; }
inline V3 operator*(float s, V3 a) { return { s * a.x, s * a.y, s * a.z }; }
inline V3 operator/(V3 a, float s) { return { a.x / s, a.y / s, a.z / s }; }
inline void operator+=(V3& a, V3 b) { a.x += b.x; a.y += b.y; a.z += b.z; }
inline void operator*=(V3& a, V3 b) { a.x *= b.x; a.y *= b.y; a.z *= b.z; }
inline void operator/=(V3& a, float s) { a.x /= s; a.y /= s; a.z /= s; }
inline float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }                // precomp.h:701
inline float sqrLength(V3 v) { return dot(v, v); }
inline float length(V3 v) { return sqrtf(dot(v, v)); }
inline float absdot(V3 a, V3 b) { return std::abs(dot(a, b)); }
inline V3 normalize(V3 v) { float inv = 1.0f / sqrtf(dot(v, v)); return v * inv; }        // precomp.h:366,735
inline V3 cross(V3 a, V3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }
inline bool IsBlack(V3 v) { return v.x == 0 && v.y == 0 && v.z == 0; }
inline V3 Faceforward(V3 v, V3 v2) { return (dot(v, v2) < 0.f) ? -v : v; }
inline V3 Lerp(float t, V3 a, V3 b) { return (1 - t) * a + t * b; }
inline V3 Reflect(V3 wo, V3 n) { return -wo + 2.0f * dot(wo, n) * n; }
inline float tmin2(float a, float b) { return a < b ? a : b; }        // template fminf (precomp.h:364)
inline float tmax2(float a, float b) { return a > b ? a : b; }        // template fmaxf (precomp.h:365)
inline float tclamp(float f, float a, float b) { return tmax2(a, tmin2(f, b)); }   // precomp.h:678

const float kPi = 3.14159265358979323846264f, kInvPi = 0.31830988618379067153777f;
const float kInv2Pi = 0.15915494309189533576888f, kTwoPi = 6.28318530717958647692528f, kEps = 0.0001f;
const float kOneMinusEps = 0x1.fffffep-1;

inline void CoordinateSystem(V3 v1, V3* v2, V3* v3o) {                                     // common.h:145-151
	if (std::abs(v1.x) > std::abs(v1.y)) *v2 = v3(-v1.z, 0, v1.x) / std::sqrt(v1.x * v1.x + v1.z * v1.z);
	else *v2 = v3(0, v1.z, -v1.y) / std::sqrt(v1.y * v1.y + v1.z * v1.z);
	*v3o = cross(v1, *v2);
}

// ---- RNG (template/template.cpp:666-685, cl/tools.cl:1-4; stream definition SURVEY 8a row 3)
inline uint32_t WangHash(uint32_t s) { s = (s ^ 61u) ^ (s >> 16); s *= 9u; s = s ^ (s >> 4); s *= 0x27d4eb2du; s = s ^ (s >> 15); return s; }
struct Rng {
	uint32_t s;
	int draws = 0;
	void Seed(uint32_t pixel, uint32_t sample) { s = WangHash(WangHash((pixel + 1u) * 17u) + sample); if (!s) s = 1u; draws = 0; }
	float Float() { s ^= s << 13; s ^= s >> 17; s ^= s << 5; draws++; return s * 2.3283064365387e-10f; }
};

// ---- scene (copies of the flattened tables) ---------------------------------------------
struct Mesh {
	std::vector<agpt_bvh_node> nodes;
	std::vector<float> verts;     // 12 floats per triangle (3 x float4), leaf order
	std::vector<int32_t> ids;
	std::vector<float> normals;   // 12 floats per triangle or empty
	std::vector<float> uvs;       // 6 floats per triangle or empty
};
struct OScene {
	std::vector<agpt_prim> prims;
	std::vector<agpt_sphere> spheres;
	std::vector<agpt_plane> planes;
	std::vector<Mesh> meshes;
	std::vector<agpt_material> mats;
	std::vector<agpt_light> lights;
	std::vector<agpt_instance> instances;    // extension: placed meshes (agpt.h)
	agpt_camera cam;
	// InfiniteAreaLight tables (lights.cpp:31-48, texture.h:41-57, sampling.h:22-35)
	int envW = 0, envH = 0;
	std::vector<float> envRgb, envFunc, envCdf;
	float envFuncInt = 0;
	bool rrByBounce = false;           // extension: Russian roulette keyed on the bounce index (see Li)
};

struct Ray {                       // camera.h:3-15
	V3 O, D;
	float t;
	Ray(V3 o, V3 d, float tt = FLT_MAX) : O(o), D(normalize(d)), t(tt) {}
	struct AsGiven {};             // object-space rays of instances keep their (unnormalised) direction: same t as in world space
	Ray(AsGiven, V3 o, V3 d, float tt) : O(o), D(d), t(tt) {}
};

// ---- EXTENSION: instances (agpt.h agpt_instance).  Parity unpinned by the reference -- it has no transforms at trace
// time; this is the statement the GPU path is checked against.  3x4 row-major affine, sums left to right.
inline V3 XformPoint(const float* m, V3 p) { return v3(m[0] * p.x + m[1] * p.y + m[2] * p.z + m[3], m[4] * p.x + m[5] * p.y + m[6] * p.z + m[7], m[8] * p.x + m[9] * p.y + m[10] * p.z + m[11]); }
inline V3 XformVector(const float* m, V3 v) { return v3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[4] * v.x + m[5] * v.y + m[6] * v.z, m[8] * v.x + m[9] * v.y + m[10] * v.z); }
inline V3 XformNormal(const float* w2o, V3 n) { return v3(w2o[0] * n.x + w2o[4] * n.y + w2o[8] * n.z, w2o[1] * n.x + w2o[5] * n.y + w2o[9] * n.z, w2o[2] * n.x + w2o[6] * n.y + w2o[10] * n.z); }   // transpose(W2O)

struct Counters {
	uint64_t raysClosest = 0, raysAny = 0, interior = 0, boxes = 0, tris = 0, analytic = 0;
	void Add(const Counters& o) { raysClosest += o.raysClosest; raysAny += o.raysAny; interior += o.interior; boxes += o.boxes; tris += o.tris; analytic += o.analytic; }
};

struct Hit {
	int prim = -1, slot = -1;
	float t = 0, b1 = 0, b2 = 0;
};

inline const Mesh& MeshOfPrim(const OScene& sc, const agpt_prim& pr) { return sc.meshes[pr.type == AGPT_PRIM_INSTANCE ? sc.instances[pr.payload].mesh : pr.payload]; }

// Bounds::Intersect (bvhtrimesh.h:18-36), per-axis early out as written upstream
bool BoundsIntersect(const agpt_bvh_node& n, const Ray& ray, float& t) {
	float tmin = 0.0f, tmax = ray.t;
	const float O[3] = { ray.O.x, ray.O.y, ray.O.z }, D[3] = { ray.D.x, ray.D.y, ray.D.z };
	for (int a = 0; a < 3; a++) {
		float t0 = tmin2((n.bmin[a] - O[a]) / D[a], (n.bmax[a] - O[a]) / D[a]);
		float t1 = tmax2((n.bmin[a] - O[a]) / D[a], (n.bmax[a] - O[a]) / D[a]);
		tmin = tmax2(t0, tmin);
		tmax = tmin2(t1, tmax);
		if ((tmax * 1.00000024f) < tmin) return false;
	}
	t = tmin;
	return true;
}

// trianglemesh.cpp:59-80: partial derivatives; false = triangle declared degenerate
bool TriangleDerivatives(V3 v0, V3 v1, V3 v2, const float* uv, V3& dpdu, V3& dpdv) {
	float duv02x = uv[0] - uv[4], duv02y = uv[1] - uv[5], duv12x = uv[2] - uv[4], duv12y = uv[3] - uv[5];
	V3 dp02 = v0 - v2, dp12 = v1 - v2;
	float determinant = duv02x * duv12y - duv02y * duv12x;
	bool degenerateUV = std::abs(determinant) < 1e-8;
	if (!degenerateUV) {
		float invdet = 1 / determinant;
		dpdu = (duv12y * dp02 - duv02y * dp12) * invdet;
		dpdv = (-duv12x * dp02 + duv02x * dp12) * invdet;
	}
	if (degenerateUV || sqrLength(cross(dpdu, dpdv)) == 0) {
		V3 ng = cross(v2 - v0, v1 - v0);
		if (sqrLength(ng) == 0) return false;
		CoordinateSystem(normalize(ng), &dpdu, &dpdv);
	}
	return true;
}

void TriangleUVs(const Mesh& m, int slot, float* uv) {
	if (!m.uvs.empty()) memcpy(uv, &m.uvs[6 * (size_t)slot], 6 * sizeof(float));
	else { const float d[6] = { 0, 0, 1, 0, 1, 1 }; memcpy(uv, d, sizeof(d)); }           // trianglemesh.cpp:52-56
}

// TriangleMesh::TriangleIntersect / TriangleIntersectP up to the point where the hit is
// committed (trianglemesh.cpp:7-43,59-83 / :117-155)
bool TriangleTest(const Mesh& m, int slot, const Ray& ray, bool anyHit, float& tOut, float& b1Out, float& b2Out) {
	const float* p = &m.verts[12 * (size_t)slot];
	V3 v0 = v3(p), v1 = v3(p + 4), v2 = v3(p + 8);
	V3 e1 = v1 - v0, e2 = v2 - v0;
	V3 pvec = cross(ray.D, e2);
	float det = dot(e1, pvec);
	if (det == 0.0f) return false;
	float inv_det = 1.0f / det;
	V3 tvec = ray.O - v0;
	float b1 = dot(tvec, pvec) * inv_det;
	if (b1 < 0.0f || b1 > 1.0f) return false;
	V3 qvec = cross(tvec, e1);
	float b2 = dot(ray.D, qvec) * inv_det;
	if (b2 < 0.0f || b1 + b2 > 1.0f) return false;
	float t = dot(e2, qvec) * inv_det;
	if (t <= 0.0f || t >= ray.t) return false;
	if (!anyHit) {
		float uv[6];
		TriangleUVs(m, slot, uv);
		V3 dpdu = v3(0.f), dpdv = v3(0.f);
		if (!TriangleDerivatives(v0, v1, v2, uv, dpdu, dpdv)) return false;               // :74-77, before ray.t = t
	}
	tOut = t; b1Out = b1; b2Out = b2;
	return true;
}

// BVHTriMesh::RecursiveHit (bvhtrimesh.h:332-384)
bool RecursiveHit(const Mesh& m, int primIndex, const agpt_bvh_node& node, Ray& ray, Hit& hit, Counters& c) {
	bool any = false;
	if (node.count > 0) {
		for (int i = 0; i < node.count; i++) {
			c.tris++;
			float t, b1, b2;
			if (TriangleTest(m, node.first + i, ray, false, t, b1, b2)) {
				any = true;
				ray.t = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = primIndex; hit.slot = node.first + i;
			}
		}
		return any;
	}
	c.interior++; c.boxes += 2;
	agpt_bvh_node left = m.nodes[node.first], right = m.nodes[node.first + 1];
	float leftDist, rightDist;
	bool traverseLeft = BoundsIntersect(left, ray, leftDist);
	bool traverseRight = BoundsIntersect(right, ray, rightDist);
	bool swapKids;
	if (traverseLeft && traverseRight) swapKids = rightDist < leftDist;
	else if (traverseLeft || traverseRight) swapKids = !traverseLeft;
	else return false;
	if (swapKids) std::swap(left, right);
	if (RecursiveHit(m, primIndex, left, ray, hit, c)) any = true;
	if (traverseLeft && traverseRight && RecursiveHit(m, primIndex, right, ray, hit, c)) any = true;
	return any;
}

// BVHTriMesh::RecursiveHitP (bvhtrimesh.h:386-413)
bool RecursiveHitP(const Mesh& m, const agpt_bvh_node& node, const Ray& ray, Counters& c) {
	if (node.count > 0) {
		for (int i = 0; i < node.count; i++) {
			c.tris++;
			float t, b1, b2;
			if (TriangleTest(m, node.first + i, ray, true, t, b1, b2)) return true;
		}
		return false;
	}
	c.interior++;
	for (int k = 0; k < 2; k++) {
		const agpt_bvh_node& child = m.nodes[node.first + k];
		float tmp;
		c.boxes++;
		if (BoundsIntersect(child, ray, tmp) && RecursiveHitP(m, child, ray, c)) return true;
	}
	return false;
}

// Sphere::Intersect / IntersectP root choice (intersectable.h:164-181,207-226)
bool SphereTest(const agpt_sphere& s, const Ray& ray, float& tOut) {
	V3 oc = ray.O - v3(s.center);
	float half_b = dot(oc, ray.D);
	float c = sqrLength(oc) - s.r2;
	float discriminant = half_b * half_b - c;
	if (discriminant < 0) return false;
	float sqrtd = sqrtf(discriminant);
	float root = -half_b - sqrtd;
	if (root < 0 || ray.t < root) {
		root = -half_b + sqrtd;
		if (root < 0 || ray.t < root) return false;
	}
	tOut = root;
	return true;
}

// Plane::Intersect / IntersectP (intersectable.h:123-150)
bool PlaneTest(const agpt_plane& p, const Ray& ray, float& tOut) {
	if (ray.D.y == 0) return false;
	float t = (p.o[1] - ray.O.y) / ray.D.y;
	if (t <= 0 || t >= ray.t) return false;
	V3 P = ray.O + t * ray.D;
	float u = (P.x - p.o[0]) / p.half_x;
	float v = (P.z - p.o[2]) / p.half_z;
	if (fabsf(u) <= 1 && fabs(v) <= 1) { tOut = t; return true; }
	return false;
}

// Scene::Intersect (scene.h:5-13)
bool SceneIntersect(const OScene& sc, Ray& ray, Hit& hit, Counters& c) {
	bool found = false;
	c.raysClosest++;
	for (size_t p = 0; p < sc.prims.size(); p++) {
		const agpt_prim& pr = sc.prims[p];
		float t;
		if (pr.type == AGPT_PRIM_SPHERE) {
			c.analytic++;
			if (SphereTest(sc.spheres[pr.payload], ray, t)) { ray.t = t; hit = Hit(); hit.t = t; hit.prim = (int)p; found = true; }
		}
		else if (pr.type == AGPT_PRIM_PLANE) {
			c.analytic++;
			if (PlaneTest(sc.planes[pr.payload], ray, t)) { ray.t = t; hit = Hit(); hit.t = t; hit.prim = (int)p; found = true; }
		}
		else if (pr.type == AGPT_PRIM_INSTANCE) {
			// extension: the same two mesh entry points on the object-space ray; t is shared
			const agpt_instance& in = sc.instances[pr.payload];
			const Mesh& m = sc.meshes[in.mesh];
			Ray local(Ray::AsGiven(), XformPoint(in.world_to_object, ray.O), XformVector(in.world_to_object, ray.D), ray.t);
			bool any = false;
			if (m.nodes.empty()) {
				for (size_t j = 0; j < m.ids.size(); j++) {
					c.tris++;
					float b1, b2;
					if (TriangleTest(m, (int)j, local, false, t, b1, b2)) { local.t = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = (int)p; hit.slot = (int)j; any = true; }
				}
			}
			else {
				float dist;
				c.boxes++;
				if (BoundsIntersect(m.nodes[0], local, dist) && RecursiveHit(m, (int)p, m.nodes[0], local, hit, c)) any = true;
			}
			if (any) { ray.t = local.t; found = true; }
		}
		else {
			const Mesh& m = sc.meshes[pr.payload];
			if (m.nodes.empty()) {                                                        // TriangleMesh::Intersect (trianglemesh.h:25-35)
				for (size_t j = 0; j < m.ids.size(); j++) {
					c.tris++;
					float b1, b2;
					if (TriangleTest(m, (int)j, ray, false, t, b1, b2)) { ray.t = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = (int)p; hit.slot = (int)j; found = true; }
				}
			}
			else {                                                                        // BVHTriMesh::Intersect (bvhtrimesh.h:185-191)
				float dist;
				c.boxes++;
				if (!BoundsIntersect(m.nodes[0], ray, dist)) continue;
				if (RecursiveHit(m, (int)p, m.nodes[0], ray, hit, c)) found = true;
			}
		}
	}
	return found;
}

// Scene::IntersectP (scene.h:15-19)
bool SceneIntersectP(const OScene& sc, const Ray& ray, Counters& c) {
	c.raysAny++;
	for (size_t p = 0; p < sc.prims.size(); p++) {
		const agpt_prim& pr = sc.prims[p];
		float t;
		if (pr.type == AGPT_PRIM_SPHERE) { c.analytic++; if (SphereTest(sc.spheres[pr.payload], ray, t)) return true; }
		else if (pr.type == AGPT_PRIM_PLANE) { c.analytic++; if (PlaneTest(sc.planes[pr.payload], ray, t)) return true; }
		else {
			const bool inst = pr.type == AGPT_PRIM_INSTANCE;
			const Mesh& m = sc.meshes[inst ? sc.instances[pr.payload].mesh : pr.payload];
			const Ray local = inst ? Ray(Ray::AsGiven(), XformPoint(sc.instances[pr.payload].world_to_object, ray.O), XformVector(sc.instances[pr.payload].world_to_object, ray.D), ray.t) : ray;
			if (m.nodes.empty()) {
				for (size_t j = 0; j < m.ids.size(); j++) { c.tris++; float b1, b2; if (TriangleTest(m, (int)j, local, true, t, b1, b2)) return true; }
			}
			else {
				float dist;
				c.boxes++;
				if (BoundsIntersect(m.nodes[0], local, dist) && RecursiveHitP(m, m.nodes[0], local, c)) return true;
			}
		}
	}
	return false;
}

// ---- SurfaceInteraction (intersectable.h:63-115) ------------------------------------------
struct Surface {
	V3 p, n, sn, sdpdu;          // point, geometric n, shading.n, shading.dpdu
	void Init(V3 pp, V3 dpdu, V3 dpdv) { p = pp; n = normalize(cross(dpdu, dpdv)); sn = n; sdpdu = dpdu; }
};

void BuildSurface(const OScene& sc, const Ray& ray, const Hit& h, Surface& s) {
	const agpt_prim& pr = sc.prims[h.prim];
	if (pr.type == AGPT_PRIM_SPHERE) {                                                    // intersectable.h:183-204
		const agpt_sphere& sp = sc.spheres[pr.payload];
		V3 p = ray.O + h.t * ray.D;
		V3 pHit = p - v3(sp.center);
		if (pHit.x == 0 && pHit.y == 0) pHit.x = kEps * sp.r;
		float theta = std::acos(tclamp(pHit.z / sp.r, -1.f, 1.f));
		float zRadius = std::sqrt(pHit.x * pHit.x + pHit.y * pHit.y);
		float invZRadius = 1 / zRadius;
		float cosPhi = pHit.x * invZRadius, sinPhi = pHit.y * invZRadius;
		V3 dpdu = v3(-kTwoPi * pHit.y, kTwoPi * pHit.x, 0);
		V3 dpdv = kPi * v3(pHit.z * cosPhi, pHit.z * sinPhi, -sp.r * std::sin(theta));
		s.Init(p, dpdv, dpdu);                                                            // swapped upstream (:200-201)
	}
	else if (pr.type == AGPT_PRIM_PLANE) s.Init(ray.O + h.t * ray.D, v3(0, 0, 1), v3(1, 0, 0));   // :128-133
	else {                                                                                // trianglemesh.cpp:45-113
		const agpt_instance* in = pr.type == AGPT_PRIM_INSTANCE ? &sc.instances[pr.payload] : nullptr;
		const Mesh& m = sc.meshes[in ? in->mesh : pr.payload];
		const float* p = &m.verts[12 * (size_t)h.slot];
		V3 v0 = v3(p), v1 = v3(p + 4), v2 = v3(p + 8);
		if (in) { v0 = XformPoint(in->object_to_world, v0); v1 = XformPoint(in->object_to_world, v1); v2 = XformPoint(in->object_to_world, v2); }   // extension
		float b0 = 1.f - h.b1 - h.b2;
		float uv[6];
		TriangleUVs(m, h.slot, uv);
		V3 dpdu = v3(0.f), dpdv = v3(0.f);
		TriangleDerivatives(v0, v1, v2, uv, dpdu, dpdv);
		s.Init(ray.O + h.t * ray.D, dpdu, dpdv);
		if (!m.normals.empty()) {
			const float* q = &m.normals[12 * (size_t)h.slot];
			V3 ns = v3(q) * b0 + v3(q + 4) * h.b1 + v3(q + 8) * h.b2;
			if (in) ns = XformNormal(in->world_to_object, ns);                                // extension
			if (sqrLength(ns) > 0.f) ns = normalize(ns);
			else ns = s.n;
			V3 ss = normalize(dpdu);
			V3 ts = cross(ss, ns);
			if (sqrLength(ts) > 0.f) { ts = normalize(ts); ss = cross(ts, ns); }
			else CoordinateSystem(ns, &ss, &ts);
			s.sn = normalize(cross(ss, ts));                                              // SetShadingGeometry (intersectable.h:80-89)
			s.n = Faceforward(s.n, s.sn);
		}
	}
}

// ---- BSDF (reflection.h, disney.h, microfacet.h) ------------------------------------------
inline float CosTheta(V3 w) { return w.z; }
inline float Cos2Theta(V3 w) { return w.z * w.z; }
inline float AbsCosTheta(V3 w) { return std::abs(w.z); }
inline float Sin2Theta(V3 w) { return std::max(0.f, 1.f - Cos2Theta(w)); }
inline float SinTheta(V3 w) { return std::sqrt(Sin2Theta(w)); }
inline float TanTheta(V3 w) { return SinTheta(w) / CosTheta(w); }
inline float Tan2Theta(V3 w) { return Sin2Theta(w) / Cos2Theta(w); }
inline float CosPhi(V3 w) { float s = SinTheta(w); return (s == 0) ? 1 : tclamp(w.x / s, -1.f, 1.f); }
inline float SinPhi(V3 w) { float s = SinTheta(w); return (s == 0) ? 0 : tclamp(w.y / s, -1.f, 1.f); }
inline float Cos2Phi(V3 w) { return CosPhi(w) * CosPhi(w); }
inline float Sin2Phi(V3 w) { return SinPhi(w) * SinPhi(w); }
inline bool SameHemisphere(V3 w, V3 wp) { return w.z * wp.z > 0; }

float FrDielectric(float cosThetaI, float etaI, float etaT) {                             // microfacet.h:180-201
	cosThetaI = tclamp(cosThetaI, -1.f, 1.f);
	bool entering = cosThetaI > 0.f;
	if (!entering) { std::swap(etaI, etaT); cosThetaI = std::abs(cosThetaI); }
	float sinThetaI = std::sqrt(std::max(0.f, 1.f - cosThetaI * cosThetaI));
	float sinThetaT = etaI / etaT * sinThetaI;
	if (sinThetaT >= 1) return 1;
	float cosThetaT = std::sqrt(std::max(0.f, 1.f - sinThetaT * sinThetaT));
	float Rparl = ((etaT * cosThetaI) - (etaI * cosThetaT)) / ((etaT * cosThetaI) + (etaI * cosThetaT));
	float Rperp = ((etaI * cosThetaI) - (etaT * cosThetaT)) / ((etaI * cosThetaI) + (etaT * cosThetaT));
	return (Rparl * Rparl + Rperp * Rperp) / 2;
}
inline float SchlickWeight(float cosTheta) { float m = tclamp(1 - cosTheta, 0.f, 1.f); return (m * m) * (m * m) * m; }   // disney.h:12-15
inline V3 FrSchlick(V3 R0, float cosTheta) { return Lerp(SchlickWeight(cosTheta), R0, v3(1.f)); }                       // disney.h:17-19
inline V3 DisneyFresnel(const agpt_material& m, float cosI) {                                                           // disney.h:62-71
	return Lerp(m.metallic, v3(FrDielectric(cosI, 1, m.eta)), FrSchlick(v3(m.spec_r0), cosI));
}
float TR_D(const agpt_material& m, V3 wh) {                                               // microfacet.h:124-132
	float tan2Theta = Tan2Theta(wh);
	if (std::isinf(tan2Theta)) return 0.;
	const float cos4Theta = Cos2Theta(wh) * Cos2Theta(wh);
	float e = (Cos2Phi(wh) / (m.alpha_x * m.alpha_x) + Sin2Phi(wh) / (m.alpha_y * m.alpha_y)) * tan2Theta;
	return 1 / (kPi * m.alpha_x * m.alpha_y * cos4Theta * (1 + e) * (1 + e));
}
float TR_Lambda(const agpt_material& m, V3 w) {                                           // microfacet.h:142-149
	float absTanTheta = std::abs(TanTheta(w));
	if (std::isinf(absTanTheta)) return 0.f;
	float alpha = std::sqrt(Cos2Phi(w) * m.alpha_x * m.alpha_x + Sin2Phi(w) * m.alpha_y * m.alpha_y);
	float alpha2Tan2Theta = (alpha * absTanTheta) * (alpha * absTanTheta);
	return (-1 + std::sqrt(1.f + alpha2Tan2Theta)) / 2;
}
inline float TR_G1(const agpt_material& m, V3 w) { return 1 / (1 + TR_Lambda(m, w)); }   // microfacet.h:100-102
inline float TR_Pdf(const agpt_material& m, V3 wo, V3 wh) { return TR_D(m, wh) * TR_G1(m, wo) * absdot(wo, wh) / AbsCosTheta(wo); }   // :107-109

void TrowbridgeReitzSample11(float cosTheta, float U1, float U2, float* slope_x, float* slope_y) {   // microfacet.h:34-73
	if (cosTheta > .9999f) {
		float r = std::sqrt(U1 / (1 - U1));
		float phi = 6.28318530718f * U2;
		*slope_x = r * std::cos(phi);
		*slope_y = r * std::sin(phi);
		return;
	}
	float sinTheta = std::sqrt(std::max(0.f, 1.f - cosTheta * cosTheta));
	float tanTheta = sinTheta / cosTheta;
	float a = 1 / tanTheta;
	float G1 = 2 / (1 + std::sqrt(1.f + 1.f / (a * a)));
	float A = 2 * U1 / G1 - 1;
	float tmp = 1.f / (A * A - 1.f);
	if (tmp > 1e10) tmp = 1e10;
	float B = tanTheta;
	float D = std::sqrt(std::max(float(B * B * tmp * tmp - (A * A - B * B) * tmp), 0.f));
	float slope_x_1 = B * tmp - D;
	float slope_x_2 = B * tmp + D;
	*slope_x = (A < 0 || slope_x_2 > 1.f / tanTheta) ? slope_x_1 : slope_x_2;
	float S;
	if (U2 > 0.5f) { S = 1.f; U2 = 2.f * (U2 - .5f); }
	else { S = -1.f; U2 = 2.f * (.5f - U2); }
	float z = (U2 * (U2 * (U2 * 0.27385f - 0.73369f) + 0.46341f)) / (U2 * (U2 * (U2 * 0.093073f + 0.309420f) - 1.000000f) + 0.597999f);
	*slope_y = S * z * std::sqrt(1.f + *slope_x * *slope_x);
}
V3 TR_Sample_wh(const agpt_material& m, V3 wo, float u0, float u1) {                      // microfacet.h:75-94,134-140
	bool flip = wo.z < 0;
	V3 wi = flip ? -wo : wo;
	V3 wiS = normalize(v3(m.alpha_x * wi.x, m.alpha_y * wi.y, wi.z));
	float sx, sy;
	TrowbridgeReitzSample11(CosTheta(wiS), u0, u1, &sx, &sy);
	float tmp = CosPhi(wiS) * sx - SinPhi(wiS) * sy;
	sy = SinPhi(wiS) * sx + CosPhi(wiS) * sy;
	sx = tmp;
	sx = m.alpha_x * sx;
	sy = m.alpha_y * sy;
	V3 wh = normalize(v3(-sx, -sy, 1.));
	if (flip) wh = -wh;
	return wh;
}

// ---- EXTENSION: rough dielectric (agpt.h AGPT_LOBE_GLASS_*) ---------------------------------
inline float TR_G(const agpt_material& m, V3 wo, V3 wi) { return 1 / (1 + TR_Lambda(m, wo) + TR_Lambda(m, wi)); }     // microfacet.h:103-105
// PBRT-v3 Refract(wi, n, eta, wt): false on total internal reflection
inline bool Refract(V3 wi, V3 n, float eta, V3* wt) {
	float cosThetaI = dot(n, wi);
	float sin2ThetaI = std::max(0.f, 1.f - cosThetaI * cosThetaI);
	float sin2ThetaT = eta * eta * sin2ThetaI;
	if (sin2ThetaT >= 1) return false;
	float cosThetaT = std::sqrt(1 - sin2ThetaT);
	*wt = eta * -wi + (eta * cosThetaI - cosThetaT) * n;
	return true;
}
// MicrofacetTransmission::f / Pdf (PBRT-v3 reflection.cpp), etaA = 1 outside, etaB = m.eta inside, TransportMode::Radiance
V3 GlassT_f(const agpt_material& m, V3 wo, V3 wi) {
	if (SameHemisphere(wo, wi)) return v3(0.f);
	float cosThetaO = CosTheta(wo), cosThetaI = CosTheta(wi);
	if (cosThetaI == 0 || cosThetaO == 0) return v3(0.f);
	float eta = CosTheta(wo) > 0 ? (m.eta / 1.f) : (1.f / m.eta);
	V3 wh = normalize(wo + wi * eta);
	if (wh.z < 0) wh = -wh;
	if (dot(wo, wh) * dot(wi, wh) > 0) return v3(0.f);
	float F = FrDielectric(dot(wo, wh), 1.f, m.eta);
	float sqrtDenom = dot(wo, wh) + eta * dot(wi, wh);
	float factor = 1 / eta;
	return (v3(1.f) - v3(F)) * v3(m.diffuse_r) *
		std::abs(TR_D(m, wh) * TR_G(m, wo, wi) * eta * eta * absdot(wi, wh) * absdot(wo, wh) * factor * factor / (cosThetaI * cosThetaO * sqrtDenom * sqrtDenom));
}
float GlassT_Pdf(const agpt_material& m, V3 wo, V3 wi) {
	if (SameHemisphere(wo, wi)) return 0;
	float eta = CosTheta(wo) > 0 ? (m.eta / 1.f) : (1.f / m.eta);
	V3 wh = normalize(wo + wi * eta);
	if (dot(wo, wh) * dot(wi, wh) > 0) return 0;
	float sqrtDenom = dot(wo, wh) + eta * dot(wi, wh);
	float dwh_dwi = std::abs((eta * eta * dot(wi, wh)) / (sqrtDenom * sqrtDenom));
	return TR_Pdf(m, wo, wh) * dwh_dwi;
}

V3 Lobe_f(const agpt_material& m, int lobe, V3 wo, V3 wi) {
	if (lobe == AGPT_LOBE_GLASS_TRANSMIT) return GlassT_f(m, wo, wi);
	if (lobe == AGPT_LOBE_GLASS_REFLECT) {                                                // reflection.h:42-54 with FresnelDielectric and the base-class G
		float cosThetaO = AbsCosTheta(wo), cosThetaI = AbsCosTheta(wi);
		V3 wh = wi + wo;
		if (cosThetaI == 0 || cosThetaO == 0) return v3(0.f);
		if (wh.x == 0 && wh.y == 0 && wh.z == 0) return v3(0.f);
		wh = normalize(wh);
		V3 F = v3(FrDielectric(dot(wi, Faceforward(wh, v3(0, 0, 1))), 1.f, m.eta));
		return v3(m.mirror_r) * TR_D(m, wh) * TR_G(m, wo, wi) * F / (4 * cosThetaI * cosThetaO);
	}
	if (lobe == AGPT_LOBE_DIFFUSE) {                                                      // disney.h:27-34
		float Fo = SchlickWeight(AbsCosTheta(wo)), Fi = SchlickWeight(AbsCosTheta(wi));
		return v3(m.diffuse_r) * kInvPi * (1 - Fo / 2) * (1 - Fi / 2);
	}
	if (lobe == AGPT_LOBE_RETRO) {                                                        // disney.h:42-54
		V3 wh = wi + wo;
		if (wh.x == 0 && wh.y == 0 && wh.z == 0) return v3(0.f);
		wh = normalize(wh);
		float cosThetaD = dot(wi, wh);
		float Fo = SchlickWeight(AbsCosTheta(wo)), Fi = SchlickWeight(AbsCosTheta(wi));
		float Rr = 2 * m.roughness * cosThetaD * cosThetaD;
		return v3(m.diffuse_r) * kInvPi * Rr * (Fo + Fi + Fo * Fi * (Rr - 1));
	}
	if (lobe == AGPT_LOBE_MICROFACET) {                                                   // reflection.h:42-54
		float cosThetaO = AbsCosTheta(wo), cosThetaI = AbsCosTheta(wi);
		V3 wh = wi + wo;
		if (cosThetaI == 0 || cosThetaO == 0) return v3(0.f);
		if (wh.x == 0 && wh.y == 0 && wh.z == 0) return v3(0.f);
		wh = normalize(wh);
		V3 F = DisneyFresnel(m, dot(wi, Faceforward(wh, v3(0, 0, 1))));
		float G = TR_G1(m, wo) * TR_G1(m, wi);                                            // disney.h:77-80
		return v3(1.f) * TR_D(m, wh) * G * F / (4 * cosThetaI * cosThetaO);
	}
	return v3(0.f);                                                                       // SpecularReflection::f (reflection.h:26-28)
}
float Lobe_Pdf(const agpt_material& m, int lobe, V3 wo, V3 wi) {
	if (lobe == AGPT_LOBE_DIFFUSE || lobe == AGPT_LOBE_RETRO) return SameHemisphere(wo, wi) ? AbsCosTheta(wi) * kInvPi : 0;   // reflection.h:16-18
	if (lobe == AGPT_LOBE_GLASS_TRANSMIT) return GlassT_Pdf(m, wo, wi);
	if (lobe == AGPT_LOBE_MICROFACET || lobe == AGPT_LOBE_GLASS_REFLECT) {                // reflection.h:67-71
		if (!SameHemisphere(wo, wi)) return 0;
		V3 wh = normalize(wo + wi);
		return TR_Pdf(m, wo, wh) / (4 * dot(wo, wh));
	}
	return 0;
}

struct Bsdf {                                                                             // reflection.h:83-201, reflection.cpp:6-11
	V3 ng, ns, ss, ts;
	const agpt_material* m;
	int lobes[4];
	int nAll;            // every BxDF, in bxdfs[] order
	Bsdf(const Surface& s, const agpt_material* mat) : ng(s.n), ns(s.sn), ss(normalize(s.sdpdu)), ts(cross(ns, ss)), m(mat) {
		nAll = 0;
		if (m->lobes & AGPT_LOBE_DIFFUSE) lobes[nAll++] = AGPT_LOBE_DIFFUSE;
		if (m->lobes & AGPT_LOBE_RETRO) lobes[nAll++] = AGPT_LOBE_RETRO;
		if (m->lobes & AGPT_LOBE_MICROFACET) lobes[nAll++] = AGPT_LOBE_MICROFACET;
		if (m->lobes & AGPT_LOBE_SPECULAR) lobes[nAll++] = AGPT_LOBE_SPECULAR;
		if (m->lobes & AGPT_LOBE_GLASS_REFLECT) lobes[nAll++] = AGPT_LOBE_GLASS_REFLECT;      // extension
		if (m->lobes & AGPT_LOBE_GLASS_TRANSMIT) lobes[nAll++] = AGPT_LOBE_GLASS_TRANSMIT;
	}
	// which lobes BSDF::f sums for a pair of directions: reflection lobes when wi, wo lie on the same side of the geometric
	// normal (reflection.h:118-121); a transmission lobe -- extension -- when they lie on opposite sides (PBRT-v3 BSDF::f)
	static bool Contributes(int lobe, bool reflect) { return lobe == AGPT_LOBE_GLASS_TRANSMIT ? !reflect : reflect; }
	static bool Matches(int lobe, bool skipSpecular) { return !skipSpecular || lobe != AGPT_LOBE_SPECULAR; }
	bool IsPerfectlySpecular() const { for (int i = 0; i < nAll; i++) if (lobes[i] != AGPT_LOBE_SPECULAR) return false; return true; }
	V3 ToLocal(V3 v) const { return v3(dot(v, ss), dot(v, ts), dot(v, ns)); }
	V3 ToWorld(V3 v) const {
		return v3(ss.x * v.x + ts.x * v.y + ns.x * v.z, ss.y * v.x + ts.y * v.y + ns.y * v.z, ss.z * v.x + ts.z * v.y + ns.z * v.z);
	}
	V3 f(V3 woW, V3 wiW, bool skipSpecular) const {
		V3 wi = ToLocal(wiW), wo = ToLocal(woW);
		if (wo.z == 0) return v3(0.f);
		bool reflect = dot(wiW, ng) * dot(woW, ng) > 0;
		V3 r = v3(0.f);
		for (int i = 0; i < nAll; i++)
			if (Matches(lobes[i], skipSpecular) && Contributes(lobes[i], reflect)) r += Lobe_f(*m, lobes[i], wo, wi);
		return r;
	}
	float Pdf(V3 woW, V3 wiW, bool skipSpecular) const {
		if (nAll == 0) return 0.f;
		V3 wo = ToLocal(woW), wi = ToLocal(wiW);
		if (wo.z == 0) return 0.f;
		float pdf = 0.f;
		int matching = 0;
		for (int i = 0; i < nAll; i++)
			if (Matches(lobes[i], skipSpecular)) { ++matching; pdf += Lobe_Pdf(*m, lobes[i], wo, wi); }
		return matching > 0 ? pdf / matching : 0.f;
	}
	V3 Sample_f(V3 woW, V3* wiW, float u0, float u1, float* pdf, bool skipSpecular, bool* sampledSpecular) const {
		int matching = 0;
		for (int i = 0; i < nAll; i++) if (Matches(lobes[i], skipSpecular)) matching++;
		if (matching == 0) { *pdf = 0; return v3(0.f); }
		int comp = std::min((int)std::floor(u0 * matching), matching - 1);
		int lobe = -1, count = comp;
		for (int i = 0; i < nAll; i++)
			if (Matches(lobes[i], skipSpecular) && count-- == 0) { lobe = lobes[i]; break; }
		float ur0 = std::min(u0 * matching - comp, kOneMinusEps), ur1 = u1;
		V3 wi = v3(0.f), wo = ToLocal(woW);
		if (wo.z == 0) return v3(0.f);
		*pdf = 0;
		bool specular = lobe == AGPT_LOBE_SPECULAR;
		if (sampledSpecular) *sampledSpecular = specular;
		V3 f = v3(0.f);
		if (specular) {                                                                   // reflection.cpp:13-17
			wi = v3(-wo.x, -wo.y, wo.z);
			*pdf = 1;
			f = v3(1.f) * v3(m->mirror_r) / AbsCosTheta(wi);
		}
		else if (lobe == AGPT_LOBE_MICROFACET || lobe == AGPT_LOBE_GLASS_REFLECT) {       // reflection.h:55-66
			V3 wh = TR_Sample_wh(*m, wo, ur0, ur1);
			if (!(dot(wo, wh) < 0)) {
				wi = Reflect(wo, wh);
				if (SameHemisphere(wo, wi)) *pdf = TR_Pdf(*m, wo, wh) / (4 * dot(wo, wh));
			}
		}
		else if (lobe == AGPT_LOBE_GLASS_TRANSMIT) {                                      // MicrofacetTransmission::Sample_f (PBRT-v3)
			V3 wh = TR_Sample_wh(*m, wo, ur0, ur1);
			if (!(dot(wo, wh) < 0)) {
				float eta = CosTheta(wo) > 0 ? (1.f / m->eta) : (m->eta / 1.f);
				if (Refract(wo, wh, eta, &wi)) *pdf = GlassT_Pdf(*m, wo, wi);
			}
		}
		else {                                                                            // reflection.h:8-15, common.h:118-143
			float ox = 2.f * ur0 - 1, oy = 2.f * ur1 - 1;
			float dx = 0, dy = 0;
			if (!(ox == 0 && oy == 0)) {
				float theta, r;
				if (std::abs(ox) > std::abs(oy)) { r = ox; theta = (kPi / 4) * (oy / ox); }
				else { r = oy; theta = (kPi / 2) - (kPi / 4) * (ox / oy); }
				dx = r * std::cos(theta); dy = r * std::sin(theta);
			}
			float z = std::sqrt(std::max(0.f, 1 - dx * dx - dy * dy));
			wi = v3(dx, dy, z);
			if (wo.z < 0) wi.z *= -1;
			*pdf = SameHemisphere(wo, wi) ? AbsCosTheta(wi) * kInvPi : 0;
		}
		if (*pdf == 0) return v3(0.f);
		*wiW = ToWorld(wi);
		if (!specular && matching > 1)
			for (int i = 0; i < nAll; i++)
				if (lobes[i] != lobe && Matches(lobes[i], skipSpecular)) *pdf += Lobe_Pdf(*m, lobes[i], wo, wi);
		if (matching > 1) *pdf /= matching;
		if (!specular) {
			bool reflect = dot(*wiW, ng) * dot(woW, ng) > 0;
			f = v3(0.f);
			for (int i = 0; i < nAll; i++)
				if (Matches(lobes[i], skipSpecular) && Contributes(lobes[i], reflect)) f += Lobe_f(*m, lobes[i], wo, wi);
		}
		return f;
	}
};

// ---- sphere light sampling (intersectable.h:230-317) --------------------------------------
void SphereSample(const agpt_sphere& sp, V3 refP, float u0, float u1, V3* pOut, V3* nOut, float* pdf) {
	V3 pCenter = v3(sp.center);
	if (sqrLength(refP - pCenter) <= sp.r2) {
		float a = 1 - 2 * u0;                                                             // common.h:84-89
		float b = std::sqrt(1 - a * a);
		float phi = 2 * kPi * u1;
		V3 pObj = pCenter + sp.r * v3(b * std::cos(phi), b * std::sin(phi), a);
		V3 n = normalize(pObj);                                                           // :233 (normalises the world position)
		*pdf = 1 / (4.f * kPi * sp.r2);
		V3 wi = pObj - refP;
		if (sqrLength(wi) == 0) *pdf = 0;
		else { wi = normalize(wi); *pdf *= sqrLength(refP - pObj) / absdot(n, -wi); }
		if (std::isinf(*pdf)) *pdf = 0;
		*pOut = pObj; *nOut = n;
		return;
	}
	float dc = length(refP - pCenter);
	float invDc = 1 / dc;
	V3 wc = (pCenter - refP) * invDc;
	V3 wcX, wcY;
	CoordinateSystem(wc, &wcX, &wcY);
	float sinThetaMax = sp.r * invDc;
	float sinThetaMax2 = sinThetaMax * sinThetaMax;
	float invSinThetaMax = 1 / sinThetaMax;
	float cosThetaMax = std::sqrt(std::max(0.f, 1 - sinThetaMax2));
	float cosTheta = (cosThetaMax - 1) * u0 + 1;
	float sinTheta2 = 1 - cosTheta * cosTheta;
	if (sinThetaMax2 < 0.00068523f) { sinTheta2 = sinThetaMax2 * u0; cosTheta = std::sqrt(1 - sinTheta2); }
	float cosAlpha = sinTheta2 * invSinThetaMax + cosTheta * std::sqrt(std::max(0.f, 1.f - sinTheta2 * invSinThetaMax * invSinThetaMax));
	float sinAlpha = std::sqrt(std::max(0.f, 1.f - cosAlpha * cosAlpha));
	float phi = u1 * 2 * kPi;
	V3 x = -wcX, y = -wcY, z = -wc;
	V3 nWorld = sinAlpha * std::cos(phi) * x + sinAlpha * std::sin(phi) * y + cosAlpha * z;   // common.h:153-156
	*pOut = pCenter + sp.r * v3(nWorld.x, nWorld.y, nWorld.z);
	*nOut = nWorld;
	*pdf = 1 / (2 * kPi * (1 - cosThetaMax));
}
float SpherePdf(const agpt_sphere& sp, V3 refP) {                                         // intersectable.h:306-317
	V3 pCenter = v3(sp.center);
	if (sqrLength(refP - pCenter) <= sp.r2) return 1 / (4 * kPi);
	float sinThetaMax2 = sp.r2 / sqrLength(refP - pCenter);
	float cosThetaMax = std::sqrt(std::max(0.f, 1 - sinThetaMax2));
	return 1 / (2 * kPi * (1 - cosThetaMax));
}

// ---- InfiniteAreaLight (lights.cpp:50-112, ILS), HDRTexture::value (texture.h:59-81), Distribution1D (sampling.h)
inline float SphericalTheta(V3 v) { return std::acos(tclamp(v.z, -1.f, 1.f)); }                        // common.h:158-160
inline float SphericalPhi(V3 v) { float p = std::atan2(v.y, v.x); return (p < 0) ? (p + kTwoPi) : p; }   // common.h:162-165
inline int EnvMod(int a, int b) { int r = a - (a / b) * b; return (r < 0) ? r + b : r; }
V3 EnvLe(const OScene& sc, V3 rayD) {
	V3 w = normalize(rayD);
	w = v3(w.x, w.z, w.y);
	float u = SphericalPhi(w) * kInv2Pi, v = SphericalTheta(w) * kInvPi;
	int s = (int)std::floor(u * sc.envW - .5f);
	int t = (int)std::floor(v * sc.envH - .5f);
	int x = EnvMod(s, sc.envW), y = EnvMod(t, sc.envH);
	return v3(&sc.envRgb[3 * ((size_t)y * sc.envW + x)]);
}
float EnvPdfLi(const OScene& sc, V3 wi) {
	V3 w = normalize(wi);
	w = v3(w.x, w.z, w.y);
	float theta = SphericalTheta(w), phi = SphericalPhi(w);
	float sinTheta = std::sin(theta);
	if (sinTheta == 0) return 0;
	int x = std::min(std::max(int(phi * kInv2Pi * sc.envW), 0), sc.envW - 1);
	int y = std::min(std::max(int(theta * kInvPi * sc.envH), 0), sc.envH - 1);
	int count = sc.envW * sc.envH;
	float discrete = sc.envFunc[y * sc.envW + x] / (sc.envFuncInt * count);
	return count * discrete / (2 * kPi * kPi * sinTheta);
}
bool EnvSampleLi(const OScene& sc, float u, V3* wi, float* pdf) {
	const int n = sc.envW * sc.envH;
	int first = 0, len = n + 1;                                                           // FindInterval (sampling.h:4-18)
	while (len > 0) {
		int half = len >> 1, middle = first + half;
		if (sc.envCdf[middle] <= u) { first = middle + 1; len -= half + 1; }
		else len = half;
	}
	int offset = std::min(std::max(first - 1, 0), n + 1 - 2);
	float du = u - sc.envCdf[offset];
	if ((sc.envCdf[offset + 1] - sc.envCdf[offset]) > 0) du /= sc.envCdf[offset + 1] - sc.envCdf[offset];
	float mapPdf = (sc.envFuncInt > 0) ? sc.envFunc[offset] / sc.envFuncInt : 0;
	float sample = (offset + du) / n;
	if (mapPdf == 0) return false;
	int idx = int(sample * n);
	float uvx = ((idx % sc.envW) + .5f) / sc.envW, uvy = ((idx / sc.envW) + .5f) / sc.envH;
	float theta = uvy * kPi, phi = uvx * kTwoPi;
	float cosTheta = std::cos(theta), sinTheta = std::sin(theta);
	float sinPhi = std::sin(phi), cosPhi = std::cos(phi);
	*wi = v3(sinTheta * cosPhi, cosTheta, sinTheta * sinPhi);
	*pdf = mapPdf / (2 * kPi * kPi * sinTheta);
	if (sinTheta == 0) *pdf = 0;
	return true;
}

inline float PowerHeuristic(int nf, float fPdf, int ng, float gPdf) { float f = nf * fPdf, g = ng * gPdf; return (f * f) / (f * f + g * g); }   // integrator.h:33-36

// EstimateDirect (integrator.h:38-93)
V3 EstimateDirect(const OScene& sc, const Surface& si, const Bsdf& bsdf, V3 wo, float uScatX, float uScatY, int lightIdx,
		float uLightX, float uLightY, Rng& rng, Counters& c) {
	const agpt_light& light = sc.lights[lightIdx];
	V3 lemit = v3(light.lemit);
	V3 Ld = v3(0.f), wi = v3(0.f);
	float lightPdf = 0, scatteringPdf = 0;
	V3 Li = v3(0.f);
	Ray vis(v3(0.f), v3(1.f, 0.f, 0.f));
	if (light.type == AGPT_LIGHT_AREA) {                                                  // lights.cpp:115-126
		const agpt_prim& lp = sc.prims[light.prim];
		if (lp.type == AGPT_PRIM_SPHERE) {
			V3 pS, nS;
			SphereSample(sc.spheres[lp.payload], si.p, uLightX, uLightY, &pS, &nS, &lightPdf);
			if (lightPdf == 0 || sqrLength(pS - si.p) == 0) lightPdf = 0;
			else {
				wi = pS - si.p;
				float dist = length(wi);
				wi /= dist;
				vis = Ray(si.p + kEps * wi, wi, dist - 10 * kEps);
				Li = lemit;
			}
		}
	}
	else if (light.type == AGPT_LIGHT_INFINITE_AREA) {                                    // lights.cpp:50-90
		float u01 = rng.Float();
		if (EnvSampleLi(sc, u01, &wi, &lightPdf)) {
			vis = Ray(si.p + kEps * si.n, wi);
			Li = EnvLe(sc, vis.D);
		}
	}
	else {                                                                                // lights.cpp:15-24, common.h:73-97
		float a = 1 - 2 * rng.Float();
		float b = std::sqrt(1 - a * a);
		float phi = 2 * kPi * rng.Float();
		V3 v = v3(1.f * b * std::cos(phi), 1.f * b * std::sin(phi), 1.f * a);
		if (dot(v, si.sn) < 0) v = -v;
		wi = v;
		lightPdf = kInv2Pi;
		vis = Ray(si.p + kEps * wi, wi);
		Li = lemit;
	}
	if (lightPdf > 0 && !IsBlack(Li)) {
		V3 f = bsdf.f(wo, wi, true) * absdot(wi, si.sn);
		scatteringPdf = bsdf.Pdf(wo, wi, true);
		if (!IsBlack(f)) {
			if (SceneIntersectP(sc, vis, c)) Li = v3(0.f);
			if (!IsBlack(Li)) {
				float weight = PowerHeuristic(1, lightPdf, 1, scatteringPdf);
				Ld += f * Li * weight / lightPdf;
			}
		}
	}
	{
		V3 f = bsdf.Sample_f(wo, &wi, uScatX, uScatY, &scatteringPdf, true, nullptr);
		f *= v3(absdot(wi, si.sn));
		if (!IsBlack(f) && scatteringPdf > 0) {
			float lp;
			if (light.type == AGPT_LIGHT_AREA) {
				const agpt_prim& lpr = sc.prims[light.prim];
				lp = lpr.type == AGPT_PRIM_SPHERE ? SpherePdf(sc.spheres[lpr.payload], si.p) : 0.f;
			}
			else if (light.type == AGPT_LIGHT_INFINITE_AREA) lp = EnvPdfLi(sc, wi);
			else lp = dot(si.n, wi) > 0 ? kInv2Pi : 0.f;                                  // lights.cpp:26-28
			if (lp == 0) return Ld;
			float weight = PowerHeuristic(1, scatteringPdf, 1, lp);
			Ray ray(si.p + kEps * wi, wi);
			Hit h;
			bool found = SceneIntersect(sc, ray, h, c);
			V3 Lr = v3(0.f);
			if (found) { if (sc.prims[h.prim].area_light == lightIdx) Lr = lemit; }
			else if (light.type == AGPT_LIGHT_UNIFORM_INFINITE) Lr = lemit;
			else if (light.type == AGPT_LIGHT_INFINITE_AREA) Lr = EnvLe(sc, ray.D);
			if (!IsBlack(Lr)) Ld += f * Lr * weight / scatteringPdf;
		}
	}
	return Ld;
}

// PathTracer::Li (integrator.h:124-191)
// sc.rrByBounce (EXTENSION, parity unpinned by the reference: it has no such rule): the roulette is keyed on the
// path's bounce index -- `bounces > 3`, as PBRT states it -- instead of on the constant depth argument.
V3 Li(const OScene& sc, Ray ray, int maxDepth, int depthArg, Rng& rng, Counters& c) {
	V3 beta = v3(1.f), L = v3(0.f);
	bool specularBounce = false;
	for (int bounces = 0;; bounces++) {
		Hit h;
		bool found = SceneIntersect(sc, ray, h, c);
		if (bounces == 0 || specularBounce) {
			if (found) {
				int al = sc.prims[h.prim].area_light;
				L += beta * (al >= 0 ? v3(sc.lights[al].lemit) : v3(0.f));
			}
			else {
				for (auto& l : sc.lights) {
					if (l.type == AGPT_LIGHT_UNIFORM_INFINITE) L += beta * v3(l.lemit);
					else if (l.type == AGPT_LIGHT_INFINITE_AREA) L += beta * EnvLe(sc, ray.D);
				}
			}
		}
		if (!found || bounces >= maxDepth) break;
		Surface si;
		BuildSurface(sc, ray, h, si);
		const agpt_prim& pr = sc.prims[h.prim];
		if (pr.material < 0) {                                                            // :152-161
			ray = Ray(si.p + kEps * ray.D, ray.D);
			bounces--;
			continue;
		}
		Bsdf bsdf(si, &sc.mats[pr.material]);
		V3 wo = -ray.D;
		if (!bsdf.IsPerfectlySpecular() && !sc.lights.empty()) {                          // :165-167, :95-105
			int nLights = (int)sc.lights.size();
			int numLight = std::min((int)(rng.Float() * nLights), nLights - 1);
			float lightPdf = 1.f / nLights;
			float uLy = rng.Float(), uLx = rng.Float();                                   // g++ evaluates float2(a(), b()) right to left
			float uSy = rng.Float(), uSx = rng.Float();
			L += beta * (EstimateDirect(sc, si, bsdf, wo, uSx, uSy, numLight, uLx, uLy, rng, c) / lightPdf);
		}
		float uy = rng.Float(), ux = rng.Float();
		V3 wi = v3(0.f);
		float pdf = 0;
		bool sampledSpecular = false;
		V3 f = bsdf.Sample_f(wo, &wi, ux, uy, &pdf, false, &sampledSpecular);
		if (IsBlack(f) || pdf == 0) break;
		beta *= f * absdot(wi, si.sn) / pdf;
		specularBounce = sampledSpecular;
		float maxComponent = std::max(beta.x, std::max(beta.y, beta.z));
		if (maxComponent < 1 && (sc.rrByBounce ? bounces : depthArg) > 3) {               // :179-185
			float q = std::max(.05f, 1 - maxComponent);
			if (rng.Float() < q) break;
			beta /= 1 - q;
		}
		ray = Ray(si.p + kEps * wi, wi);
	}
	return L;
}

// myapp.cpp:165-167, camera.h:58-64, common.h:65-71
Ray CameraRay(const OScene& sc, int W, int H, int x, int y, Rng& rng) {
	float jy = rng.Float(), jx = rng.Float();
	float px = x + jx, py = y + jy;
	float s = px / W, t = py / H;
	const agpt_camera& cam = sc.cam;
	V3 rd = v3(0.f);
	if (cam.lens_radius > 0.f) {
		while (true) {
			float ry = -1 + (1 - -1) * rng.Float();
			float rx = -1 + (1 - -1) * rng.Float();
			V3 p = v3(rx, ry, 0);
			if (sqrLength(p) >= 1) continue;
			rd = cam.lens_radius * p;
			break;
		}
	}
	V3 offset = v3(cam.u) * rd.x + v3(cam.v) * rd.y;
	V3 pixel = v3(cam.lower_left_corner) + s * v3(cam.horizontal) + t * v3(cam.vertical);
	return Ray(v3(cam.origin) + offset, pixel - v3(cam.origin) - offset);
}

template <typename F>
void ParallelRows(int y0, int y1, int threads, F&& body) {
	if (threads <= 1) { for (int y = y0; y < y1; y++) body(y); return; }
	std::atomic<int> next(y0);
	std::vector<std::thread> pool;
	for (int t = 0; t < threads; t++) pool.emplace_back([&] { for (int y; (y = next.fetch_add(1)) < y1;) body(y); });
	for (auto& t : pool) t.join();
}

} // namespace

extern "C" {

struct agpt_oracle_tables {            // what tests pass in: the flattened tables of include/agpt.h
	const agpt_prim* prims; int n_prims;
	const agpt_sphere* spheres; int n_spheres;
	const agpt_plane* planes; int n_planes;
	const agpt_mesh_desc* meshes; int n_meshes;
	const agpt_material* materials; int n_materials;
	const agpt_light* lights; int n_lights;
	agpt_camera camera;
	agpt_envmap envmap;
	const agpt_instance* instances; int n_instances;
};

void* agpt_oracle_scene_create(const agpt_oracle_tables* t) {
	auto* s = new OScene();
	s->prims.assign(t->prims, t->prims + t->n_prims);
	s->spheres.assign(t->spheres, t->spheres + t->n_spheres);
	s->planes.assign(t->planes, t->planes + t->n_planes);
	s->mats.assign(t->materials, t->materials + t->n_materials);
	s->lights.assign(t->lights, t->lights + t->n_lights);
	if (t->n_instances > 0) s->instances.assign(t->instances, t->instances + t->n_instances);
	s->cam = t->camera;
	if (t->envmap.width > 0) {
		size_t n = (size_t)t->envmap.width * t->envmap.height;
		s->envW = t->envmap.width; s->envH = t->envmap.height; s->envFuncInt = t->envmap.func_int;
		s->envRgb.assign(t->envmap.rgb, t->envmap.rgb + 3 * n);
		s->envFunc.assign(t->envmap.func, t->envmap.func + n);
		s->envCdf.assign(t->envmap.cdf, t->envmap.cdf + n + 1);
	}
	for (int i = 0; i < t->n_meshes; i++) {
		const agpt_mesh_desc& d = t->meshes[i];
		Mesh m;
		if (d.n_nodes) m.nodes.assign(d.nodes, d.nodes + d.n_nodes);
		m.verts.assign(d.tri_verts, d.tri_verts + 12 * (size_t)d.n_tris);
		m.ids.assign(d.tri_ids, d.tri_ids + d.n_tris);
		if (d.tri_normals) m.normals.assign(d.tri_normals, d.tri_normals + 12 * (size_t)d.n_tris);
		if (d.tri_uvs) m.uvs.assign(d.tri_uvs, d.tri_uvs + 6 * (size_t)d.n_tris);
		s->meshes.push_back(std::move(m));
	}
	return s;
}
void agpt_oracle_scene_destroy(void* h) { delete (OScene*)h; }
void agpt_oracle_scene_set_rr_by_bounce(void* h, int on) { ((OScene*)h)->rrByBounce = on != 0; }

// Same contract as agpt_ref_render (oracle/ref_harness.cpp).  counters_out (optional, 6):
// closest rays, any-hit rays, interior visits, box tests, triangle tests, analytic tests.
long long agpt_oracle_render(void* h, int W, int H, int x0, int y0, int x1, int y1, int s0, int ns, int sample_stride,
		int max_depth, int depth_arg, int threads, float* out_rgba, unsigned long long* counters_out) {
	const OScene& sc = *(OScene*)h;
	std::vector<Counters> per(std::max(threads, 1) + 1);
	std::atomic<int> slot(0);
	Counters total;
	std::atomic<int> lock(0);
	ParallelRows(y0, y1, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int k = 0; k < ns; k++) {
			int s = s0 + k * sample_stride;
			for (int x = x0; x < x1; x++) {
				rng.Seed((uint32_t)(y * W + x), (uint32_t)s);
				Ray ray = CameraRay(sc, W, H, x, y, rng);
				V3 clr = Li(sc, ray, max_depth, depth_arg, rng, c);
				float lum = 0.212671f * clr.x + 0.715160f * clr.y + 0.072169f * clr.z;
				if (std::isnan(clr.x) || std::isnan(clr.y) || std::isnan(clr.z) || std::isinf(lum)) clr = v3(0.f);
				float* px = out_rgba + 4 * ((size_t)(H - 1 - y) * W + x);
				px[0] += clr.x; px[1] += clr.y; px[2] += clr.z;
			}
		}
		while (lock.exchange(1)) {}
		total.Add(c);
		lock.store(0);
	});
	if (counters_out) {
		counters_out[0] = total.raysClosest; counters_out[1] = total.raysAny; counters_out[2] = total.interior;
		counters_out[3] = total.boxes; counters_out[4] = total.tris; counters_out[5] = total.analytic;
	}
	return (long long)(x1 - x0) * (y1 - y0) * ns;
}

// counters_out (optional, 3): interior visits, box tests, triangle tests of the whole table.
long long agpt_oracle_primary_hits(void* h, int W, int H, int sample, int threads, agpt_hit* out, unsigned long long* counters_out) {
	const OScene& sc = *(OScene*)h;
	Counters total;
	std::atomic<int> lock(0);
	ParallelRows(0, H, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int x = 0; x < W; x++) {
			rng.Seed((uint32_t)(y * W + x), (uint32_t)sample);
			Ray ray = CameraRay(sc, W, H, x, y, rng);
			Hit hit;
			bool found = SceneIntersect(sc, ray, hit, c);
			agpt_hit& o = out[(size_t)y * W + x];
			o.found = found ? 1u : 0u;
			o.prim = found ? hit.prim : -1;
			o.tri = (found && hit.slot >= 0) ? MeshOfPrim(sc, sc.prims[hit.prim]).ids[hit.slot] : -1;
			o.t = found ? hit.t : 0.f;
		}
		while (lock.exchange(1)) {}
		total.Add(c);
		lock.store(0);
	});
	if (counters_out) { counters_out[0] = total.interior; counters_out[1] = total.boxes; counters_out[2] = total.tris; }
	return 0;
}

// Scene::Intersect / IntersectP for caller rays (O, D normalised like the Ray ctor, tmax): same
// contract as agpt_ref_trace_rays.  counters_out (optional, 3): interior visits, box tests, triangle tests.
void agpt_oracle_trace_rays(void* h, long long n, const float* rays7, int any_hit, agpt_hit* out, unsigned long long* counters_out) {
	const OScene& sc = *(OScene*)h;
	Counters c;
	for (long long i = 0; i < n; i++) {
		const float* r = rays7 + 7 * i;
		Ray ray(v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]);
		agpt_hit& o = out[i];
		o.prim = -1; o.tri = -1; o.t = 0.f;
		if (any_hit) { o.found = SceneIntersectP(sc, ray, c) ? 1u : 0u; continue; }
		Hit hit;
		bool found = SceneIntersect(sc, ray, hit, c);
		o.found = found ? 1u : 0u;
		if (found) {
			o.prim = hit.prim; o.t = hit.t;
			o.tri = hit.slot >= 0 ? MeshOfPrim(sc, sc.prims[hit.prim]).ids[hit.slot] : -1;
		}
	}
	if (counters_out) { counters_out[0] = c.interior; counters_out[1] = c.boxes; counters_out[2] = c.tris; }
}

// radiance + number of RandomFloat() draws of single camera paths
void agpt_oracle_li_pixels(void* h, int W, int H, int n, const int* xs, const int* ys, const int* ss, int max_depth, int depth_arg,
		float* out_rgb, int* draws_out) {
	const OScene& sc = *(OScene*)h;
	Counters c;
	Rng rng;
	for (int i = 0; i < n; i++) {
		rng.Seed((uint32_t)(ys[i] * W + xs[i]), (uint32_t)ss[i]);
		Ray ray = CameraRay(sc, W, H, xs[i], ys[i], rng);
		V3 clr = Li(sc, ray, max_depth, depth_arg, rng, c);
		out_rgb[3 * i] = clr.x; out_rgb[3 * i + 1] = clr.y; out_rgb[3 * i + 2] = clr.z;
		if (draws_out) draws_out[i] = rng.draws;
	}
}

// BSDF::f / Pdf / Sample_f on a flat frame built from (dpdu, dpdv): same contract as agpt_ref_probe_bsdf
// (oracle/ref_harness.cpp) and agpt_probe_bsdf (include/agpt.h), for a material RECORD.
void agpt_oracle_probe_bsdf(int n, const agpt_material* mat, const float* in14, int skip_specular, float* out12) {
	for (int i = 0; i < n; i++) {
		const float* a = in14 + 14 * i;
		V3 dpdu = v3(a[0], a[1], a[2]), dpdv = v3(a[3], a[4], a[5]), wo = v3(a[6], a[7], a[8]), wi = v3(a[9], a[10], a[11]);
		Surface si;
		si.Init(v3(0.f), dpdu, dpdv);
		Bsdf bsdf(si, mat);
		float* o = out12 + 12 * i;
		V3 f = bsdf.f(wo, wi, skip_specular != 0);
		o[0] = f.x; o[1] = f.y; o[2] = f.z;
		o[3] = bsdf.Pdf(wo, wi, skip_specular != 0);
		V3 wis = v3(0.f);
		float pdf = 0;
		bool spec = false;
		V3 fs = bsdf.Sample_f(wo, &wis, a[12], a[13], &pdf, skip_specular != 0, &spec);
		o[4] = wis.x; o[5] = wis.y; o[6] = wis.z; o[7] = fs.x; o[8] = fs.y; o[9] = fs.z; o[10] = pdf; o[11] = spec ? 1.f : 0.f;
	}
}

void agpt_oracle_probe_stream(unsigned pixel, unsigned sample, int k, float* out) {
	Rng rng;
	rng.Seed(pixel, sample);
	for (int i = 0; i < k; i++) out[i] = rng.Float();
}

} // extern "C"
