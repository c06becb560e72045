// oracle/agpt_shape_oracle.cpp -- TEST INFRASTRUCTURE, not product code.
//
// EXTENSION (include/agpt.h AGPT_LIGHT_SAMPLE_SHAPE): the CPU statement of sampled plane and mesh area lights, the one the
// GPU path is checked against.  Parity unpinned by the reference -- its Plane and TriangleMesh inherit Sample / Pdf stubs
// that return pdf 0 (lights.cpp:115-130) -- so this is PBRT-v3's Shape::Sample / Shape::Pdf in solid angle, fitted to the
// oracle's conventions.
//
// The oracle (agpt_oracle.cpp, pinned bit for bit to the reference) is compiled into this translation unit unchanged and
// reused as it is: tables, intersection, BSDF, sphere and environment lights, camera, RNG.  Only EstimateDirect and the Li
// loop that calls it are restated here with the extension added; with no light flagged they are the oracle's functions.
// Built by __graft_entry__.build() into oracle/libagpt_shape_oracle.so with the oracle's flags (-O2, no FMA contraction).
#include "agpt_oracle.cpp"

namespace {

// Per light: total area, and for a mesh the Distribution1D (sampling.h:22-35) over its triangle areas in slot order, a
// degenerate triangle (one TriangleIntersect would reject, trianglemesh.cpp:74-77) counting 0.  Built from the scene's own
// triangles, independently of the library's tables.
struct ShapeLight {
	std::vector<float> cdf;        // meshes only
	float area = 0;                // total area; 0: the light is never sampled
};
typedef std::vector<ShapeLight> ShapeTables;

struct ShapeScene {
	OScene* sc;
	ShapeTables st;
};

inline bool SamplesShape(const OScene& sc, const agpt_light& l) {
	return l.type == AGPT_LIGHT_AREA && (l.flags & AGPT_LIGHT_SAMPLE_SHAPE) &&
		(sc.prims[l.prim].type == AGPT_PRIM_PLANE || sc.prims[l.prim].type == AGPT_PRIM_MESH || sc.prims[l.prim].type == AGPT_PRIM_BVH_MESH);
}
inline float TriangleArea(V3 v0, V3 v1, V3 v2) { return 0.5f * length(cross(v1 - v0, v2 - v0)); }
inline V3 TriangleNormal(const Mesh& m, int slot) {
	const float* p = &m.verts[12 * (size_t)slot];
	return normalize(cross(v3(p + 4) - v3(p), v3(p + 8) - v3(p)));
}

ShapeTables BuildShapeLights(const OScene& sc) {
	ShapeTables st(sc.lights.size());
	for (size_t i = 0; i < sc.lights.size(); i++) {
		if (!SamplesShape(sc, sc.lights[i])) continue;
		const agpt_prim& pr = sc.prims[sc.lights[i].prim];
		ShapeLight& sl = st[i];
		if (pr.type == AGPT_PRIM_PLANE) { sl.area = 4.f * sc.planes[pr.payload].half_x * sc.planes[pr.payload].half_z; continue; }
		const Mesh& m = sc.meshes[pr.payload];
		const int n = (int)m.ids.size();
		std::vector<float> func((size_t)n);
		float total = 0;
		for (int j = 0; j < n; j++) {
			const float* p = &m.verts[12 * (size_t)j];
			float uv[6];
			TriangleUVs(m, j, uv);
			V3 dpdu = v3(0.f), dpdv = v3(0.f);
			func[j] = TriangleDerivatives(v3(p), v3(p + 4), v3(p + 8), uv, dpdu, dpdv) ? TriangleArea(v3(p), v3(p + 4), v3(p + 8)) : 0.f;
			total += func[j];
		}
		if (n == 0) continue;
		sl.cdf.assign((size_t)n + 1, 0.f);
		for (int j = 1; j < n + 1; j++) sl.cdf[j] = sl.cdf[j - 1] + func[j - 1] / n;
		const float funcInt = sl.cdf[n];
		if (funcInt == 0) continue;                        // (Distribution1D would fall back to a uniform cdf: never sampled instead)
		for (int j = 1; j < n + 1; j++) sl.cdf[j] /= funcInt;
		sl.area = total;
	}
	return st;
}

// solid-angle pdf of a point with light normal n seen from the reference point along the unit direction wi: dist^2 / (|cos| * area)
inline float ShapeSolidAnglePdf(float d2, V3 n, V3 wi, float area) {
	float c = absdot(n, wi);
	if (c == 0) return 0;
	float pdf = d2 / (c * area);
	return std::isinf(pdf) ? 0.f : pdf;
}

// Sample_Li's point: Distribution1D::SampleDiscrete (PBRT-v3 sampling.h) on the area cdf, UniformSampleTriangle on the
// remapped u0 and u1; a plane: a uniform point of the rectangle.
void ShapeSample(const OScene& sc, const ShapeTables& st, int lightIdx, V3 refP, float u0, float u1, V3* pOut, V3* nOut, float* pdf) {
	const ShapeLight& sl = st[lightIdx];
	const agpt_prim& pr = sc.prims[sc.lights[lightIdx].prim];
	*pdf = 0; *pOut = v3(0.f); *nOut = v3(0.f);
	if (!(sl.area > 0)) return;
	V3 p, n;
	if (pr.type == AGPT_PRIM_PLANE) {
		const agpt_plane& pl = sc.planes[pr.payload];
		p = v3(pl.o[0] + (2 * u0 - 1) * pl.half_x, pl.o[1], pl.o[2] + (2 * u1 - 1) * pl.half_z);
		n = v3(0.f, 1.f, 0.f);
	}
	else {
		const Mesh& m = sc.meshes[pr.payload];
		const int size = (int)sl.cdf.size();
		int first = 0, len = size;                                                        // FindInterval (sampling.h:4-18)
		while (len > 0) {
			int half = len >> 1, middle = first + half;
			if (sl.cdf[middle] <= u0) { first = middle + 1; len -= half + 1; }
			else len = half;
		}
		int offset = std::min(std::max(first - 1, 0), size - 2);
		float width = sl.cdf[offset + 1] - sl.cdf[offset];
		if (!(width > 0)) return;                          // a zero-area triangle (u0 == 1 can land on one at the end)
		float ur = (u0 - sl.cdf[offset]) / width;
		const float* q = &m.verts[12 * (size_t)offset];
		V3 v0 = v3(q), v1 = v3(q + 4), v2 = v3(q + 8);
		float su0 = std::sqrt(ur);
		float b0 = 1 - su0, b1 = u1 * su0;
		p = b0 * v0 + b1 * v1 + (1 - b0 - b1) * v2;
		n = normalize(cross(v1 - v0, v2 - v0));
	}
	*pOut = p; *nOut = n;
	V3 wi = p - refP;
	float d2 = sqrLength(wi);
	if (d2 == 0) return;
	wi /= std::sqrt(d2);
	*pdf = ShapeSolidAnglePdf(d2, n, wi, sl.area);
}

// Pdf_Li: the MIS ray against the light's shape ALONE (Plane::Intersect, or the mesh's own TriangleIntersect / RecursiveHit
// order), 0 without a hit.
float ShapePdf(const OScene& sc, const ShapeTables& st, int lightIdx, V3 refP, V3 wi) {
	const ShapeLight& sl = st[lightIdx];
	const agpt_prim& pr = sc.prims[sc.lights[lightIdx].prim];
	if (!(sl.area > 0)) return 0;
	Ray ray(refP + kEps * wi, wi);
	V3 n;
	float t = 0;
	if (pr.type == AGPT_PRIM_PLANE) {
		if (!PlaneTest(sc.planes[pr.payload], ray, t)) return 0;
		n = v3(0.f, 1.f, 0.f);
	}
	else {
		const Mesh& m = sc.meshes[pr.payload];
		Hit h;
		Counters none;                                                                    // not a scene ray: not counted
		bool found = false;
		if (m.nodes.empty()) {
			for (size_t j = 0; j < m.ids.size(); j++) {
				float b1, b2;
				if (TriangleTest(m, (int)j, ray, false, t, b1, b2)) { ray.t = t; h.t = t; h.slot = (int)j; found = true; }
			}
		}
		else {
			float dist;
			found = BoundsIntersect(m.nodes[0], ray, dist) && RecursiveHit(m, 0, m.nodes[0], ray, h, none);
		}
		if (!found) return 0;
		t = h.t;
		n = TriangleNormal(m, h.slot);
	}
	V3 p = ray.O + t * ray.D;
	return ShapeSolidAnglePdf(sqrLength(p - refP), n, wi, sl.area);
}

// EstimateDirect (integrator.h:38-93) as the oracle states it, with the sampled plane / mesh lights added (marked "extension")
V3 ShapeEstimateDirect(const OScene& sc, const ShapeTables& st, const Surface& si, const Bsdf& bsdf, V3 wo, float uScatX, float uScatY, int lightIdx,
		float uLightX, float uLightY, Rng& rng, Counters& c) {
	const agpt_light& light = sc.lights[lightIdx];
	V3 lemit = v3(light.lemit);
	V3 Ld = v3(0.f), wi = v3(0.f);
	float lightPdf = 0, scatteringPdf = 0;
	V3 Li = v3(0.f);
	Ray vis(v3(0.f), v3(1.f, 0.f, 0.f));
	if (light.type == AGPT_LIGHT_AREA) {                                                  // lights.cpp:115-126
		const agpt_prim& lp = sc.prims[light.prim];
		if (lp.type == AGPT_PRIM_SPHERE || SamplesShape(sc, light)) {
			V3 pS, nS;
			if (lp.type == AGPT_PRIM_SPHERE) SphereSample(sc.spheres[lp.payload], si.p, uLightX, uLightY, &pS, &nS, &lightPdf);
			else ShapeSample(sc, st, lightIdx, si.p, uLightX, uLightY, &pS, &nS, &lightPdf);       // extension
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
				lp = lpr.type == AGPT_PRIM_SPHERE ? SpherePdf(sc.spheres[lpr.payload], si.p)
					: SamplesShape(sc, light) ? ShapePdf(sc, st, lightIdx, si.p, wi) : 0.f;                   // extension
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

// PathTracer::Li (integrator.h:124-191) as the oracle states it, calling ShapeEstimateDirect
// sc.rrByBounce (EXTENSION, parity unpinned by the reference: it has no such rule): the roulette is keyed on the
// path's bounce index -- `bounces > 3`, as PBRT states it -- instead of on the constant depth argument.
V3 ShapeLi(const OScene& sc, const ShapeTables& st, Ray ray, int maxDepth, int depthArg, Rng& rng, Counters& c) {
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
			L += beta * (ShapeEstimateDirect(sc, st, si, bsdf, wo, uSx, uSy, numLight, uLx, uLy, rng, c) / lightPdf);
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

} // namespace

extern "C" {

// the oracle's scene (agpt_oracle_scene_create) plus the sampling tables of its flagged lights
void* agpt_shape_oracle_scene_create(const agpt_oracle_tables* t) {
	auto* s = new ShapeScene();
	s->sc = (OScene*)agpt_oracle_scene_create(t);
	s->st = BuildShapeLights(*s->sc);
	return s;
}
void agpt_shape_oracle_scene_destroy(void* h) {
	auto* s = (ShapeScene*)h;
	agpt_oracle_scene_destroy(s->sc);
	delete s;
}
void agpt_shape_oracle_scene_set_rr_by_bounce(void* h, int on) { agpt_oracle_scene_set_rr_by_bounce(((ShapeScene*)h)->sc, on); }
void agpt_shape_oracle_trace_rays(void* h, long long n, const float* rays7, int any_hit, agpt_hit* out, unsigned long long* counters_out) {
	agpt_oracle_trace_rays(((ShapeScene*)h)->sc, n, rays7, any_hit, out, counters_out);
}

// Same contract as agpt_oracle_render.  counters_out (optional, 6):
// closest rays, any-hit rays, interior visits, box tests, triangle tests, analytic tests.
long long agpt_shape_oracle_render(void* h, int W, int H, int x0, int y0, int x1, int y1, int s0, int ns, int sample_stride,
		int max_depth, int depth_arg, int threads, float* out_rgba, unsigned long long* counters_out) {
	const OScene& sc = *((ShapeScene*)h)->sc;
	const ShapeTables& st = ((ShapeScene*)h)->st;
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
				V3 clr = ShapeLi(sc, st, ray, max_depth, depth_arg, rng, c);
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

// Same contract as agpt_oracle_li_pixels.
void agpt_shape_oracle_li_pixels(void* h, int W, int H, int n, const int* xs, const int* ys, const int* ss, int max_depth, int depth_arg,
		float* out_rgb, int* draws_out) {
	const OScene& sc = *((ShapeScene*)h)->sc;
	const ShapeTables& st = ((ShapeScene*)h)->st;
	Counters c;
	Rng rng;
	for (int i = 0; i < n; i++) {
		rng.Seed((uint32_t)(ys[i] * W + xs[i]), (uint32_t)ss[i]);
		Ray ray = CameraRay(sc, W, H, xs[i], ys[i], rng);
		V3 clr = ShapeLi(sc, st, ray, max_depth, depth_arg, rng, c);
		out_rgb[3 * i] = clr.x; out_rgb[3 * i + 1] = clr.y; out_rgb[3 * i + 2] = clr.z;
		if (draws_out) draws_out[i] = rng.draws;
	}
}

// Same contract as agpt_probe_light_sample (include/agpt.h)
void agpt_shape_oracle_probe_light_sample(void* h, int light, int n, const float* in8, float* out8) {
	const OScene& sc = *((ShapeScene*)h)->sc;
	const ShapeTables& st = ((ShapeScene*)h)->st;
	for (int i = 0; i < n; i++) {
		const float* a = in8 + 8 * i;
		float* o = out8 + 8 * i;
		V3 p, nn;
		float pdf;
		ShapeSample(sc, st, light, v3(a), a[3], a[4], &p, &nn, &pdf);
		o[0] = p.x; o[1] = p.y; o[2] = p.z; o[3] = pdf;
		o[4] = ShapePdf(sc, st, light, v3(a), v3(a + 5));
		o[5] = nn.x; o[6] = nn.y; o[7] = nn.z;
	}
}

} // extern "C"
