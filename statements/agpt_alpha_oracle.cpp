// statements/agpt_alpha_oracle.cpp -- TEST INFRASTRUCTURE, not product code.
//
// EXTENSION (include/agpt.h agpt_upload_alpha_masks): the CPU statement of alpha-masked cutout geometry, the one the GPU path is
// checked against.  The reference has no masks; what a masked hit means is defined in agpt.h.
//
// The maps statement (statements/agpt_material_maps_oracle.cpp, with the texture statement and the oracle under it) is compiled
// into this translation unit unchanged.  The mask is applied where the oracle commits a triangle or plane hit, so the oracle's
// SceneIntersect / SceneIntersectP with their recursions are restated here with that one test added, and so are the callers that
// must see it: EstimateDirect's shadow and MIS rays, the path loop, the guide record and the hit tables.  Everything else --
// camera rays, surfaces, BSDFs, light sampling, uvs and the bilinear lookup -- is the code below this file, used as it is.  With
// no mask bound every function here computes what the oracle computes.  Built by __graft_entry__.build() into
// statements/libagpt_alpha_oracle.so (-O2, no FMA contraction).
#include "agpt_material_maps_oracle.cpp"

namespace {

struct AlphaScene {
	MapsScene ms;                                    // scene, textures and map bindings
	std::vector<agpt_alpha_mask> masks;              // per material; empty: no masks
};

inline float Channel(V3 c, int k) { return k == 0 ? c.x : k == 1 ? c.y : c.z; }

// agpt.h agpt_upload_alpha_masks steps 1-3 for a candidate hit h (prim, slot, t, b1, b2) of the world-space ray `ray`
bool MaskKeeps(const AlphaScene& as, const Ray& ray, const Hit& h) {
	const OScene& sc = *as.ms.ts.sc;
	const int mat = sc.prims[h.prim].material;
	if (mat < 0 || mat >= (int)as.masks.size() || as.masks[mat].texture < 0) return true;
	const agpt_alpha_mask& m = as.masks[mat];
	float u = 0, v = 0;
	HitUV(sc, ray, h, &u, &v);
	return Channel(Lookup(as.ms.ts.tex[m.texture], u, v), m.channel) >= m.cutoff;
}
bool MaskKeepsTri(const AlphaScene& as, const Ray& world, int prim, int slot, float t, float b1, float b2) {
	Hit h;
	h.prim = prim; h.slot = slot; h.t = t; h.b1 = b1; h.b2 = b2;
	return MaskKeeps(as, world, h);
}

// oracle RecursiveHit / RecursiveHitP with the mask after TriangleTest (`world`: the world-space ray, for the plane-free uv rule)
bool MRecursiveHit(const AlphaScene& as, const Mesh& m, int primIndex, const agpt_bvh_node& node, Ray& ray, const Ray& world, Hit& hit, Counters& c) {
	bool any = false;
	if (node.count > 0) {
		for (int i = 0; i < node.count; i++) {
			c.tris++;
			float t, b1, b2;
			if (TriangleTest(m, node.first + i, ray, false, t, b1, b2) && MaskKeepsTri(as, world, primIndex, node.first + i, t, b1, b2)) {
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
	if (MRecursiveHit(as, m, primIndex, left, ray, world, hit, c)) any = true;
	if (traverseLeft && traverseRight && MRecursiveHit(as, m, primIndex, right, ray, world, hit, c)) any = true;
	return any;
}
bool MRecursiveHitP(const AlphaScene& as, const Mesh& m, int primIndex, const agpt_bvh_node& node, const Ray& ray, const Ray& world, Counters& c) {
	if (node.count > 0) {
		for (int i = 0; i < node.count; i++) {
			c.tris++;
			float t, b1, b2;
			if (TriangleTest(m, node.first + i, ray, true, t, b1, b2) && MaskKeepsTri(as, world, primIndex, node.first + i, t, b1, b2)) return true;
		}
		return false;
	}
	c.interior++;
	for (int k = 0; k < 2; k++) {
		const agpt_bvh_node& child = m.nodes[node.first + k];
		float tmp;
		c.boxes++;
		if (BoundsIntersect(child, ray, tmp) && MRecursiveHitP(as, m, primIndex, child, ray, world, c)) return true;
	}
	return false;
}

// oracle SceneIntersect with the mask
bool MSceneIntersect(const AlphaScene& as, Ray& ray, Hit& hit, Counters& c) {
	const OScene& sc = *as.ms.ts.sc;
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
			if (PlaneTest(sc.planes[pr.payload], ray, t)) {
				Hit h;
				h.t = t; h.prim = (int)p;
				if (MaskKeeps(as, ray, h)) { ray.t = t; hit = h; found = true; }
			}
		}
		else {
			const bool inst = pr.type == AGPT_PRIM_INSTANCE;
			const Mesh& m = MeshOfPrim(sc, pr);
			const Ray world = ray;
			Ray local = inst ? Ray(Ray::AsGiven(), XformPoint(sc.instances[pr.payload].world_to_object, ray.O), XformVector(sc.instances[pr.payload].world_to_object, ray.D), ray.t) : ray;
			bool any = false;
			if (m.nodes.empty()) {
				for (size_t j = 0; j < m.ids.size(); j++) {
					c.tris++;
					float b1, b2;
					if (TriangleTest(m, (int)j, local, false, t, b1, b2) && MaskKeepsTri(as, world, (int)p, (int)j, t, b1, b2)) {
						local.t = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = (int)p; hit.slot = (int)j; any = true;
					}
				}
			}
			else {
				float dist;
				c.boxes++;
				if (BoundsIntersect(m.nodes[0], local, dist) && MRecursiveHit(as, m, (int)p, m.nodes[0], local, world, hit, c)) any = true;
			}
			if (any) { ray.t = local.t; found = true; }
		}
	}
	return found;
}

// oracle SceneIntersectP with the mask
bool MSceneIntersectP(const AlphaScene& as, const Ray& ray, Counters& c) {
	const OScene& sc = *as.ms.ts.sc;
	c.raysAny++;
	for (size_t p = 0; p < sc.prims.size(); p++) {
		const agpt_prim& pr = sc.prims[p];
		float t;
		if (pr.type == AGPT_PRIM_SPHERE) { c.analytic++; if (SphereTest(sc.spheres[pr.payload], ray, t)) return true; }
		else if (pr.type == AGPT_PRIM_PLANE) {
			c.analytic++;
			if (PlaneTest(sc.planes[pr.payload], ray, t)) {
				Hit h;
				h.t = t; h.prim = (int)p;
				if (MaskKeeps(as, ray, h)) return true;
			}
		}
		else {
			const bool inst = pr.type == AGPT_PRIM_INSTANCE;
			const Mesh& m = MeshOfPrim(sc, pr);
			const Ray local = inst ? Ray(Ray::AsGiven(), XformPoint(sc.instances[pr.payload].world_to_object, ray.O), XformVector(sc.instances[pr.payload].world_to_object, ray.D), ray.t) : ray;
			if (m.nodes.empty()) {
				for (size_t j = 0; j < m.ids.size(); j++) {
					c.tris++;
					float b1, b2;
					if (TriangleTest(m, (int)j, local, true, t, b1, b2) && MaskKeepsTri(as, ray, (int)p, (int)j, t, b1, b2)) return true;
				}
			}
			else {
				float dist;
				c.boxes++;
				if (BoundsIntersect(m.nodes[0], local, dist) && MRecursiveHitP(as, m, (int)p, m.nodes[0], local, ray, c)) return true;
			}
		}
	}
	return false;
}

// oracle EstimateDirect with its shadow ray and MIS ray through the masked scene
V3 MEstimateDirect(const AlphaScene& as, const Surface& si, const Bsdf& bsdf, V3 wo, float uScatX, float uScatY, int lightIdx,
		float uLightX, float uLightY, Rng& rng, Counters& c) {
	const OScene& sc = *as.ms.ts.sc;
	const agpt_light& light = sc.lights[lightIdx];
	V3 lemit = v3(light.lemit);
	V3 Ld = v3(0.f), wi = v3(0.f);
	float lightPdf = 0, scatteringPdf = 0;
	V3 Li = v3(0.f);
	Ray vis(v3(0.f), v3(1.f, 0.f, 0.f));
	if (light.type == AGPT_LIGHT_AREA) {
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
	else if (light.type == AGPT_LIGHT_INFINITE_AREA) {
		float u01 = rng.Float();
		if (EnvSampleLi(sc, u01, &wi, &lightPdf)) {
			vis = Ray(si.p + kEps * si.n, wi);
			Li = EnvLe(sc, vis.D);
		}
	}
	else {
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
			if (MSceneIntersectP(as, vis, c)) Li = v3(0.f);
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
			else lp = dot(si.n, wi) > 0 ? kInv2Pi : 0.f;
			if (lp == 0) return Ld;
			float weight = PowerHeuristic(1, scatteringPdf, 1, lp);
			Ray ray(si.p + kEps * wi, wi);
			Hit h;
			bool found = MSceneIntersect(as, ray, h, c);
			V3 Lr = v3(0.f);
			if (found) { if (sc.prims[h.prim].area_light == lightIdx) Lr = lemit; }
			else if (light.type == AGPT_LIGHT_UNIFORM_INFINITE) Lr = lemit;
			else if (light.type == AGPT_LIGHT_INFINITE_AREA) Lr = EnvLe(sc, ray.D);
			if (!IsBlack(Lr)) Ld += f * Lr * weight / scatteringPdf;
		}
	}
	return Ld;
}

// the maps statement's MapsLi with every ray through the masked scene
V3 AlphaLi(const AlphaScene& as, Ray ray, int maxDepth, int depthArg, Rng& rng, Counters& c) {
	const OScene& sc = *as.ms.ts.sc;
	V3 beta = v3(1.f), L = v3(0.f);
	bool specularBounce = false;
	for (int bounces = 0;; bounces++) {
		Hit h;
		const Ray ray0 = ray;
		bool found = MSceneIntersect(as, ray, h, c);
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
		if (pr.material < 0) {
			ray = Ray(si.p + kEps * ray.D, ray.D);
			bounces--;
			continue;
		}
		const agpt_material mat = HitMaps(as.ms, ray0, h, si);
		Bsdf bsdf(si, &mat);
		V3 wo = -ray.D;
		if (!bsdf.IsPerfectlySpecular() && !sc.lights.empty()) {
			int nLights = (int)sc.lights.size();
			int numLight = std::min((int)(rng.Float() * nLights), nLights - 1);
			float lightPdf = 1.f / nLights;
			float uLy = rng.Float(), uLx = rng.Float();
			float uSy = rng.Float(), uSx = rng.Float();
			L += beta * (MEstimateDirect(as, si, bsdf, wo, uSx, uSy, numLight, uLx, uLy, rng, c) / lightPdf);
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
		if (maxComponent < 1 && (sc.rrByBounce ? bounces : depthArg) > 3) {
			float q = std::max(.05f, 1 - maxComponent);
			if (rng.Float() < q) break;
			beta /= 1 - q;
		}
		ray = Ray(si.p + kEps * wi, wi);
	}
	return L;
}

void SetMasks(AlphaScene& as, const agpt_alpha_mask* masks, int n) {
	as.masks.clear();
	if (masks) as.masks.assign(masks, masks + n);
}

// the six counters of agpt_alpha_oracle_render (closest, any, interior, boxes, tris, analytic) into counters_out, unless NULL
void PutCounters(const Counters& c, unsigned long long* counters_out) {
	if (!counters_out) return;
	const uint64_t v[6] = { c.raysClosest, c.raysAny, c.interior, c.boxes, c.tris, c.analytic };
	for (int i = 0; i < 6; i++) counters_out[i] = v[i];
}

} // namespace

extern "C" {

// The tables of a host-mirror scene (agpt_scene_tables) and its alpha masks (agpt_host_scene_alpha_masks; NULL, 0: none)
void* agpt_alpha_oracle_create(const agpt_scene_tables* t, const agpt_alpha_mask* masks, int n_masks) {
	auto* as = new AlphaScene();
	as->ms.ts.sc = (OScene*)agpt_oracle_scene_create((const agpt_oracle_tables*)t);
	SetTextures(as->ms, t->textures, t->n_textures, t->material_textures, t->n_material_textures);
	SetMasks(*as, masks, n_masks);
	return as;
}
// replaces the textures and bindings (agpt_upload_material_textures' arguments); like the device, this clears the masks
void agpt_alpha_oracle_set_textures(void* h, const agpt_texture* textures, int n, const agpt_material_textures* bind, int n_materials) {
	AlphaScene& as = *(AlphaScene*)h;
	SetTextures(as.ms, textures, n, bind, n_materials);
	as.masks.clear();
}
// replaces the masks (agpt_upload_alpha_masks' arguments)
void agpt_alpha_oracle_set_masks(void* h, const agpt_alpha_mask* masks, int n) { SetMasks(*(AlphaScene*)h, masks, n); }
void agpt_alpha_oracle_destroy(void* h) { AlphaScene* as = (AlphaScene*)h; agpt_oracle_scene_destroy(as->ms.ts.sc); delete as; }
void agpt_alpha_oracle_set_rr_by_bounce(void* h, int on) { ((AlphaScene*)h)->ms.ts.sc->rrByBounce = on != 0; }

// agpt_render of samples [s0, s0 + ns) into out_rgba (added to); counters_out (6, or NULL): closest, any, interior, boxes, tris, analytic
void agpt_alpha_oracle_render(void* h, int W, int H, int s0, int ns, int max_depth, int depth_arg, int threads, float* out_rgba,
		unsigned long long* counters_out) {
	const AlphaScene& as = *(AlphaScene*)h;
	Counters total;
	std::mutex lock;
	ParallelRows(0, H, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int k = 0; k < ns; k++)
			for (int x = 0; x < W; x++) {
				rng.Seed((uint32_t)(y * W + x), (uint32_t)(s0 + k));
				Ray ray = CameraRay(*as.ms.ts.sc, W, H, x, y, rng);
				V3 clr = AlphaLi(as, ray, max_depth, depth_arg, rng, c);
				float lum = 0.212671f * clr.x + 0.715160f * clr.y + 0.072169f * clr.z;
				if (std::isnan(clr.x) || std::isnan(clr.y) || std::isnan(clr.z) || std::isinf(lum)) clr = v3(0.f);
				float* px = out_rgba + 4 * ((size_t)(H - 1 - y) * W + x);
				px[0] += clr.x; px[1] += clr.y; px[2] += clr.z;
			}
		std::lock_guard<std::mutex> g(lock);
		total.Add(c);
	});
	PutCounters(total, counters_out);
}

// agpt_li_pixels: radiance of single camera paths
void agpt_alpha_oracle_li_pixels(void* h, int W, int H, int n, const int* xs, const int* ys, const int* ss, int max_depth, int depth_arg, float* out_rgb) {
	const AlphaScene& as = *(AlphaScene*)h;
	Counters c;
	Rng rng;
	for (int i = 0; i < n; i++) {
		rng.Seed((uint32_t)(ys[i] * W + xs[i]), (uint32_t)ss[i]);
		Ray ray = CameraRay(*as.ms.ts.sc, W, H, xs[i], ys[i], rng);
		V3 clr = AlphaLi(as, ray, max_depth, depth_arg, rng, c);
		out_rgb[3 * i] = clr.x; out_rgb[3 * i + 1] = clr.y; out_rgb[3 * i + 2] = clr.z;
	}
}

// agpt_trace_rays: closest or any hit of caller rays (rays7 = O, D normalised like the Ray ctor, tmax); counters_out (6, or NULL) as for agpt_alpha_oracle_render
void agpt_alpha_oracle_trace_rays(void* h, long long n, const float* rays7, int any_hit, agpt_hit* out, unsigned long long* counters_out) {
	const AlphaScene& as = *(AlphaScene*)h;
	const OScene& sc = *as.ms.ts.sc;
	Counters c;
	for (long long i = 0; i < n; i++) {
		const float* r = rays7 + 7 * i;
		Ray ray(v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]);
		agpt_hit& o = out[i];
		o.prim = -1; o.tri = -1; o.t = 0.f;
		if (any_hit) { o.found = MSceneIntersectP(as, ray, c) ? 1u : 0u; continue; }
		Hit hit;
		bool found = MSceneIntersect(as, ray, hit, c);
		o.found = found ? 1u : 0u;
		if (found) {
			o.prim = hit.prim; o.t = hit.t;
			o.tri = hit.slot >= 0 ? MeshOfPrim(sc, sc.prims[hit.prim]).ids[hit.slot] : -1;
		}
	}
	PutCounters(c, counters_out);
}

// agpt_trace_primary: the closest hit of every camera ray of sample `sample`, row-major from the top row; counters_out (6, or NULL) as for
// agpt_alpha_oracle_render
void agpt_alpha_oracle_primary_hits(void* h, int W, int H, int sample, agpt_hit* out, unsigned long long* counters_out) {
	const AlphaScene& as = *(AlphaScene*)h;
	const OScene& sc = *as.ms.ts.sc;
	Counters c;
	Rng rng;
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			rng.Seed((uint32_t)(y * W + x), (uint32_t)sample);
			Ray ray = CameraRay(sc, W, H, x, y, rng);
			Hit hit;
			bool found = MSceneIntersect(as, ray, hit, c);
			agpt_hit& o = out[(size_t)y * W + x];
			o.found = found ? 1u : 0u;
			o.prim = found ? hit.prim : -1;
			o.tri = (found && hit.slot >= 0) ? MeshOfPrim(sc, sc.prims[hit.prim]).ids[hit.slot] : -1;
			o.t = found ? hit.t : 0.f;
		}
	PutCounters(c, counters_out);
}

// agpt_render_guides: the maps statement's guide record over the masked first hit
void agpt_alpha_oracle_guides(void* h, int W, int H, int num_samples, int threads, float* albedo, float* normal_depth) {
	const AlphaScene& as = *(AlphaScene*)h;
	const OScene& sc = *as.ms.ts.sc;
	ParallelRows(0, H, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int x = 0; x < W; x++) {
			V3 a = v3(0.f), n = v3(0.f);
			float hits = 0, tsum = 0;
			for (int s = 0; s < num_samples; s++) {
				rng.Seed((uint32_t)(y * W + x), (uint32_t)s);
				Ray ray = CameraRay(sc, W, H, x, y, rng);
				const Ray ray0 = ray;
				const V3 D = ray.D;
				Hit hit;
				V3 alb = v3(1.f), nrm = v3(0.f);
				if (MSceneIntersect(as, ray, hit, c)) {
					Surface si;
					BuildSurface(sc, ray, hit, si);
					const agpt_prim& pr = sc.prims[hit.prim];
					agpt_material m;
					if (pr.material >= 0) m = HitMaps(as.ms, ray0, hit, si);
					nrm = dot(si.sn, D) > 0.f ? -si.sn : si.sn;
					if (pr.material >= 0) {
						if (m.type == AGPT_MAT_MIRROR) alb = v3(m.mirror_r);
						else if (m.type == AGPT_MAT_GLASS) alb = v3(m.mirror_r) + v3(m.diffuse_r);
						else alb = v3(m.diffuse_r) + v3(m.spec_r0);
						alb = v3(tmin2(alb.x, 1.f), tmin2(alb.y, 1.f), tmin2(alb.z, 1.f));
					}
					hits += 1.f;
					tsum += hit.t;
				}
				a += alb;
				n += nrm;
			}
			const float ns = (float)num_samples;
			float* pa = albedo + 4 * ((size_t)(H - 1 - y) * W + x);
			float* pn = normal_depth + 4 * ((size_t)(H - 1 - y) * W + x);
			pa[0] = a.x / ns; pa[1] = a.y / ns; pa[2] = a.z / ns; pa[3] = hits / ns;
			pn[0] = n.x / ns; pn[1] = n.y / ns; pn[2] = n.z / ns; pn[3] = hits > 0.f ? tsum / hits : 0.f;
		}
	});
}

// single rule, for the CPU tests: channel `channel` of the lookup of image (W x H x 3) at each uv (agpt.h steps 2)
void agpt_alpha_oracle_lookup_channel(int W, int H, const float* rgb, int channel, int n, const float* uv, float* out) {
	const Tex t = { W, H, rgb };
	for (int i = 0; i < n; i++) out[i] = Channel(Lookup(t, uv[2 * i], uv[2 * i + 1]), channel);
}

} // extern "C"
