// statements/agpt_material_maps_oracle.cpp -- TEST INFRASTRUCTURE, not product code.
//
// EXTENSION (include/agpt.h agpt_upload_material_textures): the CPU statement of roughness-metallic and normal maps on Disney
// materials, the one the GPU path is checked against.  The reference has neither; what a mapped hit means is defined in agpt.h.
//
// The texture statement (statements/agpt_texture_oracle.cpp, itself the oracle compiled unchanged plus the uv rules and the
// lookup) is compiled into this translation unit unchanged and reused as it is.  New here: dp/du and dp/dv of each shape's uv,
// the normal-map frame rule, the per-hit material derived from the maps, and the path loop, guide record and per-hit rows
// that use them.  Built by __graft_entry__.build() into statements/libagpt_material_maps_oracle.so (-O2, no FMA contraction).
#include "agpt_texture_oracle.cpp"

#include <mutex>

namespace {

struct MapsScene {
	TexScene ts;                                     // scene, textures (ts.tex) and base bindings (ts.matTex)
	std::vector<agpt_material_textures> bind;        // per material; empty: no maps
};

const agpt_material_textures* BindingOf(const MapsScene& ms, int material) {
	return material >= 0 && material < (int)ms.bind.size() ? &ms.bind[material] : nullptr;
}

// T = dp/du and B = dp/dv of the texture's uv (agpt.h maps step 2), from the quantities BuildSurface forms
void HitTangents(const OScene& sc, const Ray& ray, const Hit& h, V3* T, V3* B) {
	const agpt_prim& pr = sc.prims[h.prim];
	if (pr.type == AGPT_PRIM_SPHERE) {
		const agpt_sphere& sp = sc.spheres[pr.payload];
		V3 p = ray.O + h.t * ray.D;
		V3 pHit = p - v3(sp.center);
		if (pHit.x == 0 && pHit.y == 0) pHit.x = kEps * sp.r;
		float theta = std::acos(tclamp(pHit.z / sp.r, -1.f, 1.f));
		float zRadius = std::sqrt(pHit.x * pHit.x + pHit.y * pHit.y);
		float invZRadius = 1 / zRadius;
		float cosPhi = pHit.x * invZRadius, sinPhi = pHit.y * invZRadius;
		*T = v3(-kTwoPi * pHit.y, kTwoPi * pHit.x, 0);
		*B = kPi * v3(pHit.z * cosPhi, pHit.z * sinPhi, -sp.r * std::sin(theta));
	}
	else if (pr.type == AGPT_PRIM_PLANE) { *T = v3(1, 0, 0); *B = v3(0, 0, 1); }
	else {
		const agpt_instance* in = pr.type == AGPT_PRIM_INSTANCE ? &sc.instances[pr.payload] : nullptr;
		const Mesh& m = sc.meshes[in ? in->mesh : pr.payload];
		const float* p = &m.verts[12 * (size_t)h.slot];
		V3 v0 = v3(p), v1 = v3(p + 4), v2 = v3(p + 8);
		if (in) { v0 = XformPoint(in->object_to_world, v0); v1 = XformPoint(in->object_to_world, v1); v2 = XformPoint(in->object_to_world, v2); }
		float uv[6];
		TriangleUVs(m, h.slot, uv);
		*T = v3(0.f); *B = v3(0.f);
		TriangleDerivatives(v0, v1, v2, uv, *T, *B);
	}
}

// agpt.h maps step 2 for the looked-up texel c: false (surface untouched) in the three cases agpt.h names
bool NormalMapFrame(V3 c, float scale, V3 T, V3 B, Surface& s) {
	const V3 nts = v3(scale * (2 * c.x - 1), scale * (2 * c.y - 1), 2 * c.z - 1);
	if (nts.x == 0 && nts.y == 0 && nts.z > 0) return false;
	const V3 N = s.sn;
	V3 Tp = T - N * dot(N, T);
	if (dot(Tp, Tp) == 0) return false;
	Tp = normalize(Tp);
	V3 Bp = cross(N, Tp);
	if (dot(Bp, B) < 0) Bp = -Bp;
	V3 n = (nts.x * Tp + nts.y * Bp) + nts.z * N;
	if (!(dot(n, N) > 0)) return false;
	n = normalize(n);
	s.sn = n;
	s.sdpdu = Tp - n * dot(n, Tp);
	return true;
}

inline float Clamp01(float x) { return x < 0.f ? 0.f : x > 1.f ? 1.f : x; }

// agpt.h maps step 1 from the roughness-metallic texel c and the base colour C: DisneyMaterial's constructor arithmetic
agpt_material DeriveMaterial(const agpt_material& rec, V3 C, V3 c) {
	agpt_material m = rec;
	const float r = rec.roughness * Clamp01(c.y), k = rec.metallic * Clamp01(c.z);
	const float dw = (1 - k) * (1 - 0.f);
	const V3 d = dw > 0 ? dw * C : v3(0.f);
	const float a = std::max(.001f, std::max(.001f, r * r));
	const float r0 = ((rec.eta - 1) * (rec.eta - 1)) / ((rec.eta + 1) * (rec.eta + 1));
	const V3 s0 = Lerp(k, v3(r0), C);
	m.lobes = (dw > 0 ? (uint32_t)(AGPT_LOBE_DIFFUSE | AGPT_LOBE_RETRO) : 0u) | (uint32_t)AGPT_LOBE_MICROFACET;
	m.roughness = r; m.metallic = k;
	m.diffuse_r[0] = d.x; m.diffuse_r[1] = d.y; m.diffuse_r[2] = d.z;
	m.spec_r0[0] = s0.x; m.spec_r0[1] = s0.y; m.spec_r0[2] = s0.z;
	m.alpha_x = a; m.alpha_y = a;
	return m;
}

// the hit's material record (step 1) and, with a normal map, its mapped surface (step 2)
agpt_material HitMaps(const MapsScene& ms, const Ray& ray, const Hit& h, Surface& si) {
	const OScene& sc = *ms.ts.sc;
	const agpt_prim& pr = sc.prims[h.prim];
	const agpt_material_textures* b = BindingOf(ms, pr.material);
	if (!b) return HitMaterial(ms.ts, ray, h);
	float u = 0, v = 0;
	HitUV(sc, ray, h, &u, &v);
	if (b->normal >= 0) {
		V3 T, B;
		HitTangents(sc, ray, h, &T, &B);
		NormalMapFrame(Lookup(ms.ts.tex[b->normal], u, v), b->normal_scale, T, B, si);
	}
	if (b->roughness_metallic < 0) return HitMaterial(ms.ts, ray, h);
	const V3 C = b->base >= 0 ? Lookup(ms.ts.tex[b->base], u, v) : v3(b->color[0], b->color[1], b->color[2]);
	return DeriveMaterial(sc.mats[pr.material], C, Lookup(ms.ts.tex[b->roughness_metallic], u, v));
}

// PathTracer::Li as oracle/agpt_oracle.cpp states it (the loop of TexLi), each hit shaded with HitMaps
V3 MapsLi(const MapsScene& ms, Ray ray, int maxDepth, int depthArg, Rng& rng, Counters& c) {
	const OScene& sc = *ms.ts.sc;
	V3 beta = v3(1.f), L = v3(0.f);
	bool specularBounce = false;
	for (int bounces = 0;; bounces++) {
		Hit h;
		const Ray ray0 = ray;
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
		if (pr.material < 0) {
			ray = Ray(si.p + kEps * ray.D, ray.D);
			bounces--;
			continue;
		}
		const agpt_material mat = HitMaps(ms, ray0, h, si);
		Bsdf bsdf(si, &mat);
		V3 wo = -ray.D;
		if (!bsdf.IsPerfectlySpecular() && !sc.lights.empty()) {
			int nLights = (int)sc.lights.size();
			int numLight = std::min((int)(rng.Float() * nLights), nLights - 1);
			float lightPdf = 1.f / nLights;
			float uLy = rng.Float(), uLx = rng.Float();
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
		if (maxComponent < 1 && (sc.rrByBounce ? bounces : depthArg) > 3) {
			float q = std::max(.05f, 1 - maxComponent);
			if (rng.Float() < q) break;
			beta /= 1 - q;
		}
		ray = Ray(si.p + kEps * wi, wi);
	}
	return L;
}

void SetTextures(MapsScene& ms, const agpt_texture* textures, int n, const agpt_material_textures* bind, int nMat) {
	ms.ts.texels.clear(); ms.ts.tex.clear(); ms.ts.matTex.clear(); ms.bind.clear();
	for (int i = 0; i < n; i++) {
		const agpt_texture& x = textures[i];
		ms.ts.texels.emplace_back(x.rgb, x.rgb + 3 * (size_t)x.width * x.height);
		ms.ts.tex.push_back({ x.width, x.height, nullptr });
	}
	for (int i = 0; i < n; i++) ms.ts.tex[i].rgb = ms.ts.texels[i].data();
	if (bind) {
		ms.bind.assign(bind, bind + nMat);
		for (int i = 0; i < nMat; i++) ms.ts.matTex.push_back(bind[i].base);
	}
}

} // namespace

extern "C" {

// The tables of a host-mirror scene (agpt_scene_tables, the map bindings at its end).
void* agpt_maps_oracle_create(const agpt_scene_tables* t) {
	auto* ms = new MapsScene();
	ms->ts.sc = (OScene*)agpt_oracle_scene_create((const agpt_oracle_tables*)t);
	SetTextures(*ms, t->textures, t->n_textures, t->material_textures, t->n_material_textures);
	return ms;
}
// replaces the textures and bindings (agpt_upload_material_textures' arguments)
void agpt_maps_oracle_set_textures(void* h, const agpt_texture* textures, int n, const agpt_material_textures* bind, int n_materials) {
	SetTextures(*(MapsScene*)h, textures, n, bind, n_materials);
}
void agpt_maps_oracle_destroy(void* h) { MapsScene* ms = (MapsScene*)h; agpt_oracle_scene_destroy(ms->ts.sc); delete ms; }
void agpt_maps_oracle_set_rr_by_bounce(void* h, int on) { ((MapsScene*)h)->ts.sc->rrByBounce = on != 0; }

// agpt_render of samples [s0, s0 + ns) into out_rgba (H x W float4 in the film's row order, added to); counters_out (6, or NULL):
// the rays the reference algorithm issues, as oracle/agpt_oracle.cpp counts them (closest, any, interior, boxes, tris, analytic)
void agpt_maps_oracle_render(void* h, int W, int H, int s0, int ns, int max_depth, int depth_arg, int threads, float* out_rgba,
		unsigned long long* counters_out) {
	const MapsScene& ms = *(MapsScene*)h;
	Counters total;
	std::mutex lock;
	ParallelRows(0, H, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int k = 0; k < ns; k++)
			for (int x = 0; x < W; x++) {
				rng.Seed((uint32_t)(y * W + x), (uint32_t)(s0 + k));
				Ray ray = CameraRay(*ms.ts.sc, W, H, x, y, rng);
				V3 clr = MapsLi(ms, ray, max_depth, depth_arg, rng, c);
				float lum = 0.212671f * clr.x + 0.715160f * clr.y + 0.072169f * clr.z;
				if (std::isnan(clr.x) || std::isnan(clr.y) || std::isnan(clr.z) || std::isinf(lum)) clr = v3(0.f);
				float* px = out_rgba + 4 * ((size_t)(H - 1 - y) * W + x);
				px[0] += clr.x; px[1] += clr.y; px[2] += clr.z;
			}
		std::lock_guard<std::mutex> g(lock);
		total.Add(c);
	});
	if (counters_out) {
		const uint64_t v[6] = { total.raysClosest, total.raysAny, total.interior, total.boxes, total.tris, total.analytic };
		for (int i = 0; i < 6; i++) counters_out[i] = v[i];
	}
}

// agpt_li_pixels: radiance of single camera paths
void agpt_maps_oracle_li_pixels(void* h, int W, int H, int n, const int* xs, const int* ys, const int* ss, int max_depth, int depth_arg, float* out_rgb) {
	const MapsScene& ms = *(MapsScene*)h;
	Counters c;
	Rng rng;
	for (int i = 0; i < n; i++) {
		rng.Seed((uint32_t)(ys[i] * W + xs[i]), (uint32_t)ss[i]);
		Ray ray = CameraRay(*ms.ts.sc, W, H, xs[i], ys[i], rng);
		V3 clr = MapsLi(ms, ray, max_depth, depth_arg, rng, c);
		out_rgb[3 * i] = clr.x; out_rgb[3 * i + 1] = clr.y; out_rgb[3 * i + 2] = clr.z;
	}
}

// agpt_render_guides with the mapped normal and the per-hit albedo (agpt.h maps step 3)
void agpt_maps_oracle_guides(void* h, int W, int H, int num_samples, int threads, float* albedo, float* normal_depth) {
	const MapsScene& ms = *(MapsScene*)h;
	const OScene& sc = *ms.ts.sc;
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
				if (SceneIntersect(sc, ray, hit, c)) {
					Surface si;
					BuildSurface(sc, ray, hit, si);
					const agpt_prim& pr = sc.prims[hit.prim];
					agpt_material m;
					if (pr.material >= 0) m = HitMaps(ms, ray0, hit, si);
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

// Per-hit rows of the closest hit of each ray (rays7 = O, D as given, tmax), 32 floats: prim (-1: miss), u, v, ng3, sn3, ss3,
// ts3 (the BSDF frame), T3, B3 (dp/du, dp/dv), roughness, metallic, lobes, diffuse_r3, spec_r03.
void agpt_maps_oracle_hit_rows(void* h, int n, const float* rays7, float* out32) {
	const MapsScene& ms = *(MapsScene*)h;
	const OScene& sc = *ms.ts.sc;
	Counters c;
	for (int i = 0; i < n; i++) {
		const float* r = rays7 + 7 * i;
		float* o = out32 + 32 * i;
		for (int k = 0; k < 32; k++) o[k] = 0.f;
		o[0] = -1.f;
		Ray ray(v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]);
		const Ray ray0 = ray;
		Hit hit;
		if (!SceneIntersect(sc, ray, hit, c)) continue;
		o[0] = (float)hit.prim;
		HitUV(sc, ray0, hit, &o[1], &o[2]);
		Surface si;
		BuildSurface(sc, ray, hit, si);
		agpt_material m = sc.mats.empty() ? agpt_material() : sc.mats[0];
		if (sc.prims[hit.prim].material >= 0) m = HitMaps(ms, ray0, hit, si);
		V3 T, B;
		HitTangents(sc, ray0, hit, &T, &B);
		const Bsdf b(si, &m);
		const V3 rows[6] = { b.ng, b.ns, b.ss, b.ts, T, B };
		for (int k = 0; k < 6; k++) { o[3 + 3 * k] = rows[k].x; o[4 + 3 * k] = rows[k].y; o[5 + 3 * k] = rows[k].z; }
		o[21] = m.roughness; o[22] = m.metallic; o[23] = (float)m.lobes;
		for (int k = 0; k < 3; k++) { o[24 + k] = m.diffuse_r[k]; o[27 + k] = m.spec_r0[k]; }
	}
}

// the triangle of each closest hit, as HitTangents forms it (world-space vertices for instances): out15 = v0 v1 v2 uv0 uv1 uv2,
// all NaN where the ray misses or hits a sphere or plane
void agpt_maps_oracle_hit_triangle(void* h, int n, const float* rays7, float* out15) {
	const MapsScene& ms = *(MapsScene*)h;
	const OScene& sc = *ms.ts.sc;
	Counters c;
	for (int i = 0; i < n; i++) {
		const float* r = rays7 + 7 * i;
		float* o = out15 + 15 * i;
		for (int k = 0; k < 15; k++) o[k] = std::nanf("");
		Ray ray(v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]);
		Hit hit;
		if (!SceneIntersect(sc, ray, hit, c)) continue;
		const agpt_prim& pr = sc.prims[hit.prim];
		if (pr.type == AGPT_PRIM_SPHERE || pr.type == AGPT_PRIM_PLANE) continue;
		const agpt_instance* in = pr.type == AGPT_PRIM_INSTANCE ? &sc.instances[pr.payload] : nullptr;
		const Mesh& m = sc.meshes[in ? in->mesh : pr.payload];
		const float* p = &m.verts[12 * (size_t)hit.slot];
		V3 v[3] = { v3(p), v3(p + 4), v3(p + 8) };
		for (int k = 0; k < 3; k++) {
			if (in) v[k] = XformPoint(in->object_to_world, v[k]);
			o[3 * k] = v[k].x; o[3 * k + 1] = v[k].y; o[3 * k + 2] = v[k].z;
		}
		TriangleUVs(m, hit.slot, o + 9);
	}
}

// single rules, for the CPU tests.  frame: in12 = N3 T3 B3 texel3, scale; out7 = sn3 sdpdu3 changed (1 / 0), the surface
// given as sn = N, sdpdu = T.
void agpt_maps_oracle_frame(int n, const float* in12, const float* scale, float* out7) {
	for (int i = 0; i < n; i++) {
		const float* p = in12 + 12 * i;
		Surface s;
		s.p = v3(0.f); s.n = v3(p); s.sn = v3(p); s.sdpdu = v3(p + 3);
		const bool changed = NormalMapFrame(v3(p + 9), scale[i], v3(p + 3), v3(p + 6), s);
		float* o = out7 + 7 * i;
		o[0] = s.sn.x; o[1] = s.sn.y; o[2] = s.sn.z; o[3] = s.sdpdu.x; o[4] = s.sdpdu.y; o[5] = s.sdpdu.z; o[6] = changed ? 1.f : 0.f;
	}
}
// material: the record derived from rec with base colour C and roughness-metallic texel c
void agpt_maps_oracle_material(const agpt_material* rec, const float* C, const float* c, agpt_material* out) {
	*out = DeriveMaterial(*rec, v3(C), v3(c));
}

} // extern "C"
