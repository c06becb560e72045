// statements/agpt_emission_oracle.cpp -- TEST INFRASTRUCTURE, not product code.
//
// EXTENSION (include/agpt.h agpt_upload_emission): the CPU statement of emissive materials, the one the GPU path is checked
// against.  The reference has no emissive materials; what one adds to Li is defined in agpt.h.
//
// The alpha-mask statement (statements/agpt_alpha_oracle.cpp, with the maps and texture statements and the oracle under it) is
// compiled into this translation unit unchanged.  Emission adds one term to the path loop, so only AlphaLi is restated here, as
// EmissionLi; the scene intersection (masks included), direct lighting, surfaces, uvs and the bilinear lookup are the code below
// this file, used as it is.  The path ray at bounces == max_depth is traced on the CPU already.  With no emitting row
// EmissionLi computes what AlphaLi computes.  Built by __graft_entry__.build() into statements/libagpt_emission_oracle.so (-O2,
// no FMA contraction).
#include "agpt_alpha_oracle.cpp"

namespace {

struct EmissionScene {
	AlphaScene as;                                   // scene, textures, map bindings and alpha masks
	std::vector<agpt_emission> rows;                 // per material; empty: nothing emits
};

inline bool Emits(const agpt_emission& e) { return e.factor[0] > 0.f || e.factor[1] > 0.f || e.factor[2] > 0.f; }

// agpt.h agpt_upload_emission: E of closest hit h of `ray` (the ray as traced: O, D), or false when its material does not emit
bool EmissionOf(const EmissionScene& es, const Ray& ray, const Hit& h, V3* E) {
	const OScene& sc = *es.as.ms.ts.sc;
	const int mat = sc.prims[h.prim].material;
	if (mat < 0 || mat >= (int)es.rows.size() || !Emits(es.rows[mat])) return false;
	const agpt_emission& e = es.rows[mat];
	*E = v3(e.factor[0], e.factor[1], e.factor[2]);
	if (e.texture >= 0) {
		float u = 0, v = 0;
		HitUV(sc, ray, h, &u, &v);
		*E = *E * Lookup(es.as.ms.ts.tex[e.texture], u, v);
	}
	return true;
}

// the alpha statement's AlphaLi with the one term of emissive materials
V3 EmissionLi(const EmissionScene& es, Ray ray, int maxDepth, int depthArg, Rng& rng, Counters& c) {
	const AlphaScene& as = es.as;
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
		V3 E;
		if (found && EmissionOf(es, ray0, h, &E)) L += beta * E;      // emissive materials: every hit, whatever specularBounce says
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

void SetEmission(EmissionScene& es, const agpt_emission* rows, int n) {
	es.rows.clear();
	if (rows) es.rows.assign(rows, rows + n);
}

} // namespace

extern "C" {

// The tables of a host-mirror scene (agpt_scene_tables), its alpha masks (agpt_host_scene_alpha_masks) and its emission rows
// (agpt_host_scene_emission); NULL, 0: none
void* agpt_emission_oracle_create(const agpt_scene_tables* t, const agpt_alpha_mask* masks, int n_masks, const agpt_emission* rows, int n_rows) {
	auto* es = new EmissionScene();
	es->as.ms.ts.sc = (OScene*)agpt_oracle_scene_create((const agpt_oracle_tables*)t);
	SetTextures(es->as.ms, t->textures, t->n_textures, t->material_textures, t->n_material_textures);
	SetMasks(es->as, masks, n_masks);
	SetEmission(*es, rows, n_rows);
	return es;
}
// replaces the textures and bindings (agpt_upload_material_textures' arguments); like the device, this clears the masks and the
// emission rows
void agpt_emission_oracle_set_textures(void* h, const agpt_texture* textures, int n, const agpt_material_textures* bind, int n_materials) {
	EmissionScene& es = *(EmissionScene*)h;
	SetTextures(es.as.ms, textures, n, bind, n_materials);
	es.as.masks.clear();
	es.rows.clear();
}
// replaces the masks (agpt_upload_alpha_masks' arguments)
void agpt_emission_oracle_set_masks(void* h, const agpt_alpha_mask* masks, int n) { SetMasks(((EmissionScene*)h)->as, masks, n); }
// replaces the emission rows (agpt_upload_emission's arguments)
void agpt_emission_oracle_set_emission(void* h, const agpt_emission* rows, int n) { SetEmission(*(EmissionScene*)h, rows, n); }
void agpt_emission_oracle_destroy(void* h) { EmissionScene* es = (EmissionScene*)h; agpt_oracle_scene_destroy(es->as.ms.ts.sc); delete es; }
void agpt_emission_oracle_set_rr_by_bounce(void* h, int on) { ((EmissionScene*)h)->as.ms.ts.sc->rrByBounce = on != 0; }

// agpt_render of samples [s0, s0 + ns) into out_rgba (added to); counters_out (6, or NULL): closest, any, interior, boxes, tris, analytic
void agpt_emission_oracle_render(void* h, int W, int H, int s0, int ns, int max_depth, int depth_arg, int threads, float* out_rgba,
		unsigned long long* counters_out) {
	const EmissionScene& es = *(EmissionScene*)h;
	Counters total;
	std::mutex lock;
	ParallelRows(0, H, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int k = 0; k < ns; k++)
			for (int x = 0; x < W; x++) {
				rng.Seed((uint32_t)(y * W + x), (uint32_t)(s0 + k));
				Ray ray = CameraRay(*es.as.ms.ts.sc, W, H, x, y, rng);
				V3 clr = EmissionLi(es, ray, max_depth, depth_arg, rng, c);
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
void agpt_emission_oracle_li_pixels(void* h, int W, int H, int n, const int* xs, const int* ys, const int* ss, int max_depth, int depth_arg, float* out_rgb) {
	const EmissionScene& es = *(EmissionScene*)h;
	Counters c;
	Rng rng;
	for (int i = 0; i < n; i++) {
		rng.Seed((uint32_t)(ys[i] * W + xs[i]), (uint32_t)ss[i]);
		Ray ray = CameraRay(*es.as.ms.ts.sc, W, H, xs[i], ys[i], rng);
		V3 clr = EmissionLi(es, ray, max_depth, depth_arg, rng, c);
		out_rgb[3 * i] = clr.x; out_rgb[3 * i + 1] = clr.y; out_rgb[3 * i + 2] = clr.z;
	}
}

// agpt_li_rays: radiance of caller rays (rays7 = O, D normalised like the Ray ctor, tmax), path i drawing from xorshift32 state rng_states[i]
void agpt_emission_oracle_li_rays(void* h, int n, const float* rays7, const uint32_t* rng_states, int max_depth, int depth_arg, float* out_rgb) {
	const EmissionScene& es = *(EmissionScene*)h;
	Counters c;
	Rng rng;
	for (int i = 0; i < n; i++) {
		const float* r = rays7 + 7 * i;
		Ray ray(v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]);
		rng.s = rng_states[i]; rng.draws = 0;
		V3 clr = EmissionLi(es, ray, max_depth, depth_arg, rng, c);
		out_rgb[3 * i] = clr.x; out_rgb[3 * i + 1] = clr.y; out_rgb[3 * i + 2] = clr.z;
	}
}

} // extern "C"
