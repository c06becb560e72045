// statements/agpt_texture_oracle.cpp -- TEST INFRASTRUCTURE, not product code.
//
// EXTENSION (include/agpt.h agpt_upload_textures): the CPU statement of image textures on the base colour of Disney
// materials, the one the GPU path is checked against.  The reference has one colour per material; what a textured hit means
// is defined in agpt.h.
//
// The oracle (oracle/agpt_oracle.cpp, pinned bit for bit to the reference) is compiled into this translation unit unchanged
// and reused as it is: tables, camera ray, Scene::Intersect, the SurfaceInteraction of a hit, the BSDF and EstimateDirect.
// New here: the uv rules, the fdlibm atan2f the device states the sphere's u with, the lookup, the per-hit material, and the
// path loop and guide record that use them (PathTracer::Li as the oracle states it, with the hit's material replaced).
// Built by __graft_entry__.build() into statements/libagpt_texture_oracle.so with the oracle's flags (-O2, no FMA contraction).
#include "../oracle/agpt_oracle.cpp"
#include "agpt_host.h"

namespace {

inline float AsFloat(int i) { float f; memcpy(&f, &i, 4); return f; }
inline int AsInt(float f) { int i; memcpy(&i, &f, 4); return i; }

// Sun fdlibm s_atanf.c / e_atan2f.c in float, as agpt_device.cuh ratanfT / ratan2T state them
float FdAtanf(float x) {
	const float atanhi[4] = { 4.6364760399e-01f, 7.8539812565e-01f, 9.8279368877e-01f, 1.5707962513e+00f };
	const float atanlo[4] = { 5.0121582440e-09f, 3.7748947079e-08f, 3.4473217170e-08f, 7.5497894159e-08f };
	const float aT[11] = { 3.3333334327e-01f, -2.0000000298e-01f, 1.4285714924e-01f, -1.1111110449e-01f, 9.0908870101e-02f,
		-7.6918758452e-02f, 6.6610731184e-02f, -5.8335702866e-02f, 4.9768779427e-02f, -3.6531571299e-02f, 1.6285819933e-02f };
	int hx = AsInt(x), ix = hx & 0x7fffffff, id;
	if (ix >= 0x4c800000) {
		if (ix > 0x7f800000) return x + x;
		return hx > 0 ? atanhi[3] + atanlo[3] : -atanhi[3] - atanlo[3];
	}
	if (ix < 0x3ee00000) {
		if (ix < 0x31000000) return x;
		id = -1;
	}
	else {
		x = std::fabs(x);
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
float FdAtan2f(float y, float x) {
	const float tiny = 1.0e-30f, pi_o_4 = 7.8539818525e-01f, pi_o_2 = 1.5707963705e+00f, pi = 3.1415927410e+00f, pi_lo = -8.7422776573e-08f;
	int hx = AsInt(x), ix = hx & 0x7fffffff, hy = AsInt(y), iy = hy & 0x7fffffff;
	if (ix > 0x7f800000 || iy > 0x7f800000) return x + y;
	if (hx == 0x3f800000) return FdAtanf(y);
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
	else z = FdAtanf(std::fabs(y / x));
	switch (m) {
	case 0: return z;
	case 1: return -z;
	case 2: return pi - (z - pi_lo);
	default: return (z - pi_lo) - pi;
	}
}

struct Tex {
	int w, h;
	const float* rgb;
};

inline int Wrap(int x, int n) { return x < 0 ? x + n : x >= n ? x - n : x; }
V3 Lookup(const Tex& t, float u, float v) {
	u = std::isfinite(u) ? u - std::floor(u) : 0.f;
	v = std::isfinite(v) ? v - std::floor(v) : 0.f;
	const float s = u * (float)t.w - 0.5f, tt = v * (float)t.h - 0.5f;
	const float fs = std::floor(s), ft = std::floor(tt);
	const int x0 = Wrap((int)fs, t.w), x1 = Wrap((int)fs + 1, t.w), y0 = Wrap((int)ft, t.h), y1 = Wrap((int)ft + 1, t.h);
	const float fx = s - fs, fy = tt - ft;
	auto T = [&](int x, int y) { return v3(t.rgb + 3 * ((size_t)y * t.w + x)); };
	const V3 t00 = T(x0, y0), t10 = T(x1, y0), t01 = T(x0, y1), t11 = T(x1, y1);
	const V3 a = t00 + fx * (t10 - t00), b = t01 + fx * (t11 - t01);
	return a + fy * (b - a);
}

// the surface uv of a hit (agpt.h, step 1), from the same quantities BuildSurface forms
void HitUV(const OScene& sc, const Ray& ray, const Hit& h, float* u, float* v) {
	const agpt_prim& pr = sc.prims[h.prim];
	if (pr.type == AGPT_PRIM_SPHERE) {
		const agpt_sphere& sp = sc.spheres[pr.payload];
		V3 p = ray.O + h.t * ray.D;
		V3 pHit = p - v3(sp.center);
		if (pHit.x == 0 && pHit.y == 0) pHit.x = kEps * sp.r;
		float theta = std::acos(tclamp(pHit.z / sp.r, -1.f, 1.f));
		float phi = FdAtan2f(pHit.y, pHit.x);
		if (phi < 0) phi = phi + kTwoPi;
		*u = phi / kTwoPi; *v = theta / kPi;
	}
	else if (pr.type == AGPT_PRIM_PLANE) {
		const agpt_plane& pl = sc.planes[pr.payload];
		V3 p = ray.O + h.t * ray.D;
		*u = ((p.x - pl.o[0]) / pl.half_x + 1) * 0.5f;
		*v = ((p.z - pl.o[2]) / pl.half_z + 1) * 0.5f;
	}
	else {
		const Mesh& m = MeshOfPrim(sc, pr);
		float uv[6];
		TriangleUVs(m, h.slot, uv);
		float b0 = 1.f - h.b1 - h.b2;
		*u = (b0 * uv[0] + h.b1 * uv[2]) + h.b2 * uv[4];
		*v = (b0 * uv[1] + h.b1 * uv[3]) + h.b2 * uv[5];
	}
}

struct TexScene {
	OScene* sc;
	std::vector<std::vector<float>> texels;
	std::vector<Tex> tex;
	std::vector<int32_t> matTex;
};

// the material record of a hit (agpt.h, step 3): a textured Disney material's colours come from the texture value
agpt_material HitMaterial(const TexScene& ts, const Ray& ray, const Hit& h) {
	const agpt_prim& pr = ts.sc->prims[h.prim];
	agpt_material m = ts.sc->mats[pr.material];
	const int t = pr.material < (int)ts.matTex.size() ? ts.matTex[pr.material] : -1;
	if (t < 0) return m;
	float u, v;
	HitUV(*ts.sc, ray, h, &u, &v);
	const V3 c = Lookup(ts.tex[t], u, v);
	const float dw = (1 - m.metallic) * (1 - 0.f);
	const V3 d = dw > 0 ? dw * c : v3(0.f);
	const float r0 = ((m.eta - 1) * (m.eta - 1)) / ((m.eta + 1) * (m.eta + 1));
	const V3 s = Lerp(m.metallic, v3(r0), c);
	m.diffuse_r[0] = d.x; m.diffuse_r[1] = d.y; m.diffuse_r[2] = d.z;
	m.spec_r0[0] = s.x; m.spec_r0[1] = s.y; m.spec_r0[2] = s.z;
	return m;
}

// PathTracer::Li as oracle/agpt_oracle.cpp states it, each hit shaded with HitMaterial
V3 TexLi(const TexScene& ts, Ray ray, int maxDepth, int depthArg, Rng& rng, Counters& c) {
	const OScene& sc = *ts.sc;
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
		if (pr.material < 0) {
			ray = Ray(si.p + kEps * ray.D, ray.D);
			bounces--;
			continue;
		}
		const agpt_material mat = HitMaterial(ts, ray, h);
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

} // namespace

extern "C" {

// The tables of a host-mirror scene (agpt_scene_tables: the oracle's tables followed by the texture fields).
void* agpt_texture_oracle_create(const agpt_scene_tables* t) {
	auto* ts = new TexScene();
	ts->sc = (OScene*)agpt_oracle_scene_create((const agpt_oracle_tables*)t);
	for (int i = 0; i < t->n_textures; i++) {
		const agpt_texture& x = t->textures[i];
		ts->texels.emplace_back(x.rgb, x.rgb + 3 * (size_t)x.width * x.height);
		ts->tex.push_back({ x.width, x.height, ts->texels.back().data() });
	}
	for (int i = 0; i < (int)ts->tex.size(); i++) ts->tex[i].rgb = ts->texels[i].data();
	if (t->material_texture) ts->matTex.assign(t->material_texture, t->material_texture + t->n_material_texture);
	return ts;
}
void agpt_texture_oracle_destroy(void* h) { TexScene* ts = (TexScene*)h; agpt_oracle_scene_destroy(ts->sc); delete ts; }
void agpt_texture_oracle_set_rr_by_bounce(void* h, int on) { ((TexScene*)h)->sc->rrByBounce = on != 0; }

// agpt_render of samples [s0, s0 + ns) into out_rgba (H x W float4 in the film's row order, added to)
void agpt_texture_oracle_render(void* h, int W, int H, int s0, int ns, int max_depth, int depth_arg, int threads, float* out_rgba) {
	const TexScene& ts = *(TexScene*)h;
	ParallelRows(0, H, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int k = 0; k < ns; k++)
			for (int x = 0; x < W; x++) {
				rng.Seed((uint32_t)(y * W + x), (uint32_t)(s0 + k));
				Ray ray = CameraRay(*ts.sc, W, H, x, y, rng);
				V3 clr = TexLi(ts, ray, max_depth, depth_arg, rng, c);
				float lum = 0.212671f * clr.x + 0.715160f * clr.y + 0.072169f * clr.z;
				if (std::isnan(clr.x) || std::isnan(clr.y) || std::isnan(clr.z) || std::isinf(lum)) clr = v3(0.f);
				float* px = out_rgba + 4 * ((size_t)(H - 1 - y) * W + x);
				px[0] += clr.x; px[1] += clr.y; px[2] += clr.z;
			}
	});
}

// agpt_li_pixels: radiance of single camera paths
void agpt_texture_oracle_li_pixels(void* h, int W, int H, int n, const int* xs, const int* ys, const int* ss, int max_depth, int depth_arg, float* out_rgb) {
	const TexScene& ts = *(TexScene*)h;
	Counters c;
	Rng rng;
	for (int i = 0; i < n; i++) {
		rng.Seed((uint32_t)(ys[i] * W + xs[i]), (uint32_t)ss[i]);
		Ray ray = CameraRay(*ts.sc, W, H, xs[i], ys[i], rng);
		V3 clr = TexLi(ts, ray, max_depth, depth_arg, rng, c);
		out_rgb[3 * i] = clr.x; out_rgb[3 * i + 1] = clr.y; out_rgb[3 * i + 2] = clr.z;
	}
}

// agpt_render_guides (oracle/agpt_guides_oracle.cpp's record, with the textured albedo of agpt.h step 4)
void agpt_texture_oracle_guides(void* h, int W, int H, int num_samples, int threads, float* albedo, float* normal_depth) {
	const TexScene& ts = *(TexScene*)h;
	const OScene& sc = *ts.sc;
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
					nrm = dot(si.sn, D) > 0.f ? -si.sn : si.sn;
					const agpt_prim& pr = sc.prims[hit.prim];
					if (pr.material >= 0) {
						const agpt_material m = HitMaterial(ts, ray0, hit);
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

// single functions of the statement, for the CPU tests
void agpt_texture_oracle_lookup(int W, int H, const float* rgb, int n, const float* uv, float* out_rgb) {
	const Tex t = { W, H, rgb };
	for (int i = 0; i < n; i++) { V3 c = Lookup(t, uv[2 * i], uv[2 * i + 1]); out_rgb[3 * i] = c.x; out_rgb[3 * i + 1] = c.y; out_rgb[3 * i + 2] = c.z; }
}
void agpt_texture_oracle_atan2(int n, const float* y, const float* x, float* out) { for (int i = 0; i < n; i++) out[i] = FdAtan2f(y[i], x[i]); }
// uv of the closest hit of each ray (rays7 = O, D as given, tmax) on the scene: out3 = u, v, prim (-1: miss)
void agpt_texture_oracle_hit_uv(void* h, int n, const float* rays7, float* out3) {
	const TexScene& ts = *(TexScene*)h;
	Counters c;
	for (int i = 0; i < n; i++) {
		const float* r = rays7 + 7 * i;
		Ray ray(v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]);
		const Ray ray0 = ray;
		Hit hit;
		out3[3 * i] = out3[3 * i + 1] = 0.f; out3[3 * i + 2] = -1.f;
		if (SceneIntersect(*ts.sc, ray, hit, c)) { HitUV(*ts.sc, ray0, hit, &out3[3 * i], &out3[3 * i + 1]); out3[3 * i + 2] = (float)hit.prim; }
	}
}

} // extern "C"
