// config_scenes.h -- the five BASELINE.json configurations as procedural scenes.
//
// This file is written ONLY against the reference's public scene-building API
// (/root/reference/myapp.cpp:13-114 shows the style): Scene, Sphere, Plane, TriangleMesh,
// BVHTriMesh, index_type, DisneyMaterial::Make, MirrorMaterial::Make, UniformInfiniteLight,
// Scene::addAreaLight, CameraDesc.  It is compiled twice from this single source:
//   * against the reference's own headers  -> oracle/_ref (the CPU oracle), and
//   * against ag-pathtracer_b200/host/*.h  -> the B200 drop-in,
// which is the compile-time proof that the host mirror keeps the reference's API surface.
// The includer must have the API in scope before including this header.
//
// Scene definitions follow SURVEY.md section 8d; all assets are procedural (the reference's
// own scenes need D://models/bunny.obj and small_workshop_1k.hdr, which are not in the repo).
#pragma once

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <memory>
#include <utility>
#include <vector>

namespace agpt_scenes {

// Film/integrator defaults that go with each configuration (BASELINE.json "configs").
struct ConfigDefaults {
	int width, height, spp, max_depth, depth_arg;
	const char* name;
};

inline ConfigDefaults Defaults(int config) {
	switch (config) {
	case 1: return { 640, 360, 64, 5, 0, "cfg1_analytic_640x360_64spp_depth5" };
	case 2: return { 1920, 1080, 16, 1, 0, "cfg2_icosphere1p31M_direct_1080p_16spp" };
	case 3: return { 1920, 1080, 256, 8, 0, "cfg3_disney_multimaterial_1p31M_1080p_256spp_depth8" };
	case 4: return { 3840, 2160, 1024, 8, 0, "cfg4_8xicosphere_10p5M_4k_1024spp_depth8" };
	case 5: return { 1920, 1080, 64, 16, 4, "cfg5_closed_box_incoherent_1080p_depth16_rr" };
	case 6: return { 320, 180, 16, 5, 0, "cfg6_test_thin_lens_plain_mesh_multi_tri_leaves" };
	case 7: return { 400, 400, 64, 5, 0, "cfg7_reference_default_scene_envmap_400x400" };
	case 8: return { 640, 360, 16, 6, 4, "cfg8_test_degenerate_triangles_deep_tree_overflowing_light" };
	case 9: return { 3840, 2160, 1024, 8, 0, "cfg9_ext_cfg4_with_true_instances_one_mesh_8_placements" };
	case 10: return { 1920, 1080, 64, 16, 0, "cfg10_ext_cfg5_rough_glass_rr_by_bounce" };
	case 11: return { 1920, 1080, 64, 16, 4, "cfg11_ext_cfg5_sampled_panel_plane_and_mesh_lights" };
	case 12: return { 480, 270, 16, 8, 0, "cfg12_ext_procedural_image_textures" };
	case 13: return { 480, 270, 16, 8, 0, "cfg13_ext_procedural_roughness_metallic_and_normal_maps" };
	case 14: return { 480, 270, 16, 8, 0, "cfg14_ext_alpha_masked_cutouts" };
	case 15: return { 480, 270, 16, 8, 0, "cfg15_ext_emissive_materials" };
	default: return { 0, 0, 0, 0, 0, "unknown" };
	}
}

// ---------------------------------------------------------------------------------------
// Unit icosphere: icosahedron subdivided `level` times with shared vertices.  20*4^level
// triangles, 10*4^level+2 vertices.  Plain float arithmetic so both builds produce the same
// bits.  Per-vertex normals = unit positions; no texture coordinates (the reference then
// uses its default per-triangle uvs, trianglemesh.cpp:52-56).
// ---------------------------------------------------------------------------------------
struct IcoData {
	std::vector<float> pos;   // xyz per vertex, unit length
	std::vector<int> tri;     // 3 indices per triangle
};

inline void IcoNormalize(float* p) {
	float inv = 1.0f / std::sqrt(p[0] * p[0] + p[1] * p[1] + p[2] * p[2]);
	p[0] *= inv; p[1] *= inv; p[2] *= inv;
}

inline IcoData MakeIcoData(int level) {
	IcoData d;
	const float g = 1.6180339887498949f;
	const float base[12][3] = {
		{ -1, g, 0 }, { 1, g, 0 }, { -1, -g, 0 }, { 1, -g, 0 },
		{ 0, -1, g }, { 0, 1, g }, { 0, -1, -g }, { 0, 1, -g },
		{ g, 0, -1 }, { g, 0, 1 }, { -g, 0, -1 }, { -g, 0, 1 } };
	const int faces[20][3] = {
		{ 0, 11, 5 }, { 0, 5, 1 }, { 0, 1, 7 }, { 0, 7, 10 }, { 0, 10, 11 },
		{ 1, 5, 9 }, { 5, 11, 4 }, { 11, 10, 2 }, { 10, 7, 6 }, { 7, 1, 8 },
		{ 3, 9, 4 }, { 3, 4, 2 }, { 3, 2, 6 }, { 3, 6, 8 }, { 3, 8, 9 },
		{ 4, 9, 5 }, { 2, 4, 11 }, { 6, 2, 10 }, { 8, 6, 7 }, { 9, 8, 1 } };
	for (auto& b : base) {
		float p[3] = { b[0], b[1], b[2] };
		IcoNormalize(p);
		d.pos.insert(d.pos.end(), p, p + 3);
	}
	for (auto& f : faces) d.tri.insert(d.tri.end(), f, f + 3);

	for (int l = 0; l < level; l++) {
		std::map<std::pair<int, int>, int> midpoint;
		auto mid = [&](int a, int b) {
			std::pair<int, int> key(a < b ? a : b, a < b ? b : a);
			auto it = midpoint.find(key);
			if (it != midpoint.end()) return it->second;
			float p[3] = { (d.pos[3 * a] + d.pos[3 * b]) * 0.5f,
				(d.pos[3 * a + 1] + d.pos[3 * b + 1]) * 0.5f,
				(d.pos[3 * a + 2] + d.pos[3 * b + 2]) * 0.5f };
			IcoNormalize(p);
			int idx = (int)(d.pos.size() / 3);
			d.pos.insert(d.pos.end(), p, p + 3);
			midpoint[key] = idx;
			return idx;
		};
		std::vector<int> next;
		next.reserve(d.tri.size() * 4);
		for (size_t t = 0; t < d.tri.size(); t += 3) {
			int a = d.tri[t], b = d.tri[t + 1], c = d.tri[t + 2];
			int ab = mid(a, b), bc = mid(b, c), ca = mid(c, a);
			const int sub[12] = { a, ab, ca, b, bc, ab, c, ca, bc, ab, bc, ca };
			next.insert(next.end(), sub, sub + 12);
		}
		d.tri.swap(next);
	}
	return d;
}

// Icosphere as a reference TriangleMesh with baked world-space vertices (the reference has
// no instancing or per-primitive transforms, scene.h:5-28).
inline std::shared_ptr<TriangleMesh> MakeIcosphere(int level, const float3& center, float radius,
		std::shared_ptr<Material> mat) {
	IcoData d = MakeIcoData(level);
	std::vector<float3> vertices, normals;
	std::vector<float2> texcoords;
	std::vector<index_type> indices;
	size_t nv = d.pos.size() / 3;
	vertices.reserve(nv);
	normals.reserve(nv);
	for (size_t i = 0; i < nv; i++) {
		float3 n(d.pos[3 * i], d.pos[3 * i + 1], d.pos[3 * i + 2]);
		normals.push_back(n);
		vertices.push_back(float3(center.x + radius * n.x, center.y + radius * n.y, center.z + radius * n.z));
	}
	indices.reserve(d.tri.size());
	for (int v : d.tri) indices.push_back(index_type(v));
	return std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, mat);
}

// Axis-aligned room [lo,hi] as 12 inward-facing triangles with per-face normals.
inline std::shared_ptr<TriangleMesh> MakeRoom(const float3& lo, const float3& hi, std::shared_ptr<Material> mat) {
	std::vector<float3> vertices, normals;
	std::vector<float2> texcoords;
	std::vector<index_type> indices;
	auto quad = [&](float3 a, float3 b, float3 c, float3 d, float3 n) {
		int base = (int)vertices.size();
		vertices.push_back(a); vertices.push_back(b); vertices.push_back(c); vertices.push_back(d);
		for (int i = 0; i < 4; i++) normals.push_back(n);
		texcoords.push_back(float2(0, 0)); texcoords.push_back(float2(1, 0));
		texcoords.push_back(float2(1, 1)); texcoords.push_back(float2(0, 1));
		const int order[6] = { 0, 1, 2, 0, 2, 3 };
		for (int o : order) indices.push_back(index_type(base + o));
	};
	quad(float3(lo.x, lo.y, lo.z), float3(hi.x, lo.y, lo.z), float3(hi.x, lo.y, hi.z), float3(lo.x, lo.y, hi.z), float3(0, 1, 0));   // floor
	quad(float3(lo.x, hi.y, lo.z), float3(lo.x, hi.y, hi.z), float3(hi.x, hi.y, hi.z), float3(hi.x, hi.y, lo.z), float3(0, -1, 0));  // ceiling
	quad(float3(lo.x, lo.y, lo.z), float3(lo.x, lo.y, hi.z), float3(lo.x, hi.y, hi.z), float3(lo.x, hi.y, lo.z), float3(1, 0, 0));   // -x wall
	quad(float3(hi.x, lo.y, lo.z), float3(hi.x, hi.y, lo.z), float3(hi.x, hi.y, hi.z), float3(hi.x, lo.y, hi.z), float3(-1, 0, 0));  // +x wall
	quad(float3(lo.x, lo.y, hi.z), float3(hi.x, lo.y, hi.z), float3(hi.x, hi.y, hi.z), float3(lo.x, hi.y, hi.z), float3(0, 0, -1));  // back wall
	quad(float3(lo.x, lo.y, lo.z), float3(lo.x, hi.y, lo.z), float3(hi.x, hi.y, lo.z), float3(hi.x, lo.y, lo.z), float3(0, 0, 1));   // front wall
	return std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, mat);
}

inline float3 WarmWhite(float scale) { return float3(1.f, .941f, .914f) * scale; }

// cfg 1: reference-default-style analytic scene (plane + diffuse / mirror / gold spheres,
// a small bright sphere standing in for the point light the reference lacks, uniform sky).
inline void BuildConfig1(Scene* scene) {
	auto grey = DisneyMaterial::Make(float3(.5f, .5f, .5f), 1.f, 0.f);
	auto red = DisneyMaterial::Make(float3(.7f, .1f, .1f), .5f, 0.f);
	auto mirror = MirrorMaterial::Make(float3(.9f, .9f, .9f));
	auto gold = DisneyMaterial::Make(float3(0.944f, 0.776f, 0.373f), .3f, 1.f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -1, 0), float2(40, 40), grey));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(-2.2f, 0, 0), 1.f, red));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(0, 0, 0), 1.f, mirror));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(2.2f, 0, 0), 1.f, gold));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 6, -3), .25f, nullptr), WarmWhite(400));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.1f, .12f, .15f)));
	scene->camera.lookfrom = float3(0, 1.5f, -8);
	scene->camera.lookat = float3(0, 0, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 35;
	scene->camera.aperture = 0;
}

// cfg 2: one subdivided icosphere (level 8 = 1,310,720 triangles) in a BVHTriMesh, one
// sphere area light, direct lighting only (PathTracer(1)).
inline void BuildConfig2(Scene* scene, int level) {
	auto clay = DisneyMaterial::Make(float3(.8f, .3f, .2f), .5f, 0.f);
	auto mesh = MakeIcosphere(level, float3(0, 0, 0), 1.f, clay);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(mesh, clay, 1));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 25, -20), 1.f, nullptr), WarmWhite(200));
	scene->camera.lookfrom = float3(0, 0, -3.2f);
	scene->camera.lookat = float3(0, 0, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 45;
	scene->camera.aperture = 0;
}

// cfg 3: Disney multi-material scene: backdrop mesh, 5x5 analytic spheres sweeping
// roughness x metallic, four icospheres (level 7 -> 4 x 327,680 = 1,310,720 triangles),
// the three sphere area lights and the uniform sky of the reference's BunnyScene
// (myapp.cpp:36-51), thin-lens camera off.
inline void BuildConfig3(Scene* scene, int level) {
	const int palette[25] = {
		0xf19a91, 0xedd0ca, 0xf3b8a8, 0xf9ece6, 0xf6e7d0, 0xf5deac, 0xeecf74, 0x9ed5d8, 0x9ba6ac,
		0xaebdc4, 0xb9ddf3, 0x87abc5, 0xcbceb1, 0xf7f7f7, 0xc4ac64, 0xe2f4f6, 0xd2e4e6, 0xbfdcda,
		0x69bab3, 0x88cabc, 0xcdd1d4, 0xe6e5ea, 0x33455b, 0x5b6268, 0x778592 };
	const float rough[5] = { .1f, .25f, .5f, .75f, 1.f };
	const float metal[3] = { 0.f, .5f, 1.f };

	auto floor = DisneyMaterial::Make(hex2lin(0xcbceb1), 1.f, 0.f);
	auto backdrop = TriangleMesh::CreateBackdrop(make_float3(0, -1, 20), float3(40, 20, 40), 7.5f, 32, floor);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(backdrop, floor, 1));
	// the cfg-1 floor, kept just below the backdrop's own floor so no two surfaces coincide
	auto grey = DisneyMaterial::Make(float3(.5f, .5f, .5f), 1.f, 0.f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -1.05f, 0), float2(120, 120), grey));

	for (int i = 0; i < 25; i++) {
		int col = i % 5, row = i / 5;
		auto m = DisneyMaterial::Make(hex2lin(palette[i]), rough[col], metal[row % 3]);
		float3 c(-3.f + 1.5f * col, -1.f + .5f, -4.f + 1.5f * row);
		scene->primitives.push_back(std::make_shared<Sphere>(c, .5f, m));
	}
	auto gold = DisneyMaterial::Make(float3(0.944f, 0.776f, 0.373f), .2f, 1.f);
	auto red = DisneyMaterial::Make(rgb2lin(float3(.529f, .145f, .039f)), .25f, 0.f);
	auto cute = DisneyMaterial::Make(hex2lin(0xc5b5d2), .25f, 0.f);
	auto alu = DisneyMaterial::Make(float3(0.912f, 0.914f, 0.920f), .5f, .5f);
	struct { float3 c; float r; std::shared_ptr<Material> m; } balls[4] = {
		{ float3(-6.f, .5f, 1.f), 1.5f, gold }, { float3(6.f, .5f, 1.f), 1.5f, red },
		{ float3(-3.f, 1.f, 6.f), 2.f, cute }, { float3(3.f, 1.f, 6.f), 2.f, alu } };
	for (auto& b : balls) {
		auto mesh = MakeIcosphere(level, b.c, b.r, b.m);
		scene->primitives.push_back(std::make_shared<BVHTriMesh>(mesh, b.m, 1));
	}
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 25, -20), 1.f, nullptr), WarmWhite(200));   // key
	scene->addAreaLight(std::make_shared<Sphere>(float3(10, 25, -20), 1.f, nullptr), WarmWhite(50));   // fill
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 20, 10), 5.f, nullptr), WarmWhite(1));      // back
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.4f, .45f, .5f)));
	scene->camera.lookfrom = float3(0, 5.f, -14.f);
	scene->camera.lookat = float3(0, 0, 1.f);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 35;
	scene->camera.aperture = 0;
}

// cfg 4: eight icospheres (level 8 -> 10,485,760 triangles) as eight separate BVHTriMesh
// objects with baked translations on a 2x2x2 lattice ("instances" in the only form the
// reference can express, SURVEY D5), floor plane, two sphere lights.
inline void BuildConfig4(Scene* scene, int level) {
	auto grey = DisneyMaterial::Make(float3(.5f, .5f, .5f), 1.f, 0.f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -2.5f, 0), float2(60, 60), grey));
	const int palette[8] = { 0xf19a91, 0x9ed5d8, 0xeecf74, 0x87abc5, 0xc4ac64, 0x69bab3, 0xe57a82, 0xf7f7f7 };
	for (int i = 0; i < 8; i++) {
		float3 c(((i & 1) ? 1.25f : -1.25f), ((i & 2) ? 1.25f : -1.25f), ((i & 4) ? 1.25f : -1.25f));
		auto m = DisneyMaterial::Make(hex2lin(palette[i]), .2f + .1f * i, (i % 3 == 2) ? 1.f : 0.f);
		auto mesh = MakeIcosphere(level, c, 1.f, m);
		scene->primitives.push_back(std::make_shared<BVHTriMesh>(mesh, m, 1));
	}
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 25, -20), 1.f, nullptr), WarmWhite(200));
	scene->addAreaLight(std::make_shared<Sphere>(float3(-12, 10, -6), 1.f, nullptr), WarmWhite(60));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.2f, .22f, .25f)));
	scene->camera.lookfrom = float3(4.5f, 3.5f, -9.f);
	scene->camera.lookat = float3(0, 0, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 35;
	scene->camera.aperture = 0;
}

// cfg 5: incoherent-ray stress.  Closed room of diffuse quads, a rough metallic icosphere
// (the reference has no transmission lobe, SURVEY D3, so rough metal is its closest thing to
// "rough glass") and a diffuse icosphere, one small sphere light inside the room.  Rendered
// with PathTracer(16) and Li(..., depth=4) so the reference's Russian roulette is live (D2).
inline void BuildConfig5(Scene* scene, int level) {
	auto wall = DisneyMaterial::Make(float3(.73f, .73f, .73f), 1.f, 0.f);
	auto room = MakeRoom(float3(-4, -1, -9), float3(4, 5, 4), wall);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(room, wall, 1));
	auto roughMetal = DisneyMaterial::Make(float3(0.912f, 0.914f, 0.920f), .6f, 1.f);
	auto diffuse = DisneyMaterial::Make(float3(.2f, .45f, .7f), 1.f, 0.f);
	auto a = MakeIcosphere(level, float3(-1.4f, .2f, .5f), 1.2f, roughMetal);
	auto b = MakeIcosphere(level, float3(1.4f, .2f, -.5f), 1.2f, diffuse);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(a, roughMetal, 1));
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(b, diffuse, 1));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 4.2f, -1.f), .4f, nullptr), WarmWhite(15));
	scene->camera.lookfrom = float3(0, 1.8f, -8.5f);
	scene->camera.lookat = float3(0, .6f, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 40;
	scene->camera.aperture = 0;
}

// cfg 6 (test-only, not in BASELINE.json): small scene that reaches the corners of the
// path the five configs leave out -- thin-lens camera (rejection-sampled lens draws),
// a plain brute-force TriangleMesh, a mesh without normals, a multi-triangle BVH leaf
// (maxPrimsInNode = 4), a sphere light seen from inside a sphere.
inline void BuildConfig6(Scene* scene, int level) {
	auto floor = DisneyMaterial::Make(hex2lin(0xcbceb1), 1.f, 0.f);
	auto backdrop = TriangleMesh::CreateBackdrop(make_float3(0, -1, 20), float3(40, 20, 40), 7.5f, 8, floor);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(backdrop, floor, 4));
	auto gold = DisneyMaterial::Make(float3(0.944f, 0.776f, 0.373f), .5f, 1.f);
	scene->primitives.push_back(std::make_shared<Sphere>(float3(0, 0, 0), 1.f, gold));
	auto mirror = MirrorMaterial::Make(float3(.85f, .9f, .95f));
	auto room = MakeRoom(float3(1.6f, -.95f, -1.f), float3(3.f, .4f, .4f), mirror);
	scene->primitives.push_back(room);   // brute-force TriangleMesh::Intersect (trianglemesh.h:25-35)
	auto teal = DisneyMaterial::Make(float3(.1f, .6f, .55f), .35f, .5f);
	{
		// icosphere WITHOUT normals (geometric shading frame, default per-triangle uvs)
		IcoData d = MakeIcoData(level);
		std::vector<float3> vertices, normals;
		std::vector<float2> texcoords;
		std::vector<index_type> indices;
		for (size_t i = 0; i < d.pos.size() / 3; i++)
			vertices.push_back(float3(-2.2f + .8f * d.pos[3 * i], -.2f + .8f * d.pos[3 * i + 1], -.6f + .8f * d.pos[3 * i + 2]));
		for (int v : d.tri) indices.push_back(index_type(v));
		auto mesh = std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, teal);
		scene->primitives.push_back(std::make_shared<BVHTriMesh>(mesh, teal, 4));
	}
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 6, -3), .5f, nullptr), WarmWhite(120));
	scene->addAreaLight(std::make_shared<Sphere>(float3(-4, 1, 1), 2.5f, nullptr), WarmWhite(2));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.3f, .33f, .4f)));
	scene->camera.lookfrom = float3(-1.46f, 1.16f, -4.64f);
	scene->camera.lookat = float3(0, 0, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 45;
	scene->camera.aperture = .1f;
}

// ---------------------------------------------------------------------------------------
// Procedural environment map.  The reference's default lighting is an HDR file that is not in
// its repo (small_workshop_1k.hdr, myapp.cpp:113); this writes a deterministic stand-in --
// gradient sky, warm horizon band, ground, a small very bright sun -- as a flat (non-RLE)
// Radiance RGBE file that both stb_image (oracle) and host/texture.h read.
// ---------------------------------------------------------------------------------------
inline std::string EnvMapPath() {
	const char* dir = std::getenv("AGPT_TMPDIR");
	return std::string(dir ? dir : "/tmp") + "/agpt_procedural_sky_1k.hdr";
}
inline void WriteProceduralHdr(const std::string& path, int W = 1024, int H = 512) {
	std::vector<unsigned char> bytes((size_t)W * H * 4);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			float v = (y + .5f) / H, u = (x + .5f) / W;           // v = 0: zenith, v = 1: nadir
			float up = 1.f - 2.f * v;                              // ~cos(theta)
			float rgb[3];
			if (up > 0) { rgb[0] = .25f + .35f * (1 - up); rgb[1] = .4f + .3f * (1 - up); rgb[2] = .9f - .2f * (1 - up); }
			else { rgb[0] = .22f; rgb[1] = .2f; rgb[2] = .17f; }
			float band = 1.f - std::fabs(up) * 8.f;
			if (band > 0) { rgb[0] += .5f * band; rgb[1] += .35f * band; rgb[2] += .15f * band; }
			float du = (u - .62f) * 2.f, dv = v - .28f;
			if (du * du + dv * dv < .0002f) { rgb[0] = 120.f; rgb[1] = 108.f; rgb[2] = 90.f; }   // the sun
			float m = std::max(rgb[0], std::max(rgb[1], rgb[2]));
			unsigned char* p = &bytes[4 * ((size_t)y * W + x)];
			if (m < 1e-32f) { p[0] = p[1] = p[2] = p[3] = 0; continue; }
			int e;
			float scale = std::frexp(m, &e) * 256.f / m;
			p[0] = (unsigned char)(rgb[0] * scale); p[1] = (unsigned char)(rgb[1] * scale); p[2] = (unsigned char)(rgb[2] * scale);
			p[3] = (unsigned char)(e + 128);
		}
	FILE* f = std::fopen(path.c_str(), "wb");
	if (!f) return;
	std::fprintf(f, "#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y %d +X %d\n", H, W);
	std::fwrite(bytes.data(), 1, bytes.size(), f);
	std::fclose(f);
}

// cfg 7 (SURVEY 8f row 1): the reference's own default scene, SimpleTestScene (myapp.cpp:55-114):
// backdrop mesh + one gold Disney sphere, thin-lens camera (aperture .1), lit only by an
// InfiniteAreaLight -- with the procedural map standing in for the missing asset.
inline void BuildConfig7(Scene* scene) {
	float roughness = .5f;
	auto gold = DisneyMaterial::Make((float3(0.944f, 0.776f, 0.373f)), roughness, 1.f);
	auto floor = DisneyMaterial::Make(hex2lin(0xcbceb1), 1.f, 0.f);
	auto backdrop = TriangleMesh::CreateBackdrop(make_float3(0, -1, 20), float3(40, 20, 40), 7.5, 32, floor);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(backdrop, floor, 1));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(0, 0, 0), 1.f, gold));
	scene->camera.lookfrom = float3(-1.46, 1.16, -4.64);
	scene->camera.lookat = float3(0, 0, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 1;
	scene->camera.aperture = .1f;
	std::string path = EnvMapPath();
	WriteProceduralHdr(path);
	scene->lights.push_back(std::make_shared<InfiniteAreaLight>(path));
}

// cfg 8 (test-only): the branches no other configuration reaches.
//   * a BVHTriMesh whose SAH tree is a CHAIN: 30 equal triangles perpendicular to x at x = 1e-18 * 16^i.
//     Every binned split (bvhtrimesh.h:257-300) peels off the farthest one, so the tree is 29 levels
//     deep and a ray along +x hits both children at every level: 29 pending far children, more than
//     the traversal keeps in shared memory.  The first ten triangles lie within one ulp of x = 0 as
//     seen from a ray origin at x = -1: exact-t ties, decided by visit order;
//   * a plain TriangleMesh BETWEEN two BVH meshes and another after them (one run of four mesh
//     primitives), the first holding the
//     triangles TriangleIntersect rejects or special-cases (trianglemesh.cpp:59-80): zero area, an
//     area so small that |ng|^2 underflows while det != 0 (dropped by Intersect, kept by
//     IntersectP), zero-determinant texture coordinates on sound geometry (CoordinateSystem
//     fallback), collinear texture coordinates;
//   * a large sphere light with Lemit 3e38: next-event estimates near it overflow to inf, and
//     inf times a zero throughput channel (after the magenta mirror) is NaN -- the samples
//     MyApp::Tick zeroes (myapp.cpp:169-172);
//   * Russian roulette live (depth argument 4), mirror sphere, two infinite lights in one scene.
inline void BuildConfig8(Scene* scene, int level) {
	auto grey = DisneyMaterial::Make(float3(.6f, .6f, .6f), 1.f, 0.f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -1, 0), float2(30, 30), grey));
	auto red = DisneyMaterial::Make(float3(1.f, 0.f, 0.f), 1.f, 0.f);
	{
		std::vector<float3> vertices, normals;
		std::vector<float2> texcoords;
		std::vector<index_type> indices;
		float x = 1e-18f;
		for (int i = 0; i < 30; i++, x *= 16.f) {
			int base = (int)vertices.size();
			vertices.push_back(float3(x, -1.f, 5.f)); vertices.push_back(float3(x, 1.f, 5.f)); vertices.push_back(float3(x, 0.f, 7.f));
			for (int k = 0; k < 3; k++) indices.push_back(index_type(base + k));
		}
		auto chain = std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, red);
		scene->primitives.push_back(std::make_shared<BVHTriMesh>(chain, red, 1));
	}
	auto cream = DisneyMaterial::Make(hex2lin(0xf6e7d0), .6f, 0.f);
	{
		std::vector<float3> vertices, normals;
		std::vector<float2> texcoords;
		std::vector<index_type> indices;
		auto tri = [&](float3 a, float3 b, float3 c, float2 ta, float2 tb, float2 tc) {
			int base = (int)vertices.size();
			vertices.push_back(a); vertices.push_back(b); vertices.push_back(c);
			texcoords.push_back(ta); texcoords.push_back(tb); texcoords.push_back(tc);
			for (int k = 0; k < 3; k++) { index_type idx(base + k); idx.texcoord_index = base + k; indices.push_back(idx); }
		};
		// a sound quad with sound texture coordinates
		tri(float3(-4.f, -1.f, 2.f), float3(-2.f, -1.f, 2.f), float3(-2.f, 1.5f, 2.5f), float2(0, 0), float2(1, 0), float2(1, 1));
		tri(float3(-4.f, -1.f, 2.f), float3(-2.f, 1.5f, 2.5f), float3(-4.f, 1.5f, 2.5f), float2(0, 0), float2(1, 1), float2(0, 1));
		// zero area (two equal vertices): det == 0 for every ray
		tri(float3(-3.f, 0.f, 1.f), float3(-3.f, 0.f, 1.f), float3(-2.5f, 1.f, 1.f), float2(0, 0), float2(1, 0), float2(1, 1));
		// |ng|^2 underflows to 0 although det != 0: rejected by TriangleIntersect only after the t test,
		// accepted by TriangleIntersectP.  Texture coordinates degenerate so the ng branch is taken.
		tri(float3(0.f, 0.f, 0.f), float3(1e-12f, 0.f, 0.f), float3(0.f, 1e-12f, 0.f), float2(.5f, .5f), float2(.5f, .5f), float2(.5f, .5f));
		// sound geometry, all three texture coordinates equal: CoordinateSystem(normalize(ng)) frame
		tri(float3(-1.5f, -1.f, 3.f), float3(.5f, -1.f, 3.f), float3(-.5f, 1.2f, 3.4f), float2(.5f, .5f), float2(.5f, .5f), float2(.5f, .5f));
		// sound geometry, collinear texture coordinates: same branch through a zero determinant
		tri(float3(1.f, -1.f, 3.f), float3(3.f, -1.f, 3.f), float3(2.f, 1.2f, 3.4f), float2(0, 0), float2(1, 1), float2(2, 2));
		scene->primitives.push_back(std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, cream));   // plain: brute force
	}
	auto teal = DisneyMaterial::Make(float3(.1f, .6f, .55f), .35f, .5f);
	auto ball = MakeIcosphere(level, float3(3.f, 0.f, 0.f), 1.f, teal);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(ball, teal, 1));
	{
		// magenta mirror wall behind the overflowing light: throughput (.9, 0, .9), and what it reflects
		// is the floor around the light -- 0 * inf = NaN in the green channel
		auto magenta = MirrorMaterial::Make(float3(.9f, 0.f, .9f));
		std::vector<float3> vertices, normals;
		std::vector<float2> texcoords;
		std::vector<index_type> indices;
		vertices.push_back(float3(-4.f, -1.f, 11.5f)); vertices.push_back(float3(4.f, -1.f, 11.5f));
		vertices.push_back(float3(4.f, 3.f, 11.5f)); vertices.push_back(float3(-4.f, 3.f, 11.5f));
		const int order[6] = { 0, 1, 2, 0, 2, 3 };
		for (int o : order) indices.push_back(index_type(o));
		scene->primitives.push_back(std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, magenta));
	}
	auto mirror = MirrorMaterial::Make(float3(.9f, .9f, .9f));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(-1.2f, 0.f, -1.f), 1.f, mirror));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0.f, .4f, 9.f), 1.4f, nullptr), float3(3e38f, 3e38f, 3e38f));   // rests on the floor behind the chain; estimates near it overflow
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 8, -4), .5f, nullptr), WarmWhite(150));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.25f, .28f, .32f)));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.05f, .04f, .03f)));
	scene->camera.lookfrom = float3(4.5f, 2.5f, -8.f);      // off axis: the chain triangles (planes x = const) are seen obliquely
	scene->camera.lookat = float3(0, 0, 2.f);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 40;
	scene->camera.aperture = 0;
}

#ifdef AGPT_HAS_INSTANCES
// cfg 9 (EXTENSION, host mirror only -- the reference has no Instance class): BASELINE config 4 as its wording has it,
// "10M-triangle INSTANCED scene": ONE unit icosphere mesh (level 8 = 1,310,720 triangles, one BVH) placed eight times
// on the 2x2x2 lattice of cfg 4 through per-instance transforms, one of them scaled and rotated, each placement with
// its own material.  The scene holds 1/8 of cfg 4's geometry (215 MB instead of 1.7 GB).
inline void BuildConfig9(Scene* scene, int level) {
	auto grey = DisneyMaterial::Make(float3(.5f, .5f, .5f), 1.f, 0.f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -2.5f, 0), float2(60, 60), grey));
	const int palette[8] = { 0xf19a91, 0x9ed5d8, 0xeecf74, 0x87abc5, 0xc4ac64, 0x69bab3, 0xe57a82, 0xf7f7f7 };
	auto unit = MakeIcosphere(level, float3(0, 0, 0), 1.f, grey);
	auto shared = std::make_shared<BVHTriMesh>(unit, grey, 1);
	for (int i = 0; i < 8; i++) {
		auto m = DisneyMaterial::Make(hex2lin(palette[i]), .2f + .1f * i, (i % 3 == 2) ? 1.f : 0.f);
		mat4 xf = mat4::Translate((i & 1) ? 1.25f : -1.25f, (i & 2) ? 1.25f : -1.25f, (i & 4) ? 1.25f : -1.25f);
		if (i == 5) xf = xf * mat4::RotateY(.6f) * mat4::Scale(.8f);          // a placement that is not a pure translation
		scene->primitives.push_back(std::make_shared<Instance>(shared, xf, m));
	}
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 25, -20), 1.f, nullptr), WarmWhite(200));
	scene->addAreaLight(std::make_shared<Sphere>(float3(-12, 10, -6), 1.f, nullptr), WarmWhite(60));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.2f, .22f, .25f)));
	scene->camera.lookfrom = float3(4.5f, 3.5f, -9.f);
	scene->camera.lookat = float3(0, 0, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 35;
	scene->camera.aperture = 0;
}
#endif

#ifdef AGPT_HAS_GLASS
// cfg 10 (EXTENSION, host mirror only -- the reference has no transmission lobe): BASELINE config 5 as its wording has
// it, "rough-glass plus diffuse interreflection, 16 bounces with Russian roulette": cfg 5's closed room with the rough
// metal icosphere replaced by ROUGH GLASS (roughness .3, eta 1.5); meant to be rendered with AGPT_FLAG_RR_BY_BOUNCE.
inline void BuildConfig10(Scene* scene, int level) {
	auto wall = DisneyMaterial::Make(float3(.73f, .73f, .73f), 1.f, 0.f);
	auto room = MakeRoom(float3(-4, -1, -9), float3(4, 5, 4), wall);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(room, wall, 1));
	auto glass = GlassMaterial::Make(float3(1.f, 1.f, 1.f), float3(.95f, .97f, 1.f), .3f, 1.5f);
	auto diffuse = DisneyMaterial::Make(float3(.2f, .45f, .7f), 1.f, 0.f);
	auto a = MakeIcosphere(level, float3(-1.4f, .2f, .5f), 1.2f, glass);
	auto b = MakeIcosphere(level, float3(1.4f, .2f, -.5f), 1.2f, diffuse);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(a, glass, 1));
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(b, diffuse, 1));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(0.f, -.4f, -2.5f), .6f, GlassMaterial::Make(float3(1.f, 1.f, 1.f), float3(1.f, .9f, .8f), .05f, 1.33f)));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 4.2f, -1.f), .4f, nullptr), WarmWhite(15));
	scene->camera.lookfrom = float3(0, 1.8f, -8.5f);
	scene->camera.lookat = float3(0, .6f, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 40;
	scene->camera.aperture = 0;
}
#endif

#ifdef AGPT_HAS_SAMPLED_AREA_LIGHTS
// cfg 11 (EXTENSION, host mirror only -- the reference cannot sample a plane or a mesh): cfg 5's room and objects lit by
// three SAMPLED area lights (Scene::addSampledAreaLight) instead of the sphere: a two-triangle TriangleMesh panel just below
// the ceiling, a Plane panel a little lower (no coplanar ties with the ceiling or with the other panel) and a small
// emissive BVHTriMesh icosphere (level 2).  Without the flag the walls would be lit only through specular chains.
inline void BuildConfig11(Scene* scene, int level) {
	auto wall = DisneyMaterial::Make(float3(.73f, .73f, .73f), 1.f, 0.f);
	auto room = MakeRoom(float3(-4, -1, -9), float3(4, 5, 4), wall);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(room, wall, 1));
	auto roughMetal = DisneyMaterial::Make(float3(0.912f, 0.914f, 0.920f), .6f, 1.f);
	auto diffuse = DisneyMaterial::Make(float3(.2f, .45f, .7f), 1.f, 0.f);
	auto a = MakeIcosphere(level, float3(-1.4f, .2f, .5f), 1.2f, roughMetal);
	auto b = MakeIcosphere(level, float3(1.4f, .2f, -.5f), 1.2f, diffuse);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(a, roughMetal, 1));
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(b, diffuse, 1));
	{
		// 1.6 x 1.2 panel at y = 4.97, facing down
		std::vector<float3> vertices = { float3(-.8f, 4.97f, -2.2f), float3(.8f, 4.97f, -2.2f), float3(.8f, 4.97f, -1.f), float3(-.8f, 4.97f, -1.f) };
		std::vector<float3> normals(4, float3(0, -1, 0));
		std::vector<float2> texcoords;
		std::vector<index_type> indices;
		for (int v : { 0, 2, 1, 0, 3, 2 }) indices.push_back(index_type(v));
		scene->addSampledAreaLight(std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, nullptr), WarmWhite(6));
	}
	scene->addSampledAreaLight(std::make_shared<Plane>(float3(-2.2f, 4.93f, -5.f), float2(1.f, 1.f), nullptr), WarmWhite(8));
	scene->addSampledAreaLight(std::make_shared<BVHTriMesh>(MakeIcosphere(2, float3(2.3f, 2.2f, -3.5f), .3f, nullptr), nullptr, 1), WarmWhite(10));
	scene->camera.lookfrom = float3(0, 1.8f, -8.5f);
	scene->camera.lookat = float3(0, .6f, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 40;
	scene->camera.aperture = 0;
}
#endif

#ifdef AGPT_HAS_IMAGE_TEXTURES
// cfg 12 (EXTENSION, host mirror only -- the reference has one colour per material): procedural image textures on the base
// colour of Disney materials, laid out so every uv rule and texture shape is used: a floor plane with a 2048 x 2048 checker
// gradient, spheres with a 37 x 23 (non-power-of-two) image and a 64 x 1 strip, an 8 x 8 quad grid with per-vertex uvs over
// [0, 2]^2 (repeat wrap) and normals placed once as a plain TriangleMesh and once as an Instance of a BVHTriMesh, and one
// untextured Disney sphere.  The 37 x 23 texture is shared by two materials (flattened once).
inline std::shared_ptr<ImageTexture> ProceduralTexture(int W, int H, int kind) {
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			float* p = &rgb[3 * ((size_t)y * W + x)];
			const float fx = (x + .5f) / W, fy = (y + .5f) / H;
			if (kind == 0) {            // checker of 64-texel cells over a gradient
				const bool odd = ((x >> 6) + (y >> 6)) & 1;
				p[0] = .15f + .7f * fx; p[1] = odd ? .8f : .1f; p[2] = .15f + .7f * fy;
			}
			else if (kind == 1) {       // coarse colour blocks: every texel differs from its neighbours
				p[0] = (float)((x * 7 + y * 3) % 11) / 10.f; p[1] = (float)((x * 5 + y * 13) % 7) / 6.f; p[2] = .25f + .5f * fy;
			}
			else {                      // stripes
				p[0] = (x & 1) ? .9f : .2f; p[1] = .3f + .6f * fx; p[2] = (x % 3 == 0) ? .7f : .1f;
			}
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline std::shared_ptr<TriangleMesh> MakeQuadGrid(int n, float size, const float3& at, std::shared_ptr<Material> mat) {
	std::vector<float3> vertices, normals;
	std::vector<float2> texcoords;
	std::vector<index_type> indices;
	for (int j = 0; j <= n; j++)
		for (int i = 0; i <= n; i++) {
			const float u = (float)i / n, v = (float)j / n;
			vertices.push_back(float3(at.x + (u - .5f) * size, at.y + (v - .5f) * size, at.z + .15f * (u - .5f) * (v - .5f) * size));
			normals.push_back(float3(-.1f * (v - .5f), -.1f * (u - .5f), -1.f));
			texcoords.push_back(float2(2.f * u, 2.f * v));
		}
	for (int j = 0; j < n; j++)
		for (int i = 0; i < n; i++) {
			const int a = j * (n + 1) + i, b = a + 1, c = a + n + 2, d = a + n + 1;
			for (int k : { a, b, c, a, c, d }) indices.push_back(index_type(k));
		}
	return std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, mat);
}
inline void BuildConfig12(Scene* scene) {
	auto checker = ProceduralTexture(2048, 2048, 0);
	auto blocks = ProceduralTexture(37, 23, 1);
	auto strip = ProceduralTexture(64, 1, 2);
	auto floorMat = DisneyMaterial::Make(checker, 1.f, 0.f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -1, 0), float2(8, 8), floorMat));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(-2.4f, 0, 0), 1.f, DisneyMaterial::Make(blocks, .5f, 0.f)));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(0, 0, 1.f), 1.f, DisneyMaterial::Make(strip, .3f, .5f)));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(2.4f, 0, 0), 1.f, DisneyMaterial::Make(float3(.2f, .45f, .7f), .4f, 0.f)));
	auto gridMat = DisneyMaterial::Make(blocks, .7f, .2f);
	scene->primitives.push_back(MakeQuadGrid(8, 2.f, float3(-1.2f, 1.8f, 3.f), gridMat));
	auto placed = std::make_shared<BVHTriMesh>(MakeQuadGrid(8, 2.f, float3(0.f), gridMat), gridMat, 1);
	scene->primitives.push_back(std::make_shared<Instance>(placed, mat4::Translate(1.4f, 1.9f, 3.2f) * mat4::RotateY(-.4f), DisneyMaterial::Make(checker, .6f, 0.f)));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 8, -4), .5f, nullptr), WarmWhite(120));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.15f, .17f, .2f)));
	scene->camera.lookfrom = float3(0, 2.2f, -8.5f);
	scene->camera.lookat = float3(0, .4f, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 40;
	scene->camera.aperture = 0;
}
#endif

#ifdef AGPT_HAS_MATERIAL_MAPS
// cfg 13 (EXTENSION, host mirror only): procedural roughness-metallic and normal maps (include/agpt.h
// agpt_upload_material_textures), laid out so every shape's tangent frame and every rule of the maps is used:
// - a floor plane, colour-only material, with a roughness / metallic checker (metallic 0 and 1 tiles: the lobe set changes from
//   hit to hit) and the normal map of an analytic height field;
// - a sphere with a base-colour image, a roughness-metallic map and a bumpy normal map (its -z pole faces the camera);
// - a sphere whose normal map mixes flat texels, tilted ones and texels with z < 0.5 (the rules that leave a surface as it is);
// - an 8 x 8 quad grid with per-vertex uvs and interpolated normals, placed plainly, as a rotated, scaled instance and as a
//   sheared one;
// level 2 adds a rough glass sphere, so the instantiation that carries everything runs.
inline std::shared_ptr<ImageTexture> HeightFieldNormals(int W, int H, float amplitude, int waves) {
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			const double u = (x + .5) / W, v = (y + .5) / H, k = 2 * 3.14159265358979 * waves;
			// h = amplitude * sin(k u) sin(k v); tangent-space normal = normalize(-dh/du, -dh/dv, 1), stored as n / 2 + 1/2
			const double du = amplitude * k * std::cos(k * u) * std::sin(k * v), dv = amplitude * k * std::sin(k * u) * std::cos(k * v);
			const double l = std::sqrt(du * du + dv * dv + 1);
			float* p = &rgb[3 * ((size_t)y * W + x)];
			p[0] = (float)(-du / l * .5 + .5); p[1] = (float)(-dv / l * .5 + .5); p[2] = (float)(1 / l * .5 + .5);
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline std::shared_ptr<ImageTexture> RoughnessMetallicChecker(int W, int H, int cells) {
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			const int cx = x * cells / W, cy = y * cells / H;
			float* p = &rgb[3 * ((size_t)y * W + x)];
			p[0] = .5f;                                            // unused
			p[1] = ((cx + 2 * cy) % 3 == 0) ? .25f : ((cx + 2 * cy) % 3 == 1) ? .6f : 1.f;   // roughness factor
			p[2] = ((cx + cy) & 1) ? 1.f : 0.f;                   // metallic 0 / 1 tiles
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline std::shared_ptr<ImageTexture> MixedNormals(int W, int H) {
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			float* p = &rgb[3 * ((size_t)y * W + x)];
			const int kind = (x / 4 + y / 4) % 4;
			if (kind == 0) { p[0] = .5f; p[1] = .5f; p[2] = 1.f; }         // flat
			else if (kind == 1) { p[0] = .8f; p[1] = .4f; p[2] = .85f; }   // tilted
			else if (kind == 2) { p[0] = .6f; p[1] = .9f; p[2] = .2f; }    // z < 0.5: below the surface
			else { p[0] = .5f; p[1] = .5f; p[2] = .3f; }                   // z < 0.5 and no tilt
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline void BuildConfig13(Scene* scene, int level) {
	auto floorMat = DisneyMaterial::Make(float3(.7f, .62f, .5f), .9f, 1.f);
	floorMat->SetRoughnessMetallicMap(RoughnessMetallicChecker(64, 64, 8));
	floorMat->SetNormalMap(HeightFieldNormals(256, 256, .02f, 6), 1.f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -1, 0), float2(8, 8), floorMat));
	auto bumps = HeightFieldNormals(64, 32, .01f, 4);
	auto ballMat = DisneyMaterial::Make(ProceduralTexture(37, 23, 1), .6f, .8f);
	ballMat->SetRoughnessMetallicMap(RoughnessMetallicChecker(16, 16, 4));
	ballMat->SetNormalMap(bumps, 1.5f);
	scene->primitives.push_back(std::make_shared<Sphere>(float3(-2.2f, 0, 0), 1.f, ballMat));
	auto mixedMat = DisneyMaterial::Make(float3(.25f, .5f, .75f), .4f, 0.f);
	mixedMat->SetNormalMap(MixedNormals(32, 16), .8f);
	scene->primitives.push_back(std::make_shared<Sphere>(float3(.3f, 0, .6f), 1.f, mixedMat));
	auto gridMat = DisneyMaterial::Make(float3(.8f, .3f, .2f), .7f, .5f);
	gridMat->SetRoughnessMetallicMap(RoughnessMetallicChecker(8, 8, 2));
	gridMat->SetNormalMap(bumps, 1.f);
	scene->primitives.push_back(MakeQuadGrid(8, 2.f, float3(-1.2f, 1.8f, 3.f), gridMat));
	auto placed = std::make_shared<BVHTriMesh>(MakeQuadGrid(8, 2.f, float3(0.f), gridMat), gridMat, 1);
	scene->primitives.push_back(std::make_shared<Instance>(placed, mat4::Translate(1.6f, 1.7f, 3.2f) * mat4::RotateY(-.5f) * mat4::Scale(1.3f), gridMat));
	mat4 shear;                                    // x += .35 y, z += .2 x: a sheared placement of the same grid
	shear.cell[1] = .35f; shear.cell[8] = .2f;
	scene->primitives.push_back(std::make_shared<Instance>(placed, mat4::Translate(-3.6f, 2.0f, 3.6f) * shear, gridMat));
	if (level >= 2)
		scene->primitives.push_back(std::make_shared<Sphere>(float3(2.6f, -.2f, -.4f), .8f, GlassMaterial::Make(float3(1.f), float3(.9f, .95f, 1.f), .2f)));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 8, -4), .5f, nullptr), WarmWhite(120));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.15f, .17f, .2f)));
	scene->camera.lookfrom = float3(0, 2.2f, -8.5f);
	scene->camera.lookat = float3(0, .4f, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 40;
	scene->camera.aperture = 0;
}
#endif

#if defined(AGPT_HAS_ALPHA_MASKS) && defined(AGPT_HAS_MATERIAL_MAPS)
// cfg 14 (EXTENSION, host mirror only -- the reference's surfaces are solid): alpha-masked cutout geometry (include/agpt.h
// agpt_upload_alpha_masks), laid out so every masked path of the trace walk is used:
// - a BVHTriMesh of 1,536 leaf quads with per-vertex uvs over an elliptical leaf; the leaf image is the leaves' base colour and,
//   through its green channel, their mask; a ring of its texels equals the cutoff exactly;
// - the same leaf mesh as two rotated, scaled Instances with a second material masked by the red channel of another image;
// - a plain TriangleMesh quad with the default uvs and a checker mask;
// - a horizontal masked Plane (a grate) between the sphere area light and the floor: shadow rays go through its holes;
// - a masked mirror quad, and the sky (UniformInfiniteLight) behind every hole.
// Level 2 adds roughness-metallic and normal maps on the leaves, so masked trace runs beside the mapped shade.
inline std::shared_ptr<ImageTexture> LeafImage(int W, int H) {
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			const float u = (x + .5f) / W - .5f, v = (y + .5f) / H - .5f;
			const float e = (u * u) / (.45f * .45f) + (v * v) / (.3f * .3f);      // elliptical leaf
			float* p = &rgb[3 * ((size_t)y * W + x)];
			p[0] = .15f + .3f * (v + .5f);
			p[1] = e < .8f ? 1.f : e < 1.f ? .5f : 0.f;                             // the alpha; .5 = the cutoff, on a ring
			p[2] = .1f + .2f * (u + .5f);
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline std::shared_ptr<ImageTexture> MaskPattern(int W, int H, int kind) {
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			float* p = &rgb[3 * ((size_t)y * W + x)];
			float a;
			if (kind == 0) a = ((x + y) & 1) ? 1.f : 0.f;                                  // checker
			else if (kind == 1) a = (x % 4 == 0 || y % 4 == 0) ? 1.f : .25f;               // grate bars
			else { const float u = (x + .5f) / W - .5f, v = (y + .5f) / H - .5f; a = u * u + v * v < .2f ? .9f : .1f; }   // disc
			p[0] = a; p[1] = .5f * a; p[2] = a;
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline std::shared_ptr<TriangleMesh> MakeLeaves(int n, std::shared_ptr<Material> mat) {
	std::vector<float3> vertices, normals;
	std::vector<float2> texcoords;
	std::vector<index_type> indices;
	uint32_t s = 12345u;
	auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (float)(s >> 8) / 16777216.f; };
	for (int i = 0; i < n; i++) {
		const float3 c(-2.5f + 2.f * rnd(), 1.f + 2.2f * rnd(), -1.f + 2.f * rnd());
		const float a = 6.2831853f * rnd(), b = 1.2f * (rnd() - .5f), size = .25f + .2f * rnd();
		const float3 t(std::cos(a) * size, b * size, std::sin(a) * size), w(-std::sin(a) * .6f * size * b, .6f * size, std::cos(a) * .6f * size * b);
		const int base = (int)vertices.size();
		const float3 corner[4] = { c - t - w, c + t - w, c + t + w, c - t + w };
		const float2 uv[4] = { float2(0, 0), float2(1, 0), float2(1, 1), float2(0, 1) };
		for (int k = 0; k < 4; k++) { vertices.push_back(corner[k]); texcoords.push_back(uv[k]); }
		for (int k : { 0, 1, 2, 0, 2, 3 }) indices.push_back(index_type(base + k));
	}
	return std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, mat);
}
inline std::shared_ptr<TriangleMesh> MakeQuad(const float3& o, const float3& e1, const float3& e2, bool uvs, std::shared_ptr<Material> mat) {
	std::vector<float3> vertices = { o, o + e1, o + e1 + e2, o + e2 }, normals;
	std::vector<float2> texcoords;
	if (uvs) texcoords = { float2(0, 0), float2(1, 0), float2(1, 1), float2(0, 1) };
	std::vector<index_type> indices;
	for (int v : { 0, 1, 2, 0, 2, 3 }) indices.push_back(index_type(v));
	return std::make_shared<TriangleMesh>(indices, vertices, normals, texcoords, mat);
}
inline void BuildConfig14(Scene* scene, int level) {
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, -1, 0), float2(8, 8), DisneyMaterial::Make(float3(.6f, .58f, .55f), .9f, 0.f)));
	auto leaf = LeafImage(64, 64);
	auto leafMat = DisneyMaterial::Make(leaf, .6f, 0.f);
	leafMat->SetAlphaMask(leaf, 1, .5f);
	if (level >= 2) {
		leafMat->SetRoughnessMetallicMap(RoughnessMetallicChecker(16, 16, 4));
		leafMat->SetNormalMap(HeightFieldNormals(32, 32, .01f, 2), 1.f);
	}
	auto leaves = MakeLeaves(1536, leafMat);
	auto bvh = std::make_shared<BVHTriMesh>(leaves, leafMat, 1);
	scene->primitives.push_back(bvh);
	auto discs = MaskPattern(32, 32, 2);
	auto otherLeaf = DisneyMaterial::Make(float3(.55f, .35f, .15f), .5f, 0.f);
	otherLeaf->SetAlphaMask(discs, 0, .5f);
	scene->primitives.push_back(std::make_shared<Instance>(bvh, mat4::Translate(3.8f, -.4f, 1.5f) * mat4::RotateY(.7f) * mat4::Scale(.7f), otherLeaf));
	scene->primitives.push_back(std::make_shared<Instance>(bvh, mat4::Translate(-1.f, -.9f, 4.f) * mat4::RotateY(-.4f) * mat4::Scale(1.2f), leafMat));
	auto checkerMat = DisneyMaterial::Make(float3(.2f, .45f, .7f), .4f, 0.f);
	checkerMat->SetAlphaMask(MaskPattern(8, 8, 0), 0, .5f);
	scene->primitives.push_back(MakeQuad(float3(1.f, -1.f, -1.5f), float3(2.f, 0, .3f), float3(0, 2.f, 0), false, checkerMat));
	auto grateMat = DisneyMaterial::Make(float3(.5f, .5f, .52f), .7f, 1.f);
	grateMat->SetAlphaMask(MaskPattern(16, 16, 1), 2, .5f);
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, 4.f, 0), float2(3.f, 3.f), grateMat));
	auto mirror = MirrorMaterial::Make(float3(.9f, .9f, .9f));
	mirror->SetAlphaMask(discs, 0, .5f);
	scene->primitives.push_back(MakeQuad(float3(-4.2f, -1.f, 2.f), float3(1.8f, 0, -.6f), float3(0, 2.5f, 0), true, mirror));
	scene->addAreaLight(std::make_shared<Sphere>(float3(0, 6.f, .5f), .5f, nullptr), WarmWhite(150));
	scene->lights.push_back(std::make_shared<UniformInfiniteLight>(float3(.3f, .35f, .45f)));
	scene->camera.lookfrom = float3(0, 2.f, -8.5f);
	scene->camera.lookat = float3(0, 1.f, 0);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 45;
	scene->camera.aperture = 0;
}
#endif

#if defined(AGPT_HAS_EMISSION) && defined(AGPT_HAS_ALPHA_MASKS) && defined(AGPT_HAS_MATERIAL_MAPS)
// cfg 15 (EXTENSION, host mirror only -- the reference's only emitters are AreaLights around null-material shapes): emissive
// materials (include/agpt.h agpt_upload_emission) in a closed room, laid out so every uv rule of the emission lookup is used:
// - a screen: a BVHTriMesh of 2 x 2 quads with uvs over [0, 2]^2 (repeat wrap), a colour-bar / checker image as its emission
//   and as the base colour of the glossy Disney material under it (a BVHTriMesh of only two triangles flattens to a two-entry
//   node table, which agpt_upload_meshes refuses);
// - a constant-emission Disney sphere, and a factor-only emissive Plane strip under the ceiling;
// - a small icosphere (default uvs) placed twice as Instances, its emission a striped image;
// - a mirror on the side wall that sees the screen (specular chains).
// Level 1 lights the room with one sphere AreaLight as well, so next-event estimation and emission combine.  Level 2 has no
// light at all (every path runs with n_lights == 0) and adds an emissive sign whose letters are cut out by an alpha mask (the
// mask image is also its emission image).
inline std::shared_ptr<ImageTexture> ColourBars(int W, int H) {
	static const float bars[7][3] = { { .75f, .75f, .75f }, { .75f, .75f, 0 }, { 0, .75f, .75f }, { 0, .75f, 0 }, { .75f, 0, .75f }, { .75f, 0, 0 }, { 0, 0, .75f } };
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			float* p = &rgb[3 * ((size_t)y * W + x)];
			if (y < H / 3) { const float c = ((x / 4 + y / 4) & 1) ? 1.f : .05f; p[0] = c; p[1] = c; p[2] = c; }   // checker (row 0: v near 0)
			else { const float* b = bars[(x * 7) / W]; p[0] = b[0]; p[1] = b[1]; p[2] = b[2]; }
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline std::shared_ptr<ImageTexture> SignLetters(int W, int H) {
	std::vector<float> rgb(3 * (size_t)W * H);
	for (int y = 0; y < H; y++)
		for (int x = 0; x < W; x++) {
			const int cx = x % 8, cy = y % 16, letter = x / 8;
			// blocky strokes: a left bar, and a top, middle or bottom bar that changes from letter to letter
			const bool on = cx == 1 || cx == 2 || ((cy == 2 || cy == 3) && letter % 2 == 0) || ((cy == 7 || cy == 8) && letter % 3 != 1) ||
				((cy == 12 || cy == 13) && cx < 6) || (cx == 5 && letter % 2 == 1 && cy > 2 && cy < 13);
			float* p = &rgb[3 * ((size_t)y * W + x)];
			p[0] = on ? 1.f : 0.f; p[1] = on ? .5f + .5f * (float)letter / (W / 8) : 0.f; p[2] = on ? .25f : 0.f;
		}
	return ImageTexture::Make(W, H, std::move(rgb));
}
inline void BuildConfig15(Scene* scene, int level) {
	auto wallMat = DisneyMaterial::Make(float3(.7f, .68f, .65f), .9f, 0.f);
	scene->primitives.push_back(MakeRoom(float3(-5.f, -1.f, -6.f), float3(5.f, 5.f, 6.f), wallMat));
	auto bars = ColourBars(64, 48);
	auto screenMat = DisneyMaterial::Make(bars, .25f, 0.f);
	screenMat->SetEmission(float3(2.f, 2.f, 2.f), bars);
	scene->primitives.push_back(std::make_shared<BVHTriMesh>(MakeQuadGrid(2, 2.5f, float3(0, 1.35f, 5.5f), screenMat), screenMat, 1));
	auto ballMat = DisneyMaterial::Make(float3(.8f, .3f, .2f), .5f, 0.f);
	ballMat->SetEmission(float3(1.5f, .6f, .2f));
	scene->primitives.push_back(std::make_shared<Sphere>(float3(2.6f, -.2f, 2.f), .8f, ballMat));
	auto stripMat = DisneyMaterial::Make(float3(.9f, .9f, .9f), .8f, 0.f);
	stripMat->SetEmission(float3(4.f, 4.f, 4.5f));
	scene->primitives.push_back(std::make_shared<Plane>(float3(0, 4.9f, 1.f), float2(3.f, .2f), stripMat));
	auto icoMat = DisneyMaterial::Make(float3(.2f, .5f, .8f), .4f, 0.f);
	icoMat->SetEmission(float3(1.f, 1.f, 1.f), ProceduralTexture(64, 1, 2));
	auto unit = std::make_shared<BVHTriMesh>(MakeIcosphere(2, float3(0, 0, 0), 1.f, icoMat), icoMat, 1);
	scene->primitives.push_back(std::make_shared<Instance>(unit, mat4::Translate(-2.6f, -.5f, 1.5f) * mat4::Scale(.5f), icoMat));
	scene->primitives.push_back(std::make_shared<Instance>(unit, mat4::Translate(-.9f, -.6f, -.5f) * mat4::RotateY(.6f) * mat4::Scale(.4f), icoMat));
	auto mirror = MirrorMaterial::Make(float3(.9f, .9f, .9f));
	scene->primitives.push_back(MakeQuad(float3(-4.8f, -.5f, -1.f), float3(0, 0, 4.5f), float3(0, 3.5f, 0), true, mirror));
	if (level >= 2) {
		auto letters = SignLetters(48, 16);
		auto signMat = DisneyMaterial::Make(float3(.1f, .1f, .12f), .6f, 0.f);
		signMat->SetAlphaMask(letters, 0, .5f);
		signMat->SetEmission(float3(3.f, 1.2f, .4f), letters);
		scene->primitives.push_back(MakeQuad(float3(-1.5f, 3.1f, 4.f), float3(3.f, 0, 0), float3(0, 1.f, 0), true, signMat));
	}
	else scene->addAreaLight(std::make_shared<Sphere>(float3(0, 4.2f, 0), .35f, nullptr), WarmWhite(60));
	scene->camera.lookfrom = float3(.5f, 1.6f, -5.5f);
	scene->camera.lookat = float3(-.3f, 1.2f, 3.f);
	scene->camera.vup = float3(0, 1, 0);
	scene->camera.aspect_ratio = 16.f / 9.f;
	scene->camera.vfov = 60;
	scene->camera.aperture = 0;
}
#endif

// level <= 0 selects the BASELINE.json size of each configuration.
inline bool BuildConfig(Scene* scene, int config, int level) {
	switch (config) {
	case 1: BuildConfig1(scene); return true;
	case 2: BuildConfig2(scene, level > 0 ? level : 8); return true;
	case 3: BuildConfig3(scene, level > 0 ? level : 7); return true;
	case 4: BuildConfig4(scene, level > 0 ? level : 8); return true;
	case 5: BuildConfig5(scene, level > 0 ? level : 7); return true;
	case 6: BuildConfig6(scene, level > 0 ? level : 2); return true;
	case 7: BuildConfig7(scene); return true;
	case 8: BuildConfig8(scene, level > 0 ? level : 3); return true;
#ifdef AGPT_HAS_INSTANCES
	case 9: BuildConfig9(scene, level > 0 ? level : 8); return true;
#endif
#ifdef AGPT_HAS_GLASS
	case 10: BuildConfig10(scene, level > 0 ? level : 7); return true;
#endif
#ifdef AGPT_HAS_SAMPLED_AREA_LIGHTS
	case 11: BuildConfig11(scene, level > 0 ? level : 7); return true;
#endif
#ifdef AGPT_HAS_IMAGE_TEXTURES
	case 12: BuildConfig12(scene); return true;
#endif
#ifdef AGPT_HAS_MATERIAL_MAPS
	case 13: BuildConfig13(scene, level > 0 ? level : 1); return true;
#endif
#if defined(AGPT_HAS_ALPHA_MASKS) && defined(AGPT_HAS_MATERIAL_MAPS)
	case 14: BuildConfig14(scene, level > 0 ? level : 1); return true;
#endif
#if defined(AGPT_HAS_EMISSION) && defined(AGPT_HAS_ALPHA_MASKS) && defined(AGPT_HAS_MATERIAL_MAPS)
	case 15: BuildConfig15(scene, level > 0 ? level : 1); return true;
#endif
	default: return false;
	}
}

} // namespace agpt_scenes
