// agpt_host.cpp -- libagpt_host.so: C entry points over the host mirror (include/agpt_host.h).
#include "precomp.h"
#include "scene.h"
#include "integrator.h"
#include "scenes/config_scenes.h"
#include "agpt_host.h"

struct agpt_host_scene {
	Scene scene;
	std::unique_ptr<Camera> camera;
	std::shared_ptr<FlatScene> flat;      // cached Flatten() result
};

struct agpt_host_tracer {
	std::unique_ptr<CudaPathTracer> tracer;
};

static thread_local std::string g_hostError;
static int HostFail(const std::string& m) { g_hostError = m; return AGPT_ERR_INVALID; }
#define HOST_TRY(...) try { __VA_ARGS__ } catch (const std::exception& e) { return HostFail(e.what()); }

static int UploadFlat(const FlatScene& flat, const Camera& camera, agpt_ctx* ctx) {
	int rc;
	if ((rc = agpt_upload_meshes(ctx, flat.meshes.data(), (int)flat.meshes.size()))) return rc;
	if ((rc = agpt_upload_spheres(ctx, flat.spheres.data(), (int)flat.spheres.size()))) return rc;
	if ((rc = agpt_upload_planes(ctx, flat.planes.data(), (int)flat.planes.size()))) return rc;
	if ((rc = agpt_upload_materials(ctx, flat.materials.data(), (int)flat.materials.size()))) return rc;
	if ((rc = agpt_upload_lights(ctx, flat.lights.data(), (int)flat.lights.size()))) return rc;
	if ((rc = agpt_upload_envmap(ctx, flat.envmap.width > 0 ? &flat.envmap : nullptr))) return rc;
	if ((rc = agpt_upload_instances(ctx, flat.instances.data(), (int)flat.instances.size()))) return rc;
	if ((rc = agpt_upload_primitives(ctx, flat.prims.data(), (int)flat.prims.size()))) return rc;
	if ((rc = agpt_upload_material_textures(ctx, flat.textures.data(), (int)flat.textures.size(), flat.materialTextures.data(), (int)flat.materialTextures.size()))) return rc;
	if ((rc = agpt_upload_alpha_masks(ctx, flat.alphaMasks.data(), (int)flat.alphaMasks.size()))) return rc;   // after the textures it names
	if ((rc = agpt_upload_emission(ctx, flat.emission.data(), (int)flat.emission.size()))) return rc;          // likewise
	agpt_camera cam = camera.Export();
	return agpt_set_camera(ctx, &cam);
}

extern "C" {

const char* agpt_host_last_error(void) { return g_hostError.empty() ? agpt_last_error() : g_hostError.c_str(); }

int agpt_host_scene_create(int config, int level, agpt_host_scene** out) {
	if (!out) return HostFail("null out");
	*out = nullptr;
	HOST_TRY(
		auto s = std::make_unique<agpt_host_scene>();
		if (!agpt_scenes::BuildConfig(&s->scene, config, level)) return HostFail("unknown configuration");
		s->camera.reset(new Camera(s->scene.camera));
		*out = s.release();
	)
	g_hostError.clear();
	return AGPT_OK;
}

int agpt_host_scene_destroy(agpt_host_scene* s) { delete s; return AGPT_OK; }

int agpt_host_config_defaults(int config, int* out5, const char** name) {
	agpt_scenes::ConfigDefaults d = agpt_scenes::Defaults(config);
	if (d.width == 0) return HostFail("unknown configuration");
	out5[0] = d.width; out5[1] = d.height; out5[2] = d.spp; out5[3] = d.max_depth; out5[4] = d.depth_arg;
	if (name) *name = d.name;
	return AGPT_OK;
}

static FlatScene& Flat(agpt_host_scene* s) {
	if (!s->flat) s->flat = s->scene.Flatten();
	return *s->flat;
}

int agpt_host_scene_counts(agpt_host_scene* s, int64_t* counts4, uint64_t* bytes) {
	if (!s) return HostFail("null scene");
	HOST_TRY(
		FlatScene& f = Flat(s);
		int64_t tris = 0, nodes = 0;
		for (auto& m : f.meshes) { tris += m.n_tris; nodes += m.n_nodes; }
		if (counts4) { counts4[0] = (int64_t)f.prims.size(); counts4[1] = (int64_t)f.lights.size(); counts4[2] = tris; counts4[3] = nodes; }
		if (bytes) *bytes = f.Bytes();
	)
	return AGPT_OK;
}

int agpt_host_scene_upload(agpt_host_scene* s, agpt_ctx* ctx) {
	if (!s || !ctx) return HostFail("null argument");
	g_hostError.clear();
	HOST_TRY( return UploadFlat(Flat(s), *s->camera, ctx); )
}

int agpt_host_scene_tables(agpt_host_scene* s, agpt_scene_tables* out) {
	if (!s || !out) return HostFail("null argument");
	HOST_TRY(
		FlatScene& f = Flat(s);
		out->prims = f.prims.data(); out->n_prims = (int)f.prims.size();
		out->spheres = f.spheres.data(); out->n_spheres = (int)f.spheres.size();
		out->planes = f.planes.data(); out->n_planes = (int)f.planes.size();
		out->meshes = f.meshes.data(); out->n_meshes = (int)f.meshes.size();
		out->materials = f.materials.data(); out->n_materials = (int)f.materials.size();
		out->lights = f.lights.data(); out->n_lights = (int)f.lights.size();
		out->camera = s->camera->Export();
		out->envmap = f.envmap;
		out->instances = f.instances.data(); out->n_instances = (int)f.instances.size();
		out->textures = f.textures.empty() ? nullptr : f.textures.data(); out->material_texture = f.materialTexture.empty() ? nullptr : f.materialTexture.data();
		out->n_textures = (int)f.textures.size(); out->n_material_texture = (int)f.materialTexture.size();
		out->material_textures = f.materialTextures.empty() ? nullptr : f.materialTextures.data(); out->n_material_textures = (int)f.materialTextures.size();
	)
	return AGPT_OK;
}

int agpt_host_scene_alpha_masks(agpt_host_scene* s, const agpt_alpha_mask** out, int* n) {
	if (!s || !out || !n) return HostFail("null argument");
	HOST_TRY(
		FlatScene& f = Flat(s);
		*out = f.alphaMasks.empty() ? nullptr : f.alphaMasks.data();
		*n = (int)f.alphaMasks.size();
	)
	return AGPT_OK;
}

int agpt_host_scene_emission(agpt_host_scene* s, const agpt_emission** out, int* n) {
	if (!s || !out || !n) return HostFail("null argument");
	HOST_TRY(
		FlatScene& f = Flat(s);
		*out = f.emission.empty() ? nullptr : f.emission.data();
		*n = (int)f.emission.size();
	)
	return AGPT_OK;
}

int agpt_host_camera_export(agpt_host_scene* s, float* out19) {
	agpt_camera c = s->camera->Export();
	memcpy(out19, &c, 19 * sizeof(float));
	return AGPT_OK;
}

int agpt_host_prim_info(agpt_host_scene* s, int prim, int* kind, int* counts5, int* has_material, int* is_light) {
	if (prim < 0 || prim >= (int)s->scene.primitives.size()) return HostFail("primitive index out of range");
	const Intersectable* shape = s->scene.primitives[prim].get();
	*kind = shape->Kind();
	*has_material = shape->GetMaterial() != nullptr;
	*is_light = shape->GetAreaLight() != nullptr;
	for (int i = 0; i < 5; i++) counts5[i] = 0;
	if (*kind >= AGPT_PRIM_BVH_MESH) {
		const int payload = Flat(s).prims[prim].payload;
		const agpt_mesh_desc& m = Flat(s).meshes[*kind == AGPT_PRIM_INSTANCE ? Flat(s).instances[payload].mesh : payload];
		counts5[0] = m.n_nodes; counts5[1] = m.n_tris;
		counts5[3] = m.tri_normals ? 1 : 0; counts5[4] = m.tri_uvs ? 1 : 0;
	}
	return AGPT_OK;
}

int agpt_host_bvh_export(agpt_host_scene* s, int prim, void* nodes_out, int* leaf_tri_out) {
	if (prim < 0 || prim >= (int)s->scene.primitives.size()) return HostFail("primitive index out of range");
	auto* bvh = dynamic_cast<const BVHTriMesh*>(s->scene.primitives[prim].get());
	if (!bvh) return HostFail("not a BVHTriMesh");
	memcpy(nodes_out, bvh->Nodes().data(), bvh->Nodes().size() * sizeof(BVHNode));
	memcpy(leaf_tri_out, bvh->LeafOrder().data(), bvh->LeafOrder().size() * sizeof(int));
	return (int)bvh->Nodes().size();
}

int agpt_host_mesh_export(agpt_host_scene* s, int prim, float* tri_verts_out) {
	if (prim < 0 || prim >= (int)s->scene.primitives.size()) return HostFail("primitive index out of range");
	auto* mesh = dynamic_cast<const TriangleMesh*>(s->scene.primitives[prim].get());
	if (!mesh) return HostFail("not a TriangleMesh");
	std::vector<int32_t> order(mesh->NumTriangles());
	for (size_t i = 0; i < order.size(); i++) order[i] = (int32_t)i;
	FlatTriangles ft = mesh->ExportTriangles(order);
	for (size_t t = 0; t < order.size(); t++)
		for (int k = 0; k < 3; k++)
			for (int a = 0; a < 3; a++) tri_verts_out[9 * t + 3 * k + a] = ft.verts[12 * t + 4 * k + a];
	return (int)order.size();
}

static void MaterialTo20(const agpt_material& m, float* o) {
	for (int i = 0; i < 20; i++) o[i] = 0;
	o[0] = (float)m.type;
	if (m.type == AGPT_MAT_DISNEY) {
		if (m.lobes & AGPT_LOBE_DIFFUSE) { o[1] = m.diffuse_r[0]; o[2] = m.diffuse_r[1]; o[3] = m.diffuse_r[2]; o[18] = 1; }
		if (m.lobes & AGPT_LOBE_RETRO) { o[4] = m.diffuse_r[0]; o[5] = m.diffuse_r[1]; o[6] = m.diffuse_r[2]; o[7] = m.roughness; o[19] = 1; }
		o[8] = m.alpha_x; o[9] = m.alpha_y;
		o[10] = m.spec_r0[0]; o[11] = m.spec_r0[1]; o[12] = m.spec_r0[2]; o[13] = m.metallic; o[14] = m.eta;
	}
	else if (m.type == AGPT_MAT_MIRROR) { o[15] = m.mirror_r[0]; o[16] = m.mirror_r[1]; o[17] = m.mirror_r[2]; }
}

int agpt_host_material_export(agpt_host_scene* s, int prim, float* out20) {
	if (prim < 0 || prim >= (int)s->scene.primitives.size()) return HostFail("primitive index out of range");
	const Material* m = s->scene.primitives[prim]->GetMaterial();
	for (int i = 0; i < 20; i++) out20[i] = 0;
	if (!m) return 0;
	agpt_material rec = m->Export();
	MaterialTo20(rec, out20);
	return rec.type;
}

int agpt_host_make_material(int type, const float* c, float roughness, float metallic, agpt_material* out) {
	if (!c || !out) return HostFail("null argument");
	if (type == AGPT_MAT_DISNEY) *out = DisneyMaterial(float3(c[0], c[1], c[2]), roughness, metallic).Export();
	else if (type == AGPT_MAT_MIRROR) *out = MirrorMaterial(float3(c[0], c[1], c[2])).Export();
	else if (type == AGPT_MAT_GLASS) *out = GlassMaterial(float3(c[0], c[1], c[2]), float3(c[0], c[1], c[2]), roughness, metallic > 0 ? metallic : 1.5f).Export();   // (Kr = Kt = color; the `metallic` slot carries eta)
	else return HostFail("unknown material type");
	return AGPT_OK;
}

int agpt_host_set_build_options(int threads, const char* cache_dir) {
	BVHTriMesh::BuildOptions& opt = BVHTriMesh::Options();
	if (threads >= 1) opt.threads = threads;
	if (cache_dir) opt.cacheDir = cache_dir;
	return AGPT_OK;
}

int agpt_host_get_build_options(int* threads, char* cache_dir, int cache_dir_capacity) {
	const BVHTriMesh::BuildOptions& opt = BVHTriMesh::Options();
	if (threads) *threads = opt.threads;
	if (cache_dir && cache_dir_capacity > 0) snprintf(cache_dir, (size_t)cache_dir_capacity, "%s", opt.cacheDir.c_str());
	return AGPT_OK;
}

int agpt_host_tracer_create(int max_depth, int device, agpt_host_tracer** out) {
	if (!out) return HostFail("null out");
	*out = nullptr;
	g_hostError.clear();
	HOST_TRY(
		auto t = std::make_unique<agpt_host_tracer>();
		t->tracer.reset(new CudaPathTracer(max_depth, device));
		*out = t.release();
	)
	return AGPT_OK;
}

int agpt_host_tracer_create_multi(int max_depth, const int* devices, int n, agpt_host_tracer** out) {
	if (!out || !devices || n < 1) return HostFail("bad device list");
	*out = nullptr;
	g_hostError.clear();
	HOST_TRY(
		auto t = std::make_unique<agpt_host_tracer>();
		t->tracer.reset(new CudaPathTracer(max_depth, std::vector<int>(devices, devices + n)));
		*out = t.release();
	)
	return AGPT_OK;
}

int agpt_host_tracer_destroy(agpt_host_tracer* t) { delete t; return AGPT_OK; }

int agpt_host_tracer_ctx(agpt_host_tracer* t, agpt_ctx** out) {
	if (!t || !out) return HostFail("null argument");
	*out = t->tracer->Context();
	return AGPT_OK;
}

int agpt_host_tracer_render(agpt_host_tracer* t, agpt_host_scene* s, int width, int height, float* host_rgba,
		int first_sample, int num_samples, int depth_arg, uint32_t flags, int reupload) {
	if (!t || !s || !host_rgba) return HostFail("null argument");
	g_hostError.clear();
	HOST_TRY(
		if (reupload) t->tracer->Upload(s->scene);
		Accumulator acc(width, height, reinterpret_cast<float3*>(host_rgba));     // the caller's film, in place
		t->tracer->Render(s->scene, *s->camera, acc, first_sample, num_samples, depth_arg, flags);
	)
	return AGPT_OK;
}

int agpt_host_tracer_render_resolve(agpt_host_tracer* t, agpt_host_scene* s, int width, int height, float* host_rgba,
		int samples_so_far, int first_sample, int num_samples, int depth_arg, uint32_t flags, uint32_t* host_rgb8) {
	if (!t || !s || !host_rgba || !host_rgb8) return HostFail("null argument");
	g_hostError.clear();
	HOST_TRY(
		Accumulator acc(width, height, reinterpret_cast<float3*>(host_rgba));
		acc.SetNumSamples(samples_so_far);
		t->tracer->RenderAndResolve(s->scene, *s->camera, acc, first_sample, num_samples, host_rgb8, depth_arg, flags);
	)
	return AGPT_OK;
}

int agpt_host_tracer_render_adaptive(agpt_host_tracer* t, agpt_host_scene* s, int width, int height, float* host_rgba,
		const agpt_adaptive* params, int depth_arg, uint32_t flags, int32_t* host_counts) {
	if (!t || !s || !host_rgba || !params || !host_counts) return HostFail("null argument");
	g_hostError.clear();
	HOST_TRY(
		Accumulator acc(width, height, reinterpret_cast<float3*>(host_rgba));
		std::vector<int> counts;
		t->tracer->RenderAdaptive(s->scene, *s->camera, acc, *params, depth_arg, counts, flags);
		std::copy(counts.begin(), counts.end(), host_counts);
	)
	return AGPT_OK;
}

int agpt_host_tracer_render_adaptive_denoised(agpt_host_tracer* t, agpt_host_scene* s, int width, int height, float* host_rgba,
		const agpt_adaptive* params, const agpt_denoise_params* denoise, int guide_samples, int depth_arg, uint32_t flags, int32_t* host_counts,
		float* out_rgba, uint32_t* out_rgb8) {
	if (!t || !s || !host_rgba || !params || !denoise || !host_counts) return HostFail("null argument");
	g_hostError.clear();
	HOST_TRY(
		Accumulator acc(width, height, reinterpret_cast<float3*>(host_rgba));
		std::vector<int> counts;
		t->tracer->RenderAdaptiveDenoised(s->scene, *s->camera, acc, *params, *denoise, guide_samples, depth_arg, counts,
			reinterpret_cast<float3*>(out_rgba), out_rgb8, flags);
		std::copy(counts.begin(), counts.end(), host_counts);
	)
	return AGPT_OK;
}

// A Camera whose derived vectors are given (a viewer moved it): Export() returns them as they are.
struct GivenCamera : Camera {
	GivenCamera(const CameraDesc& d, const agpt_camera& k) : Camera(d) {
		origin = float3(k.origin[0], k.origin[1], k.origin[2]);
		lower_left_corner = float3(k.lower_left_corner[0], k.lower_left_corner[1], k.lower_left_corner[2]);
		horizontal = float3(k.horizontal[0], k.horizontal[1], k.horizontal[2]);
		vertical = float3(k.vertical[0], k.vertical[1], k.vertical[2]);
		u = float3(k.u[0], k.u[1], k.u[2]);
		v = float3(k.v[0], k.v[1], k.v[2]);
		lens_radius = k.lens_radius;
	}
};

int agpt_host_tracer_render_temporal(agpt_host_tracer* t, agpt_host_scene* s, const agpt_camera* camera, int width, int height, float* host_rgba,
		int first_sample, int num_samples, const agpt_reproject* reproject, const agpt_denoise_params* denoise, int guide_samples, int depth_arg,
		uint32_t flags, float* out_rgba, uint32_t* out_rgb8) {
	if (!t || !s || !host_rgba || !reproject || !denoise) return HostFail("null argument");
	g_hostError.clear();
	HOST_TRY(
		Accumulator acc(width, height, reinterpret_cast<float3*>(host_rgba));
		GivenCamera cam(s->scene.camera, camera ? *camera : s->camera->Export());
		t->tracer->RenderTemporal(s->scene, cam, acc, first_sample, num_samples, *reproject, *denoise, guide_samples, depth_arg,
			reinterpret_cast<float3*>(out_rgba), out_rgb8, flags);
	)
	return AGPT_OK;
}

int agpt_host_tracer_li(agpt_host_tracer* t, agpt_host_scene* s, const float* o, const float* d, int depth_arg, float* out3) {
	if (!t || !s || !o || !d || !out3) return HostFail("null argument");
	g_hostError.clear();
	HOST_TRY(
		float3 r = t->tracer->Li(Ray(float3(o[0], o[1], o[2]), float3(d[0], d[1], d[2])), s->scene, depth_arg);
		out3[0] = r.x; out3[1] = r.y; out3[2] = r.z;
	)
	return AGPT_OK;
}

} // extern "C"
