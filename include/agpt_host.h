/* agpt_host.h -- C ABI of libagpt_host.so: the host-side mirror of the reference's C++ API
 * (ag-pathtracer_b200/host/) made reachable from C / Python (ctypes) for tests and bench.py.
 *
 * The mirror itself is C++ (Scene, Sphere, Plane, TriangleMesh, BVHTriMesh, Camera,
 * DisneyMaterial, MirrorMaterial, AreaLight, UniformInfiniteLight, CudaPathTracer -- same
 * names and constructor arguments as the headers under /root/reference); these entry points build the
 * BASELINE.json configuration scenes through it (host/scenes/config_scenes.h, the same
 * source the oracle compiles against the reference's own headers), flatten them into the
 * tables of agpt.h, upload them, and render through CudaPathTracer::Render -- the call a
 * user of the reference would make instead of looping MyApp::Tick (myapp.cpp:141-187).
 * All compute goes through libagpt.so; nothing here traces or shades on the CPU.
 */
#ifndef AGPT_HOST_H
#define AGPT_HOST_H

#include "agpt.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct agpt_host_scene agpt_host_scene;
typedef struct agpt_host_tracer agpt_host_tracer;

const char* agpt_host_last_error(void);

/* config 1..5 = BASELINE.json configs[0..4]; 6 and 8 = test-only corner-case scenes, 7 = the reference default scene;
 * 9..15 = extension scenes of the host mirror (12: procedural image textures; 13: roughness-metallic and normal maps; 14: alpha masks;
 * 15: emissive materials);
 * level <= 0 picks the configuration's own icosphere subdivision level. */
int agpt_host_scene_create(int config, int level, agpt_host_scene** out);
int agpt_host_scene_destroy(agpt_host_scene* scene);
/* film / integrator defaults of a configuration: out5 = width, height, spp, max_depth, depth_arg */
int agpt_host_config_defaults(int config, int* out5, const char** name);
/* counts4 = primitives, lights, triangles, BVH nodes; bytes = flattened scene size */
int agpt_host_scene_counts(agpt_host_scene* scene, int64_t* counts4, uint64_t* bytes);
/* Scene::Flatten() + agpt_upload_* + agpt_set_camera(Camera(scene.camera)) */
int agpt_host_scene_upload(agpt_host_scene* scene, agpt_ctx* ctx);

/* Borrowed view of the flattened tables (valid while the scene lives): what
 * agpt_host_scene_upload hands to agpt_upload_*; tests feed the same tables to the CPU oracle. */
typedef struct agpt_scene_tables {
	const agpt_prim* prims; int n_prims;
	const agpt_sphere* spheres; int n_spheres;
	const agpt_plane* planes; int n_planes;
	const agpt_mesh_desc* meshes; int n_meshes;
	const agpt_material* materials; int n_materials;
	const agpt_light* lights; int n_lights;
	agpt_camera camera;
	agpt_envmap envmap;      /* width == 0: none */
	const agpt_instance* instances; int n_instances;      /* extension: placed meshes */
	const agpt_texture* textures;                          /* extension: base-colour images (agpt_upload_textures) */
	const int32_t* material_texture;                       /* per material: texture index or -1; NULL when no material has one */
	int n_textures, n_material_texture;
	const agpt_material_textures* material_textures;       /* extension: per material, all its image bindings; NULL as above */
	int n_material_textures;
} agpt_scene_tables;
int agpt_host_scene_tables(agpt_host_scene* scene, agpt_scene_tables* out);
/* extension: the flattened scene's alpha masks (agpt_upload_alpha_masks), one row per material, or (NULL, 0) when no material
 * has one; the texture indices name agpt_scene_tables.textures.  Valid while the scene lives. */
int agpt_host_scene_alpha_masks(agpt_host_scene* scene, const agpt_alpha_mask** out, int* n);
/* extension: the flattened scene's emission rows (agpt_upload_emission), one per material, or (NULL, 0) when no material
 * emits; the texture indices name agpt_scene_tables.textures.  Valid while the scene lives. */
int agpt_host_scene_emission(agpt_host_scene* scene, const agpt_emission** out, int* n);

/* exports for comparison with the oracle's view of the same scene (oracle/ref_harness.cpp) */
int agpt_host_camera_export(agpt_host_scene* scene, float* out19);
int agpt_host_prim_info(agpt_host_scene* scene, int prim, int* kind, int* counts5, int* has_material, int* is_light);
int agpt_host_bvh_export(agpt_host_scene* scene, int prim, void* nodes_out, int* leaf_tri_out);
int agpt_host_mesh_export(agpt_host_scene* scene, int prim, float* tri_verts_out);
int agpt_host_material_export(agpt_host_scene* scene, int prim, float* out20);
/* DisneyMaterial(color, roughness, metallic) / MirrorMaterial(color) -> device record */
int agpt_host_make_material(int type, const float* color3, float roughness, float metallic, agpt_material* out);

/* BVH build settings of the host mirror (SURVEY.md 8f row 3; reference: BuildRecursive +
 * FlattenBVHTree, bvhtrimesh.h:213-330, single-threaded and uncached upstream).
 * threads >= 1 sets the number of builder threads (default: AGPT_BUILD_THREADS, else the
 * hardware concurrency capped at 16); cache_dir != NULL sets the directory flattened BVHs are
 * cached in, "" turns the cache off (default: AGPT_BVH_CACHE_DIR, else off).  The arrays are
 * byte-identical whatever the settings. */
int agpt_host_set_build_options(int threads, const char* cache_dir);
int agpt_host_get_build_options(int* threads, char* cache_dir, int cache_dir_capacity);

/* CudaPathTracer(max_depth, device) */
int agpt_host_tracer_create(int max_depth, int device, agpt_host_tracer** out);
/* CudaPathTracer(max_depth, {devices...}): renders split by sample index over the listed GPUs */
int agpt_host_tracer_create_multi(int max_depth, const int* devices, int n, agpt_host_tracer** out);
int agpt_host_tracer_destroy(agpt_host_tracer* tracer);
int agpt_host_tracer_ctx(agpt_host_tracer* tracer, agpt_ctx** out);
/* CudaPathTracer::Render(scene, Camera(scene.camera), Accumulator(width,height) over
 * host_rgba, first_sample, num_samples, depth_arg): host buffers in, host buffers out.
 * reupload != 0 forces a fresh Scene::Flatten + upload inside the call. */
int agpt_host_tracer_render(agpt_host_tracer* tracer, agpt_host_scene* scene, int width, int height,
		float* host_rgba, int first_sample, int num_samples, int depth_arg, uint32_t flags, int reupload);
/* CudaPathTracer::RenderAndResolve: Render, then Accumulator::CopyToSurface of the film (which holds
 * samples_so_far samples per pixel before the call) into host_rgb8[y*W + x] = 0x00RRGGBB -- the sum over
 * GPUs and the display transform fused in one kernel per GPU. */
int agpt_host_tracer_render_resolve(agpt_host_tracer* tracer, agpt_host_scene* scene, int width, int height, float* host_rgba,
		int samples_so_far, int first_sample, int num_samples, int depth_arg, uint32_t flags, uint32_t* host_rgb8);
/* EXTENSION: CudaPathTracer::RenderAdaptive (agpt.h agpt_adaptive) on a one-device tracer: the film replaces host_rgba,
 * host_counts[y*W + x] (W*H ints) receives each pixel's sample count. */
int agpt_host_tracer_render_adaptive(agpt_host_tracer* tracer, agpt_host_scene* scene, int width, int height, float* host_rgba,
		const agpt_adaptive* params, int depth_arg, uint32_t flags, int32_t* host_counts);
/* EXTENSION: CudaPathTracer::RenderAdaptiveDenoised (agpt.h agpt_render_guides / agpt_denoise): the adaptive frame as above,
 * then the guides of samples [0, guide_samples) and the denoiser; out_rgba (W*H float4) and out_rgb8 (W*H) receive the denoised
 * image in film row order, either may be NULL. */
int agpt_host_tracer_render_adaptive_denoised(agpt_host_tracer* tracer, agpt_host_scene* scene, int width, int height, float* host_rgba,
		const agpt_adaptive* params, const agpt_denoise_params* denoise, int guide_samples, int depth_arg, uint32_t flags, int32_t* host_counts,
		float* out_rgba, uint32_t* out_rgb8);
/* EXTENSION: CudaPathTracer::RenderTemporal (agpt.h agpt_reproject_film) on a one-device tracer: one viewer frame with the
 * camera `camera` (NULL: the scene's own) -- guides, the film and moments of the last such frame carried into this view, samples
 * [first_sample, first_sample + num_samples) added, denoised.  The film replaces host_rgba; out_rgba (W*H float4) and out_rgb8
 * (W*H) receive the denoised image in film row order, either may be NULL. */
int agpt_host_tracer_render_temporal(agpt_host_tracer* tracer, agpt_host_scene* scene, const agpt_camera* camera, int width, int height,
		float* host_rgba, int first_sample, int num_samples, const agpt_reproject* reproject, const agpt_denoise_params* denoise,
		int guide_samples, int depth_arg, uint32_t flags, float* out_rgba, uint32_t* out_rgb8);
/* CudaPathTracer::Li(Ray(o, d), scene, depth_arg) */
int agpt_host_tracer_li(agpt_host_tracer* tracer, agpt_host_scene* scene, const float* o3, const float* d3, int depth_arg, float* out3);

#ifdef __cplusplus
}
#endif
#endif /* AGPT_HOST_H */
