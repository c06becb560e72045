/* agpt.h -- C ABI of the B200-native path-tracing hot path (libagpt.so).
 *
 * The reference (voxel-tracer/ag-pathtracer) has no FFI or plugin layer: its hot path is
 * entered per ray through `virtual float3 Integrator::Li(const Ray&, const Scene&, int depth)`
 * (integrator.h:28-31) and per frame through the pixel loop of `MyApp::Tick`
 * (myapp.cpp:163-175) storing through `Accumulator::AddSample` (myapp.h:17-19).  This header
 * is the boundary the drop-in inserts there: host C++ (the reference's own classes, or the
 * mirror in ag-pathtracer_b200/host/) flattens a Scene once and hands (scene, camera,
 * sample range) to the device; the device hands an accumulator back.
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative
 * agpt_status, with a message in agpt_last_error(); no exceptions cross the boundary; one
 * context per GPU; functions are thread-compatible per context (not thread-safe); all
 * pointers are HOST pointers to caller-owned memory that may be freed when the call
 * returns, unless the name says `_dev`.  There is no CPU fallback: without a usable CUDA
 * device agpt_create() fails and nothing else can be called.
 */
#ifndef AGPT_H
#define AGPT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct agpt_ctx agpt_ctx;

typedef enum agpt_status {
	AGPT_OK = 0,
	AGPT_ERR_INVALID = -1,   /* bad argument or inconsistent scene tables */
	AGPT_ERR_CUDA = -2,      /* CUDA runtime error (message carries cudaGetErrorString) */
	AGPT_ERR_STATE = -3,     /* call order: film / camera / scene not set yet */
	AGPT_ERR_NOMEM = -4
} agpt_status;

/* ---- scene tables ------------------------------------------------------------------ */

/* Verbatim BVHNode of the reference (bvhtrimesh.h:126-130): 32 bytes = 2 x 128-bit loads.
 * count > 0: leaf, `first` = offset of its first triangle in the mesh's leaf-ordered
 * triangle array; count == 0: interior, children at nodes[first] and nodes[first+1]
 * (one 64-byte line, bvhtrimesh.h:175).  Root at 0, slot 1 unused. */
typedef struct agpt_bvh_node {
	float bmin[3];
	float bmax[3];
	int32_t first;
	int32_t count;
} agpt_bvh_node;

/* One TriangleMesh / BVHTriMesh.  Triangles are LEAF-ORDERED: slot j holds the triangle
 * that `primitives[j]` refers to in the reference (bvhtrimesh.h:339), so a leaf reads
 * tri_verts[first .. first+count) directly instead of chasing
 * primitives[].index -> indices[].vertex_index -> vertices[] (SURVEY 8a row 8).
 * n_nodes == 0: plain TriangleMesh, tested brute force in slot order with no bounds test
 * (trianglemesh.h:25-35). */
typedef struct agpt_mesh_desc {
	const agpt_bvh_node* nodes;  /* n_nodes entries, or NULL */
	int32_t n_nodes;
	int32_t n_tris;
	const float* tri_verts;      /* n_tris x 3 x float4: v0 v1 v2; .w unused */
	const int32_t* tri_ids;      /* n_tris: original triangle number (indices[3*id..]) reported in agpt_hit.tri */
	const float* tri_normals;    /* n_tris x 3 x float4 (n0 n1 n2) or NULL: mesh has no normals (trianglemesh.cpp:86) */
	const float* tri_uvs;        /* n_tris x 3 x float2 or NULL: default uvs (0,0),(1,0),(1,1) (trianglemesh.cpp:52-56) */
} agpt_mesh_desc;

typedef struct agpt_sphere {     /* intersectable.h:159-162,319-321 */
	float center[3];
	float r;
	float r2;                    /* radius*radius as the Sphere ctor rounds it */
	float pad[3];
} agpt_sphere;

typedef struct agpt_plane {      /* intersectable.h:119-121,154-156: XZ plane through o, normal +y */
	float o[3];
	float half_x;
	float half_z;
	float pad[3];
} agpt_plane;

enum { AGPT_PRIM_SPHERE = 0, AGPT_PRIM_PLANE = 1, AGPT_PRIM_BVH_MESH = 2, AGPT_PRIM_MESH = 3,
       AGPT_PRIM_INSTANCE = 4 /* EXTENSION: a placed mesh, payload = index into the instance table */ };

/* EXTENSION (SURVEY 8f row 4; BASELINE config 4 says "instanced"): one placement of a mesh.  The reference has no
 * transforms at trace time (scene.h:5-28: a flat list, geometry baked); what an instance means is therefore
 * defined here and stated on the CPU in oracle/agpt_oracle.cpp (parity is against that, not against the reference):
 *   - the ray is taken to object space, O' = W2O * (O,1), D' = W2O * (D,0), D' NOT re-normalised, so the ray
 *     parameter t is the same in both spaces and ray.t is shared with the rest of the scene;
 *   - BVHTriMesh::Intersect / IntersectP run unchanged on (O', D', t) over the shared mesh;
 *   - the hit point is O + t*D (world ray); the triangle's vertices go to world space through O2W before the
 *     partial derivatives are formed, the interpolated shading normal goes through transpose(W2O).
 * Matrices are 3x4 row-major affine, rows of [R | t]; products are summed left to right ((m0*x + m1*y) + m2*z) + m3. */
typedef struct agpt_instance {
	int32_t mesh;                  /* index into the mesh table (shared by any number of instances) */
	int32_t pad[3];
	float object_to_world[12];
	float world_to_object[12];
} agpt_instance;

/* Scene::primitives in list order (scene.h:5-13,27): order decides exact-t ties. */
typedef struct agpt_prim {
	int32_t type;        /* AGPT_PRIM_* */
	int32_t payload;     /* index into the spheres / planes / meshes table of that type */
	int32_t material;    /* index into materials, -1 = nullptr material (emissive shape, integrator.h:152-161) */
	int32_t area_light;  /* index into lights of the AreaLight wrapping this shape, -1 = none; that light's
	                        `prim` must be this row (one shape per AreaLight, as upstream), else AGPT_ERR_INVALID */
} agpt_prim;

enum { AGPT_MAT_DISNEY = 1, AGPT_MAT_MIRROR = 2, AGPT_MAT_GLASS = 3 /* EXTENSION: rough dielectric */ };
enum { AGPT_LOBE_DIFFUSE = 1, AGPT_LOBE_RETRO = 2, AGPT_LOBE_MICROFACET = 4, AGPT_LOBE_SPECULAR = 8,
       /* EXTENSION (SURVEY 8f row 4; BASELINE config 5 says "rough-glass"): a rough dielectric interface as PBRT-v3's GlassMaterial
        * builds it.  GLASS_REFLECT is the reference's own MicrofacetReflection (reflection.h:38-78) over its plain
        * TrowbridgeReitzDistribution (G = 1/(1 + Lambda(wo) + Lambda(wi)), microfacet.h:103-105) and its FresnelDielectric(1, eta)
        * (microfacet.h:220-228).  GLASS_TRANSMIT -- MicrofacetTransmission (PBRT-v3 reflection.cpp, radiance transport) -- and the
        * rule that a transmission lobe contributes to BSDF::f when wi and wo lie on opposite sides of the geometric normal do not
        * exist upstream (its BSDF::f only sums when both lie on the same side, reflection.h:114-123): parity for those is against
        * oracle/agpt_oracle.cpp only.  bxdfs[] order: GLASS_REFLECT, GLASS_TRANSMIT. */
       AGPT_LOBE_GLASS_REFLECT = 16, AGPT_LOBE_GLASS_TRANSMIT = 32 };

/* Constants the reference's material constructors derive once (material.h:14-49,74-77). */
typedef struct agpt_material {
	int32_t type;         /* AGPT_MAT_* */
	uint32_t lobes;       /* AGPT_LOBE_* in BSDF::bxdfs[] order: diffuse, retro, microfacet | specular */
	float roughness;      /* DisneyRetro::roughness */
	float metallic;       /* DisneyFresnel::metallic */
	float diffuse_r[3];   /* (1-metallic)*color: R of DisneyDiffuse and DisneyRetro; GLASS: T of the transmission lobe */
	float eta;            /* 1.5 (material.h:65) */
	float spec_r0[3];     /* DisneyFresnel::R0 = Lerp(metallic, SchlickR0FromEta(eta), color) */
	float alpha_x;        /* max(.001, roughness^2) */
	float mirror_r[3];    /* SpecularReflection::R; GLASS: R of the reflection lobe */
	float alpha_y;
} agpt_material;

enum { AGPT_LIGHT_AREA = 0, AGPT_LIGHT_UNIFORM_INFINITE = 1, AGPT_LIGHT_INFINITE_AREA = 2 };

/* agpt_light.flags */
enum {
	/* EXTENSION (not reference behaviour: upstream's Plane and TriangleMesh inherit Sample / Pdf stubs that return pdf 0,
	 * so an emissive quad or mesh lights only what sees it directly or through a mirror).  On an AGPT_LIGHT_AREA light
	 * whose shape is an AGPT_PRIM_PLANE, AGPT_PRIM_MESH or AGPT_PRIM_BVH_MESH, next-event estimation samples the shape,
	 * as PBRT-v3's Shape::Sample / Shape::Pdf do, stated on the CPU in oracle/agpt_shape_oracle.cpp:
	 *   - the whole mesh is one light: a triangle is picked by Distribution1D::SampleDiscrete(uLight.x) over the triangle
	 *     areas 0.5 * |cross(v1 - v0, v2 - v0)| in slot (leaf) order, and the remapped uLight.x with uLight.y picks a point
	 *     by UniformSampleTriangle; degenerate triangles (the ones a hit would reject) have area 0 and are never picked;
	 *     a plane picks a uniform point of its rectangle, o + ((2 u.x - 1) half_x, 0, (2 u.y - 1) half_z);
	 *   - the light normal is the geometric one (plane: +y), emission stays two-sided, the solid-angle pdf is
	 *     dist^2 / (|cos| * total area) and 0 where the cosine is 0 or the total area is 0;
	 *   - the MIS pdf (Pdf_Li) intersects the MIS ray with the light's shape ALONE and is 0 when it misses;
	 *   - only the two uLight numbers the vertex draws anyway are used: every later draw of a path stays where it was.
	 * Without the flag a scene renders exactly as the reference does; on a sphere the flag changes nothing (spheres are
	 * sampled already).  The flag on a non-area light, on an instanced shape (AGPT_PRIM_INSTANCE) or any other bit set
	 * is refused with AGPT_ERR_INVALID. */
	AGPT_LIGHT_SAMPLE_SHAPE = 1u
};

/* Scene::lights in list order (lights.h:37-51,72-87). */
typedef struct agpt_light {
	int32_t type;        /* AGPT_LIGHT_* */
	int32_t prim;        /* AREA: scene primitive index of the emitting shape; else -1 */
	uint32_t flags;      /* AGPT_LIGHT_SAMPLE_SHAPE or 0 */
	float pad;
	float lemit[3];
	float pad2;
} agpt_light;

/* InfiniteAreaLight (lights.h:52-70, lights.cpp:31-112): lat-long HDR map (HDRTexture,
 * texture.h:41-84) plus the piecewise-constant distribution over its texels (Distribution1D,
 * sampling.h:20-69) that the light's constructor builds (lights.cpp:33-47).  One per scene. */
typedef struct agpt_envmap {
	int32_t width, height;
	const float* rgb;        /* width*height x 3 floats, row-major, as stbi_loadf decodes the .hdr */
	const float* func;       /* width*height: max(r,g,b) * sin(theta_row) */
	const float* cdf;        /* width*height + 1 */
	float func_int;          /* Distribution1D::funcInt */
} agpt_envmap;

/* Derived camera vectors exactly as Camera::updateCoords leaves them (camera.h:77-90);
 * computed on the host (tan, double->float), the device only adds and multiplies. */
typedef struct agpt_camera {
	float origin[3];
	float lower_left_corner[3];
	float horizontal[3];
	float vertical[3];
	float u[3];
	float v[3];
	float lens_radius;
} agpt_camera;

typedef struct agpt_hit {
	uint32_t found;
	int32_t prim;        /* index in Scene::primitives */
	int32_t tri;         /* original triangle number inside that mesh, -1 for sphere / plane */
	float t;
} agpt_hit;

typedef struct agpt_stats {
	uint64_t paths;            /* camera paths started */
	uint64_t rays_closest;     /* path rays through Scene::Intersect (integrator.h:136), skip-through rays included */
	uint64_t rays_shadow;      /* any-hit visibility rays (integrator.h:50) */
	uint64_t rays_mis;         /* closest-hit MIS rays (integrator.h:79) */
	uint64_t rays_skip;        /* of rays_closest: continuation through null-material shapes (integrator.h:158) */
	uint64_t rays_mis_culled;  /* MIS rays the reference traces but that provably cannot reach their light: not traced, not counted above.
	                            * Exact in renders made with AGPT_FLAG_COUNTERS; otherwise an upper bound (such samples are dropped before their BSDF
	                            * value is known, and the reference does not trace a sample whose value is black) */
	uint64_t rays_tail_culled; /* path rays the reference traces at bounces == MaxDepth and then discards (integrator.h:139,150): not traced, not counted above.
	                            * 0 while an emitting row is bound (agpt_upload_emission): those rays may hit an emitter, so they are traced and
	                            * counted in rays_closest */
	/* traversal work, only counted with AGPT_FLAG_COUNTERS; [0] closest-hit kernel, [1] any-hit kernel */
	uint64_t node_visits[2];   /* interior sibling pairs fetched (64 B each) */
	uint64_t box_tests[2];
	uint64_t tri_tests[2];     /* triangles fetched and tested (48 B each) */
	uint64_t analytic_tests[2];/* sphere / plane records tested (32 B each) */
	uint64_t warp_steps[2];    /* trips of the lockstep BVH walk, counted once per warp */
	uint64_t lane_steps[2];    /* lanes that had work in those trips: lane_steps / warp_steps = rays alive per step (of 32) */
	uint64_t kernel_launches;  /* launches of this library's kernels since agpt_reset_stats */
	uint64_t launches_closest; /* of which closest-hit trace, any-hit trace, shade */
	uint64_t launches_any;
	uint64_t launches_shade;
	uint64_t waves;            /* wavefront iterations */
	float ms_render;           /* device time of agpt_render calls (CUDA events on the context stream) */
	float ms_trace_closest;    /* per kernel class, only with AGPT_FLAG_TIMING */
	float ms_trace_any;
	float ms_shade;
	float ms_other;            /* ms_render minus the three above (generate, accumulate, queue bookkeeping) */
	float ms_reduce;           /* device time of this context's share of agpt_reduce_* / agpt_allreduce_* calls */
	uint32_t reduce_path;      /* how the last one ran: 1 = this library's peer-memory kernels, 2 = ncclAllReduce */
} agpt_stats;

/* agpt_render / agpt_trace_* flags */
enum {
	AGPT_FLAG_COUNTERS = 1u,      /* count node visits / box / triangle tests (slower kernels) */
	AGPT_FLAG_TIMING = 2u,        /* bracket every kernel class with CUDA events (serialises) */
	AGPT_FLAG_STRICT_BOXES = 4u,  /* every slab test with the reference's six IEEE divisions; the default is the
	                                 exact-filtered test (same decisions, divisions only inside a guard band) */
	AGPT_FLAG_RAYS_FINAL = 8u,    /* agpt_trace_rays / agpt_li_rays: directions are used as given -- the rays come from host
	                                 Ray objects, whose constructor has normalised them already (camera.h:7) */
	AGPT_FLAG_RR_BY_BOUNCE = 16u  /* EXTENSION (SURVEY 8f row 4; not reference behaviour): Russian roulette keyed on the path's own
	                                 bounce index -- live once bounces > 3, the rule BASELINE config 5 names ("16 bounces with Russian
	                                 roulette") -- instead of on Li's constant depth argument (integrator.h:180, dead for depth = 0).
	                                 rr_depth_arg is ignored.  Checked against oracle/agpt_oracle.cpp, the only statement of it. */
};

/* ---- lifecycle --------------------------------------------------------------------- */

int agpt_create(int device, agpt_ctx** out);                 /* fails loudly without CUDA */
int agpt_destroy(agpt_ctx* ctx);
const char* agpt_last_error(void);
int agpt_device_count(int* out);
/* Launch on the caller's CUDA stream (cudaStream_t as void*); NULL = the context's own. */
int agpt_set_stream(agpt_ctx* ctx, void* cuda_stream);

/* ---- scene upload (replaces the Scene the reference keeps in host memory, scene.h:27-29) */

int agpt_upload_meshes(agpt_ctx* ctx, const agpt_mesh_desc* meshes, int n);
int agpt_upload_spheres(agpt_ctx* ctx, const agpt_sphere* spheres, int n);
int agpt_upload_planes(agpt_ctx* ctx, const agpt_plane* planes, int n);
int agpt_upload_primitives(agpt_ctx* ctx, const agpt_prim* prims, int n);
int agpt_upload_instances(agpt_ctx* ctx, const agpt_instance* instances, int n);  /* EXTENSION; rows of AGPT_PRIM_INSTANCE point here */
int agpt_upload_materials(agpt_ctx* ctx, const agpt_material* materials, int n);
int agpt_upload_lights(agpt_ctx* ctx, const agpt_light* lights, int n);   /* refuses bad flags (see agpt_light.flags), scene unchanged */
int agpt_upload_envmap(agpt_ctx* ctx, const agpt_envmap* env);          /* NULL clears it;
                                                                           a refused map (AGPT_ERR_INVALID) leaves the resident one */

/* ---- image textures on the base colour of Disney materials (EXTENSION: the reference has one colour per material) -------
 * A texture is linear RGB float32, row-major: texel (x, y) at rgb[3 * (y * width + x) ..]; row 0 holds v in [0, 1/height).
 * material_texture[i] is the base-colour texture of material i (an index into `textures`) or -1.  At a hit on a material with
 * a texture, float32 with every operation rounded on its own:
 *   1. surface uv (P = the hit point O + t * D the surface is built from):
 *      - sphere: phi = atan2f(pHit.y, pHit.x), phi = phi < 0 ? phi + 2pi : phi; u = phi / 2pi, v = theta / pi, where pHit and
 *        theta are those of Sphere's SurfaceInteraction (pHit = P - centre, x nudged to EPSILON * r at the poles; theta =
 *        acos(clamp(pHit.z / r, -1, 1))) and atan2f is Sun fdlibm's e_atan2f.c in float (2pi, pi: the float constants);
 *      - plane: u = ((P.x - o.x) / half_x + 1) * 0.5, v = ((P.z - o.z) / half_z + 1) * 0.5;
 *      - triangle (instances: their mesh's uvs): b0 = 1 - b1 - b2, u = (b0 * uv0.u + b1 * uv1.u) + b2 * uv2.u, the same for v,
 *        with the mesh's uvs or the default (0,0), (1,0), (1,1);
 *   2. lookup, bilinear and repeat-wrapped, texel centres at (i + 0.5) / W:
 *        u' = isfinite(u) ? u - floorf(u) : 0 (the same for v); s = u' * W - 0.5, x0 = (int)floorf(s), fx = s - floorf(s),
 *        x1 = x0 + 1, each wrapped by x < 0 ? x + W : x >= W ? x - W : x (the same for t = v' * H - 0.5, y0, y1, fy);
 *        a = T00 + fx * (T10 - T00), b = T01 + fx * (T11 - T01), c = a + fy * (b - a), Tij = texel (xi, yj)
 *      (a constant texture returns its colour exactly; no random number is drawn: every path's draws stay where they were);
 *   3. c replaces the colour of DisneyMaterial(color, roughness, metallic) (host/material.h) in its arithmetic:
 *        dw = (1 - metallic) * (1 - 0); diffuse_r = dw > 0 ? dw * c : 0;  spec_r0 = Lerp(metallic, r0, c) = (1 - metallic) * r0
 *        + metallic * c, r0 = ((eta - 1) * (eta - 1)) / ((eta + 1) * (eta + 1));
 *      roughness, metallic, the alphas and the lobe set stay as the record has them;
 *   4. agpt_render_guides' albedo of such a hit is that diffuse_r + spec_r0 (then clamped as for every material).
 * Refused with AGPT_ERR_INVALID, leaving the resident textures as they were: a width or height < 1, width * height > 2^28, a
 * NULL rgb, a texel that is not finite, an entry of material_texture outside [-1, n_textures).  (NULL, 0, NULL, 0) clears the
 * textures.  Like every upload it makes the guides stale and drops the saved reprojection view.  At render time (with any
 * binding >= 0) n_materials must equal the resident material count and every bound material must be AGPT_MAT_DISNEY, else
 * AGPT_ERR_INVALID.  agpt_scene_bytes counts the texels (16 bytes each on the device) and the two small tables.
 * statements/agpt_texture_oracle.cpp states the same on the CPU. */
typedef struct agpt_texture {
	int32_t width, height;
	const float* rgb;        /* width * height * 3 floats */
} agpt_texture;
int agpt_upload_textures(agpt_ctx* ctx, const agpt_texture* textures, int n_textures, const int32_t* material_texture, int n_materials);

/* ---- roughness-metallic and normal maps on Disney materials (EXTENSION, beside the base-colour texture above) ----------
 * bindings[i] binds material i's maps, each an index into `textures` or -1.  agpt_upload_textures(t, n, material_texture, m)
 * is this call with only `base` set (roughness_metallic = normal = -1, normal_scale = 1, color = 0): one upload path, the same
 * refusals.  Every map is read with the uv and the lookup of agpt_upload_textures steps 1-2.  At a hit on material i, float32
 * with every operation rounded on its own:
 *   1. per-hit material.  roughness_metallic < 0: the material of agpt_upload_textures step 3 (record, or record with the base
 *      texture's colours).  Otherwise, with c the looked-up roughness-metallic texel and C the base texture's value when
 *      base >= 0, else `color`:
 *        r = roughness * clamp(c.y, 0, 1), k = metallic * clamp(c.z, 0, 1)  (clamp(x, lo, hi) = x < lo ? lo : x > hi ? hi : x;
 *        the record's roughness and metallic act as glTF factors; c.x is unused), then DisneyMaterial's constructor arithmetic
 *        (host/material.h) on (C, r, k): dw = (1 - k) * (1 - 0); lobes = (dw > 0 ? DIFFUSE | RETRO : 0) | MICROFACET;
 *        diffuse_r = dw > 0 ? dw * C : 0; alpha_x = alpha_y = max(.001, max(.001, r * r)); roughness = r; metallic = k;
 *        spec_r0 = Lerp(k, r0, C), r0 = ((eta - 1) * (eta - 1)) / ((eta + 1) * (eta + 1)).  The lobe set, and with it the lobe
 *        count and the lobe choice of Sample_f, can change from hit to hit.  A map of texels (x, 1, 1) with `color` equal to the
 *        material's own colour gives back its record bit for bit.
 *   2. normal map (normal >= 0), applied to the surface before the BSDF frame is built; emission, the light choice and the
 *      geometric normal (and with it every ray offset and Pdf_Li test) are unchanged, and whatever reads shading.n after this
 *      step (the cosine factors, UniformInfiniteLight's hemisphere) reads the mapped one.  c = the looked-up texel (linear, no sRGB decode; +y points along increasing v), s =
 *      normal_scale: n_ts = (s * (2 * c.x - 1), s * (2 * c.y - 1), 2 * c.z - 1).  T = dp/du and B = dp/dv of the texture's uv:
 *        - sphere: dpdu = (-2pi * pHit.y, 2pi * pHit.x, 0) and dpdv = pi * (pHit.z * cosPhi, pHit.z * sinPhi, -r * sin(theta))
 *          of Sphere's SurfaceInteraction, before its swap (the swapped pair is what shading.dpdu holds);
 *        - plane: T = (1, 0, 0), B = (0, 0, 1);
 *        - triangle: dpdu, dpdv of TriangleDerivatives (trianglemesh.cpp:59-80), from world-space vertices for instances.
 *      N = shading.n as the shape produces it (interpolated normals included).  Then
 *        T' = T - N * dot(N, T); if dot(T', T') == 0 the surface is left as it is; T' = normalize(T');
 *        B' = cross(N, T'), negated if dot(B', B) < 0;  n = (n_ts.x * T' + n_ts.y * B') + n_ts.z * N;
 *        if !(dot(n, N) > 0) the surface is left as it is; n = normalize(n);
 *        shading.n = n, shading.dpdu = T' - n * dot(n, T')   (the BSDF frame: ns = n, ss = normalize(shading.dpdu), ts = cross)
 *      A texel with n_ts.x == 0 && n_ts.y == 0 && n_ts.z > 0 (flat; normal_scale = 0 included) leaves the surface bit for bit.
 *   3. agpt_render_guides: the normal guide is the mapped shading.n (flipped toward the camera as for every hit), the albedo
 *      the per-hit diffuse_r + spec_r0 (then clamped).
 * No random number is drawn: every path's draws stay where they were.  Refused with AGPT_ERR_INVALID, leaving the resident
 * textures as they were: everything agpt_upload_textures refuses, an index outside [-1, n_textures), a normal_scale or color
 * that is not finite.  Like every upload it makes the guides stale and drops the saved reprojection view.  At render time
 * (with any map bound) n_materials must equal the resident material count and every material with a map must be
 * AGPT_MAT_DISNEY, else AGPT_ERR_INVALID.  statements/agpt_material_maps_oracle.cpp states the same on the CPU. */
typedef struct agpt_material_textures {
	int32_t base;                /* base-colour texture or -1 (what agpt_upload_textures binds) */
	int32_t roughness_metallic;  /* texture or -1: G = roughness, B = metallic (glTF layout); R unused */
	int32_t normal;              /* tangent-space normal map or -1 */
	float normal_scale;          /* glTF normalTexture.scale; finite */
	float color[3];              /* the material's base colour, used when base < 0 and roughness_metallic >= 0 */
} agpt_material_textures;
int agpt_upload_material_textures(agpt_ctx* ctx, const agpt_texture* textures, int n_textures,
                                  const agpt_material_textures* bindings, int n_materials);

/* ---- alpha masks: cutout geometry (EXTENSION: glTF alphaMode MASK; the reference's surfaces are solid everywhere) --------
 * masks[i] applies to material i of any type (Disney, mirror, glass): the mask is geometry, not BSDF.  Its alpha is channel
 * `channel` (0, 1, 2) of resident texture `texture` (agpt_upload_textures / agpt_upload_material_textures), which needs no
 * base or map binding of its own; -1: no mask.  A candidate hit on a primitive whose material has a mask -- one the test of
 * its ray accepts (closest-hit: the triangle or plane test and the degenerate-triangle test; any-hit: the triangle or plane
 * test) -- is then, in float32 with every operation rounded on its own:
 *   1. given a uv by agpt_upload_textures step 1: triangle b0 = 1 - b1 - b2, (b0 * uv0 + b1 * uv1) + b2 * uv2 with the mesh's
 *      uvs or the default ones (instances: their mesh's uvs and the object-space barycentrics); plane ((P - o) / half + 1) * 0.5
 *      with P = O + t * D;
 *   2. looked up by agpt_upload_textures step 2 (bilinear, repeat-wrapped, nested lerp), keeping channel `channel`: alpha;
 *   3. kept iff alpha >= cutoff.  Otherwise it is as if the triangle or plane test had returned false: ray.t is unchanged and
 *      the walk goes on, in the reference's order and with its tie rules.
 * The rule holds for every ray through Scene::Intersect / IntersectP: path, MIS and shadow rays, agpt_trace_primary,
 * agpt_trace_rays, agpt_li_*, and the rays of agpt_render_guides.  No random number is drawn: every path's draws stay where
 * they were.  Refused with AGPT_ERR_INVALID, leaving the resident masks as they were: a texture outside [-1, resident
 * textures), a channel outside [0, 2], a cutoff that is not finite.  (NULL, 0) clears the masks, and so does every successful
 * texture upload (the indices name the old table).  Like every upload it makes the guides stale and drops the saved
 * reprojection view.  At render time (with any mask bound) n_materials must equal the resident material count, and no
 * primitive whose material has a mask may be a sphere or have area_light >= 0 (masked spheres and emitters are not defined),
 * else AGPT_ERR_INVALID.  agpt_scene_bytes counts the mask table (16 bytes per material).  Scenes without a mask run the trace
 * kernels they ran before; with one, trace runs instantiations that add the test.  statements/agpt_alpha_oracle.cpp states
 * the same on the CPU. */
typedef struct agpt_alpha_mask {
	int32_t texture;   /* index into the resident textures, or -1: no mask */
	int32_t channel;   /* 0, 1, 2: which channel of that texture is the alpha */
	float cutoff;      /* glTF alphaCutoff: the surface is there where alpha >= cutoff; finite */
	int32_t pad;
} agpt_alpha_mask;
int agpt_upload_alpha_masks(agpt_ctx* ctx, const agpt_alpha_mask* masks, int n_materials);

/* ---- emissive materials (EXTENSION: glTF emissiveFactor / emissiveTexture, KHR_materials_emissive_strength folded into the
 * factor; the reference's only emitters are AreaLights around null-material shapes) ---------------------------------------
 * rows[i] belongs to material i of any type (Disney, mirror, glass); the material keeps its BSDF.  A row EMITS iff some factor
 * component is > 0.  Its emitted radiance at a hit, in float32 with every operation rounded on its own:
 *   texture < 0:  E = factor;
 *   otherwise:    E_c = factor_c * T_c, T = the lookup (agpt_upload_textures step 2: bilinear, repeat-wrapped, nested lerp) of
 *                 resident texture `texture` at the hit's uv (agpt_upload_textures step 1: sphere, plane, triangle; instances
 *                 through their mesh's uvs).  Texels are linear (no sRGB decode).  Emission is two-sided.
 * The one new term of Li: at every vertex where the path ray has a closest hit, at bounce indices 0 .. max_depth whatever
 * specularBounce says, on a primitive whose material >= 0 emits, L = L + beta * E -- after that vertex's area-light / sky term
 * and before the bounces >= maxDepth break.  Skip-through (null-material) hits never emit, and candidates an alpha mask
 * rejects are not hits.  No random number is drawn: every path's draws stay where they were.
 * Emissive materials are not lights: they are not in the light list, UniformSampleOneLight never picks them, and a shadow or
 * MIS ray that hits one sees an occluder as before.  Their light reaches other surfaces only through BSDF-sampled
 * continuations: unbiased, but noisier than next-event estimation for small bright emitters.  Because the path ray at
 * bounces == max_depth may now hit an emitter, it is traced while an emitting row is bound (it counts in rays_closest, and
 * rays_tail_culled stays 0).
 * Refused with AGPT_ERR_INVALID, leaving the resident table as it was: n_materials < 0, rows == NULL with n_materials > 0, a
 * texture outside [-1, resident textures), a factor component that is not finite or is < 0.  (NULL, 0) clears the table, and
 * so does every successful texture upload (the indices name the old table).  Like every upload it makes the guides stale and
 * drops the saved reprojection view.  At render time (with an emitting row bound) n_materials must equal the resident
 * material count, and no primitive whose material emits may have area_light >= 0 (an area light's Le and a material's
 * emission on one shape are not defined), else AGPT_ERR_INVALID.  agpt_scene_bytes counts the table (16 bytes per material).
 * agpt_render_guides ignores emission: the albedo guide stays the reflectance.  agpt_render, agpt_li_pixels, agpt_li_rays,
 * adaptive rendering and agpt_render_multi all include the term.  Scenes without an emitting row run the shade kernels they ran
 * before.  statements/agpt_emission_oracle.cpp states the same on the CPU. */
typedef struct agpt_emission {
	int32_t texture;   /* index into the resident textures, or -1: constant emission */
	float factor[3];   /* linear RGB radiance scale (glTF emissiveFactor x emissive strength); finite, >= 0 */
} agpt_emission;     /* 16 bytes */
int agpt_upload_emission(agpt_ctx* ctx, const agpt_emission* rows, int n_materials);

int agpt_set_camera(agpt_ctx* ctx, const agpt_camera* camera);          /* Camera, camera.h:38-56 */
int agpt_set_film(agpt_ctx* ctx, int width, int height);                /* Accumulator(w,h), myapp.h:10-13 */
int agpt_scene_bytes(agpt_ctx* ctx, uint64_t* out);                     /* resident scene bytes in HBM */

/* ---- the hot path -------------------------------------------------------------------- */

/* num_samples iterations of the MyApp::Tick pixel loop (myapp.cpp:163-175) for sample
 * indices [first_sample, first_sample+num_samples) stepping by sample_stride (1 on one GPU,
 * G when G GPUs split the samples s = g mod G), PathTracer(max_depth)::Li(ray, scene,
 * rr_depth_arg) per pixel, accumulated into the device float4[W*H] accumulator. */
int agpt_render(agpt_ctx* ctx, int first_sample, int num_samples, int sample_stride,
		int max_depth, int rr_depth_arg, uint32_t flags);

/* Hit table of the camera rays of one sample index: out_host[y*W + x] (parity gate). */
int agpt_trace_primary(agpt_ctx* ctx, int sample, uint32_t flags, agpt_hit* out_host);

/* Scene::Intersect (any_hit = 0) / Scene::IntersectP (any_hit != 0) for caller rays:
 * rays7 = O.xyz, D.xyz (normalised on the device like the Ray ctor, camera.h:7, unless AGPT_FLAG_RAYS_FINAL), tmax. */
int agpt_trace_rays(agpt_ctx* ctx, int64_t n, const float* rays7, int any_hit, uint32_t flags, agpt_hit* out_host);

/* Radiance of single camera paths without accumulation (Integrator::Li for the debug
 * click, myapp.cpp:196-198): pixel (xs[i], ys[i]), sample ss[i] -> out_rgb[3*i..]. */
int agpt_li_pixels(agpt_ctx* ctx, int n, const int* xs, const int* ys, const int* ss,
		int max_depth, int rr_depth_arg, uint32_t flags, float* out_rgb);

/* Integrator::Li(ray, scene, depth) for caller-supplied rays (integrator.h:28-31): rays7 as
 * in agpt_trace_rays, rng_states[i] = xorshift32 state the path starts from (the reference
 * draws from its one global generator instead). */
int agpt_li_rays(agpt_ctx* ctx, int n, const float* rays7, const uint32_t* rng_states,
		int max_depth, int rr_depth_arg, uint32_t flags, float* out_rgb);

/* ---- accumulator (Accumulator, myapp.h:8-68) ----------------------------------------- */

int agpt_clear(agpt_ctx* ctx);                                  /* Accumulator::Clear */
int agpt_accum_ptr_dev(agpt_ctx* ctx, void** dev_ptr);          /* float4[W*H] in HBM, row (H-1-y): for NCCL */
int agpt_set_accum_dev(agpt_ctx* ctx, void* dev_ptr);           /* accumulate into caller-owned device memory */
int agpt_read_accum(agpt_ctx* ctx, float* host_rgba);           /* D2H of float4[W*H] */
int agpt_write_accum(agpt_ctx* ctx, const float* host_rgba);    /* H2D (resume) */
/* The same upload, started and not waited for: it runs beside the agpt_render that follows (the film is only needed when a
 * batch is added to it, at the end) -- the batched Tick of CudaPathTracer::Render hides its H2D copy this way.  The host buffer
 * must stay untouched until the next call on this context that reads or writes the film returns (agpt_render, agpt_read_accum,
 * agpt_resolve, the reduce calls ...: each waits for the upload first).  Page-locked memory (agpt_host_alloc) for a true overlap. */
int agpt_write_accum_begin(agpt_ctx* ctx, const float* host_rgba);
/* Accumulator::CopyToSurface (myapp.h:34-41): /samples, pow(1/2.2), 8-bit pack 0x00RRGGBB. */
int agpt_resolve(agpt_ctx* ctx, int samples, uint32_t* host_rgb8);

/* ---- adaptive sampling (EXTENSION: the reference gives every pixel the same number of samples) ----------------------
 * Per-pixel moments: a second float4[W*H] owned by the context, in the film's row order (row H-1-y).  .xyz = sum of c*c per
 * channel and .w = n, the number of samples added (a float: exact up to 2^24), where c is each sample after the film's filter
 * (a sample with a NaN channel or an infinite luminance adds 0, and still counts in n), added in ascending sample order like
 * the film.  Off by default; while off, nothing about the film or the kernels that run changes.  On: the buffer is allocated
 * and zeroed, re-allocated (zeroed) by agpt_set_film and zeroed by agpt_clear, and agpt_render (any stride) adds the samples
 * it renders.  agpt_write_accum*, agpt_set_accum_dev and the multi-GPU reduce calls leave it alone: after them the caller
 * owns the consistency between film and moments. */
int agpt_set_moments(agpt_ctx* ctx, int enable);
int agpt_read_moments(agpt_ctx* ctx, float* host_rgba);            /* D2H of float4[W*H]; AGPT_ERR_STATE while moments are off */
/* H2D of float4[W*H] (resume, with agpt_write_accum).  Every .w must be an integer in [0, 2^24] (NaN and inf are not), else
 * AGPT_ERR_INVALID and the moments stay as they were; AGPT_ERR_STATE while moments are off.  Like agpt_write_accum, it leaves
 * fresh guides fresh. */
int agpt_write_moments(agpt_ctx* ctx, const float* host_rgba);

/* Convergence test.  Valid: 2 <= min_samples <= max_samples <= 1<<24, step >= 1, tolerance and floor finite and >= 0
 * (else AGPT_ERR_INVALID).  Pixel p, with film sum a, moments q and count n, is SELECTED (needs `step` more samples) iff
 * n + step <= max_samples and, for at least one channel, in float32 with every operation rounded on its own:
 *     mu = a / n;  d = q - a * mu;  v = d / (n - 1);  v = v < 0 ? 0 : v;  se = sqrt(v / n);
 *     thr = tolerance * (mu > floor ? mu : floor);  !(se <= thr)
 * (a NaN v stays NaN: a pixel whose se is not finite keeps sampling until max_samples).  oracle/adaptive.py states the same
 * rule element for element. */
typedef struct agpt_adaptive {
	int32_t min_samples, max_samples, step;
	float tolerance;   /* relative standard error of the pixel mean that is good enough */
	float floor;       /* darker pixels are held to tolerance * floor instead of tolerance * mean */
} agpt_adaptive;
/* Runs the test over the film on the device and leaves the compacted list of selected pixels there; *n_out = its length,
 * pixels_out (NULL, or W*H entries) receives the film pixel indices y*W + x.  The order of the list is unspecified (8x4 tiles
 * stay together) and never affects results. */
int agpt_adaptive_select(agpt_ctx* ctx, const agpt_adaptive* params, int32_t* pixels_out, int* n_out);
/* A frame from scratch: clears film and moments, renders samples [0, min_samples) of every pixel (agpt_render), then
 * repeats { agpt_adaptive_select; samples [n_p, n_p + step) of every selected pixel } until nothing is selected, at most
 * (max - min) / step rounds.  Each pixel of the result equals, bit for bit, the same pixel of agpt_render(0, n_p) on a cleared
 * film, n_p being its final count (moments .w): every draw of a path depends only on its pixel and sample index, and the film
 * adds a pixel's samples in ascending order whatever the batches.  *rounds_out (may be NULL) = selection rounds that rendered
 * something, *paths_out (may be NULL) = camera paths of the whole frame.  AGPT_ERR_STATE with moments off or without film,
 * scene or camera; a refused call leaves film and moments as they were. */
int agpt_render_adaptive(agpt_ctx* ctx, const agpt_adaptive* params, int max_depth, int rr_depth_arg, uint32_t flags,
		int* rounds_out, int64_t* paths_out);
/* agpt_resolve with each pixel's own sample count: ResolvePixel(film[i], moments[i].w); a pixel with n = 0 resolves to 0. */
int agpt_resolve_counts(agpt_ctx* ctx, uint32_t* host_rgb8);

/* ---- denoising (EXTENSION: the reference only divides the film by the sample count) ----------------------------------
 * Guide buffers: what the camera rays of samples [0, num_samples) of every pixel hit first -- the rays agpt_render starts
 * those samples with (same StreamSeed, CameraRay, jitter and lens draws), traced by the closest-hit kernels (flags:
 * AGPT_FLAG_COUNTERS, AGPT_FLAG_STRICT_BOXES).  Two context-owned float4[W*H] in the film's row order (row H-1-y):
 *   albedo:       .xyz = mean albedo, .w = fraction of the samples that hit something;
 *   normal/depth: .xyz = mean normal (not renormalised: shorter than 1 where the samples disagree), .w = mean hit distance t
 *                 over the samples that hit, 0 if none hit.
 * One sample: the FIRST hit of its camera ray, no skip-through.
 *   - a miss: albedo (1,1,1), normal 0, no depth (adds nothing to the hit count or the t sum);
 *   - a hit: normal = the shading normal sn of the surface rebuilt as shade rebuilds it (instances included), flipped to face
 *     the ray: dot(sn, D) > 0 ? -sn : sn; albedo by material, each channel then clamped as a < 1 ? a : 1:
 *     null material (an emitter) (1,1,1); AGPT_MAT_MIRROR mirror_r; AGPT_MAT_GLASS mirror_r + diffuse_r;
 *     otherwise (Disney) diffuse_r + spec_r0.
 * Per pixel, float32 sums in ascending sample order; then albedo.xyz = sum / num_samples, albedo.w = hits / num_samples,
 * normal.xyz = sum / num_samples, depth = hits > 0 ? t_sum / hits : 0.  Batched like agpt_render (whole samples per batch);
 * the film and moments are not touched.  The guides belong to the scene, camera and film they were traced with:
 * agpt_set_film, agpt_set_camera and every agpt_upload_* that passes its argument checks (a later failure too) make them stale (agpt_clear and agpt_render* do not).
 * oracle/agpt_guides_oracle.cpp states the same on the CPU. */
int agpt_render_guides(agpt_ctx* ctx, int num_samples, uint32_t flags);   /* 1 <= num_samples <= 1<<24 */
int agpt_read_guides(agpt_ctx* ctx, float* albedo_rgba, float* normal_depth_rgba);   /* either may be NULL; AGPT_ERR_STATE if none */

/* The spatial part of SVGF (Schied et al. 2017): the edge-avoiding a-trous wavelet filter of Dammertz et al. 2010 driven by
 * per-pixel variance, without temporal reprojection, over the resident film, moments and (fresh) guides.  float32, every
 * operation rounded on its own (+ - * / sqrt, compares, selects), stated element for element in oracle/denoise.py:
 *   per pixel (a = film, q = moments.xyz, n = moments.w, per channel c):
 *     mu_c  = n > 0 ? a_c / n : 0;
 *     var_c = n < 2 ? 0 : v / n with mu = a / n; d = q - a * mu; v = d / (n - 1); v = v < 0 ? 0 : v   (the arithmetic of the
 *             convergence test of agpt_adaptive, shared with it);
 *     al_c  = albedo_c > EPS_A ? albedo_c : EPS_A,  EPS_A = 0.01;   e_c = mu_c / al_c;
 *     lum(x) = (0.212671 * x.r + 0.715160 * x.g) + 0.072169 * x.b;
 *     v_l   = (t_r + t_g) + t_b,  t_c = ((W_c * W_c) * var_c) / (al_c * al_c),  W = the luminance weights above;
 *     missed: none of the pixel's guide samples hit (albedo.w == 0).  Its guide normal is then 0, so its w_n is 0 for every
 *     tap: a pixel that saw only sky is never filtered (w_z's miss cases decide only for guides whose normal is not 0).
 *   iteration i = 0 .. iterations-1, every pixel p from the previous iteration's (e, v_l), step = 2^i:
 *     for dy = -2..2 (outer), dx = -2..2 (inner): q = (film row of p + dy * step, column of p + dx * step); a tap outside the
 *     film is skipped;
 *       w_l = 1 / (1 + (dl * dl) / ((s_l * s_l) * v_p + EPS_L)),  dl = lum(e_p) - lum(e_q),  EPS_L = 1e-4,  s_l = sigma_luminance;
 *       w_n = m squared normal_power_log2 times (m = m * m), m = dot(n_p, n_q) (= (x*x' + y*y') + z*z'), m = m > 0 ? m : 0;
 *       w_z = 1 if both missed, 0 if exactly one missed, else 1 / (1 + |z_p - z_q| / (sigma_depth * z_p));
 *       w   = (((h[dx] * h[dy]) * w_l) * w_n) * w_z,  h = (1/16, 1/4, 3/8, 1/4, 1/16);
 *       W += w;  S_c += w * e_q,c;  V += (w * w) * v_q   (sums from 0, in tap order);
 *     e'_c = S_c / W,  v' = V / (W * W).
 *   end: out_c = e_c * al_c (out.w = 0); packed = ResolvePixel(out, 1) (agpt_resolve's lin2rgb / rgb2uint of the floats).
 *   iterations == 0: out = (mu, 0), no demodulation: the per-pixel means, and the packed pixels equal agpt_resolve_counts.
 * Non-finite values (cfg 8: sums of squares that overflow to inf): a pixel is INVALID when one of its e_c or its v_l is not
 * finite.  An invalid pixel keeps its (e, v_l) through every iteration and is skipped as a tap.  A tap whose w is not finite
 * (NaN: inf / inf, 0 / 0) is skipped.  A pixel whose W is not > 0 (sky pixels: normal 0), or whose e' or v' is not finite,
 * keeps its (e, v_l) in that iteration.  sigma_depth = 0 therefore turns the filter off: every hit pixel's centre tap is
 * 0 / 0 and every other tap that hit has w_z = 0.
 * Refused with AGPT_ERR_INVALID (params NULL, iterations outside [0, 10], a sigma not finite or < 0, normal_power_log2
 * outside [0, 10]) and AGPT_ERR_STATE (moments off, no film, guides missing or stale); a refused call writes nothing and
 * leaves film, moments and guides as they were.  out_rgba: float4[W*H] in film row order like agpt_read_accum; out_rgb8:
 * W*H packed pixels in agpt_resolve_counts' layout; either may be NULL. */
struct agpt_denoise {
	int32_t iterations;        /* a-trous passes, 0 .. 10 */
	float sigma_luminance;     /* luminance edge stop, in standard deviations of the pixel's luminance */
	float sigma_depth;         /* depth edge stop, relative to the pixel's depth */
	int32_t normal_power_log2; /* w_n = max(0, dot(n_p, n_q)) ^ (2 ^ normal_power_log2) */
};
typedef struct agpt_denoise agpt_denoise_params;
int agpt_denoise(agpt_ctx* ctx, const agpt_denoise_params* params, float* out_rgba, uint32_t* out_rgb8);

/* ---- reprojection across camera moves (EXTENSION: the reference clears the film whenever the camera moves) ---------------
 * The temporal half of SVGF for the sample statistics: the film and its moments are carried into the current camera's view, so
 * a frame after a camera move starts from the samples of the frames before it instead of from none.  What is carried is
 * "per-pixel sums + counts" as before, so agpt_denoise, agpt_resolve_counts and the convergence test apply unchanged.
 *
 * A viewer's frame, one per camera:  agpt_set_camera;  agpt_render_guides(ctx, g, 0);  agpt_reproject_film;
 * agpt_render(ctx, first, k, ...) with first = the number of sample indices used by all frames so far;  agpt_denoise or
 * agpt_resolve_counts.  The sample indices must keep advancing from frame to frame: a path's random numbers depend only on its
 * (pixel, sample index), so a frame that reuses sample indices repeats the random numbers of the history it lands on and its
 * samples are not independent of that history.
 *
 * The context keeps a SAVED VIEW: the camera and, per pixel in film row order, G = (mean guide normal, mean hit depth, or -1 for
 * a pixel whose guide samples all missed) -- the G of k_denoise_prepare.  agpt_reproject_film (moments on, a film, fresh guides):
 *   - no saved view: film and moments are left as they are; the view is saved;
 *   - the saved camera is bitwise equal to the current one: film and moments are left as they are (recomputing the identity
 *     map in float32 would put some pixel centres an ulp from a pixel edge and leak a tiny share of a neighbour into every
 *     static frame: with this rule a static camera accumulates exactly as without reprojection); the view is saved again;
 *   - otherwise, per current pixel (x, y) (film row H-1-y), float32, every operation rounded on its own:
 *     1. centre ray: s = (x + 0.5) / W, t = (y + 0.5) / H, D = normalize(((L + s*Hz) + t*Vt) - O) with normalize(v) =
 *        v * (1 / sqrt(dot(v, v))) and dot(a, b) = (a.x*b.x + a.y*b.y) + a.z*b.z (O, L, Hz, Vt: the current camera's origin,
 *        lower-left corner, horizontal, vertical: CameraRay without jitter and lens offset);
 *     2. a hit pixel (guide hit fraction > 0): X = O + depth * D, d = X - O', z = length(d) = sqrt(dot(d, d)) (primes: the
 *        saved camera); a sky pixel: d = D (a point at infinity);
 *     3. f = ((L' + 0.5*Hz') + 0.5*Vt') - O', den = dot(d, f); !(den > 0): no history.  lam = dot(f, f) / den,
 *        u = 0.5 + (lam * dot(d, Hz')) / dot(Hz', Hz'), v = 0.5 + (lam * dot(d, Vt')) / dot(Vt', Vt'), px = u * W - 0.5,
 *        py = v * H - 0.5;
 *     4. x0 = floor(px), y0 = floor(py); unless -1 <= x0 <= W - 1 and -1 <= y0 <= H - 1 (false for a px or py that is not
 *        finite) no history.  fx = px - x0, fy = py - y0, wx = (1 - fx, fx), wy = (1 - fy, fy); taps k = 0..3 in this order:
 *        (x0 + (k & 1), y0 + (k >> 1)) with w = wx[k & 1] * wy[k >> 1], read at film row H-1-(y0 + (k >> 1)).  A tap is
 *        ACCEPTED when it is inside the film, w > 0, its film and moments values are finite (all four channels each), its saved
 *        G is a hit (G'.w >= 0) exactly when the current pixel's is, and for hits |G'.w - z| <= sigma_depth * z and
 *        dot(n, n') >= min_normal_dot (n, n': current and saved guide normals);
 *     5. over the accepted taps in tap order, from 0: Wt += w; S += w * a (film, four channels); Q += w * q (moments, four
 *        channels).  Wt > 0: a' = S / Wt, q' = Q / Wt per channel, and if q'.w > max_history: k = max_history / q'.w,
 *        a' = a' * k (four channels), q'.xyz = q'.xyz * k, q'.w = max_history.  Otherwise (a disocclusion) a' = q' = 0;
 *   and the current camera and the current guides' G become the saved view.  oracle/reproject.py states the same.
 * The saved view is dropped by agpt_set_film to a new size, by every agpt_upload_* past its argument checks (the scene changed)
 * and by agpt_set_moments(0); agpt_set_camera keeps it.
 * Consequences: counts become fractional, so agpt_resolve(samples) no longer describes the film (use agpt_resolve_counts or
 * agpt_denoise), and agpt_write_moments still refuses fractional counts; agpt_render_adaptive still starts from a cleared film;
 * one GPU only (like adaptive sampling); view-dependent radiance (mirror, glass, glossy lobes) ghosts, by up to max_history
 * samples' worth.  Refused with AGPT_ERR_INVALID (params NULL, max_history outside [1, 2^24], sigma_depth not finite or <= 0,
 * min_normal_dot outside [-1, 1]) and AGPT_ERR_STATE (moments off, no film, guides missing or stale); a refused call leaves
 * film, moments and the saved view as they were.  The film keeps its address (agpt_set_accum_dev films too). */
typedef struct agpt_reproject {
	float max_history;     /* most samples a pixel may carry into the new view, 1 .. 2^24 */
	float sigma_depth;     /* relative depth tolerance of a history tap, finite, > 0 */
	float min_normal_dot;  /* least dot(normal, history normal) of a history tap, in [-1, 1] */
} agpt_reproject;
int agpt_reproject_film(agpt_ctx* ctx, const agpt_reproject* params);

/* ---- multi-GPU: sample-index sharding (SURVEY 8e; north star "NCCL reduces the accumulators over NVLink") ----
 * One context per GPU of ONE process, each holding the whole scene and a film of the same size.  GPU g of G
 * renders the samples s = first + g (mod G) into its own accumulator (agpt_render with sample_stride = G, or
 * agpt_render_multi, which runs the G renders on G host threads); the frame is the sum of the accumulators.
 *
 * agpt_reduce_accum sums them with this library's own kernel over NVLink peer memory -- each GPU owns a slice
 * of the film, loads it from all accumulators, adds in RANK ORDER and stores the sum back to all (root = -1) or
 * the root's GPU does it for the whole film (root >= 0: only ctxs[root] receives the sum).  Rank-order summation
 * makes the result reproducible and equal to ((a0 + a1) + a2) + ... .  Where some pair of GPUs has no peer access,
 * or with AGPT_REDUCE=nccl in the environment, it runs ncclAllReduce instead (libnccl is dlopen'ed on first use).
 * agpt_allreduce_accum(ctxs, n) == agpt_reduce_accum(ctxs, n, -1).
 *
 * agpt_reduce_resolve is the fused end of a render: sum + Accumulator::CopyToSurface (myapp.h:34-41) in ONE
 * kernel per GPU (its slice of the film), packed pixels straight to the host over all GPUs' PCIe links;
 * keep_sum != 0 also leaves the summed film in ctxs[0]'s accumulator. */
int agpt_render_multi(agpt_ctx** ctxs, int n, int first_sample, int num_samples, int max_depth, int rr_depth_arg, uint32_t flags);
int agpt_reduce_accum(agpt_ctx** ctxs, int n, int root);
int agpt_allreduce_accum(agpt_ctx** ctxs, int n);
int agpt_reduce_resolve(agpt_ctx** ctxs, int n, int samples, int keep_sum, uint32_t* host_rgb8);

/* The same exchange between PROCESSES (one rank per GPU: torchrun, MPI).  Each rank exports its context-owned
 * accumulator as a 64-byte CUDA IPC handle; after the ranks have exchanged the handles (any transport), each
 * opens the others' accumulators and the same peer-memory kernels run on them.  The caller provides the
 * barriers: before either call every rank must have finished rendering; after agpt_allreduce_accum_peers no
 * rank may touch its accumulator until every rank has returned.  agpt_reduce_resolve_peers runs on the root
 * rank only and writes nothing to the peers. */
int agpt_accum_ipc_handle(agpt_ctx* ctx, void* handle64);
int agpt_open_peer_accums(agpt_ctx* ctx, int rank, int world, const void* handles64 /* world x 64 bytes, rank order */);
int agpt_close_peer_accums(agpt_ctx* ctx);
int agpt_allreduce_accum_peers(agpt_ctx* ctx);
int agpt_reduce_resolve_peers(agpt_ctx* ctx, int samples, int keep_sum, uint32_t* host_rgb8);

/* Page-locked host memory for accumulator buffers (what MALLOC64 is upstream, myapp.h:11):
 * agpt_read_accum / agpt_write_accum on such a buffer run at PCIe speed. */
int agpt_host_alloc(size_t bytes, void** out);
int agpt_host_free(void* p);

/* ---- observability ------------------------------------------------------------------- */

/* Traversal work per WAVE of the renders made with AGPT_FLAG_COUNTERS since agpt_reset_stats.  Wave w of a batch
 * traces the path rays of bounce w (and the shadow / MIS rays of the vertex before it), so this is the per-bounce
 * N_int / N_tri / divergence report of SURVEY 8d (RecursiveHit, bvhtrimesh.h:332-384).  kind 0 = closest-hit kernel
 * (path + MIS rays), 1 = any-hit kernel (shadow rays).  Fills up to max_waves rows; *n_waves = rows in use. */
typedef struct agpt_wave_stats {
	uint64_t rays, node_visits, box_tests, tri_tests, analytic_tests, warp_steps, lane_steps, reserved;
} agpt_wave_stats;
int agpt_get_wave_stats(agpt_ctx* ctx, int kind, agpt_wave_stats* out, int max_waves, int* n_waves);
/* Read bandwidth (GB/s) a plain streaming kernel of this library reaches on this GPU over `bytes` of device memory
 * read `iters` times: bytes well inside the L2 size measures L2, bytes far beyond it HBM (roofline denominators). */
int agpt_probe_bandwidth(agpt_ctx* ctx, size_t bytes, int iters, float* gbs_out);
int agpt_get_stats(agpt_ctx* ctx, agpt_stats* out);
int agpt_reset_stats(agpt_ctx* ctx);
/* Builds with -DAGPT_DEBUG (libagpt_debug.so) check stack depth, node / triangle / primitive indices and queue
 * slots inside the kernels.  out4 = { failed checks, code of the first failure, its value, checks executed }
 * since the library was loaded; a release build reports 0 checks executed. */
int agpt_debug_status(agpt_ctx* ctx, uint64_t* out4);

/* ---- per-function probes (differential tests against single reference functions) ----- */

/* Bounds::Intersect (bvhtrimesh.h:18-36): boxes6 = bmin,bmax; rays7 = O,D (as given),tmax. */
int agpt_probe_bounds(agpt_ctx* ctx, int n, const float* boxes6, const float* rays7, int* out_hit, float* out_t);
/* BSDF::f / Pdf / Sample_f on a frame built from (dpdu, dpdv) (reflection.h:114-188):
 * in14 = dpdu3 dpdv3 wo3 wi3 u2; out12 = f3 pdf1 | sampled wi3 f3 pdf1 specular1. */
int agpt_probe_bsdf(agpt_ctx* ctx, int n, const agpt_material* mat, const float* in14, int skip_specular, float* out12);
/* Sphere::Sample(ref,u) / Sphere::Pdf (intersectable.h:239-317): in9 = center3 r refp3 u2;
 * out8 = p3 n3 pdf pdf_only. */
int agpt_probe_sphere_sample(agpt_ctx* ctx, int n, const float* in9, float* out8);
/* EXTENSION: Sample_Li / Pdf_Li of resident light `light`, which must be an area light with AGPT_LIGHT_SAMPLE_SHAPE on a
 * plane or mesh (agpt_light.flags): in8 = ref point3 u2 query direction3; out8 = sampled point3, its solid-angle pdf,
 * Pdf_Li(ref, query direction), light normal3 at the sampled point. */
int agpt_probe_light_sample(agpt_ctx* ctx, int light, int n, const float* in8, float* out8);
/* EXTENSION (agpt_upload_material_textures): the closest hit of each ray of rays7 (O, D normalised like agpt_trace_rays, tmax)
 * on the resident scene, shaded as the roughness-metallic / normal-map shade kernel shades it.  out32 per ray: prim (-1: miss,
 * the rest 0), u, v, ng3, ns3, ss3, ts3 (the BSDF frame after the normal map), T3, B3 (dp/du, dp/dv of the uv), roughness,
 * metallic, lobes, diffuse_r3, spec_r03 (the hit's material record; the first record for a null material).  AGPT_ERR_STATE
 * unless some material has a roughness-metallic or normal map. */
int agpt_probe_material_maps(agpt_ctx* ctx, int n, const float* rays7, float* out32);
/* First k floats of the RNG stream of (pixel_index, sample) (SURVEY 8a row 3). */
int agpt_probe_stream(agpt_ctx* ctx, uint32_t pixel_index, uint32_t sample, int k, float* out);

#ifdef __cplusplus
}
#endif
#endif /* AGPT_H */
