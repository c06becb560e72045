// agpt_api.cu -- libagpt.so: the extern "C" boundary of include/agpt.h over the sm_100a
// wavefront kernels.  Host code here only moves tables into HBM, sizes launches and drives
// the wave loop; every ray is traced and shaded on the device.  There is no CPU path: if no
// CUDA device can be opened agpt_create() fails and the caller gets the CUDA error text.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <optional>
#include <string>
#include <thread>
#include <type_traits>
#include <utility>
#include <vector>

#include "agpt_kernels.cuh"
#include "agpt_multigpu.cuh"
#include "../host/sampling.h"

static inline int Blocks(size_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---- error plumbing ----------------------------------------------------------------------
static thread_local std::string g_error;
static int Fail(int code, const std::string& msg) { g_error = msg; return code; }
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) \
	return Fail(AGPT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)
#define NEED(cond, code, msg) do { if (!(cond)) return Fail(code, msg); } while (0)

// One device allocation and its only owner: freed when the buffer goes out of scope or is assigned another by a move.
template <typename T>
struct DevBuf {
	T* p = nullptr;
	size_t n = 0;
	DevBuf() = default;
	DevBuf(DevBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), n(std::exchange(o.n, 0)) {}
	DevBuf& operator=(DevBuf&& o) noexcept {
		if (this != &o) { Free(); p = std::exchange(o.p, nullptr); n = std::exchange(o.n, 0); }
		return *this;
	}
	DevBuf(const DevBuf&) = delete; DevBuf& operator=(const DevBuf&) = delete;     // one owner per allocation
	~DevBuf() { Free(); }
	cudaError_t Alloc(size_t count) {
		Free();
		if (count == 0) return cudaSuccess;
		cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
		if (e == cudaSuccess) n = count;
		return e;
	}
	cudaError_t Upload(const T* host, size_t count, cudaStream_t s) {
		cudaError_t e = Alloc(count);
		if (e != cudaSuccess || count == 0) return e;
		return cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, s);
	}
	void Free() { if (p) cudaFree(p); p = nullptr; n = 0; }
	size_t Bytes() const { return n * sizeof(T); }
};

struct MeshStore {
	DevBuf<float4> nodes, tris, normals;
	DevBuf<float2> uvs;
	DevBuf<int> ids;
};

// A stream, event or pinned block created by the context and released with it.
template <typename H, auto Destroy>
struct Owned {
	H h{};
	Owned() = default;
	Owned(const Owned&) = delete;
	Owned& operator=(const Owned&) = delete;
	~Owned() { if (h) Destroy(h); }
	operator H() const { return h; }
};
using OwnedStream = Owned<cudaStream_t, cudaStreamDestroy>;
using OwnedEvent = Owned<cudaEvent_t, cudaEventDestroy>;

#ifndef AGPT_BATCH_LOG2
#define AGPT_BATCH_LOG2 27
#endif
// Paths in flight per batch, at most.  2^27 = 134 M slots ~ 39 GB of wavefront state + queues (sized for 180 GB of
// HBM3e; the state is allocated for the batches a caller actually asks for: 16 spp at 1080p take 33 M slots).
// Bigger batches mean fuller waves and more rays per bucket, i.e. more coherent warps: cfg 3 runs a 16-spp
// share in 106 / 98 / 94 ms with batches of 2^23 / 2^24 / 2^25 slots (round 1's kernels) and in 57.9 / 55.8 /
// 54.4 ms with 2^25 / 2^26 / 2^27 (16 / 32 / 64 spp per batch at 1080p, round 2's).
static const size_t kMaxPathsPerBatch = (size_t)1 << AGPT_BATCH_LOG2;

struct agpt_ctx {
	// (declared before every buffer: members are destroyed in reverse order, so these outlive the buffers)
	OwnedStream ownStream;
	OwnedStream sideStream;              // any-hit trace of a wave runs here, beside the closest-hit trace
	OwnedStream copyStream;              // agpt_write_accum_begin: the film upload runs here, beside the render that follows
	OwnedEvent evUpload;
	OwnedEvent evFork, evJoin;
	OwnedEvent evA, evB, evC, evD;
	OwnedEvent evRender0, evRender1;     // bracket of agpt_render (ms_render)
	Owned<int*, cudaFreeHost> hostCounts;   // pinned ring of kRing x 3 ints
	OwnedEvent ringEvents[8];
	// Work still queued may use the buffers: it finishes before the members release them.  (Failures change nothing about what
	// follows.)
	~agpt_ctx() {
		cudaSetDevice(device);
		if (uploadPending) cudaStreamSynchronize(copyStream);
		if (stream) cudaStreamSynchronize(stream);
		for (int r = 0; r < peerWorld; r++) if (r != peerRank && peerAccum[r]) cudaIpcCloseMemHandle(peerAccum[r]);
	}

	int device = 0;
	cudaStream_t stream = nullptr;       // ownStream or the caller's (agpt_set_stream)
	bool uploadPending = false;          // a film upload is in flight: k_accumulate waits for it, every other film access joins it first
	int smCount = 0;

	// scene tables
	std::vector<MeshStore> meshStore;
	DevBuf<DMesh> meshes;
	DevBuf<agpt_sphere> spheres;
	DevBuf<agpt_plane> planes;
	DevBuf<agpt_prim> prims;
	DevBuf<agpt_instance> instances;     // extension: placed meshes
	std::vector<agpt_instance> hostInstances;
	int nInstances = 0;
	bool hasGlass = false;        // some material is a rough dielectric (extension): shade runs the GLASS instantiation
	bool hasShapeLights = false;  // some area light samples its plane or mesh (extension): shade runs a SHAPES instantiation
	bool shapesDirty = true;      // the sampling tables below follow the mesh, plane, primitive and light tables
	DevBuf<DShapeLight> shapeLights;
	DevBuf<float> shapeCdf;
	std::vector<agpt_plane> hostPlanes;
	DevBuf<int> sphereRun;
	DevBuf<float4> sphereRunBox;
	DevBuf<float4> keyBoxes;         // root boxes of the meshes that do not cover the scene (ray-bucket key)
	std::vector<agpt_bvh_node> hostRoots;   // node 0 of every mesh (count < 0: the mesh has no BVH)
	std::vector<agpt_sphere> hostSpheres;
	bool runsDirty = true;
	int maxSphereRun = 1 << 20;   // AGPT_MAX_SPHERE_RUN
	DevBuf<agpt_material> mats;
	std::vector<int32_t> hostMatTypes;
	// image textures on the base colour of Disney materials (extension, agpt_upload_textures)
	DevBuf<float4> texels;
	DevBuf<DTexture> textures;
	DevBuf<int> matTex;
	DevBuf<DMatMaps> matMaps;     // roughness-metallic and normal maps (extension, agpt_upload_material_textures)
	std::vector<agpt_material_textures> hostBindings;
	bool hasTextures = false;     // some material has a texture: shade and guides run the textured instantiations
	bool hasMaps = false;         // some material has a roughness-metallic or normal map: the TEX == 2 instantiations
	DevBuf<agpt_alpha_mask> masks;            // alpha masks (extension, agpt_upload_alpha_masks), per material
	std::vector<agpt_alpha_mask> hostMasks;
	bool hasMasks = false;        // some material has a mask: trace runs the MASK instantiations
	DevBuf<agpt_emission> emission;           // emissive materials (extension, agpt_upload_emission), per material
	std::vector<agpt_emission> hostEmission;
	bool hasEmission = false;     // some row emits: k_shade_a_emit runs and tail rays are traced
	DevBuf<agpt_light> lights;
	DevBuf<float> envRgb, envFunc, envCdf;
	float envFuncInt = 0;
	int envW = 0, envH = 0;
	std::vector<agpt_prim> hostPrims;
	std::vector<agpt_light> hostLights;
	int nMeshes = 0, nSpheres = 0, nPlanes = 0, nMats = 0;
	int maxBvhDepth = 0;          // deepest uploaded tree (levels below the root), validated against the traversal stack
	agpt_camera cam;
	bool haveCam = false;
	float boundsLo[3] = { -1, -1, -1 }, boundsHi[3] = { 1, 1, 1 };   // bounded geometry (mesh roots), for ray bucketing only
	float gridLo[3] = { -1, -1, -1 }, gridHi[3] = { 1, 1, 1 };       // ... refined from where the camera's rays actually land (CalibrateBucketGrid)
	bool gridCalibrated = false;
	bool calibrateGrid = true;    // AGPT_BUCKET_CALIBRATE=0: keep the grid on the mesh bounds
	int width = 0, height = 0;

	// film
	DevBuf<float4> accumOwn;
	DevBuf<uint32_t> resolved;    // agpt_resolve's packed output, kept between calls
	float4* accum = nullptr;      // accumOwn.p or caller-owned
	// adaptive sampling (agpt_set_moments): per-pixel sum of squares and sample count, always context-owned
	bool momentsOn = false;
	DevBuf<float4> moments;
	DevBuf<int> adaptiveList;     // agpt_adaptive_select's compacted pixel list (W*H) and its length
	DevBuf<int> adaptiveCount;
	// denoising (agpt_render_guides, agpt_denoise): guides traced for the scene, camera and film of generation guidesGen
	uint64_t stateGen = 1;        // bumped by agpt_set_film, agpt_set_camera and every agpt_upload_* past its argument checks
	uint64_t guidesGen = 0;       // 0: no guides
	DevBuf<float4> guideAlbedo, guideNormal;
	DevBuf<float4> denoiseE[2], denoiseG, denoiseOut;   // ping-pong (e, v_l), the filter's guide, the result
	// reprojection (agpt_reproject_film): the saved view is viewCam and the guide G per pixel in viewG[viewCur]
	uint64_t historyGen = 1;      // bumped by what makes a saved view wrong: agpt_set_film to a new size, every agpt_upload_* past
	                              // its argument checks, agpt_set_moments(0).  Not by agpt_set_camera: carrying across it is the point
	uint64_t viewGen = 0;         // the historyGen the saved view was taken in; 0: none
	agpt_camera viewCam;
	DevBuf<float4> viewG[2];      // ping-pong: a call reads its saved G from one and saves the current G into the other
	int viewCur = 0;
	DevBuf<float4> reprojFilm, reprojMoments;   // the gathered film and moments (the gathers read the old ones)

	// wavefront state
	size_t capacity = 0;          // path slots allocated
	DevBuf<float4> f4[13];
	DevBuf<int> i32[3];
	DevBuf<uint32_t> u32[2];
	DevBuf<int> queues[6];        // closest A/B (2*cap), shadow A/B, active A/B
	DevBuf<int> sortedClosest;    // closest queue in bucket order (2*cap)
	DevBuf<unsigned short> keys[2], shadowKeys[2];
	DevBuf<int> sortedShadow;
	DevBuf<int> hist;             // AGPT_BUCKETS x { histogram, offsets, running }
	DevBuf<int> counts;           // 2 x 3
	DevBuf<int> survivors, survivorCount;   // paths k_shade_b works on this wave
	DevBuf<unsigned long long> traceCounters;   // [2][8] totals (closest-hit, any-hit), then [2][AGPT_MAX_WAVE_ROWS][8] per wave (FlushCounters)
	DevBuf<RayCounters> rayCounters;

	// multi-process sharding: the other ranks' accumulators, mapped through CUDA IPC (agpt_open_peer_accums)
	float4* peerAccum[AGPT_MAX_PEERS] = {};
	int peerRank = -1, peerWorld = 0;

	agpt_stats stats;
	bool asyncWaves = false;      // AGPT_ASYNC_WAVES=1: run one wave ahead of the landed queue counts instead of syncing
	                              // every wave.  Measured slower (N=1: 133 vs 130.5 ms/step, N=8: 142.8 vs 139.3): the loose
	                              // launch bounds and the extra empty wave cost more than the ~30 us sync gaps they remove.
	size_t maxPathsPerBatch = kMaxPathsPerBatch;   // AGPT_BATCH_LOG2 (environment) overrides the compiled-in size
	bool overlapAny = true;       // AGPT_OVERLAP_ANY=0: any-hit trace on the main stream after the closest-hit trace
	bool bucketRays = true;       // bucket pass on the ray queues (AGPT_BUCKET_RAYS=0 turns it off)
};

// Runs of sphere primitives whose payloads are consecutive: the trace kernels walk such a run
// straight through the sphere table, and skip it when no ray of the warp can reach its box.
static int BuildSphereRuns(agpt_ctx* c) {
	const int n = (int)c->hostPrims.size();
	std::vector<int> run((size_t)n, 0);
	std::vector<float4> box(3 * (size_t)n, make_float4(0.f, 0.f, 0.f, 0.f));
	const std::vector<agpt_prim>& rows = c->hostPrims;
	for (int p = n - 1; p >= 0; p--) {
		if (rows[p].type != AGPT_PRIM_SPHERE) continue;
		bool chained = p + 1 < n && rows[p + 1].type == AGPT_PRIM_SPHERE && rows[p + 1].payload == rows[p].payload + 1;
		run[p] = chained && run[p + 1] < c->maxSphereRun ? run[p + 1] + 1 : 1;     // capped: shorter runs have tighter boxes
	}
	for (int p = 0; p < n; p++) {
		if (run[p] == 0) continue;
		float lo[3] = { 1e30f, 1e30f, 1e30f }, hi[3] = { -1e30f, -1e30f, -1e30f }, rmin = 1e30f;
		bool ok = true;
		for (int j = 0; j < run[p]; j++) {
			int k = rows[p + j].payload;
			if (k < 0 || k >= (int)c->hostSpheres.size()) { ok = false; break; }
			const agpt_sphere& sp = c->hostSpheres[k];
			if (!(sp.r > 0.f)) { ok = false; break; }
			for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], sp.center[a] - sp.r); hi[a] = fmaxf(hi[a], sp.center[a] + sp.r); }
			rmin = fminf(rmin, sp.r);
		}
		float4* b = &box[3 * (size_t)p];
		if (!ok) { b[2] = make_float4(0.f, 0.f, 0.f, -1.f); continue; }      // never cull
		const float grow = 0.05f * rmin;
		float ctr[3], diag2 = 0.f;
		for (int a = 0; a < 3; a++) { lo[a] -= grow; hi[a] += grow; ctr[a] = 0.5f * (lo[a] + hi[a]); float h = 0.5f * (hi[a] - lo[a]); diag2 += h * h; }
		// Rounding of Sphere::Intersect's discriminant is at most ~22 * 2^-24 |oc|^2 = 1.3e-6 |oc|^2 (every
		// product, sum and input rounding counted against us); a ray that misses the grown box has
		// d^2 - r^2 > 2 r grow = 0.1 rmin^2.  With |oc|^2 <= 2 (|O - ctr|^2 + diag2) kept below 2e4 rmin^2 the
		// rounding stays under 0.026 rmin^2: a factor 4 of slack on a worst-case bound.
		b[0] = make_float4(lo[0], lo[1], lo[2], hi[0]);
		b[1] = make_float4(hi[1], hi[2], 0.f, 0.f);
		b[2] = make_float4(ctr[0], ctr[1], ctr[2], 1.0e4f * rmin * rmin - diag2);
	}
	// ray-bucket key: the root boxes of BVH mesh primitives that are small against the union of all of them
	std::vector<float4> kb;
	{
		float lo[3] = { 1e30f, 1e30f, 1e30f }, hi[3] = { -1e30f, -1e30f, -1e30f };
		std::vector<int> meshPrims;
		for (int p = 0; p < n; p++)
			if (rows[p].type == AGPT_PRIM_BVH_MESH && rows[p].payload >= 0 && rows[p].payload < (int)c->hostRoots.size() && c->hostRoots[rows[p].payload].count >= 0) {
				meshPrims.push_back(rows[p].payload);
				for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], c->hostRoots[rows[p].payload].bmin[a]); hi[a] = fmaxf(hi[a], c->hostRoots[rows[p].payload].bmax[a]); }
			}
		double all = 1;
		for (int a = 0; a < 3; a++) all *= fmax((double)hi[a] - lo[a], 1e-30);
		for (int m : meshPrims) {
			const agpt_bvh_node& r = c->hostRoots[m];
			double v = 1;
			for (int a = 0; a < 3; a++) v *= fmax((double)r.bmax[a] - r.bmin[a], 1e-30);
			if (v <= 0.25 * all && kb.size() < 2 * 16) { kb.push_back(make_float4(r.bmin[0], r.bmin[1], r.bmin[2], r.bmax[0])); kb.push_back(make_float4(r.bmax[1], r.bmax[2], 0.f, 0.f)); }
		}
	}
	DevBuf<float4> keyBoxes, runBox;
	DevBuf<int> runs;
	CU(keyBoxes.Upload(kb.data(), kb.size(), c->stream));
	CU(runs.Upload(run.data(), (size_t)n, c->stream));
	CU(runBox.Upload(box.data(), box.size(), c->stream));
	CU(cudaStreamSynchronize(c->stream));
	c->keyBoxes = std::move(keyBoxes); c->sphereRun = std::move(runs); c->sphereRunBox = std::move(runBox);
	c->runsDirty = false;
	return AGPT_OK;
}

// EXTENSION (agpt.h AGPT_LIGHT_SAMPLE_SHAPE): per light, the total area of a sampled plane or mesh and, for a mesh, the
// Distribution1D over its triangle areas in slot order.  The areas come from the device (k_triangle_areas, the degenerate
// flags of the upload), the sums are host/sampling.h's sequential ones.
static int BuildShapeLights(agpt_ctx* c) {
	const int nl = (int)c->hostLights.size();
	std::vector<DShapeLight> table((size_t)nl);
	std::vector<float> cdf;
	bool any = false;
	for (int i = 0; i < nl; i++) {
		DShapeLight& e = table[i];
		e.cdfOff = 0; e.n = 0; e.area = 0.f; e.pad = 0.f;
		const agpt_light& l = c->hostLights[i];
		if (l.type != AGPT_LIGHT_AREA || !(l.flags & AGPT_LIGHT_SAMPLE_SHAPE)) continue;
		const agpt_prim& pr = c->hostPrims[l.prim];
		if (pr.type == AGPT_PRIM_PLANE) {
			e.area = 4.f * c->hostPlanes[pr.payload].half_x * c->hostPlanes[pr.payload].half_z;
			any = true;
			continue;
		}
		if (pr.type != AGPT_PRIM_MESH && pr.type != AGPT_PRIM_BVH_MESH) continue;      // a sphere is sampled as a sphere anyway
		any = true;
		const int n = (int)(c->meshStore[pr.payload].tris.n / 3);
		if (n == 0) continue;
		DevBuf<float> dev;
		std::vector<float> area((size_t)n);
		CU(dev.Alloc((size_t)n));
		k_triangle_areas<<<Blocks(n, 256), 256, 0, c->stream>>>(c->meshStore[pr.payload].tris.p, n, dev.p);
		CU(cudaGetLastError());
		c->stats.kernel_launches++;
		CU(cudaMemcpyAsync(area.data(), dev.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
		CU(cudaStreamSynchronize(c->stream));
		Distribution1D d(area.data(), n);
		if (d.funcInt == 0) continue;                       // nothing to sample (Distribution1D's uniform fallback is not used)
		float total = 0;
		for (float a : area) total += a;
		e.cdfOff = (int)cdf.size(); e.n = n; e.area = total;
		cdf.insert(cdf.end(), d.cdf.begin(), d.cdf.end());
	}
	DevBuf<DShapeLight> lights;
	DevBuf<float> lightCdf;
	if (any) {
		CU(lights.Upload(table.data(), table.size(), c->stream));
		CU(lightCdf.Upload(cdf.data(), cdf.size(), c->stream));
		CU(cudaStreamSynchronize(c->stream));
	}
	c->shapeLights = std::move(lights); c->shapeCdf = std::move(lightCdf);
	c->hasShapeLights = any;
	c->shapesDirty = false;
	return AGPT_OK;
}

static void SetBucketGrid(DScene& s, const float* lo, const float* hi) {
	for (int a = 0; a < 3; a++) { s.cellLo[a] = lo[a]; float e = hi[a] - lo[a]; s.cellScale[a] = e > 0 ? (float)(1 << AGPT_CELL_BITS) / e : 0.f; }
}

static DScene MakeScene(const agpt_ctx* c) {
	DScene s;
	s.keyBoxes = c->keyBoxes.p; s.n_keyBoxes = (int)(c->keyBoxes.n / 2);
	s.prims = c->prims.p; s.sphereRun = c->sphereRun.p; s.sphereRunBox = c->sphereRunBox.p; s.spheres = c->spheres.p; s.planes = c->planes.p; s.meshes = c->meshes.p; s.instances = c->instances.p;
	s.mats = c->mats.p; s.lights = c->lights.p;
	s.n_prims = (int)c->prims.n; s.n_lights = (int)c->lights.n;
	s.envRgb = c->envRgb.p; s.envFunc = c->envFunc.p; s.envCdf = c->envCdf.p; s.envFuncInt = c->envFuncInt; s.envW = c->envW; s.envH = c->envH;
	s.width = c->width; s.height = c->height;
	SetBucketGrid(s, c->gridCalibrated ? c->gridLo : c->boundsLo, c->gridCalibrated ? c->gridHi : c->boundsHi);
	s.cam = c->cam;
	return s;
}

// ---- launch plan: which instantiation of each kernel family runs for the resident scene ------------------------------------
// Built once per call, after CheckReady has built the lazy tables.  It is the only code that turns the scene's feature flags into
// kernel choices: the launch dispatchers take it instead of flags of their own.
struct LaunchPlan {
	bool inst;                      // some primitive row is an instance: the INST trace instantiations
	bool env;                       // an environment map (InfiniteAreaLight)
	bool glass;                     // some material is a rough dielectric
	bool shapes;                    // some area light samples its plane or mesh
	int tex;                        // 1: some material is textured; 2: some material has a roughness-metallic or normal map
	DShapeTables st;
	DTexTables tt;
	std::optional<DMaskTables> mk;  // some alpha mask is bound: the *_masked trace kernels
	std::optional<DEmitTables> em;  // some emission row emits: k_shade_a_emit, and the path ray at max_depth is traced
};

static LaunchPlan PlanLaunches(const agpt_ctx* c) {
	LaunchPlan p;
	p.inst = c->nInstances > 0; p.env = c->envW > 0; p.glass = c->hasGlass; p.shapes = c->hasShapeLights;
	p.tex = c->hasMaps ? 2 : c->hasTextures ? 1 : 0;
	p.st.lights = c->shapeLights.p; p.st.cdf = c->shapeCdf.p;
	p.tt.texels = c->texels.p; p.tt.textures = c->textures.p; p.tt.matTex = c->matTex.p;
	p.tt.nTextures = (int)c->textures.n; p.tt.nTexels = (long long)c->texels.n;
	p.tt.matMaps = c->matMaps.p; p.tt.nMatMaps = (int)c->matMaps.n;
	if (c->hasMasks) p.mk = DMaskTables{ p.tt, c->masks.p, (int)c->masks.n };
	if (c->hasEmission) p.em = DEmitTables{ p.tt, c->emission.p, (int)c->emission.n };
	return p;
}

// What every call that generates paths or rays starts from: the scene, the path slots, the queues k_generate fills for the first
// wave (queue set A, counts A; no bucket keys yet) and the launch plan
struct Frame {
	DScene sc;
	PathState ps;
	WaveQueues q0;
	LaunchPlan plan;
};

static Frame MakeFrame(agpt_ctx* c) {
	Frame f{ MakeScene(c), PathState(), WaveQueues(), PlanLaunches(c) };
	PathState& p = f.ps;
	p.rayO = c->f4[0].p; p.rayD = c->f4[1].p; p.hitA = c->f4[2].p; p.beta = c->f4[3].p; p.L = c->f4[4].p;
	p.neeLight = c->f4[5].p; p.neeMis = c->f4[6].p; p.neeBeta = c->f4[7].p;
	p.shO = c->f4[8].p; p.shD = c->f4[9].p; p.misO = c->f4[10].p; p.misD = c->f4[11].p; p.Lout = c->f4[12].p;
	p.hitSlot = c->i32[0].p; p.shadowOccluded = c->i32[1].p; p.misPrim = c->i32[2].p;
	p.rng = c->u32[0].p; p.flags = c->u32[1].p;
	p.slots = (int)c->capacity;
	WaveQueues& q0 = f.q0;
	q0.closest = c->queues[0].p; q0.shadow = c->queues[2].p; q0.active = c->queues[4].p; q0.counts = c->counts.p; q0.keys = nullptr; q0.shadowKeys = nullptr;
	return f;
}

static int EnsureCapacity(agpt_ctx* c, size_t paths) {
	if (paths <= c->capacity) return AGPT_OK;
	c->capacity = 0;                 // published again only when every buffer below is there (a failed allocation must not leave a stale size)
	for (auto& b : c->f4) CU(b.Alloc(paths));
	for (auto& b : c->i32) CU(b.Alloc(paths));
	for (auto& b : c->u32) CU(b.Alloc(paths));
	const size_t slack = 1024;       // kernels read queue[i] before they know the queue length (i < grid * block)
	CU(c->queues[0].Alloc(2 * paths + slack)); CU(c->queues[1].Alloc(2 * paths + slack));
	CU(c->sortedClosest.Alloc(2 * paths + slack)); CU(c->keys[0].Alloc(2 * paths + slack)); CU(c->keys[1].Alloc(2 * paths + slack));
	CU(c->shadowKeys[0].Alloc(paths + slack)); CU(c->shadowKeys[1].Alloc(paths + slack)); CU(c->sortedShadow.Alloc(paths + slack));
	for (int k = 2; k < 6; k++) CU(c->queues[k].Alloc(paths + slack));
	CU(c->survivors.Alloc(paths + slack));
	c->capacity = paths;
	return AGPT_OK;
}

// agpt_upload_emission (extension): a row emits iff some factor component is > 0
static bool Emits(const agpt_emission& e) { return e.factor[0] > 0.f || e.factor[1] > 0.f || e.factor[2] > 0.f; }

// agpt_light.flags (extension): only AGPT_LIGHT_SAMPLE_SHAPE, and only on area lights
static int CheckLightFlags(const agpt_light& l) {
	NEED((l.flags & ~(uint32_t)AGPT_LIGHT_SAMPLE_SHAPE) == 0, AGPT_ERR_INVALID, "unknown agpt_light.flags bits");
	NEED(l.flags == 0 || l.type == AGPT_LIGHT_AREA, AGPT_ERR_INVALID, "AGPT_LIGHT_SAMPLE_SHAPE on a light that is not an area light");
	return AGPT_OK;
}

static int CheckReady(agpt_ctx* c, bool needFilm) {
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	NEED(c->prims.n > 0, AGPT_ERR_STATE, "no primitives uploaded (agpt_upload_primitives)");
	if (needFilm) {
		NEED(c->width > 0 && c->height > 0, AGPT_ERR_STATE, "film not set (agpt_set_film)");
		NEED(c->haveCam, AGPT_ERR_STATE, "camera not set (agpt_set_camera)");
	}
	// table consistency: every row must point inside its table
	for (size_t i = 0; i < c->hostPrims.size(); i++) {
		const agpt_prim& p = c->hostPrims[i];
		int limit = p.type == AGPT_PRIM_SPHERE ? c->nSpheres : p.type == AGPT_PRIM_PLANE ? c->nPlanes : p.type == AGPT_PRIM_INSTANCE ? c->nInstances : c->nMeshes;
		NEED(p.type >= 0 && p.type <= 4 && p.payload >= 0 && p.payload < limit, AGPT_ERR_INVALID, "primitive row points outside its shape table");
		NEED(p.material < c->nMats, AGPT_ERR_INVALID, "primitive row points outside the material table");
		NEED(p.area_light < (int)c->hostLights.size(), AGPT_ERR_INVALID, "primitive row points outside the light table");
	}
	for (auto& in : c->hostInstances)
		NEED(in.mesh >= 0 && in.mesh < c->nMeshes, AGPT_ERR_INVALID, "instance row points outside the mesh table");
	for (auto& l : c->hostLights)
		NEED(l.type != AGPT_LIGHT_INFINITE_AREA || c->envW > 0, AGPT_ERR_STATE, "InfiniteAreaLight without an environment map (agpt_upload_envmap)");
	for (auto& l : c->hostLights)
		NEED(l.type != AGPT_LIGHT_AREA || (l.prim >= 0 && l.prim < (int)c->hostPrims.size()), AGPT_ERR_INVALID, "area light without a primitive");
	for (auto& l : c->hostLights) {
		int rcode = CheckLightFlags(l);
		if (rcode != AGPT_OK) return rcode;
		NEED(!(l.flags & AGPT_LIGHT_SAMPLE_SHAPE) || c->hostPrims[l.prim].type != AGPT_PRIM_INSTANCE, AGPT_ERR_INVALID,
			"AGPT_LIGHT_SAMPLE_SHAPE on an instanced shape (instanced emitters are not sampled)");
	}
	// An AreaLight wraps exactly one shape upstream (scene.h addAreaLight; lights.h:70-86), and the exact
	// MIS-ray cull relies on it: the primitive a light names must be the only one that names the light.
	for (size_t i = 0; i < c->hostPrims.size(); i++) {
		int al = c->hostPrims[i].area_light;
		NEED(al < 0 || (c->hostLights[al].type == AGPT_LIGHT_AREA && c->hostLights[al].prim == (int)i), AGPT_ERR_INVALID,
			"primitive and area light do not name each other (one shape per AreaLight)");
	}
	if (c->hasTextures) {
		// textures (extension): the binding table belongs to the resident material table, and binds Disney materials only
		NEED(c->hostBindings.size() == (size_t)c->nMats, AGPT_ERR_INVALID, "texture bindings were uploaded for a different number of materials");
		for (size_t i = 0; i < c->hostBindings.size(); i++) {
			const agpt_material_textures& b = c->hostBindings[i];
			NEED((b.base < 0 && b.roughness_metallic < 0 && b.normal < 0) || c->hostMatTypes[i] == AGPT_MAT_DISNEY, AGPT_ERR_INVALID,
				"a texture is bound to a material that is not AGPT_MAT_DISNEY");
		}
	}
	if (c->hasMasks) {
		// alpha masks (extension): the mask table belongs to the resident material table; masked spheres and emitters are not defined
		NEED(c->hostMasks.size() == (size_t)c->nMats, AGPT_ERR_INVALID, "alpha masks were uploaded for a different number of materials");
		for (const agpt_prim& p : c->hostPrims) {
			if (p.material < 0 || c->hostMasks[p.material].texture < 0) continue;
			NEED(p.type != AGPT_PRIM_SPHERE, AGPT_ERR_INVALID, "an alpha mask on a sphere's material");
			NEED(p.area_light < 0, AGPT_ERR_INVALID, "an alpha mask on an emitter's material");
		}
	}
	if (c->hasEmission) {
		// emissive materials (extension): the table belongs to the resident material table; an area light's Le and a material's
		// emission on one shape are not defined
		NEED(c->hostEmission.size() == (size_t)c->nMats, AGPT_ERR_INVALID, "emission rows were uploaded for a different number of materials");
		for (const agpt_prim& p : c->hostPrims)
			NEED(p.material < 0 || p.area_light < 0 || !Emits(c->hostEmission[p.material]), AGPT_ERR_INVALID,
				"an emissive material on a primitive that is an area light");
	}
	if (c->mats.p == nullptr) {
		// a scene of null-material (emissive) shapes only is legal upstream; shade still needs a record to point idle lanes at
		CU(cudaSetDevice(c->device));
		agpt_material none;
		memset(&none, 0, sizeof(none));
		CU(c->mats.Upload(&none, 1, c->stream));
		CU(cudaStreamSynchronize(c->stream));
	}
	if (c->runsDirty) {
		CU(cudaSetDevice(c->device));
		int rcode = BuildSphereRuns(c);
		if (rcode != AGPT_OK) return rcode;
	}
	if (c->shapesDirty) {
		CU(cudaSetDevice(c->device));
		int rcode = BuildShapeLights(c);
		if (rcode != AGPT_OK) return rcode;
	}
	return AGPT_OK;
}


// A film upload started by agpt_write_accum_begin may still be in flight: whatever touches the film next waits for it.
static int JoinUpload(agpt_ctx* c) {
	if (c != nullptr && c->uploadPending) {
		CU(cudaSetDevice(c->device));
		CU(cudaStreamSynchronize(c->copyStream));
		c->uploadPending = false;
	}
	return AGPT_OK;
}
#define JOIN(c) do { int j_ = JoinUpload(c); if (j_ != AGPT_OK) return j_; } while (0)

// ---- launches ---------------------------------------------------------------------------
// f(std::bool_constant<b>...) for the run-time flags b...: one instantiation per combination of the flags given
template <typename F>
static void WithBools(F&& f) { f(); }
template <typename F, typename... B>
static void WithBools(F&& f, bool b, B... rest) {
	if (b) WithBools([&](auto... t) { f(std::true_type(), t...); }, rest...);
	else WithBools([&](auto... t) { f(std::false_type(), t...); }, rest...);
}

// k_generate for g.n paths into the frame's slots and first-wave queues; LIST, the adaptive rounds' mode, when g names a pixel list
static int Generate(agpt_ctx* c, const Frame& f, const GenParams& g) {
	WithBools([&](auto LIST) { k_generate<LIST><<<Blocks(g.n, 256), 256, 0, c->stream>>>(f.sc, f.ps, f.q0, g); }, g.list != nullptr);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	return AGPT_OK;
}

// Trace kernels take <lead..., COUNT = AGPT_FLAG_COUNTERS, FAST = !AGPT_FLAG_STRICT_BOXES, INST>; while a mask is bound the
// *_masked ones run instead, which always take the instance path and so have no INST.
template <typename Plain, typename Masked, typename... Lead>
static void LaunchTrace(const LaunchPlan& p, uint32_t flags, Plain plain, Masked masked, Lead... lead) {
	const bool count = flags & AGPT_FLAG_COUNTERS, fast = !(flags & AGPT_FLAG_STRICT_BOXES);
	if (p.mk) WithBools(masked, lead..., count, fast);
	else WithBools(plain, lead..., count, fast, p.inst);
}

static void LaunchClosest(const LaunchPlan& p, uint32_t flags, int rays, cudaStream_t st, const DScene& sc, const PathState& ps, const int* queue, const int* n,
		unsigned long long* cnt, unsigned long long* row) {
	const int b = Blocks(rays, AGPT_TRACE_THREADS);
	LaunchTrace(p, flags, [&](auto C, auto F, auto I) { k_trace_closest<C, F, I><<<b, AGPT_TRACE_THREADS, 0, st>>>(sc, ps, queue, n, cnt, row); },
		[&](auto C, auto F) { k_trace_closest_masked<C, F><<<b, AGPT_TRACE_THREADS, 0, st>>>(sc, ps, queue, n, cnt, row, *p.mk); });
}
static void LaunchAny(const LaunchPlan& p, uint32_t flags, int rays, cudaStream_t st, const DScene& sc, const PathState& ps, const int* queue, const int* n,
		unsigned long long* cnt, unsigned long long* row) {
	const int b = Blocks(rays, AGPT_TRACE_THREADS);
	LaunchTrace(p, flags, [&](auto C, auto F, auto I) { k_trace_any<C, F, I><<<b, AGPT_TRACE_THREADS, 0, st>>>(sc, ps, queue, n, cnt, row); },
		[&](auto C, auto F) { k_trace_any_masked<C, F><<<b, AGPT_TRACE_THREADS, 0, st>>>(sc, ps, queue, n, cnt, row, *p.mk); });
}
static void LaunchTable(const LaunchPlan& p, uint32_t flags, bool any, cudaStream_t st, const DScene& sc, const float4* o, const float4* d, int n, agpt_hit* out,
		unsigned long long* cnt) {
	const int b = Blocks(n, AGPT_TRACE_THREADS);
	LaunchTrace(p, flags, [&](auto A, auto C, auto F, auto I) { k_trace_table<A, C, F, I><<<b, AGPT_TRACE_THREADS, 0, st>>>(sc, o, d, n, out, cnt); },
		[&](auto A, auto C, auto F) { k_trace_table_masked<A, C, F><<<b, AGPT_TRACE_THREADS, 0, st>>>(sc, o, d, n, out, cnt, *p.mk); }, any);
}

// k_shade_a<ENV>: ENV, the scene has an environment map; k_shade_a_emit<ENV> while an emission row emits
static void LaunchShadeA(const LaunchPlan& p, int active, cudaStream_t st, const DScene& sc, const PathState& ps, const int* queue, const int* n, int* survivors,
		int* survivorCount, int max_depth) {
	if (p.em) WithBools([&](auto E) { k_shade_a_emit<E><<<Blocks(active, 256), 256, 0, st>>>(sc, ps, queue, n, survivors, survivorCount, max_depth, *p.em); }, p.env);
	else WithBools([&](auto E) { k_shade_a<E><<<Blocks(active, 256), 256, 0, st>>>(sc, ps, queue, n, survivors, survivorCount, max_depth); }, p.env);
}

// k_shade_b<ENV, GLASS, SHAPES, TEX> has ten instantiations; each carries only what it needs, or everything.
//   a plain scene:                  <ENV, GLASS, false, 0>  (four)
//   a sampled shape light:          <false, false, true, 0>, or <true, true, true, 0> with an environment map or glass
//   textures (TEX 1), maps (TEX 2): <false, false, false, TEX>, or <true, true, true, TEX> with a shape light, an
//                                   environment map or glass
static void LaunchShadeB(const LaunchPlan& p, int blocks, cudaStream_t st, const DScene& sc, const PathState& ps, const int* survivors, const WaveQueues& qout,
		const ShadeParams& sp, RayCounters* rc) {
	auto launch = [&](auto E, auto G, auto S, auto T) { k_shade_b<E, G, S, T><<<blocks, AGPT_SHADE_THREADS, 0, st>>>(sc, p.st, ps, survivors, qout, sp, rc, p.tt); };
	const bool envOrGlass = p.env || p.glass;
	if (p.tex == 2) WithBools([&](auto all) { launch(all, all, all, std::integral_constant<int, 2>()); }, envOrGlass || p.shapes);
	else if (p.tex == 1) WithBools([&](auto all) { launch(all, all, all, std::integral_constant<int, 1>()); }, envOrGlass || p.shapes);
	else if (p.shapes) WithBools([&](auto all) { launch(all, all, std::true_type(), std::integral_constant<int, 0>()); }, envOrGlass);
	else WithBools([&](auto E, auto G) { launch(E, G, std::false_type(), std::integral_constant<int, 0>()); }, p.env, p.glass);
}

// k_guides; a textured material's albedo needs the texture tables (k_guides_tex), a mapped one also its material record (k_guides_maps)
static void LaunchGuides(const LaunchPlan& p, int pixels, cudaStream_t st, const DScene& sc, const PathState& ps, int ns, bool first, int total, float4* albedo,
		float4* normalDepth) {
	const int blocks = Blocks(pixels, 256);
	if (p.tex == 2) k_guides_maps<<<blocks, 256, 0, st>>>(sc, p.tt, ps, ns, first, total, albedo, normalDepth);
	else if (p.tex == 1) k_guides_tex<<<blocks, 256, 0, st>>>(sc, p.tt, ps, ns, first, total, albedo, normalDepth);
	else k_guides<<<blocks, 256, 0, st>>>(sc, ps, ns, first, total, albedo, normalDepth);
}


extern "C" {

const char* agpt_last_error(void) { return g_error.c_str(); }

int agpt_device_count(int* out) {
	NEED(out != nullptr, AGPT_ERR_INVALID, "null out");
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess) { *out = 0; return Fail(AGPT_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e)); }
	*out = n;
	return AGPT_OK;
}

int agpt_create(int device, agpt_ctx** out) {
	NEED(out != nullptr, AGPT_ERR_INVALID, "null out");
	*out = nullptr;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0)
		return Fail(AGPT_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
			" (libagpt has no CPU path)");
	NEED(device >= 0 && device < n, AGPT_ERR_INVALID, "device index out of range");
	CU(cudaSetDevice(device));
	std::unique_ptr<agpt_ctx> c(new agpt_ctx());
	c->device = device;
	memset(&c->stats, 0, sizeof(c->stats));
	cudaDeviceProp prop;
	CU(cudaGetDeviceProperties(&prop, device));
	c->smCount = prop.multiProcessorCount;
	CU(cudaStreamCreateWithFlags(&c->ownStream.h, cudaStreamNonBlocking));
	c->stream = c->ownStream;
	CU(cudaStreamCreateWithFlags(&c->sideStream.h, cudaStreamNonBlocking));
	CU(cudaStreamCreateWithFlags(&c->copyStream.h, cudaStreamNonBlocking));
	CU(cudaEventCreateWithFlags(&c->evUpload.h, cudaEventDisableTiming));
	CU(cudaEventCreateWithFlags(&c->evFork.h, cudaEventDisableTiming)); CU(cudaEventCreateWithFlags(&c->evJoin.h, cudaEventDisableTiming));
	CU(cudaEventCreate(&c->evA.h)); CU(cudaEventCreate(&c->evB.h)); CU(cudaEventCreate(&c->evC.h)); CU(cudaEventCreate(&c->evD.h));
	CU(cudaEventCreate(&c->evRender0.h)); CU(cudaEventCreate(&c->evRender1.h));
	CU(c->counts.Alloc(6));
	CU(c->survivorCount.Alloc(1));
	CU(c->hist.Alloc(3 * AGPT_BUCKETS));
	CU(c->traceCounters.Alloc(2 * AGPT_WAVE_COUNTERS * (1 + AGPT_MAX_WAVE_ROWS)));
	CU(c->rayCounters.Alloc(1));
	CU(cudaMemset(c->traceCounters.p, 0, c->traceCounters.Bytes()));
	CU(cudaMemset(c->rayCounters.p, 0, c->rayCounters.Bytes()));
	CU(cudaMallocHost((void**)&c->hostCounts.h, 8 * 3 * sizeof(int)));
	for (auto& e : c->ringEvents) CU(cudaEventCreateWithFlags(&e.h, cudaEventDisableTiming));
	if (const char* e = getenv("AGPT_ASYNC_WAVES")) c->asyncWaves = atoi(e) != 0;
	if (const char* e = getenv("AGPT_BATCH_LOG2")) { int b = atoi(e); if (b >= 10 && b <= 28) c->maxPathsPerBatch = (size_t)1 << b; }
	if (const char* e = getenv("AGPT_BUCKET_CALIBRATE")) c->calibrateGrid = atoi(e) != 0;
	if (const char* e = getenv("AGPT_MAX_SPHERE_RUN")) { int v = atoi(e); if (v >= 1) c->maxSphereRun = v; }
	if (const char* e = getenv("AGPT_OVERLAP_ANY")) c->overlapAny = atoi(e) != 0;
	if (const char* e = getenv("AGPT_BUCKET_RAYS")) c->bucketRays = atoi(e) != 0;
	*out = c.release();
	return AGPT_OK;
}

int agpt_destroy(agpt_ctx* c) {
	delete c;               // (null: nothing to do)
	return AGPT_OK;
}

int agpt_set_stream(agpt_ctx* c, void* s) {
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	c->stream = s ? (cudaStream_t)s : c->ownStream;
	return AGPT_OK;
}

// ---- scene upload ------------------------------------------------------------------------
// One pass over a caller-supplied node table before anything is uploaded: every interior link and
// leaf range must stay inside its table, the links must form a TREE (a child reached twice -- a
// shared child or a link back to an ancestor -- would make the walk loop or double-count), and the
// tree must not be deeper than the traversal stack.  The reference recurses without a limit
// (bvhtrimesh.h:332-413); the device stack holds AGPT_STACK_SMEM + AGPT_STACK_LOCAL far children,
// far more than any SAH tree over 2^31 triangles needs, and deeper tables are refused here
// instead of corrupting memory there.
static int ValidateBvh(const agpt_mesh_desc& d, int meshIndex, int* depthOut) {
	*depthOut = 0;
	if (d.n_nodes == 0) return AGPT_OK;
	const std::string where = "mesh " + std::to_string(meshIndex) + ": ";
	NEED(d.n_nodes == 1 || d.n_nodes >= 3, AGPT_ERR_INVALID, where + "node table of 2 entries (root at 0, slot 1 unused, children from 2)");
	std::vector<unsigned char> seen((size_t)d.n_nodes, 0);
	std::vector<std::pair<int, int>> todo;      // node, depth
	todo.emplace_back(0, 0);
	seen[0] = 1;
	int maxDepth = 0;
	while (!todo.empty()) {
		auto [k, depth] = todo.back();
		todo.pop_back();
		const agpt_bvh_node& nd = d.nodes[k];
		if (depth > maxDepth) maxDepth = depth;
		if (nd.count > 0) {
			NEED(nd.first >= 0 && (long long)nd.first + nd.count <= d.n_tris, AGPT_ERR_INVALID, where + "BVH leaf range outside the triangle table");
			continue;
		}
		NEED(nd.count == 0, AGPT_ERR_INVALID, where + "BVH node with a negative count");
		NEED(nd.first >= 2 && nd.first + 1 < d.n_nodes, AGPT_ERR_INVALID, where + "BVH child link outside the node table");
		NEED(!seen[nd.first] && !seen[nd.first + 1], AGPT_ERR_INVALID, where + "BVH node table is not a tree (a child is linked twice, or links back to an ancestor)");
		seen[nd.first] = seen[nd.first + 1] = 1;
		NEED(depth + 1 <= AGPT_STACK_SMEM + AGPT_STACK_LOCAL, AGPT_ERR_INVALID,
			where + "BVH deeper than " + std::to_string(AGPT_STACK_SMEM + AGPT_STACK_LOCAL) + " levels (the device traversal stack)");
		todo.emplace_back(nd.first, depth + 1);
		todo.emplace_back(nd.first + 1, depth + 1);
	}
	*depthOut = maxDepth;
	return AGPT_OK;
}

// Every agpt_upload_* once its arguments have passed their checks: the work still queued on the old tables finishes, and the
// guides and the saved reprojection view of the old scene become stale.
static int BeginSceneChange(agpt_ctx* c) {
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	c->stateGen++;
	c->historyGen++;
	return AGPT_OK;
}

int agpt_upload_meshes(agpt_ctx* c, const agpt_mesh_desc* meshes, int n) {
	NEED(c != nullptr && n >= 0 && (n == 0 || meshes != nullptr), AGPT_ERR_INVALID, "bad mesh table");
	// validate every descriptor before touching what is resident: a refused upload leaves the old scene intact
	int maxDepth = 0;
	for (int i = 0; i < n; i++) {
		const agpt_mesh_desc& d = meshes[i];
		NEED(d.n_tris >= 0 && d.n_nodes >= 0 && (d.n_tris == 0 || (d.tri_verts && d.tri_ids)), AGPT_ERR_INVALID, "mesh without triangle data");
		NEED(d.n_nodes == 0 || d.nodes != nullptr, AGPT_ERR_INVALID, "mesh node table missing");
		int depth = 0;
		int rcode = ValidateBvh(d, i, &depth);
		if (rcode != AGPT_OK) return rcode;
		if (depth > maxDepth) maxDepth = depth;
	}
	int rcode = BeginSceneChange(c);
	if (rcode != AGPT_OK) return rcode;
	c->gridCalibrated = false;
	// the new tables are built beside the resident ones, which a failure leaves in place
	std::vector<MeshStore> store((size_t)n);
	std::vector<DMesh> table(n);
	for (int i = 0; i < n; i++) {
		const agpt_mesh_desc& d = meshes[i];
		MeshStore& st = store[i];
		CU(st.nodes.Upload((const float4*)d.nodes, 2 * (size_t)d.n_nodes, c->stream));
		CU(st.tris.Upload((const float4*)d.tri_verts, 3 * (size_t)d.n_tris, c->stream));
		CU(st.ids.Upload(d.tri_ids, (size_t)d.n_tris, c->stream));
		if (d.tri_normals) CU(st.normals.Upload((const float4*)d.tri_normals, 3 * (size_t)d.n_tris, c->stream));
		if (d.tri_uvs) CU(st.uvs.Upload((const float2*)d.tri_uvs, 3 * (size_t)d.n_tris, c->stream));
		if (d.n_tris > 0) {
			k_flag_degenerate<<<Blocks(d.n_tris, 256), 256, 0, c->stream>>>(st.tris.p, st.uvs.p, d.n_tris);
			CU(cudaGetLastError());
			c->stats.kernel_launches++;
		}
		DMesh& m = table[i];
		m.nodes = st.nodes.p; m.tris = st.tris.p; m.ids = st.ids.p; m.normals = st.normals.p; m.uvs = st.uvs.p;
		m.n_nodes = d.n_nodes; m.n_tris = d.n_tris;
	}
	DevBuf<DMesh> dtable;
	CU(dtable.Upload(table.data(), (size_t)n, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	c->meshStore = std::move(store); c->meshes = std::move(dtable);
	c->nMeshes = n;
	c->maxBvhDepth = maxDepth;
	c->hostRoots.assign((size_t)n, agpt_bvh_node());
	for (int i = 0; i < n; i++) { if (meshes[i].n_nodes > 0) c->hostRoots[i] = meshes[i].nodes[0]; else c->hostRoots[i].count = -1; }
	c->runsDirty = true;
	c->shapesDirty = true;
	bool any = false;
	for (int i = 0; i < n; i++) {
		if (meshes[i].n_nodes == 0) continue;
		const agpt_bvh_node& r = meshes[i].nodes[0];
		for (int a = 0; a < 3; a++) {
			c->boundsLo[a] = any ? (r.bmin[a] < c->boundsLo[a] ? r.bmin[a] : c->boundsLo[a]) : r.bmin[a];
			c->boundsHi[a] = any ? (r.bmax[a] > c->boundsHi[a] ? r.bmax[a] : c->boundsHi[a]) : r.bmax[a];
		}
		any = true;
	}
	return AGPT_OK;
}

// The new table replaces the resident one, and `counter` describes it, only once its upload has completed.
#define SIMPLE_UPLOAD(fn, T, member, counter) \
	int fn(agpt_ctx* c, const T* rows, int n) { \
		NEED(c != nullptr && n >= 0 && (n == 0 || rows != nullptr), AGPT_ERR_INVALID, "bad table"); \
		int rcode = BeginSceneChange(c); \
		if (rcode != AGPT_OK) return rcode; \
		DevBuf<T> table; \
		CU(table.Upload(rows, (size_t)n, c->stream)); \
		CU(cudaStreamSynchronize(c->stream)); \
		c->member = std::move(table); \
		counter; \
		return AGPT_OK; \
	}
SIMPLE_UPLOAD(agpt_upload_spheres, agpt_sphere, spheres, c->nSpheres = n; c->hostSpheres.assign(rows, rows + n); c->runsDirty = true)
SIMPLE_UPLOAD(agpt_upload_planes, agpt_plane, planes, c->nPlanes = n; c->hostPlanes.assign(rows, rows + n); c->shapesDirty = true)
SIMPLE_UPLOAD(agpt_upload_materials, agpt_material, mats, c->nMats = n; c->hasGlass = false; for (int i = 0; i < n; i++) if (rows[i].lobes & (AGPT_LOBE_GLASS_REFLECT | AGPT_LOBE_GLASS_TRANSMIT)) c->hasGlass = true;
	c->hostMatTypes.resize((size_t)n); for (int i = 0; i < n; i++) c->hostMatTypes[i] = rows[i].type)
static int UploadLights(agpt_ctx* c, const agpt_light* rows, int n);
SIMPLE_UPLOAD(UploadLights, agpt_light, lights, c->hostLights.assign(rows, rows + n); c->shapesDirty = true)
int agpt_upload_lights(agpt_ctx* c, const agpt_light* rows, int n) {
	// refused flags leave the resident scene as it was
	for (int i = 0; rows != nullptr && i < n; i++) {
		int rcode = CheckLightFlags(rows[i]);
		if (rcode != AGPT_OK) return rcode;
	}
	return UploadLights(c, rows, n);
}
SIMPLE_UPLOAD(agpt_upload_primitives, agpt_prim, prims, c->hostPrims.assign(rows, rows + n); c->runsDirty = true; c->shapesDirty = true)
SIMPLE_UPLOAD(agpt_upload_instances, agpt_instance, instances, c->nInstances = n; c->hostInstances.assign(rows, rows + n))

int agpt_upload_envmap(agpt_ctx* c, const agpt_envmap* env) {
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	const bool clear = !env || env->width == 0;
	NEED(clear || (env->width > 0 && env->height > 0 && env->rgb && env->func && env->cdf), AGPT_ERR_INVALID, "bad environment map");
	int rcode = BeginSceneChange(c);
	if (rcode != AGPT_OK) return rcode;
	if (clear) {
		c->envRgb.Free(); c->envFunc.Free(); c->envCdf.Free();
		c->envW = c->envH = 0; c->envFuncInt = 0;
		return AGPT_OK;
	}
	size_t n = (size_t)env->width * env->height;
	DevBuf<float> rgb, func, cdf;
	CU(rgb.Upload(env->rgb, 3 * n, c->stream));
	CU(func.Upload(env->func, n, c->stream));
	CU(cdf.Upload(env->cdf, n + 1, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	c->envRgb = std::move(rgb); c->envFunc = std::move(func); c->envCdf = std::move(cdf);
	c->envW = env->width; c->envH = env->height; c->envFuncInt = env->func_int;
	return AGPT_OK;
}

// EXTENSION (agpt.h agpt_upload_textures, agpt_upload_material_textures): the one upload path of textures and their bindings.
// Every argument is checked before anything resident changes.
static int UploadMaterialTextures(agpt_ctx* c, const agpt_texture* textures, int n_textures, const agpt_material_textures* bindings, int n_materials) {
	NEED(c != nullptr && n_textures >= 0 && n_materials >= 0 && (n_textures == 0 || textures != nullptr) && (n_materials == 0 || bindings != nullptr),
		AGPT_ERR_INVALID, "agpt_upload_textures: bad table");
	size_t total = 0;
	for (int i = 0; i < n_textures; i++) {
		const agpt_texture& t = textures[i];
		NEED(t.width >= 1 && t.height >= 1 && (long long)t.width * t.height <= (1ll << 28), AGPT_ERR_INVALID, "agpt_upload_textures: need 1 <= width, height and width * height <= 2^28");
		NEED(t.rgb != nullptr, AGPT_ERR_INVALID, "agpt_upload_textures: texture without texels");
		const size_t n = 3 * (size_t)t.width * t.height;
		for (size_t k = 0; k < n; k++) NEED(std::isfinite(t.rgb[k]), AGPT_ERR_INVALID, "agpt_upload_textures: texel not finite");
		total += (size_t)t.width * t.height;
	}
	for (int i = 0; i < n_materials; i++) {
		const agpt_material_textures& b = bindings[i];
		for (int32_t t : { b.base, b.roughness_metallic, b.normal })
			NEED(t >= -1 && t < n_textures, AGPT_ERR_INVALID, "agpt_upload_textures: material points outside the texture table");
		NEED(std::isfinite(b.normal_scale) && std::isfinite(b.color[0]) && std::isfinite(b.color[1]) && std::isfinite(b.color[2]), AGPT_ERR_INVALID,
			"agpt_upload_material_textures: normal_scale or color not finite");
	}
	int rcode = BeginSceneChange(c);
	if (rcode != AGPT_OK) return rcode;
	std::vector<float4> texels(total);
	std::vector<DTexture> desc((size_t)n_textures);
	size_t off = 0;
	for (int i = 0; i < n_textures; i++) {
		const agpt_texture& t = textures[i];
		desc[i].width = t.width; desc[i].height = t.height; desc[i].off = (long long)off;
		const size_t n = (size_t)t.width * t.height;
		for (size_t k = 0; k < n; k++) texels[off + k] = make_float4(t.rgb[3 * k], t.rgb[3 * k + 1], t.rgb[3 * k + 2], 0.f);
		off += n;
	}
	bool hasTextures = false, hasMaps = false;
	std::vector<int32_t> matTex((size_t)n_materials);
	std::vector<DMatMaps> maps((size_t)n_materials);
	for (int i = 0; i < n_materials; i++) {
		const agpt_material_textures& b = bindings[i];
		matTex[i] = b.base;
		maps[i] = DMatMaps{ b.base, b.roughness_metallic, b.normal, b.normal_scale, { b.color[0], b.color[1], b.color[2] }, 0.f };
		if (b.base >= 0 || b.roughness_metallic >= 0 || b.normal >= 0) hasTextures = true;
		if (b.roughness_metallic >= 0 || b.normal >= 0) hasMaps = true;
	}
	DevBuf<float4> dTexels; DevBuf<DTexture> dTextures; DevBuf<int> dMatTex; DevBuf<DMatMaps> dMatMaps;
	CU(dTexels.Upload(texels.data(), texels.size(), c->stream));
	CU(dTextures.Upload(desc.data(), desc.size(), c->stream));
	CU(dMatTex.Upload(matTex.data(), matTex.size(), c->stream));
	CU(dMatMaps.Upload(maps.data(), hasMaps ? maps.size() : 0, c->stream));     // read by the TEX == 2 kernels only
	CU(cudaStreamSynchronize(c->stream));
	c->texels = std::move(dTexels); c->textures = std::move(dTextures); c->matTex = std::move(dMatTex); c->matMaps = std::move(dMatMaps);
	c->hasTextures = hasTextures; c->hasMaps = hasMaps;
	c->hostBindings.assign(bindings, bindings + n_materials);
	c->masks.Free(); c->hostMasks.clear(); c->hasMasks = false;     // alpha masks name textures of the old table
	c->emission.Free(); c->hostEmission.clear(); c->hasEmission = false;     // ... and so do emission rows
	return AGPT_OK;
}
int agpt_upload_textures(agpt_ctx* c, const agpt_texture* textures, int n_textures, const int32_t* material_texture, int n_materials) {
	NEED(c != nullptr && n_materials >= 0 && (n_materials == 0 || material_texture != nullptr), AGPT_ERR_INVALID, "agpt_upload_textures: bad table");
	std::vector<agpt_material_textures> b((size_t)n_materials);
	for (int i = 0; i < n_materials; i++) b[i] = agpt_material_textures{ material_texture[i], -1, -1, 1.f, { 0.f, 0.f, 0.f } };
	return UploadMaterialTextures(c, textures, n_textures, b.data(), n_materials);
}
int agpt_upload_material_textures(agpt_ctx* c, const agpt_texture* textures, int n_textures, const agpt_material_textures* bindings, int n_materials) {
	return UploadMaterialTextures(c, textures, n_textures, bindings, n_materials);
}

// EXTENSION (agpt.h agpt_upload_alpha_masks).  Every argument is checked before anything resident changes.
int agpt_upload_alpha_masks(agpt_ctx* c, const agpt_alpha_mask* masks, int n_materials) {
	NEED(c != nullptr && n_materials >= 0 && (n_materials == 0 || masks != nullptr), AGPT_ERR_INVALID, "agpt_upload_alpha_masks: bad table");
	bool hasMasks = false;
	for (int i = 0; i < n_materials; i++) {
		const agpt_alpha_mask& m = masks[i];
		NEED(m.texture >= -1 && m.texture < (int)c->textures.n, AGPT_ERR_INVALID, "agpt_upload_alpha_masks: material points outside the resident textures");
		NEED(m.channel >= 0 && m.channel <= 2, AGPT_ERR_INVALID, "agpt_upload_alpha_masks: channel outside [0, 2]");
		NEED(std::isfinite(m.cutoff), AGPT_ERR_INVALID, "agpt_upload_alpha_masks: cutoff not finite");
		if (m.texture >= 0) hasMasks = true;
	}
	int rcode = BeginSceneChange(c);
	if (rcode != AGPT_OK) return rcode;
	DevBuf<agpt_alpha_mask> dMasks;
	CU(dMasks.Upload(masks, (size_t)n_materials, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	c->masks = std::move(dMasks);
	c->hostMasks.assign(masks, masks + n_materials);
	c->hasMasks = hasMasks;
	return AGPT_OK;
}

// EXTENSION (agpt.h agpt_upload_emission).  Every argument is checked before anything resident changes.
int agpt_upload_emission(agpt_ctx* c, const agpt_emission* rows, int n_materials) {
	NEED(c != nullptr && n_materials >= 0 && (n_materials == 0 || rows != nullptr), AGPT_ERR_INVALID, "agpt_upload_emission: bad table");
	bool hasEmission = false;
	for (int i = 0; i < n_materials; i++) {
		const agpt_emission& e = rows[i];
		NEED(e.texture >= -1 && e.texture < (int)c->textures.n, AGPT_ERR_INVALID, "agpt_upload_emission: material points outside the resident textures");
		for (float f : e.factor) NEED(std::isfinite(f) && f >= 0.f, AGPT_ERR_INVALID, "agpt_upload_emission: factor not finite or negative");
		if (Emits(e)) hasEmission = true;
	}
	int rcode = BeginSceneChange(c);
	if (rcode != AGPT_OK) return rcode;
	DevBuf<agpt_emission> dRows;
	CU(dRows.Upload(rows, (size_t)n_materials, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	c->emission = std::move(dRows);
	c->hostEmission.assign(rows, rows + n_materials);
	c->hasEmission = hasEmission;
	return AGPT_OK;
}

int agpt_set_camera(agpt_ctx* c, const agpt_camera* cam) {
	NEED(c != nullptr && cam != nullptr, AGPT_ERR_INVALID, "null camera");
	c->cam = *cam;
	c->haveCam = true;
	c->stateGen++;
	c->gridCalibrated = false;
	return AGPT_OK;
}

// Zeroed moments and a pixel list for a film of wh pixels: they replace the resident ones once both exist
static int AllocMoments(agpt_ctx* c, size_t wh) {
	DevBuf<float4> moments;
	DevBuf<int> list;
	CU(moments.Alloc(wh));
	CU(list.Alloc(wh));
	if (!c->adaptiveCount.p) CU(c->adaptiveCount.Alloc(1));
	CU(cudaMemsetAsync(moments.p, 0, moments.Bytes(), c->stream));
	c->moments = std::move(moments); c->adaptiveList = std::move(list);
	return AGPT_OK;
}

int agpt_set_film(agpt_ctx* c, int width, int height) {
	JOIN(c);
	NEED(c != nullptr && width > 0 && height > 0 && (long long)width * height < (1ll << 30), AGPT_ERR_INVALID, "bad film size");
	CU(cudaSetDevice(c->device));
	c->stateGen++;
	if (width == c->width && height == c->height) return AGPT_OK;
	c->historyGen++;
	CU(cudaStreamSynchronize(c->stream));
	const bool own = c->accum == c->accumOwn.p;
	DevBuf<float4> film;
	if (own) {
		CU(film.Alloc((size_t)width * height));
		CU(cudaMemsetAsync(film.p, 0, film.Bytes(), c->stream));
	}
	if (c->momentsOn) {                      // (the last step that can fail: it replaces the resident moments when it succeeds)
		int rcode = AllocMoments(c, (size_t)width * height);
		if (rcode != AGPT_OK) return rcode;
	}
	c->width = width; c->height = height;
	if (own) {
		c->accumOwn = std::move(film);
		c->accum = c->accumOwn.p;
	}
	return AGPT_OK;
}

int agpt_scene_bytes(agpt_ctx* c, uint64_t* out) {
	NEED(c != nullptr && out != nullptr, AGPT_ERR_INVALID, "null argument");
	uint64_t b = c->envRgb.Bytes() + c->envFunc.Bytes() + c->envCdf.Bytes() + c->meshes.Bytes() + c->spheres.Bytes() + c->planes.Bytes() + c->prims.Bytes() + c->instances.Bytes() + c->mats.Bytes() + c->lights.Bytes()
		+ c->shapeLights.Bytes() + c->shapeCdf.Bytes() + c->texels.Bytes() + c->textures.Bytes() + c->matTex.Bytes() + c->matMaps.Bytes() + c->masks.Bytes()
		+ c->emission.Bytes();
	for (auto& m : c->meshStore) b += m.nodes.Bytes() + m.tris.Bytes() + m.normals.Bytes() + m.uvs.Bytes() + m.ids.Bytes();
	*out = b;
	return AGPT_OK;
}

// ---- accumulator -------------------------------------------------------------------------
int agpt_clear(agpt_ctx* c) {
	JOIN(c);
	NEED(c != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "film not set");
	CU(cudaSetDevice(c->device));
	CU(cudaMemsetAsync(c->accum, 0, (size_t)c->width * c->height * sizeof(float4), c->stream));
	if (c->momentsOn) CU(cudaMemsetAsync(c->moments.p, 0, c->moments.Bytes(), c->stream));
	return AGPT_OK;
}
int agpt_accum_ptr_dev(agpt_ctx* c, void** p) {
	JOIN(c);
	NEED(c != nullptr && p != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "film not set");
	*p = c->accum;
	return AGPT_OK;
}
int agpt_set_accum_dev(agpt_ctx* c, void* p) {
	JOIN(c);
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	NEED(c->width > 0, AGPT_ERR_STATE, "film not set");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	if (p) c->accum = (float4*)p;
	else {
		if (!c->accumOwn.p) { CU(c->accumOwn.Alloc((size_t)c->width * c->height)); CU(cudaMemset(c->accumOwn.p, 0, c->accumOwn.Bytes())); }
		c->accum = c->accumOwn.p;
	}
	return AGPT_OK;
}
int agpt_read_accum(agpt_ctx* c, float* host) {
	JOIN(c);
	NEED(c != nullptr && host != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "film not set");
	CU(cudaSetDevice(c->device));
	CU(cudaMemcpyAsync(host, c->accum, (size_t)c->width * c->height * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}
int agpt_write_accum(agpt_ctx* c, const float* host) {
	JOIN(c);
	NEED(c != nullptr && host != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "film not set");
	CU(cudaSetDevice(c->device));
	CU(cudaMemcpyAsync(c->accum, host, (size_t)c->width * c->height * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}
int agpt_write_accum_begin(agpt_ctx* c, const float* host) {
	JOIN(c);
	NEED(c != nullptr && host != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "film not set");
	CU(cudaSetDevice(c->device));
	// everything queued on the render stream so far (a clear, an earlier render's accumulate) comes first
	CU(cudaEventRecord(c->evUpload, c->stream));
	CU(cudaStreamWaitEvent(c->copyStream, c->evUpload, 0));
	CU(cudaMemcpyAsync(c->accum, host, (size_t)c->width * c->height * sizeof(float4), cudaMemcpyHostToDevice, c->copyStream));
	CU(cudaEventRecord(c->evUpload, c->copyStream));
	c->uploadPending = true;
	return AGPT_OK;
}
int agpt_resolve(agpt_ctx* c, int samples, uint32_t* host) {
	JOIN(c);
	NEED(c != nullptr && host != nullptr && c->accum != nullptr && samples > 0, AGPT_ERR_STATE, "film not set or samples <= 0");
	CU(cudaSetDevice(c->device));
	int n = c->width * c->height;
	if (c->resolved.n != (size_t)n) CU(c->resolved.Alloc(n));
	k_resolve<<<Blocks(n, 256), 256, 0, c->stream>>>(c->accum, c->resolved.p, n, (float)samples);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(host, c->resolved.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

// ---- the wave loop -------------------------------------------------------------------------
// Generates the g.n paths of g (k_generate: slots 0..n-1, queues A and counts A) and runs them to
// completion.  Queue lengths stay on the device (kernels read them); the host sizes grids from
// upper bounds.  Default: after every wave the host waits for that wave's three counts (one
// 12-byte copy to pinned memory), so the bounds are exact and the loop ends with the wave that
// empties the active list.  Optional (asyncWaves): the host runs up to kMaxAhead waves ahead of
// the newest landed counts, tightening bounds as copies land (the active list only shrinks: a
// later wave has at most `active` paths, 2*active closest-hit rays and `active` shadow rays);
// empty waves launched past the end are no-ops.  AGPT_FLAG_TIMING brackets the kernel classes
// of every wave with events.
static const int kMaxAhead = 2, kRing = 8;
static const int kSmallWave = 16384;
// The bucket grid should resolve the part of the scene the rays are in, not the scene's bounding
// box (cfg 3: a 40-unit backdrop around 15 units of objects left 12 of the 512 cells in use).
// Once per scene and camera, after the first camera rays have been traced, a strided sample of
// their hit points is read back and the grid is laid over mean +- 2.5 sigma of it.  Ray order
// only: results do not depend on the grid.
static int CalibrateBucketGrid(agpt_ctx* c, const PathState& ps, int n) {
	const int samples = n < 65536 ? n : 65536;
	const size_t pitch = (size_t)(n / samples) * sizeof(float4);
	std::vector<float4> o(samples), d(samples), h(samples);
	CU(cudaMemcpy2DAsync(o.data(), sizeof(float4), (const float4*)ps.rayO, pitch, sizeof(float4), samples, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpy2DAsync(d.data(), sizeof(float4), (const float4*)ps.rayD, pitch, sizeof(float4), samples, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpy2DAsync(h.data(), sizeof(float4), (const float4*)ps.hitA, pitch, sizeof(float4), samples, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	double sum[3] = { 0, 0, 0 }, sq[3] = { 0, 0, 0 };
	long hits = 0;
	for (int i = 0; i < samples; i++) {
		int prim; memcpy(&prim, &h[i].w, sizeof(prim));
		float t = h[i].x;
		if (prim < 0 || !(t > 0.f) || !(t < 1e30f)) continue;
		double p[3] = { o[i].x + (double)t * d[i].x, o[i].y + (double)t * d[i].y, o[i].z + (double)t * d[i].z };
		for (int a = 0; a < 3; a++) { sum[a] += p[a]; sq[a] += p[a] * p[a]; }
		hits++;
	}
	c->gridCalibrated = true;
	for (int a = 0; a < 3; a++) { c->gridLo[a] = c->boundsLo[a]; c->gridHi[a] = c->boundsHi[a]; }
	if (hits < 256) return AGPT_OK;                       // too little to go by: keep the mesh bounds
	for (int a = 0; a < 3; a++) {
		double mean = sum[a] / hits, var = sq[a] / hits - mean * mean;
		double sigma = var > 0 ? sqrt(var) : 0;
		if (sigma <= 0) continue;
		c->gridLo[a] = (float)(mean - 2.5 * sigma);
		c->gridHi[a] = (float)(mean + 2.5 * sigma);
	}
	return AGPT_OK;
}

static int RunWaves(agpt_ctx* c, const Frame& f, const GenParams& g, int max_depth, int rr_depth_arg, uint32_t flags) {
	const bool count = flags & AGPT_FLAG_COUNTERS, timing = flags & AGPT_FLAG_TIMING;
	const int n = g.n;
	int rcode = Generate(c, f, g);
	if (rcode != AGPT_OK) return rcode;
	const PathState& ps = f.ps;
	DScene sc = f.sc;
	c->stats.paths += (uint64_t)n;
	c->stats.rays_closest += (uint64_t)n;     // camera rays; the rest is counted on the device
	WaveQueues q[2];
	for (int k = 0; k < 2; k++) {
		q[k].closest = c->queues[0 + k].p; q[k].shadow = c->queues[2 + k].p; q[k].active = c->queues[4 + k].p;
		q[k].counts = c->counts.p + 3 * k;
		q[k].keys = c->keys[k].p; q[k].shadowKeys = c->shadowKeys[k].p;
	}
	int* bucketHist = c->hist.p;
	int* bucketOffsets = c->hist.p + AGPT_BUCKETS;
	int* bucketRunning = c->hist.p + 2 * AGPT_BUCKETS;
	const bool bucketing = c->bucketRays;
	const bool overlap = c->overlapAny && !timing;
	float msClosest = 0, msAny = 0, msShade = 0;
	unsigned long long* cntClosest = c->traceCounters.p;
	unsigned long long* cntAny = c->traceCounters.p + AGPT_WAVE_COUNTERS;
	unsigned long long* waveRows = c->traceCounters.p + 2 * AGPT_WAVE_COUNTERS;      // [kind][wave][8]

	int ubClosest = n, ubShadow = 0, ubActive = n;   // upper bounds of the current wave's queue lengths
	int cur = 0, wave = 0;
	int ringHead = 0, ringTail = 0;                  // copies in flight: [ringTail, ringHead)
	bool done = false;
	while (!done) {
		// ---- one wave on q[cur] -> q[cur ^ 1] ----
		const int* closestQueue = q[cur].closest;
		const int* shadowQueue = q[cur].shadow;
		if (wave > 0 && bucketing) {
			// bucket pass: rays that start in the same cell going the same way end up adjacent
			// (not worth its six launches for the last few thousand rays of a batch)
			const int perBlock = 256 * AGPT_BUCKET_ITEMS;
			if (ubClosest >= kSmallWave) {
				CU(cudaMemsetAsync(bucketHist, 0, AGPT_BUCKETS * sizeof(int), c->stream));
				k_bucket_hist<<<Blocks(ubClosest, perBlock), 256, 0, c->stream>>>(q[cur].keys, q[cur].counts + 0, bucketHist);
				k_bucket_scan<<<1, 1024, 0, c->stream>>>(bucketHist, bucketOffsets, bucketRunning);
				k_bucket_scatter<<<Blocks(ubClosest, perBlock), 256, 0, c->stream>>>(q[cur].closest, q[cur].keys, q[cur].counts + 0, bucketOffsets, bucketRunning, c->sortedClosest.p);
				c->stats.kernel_launches += 3;
				closestQueue = c->sortedClosest.p;
			}
			if (ubShadow >= kSmallWave) {
				CU(cudaMemsetAsync(bucketHist, 0, AGPT_BUCKETS * sizeof(int), c->stream));
				k_bucket_hist<<<Blocks(ubShadow, perBlock), 256, 0, c->stream>>>(q[cur].shadowKeys, q[cur].counts + 1, bucketHist);
				k_bucket_scan<<<1, 1024, 0, c->stream>>>(bucketHist, bucketOffsets, bucketRunning);
				k_bucket_scatter<<<Blocks(ubShadow, perBlock), 256, 0, c->stream>>>(q[cur].shadow, q[cur].shadowKeys, q[cur].counts + 1, bucketOffsets, bucketRunning, c->sortedShadow.p);
				c->stats.kernel_launches += 3;
				shadowQueue = c->sortedShadow.p;
			}
		}
		// The two traces of a wave are independent (different queues, different result arrays):
		// unless per-kernel timing is on, the any-hit trace runs on the side stream so that each
		// fills the SMs the other's tail leaves idle.
		const bool fork = overlap && ubClosest > 0 && ubShadow > 0;
		const int row = wave < AGPT_MAX_WAVE_ROWS ? wave : AGPT_MAX_WAVE_ROWS - 1;
		if (timing) CU(cudaEventRecord(c->evA, c->stream));
		if (fork) CU(cudaEventRecord(c->evFork, c->stream));
		if (ubClosest > 0) {
			LaunchClosest(f.plan, flags, ubClosest, c->stream, sc, ps, closestQueue, q[cur].counts + 0, cntClosest, waveRows + (size_t)AGPT_WAVE_COUNTERS * row);
			c->stats.kernel_launches++; c->stats.launches_closest++;
		}
		if (wave == 0 && bucketing && !c->gridCalibrated && c->calibrateGrid && n >= 4096) {
			// first camera rays of this scene and camera: lay the bucket grid where they land
			rcode = CalibrateBucketGrid(c, ps, n);
			if (rcode != AGPT_OK) return rcode;
			SetBucketGrid(sc, c->gridLo, c->gridHi);
		}
		if (timing) CU(cudaEventRecord(c->evB, c->stream));
		if (ubShadow > 0) {
			if (fork) CU(cudaStreamWaitEvent(c->sideStream, c->evFork, 0));
			LaunchAny(f.plan, flags, ubShadow, fork ? c->sideStream : c->stream, sc, ps, shadowQueue, q[cur].counts + 1, cntAny,
				waveRows + (size_t)AGPT_WAVE_COUNTERS * (AGPT_MAX_WAVE_ROWS + row));
			c->stats.kernel_launches++; c->stats.launches_any++;
			if (fork) {
				CU(cudaEventRecord(c->evJoin, c->sideStream));
				CU(cudaStreamWaitEvent(c->stream, c->evJoin, 0));
			}
		}
		CU(cudaMemsetAsync(q[cur ^ 1].counts, 0, 3 * sizeof(int), c->stream));
		if (timing) CU(cudaEventRecord(c->evC, c->stream));
		ShadeParams sp;
		// with an emitting row bound the path ray at bounces == max_depth may hit an emitter, so k_shade_b must not cull it: it sees
		// a depth one larger (sp.max_depth is read by that cull only), while k_shade_a still ends every path at max_depth, after its
		// emission.  k_shade_b's code stays as it is.
		const int shadeDepth = f.plan.em ? (max_depth == INT_MAX ? INT_MAX : max_depth + 1) : max_depth;
		sp.count = q[cur].counts + 2; sp.max_depth = shadeDepth; sp.rr_depth_arg = rr_depth_arg; sp.rr_by_bounce = (flags & AGPT_FLAG_RR_BY_BOUNCE) ? 1 : 0; sp.exact_counts = count ? 1 : 0;
		// shade: k_shade_a (per active entry: NEE fold, emission, termination -> survivor list),
		// then k_shade_b (per survivor: the BSDF work), blocks striding over the list
		CU(cudaMemsetAsync(c->survivorCount.p, 0, sizeof(int), c->stream));
		sp.count = c->survivorCount.p;
		LaunchShadeA(f.plan, ubActive, c->stream, sc, ps, q[cur].active, q[cur].counts + 2, c->survivors.p, c->survivorCount.p, max_depth);
		// upper bound: blocks past the survivor count return at once
		LaunchShadeB(f.plan, Blocks(ubActive, AGPT_SHADE_THREADS), c->stream, sc, ps, c->survivors.p, q[cur ^ 1], sp, c->rayCounters.p);
		c->stats.kernel_launches += 2; c->stats.launches_shade++;
		CU(cudaGetLastError());
		if (timing) CU(cudaEventRecord(c->evD, c->stream));
		// counts of the NEXT wave -> pinned ring slot, marked by an event
		int slot = ringHead % kRing;
		CU(cudaMemcpyAsync(c->hostCounts + 3 * slot, q[cur ^ 1].counts, 3 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
		CU(cudaEventRecord(c->ringEvents[slot], c->stream));
		ringHead++;
		cur ^= 1; wave++;
		c->stats.waves++;
		// the next wave's bounds follow from this wave's: the active list only shrinks
		ubClosest = 2 * ubActive < (int)(2 * c->capacity) ? 2 * ubActive : (int)(2 * c->capacity);
		ubShadow = ubActive;

		// ---- consume the copies that have landed (block only when too far ahead, or when timing) ----
		while (ringTail < ringHead) {
			int s = ringTail % kRing;
			// small waves (the stragglers at the end of a batch) are launched from the last known
			// bounds without waiting for their counts: nothing to lose on a few thousand entries
			bool runAhead = c->asyncWaves || ubActive < kSmallWave;
			bool mustWait = timing || !runAhead || (ringHead - ringTail) >= kMaxAhead;
			cudaError_t e = mustWait ? cudaEventSynchronize(c->ringEvents[s]) : cudaEventQuery(c->ringEvents[s]);
			if (e == cudaErrorNotReady) break;
			if (e != cudaSuccess) return Fail(AGPT_ERR_CUDA, std::string("wave loop: ") + cudaGetErrorString(e));
			const int* hc = c->hostCounts + 3 * s;        // (closest, shadow, active) of wave ringTail + 1
			int landedWave = ringTail + 1;
			ringTail++;
			if (hc[2] == 0) { done = true; break; }
			if (landedWave == wave) { ubClosest = hc[0]; ubShadow = hc[1]; ubActive = hc[2]; }
			else {
				// older than the wave about to be launched: still bounds it
				if (hc[2] < ubActive) ubActive = hc[2];
				if (2 * hc[2] < ubClosest) ubClosest = 2 * hc[2];
				if (hc[2] < ubShadow) ubShadow = hc[2];
			}
		}
		if (timing) {
			float a = 0, b = 0, d = 0;
			cudaEventElapsedTime(&a, c->evA, c->evB);
			cudaEventElapsedTime(&b, c->evB, c->evC);
			cudaEventElapsedTime(&d, c->evC, c->evD);
			msClosest += a; msAny += b; msShade += d;
		}
	}
	c->stats.ms_trace_closest += msClosest; c->stats.ms_trace_any += msAny; c->stats.ms_shade += msShade;
	return AGPT_OK;
}

// Samples per pixel in one batch of a whole-film call: as many as maxPathsPerBatch holds, at least one, at most num_samples (>= 1)
static int SamplesPerBatch(const agpt_ctx* c, int num_samples) {
	const int fit = (int)(c->maxPathsPerBatch / ((size_t)c->width * c->height));
	return std::min(std::max(fit, 1), num_samples);
}

int agpt_render(agpt_ctx* c, int first_sample, int num_samples, int sample_stride, int max_depth, int rr_depth_arg, uint32_t flags) {
	int rcode = CheckReady(c, true);
	if (rcode != AGPT_OK) return rcode;
	NEED(num_samples >= 0 && sample_stride >= 1 && max_depth >= 0, AGPT_ERR_INVALID, "bad sample range or depth");
	NEED(c->accum != nullptr, AGPT_ERR_STATE, "no accumulator");
	CU(cudaSetDevice(c->device));
	if (num_samples == 0) return AGPT_OK;
	const size_t wh = (size_t)c->width * c->height;
	const int perBatch = SamplesPerBatch(c, num_samples);
	rcode = EnsureCapacity(c, wh * perBatch);
	if (rcode != AGPT_OK) return rcode;
	const Frame f = MakeFrame(c);
	// evA/evC/evD are reused inside RunWaves when timing; the render bracket has its own pair
	cudaEvent_t r0 = c->evRender0, r1 = c->evRender1;
	CU(cudaEventRecord(r0, c->stream));
	for (int done = 0; done < num_samples; done += perBatch) {
		int ns = num_samples - done < perBatch ? num_samples - done : perBatch;
		GenParams g{};
		g.n = (int)(wh * ns); g.first_sample = first_sample + done * sample_stride; g.sample_stride = sample_stride; g.tiled = 1; g.samples = ns;
		rcode = RunWaves(c, f, g, max_depth, rr_depth_arg, flags);
		if (rcode != AGPT_OK) return rcode;
		if (c->uploadPending) CU(cudaStreamWaitEvent(c->stream, c->evUpload, 0));      // the film this batch adds to may still be on its way (agpt_write_accum_begin)
		if (c->momentsOn) k_accumulate<true, false><<<Blocks(wh, 256), 256, 0, c->stream>>>(f.ps.Lout, c->accum, c->width, c->height, ns, c->moments.p);
		else k_accumulate<false, false><<<Blocks(wh, 256), 256, 0, c->stream>>>(f.ps.Lout, c->accum, c->width, c->height, ns);
		CU(cudaGetLastError());
		c->stats.kernel_launches++;
	}
	CU(cudaEventRecord(r1, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	c->uploadPending = false;        // k_accumulate waited for it
	float ms = 0;
	cudaEventElapsedTime(&ms, r0, r1);
	c->stats.ms_render += ms;
	return AGPT_OK;
}

// ---- adaptive sampling (EXTENSION, agpt.h agpt_adaptive) ----------------------------------------------------------------
int agpt_set_moments(agpt_ctx* c, int enable) {
	JOIN(c);
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	if (!enable) {
		c->momentsOn = false;
		c->historyGen++;
		c->moments.Free(); c->adaptiveList.Free(); c->adaptiveCount.Free(); c->reprojMoments.Free();
		return AGPT_OK;
	}
	if (c->momentsOn) return AGPT_OK;
	if (c->width > 0) {                      // (else agpt_set_film allocates them)
		int rcode = AllocMoments(c, (size_t)c->width * c->height);
		if (rcode != AGPT_OK) return rcode;
	}
	c->momentsOn = true;
	return AGPT_OK;
}

int agpt_read_moments(agpt_ctx* c, float* host) {
	JOIN(c);
	NEED(c != nullptr && host != nullptr, AGPT_ERR_INVALID, "null argument");
	NEED(c->momentsOn && c->moments.p != nullptr, AGPT_ERR_STATE, "moments are off (agpt_set_moments) or film not set");
	CU(cudaSetDevice(c->device));
	CU(cudaMemcpyAsync(host, c->moments.p, c->moments.Bytes(), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

int agpt_write_moments(agpt_ctx* c, const float* host) {
	JOIN(c);
	NEED(c != nullptr && host != nullptr, AGPT_ERR_INVALID, "null argument");
	NEED(c->momentsOn && c->moments.p != nullptr, AGPT_ERR_STATE, "moments are off (agpt_set_moments) or film not set");
	// k_generate<true> seeds a listed pixel's paths from (int)moments.w: every count must be one it can hold
	for (size_t i = 0; i < c->moments.n; i++) {
		const float w = host[4 * i + 3];
		NEED(w >= 0.f && w <= 16777216.f && w == std::floor(w), AGPT_ERR_INVALID, "agpt_write_moments: every .w must be an integer in [0, 2^24]");
	}
	CU(cudaSetDevice(c->device));
	CU(cudaMemcpyAsync(c->moments.p, host, c->moments.Bytes(), cudaMemcpyHostToDevice, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

static int CheckAdaptive(const agpt_adaptive* p) {
	NEED(p != nullptr, AGPT_ERR_INVALID, "null agpt_adaptive");
	NEED(p->min_samples >= 2 && p->min_samples <= p->max_samples && p->max_samples <= (1 << 24), AGPT_ERR_INVALID,
		"agpt_adaptive: need 2 <= min_samples <= max_samples <= 1<<24");
	NEED(p->step >= 1, AGPT_ERR_INVALID, "agpt_adaptive: step < 1");
	NEED(std::isfinite(p->tolerance) && p->tolerance >= 0.f && std::isfinite(p->floor) && p->floor >= 0.f, AGPT_ERR_INVALID,
		"agpt_adaptive: tolerance and floor must be finite and >= 0");
	return AGPT_OK;
}

// The convergence test over the film -> c->adaptiveList[0, *count) on the device, *count on the host.
static int SelectPixels(agpt_ctx* c, const agpt_adaptive& a, int* count) {
	const int wh = c->width * c->height;
	CU(cudaMemsetAsync(c->adaptiveCount.p, 0, sizeof(int), c->stream));
	k_adaptive_select<<<Blocks(wh, 256), 256, 0, c->stream>>>(c->accum, c->moments.p, c->width, c->height, a.max_samples, a.step, a.tolerance, a.floor,
		c->adaptiveList.p, c->adaptiveCount.p);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(count, c->adaptiveCount.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

int agpt_adaptive_select(agpt_ctx* c, const agpt_adaptive* params, int32_t* pixels_out, int* n_out) {
	JOIN(c);
	NEED(c != nullptr && n_out != nullptr, AGPT_ERR_INVALID, "null argument");
	int rcode = CheckAdaptive(params);
	if (rcode != AGPT_OK) return rcode;
	NEED(c->momentsOn && c->moments.p != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "moments are off (agpt_set_moments) or film not set");
	CU(cudaSetDevice(c->device));
	int n = 0;
	rcode = SelectPixels(c, *params, &n);
	if (rcode != AGPT_OK) return rcode;
	if (pixels_out && n > 0) {
		CU(cudaMemcpyAsync(pixels_out, c->adaptiveList.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
		CU(cudaStreamSynchronize(c->stream));
	}
	*n_out = n;
	return AGPT_OK;
}

// One adaptive round: samples [n_p, n_p + step) of the `count` pixels of c->adaptiveList, through the wave loop of agpt_render.
// A batch holds whole pixels (at most maxPathsPerBatch / step of them, at least one).
static int RenderListed(agpt_ctx* c, int count, int step, int maxSamples, int max_depth, int rr_depth_arg, uint32_t flags) {
	size_t perBatch = c->maxPathsPerBatch / (size_t)step;
	if (perBatch < 1) perBatch = 1;
	if (perBatch > (size_t)count) perBatch = (size_t)count;
	int rcode = EnsureCapacity(c, perBatch * step);
	if (rcode != AGPT_OK) return rcode;
	const Frame f = MakeFrame(c);
	CU(cudaEventRecord(c->evRender0, c->stream));
	for (int done = 0; done < count; done += (int)perBatch) {
		const int np = count - done < (int)perBatch ? count - done : (int)perBatch;
		GenParams g{};
		g.n = np * step; g.samples = step; g.list = c->adaptiveList.p; g.listBase = done; g.listCount = count; g.moments = c->moments.p; g.maxSamples = maxSamples;
		rcode = RunWaves(c, f, g, max_depth, rr_depth_arg, flags);
		if (rcode != AGPT_OK) return rcode;
		k_accumulate<true, true><<<Blocks(np, 256), 256, 0, c->stream>>>(f.ps.Lout, c->accum, c->width, c->height, step, c->moments.p, c->adaptiveList.p + done, np, maxSamples);
		CU(cudaGetLastError());
		c->stats.kernel_launches++;
	}
	CU(cudaEventRecord(c->evRender1, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	float ms = 0;
	cudaEventElapsedTime(&ms, c->evRender0, c->evRender1);
	c->stats.ms_render += ms;
	return AGPT_OK;
}

int agpt_render_adaptive(agpt_ctx* c, const agpt_adaptive* params, int max_depth, int rr_depth_arg, uint32_t flags, int* rounds_out, int64_t* paths_out) {
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	int rcode = CheckAdaptive(params);
	if (rcode != AGPT_OK) return rcode;
	NEED(max_depth >= 0, AGPT_ERR_INVALID, "bad depth");
	NEED(c->momentsOn, AGPT_ERR_STATE, "moments are off (agpt_set_moments)");
	rcode = CheckReady(c, true);
	if (rcode != AGPT_OK) return rcode;
	NEED(c->accum != nullptr && c->moments.p != nullptr, AGPT_ERR_STATE, "no accumulator");
	const agpt_adaptive a = *params;
	rcode = agpt_clear(c);                                  // film and moments
	if (rcode != AGPT_OK) return rcode;
	rcode = agpt_render(c, 0, a.min_samples, 1, max_depth, rr_depth_arg, flags);
	if (rcode != AGPT_OK) return rcode;
	int64_t paths = (int64_t)c->width * c->height * a.min_samples;
	int rounds = 0;
	while (true) {
		int n = 0;
		rcode = SelectPixels(c, a, &n);
		if (rcode != AGPT_OK) return rcode;
		if (n == 0) break;
		rcode = RenderListed(c, n, a.step, a.max_samples, max_depth, rr_depth_arg, flags);
		if (rcode != AGPT_OK) return rcode;
		rounds++;
		paths += (int64_t)n * a.step;
	}
	if (rounds_out) *rounds_out = rounds;
	if (paths_out) *paths_out = paths;
	return AGPT_OK;
}

int agpt_resolve_counts(agpt_ctx* c, uint32_t* host) {
	JOIN(c);
	NEED(c != nullptr && host != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "film not set");
	NEED(c->momentsOn && c->moments.p != nullptr, AGPT_ERR_STATE, "moments are off (agpt_set_moments)");
	CU(cudaSetDevice(c->device));
	int n = c->width * c->height;
	if (c->resolved.n != (size_t)n) CU(c->resolved.Alloc(n));
	k_resolve_counts<<<Blocks(n, 256), 256, 0, c->stream>>>(c->accum, c->moments.p, c->resolved.p, n);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(host, c->resolved.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

// ---- denoising (EXTENSION, agpt.h agpt_render_guides / agpt_denoise) ------------------------------------------------------
// The camera rays of samples [0, num_samples) as agpt_render generates them (k_generate<false>, tiled), batch by batch through
// the closest-hit trace alone; k_guides folds each batch into the guide sums.
int agpt_render_guides(agpt_ctx* c, int num_samples, uint32_t flags) {
	int rcode = CheckReady(c, true);
	if (rcode != AGPT_OK) return rcode;
	NEED(num_samples >= 1 && num_samples <= (1 << 24), AGPT_ERR_INVALID, "agpt_render_guides: need 1 <= num_samples <= 1<<24");
	CU(cudaSetDevice(c->device));
	const size_t wh = (size_t)c->width * c->height;
	const int perBatch = SamplesPerBatch(c, num_samples);
	rcode = EnsureCapacity(c, wh * perBatch);
	if (rcode != AGPT_OK) return rcode;
	c->guidesGen = 0;                                    // valid again only once this call has completed
	if (c->guideAlbedo.n != wh) { CU(c->guideAlbedo.Alloc(wh)); CU(c->guideNormal.Alloc(wh)); }
	const Frame f = MakeFrame(c);
	for (int done = 0; done < num_samples; done += perBatch) {
		const int ns = num_samples - done < perBatch ? num_samples - done : perBatch;
		const int n = (int)(wh * ns);
		GenParams g{};
		g.n = n; g.first_sample = done; g.sample_stride = 1; g.tiled = 1; g.samples = ns;
		rcode = Generate(c, f, g);
		if (rcode != AGPT_OK) return rcode;
		LaunchClosest(f.plan, flags, n, c->stream, f.sc, f.ps, f.q0.closest, f.q0.counts + 0, c->traceCounters.p, nullptr);
		LaunchGuides(f.plan, (int)wh, c->stream, f.sc, f.ps, ns, done == 0, done + ns == num_samples ? num_samples : 0, c->guideAlbedo.p, c->guideNormal.p);
		CU(cudaGetLastError());
		c->stats.kernel_launches += 2; c->stats.launches_closest++;
	}
	CU(cudaStreamSynchronize(c->stream));
	c->guidesGen = c->stateGen;
	return AGPT_OK;
}

static bool GuidesFresh(const agpt_ctx* c) {
	return c->guidesGen != 0 && c->guidesGen == c->stateGen && c->guideAlbedo.n == (size_t)c->width * c->height;
}

int agpt_read_guides(agpt_ctx* c, float* albedo_rgba, float* normal_depth_rgba) {
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	NEED(GuidesFresh(c), AGPT_ERR_STATE, "no guides for the current scene, camera and film (agpt_render_guides)");
	CU(cudaSetDevice(c->device));
	if (albedo_rgba) CU(cudaMemcpyAsync(albedo_rgba, c->guideAlbedo.p, c->guideAlbedo.Bytes(), cudaMemcpyDeviceToHost, c->stream));
	if (normal_depth_rgba) CU(cudaMemcpyAsync(normal_depth_rgba, c->guideNormal.p, c->guideNormal.Bytes(), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

static int CheckDenoise(const agpt_denoise_params* p) {
	NEED(p != nullptr, AGPT_ERR_INVALID, "null agpt_denoise");
	NEED(p->iterations >= 0 && p->iterations <= 10, AGPT_ERR_INVALID, "agpt_denoise: need 0 <= iterations <= 10");
	NEED(std::isfinite(p->sigma_luminance) && p->sigma_luminance >= 0.f && std::isfinite(p->sigma_depth) && p->sigma_depth >= 0.f, AGPT_ERR_INVALID,
		"agpt_denoise: sigmas must be finite and >= 0");
	NEED(p->normal_power_log2 >= 0 && p->normal_power_log2 <= 10, AGPT_ERR_INVALID, "agpt_denoise: need 0 <= normal_power_log2 <= 10");
	return AGPT_OK;
}

// k_denoise_prepare, then one k_denoise_atrous per iteration ping-ponging between denoiseE[0] and [1]; the last writes the
// remodulated floats and the packed pixels.
int agpt_denoise(agpt_ctx* c, const agpt_denoise_params* params, float* out_rgba, uint32_t* out_rgb8) {
	JOIN(c);
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	int rcode = CheckDenoise(params);
	if (rcode != AGPT_OK) return rcode;
	NEED(c->momentsOn && c->moments.p != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "moments are off (agpt_set_moments) or film not set");
	NEED(GuidesFresh(c), AGPT_ERR_STATE, "guides missing or stale: agpt_render_guides after the last agpt_set_film / agpt_set_camera / agpt_upload_*");
	const agpt_denoise_params p = *params;
	CU(cudaSetDevice(c->device));
	const int W = c->width, H = c->height, n = W * H;
	if (c->denoiseOut.n != (size_t)n) CU(c->denoiseOut.Alloc(n));
	if (c->resolved.n != (size_t)n) CU(c->resolved.Alloc(n));
	if (p.iterations > 0 && c->denoiseG.n != (size_t)n) { CU(c->denoiseE[0].Alloc(n)); CU(c->denoiseE[1].Alloc(n)); CU(c->denoiseG.Alloc(n)); }
	k_denoise_prepare<<<Blocks(n, 256), 256, 0, c->stream>>>(c->accum, c->moments.p, c->guideAlbedo.p, c->guideNormal.p, n, c->denoiseE[0].p, c->denoiseG.p,
		p.iterations == 0 ? c->denoiseOut.p : nullptr, c->resolved.p);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	const dim3 block(32, 8), grid(Blocks(W, 32), Blocks(H, 8));
	for (int i = 0; i < p.iterations; i++) {
		const float4* in = c->denoiseE[i & 1].p;
		if (i == p.iterations - 1)
			k_denoise_atrous<true><<<grid, block, 0, c->stream>>>(in, c->denoiseG.p, c->guideAlbedo.p, W, H, 1 << i, p.sigma_luminance, p.sigma_depth, p.normal_power_log2,
				c->denoiseOut.p, c->resolved.p);
		else
			k_denoise_atrous<false><<<grid, block, 0, c->stream>>>(in, c->denoiseG.p, c->guideAlbedo.p, W, H, 1 << i, p.sigma_luminance, p.sigma_depth, p.normal_power_log2,
				c->denoiseE[(i + 1) & 1].p, nullptr);
		CU(cudaGetLastError());
		c->stats.kernel_launches++;
	}
	if (out_rgba) CU(cudaMemcpyAsync(out_rgba, c->denoiseOut.p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
	if (out_rgb8) CU(cudaMemcpyAsync(out_rgb8, c->resolved.p, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

// ---- reprojection (EXTENSION, agpt.h agpt_reproject_film) -----------------------------------------------------------------------
static int CheckReproject(const agpt_reproject* p) {
	NEED(p != nullptr, AGPT_ERR_INVALID, "null agpt_reproject");
	NEED(p->max_history >= 1.f && p->max_history <= 16777216.f, AGPT_ERR_INVALID, "agpt_reproject: need 1 <= max_history <= 2^24");
	NEED(std::isfinite(p->sigma_depth) && p->sigma_depth > 0.f, AGPT_ERR_INVALID, "agpt_reproject: sigma_depth must be finite and > 0");
	NEED(p->min_normal_dot >= -1.f && p->min_normal_dot <= 1.f, AGPT_ERR_INVALID, "agpt_reproject: need -1 <= min_normal_dot <= 1");
	return AGPT_OK;
}

// One k_reproject_film: CARRY gathers film and moments from the saved view into reprojFilm / reprojMoments, which then replace
// them (the film by a copy, so that a caller-owned or exported film keeps its address); either way the current G goes into the
// other viewG buffer, which becomes the saved view.
int agpt_reproject_film(agpt_ctx* c, const agpt_reproject* params) {
	JOIN(c);
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	int rcode = CheckReproject(params);
	if (rcode != AGPT_OK) return rcode;
	NEED(c->momentsOn && c->moments.p != nullptr && c->accum != nullptr, AGPT_ERR_STATE, "moments are off (agpt_set_moments) or film not set");
	NEED(GuidesFresh(c), AGPT_ERR_STATE, "guides missing or stale: agpt_render_guides after the last agpt_set_film / agpt_set_camera / agpt_upload_*");
	const agpt_reproject p = *params;
	CU(cudaSetDevice(c->device));
	const int W = c->width, H = c->height;
	const size_t n = (size_t)W * H;
	const bool saved = c->viewGen != 0 && c->viewGen == c->historyGen && c->viewG[c->viewCur].n == n;
	// A static camera keeps film and moments as they are.  Recomputing the identity map in float rounds some pixel centres to
	// within an ulp of a pixel edge, and their bilinear weights would leak a tiny share of a neighbour into every static frame;
	// with this rule a static camera accumulates exactly as without reprojection.
	const bool carry = saved && memcmp(&c->viewCam, &c->cam, sizeof(agpt_camera)) != 0;
	const int next = c->viewCur ^ 1;
	if (c->viewG[next].n != n) CU(c->viewG[next].Alloc(n));
	if (carry && c->reprojFilm.n != n) CU(c->reprojFilm.Alloc(n));
	if (carry && c->reprojMoments.n != n) CU(c->reprojMoments.Alloc(n));     // (agpt_set_moments(0) frees it)
	const dim3 block(32, 8), grid(Blocks(W, 32), Blocks(H, 8));
	if (carry)
		k_reproject_film<true><<<grid, block, 0, c->stream>>>(c->accum, c->moments.p, c->viewG[c->viewCur].p, c->guideAlbedo.p, c->guideNormal.p, W, H,
			c->cam, c->viewCam, p.max_history, p.sigma_depth, p.min_normal_dot, c->reprojFilm.p, c->reprojMoments.p, c->viewG[next].p);
	else
		k_reproject_film<false><<<grid, block, 0, c->stream>>>(nullptr, nullptr, nullptr, c->guideAlbedo.p, c->guideNormal.p, W, H,
			c->cam, c->cam, p.max_history, p.sigma_depth, p.min_normal_dot, nullptr, nullptr, c->viewG[next].p);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	if (carry) {
		CU(cudaMemcpyAsync(c->accum, c->reprojFilm.p, n * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
		std::swap(c->moments, c->reprojMoments);
	}
	CU(cudaStreamSynchronize(c->stream));
	c->viewCur = next;
	c->viewCam = c->cam;
	c->viewGen = c->historyGen;
	return AGPT_OK;
}

// The g.n rays k_generate makes from g, traced into a hit table on the host
static int TraceTable(agpt_ctx* c, const Frame& f, const GenParams& g, int any_hit, uint32_t flags, agpt_hit* out_host) {
	const int n = g.n;
	int rcode = Generate(c, f, g);
	if (rcode != AGPT_OK) return rcode;
	DevBuf<agpt_hit> out;
	CU(out.Alloc(n));
	LaunchTable(f.plan, flags, any_hit != 0, c->stream, f.sc, f.ps.rayO, f.ps.rayD, n, out.p, c->traceCounters.p + (any_hit ? AGPT_WAVE_COUNTERS : 0));
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(out_host, out.p, (size_t)n * sizeof(agpt_hit), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

// A rays7 table (O, D, tmax per ray) on the device with an RNG seed per ray, the caller's or zeros; g names them.
struct RayTable {
	DevBuf<float> rays;
	DevBuf<uint32_t> seeds;
};
static int UploadRays(agpt_ctx* c, RayTable& t, int n, const float* rays7, const uint32_t* seeds, uint32_t flags, GenParams& g) {
	CU(t.rays.Upload(rays7, 7 * (size_t)n, c->stream));
	if (seeds) CU(t.seeds.Upload(seeds, (size_t)n, c->stream));
	else { CU(t.seeds.Alloc((size_t)n)); CU(cudaMemsetAsync(t.seeds.p, 0, t.seeds.Bytes(), c->stream)); }
	g.n = n; g.rays7 = t.rays.p; g.seeds = t.seeds.p; g.raysFinal = (flags & AGPT_FLAG_RAYS_FINAL) ? 1 : 0;
	return AGPT_OK;
}

int agpt_trace_primary(agpt_ctx* c, int sample, uint32_t flags, agpt_hit* out_host) {
	int rcode = CheckReady(c, true);
	if (rcode != AGPT_OK) return rcode;
	NEED(out_host != nullptr, AGPT_ERR_INVALID, "null output");
	CU(cudaSetDevice(c->device));
	const size_t wh = (size_t)c->width * c->height;
	rcode = EnsureCapacity(c, wh);
	if (rcode != AGPT_OK) return rcode;
	GenParams g{};
	g.n = (int)wh; g.first_sample = sample; g.sample_stride = 1;
	return TraceTable(c, MakeFrame(c), g, 0, flags, out_host);
}

int agpt_trace_rays(agpt_ctx* c, int64_t n, const float* rays7, int any_hit, uint32_t flags, agpt_hit* out_host) {
	int rcode = CheckReady(c, false);
	if (rcode != AGPT_OK) return rcode;
	NEED(n >= 0 && n < (1ll << 30) && (n == 0 || (rays7 && out_host)), AGPT_ERR_INVALID, "bad ray table");
	if (n == 0) return AGPT_OK;
	CU(cudaSetDevice(c->device));
	// same normalisation as the Ray constructor, done on the device by k_generate
	rcode = EnsureCapacity(c, (size_t)n);
	if (rcode != AGPT_OK) return rcode;
	RayTable t;
	GenParams g{};
	rcode = UploadRays(c, t, (int)n, rays7, nullptr, flags, g);
	if (rcode != AGPT_OK) return rcode;
	return TraceTable(c, MakeFrame(c), g, any_hit, flags, out_host);
}

static int LiGeneric(agpt_ctx* c, GenParams g, int max_depth, int rr_depth_arg, uint32_t flags, float* out_rgb) {
	int n = g.n;
	int rcode = EnsureCapacity(c, (size_t)n);
	if (rcode != AGPT_OK) return rcode;
	const Frame f = MakeFrame(c);
	rcode = RunWaves(c, f, g, max_depth, rr_depth_arg, flags & AGPT_FLAG_RR_BY_BOUNCE);
	if (rcode != AGPT_OK) return rcode;
	std::vector<float4> host(n);
	CU(cudaMemcpyAsync(host.data(), f.ps.Lout, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	for (int i = 0; i < n; i++) { out_rgb[3 * i] = host[i].x; out_rgb[3 * i + 1] = host[i].y; out_rgb[3 * i + 2] = host[i].z; }
	return AGPT_OK;
}

int agpt_li_pixels(agpt_ctx* c, int n, const int* xs, const int* ys, const int* ss, int max_depth, int rr_depth_arg, uint32_t flags, float* out_rgb) {
	int rcode = CheckReady(c, true);
	if (rcode != AGPT_OK) return rcode;
	NEED(n >= 0 && (n == 0 || (xs && ys && ss && out_rgb)), AGPT_ERR_INVALID, "bad pixel list");
	if (n == 0) return AGPT_OK;
	CU(cudaSetDevice(c->device));
	DevBuf<int> dx, dy, ds;
	CU(dx.Upload(xs, n, c->stream)); CU(dy.Upload(ys, n, c->stream)); CU(ds.Upload(ss, n, c->stream));
	GenParams g{};
	g.n = n; g.xs = dx.p; g.ys = dy.p; g.ss = ds.p;
	return LiGeneric(c, g, max_depth, rr_depth_arg, flags, out_rgb);
}

int agpt_li_rays(agpt_ctx* c, int n, const float* rays7, const uint32_t* rng_states, int max_depth, int rr_depth_arg, uint32_t flags, float* out_rgb) {
	int rcode = CheckReady(c, false);
	if (rcode != AGPT_OK) return rcode;
	NEED(n >= 0 && (n == 0 || (rays7 && rng_states && out_rgb)), AGPT_ERR_INVALID, "bad ray list");
	if (n == 0) return AGPT_OK;
	CU(cudaSetDevice(c->device));
	RayTable t;
	GenParams g{};
	rcode = UploadRays(c, t, n, rays7, rng_states, flags, g);
	if (rcode != AGPT_OK) return rcode;
	return LiGeneric(c, g, max_depth, rr_depth_arg, flags, out_rgb);
}

// ---- multi-GPU: sample-index sharding (SURVEY 8e) ---------------------------------------------
// One context per GPU, every context holds the whole scene; GPU g renders s = first + g, first + g + G, ...
static int CheckGroup(agpt_ctx** ctxs, int n) {
	for (int g = 0; ctxs != nullptr && g < n; g++) JOIN(ctxs[g]);
	NEED(ctxs != nullptr && n >= 1 && n <= AGPT_MAX_PEERS, AGPT_ERR_INVALID, "bad context list (1.." + std::to_string(AGPT_MAX_PEERS) + " contexts)");
	for (int g = 0; g < n; g++) {
		NEED(ctxs[g] != nullptr && ctxs[g]->accum != nullptr, AGPT_ERR_STATE, "context " + std::to_string(g) + ": film not set");
		NEED(ctxs[g]->width == ctxs[0]->width && ctxs[g]->height == ctxs[0]->height, AGPT_ERR_INVALID, "contexts have different film sizes");
		for (int h = 0; h < g; h++) NEED(ctxs[h] != ctxs[g] && ctxs[h]->device != ctxs[g]->device, AGPT_ERR_INVALID, "two contexts on one GPU");
	}
	return AGPT_OK;
}

// Peer access between every pair of the group's GPUs; *all = false if some pair has none.
static int EnablePeerAccess(agpt_ctx** ctxs, int n, bool* all) {
	*all = true;
	for (int a = 0; a < n; a++)
		for (int b = 0; b < n; b++) {
			if (a == b) continue;
			int can = 0;
			CU(cudaDeviceCanAccessPeer(&can, ctxs[a]->device, ctxs[b]->device));
			if (!can) { *all = false; continue; }
			CU(cudaSetDevice(ctxs[a]->device));
			cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[b]->device, 0);
			if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
			else if (e != cudaSuccess) return Fail(AGPT_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
		}
	return AGPT_OK;
}

static int SyncGroup(agpt_ctx** ctxs, int n) {
	for (int g = 0; g < n; g++) { CU(cudaSetDevice(ctxs[g]->device)); CU(cudaStreamSynchronize(ctxs[g]->stream)); }
	return AGPT_OK;
}

static NcclApi g_nccl;
static std::vector<int> g_ncclDevices;
static std::vector<agpt_ncclComm_t> g_ncclComms;

static int NcclAllReduce(agpt_ctx** ctxs, int n) {
	NEED(g_nccl.Load(), AGPT_ERR_STATE, g_nccl.error);
	std::vector<int> devs(n);
	for (int g = 0; g < n; g++) devs[g] = ctxs[g]->device;
	if (devs != g_ncclDevices) {
		for (auto cm : g_ncclComms) g_nccl.CommDestroy(cm);
		g_ncclComms.assign(n, nullptr);
		int r = g_nccl.CommInitAll(g_ncclComms.data(), n, devs.data());
		if (r != 0) { g_ncclComms.clear(); g_ncclDevices.clear(); return Fail(AGPT_ERR_CUDA, std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(r)); }
		g_ncclDevices = devs;
	}
	const size_t count = 4 * (size_t)ctxs[0]->width * ctxs[0]->height;
	int r = g_nccl.GroupStart();
	for (int g = 0; g < n && r == 0; g++) {
		CU(cudaSetDevice(ctxs[g]->device));
		r = g_nccl.AllReduce(ctxs[g]->accum, ctxs[g]->accum, count, /*ncclFloat*/ 7, /*ncclSum*/ 0, g_ncclComms[g], ctxs[g]->stream);
	}
	int r2 = g_nccl.GroupEnd();
	if (r != 0 || r2 != 0) return Fail(AGPT_ERR_CUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(r != 0 ? r : r2));
	return AGPT_OK;
}

static bool WantNccl() { const char* e = getenv("AGPT_REDUCE"); return e && std::string(e) == "nccl"; }

static void SliceOf(int g, int n, size_t wh, int* first, int* count) {
	size_t a = wh * (size_t)g / n, b = wh * (size_t)(g + 1) / n;
	*first = (int)a; *count = (int)(b - a);
}

int agpt_reduce_accum(agpt_ctx** ctxs, int n, int root) {
	int rcode = CheckGroup(ctxs, n);
	if (rcode != AGPT_OK) return rcode;
	NEED(root >= -1 && root < n, AGPT_ERR_INVALID, "bad root");
	if (n == 1) return AGPT_OK;
	bool peers = false;
	rcode = EnablePeerAccess(ctxs, n, &peers);
	if (rcode != AGPT_OK) return rcode;
	rcode = SyncGroup(ctxs, n);                    // every render has landed before any accumulator is read
	if (rcode != AGPT_OK) return rcode;
	const size_t wh = (size_t)ctxs[0]->width * ctxs[0]->height;
	for (int g = 0; g < n; g++) { CU(cudaSetDevice(ctxs[g]->device)); CU(cudaEventRecord(ctxs[g]->evRender0, ctxs[g]->stream)); }
	int path = 1;
	if (!peers || WantNccl()) {
		path = 2;
		rcode = NcclAllReduce(ctxs, n);
		if (rcode != AGPT_OK) return rcode;
	}
	else {
		PeerAccums pa;
		pa.n = n;
		for (int g = 0; g < n; g++) pa.p[g] = ctxs[g]->accum;
		for (int g = 0; g < n; g++) {
			if (root >= 0 && g != root) continue;
			int first = 0, count = (int)wh;
			if (root < 0) SliceOf(g, n, wh, &first, &count);
			CU(cudaSetDevice(ctxs[g]->device));
			if (root < 0) k_allreduce_slice<<<Blocks(count, 256), 256, 0, ctxs[g]->stream>>>(pa, first, count);
			else k_reduce_resolve<<<Blocks(count, 256), 256, 0, ctxs[g]->stream>>>(pa, first, count, 1.f, ctxs[g]->accum, nullptr);
			CU(cudaGetLastError());
			ctxs[g]->stats.kernel_launches++;
		}
	}
	for (int g = 0; g < n; g++) { CU(cudaSetDevice(ctxs[g]->device)); CU(cudaEventRecord(ctxs[g]->evRender1, ctxs[g]->stream)); }
	rcode = SyncGroup(ctxs, n);
	if (rcode != AGPT_OK) return rcode;
	for (int g = 0; g < n; g++) {
		float ms = 0;
		cudaEventElapsedTime(&ms, ctxs[g]->evRender0, ctxs[g]->evRender1);
		ctxs[g]->stats.ms_reduce += ms; ctxs[g]->stats.reduce_path = (uint32_t)path;
	}
	return AGPT_OK;
}

int agpt_allreduce_accum(agpt_ctx** ctxs, int n) { return agpt_reduce_accum(ctxs, n, -1); }

// Fused reduce + CopyToSurface: GPU g sums ITS slice of the film over all accumulators (rank order, peer
// loads) and packs it; the G slices go to the host over G PCIe links at once.  keep_sum != 0 also leaves
// the summed film in ctxs[0]'s accumulator (slices written there by peer stores).
int agpt_reduce_resolve(agpt_ctx** ctxs, int n, int samples, int keep_sum, uint32_t* host_rgb8) {
	int rcode = CheckGroup(ctxs, n);
	if (rcode != AGPT_OK) return rcode;
	NEED(samples > 0 && host_rgb8 != nullptr, AGPT_ERR_INVALID, "samples <= 0 or null output");
	bool peers = n == 1;
	if (n > 1) { rcode = EnablePeerAccess(ctxs, n, &peers); if (rcode != AGPT_OK) return rcode; }
	if (!peers || (n > 1 && WantNccl())) {
		// no peer memory between some pair: NCCL all-reduce, then the single-GPU resolve
		rcode = agpt_reduce_accum(ctxs, n, -1);
		if (rcode != AGPT_OK) return rcode;
		return agpt_resolve(ctxs[0], samples, host_rgb8);
	}
	rcode = SyncGroup(ctxs, n);
	if (rcode != AGPT_OK) return rcode;
	const size_t wh = (size_t)ctxs[0]->width * ctxs[0]->height;
	PeerAccums pa;
	pa.n = n;
	for (int g = 0; g < n; g++) pa.p[g] = ctxs[g]->accum;
	for (int g = 0; g < n; g++) {
		agpt_ctx* c = ctxs[g];
		int first, count;
		SliceOf(g, n, wh, &first, &count);
		CU(cudaSetDevice(c->device));
		if (c->resolved.n != wh) CU(c->resolved.Alloc(wh));
		CU(cudaEventRecord(c->evRender0, c->stream));
		// (the sum may be written over ctxs[0]'s own addend: pixel i is read and written by this one thread only)
		k_reduce_resolve<<<Blocks(count, 256), 256, 0, c->stream>>>(pa, first, count, (float)samples, keep_sum ? ctxs[0]->accum : nullptr, c->resolved.p);
		CU(cudaGetLastError());
		c->stats.kernel_launches++;
		CU(cudaEventRecord(c->evRender1, c->stream));
		CU(cudaMemcpyAsync(host_rgb8 + first, c->resolved.p + first, (size_t)count * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	}
	rcode = SyncGroup(ctxs, n);
	if (rcode != AGPT_OK) return rcode;
	for (int g = 0; g < n; g++) {
		float ms = 0;
		cudaEventElapsedTime(&ms, ctxs[g]->evRender0, ctxs[g]->evRender1);
		ctxs[g]->stats.ms_reduce += ms; ctxs[g]->stats.reduce_path = 1;
	}
	return AGPT_OK;
}

// num_samples Tick bodies split over the group: context g renders first_sample + g, + g + n, ... (one host
// thread per GPU: agpt_render paces its waves from the host).
int agpt_render_multi(agpt_ctx** ctxs, int n, int first_sample, int num_samples, int max_depth, int rr_depth_arg, uint32_t flags) {
	int rcode = CheckGroup(ctxs, n);
	if (rcode != AGPT_OK) return rcode;
	NEED(num_samples >= 0, AGPT_ERR_INVALID, "bad sample range");
	std::vector<int> rc((size_t)n, AGPT_OK);
	std::vector<std::string> msg((size_t)n);
	std::vector<std::thread> pool;
	for (int g = 0; g < n; g++) {
		int count = num_samples > g ? (num_samples - g + n - 1) / n : 0;
		pool.emplace_back([=, &rc, &msg] {
			if (count > 0) rc[g] = agpt_render(ctxs[g], first_sample + g, count, n, max_depth, rr_depth_arg, flags);
			if (rc[g] != AGPT_OK) msg[g] = g_error;         // (thread-local message of the worker)
		});
	}
	for (auto& t : pool) t.join();
	for (int g = 0; g < n; g++) if (rc[g] != AGPT_OK) return Fail(rc[g], "GPU " + std::to_string(ctxs[g]->device) + ": " + msg[g]);
	return AGPT_OK;
}

// ---- multi-process sharding (one rank per GPU: torchrun, MPI): peers' accumulators through CUDA IPC ----
int agpt_accum_ipc_handle(agpt_ctx* c, void* handle64) {
	JOIN(c);
	NEED(c != nullptr && handle64 != nullptr, AGPT_ERR_INVALID, "null argument");
	NEED(c->accum != nullptr && c->accum == c->accumOwn.p, AGPT_ERR_STATE, "the context must own its accumulator (agpt_set_film, no agpt_set_accum_dev)");
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
	CU(cudaSetDevice(c->device));
	cudaIpcMemHandle_t h;
	CU(cudaIpcGetMemHandle(&h, c->accumOwn.p));
	memcpy(handle64, &h, sizeof(h));
	return AGPT_OK;
}

int agpt_close_peer_accums(agpt_ctx* c) {
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	for (int r = 0; r < c->peerWorld; r++) if (r != c->peerRank && c->peerAccum[r]) cudaIpcCloseMemHandle(c->peerAccum[r]);
	memset(c->peerAccum, 0, sizeof(c->peerAccum));
	c->peerWorld = 0; c->peerRank = -1;
	return AGPT_OK;
}

int agpt_open_peer_accums(agpt_ctx* c, int rank, int world, const void* handles64) {
	JOIN(c);
	NEED(c != nullptr && handles64 != nullptr && world >= 1 && world <= AGPT_MAX_PEERS && rank >= 0 && rank < world, AGPT_ERR_INVALID, "bad rank / world / handles");
	NEED(c->accum != nullptr, AGPT_ERR_STATE, "film not set");
	int rcode = agpt_close_peer_accums(c);
	if (rcode != AGPT_OK) return rcode;
	for (int r = 0; r < world; r++) {
		if (r == rank) { c->peerAccum[r] = c->accum; continue; }
		cudaIpcMemHandle_t h;
		memcpy(&h, (const char*)handles64 + 64 * (size_t)r, sizeof(h));
		void* p = nullptr;
		cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
		if (e != cudaSuccess) { c->peerWorld = r; c->peerRank = rank; agpt_close_peer_accums(c); return Fail(AGPT_ERR_CUDA, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(r) + "): " + cudaGetErrorString(e)); }
		c->peerAccum[r] = (float4*)p;
	}
	c->peerRank = rank; c->peerWorld = world;
	return AGPT_OK;
}

static int PeerTable(agpt_ctx* c, PeerAccums* pa) {
	NEED(c != nullptr && c->peerWorld >= 1, AGPT_ERR_STATE, "peer accumulators not open (agpt_open_peer_accums)");
	pa->n = c->peerWorld;
	for (int r = 0; r < c->peerWorld; r++) pa->p[r] = c->peerAccum[r];
	pa->p[c->peerRank] = c->accum;
	return AGPT_OK;
}

// This rank's slice of the all-reduce.  The CALLER provides the two barriers: every rank has finished
// rendering before any rank calls, and no rank reads its accumulator before every rank has returned.
int agpt_allreduce_accum_peers(agpt_ctx* c) {
	JOIN(c);
	PeerAccums pa;
	int rcode = PeerTable(c, &pa);
	if (rcode != AGPT_OK) return rcode;
	CU(cudaSetDevice(c->device));
	int first, count;
	SliceOf(c->peerRank, c->peerWorld, (size_t)c->width * c->height, &first, &count);
	CU(cudaEventRecord(c->evRender0, c->stream));
	k_allreduce_slice<<<Blocks(count, 256), 256, 0, c->stream>>>(pa, first, count);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaEventRecord(c->evRender1, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	float ms = 0;
	cudaEventElapsedTime(&ms, c->evRender0, c->evRender1);
	c->stats.ms_reduce += ms; c->stats.reduce_path = 1;
	return AGPT_OK;
}

// The whole film on this rank (the root): sum of all ranks' accumulators in rank order -> packed pixels on the
// host; keep_sum != 0 also stores the sum in this rank's accumulator.  Reads the peers, writes none of them:
// only the barrier BEFORE the call is needed.
int agpt_reduce_resolve_peers(agpt_ctx* c, int samples, int keep_sum, uint32_t* host_rgb8) {
	JOIN(c);
	PeerAccums pa;
	int rcode = PeerTable(c, &pa);
	if (rcode != AGPT_OK) return rcode;
	NEED(samples > 0 && host_rgb8 != nullptr, AGPT_ERR_INVALID, "samples <= 0 or null output");
	CU(cudaSetDevice(c->device));
	const size_t wh = (size_t)c->width * c->height;
	if (c->resolved.n != wh) CU(c->resolved.Alloc(wh));
	CU(cudaEventRecord(c->evRender0, c->stream));
	k_reduce_resolve<<<Blocks(wh, 256), 256, 0, c->stream>>>(pa, 0, (int)wh, (float)samples, keep_sum ? c->accum : nullptr, c->resolved.p);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaEventRecord(c->evRender1, c->stream));
	CU(cudaMemcpyAsync(host_rgb8, c->resolved.p, wh * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	float ms = 0;
	cudaEventElapsedTime(&ms, c->evRender0, c->evRender1);
	c->stats.ms_reduce += ms; c->stats.reduce_path = 1;
	return AGPT_OK;
}

// ---- pinned host memory for accumulators (fast H2D/D2H of the float4 film) --------------------
int agpt_host_alloc(size_t bytes, void** out) {
	NEED(out != nullptr && bytes > 0, AGPT_ERR_INVALID, "bad allocation request");
	*out = nullptr;
	CU(cudaMallocHost(out, bytes));
	return AGPT_OK;
}
int agpt_host_free(void* p) {
	if (p) CU(cudaFreeHost(p));
	return AGPT_OK;
}

// ---- observability -----------------------------------------------------------------------
int agpt_get_stats(agpt_ctx* c, agpt_stats* out) {
	NEED(c != nullptr && out != nullptr, AGPT_ERR_INVALID, "null argument");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	unsigned long long tc[2 * AGPT_WAVE_COUNTERS];
	RayCounters rc;
	CU(cudaMemcpy(tc, c->traceCounters.p, sizeof(tc), cudaMemcpyDeviceToHost));
	CU(cudaMemcpy(&rc, c->rayCounters.p, sizeof(rc), cudaMemcpyDeviceToHost));
	*out = c->stats;
	for (int k = 0; k < 2; k++) {
		const unsigned long long* t = tc + AGPT_WAVE_COUNTERS * k;
		out->node_visits[k] = t[1]; out->box_tests[k] = t[2]; out->tri_tests[k] = t[3]; out->analytic_tests[k] = t[4];
		out->warp_steps[k] = t[5]; out->lane_steps[k] = t[6];
	}
	out->rays_closest += rc.rays_closest; out->rays_shadow = rc.rays_shadow; out->rays_mis = rc.rays_mis; out->rays_skip = rc.rays_skip; out->rays_mis_culled = rc.rays_mis_culled; out->rays_tail_culled = rc.rays_tail_culled;
	out->ms_other = out->ms_render - out->ms_trace_closest - out->ms_trace_any - out->ms_shade;
	return AGPT_OK;
}
int agpt_get_wave_stats(agpt_ctx* c, int kind, agpt_wave_stats* out, int max_waves, int* n_waves) {
	NEED(c != nullptr && out != nullptr && n_waves != nullptr && (kind == 0 || kind == 1) && max_waves >= 1, AGPT_ERR_INVALID, "bad argument");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	std::vector<unsigned long long> rows((size_t)AGPT_MAX_WAVE_ROWS * AGPT_WAVE_COUNTERS);
	CU(cudaMemcpy(rows.data(), c->traceCounters.p + 2 * AGPT_WAVE_COUNTERS + (size_t)kind * AGPT_MAX_WAVE_ROWS * AGPT_WAVE_COUNTERS, rows.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
	int n = 0;
	for (int w = 0; w < AGPT_MAX_WAVE_ROWS && w < max_waves; w++) {
		const unsigned long long* r = &rows[(size_t)w * AGPT_WAVE_COUNTERS];
		out[w].rays = r[0]; out[w].node_visits = r[1]; out[w].box_tests = r[2]; out[w].tri_tests = r[3]; out[w].analytic_tests = r[4];
		out[w].warp_steps = r[5]; out[w].lane_steps = r[6]; out[w].reserved = 0;
		if (r[0]) n = w + 1;
	}
	*n_waves = n;
	return AGPT_OK;
}

int agpt_probe_bandwidth(agpt_ctx* c, size_t bytes, int iters, float* gbs_out) {
	NEED(c != nullptr && gbs_out != nullptr && bytes >= 4096 && iters >= 1, AGPT_ERR_INVALID, "bad probe arguments");
	CU(cudaSetDevice(c->device));
	DevBuf<uint4> buf;
	DevBuf<unsigned> sink;
	const size_t n16 = bytes / 16;
	CU(buf.Alloc(n16)); CU(sink.Alloc(1));
	CU(cudaMemsetAsync(buf.p, 0, n16 * 16, c->stream));
	const int blocks = c->smCount * 4;
	k_probe_bandwidth<<<blocks, 512, 0, c->stream>>>(buf.p, n16, 1, sink.p);          // warm-up: page in, fill L2
	CU(cudaEventRecord(c->evA, c->stream));
	k_probe_bandwidth<<<blocks, 512, 0, c->stream>>>(buf.p, n16, iters, sink.p);
	CU(cudaEventRecord(c->evB, c->stream));
	CU(cudaGetLastError());
	c->stats.kernel_launches += 2;
	CU(cudaStreamSynchronize(c->stream));
	float ms = 0;
	cudaEventElapsedTime(&ms, c->evA, c->evB);
	*gbs_out = ms > 0 ? (float)((double)n16 * 16 * iters / (ms * 1e-3) / 1e9) : 0.f;
	return AGPT_OK;
}

int agpt_debug_status(agpt_ctx* c, uint64_t* out4) {
	NEED(c != nullptr && out4 != nullptr, AGPT_ERR_INVALID, "null argument");
	out4[0] = out4[1] = out4[2] = out4[3] = 0;
#ifdef AGPT_DEBUG
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	unsigned long long v[4];
	CU(cudaMemcpyFromSymbol(v, g_agptDebug, sizeof(v)));
	for (int k = 0; k < 4; k++) out4[k] = v[k];
#endif
	return AGPT_OK;
}
int agpt_reset_stats(agpt_ctx* c) {
	NEED(c != nullptr, AGPT_ERR_INVALID, "null context");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	memset(&c->stats, 0, sizeof(c->stats));
	CU(cudaMemset(c->traceCounters.p, 0, c->traceCounters.Bytes()));
	CU(cudaMemset(c->rayCounters.p, 0, c->rayCounters.Bytes()));
	return AGPT_OK;
}

} // extern "C"

// ---- per-function probes -------------------------------------------------------------------
__global__ void k_probe_bounds(int n, const float* boxes6, const float* rays7, int* out_hit, float* out_t) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float* b = boxes6 + 6 * i;
	const float* r = rays7 + 7 * i;
	float t = 0;
	bool h = BoundsIntersect(f3(b[0], b[1], b[2]), f3(b[3], b[4], b[5]), f3(r[0], r[1], r[2]), f3(r[3], r[4], r[5]), r[6], t);
	out_hit[i] = h ? 1 : 0;
	out_t[i] = h ? t : 0.f;
}

// BSDF::f / Pdf / Sample_f through the SAME functions k_shade_b runs (VertexBsdfInit, EvalLobes,
// FinishEval, SampleLobeDir, FinishSample), against golden vectors of the reference's own methods.
__global__ void k_probe_bsdf(int n, agpt_material mat, const float* in14, int skipSpecular, float* out12) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float* a = in14 + 14 * i;
	float3 dpdu = f3(a[0], a[1], a[2]), dpdv = f3(a[3], a[4], a[5]), wo = f3(a[6], a[7], a[8]), wi = f3(a[9], a[10], a[11]);
	float2 u = make_float2(a[12], a[13]);
	DSurface si;
	SurfaceInit(si, f3(0.f), dpdu, dpdv);
	VertexBsdf vb;
	VertexBsdfInit<true>(vb, si, &mat, wo);
	float* o = out12 + 12 * i;
	// f(wo, wi) and Pdf(wo, wi): zero when wo.z == 0 (reflection.h:117,178)
	float3 f = f3(0.f);
	float pdf = 0.f;
	LobeEval ev;
	if (vb.woOk) {
		EvalLobes<true>(vb, WorldToLocal(vb.b, wi), ev);
		f = FinishEval<true>(vb, ev, wi, &pdf);
	}
	o[0] = f.x; o[1] = f.y; o[2] = f.z; o[3] = pdf;
	// Sample_f(wo, &wi, u, &pdf, skipSpecular, &sampledSpecular)
	DirSample smp;
	SampleLobeDir<true>(vb, u, skipSpecular != 0, smp);
	float3 wis = f3(0.f), fs = f3(0.f);
	float pdfs = 0.f;
	if (smp.ok) {
		ev.f = f3(0.f); ev.pdfCos = 0.f; ev.pdfMicro = 0.f; ev.fT = f3(0.f); ev.pdfT = 0.f;
		if (smp.lobe != AGPT_LOBE_SPECULAR) EvalLobes<true>(vb, smp.wi, ev);
		wis = LocalToWorld(vb.b, smp.wi);
		fs = FinishSample<true>(vb, smp, ev, wis, &pdfs);
	}
	bool spec = vb.woOk && smp.matching > 0 && smp.lobe == AGPT_LOBE_SPECULAR;
	o[4] = wis.x; o[5] = wis.y; o[6] = wis.z; o[7] = fs.x; o[8] = fs.y; o[9] = fs.z; o[10] = pdfs; o[11] = spec ? 1.f : 0.f;
}

__global__ void k_probe_sphere_sample(int n, const float* in9, float* out8) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float* a = in9 + 9 * i;
	agpt_sphere s;
	s.center[0] = a[0]; s.center[1] = a[1]; s.center[2] = a[2]; s.r = a[3]; s.r2 = a[3] * a[3];
	float3 p, nn;
	float pdf = 0;
	SphereSampleFrom(s, f3(a[4], a[5], a[6]), make_float2(a[7], a[8]), &p, &nn, &pdf);
	float* o = out8 + 8 * i;
	o[0] = p.x; o[1] = p.y; o[2] = p.z; o[3] = nn.x; o[4] = nn.y; o[5] = nn.z; o[6] = pdf;
	o[7] = SpherePdfFrom(s, f3(a[4], a[5], a[6]));
}

// EXTENSION: Sample_Li / Pdf_Li of one sampled plane / mesh light through the same functions k_shade_b runs.  No early
// return: the mesh walk of Pdf_Li votes with the whole warp.
__global__ void __launch_bounds__(128) k_probe_light_sample(DScene sc, DShapeTables st, int light, int n, const float* in8, float* out8) {
	__shared__ unsigned stack[AGPT_SHADE_STACK_SMEM * 128];
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	const bool lane = i < n;
	const float* a = in8 + 8 * (lane ? i : 0);
	const float3 refP = f3(a[0], a[1], a[2]);
	float3 p = f3(0.f), nn = f3(0.f);
	float pdf = 0.f;
	if (lane) ShapeSampleFrom(sc, st, light, sc.prims[sc.lights[light].prim], refP, make_float2(a[3], a[4]), &p, &nn, &pdf);
	const float pdfLi = ShapePdfLi<AGPT_SHADE_STACK_SMEM>(sc, st, light, refP, f3(a[5], a[6], a[7]), stack + threadIdx.x, 128, lane);
	if (lane) {
		float* o = out8 + 8 * i;
		o[0] = p.x; o[1] = p.y; o[2] = p.z; o[3] = pdf; o[4] = pdfLi; o[5] = nn.x; o[6] = nn.y; o[7] = nn.z;
	}
}

__global__ void k_probe_stream(uint32_t pixel, uint32_t sample, int k, float* out) {
	uint32_t s = StreamSeed(pixel, sample);
	for (int i = 0; i < k; i++) out[i] = RandomFloat(s);
}

template <typename TIn, typename TOut, typename Launch>
static int ProbeRun(agpt_ctx* c, const TIn* in, size_t nIn, TOut* out, size_t nOut, Launch launch) {
	DevBuf<TIn> din;
	DevBuf<TOut> dout;
	CU(din.Upload(in, nIn, c->stream));
	CU(dout.Alloc(nOut));
	launch(din.p, dout.p);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(out, dout.p, nOut * sizeof(TOut), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

extern "C" {

int agpt_probe_bounds(agpt_ctx* c, int n, const float* boxes6, const float* rays7, int* out_hit, float* out_t) {
	NEED(c != nullptr && n > 0 && boxes6 && rays7 && out_hit && out_t, AGPT_ERR_INVALID, "bad probe arguments");
	CU(cudaSetDevice(c->device));
	DevBuf<float> db, dr, dt;
	DevBuf<int> dh;
	CU(db.Upload(boxes6, 6 * (size_t)n, c->stream)); CU(dr.Upload(rays7, 7 * (size_t)n, c->stream));
	CU(dh.Alloc(n)); CU(dt.Alloc(n));
	k_probe_bounds<<<Blocks(n, 128), 128, 0, c->stream>>>(n, db.p, dr.p, dh.p, dt.p);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(out_hit, dh.p, n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(out_t, dt.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

int agpt_probe_bsdf(agpt_ctx* c, int n, const agpt_material* mat, const float* in14, int skip_specular, float* out12) {
	NEED(c != nullptr && n > 0 && mat && in14 && out12, AGPT_ERR_INVALID, "bad probe arguments");
	CU(cudaSetDevice(c->device));
	agpt_material m = *mat;
	return ProbeRun(c, in14, 14 * (size_t)n, out12, 12 * (size_t)n, [&](const float* din, float* dout) {
		k_probe_bsdf<<<Blocks(n, 128), 128, 0, c->stream>>>(n, m, din, skip_specular, dout);
	});
}

// EXTENSION (agpt.h agpt_probe_material_maps): the rays are traced as agpt_trace_rays traces them (k_generate<false>, closest hit)
int agpt_probe_material_maps(agpt_ctx* c, int n, const float* rays7, float* out32) {
	NEED(c != nullptr && n > 0 && rays7 && out32, AGPT_ERR_INVALID, "bad probe arguments");
	int rcode = CheckReady(c, false);
	if (rcode != AGPT_OK) return rcode;
	NEED(c->hasMaps, AGPT_ERR_STATE, "agpt_probe_material_maps: no material has a roughness-metallic or normal map");
	CU(cudaSetDevice(c->device));
	rcode = EnsureCapacity(c, (size_t)n);
	if (rcode != AGPT_OK) return rcode;
	const Frame f = MakeFrame(c);
	RayTable t;
	GenParams g{};
	rcode = UploadRays(c, t, n, rays7, nullptr, 0, g);
	if (rcode != AGPT_OK) return rcode;
	DevBuf<float> out;
	CU(out.Alloc(32 * (size_t)n));
	rcode = Generate(c, f, g);
	if (rcode != AGPT_OK) return rcode;
	LaunchClosest(f.plan, 0, n, c->stream, f.sc, f.ps, f.q0.closest, f.q0.counts + 0, c->traceCounters.p, nullptr);
	k_probe_material_maps<<<Blocks(n, 256), 256, 0, c->stream>>>(f.sc, f.plan.tt, f.ps, n, out.p);
	CU(cudaGetLastError());
	c->stats.kernel_launches += 2;
	CU(cudaMemcpyAsync(out32, out.p, out.Bytes(), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

int agpt_probe_sphere_sample(agpt_ctx* c, int n, const float* in9, float* out8) {
	NEED(c != nullptr && n > 0 && in9 && out8, AGPT_ERR_INVALID, "bad probe arguments");
	CU(cudaSetDevice(c->device));
	return ProbeRun(c, in9, 9 * (size_t)n, out8, 8 * (size_t)n, [&](const float* din, float* dout) {
		k_probe_sphere_sample<<<Blocks(n, 128), 128, 0, c->stream>>>(n, din, dout);
	});
}

int agpt_probe_light_sample(agpt_ctx* c, int light, int n, const float* in8, float* out8) {
	NEED(c != nullptr && n > 0 && in8 && out8, AGPT_ERR_INVALID, "bad probe arguments");
	int rcode = CheckReady(c, false);
	if (rcode != AGPT_OK) return rcode;
	NEED(light >= 0 && light < (int)c->hostLights.size(), AGPT_ERR_INVALID, "light index out of range");
	const agpt_light& l = c->hostLights[light];
	NEED(l.type == AGPT_LIGHT_AREA && (l.flags & AGPT_LIGHT_SAMPLE_SHAPE) && c->hostPrims[l.prim].type != AGPT_PRIM_SPHERE, AGPT_ERR_INVALID,
		"not an area light that samples its plane or mesh (AGPT_LIGHT_SAMPLE_SHAPE)");
	CU(cudaSetDevice(c->device));
	const DScene sc = MakeScene(c);
	const DShapeTables st = PlanLaunches(c).st;
	return ProbeRun(c, in8, 8 * (size_t)n, out8, 8 * (size_t)n, [&](const float* din, float* dout) {
		k_probe_light_sample<<<Blocks(n, 128), 128, 0, c->stream>>>(sc, st, light, n, din, dout);
	});
}

int agpt_probe_stream(agpt_ctx* c, uint32_t pixel_index, uint32_t sample, int k, float* out) {
	NEED(c != nullptr && k > 0 && out, AGPT_ERR_INVALID, "bad probe arguments");
	CU(cudaSetDevice(c->device));
	DevBuf<float> d;
	CU(d.Alloc(k));
	k_probe_stream<<<1, 1, 0, c->stream>>>(pixel_index, sample, k, d.p);
	CU(cudaGetLastError());
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(out, d.p, k * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return AGPT_OK;
}

} // extern "C"
