// host/integrator.h -- Integrator (reference surface, /root/reference/integrator.h:28-31)
// and CudaPathTracer, the B200 implementation of PathTracer (integrator.h:120-196).
//
// CudaPathTracer::Render is the batched form of MyApp::Tick's pixel loop
// (myapp.cpp:163-175): numSamples passes over every pixel of the accumulator, executed as
// wavefront kernels on the device through the C ABI (include/agpt.h).  Li() keeps the
// per-ray entry point (used upstream by the debug click, myapp.cpp:196-198) by tracing a
// one-path batch on the device.  No CPU integrator exists here: if libagpt cannot create a
// CUDA context the constructor throws.
//
// Constructed with a list of devices it shards a render by sample index (SURVEY 8e): GPU g of G
// renders the samples s = firstSample + g (mod G) of every pixel, and the G accumulators are
// summed in rank order over NVLink peer memory (agpt_reduce_accum) -- or summed AND resolved to
// display pixels in one fused kernel (RenderAndResolve = Render + Accumulator::CopyToSurface).
#pragma once

#include <stdexcept>
#include <string>
#include <vector>

#include "precomp.h"
#include "scene.h"
#include "accumulator.h"

class Integrator {
public:
	virtual ~Integrator() {}
	virtual float3 Li(const Ray& ray, const Scene& scene, int depth = 0) const = 0;
};

class CudaPathTracer : public Integrator {
public:
	explicit CudaPathTracer(int maxDepth = 5, int device = 0) : CudaPathTracer(maxDepth, std::vector<int>{ device }) {}
	CudaPathTracer(int maxDepth, const std::vector<int>& devices) : MaxDepth(maxDepth) {
		if (devices.empty()) throw std::runtime_error("CudaPathTracer: empty device list");
		for (int d : devices) {
			agpt_ctx* c = nullptr;
			if (agpt_create(d, &c) != AGPT_OK) { std::string m = agpt_last_error(); Destroy(); throw std::runtime_error("CudaPathTracer: " + m); }
			ctxs.push_back(c);
		}
	}
	~CudaPathTracer() override { Destroy(); }
	CudaPathTracer(const CudaPathTracer&) = delete;
	CudaPathTracer& operator=(const CudaPathTracer&) = delete;

	// Upload (or re-upload) the flattened scene to every GPU.  Called implicitly by Render/Li whenever
	// the scene's fingerprint differs from the resident one (another Scene object, or primitives /
	// lights added since).
	void Upload(const Scene& scene) const {
		temporalW = temporalH = 0;
		auto flat = scene.Flatten();
		for (agpt_ctx* ctx : ctxs) {
			Check(agpt_upload_meshes(ctx, flat->meshes.data(), (int)flat->meshes.size()));
			Check(agpt_upload_spheres(ctx, flat->spheres.data(), (int)flat->spheres.size()));
			Check(agpt_upload_planes(ctx, flat->planes.data(), (int)flat->planes.size()));
			Check(agpt_upload_materials(ctx, flat->materials.data(), (int)flat->materials.size()));
			Check(agpt_upload_lights(ctx, flat->lights.data(), (int)flat->lights.size()));
			Check(agpt_upload_envmap(ctx, flat->envmap.width > 0 ? &flat->envmap : nullptr));
			Check(agpt_upload_instances(ctx, flat->instances.data(), (int)flat->instances.size()));
			Check(agpt_upload_primitives(ctx, flat->prims.data(), (int)flat->prims.size()));
			Check(agpt_upload_material_textures(ctx, flat->textures.data(), (int)flat->textures.size(), flat->materialTextures.data(), (int)flat->materialTextures.size()));
			Check(agpt_upload_alpha_masks(ctx, flat->alphaMasks.data(), (int)flat->alphaMasks.size()));   // after the textures it names
			Check(agpt_upload_emission(ctx, flat->emission.data(), (int)flat->emission.size()));          // likewise
		}
		uploaded = scene.Fingerprint();
	}

	// numSamples Tick bodies: samples firstSample .. firstSample+numSamples-1 of every pixel,
	// added to `acc` (which keeps its earlier contents, like successive Ticks do).
	void Render(const Scene& scene, const Camera& camera, Accumulator& acc, int firstSample, int numSamples,
			int depth = 0, uint32_t flags = 0) const {
		RenderShards(scene, camera, acc, firstSample, numSamples, depth, flags);
		if (ctxs.size() > 1) Check(agpt_reduce_accum(ctxs.data(), (int)ctxs.size(), 0));      // rank-order sum into GPU 0
		Check(agpt_read_accum(ctxs[0], &acc.Pixels()->x));
		acc.SetNumSamples(acc.NumSamples() + numSamples);
	}

	// Render followed by Accumulator::CopyToSurface (myapp.h:34-41): rgb8[y*W + x] = 0x00RRGGBB, row 0 = top.
	// The sum over GPUs, the division by the sample count, the gamma curve and the 8-bit pack are ONE kernel
	// per GPU over its slice of the film (agpt_reduce_resolve).
	void RenderAndResolve(const Scene& scene, const Camera& camera, Accumulator& acc, int firstSample, int numSamples,
			uint32_t* rgb8, int depth = 0, uint32_t flags = 0) const {
		RenderShards(scene, camera, acc, firstSample, numSamples, depth, flags);
		acc.SetNumSamples(acc.NumSamples() + numSamples);
		Check(agpt_reduce_resolve(ctxs.data(), (int)ctxs.size(), acc.NumSamples(), 1, rgb8));
		Check(agpt_read_accum(ctxs[0], &acc.Pixels()->x));
	}

	// EXTENSION (agpt.h agpt_adaptive): a frame rendered adaptively on the tracer's one GPU -- every pixel gets min_samples,
	// then `step` more per round while its standard error is above tolerance, up to max_samples.  The film replaces acc's
	// contents (acc.NumSamples() is set to 0: pixels differ in their sample counts) and counts[y*W + x] receives each
	// pixel's number of samples; film pixel (H-1-y)*W + x divided by it is the pixel's mean.  Throws for a device list (the
	// moments would have to be reduced with the film every round).
	void RenderAdaptive(const Scene& scene, const Camera& camera, Accumulator& acc, const agpt_adaptive& params, int depth,
			std::vector<int>& counts, uint32_t flags = 0) const {
		AdaptiveFrame(scene, camera, acc, params, nullptr, 0, depth, counts, nullptr, nullptr, flags);
	}

	// EXTENSION (agpt.h agpt_render_guides / agpt_denoise): RenderAdaptive, then the guides of samples [0, guideSamples) and the
	// denoiser over the film, before the moments are switched off again.  min == max gives a uniform frame.  out (W*H, film row
	// order like acc) and rgb8 (W*H packed pixels, film row order) receive the denoised image; either may be null.
	void RenderAdaptiveDenoised(const Scene& scene, const Camera& camera, Accumulator& acc, const agpt_adaptive& params, const agpt_denoise_params& denoise,
			int guideSamples, int depth, std::vector<int>& counts, float3* out, uint32_t* rgb8, uint32_t flags = 0) const {
		AdaptiveFrame(scene, camera, acc, params, &denoise, guideSamples, depth, counts, out, rgb8, flags);
	}

	// EXTENSION (agpt.h agpt_reproject_film): one frame of a viewer whose camera may have moved since the last frame, on a
	// one-GPU tracer: the guides of samples [0, guideSamples) of this camera, the film and moments carried over from the last
	// RenderTemporal frame into this view, samples [firstSample, firstSample + numSamples) added, and the denoiser.  Film,
	// moments and the saved view stay on the device between the calls; the first frame, a new film size or a new scene start
	// from a cleared film.  firstSample must keep advancing from frame to frame (agpt.h says why).  acc receives the film
	// (acc.NumSamples() is set to 0: the counts are per pixel and fractional); out and rgb8 (film row order) the denoised image,
	// either may be null.  Throws for a device list.
	void RenderTemporal(const Scene& scene, const Camera& camera, Accumulator& acc, int firstSample, int numSamples, const agpt_reproject& reproject,
			const agpt_denoise_params& denoise, int guideSamples, int depth, float3* out, uint32_t* rgb8, uint32_t flags = 0) const {
		if (ctxs.size() != 1) throw std::runtime_error("CudaPathTracer: temporal frames render on one device only");
		if (uploaded != scene.Fingerprint()) Upload(scene);
		agpt_camera cam = camera.Export();
		agpt_ctx* c = ctxs[0];
		Check(agpt_set_camera(c, &cam));
		Check(agpt_set_film(c, acc.width, acc.height));
		Check(agpt_set_moments(c, 1));
		if (temporalW != acc.width || temporalH != acc.height) Check(agpt_clear(c));
		temporalW = temporalH = 0;
		Check(agpt_render_guides(c, guideSamples, flags & (AGPT_FLAG_COUNTERS | AGPT_FLAG_STRICT_BOXES)));
		Check(agpt_reproject_film(c, &reproject));
		Check(agpt_render(c, firstSample, numSamples, 1, MaxDepth, depth, flags));
		Check(agpt_read_accum(c, &acc.Pixels()->x));
		Check(agpt_denoise(c, &denoise, out ? &out->x : nullptr, rgb8));
		temporalW = acc.width; temporalH = acc.height;
		acc.SetNumSamples(0);
	}

	// Single-ray entry point.  The reference's Li draws from the global generator; here the
	// ray gets the RNG stream of (pixel 0, sample liCalls++), film/camera are not involved.
	float3 Li(const Ray& ray, const Scene& scene, int depth = 0) const override;

	agpt_ctx* Context(int i = 0) const { return ctxs[i]; }
	int NumDevices() const { return (int)ctxs.size(); }
	int GetMaxDepth() const { return MaxDepth; }

protected:
	static void Check(int status) {
		if (status != AGPT_OK) throw std::runtime_error(std::string("agpt: ") + agpt_last_error());
	}
	void Destroy() { for (agpt_ctx* c : ctxs) agpt_destroy(c); ctxs.clear(); }
	// RenderAdaptive, and with `denoise` the guides and the denoiser, all while the moments are on
	void AdaptiveFrame(const Scene& scene, const Camera& camera, Accumulator& acc, const agpt_adaptive& params, const agpt_denoise_params* denoise,
			int guideSamples, int depth, std::vector<int>& counts, float3* out, uint32_t* rgb8, uint32_t flags) const {
		if (ctxs.size() != 1) throw std::runtime_error("CudaPathTracer: adaptive frames render on one device only");
		if (uploaded != scene.Fingerprint()) Upload(scene);
		temporalW = temporalH = 0;
		agpt_camera cam = camera.Export();
		agpt_ctx* c = ctxs[0];
		Check(agpt_set_camera(c, &cam));
		Check(agpt_set_film(c, acc.width, acc.height));
		Check(agpt_set_moments(c, 1));
		int rc = agpt_render_adaptive(c, &params, MaxDepth, depth, flags, nullptr, nullptr);
		std::vector<float> m(rc == AGPT_OK ? 4 * (size_t)acc.width * acc.height : 0);
		if (rc == AGPT_OK) rc = agpt_read_accum(c, &acc.Pixels()->x);
		if (rc == AGPT_OK) rc = agpt_read_moments(c, m.data());
		if (rc == AGPT_OK && denoise) rc = agpt_render_guides(c, guideSamples, flags & (AGPT_FLAG_COUNTERS | AGPT_FLAG_STRICT_BOXES));
		if (rc == AGPT_OK && denoise) rc = agpt_denoise(c, denoise, out ? &out->x : nullptr, rgb8);
		std::string err = rc == AGPT_OK ? "" : agpt_last_error();
		agpt_set_moments(c, 0);             // plain Render calls stay as they were
		if (rc != AGPT_OK) throw std::runtime_error("agpt: " + err);
		counts.resize((size_t)acc.width * acc.height);
		for (int y = 0; y < acc.height; y++)
			for (int x = 0; x < acc.width; x++) counts[(size_t)y * acc.width + x] = (int)m[4 * ((size_t)(acc.height - 1 - y) * acc.width + x) + 3];
		acc.SetNumSamples(0);
	}
	// every GPU's share of the samples into its own accumulator; GPU 0's starts from the caller's film
	void RenderShards(const Scene& scene, const Camera& camera, Accumulator& acc, int firstSample, int numSamples, int depth, uint32_t flags) const {
		if (uploaded != scene.Fingerprint()) Upload(scene);
		temporalW = temporalH = 0;
		agpt_camera cam = camera.Export();
		for (size_t g = 0; g < ctxs.size(); g++) {
			Check(agpt_set_camera(ctxs[g], &cam));
			Check(agpt_set_film(ctxs[g], acc.width, acc.height));
			if (g == 0) Check(agpt_write_accum_begin(ctxs[g], &acc.Pixels()->x));      // lands while the batch is traced; k_accumulate waits for it
			else Check(agpt_clear(ctxs[g]));
		}
		if (ctxs.size() == 1) Check(agpt_render(ctxs[0], firstSample, numSamples, 1, MaxDepth, depth, flags));
		else Check(agpt_render_multi(ctxs.data(), (int)ctxs.size(), firstSample, numSamples, MaxDepth, depth, flags));
	}
	int MaxDepth;
	mutable std::vector<agpt_ctx*> ctxs;
	mutable uint64_t uploaded = 0;     // Scene::Fingerprint() of the resident tables (0: none)
	mutable unsigned liCalls = 0;
	mutable int temporalW = 0, temporalH = 0;   // film size of the last RenderTemporal frame, whose film and view are resident (0: none)
};

// (defined here so that the mirror stays header-only; libagpt.so is the only link dependency)
inline float3 CudaPathTracer::Li(const Ray& ray, const Scene& scene, int depth) const {
	if (uploaded != scene.Fingerprint()) Upload(scene);
	float r7[7] = { ray.O.x, ray.O.y, ray.O.z, ray.D.x, ray.D.y, ray.D.z, ray.t };
	uint32_t seed = 0x12345678u + 0x9e3779b9u * liCalls++;   // upstream's global seed, advanced per call
	float out[3] = { 0, 0, 0 };
	Check(agpt_li_rays(ctxs[0], 1, r7, &seed, MaxDepth, depth, AGPT_FLAG_RAYS_FINAL, out));      // ray.D is final: the Ray ctor normalised it
	return float3(out[0], out[1], out[2]);
}

using PathTracer = CudaPathTracer;   // scene code written against the reference keeps compiling
