// examples/render_ppm.cpp -- scene code written in the reference's style (compare
// /root/reference/myapp.cpp:13-114,121-135) compiled against the B200 host mirror, rendering
// headless on one or several GPUs and writing the displayed frame (Accumulator::CopyToSurface
// semantics) as a PPM.
//
//   make -C ag-pathtracer_b200 example && build/render_ppm out.ppm <config 1..11> <spp> [gpus]
//
// With gpus > 1 the samples are split by index over the GPUs (SURVEY 8e) and the accumulators are
// summed and resolved by one fused kernel per GPU over NVLink peer memory (agpt_reduce_resolve).
#include "precomp.h"
#include "scene.h"
#include "integrator.h"
#include "scenes/config_scenes.h"

int main(int argc, char** argv) {
	const char* out = argc > 1 ? argv[1] : "out.ppm";
	int config = argc > 2 ? atoi(argv[2]) : 7;
	int spp = argc > 3 ? atoi(argv[3]) : 64;
	int gpus = argc > 4 ? atoi(argv[4]) : 1;
	auto defaults = agpt_scenes::Defaults(config);
	int W = defaults.width ? defaults.width : 400, H = defaults.height ? defaults.height : 400;
	int maxDepth = defaults.max_depth ? defaults.max_depth : 5;

	auto scene = std::make_shared<Scene>();                 // MyApp::Init (myapp.cpp:121-135)
	if (!agpt_scenes::BuildConfig(scene.get(), config, 0)) { fprintf(stderr, "unknown config\n"); return 1; }
	Camera camera(scene->camera);
	std::vector<int> devices;
	for (int g = 0; g < gpus; g++) devices.push_back(g);
	std::vector<uint32_t> rgb((size_t)W * H);
	try {
		auto integrator = std::make_shared<PathTracer>(maxDepth, devices);    // PathTracer == CudaPathTracer here
		Accumulator accumulator(W, H);
		// spp x MyApp::Tick + Accumulator::CopyToSurface
		integrator->RenderAndResolve(*scene, camera, accumulator, 0, spp, rgb.data(), defaults.depth_arg);
		double ms = 0, rays = 0, msReduce = 0;
		for (int g = 0; g < integrator->NumDevices(); g++) {
			agpt_stats st;
			agpt_get_stats(integrator->Context(g), &st);
			ms = st.ms_render > ms ? st.ms_render : ms;
			msReduce = st.ms_reduce > msReduce ? st.ms_reduce : msReduce;
			rays += (double)(st.rays_closest + st.rays_shadow + st.rays_mis);
		}
		printf("%s: %dx%d, %d spp on %d GPU(s), %.1f ms render (max over GPUs) + %.3f ms reduce-resolve, %.1f Mrays/s\n", out, W, H, spp, gpus, ms, msReduce, rays / ms / 1e3);
	}
	catch (const std::exception& e) { fprintf(stderr, "%s\n", e.what()); return 1; }
	FILE* f = fopen(out, "wb");
	if (!f) return 1;
	fprintf(f, "P6\n%d %d\n255\n", W, H);
	for (uint32_t p : rgb) { unsigned char c[3] = { (unsigned char)(p >> 16), (unsigned char)(p >> 8), (unsigned char)p }; fwrite(c, 1, 3, f); }
	fclose(f);
	return 0;
}
