// oracle/agpt_guides_oracle.cpp -- TEST INFRASTRUCTURE, not product code.
//
// EXTENSION (include/agpt.h agpt_render_guides): the CPU statement of the denoiser's guide buffers, the one the GPU path is
// checked against.  The reference has no guides; what one sample contributes is defined in agpt.h.
//
// The oracle (agpt_oracle.cpp, pinned bit for bit to the reference) is compiled into this translation unit unchanged and
// reused as it is: tables, camera ray, Scene::Intersect and the SurfaceInteraction of a hit.  Only the per-sample guide record
// and the per-pixel sums are new.  Built by __graft_entry__.build() into oracle/libagpt_guides_oracle.so with the oracle's
// flags (-O2, no FMA contraction).
#include "agpt_oracle.cpp"

extern "C" {

// One camera sample's first hit: what agpt_render_guides adds for it.
struct agpt_guide_sample {
	float albedo[3];
	float normal[3];      // shading normal facing the ray; 0 on a miss
	float dir[3];         // the camera ray's (normalised) direction
	float t;              // hit distance, 0 on a miss
	int32_t prim;         // primitive hit, -1 on a miss
};

// Samples [0, num_samples) of every pixel of a W x H film.  per_sample (may be NULL): num_samples x H x W records, sample-major,
// image row y at y*W + x (the layout of agpt_oracle_primary_hits).  albedo / normal_depth: H x W float4 each, in the film's row
// order (row H-1-y), as agpt_read_guides returns them.
void agpt_guides_oracle(void* h, int W, int H, int num_samples, int threads, agpt_guide_sample* per_sample, float* albedo, float* normal_depth) {
	const OScene& sc = *(OScene*)h;
	ParallelRows(0, H, threads, [&](int y) {
		Counters c;
		Rng rng;
		for (int x = 0; x < W; x++) {
			V3 a = v3(0.f), n = v3(0.f);
			float hits = 0, tsum = 0;
			for (int s = 0; s < num_samples; s++) {
				rng.Seed((uint32_t)(y * W + x), (uint32_t)s);
				Ray ray = CameraRay(sc, W, H, x, y, rng);
				const V3 D = ray.D;
				Hit hit;
				agpt_guide_sample g;
				V3 alb = v3(1.f), nrm = v3(0.f);
				g.t = 0.f; g.prim = -1;
				if (SceneIntersect(sc, ray, hit, c)) {
					Surface si;
					BuildSurface(sc, ray, hit, si);
					nrm = dot(si.sn, D) > 0.f ? -si.sn : si.sn;
					const agpt_prim& pr = sc.prims[hit.prim];
					if (pr.material >= 0) {
						const agpt_material& m = sc.mats[pr.material];
						if (m.type == AGPT_MAT_MIRROR) alb = v3(m.mirror_r);
						else if (m.type == AGPT_MAT_GLASS) alb = v3(m.mirror_r) + v3(m.diffuse_r);
						else alb = v3(m.diffuse_r) + v3(m.spec_r0);
						alb = v3(tmin2(alb.x, 1.f), tmin2(alb.y, 1.f), tmin2(alb.z, 1.f));
					}
					g.t = hit.t; g.prim = hit.prim;
					hits += 1.f;
					tsum += hit.t;
				}
				a += alb;
				n += nrm;
				g.albedo[0] = alb.x; g.albedo[1] = alb.y; g.albedo[2] = alb.z;
				g.normal[0] = nrm.x; g.normal[1] = nrm.y; g.normal[2] = nrm.z;
				g.dir[0] = D.x; g.dir[1] = D.y; g.dir[2] = D.z;
				if (per_sample) per_sample[((size_t)s * H + y) * W + x] = g;
			}
			const float ns = (float)num_samples;
			float* pa = albedo + 4 * ((size_t)(H - 1 - y) * W + x);
			float* pn = normal_depth + 4 * ((size_t)(H - 1 - y) * W + x);
			pa[0] = a.x / ns; pa[1] = a.y / ns; pa[2] = a.z / ns; pa[3] = hits / ns;
			pn[0] = n.x / ns; pn[1] = n.y / ns; pn[2] = n.z / ns; pn[3] = hits > 0.f ? tsum / hits : 0.f;
		}
	});
}

} // extern "C"
