// agpt_kernels.cuh -- the wavefront: path generation, trace, shade, accumulate, resolve.
//
// One wave = { closest-hit trace of the path rays + MIS rays queued by the previous shade,
// any-hit trace of its shadow rays, shade }.  Shade realises one iteration of the loop of
// PathTracer::Li (integrator.h:132-188) per path: it first folds the next-event estimate
// of the PREVIOUS vertex into L (its shadow / MIS rays have just been traced), then handles
// the new hit: emission, termination, null-material skip-through, light sampling
// (UniformSampleOneLight + EstimateDirect, integrator.h:38-105), BSDF sampling, Russian
// roulette, and queues the rays of the next wave (warp ballots + a shared-memory prefix over the
// block's warps: one atomic per queue per block).
// The per-path RNG state lives in HBM, so the draw order inside a path is the reference's
// whatever the scheduling (SURVEY 8a row 3).
#pragma once

#include "agpt_bsdf.cuh"
#include "agpt_trace.cuh"

// path flag bits (PathState::flags)
#define PF_SPECULAR      1u     // specularBounce (integrator.h:129,177)
#define PF_NEE_SHADOW    2u     // a shadow ray of the previous vertex is in flight
#define PF_NEE_MIS       4u     // a MIS ray of the previous vertex is in flight
#define PF_NO_CONTINUE   8u     // path ended at the previous vertex; only its NEE is left to fold in
#define PF_BOUNCE_SHIFT  8

// Path state is plain SoA in HBM.  (Cache-streaming hints -- ld/st.global.cs -- on these accesses,
// to keep the state from pushing BVH nodes out of L2, measured +-0.5 %: not kept.)
template <typename T>
using StateArray = T*;

struct PathState {
	StateArray<float4> rayO;        // O.xyz, tmax
	StateArray<float4> rayD;        // D.xyz
	StateArray<float4> hitA;        // t, b1, b2, int_as_float(prim)
	StateArray<int> hitSlot;
	StateArray<float4> beta;        // throughput
	StateArray<float4> L;           // radiance so far
	StateArray<uint32_t> rng;
	StateArray<uint32_t> flags;
	StateArray<float4> neeLight;    // f*Li*weight/lightPdf of the light-sampling strategy (integrator.h:57)
	StateArray<float4> neeMis;      // f*Lemit*weight/scatteringPdf of the BSDF strategy (integrator.h:88); w = int_as_float(light index)
	StateArray<float4> neeBeta;     // beta at the vertex the estimate belongs to
	StateArray<float4> shO;         // shadow ray O.xyz, tmax
	StateArray<float4> shD;
	StateArray<float4> misO;        // MIS ray
	StateArray<float4> misD;
	StateArray<int> shadowOccluded;
	StateArray<int> misPrim;        // primitive hit by the MIS ray, -1 = none
	StateArray<float4> Lout;        // finished radiance per path slot
	int slots;                      // allocated path slots (debug checks)
};

#ifndef AGPT_CELL_BITS
#define AGPT_CELL_BITS 3
#endif
#define AGPT_BUCKETS (16 << (3 * AGPT_CELL_BITS))  // ray buckets: 4 bits direction code | 3 x AGPT_CELL_BITS bits grid cell of the ray origin

struct WaveQueues {
	int* closest;        // entries path*2 + kind (0 = path ray, 1 = MIS ray)
	unsigned short* keys; // bucket key of each closest-queue entry
	int* shadow;         // path indices with a shadow ray
	unsigned short* shadowKeys;
	int* active;         // path indices shade works on
	int* counts;         // [0] closest, [1] shadow, [2] active
};

struct RayCounters {     // device-side totals, see agpt_stats
	unsigned long long rays_closest, rays_shadow, rays_mis, rays_skip, rays_mis_culled, rays_tail_culled;
};

// Ray bucket: rays that start in the same cell and go the same way walk similar parts of the trees in the same
// near/far order, so putting them next to each other in the queue raises both the SIMT efficiency of the
// lockstep walk and the L1/L2 hit rate.  Key = 9 bits Morton cell of the origin | 4 bits direction code:
//   closest-hit queue (path and MIS rays): octant (3 bits) | "meets the root box of a mesh" (1 bit);
//   shadow ray to an area light:           8 | light & 3 (2 bits) | "meets ..." (1 bit) -- rays from one cell to
//                                          one small light are as alike as rays get;
//   shadow ray to an infinite light:       octant.
// The "meets" bit (round 2) separates rays that will walk a tree for tens of steps from rays that are done with
// the mesh run at once -- it is lanes finishing at very different times, not memory, that limits the walk
// (13.8 of 32 rays alive per step).  It replaced the "mostly vertical" bit: closest-hit -6 % (cfg 3) / -15 %
// (cfg 5) against -3 % for that one; both at the price of a cell bit was worse (profiles/r2_experiments.md).
// Boxes = roots of the BVH meshes that are small against the union of all roots (a backdrop or a room meets
// every ray and tells nothing).  Sort key only: approximate arithmetic (MUFU reciprocal), results never depend on it.
__device__ __forceinline__ bool RayMeetsMeshBox(const DScene& sc, float3 O, float3 D, float tmax) {
	float3 rD;        // one MUFU each: a sort key needs no more
	asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rD.x) : "f"(D.x));
	asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rD.y) : "f"(D.y));
	asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rD.z) : "f"(D.z));
	bool any = false;
	for (int k = 0; k < sc.n_keyBoxes; k++) {
		const float4 a = __ldg(sc.keyBoxes + 2 * k), b = __ldg(sc.keyBoxes + 2 * k + 1);
		float tn, tx;
		SlabApprox(f3(a.x, a.y, a.z), f3(a.w, b.x, b.y), O, rD, tmax, tn, tx);
		any = any || tn <= tx;
	}
	return any;
}
__device__ __forceinline__ int RayBucket(const DScene& sc, float3 O, float3 D, int areaLight = -1, bool closestQueue = false, float tmax = 3.0e38f) {
	const int hi = (1 << AGPT_CELL_BITS) - 1;
	int cx = min(max((int)((O.x - sc.cellLo[0]) * sc.cellScale[0]), 0), hi);
	int cy = min(max((int)((O.y - sc.cellLo[1]) * sc.cellScale[1]), 0), hi);
	int cz = min(max((int)((O.z - sc.cellLo[2]) * sc.cellScale[2]), 0), hi);
	// Morton-interleave the cell so neighbouring buckets are neighbouring cells
	int cell = 0;
#pragma unroll
	for (int b = 0; b < AGPT_CELL_BITS; b++) cell |= (((cx >> b) & 1) << (3 * b)) | (((cy >> b) & 1) << (3 * b + 1)) | (((cz >> b) & 1) << (3 * b + 2));
	if (areaLight >= 0) return (cell << 4) | 8 | ((areaLight & 3) << 1) | (RayMeetsMeshBox(sc, O, D, tmax) ? 1 : 0);
	const int octant = (D.x < 0.f ? 1 : 0) | (D.y < 0.f ? 2 : 0) | (D.z < 0.f ? 4 : 0);   // (octant-major order measured no better)
	if (closestQueue) return (cell << 4) | (octant << 1) | (RayMeetsMeshBox(sc, O, D, tmax) ? 1 : 0);
	return (cell << 4) | octant;
}
// ---- bucket pass between shade and the next trace: counting sort of a ray queue by key ------
// k_bucket_hist (entries per bucket) -> k_bucket_scan (exclusive offsets, one block) ->
// k_bucket_scatter.  Neighbouring queue entries come from neighbouring paths and so carry the
// same few keys: global atomics per warp would all land on the same addresses at the same time
// and serialise in L2.  Both kernels therefore count in block-private shared-memory bins first
// (1024 entries per block) and touch each global counter once per block.  The order inside a
// bucket is free: every path's arithmetic is independent of its queue position.
#define AGPT_BUCKET_ITEMS 4      // entries per thread of the 256-thread bucket kernels

// rank of this lane among the lanes of its warp with the same key, plus the warp's claim on the
// block's bin (one shared-memory atomic per distinct key per warp).  All 32 lanes must call.
__device__ __forceinline__ int BlockBinClaim(bool valid, int key, int* bins) {
	int lane = threadIdx.x & 31;
	unsigned m = __match_any_sync(0xffffffffu, valid ? key : (AGPT_BUCKETS + lane));
	int leader = __ffs(m) - 1;
	int base = 0;
	if (valid && lane == leader) base = atomicAdd(bins + key, __popc(m));
	base = __shfl_sync(0xffffffffu, base, leader);
	return base + __popc(m & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(256) k_bucket_hist(const unsigned short* __restrict__ keys, const int* __restrict__ countPtr, int* hist) {
	__shared__ int bins[AGPT_BUCKETS];
	for (int b = threadIdx.x; b < AGPT_BUCKETS; b += 256) bins[b] = 0;
	__syncthreads();
	const int count = *countPtr;
	const int base = blockIdx.x * 256 * AGPT_BUCKET_ITEMS;
#pragma unroll
	for (int k = 0; k < AGPT_BUCKET_ITEMS; k++) {
		int i = base + k * 256 + threadIdx.x;
		int key = keys[i];                 // (allocation slack: unconditional)
		BlockBinClaim(i < count, key, bins);
	}
	__syncthreads();
	for (int b = threadIdx.x; b < AGPT_BUCKETS; b += 256) { int c = bins[b]; if (c) atomicAdd(hist + b, c); }
}

__global__ void __launch_bounds__(1024) k_bucket_scan(const int* hist, int* offsets, int* running) {
	__shared__ int warpSums[32];
	const int PER = AGPT_BUCKETS / 1024;   // AGPT_BUCKETS is a multiple of 1024 for AGPT_CELL_BITS >= 3
	int t = threadIdx.x;
	int v[PER], sum = 0;
	for (int k = 0; k < PER; k++) { v[k] = hist[t * PER + k]; sum += v[k]; }
	// block-wide exclusive scan of `sum`
	int lane = t & 31, w = t >> 5, x = sum;
	for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
	if (lane == 31) warpSums[w] = x;
	__syncthreads();
	if (w == 0) {
		int s2 = warpSums[lane];
		for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, s2, o); if (lane >= o) s2 += y; }
		warpSums[lane] = s2;
	}
	__syncthreads();
	int base = x - sum + (w > 0 ? warpSums[w - 1] : 0);
	for (int k = 0; k < PER; k++) { offsets[t * PER + k] = base; running[t * PER + k] = 0; base += v[k]; }
}

__global__ void __launch_bounds__(256) k_bucket_scatter(const int* __restrict__ in, const unsigned short* __restrict__ keys, const int* __restrict__ countPtr,
		const int* __restrict__ offsets, int* running, int* __restrict__ out) {
	__shared__ int bins[AGPT_BUCKETS];     // entries of this block per bucket, then: where the block's group starts in `out`
	for (int b = threadIdx.x; b < AGPT_BUCKETS; b += 256) bins[b] = 0;
	__syncthreads();
	const int count = *countPtr;
	const int base = blockIdx.x * 256 * AGPT_BUCKET_ITEMS;
	int entry[AGPT_BUCKET_ITEMS], key[AGPT_BUCKET_ITEMS], rank[AGPT_BUCKET_ITEMS];
#pragma unroll
	for (int k = 0; k < AGPT_BUCKET_ITEMS; k++) {
		int i = base + k * 256 + threadIdx.x;
		entry[k] = in[i]; key[k] = keys[i];
		rank[k] = BlockBinClaim(i < count, key[k], bins);
	}
	__syncthreads();
	for (int b = threadIdx.x; b < AGPT_BUCKETS; b += 256) { int c = bins[b]; if (c) bins[b] = offsets[b] + atomicAdd(running + b, c); }
	__syncthreads();
#pragma unroll
	for (int k = 0; k < AGPT_BUCKET_ITEMS; k++) {
		int i = base + k * 256 + threadIdx.x;
		if (i < count) out[bins[key[k]] + rank[k]] = entry[k];
	}
}

// ---- path generation: myapp.cpp:165-167 + Camera::GetRay (camera.h:58-64) ----------------
__device__ __forceinline__ DRay CameraRay(const DScene& sc, int x, int y, uint32_t& rng) {
	// float2 p(x + RandomFloat(), y + RandomFloat()): g++ evaluates the arguments right to
	// left, so the y jitter is drawn first (oracle probe agpt_ref_probe_draw_order).
	float jy = RandomFloat(rng);
	float jx = RandomFloat(rng);
	float px = x + jx, py = y + jy;
	float s = px / sc.width, t = py / sc.height;            // Accumulator::PixelToFilm (myapp.h:57-59)
	const agpt_camera& c = sc.cam;
	float3 rd = f3(0.f);
	if (c.lens_radius > 0.f) {
		// RandomInUnitDisk (common.h:65-71): rejection loop, y drawn before x each round
		while (true) {
			float ry = -1 + (1 - -1) * RandomFloat(rng);
			float rx = -1 + (1 - -1) * RandomFloat(rng);
			float3 p = f3(rx, ry, 0);
			if (sqrLength(p) >= 1) continue;
			rd = c.lens_radius * p;
			break;
		}
	}
	float3 offset = f3(c.u) * rd.x + f3(c.v) * rd.y;
	float3 pixel = f3(c.lower_left_corner) + s * f3(c.horizontal) + t * f3(c.vertical);
	return MakeRay(f3(c.origin) + offset, pixel - f3(c.origin) - offset);
}

struct GenParams {
	int n;                 // paths to start
	int first_sample, sample_stride;
	const int* xs;         // optional explicit pixel list (li_pixels); nullptr = whole film
	const int* ys;
	const int* ss;
	const float* rays7;    // optional explicit rays (li_rays); O, D, tmax
	const uint32_t* seeds;
	int raysFinal;         // rays7 directions are unit length already (a host Ray object): use as given
	int tiled;             // whole-film mode of agpt_render: slot = tile-order pixel slot * samples + sample (else sample-major rows)
	int samples;           // samples per pixel in this batch (tiled mode)
	// list mode (k_generate<true>, adaptive rounds): slot = (list entry - listBase) * samples + j renders sample n_p + j of
	// pixel list[entry], n_p = the pixel's moments .w (the samples it has so far)
	const int* list;       // film pixel indices y * W + x
	int listBase, listCount;
	const float4* moments; // per pixel, film row order (H-1-y)
	int maxSamples;        // (debug checks) no pixel may pass it
};

// Path slot <-> pixel.  Rendering keeps the samples of a pixel in neighbouring slots and orders
// the pixels in 8x4 tiles, so a warp's 32 camera rays cover a compact patch of the film (at 16
// samples per batch: two pixels) instead of a 32x1 strip of one sample: they walk the same nodes
// and mostly shade the same material.  (Every draw of a path depends on its pixel and
// sample index only, never on its slot.)  Films whose size is not a multiple of the tile, and
// the hit-table entry points, use the row-major order.
__device__ __forceinline__ void SlotToPixel(int slot, int width, int height, bool tiled, int& x, int& y) {
	if (tiled && (width & 7) == 0 && (height & 3) == 0) {
		int tile = slot >> 5, within = slot & 31, tilesX = width >> 3;
		x = (tile % tilesX) * 8 + (within & 7);
		y = (tile / tilesX) * 4 + (within >> 3);
	}
	else { x = slot % width; y = slot / width; }
}
__device__ __forceinline__ int PixelToSlot(int x, int y, int width, int height, bool tiled) {
	if (tiled && (width & 7) == 0 && (height & 3) == 0) return ((y >> 2) * (width >> 3) + (x >> 3)) * 32 + (y & 3) * 8 + (x & 7);
	return y * width + x;
}

template <bool LIST>
__global__ void __launch_bounds__(256) k_generate(DScene sc, PathState ps, WaveQueues q, GenParams g) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i == 0 && q.counts) { q.counts[0] = g.n; q.counts[1] = 0; q.counts[2] = g.n; }   // wave 0: n camera rays, n paths to shade
	if (i >= g.n) return;
	DRay ray;
	uint32_t rng;
	if constexpr (LIST) {
		// the step samples of a listed pixel sit next to each other, like the samples of a pixel in the tiled mode
		const int entry = g.listBase + i / g.samples, j = i % g.samples;
		AGPT_CHECK(entry >= 0 && entry < g.listCount, AGPT_DBG_LIST, entry);
		const int pixel = g.list[entry];
		AGPT_CHECK(pixel >= 0 && pixel < sc.width * sc.height, AGPT_DBG_LIST, pixel);
		const int x = pixel % sc.width, y = pixel / sc.width;
		const int have = (int)g.moments[(size_t)(sc.height - 1 - y) * sc.width + x].w;
		AGPT_CHECK(have >= 0 && have + g.samples <= g.maxSamples, AGPT_DBG_SAMPLE, have);
		rng = StreamSeed((uint32_t)pixel, (uint32_t)(have + j));
		ray = CameraRay(sc, x, y, rng);
	}
	else if (g.rays7) {
		const float* r = g.rays7 + 7 * (size_t)i;
		if (g.raysFinal) { ray.O = f3(r[0], r[1], r[2]); ray.D = f3(r[3], r[4], r[5]); ray.t = r[6]; }
		else ray = MakeRay(f3(r[0], r[1], r[2]), f3(r[3], r[4], r[5]), r[6]);
		rng = g.seeds[i] ? g.seeds[i] : 1u;
	}
	else {
		int x, y, sample;
		if (g.xs) { x = g.xs[i]; y = g.ys[i]; sample = g.ss[i]; }
		else {
			int wh = sc.width * sc.height;
			if (g.tiled) {
				// samples of a pixel sit next to each other, pixels in 8x4 tiles
				SlotToPixel(i / g.samples, sc.width, sc.height, true, x, y);
				sample = g.first_sample + (i % g.samples) * g.sample_stride;
			}
			else {
				SlotToPixel(i % wh, sc.width, sc.height, false, x, y);
				sample = g.first_sample + (i / wh) * g.sample_stride;
			}
		}
		rng = StreamSeed((uint32_t)(y * sc.width + x), (uint32_t)sample);
		ray = CameraRay(sc, x, y, rng);
	}
	ps.rayO[i] = make_float4(ray.O.x, ray.O.y, ray.O.z, ray.t);
	ps.rayD[i] = make_float4(ray.D.x, ray.D.y, ray.D.z, 0.f);
	ps.beta[i] = make_float4(1.f, 1.f, 1.f, 0.f);
	ps.L[i] = make_float4(0.f, 0.f, 0.f, 0.f);
	ps.rng[i] = rng;
	ps.flags[i] = 0u;
	q.closest[i] = i * 2;
	q.active[i] = i;
}

// ---- trace kernels ---------------------------------------------------------------------
// The bodies are shared with the MASK entry points below (extension, alpha masks: mk is read by those only).
template <bool COUNT, bool FAST, bool INST, bool MASK>
__device__ __forceinline__ void TraceClosest(const DScene& sc, const PathState& ps, const int* __restrict__ queue, const int* __restrict__ countPtr,
		unsigned long long* counters, unsigned long long* waveRow, unsigned* stackMem, const DMaskTables& mk) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	TraceCounters cnt = { 0, 0, 0, 0, 0, 0 };
	// The queue length lives on the device (the host launches an upper bound of blocks).  The
	// entry is fetched unconditionally -- queues are allocated with slack past any launchable
	// index -- so that the two loads overlap instead of costing two dependent round trips.
	int e = queue[i];
	const int count = *countPtr;
	bool lane = i < count;
	if (!lane) e = 0;
	int path = e >> 1, kind = e & 1;
	AGPT_CHECK(path >= 0 && path < ps.slots, AGPT_DBG_PATH, path);
	float4 o = make_float4(0.f, 0.f, 0.f, 0.f), d = make_float4(1.f, 0.f, 0.f, 0.f);
	if (lane) {
		o = kind ? ps.misO[path] : ps.rayO[path];
		d = kind ? ps.misD[path] : ps.rayD[path];
	}
	HitRecord hit;
	TraceScene<false, COUNT, FAST, INST, MASK>(sc, f3(o.x, o.y, o.z), f3(d.x, d.y, d.z), o.w, hit, stackMem + threadIdx.x, AGPT_TRACE_THREADS, cnt, lane, mk);
	if (lane) {
		if (kind == 0) {
			ps.hitA[path] = make_float4(hit.t, hit.b1, hit.b2, __int_as_float(hit.prim));
			ps.hitSlot[path] = hit.slot;
		}
		else ps.misPrim[path] = hit.prim;
	}
	if (COUNT) FlushCounters(cnt, lane, counters, waveRow);
}
template <bool COUNT, bool FAST, bool INST>
__global__ void __launch_bounds__(AGPT_TRACE_THREADS, AGPT_TRACE_MIN_BLOCKS) k_trace_closest(DScene sc, PathState ps, const int* __restrict__ queue, const int* __restrict__ countPtr,
		unsigned long long* counters, unsigned long long* waveRow) {
	__shared__ unsigned stackMem[AGPT_STACK_SMEM * AGPT_TRACE_THREADS];
	TraceClosest<COUNT, FAST, INST, false>(sc, ps, queue, countPtr, counters, waveRow, stackMem, DMaskTables());
}

template <bool COUNT, bool FAST, bool INST, bool MASK>
__device__ __forceinline__ void TraceAny(const DScene& sc, const PathState& ps, const int* __restrict__ queue, const int* __restrict__ countPtr,
		unsigned long long* counters, unsigned long long* waveRow, unsigned* stackMem, const DMaskTables& mk) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	TraceCounters cnt = { 0, 0, 0, 0, 0, 0 };
	int path = queue[i];
	const int count = *countPtr;
	bool lane = i < count;
	if (!lane) path = 0;
	AGPT_CHECK(path >= 0 && path < ps.slots, AGPT_DBG_PATH, path);
	float4 o = make_float4(0.f, 0.f, 0.f, 0.f), d = make_float4(1.f, 0.f, 0.f, 0.f);
	if (lane) { o = ps.shO[path]; d = ps.shD[path]; }
	HitRecord hit;
	bool occluded = TraceScene<true, COUNT, FAST, INST, MASK>(sc, f3(o.x, o.y, o.z), f3(d.x, d.y, d.z), o.w, hit, stackMem + threadIdx.x, AGPT_TRACE_THREADS, cnt, lane, mk);
	if (lane) ps.shadowOccluded[path] = occluded ? 1 : 0;
	if (COUNT) FlushCounters(cnt, lane, counters, waveRow);
}
template <bool COUNT, bool FAST, bool INST>
__global__ void __launch_bounds__(AGPT_TRACE_THREADS, AGPT_TRACE_MIN_BLOCKS) k_trace_any(DScene sc, PathState ps, const int* __restrict__ queue, const int* __restrict__ countPtr,
		unsigned long long* counters, unsigned long long* waveRow) {
	__shared__ unsigned stackMem[AGPT_STACK_SMEM * AGPT_TRACE_THREADS];
	TraceAny<COUNT, FAST, INST, false>(sc, ps, queue, countPtr, counters, waveRow, stackMem, DMaskTables());
}

// Standalone rays (agpt_trace_rays / agpt_trace_primary): hit table out.
template <bool ANY, bool COUNT, bool FAST, bool INST, bool MASK>
__device__ __forceinline__ void TraceTable(const DScene& sc, const float4* __restrict__ rayO, const float4* __restrict__ rayD,
		int count, agpt_hit* out, unsigned long long* counters, unsigned* stackMem, const DMaskTables& mk) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	TraceCounters cnt = { 0, 0, 0, 0, 0, 0 };
	bool lane = i < count;
	float4 o = make_float4(0.f, 0.f, 0.f, 0.f), d = make_float4(1.f, 0.f, 0.f, 0.f);
	if (lane) { o = rayO[i]; d = rayD[i]; }
	HitRecord hit;
	bool found = TraceScene<ANY, COUNT, FAST, INST, MASK>(sc, f3(o.x, o.y, o.z), f3(d.x, d.y, d.z), o.w, hit, stackMem + threadIdx.x, AGPT_TRACE_THREADS, cnt, lane, mk);
	if (lane) {
		agpt_hit h;
		h.found = found ? 1u : 0u;
		h.prim = (found && !ANY) ? hit.prim : -1;
		h.tri = -1;
		if (found && !ANY && hit.slot >= 0) h.tri = MeshOfPrim<INST>(sc, sc.prims[hit.prim]).ids[hit.slot];
		h.t = (found && !ANY) ? hit.t : 0.f;
		out[i] = h;
	}
	if (COUNT) FlushCounters(cnt, lane, counters, nullptr);
}
template <bool ANY, bool COUNT, bool FAST, bool INST>
__global__ void __launch_bounds__(AGPT_TRACE_THREADS) k_trace_table(DScene sc, const float4* __restrict__ rayO, const float4* __restrict__ rayD,
		int count, agpt_hit* out, unsigned long long* counters) {
	__shared__ unsigned stackMem[AGPT_STACK_SMEM * AGPT_TRACE_THREADS];
	TraceTable<ANY, COUNT, FAST, INST, false>(sc, rayO, rayD, count, out, counters, stackMem, DMaskTables());
}

// EXTENSION: alpha masks (agpt.h agpt_upload_alpha_masks).  The three trace kernels with the mask test, run only while some
// mask is bound; INST is always on (its path is also right for scenes without instances), which keeps the count at 4 + 4 + 8.
#ifndef AGPT_MASK_MIN_BLOCKS
#define AGPT_MASK_MIN_BLOCKS AGPT_TRACE_MIN_BLOCKS   // they spill a little under it, yet 8 (fewer spills) measured 10-12 % slower (DESIGN.md section 10)
#endif
template <bool COUNT, bool FAST>
__global__ void __launch_bounds__(AGPT_TRACE_THREADS, AGPT_MASK_MIN_BLOCKS) k_trace_closest_masked(DScene sc, PathState ps, const int* __restrict__ queue,
		const int* __restrict__ countPtr, unsigned long long* counters, unsigned long long* waveRow, DMaskTables mk) {
	__shared__ unsigned stackMem[AGPT_STACK_SMEM * AGPT_TRACE_THREADS];
	TraceClosest<COUNT, FAST, true, true>(sc, ps, queue, countPtr, counters, waveRow, stackMem, mk);
}
template <bool COUNT, bool FAST>
__global__ void __launch_bounds__(AGPT_TRACE_THREADS, AGPT_MASK_MIN_BLOCKS) k_trace_any_masked(DScene sc, PathState ps, const int* __restrict__ queue,
		const int* __restrict__ countPtr, unsigned long long* counters, unsigned long long* waveRow, DMaskTables mk) {
	__shared__ unsigned stackMem[AGPT_STACK_SMEM * AGPT_TRACE_THREADS];
	TraceAny<COUNT, FAST, true, true>(sc, ps, queue, countPtr, counters, waveRow, stackMem, mk);
}
template <bool ANY, bool COUNT, bool FAST>
__global__ void __launch_bounds__(AGPT_TRACE_THREADS) k_trace_table_masked(DScene sc, const float4* __restrict__ rayO, const float4* __restrict__ rayD,
		int count, agpt_hit* out, unsigned long long* counters, DMaskTables mk) {
	__shared__ unsigned stackMem[AGPT_STACK_SMEM * AGPT_TRACE_THREADS];
	TraceTable<ANY, COUNT, FAST, true, true>(sc, rayO, rayD, count, out, counters, stackMem, mk);
}

// ---- shade -------------------------------------------------------------------------------
struct ShadeParams {
	const int* count;     // entries in the survivor list (this wave), on the device
	int max_depth;
	int rr_depth_arg;     // the `depth` argument of Li (integrator.h:124,181)
	int rr_by_bounce;     // AGPT_FLAG_RR_BY_BOUNCE: roulette keyed on the bounce index instead (extension)
	int exact_counts;     // AGPT_FLAG_COUNTERS: rays_mis_culled must be exact, so no MIS sample is dropped before its BSDF value is known
};

// EXTENSION: emissive materials (agpt.h agpt_upload_emission).  E of the closest hit of `path` on primitive `prim`, or false
// when its material does not emit (null materials never do).  The uv is the one k_shade_b's surface helpers give: SphereSurface;
// PlaneUV at O + t * D, the point PlaneSurface builds; a triangle's TriangleUVs and BaryUV, as in TriangleSurface (instances: their
// mesh's uvs and the object-space barycentrics).  The 16-byte row is read only here, at a hit.
__device__ __forceinline__ bool EmissionAt(const DScene& sc, const PathState& ps, const DEmitTables& em, int path, const agpt_prim& prim, float4 h,
		float3& E) {
	if (prim.material < 0) return false;
	AGPT_CHECK(prim.material < em.nRows, AGPT_DBG_EMIT, prim.material);
	const float4 r = __ldg(reinterpret_cast<const float4*>(em.rows + prim.material));
	E = f3(r.y, r.z, r.w);
	if (!(E.x > 0.f || E.y > 0.f || E.z > 0.f)) return false;
	const int tex = __float_as_int(r.x);
	if (tex < 0) return true;
	float2 uv;
	if (prim.type == AGPT_PRIM_SPHERE || prim.type == AGPT_PRIM_PLANE) {
		const float4 o4 = ps.rayO[path], d4 = ps.rayD[path];
		const float3 O = f3(o4.x, o4.y, o4.z), D = f3(d4.x, d4.y, d4.z);
		if (prim.type == AGPT_PRIM_SPHERE) { DSurface si; SphereSurface(sc.spheres[prim.payload], O, D, h.x, si, &uv); }
		else uv = PlaneUV(sc.planes[prim.payload], O + h.x * D);
	}
	else {
		const DMesh& mesh = sc.meshes[prim.type == AGPT_PRIM_INSTANCE ? sc.instances[prim.payload].mesh : prim.payload];
		float2 uv0, uv1, uv2;
		TriangleUVs(mesh, ps.hitSlot[path], uv0, uv1, uv2);
		uv = BaryUV(h.y, h.z, uv0, uv1, uv2);
	}
	E = E * TexLookup(em.tt, tex, uv);
	return true;
}

// ENV: the scene has an InfiniteAreaLight; scenes without one run the leaner instantiation.
//
// Shade is two kernels.  Most entries of the active list need almost no work: their path left
// the scene, hit max depth or only waited for its last next-event estimate (cfg 3, second wave:
// 2 of 3).  Shading them in place would leave the expensive part -- light sampling and three
// BSDF evaluations -- running on a third of each warp.
//   k_shade_a  one thread per active entry, small and memory-bound: folds the previous vertex's
//              NEE into L, adds emission, finishes the paths that end here and appends the
//              SURVIVORS (paths with a surface to shade) to a dense list;
//   k_shade_b  one thread per survivor: phases B..E.
// (A single kernel with the survivors compacted through a shared-memory ring was measured too:
// per-block rings with two barriers per round -22 % shade on cfg 3 but +10 % in closed rooms;
// per-warp rings without barriers desynchronise the warps and stall on instruction fetch.)
//
// EMIT (extension, emissive materials): the body also adds the emission of the hit's material at every vertex (EmissionAt).
// k_shade_a is <ENV, false>; k_shade_a_emit, run only while an emitting row is bound, is <ENV, true>.  tid is threadIdx.x as
// the entry points read it: there the compiler knows its range from their launch bound, and the survivor append's shared-memory
// indexing stays what it was.
template <bool ENV, bool EMIT>
__device__ __forceinline__ void ShadeA(const DScene& sc, const PathState& ps, const int* __restrict__ active, const int* __restrict__ activeCount,
		int* __restrict__ survivors, int* survivorCount, int max_depth, const DEmitTables& em, unsigned tid) {
	const int i = blockIdx.x * blockDim.x + tid;
	int path = active[i];              // unconditional (allocation slack), overlaps with the count load
	const bool valid = i < *activeCount;
	if (!valid) path = 0;
	AGPT_CHECK(path >= 0 && path < ps.slots, AGPT_DBG_PATH, path);
	bool survive = false;
	if (valid) {
		// (loading the NEE terms unconditionally, to save the dependent round trip, measured slower:
		// the kernel then moves ~60 B more per entry and it is those bytes that cost)
		uint32_t flags = ps.flags[path];
		const uint32_t flags0 = flags;
		float4 h = ps.hitA[path];
		float4 L4 = ps.L[path];
		float3 L = f3(L4.x, L4.y, L4.z);
		const float lightSelPdf = sc.n_lights > 0 ? 1.f / sc.n_lights : 0.f;

		// (1) fold in the next-event estimate of the previous vertex (integrator.h:53-58,80-88,104,166)
		if (flags & (PF_NEE_SHADOW | PF_NEE_MIS)) {
			float3 Ld = f3(0.f);
			if ((flags & PF_NEE_SHADOW) && !ps.shadowOccluded[path]) {
				float4 t = ps.neeLight[path];
				Ld += f3(t.x, t.y, t.z);
			}
			if (flags & PF_NEE_MIS) {
				float4 t = ps.neeMis[path];
				int lightIdx = __float_as_int(t.w);
				int misHit = ps.misPrim[path];
				bool lit;
				if (misHit >= 0) lit = sc.prims[misHit].area_light == lightIdx;            // lightIsect.shape->GetAreaLight() == &light
				else lit = sc.lights[lightIdx].type != AGPT_LIGHT_AREA;                 // light.Le(ray): only infinite lights emit
				if (lit) Ld += f3(t.x, t.y, t.z);      // the term already carries Li (a black Li adds zero, like upstream's skip)
			}
			float4 nb = ps.neeBeta[path];
			L += f3(nb.x, nb.y, nb.z) * (Ld / lightSelPdf);
			flags &= ~(PF_NEE_SHADOW | PF_NEE_MIS);
		}

		if (!(flags & PF_NO_CONTINUE)) {
			// (2) the new vertex: did the ray hit, and is there emission to add (integrator.h:139-147)
			int hitPrim = __float_as_int(h.w);
			AGPT_CHECK(hitPrim < sc.n_prims, AGPT_DBG_PRIM, hitPrim);
			bool found = hitPrim >= 0;
			int bounces = (int)(flags >> PF_BOUNCE_SHIFT);
			if (bounces == 0 || (flags & PF_SPECULAR)) {
				float4 b4 = ps.beta[path];
				float3 beta = f3(b4.x, b4.y, b4.z);
				if (found) {
					int al = sc.prims[hitPrim].area_light;
					if (al >= 0) L += beta * f3(sc.lights[al].lemit);
					else L += beta * f3(0.f);
				}
				else {
					for (int l = 0; l < sc.n_lights; l++) {
						if (sc.lights[l].type == AGPT_LIGHT_UNIFORM_INFINITE) L += beta * f3(sc.lights[l].lemit);
						else if (ENV && sc.lights[l].type == AGPT_LIGHT_INFINITE_AREA) {
							float4 d4 = ps.rayD[path];
							L += beta * EnvLe(sc, f3(d4.x, d4.y, d4.z));
						}
					}
				}
			}
			// (2b) emissive materials (extension): at every hit, after the area-light / sky term, before the max-depth end
			if (EMIT && found) {
				float3 E;
				if (EmissionAt(sc, ps, em, path, sc.prims[hitPrim], h, E)) {
					float4 b4 = ps.beta[path];
					L += f3(b4.x, b4.y, b4.z) * E;
				}
			}
			survive = found && bounces < max_depth;     // integrator.h:150
		}
		if (!survive) ps.Lout[path] = make_float4(L.x, L.y, L.z, 0.f);      // the path is complete
		else {
			ps.L[path] = make_float4(L.x, L.y, L.z, 0.f);
			if (flags != flags0) ps.flags[path] = flags;
		}
	}
	// append the survivors: one atomic per BLOCK (a million same-address atomics per launch, one
	// per warp, are what the kernel would otherwise wait for), order inside the block kept
	__shared__ int warpBase[8];
	__shared__ int blockBase;
	const int lane = tid & 31, warp = tid >> 5;
	const unsigned m = __ballot_sync(0xffffffffu, survive);
	if (lane == 0) warpBase[warp] = __popc(m);
	__syncthreads();
	if (tid == 0) {
		int total = 0;
		for (int w = 0; w < 8; w++) { int c = warpBase[w]; warpBase[w] = total; total += c; }
		blockBase = total ? atomicAdd(survivorCount, total) : 0;
	}
	__syncthreads();
	if (survive) survivors[blockBase + warpBase[warp] + __popc(m & ((1u << lane) - 1u))] = path;
}
template <bool ENV>
__global__ void __launch_bounds__(256) k_shade_a(DScene sc, PathState ps, const int* __restrict__ active, const int* __restrict__ activeCount,
		int* __restrict__ survivors, int* survivorCount, int max_depth) {
	ShadeA<ENV, false>(sc, ps, active, activeCount, survivors, survivorCount, max_depth, DEmitTables(), threadIdx.x);
}
template <bool ENV>
__global__ void __launch_bounds__(256) k_shade_a_emit(DScene sc, PathState ps, const int* __restrict__ active, const int* __restrict__ activeCount,
		int* __restrict__ survivors, int* survivorCount, int max_depth, DEmitTables em) {
	ShadeA<ENV, true>(sc, ps, active, activeCount, survivors, survivorCount, max_depth, em, threadIdx.x);
}

// The kernel is ~100 KB of SASS (IEEE division / sqrt sequences, double-precision sincos), far
// more than the instruction cache holds, so it matters that the resident warps walk the same
// code at roughly the same time: one large block per SM (measured, cfg 3 / cfg 5 shade ms per
// 4 spp: 128-thread blocks 11.5 / 22.4, 512-thread blocks 9.9 / 20.9; 768 threads at 80
// registers another -7 % / -3 %).
#ifndef AGPT_SHADE_THREADS
#define AGPT_SHADE_THREADS 768
#endif
#ifndef AGPT_SHADE_MIN_BLOCKS
#define AGPT_SHADE_MIN_BLOCKS 1
#endif
// SHAPES instantiation: traversal-stack entries per thread in shared memory for the light-only walk of a mesh light (the
// rest in local memory, as in the trace kernels).  8 x 768 threads = 24 KB: emissive meshes are small, their trees shallow.
#define AGPT_SHADE_STACK_SMEM 8

// SHAPES (extension): some area light samples its plane or mesh (AGPT_LIGHT_SAMPLE_SHAPE); other scenes run the
// instantiations without that code.  TEX (extension): 1, some Disney material has an image texture on its base colour
// (agpt_upload_textures): two instantiations run, <false, false, false, 1> and <true, true, true, 1>; `tt` is read only by
// them (the others take it last, after every parameter they had before, and their code is what it was).  2, some Disney
// material has a roughness-metallic or normal map (agpt_upload_material_textures): <false, false, false, 2> and
// <true, true, true, 2> shade with the hit's own material record, built once per vertex before the BSDF frame.
template <bool ENV, bool GLASS, bool SHAPES, int TEX>
__global__ void __launch_bounds__(AGPT_SHADE_THREADS, AGPT_SHADE_MIN_BLOCKS) k_shade_b(DScene sc, DShapeTables st, PathState ps, const int* __restrict__ survivors, WaveQueues qout, ShadeParams sp,
		RayCounters* rc, DTexTables tt) {
	__shared__ unsigned shapeStack[SHAPES ? AGPT_SHADE_STACK_SMEM * AGPT_SHADE_THREADS : 1];
	const int lane = threadIdx.x & 31;
	const int count = *sp.count;
	// one block-sized piece of the list per block, no loop: warps that start together stay together
	for (int base = blockIdx.x * AGPT_SHADE_THREADS; base < count; base = count) {
		const int i = base + threadIdx.x;
		const bool valid = i < count;
		int path = 0;
		uint32_t flags = 0;
		float3 beta = f3(0.f);
		float4 o4 = make_float4(0.f, 0.f, 0.f, 0.f), d4 = o4, h = o4;
		int hitSlot = 0;
		uint32_t rng = 0;
		if (valid) {
			path = survivors[i];
			AGPT_CHECK(path >= 0 && path < ps.slots, AGPT_DBG_PATH, path);
			flags = ps.flags[path];
			o4 = ps.rayO[path]; d4 = ps.rayD[path]; h = ps.hitA[path];
			float4 b4 = ps.beta[path];
			hitSlot = ps.hitSlot[path]; rng = ps.rng[path];        // (requested now: one round trip for all per-path state)
			beta = f3(b4.x, b4.y, b4.z);
		}
		const float3 O = f3(o4.x, o4.y, o4.z), D = f3(d4.x, d4.y, d4.z);

		bool emitExtend = false, emitShadow = false, emitMis = false, stayActive = false, skipRay = false, misCulled = false, tailCulled = false;
		int keyExtend = 0, keyMis = 0, keyShadow = 0;
		bool finished = false, full = false;
		bool specularBounce = flags & PF_SPECULAR;
		int bounces = (int)(flags >> PF_BOUNCE_SHIFT);
		DSurface si;
		si.p = f3(0.f); si.n = f3(0.f); si.sn = f3(0.f); si.sdpdu = f3(0.f);
		const agpt_material* mat = sc.mats;      // (never null: agpt keeps one dummy record resident when the scene has no materials)
		float2 uv = make_float2(0.f, 0.f);       // TEX: surface uv of the hit
		TexColors tc;                            // TEX: the hit's diffuse reflectance and Schlick R0
		tc.diffuse = f3(0.f); tc.spec0 = f3(0.f);
		float3 dpdu = f3(0.f), dpdv = f3(0.f);   // TEX == 2: dp/du, dp/dv of the uv (normal maps)
		agpt_material hm;                        // TEX == 2: the hit's material record; idle lanes keep the first record
		if (TEX == 2) hm = sc.mats[0];

		// the surface at the hit (a survivor has one); null materials pass straight through
		if (valid) {
			AGPT_CHECK(__float_as_int(h.w) >= 0 && __float_as_int(h.w) < sc.n_prims, AGPT_DBG_PRIM, __float_as_int(h.w));
			agpt_prim prim = sc.prims[__float_as_int(h.w)];
			// SurfaceInteraction of the closest hit
			if (prim.type == AGPT_PRIM_SPHERE) SphereSurface(sc.spheres[prim.payload], O, D, h.x, si, TEX ? &uv : nullptr, TEX == 2 ? &dpdu : nullptr, TEX == 2 ? &dpdv : nullptr);
			else if (prim.type == AGPT_PRIM_PLANE) PlaneSurface(O, D, h.x, si);
			else if (prim.type == AGPT_PRIM_INSTANCE) {          // extension: a placed mesh
				const agpt_instance& in = sc.instances[prim.payload];
				TriangleSurface(sc.meshes[in.mesh], hitSlot, O, D, h.x, h.y, h.z, si, &in, TEX ? &uv : nullptr, TEX == 2 ? &dpdu : nullptr, TEX == 2 ? &dpdv : nullptr);
			}
			else TriangleSurface(sc.meshes[prim.payload], hitSlot, O, D, h.x, h.y, h.z, si, nullptr, TEX ? &uv : nullptr, TEX == 2 ? &dpdu : nullptr, TEX == 2 ? &dpdv : nullptr);
			if (TEX && prim.type == AGPT_PRIM_PLANE) { uv = PlaneUV(sc.planes[prim.payload], si.p); dpdu = f3(1.f, 0.f, 0.f); dpdv = f3(0.f, 0.f, 1.f); }

			if (prim.material < 0) {
				// null material: pass straight through, bounce count unchanged (integrator.h:152-161)
				DRay nr = MakeRay(si.p + AGPT_EPSILON * D, D);
				ps.rayO[path] = make_float4(nr.O.x, nr.O.y, nr.O.z, nr.t);
				ps.rayD[path] = make_float4(nr.D.x, nr.D.y, nr.D.z, 0.f);
				emitExtend = true; skipRay = true; stayActive = true;
				keyExtend = RayBucket(sc, nr.O, nr.D, -1, true);
			}
			else {
				full = true; mat = sc.mats + prim.material;
				if (TEX == 1) tc = HitColors(tt, prim.material, *mat, uv);     // the one lookup of this vertex
				if (TEX == 2) hm = HitMaps(tt, prim.material, *mat, uv, dpdu, dpdv, si);   // the lookups of this vertex
			}
		}
		if (TEX == 2) mat = &hm;

		// ================= phase B: BSDF frame, random numbers, light sample =================
		const float3 wo = -D;
		VertexBsdf vb;
		bool doNee = false;
		int numLight = 0;
		float2 uLight = make_float2(0, 0), uScattering = make_float2(0, 0), u = make_float2(0, 0);
		float3 wiL = f3(0.f), Li = f3(0.f), lemit = f3(0.f);
		float lightPdf = 0;
		DRay vis;
		vis.O = f3(0.f); vis.D = f3(0.f); vis.t = 0.f;
		int lightType = -1, lightPrimType = -1, lightPayload = 0;
		bool lightShape = false;          // SHAPES: the chosen light samples its plane or mesh
		VertexBsdfInit<GLASS>(vb, si, mat, wo);       // cheap enough to run unconditionally (keeps vb defined for idle threads)
		if (full) {
			doNee = !BSDF_IsPerfectlySpecular(vb.b) && sc.n_lights > 0;
			// ---- all RNG draws of this vertex up to the BSDF sample, in the reference's order ----
			// UniformSampleOneLight (integrator.h:95-105): light pick, uLight, uScattering
			// (float2 arguments are evaluated right to left: .y first), then the extra draws the
			// infinite lights' Sample_Li make (lights.cpp:15-24,50-55), then u (:171).
			if (doNee) {
				int nLights = sc.n_lights;
				numLight = min((int)(RandomFloat(rng) * nLights), nLights - 1);
				uLight.y = RandomFloat(rng); uLight.x = RandomFloat(rng);
				uScattering.y = RandomFloat(rng); uScattering.x = RandomFloat(rng);
				const agpt_light& light = sc.lights[numLight];
				lemit = f3(light.lemit);
				lightType = light.type;
				if (lightType == AGPT_LIGHT_AREA) {
					// AreaLight::Sample_Li (lights.cpp:115-126); upstream can sample spheres only, the extension planes and meshes
					const agpt_prim& lp = sc.prims[light.prim];
					lightPrimType = lp.type; lightPayload = lp.payload;
					lightShape = SHAPES && lp.type != AGPT_PRIM_SPHERE && (light.flags & AGPT_LIGHT_SAMPLE_SHAPE);
					if (lp.type == AGPT_PRIM_SPHERE || lightShape) {
						float3 pS, nS;
						if (lp.type == AGPT_PRIM_SPHERE) SphereSampleFrom(sc.spheres[lp.payload], si.p, uLight, &pS, &nS, &lightPdf);
						else ShapeSampleFrom(sc, st, numLight, lp, si.p, uLight, &pS, &nS, &lightPdf);
						if (lightPdf == 0 || sqrLength(pS - si.p) == 0) lightPdf = 0;
						else {
							wiL = pS - si.p;
							float dist = length(wiL);
							wiL /= dist;
							vis = MakeRay(si.p + AGPT_EPSILON * wiL, wiL, dist - 10 * AGPT_EPSILON);
							Li = lemit;
						}
					}
				}
				else if (ENV && lightType == AGPT_LIGHT_INFINITE_AREA) {
					// InfiniteAreaLight::Sample_Li (lights.cpp:50-90): ignores u, one extra draw;
					// the visibility ray starts EPSILON along the GEOMETRIC normal
					float u01 = RandomFloat(rng);
					if (EnvSampleLi(sc, u01, &wiL, &lightPdf)) {
						vis = MakeRay(si.p + AGPT_EPSILON * si.n, wiL);
						Li = EnvLe(sc, vis.D);
					}
				}
				else {
					// UniformInfiniteLight::Sample_Li: RandomInHemisphere(shading.n), pdf 1/2pi
					float a = 1 - 2 * RandomFloat(rng);
					float b = sqrtf(1 - a * a);
					float phi = 2 * AGPT_PI * RandomFloat(rng);
					float sphi, cphi;
					rsincos(phi, &sphi, &cphi);
					float3 v = f3(1.f * b * cphi, 1.f * b * sphi, 1.f * a);
					if (dot(v, si.sn) < 0) v = -v;
					wiL = v;
					lightPdf = AGPT_INV2PI;
					vis = MakeRay(si.p + AGPT_EPSILON * wiL, wiL);
					Li = lemit;
				}
			}
			u.y = RandomFloat(rng); u.x = RandomFloat(rng);
		}
		const bool evalLight = doNee && lightPdf > 0 && !IsBlack(Li);

		// ================= phase C: sample the MIS and the continuation directions =================
		// Everything a vertex carries between the phases stays in REGISTERS: the two loops below are
		// not unrolled (one copy of the sampling and of the evaluation code, as with an out-of-line
		// function) but their bodies are inlined and their results land in named variables through
		// selects, not in arrays indexed by the loop counter -- those, and structs passed by reference
		// to out-of-line functions, live in local memory, and local stores go through to L2 (ncu,
		// first wave, before: 1.85 KB of L2 traffic and 380 B of DRAM writes per vertex).
		DirSample smpMis, smpCont;
		smpMis.ok = false; smpMis.lobe = 0; smpMis.matching = 0; smpMis.pdf = 0; smpMis.wi = f3(0.f); smpMis.fSpec = f3(0.f);
		smpCont = smpMis;
	#pragma unroll 1
		for (int k = 0; k < 2; k++) {
			bool want = full && (k == 0 ? doNee : true);
			if (want) {
				DirSample s;
				SampleLobeDir<GLASS>(vb, k == 0 ? uScattering : u, k == 0, s);
				if (k == 0) smpMis = s; else smpCont = s;
			}
		}

		// The BSDF-strategy sample of EstimateDirect (integrator.h:62-90) matters only if its ray can end on the chosen
		// light: a sphere light's ray must meet that sphere (the exact MIS cull of phase E: Sphere::Intersect with the
		// largest possible ray.t), a uniform sky needs Pdf_Li != 0 (lights.cpp:26-28).  Where it cannot, the BSDF value at
		// that direction -- one of this vertex's three evaluations -- is never used, and is not computed.  (With
		// AGPT_FLAG_COUNTERS it is: whether the reference would have traced the ray depends on that value being non-black.)
		// A sampled plane / mesh light's Pdf_Li is exact for the same reason the sky's is: it depends on the direction only.  It is
		// the light-only intersection phase E needs as the MIS pdf, taken here by the whole warp (the mesh walk votes).
		float shapeLp = 0.f;
		if (SHAPES) {
			const bool q = full && doNee && smpMis.ok && lightShape;
			shapeLp = ShapePdfLi<AGPT_SHADE_STACK_SMEM>(sc, st, numLight, si.p, q ? LocalToWorld(vb.b, smpMis.wi) : f3(0.f, 1.f, 0.f), shapeStack + threadIdx.x,
				AGPT_SHADE_THREADS, q);
		}
		bool misUseful = true;
		if (full && doNee && smpMis.ok && !sp.exact_counts) {
			const float3 wim = LocalToWorld(vb.b, smpMis.wi);
			if (lightType == AGPT_LIGHT_AREA) {
				misUseful = false;
				if (lightPrimType == AGPT_PRIM_SPHERE) {
					const DRay mr = MakeRay(si.p + AGPT_EPSILON * wim, wim);
					float tLight;
					misUseful = SphereTest(sc.spheres[lightPayload], mr.O, mr.D, mr.t, tLight);
				}
				else if (SHAPES && lightShape) misUseful = shapeLp != 0;
			}
			else if (!(ENV && lightType == AGPT_LIGHT_INFINITE_AREA)) misUseful = dot(si.n, wim) > 0;
		}
		const bool misDropped = full && doNee && smpMis.ok && !misUseful;

		// ================= phase D: one evaluator, three directions (light, MIS, continuation) =================
		float3 fLight = f3(0.f), fMis = f3(0.f), fCont = f3(0.f);
		float pdfLight = 0.f, pdfMis = 0.f, pdfCont = 0.f;
		float3 wiMis = f3(0.f), wiCont = f3(0.f);
	#pragma unroll 1
		for (int k = 0; k < 3; k++) {
			const bool sampledOk = k == 1 ? smpMis.ok : smpCont.ok;
			const int sampledLobe = k == 1 ? smpMis.lobe : smpCont.lobe;
			const float3 sampledWi = k == 1 ? smpMis.wi : smpCont.wi;
			bool sampled = k > 0 && sampledOk;
			bool need = full && (k == 0 ? (evalLight && vb.woOk) : (sampled && sampledLobe != AGPT_LOBE_SPECULAR && (k == 2 || misUseful)));
			float3 wiLoc = k == 0 ? WorldToLocal(vb.b, wiL) : sampledWi;
			LobeEval ev;
			ev.f = f3(0.f); ev.pdfCos = 0.f; ev.pdfMicro = 0.f; ev.fT = f3(0.f); ev.pdfT = 0.f;
			if (need) EvalLobes<GLASS, TEX == 1>(vb, wiLoc, ev, tc);
			if (k == 0) {
				if (need) fLight = FinishEval<GLASS>(vb, ev, wiL, &pdfLight);     // BSDF::f and BSDF::Pdf at the light direction
			}
			else if (full && sampled) {
				float3 w = LocalToWorld(vb.b, sampledWi);
				float p = 0.f;
				float3 f = FinishSample<GLASS>(vb, k == 1 ? smpMis : smpCont, ev, w, &p);
				if (k == 1) { wiMis = w; fMis = f; pdfMis = p; } else { wiCont = w; fCont = f; pdfCont = p; }
			}
		}

		// ================= phase E: EstimateDirect terms, throughput, next rays =================
		if (full) {
			// (3) EstimateDirect (integrator.h:38-93)
			if (doNee) {
				float scatteringPdf = 0;
				if (evalLight) {
					float3 f = fLight * absdot(wiL, si.sn);
					scatteringPdf = pdfLight;
					if (!IsBlack(f)) {
						float weight = PowerHeuristic(1, lightPdf, 1, scatteringPdf);
						float3 term = f * Li * weight / lightPdf;
						ps.neeLight[path] = make_float4(term.x, term.y, term.z, 0.f);
						ps.shO[path] = make_float4(vis.O.x, vis.O.y, vis.O.z, vis.t);
						ps.shD[path] = make_float4(vis.D.x, vis.D.y, vis.D.z, 0.f);
						emitShadow = true;
						keyShadow = RayBucket(sc, vis.O, vis.D, lightType == AGPT_LIGHT_AREA ? numLight : -1, false, vis.t);
					}
				}
				// (a dropped sphere-light sample counts as a culled ray -- an upper bound without AGPT_FLAG_COUNTERS, since a black
				// BSDF value would not have been traced upstream either; a sky sample with Pdf_Li == 0 is no ray upstream)
				if (misDropped) misCulled = lightType == AGPT_LIGHT_AREA && lightPrimType == AGPT_PRIM_SPHERE;
				else if (smpMis.ok) {
					float3 wim = wiMis;
					float3 f = fMis;
					scatteringPdf = pdfMis;
					f *= absdot(wim, si.sn);
					if (!IsBlack(f) && scatteringPdf > 0) {
						float lp;
						if (lightType == AGPT_LIGHT_AREA) lp = lightPrimType == AGPT_PRIM_SPHERE ? SpherePdfFrom(sc.spheres[lightPayload], si.p) : (SHAPES && lightShape) ? shapeLp : 0.f;
						else if (ENV && lightType == AGPT_LIGHT_INFINITE_AREA) lp = EnvPdfLi(sc, wim);
						else lp = dot(si.n, wim) > 0 ? AGPT_INV2PI : 0.f;       // lights.cpp:26-28 (geometric n)
						if (lp != 0) {
							float weight = PowerHeuristic(1, scatteringPdf, 1, lp);
							DRay mr = MakeRay(si.p + AGPT_EPSILON * wim, wim);
							// radiance the MIS ray returns if it reaches this light (integrator.h:81-87)
							float3 LiMis = (ENV && lightType == AGPT_LIGHT_INFINITE_AREA) ? EnvLe(sc, mr.D) : lemit;
							float3 term = f * LiMis * weight / scatteringPdf;
							// An area light's MIS ray only ever contributes if its closest hit IS the light's
							// shape (integrator.h:82-85).  If the ray misses that sphere outright -- the very
							// Sphere::Intersect test Scene::Intersect would run, with the largest possible
							// ray.t -- nothing it could hit matters, so it is not traced.  Same result, far
							// fewer closest-hit rays for small or distant lights (Sphere::Pdf never checks
							// that wi points at the sphere, intersectable.h:306-317, so upstream traces them all).  A sampled plane / mesh
							// light's ray met the shape already (lp != 0).
							float tLight;
							bool canReachLight = lightType != AGPT_LIGHT_AREA || (SHAPES && lightShape) || SphereTest(sc.spheres[lightPayload], mr.O, mr.D, mr.t, tLight);
							misCulled = !canReachLight;
							ps.neeMis[path] = make_float4(term.x, term.y, term.z, __int_as_float(numLight));
							ps.misO[path] = make_float4(mr.O.x, mr.O.y, mr.O.z, mr.t);
							ps.misD[path] = make_float4(mr.D.x, mr.D.y, mr.D.z, 0.f);
							if (canReachLight) {
								emitMis = true;
								keyMis = RayBucket(sc, mr.O, mr.D, -1, true);
							}
						}
					}
				}
				if (emitShadow || emitMis) ps.neeBeta[path] = make_float4(beta.x, beta.y, beta.z, 0.f);
			}

			// (4) the new path direction (integrator.h:169-185)
			float3 wi = wiCont;
			float pdf = pdfCont;
			float3 f = fCont;
			bool sampledSpecular = smpCont.lobe == AGPT_LOBE_SPECULAR;
			bool alive = smpCont.ok && !(IsBlack(f) || pdf == 0);
			if (alive) {
				beta *= f * absdot(wi, si.sn) / pdf;
				specularBounce = sampledSpecular;
				// Russian roulette (integrator.h:179-185): live only if the caller passed depth > 3
				float maxComponent = smax(beta.x, smax(beta.y, beta.z));
				if (maxComponent < 1 && (sp.rr_by_bounce ? bounces : sp.rr_depth_arg) > 3) {
					float q = smax(.05f, 1 - maxComponent);
					if (RandomFloat(rng) < q) alive = false;
					else beta /= 1 - q;
				}
			}
			if (alive) {
				bounces++;
				// the vertex at bounces == max_depth only adds emission, and only after a
				// specular bounce (integrator.h:139,150): otherwise its ray need not be traced
				if (bounces >= sp.max_depth && !specularBounce) { alive = false; tailCulled = true; }
			}
			if (alive) {
				DRay nr = MakeRay(si.p + AGPT_EPSILON * wi, wi);
				ps.rayO[path] = make_float4(nr.O.x, nr.O.y, nr.O.z, nr.t);
				ps.rayD[path] = make_float4(nr.D.x, nr.D.y, nr.D.z, 0.f);
				ps.beta[path] = make_float4(beta.x, beta.y, beta.z, 0.f);
				emitExtend = true; stayActive = true;
				keyExtend = RayBucket(sc, nr.O, nr.D, -1, true);
			}
			else if (emitShadow || emitMis) { flags |= PF_NO_CONTINUE; stayActive = true; }
			else finished = true;
			ps.rng[path] = rng;
			flags = (flags & 0xffu & ~PF_SPECULAR) | (specularBounce ? PF_SPECULAR : 0u) | ((uint32_t)bounces << PF_BOUNCE_SHIFT);
			if (emitShadow) flags |= PF_NEE_SHADOW;
			if (emitMis) flags |= PF_NEE_MIS;
		}
		if (valid) {
			ps.flags[path] = flags;
			if (finished) { float4 Lf = ps.L[path]; ps.Lout[path] = Lf; }       // L was completed by k_shade_a; nothing is added here
		}

		// (5) queue the next wave.  One atomic per queue per BLOCK: the counters are single
		// addresses, and one atomic per warp (a million a launch) serialises in L2 -- measured
		// on k_shade_a: -3 ms per step from this alone.  Every thread of the block gets here.
		__shared__ int warpCount[AGPT_SHADE_THREADS / 32][4];      // extend, MIS, shadow, active; then: offsets
		__shared__ int queueBase[3];
		__shared__ int blockStats[6];
		const int warp = threadIdx.x >> 5;
		const unsigned below = (1u << lane) - 1u;
		const unsigned mE = __ballot_sync(0xffffffffu, emitExtend), mM = __ballot_sync(0xffffffffu, emitMis);
		const unsigned mS = __ballot_sync(0xffffffffu, emitShadow), mA = __ballot_sync(0xffffffffu, stayActive);
		if (threadIdx.x < 6) blockStats[threadIdx.x] = 0;
		if (lane == 0) { warpCount[warp][0] = __popc(mE); warpCount[warp][1] = __popc(mM); warpCount[warp][2] = __popc(mS); warpCount[warp][3] = __popc(mA); }
		__syncthreads();
		if (threadIdx.x < 3) {
			// thread 0: closest queue (a warp's path rays, then its MIS rays), 1: shadow queue, 2: active list
			int total = 0;
			for (int w = 0; w < AGPT_SHADE_THREADS / 32; w++) {
				if (threadIdx.x == 0) {
					int c0 = warpCount[w][0], c1 = warpCount[w][1];
					warpCount[w][0] = total; total += c0;
					warpCount[w][1] = total; total += c1;
				}
				else {
					int c = warpCount[w][threadIdx.x + 1];
					warpCount[w][threadIdx.x + 1] = total; total += c;
				}
			}
			queueBase[threadIdx.x] = total ? atomicAdd(qout.counts + threadIdx.x, total) : 0;
		}
		// ray statistics, first into the block's counters
		const unsigned mSkip = __ballot_sync(0xffffffffu, skipRay), mMc = __ballot_sync(0xffffffffu, misCulled), mTc = __ballot_sync(0xffffffffu, tailCulled);
		if (lane == 0) {
			if (mE) atomicAdd(&blockStats[0], __popc(mE));
			if (mM) atomicAdd(&blockStats[1], __popc(mM));
			if (mS) atomicAdd(&blockStats[2], __popc(mS));
			if (mSkip) atomicAdd(&blockStats[3], __popc(mSkip));
			if (mMc) atomicAdd(&blockStats[4], __popc(mMc));
			if (mTc) atomicAdd(&blockStats[5], __popc(mTc));
		}
		__syncthreads();
		AGPT_CHECK(queueBase[0] + warpCount[warp][1] + __popc(mM) <= 2 * ps.slots && queueBase[1] + warpCount[warp][2] + __popc(mS) <= ps.slots &&
			queueBase[2] + warpCount[warp][3] + __popc(mA) <= ps.slots, AGPT_DBG_QUEUE, queueBase[0]);
		if (emitExtend) { int slot = queueBase[0] + warpCount[warp][0] + __popc(mE & below); qout.closest[slot] = path * 2; qout.keys[slot] = (unsigned short)keyExtend; }
		if (emitMis) { int slot = queueBase[0] + warpCount[warp][1] + __popc(mM & below); qout.closest[slot] = path * 2 + 1; qout.keys[slot] = (unsigned short)keyMis; }
		if (emitShadow) { int slot = queueBase[1] + warpCount[warp][2] + __popc(mS & below); qout.shadow[slot] = path; qout.shadowKeys[slot] = (unsigned short)keyShadow; }
		if (stayActive) { int slot = queueBase[2] + warpCount[warp][3] + __popc(mA & below); qout.active[slot] = path; }

		// ray statistics: one atomic per counter per block
		if (threadIdx.x < 6 && blockStats[threadIdx.x]) {
			unsigned long long* dst = threadIdx.x == 0 ? &rc->rays_closest : threadIdx.x == 1 ? &rc->rays_mis : threadIdx.x == 2 ? &rc->rays_shadow :
				threadIdx.x == 3 ? &rc->rays_skip : threadIdx.x == 4 ? &rc->rays_mis_culled : &rc->rays_tail_culled;
			atomicAdd(dst, (unsigned long long)blockStats[threadIdx.x]);
		}
	}
}

// ---- accumulate: myapp.cpp:169-173 + Accumulator::AddSample (myapp.h:17-19) --------------
// One thread per pixel adds its samples of this batch in ascending sample order, the order
// the reference's successive Ticks add them in.
// MOMENTS (agpt_set_moments): the same filtered sample c also adds c * c per channel to moments.xyz and 1 to moments.w, in the
// same order.  LIST (adaptive rounds): one thread per entry of list[0, listCount), whose samplesInBatch samples sit at
// Lout[entry * samplesInBatch ..] (k_generate<true>); film and moments of pixel list[entry].  <false, false> is agpt_render's.
template <bool MOMENTS, bool LIST>
__global__ void __launch_bounds__(256) k_accumulate(const float4* __restrict__ Lout, float4* accum, int width, int height, int samplesInBatch,
		float4* moments = nullptr, const int* __restrict__ list = nullptr, int listCount = 0, int maxSamples = 0) {
	int pixel = blockIdx.x * blockDim.x + threadIdx.x;
	int wh = width * height;
	size_t slot;
	if constexpr (LIST) {
		if (pixel >= listCount) return;
		slot = (size_t)pixel * samplesInBatch;
		pixel = list[pixel];
		AGPT_CHECK(pixel >= 0 && pixel < wh, AGPT_DBG_LIST, pixel);
	}
	else if (pixel >= wh) return;
	int x = pixel % width, y = pixel / width;
	if constexpr (!LIST) slot = (size_t)PixelToSlot(x, y, width, height, true) * samplesInBatch;       // agpt_render generates tiled
	float4* dst = accum + (size_t)(height - 1 - y) * width + x;
	float4 a = *dst;
	float4 m;
	if constexpr (MOMENTS) {
		m = moments[dst - accum];
		AGPT_CHECK(!LIST || (int)m.w + samplesInBatch <= maxSamples, AGPT_DBG_SAMPLE, (int)m.w);
	}
	for (int s = 0; s < samplesInBatch; s++) {
		float4 c = Lout[slot + s];
		float lum = 0.212671f * c.x + 0.715160f * c.y + 0.072169f * c.z;     // Luminance (precomp.h:717)
		if (isnan(c.x) || isnan(c.y) || isnan(c.z) || isinf(lum)) c = make_float4(0.f, 0.f, 0.f, 0.f);
		a.x += c.x; a.y += c.y; a.z += c.z;
		if constexpr (MOMENTS) { m.x += c.x * c.x; m.y += c.y * c.y; m.z += c.z * c.z; m.w += 1.f; }
	}
	*dst = a;
	if constexpr (MOMENTS) moments[dst - accum] = m;
}

// ---- adaptive sampling: the convergence test of agpt_adaptive_select (agpt.h), per pixel ------------------------------
// Film sum a, moments q and count n of one channel; every operation rounded on its own (--fmad=false, IEEE / and sqrt).
// The variance of the channel's mean, v / n (and the mean mu), as the convergence test and the denoiser both estimate it.
__device__ __forceinline__ float ChannelVarianceOfMean(float a, float q, float n, float& mu) {
	mu = a / n;
	float d = q - a * mu;
	float v = d / (n - 1.f);
	v = v < 0.f ? 0.f : v;                      // (a NaN stays NaN)
	return v / n;
}
// True: the channel's standard error is not (yet) within tolerance, or not finite.
__device__ __forceinline__ bool ChannelUnconverged(float a, float q, float n, float tolerance, float floor_) {
	float mu;
	float se = sqrtf(ChannelVarianceOfMean(a, q, n, mu));
	float thr = tolerance * (mu > floor_ ? mu : floor_);
	return !(se <= thr);
}
__device__ __forceinline__ bool PixelSelected(float4 a, float4 q, int maxSamples, int step, float tolerance, float floor_) {
	if (!((long long)q.w + step <= maxSamples)) return false;
	return ChannelUnconverged(a.x, q.x, q.w, tolerance, floor_) || ChannelUnconverged(a.y, q.y, q.w, tolerance, floor_) ||
		ChannelUnconverged(a.z, q.z, q.w, tolerance, floor_);
}
// One thread per pixel, pixels in the tiled slot order of agpt_render (8x4 tiles), so neighbouring list entries are
// neighbouring pixels and a round's warps cover compact patches.  The selected pixels of a block are compacted with
// warp ballots and a shared-memory prefix over the warps, one global atomic per block, as the queue appends of k_shade_b.
__global__ void __launch_bounds__(256) k_adaptive_select(const float4* __restrict__ accum, const float4* __restrict__ moments, int width, int height,
		int maxSamples, int step, float tolerance, float floor_, int* __restrict__ list, int* count) {
	__shared__ int warpCount[8];
	__shared__ int blockBase;
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	bool sel = false;
	int pixel = 0;
	if (i < width * height) {
		int x, y;
		SlotToPixel(i, width, height, true, x, y);
		pixel = y * width + x;
		const size_t f = (size_t)(height - 1 - y) * width + x;
		sel = PixelSelected(accum[f], moments[f], maxSamples, step, tolerance, floor_);
	}
	const unsigned m = __ballot_sync(0xffffffffu, sel);
	if (lane == 0) warpCount[warp] = __popc(m);
	__syncthreads();
	if (threadIdx.x == 0) {
		int total = 0;
		for (int w = 0; w < 8; w++) { int c = warpCount[w]; warpCount[w] = total; total += c; }
		blockBase = total ? atomicAdd(count, total) : 0;
	}
	__syncthreads();
	if (sel) {
		const int at = blockBase + warpCount[warp] + __popc(m & ((1u << lane) - 1u));
		AGPT_CHECK(at >= 0 && at < width * height, AGPT_DBG_LIST, at);
		list[at] = pixel;
	}
}

// ---- resolve: Accumulator::CopyToSurface (myapp.h:34-41) + lin2rgb / rgb2uint (common.h:41-51)
// One pixel of CopyToSurface: pixels / (float)samples -> lin2rgb -> rgb2uint.  powf is glibc's
// (rpowf), so the packed bytes equal the reference's for every float input, not just "within 1 LSB".
// rgb2uint's clamp(clr.x, 0.0, 0.999) resolves to the template's float overload (precomp.h:678):
// fmaxf(0.f, fminf(f, 0.999f)) with the a<b?a:b / a>b?a:b semantics (a NaN channel comes out 255).
__device__ __forceinline__ uint32_t ResolvePixel(float4 a, float samples) {
	const float e = 1 / 2.2f;
	float3 c = f3(rpowf(a.x / samples, e), rpowf(a.y / samples, e), rpowf(a.z / samples, e));
	int r = (int)(256 * rclamp(c.x, 0.0f, 0.999f)), g = (int)(256 * rclamp(c.y, 0.0f, 0.999f)), b = (int)(256 * rclamp(c.z, 0.0f, 0.999f));
	return (uint32_t)((r << 16) + (g << 8) + b);
}
__global__ void __launch_bounds__(256) k_resolve(const float4* __restrict__ accum, uint32_t* out, int n, float samples) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	out[i] = ResolvePixel(accum[i], samples);
}
// agpt_resolve_counts: each pixel divided by its own sample count (moments .w); a pixel without samples resolves to 0
__global__ void __launch_bounds__(256) k_resolve_counts(const float4* __restrict__ accum, const float4* __restrict__ moments, uint32_t* out, int n) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float s = moments[i].w;
	out[i] = s > 0.f ? ResolvePixel(accum[i], s) : 0u;
}

// ---- EXTENSION: denoising (agpt.h agpt_render_guides / agpt_denoise; CPU statements oracle/agpt_guides_oracle.cpp and
// oracle/denoise.py) --------------------------------------------------------------------------------------------------------
// k_guides: one thread per pixel after k_generate<false> (tiled) and k_trace_closest have run the batch's camera rays.  It walks
// the pixel's slots in sample order and adds each sample's first hit to the running sums in albedo (.xyz, .w = hits) and
// normalDepth (.xyz, .w = t sum).  `total` > 0 on the last batch: the sums become the means of all `total` samples.
// TEX (extension): 1, a textured Disney material's albedo is the hit's textured diffuse_r + spec_r0 (k_guides_tex); 2, the
// hit's material record and mapped shading normal of k_shade_b<..., 2> give albedo and normal (k_guides_maps).
template <int TEX>
__device__ __forceinline__ void Guides(DScene sc, DTexTables tt, PathState ps, int samplesInBatch, bool firstBatch, int total, float4* albedo, float4* normalDepth) {
	const int pixel = blockIdx.x * blockDim.x + threadIdx.x;
	const int width = sc.width, height = sc.height;
	if (pixel >= width * height) return;
	const int x = pixel % width, y = pixel / width;
	const size_t f = (size_t)(height - 1 - y) * width + x;
	float4 a = make_float4(0.f, 0.f, 0.f, 0.f), nd = a;
	if (!firstBatch) { a = albedo[f]; nd = normalDepth[f]; }
	const size_t base = (size_t)PixelToSlot(x, y, width, height, true) * samplesInBatch;     // k_generate's tiled slots
	for (int s = 0; s < samplesInBatch; s++) {
		const size_t slot = base + s;
		AGPT_CHECK(slot < (size_t)ps.slots, AGPT_DBG_GUIDE, slot);
		const float4 h = ps.hitA[slot];
		const int hitPrim = __float_as_int(h.w);
		AGPT_CHECK(hitPrim < sc.n_prims, AGPT_DBG_PRIM, hitPrim);
		float3 alb = f3(1.f), n = f3(0.f);
		if (hitPrim >= 0) {
			const float4 o4 = ps.rayO[slot], d4 = ps.rayD[slot];
			const float3 O = f3(o4.x, o4.y, o4.z), D = f3(d4.x, d4.y, d4.z);
			const agpt_prim prim = sc.prims[hitPrim];
			DSurface si;
			float2 uv = make_float2(0.f, 0.f);
			float3 dpdu = f3(0.f), dpdv = f3(0.f);
			agpt_material hm;
			// the surface of the closest hit as k_shade_b rebuilds it
			if (prim.type == AGPT_PRIM_SPHERE) SphereSurface(sc.spheres[prim.payload], O, D, h.x, si, TEX ? &uv : nullptr, TEX == 2 ? &dpdu : nullptr, TEX == 2 ? &dpdv : nullptr);
			else if (prim.type == AGPT_PRIM_PLANE) PlaneSurface(O, D, h.x, si);
			else if (prim.type == AGPT_PRIM_INSTANCE) {
				const agpt_instance& in = sc.instances[prim.payload];
				TriangleSurface(sc.meshes[in.mesh], ps.hitSlot[slot], O, D, h.x, h.y, h.z, si, &in, TEX ? &uv : nullptr, TEX == 2 ? &dpdu : nullptr, TEX == 2 ? &dpdv : nullptr);
			}
			else TriangleSurface(sc.meshes[prim.payload], ps.hitSlot[slot], O, D, h.x, h.y, h.z, si, nullptr, TEX ? &uv : nullptr, TEX == 2 ? &dpdu : nullptr, TEX == 2 ? &dpdv : nullptr);
			if (TEX && prim.type == AGPT_PRIM_PLANE) { uv = PlaneUV(sc.planes[prim.payload], si.p); dpdu = f3(1.f, 0.f, 0.f); dpdv = f3(0.f, 0.f, 1.f); }
			if (TEX == 2 && prim.material >= 0) hm = HitMaps(tt, prim.material, sc.mats[prim.material], uv, dpdu, dpdv, si);
			n = dot(si.sn, D) > 0.f ? -si.sn : si.sn;
			if (prim.material >= 0) {
				const agpt_material& m = sc.mats[prim.material];
				if (m.type == AGPT_MAT_MIRROR) alb = f3(m.mirror_r);
				else if (m.type == AGPT_MAT_GLASS) alb = f3(m.mirror_r) + f3(m.diffuse_r);
				else if (TEX == 2) alb = f3(hm.diffuse_r) + f3(hm.spec_r0);
				else if (TEX) { const TexColors tc = HitColors(tt, prim.material, m, uv); alb = tc.diffuse + tc.spec0; }
				else alb = f3(m.diffuse_r) + f3(m.spec_r0);
				alb = f3(alb.x < 1.f ? alb.x : 1.f, alb.y < 1.f ? alb.y : 1.f, alb.z < 1.f ? alb.z : 1.f);
			}
			a.w += 1.f;
			nd.w += h.x;
		}
		a.x += alb.x; a.y += alb.y; a.z += alb.z;
		nd.x += n.x; nd.y += n.y; nd.z += n.z;
	}
	if (total > 0) {
		const float t = (float)total;
		nd.w = a.w > 0.f ? nd.w / a.w : 0.f;
		a = make_float4(a.x / t, a.y / t, a.z / t, a.w / t);
		nd.x /= t; nd.y /= t; nd.z /= t;
	}
	albedo[f] = a;
	normalDepth[f] = nd;
}
__global__ void __launch_bounds__(256) k_guides(DScene sc, PathState ps, int samplesInBatch, bool firstBatch, int total, float4* albedo, float4* normalDepth) {
	Guides<0>(sc, DTexTables(), ps, samplesInBatch, firstBatch, total, albedo, normalDepth);
}
__global__ void __launch_bounds__(256) k_guides_tex(DScene sc, DTexTables tt, PathState ps, int samplesInBatch, bool firstBatch, int total, float4* albedo, float4* normalDepth) {
	Guides<1>(sc, tt, ps, samplesInBatch, firstBatch, total, albedo, normalDepth);
}
__global__ void __launch_bounds__(256) k_guides_maps(DScene sc, DTexTables tt, PathState ps, int samplesInBatch, bool firstBatch, int total, float4* albedo, float4* normalDepth) {
	Guides<2>(sc, tt, ps, samplesInBatch, firstBatch, total, albedo, normalDepth);
}

// EXTENSION probe (agpt.h agpt_probe_material_maps): for each closest hit of a ray table (k_generate<false> with rays7, then the
// closest-hit trace), the uv, the BSDF frame and the material record of k_shade_b<..., 2>, through the calls that kernel makes.
// out32 per ray: prim (-1: miss), u, v, ng3, ns3, ss3, ts3, T3, B3 (dp/du, dp/dv), roughness, metallic, lobes, diffuse_r3, spec_r03.
__global__ void __launch_bounds__(256) k_probe_material_maps(DScene sc, DTexTables tt, PathState ps, int n, float* out32) {
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	float* o = out32 + 32 * (size_t)i;
	for (int k = 0; k < 32; k++) o[k] = 0.f;
	o[0] = -1.f;
	const float4 h = ps.hitA[i];
	const int hitPrim = __float_as_int(h.w);
	AGPT_CHECK(hitPrim < sc.n_prims, AGPT_DBG_PRIM, hitPrim);
	if (hitPrim < 0) return;
	const float4 o4 = ps.rayO[i], d4 = ps.rayD[i];
	const float3 O = f3(o4.x, o4.y, o4.z), D = f3(d4.x, d4.y, d4.z);
	const agpt_prim prim = sc.prims[hitPrim];
	DSurface si;
	float2 uv = make_float2(0.f, 0.f);
	float3 dpdu = f3(0.f), dpdv = f3(0.f);
	if (prim.type == AGPT_PRIM_SPHERE) SphereSurface(sc.spheres[prim.payload], O, D, h.x, si, &uv, &dpdu, &dpdv);
	else if (prim.type == AGPT_PRIM_PLANE) PlaneSurface(O, D, h.x, si);
	else if (prim.type == AGPT_PRIM_INSTANCE) {
		const agpt_instance& in = sc.instances[prim.payload];
		TriangleSurface(sc.meshes[in.mesh], ps.hitSlot[i], O, D, h.x, h.y, h.z, si, &in, &uv, &dpdu, &dpdv);
	}
	else TriangleSurface(sc.meshes[prim.payload], ps.hitSlot[i], O, D, h.x, h.y, h.z, si, nullptr, &uv, &dpdu, &dpdv);
	if (prim.type == AGPT_PRIM_PLANE) { uv = PlaneUV(sc.planes[prim.payload], si.p); dpdu = f3(1.f, 0.f, 0.f); dpdv = f3(0.f, 0.f, 1.f); }
	agpt_material hm = sc.mats[0];
	if (prim.material >= 0) hm = HitMaps(tt, prim.material, sc.mats[prim.material], uv, dpdu, dpdv, si);
	const DBSDF b = MakeBSDF(si, &hm);
	const float3 rows[6] = { b.ng, b.ns, b.ss, b.ts, dpdu, dpdv };
	o[0] = (float)hitPrim; o[1] = uv.x; o[2] = uv.y;
	for (int k = 0; k < 6; k++) { o[3 + 3 * k] = rows[k].x; o[4 + 3 * k] = rows[k].y; o[5 + 3 * k] = rows[k].z; }
	o[21] = hm.roughness; o[22] = hm.metallic; o[23] = (float)hm.lobes;
	for (int k = 0; k < 3; k++) { o[24 + k] = hm.diffuse_r[k]; o[27 + k] = hm.spec_r0[k]; }
}

#define AGPT_DENOISE_ALBEDO_EPS 0.01f
#define AGPT_DENOISE_LUM_EPS 1e-4f
__device__ __forceinline__ float DenoiseLum(float4 e) { return 0.212671f * e.x + 0.715160f * e.y + 0.072169f * e.z; }
__device__ __forceinline__ float3 DenoiseAlbedo(float4 a) {
	return f3(a.x > AGPT_DENOISE_ALBEDO_EPS ? a.x : AGPT_DENOISE_ALBEDO_EPS, a.y > AGPT_DENOISE_ALBEDO_EPS ? a.y : AGPT_DENOISE_ALBEDO_EPS,
		a.z > AGPT_DENOISE_ALBEDO_EPS ? a.z : AGPT_DENOISE_ALBEDO_EPS);
}
__device__ __forceinline__ bool Finite4(float4 v) { return isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w); }

// k_denoise_prepare: one thread per film pixel.  iterations > 0: the demodulated mean and its luminance variance into E, the
// filter's guide (normal, depth or -1 for a pixel that missed) into G.  iterations == 0 (out != nullptr): the means themselves
// into out and their packed pixels into rgb8.
__global__ void __launch_bounds__(256) k_denoise_prepare(const float4* __restrict__ accum, const float4* __restrict__ moments, const float4* __restrict__ albedo,
		const float4* __restrict__ normalDepth, int n, float4* __restrict__ E, float4* __restrict__ G, float4* __restrict__ out, uint32_t* __restrict__ rgb8) {
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float4 a = accum[i], q = moments[i];
	float3 mu = f3(0.f), var = f3(0.f);
	if (q.w > 0.f) { mu = f3(a.x / q.w, a.y / q.w, a.z / q.w); }
	if (out) {
		const float4 o = make_float4(mu.x, mu.y, mu.z, 0.f);
		out[i] = o;
		rgb8[i] = ResolvePixel(o, 1.f);
		return;
	}
	if (q.w >= 2.f) {
		float m;
		var = f3(ChannelVarianceOfMean(a.x, q.x, q.w, m), ChannelVarianceOfMean(a.y, q.y, q.w, m), ChannelVarianceOfMean(a.z, q.z, q.w, m));
	}
	const float4 alb = albedo[i], nd = normalDepth[i];
	const float3 al = DenoiseAlbedo(alb);
	const float wr = 0.212671f * 0.212671f, wg = 0.715160f * 0.715160f, wb = 0.072169f * 0.072169f;
	const float vl = ((wr * var.x) / (al.x * al.x) + (wg * var.y) / (al.y * al.y)) + (wb * var.z) / (al.z * al.z);
	E[i] = make_float4(mu.x / al.x, mu.y / al.y, mu.z / al.z, vl);
	G[i] = make_float4(nd.x, nd.y, nd.z, alb.w == 0.f ? -1.f : nd.w);
}

// k_denoise_atrous: one a-trous pass at tap spacing `step`, one thread per pixel (a 32 x 8 block covers a film patch).  The 25
// taps are plain loads: neighbouring threads share most of them through L1.  LAST: remodulated by the albedo into out, packed
// into rgb8.
template <bool LAST>
__global__ void __launch_bounds__(256) k_denoise_atrous(const float4* __restrict__ Ein, const float4* __restrict__ G, const float4* __restrict__ albedo, int width, int height,
		int step, float sigmaL, float sigmaZ, int normalPow, float4* __restrict__ Eout, uint32_t* __restrict__ rgb8) {
	const int x = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
	if (x >= width || r >= height) return;
	const int p = r * width + x;
	const float h[5] = { 1.f / 16, 1.f / 4, 3.f / 8, 1.f / 4, 1.f / 16 };
	const float4 ep = Ein[p];
	float4 res = ep;
	if (Finite4(ep)) {
		const float4 gp = G[p];
		const bool missP = gp.w < 0.f;
		const float lp = DenoiseLum(ep);
		const float den = (sigmaL * sigmaL) * ep.w + AGPT_DENOISE_LUM_EPS;
		float sw = 0.f, sv = 0.f;
		float3 se = f3(0.f);
#pragma unroll
		for (int dy = -2; dy <= 2; dy++) {
			const int rq = r + dy * step;
			if (rq < 0 || rq >= height) continue;
#pragma unroll
			for (int dx = -2; dx <= 2; dx++) {
				const int xq = x + dx * step;
				if (xq < 0 || xq >= width) continue;
				const int q = rq * width + xq;
				AGPT_CHECK(q >= 0 && q < width * height, AGPT_DBG_TAP, q);
				const float4 eq = Ein[q];
				if (!Finite4(eq)) continue;
				const float4 gq = G[q];
				const float dl = lp - DenoiseLum(eq);
				const float wl = 1.f / (1.f + (dl * dl) / den);
				float m = gp.x * gq.x + gp.y * gq.y + gp.z * gq.z;
				m = m > 0.f ? m : 0.f;
				for (int k = 0; k < normalPow; k++) m = m * m;
				const bool missQ = gq.w < 0.f;
				const float wz = (missP && missQ) ? 1.f : (missP != missQ) ? 0.f : 1.f / (1.f + fabsf(gp.w - gq.w) / (sigmaZ * gp.w));
				const float w = (((h[dx + 2] * h[dy + 2]) * wl) * m) * wz;
				if (!isfinite(w)) continue;
				sw += w;
				se.x += w * eq.x; se.y += w * eq.y; se.z += w * eq.z;
				sv += (w * w) * eq.w;
			}
		}
		if (sw > 0.f) {
			const float4 e2 = make_float4(se.x / sw, se.y / sw, se.z / sw, sv / (sw * sw));
			if (Finite4(e2)) res = e2;
		}
	}
	if (LAST) {
		const float3 al = DenoiseAlbedo(albedo[p]);
		const float4 o = make_float4(res.x * al.x, res.y * al.y, res.z * al.z, 0.f);
		Eout[p] = o;
		rgb8[p] = ResolvePixel(o, 1.f);
	}
	else Eout[p] = res;
}

// ---- EXTENSION: reprojection of the film and its moments across a camera move (agpt.h agpt_reproject_film; CPU statement
// oracle/reproject.py) -------------------------------------------------------------------------------------------------------
// k_reproject_film: one thread per film pixel (a 32 x 8 block covers a film patch).  Every pixel writes its guide G (normal,
// depth or -1 for a pixel whose guide samples all missed, as k_denoise_prepare builds it) into Gout, the view the next call
// reprojects from.  CARRY: the pixel's centre ray is projected into the saved camera `prev` and the film and moments are
// gathered from the accepted bilinear taps of the old film (accumIn, momentsIn, Gin) into accumOut and momentsOut.
template <bool CARRY>
__global__ void __launch_bounds__(256) k_reproject_film(const float4* __restrict__ accumIn, const float4* __restrict__ momentsIn, const float4* __restrict__ Gin,
		const float4* __restrict__ albedo, const float4* __restrict__ normalDepth, int width, int height, agpt_camera cur, agpt_camera prev,
		float maxHistory, float sigmaDepth, float minNormalDot, float4* __restrict__ accumOut, float4* __restrict__ momentsOut, float4* __restrict__ Gout) {
	const int x = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
	if (x >= width || r >= height) return;
	const int p = r * width + x, y = height - 1 - r;
	const float4 nd = normalDepth[p];
	const float4 gp = make_float4(nd.x, nd.y, nd.z, albedo[p].w == 0.f ? -1.f : nd.w);
	const bool hitP = gp.w >= 0.f;
	Gout[p] = gp;
	if (!CARRY) return;
	const float W = (float)width, Hf = (float)height;
	const float s = (x + 0.5f) / W, t = (y + 0.5f) / Hf;
	const float3 O = f3(cur.origin), O1 = f3(prev.origin), H1 = f3(prev.horizontal), V1 = f3(prev.vertical);
	const float3 D = normalize(((f3(cur.lower_left_corner) + s * f3(cur.horizontal)) + t * f3(cur.vertical)) - O);
	float3 d = D;
	float z = 0.f;
	if (hitP) {
		d = (O + gp.w * D) - O1;
		z = length(d);
	}
	float4 A = make_float4(0.f, 0.f, 0.f, 0.f), Q = A;
	float sw = 0.f;
	const float3 f = ((f3(prev.lower_left_corner) + 0.5f * H1) + 0.5f * V1) - O1;
	const float den = dot(d, f);
	if (den > 0.f) {
		const float lam = dot(f, f) / den;
		const float u = 0.5f + (lam * dot(d, H1)) / dot(H1, H1);
		const float v = 0.5f + (lam * dot(d, V1)) / dot(V1, V1);
		const float px = u * W - 0.5f, py = v * Hf - 0.5f;
		const float x0 = floorf(px), y0 = floorf(py);
		// (a NaN or infinite px / py fails these compares too; within them the tap indices fit an int)
		if (x0 >= -1.f && x0 <= W - 1.f && y0 >= -1.f && y0 <= Hf - 1.f) {
			const float fx = px - x0, fy = py - y0;
			const float wx[2] = { 1.f - fx, fx }, wy[2] = { 1.f - fy, fy };
			const int ix = (int)x0, iy = (int)y0;
#pragma unroll
			for (int k = 0; k < 4; k++) {
				const int tx = ix + (k & 1), ty = iy + (k >> 1);
				const float w = wx[k & 1] * wy[k >> 1];
				if (tx < 0 || tx >= width || ty < 0 || ty >= height || !(w > 0.f)) continue;
				const int q = (height - 1 - ty) * width + tx;
				AGPT_CHECK(q >= 0 && q < width * height, AGPT_DBG_TAP, q);
				const float4 a = accumIn[q], m = momentsIn[q], g = Gin[q];
				if (!Finite4(a) || !Finite4(m)) continue;
				const bool hitQ = g.w >= 0.f;
				if (hitQ != hitP) continue;
				if (hitP && !(fabsf(g.w - z) <= sigmaDepth * z && (gp.x * g.x + gp.y * g.y) + gp.z * g.z >= minNormalDot)) continue;
				sw += w;
				A.x += w * a.x; A.y += w * a.y; A.z += w * a.z; A.w += w * a.w;
				Q.x += w * m.x; Q.y += w * m.y; Q.z += w * m.z; Q.w += w * m.w;
			}
		}
	}
	if (sw > 0.f) {
		A = make_float4(A.x / sw, A.y / sw, A.z / sw, A.w / sw);
		Q = make_float4(Q.x / sw, Q.y / sw, Q.z / sw, Q.w / sw);
		if (Q.w > maxHistory) {
			const float k = maxHistory / Q.w;
			A = make_float4(A.x * k, A.y * k, A.z * k, A.w * k);
			Q = make_float4(Q.x * k, Q.y * k, Q.z * k, maxHistory);
		}
	}
	else { A = make_float4(0.f, 0.f, 0.f, 0.f); Q = A; }
	accumOut[p] = A;
	momentsOut[p] = Q;
}

// ---- bandwidth probe: what a plain streaming read of this library's own making reaches on this GPU ----
// `n16` 16-byte words read `iters` times by a persistent grid with 128-bit loads.  A buffer that fits in L2
// measures L2 bandwidth (the roofline denominator for the trace kernels' L2 traffic), one far larger than L2
// measures HBM read bandwidth.
__global__ void __launch_bounds__(512) k_probe_bandwidth(const uint4* __restrict__ data, size_t n16, int iters, unsigned* sink) {
	unsigned acc = 0;
	const size_t stride = (size_t)gridDim.x * blockDim.x;
	for (int it = 0; it < iters; it++)
		for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) {
			uint4 v = __ldcg(data + i);        // cached in L2 only: a second pass must not be served from L1
			acc ^= v.x ^ v.y ^ v.z ^ v.w;
		}
	if (acc == 0x9e3779b9u) sink[0] = acc;      // (never true for the zero-filled buffer: keeps the loads alive)
}

// ---- upload-time pass: flag triangles upstream would reject as degenerate (trianglemesh.cpp:71-77)
__global__ void k_flag_degenerate(float4* tris, const float2* uvs, int n) {
	int j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	float4 a = tris[3 * j], b = tris[3 * j + 1], c = tris[3 * j + 2];
	float2 uv0 = make_float2(0, 0), uv1 = make_float2(1, 0), uv2 = make_float2(1, 1);
	if (uvs) { uv0 = uvs[3 * j]; uv1 = uvs[3 * j + 1]; uv2 = uvs[3 * j + 2]; }
	float3 dpdu, dpdv;
	bool ok = TriangleDerivatives(f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), f3(c.x, c.y, c.z), uv0, uv1, uv2, dpdu, dpdv);
	tris[3 * j].w = ok ? 0.f : 1.f;
}

// ---- EXTENSION: sampling tables of the plane / mesh area lights (AGPT_LIGHT_SAMPLE_SHAPE): triangle areas in slot order,
// 0 for a triangle k_flag_degenerate marked (CPU statement: oracle/agpt_shape_oracle.cpp BuildShapeLights)
__global__ void k_triangle_areas(const float4* __restrict__ tris, int n, float* area) {
	int j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	float4 a = tris[3 * j], b = tris[3 * j + 1], c = tris[3 * j + 2];
	float3 v0 = f3(a.x, a.y, a.z);
	area[j] = a.w != 0.f ? 0.f : 0.5f * length(cross(f3(b.x, b.y, b.z) - v0, f3(c.x, c.y, c.z) - v0));
}
