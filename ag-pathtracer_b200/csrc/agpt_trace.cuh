// agpt_trace.cuh -- Scene::Intersect / Scene::IntersectP on the device.
//
// Closest-hit: scene.h:5-13 -> per primitive in list order, BVHTriMesh::Intersect
// (bvhtrimesh.h:185-191) -> RecursiveHit (:332-384) as an iterative, near-first walk with an
// explicit stack.  Any-hit: scene.h:15-19 -> RecursiveHitP (:386-413), order-free, early out.
//
// Result equivalence with the recursion: the near child is descended first, the far child
// is pushed iff both boxes were hit (swap iff rightDist < leftDist, :359-372) and is NOT
// re-tested against the shrunken ray.t when popped (upstream does not either, :379) -- its
// leaves' triangles are simply rejected by t >= ray.t.  Equal-t ties therefore go to the
// triangle upstream visits first.
//
// Node fetch: a sibling pair is one 64-byte line = four 128-bit loads (north star item 1);
// a leaf-ordered triangle is three 128-bit loads.
#pragma once

#include "agpt_device.cuh"
#include "agpt_bsdf.cuh"      // the texture lookup of alpha masks

#ifndef AGPT_STACK_SMEM
#define AGPT_STACK_SMEM 24      // stack entries per thread kept in shared memory
#endif
#ifndef AGPT_TRACE_MIN_BLOCKS
#define AGPT_TRACE_MIN_BLOCKS 16  // <= 64 registers: 1024 threads per SM (measured: 71 registers is 7 % slower)
#endif
#ifndef AGPT_STACK_LOCAL
#define AGPT_STACK_LOCAL 104    // overflow entries in local memory: 128 levels in all.  SAH trees over real meshes are <= ~30
                                // deep (the shared-memory part); agpt_upload_meshes refuses trees deeper than the stack.
#endif
#ifndef AGPT_TRACE_THREADS
#define AGPT_TRACE_THREADS 64     // small blocks retire early when their rays are short (128: +1 %, 256: +8 %, 512: +25 % trace time)
#endif

struct TraceCounters {
	unsigned long long node_visits, box_tests, tri_tests, analytic_tests;
	unsigned long long warp_steps, lane_steps;     // trips of the lockstep walk (counted by lane 0) and lanes with work in them: lane_steps / warp_steps = rays alive per step
};

struct HitRecord {
	float t;
	float b1, b2;     // barycentrics of a triangle hit (trianglemesh.cpp:28,35)
	int prim;         // index in Scene::primitives, -1 = miss
	int slot;         // leaf-order triangle slot inside the mesh, -1 for sphere / plane
};

// Stack entry encoding: bit 31 set -> single-triangle leaf, low bits = triangle slot;
// otherwise bit 30 set -> multi-triangle leaf, low bits = node index (re-read first/count);
// otherwise interior node, value = index of its left child (the pair base).
#define AGPT_ENT_LEAF1 0x80000000u
#define AGPT_ENT_LEAFN 0x40000000u

__device__ __forceinline__ unsigned EncodeNode(int nodeIndex, int first, int count) {
	if (count == 0) return (unsigned)first;
	if (count == 1) return AGPT_ENT_LEAF1 | (unsigned)first;
	return AGPT_ENT_LEAFN | (unsigned)nodeIndex;
}

struct NodeBox {
	float3 bmin, bmax;
	int first, count;
};
__device__ __forceinline__ float4 LoadTable(const float4* __restrict__ p) { return __ldg(p); }
__device__ __forceinline__ NodeBox LoadNode(const float4* __restrict__ nodes, int i) {
	float4 a = LoadTable(nodes + 2 * i), b = LoadTable(nodes + 2 * i + 1);
	NodeBox n;
	n.bmin = f3(a.x, a.y, a.z);
	n.bmax = f3(a.w, b.x, b.y);
	n.first = __float_as_int(b.z);
	n.count = __float_as_int(b.w);
	return n;
}

// Exact hit/miss decision of Bounds::Intersect (bvhtrimesh.h:18-36): filtered arithmetic first,
// the reference's divisions only when a comparison falls inside the guard band.
template <bool FAST>
__device__ __forceinline__ bool ExactBoxHit(float3 bmin, float3 bmax, float3 O, float3 D, float3 rD, bool filterOk, float rayT) {
	if (FAST && filterOk) {
		float tn, tx;
		SlabApprox(bmin, bmax, O, rD, rayT, tn, tx);
		int c = SlabDecision(tn, tx);
		if (c >= 0) return c == 1;
	}
	float dist;
	return BoundsIntersect(bmin, bmax, O, D, rayT, dist);
}

// exact-filtered slab test (agpt_device.cuh): valid only for sane direction and origin components
template <bool FAST>
__device__ __forceinline__ bool FilterOk(float3 O, float3 D) {
	return FAST && fabsf(D.x) >= 1e-18f && fabsf(D.y) >= 1e-18f && fabsf(D.z) >= 1e-18f &&
		fabsf(D.x) <= 2.0f && fabsf(D.y) <= 2.0f && fabsf(D.z) <= 2.0f && fabsf(O.x) < 1e15f && fabsf(O.y) < 1e15f && fabsf(O.z) < 1e15f;
}

// EXTENSION: instances (agpt.h agpt_instance); the transforms themselves are in agpt_device.cuh.
template <bool FAST>
__device__ __forceinline__ void ObjectSpaceRay(const agpt_instance& in, float3 O, float3 D, float3& o, float3& d, float3& rd, bool& filterOk) {
	o = XformPoint(in.world_to_object, O);
	d = XformVector(in.world_to_object, D);        // not re-normalised: t means the same in both spaces
	rd = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
	filterOk = FilterOk<FAST>(o, d);
}
template <bool INST>
__device__ __forceinline__ const DMesh& MeshOfPrim(const DScene& sc, const agpt_prim& pr) {
	return sc.meshes[(INST && pr.type == AGPT_PRIM_INSTANCE) ? sc.instances[pr.payload].mesh : pr.payload];
}

// EXTENSION: alpha masks (agpt.h agpt_upload_alpha_masks).  A candidate hit the triangle or plane test accepted on a primitive
// of material `material` stands iff that material has no mask or the mask's channel at the hit's uv is >= its cutoff.  The
// record is read only here, on a geometric hit: the walk keeps just the material index of the mesh it is in.
__device__ __forceinline__ bool MaskOf(const DMaskTables& mk, int material, int& texture, int& channel, float& cutoff) {
	if (material < 0) return false;
	AGPT_CHECK(material < mk.nMasks, AGPT_DBG_MASK, material);
	const agpt_alpha_mask m = mk.masks[material];
	texture = m.texture; channel = m.channel; cutoff = m.cutoff;
	return texture >= 0;
}
template <bool INST>
__device__ __forceinline__ bool MaskTriangle(const DScene& sc, const DMaskTables& mk, int material, int primIndex, int slot, float b1, float b2) {
	int texture, channel;
	float cutoff;
	if (!MaskOf(mk, material, texture, channel, cutoff)) return true;
	float2 uv0, uv1, uv2;
	TriangleUVs(MeshOfPrim<INST>(sc, sc.prims[primIndex]), slot, uv0, uv1, uv2);
	return TexLookupChannel(mk.tt, texture, channel, BaryUV(b1, b2, uv0, uv1, uv2)) >= cutoff;
}
__device__ __forceinline__ bool MaskPlane(const DMaskTables& mk, int material, const agpt_plane& pl, float3 O, float3 D, float t) {
	int texture, channel;
	float cutoff;
	if (!MaskOf(mk, material, texture, channel, cutoff)) return true;
	return TexLookupChannel(mk.tt, texture, channel, PlaneUV(pl, O + t * D)) >= cutoff;
}
#ifndef AGPT_ANY_NEAR_FIRST
#define AGPT_ANY_NEAR_FIRST 1
#endif
#ifndef AGPT_RUN_CULL_MIN
#define AGPT_RUN_CULL_MIN 4        // sphere runs at least this long get a bounding-box pre-test
#endif

// A RUN of at most 32 consecutive mesh primitives [p0, p1) of Scene::primitives.  `stack` points
// at this thread's shared-memory column (stride = blockDim.x).  ANY: stop at the first accepted
// triangle.  Otherwise updates hit / rayT.
//
// Convergence: the walk is a WARP-SYNCHRONOUS loop.  All 32 lanes stay in the loop until
// every lane is done (`__any_sync` on the loop condition); a finished or invalid lane is
// predicated off.  The loop has one back edge and every path through the body merges before
// it, so the hardware re-converges the warp once per step instead of letting lanes that
// `continue`d early run ahead as separate fragments (measured: 2.3-3.1 of 32 threads active
// per instruction with the naive while/continue form, 7-23 with this one).
//
// Root prepass: the root boxes of all meshes of the run (BVHTriMesh::Intersect,
// bvhtrimesh.h:185-191) are first tested by the whole warp together against the ray's CURRENT
// extent.  A root missed now is also missed later (ray.t only shrinks), so the walk proper
// only enters the remaining candidates -- each lane on its own, in list order -- and repeats
// the root test there when ray.t has shrunk since.  Per ray the sequence of box and triangle
// tests is the reference's; the root tests just happen in lockstep instead of one loop step
// each (a typical ray hits 1-2 of 5 roots).
// `lane` is false for threads without a ray; they must still call (full-mask votes).
// SMEM: stack entries per thread in shared memory (the rest of the AGPT_STACK_SMEM + AGPT_STACK_LOCAL levels in local memory).
// MASK (extension, alpha masks): a triangle hit must also pass MaskTriangle.
template <bool ANY, bool COUNT, bool FAST, bool INST, int SMEM = AGPT_STACK_SMEM, bool MASK = false>
__device__ __forceinline__ bool TraceMeshRun(const DScene& sc, int p0, int p1, float3 O, float3 D, float3 rD, bool filterOk, float& rayT, HitRecord& hit,
		unsigned* stack, int stackStride, TraceCounters& cnt, bool lane, const DMaskTables& mk = DMaskTables()) {
	bool found = false;
	unsigned local[AGPT_STACK_SMEM + AGPT_STACK_LOCAL - SMEM];
	unsigned cand = 0;               // meshes of the run this lane still has to enter (bit m - p0)
	unsigned bvhMask = 0;            // meshes of the run that have a root box
	const float rayT0 = rayT;
	// INST (the scene has instances, agpt.h agpt_instance): a mesh of the run may be a placed one; its boxes and
	// triangles are then tested against the object-space ray (cO, cD), which shares the parameter t with the world ray.
	float3 cO = O, cD = D, crD = rD;
	bool cFilt = filterOk;
	for (int m = p0; m < p1; m++) {
		const agpt_prim pr = sc.prims[m];
		const DMesh& mesh = MeshOfPrim<INST>(sc, pr);
		bool c = lane;
		if (COUNT && mesh.nodes != nullptr) bvhMask |= 1u << (m - p0);
		if (c && mesh.nodes != nullptr) {
			NodeBox root = LoadNode(mesh.nodes, 0);
			if (INST && pr.type == AGPT_PRIM_INSTANCE) {
				float3 o, d, rd;
				bool f;
				ObjectSpaceRay<FAST>(sc.instances[pr.payload], O, D, o, d, rd, f);
				c = ExactBoxHit<FAST>(root.bmin, root.bmax, o, d, rd, f, rayT0);
			}
			else c = ExactBoxHit<FAST>(root.bmin, root.bmax, O, D, rD, filterOk, rayT0);
		}
		if (c) cand |= 1u << (m - p0);
	}
	int mp = p1 - 1;                 // this lane's current mesh primitive
	int mat = -1;                    // MASK: the material of mesh mp
	bool inside = false;             // walking mesh mp (else: about to enter the next candidate)
	const float4* nodes = nullptr;
	const float4* tris = nullptr;
	unsigned cur = 0;
	int sp = 0;
	bool active = lane;
	while (__any_sync(0xffffffffu, active && (inside || cand != 0u))) {
		if (COUNT) { if ((threadIdx.x & 31) == 0) cnt.warp_steps++; if (active && (inside || cand != 0u)) cnt.lane_steps++; }
		if (active && (inside || cand != 0u)) {
			if (!inside) {
				// enter the next candidate mesh
				int bit = __ffs((int)cand) - 1;
				cand &= cand - 1u;
				mp = p0 + bit;
				const agpt_prim pr = sc.prims[mp];
				const DMesh& mesh = MeshOfPrim<INST>(sc, pr);
				nodes = mesh.nodes; tris = mesh.tris;
				if (MASK) mat = pr.material;
				if (INST) {
					if (pr.type == AGPT_PRIM_INSTANCE) ObjectSpaceRay<FAST>(sc.instances[pr.payload], O, D, cO, cD, crD, cFilt);
					else { cO = O; cD = D; crD = rD; cFilt = filterOk; }
				}
				if (nodes == nullptr) {
					// plain TriangleMesh: every triangle in order, no bounds test (trianglemesh.h:25-41)
					for (int j = 0; j < mesh.n_tris; j++) {
						float4 a = LoadTable(tris + 3 * j), b = LoadTable(tris + 3 * j + 1), c = LoadTable(tris + 3 * j + 2);
						if (COUNT) cnt.tri_tests++;
						float t, b1, b2;
						if constexpr (MASK) {
							if ((ANY || a.w == 0.f) && TriangleTest(f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), f3(c.x, c.y, c.z), cO, cD, rayT, t, b1, b2) && MaskTriangle<INST>(sc, mk, mat, mp, j, b1, b2)) {
								found = true;
								if (ANY) break;
								rayT = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = mp; hit.slot = j;
							}
						}
						else if ((ANY || a.w == 0.f) && TriangleTest(f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), f3(c.x, c.y, c.z), cO, cD, rayT, t, b1, b2)) {
							found = true;
							if (ANY) break;
							rayT = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = mp; hit.slot = j;
						}
					}
				}
				else {
					NodeBox root = LoadNode(nodes, 0);
					// ray.t unchanged since the prepass: same decision; else redo it with the shrunken extent
					if (rayT == rayT0 || ExactBoxHit<FAST>(root.bmin, root.bmax, cO, cD, crD, cFilt, rayT)) {
						cur = EncodeNode(0, root.first, root.count); sp = 0; inside = true;
					}
				}
			}
			else {
				bool pop = true;
				if (!(cur & (AGPT_ENT_LEAF1 | AGPT_ENT_LEAFN))) {
					// interior: fetch the sibling pair (64 B), test both boxes
					AGPT_CHECK((int)cur >= 2 && (int)cur + 1 < MeshOfPrim<INST>(sc, sc.prims[mp]).n_nodes, AGPT_DBG_NODE, cur);
					NodeBox l = LoadNode(nodes, (int)cur), r = LoadNode(nodes, (int)cur + 1);
					if (COUNT) { cnt.node_visits++; cnt.box_tests += 2; }
					float dl, dr;
					bool hl, hr, swapKids;
					bool strict = !cFilt;
					if (!strict) {
						float xl, xr;
						SlabApprox(l.bmin, l.bmax, cO, crD, rayT, dl, xl);
						SlabApprox(r.bmin, r.bmax, cO, crD, rayT, dr, xr);
						int cl = SlabDecision(dl, xl), cr = SlabDecision(dr, xr);
						if (ANY && !COUNT && AGPT_ANY_NEAR_FIRST) {
							// Occlusion does not depend on the order of the walk (upstream: left first,
							// bvhtrimesh.h:400-411), nor on visiting a box that a borderline test would
							// have skipped: nearer child first finds occluders sooner, and a comparison
							// inside the guard band simply counts as a hit.  The counting instantiation
							// keeps upstream's order so its visit counts stay comparable.
							hl = cl != 0; hr = cr != 0; swapKids = dr < dl;
						}
						else {
							int cs = (ANY || cl != 1 || cr != 1) ? 0 : NearerDecision(dl, dr);
							hl = cl == 1; hr = cr == 1; swapKids = cs == 1;
							strict = (cl | cr | cs) < 0;       // some comparison fell inside the guard band
						}
					}
					if (strict) {
						hl = BoundsIntersect(l.bmin, l.bmax, cO, cD, rayT, dl);
						hr = BoundsIntersect(r.bmin, r.bmax, cO, cD, rayT, dr);
						// closest-hit: near first, far pushed iff both hit (swap iff rightDist < leftDist,
						// bvhtrimesh.h:359-372); any-hit: left first (:400-411)
						swapKids = ANY ? false : (dr < dl);
					}
					unsigned el = EncodeNode((int)cur, l.first, l.count), er = EncodeNode((int)cur + 1, r.first, r.count);
					if (hl && hr) {
						unsigned farE = swapKids ? el : er;
						AGPT_CHECK(sp < AGPT_STACK_SMEM + AGPT_STACK_LOCAL, AGPT_DBG_STACK, sp);
						if (sp < SMEM) stack[sp * stackStride] = farE; else local[sp - SMEM] = farE;
						sp++;
						cur = swapKids ? er : el;
						pop = false;
					}
					else if (hl || hr) { cur = hl ? el : er; pop = false; }
				}
				else {
					int first, count;
					if (cur & AGPT_ENT_LEAF1) { first = (int)(cur & 0x7fffffffu); count = 1; }
					else {
						NodeBox n = LoadNode(nodes, (int)(cur & 0x3fffffffu));
						first = n.first; count = n.count;
					}
					AGPT_CHECK(first >= 0 && first + count <= MeshOfPrim<INST>(sc, sc.prims[mp]).n_tris, AGPT_DBG_TRI, first);
					for (int j = first; j < first + count; j++) {
						float4 a = LoadTable(tris + 3 * j), b = LoadTable(tris + 3 * j + 1), c = LoadTable(tris + 3 * j + 2);
						if (COUNT) cnt.tri_tests++;
						float t, b1, b2;
						if constexpr (MASK) {
							if ((ANY || a.w == 0.f) && TriangleTest(f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), f3(c.x, c.y, c.z), cO, cD, rayT, t, b1, b2) && MaskTriangle<INST>(sc, mk, mat, mp, j, b1, b2)) {
								found = true;
								if (ANY) break;
								rayT = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = mp; hit.slot = j;
							}
						}
						else if ((ANY || a.w == 0.f) && TriangleTest(f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), f3(c.x, c.y, c.z), cO, cD, rayT, t, b1, b2)) {
							found = true;
							if (ANY) break;
							rayT = t; hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = mp; hit.slot = j;
						}
					}
				}
				if (pop) {
					if (sp == 0) inside = false;
					else {
						sp--;
						cur = (sp < SMEM) ? stack[sp * stackStride] : local[sp - SMEM];
					}
				}
			}
			if (ANY && found) active = false;
		}
	}
	// one root test per mesh the reference reaches: all of the run, or up to the occluder (scene.h:15-19)
	if (COUNT && lane) {
		int last = ((ANY && found) ? mp : p1 - 1) - p0;
		cnt.box_tests += (unsigned long long)__popc(bvhMask & (0xffffffffu >> (31 - last)));
	}
	return found;
}

// Scene::Intersect (ANY=false) / Scene::IntersectP (ANY=true): primitives in list order.
// Every lane of the warp must call (lane=false for threads without a ray).
// (Testing the spheres and planes first and the meshes afterwards, with an exact tie-aware merge,
// was measured: closest-hit +13 % on cfg 3, +10 % in the closed room -- a second pass over the
// primitive list for little extra pruning.  Not kept; numbers in DESIGN.md.)
// MASK (extension, alpha masks): plane and triangle hits must also pass MaskPlane / MaskTriangle (mk: the mask tables).
template <bool ANY, bool COUNT, bool FAST, bool INST, bool MASK = false>
__device__ __forceinline__ bool TraceScene(const DScene& sc, float3 O, float3 D, float rayT, HitRecord& hit,
		unsigned* stack, int stackStride, TraceCounters& cnt, bool lane, const DMaskTables& mk = DMaskTables()) {
	hit.prim = -1; hit.slot = -1; hit.t = 0.f; hit.b1 = 0.f; hit.b2 = 0.f;
	bool found = false;
	// exact-filtered slab test (agpt_device.cuh): reciprocal direction, valid only for sane components
	const float3 rD = f3(1.0f / D.x, 1.0f / D.y, 1.0f / D.z);
	const bool filterOk = FilterOk<FAST>(O, D);
	int p = 0;
	while (p < sc.n_prims) {
		agpt_prim prim = sc.prims[p];
		bool test = lane && !(ANY && found);
		if (ANY && !__any_sync(0xffffffffu, test)) break;     // warp-uniform early out of IntersectP
		if (prim.type == AGPT_PRIM_SPHERE) {
			// a run of spheres with consecutive payloads: straight through the sphere table
			const int len = sc.sphereRun[p];
			const agpt_sphere* sp = sc.spheres + prim.payload;
			if (len >= AGPT_RUN_CULL_MIN) {
				// Exact cull of the whole run: its spheres sit in a box grown by 5 % of the smallest
				// radius.  A ray that certainly misses that box passes every sphere at more than
				// r + 0.05 r, and as long as the origin is near enough (runBox.w: |oc|^2 below
				// 2e4 r^2) the rounding of Sphere::Intersect's discriminant, < 1.3e-6 |oc|^2, is far
				// too small to turn such a miss into a hit.  If no lane of the warp can hit the
				// box the run is skipped (analytic_tests counts the records really read).
				const float4 b0 = __ldg(sc.sphereRunBox + 3 * p), b1 = __ldg(sc.sphereRunBox + 3 * p + 1), b2 = __ldg(sc.sphereRunBox + 3 * p + 2);
				bool maybe = test;
				if (test && filterOk) {
					float3 oc = O - f3(b2.x, b2.y, b2.z);
					if (sqrLength(oc) < b2.w) {
						float tn, tx;
						SlabApprox(f3(b0.x, b0.y, b0.z), f3(b0.w, b1.x, b1.y), O, rD, rayT, tn, tx);
						maybe = SlabDecision(tn, tx) != 0;
					}
				}
				if (COUNT && test) cnt.analytic_tests++;          // the box record counts as one analytic record read
				if (!__any_sync(0xffffffffu, maybe)) { p += len; continue; }
			}
			for (int j = 0; j < len; j++) {
				bool tj = test && !(ANY && found);
				if (COUNT && tj) cnt.analytic_tests++;
				float t;
				if (tj && SphereTest(sp[j], O, D, rayT, t)) {
					if (!ANY) { rayT = t; hit.t = t; hit.prim = p + j; hit.slot = -1; }
					found = true;
				}
			}
			p += len;
		}
		else if (prim.type == AGPT_PRIM_PLANE) {
			if (COUNT && test) cnt.analytic_tests++;
			float t;
			if constexpr (MASK) {
				if (test && PlaneTest(sc.planes[prim.payload], O, D, rayT, t) && MaskPlane(mk, prim.material, sc.planes[prim.payload], O, D, t)) {
					if (!ANY) { rayT = t; hit.t = t; hit.prim = p; hit.slot = -1; }
					found = true;
				}
			}
			else if (test && PlaneTest(sc.planes[prim.payload], O, D, rayT, t)) {
				if (!ANY) { rayT = t; hit.t = t; hit.prim = p; hit.slot = -1; }
				found = true;
			}
			p++;
		}
		else {
			int q = p + 1;                                     // run of consecutive mesh primitives (<= 32 per call)
			while (q < sc.n_prims && q < p + 32 && sc.prims[q].type >= AGPT_PRIM_BVH_MESH) q++;
			if (TraceMeshRun<ANY, COUNT, FAST, INST, AGPT_STACK_SMEM, MASK>(sc, p, q, O, D, rD, filterOk, rayT, hit, stack, stackStride, cnt, test, mk)) found = true;
			p = q;
		}
	}
	return found;
}

// EXTENSION: Pdf_Li of a plane or mesh area light with AGPT_LIGHT_SAMPLE_SHAPE (agpt.h; CPU statement: oracle/agpt_shape_oracle.cpp
// ShapePdf) -- PBRT-v3's Shape::Pdf(ref, wi): the ray MakeRay(refP + EPSILON wi, wi) against the light's shape ALONE
// (Plane::Intersect, or the mesh's own closest-hit walk, TraceMeshRun over the one-primitive run), 0 without a hit, else
// dist^2 / (|cos| * area) at the hit.  Every lane of the warp must call (lane = false: no query): the walk votes with full masks.
template <int SMEM>
__device__ __forceinline__ float ShapePdfLi(const DScene& sc, const DShapeTables& st, int light, float3 refP, float3 wi, unsigned* stack, int stackStride, bool lane) {
	DShapeLight sl;
	sl.area = 0.f;
	if (lane) sl = st.lights[light];
	lane = lane && sl.area > 0;
	const int primIdx = lane ? sc.lights[light].prim : 0;
	const agpt_prim pr = sc.prims[primIdx];
	DRay r;
	r.O = refP; r.D = f3(1.f, 0.f, 0.f); r.t = FLT_MAX;
	if (lane) r = MakeRay(refP + AGPT_EPSILON * wi, wi);
	bool found = false;
	float t = 0.f;
	float3 n = f3(0.f, 1.f, 0.f);
	if (lane && pr.type == AGPT_PRIM_PLANE) found = PlaneTest(sc.planes[pr.payload], r.O, r.D, r.t, t);
	const bool mesh = lane && pr.type != AGPT_PRIM_PLANE;
	if (__any_sync(0xffffffffu, mesh)) {
		HitRecord hit;
		hit.prim = -1; hit.slot = -1; hit.t = 0.f; hit.b1 = 0.f; hit.b2 = 0.f;
		TraceCounters cnt = { 0, 0, 0, 0, 0, 0 };
		float rayT = r.t;
		const float3 rD = f3(1.0f / r.D.x, 1.0f / r.D.y, 1.0f / r.D.z);
		if (TraceMeshRun<false, false, true, false, SMEM>(sc, primIdx, primIdx + 1, r.O, r.D, rD, FilterOk<true>(r.O, r.D), rayT, hit, stack, stackStride, cnt, mesh)) {
			found = true;
			t = hit.t;
			n = TriangleGeomNormal(sc.meshes[pr.payload].tris + 3 * hit.slot);
		}
	}
	if (!found) return 0.f;
	float3 p = r.O + t * r.D;
	return ShapeSolidAnglePdf(sqrLength(p - refP), n, wi, sl.area);
}

// Warp-aggregated flush of per-thread counters: one atomic per counter per warp.  `totals` = 8 counters of
// the kernel class (agpt_stats), `waveRow` = the same 8 for the current wave (agpt_get_wave_stats) or nullptr:
// rays, node visits, box tests, triangle tests, analytic records, warp steps, lane steps, -.
#define AGPT_WAVE_COUNTERS 8
#define AGPT_MAX_WAVE_ROWS 64
__device__ __forceinline__ void FlushCounters(const TraceCounters& c, bool hasRay, unsigned long long* totals, unsigned long long* waveRow) {
	unsigned long long v[7] = { hasRay ? 1ull : 0ull, c.node_visits, c.box_tests, c.tri_tests, c.analytic_tests, c.warp_steps, c.lane_steps };
#pragma unroll
	for (int k = 0; k < 7; k++) {
		unsigned long long x = v[k];
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
		if ((threadIdx.x & 31) == 0 && x) { atomicAdd(totals + k, x); if (waveRow) atomicAdd(waveRow + k, x); }
	}
}
