// host/scene.h -- Scene with the reference's surface (/root/reference/scene.h:3-30): a flat
// list of primitives in insertion order, a list of lights, a CameraDesc -- plus Flatten(),
// which turns the object graph into the typed tables of include/agpt.h.
//
// Scene::Intersect / IntersectP (scene.h:5-19) are the device's closest-hit and any-hit
// kernels; list ORDER is preserved in the primitive table because it decides exact-t ties
// (a sphere accepts root == ray.t, triangles and planes reject t >= ray.t).
#pragma once

#include <atomic>
#include <map>
#include <stdexcept>

#include "precomp.h"
#include "camera.h"
#include "intersectable.h"
#include "trianglemesh.h"
#include "bvhtrimesh.h"
#include "lights.h"

// EXTENSION (SURVEY 8f row 4; not a reference class -- upstream bakes transforms into vertices, scene.h:5-28,
// trianglemesh.cpp:157): one placement of a shared mesh.  `objectToWorld` is an affine mat4 (rows of [R | t]);
// what tracing an instance means is defined in include/agpt.h (agpt_instance) and stated on the CPU in
// oracle/agpt_oracle.cpp.  The material belongs to the placement, the geometry and its BVH to the shared mesh.
#define AGPT_HAS_INSTANCES 1
class Instance : public Intersectable {
public:
	Instance(shared_ptr<TriangleMesh> mesh, const mat4& objectToWorld, shared_ptr<Material> material)
		: Intersectable(material), Mesh(mesh), ObjectToWorld(objectToWorld) {}
	int Kind() const override { return AGPT_PRIM_INSTANCE; }
	// affine inverse in double: both the GPU and the CPU statement consume the same two float matrices
	agpt_instance Export(int meshIndex) const {
		agpt_instance r;
		memset(&r, 0, sizeof(r));
		r.mesh = meshIndex;
		const float* m = ObjectToWorld.cell;
		double a[3][3] = { { m[0], m[1], m[2] }, { m[4], m[5], m[6] }, { m[8], m[9], m[10] } }, t[3] = { m[3], m[7], m[11] };
		double det = a[0][0] * (a[1][1] * a[2][2] - a[1][2] * a[2][1]) - a[0][1] * (a[1][0] * a[2][2] - a[1][2] * a[2][0]) + a[0][2] * (a[1][0] * a[2][1] - a[1][1] * a[2][0]);
		if (det == 0) throw std::runtime_error("Instance: singular transform");
		double inv[3][3];
		for (int i = 0; i < 3; i++)
			for (int j = 0; j < 3; j++) {
				int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
				inv[j][i] = (a[i1][j1] * a[i2][j2] - a[i1][j2] * a[i2][j1]) / det;
			}
		for (int i = 0; i < 3; i++) {
			for (int j = 0; j < 3; j++) { r.object_to_world[4 * i + j] = (float)a[i][j]; r.world_to_object[4 * i + j] = (float)inv[i][j]; }
			r.object_to_world[4 * i + 3] = (float)t[i];
			r.world_to_object[4 * i + 3] = (float)-(inv[i][0] * t[0] + inv[i][1] * t[1] + inv[i][2] * t[2]);
		}
		return r;
	}
	shared_ptr<TriangleMesh> Mesh;
	mat4 ObjectToWorld;
};

// Everything agpt_upload_* needs, owned in one place so the pointers in `meshes` stay valid.
struct FlatScene {
	std::vector<agpt_prim> prims;
	std::vector<agpt_sphere> spheres;
	std::vector<agpt_plane> planes;
	std::vector<agpt_material> materials;
	std::vector<agpt_light> lights;
	std::vector<agpt_mesh_desc> meshes;
	std::vector<FlatTriangles> meshTris;
	std::vector<agpt_instance> instances;      // extension: placed meshes
	agpt_envmap envmap = { 0, 0, nullptr, nullptr, nullptr, 0.f };   // borrowed from the scene's InfiniteAreaLight
	std::vector<agpt_texture> textures;        // extension: base-colour images, texels borrowed from the materials
	std::vector<int32_t> materialTexture;      // per material: index into textures or -1 (empty when no material has one)
	std::vector<agpt_material_textures> materialTextures;   // extension: per material, all its image bindings (empty as above)
	std::vector<agpt_alpha_mask> alphaMasks;   // extension: per material, its alpha mask (empty when no material has one)
	std::vector<agpt_emission> emission;       // extension: per material, its emission (empty when no material emits)
	bool HasMaps() const { for (auto& b : materialTextures) if (b.roughness_metallic >= 0 || b.normal >= 0) return true; return false; }
	uint64_t Bytes() const {
		uint64_t b = prims.size() * sizeof(agpt_prim) + spheres.size() * sizeof(agpt_sphere) + planes.size() * sizeof(agpt_plane)
			+ materials.size() * sizeof(agpt_material) + lights.size() * sizeof(agpt_light);
		b += instances.size() * sizeof(agpt_instance);
		for (auto& m : meshes) b += (uint64_t)m.n_nodes * 32 + (uint64_t)m.n_tris * (48 + 4 + (m.tri_normals ? 48 : 0) + (m.tri_uvs ? 24 : 0));
		for (auto& t : textures) b += (uint64_t)t.width * t.height * 16 + 16;   // float4 texels and a descriptor on the device
		b += materialTexture.size() * 4;
		if (HasMaps()) b += materialTextures.size() * 32;                      // the map binding table
		b += alphaMasks.size() * sizeof(agpt_alpha_mask);
		b += emission.size() * sizeof(agpt_emission);
		return b;
	}
};

class Scene {
public:
	void addAreaLight(std::shared_ptr<Intersectable> shape, const float3& L) {
		primitives.push_back(shape);
		lights.push_back(make_shared<AreaLight>(shape, L));
	}
	// EXTENSION: the same, with the shape sampled for next-event estimation (host/lights.h SampledAreaLight)
	void addSampledAreaLight(std::shared_ptr<Intersectable> shape, const float3& L) {
		primitives.push_back(shape);
		lights.push_back(make_shared<SampledAreaLight>(shape, L));
	}

	// Object graph -> device tables.  Materials are de-duplicated by pointer.
	std::shared_ptr<FlatScene> Flatten() const {
		auto flat = std::make_shared<FlatScene>();
		std::map<const Material*, int> matIndex;
		std::map<const ImageTexture*, int> texIndex;         // extension: textures de-duplicated by pointer
		std::map<const Light*, int> lightIndex;
		std::map<const Intersectable*, int> primIndex;
		std::map<const TriangleMesh*, int> sharedMesh;       // meshes referenced by instances: flattened once
		for (size_t i = 0; i < lights.size(); i++) lightIndex[lights[i].get()] = (int)i;
		flat->meshTris.reserve(2 * primitives.size());
		auto flattenMesh = [&](const TriangleMesh* mesh) {
			agpt_mesh_desc d;
			memset(&d, 0, sizeof(d));
			std::vector<int32_t> order;
			if (mesh->Kind() == AGPT_PRIM_BVH_MESH) {
				const BVHTriMesh* bvh = static_cast<const BVHTriMesh*>(mesh);
				d.nodes = reinterpret_cast<const agpt_bvh_node*>(bvh->Nodes().data());   // owned by the mesh
				d.n_nodes = (int)bvh->Nodes().size();
				order = bvh->LeafOrder();
			}
			else {
				order.resize(mesh->NumTriangles());
				for (size_t t = 0; t < order.size(); t++) order[t] = (int32_t)t;
			}
			flat->meshTris.push_back(mesh->ExportTriangles(order));
			const FlatTriangles& ft = flat->meshTris.back();
			d.n_tris = (int)ft.ids.size();
			d.tri_verts = ft.verts.data();
			d.tri_ids = ft.ids.data();
			d.tri_normals = ft.normals.empty() ? nullptr : ft.normals.data();
			d.tri_uvs = ft.uvs.empty() ? nullptr : ft.uvs.data();
			flat->meshes.push_back(d);
			return (int)flat->meshes.size() - 1;
		};
		for (size_t i = 0; i < primitives.size(); i++) {
			const Intersectable* shape = primitives[i].get();
			primIndex[shape] = (int)i;
			agpt_prim row;
			row.type = shape->Kind();
			row.material = -1;
			if (const Material* m = shape->GetMaterial()) {
				auto it = matIndex.find(m);
				if (it == matIndex.end()) {
					it = matIndex.emplace(m, (int)flat->materials.size()).first;
					flat->materials.push_back(m->Export());
					auto index = [&](const ImageTexture* t) {
						if (!t) return -1;
						auto ti = texIndex.find(t);
						if (ti == texIndex.end()) { ti = texIndex.emplace(t, (int)flat->textures.size()).first; flat->textures.push_back(t->Export()); }
						return ti->second;
					};
					const MaterialMaps mm = m->Maps();
					agpt_material_textures b;
					b.base = index(mm.base); b.roughness_metallic = index(mm.roughnessMetallic); b.normal = index(mm.normal);
					b.normal_scale = mm.normalScale;
					b.color[0] = mm.color.x; b.color[1] = mm.color.y; b.color[2] = mm.color.z;
					flat->materialTexture.push_back(b.base);
					flat->materialTextures.push_back(b);
					const MaterialAlphaMask am = m->AlphaMask();
					flat->alphaMasks.push_back(agpt_alpha_mask{ index(am.image), am.channel, am.cutoff, 0 });
					const MaterialEmission me = m->Emission();
					flat->emission.push_back(agpt_emission{ index(me.image), { me.factor.x, me.factor.y, me.factor.z } });
				}
				row.material = it->second;
			}
			row.area_light = -1;
			if (const AreaLight* al = shape->GetAreaLight()) {
				auto it = lightIndex.find(al);
				if (it != lightIndex.end()) row.area_light = it->second;
			}
			switch (row.type) {
			case AGPT_PRIM_SPHERE:
				row.payload = (int)flat->spheres.size();
				flat->spheres.push_back(static_cast<const Sphere*>(shape)->Export());
				break;
			case AGPT_PRIM_PLANE:
				row.payload = (int)flat->planes.size();
				flat->planes.push_back(static_cast<const Plane*>(shape)->Export());
				break;
			case AGPT_PRIM_INSTANCE: {
				const Instance* inst = static_cast<const Instance*>(shape);
				auto it = sharedMesh.find(inst->Mesh.get());
				if (it == sharedMesh.end()) it = sharedMesh.emplace(inst->Mesh.get(), flattenMesh(inst->Mesh.get())).first;
				row.payload = (int)flat->instances.size();
				flat->instances.push_back(inst->Export(it->second));
			} break;
			default:
				row.payload = flattenMesh(static_cast<const TriangleMesh*>(shape));
				break;
			}
			flat->prims.push_back(row);
		}
		if (flat->textures.empty()) { flat->materialTexture.clear(); flat->materialTextures.clear(); }
		bool masked = false;
		for (auto& am : flat->alphaMasks) masked = masked || am.texture >= 0;
		if (!masked) flat->alphaMasks.clear();
		bool emits = false;
		for (auto& e : flat->emission) emits = emits || e.factor[0] > 0.f || e.factor[1] > 0.f || e.factor[2] > 0.f;
		if (!emits) flat->emission.clear();
		for (auto& l : lights) {
			agpt_light rec;
			memset(&rec, 0, sizeof(rec));
			rec.type = l->Kind();
			rec.flags = l->Flags();
			rec.prim = -1;
			if (rec.type == AGPT_LIGHT_AREA) {
				auto it = primIndex.find(static_cast<const AreaLight*>(l.get())->Shape.get());
				if (it != primIndex.end()) rec.prim = it->second;
			}
			if (rec.type == AGPT_LIGHT_INFINITE_AREA) flat->envmap = static_cast<const InfiniteAreaLight*>(l.get())->Export();
			float3 e = l->Emission();
			rec.lemit[0] = e.x; rec.lemit[1] = e.y; rec.lemit[2] = e.z;
			flat->lights.push_back(rec);
		}
		return flat;
	}

	// What an uploaded copy of this scene is keyed on (CudaPathTracer): the object's serial number --
	// a different Scene later constructed at the same address gets a new one -- mixed with the
	// identities of its primitives and lights, so push_back / addAreaLight after an upload are seen.
	// Shapes, materials and lights are immutable after construction upstream, so identity is content.
	uint64_t Fingerprint() const {
		uint64_t h = 0xcbf29ce484222325ull ^ serial;
		auto mix = [&h](uint64_t v) { h = (h ^ v) * 0x100000001b3ull; };
		mix(primitives.size()); mix(lights.size());
		for (auto& p : primitives) mix((uint64_t)(uintptr_t)p.get());
		for (auto& l : lights) mix((uint64_t)(uintptr_t)l.get());
		return h;
	}

	vector<shared_ptr<Intersectable>> primitives;
	vector<shared_ptr<Light>> lights;
	CameraDesc camera;

private:
	static uint64_t NextSerial() { static std::atomic<uint64_t> next(1); return next.fetch_add(1); }
	uint64_t serial = NextSerial();
};
