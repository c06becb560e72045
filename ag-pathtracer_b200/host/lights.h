// host/lights.h -- Light, UniformInfiniteLight, AreaLight with the reference's
// construction surface (/root/reference/lights.h:23-87).
//
// Host lights are descriptors.  Sample_Li / Pdf_Li / Le (lights.cpp:10-28,115-130) and the
// visibility test (lights.cpp:10-12) are evaluated on the device by the shade and any-hit
// kernels.  InfiniteAreaLight (HDR environment map, lights.cpp:31-112) loads its lat-long map
// and builds the texel distribution on the host exactly as upstream's constructor does
// (lights.cpp:31-48); lookups and importance sampling run on the device.
#pragma once

#include "precomp.h"
#include "intersectable.h"
#include "texture.h"
#include "sampling.h"

class Light {
public:
	virtual ~Light() {}
	virtual bool IsInfinite() const { return false; }
	virtual int Kind() const = 0;      // AGPT_LIGHT_*
	virtual float3 Emission() const = 0;
	virtual uint32_t Flags() const { return 0; }   // agpt_light.flags
};

class UniformInfiniteLight : public Light {
public:
	UniformInfiniteLight(const float3& l) : Lemit(l) {}
	bool IsInfinite() const override { return true; }
	int Kind() const override { return AGPT_LIGHT_UNIFORM_INFINITE; }
	float3 Emission() const override { return Lemit; }
protected:
	const float3 Lemit;
};

// Wraps any Intersectable; as upstream, only Sphere can be sampled (others emit when hit
// by camera / specular rays only, SURVEY D8).  Emission is two-sided (lights.h:82).
class AreaLight : public Light {
public:
	AreaLight(shared_ptr<Intersectable> shape, const float3& l) : Shape(shape), Lemit(l) { shape->SetAreaLight(this); }
	int Kind() const override { return AGPT_LIGHT_AREA; }
	float3 Emission() const override { return Lemit; }
	shared_ptr<Intersectable> Shape;
protected:
	const float3 Lemit;
};

// EXTENSION (not a reference class; agpt.h AGPT_LIGHT_SAMPLE_SHAPE): an AreaLight whose Plane, TriangleMesh or BVHTriMesh
// next-event estimation samples (PBRT-v3's Shape::Sample / Pdf, one light for the whole mesh).  Emission stays two-sided.
// Scene::addSampledAreaLight makes one; a plain AreaLight keeps the reference's behaviour.
#define AGPT_HAS_SAMPLED_AREA_LIGHTS 1
class SampledAreaLight : public AreaLight {
public:
	SampledAreaLight(shared_ptr<Intersectable> shape, const float3& l) : AreaLight(shape, l) {}
	uint32_t Flags() const override { return AGPT_LIGHT_SAMPLE_SHAPE; }
};

// Environment light over a lat-long HDR map with importance sampling (upstream builds with ILS
// defined, lights.h:9).  func[idx] = max(r,g,b) * sin(theta of the texel row) (lights.cpp:36-45).
class InfiniteAreaLight : public Light {
public:
	InfiniteAreaLight(const std::string& texmap) {
		Lmap = std::make_shared<HDRTexture>(texmap);
		std::vector<float> pdf((size_t)Lmap->Width() * Lmap->Height());
		for (int idx = 0; idx < (int)pdf.size(); idx++) {
			int x = idx % Lmap->Width();
			int y = idx / Lmap->Width();
			float th = (y + .5f) * PI / Lmap->Height();
			float3 value = Lmap->GetPixel(x, y);
			float maxComponent = std::max(value.x, std::max(value.y, value.z));
			pdf[idx] = maxComponent * std::sin(th);
		}
		distrib = std::make_shared<Distribution1D>(pdf.empty() ? nullptr : &pdf[0], (int)pdf.size());
	}
	bool IsInfinite() const override { return true; }
	int Kind() const override { return AGPT_LIGHT_INFINITE_AREA; }
	float3 Emission() const override { return float3(0.f); }
	agpt_envmap Export() const {
		agpt_envmap e;
		e.width = Lmap->Width(); e.height = Lmap->Height();
		e.rgb = Lmap->Data().data(); e.func = distrib->func.data(); e.cdf = distrib->cdf.data(); e.func_int = distrib->funcInt;
		return e;
	}
private:
	std::shared_ptr<HDRTexture> Lmap;
	std::shared_ptr<Distribution1D> distrib;
};
