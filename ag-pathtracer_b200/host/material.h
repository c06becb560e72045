// host/material.h -- Material, DisneyMaterial, MirrorMaterial with the reference's
// construction surface (/root/reference/material.h:6-88).
//
// On the host a material is just its parameters: the constructor derives, with the
// reference's float arithmetic, the constants its BxDF objects would hold (diffuse/retro
// reflectance, Trowbridge-Reitz alphas, Schlick R0; material.h:14-49, disney.h:22) and
// Export() packs them into the 64-byte agpt_material record the shade kernel reads.
// BSDF evaluation and sampling run on the device only.
#pragma once

#include "precomp.h"
#include "agpt.h"
#include "texture.h"

// EXTENSION: a material's image bindings (include/agpt.h agpt_material_textures), with the images as pointers
struct MaterialMaps {
	const ImageTexture* base = nullptr;
	const ImageTexture* roughnessMetallic = nullptr;   // G = roughness, B = metallic
	const ImageTexture* normal = nullptr;              // tangent-space normal map
	float normalScale = 1.f;
	float3 color = float3(0.f);                        // the base colour, used when base is null and roughnessMetallic is not
};

// EXTENSION: a material's alpha mask (include/agpt.h agpt_alpha_mask), with the image as a pointer
struct MaterialAlphaMask {
	const ImageTexture* image = nullptr;   // null: no mask
	int channel = 0;                       // 0, 1, 2
	float cutoff = 0.5f;                   // the surface is there where the channel >= cutoff
};

// EXTENSION: a material's emission (include/agpt.h agpt_emission), with the image as a pointer
struct MaterialEmission {
	const ImageTexture* image = nullptr;   // null: constant emission
	float3 factor = float3(0.f);           // linear RGB radiance scale; the material emits iff some component is > 0
};

#define AGPT_HAS_ALPHA_MASKS 1         // extension: Material::SetAlphaMask
#define AGPT_HAS_EMISSION 1            // extension: Material::SetEmission
class Material {
public:
	virtual ~Material() {}
	virtual agpt_material Export() const = 0;
	virtual const ImageTexture* BaseColorTexture() const { return nullptr; }   // extension: DisneyMaterial with an image
	virtual MaterialMaps Maps() const { MaterialMaps m; m.base = BaseColorTexture(); return m; }   // extension: all its images
	// EXTENSION (include/agpt.h agpt_upload_alpha_masks): cutout geometry on a material of any type -- channel `channel` of
	// `image` at the hit's uv decides whether a ray hits the surface (glTF alphaMode MASK with alphaCutoff `cutoff`).  Set it before
	// the scene's first render: CudaPathTracer re-uploads a scene when its primitive or light list changes (Scene::Fingerprint,
	// which takes materials as immutable), so a mask set later needs an explicit CudaPathTracer::Upload.
	void SetAlphaMask(std::shared_ptr<ImageTexture> image, int channel = 0, float cutoff = 0.5f) {
		if (channel < 0 || channel > 2 || !std::isfinite(cutoff)) throw std::runtime_error("SetAlphaMask: need a channel in [0, 2] and a finite cutoff");
		maskImage = std::move(image); mask.image = maskImage.get(); mask.channel = channel; mask.cutoff = cutoff;
	}
	MaterialAlphaMask AlphaMask() const { return mask; }
	// EXTENSION (include/agpt.h agpt_upload_emission): the material emits factor, or factor * image at the hit's uv (glTF
	// emissiveFactor x emissive strength, emissiveTexture; linear texels), wherever a path ray hits it, on a material of any type
	// that keeps its BSDF.  Emissive materials are not lights: they are not sampled by next-event estimation.  Set it before the
	// scene's first render, for the reason SetAlphaMask gives.
	void SetEmission(float3 factor, std::shared_ptr<ImageTexture> image = nullptr) {
		for (float f : { factor.x, factor.y, factor.z })
			if (!std::isfinite(f) || f < 0.f) throw std::runtime_error("SetEmission: need a finite factor >= 0");
		emissionImage = std::move(image); emission.image = emissionImage.get(); emission.factor = factor;
	}
	MaterialEmission Emission() const { return emission; }
private:
	std::shared_ptr<ImageTexture> maskImage;
	MaterialAlphaMask mask;
	std::shared_ptr<ImageTexture> emissionImage;
	MaterialEmission emission;
};

#define AGPT_HAS_IMAGE_TEXTURES 1      // extension: DisneyMaterial(ImageTexture, roughness, metallic)
#define AGPT_HAS_MATERIAL_MAPS 1       // extension: DisneyMaterial::SetRoughnessMetallicMap / SetNormalMap
class DisneyMaterial : public Material {
public:
	DisneyMaterial(const float3& color, float roughness, float metallic) : color(color) {
		memset(&rec, 0, sizeof(rec));
		rec.type = AGPT_MAT_DISNEY;
		rec.eta = 1.5f;
		rec.roughness = roughness;
		rec.metallic = metallic;
		const float strans = 0.f;   // no transmission upstream (material.h:19)
		float diffuseWeight = (1 - metallic) * (1 - strans);
		if (diffuseWeight > 0) {    // diffuse + retro lobes exist iff metallic < 1 (material.h:27-36)
			float3 R = diffuseWeight * color;
			rec.diffuse_r[0] = R.x; rec.diffuse_r[1] = R.y; rec.diffuse_r[2] = R.z;
			rec.lobes |= AGPT_LOBE_DIFFUSE | AGPT_LOBE_RETRO;
		}
		const float aspect = 1.f;
		float ax = std::max(.001f, sqr(roughness) / aspect);
		float ay = std::max(.001f, sqr(roughness) * aspect);
		rec.alpha_x = std::max(0.001f, ax);   // clamped again by TrowbridgeReitzDistribution (microfacet.h:120-122)
		rec.alpha_y = std::max(0.001f, ay);
		const float specTint = 0.f;
		float r0 = sqr(rec.eta - 1) / sqr(rec.eta + 1);   // SchlickR0FromEta (disney.h:22)
		float3 Cspec0 = Lerp(metallic, r0 * Lerp(specTint, float3(1.f), float3(1.f)), color);
		rec.spec_r0[0] = Cspec0.x; rec.spec_r0[1] = Cspec0.y; rec.spec_r0[2] = Cspec0.z;
		rec.lobes |= AGPT_LOBE_MICROFACET;
	}
	// EXTENSION: the base colour is an image (include/agpt.h agpt_upload_textures).  The record holds white's colours; the
	// device replaces them at every hit by the texture value's, through the same arithmetic as the constructor above.
	DisneyMaterial(std::shared_ptr<ImageTexture> texture, float roughness, float metallic)
		: DisneyMaterial(float3(1.f), roughness, metallic) { this->texture = std::move(texture); }
	agpt_material Export() const override { return rec; }
	const ImageTexture* BaseColorTexture() const override { return texture.get(); }
	// EXTENSION (include/agpt.h agpt_upload_material_textures): a roughness-metallic map (G scales the roughness, B the metallic
	// of this material per hit) and a tangent-space normal map.  The colour the material was made with is kept: it is the base
	// colour of a material with maps and without a base-colour image.
	void SetRoughnessMetallicMap(std::shared_ptr<ImageTexture> map) { roughnessMetallic = std::move(map); }
	void SetNormalMap(std::shared_ptr<ImageTexture> map, float scale = 1.f) { normal = std::move(map); normalScale = scale; }
	MaterialMaps Maps() const override {
		MaterialMaps m;
		m.base = texture.get(); m.roughnessMetallic = roughnessMetallic.get(); m.normal = normal.get();
		m.normalScale = normalScale; m.color = color;
		return m;
	}
	static std::shared_ptr<DisneyMaterial> Make(const float3& color, float roughness, float metallic) {
		return std::make_shared<DisneyMaterial>(color, roughness, metallic);
	}
	static std::shared_ptr<DisneyMaterial> Make(std::shared_ptr<ImageTexture> texture, float roughness, float metallic) {
		return std::make_shared<DisneyMaterial>(std::move(texture), roughness, metallic);
	}
private:
	agpt_material rec;
	std::shared_ptr<ImageTexture> texture;
	float3 color;
	std::shared_ptr<ImageTexture> roughnessMetallic, normal;
	float normalScale = 1.f;
};

class MirrorMaterial : public Material {
public:
	MirrorMaterial(const float3& r) {
		memset(&rec, 0, sizeof(rec));
		rec.type = AGPT_MAT_MIRROR;
		rec.lobes = AGPT_LOBE_SPECULAR;
		rec.mirror_r[0] = r.x; rec.mirror_r[1] = r.y; rec.mirror_r[2] = r.z;
	}
	agpt_material Export() const override { return rec; }
	static std::shared_ptr<MirrorMaterial> Make(const float3& r) { return std::make_shared<MirrorMaterial>(r); }
private:
	agpt_material rec;
};

// EXTENSION (SURVEY 8f row 4; not a reference class): a rough dielectric interface as PBRT-v3's GlassMaterial builds
// it -- MicrofacetReflection(Kr, TrowbridgeReitz(alpha), FresnelDielectric(1, eta)), which the reference's own classes
// can express (reflection.h:38-78, microfacet.h:112-153,220-228), plus MicrofacetTransmission(Kt, ...), which they
// cannot.  alpha = max(.001, roughness^2) like DisneyMaterial (material.h:39-41).  transmit = false keeps the
// reflection lobe alone (the half that can be checked against the reference).  See include/agpt.h AGPT_LOBE_GLASS_*.
#define AGPT_HAS_GLASS 1
class GlassMaterial : public Material {
public:
	GlassMaterial(const float3& Kr, const float3& Kt, float roughness, float eta = 1.5f, bool transmit = true) {
		memset(&rec, 0, sizeof(rec));
		rec.type = AGPT_MAT_GLASS;
		rec.lobes = AGPT_LOBE_GLASS_REFLECT | (transmit ? AGPT_LOBE_GLASS_TRANSMIT : 0);
		rec.roughness = roughness;
		rec.eta = eta;
		rec.mirror_r[0] = Kr.x; rec.mirror_r[1] = Kr.y; rec.mirror_r[2] = Kr.z;
		rec.diffuse_r[0] = Kt.x; rec.diffuse_r[1] = Kt.y; rec.diffuse_r[2] = Kt.z;
		rec.alpha_x = rec.alpha_y = std::max(0.001f, std::max(.001f, sqr(roughness)));
	}
	agpt_material Export() const override { return rec; }
	static std::shared_ptr<GlassMaterial> Make(const float3& Kr, const float3& Kt, float roughness, float eta = 1.5f, bool transmit = true) {
		return std::make_shared<GlassMaterial>(Kr, Kt, roughness, eta, transmit);
	}
private:
	agpt_material rec;
};
