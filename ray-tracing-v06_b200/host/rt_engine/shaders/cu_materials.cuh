// Host mirror of main/src/rt_engine/shaders/cu_materials.cuh:17-144 (same class names, template
// parameters and constructor arguments) plus Book 2's diffuse_light and isotropic.  The Scatter
// bodies live in the shade kernel (csrc/rtb_kernels.cu).
#pragma once
#include <glm/glm.hpp>

#include "../../rtb_context.h"
#include "cu_Textures.cuh"
#include "material.cuh"

template <Geometry_t GeoType>
class LambertianTexture : public GeometryDependantMaterial<GeoType> {
public:
	LambertianTexture(glm::vec3 c1, glm::vec3 c2, float scale) {   // checker of two solids, cu_materials.cuh:23-27
		solid_texture a(c1), b(c2);
		checker_texture tex(&a, &b, scale);
		this->rtb_material = rtb_host::check(rtb_add_lambertian(rtb_host::scene(), tex.rtb_texture), "LambertianTexture");
	}
	explicit LambertianTexture(const Texture* tex) {
		this->rtb_material = rtb_host::check(rtb_add_lambertian(rtb_host::scene(), tex->rtb_texture), "LambertianTexture");
	}
};

template <Geometry_t GeoType>
class LambertianAbstract : public GeometryDependantMaterial<GeoType> {
public:
	LambertianAbstract() : LambertianAbstract(glm::vec3(1.0f)) {}
	LambertianAbstract(glm::vec3 albedo) { this->rtb_material = rtb_host::check(rtb_add_lambertian_color(rtb_host::scene(), &albedo.x), "LambertianAbstract"); }
};

template <Geometry_t GeoType>
class MetalAbstract : public GeometryDependantMaterial<GeoType> {
public:
	MetalAbstract() : MetalAbstract(glm::vec3(1.0f), 0.0f) {}
	MetalAbstract(glm::vec3 albedo, float fuzz) { this->rtb_material = rtb_host::check(rtb_add_metal(rtb_host::scene(), &albedo.x, fuzz), "MetalAbstract"); }
};

template <Geometry_t GeoType>
class DielectricAbstract : public GeometryDependantMaterial<GeoType> {
public:
	DielectricAbstract() : DielectricAbstract(glm::vec3(1.0f), 1.333f) {}
	DielectricAbstract(glm::vec3 albedo, float ior) { this->rtb_material = rtb_host::check(rtb_add_dielectric(rtb_host::scene(), &albedo.x, ior), "DielectricAbstract"); }
};

// Geometry-independent materials (material.cuh:31-36 reserves the base class for exactly this).
class Lambertian : public GeoIndependantMaterial {
public:
	Lambertian(glm::vec3 albedo) { rtb_material = rtb_host::check(rtb_add_lambertian_color(rtb_host::scene(), &albedo.x), "Lambertian"); }
	explicit Lambertian(const Texture* tex) { rtb_material = rtb_host::check(rtb_add_lambertian(rtb_host::scene(), tex->rtb_texture), "Lambertian"); }
};
class Metal : public GeoIndependantMaterial {
public:
	Metal(glm::vec3 albedo, float fuzz) { rtb_material = rtb_host::check(rtb_add_metal(rtb_host::scene(), &albedo.x, fuzz), "Metal"); }
};
class Dielectric : public GeoIndependantMaterial {
public:
	Dielectric(glm::vec3 albedo, float ior) { rtb_material = rtb_host::check(rtb_add_dielectric(rtb_host::scene(), &albedo.x, ior), "Dielectric"); }
};
// GGX microfacet materials (DESIGN.md §5f; not in the reference): width alpha in [0.001, 1].
class RoughMetal : public GeoIndependantMaterial {
public:
	RoughMetal(glm::vec3 f0, float alpha) { rtb_material = rtb_host::check(rtb_add_rough_metal(rtb_host::scene(), &f0.x, alpha), "RoughMetal"); }
};
class RoughDielectric : public GeoIndependantMaterial {
public:
	RoughDielectric(float ior, float alpha, glm::vec3 albedo = glm::vec3(1.0f)) {
		rtb_material = rtb_host::check(rtb_add_rough_dielectric(rtb_host::scene(), &albedo.x, ior, alpha), "RoughDielectric");
	}
};
class diffuse_light : public GeoIndependantMaterial {
public:
	diffuse_light(glm::vec3 emit) { solid_texture t(emit); rtb_material = rtb_host::check(rtb_add_diffuse_light(rtb_host::scene(), t.rtb_texture), "diffuse_light"); }
	explicit diffuse_light(const Texture* tex) { rtb_material = rtb_host::check(rtb_add_diffuse_light(rtb_host::scene(), tex->rtb_texture), "diffuse_light"); }
};
class isotropic : public GeoIndependantMaterial {
public:
	isotropic(glm::vec3 albedo) { solid_texture t(albedo); rtb_material = rtb_host::check(rtb_add_isotropic(rtb_host::scene(), t.rtb_texture), "isotropic"); }
	explicit isotropic(const Texture* tex) { rtb_material = rtb_host::check(rtb_add_isotropic(rtb_host::scene(), tex->rtb_texture), "isotropic"); }
};
