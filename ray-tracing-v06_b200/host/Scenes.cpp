// Scenes.cpp — scene builders written against the host mirror of the reference's API.
//
//   SceneBook2BVH::Factory   follows main/src/rt_engine/geometry/Scenes.cu:189-314 statement by
//                            statement (bouncing spheres, 488 objects, flat BVH, top-down median).
//   book1_final              the #if 0'd SceneBook1 recipe (Scenes.cu:57-136) with static spheres.
//   book2_* (textures, Cornell box with smoke, final scene)  do not exist in the reference; they are
//                            "Ray Tracing: The Next Week" scenes in the reference idiom (SURVEY.md App. B).
//
// Random draws come from cuHostRND(512, 1984) like the reference.  The reference draws several
// uniforms inside one expression (Scenes.cu:232,235,236,242), whose evaluation order C++ leaves
// unspecified; nvcc + g++ 13 evaluates those arguments right to left, and that order is written
// out explicitly here so the scene does not depend on the compiler.
#include "rt_engine/geometry/Scenes.h"

#include <cmath>
#include <cstdlib>
#include <unistd.h>
#include <cstring>
#include <functional>
#include <initializer_list>
#include <map>
#include <memory>
#include <string>
#include <tuple>

#include "rt_engine/geometry/BVH.cuh"
#include "rt_engine/geometry/HittableList.cuh"
#include "rt_engine/geometry/Mesh.cuh"
#include "rt_engine/geometry/Quad.cuh"
#include "rt_engine/geometry/SphereHittable.cuh"
#include "rt_engine/shaders/cu_Cameras.cuh"
#include "rt_engine/shaders/cu_materials.cuh"
#include "utilities/cuda_utilities/cuHostRND.h"
#include "utilities/cuda_utilities/cuda_utils.cuh"

// ------------------------------------------------------------------ SceneBook2BVH (reference scene)

SceneBook2BVH::SceneBook2BVH() = default;
SceneBook2BVH::~SceneBook2BVH() { _delete(); }
void SceneBook2BVH::_delete() {
	delete bvh; delete world_bounds; sphere_handles.clear();
	bvh = nullptr; world_bounds = nullptr;
}
SceneBook2BVH::SceneBook2BVH(SceneBook2BVH&& scene) : bvh(scene.bvh), world_bounds(scene.world_bounds), sphere_handles(std::move(scene.sphere_handles)) {
	scene.bvh = nullptr; scene.world_bounds = nullptr;
}
SceneBook2BVH& SceneBook2BVH::operator=(SceneBook2BVH&& scene) {
	_delete();
	bvh = scene.bvh; world_bounds = scene.world_bounds; sphere_handles = std::move(scene.sphere_handles);
	scene.bvh = nullptr; scene.world_bounds = nullptr;
	return *this;
}
const Hittable* SceneBook2BVH::getWorldPtr() const { return bvh->getBVHPtr(); }

SceneBook2BVH::Factory::Factory() { host_rnd = new cuHostRND(512, 1984); }
SceneBook2BVH::Factory::~Factory() { _delete(); }
void SceneBook2BVH::Factory::_delete() { delete host_rnd; sphere_handles.clear(); host_rnd = nullptr; }
SceneBook2BVH::Factory::Factory(Factory&& f) : host_rnd(f.host_rnd), sphere_handles(std::move(f.sphere_handles)) { f.host_rnd = nullptr; }
SceneBook2BVH::Factory& SceneBook2BVH::Factory::operator=(Factory&& f) {
	_delete();
	host_rnd = f.host_rnd; sphere_handles = std::move(f.sphere_handles); f.host_rnd = nullptr;
	return *this;
}

namespace {

// The 22 x 22 grid of small spheres shared by Book 1's final scene and Book 2's bouncing spheres
// (Scenes.cu:225-254).  `moving` selects MovingSphere Lambertians (Book 2) or static ones (Book 1).
void populate_random_grid(cuHostRND& host_rnd, std::vector<SphereHandle>& sphere_handles, bool moving) {
	auto rnd = [&]() { return host_rnd.next(); };
	for (int a = -11; a < 11; a++) {
		for (int b = -11; b < 11; b++) {
			float choose_mat = rnd();
			// glm::vec3 center(a + rnd, 0.2f, b + rnd): last argument first
			float cz = b + rnd();
			float cx = a + rnd();
			glm::vec3 center(cx, 0.2f, cz);

			if (choose_mat < 0.8f) {
				// glm::vec3(rnd * rnd, rnd * rnd, rnd * rnd): blue, green, red
				float bl = rnd() * rnd();
				float gr = rnd() * rnd();
				float rd = rnd() * rnd();
				if (moving) {
					auto material = newOnDevice<LambertianAbstract<MovingSphere>>(glm::vec3(rd, gr, bl));
					glm::vec3 center1 = center + glm::vec3(0, rnd() * 0.5f, 0);
					auto moving_sphere = MovingSphere(center, center1, 0.2f);
					sphere_handles.push_back(SphereHandle::MakeMovingSphere(moving_sphere, material));
				} else {
					auto material = newOnDevice<LambertianAbstract<Sphere>>(glm::vec3(rd, gr, bl));
					sphere_handles.push_back(SphereHandle::MakeSphere(Sphere(center, 0.2f), material));
				}
			} else if (choose_mat < 0.95f) {
				// newOnDevice<Metal>(glm::vec3(.5(1+rnd), .5(1+rnd), .5(1+rnd)), 0.5f * rnd): fuzz first, then b, g, r
				float fuzz = 0.5f * rnd();
				float bl = 0.5f * (1.0f + rnd());
				float gr = 0.5f * (1.0f + rnd());
				float rd = 0.5f * (1.0f + rnd());
				auto material = newOnDevice<MetalAbstract<Sphere>>(glm::vec3(rd, gr, bl), fuzz);
				sphere_handles.push_back(SphereHandle::MakeSphere(Sphere(center, 0.2f), material));
			} else {
				auto material = newOnDevice<DielectricAbstract<Sphere>>(glm::vec3(1.0f), 1.5f);
				sphere_handles.push_back(SphereHandle::MakeSphere(Sphere(center, 0.2f), material));
			}
		}
	}
}

void populate_spheres_world(cuHostRND& host_rnd, std::vector<SphereHandle>& sphere_handles, bool moving) {
	Sphere ground_sphere = Sphere(glm::vec3(0, -1000, 0), 1000.0f);
	auto ground_mat = newOnDevice<LambertianAbstract<Sphere>>(glm::vec3(0.5f));
	sphere_handles.push_back(SphereHandle::MakeSphere(ground_sphere, ground_mat));

	populate_random_grid(host_rnd, sphere_handles, moving);

	auto center_mat = newOnDevice<DielectricAbstract<Sphere>>(glm::vec3(1.0f), 1.5f);
	sphere_handles.push_back(SphereHandle::MakeSphere(Sphere(glm::vec3(0, 1, 0), 1), center_mat));
	auto left_mat = newOnDevice<LambertianAbstract<Sphere>>(glm::vec3(0.4f, 0.2f, 0.1f));
	sphere_handles.push_back(SphereHandle::MakeSphere(Sphere(glm::vec3(-4, 1, 0), 1), left_mat));
	auto right_mat = newOnDevice<MetalAbstract<Sphere>>(glm::vec3(0.7f, 0.6f, 0.5f), 0);
	sphere_handles.push_back(SphereHandle::MakeSphere(Sphere(glm::vec3(4, 1, 0), 1), right_mat));
}

}  // namespace

void SceneBook2BVH::Factory::_populate_world() { populate_spheres_world(*host_rnd, sphere_handles, true); }

SceneBook2BVH* SceneBook2BVH::Factory::MakeScene() {
	_populate_world();

	std::vector<std::tuple<aabb, const Hittable*>> objects;
	objects.reserve(sphere_handles.size());
	for (size_t i = 0; i < sphere_handles.size(); i++)
		objects.push_back(std::make_tuple(sphere_handles[i].getBounds(), sphere_handles[i].getHittablePtr()));

	BVH_Handle::Factory bvh_factory(objects);
	bvh_factory.BuildBVH_TopDown();
	BVH_Handle* bvh_handle = bvh_factory.MakeHandle();

	auto scene = new SceneBook2BVH();
	scene->bvh = bvh_handle;
	scene->world_bounds = new aabb(scene->bvh->getBounds());
	scene->sphere_handles = std::move(sphere_handles);
	return scene;
}

// ------------------------------------------------------------------ registry of the BASELINE.json scenes

namespace {

thread_local std::string g_scene_err;

// Keeps handles (and the host proxies they own) alive until the scene is finished.  Materials and
// textures registered here are shared between objects, so handles are created non-owning.
struct Keep {
	std::vector<SphereHandle> spheres;
	std::vector<GeoHandle> geos;
	std::vector<std::unique_ptr<BVH_Handle>> bvhs;
	std::vector<std::unique_ptr<HittableList>> lists;
	std::vector<std::unique_ptr<Texture>> textures;
	std::vector<std::unique_ptr<Material>> materials;

	template <typename M> M* mat(M* m) { materials.emplace_back(m); return m; }
	template <typename T> T* tex(T* t) { textures.emplace_back(t); return t; }
	template <typename M> const Hittable* sphere(const Sphere& s, M* m) {
		spheres.push_back(SphereHandle::MakeSphere(s, m, false)); return spheres.back().getHittablePtr();
	}
	template <typename M> const Hittable* moving_sphere(const MovingSphere& s, M* m) {
		spheres.push_back(SphereHandle::MakeMovingSphere(s, m, false)); return spheres.back().getHittablePtr();
	}
	template <typename M> const Hittable* quad(glm::vec3 Q, glm::vec3 u, glm::vec3 v, M* m) {
		geos.push_back(GeoHandle::MakeQuad(Quad(Q, u, v), m)); return geos.back().getHittablePtr();
	}
	template <typename M> const Hittable* box(glm::vec3 a, glm::vec3 b, M* m) {
		geos.push_back(GeoHandle::MakeBox(Box(a, b), m)); return geos.back().getHittablePtr();
	}
	const Hittable* translate(const Hittable* c, glm::vec3 off) { geos.push_back(GeoHandle::MakeTranslate(c, off)); return geos.back().getHittablePtr(); }
	const Hittable* rotate_y(const Hittable* c, float deg) { geos.push_back(GeoHandle::MakeRotateY(c, deg)); return geos.back().getHittablePtr(); }
	template <typename M> const Hittable* medium(const Hittable* boundary, float density, M* phase) {
		geos.push_back(GeoHandle::MakeConstantMedium(boundary, density, phase)); return geos.back().getHittablePtr();
	}
	aabb bounds_of(const Hittable* h) {
		float b[6]; rtb_host::check(rtb_object_bounds(rtb_host::scene(), h->rtb_object, b), "rtb_object_bounds");
		return aabb(glm::vec3(b[0], b[1], b[2]), glm::vec3(b[3], b[4], b[5]));
	}
	const Hittable* list(std::vector<const Hittable*>& objs) {
		aabb bounds;
		for (auto* o : objs) bounds += bounds_of(o);
		lists.emplace_back(new HittableList(objs.data(), (int)objs.size(), bounds));
		return lists.back().get();
	}
	const Hittable* bvh(std::vector<const Hittable*>& objs) {   // bvh_node of the book = flat BVH, top-down median (BVH.cu:166-210)
		std::vector<std::tuple<aabb, const Hittable*>> arr;
		for (auto* o : objs) arr.push_back(std::make_tuple(bounds_of(o), o));
		BVH_Handle::Factory f(arr);
		f.BuildBVH_TopDown();
		bvhs.emplace_back(f.MakeHandle());
		return bvhs.back()->getBVHPtr();
	}
};

// `lights`: the emitters a user would hand to light sampling (rtb_scene_info::lights); they are only listed, not set.
void finish(rtb_scene_info* info, const Hittable* world, const rtb_camera& cam, int w, int h, int spp, int depth, bool black_background,
            std::initializer_list<const Hittable*> lights = {}) {
	rtb_host::check(rtb_scene_set_root(rtb_host::scene(), world->rtb_object), "rtb_scene_set_root");
	const float black[3] = {0, 0, 0};
	rtb_host::check(rtb_scene_set_background(rtb_host::scene(), black_background ? RTB_BG_CONSTANT : RTB_BG_SKY_GRADIENT, black), "rtb_scene_set_background");
	if (info) {
		info->camera = cam; info->width = w; info->height = h; info->spp = spp; info->max_depth = depth;
		info->n_lights = 0;
		for (const Hittable* l : lights) if (info->n_lights < 8) info->lights[info->n_lights++] = l->rtb_object;
	}
}

rtb_camera book2_camera(glm::vec3 from, glm::vec3 at, float vfov, float aspect) {
	// Book 2 cameras: no defocus, shutter [0,1)
	return MotionBlurCamera(from, at, glm::vec3(0, 1, 0), vfov, aspect, 0.0f, 1.0f).to_rtb();
}

// Config 1 — Book 1 final scene: SceneBook1's recipe (Scenes.cu:57-136, HittableList world) with the
// book's static Lambertian spheres and defocus camera.
void build_book1_final(rtb_scene_info* info) {
	std::vector<SphereHandle> handles;
	cuHostRND rnd(512, 1984);
	populate_spheres_world(rnd, handles, false);
	std::vector<const Hittable*> objs;
	aabb bounds;
	for (auto& s : handles) { objs.push_back(s.getHittablePtr()); bounds += s.getBounds(); }
	HittableList world(objs.data(), (int)objs.size(), bounds);
	DefocusBlurCamera cam(glm::vec3(13, 2, 3), glm::vec3(0, 0, 0), glm::vec3(0, 1, 0), 20.0f, 1200.0f / 675.0f, 0.1f, 10.0f);
	finish(info, &world, cam.to_rtb(), 1200, 675, 10, 50, false);
}

// Config 2 — Book 2 bouncing spheres = the reference's SceneBook2BVH, camera of FirstApp.cpp:24-30.
void build_book2_bouncing(rtb_scene_info* info) {
	SceneBook2BVH::Factory factory{};
	std::unique_ptr<SceneBook2BVH> scene(factory.MakeScene());
	MotionBlurCamera cam(glm::vec3(13, 2, 3), glm::vec3(0, 0, 0), glm::vec3(0, 1, 0), 30.0f, 400.0f / 225.0f, 0.1f, 1.0f);
	finish(info, scene->getWorldPtr(), cam.to_rtb(), 400, 225, 100, 50, false);
}

// Config 3a — checkered spheres
void build_book2_checker(rtb_scene_info* info) {
	Keep k;
	auto even = k.tex(new solid_texture(glm::vec3(.2f, .3f, .1f)));
	auto odd = k.tex(new solid_texture(glm::vec3(.9f, .9f, .9f)));
	auto checker = k.tex(new checker_texture(even, odd, 0.32f));
	auto m = k.mat(new Lambertian(checker));
	std::vector<const Hittable*> objs{k.sphere(Sphere(glm::vec3(0, -10, 0), 10), m), k.sphere(Sphere(glm::vec3(0, 10, 0), 10), m)};
	finish(info, k.list(objs), book2_camera(glm::vec3(13, 2, 3), glm::vec3(0), 20.0f, 400.0f / 225.0f), 400, 225, 100, 50, false);
}

// A procedural latitude/longitude "globe" standing in for the book's earthmap.jpg (the reference ships no
// earth map; its only images live outside this repository).
std::vector<uint8_t> make_globe_image(int W, int H) {
	std::vector<uint8_t> px((size_t)W * H * 3);
	for (int j = 0; j < H; ++j) for (int i = 0; i < W; ++i) {
		float lon = (i + 0.5f) / W * 6.2831853f, lat = ((j + 0.5f) / H - 0.5f) * 3.14159265f;
		float land = sinf(3.0f * lon + 1.3f) * cosf(2.0f * lat) + 0.6f * sinf(5.0f * lon - 2.0f * lat) + 0.4f * cosf(7.0f * lat + lon);
		float r, g, b;
		if (fabsf(lat) > 1.35f) { r = g = b = 0.92f; }
		else if (land > 0.35f) { float h = fminf((land - 0.35f) * 1.5f, 1.0f); r = 0.25f + 0.45f * h; g = 0.55f - 0.15f * h; b = 0.18f + 0.1f * h; }
		else { float d = fminf((0.35f - land) * 0.6f, 1.0f); r = 0.05f; g = 0.25f - 0.12f * d; b = 0.65f - 0.3f * d; }
		bool grid = (i % (W / 24) == 0) || (j % (H / 12) == 0);
		if (grid) { r *= 0.8f; g *= 0.8f; b *= 0.8f; }
		uint8_t* p = &px[3 * ((size_t)j * W + i)];
		p[0] = (uint8_t)(r * 255.0f); p[1] = (uint8_t)(g * 255.0f); p[2] = (uint8_t)(b * 255.0f);
	}
	return px;
}

// Config 3b — image-textured sphere
void build_book2_earth(rtb_scene_info* info) {
	Keep k;
	auto img = make_globe_image(1024, 512);
	auto tex = k.tex(new image_texture(img.data(), 1024, 512, 3));
	auto m = k.mat(new Lambertian(tex));
	std::vector<const Hittable*> objs{k.sphere(Sphere(glm::vec3(0, 0, 0), 2), m)};
	finish(info, k.list(objs), book2_camera(glm::vec3(0, 0, 12), glm::vec3(0), 20.0f, 400.0f / 225.0f), 400, 225, 100, 50, false);
}

// Config 3c — Perlin marble spheres
void build_book2_perlin(rtb_scene_info* info) {
	Keep k;
	auto tex = k.tex(new noise_texture(4.0f, 1984));
	auto m = k.mat(new Lambertian(tex));
	std::vector<const Hittable*> objs{k.sphere(Sphere(glm::vec3(0, -1000, 0), 1000), m), k.sphere(Sphere(glm::vec3(0, 2, 0), 2), m)};
	finish(info, k.list(objs), book2_camera(glm::vec3(13, 2, 3), glm::vec3(0), 20.0f, 400.0f / 225.0f), 400, 225, 100, 50, false);
}

// Book 2 "quads" scene (five coloured quads)
void build_book2_quads(rtb_scene_info* info) {
	Keep k;
	auto red = k.mat(new Lambertian(glm::vec3(1.0f, 0.2f, 0.2f))), green = k.mat(new Lambertian(glm::vec3(0.2f, 1.0f, 0.2f)));
	auto blue = k.mat(new Lambertian(glm::vec3(0.2f, 0.2f, 1.0f))), orange = k.mat(new Lambertian(glm::vec3(1.0f, 0.5f, 0.0f)));
	auto teal = k.mat(new Lambertian(glm::vec3(0.2f, 0.8f, 0.8f)));
	std::vector<const Hittable*> objs{
	    k.quad(glm::vec3(-3, -2, 5), glm::vec3(0, 0, -4), glm::vec3(0, 4, 0), red), k.quad(glm::vec3(-2, -2, 0), glm::vec3(4, 0, 0), glm::vec3(0, 4, 0), green),
	    k.quad(glm::vec3(3, -2, 1), glm::vec3(0, 0, 4), glm::vec3(0, 4, 0), blue), k.quad(glm::vec3(-2, 3, 1), glm::vec3(4, 0, 0), glm::vec3(0, 0, 4), orange),
	    k.quad(glm::vec3(-2, -3, 5), glm::vec3(4, 0, 0), glm::vec3(0, 0, -4), teal)};
	finish(info, k.list(objs), book2_camera(glm::vec3(0, 0, 9), glm::vec3(0), 80.0f, 1.0f), 400, 400, 100, 50, false);
}

// Book 2 "simple light" scene (Perlin spheres lit by a quad and a sphere light)
void build_book2_simple_light(rtb_scene_info* info) {
	Keep k;
	auto pertext = k.tex(new noise_texture(4.0f, 1984));
	auto m = k.mat(new Lambertian(pertext));
	auto light = k.mat(new diffuse_light(glm::vec3(4, 4, 4)));
	std::vector<const Hittable*> objs{k.sphere(Sphere(glm::vec3(0, -1000, 0), 1000), m), k.sphere(Sphere(glm::vec3(0, 2, 0), 2), m),
	                                  k.sphere(Sphere(glm::vec3(0, 7, 0), 2), light), k.quad(glm::vec3(3, 1, -2), glm::vec3(2, 0, 0), glm::vec3(0, 2, 0), light)};
	finish(info, k.list(objs), book2_camera(glm::vec3(26, 3, 6), glm::vec3(0, 2, 0), 20.0f, 400.0f / 225.0f), 400, 225, 100, 50, true, {objs[2], objs[3]});
}

void cornell_walls(Keep& k, std::vector<const Hittable*>& objs, glm::vec3 light_q, glm::vec3 light_u, glm::vec3 light_v, glm::vec3 emit) {
	auto red = k.mat(new Lambertian(glm::vec3(.65f, .05f, .05f))), white = k.mat(new Lambertian(glm::vec3(.73f, .73f, .73f)));
	auto green = k.mat(new Lambertian(glm::vec3(.12f, .45f, .15f)));
	auto light = k.mat(new diffuse_light(emit));
	objs.push_back(k.quad(glm::vec3(555, 0, 0), glm::vec3(0, 555, 0), glm::vec3(0, 0, 555), green));
	objs.push_back(k.quad(glm::vec3(0, 0, 0), glm::vec3(0, 555, 0), glm::vec3(0, 0, 555), red));
	objs.push_back(k.quad(light_q, light_u, light_v, light));
	objs.push_back(k.quad(glm::vec3(0, 0, 0), glm::vec3(555, 0, 0), glm::vec3(0, 0, 555), white));
	objs.push_back(k.quad(glm::vec3(555, 555, 555), glm::vec3(-555, 0, 0), glm::vec3(0, 0, -555), white));
	objs.push_back(k.quad(glm::vec3(0, 0, 555), glm::vec3(555, 0, 0), glm::vec3(0, 555, 0), white));
}

// Book 2 Cornell box with two rotated solid boxes
void build_book2_cornell(rtb_scene_info* info) {
	Keep k; std::vector<const Hittable*> objs;
	cornell_walls(k, objs, glm::vec3(343, 554, 332), glm::vec3(-130, 0, 0), glm::vec3(0, 0, -105), glm::vec3(15, 15, 15));
	auto white = k.mat(new Lambertian(glm::vec3(.73f, .73f, .73f)));
	objs.push_back(k.translate(k.rotate_y(k.box(glm::vec3(0, 0, 0), glm::vec3(165, 330, 165), white), 15.0f), glm::vec3(265, 0, 295)));
	objs.push_back(k.translate(k.rotate_y(k.box(glm::vec3(0, 0, 0), glm::vec3(165, 165, 165), white), -18.0f), glm::vec3(130, 0, 65)));
	finish(info, k.list(objs), book2_camera(glm::vec3(278, 278, -800), glm::vec3(278, 278, 0), 40.0f, 1.0f), 600, 600, 200, 50, true, {objs[2]});
}

// Config 4 — Cornell box, the two rotated boxes as smoke / fog
void build_book2_cornell_smoke(rtb_scene_info* info) {
	Keep k; std::vector<const Hittable*> objs;
	cornell_walls(k, objs, glm::vec3(113, 554, 127), glm::vec3(330, 0, 0), glm::vec3(0, 0, 305), glm::vec3(7, 7, 7));
	auto white = k.mat(new Lambertian(glm::vec3(.73f, .73f, .73f)));
	auto box1 = k.translate(k.rotate_y(k.box(glm::vec3(0, 0, 0), glm::vec3(165, 330, 165), white), 15.0f), glm::vec3(265, 0, 295));
	auto box2 = k.translate(k.rotate_y(k.box(glm::vec3(0, 0, 0), glm::vec3(165, 165, 165), white), -18.0f), glm::vec3(130, 0, 65));
	objs.push_back(k.medium(box1, 0.01f, k.mat(new isotropic(glm::vec3(0, 0, 0)))));
	objs.push_back(k.medium(box2, 0.01f, k.mat(new isotropic(glm::vec3(1, 1, 1)))));
	finish(info, k.list(objs), book2_camera(glm::vec3(278, 278, -800), glm::vec3(278, 278, 0), 40.0f, 1.0f), 600, 600, 1000, 50, true, {objs[2]});
}

// Config 5 — Book 2 final scene.  Random draws from cuHostRND(512, 1984), one per statement.
void build_book2_final(rtb_scene_info* info) {
	Keep k;
	cuHostRND rnd(512, 1984);
	auto ground = k.mat(new Lambertian(glm::vec3(0.48f, 0.83f, 0.53f)));
	std::vector<const Hittable*> boxes1;
	const int boxes_per_side = 20;
	for (int i = 0; i < boxes_per_side; i++) for (int j = 0; j < boxes_per_side; j++) {
		float w = 100.0f;
		float x0 = -1000.0f + i * w, z0 = -1000.0f + j * w, y0 = 0.0f;
		float x1 = x0 + w, y1 = 1.0f + 100.0f * rnd.next(), z1 = z0 + w;
		boxes1.push_back(k.box(glm::vec3(x0, y0, z0), glm::vec3(x1, y1, z1), ground));
	}
	std::vector<const Hittable*> world;
	world.push_back(k.bvh(boxes1));

	auto light = k.mat(new diffuse_light(glm::vec3(7, 7, 7)));
	world.push_back(k.quad(glm::vec3(123, 554, 147), glm::vec3(300, 0, 0), glm::vec3(0, 0, 265), light));

	auto sphere_material = k.mat(new Lambertian(glm::vec3(0.7f, 0.3f, 0.1f)));
	world.push_back(k.moving_sphere(MovingSphere(glm::vec3(400, 400, 200), glm::vec3(430, 400, 200), 50), sphere_material));

	world.push_back(k.sphere(Sphere(glm::vec3(260, 150, 45), 50), k.mat(new Dielectric(glm::vec3(1.0f), 1.5f))));
	world.push_back(k.sphere(Sphere(glm::vec3(0, 150, 145), 50), k.mat(new Metal(glm::vec3(0.8f, 0.8f, 0.9f), 1.0f))));

	auto boundary = k.sphere(Sphere(glm::vec3(360, 150, 145), 70), k.mat(new Dielectric(glm::vec3(1.0f), 1.5f)));
	world.push_back(boundary);
	world.push_back(k.medium(boundary, 0.2f, k.mat(new isotropic(glm::vec3(0.2f, 0.4f, 0.9f)))));
	auto fog_boundary = k.sphere(Sphere(glm::vec3(0, 0, 0), 5000), k.mat(new Dielectric(glm::vec3(1.0f), 1.5f)));
	world.push_back(k.medium(fog_boundary, 0.0001f, k.mat(new isotropic(glm::vec3(1, 1, 1)))));

	auto img = make_globe_image(1024, 512);
	auto emat = k.mat(new Lambertian(k.tex(new image_texture(img.data(), 1024, 512, 3))));
	world.push_back(k.sphere(Sphere(glm::vec3(400, 200, 400), 100), emat));
	auto pertext = k.tex(new noise_texture(0.2f, 1984));
	world.push_back(k.sphere(Sphere(glm::vec3(220, 280, 300), 80), k.mat(new Lambertian(pertext))));

	std::vector<const Hittable*> boxes2;
	auto white = k.mat(new Lambertian(glm::vec3(.73f, .73f, .73f)));
	for (int j = 0; j < 1000; j++) {
		float x = 165.0f * rnd.next();
		float y = 165.0f * rnd.next();
		float z = 165.0f * rnd.next();
		boxes2.push_back(k.sphere(Sphere(glm::vec3(x, y, z), 10), white));
	}
	world.push_back(k.translate(k.rotate_y(k.bvh(boxes2), 15.0f), glm::vec3(-100, 270, 395)));

	finish(info, k.list(world), book2_camera(glm::vec3(478, 278, -600), glm::vec3(278, 278, 0), 40.0f, 1.0f), 800, 800, 10000, 40, true, {world[1]});
}

// A procedural triangle mesh (a subdivided icosahedron, 1,280 faces) written to and read back through the OBJ
// loader: the triangle path of the renderer on a closed mesh, glass over a checkered ground, next to a metal copy.
std::string write_icosphere_obj(int subdivisions) {
	std::vector<glm::vec3> v; std::vector<int> f;
	const float t = (1.0f + sqrtf(5.0f)) * 0.5f;
	const float P[12][3] = {{-1, t, 0}, {1, t, 0}, {-1, -t, 0}, {1, -t, 0}, {0, -1, t}, {0, 1, t}, {0, -1, -t}, {0, 1, -t}, {t, 0, -1}, {t, 0, 1}, {-t, 0, -1}, {-t, 0, 1}};
	const int F[20][3] = {{0, 11, 5}, {0, 5, 1}, {0, 1, 7}, {0, 7, 10}, {0, 10, 11}, {1, 5, 9}, {5, 11, 4}, {11, 10, 2}, {10, 7, 6}, {7, 1, 8},
	                      {3, 9, 4}, {3, 4, 2}, {3, 2, 6}, {3, 6, 8}, {3, 8, 9}, {4, 9, 5}, {2, 4, 11}, {6, 2, 10}, {8, 6, 7}, {9, 8, 1}};
	for (auto& p : P) v.push_back(glm::normalize(glm::vec3(p[0], p[1], p[2])));
	for (auto& q : F) { f.push_back(q[0]); f.push_back(q[1]); f.push_back(q[2]); }
	for (int s = 0; s < subdivisions; ++s) {
		std::vector<int> nf; std::map<std::pair<int, int>, int> mid;
		auto midpoint = [&](int a, int b) {
			auto key = std::make_pair(a < b ? a : b, a < b ? b : a);
			auto it = mid.find(key); if (it != mid.end()) return it->second;
			v.push_back(glm::normalize((v[a] + v[b]) * 0.5f)); return mid[key] = (int)v.size() - 1;
		};
		for (size_t k = 0; k < f.size(); k += 3) {
			int a = f[k], b = f[k + 1], c = f[k + 2], ab = midpoint(a, b), bc = midpoint(b, c), ca = midpoint(c, a);
			int tri[12] = {a, ab, ca, b, bc, ab, c, ca, bc, ab, bc, ca};
			nf.insert(nf.end(), tri, tri + 12);
		}
		f.swap(nf);
	}
	// a private temporary file (several ranks build this scene at the same time): mkstemp, unlinked by the caller after loading
	char tmpl[] = "/tmp/rtb_icosphere_XXXXXX";
	const int fd = mkstemp(tmpl);
	if (fd < 0) throw std::runtime_error("cannot create a temporary file for the icosphere");
	std::string path = tmpl;
	FILE* o = fdopen(fd, "w");
	if (!o) { close(fd); throw std::runtime_error("cannot write " + path); }
	fprintf(o, "# icosphere, %zu vertices, %zu faces\n", v.size(), f.size() / 3);
	for (auto& p : v) fprintf(o, "v %.9g %.9g %.9g\n", p.x, p.y, p.z);
	for (size_t k = 0; k < f.size(); k += 3) fprintf(o, "f %d//%d %d//%d %d//%d\n", f[k] + 1, f[k] + 1, f[k + 1] + 1, f[k + 1] + 1, f[k + 2] + 1, f[k + 2] + 1);
	fclose(o);
	return path;
}

void build_mesh_icospheres(rtb_scene_info* info) {
	Keep k;
	const std::string obj = write_icosphere_obj(3);
	Mesh mesh = MeshHandle::LoadObj(obj);
	unlink(obj.c_str());
	auto even = k.tex(new solid_texture(glm::vec3(.2f, .3f, .1f)));
	auto odd = k.tex(new solid_texture(glm::vec3(.9f, .9f, .9f)));
	auto ground = k.mat(new Lambertian(k.tex(new checker_texture(even, odd, 0.8f))));
	auto glass = k.mat(new Dielectric(glm::vec3(1.0f), 1.5f));
	auto metal = k.mat(new Metal(glm::vec3(0.8f, 0.6f, 0.2f), 0.05f));
	std::vector<MeshHandle> meshes;
	meshes.push_back(MeshHandle::MakeMesh(mesh, glass));
	meshes.push_back(MeshHandle::MakeMesh(mesh, metal));
	std::vector<const Hittable*> objs{k.quad(glm::vec3(-20, -1, -20), glm::vec3(40, 0, 0), glm::vec3(0, 0, 40), ground),
	                                  k.translate(meshes[0].getHittablePtr(), glm::vec3(-1.2f, 0, 0)),
	                                  k.translate(k.rotate_y(meshes[1].getHittablePtr(), 30.0f), glm::vec3(1.2f, 0, 0.5f))};
	finish(info, k.list(objs), book2_camera(glm::vec3(0, 1.5f, -6), glm::vec3(0, 0, 0), 35.0f, 400.0f / 225.0f), 400, 225, 100, 50, false);
}

struct Entry { const char* name; void (*build)(rtb_scene_info*); };
const Entry kScenes[] = {
    {"book1_final", build_book1_final},           {"book2_bouncing", build_book2_bouncing},
    {"book2_checker", build_book2_checker},       {"book2_earth", build_book2_earth},
    {"book2_perlin", build_book2_perlin},         {"book2_quads", build_book2_quads},
    {"book2_simple_light", build_book2_simple_light}, {"book2_cornell", build_book2_cornell},
    {"book2_cornell_smoke", build_book2_cornell_smoke}, {"book2_final", build_book2_final},
    {"mesh_icospheres", build_mesh_icospheres},
};

}  // namespace

extern "C" {

int rtb_scenes_count(void) { return (int)(sizeof(kScenes) / sizeof(kScenes[0])); }
const char* rtb_scenes_name(int i) { return (i >= 0 && i < rtb_scenes_count()) ? kScenes[i].name : nullptr; }
const char* rtb_scenes_last_error(void) { return g_scene_err.c_str(); }

rtb_scene* rtb_scenes_build(const char* name, rtb_scene_info* info) {
	if (!name) { g_scene_err = "null scene name"; return nullptr; }
	for (const Entry& e : kScenes) {
		if (strcmp(e.name, name) != 0) continue;
		try {
			rtb_host::new_scene();
			e.build(info);
			return rtb_host::release_scene();
		} catch (const std::exception& ex) {
			g_scene_err = ex.what();
			rtb_host::new_scene();
			return nullptr;
		}
	}
	g_scene_err = std::string("unknown scene: ") + name;
	return nullptr;
}

}  // extern "C"
