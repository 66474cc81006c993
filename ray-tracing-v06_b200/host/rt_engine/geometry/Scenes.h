// Host mirror of main/src/rt_engine/geometry/Scenes.h:55-92 (SceneBook2BVH and its Factory, same
// public surface) plus a registry of the scenes BASELINE.json's configs name.  Definitions in
// host/Scenes.cpp.
#pragma once
#include <vector>

#include "rtb.h"

class aabb; class BVH_Handle; class cuHostRND; class Hittable; class SphereHandle;

// The scene object FirstApp keeps alive while rendering: it owns the sphere handles (and through them the
// materials), the BVH handle and the world bounds.  Built only by its Factory; move-only.
class SceneBook2BVH {
public:
	class Factory;
	SceneBook2BVH(SceneBook2BVH&& scene);
	SceneBook2BVH& operator=(SceneBook2BVH&& scene);
	~SceneBook2BVH();
	const Hittable* getWorldPtr() const;   // what Renderer::MakeRenderer takes as d_world_ptr

private:
	SceneBook2BVH();
	void _delete();
	BVH_Handle* bvh; aabb* world_bounds;              // (declaration order = initialisation order of the constructors)
	std::vector<SphereHandle> sphere_handles;
};

// Draws the 22 x 22 grid of random spheres from a host generator (cuHostRND(512, 1984)) and hands the finished
// world over: Factory{}.MakeScene() is the whole public protocol (FirstApp.cpp:34-35).
class SceneBook2BVH::Factory {
public:
	Factory();
	Factory(Factory&& factory);
	Factory& operator=(Factory&& factory);
	~Factory();
	SceneBook2BVH* MakeScene();

private:
	void _populate_world();
	void _delete();
	cuHostRND* host_rnd;
	std::vector<SphereHandle> sphere_handles;
};

// ---- C accessors used by the Python tests / bench (exported from librtb200_scenes.so)
extern "C" {
typedef struct rtb_scene_info {
	rtb_camera camera;
	int32_t width, height, spp, max_depth;
	// The scene's emitters as its author names them for light sampling (Book 3's `lights` list): pass them to
	// rtb_scene_set_sampled_lights to turn it on.  The named scenes never do that themselves.
	int32_t n_lights, lights[8];
} rtb_scene_info;

int rtb_scenes_count(void);
const char* rtb_scenes_name(int index);
// Builds the named scene through the host mirror API; the caller owns the returned rtb_scene
// (root and background already set).  NULL on error (rtb_last_error / rtb_scenes_last_error).
rtb_scene* rtb_scenes_build(const char* name, rtb_scene_info* info);
const char* rtb_scenes_last_error(void);
}
