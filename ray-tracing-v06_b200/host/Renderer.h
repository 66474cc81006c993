// Host mirror of main/src/Renderer.{h,cu}: Renderer::MakeRenderer / Render / DownloadRenderbuffer
// with the reference's signatures (Renderer.h:38-46).  MakeRenderer flattens and uploads the scene
// that `d_world_ptr` is the root of; Render launches the wavefront kernels through rtb_render and
// waits (the reference's Render is synchronous too, Renderer.cu:132-133); the camera is read at
// Render time (Renderer.cu:117).  Overloads for the other two camera PODs are an extension, and so is the number of GPUs:
// with RTB_GPUS=<n> in the environment (or Renderer::UseGpus(n) before MakeRenderer) the same three calls drive n GPUs of
// the box through rtb_multi_renderer - the sample range split over the devices, one reduction of the radiance sums.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <glm/glm.hpp>
#include <stdexcept>
#include <string>
#include <vector>

#include "rt_engine/geometry/HittableList.cuh"
#include "rt_engine/geometry/hittable.cuh"
#include "rt_engine/shaders/cu_Cameras.cuh"
#include "rtb_context.h"

class Renderer {
	struct M {
		uint32_t render_width{}, render_height{};
		uint32_t samples_per_pixel{}, max_depth{};
		const MotionBlurCamera* cam{};
		const DefocusBlurCamera* defocus_cam{};
		const PinholeCamera* pinhole_cam{};
		rtb_renderer* r{};
		rtb_multi_renderer* mr{};
		rtb_scene* scene{};
		uint32_t seed{1984};
		float noise_tolerance{-1.0f};   // < 0: uniform sampling
		uint32_t noise_min_spp{};
		rtb_adaptive_stats last_adaptive{};
		double last_render_ms{};
		uint64_t last_rays{}, last_paths{};
	} m;

	static int& _gpus() { static int n = 0; return n; }
	void _delete() { if (m.r) rtb_renderer_destroy(m.r); if (m.mr) rtb_multi_renderer_destroy(m.mr); m.r = nullptr; m.mr = nullptr; }
	Renderer(M m) : m(m) {}
	Renderer(const Renderer&) = delete;
	Renderer& operator=(const Renderer&) = delete;

	static Renderer _make(uint32_t w, uint32_t h, uint32_t spp, uint32_t depth, const Hittable* world, M m) {
		rtb_scene* s = rtb_host::scene();
		rtb_host::check(rtb_scene_set_root(s, world->rtb_object), "rtb_scene_set_root");
		int gpus = _gpus();
		if (gpus <= 0) if (const char* e = getenv("RTB_GPUS")) gpus = atoi(e);
		if (gpus > 1) {
			rtb_host::check(rtb_multi_renderer_create(&m.mr, nullptr, gpus, RTB_REDUCE_AUTO), "rtb_multi_renderer_create");
			rtb_host::check(rtb_multi_set_scene(m.mr, s), "rtb_multi_set_scene");
		} else {
			rtb_host::check(rtb_renderer_create(&m.r, 0), "rtb_renderer_create");
			rtb_host::check(rtb_renderer_set_scene(m.r, s), "rtb_renderer_set_scene");
		}
		m.render_width = w; m.render_height = h; m.samples_per_pixel = spp; m.max_depth = depth; m.scene = s;
		return Renderer(m);
	}

public:
	~Renderer() { _delete(); }
	Renderer(Renderer&& o) noexcept : m(o.m) { o.m.r = nullptr; o.m.mr = nullptr; }
	Renderer& operator=(Renderer&& o) noexcept { if (this != &o) { _delete(); m = o.m; o.m.r = nullptr; o.m.mr = nullptr; } return *this; }

	// How many GPUs of the box the next MakeRenderer uses (0: RTB_GPUS from the environment, else one).
	static void UseGpus(int n) { _gpus() = n; }
	void SetSeed(uint32_t seed) { m.seed = seed; }
	// Adaptive sampling (rtb_render_adaptive): from now on Render() gives every pixel min_spp samples, then more only where
	// the display-space standard error of its 3x3 neighbourhood is above `tolerance` (10^(-D/20) for about D dB), with
	// samples_per_pixel as the cap.  One GPU only: a renderer on several throws.
	void SetNoiseTarget(float tolerance, uint32_t min_spp) {
		if (m.mr) throw std::runtime_error("Renderer::SetNoiseTarget: adaptive sampling renders on one GPU (this renderer uses " + std::to_string(gpuCount()) + ")");
		m.noise_tolerance = tolerance; m.noise_min_spp = min_spp;
	}

	static Renderer MakeRenderer(uint32_t render_width, uint32_t render_height, uint32_t samples_per_pixel, uint32_t max_depth,
	                             const MotionBlurCamera* cam, const Hittable* d_world_ptr) {
		M m{}; m.cam = cam; return _make(render_width, render_height, samples_per_pixel, max_depth, d_world_ptr, m);
	}
	static Renderer MakeRenderer(uint32_t render_width, uint32_t render_height, uint32_t samples_per_pixel, uint32_t max_depth,
	                             const DefocusBlurCamera* cam, const Hittable* d_world_ptr) {
		M m{}; m.defocus_cam = cam; return _make(render_width, render_height, samples_per_pixel, max_depth, d_world_ptr, m);
	}
	static Renderer MakeRenderer(uint32_t render_width, uint32_t render_height, uint32_t samples_per_pixel, uint32_t max_depth,
	                             const PinholeCamera* cam, const Hittable* d_world_ptr) {
		M m{}; m.pinhole_cam = cam; return _make(render_width, render_height, samples_per_pixel, max_depth, d_world_ptr, m);
	}
	// Book 3's cam.render(world, lights): the same renderer with light importance sampling towards `lights` - a HittableList
	// of spheres / quads (each optionally under translate / rotate_y), or one such object (rtb_scene_set_sampled_lights).
	template <typename Cam>
	static Renderer MakeRenderer(uint32_t render_width, uint32_t render_height, uint32_t samples_per_pixel, uint32_t max_depth,
	                             const Cam* cam, const Hittable* d_world_ptr, const Hittable* lights) {
		std::vector<int> ids;
		if (const HittableList* l = dynamic_cast<const HittableList*>(lights)) ids = l->memberIds();
		else if (lights) ids.push_back(lights->rtb_object);
		rtb_host::check(rtb_scene_set_sampled_lights(rtb_host::scene(), ids.data(), (int)ids.size()), "rtb_scene_set_sampled_lights");
		return MakeRenderer(render_width, render_height, samples_per_pixel, max_depth, cam, d_world_ptr);
	}

	void Render() {
		rtb_camera c = m.cam ? m.cam->to_rtb() : (m.defocus_cam ? m.defocus_cam->to_rtb() : m.pinhole_cam->to_rtb());
		rtb_render_params p{};
		p.width = m.render_width; p.height = m.render_height; p.sample_begin = 0; p.sample_end = m.samples_per_pixel;
		p.max_depth = m.max_depth; p.seed = m.seed; p.flags = RTB_RENDER_CLEAR;
		printf("Running render kernel...\n");
		rtb_counters k{};
		if (m.mr) {
			rtb_host::check(rtb_multi_set_camera(m.mr, &c), "rtb_multi_set_camera");
			rtb_host::check(rtb_multi_reset_counters(m.mr), "rtb_multi_reset_counters");
			rtb_host::check(rtb_multi_render(m.mr, &p), "rtb_multi_render");
			rtb_host::check(rtb_multi_synchronize(m.mr), "rtb_multi_synchronize");
			rtb_multi_get_counters(m.mr, &k);
		} else {
			rtb_host::check(rtb_renderer_set_camera(m.r, &c), "rtb_renderer_set_camera");
			rtb_host::check(rtb_reset_counters(m.r), "rtb_reset_counters");
			if (m.noise_tolerance >= 0.0f) {
				rtb_adaptive_params a{m.noise_tolerance, m.noise_min_spp, 0, 0};
				rtb_host::check(rtb_render_adaptive(m.r, &p, &a, &m.last_adaptive, nullptr), "rtb_render_adaptive");
			} else rtb_host::check(rtb_render(m.r, &p, nullptr), "rtb_render");
			rtb_host::check(rtb_synchronize(m.r), "rtb_synchronize");
			rtb_get_counters(m.r, &k);
		}
		m.last_render_ms = k.render_ms; m.last_rays = k.rays; m.last_paths = k.paths;
		printf("Rendering finished in %fms.\n", k.render_ms);
	}
	void DownloadRenderbuffer(glm::vec4* host_dst) const {
		if (m.mr) rtb_host::check(rtb_multi_download(m.mr, &host_dst->x), "rtb_multi_download");
		else rtb_host::check(rtb_download(m.r, &host_dst->x), "rtb_download");
	}
	// The 8-bit picture write_renderbuffer would make of the render buffer (FirstApp.cpp:108-122), quantised on the device:
	// width * height * 3 bytes, top row first when flip_rows is set.
	void DownloadRenderbufferRgb8(uint8_t* host_dst, bool flip_rows = true) const {
		if (m.mr) rtb_host::check(rtb_multi_download_rgb8(m.mr, host_dst, flip_rows ? 1 : 0), "rtb_multi_download_rgb8");
		else rtb_host::check(rtb_download_rgb8(m.r, host_dst, flip_rows ? 1 : 0), "rtb_download_rgb8");
	}
	int gpuCount() const { return m.mr ? rtb_multi_device_count(m.mr) : 1; }
	double lastRenderMs() const { return m.last_render_ms; }
	uint64_t lastRays() const { return m.last_rays; }
	uint64_t lastPaths() const { return m.last_paths; }
	const rtb_adaptive_stats& lastAdaptiveStats() const { return m.last_adaptive; }
	rtb_renderer* handle() const { return m.r; }
};
