// rtb_app — a Linux command-line shell around the renderer, written against the host mirror the way
// the reference's RT application is (main/src/main.cpp:22-32, main/src/FirstApp.cpp:20-56,94-122):
// build the camera, build the scene, MakeRenderer, Render, DownloadRenderbuffer, write the image.
//
//   rtb_app [scene] [--width W] [--height H] [--spp N] [--depth D] [--seed S] [--gpus N]
//           [--out image.png|image.ppm|image.pfm] [--resume ckpt.rtba] [--checkpoint ckpt.rtba] [--sample-lights]
//           [--target-db D [--min-spp N]] [--env map.pfm [--env-scale S] [--sample-env]]
//   rtb_app --obj model.obj [--smooth [--obj-texture image.ppm]] [--obj-material clay|rough-metal|rough-glass [--alpha A]] [...]
//                                     a Wavefront OBJ mesh (MeshHandle) on a checkered floor under the sky
//
// scene = one of rtb_scenes_name(i) (default book2_bouncing, which goes through SceneBook2BVH::Factory
// and Renderer::MakeRenderer exactly like FirstApp::MakeApp).  --gpus N renders on N GPUs of the box (sample range split,
// one reduction; RTB_GPUS does the same for the Renderer mirror).  The 8-bit picture follows write_renderbuffer
// (FirstApp.cpp:108-122) - uint8 = value * 255.999f, RGB, rows flipped (row 0 of the float buffer is the bottom of the
// image) - and is quantised on the device; .png / .ppm carry it, .pfm keeps the raw floats.  --checkpoint saves the
// radiance sums after the render; --resume loads such a file and renders --spp MORE samples on top of it (single GPU).
// --sample-lights turns on light importance sampling (rtb_scene_set_sampled_lights) towards the emitters the named scene
// lists (rtb_scene_info::lights): the same converged image with less noise per sample; refused for scenes that list none.
// --target-db D samples adaptively (rtb_render_adaptive, DESIGN.md §5c): every pixel gets --min-spp samples (default 64),
// then more only where its estimated error is above 10^(-D/20), with --spp as the cap per pixel; it prints the rounds, the
// mean samples per pixel and the render time.  With --resume it continues adaptively from the checkpoint's cursor (a
// checkpoint written by an adaptive run: it needs the sums of squares), still up to --spp in all.  One GPU only.
// --env map.pfm lights the scene (any named scene or --obj) with an HDR environment map (rtb_scene_set_environment,
// DESIGN.md §5d): an equirectangular PFM, +y up, which every ray that leaves the scene reads instead of the background;
// --env-scale S multiplies its texels by S, and --sample-env importance-samples it (same converged image, less noise).
// --smooth loads the --obj model with MeshHandle::LoadObjShaded: smooth shading from its `vn` normals (computed from the faces
// when it has none) and its `vt` texture coordinates (DESIGN.md §5e).  --obj-texture image.ppm (binary P6) then maps that
// image onto the model through its texture coordinates; it needs --smooth and a model with `vt` on every corner.
// --obj-material picks the model's material: clay (the default Lambertian), rough-metal (a copper-coloured GGX conductor) or
// rough-glass (GGX glass, ior 1.5), of width --alpha A (default 0.2; DESIGN.md §5f).  --obj-texture implies the textured
// Lambertian, so it takes no rough material; --alpha needs a rough one.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "Renderer.h"
#include "rt_engine/geometry/BVH.cuh"
#include "rt_engine/geometry/HittableList.cuh"
#include "rt_engine/geometry/Mesh.cuh"
#include "rt_engine/geometry/Scenes.h"
#include "rt_engine/geometry/SphereHittable.cuh"
#include "rt_engine/shaders/cu_Cameras.cuh"
#include "rt_engine/shaders/cu_Textures.cuh"
#include "rt_engine/shaders/cu_materials.cuh"
#include "utilities/image_write.h"

// fb = float render buffer (row 0 = bottom); rgb8 = the device-quantised picture (row 0 = top).
static bool write_image(const std::string& path, uint32_t width, uint32_t height, const std::vector<glm::vec4>& fb, const std::vector<uint8_t>& rgb8) {
	if (rtb_host::has_suffix(path, ".pfm")) return rtb_host::write_pfm(path, width, height, &fb[0].x);
	if (rtb_host::has_suffix(path, ".png")) return rtb_host::write_png(path, width, height, rgb8.data());
	return rtb_host::write_ppm(path, width, height, rgb8.data());
}

int main(int argc, char** argv) {
	std::string scene_name = "book2_bouncing", out = "render.ppm", obj_path, resume_path, checkpoint_path;
	int width = 0, height = 0, spp = 0, depth = 0, gpus = 0;
	bool sample_lights = false;
	double target_db = -1.0;
	int min_spp = 64;
	std::string env_path, obj_texture, obj_material;
	float alpha = -1.0f;
	bool smooth = false;
	float env_scale = 1.0f;
	bool sample_env = false;
	uint32_t seed = 1984;   // the reference's seed (Renderer.cu:51, Scenes.cu:190)
	for (int i = 1; i < argc; ++i) {
		std::string a = argv[i];
		auto next = [&]() { return i + 1 < argc ? atoi(argv[++i]) : 0; };
		if (a == "--width") width = next();
		else if (a == "--height") height = next();
		else if (a == "--spp") spp = next();
		else if (a == "--depth") depth = next();
		else if (a == "--seed") seed = (uint32_t)strtoul(i + 1 < argc ? argv[++i] : "1984", nullptr, 10);
		else if (a == "--gpus") gpus = next();
		else if (a == "--resume" && i + 1 < argc) resume_path = argv[++i];
		else if (a == "--checkpoint" && i + 1 < argc) checkpoint_path = argv[++i];
		else if (a == "--out" && i + 1 < argc) out = argv[++i];
		else if (a == "--obj" && i + 1 < argc) obj_path = argv[++i];
		else if (a == "--sample-lights") sample_lights = true;
		else if (a == "--target-db" && i + 1 < argc) target_db = atof(argv[++i]);
		else if (a == "--min-spp") min_spp = next();
		else if (a == "--env" && i + 1 < argc) env_path = argv[++i];
		else if (a == "--env-scale" && i + 1 < argc) env_scale = (float)atof(argv[++i]);
		else if (a == "--sample-env") sample_env = true;
		else if (a == "--smooth") smooth = true;
		else if (a == "--obj-texture" && i + 1 < argc) obj_texture = argv[++i];
		else if (a == "--obj-material" && i + 1 < argc) obj_material = argv[++i];
		else if (a == "--alpha" && i + 1 < argc) alpha = (float)atof(argv[++i]);
		else if (a == "--list") { for (int k = 0; k < rtb_scenes_count(); ++k) printf("%s\n", rtb_scenes_name(k)); return 0; }
		else scene_name = a;
	}
	if (sample_lights && (!obj_path.empty() || scene_name == "book2_bouncing")) {
		fprintf(stderr, "rtb_app: --sample-lights: %s lists no lights to sample\n", obj_path.empty() ? scene_name.c_str() : obj_path.c_str());
		return 1;
	}
	if ((smooth || !obj_texture.empty()) && obj_path.empty()) { fprintf(stderr, "rtb_app: --smooth and --obj-texture apply to an --obj model\n"); return 1; }
	if (!obj_texture.empty() && !smooth) { fprintf(stderr, "rtb_app: --obj-texture needs --smooth (the texture coordinates come with LoadObjShaded)\n"); return 1; }
	const bool rough = obj_material == "rough-metal" || obj_material == "rough-glass";
	if ((!obj_material.empty() || alpha >= 0.0f) && obj_path.empty()) { fprintf(stderr, "rtb_app: --obj-material and --alpha apply to an --obj model\n"); return 1; }
	if (!obj_material.empty() && !rough && obj_material != "clay") { fprintf(stderr, "rtb_app: --obj-material: expected clay, rough-metal or rough-glass, got %s\n", obj_material.c_str()); return 1; }
	if (alpha >= 0.0f && !rough) { fprintf(stderr, "rtb_app: --alpha needs --obj-material rough-metal or rough-glass\n"); return 1; }
	if (rough && !obj_texture.empty()) { fprintf(stderr, "rtb_app: --obj-texture makes the model a textured Lambertian; drop --obj-material %s\n", obj_material.c_str()); return 1; }
	if (rough && alpha < 0.0f) alpha = 0.2f;
	if (rough && !(alpha >= RTB_ROUGH_ALPHA_MIN && alpha <= 1.0f)) { fprintf(stderr, "rtb_app: --alpha must be in [0.001, 1]\n"); return 1; }
	if (sample_env && env_path.empty()) { fprintf(stderr, "rtb_app: --sample-env needs --env map.pfm\n"); return 1; }
	std::vector<float> env_rgb;
	int env_w = 0, env_h = 0;
	if (!env_path.empty()) {
		std::string err;
		if (!rtb_host::read_pfm(env_path, env_rgb, env_w, env_h, err)) { fprintf(stderr, "rtb_app: --env: %s\n", err.c_str()); return 1; }
	}
	// the map goes on the scene before the renderer flattens it
	auto set_env = [&](rtb_scene* s) {
		if (env_rgb.empty()) return;
		const float scale[3] = {env_scale, env_scale, env_scale};
		rtb_host::check(rtb_scene_set_environment(s, env_rgb.data(), env_w, env_h, scale, sample_env ? RTB_ENV_SAMPLE : 0), "rtb_scene_set_environment");
		printf("Environment map %s: %dx%d%s.\n", env_path.c_str(), env_w, env_h, sample_env ? ", sampled" : "");
	};
	const bool adaptive = target_db >= 0.0;
	const float tolerance = adaptive ? (float)std::pow(10.0, -target_db / 20.0) : 0.0f;
	if (adaptive && gpus > 1) { fprintf(stderr, "rtb_app: --target-db renders on one GPU (adaptive sampling has no multi-GPU path); drop --gpus %d\n", gpus); return 1; }
	if (gpus > 1) Renderer::UseGpus(gpus);
	try {
		std::vector<glm::vec4> fb; std::vector<uint8_t> rgb8;
		if (!obj_path.empty()) {
			// A mesh scene assembled the way FirstApp assembles its world: materials, handles, a HittableList, MakeRenderer.
			uint32_t _width = width ? width : 800, _height = height ? height : 600;
			printf("Loading %s... ", obj_path.c_str());
			Mesh mesh = smooth ? MeshHandle::LoadObjShaded(obj_path) : MeshHandle::LoadObj(obj_path);
			Lambertian clay(glm::vec3(0.73f, 0.73f, 0.73f));
			std::unique_ptr<image_texture> skin;
			std::unique_ptr<Lambertian> skin_mat;
			if (!obj_texture.empty()) {
				if (mesh.uvs.empty()) { fprintf(stderr, "\nrtb_app: --obj-texture: %s has no texture coordinates (`vt` on every face corner)\n", obj_path.c_str()); return 1; }
				std::vector<uint8_t> px; int tw = 0, th = 0; std::string err;
				if (!rtb_host::read_ppm(obj_texture, px, tw, th, err)) { fprintf(stderr, "\nrtb_app: --obj-texture: %s\n", err.c_str()); return 1; }
				skin = std::make_unique<image_texture>(px.data(), tw, th, 3);
				skin_mat = std::make_unique<Lambertian>(skin.get());
			}
			std::unique_ptr<GeoIndependantMaterial> rough_mat;
			if (obj_material == "rough-metal") rough_mat = std::make_unique<RoughMetal>(glm::vec3(0.95f, 0.64f, 0.54f), alpha);
			else if (obj_material == "rough-glass") rough_mat = std::make_unique<RoughDielectric>(1.5f, alpha);
			GeoIndependantMaterial* model_mat = skin_mat ? static_cast<GeoIndependantMaterial*>(skin_mat.get()) : rough_mat ? rough_mat.get() : &clay;
			MeshHandle model = MeshHandle::MakeMesh(mesh, model_mat);
			printf("%d triangles%s%s.\n", model.triangleCount(), smooth ? (skin ? ", smooth, textured" : ", smooth") : "", rough ? (obj_material == "rough-metal" ? ", rough metal" : ", rough glass") : "");
			const glm::vec3 lo = model.getBounds().getMin(), hi = model.getBounds().getMax(), mid = (lo + hi) * 0.5f;
			const float size = glm::length(hi - lo);
			solid_texture dark(glm::vec3(.2f, .3f, .1f)), light(glm::vec3(.9f, .9f, .9f));
			checker_texture checks(&dark, &light, 8.0f / size);
			Lambertian floor_mat(&checks);
			GeoHandle floor = GeoHandle::MakeQuad(Quad(glm::vec3(mid.x - 10 * size, lo.y, mid.z - 10 * size), glm::vec3(20 * size, 0, 0), glm::vec3(0, 0, 20 * size)), &floor_mat);
			const Hittable* objs[2] = {floor.getHittablePtr(), model.getHittablePtr()};
			aabb bounds = model.getBounds(); bounds += floor.getBounds();
			HittableList world(objs, 2, bounds);
			MotionBlurCamera cam(mid + glm::vec3(0.55f, 0.35f, 1.1f) * size, mid, glm::vec3(0, 1, 0), 40.0f, _width / (float)_height, 0.0f, 1.0f);
			set_env(rtb_host::scene());   // the scene the mirror's constructors recorded into, before MakeRenderer flattens it
			Renderer renderer = Renderer::MakeRenderer(_width, _height, spp ? spp : 64, depth ? depth : 16, &cam, &world);
			renderer.SetSeed(seed);
			if (adaptive) renderer.SetNoiseTarget(tolerance, (uint32_t)min_spp);
			renderer.Render();
			fb.resize((size_t)_width * _height); rgb8.resize((size_t)_width * _height * 3);
			renderer.DownloadRenderbuffer(fb.data()); renderer.DownloadRenderbufferRgb8(rgb8.data());
			width = _width; height = _height;
		} else if (scene_name == "book2_bouncing") {
			// FirstApp::MakeApp, statement for statement, with the resolution / spp / depth made arguments
			uint32_t _width = width ? width : 1280, _height = height ? height : 720;
			printf("Building MotionBlurCamera object... ");
			auto cam = std::make_unique<MotionBlurCamera>(glm::vec3(13, 2, 3), glm::vec3(0, 0, 0), glm::vec3(0, 1, 0), 30.0f, _width / (float)_height, 0.1f, 1.0f);
			printf("done.\nBuilding SceneBook2BVH object...\n");
			SceneBook2BVH::Factory scene_factory{};
			std::unique_ptr<SceneBook2BVH> scene_ptr(scene_factory.MakeScene());
			printf("SceneBook2BVH object built.\nMaking Renderer object...\n");
			set_env(rtb_host::scene());
			Renderer renderer = Renderer::MakeRenderer(_width, _height, spp ? spp : 1, depth ? depth : 4, cam.get(), scene_ptr->getWorldPtr());
			renderer.SetSeed(seed);
			if (adaptive) renderer.SetNoiseTarget(tolerance, (uint32_t)min_spp);
			printf("Renderer object built (%d GPU%s).\nRendering scene...\n", renderer.gpuCount(), renderer.gpuCount() > 1 ? "s" : "");
			renderer.Render();
			fb.resize((size_t)_width * _height); rgb8.resize((size_t)_width * _height * 3);
			renderer.DownloadRenderbuffer(fb.data()); renderer.DownloadRenderbufferRgb8(rgb8.data());
			width = _width; height = _height;
		} else {
			rtb_scene_info info{};
			rtb_scene* s = rtb_scenes_build(scene_name.c_str(), &info);
			if (!s) { fprintf(stderr, "rtb_app: %s\n", rtb_scenes_last_error()); return 1; }
			if (sample_lights) {
				if (info.n_lights == 0) { fprintf(stderr, "rtb_app: --sample-lights: %s lists no lights to sample\n", scene_name.c_str()); rtb_scene_destroy(s); return 1; }
				rtb_host::check(rtb_scene_set_sampled_lights(s, info.lights, info.n_lights), "rtb_scene_set_sampled_lights");
				printf("Sampling %d light%s.\n", info.n_lights, info.n_lights > 1 ? "s" : "");
			}
			set_env(s);
			if (!width) width = info.width;
			if (!height) height = info.height;
			rtb_render_params p{};
			p.width = width; p.height = height; p.sample_end = spp ? spp : info.spp; p.max_depth = depth ? depth : info.max_depth; p.seed = seed; p.flags = RTB_RENDER_CLEAR;
			fb.resize((size_t)width * height); rgb8.resize((size_t)width * height * 3);
			rtb_counters k{};
			if (gpus > 1) {
				if (!resume_path.empty() || !checkpoint_path.empty()) { fprintf(stderr, "rtb_app: --resume / --checkpoint work on one GPU\n"); return 1; }
				rtb_multi_renderer* mr = nullptr;
				rtb_host::check(rtb_multi_renderer_create(&mr, nullptr, gpus, RTB_REDUCE_AUTO), "rtb_multi_renderer_create");
				rtb_host::check(rtb_multi_set_scene(mr, s), "rtb_multi_set_scene");
				rtb_host::check(rtb_multi_set_camera(mr, &info.camera), "rtb_multi_set_camera");
				printf("Running render kernel on %d GPUs (%s reduction)...\n", gpus, rtb_multi_reduce_mode(mr) == RTB_REDUCE_NCCL ? "NCCL" : "peer-memory");
				if (getenv("RTB_APP_WARMUP")) { rtb_host::check(rtb_multi_render(mr, &p), "rtb_multi_render"); rtb_host::check(rtb_multi_synchronize(mr), "rtb_multi_synchronize"); rtb_multi_reset_counters(mr); }
				rtb_host::check(rtb_multi_render(mr, &p), "rtb_multi_render");
				rtb_host::check(rtb_multi_synchronize(mr), "rtb_multi_synchronize");
				rtb_multi_get_counters(mr, &k);
				rtb_host::check(rtb_multi_download(mr, &fb[0].x), "rtb_multi_download");
				rtb_host::check(rtb_multi_download_rgb8(mr, rgb8.data(), 1), "rtb_multi_download_rgb8");
				rtb_multi_renderer_destroy(mr);
			} else {
				rtb_renderer* r = nullptr;
				rtb_host::check(rtb_renderer_create(&r, 0), "rtb_renderer_create");
				rtb_host::check(rtb_renderer_set_scene(r, s), "rtb_renderer_set_scene");
				rtb_host::check(rtb_renderer_set_camera(r, &info.camera), "rtb_renderer_set_camera");
				if (!resume_path.empty()) {   // continue a checkpointed render: --spp more samples from its cursor on (adaptive: up to --spp)
					uint32_t cw = 0, ch = 0, cursor = 0;
					rtb_host::check(rtb_load_accum(r, resume_path.c_str(), &cw, &ch, &cursor), "rtb_load_accum");
					if ((int)cw != width || (int)ch != height) { fprintf(stderr, "rtb_app: the checkpoint is %ux%u, the render %dx%d\n", cw, ch, width, height); return 1; }
					if (!adaptive) { p.sample_begin = cursor; p.sample_end += cursor; }
					p.flags = 0;
					printf("Resuming at sample %u.\n", cursor);
				}
				printf("Running render kernel...\n");
				if (adaptive) {
					rtb_adaptive_params a{tolerance, (uint32_t)min_spp, 0, 0};
					rtb_adaptive_stats as{};
					rtb_host::check(rtb_render_adaptive(r, &p, &a, &as, nullptr), "rtb_render_adaptive");
					rtb_get_counters(r, &k);
					std::vector<float> acc((size_t)width * height * 4);
					rtb_host::check(rtb_download_accum(r, acc.data(), nullptr), "rtb_download_accum");
					double n = 0.0;
					for (size_t i = 0; i < (size_t)width * height; ++i) n += acc[4 * i + 3];
					printf("Adaptive: target %.1f dB (tolerance %.3g), %u rounds, mean %.1f spp (cap %u), render %.1f ms.\n",
					       target_db, tolerance, as.rounds, n / ((double)width * height), p.sample_end, k.render_ms);
				} else {
					if (getenv("RTB_APP_WARMUP") && resume_path.empty()) { rtb_host::check(rtb_render(r, &p, nullptr), "rtb_render"); rtb_host::check(rtb_synchronize(r), "rtb_synchronize"); rtb_reset_counters(r); }
					rtb_host::check(rtb_render(r, &p, nullptr), "rtb_render");
					rtb_host::check(rtb_synchronize(r), "rtb_synchronize");
					rtb_get_counters(r, &k);
				}
				if (!checkpoint_path.empty()) { rtb_host::check(rtb_save_accum(r, checkpoint_path.c_str()), "rtb_save_accum"); printf("Checkpoint written (%s, %u samples).\n", checkpoint_path.c_str(), rtb_renderer_sample_cursor(r)); }
				rtb_host::check(rtb_download(r, &fb[0].x), "rtb_download");
				rtb_host::check(rtb_download_rgb8(r, rgb8.data(), 1), "rtb_download_rgb8");
				rtb_renderer_destroy(r);
			}
			printf("Rendering finished in %fms (%.1f Mrays/s, %.1f Mpaths/s).\n", k.render_ms, k.rays / k.render_ms * 1e-3, k.paths / k.render_ms * 1e-3);
			rtb_scene_destroy(s);
		}
		printf("Writing render to disk... ");
		if (!write_image(out, width, height, fb, rgb8)) { fprintf(stderr, "cannot write %s\n", out.c_str()); return 1; }
		printf("done (%s).\n", out.c_str());
	} catch (const std::exception& e) {
		fprintf(stderr, "rtb_app: %s\n", e.what());
		return 1;
	}
	return 0;
}
