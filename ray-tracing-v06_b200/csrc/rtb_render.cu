// rtb_render.cu — renderer object behind the C ABI: device memory, batch scheduling, CUDA-graph
// replay of the per-batch wavefront sequence, download and the parity hooks.
//
// Replaces Renderer::MakeRenderer / Render / DownloadRenderbuffer (main/src/Renderer.cu:31-137) and the
// scene upload of BVH_Handle's ctor (main/src/rt_engine/geometry/BVH.cu:110-120): one arena of aligned
// SoA buffers instead of ~3 device allocations + a <<<1,1>>> constructor launch per object.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "rtb_renderer.h"

using namespace rtb;

static void prof_begin(rtb_renderer* r, int cls, cudaStream_t st) {
	if (!r->profiling) return;
	if (r->prof_used == r->prof_class.size()) {
		cudaEvent_t a = nullptr, b = nullptr;
		if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) {   // no events: this launch goes untimed
			if (a) cudaEventDestroy(a);
			cudaGetLastError(); r->profiling = false; return;
		}
		r->prof_events.push_back(a); r->prof_events.push_back(b); r->prof_class.push_back(cls);
	}
	r->prof_class[r->prof_used] = cls;
	cudaEventRecord(r->prof_events[2 * r->prof_used], st);
}
static void prof_end(rtb_renderer* r, cudaStream_t st) {
	if (!r->profiling) return;
	cudaEventRecord(r->prof_events[2 * r->prof_used + 1], st);
	r->prof_used++;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static int upload_staged_scene(rtb_renderer* r);

static void free_graph(rtb_renderer* r) {
	if (r->graph_exec) { cudaGraphExecDestroy(r->graph_exec); r->graph_exec = nullptr; }
	if (r->graph_exec2) { cudaGraphExecDestroy(r->graph_exec2); r->graph_exec2 = nullptr; }
	r->graph_valid = false;
}

extern "C" {

int rtb_device_count(void) {
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n;
}

int rtb_renderer_create(rtb_renderer** out, int device) {
	if (!out) return fail(RTB_ERR_INVALID, "rtb_renderer_create: null out");
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0) {
		cudaGetLastError();
		return fail(RTB_ERR_CUDA, std::string("rtb_renderer_create: no usable CUDA device (") + cudaGetErrorString(e) +
		                              "); this library has no CPU fallback");
	}
	if (device < 0 || device >= n) return fail(RTB_ERR_INVALID, "rtb_renderer_create: bad device index");
	CUDA_TRY(cudaSetDevice(device));
	rtb_renderer* r = new rtb_renderer();
	r->device = device;
	const int rc_init = [&]() -> int {   // (a failure past this point must not leak the half-built object)
		CUDA_TRY(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking));
		CUDA_TRY(cudaEventCreateWithFlags(&r->ev_in, cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreateWithFlags(&r->ev_out, cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreate(&r->ev_t0));
		CUDA_TRY(cudaEventCreate(&r->ev_t1));
		return RTB_OK;
	}();
	if (rc_init != RTB_OK) { rtb_renderer_destroy(r); return rc_init; }
	query_occupancy(device, r->lc);
	r->tail_threshold = (uint32_t)r->lc.sms * 768u;   // ~6 warps of rays per SM sub-partition
	if (const char* e = getenv("RTB_TAIL_THRESHOLD")) r->tail_threshold = (uint32_t)strtoul(e, nullptr, 10);
	if (const char* e = getenv("RTB_LANES")) r->lanes = atoi(e) >= 2 ? 2 : 1;
	if (const char* e = getenv("RTB_BIN_BITS")) { int a = 0, b = 0; if (sscanf(e, "%d,%d", &a, &b) == 2 && a >= 0 && a <= 8 && b >= 0 && b <= 6 && 3 * a + 2 * b <= 26) { r->bin_org_bits = a; r->bin_dir_bits = b; } }
	if (const char* e = getenv("RTB_BIN_MASK")) { r->bin_mask = strtoull(e, nullptr, 16); r->bin_forced = true; }
	*out = r;
	return RTB_OK;
}

void rtb_renderer_destroy(rtb_renderer* r) {
	if (!r) return;
	cudaSetDevice(r->device);
	if (r->stream) cudaStreamSynchronize(r->stream);
	free_graph(r);
	free_gpu_scratch(r->build_scratch);
	for (cudaEvent_t e : r->prof_events) cudaEventDestroy(e);
	if (r->stream2) cudaStreamSynchronize(r->stream2);
	cudaFree(r->d_scene); cudaFree(r->d_accum); cudaFree(r->d_accum2); cudaFree(r->d_out); cudaFree(r->d_wave); cudaFree(r->d_wave2); cudaFree(r->d_rgb8);
	cudaFree(r->d_err); cudaFree(r->d_list); cudaFree(r->d_block); cudaFree(r->d_select);
	if (r->h_select) cudaFreeHost(r->h_select);
	for (cudaEvent_t e : {r->ev_lane[0], r->ev_lane[1], r->ev_fork}) if (e) cudaEventDestroy(e);
	if (r->stream2) cudaStreamDestroy(r->stream2);
	for (cudaEvent_t e : {r->ev_in, r->ev_out, r->ev_t0, r->ev_t1}) if (e) cudaEventDestroy(e);
	if (r->stream) cudaStreamDestroy(r->stream);
	cudaGetLastError();
	delete r;
}

int rtb_renderer_scene_stats(const rtb_renderer* r, rtb_scene_stats* out) {
	if (!r || !out) return fail(RTB_ERR_INVALID, "rtb_renderer_scene_stats: null argument");
	if (!r->has_scene) return fail(RTB_ERR_STATE, "rtb_renderer_scene_stats: no scene set");
	*out = r->scene_stats;
	return RTB_OK;
}

int rtb_renderer_set_scene(rtb_renderer* r, rtb_scene* s) {
	if (!r || !s) return fail(RTB_ERR_INVALID, "rtb_renderer_set_scene: null argument");
	CUDA_TRY(cudaSetDevice(r->device));
	// An unchanged scene (same object, same version) is not flattened again: only the arena is re-sent.
	const bool cached = r->staged_uid == s->uid && r->staged_version == s->version && !r->staging.empty();
	if (!cached) {
		FlatScene fs;
		GpuBuildContext gpu{r->device, r->stream, &r->build_scratch};
		int rc = flatten(*s, fs, &gpu);
		if (rc) return rc;
		r->scene_stats = rtb_scene_stats{fs.n_items, (int32_t)fs.prims.size(), (int32_t)fs.nodes.size(), fs.max_depth_nodes, fs.builder, fs.flatten_ms, fs.bvh_build_ms, 0};
		// one arena, every section 256-byte aligned
		size_t off_nodes = 0;
		size_t off_prims = align_up(off_nodes + fs.nodes.size() * sizeof(DevNode), 256);
		size_t off_info = align_up(off_prims + fs.prims.size() * sizeof(DevPrim), 256);
		size_t off_mats = align_up(off_info + fs.prim_info.size() * sizeof(DevPrimInfo), 256);
		size_t off_texs = align_up(off_mats + fs.materials.size() * sizeof(DevMaterial), 256);
		size_t off_blob = align_up(off_texs + fs.textures.size() * sizeof(DevTexture), 256);
		size_t off_pre = align_up(off_blob + fs.blob.size(), 256);
		size_t off_lights = align_up(off_pre + fs.pre_list.size() * 4, 256);   // (no lights: the arena is what it was without them)
		size_t off_env = align_up(off_lights + fs.lights.size() * (sizeof(DevPrim) + sizeof(DevLightInfo)), 256);   // (likewise without a map)
		size_t off_attr = align_up(off_env + fs.env.size() * sizeof(DevEnvTexel) + fs.env_cdf.size() * sizeof(float), 256);   // (likewise without attributes)
		size_t total = align_up(off_attr + fs.tri_attr.size() * sizeof(DevTriAttr) + fs.attr_slot.size() * sizeof(int32_t), 256) + 256;
		r->staging.assign(total, 0);
		uint8_t* st = r->staging.data();
		if (!fs.nodes.empty()) memcpy(st + off_nodes, fs.nodes.data(), fs.nodes.size() * sizeof(DevNode));
		memcpy(st + off_prims, fs.prims.data(), fs.prims.size() * sizeof(DevPrim));
		memcpy(st + off_info, fs.prim_info.data(), fs.prim_info.size() * sizeof(DevPrimInfo));
		if (!fs.materials.empty()) memcpy(st + off_mats, fs.materials.data(), fs.materials.size() * sizeof(DevMaterial));
		if (!fs.textures.empty()) memcpy(st + off_texs, fs.textures.data(), fs.textures.size() * sizeof(DevTexture));
		if (!fs.blob.empty()) memcpy(st + off_blob, fs.blob.data(), fs.blob.size());
		if (!fs.pre_list.empty()) memcpy(st + off_pre, fs.pre_list.data(), fs.pre_list.size() * 4);
		if (!fs.lights.empty()) {
			memcpy(st + off_lights, fs.lights.data(), fs.lights.size() * sizeof(DevPrim));
			memcpy(st + off_lights + fs.lights.size() * sizeof(DevPrim), fs.light_info.data(), fs.light_info.size() * sizeof(DevLightInfo));
		}
		r->off[0] = off_nodes; r->off[1] = off_prims; r->off[2] = off_info; r->off[3] = off_mats; r->off[4] = off_texs; r->off[5] = off_blob; r->off[6] = off_pre;
		if (!fs.env.empty()) {   // the CDFs follow the texels directly: the kernels find them at env + width * height
			memcpy(st + off_env, fs.env.data(), fs.env.size() * sizeof(DevEnvTexel));
			memcpy(st + off_env + fs.env.size() * sizeof(DevEnvTexel), fs.env_cdf.data(), fs.env_cdf.size() * sizeof(float));
		}
		if (!fs.tri_attr.empty()) {   // the per-slot record indices follow the records directly
			memcpy(st + off_attr, fs.tri_attr.data(), fs.tri_attr.size() * sizeof(DevTriAttr));
			memcpy(st + off_attr + fs.tri_attr.size() * sizeof(DevTriAttr), fs.attr_slot.data(), fs.attr_slot.size() * sizeof(int32_t));
		}
		r->off[7] = off_lights; r->off[8] = off_env; r->off[9] = off_attr;
		r->staged_sv = SceneView{};
		r->staged_sv.root_ref = fs.root_ref;
		r->staged_sv.n_prims = (int32_t)fs.prims.size();
		r->staged_sv.n_nodes = (int32_t)fs.nodes.size(); r->staged_sv.n_materials = (int32_t)fs.materials.size();
		r->staged_sv.n_textures = (int32_t)fs.textures.size(); r->staged_sv.n_blob = (uint32_t)fs.blob.size();
		r->staged_sv.tree_depth = fs.max_depth_nodes;
		r->staged_sv.n_pre = (int32_t)fs.pre_list.size();
		r->staged_sv.bvh_empty = fs.bvh_empty;
		r->staged_sv.n_lights = (int32_t)fs.lights.size();
		r->staged_sv.env_width = fs.env_width; r->staged_sv.env_height = fs.env_height; r->staged_sv.env_sample = fs.env_sample;
		r->staged_sv.n_tri_attr = (int32_t)fs.tri_attr.size();
		r->staged_sv.has_media = fs.n_media == 0 ? 0 : (fs.n_media <= (int32_t)fs.pre_list.size() ? 1 : 2);
		// The scene's part of the feature word that selects the shade and tail kernels (rtb_kernels.h), decided here only.
		// (A sampled map is a strategy of the light mixture, so it needs the LIGHTS kernels even without a light list.)
		uint32_t flags = 0;
		if (fs.lights.size() > 0 || (fs.env_width > 0 && fs.env_sample)) flags |= F_LIGHTS;
		if (fs.env_width > 0) flags |= F_ENV;
		if (!fs.tri_attr.empty()) flags |= F_ATTR;
		for (size_t i = 0; i < fs.materials.size(); ++i) {
			const DevMaterial& m = fs.materials[i];
			if (m.tex >= 0 && m.kind != RTB_MAT_DIFFUSE_LIGHT && (fs.textures[m.tex].kind == RTB_TEX_NOISE || fs.textures[m.tex].kind == RTB_TEX_IMAGE)) flags |= SV_DEFERRED_TEX;
			if (m.kind == RTB_MAT_ROUGH_METAL || m.kind == RTB_MAT_ROUGH_DIELECTRIC) flags |= F_ROUGH;
		}
		r->staged_sv.launch_flags = (int32_t)flags;
		r->staged_sv.background_mode = fs.background_mode;
		r->staged_sv.bg_r = fs.background[0]; r->staged_sv.bg_g = fs.background[1]; r->staged_sv.bg_b = fs.background[2];
		for (int k = 0; k < 3; ++k) { r->world_min[k] = fs.world_min[k]; r->world_max[k] = fs.world_max[k]; }
		r->staged_sv.bin_org_bits = r->bin_org_bits; r->staged_sv.bin_dir_bits = r->bin_dir_bits;
		for (int k = 0; k < 3; ++k) {
			const float ext = fs.bin_max[k] - fs.bin_min[k];
			r->staged_sv.bin_min[k] = fs.bin_min[k];
			r->staged_sv.bin_scale[k] = ext > 0.0f ? (float)(1 << r->bin_org_bits) / ext : 0.0f;
		}
		r->staged_uid = s->uid; r->staged_version = s->version;
	}
	const int rc_up = upload_staged_scene(r);
	if (rc_up) return rc_up;
	if (!cached) r->scene_version++;   // same bytes at the same addresses: the cached graph stays valid
	return RTB_OK;
}

int rtb_renderer_share_scene(rtb_renderer* r, const rtb_renderer* src) {
	if (!r || !src) return fail(RTB_ERR_INVALID, "rtb_renderer_share_scene: null argument");
	if (src->staging.empty()) return fail(RTB_ERR_STATE, "rtb_renderer_share_scene: the source renderer has no scene");
	if (r == src) return RTB_OK;
	CUDA_TRY(cudaSetDevice(r->device));
	const bool same = r->staged_uid == src->staged_uid && r->staged_version == src->staged_version && r->staging.size() == src->staging.size() && r->has_scene;
	if (!same) {
		r->staging = src->staging;
		for (int i = 0; i < 10; ++i) r->off[i] = src->off[i];
		r->staged_sv = src->staged_sv; r->staged_uid = src->staged_uid; r->staged_version = src->staged_version;
		for (int k = 0; k < 3; ++k) r->staged_sv.bin_scale[k] *= (float)(1 << r->bin_org_bits) / (float)(1 << src->bin_org_bits);   // (this renderer's own bin settings)
		r->staged_sv.bin_org_bits = r->bin_org_bits; r->staged_sv.bin_dir_bits = r->bin_dir_bits;
		for (int k = 0; k < 3; ++k) { r->world_min[k] = src->world_min[k]; r->world_max[k] = src->world_max[k]; }
		r->scene_stats = src->scene_stats;
	}
	const int rc_up = upload_staged_scene(r);
	if (rc_up) return rc_up;
	if (!same) r->scene_version++;
	return RTB_OK;
}

}  // extern "C"

// The staged arena -> device (one copy), and the device views of its sections.
static int upload_staged_scene(rtb_renderer* r) {
	const size_t total = r->staging.size();
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	if (total > r->scene_bytes) {
		cudaFree(r->d_scene); r->d_scene = nullptr; r->scene_bytes = 0;
		CUDA_TRY(cudaMalloc(&r->d_scene, total));
		r->scene_bytes = total;
	}
	CUDA_TRY(cudaMemcpy(r->d_scene, r->staging.data(), total, cudaMemcpyHostToDevice));
	uint8_t* base = static_cast<uint8_t*>(r->d_scene);
	r->sv = r->staged_sv;
	r->sv.nodes = reinterpret_cast<const float4*>(base + r->off[0]);
	r->sv.prims = reinterpret_cast<const float4*>(base + r->off[1]);
	r->sv.prim_info = reinterpret_cast<const int2*>(base + r->off[2]);
	r->sv.materials = reinterpret_cast<const float4*>(base + r->off[3]);
	r->sv.textures = reinterpret_cast<const float4*>(base + r->off[4]);
	r->sv.blob = base + r->off[5];
	r->sv.pre_list = reinterpret_cast<const int32_t*>(base + r->off[6]);
	r->sv.lights = r->sv.n_lights > 0 ? reinterpret_cast<const float4*>(base + r->off[7]) : nullptr;
	r->sv.env = r->sv.env_width > 0 ? reinterpret_cast<const float4*>(base + r->off[8]) : nullptr;
	r->sv.tri_attr = r->sv.n_tri_attr > 0 ? reinterpret_cast<const float4*>(base + r->off[9]) : nullptr;
	r->sv.attr_slot = r->sv.n_tri_attr > 0 ? reinterpret_cast<const int32_t*>(base + r->off[9] + (size_t)r->sv.n_tri_attr * sizeof(DevTriAttr)) : nullptr;
	r->has_scene = true;
	r->scene_upload_bytes = total;
	return RTB_OK;
}

extern "C" {

size_t rtb_renderer_scene_bytes(const rtb_renderer* r) { return r ? r->scene_upload_bytes : 0; }

int rtb_renderer_set_camera(rtb_renderer* r, const rtb_camera* cam) {
	if (!r || !cam) return fail(RTB_ERR_INVALID, "rtb_renderer_set_camera: null argument");
	if (cam->kind < RTB_CAM_PINHOLE || cam->kind > RTB_CAM_MOTION) return fail(RTB_ERR_INVALID, "rtb_renderer_set_camera: bad kind");
	r->cam = *cam; r->has_cam = true;
	return RTB_OK;
}

static int ensure_framebuffer(rtb_renderer* r, uint32_t w, uint32_t h) {
	if (r->width == w && r->height == h && r->d_accum) return RTB_OK;
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	cudaFree(r->d_accum); cudaFree(r->d_accum2); cudaFree(r->d_out); cudaFree(r->d_rgb8);
	cudaFree(r->d_err); cudaFree(r->d_list); cudaFree(r->d_block); cudaFree(r->d_select);
	r->d_accum = r->d_accum2 = r->d_out = nullptr; r->d_rgb8 = nullptr; r->sample_cursor = 0;
	r->d_err = nullptr; r->d_list = r->d_block = r->d_select = nullptr;
	size_t bytes = (size_t)w * h * sizeof(float4);
	CUDA_TRY(cudaMalloc(&r->d_accum, bytes));
	CUDA_TRY(cudaMalloc(&r->d_accum2, bytes));
	CUDA_TRY(cudaMalloc(&r->d_out, bytes));
	// (zeroed on the renderer's stream: it is non-blocking, so a cudaMemset on the legacy stream would not be ordered
	// before the work enqueued on it next)
	CUDA_TRY(cudaMemsetAsync(r->d_accum, 0, bytes, r->stream));
	CUDA_TRY(cudaMemsetAsync(r->d_accum2, 0, bytes, r->stream));
	CUDA_TRY(cudaMemsetAsync(r->d_out, 0, bytes, r->stream));
	r->width = w; r->height = h;
	free_graph(r);
	return RTB_OK;
}

// Buffers of the adaptive select step, for the current framebuffer size (allocated by the first adaptive render after each
// resize, so that uniform renders allocate exactly what they did before adaptive sampling existed).
static int ensure_adaptive_buffers(rtb_renderer* r) {
	if (r->d_err && r->d_list && r->d_block && r->d_select && r->h_select) return RTB_OK;
	// all or nothing: a failure part-way leaves every device pointer null, and the next call starts over
	cudaFree(r->d_err); cudaFree(r->d_list); cudaFree(r->d_block); cudaFree(r->d_select);
	r->d_err = nullptr; r->d_list = r->d_block = r->d_select = nullptr;
	const size_t n = (size_t)r->width * r->height;
	cudaError_t e = cudaMalloc(&r->d_err, n * sizeof(float));
	if (e == cudaSuccess) e = cudaMalloc(&r->d_list, n * sizeof(uint32_t));
	if (e == cudaSuccess) e = cudaMalloc(&r->d_block, (size_t)adaptive_select_blocks((uint32_t)n) * sizeof(uint32_t));
	if (e == cudaSuccess) e = cudaMalloc(&r->d_select, 256);
	if (e == cudaSuccess && !r->h_select) e = cudaMallocHost(&r->h_select, 2 * sizeof(uint32_t));
	if (e != cudaSuccess) {
		cudaFree(r->d_err); cudaFree(r->d_list); cudaFree(r->d_block); cudaFree(r->d_select);
		r->d_err = nullptr; r->d_list = r->d_block = r->d_select = nullptr;
		cudaGetLastError();
		return fail(RTB_ERR_NOMEM, std::string("rtb_render_adaptive: allocating the select buffers: ") + cudaGetErrorString(e));
	}
	return RTB_OK;
}

// Queues of one lane (0: the renderer's own stream; 1: the second stream multi-batch renders deal every other batch to).
static int ensure_wave(rtb_renderer* r, int lane, size_t paths, uint32_t depth) {
	void*& d_wave = lane ? r->d_wave2 : r->d_wave;
	size_t& wave_paths = lane ? r->wave2_paths : r->wave_paths;
	uint32_t& wave_depth = lane ? r->wave2_depth : r->wave_depth;
	WaveView& wv = lane ? r->wv2 : r->wv;
	if (paths <= wave_paths && depth <= wave_depth && d_wave) return RTB_OK;
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	if (r->stream2) CUDA_TRY(cudaStreamSynchronize(r->stream2));
	free_graph(r);
	// the path / ray totals (rtb_get_counters) live in the queue buffer: carry them over to the new one
	unsigned long long totals[2] = {0, 0};
	if (d_wave) CUDA_TRY(cudaMemcpy(totals, wv.totals, sizeof totals, cudaMemcpyDeviceToHost));
	cudaFree(d_wave); d_wave = nullptr;
	if (paths < wave_paths) paths = wave_paths;     // grow-only in both dimensions: alternating sizes do not thrash
	if (depth < wave_depth) depth = wave_depth;
	wave_paths = 0; wave_depth = 0;
	size_t P = align_up(paths, 256);
	size_t off = 0;
	auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
	size_t o_od0 = take(P * 32), o_od1 = take(P * 32);
	size_t o_t0 = take(P * 16), o_t1 = take(P * 16), o_hit = take(P * 8), o_con = take(P * 16);
	size_t o_live = take((depth + 2) * 4), o_work = take(2 * (depth + 2) * 4), o_batch = take(256), o_tot = take(256);
	size_t o_tex = take(P * 32), o_ntex = take((depth + 2) * 4);
	const size_t nbins = (size_t)1 << (3 * r->bin_org_bits + 2 * r->bin_dir_bits);
	size_t o_bcnt = take(nbins * 4), o_bcur = take(nbins * 4);
	cudaError_t e = cudaMalloc(&d_wave, off);
	if (e != cudaSuccess) { d_wave = nullptr; cudaGetLastError(); return fail(RTB_ERR_NOMEM, std::string("cudaMalloc of the wavefront queues: ") + cudaGetErrorString(e)); }
	CUDA_TRY(cudaMemsetAsync(d_wave, 0, off, r->stream));   // (ordered before the batch that follows; lane 1 starts after an event on this stream)
	uint8_t* b = static_cast<uint8_t*>(d_wave);
	wv.ray_od[0] = (float4*)(b + o_od0); wv.ray_od[1] = (float4*)(b + o_od1);
	wv.thr[0] = (float4*)(b + o_t0); wv.thr[1] = (float4*)(b + o_t1);
	wv.hit = (int2*)(b + o_hit); wv.contrib = (float4*)(b + o_con);
	wv.n_live = (uint32_t*)(b + o_live); wv.work = (uint32_t*)(b + o_work);
	wv.tex_work = (float4*)(b + o_tex); wv.n_tex = (uint32_t*)(b + o_ntex);
	wv.bin_count = (uint32_t*)(b + o_bcnt); wv.bin_cursor = (uint32_t*)(b + o_bcur);
	wv.capacity = (uint32_t)P; wv.n_bins = (uint32_t)nbins;
	wv.batch_index = (uint32_t*)(b + o_batch); wv.tail_from = wv.batch_index + 1; wv.totals = (unsigned long long*)(b + o_tot);
	wv.call_params = wv.batch_index + 8;   // (same 256-byte block)
	if (totals[0] || totals[1]) {
		CUDA_TRY(cudaMemcpyAsync(wv.totals, totals, sizeof totals, cudaMemcpyHostToDevice, r->stream));
		CUDA_TRY(cudaStreamSynchronize(r->stream));   // (the source is on this stack frame)
	}
	wave_paths = P; wave_depth = depth;
	return RTB_OK;
}

#define RTB_WAVE_BYTES_PER_PATH 152ull   // 2 x (32 ray + 16 throughput), double buffered, + 8 (hit) + 16 (contribution) + 32 (texture work list)

// Bounces before which the fused tail kernel checks whether the live queue has become short.
static bool tail_checkpoint(uint32_t b) {
	static const uint32_t pts[] = {2, 3, 4, 5, 6, 8, 10, 12, 15, 18, 22, 27, 33, 40, 48, 58, 70, 85, 100};
	for (uint32_t p : pts) if (p == b) return true;
	return b > 100 && b % 25 == 0;
}
static uint32_t count_tail_checkpoints(uint32_t depth) { uint32_t c = 0; for (uint32_t b = 0; b < depth; ++b) c += tail_checkpoint(b) ? 1 : 0; return c; }

// Which bounces' queues are binned before they are traversed (bit b of the mask), and how finely: RTB_BIN_MASK (hex),
// RTB_BIN_BITS=<origin bits per axis>,<direction bits per axis> (0,0 = off).
static bool binned_bounce(const rtb_renderer* r, uint32_t b) {
	if (r->sv.bin_org_bits + r->sv.bin_dir_bits == 0 || b == 0 || !r->bin_on) return false;
	return b < 64 ? ((r->bin_mask >> b) & 1ull) != 0 : false;
}
static uint32_t count_binned_bounces(const rtb_renderer* r, uint32_t depth) { uint32_t c = 0; for (uint32_t b = 1; b < depth; ++b) c += binned_bounce(r, b) ? 1 : 0; return c; }

// One batch of the wavefront on `st` with the queues `wv`.  The accumulation of the batch into the framebuffer is part of it
// unless the caller orders it itself (two lanes: the accumulations of consecutive batches must not overlap).
static void enqueue_batch(rtb_renderer* r, const WaveView& wv, const BatchParams& bp, cudaStream_t st, bool with_accumulate) {
	prof_begin(r, 0, st); launch_generate(bp, r->cam, wv, r->lc, st); prof_end(r, st);
	int q = 0;   // the queue that holds the rays of bounce b
	for (uint32_t b = 0; b < bp.max_depth; ++b) {
		if (r->tail_threshold && tail_checkpoint(b)) { prof_begin(r, 4, st); launch_tail(r->sv, bp, wv, b, q, r->tail_threshold, r->lc, st); prof_end(r, st); }
		prof_begin(r, 1, st); launch_traverse(r->sv, bp, wv, b, q, r->lc, st); prof_end(r, st);
		const bool bin_next = b + 1 < bp.max_depth && binned_bounce(r, b + 1);
		prof_begin(r, 2, st); launch_shade(r->sv, bp, wv, b, q, r->lc, st);
		if ((r->sv.launch_flags & SV_DEFERRED_TEX) && b + 1 < bp.max_depth) launch_texture(r->sv, wv, b, q ^ 1, r->lc, st);
		prof_end(r, st);
		if (bin_next) { prof_begin(r, 5, st); launch_bin_rays(r->sv, wv, b + 1, q ^ 1, r->lc, st); prof_end(r, st); }   // ... and back into queue q
		else q ^= 1;
	}
	if (with_accumulate) { prof_begin(r, 3, st); launch_accumulate(bp, wv, r->d_accum, r->d_accum2, r->lc, st); prof_end(r, st); }
}

static int capture_batch_graph(rtb_renderer* r, const WaveView& wv, const BatchParams& bp, cudaStream_t st, bool with_accumulate, cudaGraphExec_t* out) {
	cudaGraph_t graph = nullptr;
	CUDA_TRY(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
	enqueue_batch(r, wv, bp, st, with_accumulate);
	cudaError_t e = cudaStreamEndCapture(st, &graph);
	if (e != cudaSuccess) return fail(RTB_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
	e = cudaGraphInstantiate(out, graph, 0);
	cudaGraphDestroy(graph);
	if (e != cudaSuccess) return fail(RTB_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
	return RTB_OK;
}

// Paths one batch of an automatic batch size aims at, for `npix` pixels: 64 M (~9.7 GB of queues; larger batches keep
// late, thin bounces full), RTB_BATCH_PATHS, or less when device memory is short.
static uint64_t batch_path_budget(rtb_renderer* r, uint64_t npix, uint32_t samples_per_batch) {
	uint64_t target_paths = 64ull << 20;
	if (const char* e = getenv("RTB_BATCH_PATHS")) { uint64_t v = strtoull(e, nullptr, 10); if (v > 0) target_paths = v; }
	if (!samples_per_batch && target_paths > r->wave_paths) {
		// the queues cost RTB_WAVE_BYTES_PER_PATH per path: an automatic batch never asks for more than half of what is free
		// (a smaller device, several renderers per device, a large scene) - it gets smaller instead of failing
		size_t free_b = 0, total_b = 0;
		if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
			const uint64_t cap = (uint64_t)(free_b / 2 + r->wave_paths * RTB_WAVE_BYTES_PER_PATH) / RTB_WAVE_BYTES_PER_PATH;
			if (target_paths > cap) target_paths = cap > npix ? cap : npix;
		} else cudaGetLastError();
	}
	return target_paths;
}

// Samples per batch for `spp` samples of `npix` pixels: the caller's samples_per_batch, else as many as the budget holds,
// evened out so that every batch has the same size.
static uint64_t batch_samples(uint64_t target_paths, uint64_t npix, uint32_t spp, uint32_t samples_per_batch) {
	uint64_t S = samples_per_batch ? samples_per_batch : target_paths / npix;
	if (S < 1) S = 1;
	if (S > spp) S = spp ? spp : 1;
	if (!samples_per_batch && spp) { uint64_t nb = (spp + S - 1) / S; S = (spp + nb - 1) / nb; }   // equal-sized batches
	return S;
}

int rtb_render(rtb_renderer* r, const rtb_render_params* p, void* user_stream) {
	if (!r || !p) return fail(RTB_ERR_INVALID, "rtb_render: null argument");
	if (!r->has_scene) return fail(RTB_ERR_STATE, "rtb_render: no scene (rtb_renderer_set_scene)");
	if (!r->has_cam) return fail(RTB_ERR_STATE, "rtb_render: no camera (rtb_renderer_set_camera)");
	if (p->width == 0 || p->height == 0 || p->max_depth == 0) return fail(RTB_ERR_INVALID, "rtb_render: zero width/height/max_depth");
	if (p->sample_end < p->sample_begin) return fail(RTB_ERR_INVALID, "rtb_render: sample_end < sample_begin");
	uint32_t row_begin = p->row_begin, row_end = p->row_end;
	if (row_begin == 0 && row_end == 0) row_end = p->height;
	if (row_end > p->height || row_begin >= row_end) return fail(RTB_ERR_INVALID, "rtb_render: bad row range");
	if ((uint64_t)p->width * p->height >= (1ull << 31)) return fail(RTB_ERR_INVALID, "rtb_render: image too large");
	CUDA_TRY(cudaSetDevice(r->device));
	int rc = ensure_framebuffer(r, p->width, p->height);
	if (rc) return rc;

	const uint32_t spp = p->sample_end - p->sample_begin;
	const uint64_t npix = (uint64_t)p->width * (row_end - row_begin);
	const uint64_t S = batch_samples(batch_path_budget(r, npix, p->samples_per_batch), npix, spp, p->samples_per_batch);
	if (npix * S >= (1ull << 31)) return fail(RTB_ERR_INVALID, "rtb_render: batch too large (lower samples_per_batch)");
	rc = ensure_wave(r, 0, (size_t)(npix * S), p->max_depth);
	if (rc) return rc;
	const uint32_t n_batches = spp ? (uint32_t)((spp + S - 1) / S) : 0;
	const bool use_graph = getenv("RTB_NO_GRAPH") == nullptr && n_batches > 0 && !r->profiling;
	// Two lanes: every other batch goes to a second stream with queues of its own, so that the thin late bounces of one batch
	// (a few million rays per launch, tens of launches) overlap the full early bounces of the next.  The accumulations stay in
	// batch order (events), so the image is bit for bit the one-lane image.  Falls back to one lane when memory is short.
	bool two_lanes = use_graph && n_batches >= 2 && r->lanes >= 2;
	if (two_lanes) {
		if (!r->stream2) {
			CUDA_TRY(cudaStreamCreateWithFlags(&r->stream2, cudaStreamNonBlocking));
			for (int k = 0; k < 2; ++k) CUDA_TRY(cudaEventCreateWithFlags(&r->ev_lane[k], cudaEventDisableTiming));
			CUDA_TRY(cudaEventCreateWithFlags(&r->ev_fork, cudaEventDisableTiming));
		}
		if (!(r->d_wave2 && r->wave2_paths >= npix * S && r->wave2_depth >= p->max_depth)) {
			size_t free_b = 0, total_b = 0;
			const bool room = cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && free_b > (size_t)(npix * S) * RTB_WAVE_BYTES_PER_PATH * 5 / 4;
			if (!room || ensure_wave(r, 1, (size_t)(npix * S), p->max_depth) != RTB_OK) { cudaGetLastError(); two_lanes = false; }
		}
	}

	// Binning pays where walks are long and queues large: a tree of some size (the 20 primitives of a Cornell box are
	// walked in a few steps whatever the order of the rays: measured 179 vs 157 ms on config 4 with / without) and batches
	// big enough that the three extra launches per binned bounce are noise.  RTB_BIN_MASK forces the schedule.
	r->bin_on = r->bin_forced || (r->sv.n_nodes >= 512 && npix * S >= (8ull << 20));
	BatchParams bp{};
	bp.width = p->width; bp.height = p->height; bp.row_begin = row_begin; bp.n_rows = row_end - row_begin;
	bp.npix = (uint32_t)npix; bp.sample_begin = p->sample_begin; bp.sample_end = p->sample_end;
	bp.samples_per_batch = (uint32_t)S; bp.max_depth = p->max_depth; bp.seed = p->seed;
	bp.variance = (p->flags & RTB_RENDER_VARIANCE) ? 1u : 0u;
	bp.batch_base = 0; bp.batch_stride = two_lanes ? 2u : 1u;

	cudaStream_t us = static_cast<cudaStream_t>(user_stream);
	cudaStream_t st = r->stream;
	// order this render after whatever the caller queued on its stream
	CUDA_TRY(cudaEventRecord(r->ev_in, us));
	CUDA_TRY(cudaStreamWaitEvent(st, r->ev_in, 0));
	if (p->flags & RTB_RENDER_CLEAR) {
		size_t bytes = (size_t)p->width * p->height * sizeof(float4);
		CUDA_TRY(cudaMemsetAsync(r->d_accum, 0, bytes, st));
		CUDA_TRY(cudaMemsetAsync(r->d_accum2, 0, bytes, st));
	}
	CUDA_TRY(cudaMemsetAsync(r->wv.batch_index, 0, sizeof(uint32_t), st));
	r->call_params[0] = bp.sample_begin; r->call_params[1] = bp.sample_end; r->call_params[2] = bp.seed; r->call_params[3] = 0;
	CUDA_TRY(cudaMemcpyAsync(const_cast<uint32_t*>(r->wv.call_params), r->call_params, sizeof r->call_params, cudaMemcpyHostToDevice, st));   // (pageable source: staged before the call returns)
	CUDA_TRY(cudaEventRecord(r->ev_t0, st));

	const uint64_t launches_per_batch = 3 + 2ull * bp.max_depth + (r->tail_threshold ? count_tail_checkpoints(bp.max_depth) : 0) +
	                                    ((r->sv.launch_flags & SV_DEFERRED_TEX) ? bp.max_depth - 1 : 0) + 3ull * count_binned_bounces(r, bp.max_depth);
	if (use_graph) {
		BatchParams key = bp; key.sample_begin = key.sample_end = key.seed = 0;   // (those three travel through device memory: call_params)
		bool reuse = r->graph_valid && r->graph_bin_on == r->bin_on && memcmp(&r->graph_bp, &key, sizeof key) == 0 && memcmp(&r->graph_cam, &r->cam, sizeof r->cam) == 0 &&
		             memcmp(&r->graph_sv, &r->sv, sizeof r->sv) == 0 && r->graph_accum == r->d_accum && (!two_lanes || r->graph_exec2);
		// (The kernels see the scene only through the SceneView they are launched with - section pointers and sizes, tree depth, bin
		// grid - and the memory behind it: a scene that was edited and flattened again into the same layout, an animation step
		// for instance, needs no new graph.  Round 2 first keyed the graph on a scene version and re-captured ~300 nodes per change.)
		if (!reuse) {
			free_graph(r);
			rc = capture_batch_graph(r, r->wv, bp, st, !two_lanes, &r->graph_exec);
			if (rc) return rc;
			if (two_lanes) {
				BatchParams bp1 = bp; bp1.batch_base = 1;
				rc = capture_batch_graph(r, r->wv2, bp1, r->stream2, false, &r->graph_exec2);
				if (rc) return rc;
			}
			r->graph_bp = key; r->graph_bin_on = r->bin_on; r->graph_cam = r->cam; r->graph_sv = r->sv; r->graph_accum = r->d_accum;
			r->graph_valid = true;
		}
		if (!two_lanes) {
			for (uint32_t b = 0; b < n_batches; ++b) CUDA_TRY(cudaGraphLaunch(r->graph_exec, st));
		} else {
			BatchParams bpl[2] = {bp, bp}; bpl[1].batch_base = 1;
			const WaveView* wvl[2] = {&r->wv, &r->wv2};
			cudaStream_t stl[2] = {st, r->stream2};
			CUDA_TRY(cudaEventRecord(r->ev_fork, st));                               // lane 1 starts after the clears above
			CUDA_TRY(cudaStreamWaitEvent(r->stream2, r->ev_fork, 0));
			CUDA_TRY(cudaMemsetAsync(r->wv2.batch_index, 0, sizeof(uint32_t), r->stream2));
			CUDA_TRY(cudaMemcpyAsync(const_cast<uint32_t*>(r->wv2.call_params), r->call_params, sizeof r->call_params, cudaMemcpyHostToDevice, r->stream2));
			for (uint32_t b = 0; b < n_batches; ++b) {
				const int L = (int)(b & 1u);
				CUDA_TRY(cudaGraphLaunch(L ? r->graph_exec2 : r->graph_exec, stl[L]));
				if (b > 0) CUDA_TRY(cudaStreamWaitEvent(stl[L], r->ev_lane[L ^ 1], 0));   // batch b - 1 is in the framebuffer
				launch_accumulate(bpl[L], *wvl[L], r->d_accum, r->d_accum2, r->lc, stl[L]);
				CUDA_TRY(cudaEventRecord(r->ev_lane[L], stl[L]));
			}
			CUDA_TRY(cudaStreamWaitEvent(st, r->ev_lane[1], 0));                      // join (lane 1 ran at least one batch)
		}
	} else {
		for (uint32_t b = 0; b < n_batches; ++b) enqueue_batch(r, r->wv, bp, st, true);
	}
	CUDA_TRY(cudaGetLastError());
	r->launches += launches_per_batch * n_batches;
	r->batches += n_batches;
	CUDA_TRY(cudaEventRecord(r->ev_t1, st));
	r->timed = true;
	if ((p->flags & RTB_RENDER_CLEAR) || p->sample_end > r->sample_cursor) r->sample_cursor = p->sample_end;
	// ... and let the caller's stream see the result
	CUDA_TRY(cudaEventRecord(r->ev_out, st));
	CUDA_TRY(cudaStreamWaitEvent(us, r->ev_out, 0));
	return RTB_OK;
}

// Adaptive sampling (DESIGN.md §5c).  Each round: the select step on the device writes the ascending list of active pixels
// and their count, the host reads the count (one sync per round), and the round renders samples [c, c + k) of every listed
// pixel through enqueue_batch in list mode.  The shape of a round (pixel count, batch size) changes from round to round,
// so rounds run on one lane and without a CUDA graph.
int rtb_render_adaptive(rtb_renderer* r, const rtb_render_params* p, const rtb_adaptive_params* a, rtb_adaptive_stats* out, void* user_stream) {
	if (!r || !p || !a) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: null argument");
	if (!r->has_scene) return fail(RTB_ERR_STATE, "rtb_render_adaptive: no scene (rtb_renderer_set_scene)");
	if (!r->has_cam) return fail(RTB_ERR_STATE, "rtb_render_adaptive: no camera (rtb_renderer_set_camera)");
	if (p->width == 0 || p->height == 0 || p->max_depth == 0) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: zero width/height/max_depth");
	if (p->sample_begin != 0) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: sample_begin must be 0 (the call continues from the accumulator's own cursor)");
	if (a->min_spp < 2) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: min_spp must be at least 2");
	if (p->sample_end < a->min_spp || p->sample_end > (1u << 24)) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: need min_spp <= sample_end <= 2^24");
	if (!(a->tolerance >= 0.0f) || !(a->tolerance <= 3.402823466e+38f)) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: tolerance must be finite and >= 0");
	uint32_t row_begin = p->row_begin, row_end = p->row_end;
	if (row_begin == 0 && row_end == 0) row_end = p->height;
	if (row_end > p->height || row_begin >= row_end) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: bad row range");
	if ((uint64_t)p->width * p->height >= (1ull << 31)) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: image too large");
	const bool clear = (p->flags & RTB_RENDER_CLEAR) != 0;
	if (!clear && r->d_accum && (r->width != p->width || r->height != p->height))
		return fail(RTB_ERR_STATE, "rtb_render_adaptive: the accumulator holds another image size (pass RTB_RENDER_CLEAR)");
	CUDA_TRY(cudaSetDevice(r->device));
	int rc = ensure_framebuffer(r, p->width, p->height);
	if (rc) return rc;
	rc = ensure_adaptive_buffers(r);
	if (rc) return rc;

	const uint64_t npix_range = (uint64_t)p->width * (row_end - row_begin);
	const uint32_t max_spp = p->sample_end;
	const uint64_t budget = batch_path_budget(r, npix_range, p->samples_per_batch);
	uint32_t c = clear ? 0u : r->sample_cursor;
	AdaptiveView av{};
	av.accum = r->d_accum; av.accum2 = r->d_accum2; av.err = r->d_err; av.list = r->d_list; av.block_count = r->d_block; av.result = r->d_select;
	av.width = p->width; av.row_begin = row_begin; av.n_rows = row_end - row_begin;
	av.min_spp = a->min_spp; av.max_spp = max_spp; av.tolerance = a->tolerance;

	cudaStream_t us = static_cast<cudaStream_t>(user_stream);
	cudaStream_t st = r->stream;
	CUDA_TRY(cudaEventRecord(r->ev_in, us));
	CUDA_TRY(cudaStreamWaitEvent(st, r->ev_in, 0));
	if (clear) {
		size_t bytes = (size_t)p->width * p->height * sizeof(float4);
		CUDA_TRY(cudaMemsetAsync(r->d_accum, 0, bytes, st));
		CUDA_TRY(cudaMemsetAsync(r->d_accum2, 0, bytes, st));
	}
	CUDA_TRY(cudaEventRecord(r->ev_t0, st));
	rtb_adaptive_stats stats{};
	uint32_t n_active = 0;
	const int rc_rounds = [&]() -> int {
		for (;;) {
			// select step: error, window, candidates, ascending list; then the one read-back of the round
			av.cursor = c;
			CUDA_TRY(cudaMemsetAsync(r->d_select, 0, 2 * sizeof(uint32_t), st));
			prof_begin(r, 6, st); launch_adaptive_select(av, r->lc, st); prof_end(r, st);
			r->launches += (c >= a->min_spp ? 4 : 3);
			CUDA_TRY(cudaGetLastError());
			CUDA_TRY(cudaMemcpyAsync(r->h_select, r->d_select, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaStreamSynchronize(st));
			n_active = r->h_select[0];
			if (r->h_select[1]) return fail(RTB_ERR_STATE, "rtb_render_adaptive: the accumulator has no sums of squares (render it with RTB_RENDER_VARIANCE)");
			if (n_active == 0 || (a->max_rounds && stats.rounds >= a->max_rounds)) break;

			// round size: up to min_spp first; after that at most one doubling of the cursor and at most one batch of paths
			const uint64_t fill = budget / n_active > 1 ? budget / n_active : 1;
			const uint32_t k = (uint32_t)std::min<uint64_t>(max_spp - c, c < a->min_spp ? (uint64_t)(a->min_spp - c) : std::min<uint64_t>(c, fill));
			const uint64_t S = batch_samples(budget, n_active, k, p->samples_per_batch);
			if ((uint64_t)n_active * S >= (1ull << 31)) return fail(RTB_ERR_INVALID, "rtb_render_adaptive: batch too large (lower samples_per_batch)");
			rc = ensure_wave(r, 0, (size_t)(n_active * S), p->max_depth);
			if (rc) return rc;
			r->bin_on = r->bin_forced || (r->sv.n_nodes >= 512 && n_active * S >= (8ull << 20));
			BatchParams bp{};
			bp.width = p->width; bp.height = p->height; bp.row_begin = row_begin; bp.n_rows = row_end - row_begin;
			bp.npix = n_active; bp.sample_begin = c; bp.sample_end = c + k;
			bp.samples_per_batch = (uint32_t)S; bp.max_depth = p->max_depth; bp.seed = p->seed;
			bp.variance = 1u; bp.batch_base = 0; bp.batch_stride = 1u;
			bp.set_pixel_list(r->d_list);
			CUDA_TRY(cudaMemsetAsync(r->wv.batch_index, 0, sizeof(uint32_t), st));
			r->call_params[0] = bp.sample_begin; r->call_params[1] = bp.sample_end; r->call_params[2] = bp.seed; r->call_params[3] = 0;
			CUDA_TRY(cudaMemcpyAsync(const_cast<uint32_t*>(r->wv.call_params), r->call_params, sizeof r->call_params, cudaMemcpyHostToDevice, st));
			const uint32_t n_batches = (uint32_t)((k + S - 1) / S);
			for (uint32_t b = 0; b < n_batches; ++b) enqueue_batch(r, r->wv, bp, st, true);
			CUDA_TRY(cudaGetLastError());
			r->launches += (3 + 2ull * bp.max_depth + (r->tail_threshold ? count_tail_checkpoints(bp.max_depth) : 0) +
			                ((r->sv.launch_flags & SV_DEFERRED_TEX) ? bp.max_depth - 1 : 0) + 3ull * count_binned_bounces(r, bp.max_depth)) * n_batches;
			r->batches += n_batches;
			stats.samples += (uint64_t)n_active * k;
			stats.rounds++;
			c += k;
		}
		return RTB_OK;
	}();
	// However the rounds ended - an error included - the cursor covers every round rendered (a later call or checkpoint
	// continues from it) and the caller's stream is ordered after the work.
	r->sample_cursor = c;
	r->timed = true;
	const cudaError_t e_end[3] = {cudaEventRecord(r->ev_t1, st), cudaEventRecord(r->ev_out, st), cudaStreamWaitEvent(us, r->ev_out, 0)};
	stats.cursor = c; stats.active_pixels = n_active;
	if (out) *out = stats;
	if (rc_rounds) return rc_rounds;
	for (cudaError_t e : e_end) if (e != cudaSuccess) return fail(RTB_ERR_CUDA, std::string("rtb_render_adaptive: joining the caller's stream: ") + cudaGetErrorString(e));
	return RTB_OK;
}

int rtb_synchronize(rtb_renderer* r) {
	if (!r) return fail(RTB_ERR_INVALID, "rtb_synchronize: null renderer");
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	return RTB_OK;
}

void* rtb_renderer_accum_ptr(rtb_renderer* r) { return r ? r->d_accum : nullptr; }
void* rtb_renderer_accum2_ptr(rtb_renderer* r) { return r ? r->d_accum2 : nullptr; }

int rtb_resolve(rtb_renderer* r, void* d_out, void* user_stream) {
	if (!r || !r->d_accum) return fail(RTB_ERR_STATE, "rtb_resolve: nothing rendered");
	return rtb_resolve_from(r, r->d_accum, d_out, user_stream);
}

}  // extern "C"

int rtb_resolve_from(rtb_renderer* r, const float4* accum, void* d_out, void* user_stream) {
	CUDA_TRY(cudaSetDevice(r->device));
	cudaStream_t us = static_cast<cudaStream_t>(user_stream);
	CUDA_TRY(cudaEventRecord(r->ev_in, us));
	CUDA_TRY(cudaStreamWaitEvent(r->stream, r->ev_in, 0));
	launch_resolve(accum, d_out ? static_cast<float4*>(d_out) : r->d_out, r->width * r->height, r->stream);
	r->launches += 1;
	CUDA_TRY(cudaGetLastError());
	CUDA_TRY(cudaEventRecord(r->ev_out, r->stream));
	CUDA_TRY(cudaStreamWaitEvent(us, r->ev_out, 0));
	return RTB_OK;
}

// 8-bit image the way write_renderbuffer makes it (FirstApp.cpp:108-122): uint8 = value * 255.999f of the resolved
// image, RGB only, rows flipped when asked (row 0 of the float buffer is the bottom of the picture) - quantised on the
// device, so the copy to the host is 3 bytes per pixel instead of 16.
int rtb_quantize_from(rtb_renderer* r, const float4* accum, uint8_t* host_rgb, int flip_rows) {
	CUDA_TRY(cudaSetDevice(r->device));
	const size_t n = (size_t)r->width * r->height;
	if (!r->d_rgb8) CUDA_TRY(cudaMalloc(&r->d_rgb8, n * 3));
	launch_quantize(accum, r->d_rgb8, r->width, r->height, flip_rows, r->stream);
	r->launches += 1;
	CUDA_TRY(cudaGetLastError());
	CUDA_TRY(cudaMemcpyAsync(host_rgb, r->d_rgb8, n * 3, cudaMemcpyDeviceToHost, r->stream));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	return RTB_OK;
}

extern "C" {

int rtb_download_rgb8(rtb_renderer* r, uint8_t* host_rgb, int flip_rows) {
	if (!r || !host_rgb) return fail(RTB_ERR_INVALID, "rtb_download_rgb8: null argument");
	if (!r->d_accum) return fail(RTB_ERR_STATE, "rtb_download_rgb8: nothing rendered");
	return rtb_quantize_from(r, r->d_accum, host_rgb, flip_rows);
}

int rtb_download(rtb_renderer* r, float* host_rgba) {
	if (!r || !host_rgba) return fail(RTB_ERR_INVALID, "rtb_download: null argument");
	int rc = rtb_resolve(r, nullptr, nullptr);
	if (rc) return rc;
	CUDA_TRY(cudaMemcpyAsync(host_rgba, r->d_out, (size_t)r->width * r->height * sizeof(float4), cudaMemcpyDeviceToHost, r->stream));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	return RTB_OK;
}

int rtb_download_accum(rtb_renderer* r, float* host_sum, float* host_sum2) {
	if (!r || !r->d_accum) return fail(RTB_ERR_STATE, "rtb_download_accum: nothing rendered");
	CUDA_TRY(cudaSetDevice(r->device));
	size_t bytes = (size_t)r->width * r->height * sizeof(float4);
	if (host_sum) CUDA_TRY(cudaMemcpyAsync(host_sum, r->d_accum, bytes, cudaMemcpyDeviceToHost, r->stream));
	if (host_sum2) CUDA_TRY(cudaMemcpyAsync(host_sum2, r->d_accum2, bytes, cudaMemcpyDeviceToHost, r->stream));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	return RTB_OK;
}

// Checkpoint of a progressive render: the radiance sums, the sums of squares and the sample cursor.
//   header: "RTBA", version 1, width, height, sample_cursor, reserved[3] (8 x uint32), then 2 x width*height float4.
struct AccumFileHeader { uint32_t magic, version, width, height, sample_cursor, reserved[3]; };
static const uint32_t ACCUM_MAGIC = 0x41425452u;   // "RTBA"

int rtb_save_accum(rtb_renderer* r, const char* path) {
	if (!r || !path) return fail(RTB_ERR_INVALID, "rtb_save_accum: null argument");
	if (!r->d_accum) return fail(RTB_ERR_STATE, "rtb_save_accum: nothing rendered");
	const size_t n = (size_t)r->width * r->height;
	std::vector<float> sum(4 * n), sum2(4 * n);
	int rc = rtb_download_accum(r, sum.data(), sum2.data());
	if (rc) return rc;
	FILE* f = fopen(path, "wb");
	if (!f) return fail(RTB_ERR_INVALID, std::string("rtb_save_accum: cannot open ") + path);
	AccumFileHeader h{ACCUM_MAGIC, 1u, r->width, r->height, r->sample_cursor, {0, 0, 0}};
	bool ok = fwrite(&h, sizeof h, 1, f) == 1 && fwrite(sum.data(), 16, n, f) == n && fwrite(sum2.data(), 16, n, f) == n;
	ok = (fclose(f) == 0) && ok;
	return ok ? RTB_OK : fail(RTB_ERR_INVALID, std::string("rtb_save_accum: short write to ") + path);
}

int rtb_load_accum(rtb_renderer* r, const char* path, uint32_t* width_out, uint32_t* height_out, uint32_t* sample_cursor_out) {
	if (!r || !path) return fail(RTB_ERR_INVALID, "rtb_load_accum: null argument");
	FILE* f = fopen(path, "rb");
	if (!f) return fail(RTB_ERR_INVALID, std::string("rtb_load_accum: cannot open ") + path);
	AccumFileHeader h{};
	if (fread(&h, sizeof h, 1, f) != 1 || h.magic != ACCUM_MAGIC || h.version != 1u || h.width == 0 || h.height == 0 ||
	    (uint64_t)h.width * h.height >= (1ull << 31)) { fclose(f); return fail(RTB_ERR_INVALID, std::string("rtb_load_accum: not an accumulator checkpoint: ") + path); }
	const size_t n = (size_t)h.width * h.height;
	std::vector<float> sum(4 * n), sum2(4 * n);
	const bool ok = fread(sum.data(), 16, n, f) == n && fread(sum2.data(), 16, n, f) == n;
	fclose(f);
	if (!ok) return fail(RTB_ERR_INVALID, std::string("rtb_load_accum: truncated file ") + path);
	CUDA_TRY(cudaSetDevice(r->device));
	int rc = ensure_framebuffer(r, h.width, h.height);
	if (rc) return rc;
	CUDA_TRY(cudaMemcpyAsync(r->d_accum, sum.data(), 16 * n, cudaMemcpyHostToDevice, r->stream));
	CUDA_TRY(cudaMemcpyAsync(r->d_accum2, sum2.data(), 16 * n, cudaMemcpyHostToDevice, r->stream));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	r->sample_cursor = h.sample_cursor;
	if (width_out) *width_out = h.width;
	if (height_out) *height_out = h.height;
	if (sample_cursor_out) *sample_cursor_out = h.sample_cursor;
	return RTB_OK;
}

uint32_t rtb_renderer_sample_cursor(const rtb_renderer* r) { return r ? r->sample_cursor : 0; }

int rtb_get_counters(rtb_renderer* r, rtb_counters* out) {
	if (!r || !out) return fail(RTB_ERR_INVALID, "rtb_get_counters: null argument");
	memset(out, 0, sizeof *out);
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	if (r->stream2) CUDA_TRY(cudaStreamSynchronize(r->stream2));
	for (int lane = 0; lane < 2; ++lane) {
		if (!(lane ? r->d_wave2 : r->d_wave)) continue;
		unsigned long long tot[2] = {0, 0};
		CUDA_TRY(cudaMemcpy(tot, (lane ? r->wv2 : r->wv).totals, sizeof tot, cudaMemcpyDeviceToHost));
		out->paths += tot[0]; out->rays += tot[1];
	}
	out->launches = r->launches; out->batches = r->batches;
	if (r->timed) { float ms = 0.0f; if (cudaEventElapsedTime(&ms, r->ev_t0, r->ev_t1) == cudaSuccess) out->render_ms = ms; else cudaGetLastError(); }
	return RTB_OK;
}

int rtb_renderer_set_profiling(rtb_renderer* r, int on) {
	if (!r) return fail(RTB_ERR_INVALID, "rtb_renderer_set_profiling: null renderer");
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	r->profiling = on != 0;
	r->prof_used = 0;
	return RTB_OK;
}

int rtb_get_profile(rtb_renderer* r, rtb_profile* out) {
	if (!r || !out) return fail(RTB_ERR_INVALID, "rtb_get_profile: null argument");
	memset(out, 0, sizeof *out);
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	double ms[7] = {0, 0, 0, 0, 0, 0, 0}; uint64_t cnt[7] = {0, 0, 0, 0, 0, 0, 0};   // (class 6, the adaptive select step, is reported per launch only)
	for (size_t i = 0; i < r->prof_used; ++i) {
		float t = 0.0f;
		CUDA_TRY(cudaEventElapsedTime(&t, r->prof_events[2 * i], r->prof_events[2 * i + 1]));
		ms[r->prof_class[i]] += t; cnt[r->prof_class[i]]++;
	}
	out->generate_ms = ms[0]; out->traverse_ms = ms[1]; out->shade_ms = ms[2]; out->accumulate_ms = ms[3];
	out->tail_ms = ms[4]; out->tail_launches = cnt[4];
	out->bin_ms = ms[5]; out->bin_launches = 3 * cnt[5];
	out->generate_launches = cnt[0]; out->traverse_launches = cnt[1]; out->shade_launches = cnt[2]; out->accumulate_launches = 2 * cnt[3];
	r->prof_used = 0;
	return RTB_OK;
}

int rtb_get_profile_launches(rtb_renderer* r, float* ms_out, int32_t* class_out, int cap) {
	if (!r || cap < 0 || (cap && (!ms_out || !class_out))) return fail(RTB_ERR_INVALID, "rtb_get_profile_launches: bad argument");
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	for (size_t i = 0; i < r->prof_used && (int)i < cap; ++i) {
		float t = 0.0f;
		CUDA_TRY(cudaEventElapsedTime(&t, r->prof_events[2 * i], r->prof_events[2 * i + 1]));
		ms_out[i] = t; class_out[i] = r->prof_class[i];
	}
	return (int)r->prof_used;
}

int rtb_queue_lengths(rtb_renderer* r, uint32_t* out, int cap) {
	if (!r || !out || cap <= 0) return fail(RTB_ERR_INVALID, "rtb_queue_lengths: bad argument");
	if (!r->d_wave) return fail(RTB_ERR_STATE, "rtb_queue_lengths: nothing rendered");
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	int n = (int)r->wave_depth < cap ? (int)r->wave_depth : cap;
	CUDA_TRY(cudaMemcpy(out, r->wv.n_live, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
	return (int)r->wave_depth;
}

int rtb_reset_counters(rtb_renderer* r) {
	if (!r) return fail(RTB_ERR_INVALID, "rtb_reset_counters: null renderer");
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	if (r->stream2) CUDA_TRY(cudaStreamSynchronize(r->stream2));
	if (r->d_wave) CUDA_TRY(cudaMemsetAsync(r->wv.totals, 0, 2 * sizeof(unsigned long long), r->stream));
	if (r->d_wave2) CUDA_TRY(cudaMemsetAsync(r->wv2.totals, 0, 2 * sizeof(unsigned long long), r->stream));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	r->launches = 0; r->batches = 0;
	return RTB_OK;
}

int rtb_debug_bounds_report(rtb_renderer* r, uint64_t* violations_out, int cap, uint64_t* checks_out) {
	if (!r || !violations_out || cap < 0) return fail(RTB_ERR_INVALID, "rtb_debug_bounds_report: bad argument");
	CUDA_TRY(cudaSetDevice(r->device));
	CUDA_TRY(cudaStreamSynchronize(r->stream));
	unsigned long long v[RTB_BOUNDS_CLASSES] = {0}, checks = 0;
	const int rc = debug_bounds_report(v, &checks);
	if (rc == 0) return fail(RTB_ERR_UNSUPPORTED, "rtb_debug_bounds_report: this library was not built with -DRTB_DEBUG_BOUNDS=1 (use librtb200_debug.so)");
	if (rc < 0) return fail(RTB_ERR_CUDA, "rtb_debug_bounds_report: cannot read the counters");
	for (int i = 0; i < cap; ++i) violations_out[i] = i < RTB_BOUNDS_CLASSES ? v[i] : 0;
	if (checks_out) *checks_out = checks;
	return RTB_BOUNDS_CLASSES;
}

int rtb_trace_rays(rtb_renderer* r, const rtb_ray* rays, size_t n, rtb_hit* hits_out) {
	if (!r || (n && (!rays || !hits_out))) return fail(RTB_ERR_INVALID, "rtb_trace_rays: null argument");
	if (!r->has_scene) return fail(RTB_ERR_STATE, "rtb_trace_rays: no scene");
	if (n == 0) return RTB_OK;
	if (n >= (1ull << 31)) return fail(RTB_ERR_INVALID, "rtb_trace_rays: too many rays");
	if (r->sv.bvh_empty) {   // nothing but pre-listed media (which this hook skips): every ray misses, and there is no node 0 to start from
		for (size_t i = 0; i < n; ++i) { rtb_hit h{}; h.t = 3.402823466e+38f; h.prim = h.object = h.material = -1; hits_out[i] = h; }
		return RTB_OK;
	}
	CUDA_TRY(cudaSetDevice(r->device));
	std::vector<float4> ho(n), hd(n);
	for (size_t i = 0; i < n; ++i) {
		ho[i] = make_float4(rays[i].o[0], rays[i].o[1], rays[i].o[2], rays[i].time);
		hd[i] = make_float4(rays[i].d[0], rays[i].d[1], rays[i].d[2], 0.0f);
	}
	float4 *d_o = nullptr, *d_d = nullptr; int2 *d_hit = nullptr, *d_stats = nullptr; rtb_hit* d_rec = nullptr; uint32_t* d_cnt = nullptr;
	int rc = RTB_OK;
	auto cleanup = [&]() { cudaFree(d_o); cudaFree(d_d); cudaFree(d_hit); cudaFree(d_stats); cudaFree(d_rec); cudaFree(d_cnt); };
#define TRY_OR_CLEAN(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { cleanup(); return fail(RTB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); } } while (0)
	TRY_OR_CLEAN(cudaMalloc(&d_o, n * 16));
	TRY_OR_CLEAN(cudaMalloc(&d_d, n * 16));
	TRY_OR_CLEAN(cudaMalloc(&d_hit, n * 8));
	TRY_OR_CLEAN(cudaMalloc(&d_stats, n * 8));
	TRY_OR_CLEAN(cudaMalloc(&d_rec, n * sizeof(rtb_hit)));
	TRY_OR_CLEAN(cudaMalloc(&d_cnt, 256));
	TRY_OR_CLEAN(cudaMemcpyAsync(d_o, ho.data(), n * 16, cudaMemcpyHostToDevice, r->stream));
	TRY_OR_CLEAN(cudaMemcpyAsync(d_d, hd.data(), n * 16, cudaMemcpyHostToDevice, r->stream));
	launch_trace_rays(r->sv, d_o, d_d, (uint32_t)n, d_hit, d_stats, d_rec, d_cnt, r->lc, r->stream);
	r->launches += 2;
	TRY_OR_CLEAN(cudaGetLastError());
	TRY_OR_CLEAN(cudaMemcpyAsync(hits_out, d_rec, n * sizeof(rtb_hit), cudaMemcpyDeviceToHost, r->stream));
	TRY_OR_CLEAN(cudaStreamSynchronize(r->stream));
#undef TRY_OR_CLEAN
	cleanup();
	return rc;
}

}  // extern "C"
