// rtb_renderer.h — the renderer object shared by rtb_render.cu (single device) and rtb_multi.cu (several devices of one
// box): device memory, the staged scene arena, the cached per-batch CUDA graph.  Private to the library.
#ifndef RTB_RENDERER_H
#define RTB_RENDERER_H

#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "rtb_kernels.h"
#include "rtb_scene.h"

#define CUDA_TRY(expr)                                                                                  \
	do {                                                                                                \
		cudaError_t _e = (expr);                                                                        \
		if (_e != cudaSuccess)                                                                          \
			return rtb::fail(RTB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                 \
	} while (0)

struct rtb_renderer {
	using SceneView = rtb::SceneView; using WaveView = rtb::WaveView; using LaunchCfg = rtb::LaunchCfg;
	using BatchParams = rtb::BatchParams; using GpuScratch = rtb::GpuScratch;
	int device = 0;
	cudaStream_t stream = nullptr;
	cudaEvent_t ev_in = nullptr, ev_out = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
	bool timed = false;

	// scene arena
	void* d_scene = nullptr; size_t scene_bytes = 0, scene_upload_bytes = 0;
	SceneView sv{};
	std::vector<uint8_t> staging;           // host copy of the arena of the last flattened scene
	size_t off[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // arena sections: nodes, prims, prim info, materials, textures, blob, pre-test list, lights, environment map, triangle attributes
	SceneView staged_sv{};
	uint64_t staged_uid = 0, staged_version = 0;
	bool has_scene = false;
	rtb_scene_stats scene_stats{};
	GpuScratch build_scratch;   // grow-only scratch of the GPU BVH build
	uint64_t scene_version = 0;
	float world_min[3] = {0, 0, 0}, world_max[3] = {0, 0, 0};   // bounds of the world BVH
	rtb_camera cam{};
	bool has_cam = false;

	// framebuffers
	uint32_t width = 0, height = 0;
	float4 *d_accum = nullptr, *d_accum2 = nullptr, *d_out = nullptr;
	uint8_t* d_rgb8 = nullptr;              // 8-bit output (rtb_download_rgb8)
	uint32_t sample_cursor = 0;             // one past the last sample index accumulated since the last clear (checkpoints)
	// adaptive select step (rtb_render_adaptive; allocated by the first adaptive render after a resize of the framebuffer):
	// per-pixel error, the list of active pixels, per-block counts, (count, missing sums of squares) on the device and in
	// pinned host memory
	float* d_err = nullptr; uint32_t *d_list = nullptr, *d_block = nullptr, *d_select = nullptr, *h_select = nullptr;

	// wavefront queues
	void* d_wave = nullptr; size_t wave_paths = 0; uint32_t wave_depth = 0;
	WaveView wv{};
	LaunchCfg lc{};
	// second lane (rtb_render deals the batches of a multi-batch render to two streams): its own queues, stream and graph
	void* d_wave2 = nullptr; size_t wave2_paths = 0; uint32_t wave2_depth = 0;
	WaveView wv2{};
	cudaStream_t stream2 = nullptr;
	cudaEvent_t ev_lane[2] = {nullptr, nullptr}, ev_fork = nullptr;
	cudaGraphExec_t graph_exec2 = nullptr;
	int lanes = 2;                            // RTB_LANES=1 switches the second lane off
	uint32_t call_params[4] = {0, 0, 0, 0};   // host copy of WaveView::call_params

	// cached per-batch graph
	cudaGraphExec_t graph_exec = nullptr;
	BatchParams graph_bp{}; rtb_camera graph_cam{}; SceneView graph_sv{}; bool graph_valid = false;   // what the captured launches were made with
	float4 *graph_accum = nullptr;

	uint64_t launches = 0, batches = 0;
	int bin_org_bits = 4, bin_dir_bits = 3;                  // ray binning: 2^(3 * 4 + 2 * 3) = 262,144 bins
	unsigned long long bin_mask = 0x116ull;                   // bounces whose queue is binned before it is traversed (1, 2, 4, 8: the order persists in between)
	bool bin_on = false, bin_forced = false, graph_bin_on = false;   // binning applies to this render / RTB_BIN_MASK was given / what the cached graph was built with
	uint32_t tail_threshold = 0;   // live-queue length below which the fused tail kernel takes a batch over

	// optional per-launch event timing (rtb_renderer_set_profiling)
	bool profiling = false;
	std::vector<cudaEvent_t> prof_events;      // pairs (begin, end)
	std::vector<int> prof_class;               // 0 generate, 1 traverse, 2 shade, 3 accumulate, 4 tail, 5 binning, 6 adaptive select
	size_t prof_used = 0;
};


// Resolve (mean -> clamp -> sqrt) of an arbitrary accumulator on this renderer's device and stream (rtb_multi.cu resolves
// the cross-device total with it).
int rtb_resolve_from(rtb_renderer* r, const float4* accum, void* d_out, void* user_stream);
int rtb_quantize_from(rtb_renderer* r, const float4* accum, uint8_t* host_rgb, int flip_rows);

#endif
