// rtb_kernels.h — launch interface of the wavefront kernels (rtb_kernels.cu).
#ifndef RTB_KERNELS_H
#define RTB_KERNELS_H

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rtb.h"

namespace rtb {

// Device views of the flattened scene (all pointers 64-byte aligned).
struct SceneView {
	const float4* nodes;        // 4 x float4 per inner node
	const float4* prims;        // 4 x float4 per primitive
	const int2* prim_info;      // (material, object)
	const float4* materials;    // 2 x float4 per material
	const float4* textures;     // 3 x float4 per texture
	const uint8_t* blob;        // image texels / Perlin tables
	const int32_t* pre_list;    // leaf codes of media tested before the BVH walk
	int32_t n_pre;
	int32_t bvh_empty;
	int32_t root_ref;
	int32_t n_prims;            // record slots
	int32_t n_nodes, n_materials, n_textures;   // (sizes of the sections: the debug build checks every index against them)
	uint32_t n_blob;
	int32_t tree_depth;         // depth of the world BVH in nodes (selects the stack size of the traverse kernel)
	int32_t has_media;          // 0 none, 1 all media in the pre-test list, 2 some media are BVH leaves (selects the traverse variant)
	int32_t launch_flags;       // the scene's part of the feature word (below); SV_DEFERRED_TEX: some material has an image /
	                            // noise albedo, texture_kernel is launched after shade
	int32_t background_mode;
	float bg_r, bg_g, bg_b;
	// Ray binning (bin_scan / bin_permute kernels): origin cells are counted on a 2^org_bits cube over the world BVH's
	// bounds, directions on a 2^dir_bits square of the octahedral map; 0 / 0 switches binning off.
	float bin_min[3], bin_scale[3];   // cell coordinate = (o - bin_min) * bin_scale, clamped to [0, 2^org_bits)
	int32_t bin_org_bits, bin_dir_bits;
	int32_t n_tri_attr;         // triangle attribute records (in the padding before `lights`)
	// Sampled lights (DESIGN.md §5b): n_lights world-space records (4 x float4, SPHERE / QUAD layout), then n_lights
	// float4 (type bits, quad area, 0, 0).  n_lights = 0: no light sampling (the kernels without it are launched).
	const float4* lights;
	int32_t n_lights;
	// Environment map (DESIGN.md §5d): env_width x env_height float4 texels (r, g, b, pdf numerator), row 0 = top, then the
	// marginal CDF (env_height + 1 floats) and env_height conditional CDFs (env_width + 1 floats each).  env = null: no map
	// (the kernels without one are launched).  env_sample: the map is one more strategy of the light mixture.
	int32_t env_width;
	const float4* env;
	int32_t env_height, env_sample;
	// Triangle attributes (DESIGN.md §5e): n_tri_attr records of 4 x float4 (DevTriAttr), and per record slot the index of its
	// triangle's record or -1.  tri_attr = null: no attributes (the kernels without them are launched).
	const float4* tri_attr;
	const int32_t* attr_slot;
};
// The feature word F of the shade and tail kernels (their last template parameter): which code a scene or a batch needs.
// Each bit is one feature, and a kernel without a feature's bit is the kernel of scenes without that feature.  A new
// feature takes the next bit, so every existing word, and the instantiation and kernel name it stands for, stays.
//   F_LIGHTS  the light mixture (DESIGN.md §5b): sampled lights, or a sampled environment map (one more strategy of it)
//   F_LIST    an adaptive round (DESIGN.md §5c): local pixels come from BatchParams::pixel_list()
//   F_ENV     an environment map (DESIGN.md §5d): a miss returns its texel
//   F_ATTR    triangle attributes (DESIGN.md §5e)
//   F_ROUGH   GGX materials (DESIGN.md §5f)
enum : uint32_t { F_LIGHTS = 1, F_LIST = 2, F_ENV = 4, F_ATTR = 8, F_ROUGH = 16, F_WORDS = 32 };
// SceneView::launch_flags (read by the launchers only, never on the device): the word's scene bits, computed once where the
// scene is staged (every bit but F_LIST, which the launchers add from the batch), and SV_DEFERRED_TEX above the word.
enum : uint32_t { SV_DEFERRED_TEX = 1u << 16 };
// The map's fields fill the padding after n_lights and add 16 bytes, the attribute count fills the padding before `lights`
// and its two pointers add 16 more, so every kernel parameter after the SceneView keeps its offset modulo 16 (see BatchParams
// below for what a moved parameter costs).
// The scene's feature bits are part of launch_flags, not fields of their own, for the same reason.
static_assert(alignof(SceneView) == 8 && sizeof(SceneView) == 200 && offsetof(SceneView, launch_flags) == 96 && offsetof(SceneView, n_tri_attr) == 148 &&
              offsetof(SceneView, lights) == 152 && offsetof(SceneView, n_lights) == 160 && offsetof(SceneView, env_width) == 164 &&
              offsetof(SceneView, env) == 168 && offsetof(SceneView, tri_attr) == 184, "SceneView layout changed");

// One batch = `samples_per_batch` consecutive samples of every pixel of the row range.
struct BatchParams {
	uint32_t width, height;
	uint32_t row_begin, n_rows;
	uint32_t npix;              // width * n_rows
	uint32_t sample_begin, sample_end;
	uint32_t samples_per_batch;
	uint32_t max_depth;
	uint32_t seed;
	uint32_t variance;
	// A render's batches can be dealt to two lanes (two streams with their own queues, so that the thin late bounces of one
	// batch overlap the full early bounces of the next): the lane's k-th batch is batch_base + k * batch_stride.
	uint32_t batch_base, batch_stride;
	// Adaptive rounds (DESIGN.md §5c): npix = the number of listed pixels, and local pixel pl is pixel_list()[pl] instead of
	// row_begin * width + pl.  Null = dense (every pixel of the row range); the launchers pick the list-mode kernels by it.
	// (Kept as two 32-bit words after two unused ones: the struct stays 4-byte aligned and grows by 16 bytes, so every kernel
	// parameter after it keeps its offset modulo 16.  With 8 bytes more, the camera parameter of generate_kernel moved to
	// another alignment, the compiler picked other constant loads, and bench.py measured that layout 0.18 % slower.)
	uint32_t unused[2];
	uint32_t pixel_list_lo, pixel_list_hi;
	__host__ __device__ const uint32_t* pixel_list() const {
		return reinterpret_cast<const uint32_t*>(((uint64_t)pixel_list_hi << 32) | pixel_list_lo);
	}
	__host__ __device__ void set_pixel_list(const uint32_t* p) {
		pixel_list_lo = (uint32_t)(uintptr_t)p; pixel_list_hi = (uint32_t)((uint64_t)(uintptr_t)p >> 32);
	}
};
// The layout the comment above depends on.  A field added to BatchParams moves every kernel parameter after it: keep the
// size a multiple of 16 bytes more than the 52 of the fields before the list (tools/sass_diff.py against the previous build
// shows whether the dense kernels still compile to the same instructions), then update these numbers.
static_assert(alignof(BatchParams) == 4 && sizeof(BatchParams) == 68 && offsetof(BatchParams, unused) == 52 &&
              offsetof(BatchParams, pixel_list_lo) == 60, "BatchParams layout changed: see the comment above");

// Buffers and parameters of the adaptive select step (rtb_render_adaptive): the error of every pixel of the row range, then
// the ascending list of the pixels the next round renders and its length.
struct AdaptiveView {
	const float4* accum;        // (sums, count)
	const float4* accum2;       // (sums of squares, count)
	float* err;                 // [width * height] display-space standard error e_p
	uint32_t* list;             // [width * height] the active pixels, ascending
	uint32_t* block_count;      // [blocks of the select step] active pixels per block, then their exclusive prefix sums
	uint32_t* result;           // [0] active pixels, [1] nonzero when a pixel holding the cursor has no sums of squares
	uint32_t width, row_begin, n_rows;
	uint32_t cursor, min_spp, max_spp;
	float tolerance;
};

// Wavefront queues, double buffered.  A ray is a 32-byte record (o.xyz, time)(d.xyz, path id bits) - one DRAM sector, so
// the binning pass, which scatters rays, writes whole sectors - plus its throughput in a parallel array.
struct WaveView {
	float4* ray_od[2];          // 2 x float4 per ray: (o.xyz, time), (d.xyz, path id bits)
	float4* thr[2];             // (throughput rgb, -)
	int2* hit;                  // (t bits, leaf code or -1)
	float4* contrib;            // per path: radiance carried by the terminated path
	uint32_t* n_live;           // [max_depth + 1] queue lengths per bounce
	uint32_t* work;             // [2 * (max_depth + 1)] dynamic work counters (traverse, shade)
	float4* tex_work;           // deferred texture evaluations: 2 x float4 per entry
	uint32_t* n_tex;            // [max_depth + 1] entries per bounce
	uint32_t capacity;          // paths the queues hold
	uint32_t n_bins;
	uint32_t* bin_count;        // [2^(3 org_bits + 2 dir_bits)] rays of the next queue per bin (zero between uses)
	uint32_t* bin_cursor;       // same size: where the next ray of each bin goes
	const uint32_t* call_params; // [4] sample_begin, sample_end, seed of the current rtb_render call (BatchParams carries stale copies in a replayed graph)
	uint32_t* batch_index;      // device-side batch counter (graph replays need no new arguments)
	uint32_t* tail_from;        // first bounce handled by the fused tail kernel (0xFFFFFFFF: none yet)
	unsigned long long* totals; // [0] paths, [1] rays
};

struct LaunchCfg { int blocks_traverse, blocks_shade, blocks_stream, blocks_tail, blocks_bin, sms; };

void launch_generate(const BatchParams& bp, const rtb_camera& cam, const WaveView& wv, const LaunchCfg& lc, cudaStream_t st);
// `q` = which of the two ray queues holds the rays of `bounce` (the renderer's static schedule: the queues alternate from
// bounce to bounce, except that a binned bounce is permuted back into the queue its predecessor was read from).
void launch_traverse(const SceneView& sv, const BatchParams& bp, const WaveView& wv, uint32_t bounce, int q, const LaunchCfg& lc, cudaStream_t st);
void launch_tail(const SceneView& sv, const BatchParams& bp, const WaveView& wv, uint32_t bounce, int q, uint32_t threshold, const LaunchCfg& lc, cudaStream_t st);
// shade reads queue q and writes the survivors to queue q ^ 1
void launch_shade(const SceneView& sv, const BatchParams& bp, const WaveView& wv, uint32_t bounce, int q, const LaunchCfg& lc, cudaStream_t st);
void launch_texture(const SceneView& sv, const WaveView& wv, uint32_t bounce, int q_out, const LaunchCfg& lc, cudaStream_t st);
// Binning of the rays of `bounce` (a counting sort by ray_bin: count, prefix sums, permute): every ray of queue q_from
// moves to its bin's range in queue q_from ^ 1.
void launch_bin_rays(const SceneView& sv, const WaveView& wv, uint32_t bounce, int q_from, const LaunchCfg& lc, cudaStream_t st);
void launch_accumulate(const BatchParams& bp, const WaveView& wv, float4* accum, float4* accum2, const LaunchCfg& lc, cudaStream_t st);
// Adaptive select step: per-pixel error (skipped while cursor < min_spp: every candidate is active then), window and
// candidate test, ascending compaction into av.list; av.result[0..1] must be zero before.  Blocks of the select step:
uint32_t adaptive_select_blocks(uint32_t n_pixels);
void launch_adaptive_select(const AdaptiveView& av, const LaunchCfg& lc, cudaStream_t st);
void launch_resolve(const float4* accum, float4* out, uint32_t n, cudaStream_t st);
void launch_quantize(const float4* accum, uint8_t* rgb, uint32_t width, uint32_t height, int flip_rows, cudaStream_t st);

// Parity hook: closest hits + full hit records for explicit rays (media skipped).
void launch_trace_rays(const SceneView& sv, const float4* ray_o, const float4* ray_d, uint32_t n, int2* hit_tmp, int2* stats_tmp,
                       rtb_hit* hits_out, uint32_t* work_counter, const LaunchCfg& lc, cudaStream_t st);

void query_occupancy(int device, LaunchCfg& lc);

// -DRTB_DEBUG_BOUNDS=1 builds: per-class counts of out-of-range indices seen by the kernels on the current device.
enum { RTB_BOUNDS_STACK = 0, RTB_BOUNDS_NODE, RTB_BOUNDS_PRIM, RTB_BOUNDS_MATERIAL, RTB_BOUNDS_TEXTURE, RTB_BOUNDS_QUEUE, RTB_BOUNDS_PATH, RTB_BOUNDS_BIN, RTB_BOUNDS_CLASSES };
int debug_bounds_report(unsigned long long* violations, unsigned long long* checks);   // 1 = filled, 0 = not a debug build, -1 = CUDA error

}  // namespace rtb
#endif
