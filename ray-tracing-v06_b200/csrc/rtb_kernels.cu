// rtb_kernels.cu — the wavefront path tracer's CUDA kernels (sm_100a).
//
//   generate    camera rays for one batch of (pixel, sample) paths          Renderer.cu:183-204, cu_Cameras.cuh:27-30,54-64,87-89
//   traverse    closest hit through the 64-byte two-box BVH nodes           BVH.cu:54-106, aabb.cuh:30-44, SphereHittable.cuh:15-33
//   shade       material scatter + texture evaluation + queue compaction    Renderer.cu:139-181, cu_materials.cuh:17-144, cu_Textures.cuh:9-40
//   accumulate  per-pixel sum of the batch's path contributions             Renderer.cu:204-206
//   resolve     mean -> clamp -> sqrt -> float4                             Renderer.cu:206-216
//
// Compiled with -fmad=false: every fused multiply-add below is explicit (see rtmath.h), so the
// CPU oracle reproduces the geometry bit for bit.  No tensor cores: nothing here is a dense
// contraction.  All kernels are persistent (grid = SMs x resident blocks) and pull work in
// warp- or block-sized chunks from a device counter, so the same launch sequence (and the same
// CUDA graph) serves every bounce regardless of how many paths are still alive.
//
// The device code shared with the shade and tail kernels, and those kernels, are in rtb_device.h; rtb_shade.cu and
// rtb_tail.cu instantiate them in objects of their own, and the launchers below pick them by feature word.
#include "rtb_device.h"

namespace rtb {

#if RTB_DEBUG_BOUNDS
__device__ unsigned long long g_bounds_violations[RTB_BOUNDS_CLASSES];
__device__ unsigned long long g_bounds_checks;
#endif

// ------------------------------------------------------------------------------------------------
// generate

template <bool LIST>
__global__ void __launch_bounds__(STREAM_THREADS)
generate_kernel(BatchParams bp_in, rtb_camera cam, WaveView wv) {
	const BatchParams bp = with_call_params(bp_in, wv);
	const uint32_t batch = bp.batch_base + *wv.batch_index * bp.batch_stride;
	const uint32_t ns = batch_sample_count(bp, batch);
	const uint32_t n = ns * bp.npix;
	const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t stride = gridDim.x * blockDim.x;

	// Reset the per-bounce queue lengths and work counters of this batch.
	if (blockIdx.x == 0) {
		for (uint32_t i = threadIdx.x; i <= bp.max_depth; i += blockDim.x) wv.n_live[i] = (i == 0) ? n : 0u;
		for (uint32_t i = threadIdx.x; i < 2 * (bp.max_depth + 1); i += blockDim.x) wv.work[i] = 0u;
		for (uint32_t i = threadIdx.x; i <= bp.max_depth; i += blockDim.x) wv.n_tex[i] = 0u;
		if (threadIdx.x == 0) *wv.tail_from = 0xFFFFFFFFu;
	}

	const float px = 1.0f / (float)bp.width, py = 1.0f / (float)bp.height;   // pixel_size  Renderer.cu:188
	for (uint32_t path = tid; path < n; path += stride) {
		uint32_t pixel, sample;
		path_pixel_sample<LIST>(bp, batch, path, pixel, sample);
		uint32_t y = pixel / bp.width, x = pixel - y * bp.width;
		rt::f4 r = rt::rng4(bp.seed, pixel, sample, RT_CAMERA_BOUNCE, rt::STREAM_SCATTER);
		// ndc = (vec2(x,y) + 0.5) * pixel_size * 2 - 1 ; jitter = point in unit disc * pixel_size   Renderer.cu:192,199
		float ndcx = fmaf(((float)x + 0.5f) * px, 2.0f, -1.0f);
		float ndcy = fmaf(((float)y + 0.5f) * py, 2.0f, -1.0f);
		float jx, jy; rt::unit_disc(r.x, r.y, jx, jy);
		float s = fmaf(jx, px, ndcx), t = fmaf(jy, py, ndcy);
		v3 o = rt::mk(cam.o[0], cam.o[1], cam.o[2]);
		v3 cu = rt::mk(cam.u[0], cam.u[1], cam.u[2]), cv = rt::mk(cam.v[0], cam.v[1], cam.v[2]), cw = rt::mk(cam.w[0], cam.w[1], cam.w[2]);
		v3 d; float time = 0.0f;
		if (cam.kind == RTB_CAM_DEFOCUS) {
			// DefocusBlurCamera::sample_ray  cu_Cameras.cuh:54-64
			rt::f4 l = rt::rng4(bp.seed, pixel, sample, RT_CAMERA_BOUNCE, rt::STREAM_LENS);
			float lx, ly; rt::unit_disc(l.x, l.y, lx, ly);
			v3 off = rt::mul(rt::mk(fmaf(cv.x, ly, cu.x * lx), fmaf(cv.y, ly, cu.y * lx), fmaf(cv.z, ly, cu.z * lx)), cam.lens_radius);
			v3 fwd = rt::mul(cw, cam.focus_dist);
			v3 hori = rt::mul(rt::mul(cu, cam.viewport_width), cam.focus_dist);
			v3 vert = rt::mul(rt::mul(cv, cam.viewport_height), cam.focus_dist);
			d = rt::sub(rt::madd(vert, t, rt::madd(hori, s, fwd)), off);
			o = rt::add(o, off);
			time = rt::mixf(cam.t0, cam.t1, r.z);
		} else {
			// PinholeCamera / MotionBlurCamera::sample_ray  cu_Cameras.cuh:27-30,87-89
			d = rt::madd(cv, t, rt::madd(cu, s, cw));
			if (cam.kind == RTB_CAM_MOTION) time = rt::mixf(cam.t0, cam.t1, r.z);
		}
		st_ray(wv.ray_od[0] + 2 * (size_t)path, make_float4(o.x, o.y, o.z, time), make_float4(d.x, d.y, d.z, __uint_as_float(path)));
		stq(wv.thr[0] + path, make_float4(1.0f, 1.0f, 1.0f, 0.0f));
		stq(wv.contrib + path, make_float4(0.0f, 0.0f, 0.0f, 0.0f));
	}
}

#ifndef TRAVERSE_MIN_BLOCKS
#define TRAVERSE_MIN_BLOCKS 8   // 8 x 128 threads x 64 registers = the whole register file
#endif
// STACK = entries of the per-thread stack in shared memory: 16 when the tree is shallow enough (8 KB per
// block instead of 16 KB leaves 64 KB more L1 per SM: -2 % on the Book 2 final scene), 32 otherwise.
// LIST (adaptive rounds, media only: without media the walk never derives a pixel): the media RNG gathers the pixel.
template <int MEDIA, int STACK, bool LIST>
__global__ void __launch_bounds__(TRAVERSE_THREADS, TRAVERSE_MIN_BLOCKS)
traverse_kernel(SceneView sv, BatchParams bp_in, WaveView wv, uint32_t bounce, int q) {
	const BatchParams bp = with_call_params(bp_in, wv);
	__shared__ int s_stack[STACK * TRAVERSE_THREADS];
	if (bounce >= *wv.tail_from) return;
	const uint32_t n = wv.n_live[bounce];
	if (n == 0) return;
	if (blockIdx.x == 0 && threadIdx.x == 0) { RTB_COUNT_CHECKS(n); RTB_CHECK(n <= wv.capacity, RTB_BOUNDS_QUEUE); }
	const uint32_t batch = bp.batch_base + *wv.batch_index * bp.batch_stride;
	const int lane = threadIdx.x & 31;
	const float4* __restrict__ rod = q ? wv.ray_od[1] : wv.ray_od[0];
	uint32_t* counter = wv.work + 2 * bounce;
	// Every warp owns one static chunk of 32 rays; only when the queue is longer than the whole
	// grid do warps pull further chunks from the device counter (short queues cost no atomics).
	const uint32_t warps_total = gridDim.x * (TRAVERSE_THREADS / 32);
	uint32_t base = (blockIdx.x * (TRAVERSE_THREADS / 32) + (threadIdx.x >> 5)) * 32u;
	const uint32_t static_span = warps_total * 32u;
	while (base < n) {
		const uint32_t i = base + lane;
		if (i < n) {
			float4 fo, fd; ld_ray(rod + 2 * (size_t)i, fo, fd);
			MediumRngT<LIST> mr = make_medium_rng<LIST>(bp, batch, __float_as_uint(fd.w), bounce);
			float t; int code;
			trace_ray<MEDIA>(sv, xyz(fo), xyz(fd), fo.w, mr, s_stack + threadIdx.x, STACK, t, code);
			RTB_CHECK(i < wv.capacity, RTB_BOUNDS_QUEUE);
			stq(wv.hit + i, make_int2(__float_as_int(t), code));
		}
		__syncwarp();
		if (n <= static_span) break;
		uint32_t nb = 0;
		if (lane == 0) nb = atomicAdd(counter, 32u);
		base = static_span + __shfl_sync(FULL_MASK, nb, 0);
	}
}

// Bin of a ray for the binning pass: Morton code of the origin's cell on a 2^org_bits cube over the world bounds, then the
// cell of the direction on a 2^dir_bits square of the octahedral map.  Rays of one bin start close together and head the
// same way, so the lanes of a warp walk the same nodes (measured on B200: 12 -> 20+ active lanes on secondary bounces).
__device__ __forceinline__ uint32_t spread3(uint32_t v) {   // 10 bits -> every third bit
	v = (v | (v << 16)) & 0x030000FFu; v = (v | (v << 8)) & 0x0300F00Fu; v = (v | (v << 4)) & 0x030C30C3u; v = (v | (v << 2)) & 0x09249249u;
	return v;
}
__device__ __forceinline__ uint32_t ray_bin(const SceneView& sv, const float4& o, const float4& d) {
	const int qo = 1 << sv.bin_org_bits;
	int ix = (int)((o.x - sv.bin_min[0]) * sv.bin_scale[0]), iy = (int)((o.y - sv.bin_min[1]) * sv.bin_scale[1]), iz = (int)((o.z - sv.bin_min[2]) * sv.bin_scale[2]);
	ix = min(max(ix, 0), qo - 1); iy = min(max(iy, 0), qo - 1); iz = min(max(iz, 0), qo - 1);
	uint32_t key = spread3((uint32_t)ix) | (spread3((uint32_t)iy) << 1) | (spread3((uint32_t)iz) << 2);
	if (sv.bin_dir_bits > 0) {
		const float s = 1.0f / (fabsf(d.x) + fabsf(d.y) + fabsf(d.z) + 1e-30f);
		float u = d.x * s, v = d.z * s;
		if (d.y < 0.0f) { const float uu = (1.0f - fabsf(v)) * (u >= 0.0f ? 1.0f : -1.0f), vv = (1.0f - fabsf(u)) * (v >= 0.0f ? 1.0f : -1.0f); u = uu; v = vv; }
		const int qd = 1 << sv.bin_dir_bits;
		int iu = (int)((u * 0.5f + 0.5f) * (float)qd), iv = (int)((v * 0.5f + 0.5f) * (float)qd);
		iu = min(max(iu, 0), qd - 1); iv = min(max(iv, 0), qd - 1);
		key = (key << (2 * sv.bin_dir_bits)) | (uint32_t)(iv * qd + iu);
	}
	return key;
}
// Shared-memory hash table of (bin, rays) used by the binning kernels (see "binning" below).
// (B200, r2: tiles of 1,024 / 2,048 / 4,096 rays = 256 / 512 / 1,024 threads x 4: binning 4.75 / 4.05 / 4.17 ms per batch - a global
// counter is touched once per distinct key of a TILE, so larger tiles send fewer atomics, until one block per SM is too few.)
#ifndef BIN_THREADS
#define BIN_THREADS 512
#endif
#ifndef BIN_ITEMS
#define BIN_ITEMS 4                                  // rays per thread per tile
#endif
#define BIN_TILE (BIN_THREADS * BIN_ITEMS)
#ifndef BIN_SLOTS_LOG2
#define BIN_SLOTS_LOG2 12
#endif
#ifndef BIN_MIN_BLOCKS
#define BIN_MIN_BLOCKS 2                             // 2 x 512 threads x 64 registers
#endif
#define BIN_LAUNCH_BOUNDS __launch_bounds__(BIN_THREADS, BIN_MIN_BLOCKS)
#define BIN_SLOTS (1 << BIN_SLOTS_LOG2)              // hash slots per block: at most half full with one tile's keys
#define BIN_EMPTY 0xFFFFFFFFu
#define BIN_COUNT_SMEM (2 * BIN_SLOTS * sizeof(uint32_t))
#define BIN_PERMUTE_SMEM (3 * BIN_SLOTS * sizeof(uint32_t))

// Finds or claims the slot of `key` and counts one ray in it (linear probing; callers keep the table at most half full).
// Returns the slot, with the top bit set when this call claimed it.
__device__ __forceinline__ uint32_t bin_table_add(uint32_t* s_key, uint32_t* s_cnt, uint32_t key) {
	uint32_t h = (key * 2654435761u) >> (32 - BIN_SLOTS_LOG2);  // Fibonacci hash to log2(BIN_SLOTS) bits
	for (;;) {
		const uint32_t prev = atomicCAS(s_key + h, BIN_EMPTY, key);
		if (prev == BIN_EMPTY || prev == key) { atomicAdd(s_cnt + h, 1u); return prev == BIN_EMPTY ? (h | 0x80000000u) : h; }
		h = (h + 1u) & (BIN_SLOTS - 1u);
	}
}

// One global atomic per bin the table holds, then the table is empty again (all threads of the block).
__device__ __forceinline__ void bin_table_flush(uint32_t* s_key, uint32_t* s_cnt, uint32_t* bin_count, uint32_t n_bins, int threads) {
	for (uint32_t s = threadIdx.x; s < BIN_SLOTS; s += threads) {
		const uint32_t key = s_key[s];
		if (key != BIN_EMPTY) { RTB_CHECK(key < n_bins, RTB_BOUNDS_BIN); atomicAdd(bin_count + key, s_cnt[s]); s_key[s] = BIN_EMPTY; s_cnt[s] = 0u; }
	}
}

// ------------------------------------------------------------------------------------------------
// texture: evaluates the image / Perlin albedos that shade deferred, with dense warps, and folds them
// into the throughput of the scattered rays (thr * value is the same single product either way).

__global__ void __launch_bounds__(STREAM_THREADS)
texture_kernel(SceneView sv, WaveView wv, uint32_t bounce, int q_out) {
	if (bounce >= *wv.tail_from) return;
	const uint32_t n = wv.n_tex[bounce];
	if (n == 0) return;
	float4* __restrict__ wt = q_out ? wv.thr[1] : wv.thr[0];
	const uint32_t stride = gridDim.x * blockDim.x;
	for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
		const float4 a = wv.tex_work[2 * (size_t)k], b = wv.tex_work[2 * (size_t)k + 1];
		const v3 val = texture_value(sv, __float_as_int(b.w), b.x, b.y, xyz(a));
		const uint32_t pos = __float_as_uint(a.w);
		RTB_CHECK(pos < wv.capacity && __float_as_int(b.w) >= 0 && __float_as_int(b.w) < sv.n_textures, RTB_BOUNDS_QUEUE);
		float4 t = wt[pos];
		t.x *= val.x; t.y *= val.y; t.z *= val.z;
		wt[pos] = t;
	}
}

// ------------------------------------------------------------------------------------------------
// binning: a counting sort of the live queue by ray_bin between shade(b - 1) and traverse(b), in three launches.
//   bin_count    rays per bin
//   bin_scan     exclusive prefix sums of the counts = the first slot of every bin
//   bin_permute  every ray moves to the next free slot of its bin in the other queue
// Rays pile up in few bins (a third of the late-bounce rays of the Book 2 final scene scatter inside one sphere of
// smoke), so neither kernel sends one global atomic per ray: each block aggregates the keys of its rays in a small
// shared-memory hash table first - same-address atomics are cheap there - and touches a global counter once per distinct
// key.  Where a ray sits in a queue changes nothing about the image - contributions are stored by path id and summed per
// pixel in sample order - only which rays share a warp.

// Rays per bin.  A block's counts gather in its table over many tiles and go to the global counters when the table might
// not hold another tile's keys, and at the end.
__global__ void BIN_LAUNCH_BOUNDS
bin_count_kernel(SceneView sv, WaveView wv, uint32_t bounce, int q) {
	extern __shared__ uint32_t s_bin[];                   // BIN_COUNT_SMEM bytes
	uint32_t* const s_key = s_bin; uint32_t* const s_cnt = s_bin + BIN_SLOTS;
	__shared__ uint32_t s_used;
	if (bounce >= *wv.tail_from) return;
	const uint32_t n = wv.n_live[bounce];
	if (n == 0) return;
	const float4* __restrict__ rod = q ? wv.ray_od[1] : wv.ray_od[0];
	for (uint32_t s = threadIdx.x; s < BIN_SLOTS; s += BIN_THREADS) { s_key[s] = BIN_EMPTY; s_cnt[s] = 0u; }
	if (threadIdx.x == 0) s_used = 0u;
	__syncthreads();
	for (uint32_t base = blockIdx.x * BIN_TILE; base < n; base += gridDim.x * BIN_TILE) {
		uint32_t claimed = 0;
#pragma unroll
		for (int k = 0; k < BIN_ITEMS; ++k) {
			const uint32_t i = base + k * BIN_THREADS + threadIdx.x;
			if (i < n) { float4 o, d; ld_ray(rod + 2 * (size_t)i, o, d); claimed += bin_table_add(s_key, s_cnt, ray_bin(sv, o, d)) >> 31; }
		}
		if (claimed) atomicAdd(&s_used, claimed);
		__syncthreads();
		if (s_used > BIN_SLOTS / 2 - BIN_TILE / 2) {          // (a tile adds at most BIN_TILE keys; past this mark, flush)
			__syncthreads();
			bin_table_flush(s_key, s_cnt, wv.bin_count, wv.n_bins, BIN_THREADS);
			if (threadIdx.x == 0) s_used = 0u;
			__syncthreads();
		}
	}
	bin_table_flush(s_key, s_cnt, wv.bin_count, wv.n_bins, BIN_THREADS);
}

// Block b owns bins [b * 4096, (b + 1) * 4096): it adds up everything before them (the counts are re-read from L2 - at
// most 1 MB - instead of passing block totals around), then scans its own.  The counters are zeroed by bin_permute.
#define BIN_SCAN_THREADS 1024
#define BIN_SCAN_PER_BLOCK 4096
__global__ void __launch_bounds__(BIN_SCAN_THREADS)
bin_scan_kernel(WaveView wv, uint32_t bounce) {
	__shared__ uint32_t s_part[BIN_SCAN_THREADS];
	__shared__ uint32_t s_before;
	if (bounce >= *wv.tail_from || wv.n_live[bounce] == 0) return;
	const uint32_t first = blockIdx.x * BIN_SCAN_PER_BLOCK;
	uint32_t sum = 0;
	for (uint32_t b = threadIdx.x; b < first; b += BIN_SCAN_THREADS) sum += wv.bin_count[b];
	s_part[threadIdx.x] = sum;
	__syncthreads();
	for (uint32_t off = BIN_SCAN_THREADS / 2; off > 0; off >>= 1) {
		if (threadIdx.x < off) s_part[threadIdx.x] += s_part[threadIdx.x + off];
		__syncthreads();
	}
	if (threadIdx.x == 0) s_before = s_part[0];
	__syncthreads();
	// own bins: 4 consecutive bins per thread (one 16-byte load), block-wide inclusive scan of the per-thread sums
	const uint32_t b0 = first + 4u * threadIdx.x;
	uint4 c = make_uint4(0, 0, 0, 0);
	if (b0 + 3u < wv.n_bins) c = *reinterpret_cast<const uint4*>(wv.bin_count + b0);
	else { if (b0 < wv.n_bins) c.x = wv.bin_count[b0]; if (b0 + 1u < wv.n_bins) c.y = wv.bin_count[b0 + 1u]; if (b0 + 2u < wv.n_bins) c.z = wv.bin_count[b0 + 2u]; }
	const uint32_t mine = c.x + c.y + c.z + c.w;
	__syncthreads();
	s_part[threadIdx.x] = mine;
	__syncthreads();
	for (uint32_t off = 1; off < BIN_SCAN_THREADS; off <<= 1) {
		const uint32_t v = threadIdx.x >= off ? s_part[threadIdx.x - off] : 0u;
		__syncthreads();
		s_part[threadIdx.x] += v;
		__syncthreads();
	}
	uint32_t run = s_before + s_part[threadIdx.x] - mine;
	if (b0 < wv.n_bins) wv.bin_cursor[b0] = run; run += c.x;
	if (b0 + 1u < wv.n_bins) wv.bin_cursor[b0 + 1u] = run; run += c.y;
	if (b0 + 2u < wv.n_bins) wv.bin_cursor[b0 + 2u] = run; run += c.z;
	if (b0 + 3u < wv.n_bins) wv.bin_cursor[b0 + 3u] = run;
}

__global__ void BIN_LAUNCH_BOUNDS
bin_permute_kernel(SceneView sv, WaveView wv, uint32_t bounce, int q_from) {
	extern __shared__ uint32_t s_bin[];                   // BIN_PERMUTE_SMEM bytes
	uint32_t* const s_key = s_bin; uint32_t* const s_cnt = s_bin + BIN_SLOTS; uint32_t* const s_base = s_bin + 2 * BIN_SLOTS;
	if (bounce >= *wv.tail_from) return;
	const uint32_t n = wv.n_live[bounce];
	if (n == 0) return;
	// the counters of this bounce are dead once bin_scan has run: leave them zero for the next binned bounce
	for (uint32_t b = blockIdx.x * BIN_THREADS + threadIdx.x; b < wv.n_bins; b += gridDim.x * BIN_THREADS) wv.bin_count[b] = 0u;
	const float4* __restrict__ rod = q_from ? wv.ray_od[1] : wv.ray_od[0];
	const float4* __restrict__ rt_ = q_from ? wv.thr[1] : wv.thr[0];
	float4* __restrict__ wod = q_from ? wv.ray_od[0] : wv.ray_od[1];
	float4* __restrict__ wt = q_from ? wv.thr[0] : wv.thr[1];
	for (uint32_t s = threadIdx.x; s < BIN_SLOTS; s += BIN_THREADS) { s_key[s] = BIN_EMPTY; s_cnt[s] = 0u; }
	__syncthreads();
	for (uint32_t base = blockIdx.x * BIN_TILE; base < n; base += gridDim.x * BIN_TILE) {
		float4 o[BIN_ITEMS], d[BIN_ITEMS], t[BIN_ITEMS];
		uint32_t slot[BIN_ITEMS];
#pragma unroll
		for (int k = 0; k < BIN_ITEMS; ++k) {
			const uint32_t i = base + k * BIN_THREADS + threadIdx.x;
			if (i < n) { ld_ray(rod + 2 * (size_t)i, o[k], d[k]); t[k] = ldq(rt_ + i); }
		}
#pragma unroll
		for (int k = 0; k < BIN_ITEMS; ++k) {
			const uint32_t i = base + k * BIN_THREADS + threadIdx.x;
			slot[k] = i < n ? (bin_table_add(s_key, s_cnt, ray_bin(sv, o[k], d[k])) & 0x7FFFFFFFu) : 0u;
		}
		__syncthreads();
		// a run of slots in the other queue for every distinct key of the tile
		for (uint32_t s = threadIdx.x; s < BIN_SLOTS; s += BIN_THREADS) {
			const uint32_t key = s_key[s];
			if (key != BIN_EMPTY) { RTB_CHECK(key < wv.n_bins, RTB_BOUNDS_BIN); s_base[s] = atomicAdd(wv.bin_cursor + key, s_cnt[s]); s_cnt[s] = 0u; }
		}
		__syncthreads();
#pragma unroll
		for (int k = 0; k < BIN_ITEMS; ++k) {
			const uint32_t i = base + k * BIN_THREADS + threadIdx.x;
			if (i < n) {
				const uint32_t pos = s_base[slot[k]] + atomicAdd(s_cnt + slot[k], 1u);
				RTB_CHECK(pos < n && pos < wv.capacity, RTB_BOUNDS_QUEUE);
				st_ray(wod + 2 * (size_t)pos, o[k], d[k]); wt[pos] = t[k];   // (the 32-byte ray record is one whole sector)
			}
		}
		__syncthreads();
		for (uint32_t s = threadIdx.x; s < BIN_SLOTS; s += BIN_THREADS) { s_key[s] = BIN_EMPTY; s_cnt[s] = 0u; }
		__syncthreads();
	}
}

// ------------------------------------------------------------------------------------------------
// accumulate + batch epilogue + resolve

// LIST: the sums of local pixel pl go to pixel_list[pl], with the same float operations as dense, and the sums of squares
// are always kept (the stopping rule needs them).
template <bool LIST>
__global__ void __launch_bounds__(STREAM_THREADS)
accumulate_kernel(BatchParams bp_in, WaveView wv, float4* __restrict__ accum, float4* __restrict__ accum2) {
	const BatchParams bp = with_call_params(bp_in, wv);
	const uint32_t batch = bp.batch_base + *wv.batch_index * bp.batch_stride;
	const uint32_t ns = batch_sample_count(bp, batch);
	if (ns == 0) return;
	const uint32_t stride = gridDim.x * blockDim.x;
	for (uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x; pl < bp.npix; pl += stride) {
		float sx = 0.0f, sy = 0.0f, sz = 0.0f, qx = 0.0f, qy = 0.0f, qz = 0.0f;
		for (uint32_t s = 0; s < ns; ++s) {   // fixed sample order: deterministic sums
			const float4 c = wv.contrib[(size_t)s * bp.npix + pl];
			sx += c.x; sy += c.y; sz += c.z;
			if (LIST || bp.variance) { qx = fmaf(c.x, c.x, qx); qy = fmaf(c.y, c.y, qy); qz = fmaf(c.z, c.z, qz); }
		}
		const uint32_t gid = LIST ? listed_pixel(bp.pixel_list(), pl, bp.row_begin * bp.width, bp.n_rows * bp.width) : bp.row_begin * bp.width + pl;
		float4 a = accum[gid];
		a.x += sx; a.y += sy; a.z += sz; a.w += (float)ns;
		accum[gid] = a;
		if (LIST || bp.variance) {
			float4 q = accum2[gid];
			q.x += qx; q.y += qy; q.z += qz; q.w += (float)ns;
			accum2[gid] = q;
		}
	}
}

__global__ void end_batch_kernel(BatchParams bp_in, WaveView wv) {
	const BatchParams bp = with_call_params(bp_in, wv);
	if (threadIdx.x != 0 || blockIdx.x != 0) return;
	unsigned long long rays = 0;
	for (uint32_t b = 0; b < bp.max_depth; ++b) rays += wv.n_live[b];
	wv.totals[0] += wv.n_live[0];
	wv.totals[1] += rays;
	*wv.batch_index += 1;
}

__global__ void __launch_bounds__(STREAM_THREADS)
resolve_kernel(const float4* __restrict__ accum, float4* __restrict__ out, uint32_t n) {
	const uint32_t stride = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
		const float4 a = accum[i];
		const float inv = 1.0f / a.w;                              // radiance *= 1.0f / spp   Renderer.cu:206
		float r = a.x * inv, g = a.y * inv, b = a.z * inv;
		r = fminf(fmaxf(r, 0.0f), 1.0f); g = fminf(fmaxf(g, 0.0f), 1.0f); b = fminf(fmaxf(b, 0.0f), 1.0f);
		out[i] = make_float4(sqrtf(r), sqrtf(g), sqrtf(b), 1.0f);  // clamp, gamma 2, alpha 1   :209-214
	}
}

// ------------------------------------------------------------------------------------------------
// adaptive select step (DESIGN.md §5c): which pixels the next round of rtb_render_adaptive renders
//   adaptive_error   e_p = one standard error of the pixel's mean in display space (clamp, then sqrt, as resolve does)
//   adaptive_count   window maximum W_p of e over the 3x3 neighbourhood + candidate test, active pixels per block
//   adaptive_scan    exclusive prefix sums of the block counts, and the total
//   adaptive_write   every active pixel to its slot of the list: ascending pixel order, so camera rays stay coherent
// The rule is evaluated in binary32 in the order DESIGN.md writes it (-fmad=false: nothing is contracted), so
// tests/adaptive_rule.py reproduces every decision.  Maxima and minima propagate NaN.

__device__ __forceinline__ float nan_max(float a, float b) { return a != a ? a : (b != b ? b : fmaxf(a, b)); }
__device__ __forceinline__ float nan_min(float a, float b) { return a != a ? a : (b != b ? b : fminf(a, b)); }

__device__ __forceinline__ float display_error(float S, float Q, float n) {
	const float m = S / n;
	const float v = nan_max((Q - S * m) / (n - 1.0f), 0.0f);
	const float s = sqrtf(v / n);
	const float hi = sqrtf(nan_min(nan_max(m + s, 0.0f), 1.0f)), lo = sqrtf(nan_min(nan_max(m - s, 0.0f), 1.0f));
	return (hi - lo) * 0.5f;
}

__global__ void __launch_bounds__(STREAM_THREADS)
adaptive_error_kernel(AdaptiveView av) {
	const uint32_t n = av.width * av.n_rows, first = av.row_begin * av.width;
	const uint32_t stride = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
		const float4 a = av.accum[first + i], q = av.accum2[first + i];
		const float er = display_error(a.x, q.x, a.w), eg = display_error(a.y, q.y, a.w), eb = display_error(a.z, q.z, a.w);
		av.err[first + i] = nan_max(nan_max(er, eg), eb);
	}
}

#define SELECT_THREADS 1024   // pixels per block of the select step (one per thread)

// Whether pixel first + i takes part in the next round; `no_sq` = it holds the cursor's samples but no sums of squares, so
// the rule cannot be evaluated for it (checked before the window: without sums of squares every error reads as 0).
__device__ __forceinline__ bool adaptive_active(const AdaptiveView& av, uint32_t i, bool& no_sq) {
	no_sq = false;
	if (i >= av.width * av.n_rows) return false;
	const uint32_t first = av.row_begin * av.width;
	const float4 a = av.accum[first + i];
	if (!(a.w == (float)av.cursor)) return false;                 // missed a round: never comes back
	no_sq = !(av.accum2[first + i].w == a.w);
	if (no_sq || av.cursor >= av.max_spp) return false;
	if (av.cursor >= av.min_spp) {
		const int y = (int)(i / av.width), x = (int)(i - (uint32_t)y * av.width);
		const int y0 = max(y - 1, 0), y1 = min(y + 1, (int)av.n_rows - 1), x0 = max(x - 1, 0), x1 = min(x + 1, (int)av.width - 1);
		float w = 0.0f;
		for (int yy = y0; yy <= y1; ++yy)
			for (int xx = x0; xx <= x1; ++xx) {
				const float e = av.err[first + (uint32_t)yy * av.width + (uint32_t)xx];
				w = fmaxf(w, e != e ? INFINITY : e);
			}
		if (w <= av.tolerance) return false;
	}
	return true;
}

__global__ void __launch_bounds__(SELECT_THREADS)
adaptive_count_kernel(AdaptiveView av) {
	__shared__ uint32_t s_count;
	if (threadIdx.x == 0) s_count = 0u;
	__syncthreads();
	bool no_sq;
	const bool active = adaptive_active(av, blockIdx.x * SELECT_THREADS + threadIdx.x, no_sq);
	if (no_sq) atomicOr(av.result + 1, 1u);
	const uint32_t mask = __ballot_sync(FULL_MASK, active);
	if ((threadIdx.x & 31) == 0 && mask) atomicAdd(&s_count, (uint32_t)__popc(mask));
	__syncthreads();
	if (threadIdx.x == 0) av.block_count[blockIdx.x] = s_count;
}

// One block: exclusive prefix sums of the block counts in place, in chunks of SELECT_THREADS, and the total.
__global__ void __launch_bounds__(SELECT_THREADS)
adaptive_scan_kernel(AdaptiveView av, uint32_t n_blocks) {
	__shared__ uint32_t s_part[SELECT_THREADS];
	uint32_t carry = 0;
	for (uint32_t base = 0; base < n_blocks; base += SELECT_THREADS) {
		const uint32_t b = base + threadIdx.x;
		const uint32_t c = b < n_blocks ? av.block_count[b] : 0u;
		s_part[threadIdx.x] = c;
		__syncthreads();
		for (uint32_t off = 1; off < SELECT_THREADS; off <<= 1) {
			const uint32_t v = threadIdx.x >= off ? s_part[threadIdx.x - off] : 0u;
			__syncthreads();
			s_part[threadIdx.x] += v;
			__syncthreads();
		}
		if (b < n_blocks) av.block_count[b] = carry + s_part[threadIdx.x] - c;
		carry += s_part[SELECT_THREADS - 1];
		__syncthreads();
	}
	if (threadIdx.x == 0) av.result[0] = carry;
}

__global__ void __launch_bounds__(SELECT_THREADS)
adaptive_write_kernel(AdaptiveView av) {
	__shared__ uint32_t s_warp[SELECT_THREADS / 32];
	const uint32_t i = blockIdx.x * SELECT_THREADS + threadIdx.x;
	bool no_sq;
	const bool active = adaptive_active(av, i, no_sq);
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t mask = __ballot_sync(FULL_MASK, active);
	if (lane == 0) s_warp[warp] = __popc(mask);
	__syncthreads();
	if (threadIdx.x == 0) {
		uint32_t tot = 0;
		for (int w = 0; w < SELECT_THREADS / 32; ++w) { const uint32_t c = s_warp[w]; s_warp[w] = tot; tot += c; }
	}
	__syncthreads();
	if (active) {
		const uint32_t pos = av.block_count[blockIdx.x] + s_warp[warp] + __popc(mask & ((1u << lane) - 1u));
		RTB_CHECK(pos < av.width * av.n_rows, RTB_BOUNDS_PATH);
		av.list[pos] = av.row_begin * av.width + i;
	}
}

// Output stage of FirstApp::write_renderbuffer (FirstApp.cpp:108-122) on the device: mean -> clamp -> sqrt (as resolve),
// uint8 = value * 255.999f, RGB, optionally with the rows flipped (the float buffer's row 0 is the bottom of the picture).
__global__ void __launch_bounds__(STREAM_THREADS)
quantize_kernel(const float4* __restrict__ accum, uint8_t* __restrict__ rgb, uint32_t width, uint32_t height, int flip_rows) {
	const uint32_t n = width * height, stride = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
		const uint32_t y = i / width, x = i - y * width;
		const float4 a = accum[(size_t)(flip_rows ? height - 1 - y : y) * width + x];
		const float inv = 1.0f / a.w;
		const float r = sqrtf(fminf(fmaxf(a.x * inv, 0.0f), 1.0f)), g = sqrtf(fminf(fmaxf(a.y * inv, 0.0f), 1.0f)), b = sqrtf(fminf(fmaxf(a.z * inv, 0.0f), 1.0f));
		rgb[3 * (size_t)i] = (uint8_t)(r * 255.999f); rgb[3 * (size_t)i + 1] = (uint8_t)(g * 255.999f); rgb[3 * (size_t)i + 2] = (uint8_t)(b * 255.999f);
	}
}

// ------------------------------------------------------------------------------------------------
// hit-record parity hook

template <int STACK>
__global__ void __launch_bounds__(TRAVERSE_THREADS)
trace_rays_kernel(SceneView sv, const float4* __restrict__ ro, const float4* __restrict__ rd, uint32_t n,
                  int2* __restrict__ hit, int2* __restrict__ stats, uint32_t* counter) {
	__shared__ int s_stack[STACK * TRAVERSE_THREADS];
	const int lane = threadIdx.x & 31;
	for (;;) {
		uint32_t base = 0;
		if (lane == 0) base = atomicAdd(counter, 32u);
		base = __shfl_sync(FULL_MASK, base, 0);
		if (base >= n) break;
		uint32_t i = base + lane;
		if (i < n) {
			float4 fo = ro[i], fd = rd[i];
			MediumRng mr = make_medium_rng(BatchParams{}, 0, 0, 0);
			float t; int code;
			int st[2];
			trace_ray<0, true>(sv, xyz(fo), xyz(fd), fo.w, mr, s_stack + threadIdx.x, STACK, t, code, st);
			hit[i] = make_int2(__float_as_int(t), code);
			stats[i] = make_int2(st[0], st[1]);
		}
		__syncwarp();
	}
}

__global__ void __launch_bounds__(STREAM_THREADS)
hit_record_kernel(SceneView sv, const float4* __restrict__ ro, const float4* __restrict__ rd, const int2* __restrict__ hit,
                  const int2* __restrict__ stats, uint32_t n, rtb_hit* __restrict__ out) {
	const uint32_t stride = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
		rtb_hit r;
		const int2 h = hit[i];
		r.t = __int_as_float(h.x);
		r.nodes_visited = stats[i].x; r.prims_tested = stats[i].y; r.pad = 0;   // inner nodes visited, primitives tested
		if (h.y < 0) {
			r.t = FLT_MAX; r.prim = -1; r.object = -1; r.material = -1; r.front_face = 0; r.u = r.v = 0.0f;
			r.p[0] = r.p[1] = r.p[2] = 0.0f; r.n[0] = r.n[1] = r.n[2] = 0.0f;
		} else {
			const float4 fo = ro[i], fd = rd[i];
			const int2 info = __ldg(sv.prim_info + (h.y >> RTB_LEAF_TYPE_BITS));
			Surface s;
			if (sv.tri_attr) reconstruct<true>(sv, h.y, xyz(fo), xyz(fd), fo.w, r.t, true, s);
			else reconstruct<false>(sv, h.y, xyz(fo), xyz(fd), fo.w, r.t, true, s);
			r.prim = h.y >> RTB_LEAF_TYPE_BITS; r.object = info.y; r.material = info.x;
			r.p[0] = s.p.x; r.p[1] = s.p.y; r.p[2] = s.p.z;
			r.n[0] = s.n_shade.x; r.n[1] = s.n_shade.y; r.n[2] = s.n_shade.z;
			r.front_face = rt::dot(xyz(fd), s.n_geom) > 0.0f ? 0 : 1;
			r.u = s.u; r.v = s.v;
		}
		out[i] = r;
	}
}

// ------------------------------------------------------------------------------------------------
// host launch wrappers

int debug_bounds_report(unsigned long long* violations, unsigned long long* checks) {
#if RTB_DEBUG_BOUNDS
	if (cudaMemcpyFromSymbol(violations, g_bounds_violations, sizeof(unsigned long long) * RTB_BOUNDS_CLASSES) != cudaSuccess) return -1;
	if (cudaMemcpyFromSymbol(checks, g_bounds_checks, sizeof(unsigned long long)) != cudaSuccess) return -1;
	return 1;
#else
	(void)violations; (void)checks;
	return 0;
#endif
}

void query_occupancy(int device, LaunchCfg& lc) {
	cudaDeviceProp prop{};
	cudaGetDeviceProperties(&prop, device);
	int sms = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
	int occ_t = 0, occ_tm = 0, occ_s = 0, occ_g = 0;
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_t, traverse_kernel<0, STACK_SIZE, false>, TRAVERSE_THREADS, 0);
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_tm, traverse_kernel<2, STACK_SIZE, false>, TRAVERSE_THREADS, 0);
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_s, shade_kernel_for(0), SHADE_THREADS, 0);   // shade_kernel<0>
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_g, generate_kernel<false>, STREAM_THREADS, 0);
	int occ_trav = occ_t < occ_tm ? occ_t : occ_tm;
	int occ_l = 0, occ_lm = 0;
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_l, tail_kernel_for<false, false>(0), TRAVERSE_THREADS, 0);   // tail_kernel<false, STACK_SIZE, 0>
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_lm, tail_kernel_for<true, false>(0), TRAVERSE_THREADS, 0);
	int occ_tail = occ_l < occ_lm ? occ_l : occ_lm;
	lc.blocks_tail = sms * (occ_tail > 0 ? occ_tail : 1);
	lc.sms = sms;
	lc.blocks_traverse = sms * (occ_trav > 0 ? occ_trav : 1);
	lc.blocks_shade = sms * (occ_s > 0 ? occ_s : 1);
	lc.blocks_stream = sms * (occ_g > 0 ? occ_g : 1);
	int occ_b = 0;
	cudaFuncSetAttribute(bin_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BIN_COUNT_SMEM);
	cudaFuncSetAttribute(bin_permute_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BIN_PERMUTE_SMEM);
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_b, bin_permute_kernel, BIN_THREADS, BIN_PERMUTE_SMEM);
	lc.blocks_bin = sms * (occ_b > 0 ? occ_b : 1);
}

void launch_generate(const BatchParams& bp, const rtb_camera& cam, const WaveView& wv, const LaunchCfg& lc, cudaStream_t st) {
	if (bp.pixel_list()) generate_kernel<true><<<lc.blocks_stream, STREAM_THREADS, 0, st>>>(bp, cam, wv);
	else generate_kernel<false><<<lc.blocks_stream, STREAM_THREADS, 0, st>>>(bp, cam, wv);
}
void launch_traverse(const SceneView& sv, const BatchParams& bp, const WaveView& wv, uint32_t bounce, int q, const LaunchCfg& lc, cudaStream_t st) {
	// media need the per-path RNG inside traversal; scenes without media skip that code entirely
	// a walk keeps at most depth - 1 entries on its stack: 16 entries for shallow trees, 32 normally, 64 for the deep
	// trees a linear BVH over a large mesh can be (the flattener never hands over more than RTB_TREE_DEPTH_MAX levels)
	const bool small = sv.tree_depth <= 17, deep = sv.tree_depth > STACK_SIZE - 2;
	// (adaptive rounds: only the walks with media derive a pixel, so only they have list-mode instantiations)
#define RTB_LAUNCH_TRAVERSE(M, L) \
	do { if (small) traverse_kernel<M, 16, L><<<lc.blocks_traverse, TRAVERSE_THREADS, 0, st>>>(sv, bp, wv, bounce, q); \
	     else if (deep) traverse_kernel<M, DEEP_STACK_SIZE, L><<<lc.blocks_traverse, TRAVERSE_THREADS, 0, st>>>(sv, bp, wv, bounce, q); \
	     else traverse_kernel<M, STACK_SIZE, L><<<lc.blocks_traverse, TRAVERSE_THREADS, 0, st>>>(sv, bp, wv, bounce, q); } while (0)
	if (sv.has_media == 0) RTB_LAUNCH_TRAVERSE(0, false);
	else if (sv.has_media == 1) { if (bp.pixel_list()) RTB_LAUNCH_TRAVERSE(1, true); else RTB_LAUNCH_TRAVERSE(1, false); }
	else { if (bp.pixel_list()) RTB_LAUNCH_TRAVERSE(2, true); else RTB_LAUNCH_TRAVERSE(2, false); }
#undef RTB_LAUNCH_TRAVERSE
}
// The feature word of a launch: the scene's bits, staged with the scene, and F_LIST for an adaptive round.
static uint32_t feature_word(const SceneView& sv, const BatchParams& bp) {
	return ((uint32_t)sv.launch_flags & (F_WORDS - 1)) | (bp.pixel_list() ? F_LIST : 0u);
}
void launch_tail(const SceneView& sv, const BatchParams& bp, const WaveView& wv, uint32_t bounce, int q, uint32_t threshold, const LaunchCfg& lc, cudaStream_t st) {
	const bool deep = sv.tree_depth > STACK_SIZE - 2;
	const uint32_t f = feature_word(sv, bp);
	const TailKernel k = sv.has_media ? (deep ? tail_kernel_for<true, true>(f) : tail_kernel_for<true, false>(f))
	                                  : (deep ? tail_kernel_for<false, true>(f) : tail_kernel_for<false, false>(f));
	k<<<lc.blocks_tail, TRAVERSE_THREADS, 0, st>>>(sv, bp, wv, bounce, q, threshold);
}
void launch_shade(const SceneView& sv, const BatchParams& bp, const WaveView& wv, uint32_t bounce, int q, const LaunchCfg& lc, cudaStream_t st) {
	shade_kernel_for(feature_word(sv, bp))<<<lc.blocks_shade, SHADE_THREADS, 0, st>>>(sv, bp, wv, bounce, q);
}
void launch_texture(const SceneView& sv, const WaveView& wv, uint32_t bounce, int q_out, const LaunchCfg& lc, cudaStream_t st) {
	const int blocks = lc.sms * 2 < lc.blocks_stream ? lc.sms * 2 : lc.blocks_stream;   // short work lists: a small grid keeps the launch cheap
	texture_kernel<<<blocks, STREAM_THREADS, 0, st>>>(sv, wv, bounce, q_out);
}
void launch_bin_rays(const SceneView& sv, const WaveView& wv, uint32_t bounce, int q_from, const LaunchCfg& lc, cudaStream_t st) {
	const uint32_t nbins = 1u << (3 * sv.bin_org_bits + 2 * sv.bin_dir_bits);
	bin_count_kernel<<<lc.blocks_bin, BIN_THREADS, BIN_COUNT_SMEM, st>>>(sv, wv, bounce, q_from);
	bin_scan_kernel<<<(nbins + BIN_SCAN_PER_BLOCK - 1) / BIN_SCAN_PER_BLOCK, BIN_SCAN_THREADS, 0, st>>>(wv, bounce);
	bin_permute_kernel<<<lc.blocks_bin, BIN_THREADS, BIN_PERMUTE_SMEM, st>>>(sv, wv, bounce, q_from);
}
void launch_accumulate(const BatchParams& bp, const WaveView& wv, float4* accum, float4* accum2, const LaunchCfg& lc, cudaStream_t st) {
	if (bp.pixel_list()) accumulate_kernel<true><<<lc.blocks_stream, STREAM_THREADS, 0, st>>>(bp, wv, accum, accum2);
	else accumulate_kernel<false><<<lc.blocks_stream, STREAM_THREADS, 0, st>>>(bp, wv, accum, accum2);
	end_batch_kernel<<<1, 32, 0, st>>>(bp, wv);
}
uint32_t adaptive_select_blocks(uint32_t n_pixels) { return (n_pixels + SELECT_THREADS - 1) / SELECT_THREADS; }
void launch_adaptive_select(const AdaptiveView& av, const LaunchCfg& lc, cudaStream_t st) {
	const uint32_t n = av.width * av.n_rows, nb = adaptive_select_blocks(n);
	if (av.cursor >= av.min_spp) {   // (before min_spp every candidate is active whatever its error)
		int blocks = (int)((n + STREAM_THREADS - 1) / STREAM_THREADS); if (blocks > lc.blocks_stream) blocks = lc.blocks_stream; if (blocks < 1) blocks = 1;
		adaptive_error_kernel<<<blocks, STREAM_THREADS, 0, st>>>(av);
	}
	adaptive_count_kernel<<<nb, SELECT_THREADS, 0, st>>>(av);
	adaptive_scan_kernel<<<1, SELECT_THREADS, 0, st>>>(av, nb);
	adaptive_write_kernel<<<nb, SELECT_THREADS, 0, st>>>(av);
}
void launch_resolve(const float4* accum, float4* out, uint32_t n, cudaStream_t st) {
	int blocks = (int)((n + STREAM_THREADS - 1) / STREAM_THREADS); if (blocks > 148 * 8) blocks = 148 * 8; if (blocks < 1) blocks = 1;
	resolve_kernel<<<blocks, STREAM_THREADS, 0, st>>>(accum, out, n);
}
void launch_quantize(const float4* accum, uint8_t* rgb, uint32_t width, uint32_t height, int flip_rows, cudaStream_t st) {
	const uint32_t n = width * height;
	int blocks = (int)((n + STREAM_THREADS - 1) / STREAM_THREADS); if (blocks > 148 * 8) blocks = 148 * 8; if (blocks < 1) blocks = 1;
	quantize_kernel<<<blocks, STREAM_THREADS, 0, st>>>(accum, rgb, width, height, flip_rows);
}
void launch_trace_rays(const SceneView& sv, const float4* ray_o, const float4* ray_d, uint32_t n, int2* hit_tmp, int2* stats_tmp,
                       rtb_hit* hits_out, uint32_t* work_counter, const LaunchCfg& lc, cudaStream_t st) {
	cudaMemsetAsync(work_counter, 0, sizeof(uint32_t), st);
	if (sv.tree_depth > STACK_SIZE - 2) trace_rays_kernel<DEEP_STACK_SIZE><<<lc.blocks_traverse, TRAVERSE_THREADS, 0, st>>>(sv, ray_o, ray_d, n, hit_tmp, stats_tmp, work_counter);
	else trace_rays_kernel<STACK_SIZE><<<lc.blocks_traverse, TRAVERSE_THREADS, 0, st>>>(sv, ray_o, ray_d, n, hit_tmp, stats_tmp, work_counter);
	hit_record_kernel<<<lc.blocks_stream, STREAM_THREADS, 0, st>>>(sv, ray_o, ray_d, hit_tmp, stats_tmp, n, hits_out);
}

}  // namespace rtb
