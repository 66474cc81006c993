// rtb_device.h — device code shared by the kernel objects: helpers, traversal, surfaces, textures, the environment map,
// light sampling, materials, and the shade and tail kernel templates.  rtb_kernels.cu holds the other kernels and every
// launcher; rtb_shade.cu and rtb_tail.cu instantiate shade_kernel and tail_kernel, one object per (MEDIA, stack) for the
// tail, so that the instantiations compile in parallel.
#ifndef RTB_DEVICE_H
#define RTB_DEVICE_H

#include "rtb_kernels.h"

#include <cfloat>

#include "../../include/rtb_scene_format.h"
#include "rtb_types.h"
#include "rtmath.h"

namespace rtb {

using rt::v3;

#ifndef TRAVERSE_THREADS
#define TRAVERSE_THREADS 128
#endif
#ifndef SHADE_THREADS
#define SHADE_THREADS 128   // (B200, r2: 64 / 96 / 128 / 256 / 512 threads: shade 9.8 / 10.3 / 10.1 / 10.6 / 11.3 ms per batch, step 36.6-37.0 / 37.1 / 36.7 / 37.0 / 37.6:
#endif                      //  smaller blocks wait less at the compaction barriers, but interleave the survivors more finely for the next traverse)
#define STREAM_THREADS 256
#define DEEP_STACK_SIZE 64
#ifndef STACK_SIZE
#define STACK_SIZE 32
#endif
#define FULL_MASK 0xFFFFFFFFu

// ------------------------------------------------------------------------------------------------
// -DRTB_DEBUG_BOUNDS=1 (librtb200_debug.so): every index the kernels form from scene or queue data is checked against
// the size of what it indexes, and violations are counted per class instead of trapping (compute-sanitizer is not
// available on the pool this was developed on).  rtb_debug_bounds_report returns the counters; the release build
// compiles the checks away.
#ifndef RTB_DEBUG_BOUNDS
#define RTB_DEBUG_BOUNDS 0
#endif
#if RTB_DEBUG_BOUNDS
// One set of counters for the whole library, defined in rtb_kernels.cu: every object of the debug build is compiled with
// -rdc=true, so that they all count into it (whole-program objects would each get a copy of their own).
#ifndef __CUDACC_RDC__
#error "RTB_DEBUG_BOUNDS=1 needs -rdc=true"
#endif
extern __device__ unsigned long long g_bounds_violations[RTB_BOUNDS_CLASSES];
extern __device__ unsigned long long g_bounds_checks;
#define RTB_CHECK(ok, cls) do { if (!(ok)) atomicAdd(&g_bounds_violations[cls], 1ull); } while (0)
#define RTB_COUNT_CHECKS(n) atomicAdd(&g_bounds_checks, (unsigned long long)(n))
#else
#define RTB_CHECK(ok, cls) do { } while (0)
#define RTB_COUNT_CHECKS(n) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------
// small device helpers

__device__ __forceinline__ v3 xyz(const float4& f) { return rt::mk(f.x, f.y, f.z); }

__device__ __forceinline__ float4 ldg4(const float4* p) { return __ldg(p); }
// Two consecutive float4 (32 bytes, 32-byte aligned).  sm_100 has 256-bit global loads (LDG.E.256): with
// -DRTB_LDG256=1 a 64-byte node is two requests instead of four.  Measured neutral on B200 (traverse 30.1 vs 29.9 ms
// per step, profiles/r1_experiments.md), so the default stays with 128-bit loads.
#ifndef RTB_LDG256
#define RTB_LDG256 0
#endif
__device__ __forceinline__ void ldg8(const float4* p, float4& a, float4& b) {
#if RTB_LDG256
	asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
	    : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p));
#else
	a = __ldg(p); b = __ldg(p + 1);
#endif
}

// Wavefront queue records are touched once per kernel.  -DRTB_STREAM_HINTS=1 marks those accesses streaming (evict-first,
// ld/st.global.cs) to keep them from pushing BVH nodes and primitive records out of L1 / L2.  Measured on B200 (round 2):
// traverse 28.4 vs 28.5 ms per step, shade 11.9 vs 11.4 ms - the queues are not what evicts the tree, and shade's stores
// do better write-back cached.  Off by default.
#ifndef RTB_STREAM_HINTS
#define RTB_STREAM_HINTS 0
#endif
#if RTB_STREAM_HINTS
__device__ __forceinline__ float4 ldq(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ int2 ldq(const int2* p) { return __ldcs(p); }
__device__ __forceinline__ void stq(float4* p, float4 v) { __stcs(p, v); }
__device__ __forceinline__ void stq(int2* p, int2 v) { __stcs(p, v); }
#else
__device__ __forceinline__ float4 ldq(const float4* p) { return *p; }
__device__ __forceinline__ int2 ldq(const int2* p) { return *p; }
__device__ __forceinline__ void stq(float4* p, float4 v) { *p = v; }
__device__ __forceinline__ void stq(int2* p, int2 v) { *p = v; }
#endif

// A ray record is 32 bytes, 32-byte aligned: one 256-bit access (LDG / STG.E.256 of sm_100) moves it, so a warp reading or
// writing 32 consecutive records touches 1 KB exactly once (two 128-bit accesses at a 32-byte stride ask L1 for every
// sector twice: shade measured 9 % slower that way).
__device__ __forceinline__ void ld_ray(const float4* rec, float4& o, float4& d) {
	asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
	             : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w), "=f"(d.x), "=f"(d.y), "=f"(d.z), "=f"(d.w) : "l"(rec));
}
__device__ __forceinline__ void st_ray(float4* rec, const float4& o, const float4& d) {
	asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
	             :: "l"(rec), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w), "f"(d.x), "f"(d.y), "f"(d.z), "f"(d.w) : "memory");
}

// What changes from one rtb_render call to the next - the sample range and the seed - is read from device memory, so
// that the CUDA graph of a batch (whose kernel arguments are frozen at capture) serves every call on the same image size.
__device__ __forceinline__ BatchParams with_call_params(const BatchParams& in, const WaveView& wv) {
	BatchParams bp = in;
	bp.sample_begin = wv.call_params[0]; bp.sample_end = wv.call_params[1]; bp.seed = wv.call_params[2];
	return bp;
}

// Local pixel -> global pixel of an adaptive round: entry pl of the list, which holds pixels of the row range
// [first, first + count) and is at most `count` long.
__device__ __forceinline__ uint32_t listed_pixel(const uint32_t* list, uint32_t pl, uint32_t first, uint32_t count) {
	RTB_CHECK(pl < count, RTB_BOUNDS_PATH);
	const uint32_t p = __ldg(list + pl);
	RTB_CHECK(p - first < count, RTB_BOUNDS_PATH);
	return p;
}

// Path id -> (global pixel index, absolute sample index).  Paths of a batch are laid out
// sample-major: id = local_sample * npix + local_pixel, local pixels row-major from row_begin
// (LIST: local pixel pl is bp.pixel_list[pl]).
template <bool LIST = false>
__device__ __forceinline__ void path_pixel_sample(const BatchParams& bp, uint32_t batch, uint32_t path,
                                                  uint32_t& pixel, uint32_t& sample) {
	uint32_t sl = path / bp.npix;
	uint32_t pl = path - sl * bp.npix;
	pixel = LIST ? listed_pixel(bp.pixel_list(), pl, bp.row_begin * bp.width, bp.n_rows * bp.width) : bp.row_begin * bp.width + pl;
	sample = bp.sample_begin + batch * bp.samples_per_batch + sl;
}

__device__ __forceinline__ uint32_t batch_sample_count(const BatchParams& bp, uint32_t batch) {
	uint64_t s0 = (uint64_t)bp.sample_begin + (uint64_t)batch * bp.samples_per_batch;
	if (s0 >= bp.sample_end) return 0;
	uint64_t left = bp.sample_end - s0;
	return (uint32_t)(left < bp.samples_per_batch ? left : bp.samples_per_batch);
}

// ------------------------------------------------------------------------------------------------
// primitive tests (shared by traverse and the hit-record hook)

// _sphere_closest_intersection  SphereHittable.cuh:15-33 (a = d.d hoisted per ray)
__device__ __forceinline__ float sphere_closest(v3 o, v3 d, float a, v3 c, float r) {
	v3 oc = rt::sub(o, c);
	float hb = rt::dot(d, oc);
	float cc = fmaf(-r, r, rt::dot(oc, oc));
	float disc = fmaf(hb, hb, -(a * cc));
	if (!(disc > 0.0f)) return FLT_MAX;
	float sq = sqrtf(disc);
	float t = (-hb - sq) / a;
	if (t < 0.0f) {
		t = (-hb + sq) / a;
		if (t < 0.0f) return FLT_MAX;
	}
	return t;
}

// Book quad::hit / triangle with the reference's t policy (t >= 0, strictly closer than the best).
__device__ __forceinline__ float planar_hit(v3 o, v3 d, const float4* pp, float4 q0, bool tri, float tbest) {
	float4 q1 = ldg4(pp + 1), q2, q3;
	ldg8(pp + 2, q2, q3);
	v3 N = rt::mk(q1.w, q2.w, q3.w);
	float denom = rt::dot(N, d);
	if (fabsf(denom) < 1e-8f) return FLT_MAX;
	float t = (q0.w - rt::dot(N, o)) / denom;
	if (!(t >= 0.0f) || !(t < tbest)) return FLT_MAX;
	v3 P = rt::madd(d, t, o);
	v3 planar = rt::sub(P, xyz(q0));
	v3 w = xyz(q3);
	float alpha = rt::dot(w, rt::cross(planar, xyz(q2)));
	float beta = rt::dot(w, rt::cross(xyz(q1), planar));
	if (tri) { if (alpha < 0.0f || beta < 0.0f || alpha + beta > 1.0f) return FLT_MAX; }
	else { if (alpha < 0.0f || alpha > 1.0f || beta < 0.0f || beta > 1.0f) return FLT_MAX; }
	return t;
}

// A book box() is six quads.  One BVH leaf holds a (min, max) record followed by the six ordinary quad records; a slab
// test on (min, max) only SELECTS which faces the ray can meet (the entry faces, then the exit faces, with a tolerance
// far above the rounding of either computation, in list order), and the hit itself is the exact quad test on those
// records - so the result is the one testing all six quads gives, and it is reported on the quad (`face_code`).
//   rec_stride = float4s from one record to the next (4, or 8 when every record is followed by its transform).
__device__ __forceinline__ float box_hit(v3 o, v3 d, float idx, float idy, float idz, float oix, float oiy, float oiz,
                                         const float4* pp, float4 q0, int rec_stride, float tbest, int& face) {
	const float4 q1 = ldg4(pp + 1);                         // q0 = (min.xyz, max.x), q1 = (max.y, max.z, -, -)
	const float ax = fmaf(q0.x, idx, oix), bx = fmaf(q0.w, idx, oix);
	const float ay = fmaf(q0.y, idy, oiy), by = fmaf(q1.x, idy, oiy);
	const float az = fmaf(q0.z, idz, oiz), bz = fmaf(q1.y, idz, oiz);
	const float t0x = fminf(ax, bx), t1x = fmaxf(ax, bx), t0y = fminf(ay, by), t1y = fmaxf(ay, by), t0z = fminf(az, bz), t1z = fmaxf(az, bz);
	const float tenter = fmaxf(fmaxf(t0x, t0y), t0z), texit = fminf(fminf(t1x, t1y), t1z);
	const float scale = fmaxf(fmaxf(fmaxf(fabsf(oix), fabsf(oiy)), fabsf(oiz)), fmaxf(fabsf(tenter), fabsf(texit)));
	const float tol = 2e-5f * scale;
	face = -1;
	if (tenter > texit + tol || texit < -tol || tenter - tol >= tbest) return FLT_MAX;
	// faces in list order: 0 front (z max), 1 right (x max), 2 back (z min), 3 left (x min), 4 top (y max), 5 bottom (y min)
	const int nfx = ax <= bx ? 3 : 1, nfy = ay <= by ? 5 : 4, nfz = az <= bz ? 2 : 0;
	unsigned entry = 0, exits = 0;
	if (t0x >= tenter - tol) entry |= 1u << nfx;
	if (t0y >= tenter - tol) entry |= 1u << nfy;
	if (t0z >= tenter - tol) entry |= 1u << nfz;
	if (t1x <= texit + tol) exits |= 1u << (4 - nfx);       // the opposite face: 3 <-> 1
	if (t1y <= texit + tol) exits |= 1u << (9 - nfy);       // 5 <-> 4
	if (t1z <= texit + tol) exits |= 1u << (2 - nfz);       // 2 <-> 0
	unsigned mask = tenter >= -tol ? entry : 0u;
	if (texit - tenter <= tol) mask |= exits;                // paper-thin along the ray: the order of entry and exit is not reliable
	float best = FLT_MAX;
	for (int pass = 0; pass < 2; ++pass) {
		for (unsigned m = mask; m; m &= m - 1) {
			const int f = __ffs(m) - 1;
			const float4* fp = pp + rec_stride * (1 + f);
			const float t = planar_hit(o, d, fp, ldg4(fp), false, fminf(tbest, best));
			if (t < best) { best = t; face = f; }
		}
		if (best < FLT_MAX) break;
		mask = exits & ~mask;
	}
	return best;
}

// Free-flight uniforms of the media a ray meets.  Medium m of a path segment uses component (m & 3)
// of Philox(seed, pixel; sample, bounce, STREAM_MEDIUM0 + (m >> 2)); the block is generated lazily,
// only when some medium's boundary interval survives the geometric rejections, and shared by up to
// four media.  LIST: the batch is an adaptive round, and the pixel is gathered from its list - lazily too.
template <bool LIST> struct MediumRngList {};
template <> struct MediumRngList<true> { const uint32_t* list; uint32_t range; };   // the pixel list; pixels of the row range
template <bool LIST>
struct MediumRngT : MediumRngList<LIST> {
	uint32_t seed, path, bounce;
	uint32_t npix, pixel0, sample0;   // batch layout (warp-uniform): the path's pixel and sample are only worked out
	                                  // (an integer division) when a block of uniforms is actually drawn
	uint32_t block;    // cached block index, 0xFFFFFFFF = none
	rt::f4 u;
	__device__ __forceinline__ float get(uint32_t m) {
		const uint32_t b = m >> 2;
		if (b != block) {
			const uint32_t sl = path / npix, pl = path - sl * npix;      // path_pixel_sample
			uint32_t pixel;
			if constexpr (LIST) pixel = listed_pixel(this->list, pl, pixel0, this->range);
			else pixel = pixel0 + pl;
			u = rt::rng4(seed, pixel, sample0 + sl, bounce, rt::STREAM_MEDIUM0 + b); block = b;
		}
		const uint32_t c = m & 3u;
		return c == 0 ? u.x : (c == 1 ? u.y : (c == 2 ? u.z : u.w));
	}
};
using MediumRng = MediumRngT<false>;
template <bool LIST = false>
__device__ __forceinline__ MediumRngT<LIST> make_medium_rng(const BatchParams& bp, uint32_t batch, uint32_t path, uint32_t bounce) {
	MediumRngT<LIST> r; r.seed = bp.seed; r.path = path; r.bounce = bounce; r.block = 0xFFFFFFFFu;
	r.npix = bp.npix; r.pixel0 = bp.row_begin * bp.width; r.sample0 = bp.sample_begin + batch * bp.samples_per_batch;
	if constexpr (LIST) { r.list = bp.pixel_list(); r.range = bp.n_rows * bp.width; }
	r.u.x = r.u.y = r.u.z = r.u.w = 0.0f; return r;
}

// constant_medium::hit (book) over a convex boundary interval [t1,t2] found for any-sign t.
template <class MR>
__device__ __forceinline__ float medium_sample(float t1, float t2, float a, float neg_inv_density, MR& mr, uint32_t medium, float tbest) {
	if (!(t2 > t1 + 0.0001f)) return FLT_MAX;     // second boundary query: interval(t1 + 0.0001, inf)
	if (t1 < 0.0f) t1 = 0.0f;                     // ray_t.min (the reference accepts t >= 0)
	if (t2 > tbest) t2 = tbest;                   // ray_t.max = closest so far
	if (t1 >= t2) return FLT_MAX;
	float len = sqrtf(a);
	float dist_inside = (t2 - t1) * len;
	float hit_distance = neg_inv_density * rt::logpos(mr.get(medium));
	if (hit_distance > dist_inside) return FLT_MAX;
	return t1 + hit_distance / len;
}

template <class MR>
__device__ __forceinline__ float medium_sphere_hit(v3 o, v3 d, float a, float4 q0, float nid, MR& mr, uint32_t medium, float tbest) {
	v3 oc = rt::sub(o, xyz(q0));
	float hb = rt::dot(d, oc);
	float cc = fmaf(-q0.w, q0.w, rt::dot(oc, oc));
	float disc = fmaf(hb, hb, -(a * cc));
	if (!(disc > 0.0f)) return FLT_MAX;
	float sq = sqrtf(disc);
	return medium_sample((-hb - sq) / a, (-hb + sq) / a, a, nid, mr, medium, tbest);
}

template <class MR>
__device__ __forceinline__ float medium_box_hit(v3 o, v3 d, float a, float4 q0, float4 q1, float4 q2, MR& mr, uint32_t medium, float tbest) {
	// world -> object: translate back, rotate by -theta about y (book translate::hit / rotate_y::hit)
	float cs = q0.w, sn = q1.w;
	v3 ot = rt::sub(o, xyz(q2));
	v3 oo = rt::mk(fmaf(cs, ot.x, -(sn * ot.z)), ot.y, fmaf(sn, ot.x, cs * ot.z));
	v3 dd = rt::mk(fmaf(cs, d.x, -(sn * d.z)), d.y, fmaf(sn, d.x, cs * d.z));
	float tn = -FLT_MAX, tf = FLT_MAX;
	const float bmin[3] = {q0.x, q0.y, q0.z}, bmax[3] = {q1.x, q1.y, q1.z};
	const float oc[3] = {oo.x, oo.y, oo.z}, dc[3] = {dd.x, dd.y, dd.z};
#pragma unroll
	for (int k = 0; k < 3; ++k) {
		if (dc[k] == 0.0f) { if (oc[k] < bmin[k] || oc[k] > bmax[k]) return FLT_MAX; continue; }
		float ta = (bmin[k] - oc[k]) / dc[k], tb = (bmax[k] - oc[k]) / dc[k];
		float lo = ta < tb ? ta : tb, hi = ta < tb ? tb : ta;
		tn = lo > tn ? lo : tn; tf = hi < tf ? hi : tf;
	}
	if (!(tn < tf)) return FLT_MAX;
	return medium_sample(tn, tf, a, q2.w, mr, medium, tbest);
}

// Instances.  T = (cos, sin, off.x, off.y), (off.z, -, -, -) with world = R_y(theta) * object + off.
__device__ __forceinline__ int xf_offset(int base) { return base == PRIM_SPHERE ? 1 : (base == PRIM_MOVING_SPHERE ? 2 : 4); }   // quads, triangles, boxes: the next record

// world ray -> object ray: origin - offset (book translate::hit), then rotate by -theta (book rotate_y::hit)
__device__ __forceinline__ void xf_ray(const float4* tp, v3 o, v3 d, v3& oo, v3& dd) {
	const float4 t0 = ldg4(tp), t1 = ldg4(tp + 1);
	const float cs = t0.x, sn = t0.y;
	const v3 ot = rt::sub(o, rt::mk(t0.z, t0.w, t1.x));
	if (t1.y == 0.0f) { oo = ot; dd = d; return; }   // translate only: the book's translate::hit leaves the direction alone (signed zeros included)
	oo = rt::mk(fmaf(cs, ot.x, -(sn * ot.z)), ot.y, fmaf(sn, ot.x, cs * ot.z));
	dd = rt::mk(fmaf(cs, d.x, -(sn * d.z)), d.y, fmaf(sn, d.x, cs * d.z));
}
// object vector -> world (book rotate_y::hit, normal back-rotation)
__device__ __forceinline__ v3 xf_vec_to_world(const float4* tp, v3 v) {
	const float4 t0 = ldg4(tp);
	const float cs = t0.x, sn = t0.y;
	if (ldg4(tp + 1).y == 0.0f) return v;   // translate only
	return rt::mk(fmaf(cs, v.x, sn * v.z), v.y, fmaf(-sn, v.x, cs * v.z));
}

// ------------------------------------------------------------------------------------------------
// traverse


// One primitive against one ray: the t of the hit if it is closer than tbest, else FLT_MAX.
// `hit_code` is what a hit is reported on: the leaf itself, or for a box the quad record of the face that was hit.
// (idx.. oiz: the ray's slab-test reciprocals, used to pick the faces of a box.)
struct RaySlab { float idx, idy, idz, oix, oiy, oiz; };

// Per-ray reciprocal of the slab tests.  A component that is (nearly) zero is nudged to +-1e-20 with the sign of the
// component - signed zeros included, and every later sign decision is taken from the nudged value - so 0 * inf never appears.
__device__ __forceinline__ float slab_dir(float d) { return fabsf(d) < 1e-20f ? copysignf(1e-20f, d) : d; }

#ifndef RTB_UNIFIED_LEAF
#define RTB_UNIFIED_LEAF 1
#endif
template <bool MEDIA, class MR>
__device__ __forceinline__ float leaf_test(const SceneView& sv, int code, v3 o, v3 d, float a, float time, MR& mr, float tbest,
                                           const RaySlab& rs, int& hit_code) {
	hit_code = code;
	const int type = code & 15;
	RTB_CHECK(code >= 0 && (code >> RTB_LEAF_TYPE_BITS) < sv.n_prims, RTB_BOUNDS_PRIM);
	const float4* pp = sv.prims + 4 * (size_t)(code >> RTB_LEAF_TYPE_BITS);
	const float4 q0 = ldg4(pp);
	float t = FLT_MAX;
#if RTB_UNIFIED_LEAF
	// The lanes of a warp meet different flavours of the same shape (sphere / moving sphere / instanced sphere; box /
	// instanced box): the instance transform and the moving centre are short predicated preludes, and the long part -
	// the quadratic, the face tests - is ONE code path per shape that all those lanes run together.
	const int base = type & 7;
	if (MEDIA && (type == PRIM_MEDIUM_SPHERE || type == PRIM_MEDIUM_BOX)) {
		const float4 q1 = ldg4(pp + 1);
		if (type == PRIM_MEDIUM_SPHERE) return medium_sphere_hit(o, d, a, q0, q1.x, mr, __float_as_uint(q1.y), tbest);
		const float4 q2 = ldg4(pp + 2), q3 = ldg4(pp + 3);
		return medium_box_hit(o, d, a, q0, q1, q2, mr, __float_as_uint(q3.x), tbest);
	}
	const bool xf = (type & PRIM_XF) != 0;
	v3 oo = o, dd = d; float a2 = a;
	if (xf) {   // instance: take the ray into the primitive's frame (book translate::hit, rotate_y::hit)
		xf_ray(pp + xf_offset(base), o, d, oo, dd);
		a2 = rt::dot(dd, dd);
	}
	if (base <= PRIM_MOVING_SPHERE) {
		v3 c = xyz(q0);
		if (base == PRIM_MOVING_SPHERE) c = rt::mix(c, xyz(ldg4(pp + 1)), time);   // center = mix(center0, center1, ray.time)   SphereHittable.cu:92
		t = sphere_closest(oo, dd, a2, c, q0.w);
	} else if (base == PRIM_BOX) {
		// the box in its own frame; when instanced, every record (the box's and each face's) is followed by the transform
		RaySlab bs = rs;
		if (xf) {
			bs.idx = __frcp_rn(slab_dir(dd.x)); bs.idy = __frcp_rn(slab_dir(dd.y)); bs.idz = __frcp_rn(slab_dir(dd.z));
			bs.oix = -(oo.x * bs.idx); bs.oiy = -(oo.y * bs.idy); bs.oiz = -(oo.z * bs.idz);
		}
		const int stride = xf ? 8 : 4;
		int face;
		t = box_hit(oo, dd, bs.idx, bs.idy, bs.idz, bs.oix, bs.oiy, bs.oiz, pp, q0, stride, tbest, face);
		if (face >= 0) hit_code = (((code >> RTB_LEAF_TYPE_BITS) + (stride >> 2) * (1 + face)) << RTB_LEAF_TYPE_BITS) | PRIM_QUAD | (type & PRIM_XF);
	} else {
		t = planar_hit(oo, dd, pp, q0, base == PRIM_TRIANGLE, tbest);
	}
#else
	if (type == PRIM_SPHERE) {
		t = sphere_closest(o, d, a, xyz(q0), q0.w);
	} else if (type == PRIM_MOVING_SPHERE) {
		// center = mix(center0, center1, ray.time)   SphereHittable.cu:92
		const float4 q1 = ldg4(pp + 1);
		t = sphere_closest(o, d, a, rt::mix(xyz(q0), xyz(q1), time), q0.w);
	} else if (type == PRIM_QUAD || type == PRIM_TRIANGLE) {
		t = planar_hit(o, d, pp, q0, type == PRIM_TRIANGLE, tbest);
	} else if (type == PRIM_BOX) {
		int face;
		t = box_hit(o, d, rs.idx, rs.idy, rs.idz, rs.oix, rs.oiy, rs.oiz, pp, q0, 4, tbest, face);
		if (face >= 0) hit_code = (((code >> RTB_LEAF_TYPE_BITS) + 1 + face) << RTB_LEAF_TYPE_BITS) | PRIM_QUAD;
	} else if (type & PRIM_XF) {
		// instance: take the ray into the primitive's frame (book translate::hit, rotate_y::hit)
		const int base = type & 7;
		v3 oo, dd;
		xf_ray(pp + xf_offset(base), o, d, oo, dd);
		const float a2 = rt::dot(dd, dd);
		if (base == PRIM_SPHERE) t = sphere_closest(oo, dd, a2, xyz(q0), q0.w);
		else if (base == PRIM_MOVING_SPHERE) t = sphere_closest(oo, dd, a2, rt::mix(xyz(q0), xyz(ldg4(pp + 1)), time), q0.w);
		else if (base == PRIM_BOX) {
			// the box in its own frame; every record (the box's and each face's) is followed by the transform
			const float jx = __frcp_rn(slab_dir(dd.x)), jy = __frcp_rn(slab_dir(dd.y)), jz = __frcp_rn(slab_dir(dd.z));
			int face;
			t = box_hit(oo, dd, jx, jy, jz, -(oo.x * jx), -(oo.y * jy), -(oo.z * jz), pp, q0, 8, tbest, face);
			if (face >= 0) hit_code = (((code >> RTB_LEAF_TYPE_BITS) + 2 * (1 + face)) << RTB_LEAF_TYPE_BITS) | PRIM_QUAD | PRIM_XF;
		}
		else t = planar_hit(oo, dd, pp, q0, base == PRIM_TRIANGLE, tbest);
	} else if (MEDIA) {
		const float4 q1 = ldg4(pp + 1);
		if (type == PRIM_MEDIUM_SPHERE) {
			t = medium_sphere_hit(o, d, a, q0, q1.x, mr, __float_as_uint(q1.y), tbest);
		} else {
			const float4 q2 = ldg4(pp + 2), q3 = ldg4(pp + 3);
			t = medium_box_hit(o, d, a, q0, q1, q2, mr, __float_as_uint(q3.x), tbest);
		}
	}
#endif
	return t;
}

#ifndef TRAV_WHILE_WHILE
#define TRAV_WHILE_WHILE 1
#endif
#ifndef RTB_ROBUST_SLAB
#define RTB_ROBUST_SLAB 1
#endif
#ifndef RTB_REG_STACK
#define RTB_REG_STACK 0
#endif
#define TRAV_END ((int)0x80000000)

// MEDIA: 0 = the scene has no media; 1 = all of them are in the pre-test list (the walk itself never meets
// one: no RNG state is carried through the loop); 2 = more than the list holds, the rest are BVH leaves.
template <int MEDIA, bool STATS = false, class MR>
__device__ __forceinline__ void trace_ray(const SceneView& sv, v3 o, v3 d, float time, MR& mr,
                                          int* __restrict__ stack, int stack_cap, float& tbest_out, int& code_out, int* stats_out = nullptr) {
	const float a = rt::dot(d, d);
	float tbest = FLT_MAX;
	int best = -1;
	if (MEDIA) {   // media first: a scatter inside a medium bounds the BVH walk tightly
		for (int k = 0; k < sv.n_pre; ++k) {
			const int code = __ldg(sv.pre_list + k);
			int hit_code;
			const float t = leaf_test<true>(sv, code, o, d, a, time, mr, tbest, RaySlab{}, hit_code);   // (media only: no slab data needed)
			if (t < tbest) { tbest = t; best = hit_code; }
		}
		if (sv.bvh_empty) { tbest_out = tbest; code_out = best; return; }
	}
	// Slab test with a per-ray reciprocal (slab_dir: zero components, signed zeros included, are nudged).
	const float gx = slab_dir(d.x), gy = slab_dir(d.y), gz = slab_dir(d.z);
	const float idx = __frcp_rn(gx), idy = __frcp_rn(gy), idz = __frcp_rn(gz);
	const float oix = -(o.x * idx), oiy = -(o.y * idy), oiz = -(o.z * idz);
	// Near / far slab planes are picked by the direction signs with FMAs instead of min/max pairs:
	// t(min plane) = min * (1/d) - o/d, and the max plane adds ext * (1/d) on the side the sign says.
	// (ncu: the min/max version kept the ALU pipe 66 % busy with the FMA pipe at 20 %.)
	// The sign is that of the value the reciprocal was taken of, so a -0.0 component picks the planes its -1e20 reciprocal needs.
	const float nx = gx < 0.0f ? idx : 0.0f, fx = gx < 0.0f ? 0.0f : idx;
	const float ny = gy < 0.0f ? idy : 0.0f, fy = gy < 0.0f ? 0.0f : idy;
	const float nz = gz < 0.0f ? idz : 0.0f, fz = gz < 0.0f ? 0.0f : idz;
#if RTB_ROBUST_SLAB
	// The cull must never lose a box the exact primitive test would hit (aabb::intersects computes (min - o) / d, which
	// cancels exactly; plane * (1/d) - o/d does not): the rounding of o/d is up to 2^-24 |o/d| per plane, the reciprocal and
	// the two fused multiply-adds add a few 2^-24 of t.  The far distance is widened by both bounds before it is compared -
	// one FMA per box; a box thinner than the rounding (a 1e-4 quad seen from 10,000 units) is then always entered.
	const float slab_abs = 2.4e-7f * fmaxf(fmaxf(fabsf(oix), fabsf(oiy)), fabsf(oiz));   // 2 x 2^-23 max |o/d|
	const float slab_rel = 1.0f + 9.6e-7f;                                                // 1 + 8 x 2^-23
#endif

#if RTB_NODE_PAIRED
	const float2 id_xy = make_float2(idx, idy), oi_xy = make_float2(oix, oiy), n_xy = make_float2(nx, ny), f_xy = make_float2(fx, fy);
	const float2 id_zz = make_float2(idz, idz), oi_zz = make_float2(oiz, oiz), n_zz = make_float2(nz, nz), f_zz = make_float2(fz, fz);
#endif
	int cur = sv.root_ref;
	int sp = 0;
	// -DRTB_REG_STACK=1 (experiment): the two youngest stack entries live in registers and only older ones spill to shared
	// memory - the "short stack in registers" of the brief.  Measured on B200 (round 2): see profiles/r2_experiments.md.
#if RTB_REG_STACK
	int top0 = 0, top1 = 0;   // top0 = youngest
#define STACK_PUSH(v) do { if (sp >= 2) stack[(sp - 2) * TRAVERSE_THREADS] = top1; top1 = top0; top0 = (v); ++sp; } while (0)
#define STACK_POP(dst) do { dst = top0; top0 = top1; --sp; if (sp >= 2) top1 = stack[(sp - 2) * TRAVERSE_THREADS]; } while (0)
#else
#define STACK_PUSH(v) do { stack[sp * TRAVERSE_THREADS] = (v); ++sp; } while (0)
#define STACK_POP(dst) do { --sp; dst = stack[sp * TRAVERSE_THREADS]; } while (0)
#endif
	int n_inner = 0, n_leaf = 0;   // STATS only
	// "while-while" walk: lanes first descend inner nodes together, then test their leaf primitive
	// together (a leaf reference is negative; TRAV_END marks an exhausted walk).
	for (;;) {
		while (cur >= 0) {
			if (STATS) ++n_inner;
			RTB_CHECK(cur < sv.n_nodes, RTB_BOUNDS_NODE);
			const float4* np = sv.nodes + 4 * (size_t)cur;
			float4 n0, n1, n2, n3f;
			ldg8(np, n0, n1); ldg8(np + 2, n2, n3f);
			const int2 n3 = make_int2(__float_as_int(n3f.x), __float_as_int(n3f.y));
#if RTB_NODE_PAIRED
			// the same 18 fused multiply-adds, two per instruction (FFMA2): x and y of one child share an instruction,
			// z of the two children share one; every component is an IEEE fma, so the results are the bits of the scalar form
			const float2 l_xy = __ffma2_rn(make_float2(n0.x, n0.y), id_xy, oi_xy);
			const float2 r_xy = __ffma2_rn(make_float2(n1.x, n1.y), id_xy, oi_xy);
			const float2 lr_z = __ffma2_rn(make_float2(n2.x, n2.y), id_zz, oi_zz);
			const float2 ln_xy = __ffma2_rn(make_float2(n0.z, n0.w), n_xy, l_xy), lf_xy = __ffma2_rn(make_float2(n0.z, n0.w), f_xy, l_xy);
			const float2 rn_xy = __ffma2_rn(make_float2(n1.z, n1.w), n_xy, r_xy), rf_xy = __ffma2_rn(make_float2(n1.z, n1.w), f_xy, r_xy);
			const float2 lrn_z = __ffma2_rn(make_float2(n2.z, n2.w), n_zz, lr_z), lrf_z = __ffma2_rn(make_float2(n2.z, n2.w), f_zz, lr_z);
			const float ltmin = fmaxf(fmaxf(ln_xy.x, ln_xy.y), lrn_z.x);
			const float ltmax = fminf(fminf(lf_xy.x, lf_xy.y), lrf_z.x);
			const float rtmin = fmaxf(fmaxf(rn_xy.x, rn_xy.y), lrn_z.y);
			const float rtmax = fminf(fminf(rf_xy.x, rf_xy.y), lrf_z.y);
#else
			const float lx = fmaf(n0.x, idx, oix), ly = fmaf(n0.y, idy, oiy), lz = fmaf(n0.z, idz, oiz);
			const float rx = fmaf(n1.z, idx, oix), ry = fmaf(n1.w, idy, oiy), rz = fmaf(n2.x, idz, oiz);
			const float ltmin = fmaxf(fmaxf(fmaf(n0.w, nx, lx), fmaf(n1.x, ny, ly)), fmaf(n1.y, nz, lz));
			const float ltmax = fminf(fminf(fmaf(n0.w, fx, lx), fmaf(n1.x, fy, ly)), fmaf(n1.y, fz, lz));
			const float rtmin = fmaxf(fmaxf(fmaf(n2.y, nx, rx), fmaf(n2.z, ny, ry)), fmaf(n2.w, nz, rz));
			const float rtmax = fminf(fminf(fmaf(n2.y, fx, rx), fmaf(n2.z, fy, ry)), fmaf(n2.w, fz, rz));
#endif
			// aabb::intersects: tmin <= tmax && tmin < ray_max && tmax > 0   aabb.cuh:41
#if RTB_ROBUST_SLAB
#if RTB_NODE_PAIRED
			const float2 tmax_c = __ffma2_rn(make_float2(ltmax, rtmax), make_float2(slab_rel, slab_rel), make_float2(slab_abs, slab_abs));
			const float ltmax_c = tmax_c.x, rtmax_c = tmax_c.y;
#else
			const float ltmax_c = fmaf(ltmax, slab_rel, slab_abs), rtmax_c = fmaf(rtmax, slab_rel, slab_abs);
#endif
			const bool hl = ltmin <= ltmax_c && ltmin < tbest && ltmax_c > 0.0f;
			const bool hr = rtmin <= rtmax_c && rtmin < tbest && rtmax_c > 0.0f;
#else
			const bool hl = ltmin <= ltmax && ltmin < tbest && ltmax > 0.0f;
			const bool hr = rtmin <= rtmax && rtmin < tbest && rtmax > 0.0f;
#endif
			if (hl && hr) {
				// nearer child next, farther child on the stack (BVH.cu:91-97); boxes that both contain
				// the origin are ordered by where the ray leaves them
				const float lk = fmaxf(ltmin, 0.0f), rk = fmaxf(rtmin, 0.0f);
				const bool sw = lk > rk || (lk == rk && ltmax > rtmax);
				RTB_CHECK(sp >= 0 && sp < stack_cap, RTB_BOUNDS_STACK);
				STACK_PUSH(sw ? n3.x : n3.y);
				cur = sw ? n3.y : n3.x;
			} else if (hl) cur = n3.x;
			else if (hr) cur = n3.y;
			else if (sp > 0) { STACK_POP(cur); }
			else cur = TRAV_END;

#if !TRAV_WHILE_WHILE
			break;   // if-if flavour: at most one inner node per trip
#endif
		}
		if (cur == TRAV_END) break;
		if (cur < 0) {
			if (STATS) ++n_leaf;
			const int code = ~cur;
			int hit_code;
			const float t = leaf_test<(MEDIA == 2)>(sv, code, o, d, a, time, mr, tbest, RaySlab{idx, idy, idz, oix, oiy, oiz}, hit_code);
			if (t < tbest) { tbest = t; best = hit_code; }   // "if (t >= rec.distance) return false"  SphereHittable.cu:58
			if (sp == 0) break;
			STACK_POP(cur);
		}
	}
	if (STATS) { stats_out[0] = n_inner; stats_out[1] = n_leaf; }
	tbest_out = tbest; code_out = best;
#undef STACK_PUSH
#undef STACK_POP
}

// ------------------------------------------------------------------------------------------------
// surface reconstruction + textures + materials

// n_diel (ATTR only): the normal the dielectric refracts about - the shading normal on the geometric normal's side
// (DESIGN.md §5e); the geometric normal itself everywhere else.
struct Surface { v3 p, n_shade, n_geom, n_diel; float u, v; };

// What Sphere::getNormal / MovingSphere::getNormal hand to materials: the outward normal
// (p - c) / r, never flipped (SphereHittable.cu:43-50,64,100).  Quads face the ray (book).
// ATTR: the scene has triangle attributes; a triangle that carries them is shaded with its interpolated normal and reads its
// interpolated UVs (DESIGN.md §5e), in its own frame, before the instance transform.
template <bool ATTR>
__device__ __forceinline__ void reconstruct(const SceneView& sv, int code, v3 o, v3 d, float time, float t, bool want_uv, Surface& s) {
	const int type = code & 15, base = type & 7;
	const bool xf = (type & PRIM_XF) != 0;
	RTB_CHECK(code >= 0 && (code >> RTB_LEAF_TYPE_BITS) + (xf && base >= PRIM_QUAD ? 1 : 0) < sv.n_prims, RTB_BOUNDS_PRIM);
	const float4* pp = sv.prims + 4 * (size_t)(code >> RTB_LEAF_TYPE_BITS);
	const float4 q0 = ldg4(pp);
	s.p = rt::madd(d, t, o);          // Material::Scatter uses in_ray.at(rec.distance): the world ray
	s.u = 0.0f; s.v = 0.0f;
	if (type == PRIM_MEDIUM_SPHERE || type == PRIM_MEDIUM_BOX) {   // normal arbitrary (book constant_medium::hit)
		s.n_geom = rt::mk(1.0f, 0.0f, 0.0f);
		s.n_shade = s.n_geom;
		if (ATTR) s.n_diel = s.n_geom;
		return;
	}
	v3 oo = o, dd = d;                // the ray in the primitive's own frame
	const float4* tp = pp + xf_offset(base);
	if (xf) xf_ray(tp, o, d, oo, dd);
	if (base == PRIM_SPHERE || base == PRIM_MOVING_SPHERE) {
		v3 c = xyz(q0);
		if (base == PRIM_MOVING_SPHERE) c = rt::mix(c, xyz(ldg4(pp + 1)), time);
		v3 n = rt::divs(rt::sub(rt::madd(dd, t, oo), c), q0.w);   // (ray.at(t) - center) / radius   SphereHittable.cu:64,100
		if (want_uv) {   // book sphere::get_sphere_uv on the outward normal in the sphere's own frame
			float theta = acosf(-n.y);
			float phi = atan2f(-n.z, n.x) + 3.14159265358979323846f;
			s.u = phi / 6.28318530717958647692f;
			s.v = theta / 3.14159265358979323846f;
		}
		if (xf) n = xf_vec_to_world(tp, n);
		s.n_geom = n; s.n_shade = n;
		if (ATTR) s.n_diel = n;
	} else {
		const float4 q1 = ldg4(pp + 1), q2 = ldg4(pp + 2), q3 = ldg4(pp + 3);
		v3 N = rt::mk(q1.w, q2.w, q3.w);
		v3 ns = rt::dot(dd, N) > 0.0f ? rt::neg(N) : N;             // book set_face_normal
		v3 m = N;
		int ai = -1;
		if (ATTR && base == PRIM_TRIANGLE) {
			ai = __ldg(sv.attr_slot + (code >> RTB_LEAF_TYPE_BITS));
			RTB_CHECK(ai >= -1 && ai < sv.n_tri_attr, RTB_BOUNDS_PRIM);
		}
		if (ATTR && ai >= 0) {
			// (alpha, beta) always: the normal needs them.  x interpolates as fma(x2, beta, fma(x1, alpha, x0 * w)).
			const v3 planar = rt::sub(rt::madd(dd, t, oo), xyz(q0));
			const float alpha = rt::dot(xyz(q3), rt::cross(planar, xyz(q2)));
			const float beta = rt::dot(xyz(q3), rt::cross(xyz(q1), planar));
			const float w = (1.0f - alpha) - beta;
			const float4* ap = sv.tri_attr + 4 * (size_t)ai;
			const float4 a0 = ldg4(ap), a1 = ldg4(ap + 1), a2 = ldg4(ap + 2), a3 = ldg4(ap + 3);
			const uint32_t flags = __float_as_uint(a3.w);
			if (flags & RTBS_ATTR_NORMALS) {
				m = rt::mk(fmaf(a2.x, beta, fmaf(a1.x, alpha, a0.x * w)), fmaf(a2.y, beta, fmaf(a1.y, alpha, a0.y * w)),
				           fmaf(a2.z, beta, fmaf(a1.z, alpha, a0.z * w)));
				m = rt::dot(m, m) > 0.0f ? rt::normalize(m) : N;
				if (rt::dot(m, N) < 0.0f) m = rt::neg(m);                  // on the face normal's side
				ns = rt::dot(dd, N) > 0.0f ? rt::neg(m) : m;               // set_face_normal with m in place of N
			}
			if (flags & RTBS_ATTR_UVS) {
				s.u = fmaf(a3.y, beta, fmaf(a2.w, alpha, a0.w * w));
				s.v = fmaf(a3.z, beta, fmaf(a3.x, alpha, a1.w * w));
			} else {
				s.u = alpha; s.v = beta;
			}
		} else if (want_uv) {
			v3 planar = rt::sub(rt::madd(dd, t, oo), xyz(q0));
			s.u = rt::dot(xyz(q3), rt::cross(planar, xyz(q2)));
			s.v = rt::dot(xyz(q3), rt::cross(xyz(q1), planar));
		}
		if (xf) { N = xf_vec_to_world(tp, N); ns = xf_vec_to_world(tp, ns); if (ATTR) m = xf_vec_to_world(tp, m); }
		s.n_geom = N; s.n_shade = ns;
		if (ATTR) s.n_diel = m;
	}
}

__device__ __forceinline__ float sin_any(float x) {
	float r = x * 0.15915494309189535f;
	r = r - floorf(r);
	float s, c; rt::sincos2pi(r, s, c);
	return s;
}

// Book perlin::noise with Hermite-smoothed trilinear interpolation of gradient dot products.  (This and texture_value are
// not inline: static, so that every object including this header has its own copy, as under -rdc=true it must.)
static __device__ float perlin_noise(const float* __restrict__ grad, const int* __restrict__ perm, v3 p) {
	float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
	float u = p.x - fx, v = p.y - fy, w = p.z - fz;
	int i = (int)fx, j = (int)fy, k = (int)fz;
	float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
	float accum = 0.0f;
#pragma unroll
	for (int di = 0; di < 2; ++di)
#pragma unroll
		for (int dj = 0; dj < 2; ++dj)
#pragma unroll
			for (int dk = 0; dk < 2; ++dk) {
				int g = perm[(i + di) & 255] ^ perm[256 + ((j + dj) & 255)] ^ perm[512 + ((k + dk) & 255)];
				v3 c = rt::mk(grad[3 * g], grad[3 * g + 1], grad[3 * g + 2]);
				v3 wv = rt::mk(u - (float)di, v - (float)dj, w - (float)dk);
				float wi = di ? uu : 1.0f - uu, wj = dj ? vv : 1.0f - vv, wk = dk ? ww : 1.0f - ww;
				accum = fmaf(wi * wj * wk, rt::dot(c, wv), accum);
			}
	return accum;
}

static __device__ v3 texture_value(const SceneView& sv, int tex, float u, float v, v3 p) {
	for (int guard = 0; guard < 16; ++guard) {
		RTB_CHECK(tex >= 0 && tex < sv.n_textures, RTB_BOUNDS_TEXTURE);
		const float4 t0 = ldg4(sv.textures + 3 * tex);
		const int kind = __float_as_int(t0.x);
		if (kind == RTB_TEX_SOLID) { return xyz(ldg4(sv.textures + 3 * tex + 1)); }
		if (kind == RTB_TEX_CHECKER) {
			// checker_texture::value  cu_Textures.cuh:32-39: C cast (truncation) and C '%'
			float inv = t0.w;
			int sum = (int)(p.x * inv) + (int)(p.y * inv) + (int)(p.z * inv);
			tex = (sum % 2 == 0) ? __float_as_int(t0.y) : __float_as_int(t0.z);
			continue;
		}
		const float4 t2 = ldg4(sv.textures + 3 * tex + 2);
		const int w = __float_as_int(t2.x), h = __float_as_int(t2.y);
		const uint32_t off = __float_as_uint(t2.z);
		if (kind == RTB_TEX_IMAGE) {   // book image_texture::value (nearest texel, bytes / 255)
			float uc = fminf(fmaxf(u, 0.0f), 1.0f), vc = 1.0f - fminf(fmaxf(v, 0.0f), 1.0f);
			int i = (int)(uc * (float)w), j = (int)(vc * (float)h);
			i = i < w - 1 ? i : w - 1; j = j < h - 1 ? j : h - 1;
			RTB_CHECK(i >= 0 && j >= 0 && off + 3 * ((size_t)j * w + i) + 2 < sv.n_blob, RTB_BOUNDS_TEXTURE);
			const uint8_t* px = sv.blob + off + 3 * ((size_t)j * w + i);
			const float sc = 1.0f / 255.0f;
			return rt::mk(sc * (float)px[0], sc * (float)px[1], sc * (float)px[2]);
		}
		// RTB_TEX_NOISE: book noise_texture::value = 0.5 * (1 + sin(scale * p.z + 10 * turb(p, 7)))
		const float* grad = reinterpret_cast<const float*>(sv.blob + off);
		const int* perm = reinterpret_cast<const int*>(sv.blob + off + 256 * 3 * 4);
		float accum = 0.0f, weight = 1.0f; v3 tp = p;
		for (int k = 0; k < 7; ++k) {
			accum = fmaf(weight, perlin_noise(grad, perm, tp), accum);
			weight *= 0.5f; tp = rt::mul(tp, 2.0f);
		}
		float turb = fabsf(accum);
		float val = 0.5f * (1.0f + sin_any(fmaf(t0.w, p.z, 10.0f * turb)));
		return rt::mk(val, val, val);
	}
	return rt::mk(0.0f, 0.0f, 0.0f);
}

__device__ __forceinline__ bool texture_needs_uv(const SceneView& sv, int tex) {
	if (tex < 0) return false;
	const int kind = __float_as_int(ldg4(sv.textures + 3 * tex).x);
	return kind != RTB_TEX_SOLID && kind != RTB_TEX_NOISE;   // checker children may be images
}

// ------------------------------------------------------------------------------------------------
// environment map (DESIGN.md §5d): nearest-texel lookup of a miss direction, the pdf per solid angle of the map's own
// sampling, and a direction drawn from it

// Texel of direction d: the unit vector as the sky gradient computes it, the sphere (u, v) of sphere textures, then
// nearest-texel indexing as image textures index (row 0 = top); sin_theta of the unit vector for the pdf.
__device__ __forceinline__ const float4* env_texel(const SceneView& sv, v3 d, float& sin_theta) {
	const float inv = 1.0f / sqrtf(rt::dot(d, d));
	const v3 n = rt::mk(d.x * inv, d.y * inv, d.z * inv);
	const float theta = acosf(-n.y);
	const float phi = atan2f(-n.z, n.x) + 3.14159265358979323846f;
	const float u = phi / 6.28318530717958647692f, v = theta / 3.14159265358979323846f;
	const int W = sv.env_width, H = sv.env_height;
	int i = (int)(u * (float)W), j = (int)((1.0f - v) * (float)H);
	i = i < W - 1 ? i : W - 1; j = j < H - 1 ? j : H - 1;
	RTB_CHECK(i >= 0 && j >= 0 && i < W && j < H, RTB_BOUNDS_TEXTURE);
	sin_theta = sqrtf(fmaf(n.x, n.x, n.z * n.z));
	return sv.env + (size_t)j * W + i;
}
__device__ __forceinline__ v3 env_radiance(const SceneView& sv, v3 d) {
	float st;
	return xyz(ldg4(env_texel(sv, d, st)));
}
// pdf numerator p_ij W H / (2 pi^2) over sin theta; 0 at the poles
__device__ __forceinline__ float env_pdf(const SceneView& sv, v3 u) {
	float st;
	const float num = ldg4(env_texel(sv, u, st)).w;
	return st > 0.0f ? num / st : 0.0f;
}
// Continuous inversion of a CDF of n + 1 entries (c[0] = 0, c[n] = 1) at x: the index k with c[k] <= x < c[k + 1] and the
// fraction of x inside [c[k], c[k + 1]).  x is clamped below 1 first (uniform01 can round to 1).
__device__ __forceinline__ int cdf_invert(const float* __restrict__ c, int n, float x, float& frac) {
	x = fminf(x, 0.99999994f);
	int lo = 0, hi = n;
	while (hi - lo > 1) {
		const int mid = (lo + hi) >> 1;
		if (__ldg(c + mid) <= x) lo = mid; else hi = mid;
	}
	RTB_CHECK(lo >= 0 && lo < n, RTB_BOUNDS_TEXTURE);
	const float c0 = __ldg(c + lo), c1 = __ldg(c + lo + 1);
	frac = (x - c0) / (c1 - c0);
	return lo;
}
// A direction drawn from the map's own sampling with the uniforms (zr row, zc column)
__device__ __forceinline__ v3 env_direction(const SceneView& sv, float zr, float zc) {
	const int W = sv.env_width, H = sv.env_height;
	const float* cm = reinterpret_cast<const float*>(sv.env + (size_t)W * H);
	float fr, fc;
	const int j = cdf_invert(cm, H, zr, fr);
	const int i = cdf_invert(cm + (H + 1) + (size_t)j * (W + 1), W, zc, fc);
	const float v = 1.0f - ((float)j + fr) / (float)H;
	const float u = ((float)i + fc) / (float)W;
	float st, ct, sp, cp;
	rt::sincos2pi(0.5f * v, st, ct);
	rt::sincos2pi(u, sp, cp);
	return rt::mk(-(st * cp), -ct, st * sp);
}

// ------------------------------------------------------------------------------------------------
// light sampling: the half-and-half mixture of the material's own directions and directions towards the sampled lights
// (DESIGN.md §5b, "Ray Tracing: The Rest of Your Life")

struct LightKey { uint32_t seed, pixel, sample, bounce; };   // what the STREAM_LIGHT block of a scatter is drawn from

// pdf (per solid angle) of light i's own sampling for the direction u (unit) from p
__device__ __forceinline__ float light_pdf(const SceneView& sv, int i, v3 p, v3 u) {
	const float4* lp = sv.lights + 4 * i;
	const float4 q0 = ldg4(lp);
	const float4 info = ldg4(sv.lights + 4 * sv.n_lights + i);
	if (__float_as_int(info.x) == PRIM_QUAD) {
		const float t = planar_hit(p, u, lp, q0, false, FLT_MAX);
		if (!(t > 0.0f) || !(t < FLT_MAX)) return 0.0f;
		const v3 N = rt::mk(ldg4(lp + 1).w, ldg4(lp + 2).w, ldg4(lp + 3).w);
		return (t * t) / (fabsf(rt::dot(u, N)) * info.y);
	}
	const v3 e = rt::sub(xyz(q0), p);
	const float d2 = rt::dot(e, e), R2 = q0.w * q0.w;
	if (!(d2 > R2)) return 0.0f;                                     // inside or on the light: it cannot be sampled
	if (!(sphere_closest(p, u, rt::dot(u, u), xyz(q0), q0.w) < FLT_MAX)) return 0.0f;
	return rt::cone_pdf(rt::cone_cos_max(d2, R2));
}

// Direction and weight (scattering pdf / mixture pdf) of a Lambertian (ISO = false) or isotropic scatter; false: the
// path ends black.  ENV: a sampled environment map is strategy n (of n + 1), its pdf the last term of the sum.
template <bool ISO, bool ENV>
__device__ __forceinline__ bool light_mix(const SceneView& sv, const Surface& s, const rt::f4& r, const LightKey& lk, v3& dir, float& w) {
	const rt::f4 l = rt::rng4(lk.seed, lk.pixel, lk.sample, lk.bounce, rt::STREAM_LIGHT);
	const int n = sv.n_lights;
	const bool env = ENV && sv.env_sample;
	const int m = env ? n + 1 : n;                                   // strategies
	if (l.x < 0.5f) {                                                // towards a point on light k, or the map (k = n)
		int k = (int)(l.y * (float)m); k = k < m - 1 ? k : m - 1;
		if (env && k == n) {
			dir = env_direction(sv, l.z, l.w);
		} else {
			RTB_CHECK(k >= 0 && k < sv.n_lights, RTB_BOUNDS_PRIM);
			const float4* lp = sv.lights + 4 * k;
			const float4 q0 = ldg4(lp);
			if (__float_as_int(ldg4(sv.lights + 4 * n + k).x) == PRIM_QUAD) {
				const v3 e = rt::sub(rt::madd(xyz(ldg4(lp + 2)), l.w, rt::madd(xyz(ldg4(lp + 1)), l.z, xyz(q0))), s.p);
				if (!(rt::dot(e, e) > 0.0f)) return false;
				dir = rt::normalize(e);
			} else {
				const v3 e = rt::sub(xyz(q0), s.p);
				const float d2 = rt::dot(e, e), R2 = q0.w * q0.w;
				if (!(d2 > R2)) return false;
				dir = rt::cone_direction(e, rt::cone_cos_max(d2, R2), l.z, l.w);
			}
		}
	} else if (ISO) {
		dir = rt::unit_sphere(r.x, r.y);
	} else {
		dir = rt::add(s.n_shade, rt::unit_sphere(r.x, r.y));
		if (rt::near_zero(dir, 1e-9f)) return false;
	}
	const v3 u = rt::normalize(dir);
	const float spdf = ISO ? RT_INV_4PI : fmaxf(0.0f, rt::dot(s.n_shade, u)) * RT_INV_PI;
	if (!(spdf > 0.0f)) return false;
	float sum = 0.0f;
	for (int i = 0; i < n; ++i) sum += light_pdf(sv, i, s.p, u);
	if (env) sum += env_pdf(sv, u);
	w = rt::mixture_weight(spdf, sum / (float)m);
	return w > 0.0f;
}

// ------------------------------------------------------------------------------------------------
// GGX microfacet materials (DESIGN.md §5f): visible-normal sampling (Dupuy & Benyoub 2023, spherical caps), weight G2 / G1
// of the height-correlated Smith term; no pdf is evaluated and the light mixture is not involved.

// Smith Lambda of a local direction for the GGX width a2 = alpha^2
__device__ __forceinline__ float ggx_lambda(v3 w, float a2) {
	const float t = fmaf(w.y, w.y, w.x * w.x) / (w.z * w.z);
	return (sqrtf(fmaf(a2, t, 1.0f)) - 1.0f) * 0.5f;
}

// Rough metal (DIEL = false: F0 = albedo, frame normal n_shade) or rough dielectric (DIEL: the dielectric's normal, which
// the caller passes as n with its ior ratio).  0 = the path ends black, 1 = scattered.
template <bool DIEL>
__device__ __forceinline__ int rough_scatter(v3 n, v3 d, const rt::f4& r, float alpha, float ratio, v3 albedo, v3& dir, v3& att) {
	// frame (U, V, W = n) as rt::cone_direction builds it; wo local
	const v3 ud = rt::normalize(d);
	const v3 wo_w = rt::neg(ud);
	const v3 A = fabsf(n.x) > 0.9f ? rt::mk(0.0f, 1.0f, 0.0f) : rt::mk(1.0f, 0.0f, 0.0f);
	const v3 V = rt::normalize(rt::cross(n, A));
	const v3 U = rt::cross(n, V);
	const v3 wo = rt::mk(rt::dot(wo_w, U), rt::dot(wo_w, V), rt::dot(wo_w, n));
	if (!(wo.z > 0.0f)) return 0;
	// visible normal: spherical cap around the stretched wo
	const v3 wh = rt::normalize(rt::mk(alpha * wo.x, alpha * wo.y, wo.z));
	float sn, cs; rt::sincos2pi(r.x, sn, cs);
	const float z = fmaf(1.0f - r.y, 1.0f + wh.z, -wh.z);
	const float st = sqrtf(fmaxf(0.0f, fmaf(-z, z, 1.0f)));
	const v3 h = rt::mk(st * cs + wh.x, st * sn + wh.y, z + wh.z);
	if (!(rt::dot(h, h) > 0.0f)) return 0;
	const v3 wm = rt::normalize(rt::mk(alpha * h.x, alpha * h.y, h.z));
	const float cos_om = rt::dot(wo, wm);
	if (!(cos_om > 0.0f)) return 0;
	v3 wi;
	if (!DIEL) {
		wi = rt::reflect(rt::neg(wo), wm);
		if (!(wi.z > 0.0f)) return 0;
	} else {                                     // the dielectric of scatter() about wm
		const v3 ui = rt::neg(wo);
		const float cos_theta = fminf(cos_om, 1.0f);
		const float sin_theta = sqrtf(fmaf(-cos_theta, cos_theta, 1.0f));
		float r0 = (1.0f - ratio) / (1.0f + ratio); r0 = r0 * r0;
		const float x = 1.0f - cos_theta, x2 = x * x;
		const float prob = fmaf(1.0f - r0, x2 * x2 * x, r0);
		if (ratio * sin_theta > 1.0f || prob > r.z) {
			wi = rt::reflect(ui, wm);
			if (!(wi.z > 0.0f)) return 0;
		} else {
			const float dv = rt::dot(wm, ui);
			const float k = fmaf(-(ratio * ratio), fmaf(-dv, dv, 1.0f), 1.0f);
			if (k < 0.0f) return 0;
			const float coef = fmaf(ratio, dv, sqrtf(k));
			wi = rt::mk(fmaf(-coef, wm.x, ratio * ui.x), fmaf(-coef, wm.y, ratio * ui.y), fmaf(-coef, wm.z, ratio * ui.z));
			if (!(wi.z < 0.0f)) return 0;
		}
	}
	const float a2 = alpha * alpha;
	const float lo = 1.0f + ggx_lambda(wo, a2);
	const float g = lo / (lo + ggx_lambda(wi, a2));
	if (!DIEL) {
		const float x = 1.0f - cos_om, x2 = x * x, x5 = x2 * x2 * x;
		att = rt::mk(fmaf(1.0f - albedo.x, x5, albedo.x) * g, fmaf(1.0f - albedo.y, x5, albedo.y) * g, fmaf(1.0f - albedo.z, x5, albedo.z) * g);
	} else {
		att = rt::mul(albedo, g);
	}
	dir = rt::mk(fmaf(wi.z, n.x, fmaf(wi.y, V.x, wi.x * U.x)), fmaf(wi.z, n.y, fmaf(wi.y, V.y, wi.x * U.y)), fmaf(wi.z, n.z, fmaf(wi.y, V.z, wi.x * U.z)));
	return 1;
}

// Material::Scatter for every material kind.  Returns 0 = absorbed (path ends black),
// 1 = scattered (dir/attenuation valid), 2 = emitted (attenuation holds the emitted radiance).
// With DEFER, an image / noise albedo of a scattering material is not evaluated here: attenuation is
// left at 1 and defer_tex names the texture, to be multiplied in later by texture_kernel (dense warps).
// F is the feature word (rtb_kernels.h).
// With LIGHTS, Lambertian and isotropic scatters draw from the light mixture and set w (1 otherwise); ENV: with the map.
// ATTR: the dielectric refracts about s.n_diel (its inside / outside test stays with the geometric normal).
// ROUGH: the scene has GGX materials (their width is the material's fourth word); never part of the light mixture.
template <bool DEFER, uint32_t F>
__device__ __forceinline__ int scatter(const SceneView& sv, int mat, const Surface& s, v3 d, const rt::f4& r, const LightKey& lk,
                                       v3& dir, v3& att, float& w, int& defer_tex) {
	constexpr bool LIGHTS = (F & F_LIGHTS) != 0, ENV = (F & F_ENV) != 0, ATTR = (F & F_ATTR) != 0, ROUGH = (F & F_ROUGH) != 0;
	RTB_CHECK(mat >= 0 && mat < sv.n_materials, RTB_BOUNDS_MATERIAL);
	const float4 m0 = ldg4(sv.materials + 2 * mat), m1 = ldg4(sv.materials + 2 * mat + 1);
	const int kind = __float_as_int(m0.x), tex = __float_as_int(m0.y);
	const float param = m0.z;
	defer_tex = -1;
	v3 albedo;
	if (tex < 0) albedo = xyz(m1);
	else {
		const int tkind = __float_as_int(ldg4(sv.textures + 3 * tex).x);
		if (DEFER && kind != RTB_MAT_DIFFUSE_LIGHT && (tkind == RTB_TEX_NOISE || tkind == RTB_TEX_IMAGE)) { defer_tex = tex; albedo = rt::mk(1.0f, 1.0f, 1.0f); }
		else albedo = texture_value(sv, tex, s.u, s.v, s.p);
	}
	if (ROUGH && kind == RTB_MAT_ROUGH_METAL) return rough_scatter<false>(s.n_shade, d, r, m0.w, 0.0f, albedo, dir, att);
	if (ROUGH && kind == RTB_MAT_ROUGH_DIELECTRIC) {   // the dielectric's normal and ratio (below)
		v3 n = s.n_geom;
		const bool back = rt::dot(d, n) > 0.0f;
		if (ATTR) n = s.n_diel;
		if (back) n = rt::neg(n);
		return rough_scatter<true>(n, d, r, m0.w, back ? param : 1.0f / param, albedo, dir, att);
	}
	switch (kind) {
	case RTB_MAT_LAMBERTIAN: {   // LambertianAbstract / LambertianTexture  cu_materials.cuh:26-40,52-64
		if (LIGHTS) { att = albedo; return light_mix<false, ENV>(sv, s, r, lk, dir, w) ? 1 : 0; }
		dir = rt::add(s.n_shade, rt::unit_sphere(r.x, r.y));
		if (rt::near_zero(dir, 1e-9f)) return 0;
		att = albedo; return 1;
	}
	case RTB_MAT_METAL: {        // MetalAbstract  cu_materials.cuh:77-95 (in_ray.d is not normalised)
		dir = rt::madd(rt::unit_sphere(r.x, r.y), param, rt::reflect(d, s.n_shade));
		if (rt::dot(dir, s.n_shade) < 0.0f || rt::near_zero(dir, 1e-9f)) return 0;
		att = albedo; return 1;
	}
	case RTB_MAT_DIELECTRIC: {   // DielectricAbstract  cu_materials.cuh:115-143, reflectance :99-104
		v3 n = s.n_geom;
		bool back = rt::dot(d, n) > 0.0f;          // isBackfacing  ray_data.cuh:44-46
		if (ATTR) n = s.n_diel;
		if (back) n = rt::neg(n);
		float ratio = back ? param : 1.0f / param;
		v3 ud = rt::normalize(d);
		float cos_theta = fminf(rt::dot(rt::neg(ud), n), 1.0f);
		float sin_theta = sqrtf(fmaf(-cos_theta, cos_theta, 1.0f));
		float r0 = (1.0f - ratio) / (1.0f + ratio); r0 = r0 * r0;
		float x = 1.0f - cos_theta, x2 = x * x;
		float prob = fmaf(1.0f - r0, x2 * x2 * x, r0);   // powf(1 - cos, 5) as exact products
		if (ratio * sin_theta > 1.0f || prob > r.z) {
			dir = rt::reflect(ud, n);
		} else {                                   // glm::refract  func_geometric.inl:113-124
			float dv = rt::dot(n, ud);
			float k = fmaf(-(ratio * ratio), fmaf(-dv, dv, 1.0f), 1.0f);
			if (k < 0.0f) return 0;
			float coef = fmaf(ratio, dv, sqrtf(k));
			dir = rt::mk(fmaf(-coef, n.x, ratio * ud.x), fmaf(-coef, n.y, ratio * ud.y), fmaf(-coef, n.z, ratio * ud.z));
		}
		if (dir.x == 0.0f && dir.y == 0.0f && dir.z == 0.0f) return 0;
		att = albedo; return 1;
	}
	case RTB_MAT_ISOTROPIC: {    // book isotropic::scatter
		if (LIGHTS) { att = albedo; return light_mix<true, ENV>(sv, s, r, lk, dir, w) ? 1 : 0; }
		dir = rt::unit_sphere(r.x, r.y);
		att = albedo; return 1;
	}
	default:                     // RTB_MAT_DIFFUSE_LIGHT: emits, never scatters (book diffuse_light)
		att = albedo; return 2;
	}
}

__device__ __forceinline__ v3 background(const SceneView& sv, v3 d) {
	if (sv.background_mode == RTB_BG_CONSTANT) return rt::mk(sv.bg_r, sv.bg_g, sv.bg_b);
	// Renderer.cu:149-151: t = normalize(d).y * 0.5 + 0.5; lerp((0.1,0.2,0.4), (0.9,0.9,0.99), t)
	float ny = d.y * (1.0f / sqrtf(rt::dot(d, d)));
	float t = fmaf(ny, 0.5f, 0.5f);
	return rt::mk(fmaf(0.9f - 0.1f, t, 0.1f), fmaf(0.9f - 0.2f, t, 0.2f), fmaf(0.99f - 0.4f, t, 0.4f));
}

// ------------------------------------------------------------------------------------------------
// shade: one path segment of sample_world (Renderer.cu:146-176) + block-level queue compaction

// Shades one traversed segment.  Returns true when the path continues (no/nd/nthr hold the scattered
// ray and the updated throughput); otherwise the path has ended and its contribution (if any) has
// been written to contrib[path].
struct DeferredTex { int tex; float u, v; v3 p; };

// F: the feature word.  ENV: a miss returns the environment map's texel instead of the background.
template <bool DEFER, uint32_t F>
__device__ __forceinline__ bool shade_segment(const SceneView& sv, const BatchParams& bp, const WaveView& wv, uint32_t batch, uint32_t bounce,
                                              const float4& fo, const float4& fd, v3 thr, float t, int code,
                                              float4& no, float4& nd, v3& nthr, DeferredTex& dt) {
	constexpr bool LIGHTS = (F & F_LIGHTS) != 0, LIST = (F & F_LIST) != 0, ENV = (F & F_ENV) != 0, ATTR = (F & F_ATTR) != 0;
	dt.tex = -1;
	const uint32_t path = __float_as_uint(fd.w);
	const v3 o = xyz(fo), d = xyz(fd);
	if (code < 0) {
		v3 c = rt::mulv(thr, ENV ? env_radiance(sv, d) : background(sv, d));   // miss: throughput * sky   Renderer.cu:153
		wv.contrib[path] = make_float4(c.x, c.y, c.z, 0.0f);
		return false;
	}
	RTB_CHECK((code >> RTB_LEAF_TYPE_BITS) < sv.n_prims, RTB_BOUNDS_PRIM);
	const int2 info = __ldg(sv.prim_info + (code >> RTB_LEAF_TYPE_BITS));
	RTB_CHECK(info.x >= 0 && info.x < sv.n_materials, RTB_BOUNDS_MATERIAL);
	RTB_CHECK(path < wv.capacity, RTB_BOUNDS_PATH);
	const int tex = __float_as_int(ldg4(sv.materials + 2 * info.x).y);
	Surface s;
	reconstruct<ATTR>(sv, code, o, d, fo.w, t, texture_needs_uv(sv, tex), s);
	uint32_t pixel, sample;
	path_pixel_sample<LIST>(bp, batch, path, pixel, sample);
	const rt::f4 r = rt::rng4(bp.seed, pixel, sample, bounce, rt::STREAM_SCATTER);
	v3 dir, att;
	float w = 1.0f;
	const int res = scatter<DEFER, F>(sv, info.x, s, d, r, LightKey{bp.seed, pixel, sample, bounce}, dir, att, w, dt.tex);
	dt.u = s.u; dt.v = s.v; dt.p = s.p;
	if (res == 2) {                                       // emitter: throughput * emitted, path ends
		v3 c = rt::mulv(thr, att);
		wv.contrib[path] = make_float4(c.x, c.y, c.z, 0.0f);
		return false;
	}
	if (res != 1 || bounce + 1 >= bp.max_depth) { dt.tex = -1; return false; }   // absorbed, or out of depth: black   Renderer.cu:164,180
	// scatter_ray = Ray(at(t), dir, time); o += d * 0.001   Renderer.cu:168-175
	v3 o2 = rt::madd(dir, 0.001f, s.p);
	nthr = LIGHTS ? rt::mulv(rt::mul(thr, w), att) : rt::mulv(thr, att);   // (thr * w) * albedo: the order texture_kernel keeps
	no = make_float4(o2.x, o2.y, o2.z, fo.w);
	nd = make_float4(dir.x, dir.y, dir.z, fd.w);
	return true;
}

#ifndef SHADE_MIN_BLOCKS
#define SHADE_MIN_BLOCKS 8   // 8 x 128 threads x 64 registers = the whole register file (6 / 9 / 10 blocks: 11.7 / 10.9 / 12.4 ms)
#endif
template <uint32_t F>
__global__ void __launch_bounds__(SHADE_THREADS, SHADE_MIN_BLOCKS)
shade_kernel(SceneView sv, BatchParams bp_in, WaveView wv, uint32_t bounce, int q) {
	const BatchParams bp = with_call_params(bp_in, wv);
	__shared__ uint32_t s_chunk, s_base;
	__shared__ uint32_t s_warp[SHADE_THREADS / 32];
	if (bounce >= *wv.tail_from) return;
	const uint32_t n = wv.n_live[bounce];
	if (n == 0) return;
	const uint32_t batch = bp.batch_base + *wv.batch_index * bp.batch_stride;
	const int in = q, out = in ^ 1;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const float4* __restrict__ rod = in ? wv.ray_od[1] : wv.ray_od[0];
	const float4* __restrict__ rt_ = in ? wv.thr[1] : wv.thr[0];
	float4* __restrict__ wod = out ? wv.ray_od[1] : wv.ray_od[0];
	float4* __restrict__ wt = out ? wv.thr[1] : wv.thr[0];
	uint32_t* counter = wv.work + 2 * bounce + 1;

	// the first chunk of every block is static; further chunks come from the device counter
	uint32_t base = blockIdx.x * SHADE_THREADS;
	const uint32_t static_span = gridDim.x * SHADE_THREADS;
	for (;;) {
		if (base >= n) break;
		const uint32_t i = base + threadIdx.x;
		bool alive = false;
		float4 no = make_float4(0, 0, 0, 0), nd = no; v3 nthr = rt::mk(0, 0, 0);
		DeferredTex dt; dt.tex = -1; dt.u = dt.v = 0.0f; dt.p = rt::mk(0, 0, 0);
		if (i < n) {
			float4 fo, fd; ld_ray(rod + 2 * (size_t)i, fo, fd);
			const float4 ft = ldq(rt_ + i);
			const int2 h = ldq(wv.hit + i);
			alive = shade_segment<true, F>(sv, bp, wv, batch, bounce, fo, fd, xyz(ft), __int_as_float(h.x), h.y, no, nd, nthr, dt);
		}
		// live-path compaction: warp ballot/popc, one global atomic per block
		const uint32_t mask = __ballot_sync(FULL_MASK, alive);
		if (lane == 0) s_warp[warp] = __popc(mask);
		__syncthreads();
		if (threadIdx.x == 0) {
			uint32_t tot = 0;
#pragma unroll
			for (int w = 0; w < SHADE_THREADS / 32; ++w) { uint32_t c = s_warp[w]; s_warp[w] = tot; tot += c; }
			s_base = tot ? atomicAdd(wv.n_live + bounce + 1, tot) : 0u;
			s_chunk = (n > static_span) ? static_span + atomicAdd(counter, (uint32_t)SHADE_THREADS) : n;
		}
		__syncthreads();
		if (alive) {
			const uint32_t pos = s_base + s_warp[warp] + __popc(mask & ((1u << lane) - 1u));
			RTB_CHECK(pos < wv.capacity && pos < n, RTB_BOUNDS_QUEUE);
			st_ray(wod + 2 * (size_t)pos, no, nd); stq(wt + pos, make_float4(nthr.x, nthr.y, nthr.z, 0.0f));
			// texture work list: (p, queue slot), (u, v, -, texture id)
			const bool defer = dt.tex >= 0;
			const uint32_t act = __activemask();
			const uint32_t dmask = __ballot_sync(act, defer);
			if (dmask) {
				const int leader = __ffs(dmask) - 1;
				uint32_t tb = 0;
				if (lane == leader) tb = atomicAdd(wv.n_tex + bounce, (uint32_t)__popc(dmask));
				tb = __shfl_sync(act, tb, leader);
				if (defer) {
					const uint32_t k = tb + __popc(dmask & ((1u << lane) - 1u));
					wv.tex_work[2 * (size_t)k] = make_float4(dt.p.x, dt.p.y, dt.p.z, __uint_as_float(pos));
					wv.tex_work[2 * (size_t)k + 1] = make_float4(dt.u, dt.v, 0.0f, __int_as_float(dt.tex));
				}
			}
		}
		base = s_chunk;
		__syncthreads();
	}
}

// ------------------------------------------------------------------------------------------------
// tail: once the live queue is too short to fill the machine, per-bounce launches are pure latency.
// One persistent launch then runs every remaining path to completion (traverse + shade fused, one
// thread per path); later traverse/shade launches of the batch see tail_from and return at once.

template <bool MEDIA, int STACK, uint32_t F>
__global__ void __launch_bounds__(TRAVERSE_THREADS)
tail_kernel(SceneView sv, BatchParams bp_in, WaveView wv, uint32_t bounce0, int q, uint32_t threshold) {
	const BatchParams bp = with_call_params(bp_in, wv);
	__shared__ int s_stack[STACK * TRAVERSE_THREADS];
	if (*wv.tail_from < bounce0) return;                 // an earlier checkpoint already took the batch over
	const uint32_t n = wv.n_live[bounce0];
	if (n == 0 || n > threshold) return;
	if (blockIdx.x == 0 && threadIdx.x == 0) *wv.tail_from = bounce0;
	const uint32_t batch = bp.batch_base + *wv.batch_index * bp.batch_stride;
	const int in = q;
	const float4* __restrict__ rod = in ? wv.ray_od[1] : wv.ray_od[0];
	const float4* __restrict__ rt_ = in ? wv.thr[1] : wv.thr[0];
	unsigned long long extra = 0;
	const uint32_t stride = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
		float4 fo, fd; ld_ray(rod + 2 * (size_t)i, fo, fd);
		v3 thr = xyz(rt_[i]);
		constexpr bool LIST = (F & F_LIST) != 0;
		MediumRngT<LIST> mr = make_medium_rng<LIST>(bp, batch, __float_as_uint(fd.w), bounce0);
		for (uint32_t b = bounce0; b < bp.max_depth; ++b) {
			if (b > bounce0) ++extra;
			mr.bounce = b; mr.block = 0xFFFFFFFFu;
			float t; int code;
			trace_ray<(MEDIA ? 2 : 0)>(sv, xyz(fo), xyz(fd), fo.w, mr, s_stack + threadIdx.x, STACK, t, code);
			float4 no, nd; v3 nthr;
			DeferredTex dt;
			if (!shade_segment<false, F>(sv, bp, wv, batch, b, fo, fd, thr, t, code, no, nd, nthr, dt)) break;
			fo = no; fd = nd; thr = nthr;
		}
	}
	// ray segments traced beyond the first one of each path (that one is counted through n_live)
	for (int off = 16; off > 0; off >>= 1) extra += __shfl_down_sync(FULL_MASK, extra, off);
	if ((threadIdx.x & 31) == 0 && extra) atomicAdd(wv.totals + 1, extra);
}

// Kernel pointers by feature word, exported by the instantiation objects (rtb_shade.cu, rtb_tail.cu).
using ShadeKernel = void (*)(SceneView, BatchParams, WaveView, uint32_t, int);
using TailKernel = void (*)(SceneView, BatchParams, WaveView, uint32_t, int, uint32_t);
ShadeKernel shade_kernel_for(uint32_t f);
template <bool MEDIA, bool DEEP> TailKernel tail_kernel_for(uint32_t f);   // DEEP: the DEEP_STACK_SIZE stack, else STACK_SIZE

}  // namespace rtb
#endif
