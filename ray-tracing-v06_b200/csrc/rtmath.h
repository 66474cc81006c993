// rtmath.h — the arithmetic spec of the B200 path tracer (host + device).
//
// Every geometric quantity on the hot path is computed from IEEE-754 binary32
// +, -, *, /, sqrt and *explicit* fused multiply-adds, in the operation order written
// here.  The CUDA sources are compiled with -fmad=false (no implicit contraction),
// -prec-div=true, -prec-sqrt=true, -ftz=false, so the same sequence evaluated on a CPU
// (oracle/, written independently against DESIGN.md "Arithmetic spec") yields the same
// bits.  Functions that would otherwise need libm (sin/cos of a uniform angle, log of a
// uniform) are polynomial kernels defined here for the same reason.
#ifndef RTB_RTMATH_H
#define RTB_RTMATH_H

#include <stdint.h>
#include <math.h>
#include <string.h>

#ifdef __CUDACC__
#define RT_HD __host__ __device__ __forceinline__
#else
#define RT_HD inline
#endif

namespace rt {

struct v3 { float x, y, z; };

RT_HD v3 mk(float x, float y, float z) { v3 r; r.x = x; r.y = y; r.z = z; return r; }
RT_HD v3 add(v3 a, v3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
RT_HD v3 sub(v3 a, v3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
RT_HD v3 mul(v3 a, float s) { return mk(a.x * s, a.y * s, a.z * s); }
RT_HD v3 mulv(v3 a, v3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); }
RT_HD v3 divs(v3 a, float s) { return mk(a.x / s, a.y / s, a.z / s); }
RT_HD v3 neg(v3 a) { return mk(-a.x, -a.y, -a.z); }
// a*s + b, one fma per component  (Ray::at, ray_data.cuh:14)
RT_HD v3 madd(v3 a, float s, v3 b) { return mk(fmaf(a.x, s, b.x), fmaf(a.y, s, b.y), fmaf(a.z, s, b.z)); }
// glm::dot for vec3, contracted x -> y -> z
RT_HD float dot(v3 a, v3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)); }
RT_HD v3 cross(v3 a, v3 b) {
	return mk(fmaf(a.y, b.z, -(a.z * b.y)), fmaf(a.z, b.x, -(a.x * b.z)), fmaf(a.x, b.y, -(a.y * b.x)));
}
// glm::normalize: v * inversesqrt(dot(v,v)), inversesqrt = 1/sqrt (func_geometric.inl:81-90)
RT_HD v3 normalize(v3 a) { return mul(a, 1.0f / sqrtf(dot(a, a))); }
// glm::mix(x, y, a) = x*(1-a) + y*a
RT_HD float mixf(float x, float y, float a) { return fmaf(y, a, x * (1.0f - a)); }
RT_HD v3 mix(v3 x, v3 y, float a) {
	float b = 1.0f - a;
	return mk(fmaf(y.x, a, x.x * b), fmaf(y.y, a, x.y * b), fmaf(y.z, a, x.z * b));
}
// glm::near_zero from glm_utils.h:15-25 (all |c| <= eps)
RT_HD bool near_zero(v3 a, float eps) { return !(fabsf(a.x) > eps) && !(fabsf(a.y) > eps) && !(fabsf(a.z) > eps); }
// glm::reflect: I - N * dot(N, I) * 2
RT_HD v3 reflect(v3 I, v3 N) {
	float k = dot(N, I) * 2.0f;
	return mk(fmaf(-N.x, k, I.x), fmaf(-N.y, k, I.y), fmaf(-N.z, k, I.z));
}

RT_HD float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
RT_HD uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

// ---------------------------------------------------------------- Philox4x32-10
struct u4 { uint32_t x, y, z, w; };

RT_HD void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#ifdef __CUDA_ARCH__
	lo = a * b; hi = __umulhi(a, b);
#else
	uint64_t p = (uint64_t)a * b; lo = (uint32_t)p; hi = (uint32_t)(p >> 32);
#endif
}

RT_HD u4 philox4x32_10(u4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
	for (int r = 0; r < 10; ++r) {
		uint32_t hi0, lo0, hi1, lo1;
		mulhilo(0xD2511F53u, c.x, hi0, lo0);
		mulhilo(0xCD9E8D57u, c.z, hi1, lo1);
		u4 n; n.x = hi1 ^ c.y ^ k0; n.y = lo1; n.z = hi0 ^ c.w ^ k1; n.w = lo0;
		c = n; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
	}
	return c;
}

// curand_uniform's mapping (curand_uniform.h:69-72): x*2^-32 + 2^-33, in (0,1]
RT_HD float uniform01(uint32_t x) { return fmaf((float)x, 2.3283064365386963e-10f, 1.1641532182693481e-10f); }

// Stream ids (counter word z)
enum { STREAM_SCATTER = 0, STREAM_LENS = 1, STREAM_LIGHT = 2, STREAM_MEDIUM0 = 16 };
#define RT_CAMERA_BOUNCE 0xFFFFFFFFu

struct f4 { float x, y, z, w; };
// key = (seed, pixel), counter = (sample, bounce, stream, 0)
RT_HD f4 rng4(uint32_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t stream) {
	u4 c; c.x = sample; c.y = bounce; c.z = stream; c.w = 0u;
	u4 r = philox4x32_10(c, seed, pixel);
	f4 o; o.x = uniform01(r.x); o.y = uniform01(r.y); o.z = uniform01(r.z); o.w = uniform01(r.w);
	return o;
}

// ---------------------------------------------------------------- sin/cos(2*pi*u), u in (0,1]
RT_HD void sincos2pi(float u, float& s_out, float& c_out) {
	float x = u * 8.0f;
	int k = (int)x;                 // 0..8
	float f = x - (float)k;         // [0,1)
	int q = k & 7;
	int odd = q & 1;
	float g = odd ? (1.0f - f) : f;
	float a = g * 0.78539816339744831f;   // pi/4
	float a2 = a * a;
	float sp = fmaf(a2, 2.7557319223985893e-6f, -1.9841269841269841e-4f);
	sp = fmaf(a2, sp, 8.3333333333333332e-3f);
	sp = fmaf(a2, sp, -1.6666666666666666e-1f);
	float s = fmaf(a * a2, sp, a);
	float cp = fmaf(a2, -2.7557319223985888e-7f, 2.4801587301587302e-5f);
	cp = fmaf(a2, cp, -1.3888888888888889e-3f);
	cp = fmaf(a2, cp, 4.1666666666666664e-2f);
	cp = fmaf(a2, cp, -0.5f);
	float c = fmaf(a2, cp, 1.0f);
	int m = (q + odd) >> 1;         // quarter turns: even q: q/2 ; odd q: (q+1)/2
	// even: angle = m*pi/2 + a ; odd: angle = m*pi/2 - a
	float sa = odd ? -s : s;        // sin(+-a), cos(+-a) = c
	float rs, rc;
	switch (m & 3) {
	case 0: rs = sa; rc = c; break;
	case 1: rs = c; rc = -sa; break;
	case 2: rs = -sa; rc = -c; break;
	default: rs = -c; rc = sa; break;
	}
	s_out = rs; c_out = rc;
}

// ---------------------------------------------------------------- natural log, x > 0 normal
RT_HD float logpos(float x) {
	uint32_t b = f2u(x);
	int e = (int)(b >> 23) - 127;
	float m = u2f((b & 0x007FFFFFu) | 0x3F800000u);   // [1,2)
	if (m > 1.41421356f) { m = m * 0.5f; e += 1; }
	float s = (m - 1.0f) / (m + 1.0f);
	float s2 = s * s;
	float p = fmaf(s2, 0.1111111111f, 0.1428571429f);
	p = fmaf(s2, p, 0.2f);
	p = fmaf(s2, p, 0.3333333333f);
	p = fmaf(s2, p, 1.0f);
	p = (2.0f * s) * p;
	return fmaf((float)e, 0.69314718056f, p);
}

// Uniform direction on the unit sphere from two uniforms (replaces cuRandomOnUnit<3>,
// glm_utils.h:92-98, distributionally): z = 1-2u0, azimuth 2*pi*u1.
RT_HD v3 unit_sphere(float u0, float u1) {
	float z = fmaf(-2.0f, u0, 1.0f);
	float r2 = fmaf(-z, z, 1.0f);
	float r = sqrtf(r2 < 0.0f ? 0.0f : r2);
	float s, c; sincos2pi(u1, s, c);
	return mk(r * c, r * s, z);
}
// Uniform point in the unit disc (replaces cuRandomInUnit<2>, glm_utils.h:84-90).
RT_HD void unit_disc(float u0, float u1, float& dx, float& dy) {
	float r = sqrtf(u0);
	float s, c; sincos2pi(u1, s, c);
	dx = r * c; dy = r * s;
}

// ---------------------------------------------------------------- light sampling (DESIGN.md §5b)
#define RT_INV_PI 0.31830988618379067f
#define RT_INV_4PI 0.07957747154594767f
#define RT_2PI 6.28318530717958647692f

// cos of the half-angle of the cone a sphere of squared radius R2 subtends from squared distance d2 (> R2)
RT_HD float cone_cos_max(float d2, float R2) { return sqrtf(1.0f - R2 / d2); }
// Book 3 sphere::pdf_value: 1 / solid angle of that cone
RT_HD float cone_pdf(float cmax) { return 1.0f / (RT_2PI * (1.0f - cmax)); }
// Book 3 random_to_sphere in the orthonormal basis around e = centre - p (d2 = dot(e, e) > R2): a unit direction
// uniform in the cone, from the uniforms (u0 azimuth, u1 height).
RT_HD v3 cone_direction(v3 e, float cmax, float u0, float u1) {
	const float z = fmaf(u1, cmax - 1.0f, 1.0f);
	const float z2 = fmaf(-z, z, 1.0f);
	const float sz = sqrtf(z2 < 0.0f ? 0.0f : z2);
	float sn, cs; sincos2pi(u0, sn, cs);
	const float x = cs * sz, y = sn * sz;
	const v3 W = normalize(e);
	const v3 A = fabsf(W.x) > 0.9f ? mk(0.0f, 1.0f, 0.0f) : mk(1.0f, 0.0f, 0.0f);
	const v3 V = normalize(cross(W, A));
	const v3 U = cross(W, V);
	return normalize(mk(fmaf(z, W.x, fmaf(y, V.x, x * U.x)), fmaf(z, W.y, fmaf(y, V.y, x * U.y)), fmaf(z, W.z, fmaf(y, V.z, x * U.z))));
}
// Weight of a direction drawn from the half-and-half mixture: scattering pdf / mixture pdf (<= 0: the path ends black)
RT_HD float mixture_weight(float spdf, float lpdf) {
	const float mix = fmaf(0.5f, lpdf, 0.5f * spdf);
	return mix > 0.0f ? spdf / mix : 0.0f;
}

}  // namespace rt
#endif
