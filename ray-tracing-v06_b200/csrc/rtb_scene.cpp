// rtb_scene.cpp — host side of the C ABI: scene graph, serialisation, the reference's BVH
// builders restated, and the flattener that bakes instances into world-space SoA records.
//
// Reference behaviour followed (paths relative to the reference checkout):
//   bounds         getSphereBounds / getMovingSphereBounds   main/src/rt_engine/geometry/SphereHittable.cu:52-54,85-89
//   aabb           union, longest_axis, surface_area, centeroid   main/src/rt_engine/geometry/aabb.cuh:17-68
//   BVH builders   BVH_Handle::Factory                        main/src/rt_engine/geometry/BVH.cu:166-383
//   cameras        Pinhole/DefocusBlur/MotionBlurCamera ctors main/src/rt_engine/shaders/cu_Cameras.cuh:15-25,39-52,73-85
// Quads, boxes, instances, media follow "Ray Tracing: The Next Week" (SURVEY.md App. B).
#include "rtb_scene.h"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstring>
#include <functional>
#include <future>
#include <string>
#include <thread>

#include "rtmath.h"

namespace rtb {

static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg) { g_last_error = msg; return code; }

}  // namespace rtb

using namespace rtb;

// ============================================================== small helpers

static Box3 empty_box() {  // aabb() : min(1e9f), max(-1e9f)   aabb.cuh:17
	Box3 b; for (int i = 0; i < 3; ++i) { b.mn[i] = 1e9f; b.mx[i] = -1e9f; } return b;
}
static void grow(Box3& a, const Box3& b) {  // operator+=  aabb.cuh:24  (glm::min/max: (y<x)?y:x / (x<y)?y:x)
	for (int i = 0; i < 3; ++i) {
		a.mn[i] = (b.mn[i] < a.mn[i]) ? b.mn[i] : a.mn[i];
		a.mx[i] = (a.mx[i] < b.mx[i]) ? b.mx[i] : a.mx[i];
	}
}
static Box3 box_of_points(const float (*p)[3], int n) {
	Box3 b; for (int i = 0; i < 3; ++i) { b.mn[i] = p[0][i]; b.mx[i] = p[0][i]; }
	for (int k = 1; k < n; ++k) for (int i = 0; i < 3; ++i) {
		b.mn[i] = std::min(b.mn[i], p[k][i]); b.mx[i] = std::max(b.mx[i], p[k][i]);
	}
	return b;
}
static void pad_to_minimum(Box3& b) {  // book: aabb::pad_to_minimums, delta = 1e-4
	const float delta = 0.0001f;
	for (int i = 0; i < 3; ++i) if (b.mx[i] - b.mn[i] < delta) { b.mn[i] -= delta * 0.5f; b.mx[i] += delta * 0.5f; }
}
static int longest_axis(const Box3& b) {  // aabb.cuh:46-53
	float sx = std::fabs(b.mx[0] - b.mn[0]), sy = std::fabs(b.mx[1] - b.mn[1]), sz = std::fabs(b.mx[2] - b.mn[2]);
	if (sx > sy) return sx > sz ? 0 : 2;
	return sy > sz ? 1 : 2;
}
static float surface_area(const Box3& b) {  // aabb.cuh:55-64
	float sx = b.mx[0] - b.mn[0], sy = b.mx[1] - b.mn[1], sz = b.mx[2] - b.mn[2];
	if (sx < 0 || sy < 0 || sz < 0) return 0.0f;
	float cost = 0.0f; cost += sx * sy; cost += sx * sz; cost += sy * sz;
	return 2.0f * cost;
}

// World-from-object transform: rotation about +y by (c,s) then translation.
struct Xf {
	float c = 1.0f, s = 0.0f, off[3] = {0, 0, 0};
	bool rot = false, tr = false;
	void point(const float in[3], float out[3]) const {
		float x = in[0], y = in[1], z = in[2];
		if (rot) { float nx = fmaf(c, x, s * z); float nz = fmaf(c, z, -(s * x)); x = nx; z = nz; }
		if (tr) { x += off[0]; y += off[1]; z += off[2]; }
		out[0] = x; out[1] = y; out[2] = z;
	}
	void vec(const float in[3], float out[3]) const {
		float x = in[0], y = in[1], z = in[2];
		if (rot) { float nx = fmaf(c, x, s * z); float nz = fmaf(c, z, -(s * x)); x = nx; z = nz; }
		out[0] = x; out[1] = y; out[2] = z;
	}
};

// ============================================================== C ABI: scene assembly

extern "C" {

int rtb_abi_version(void) { return RTB_ABI_VERSION; }
const char* rtb_last_error(void) { return g_last_error.c_str(); }

int rtb_scene_create(rtb_scene** out) {
	if (!out) return fail(RTB_ERR_INVALID, "rtb_scene_create: null out");
	static std::atomic<uint64_t> next_uid{1};
	*out = new rtb_scene();
	(*out)->uid = next_uid.fetch_add(1);
	return RTB_OK;
}
void rtb_scene_destroy(rtb_scene* s) { delete s; }

static bool tex_ok(const rtb_scene* s, int t) { return t >= 0 && t < (int)s->textures.size(); }
static bool mat_ok(const rtb_scene* s, int m) { return m >= 0 && m < (int)s->materials.size(); }
static bool obj_ok(const rtb_scene* s, int o) { return o >= 0 && o < (int)s->objects.size(); }

static int push_texture(rtb_scene* s, const rtbs_texture& t) { s->version++; s->textures.push_back(t); return (int)s->textures.size() - 1; }

int rtb_add_solid_texture(rtb_scene* s, const float rgb[3]) {
	if (!s || !rgb) return fail(RTB_ERR_INVALID, "rtb_add_solid_texture: null argument");
	rtbs_texture t{}; t.kind = RTB_TEX_SOLID; t.even = t.odd = -1; t.scale = 1.0f;
	t.rgb[0] = rgb[0]; t.rgb[1] = rgb[1]; t.rgb[2] = rgb[2];
	return push_texture(s, t);
}
int rtb_add_checker_texture(rtb_scene* s, float scale, int even_tex, int odd_tex) {
	if (!s || !tex_ok(s, even_tex) || !tex_ok(s, odd_tex)) return fail(RTB_ERR_INVALID, "rtb_add_checker_texture: bad texture id");
	if (!(scale != 0.0f)) return fail(RTB_ERR_INVALID, "rtb_add_checker_texture: scale must be non-zero");
	rtbs_texture t{}; t.kind = RTB_TEX_CHECKER; t.even = even_tex; t.odd = odd_tex; t.scale = scale;
	return push_texture(s, t);
}
int rtb_add_image_texture(rtb_scene* s, const uint8_t* px, int w, int h, int ch) {
	if (!s || !px || w <= 0 || h <= 0 || !(ch == 1 || ch == 3 || ch == 4))
		return fail(RTB_ERR_INVALID, "rtb_add_image_texture: bad image");
	rtbs_texture t{}; t.kind = RTB_TEX_IMAGE; t.even = t.odd = -1; t.scale = 1.0f; t.width = w; t.height = h;
	while (s->blob.size() % 4) s->blob.push_back(0);
	t.blob_offset = (uint32_t)s->blob.size();
	s->blob.resize(s->blob.size() + (size_t)w * h * 3);
	uint8_t* dst = s->blob.data() + t.blob_offset;
	for (size_t i = 0; i < (size_t)w * h; ++i) {
		if (ch == 1) { dst[3 * i] = dst[3 * i + 1] = dst[3 * i + 2] = px[i]; }
		else { dst[3 * i] = px[ch * i]; dst[3 * i + 1] = px[ch * i + 1]; dst[3 * i + 2] = px[ch * i + 2]; }
	}
	return push_texture(s, t);
}
int rtb_add_noise_texture(rtb_scene* s, float scale, uint32_t seed) {
	if (!s) return fail(RTB_ERR_INVALID, "rtb_add_noise_texture: null scene");
	rtbs_texture t{}; t.kind = RTB_TEX_NOISE; t.even = t.odd = -1; t.scale = scale; t.seed = seed;
	while (s->blob.size() % 4) s->blob.push_back(0);
	t.blob_offset = (uint32_t)s->blob.size();
	s->blob.resize(s->blob.size() + RTBS_PERLIN_BYTES);
	float* grad = reinterpret_cast<float*>(s->blob.data() + t.blob_offset);
	int32_t* perm = reinterpret_cast<int32_t*>(s->blob.data() + t.blob_offset + 256 * 3 * 4);
	// book perlin(): randvec[i] = unit_vector(random(-1,1)^3); three Fisher-Yates shuffles.
	const uint32_t key1 = 0x5045524Cu;  // "PERL"
	for (uint32_t i = 0; i < 256; ++i) {
		rt::u4 c; c.x = i; c.y = 0; c.z = 0; c.w = 0;
		rt::u4 r = rt::philox4x32_10(c, seed, key1);
		float x = 2.0f * rt::uniform01(r.x) - 1.0f, y = 2.0f * rt::uniform01(r.y) - 1.0f, z = 2.0f * rt::uniform01(r.z) - 1.0f;
		float len = std::sqrt(x * x + y * y + z * z);
		if (!(len > 0.0f)) { x = 1.0f; y = z = 0.0f; len = 1.0f; }
		grad[3 * i] = x / len; grad[3 * i + 1] = y / len; grad[3 * i + 2] = z / len;
	}
	for (uint32_t tbl = 0; tbl < 3; ++tbl) {
		int32_t* p = perm + 256 * tbl;
		for (int i = 0; i < 256; ++i) p[i] = i;
		for (int i = 255; i > 0; --i) {
			rt::u4 c; c.x = (uint32_t)i; c.y = 1 + tbl; c.z = 0; c.w = 0;
			rt::u4 r = rt::philox4x32_10(c, seed, key1);
			int target = (int)(((uint64_t)r.x * (uint64_t)(i + 1)) >> 32);  // uniform int in [0,i]
			std::swap(p[i], p[target]);
		}
	}
	return push_texture(s, t);
}

static int push_material(rtb_scene* s, int kind, int tex, const float a[3], float param, float alpha = 0.0f) {
	rtbs_material m{}; m.kind = kind; m.tex = tex; m.param = param;
	m.albedo[0] = a ? a[0] : 1.0f; m.albedo[1] = a ? a[1] : 1.0f; m.albedo[2] = a ? a[2] : 1.0f;
	s->version++; s->materials.push_back(m); s->mat_alpha.push_back(alpha); return (int)s->materials.size() - 1;
}
int rtb_add_lambertian(rtb_scene* s, int tex) {
	if (!s || !tex_ok(s, tex)) return fail(RTB_ERR_INVALID, "rtb_add_lambertian: bad texture id");
	return push_material(s, RTB_MAT_LAMBERTIAN, tex, nullptr, 0.0f);
}
int rtb_add_lambertian_color(rtb_scene* s, const float albedo[3]) {
	if (!s || !albedo) return fail(RTB_ERR_INVALID, "rtb_add_lambertian_color: null argument");
	return push_material(s, RTB_MAT_LAMBERTIAN, -1, albedo, 0.0f);
}
int rtb_add_metal(rtb_scene* s, const float albedo[3], float fuzz) {
	if (!s || !albedo) return fail(RTB_ERR_INVALID, "rtb_add_metal: null argument");
	return push_material(s, RTB_MAT_METAL, -1, albedo, fuzz);   // fuzz not clamped: cu_materials.cuh:75
}
int rtb_add_dielectric(rtb_scene* s, const float albedo[3], float ior) {
	if (!s || !albedo) return fail(RTB_ERR_INVALID, "rtb_add_dielectric: null argument");
	return push_material(s, RTB_MAT_DIELECTRIC, -1, albedo, ior);
}
// GGX materials (DESIGN.md §5f): everything is checked before the scene is touched.
static bool rough_args_ok(const float c[3], float alpha) {
	return c && std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]) && alpha >= RTB_ROUGH_ALPHA_MIN && alpha <= 1.0f;
}
int rtb_add_rough_metal(rtb_scene* s, const float f0[3], float alpha) {
	if (!s || !rough_args_ok(f0, alpha)) return fail(RTB_ERR_INVALID, "rtb_add_rough_metal: needs a finite f0 and alpha in [0.001, 1]");
	return push_material(s, RTB_MAT_ROUGH_METAL, -1, f0, 0.0f, alpha);
}
int rtb_add_rough_dielectric(rtb_scene* s, const float albedo[3], float ior, float alpha) {
	if (!s || !rough_args_ok(albedo, alpha) || !(ior > 0.0f) || !std::isfinite(ior))
		return fail(RTB_ERR_INVALID, "rtb_add_rough_dielectric: needs a finite albedo, a finite ior > 0 and alpha in [0.001, 1]");
	return push_material(s, RTB_MAT_ROUGH_DIELECTRIC, -1, albedo, ior, alpha);
}
int rtb_add_diffuse_light(rtb_scene* s, int tex) {
	if (!s || !tex_ok(s, tex)) return fail(RTB_ERR_INVALID, "rtb_add_diffuse_light: bad texture id");
	return push_material(s, RTB_MAT_DIFFUSE_LIGHT, tex, nullptr, 0.0f);
}
int rtb_add_isotropic(rtb_scene* s, int tex) {
	if (!s || !tex_ok(s, tex)) return fail(RTB_ERR_INVALID, "rtb_add_isotropic: bad texture id");
	return push_material(s, RTB_MAT_ISOTROPIC, tex, nullptr, 0.0f);
}

static int push_object(rtb_scene* s, const rtbs_object& o) { s->version++; s->objects.push_back(o); return (int)s->objects.size() - 1; }
static rtbs_object blank_object(int kind, int mat) {
	rtbs_object o{}; o.kind = kind; o.mat = mat; o.child_begin = 0; o.child_count = 0; o.aux = 0; return o;
}

int rtb_add_sphere(rtb_scene* s, const float c[3], float r, int mat) {
	if (!s || !c || !mat_ok(s, mat)) return fail(RTB_ERR_INVALID, "rtb_add_sphere: bad argument");
	if (!(std::fabs(r) > 0.0f) || !std::isfinite(r)) return fail(RTB_ERR_INVALID, "rtb_add_sphere: the radius must be finite and non-zero");
	rtbs_object o = blank_object(RTB_OBJ_SPHERE, mat);
	o.f[0] = c[0]; o.f[1] = c[1]; o.f[2] = c[2]; o.f[3] = r;
	return push_object(s, o);
}
int rtb_add_moving_sphere(rtb_scene* s, const float c0[3], const float c1[3], float r, int mat) {
	if (!s || !c0 || !c1 || !mat_ok(s, mat)) return fail(RTB_ERR_INVALID, "rtb_add_moving_sphere: bad argument");
	if (!(std::fabs(r) > 0.0f) || !std::isfinite(r)) return fail(RTB_ERR_INVALID, "rtb_add_moving_sphere: the radius must be finite and non-zero");
	rtbs_object o = blank_object(RTB_OBJ_MOVING_SPHERE, mat);
	o.f[0] = c0[0]; o.f[1] = c0[1]; o.f[2] = c0[2]; o.f[3] = r; o.f[4] = c1[0]; o.f[5] = c1[1]; o.f[6] = c1[2];
	return push_object(s, o);
}
static int add_planar(rtb_scene* s, int kind, const float Q[3], const float u[3], const float v[3], int mat) {
	if (!s || !Q || !u || !v || !mat_ok(s, mat)) return fail(RTB_ERR_INVALID, "rtb_add_quad/triangle: bad argument");
	rtbs_object o = blank_object(kind, mat);
	for (int i = 0; i < 3; ++i) { o.f[i] = Q[i]; o.f[3 + i] = u[i]; o.f[6 + i] = v[i]; }
	return push_object(s, o);
}
int rtb_add_quad(rtb_scene* s, const float Q[3], const float u[3], const float v[3], int mat) { return add_planar(s, RTB_OBJ_QUAD, Q, u, v, mat); }
int rtb_add_triangle(rtb_scene* s, const float Q[3], const float u[3], const float v[3], int mat) { return add_planar(s, RTB_OBJ_TRIANGLE, Q, u, v, mat); }
int rtb_add_box(rtb_scene* s, const float a[3], const float b[3], int mat) {
	if (!s || !a || !b || !mat_ok(s, mat)) return fail(RTB_ERR_INVALID, "rtb_add_box: bad argument");
	rtbs_object o = blank_object(RTB_OBJ_BOX, mat);
	for (int i = 0; i < 3; ++i) { o.f[i] = std::fmin(a[i], b[i]); o.f[3 + i] = std::fmax(a[i], b[i]); }
	return push_object(s, o);
}
static int add_group(rtb_scene* s, int kind, const int* ch, int n, int aux) {
	if (!s || n < 0 || (n > 0 && !ch)) return fail(RTB_ERR_INVALID, "rtb_add_list/bvh: bad argument");
	for (int i = 0; i < n; ++i) if (!obj_ok(s, ch[i])) return fail(RTB_ERR_INVALID, "rtb_add_list/bvh: bad child id");
	rtbs_object o = blank_object(kind, -1);
	o.child_begin = (int)s->children.size(); o.child_count = n; o.aux = aux;
	s->children.insert(s->children.end(), ch, ch + n);
	return push_object(s, o);
}
int rtb_add_list(rtb_scene* s, const int* ch, int n) { return add_group(s, RTB_OBJ_LIST, ch, n, 0); }
int rtb_add_bvh(rtb_scene* s, const int* ch, int n, int builder) {
	if (builder < RTB_BVH_TOPDOWN_MEDIAN || builder > RTB_BVH_BOTTOMUP) return fail(RTB_ERR_INVALID, "rtb_add_bvh: bad builder");
	if (n < 1) return fail(RTB_ERR_INVALID, "rtb_add_bvh: needs at least one child");
	return add_group(s, RTB_OBJ_BVH, ch, n, builder);
}
// Corner normal k of a mesh_ex call: normalised in double when non-zero, zero kept.
static void put_corner_normal(const float* n, float out[3]) {
	const double x = n[0], y = n[1], z = n[2], len = std::sqrt(x * x + y * y + z * z);
	for (int c = 0; c < 3; ++c) out[c] = len > 0.0 ? (float)((double)n[c] / len) : 0.0f;
}
static int add_mesh(rtb_scene* s, const float* vertices, int n_vertices, const int* indices, int n_triangles,
                    const float* normals, const float* uvs, int mat) {
	if (!s || !vertices || !indices || n_vertices < 3 || n_triangles < 1 || !mat_ok(s, mat)) return fail(RTB_ERR_INVALID, "rtb_add_mesh: bad argument");
	for (int i = 0; i < 3 * n_triangles; ++i) if (indices[i] < 0 || indices[i] >= n_vertices) return fail(RTB_ERR_INVALID, "rtb_add_mesh: vertex index out of range");
	for (size_t i = 0; normals && i < 3 * (size_t)n_vertices; ++i)
		if (!std::isfinite(normals[i])) return fail(RTB_ERR_INVALID, "rtb_add_mesh_ex: normal of vertex " + std::to_string(i / 3) + " is not finite");
	for (size_t i = 0; uvs && i < 2 * (size_t)n_vertices; ++i)
		if (!std::isfinite(uvs[i])) return fail(RTB_ERR_INVALID, "rtb_add_mesh_ex: UV of vertex " + std::to_string(i / 2) + " is not finite");
	std::vector<int> ids; ids.reserve(n_triangles);
	s->objects.reserve(s->objects.size() + (size_t)n_triangles + 1);
	for (int t = 0; t < n_triangles; ++t) {
		const float* a = vertices + 3 * (size_t)indices[3 * t];
		const float* b = vertices + 3 * (size_t)indices[3 * t + 1];
		const float* c = vertices + 3 * (size_t)indices[3 * t + 2];
		const float u[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, v[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
		// no area: nothing to hit, and the quad constants would be NaN.  (Plain products here, not the path's fma cross:
		// fma(a, b, -(b * a)) is the rounding residue of the product, so cross(u, u) would not be exactly zero.)
		const float nx = u[1] * v[2] - u[2] * v[1], ny = u[2] * v[0] - u[0] * v[2], nz = u[0] * v[1] - u[1] * v[0];
		if (!(nx * nx + ny * ny + nz * nz > 0.0f)) continue;
		ids.push_back(add_planar(s, RTB_OBJ_TRIANGLE, a, u, v, mat));
		if (normals || uvs) {
			rtbs_tri_attr at{};
			for (int k = 0; k < 3; ++k) {
				const size_t vi = (size_t)indices[3 * t + k];
				if (normals) put_corner_normal(normals + 3 * vi, at.n[k]);
				if (uvs) { at.uv[k][0] = uvs[2 * vi]; at.uv[k][1] = uvs[2 * vi + 1]; }
			}
			at.flags = (normals ? RTBS_ATTR_NORMALS : 0) | (uvs ? RTBS_ATTR_UVS : 0);
			s->tri_attrs.push_back(at);
			s->objects.back().aux = (int32_t)s->tri_attrs.size();
		}
	}
	if (ids.empty()) return fail(RTB_ERR_INVALID, "rtb_add_mesh: no triangle has an area");
	return add_group(s, RTB_OBJ_BVH, ids.data(), (int)ids.size(), RTB_BVH_TOPDOWN_MEDIAN);
}
int rtb_add_mesh(rtb_scene* s, const float* vertices, int n_vertices, const int* indices, int n_triangles, int mat) {
	return add_mesh(s, vertices, n_vertices, indices, n_triangles, nullptr, nullptr, mat);
}
int rtb_add_mesh_ex(rtb_scene* s, const float* vertices, int n_vertices, const int* indices, int n_triangles,
                    const float* normals, const float* uvs, int mat) {
	return add_mesh(s, vertices, n_vertices, indices, n_triangles, normals, uvs, mat);
}
int rtb_add_translate(rtb_scene* s, int child, const float off[3]) {
	if (!s || !off || !obj_ok(s, child)) return fail(RTB_ERR_INVALID, "rtb_add_translate: bad argument");
	rtbs_object o = blank_object(RTB_OBJ_TRANSLATE, -1);
	o.child_begin = (int)s->children.size(); o.child_count = 1; s->children.push_back(child);
	o.f[0] = off[0]; o.f[1] = off[1]; o.f[2] = off[2];
	return push_object(s, o);
}
int rtb_add_rotate_y(rtb_scene* s, int child, float degrees) {
	if (!s || !obj_ok(s, child)) return fail(RTB_ERR_INVALID, "rtb_add_rotate_y: bad argument");
	rtbs_object o = blank_object(RTB_OBJ_ROTATE_Y, -1);
	o.child_begin = (int)s->children.size(); o.child_count = 1; s->children.push_back(child);
	float radians = degrees * 0.01745329251994329576923690768489f;  // glm::radians
	o.f[0] = degrees; o.f[1] = sinf(radians); o.f[2] = cosf(radians);
	return push_object(s, o);
}
int rtb_add_constant_medium(rtb_scene* s, int boundary, float density, int phase_mat) {
	if (!s || !obj_ok(s, boundary) || !mat_ok(s, phase_mat)) return fail(RTB_ERR_INVALID, "rtb_add_constant_medium: bad argument");
	if (!(density > 0.0f)) return fail(RTB_ERR_INVALID, "rtb_add_constant_medium: density must be > 0");
	rtbs_object o = blank_object(RTB_OBJ_CONSTANT_MEDIUM, phase_mat);
	o.child_begin = (int)s->children.size(); o.child_count = 1; s->children.push_back(boundary);
	o.f[0] = density; o.f[1] = -1.0f / density;
	return push_object(s, o);
}
int rtb_scene_set_root(rtb_scene* s, int object) {
	if (!s || !obj_ok(s, object)) return fail(RTB_ERR_INVALID, "rtb_scene_set_root: bad object id");
	s->root = object; s->version++; return RTB_OK;
}
int rtb_scene_set_world_bvh(rtb_scene* s, int mode) {
	if (!s || (mode != RTB_WORLD_BVH_QUALITY && mode != RTB_WORLD_BVH_AS_BUILT && mode != RTB_WORLD_BVH_GPU_LBVH)) return fail(RTB_ERR_INVALID, "rtb_scene_set_world_bvh: bad mode");
	s->world_bvh_mode = mode; s->version++; return RTB_OK;
}
int rtb_scene_set_background(rtb_scene* s, int mode, const float rgb[3]) {
	if (!s || (mode != RTB_BG_SKY_GRADIENT && mode != RTB_BG_CONSTANT)) return fail(RTB_ERR_INVALID, "rtb_scene_set_background: bad mode");
	s->background_mode = mode; s->version++;
	if (rgb) { s->background[0] = rgb[0]; s->background[1] = rgb[1]; s->background[2] = rgb[2]; }
	return RTB_OK;
}
int rtb_scene_num_objects(const rtb_scene* s) { return s ? (int)s->objects.size() : RTB_ERR_INVALID; }
int rtb_scene_num_children(const rtb_scene* s, int object) {
	if (!s || !obj_ok(s, object)) return fail(RTB_ERR_INVALID, "rtb_scene_num_children: bad argument");
	return s->objects[object].child_count;
}

}  // extern "C"

// ============================================================== bounds

static void quad_corners(const float* f, float p[4][3]) {
	for (int i = 0; i < 3; ++i) { p[0][i] = f[i]; p[1][i] = f[i] + f[3 + i]; p[2][i] = f[i] + f[6 + i]; p[3][i] = f[i] + f[3 + i] + f[6 + i]; }
}

// Bounds of `obj` in its parent's frame.
static int object_bounds(const rtb_scene* s, int id, Box3& out, int depth = 0) {
	if (depth > 64) return fail(RTB_ERR_INVALID, "object graph too deep / cyclic");
	const rtbs_object& o = s->objects[id];
	switch (o.kind) {
	case RTB_OBJ_SPHERE:
		for (int i = 0; i < 3; ++i) { out.mn[i] = o.f[i] - o.f[3]; out.mx[i] = o.f[i] + o.f[3]; }
		return RTB_OK;
	case RTB_OBJ_MOVING_SPHERE: {
		Box3 b0, b1;
		for (int i = 0; i < 3; ++i) { b0.mn[i] = o.f[i] - o.f[3]; b0.mx[i] = o.f[i] + o.f[3]; b1.mn[i] = o.f[4 + i] - o.f[3]; b1.mx[i] = o.f[4 + i] + o.f[3]; }
		for (int i = 0; i < 3; ++i) { out.mn[i] = (b1.mn[i] < b0.mn[i]) ? b1.mn[i] : b0.mn[i]; out.mx[i] = (b0.mx[i] < b1.mx[i]) ? b1.mx[i] : b0.mx[i]; }
		return RTB_OK;
	}
	case RTB_OBJ_QUAD: case RTB_OBJ_TRIANGLE: {
		float p[4][3]; quad_corners(o.f, p);
		out = box_of_points(p, o.kind == RTB_OBJ_QUAD ? 4 : 3); pad_to_minimum(out);
		return RTB_OK;
	}
	case RTB_OBJ_BOX:
		for (int i = 0; i < 3; ++i) { out.mn[i] = o.f[i]; out.mx[i] = o.f[3 + i]; }
		pad_to_minimum(out);
		return RTB_OK;
	case RTB_OBJ_LIST: case RTB_OBJ_BVH: {
		out = empty_box();
		for (int k = 0; k < o.child_count; ++k) {
			Box3 b; int rc = object_bounds(s, s->children[o.child_begin + k], b, depth + 1); if (rc) return rc;
			grow(out, b);
		}
		return RTB_OK;
	}
	case RTB_OBJ_TRANSLATE: {
		Box3 b; int rc = object_bounds(s, s->children[o.child_begin], b, depth + 1); if (rc) return rc;
		for (int i = 0; i < 3; ++i) { out.mn[i] = b.mn[i] + o.f[i]; out.mx[i] = b.mx[i] + o.f[i]; }
		return RTB_OK;
	}
	case RTB_OBJ_ROTATE_Y: {  // book rotate_y ctor: box of the 8 rotated corners
		Box3 b; int rc = object_bounds(s, s->children[o.child_begin], b, depth + 1); if (rc) return rc;
		float sn = o.f[1], cs = o.f[2];
		float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
		for (int i = 0; i < 2; ++i) for (int j = 0; j < 2; ++j) for (int k = 0; k < 2; ++k) {
			float x = i ? b.mx[0] : b.mn[0], y = j ? b.mx[1] : b.mn[1], z = k ? b.mx[2] : b.mn[2];
			float t[3] = {cs * x + sn * z, y, -sn * x + cs * z};
			for (int c = 0; c < 3; ++c) { mn[c] = std::fmin(mn[c], t[c]); mx[c] = std::fmax(mx[c], t[c]); }
		}
		for (int c = 0; c < 3; ++c) { out.mn[c] = mn[c]; out.mx[c] = mx[c]; }
		return RTB_OK;
	}
	case RTB_OBJ_CONSTANT_MEDIUM:
		return object_bounds(s, s->children[o.child_begin], out, depth + 1);
	}
	return fail(RTB_ERR_INVALID, "unknown object kind");
}

extern "C" int rtb_object_bounds(const rtb_scene* s, int object, float out6[6]) {
	if (!s || !out6 || !obj_ok(s, object)) return fail(RTB_ERR_INVALID, "rtb_object_bounds: bad argument");
	Box3 b; int rc = object_bounds(s, object, b); if (rc) return rc;
	for (int i = 0; i < 3; ++i) { out6[i] = b.mn[i]; out6[3 + i] = b.mx[i]; }
	return RTB_OK;
}

// ============================================================== serialisation

static_assert(sizeof(rtbs_tri_attr) == 64, "rtbs_tri_attr is a 64-byte record");

extern "C" size_t rtb_scene_serialize(const rtb_scene* s, void* buf, size_t cap) {
	if (!s) return 0;
	// A scene without sampled lights or a map is written as RTBS v1, byte for byte; one with lights only as v2 (the list
	// appended); one with a map as v3 (the list, possibly empty, then the map).
	// One with triangle attributes as v4: the v3 content (an empty map record when there is no map), then the attributes.
	// One with a rough material as v5: the v4 content (possibly no attributes), then the GGX width of every material.
	const bool rough = s->has_rough();
	const bool attr = !s->tri_attrs.empty() || rough;
	const bool env = s->env_width > 0 || attr;
	const bool lights = !s->sampled_lights.empty() || env;
	const size_t env_floats = (size_t)s->env_width * s->env_height * 3;
	size_t need = sizeof(rtbs_header) + s->textures.size() * sizeof(rtbs_texture) + s->materials.size() * sizeof(rtbs_material) +
	              s->objects.size() * sizeof(rtbs_object) + s->children.size() * 4 + s->blob.size() +
	              (lights ? 4 + s->sampled_lights.size() * 4 : 0) + (env ? sizeof(rtbs_env) + env_floats * 4 : 0) +
	              (attr ? 4 + s->tri_attrs.size() * sizeof(rtbs_tri_attr) : 0) + (rough ? 4 + s->mat_alpha.size() * 4 : 0);
	if (!buf || cap < need) return need;
	rtbs_header h{}; h.magic = RTBS_MAGIC;
	h.version = rough ? RTBS_VERSION_ROUGH : attr ? RTBS_VERSION_ATTR : env ? RTBS_VERSION_ENV : lights ? RTBS_VERSION_LIGHTS : RTBS_VERSION;
	h.n_textures = (uint32_t)s->textures.size(); h.n_materials = (uint32_t)s->materials.size();
	h.n_objects = (uint32_t)s->objects.size(); h.n_children = (uint32_t)s->children.size();
	h.n_blob_bytes = (uint32_t)s->blob.size(); h.root_object = s->root; h.background_mode = s->background_mode;
	memcpy(h.background, s->background, 12);
	uint8_t* p = static_cast<uint8_t*>(buf);
	auto put = [&p](const void* src, size_t n) { if (n) { memcpy(p, src, n); p += n; } };
	put(&h, sizeof h);
	put(s->textures.data(), s->textures.size() * sizeof(rtbs_texture));
	put(s->materials.data(), s->materials.size() * sizeof(rtbs_material));
	put(s->objects.data(), s->objects.size() * sizeof(rtbs_object));
	put(s->children.data(), s->children.size() * 4);
	put(s->blob.data(), s->blob.size());
	if (lights) {
		const int32_t n = (int32_t)s->sampled_lights.size();
		put(&n, 4);
		put(s->sampled_lights.data(), s->sampled_lights.size() * 4);
	}
	if (env) {
		rtbs_env e{};
		e.width = s->env_width; e.height = s->env_height; e.flags = s->env_flags;
		memcpy(e.scale, s->env_scale, 12);
		put(&e, sizeof e);
		put(s->env_rgb.data(), env_floats * 4);
	}
	if (attr) {
		const uint32_t n = (uint32_t)s->tri_attrs.size();
		put(&n, 4);
		put(s->tri_attrs.data(), s->tri_attrs.size() * sizeof(rtbs_tri_attr));
	}
	if (rough) {
		const uint32_t n = (uint32_t)s->mat_alpha.size();
		put(&n, 4);
		put(s->mat_alpha.data(), s->mat_alpha.size() * 4);
	}
	return need;
}

// ============================================================== BVH builders (BVH.cu:166-383 restated)

namespace rtb {

namespace {
struct Item { Box3 box; int idx; };

struct Builder {
	std::vector<Item> arr;
	std::vector<rtb_bvh_node> nodes;

	Box3 partition_bounds(int start, int end) const {  // _get_partition_bounds  BVH.cu:306-312
		Box3 b = empty_box();
		for (int i = start; i < end; ++i) grow(b, arr[i].box);
		return b;
	}
	int push_node(const Box3& b, int left, int right) {
		rtb_bvh_node n; memcpy(n.bmin, b.mn, 12); memcpy(n.bmax, b.mx, 12);
		n.left_child_idx = left; n.right_child_hittable_idx = right;
		nodes.push_back(n); return (int)nodes.size() - 1;
	}
	// _build_bvh_rec1  BVH.cu:180-210: sort the range by min[longest axis], split at the middle,
	// children first (left, then right), node last => post-order array, root = last index.
	int rec_median(int start, int end) {
		Box3 bounds = partition_bounds(start, end);
		int axis = longest_axis(bounds);
		if (end - start == 1) return push_node(bounds, -1, start);
		std::sort(arr.begin() + start, arr.begin() + end,
		          [axis](const Item& a, const Item& b) { return a.box.mn[axis] < b.box.mn[axis]; });
		int mid = (start + end) / 2;
		int l = rec_median(start, mid);
		int r = rec_median(mid, end);
		return push_node(bounds, l, r);
	}
	// _find_optimal_split  BVH.cu:245-283: 16 planes x 3 axes on the partition bounds, cost = SA*count.
	void find_split(int start, int end, const Box3& bounds, int& best_axis, float& best_split) const {
		const int split_points = 16;
		float best_cost = FLT_MAX;
		for (int axis = 0; axis < 3; ++axis) for (int split = 0; split < split_points; ++split) {
			float pos = (split + 1.0f) / (split_points + 1.0f);
			float lo = bounds.mn[axis], hi = bounds.mx[axis];
			pos = lo * (1.0f - pos) + hi * pos;  // glm::mix
			Box3 lb = empty_box(), rb = empty_box(); int lc = 0, rc = 0;
			for (int i = start; i < end; ++i) {
				const Box3& b = arr[i].box;
				float cen = (b.mx[axis] + b.mn[axis]) * 0.5f;  // centeroid  aabb.cuh:66-68
				if (cen < pos) { grow(lb, b); lc++; } else { grow(rb, b); rc++; }
			}
			float cost = surface_area(lb) * lc + surface_area(rb) * rc;
			if (cost < best_cost) { best_cost = cost; best_axis = axis; best_split = pos; }
		}
	}
	// _partition_by_split  BVH.cu:285-304
	int partition(int start, int end, int axis, float pos) {
		int i = start, j = end;
		while (i < j) {
			const Box3& b = arr[i].box;
			float cen = (b.mx[axis] + b.mn[axis]) * 0.5f;
			if (cen < pos) i++; else std::swap(arr[i], arr[--j]);
		}
		return i;
	}
	// _build_bvh_rec2  BVH.cu:212-239.  The reference recurses forever when a split leaves one side
	// empty; here such a range falls back to the median split (documented deviation).
	int rec_sah(int start, int end) {
		Box3 bounds = partition_bounds(start, end);
		if (end - start == 1) return push_node(bounds, -1, start);
		int axis = 0; float split = 0.0f;
		find_split(start, end, bounds, axis, split);
		int mid = partition(start, end, axis, split);
		if (mid == start || mid == end) {
			int ax = longest_axis(bounds);
			std::sort(arr.begin() + start, arr.begin() + end,
			          [ax](const Item& a, const Item& b) { return a.box.mn[ax] < b.box.mn[ax]; });
			mid = (start + end) / 2;
		}
		int l = rec_sah(start, mid);
		int r = rec_sah(mid, end);
		return push_node(bounds, l, r);
	}
};
}  // namespace

static int build_bottom_up(const std::vector<Box3>& boxes, std::vector<rtb_bvh_node>& nodes, std::vector<int>& order, int& root) {
	// BuildBVH_BottomUp  BVH.cu:315-383: leaves first in input order, then repeatedly merge the pair
	// with the smallest surface_area(union) * hittable_count (first minimum in (a,b) scan order).
	struct Work { Box3 box; int count; int node; };
	std::vector<Work> work;
	nodes.clear(); order.clear();
	for (int i = 0; i < (int)boxes.size(); ++i) {
		rtb_bvh_node n; memcpy(n.bmin, boxes[i].mn, 12); memcpy(n.bmax, boxes[i].mx, 12);
		n.left_child_idx = -1; n.right_child_hittable_idx = i;
		order.push_back(i);
		work.push_back({boxes[i], 1, (int)nodes.size()});
		nodes.push_back(n);
	}
	while (work.size() > 1) {
		float best = FLT_MAX; int ai = 0, bi = 1;
		for (int a = 0; a < (int)work.size(); ++a) for (int b = a + 1; b < (int)work.size(); ++b) {
			Box3 u = work[a].box; grow(u, work[b].box);
			float cost = surface_area(u) * (work[a].count + work[b].count);
			if (cost < best) { ai = a; bi = b; best = cost; }
		}
		Box3 u = work[ai].box; grow(u, work[bi].box);
		rtb_bvh_node n; memcpy(n.bmin, u.mn, 12); memcpy(n.bmax, u.mx, 12);
		n.left_child_idx = work[ai].node; n.right_child_hittable_idx = work[bi].node;
		Work merged{u, work[ai].count + work[bi].count, (int)nodes.size()};
		work.erase(work.begin() + bi); work.erase(work.begin() + ai);
		work.push_back(merged);
		nodes.push_back(n);
	}
	root = work[0].node;
	return (int)nodes.size();
}

int build_bvh(const std::vector<Box3>& boxes, int builder, std::vector<rtb_bvh_node>& nodes, std::vector<int>& order, int& root) {
	if (boxes.empty()) return fail(RTB_ERR_INVALID, "build_bvh: no primitives");
	if (builder == RTB_BVH_BOTTOMUP) return build_bottom_up(boxes, nodes, order, root);
	Builder b; b.arr.resize(boxes.size());
	for (int i = 0; i < (int)boxes.size(); ++i) { b.arr[i].box = boxes[i]; b.arr[i].idx = i; }
	b.nodes.reserve(2 * boxes.size());
	if (builder == RTB_BVH_TOPDOWN_MEDIAN) root = b.rec_median(0, (int)boxes.size());
	else if (builder == RTB_BVH_TOPDOWN_SAH) root = b.rec_sah(0, (int)boxes.size());
	else return fail(RTB_ERR_INVALID, "build_bvh: unknown builder");
	nodes.swap(b.nodes);
	order.resize(boxes.size());
	for (int i = 0; i < (int)boxes.size(); ++i) order[i] = b.arr[i].idx;  // BVH.cu:174-177
	return (int)nodes.size();
}

// Binned SAH over centroid bounds (32 bins), leaves of one primitive, depth-capped: the quality
// builder for world BVHs that are not pinned to a reference topology.
int build_bvh_world_sah(const std::vector<Box3>& boxes, std::vector<rtb_bvh_node>& nodes, std::vector<int>& order, int& root) {
	if (boxes.empty()) return fail(RTB_ERR_INVALID, "build_bvh_world_sah: no primitives");
	const int n = (int)boxes.size();
	std::vector<int> idx(n); for (int i = 0; i < n; ++i) idx[i] = i;
	std::vector<float> cen(3 * (size_t)n);
	for (int i = 0; i < n; ++i) for (int a = 0; a < 3; ++a) cen[3 * (size_t)i + a] = 0.5f * (boxes[i].mn[a] + boxes[i].mx[a]);
	// Nodes are stored in post-order (children before their parent, root last, like the reference's builders).  A
	// subtree over k leaves then owns 2k - 1 consecutive slots starting at a base known before it is built (left child:
	// the parent's base; right child: past the left subtree), whatever the splits inside it are, so large subtrees are
	// built by concurrent tasks writing disjoint slot and index ranges: the same array as a serial build.
	nodes.assign(2 * (size_t)n - 1, rtb_bvh_node{});
	auto put = [&](int slot, const Box3& b, int l, int r) {
		rtb_bvh_node& nd = nodes[slot]; memcpy(nd.bmin, b.mn, 12); memcpy(nd.bmax, b.mx, 12); nd.left_child_idx = l; nd.right_child_hittable_idx = r;
		return slot;
	};
	const int NB = 32, MAX_DEPTH = 26, PARALLEL_MIN = 16384;
	const char* serial_env = getenv("RTB_FLATTEN_SERIAL");   // =1: build on the calling thread only (the result is the same)
	const bool serial = serial_env && serial_env[0] == '1';
	const int max_fork_depth = serial ? 0 : n >= 2 * PARALLEL_MIN ? std::min(6, (int)std::ceil(std::log2(std::max(2u, std::thread::hardware_concurrency())))) + 1 : 0;
	std::function<int(int, int, int, int)> rec = [&](int start, int end, int depth, int base) -> int {
		const int slot = base + 2 * (end - start) - 2;      // this subtree's root: last of its 2 (end - start) - 1 slots
		Box3 bounds = empty_box();
		for (int i = start; i < end; ++i) grow(bounds, boxes[idx[i]]);
		if (end - start == 1) return put(slot, bounds, -1, start);
		float cmn[3] = {INFINITY, INFINITY, INFINITY}, cmx[3] = {-INFINITY, -INFINITY, -INFINITY};
		for (int i = start; i < end; ++i) for (int a = 0; a < 3; ++a) {
			float c = cen[3 * (size_t)idx[i] + a]; cmn[a] = std::fmin(cmn[a], c); cmx[a] = std::fmax(cmx[a], c);
		}
		int best_axis = -1, best_bin = -1; float best_cost = INFINITY;
		if (depth < MAX_DEPTH && end - start > 2) {
			for (int a = 0; a < 3; ++a) {
				float ext = cmx[a] - cmn[a];
				if (!(ext > 0.0f)) continue;
				Box3 bb[NB]; int bc[NB];
				for (int b = 0; b < NB; ++b) { bb[b] = empty_box(); bc[b] = 0; }
				float scale = NB / ext;
				for (int i = start; i < end; ++i) {
					int b = (int)((cen[3 * (size_t)idx[i] + a] - cmn[a]) * scale); if (b >= NB) b = NB - 1; if (b < 0) b = 0;
					grow(bb[b], boxes[idx[i]]); bc[b]++;
				}
				float right_area[NB]; int right_cnt[NB];
				Box3 acc = empty_box(); int cnt = 0;
				for (int b = NB - 1; b > 0; --b) { grow(acc, bb[b]); cnt += bc[b]; right_area[b] = surface_area(acc); right_cnt[b] = cnt; }
				acc = empty_box(); cnt = 0;
				for (int b = 0; b < NB - 1; ++b) {
					grow(acc, bb[b]); cnt += bc[b];
					if (cnt == 0 || right_cnt[b + 1] == 0) continue;
					float cost = surface_area(acc) * cnt + right_area[b + 1] * right_cnt[b + 1];
					if (cost < best_cost) { best_cost = cost; best_axis = a; best_bin = b; }
				}
			}
		}
		int mid;
		if (best_axis >= 0) {
			float ext = cmx[best_axis] - cmn[best_axis], scale = NB / ext;
			auto it = std::partition(idx.begin() + start, idx.begin() + end, [&](int id) {
				int b = (int)((cen[3 * (size_t)id + best_axis] - cmn[best_axis]) * scale); if (b >= NB) b = NB - 1; if (b < 0) b = 0;
				return b <= best_bin;
			});
			mid = (int)(it - idx.begin());
		} else mid = start;
		if (mid == start || mid == end) {  // degenerate: balanced median on the widest centroid axis
			int ax = 0; float w = -1.0f;
			for (int a = 0; a < 3; ++a) if (cmx[a] - cmn[a] > w) { w = cmx[a] - cmn[a]; ax = a; }
			mid = (start + end) / 2;
			std::nth_element(idx.begin() + start, idx.begin() + mid, idx.begin() + end, [&](int x, int y) {
				float cx = cen[3 * (size_t)x + ax], cy = cen[3 * (size_t)y + ax];
				return cx < cy || (cx == cy && x < y);
			});
		}
		int l, r;
		if (depth < max_fork_depth && end - start >= 2 * PARALLEL_MIN && mid - start >= PARALLEL_MIN / 4 && end - mid >= PARALLEL_MIN / 4) {
			std::future<int> left = std::async(std::launch::async, [&rec, start, mid, depth, base] { return rec(start, mid, depth + 1, base); });
			r = rec(mid, end, depth + 1, base + 2 * (mid - start) - 1);
			l = left.get();
		} else {
			l = rec(start, mid, depth + 1, base);
			r = rec(mid, end, depth + 1, base + 2 * (mid - start) - 1);
		}
		return put(slot, bounds, l, r);
	};
	root = rec(0, n, 0, 0);
	order = idx;
	return (int)nodes.size();
}

int bvh_depth(const std::vector<rtb_bvh_node>& nodes, int root) {
	std::vector<std::pair<int, int>> st; st.push_back({root, 1}); int best = 0;
	while (!st.empty()) {
		auto [i, d] = st.back(); st.pop_back();
		best = std::max(best, d);
		if (nodes[i].left_child_idx != -1) { st.push_back({nodes[i].left_child_idx, d + 1}); st.push_back({nodes[i].right_child_hittable_idx, d + 1}); }
	}
	return best;
}

}  // namespace rtb

extern "C" int rtb_bvh_build(const float* aabbs, int n, int builder, rtb_bvh_node* nodes_out, int* order_out, int* root_out) {
	if (!aabbs || n <= 0 || !nodes_out || !order_out || !root_out) return fail(RTB_ERR_INVALID, "rtb_bvh_build: bad argument");
	std::vector<Box3> boxes(n);
	for (int i = 0; i < n; ++i) { memcpy(boxes[i].mn, aabbs + 6 * (size_t)i, 12); memcpy(boxes[i].mx, aabbs + 6 * (size_t)i + 3, 12); }
	std::vector<rtb_bvh_node> nodes; std::vector<int> order; int root = -1;
	int rc = build_bvh(boxes, builder, nodes, order, root);
	if (rc < 0) return rc;
	memcpy(nodes_out, nodes.data(), nodes.size() * sizeof(rtb_bvh_node));
	memcpy(order_out, order.data(), order.size() * sizeof(int));
	*root_out = root;
	return (int)nodes.size();
}

extern "C" int rtb_scene_world_bvh(const rtb_scene* s, rtb_bvh_node* nodes_out, int cap, int* root_out) {
	if (!s) return fail(RTB_ERR_INVALID, "rtb_scene_world_bvh: null scene");
	if (s->world_nodes.empty()) return fail(RTB_ERR_STATE, "rtb_scene_world_bvh: scene has not been flattened (rtb_renderer_set_scene / rtb_scene_flatten)");
	if (nodes_out) {
		if (cap < (int)s->world_nodes.size()) return fail(RTB_ERR_INVALID, "rtb_scene_world_bvh: buffer too small");
		memcpy(nodes_out, s->world_nodes.data(), s->world_nodes.size() * sizeof(rtb_bvh_node));
	}
	if (root_out) *root_out = s->world_root;
	return (int)s->world_nodes.size();
}

// ============================================================== flattener

namespace rtb {

namespace {
// Splits [0, n) over the host threads when the range is large enough to pay for starting them.
template <typename F>
void parallel_for(size_t n, F&& body) {
	const size_t workers = n < 65536 ? 1 : std::min<size_t>(16, std::max(1u, std::thread::hardware_concurrency()));
	if (workers <= 1) { body((size_t)0, n); return; }
	std::vector<std::thread> pool;
	const size_t chunk = (n + workers - 1) / workers;
	for (size_t w = 1; w < workers; ++w) {
		size_t a = std::min(n, w * chunk), b = std::min(n, a + chunk);
		if (a < b) pool.emplace_back([&body, a, b] { body(a, b); });
	}
	body((size_t)0, std::min(n, chunk));
	for (std::thread& t : pool) t.join();
}

struct Flattener {
	rtb_scene& s;
	FlatScene& out;
	// One item per logical primitive (= one BVH leaf); an item owns one or two 64-byte record slots.
	// Records live in one pool; rec_type tags the first slot of everything a hit can name (-1 = continuation slot).
	struct Item { int first; int nrec; int type; DevPrimInfo info; int attr = -1; };   // attr: index of the triangle's attributes
	std::vector<Item> items;
	std::vector<Box3> prim_boxes;
	std::vector<DevPrim> recs;
	std::vector<int> rec_type;
	bool box_as_quads = false;   // RTB_BOX_AS_QUADS=1: a box is six independent BVH leaves (the layout before PRIM_BOX)

	void emit(int type, const DevPrim& p, const Box3& b, int mat, int obj, const DevPrim* second = nullptr) {
		Item it{}; it.first = (int)recs.size(); it.nrec = 1; it.type = type; it.info.material = mat; it.info.object = obj;
		recs.push_back(p); rec_type.push_back(type);
		if (second) { recs.push_back(*second); rec_type.push_back(-1); it.nrec = 2; }
		items.push_back(it);
		prim_boxes.push_back(b);
	}
	static bool is_identity(const Xf& x) { return !x.rot && !x.tr; }
	static void put_xf(float* q, const Xf& x) {   // (cos, sin, off.x, off.y), (off.z, rotates ? 1 : 0, 0, 0)
		q[0] = x.rot ? x.c : 1.0f; q[1] = x.rot ? x.s : 0.0f; q[2] = x.off[0]; q[3] = x.off[1]; q[4] = x.off[2];
		q[5] = x.rot ? 1.0f : 0.0f;   // a translate-only instance must not run vectors through an identity rotation: fma(1, -0, 0 * z) is +0
	}
	// World bounds of an instanced primitive are computed with host rounding, the hit with the
	// kernel's ray transform: pad so the box always contains what the kernel can hit.
	static void pad_instance_box(Box3& b) {
		for (int i = 0; i < 3; ++i) {
			float m = std::fmax(std::fabs(b.mn[i]), std::fabs(b.mx[i]));
			float e = std::fmax(1e-4f, 4e-6f * m);
			b.mn[i] -= e; b.mx[i] += e;
		}
	}
	void emit_sphere(const rtbs_object& o, int id, const Xf& x) {
		float c[3]; x.point(o.f, c);
		DevPrim p{};
		const float rad = std::fabs(o.f[3]);   // (a negative radius - the book's hollow glass ball - turns the normal inside out, not the box)
		Box3 b; for (int i = 0; i < 3; ++i) { b.mn[i] = c[i] - rad; b.mx[i] = c[i] + rad; }
		if (is_identity(x)) {
			p.q[0] = c[0]; p.q[1] = c[1]; p.q[2] = c[2]; p.q[3] = o.f[3];
			emit(PRIM_SPHERE, p, b, o.mat, id);
		} else {
			p.q[0] = o.f[0]; p.q[1] = o.f[1]; p.q[2] = o.f[2]; p.q[3] = o.f[3];
			put_xf(p.q + 4, x); pad_instance_box(b);
			emit(PRIM_SPHERE | PRIM_XF, p, b, o.mat, id);
		}
	}
	void emit_moving_sphere(const rtbs_object& o, int id, const Xf& x) {
		float c0[3], c1[3]; x.point(o.f, c0); x.point(o.f + 4, c1);
		DevPrim p{};
		Box3 b;
		for (int i = 0; i < 3; ++i) {
			const float rad = std::fabs(o.f[3]);
			float a0 = c0[i] - rad, a1 = c1[i] - rad, b0 = c0[i] + rad, b1 = c1[i] + rad;
			b.mn[i] = (a1 < a0) ? a1 : a0; b.mx[i] = (b0 < b1) ? b1 : b0;
		}
		if (is_identity(x)) {
			p.q[0] = c0[0]; p.q[1] = c0[1]; p.q[2] = c0[2]; p.q[3] = o.f[3]; p.q[4] = c1[0]; p.q[5] = c1[1]; p.q[6] = c1[2];
			emit(PRIM_MOVING_SPHERE, p, b, o.mat, id);
		} else {
			p.q[0] = o.f[0]; p.q[1] = o.f[1]; p.q[2] = o.f[2]; p.q[3] = o.f[3]; p.q[4] = o.f[4]; p.q[5] = o.f[5]; p.q[6] = o.f[6];
			put_xf(p.q + 8, x); pad_instance_box(b);
			emit(PRIM_MOVING_SPHERE | PRIM_XF, p, b, o.mat, id);
		}
	}
	// book quad ctor, in the primitive's own frame: n = cross(u,v); normal = unit(n); D = dot(normal,Q); w = n / dot(n,n)
	static DevPrim planar_record(const float Q[3], const float u[3], const float v[3]) {
		rt::v3 U = rt::mk(u[0], u[1], u[2]), V = rt::mk(v[0], v[1], v[2]), QQ = rt::mk(Q[0], Q[1], Q[2]);
		rt::v3 n = rt::cross(U, V);
		rt::v3 N = rt::normalize(n);
		float D = rt::dot(N, QQ);
		rt::v3 w = rt::divs(n, rt::dot(n, n));
		DevPrim p{};
		p.q[0] = Q[0]; p.q[1] = Q[1]; p.q[2] = Q[2]; p.q[3] = D;
		p.q[4] = u[0]; p.q[5] = u[1]; p.q[6] = u[2]; p.q[7] = N.x;
		p.q[8] = v[0]; p.q[9] = v[1]; p.q[10] = v[2]; p.q[11] = N.y;
		p.q[12] = w.x; p.q[13] = w.y; p.q[14] = w.z; p.q[15] = N.z;
		return p;
	}
	static Box3 planar_box(int type, const float Q[3], const float u[3], const float v[3], const Xf& x) {
		float f[9]; memcpy(f, Q, 12); memcpy(f + 3, u, 12); memcpy(f + 6, v, 12);
		float pts[4][3]; quad_corners(f, pts);
		const int cnt = type == PRIM_QUAD ? 4 : 3;
		if (is_identity(x)) { Box3 b = box_of_points(pts, cnt); pad_to_minimum(b); return b; }
		float wp[4][3];
		for (int i = 0; i < cnt; ++i) x.point(pts[i], wp[i]);
		Box3 b = box_of_points(wp, cnt); pad_to_minimum(b); pad_instance_box(b);
		return b;
	}
	void emit_planar(int type, const float Q[3], const float u[3], const float v[3], int mat, int id, const Xf& x) {
		const DevPrim p = planar_record(Q, u, v);
		const Box3 b = planar_box(type, Q, u, v, x);
		if (is_identity(x)) {
			emit(type, p, b, mat, id);
		} else {
			DevPrim t{}; put_xf(t.q, x);          // second slot: the transform
			emit(type | PRIM_XF, p, b, mat, id, &t);
		}
	}
	void emit_box(const rtbs_object& o, int id, const Xf& x) {
		// book box(a,b): six quads with outward normals (front, right, back, left, top, bottom)
		const float* mn = o.f; const float* mx = o.f + 3;
		float dx[3] = {mx[0] - mn[0], 0, 0}, dy[3] = {0, mx[1] - mn[1], 0}, dz[3] = {0, 0, mx[2] - mn[2]};
		float ndx[3] = {-dx[0], -dx[1], -dx[2]}, ndz[3] = {-dz[0], -dz[1], -dz[2]};   // full negation (signed zeros as in -dx)
		const float q[6][3] = {{mn[0], mn[1], mx[2]}, {mx[0], mn[1], mx[2]}, {mx[0], mn[1], mn[2]}, {mn[0], mn[1], mn[2]}, {mn[0], mx[1], mx[2]}, {mn[0], mn[1], mn[2]}};
		const float* us[6] = {dx, ndz, ndx, dz, dx, dx};
		const float* vs[6] = {dy, dy, dy, dy, ndz, dz};
		if (box_as_quads) {
			for (int f = 0; f < 6; ++f) emit_planar(PRIM_QUAD, q[f], us[f], vs[f], o.mat, id, x);
			return;
		}
		// One BVH leaf: a (min, max) record the kernel uses to pick which faces the ray can hit, then the same six quad
		// records as above; the kernel runs the ordinary quad test on the picked ones and reports the hit on that quad.
		const bool inst = !is_identity(x);
		Item it{}; it.first = (int)recs.size(); it.type = inst ? (PRIM_BOX | PRIM_XF) : PRIM_BOX; it.info.material = o.mat; it.info.object = id;
		DevPrim t{}; if (inst) put_xf(t.q, x);
		DevPrim bp{};
		bp.q[0] = mn[0]; bp.q[1] = mn[1]; bp.q[2] = mn[2]; bp.q[3] = mx[0]; bp.q[4] = mx[1]; bp.q[5] = mx[2];
		recs.push_back(bp); rec_type.push_back(it.type);
		if (inst) { recs.push_back(t); rec_type.push_back(-1); }
		Box3 b = empty_box();
		for (int f = 0; f < 6; ++f) {
			recs.push_back(planar_record(q[f], us[f], vs[f])); rec_type.push_back(inst ? (PRIM_QUAD | PRIM_XF) : PRIM_QUAD);
			if (inst) { recs.push_back(t); rec_type.push_back(-1); }
			grow(b, planar_box(PRIM_QUAD, q[f], us[f], vs[f], x));
		}
		it.nrec = (int)recs.size() - it.first;
		items.push_back(it);
		prim_boxes.push_back(b);
	}
	// Resolve a medium boundary: SPHERE or BOX under any chain of translate / rotate_y.
	int emit_medium(const rtbs_object& med, int id, Xf x) {
		int cur = s.children[med.child_begin];
		for (int guard = 0; guard < 64; ++guard) {
			const rtbs_object& o = s.objects[cur];
			if (o.kind == RTB_OBJ_TRANSLATE) { x = compose_translate(x, o.f); cur = s.children[o.child_begin]; continue; }
			if (o.kind == RTB_OBJ_ROTATE_Y) { x = compose_rotate(x, o.f[1], o.f[2]); cur = s.children[o.child_begin]; continue; }
			int medium_index = out.n_media++;
			if (o.kind == RTB_OBJ_SPHERE) {
				float c[3]; x.point(o.f, c);
				DevPrim p{}; p.q[0] = c[0]; p.q[1] = c[1]; p.q[2] = c[2]; p.q[3] = o.f[3]; p.q[4] = med.f[1];
				p.q[5] = rt::u2f((uint32_t)medium_index);
				Box3 b; for (int i = 0; i < 3; ++i) { b.mn[i] = c[i] - std::fabs(o.f[3]); b.mx[i] = c[i] + std::fabs(o.f[3]); }
				emit(PRIM_MEDIUM_SPHERE, p, b, med.mat, id);
				return RTB_OK;
			}
			if (o.kind == RTB_OBJ_BOX) {
				DevPrim p{};
				p.q[0] = o.f[0]; p.q[1] = o.f[1]; p.q[2] = o.f[2]; p.q[3] = x.c;
				p.q[4] = o.f[3]; p.q[5] = o.f[4]; p.q[6] = o.f[5]; p.q[7] = x.s;
				p.q[8] = x.off[0]; p.q[9] = x.off[1]; p.q[10] = x.off[2]; p.q[11] = med.f[1];
				p.q[12] = rt::u2f((uint32_t)medium_index);
				float pts[8][3]; int k = 0;
				for (int i = 0; i < 2; ++i) for (int j = 0; j < 2; ++j) for (int l = 0; l < 2; ++l) {
					float c[3] = {i ? o.f[3] : o.f[0], j ? o.f[4] : o.f[1], l ? o.f[5] : o.f[2]};
					x.point(c, pts[k++]);
				}
				Box3 b = box_of_points(pts, 8); pad_to_minimum(b);
				emit(PRIM_MEDIUM_BOX, p, b, med.mat, id);
				return RTB_OK;
			}
			return fail(RTB_ERR_UNSUPPORTED, "constant_medium boundary must be a sphere or a box (optionally under translate / rotate_y)");
		}
		return fail(RTB_ERR_INVALID, "constant_medium boundary chain too deep");
	}
	static Xf compose_translate(const Xf& x, const float off[3]) {
		Xf r = x; float o[3]; x.point(off, o);  // world = X(p + off) => offset' = X(off)
		r.off[0] = o[0]; r.off[1] = o[1]; r.off[2] = o[2]; r.tr = true; return r;
	}
	static Xf compose_rotate(const Xf& x, float sn, float cs) {
		Xf r = x;
		if (x.rot) { r.c = x.c * cs - x.s * sn; r.s = x.s * cs + x.c * sn; }
		else { r.c = cs; r.s = sn; }
		r.rot = true; return r;
	}
	int walk(int id, const Xf& x, int depth) {
		if (depth > 64) return fail(RTB_ERR_INVALID, "object graph too deep / cyclic");
		const rtbs_object& o = s.objects[id];
		switch (o.kind) {
		case RTB_OBJ_SPHERE: emit_sphere(o, id, x); return RTB_OK;
		case RTB_OBJ_MOVING_SPHERE: emit_moving_sphere(o, id, x); return RTB_OK;
		case RTB_OBJ_QUAD: emit_planar(PRIM_QUAD, o.f, o.f + 3, o.f + 6, o.mat, id, x); return RTB_OK;
		case RTB_OBJ_TRIANGLE:
			emit_planar(PRIM_TRIANGLE, o.f, o.f + 3, o.f + 6, o.mat, id, x);
			if (o.aux > 0) {
				if ((size_t)o.aux > s.tri_attrs.size()) return fail(RTB_ERR_INVALID, "triangle " + std::to_string(id) + ": bad attribute index");
				items.back().attr = o.aux - 1;
			}
			return RTB_OK;
		case RTB_OBJ_BOX: emit_box(o, id, x); return RTB_OK;
		case RTB_OBJ_LIST: case RTB_OBJ_BVH: {
			for (int k = 0; k < o.child_count; ++k) { int rc = walk(s.children[o.child_begin + k], x, depth + 1); if (rc) return rc; }
			return RTB_OK;
		}
		case RTB_OBJ_TRANSLATE: return walk(s.children[o.child_begin], compose_translate(x, o.f), depth + 1);
		case RTB_OBJ_ROTATE_Y: return walk(s.children[o.child_begin], compose_rotate(x, o.f[1], o.f[2]), depth + 1);
		case RTB_OBJ_CONSTANT_MEDIUM: return emit_medium(o, id, x);
		}
		return fail(RTB_ERR_INVALID, "unknown object kind");
	}
};

// Sampled light `id` (DESIGN.md §5b): its translate / rotate_y chain composed into one world-from-object transform, the
// sphere or quad at its end as a world-space record (the SPHERE / QUAD layout of DevPrim) and its DevLightInfo.
int light_record(const rtb_scene& s, int id, DevPrim& rec, DevLightInfo& info) {
	if (id < 0 || id >= (int)s.objects.size()) return fail(RTB_ERR_INVALID, "sampled light: bad object id " + std::to_string(id));
	Xf x;
	int cur = id;
	for (int guard = 0; guard < 64; ++guard) {
		const rtbs_object& o = s.objects[cur];
		if (o.kind == RTB_OBJ_TRANSLATE) { x = Flattener::compose_translate(x, o.f); cur = s.children[o.child_begin]; continue; }
		if (o.kind == RTB_OBJ_ROTATE_Y) { x = Flattener::compose_rotate(x, o.f[1], o.f[2]); cur = s.children[o.child_begin]; continue; }
		rec = DevPrim{}; info = DevLightInfo{};
		if (o.kind == RTB_OBJ_SPHERE) {
			float c[3]; x.point(o.f, c);
			const float r = std::fabs(o.f[3]);
			if (!(r > 0.0f) || !std::isfinite(r)) return fail(RTB_ERR_INVALID, "sampled light " + std::to_string(id) + ": the sphere has no radius");
			rec.q[0] = c[0]; rec.q[1] = c[1]; rec.q[2] = c[2]; rec.q[3] = r;
			info.type = PRIM_SPHERE;
			return RTB_OK;
		}
		if (o.kind == RTB_OBJ_QUAD) {
			float Q[3], u[3], v[3]; x.point(o.f, Q); x.vec(o.f + 3, u); x.vec(o.f + 6, v);
			rec = Flattener::planar_record(Q, u, v);
			const rt::v3 n = rt::cross(rt::mk(u[0], u[1], u[2]), rt::mk(v[0], v[1], v[2]));
			const float area = sqrtf(rt::dot(n, n));
			if (!(area > 0.0f) || !std::isfinite(area)) return fail(RTB_ERR_INVALID, "sampled light " + std::to_string(id) + ": the quad has no area");
			info.type = PRIM_QUAD; info.area = area;
			return RTB_OK;
		}
		return fail(RTB_ERR_UNSUPPORTED, "sampled light " + std::to_string(id) +
		                                     ": only spheres and quads (optionally under translate / rotate_y) can be sampled");
	}
	return fail(RTB_ERR_INVALID, "sampled light " + std::to_string(id) + ": instance chain too deep");
}
}  // namespace

int flatten(rtb_scene& s, FlatScene& out, const GpuBuildContext* gpu) {
	if (s.root < 0) return fail(RTB_ERR_STATE, "scene has no root object (rtb_scene_set_root)");
	if (s.world_bvh_mode == RTB_WORLD_BVH_GPU_LBVH && !gpu)
		return fail(RTB_ERR_STATE, "RTB_WORLD_BVH_GPU_LBVH is built on a renderer's device: use rtb_renderer_set_scene / rtb_renderer_scene_stats");
	const auto t_start = std::chrono::steady_clock::now();
	const bool trace = getenv("RTB_LBVH_TRACE") != nullptr;
	auto t_lap = t_start;
	auto lap = [&](const char* what) {
		if (!trace) return;
		auto t1 = std::chrono::steady_clock::now();
		fprintf(stderr, "[flatten] %-12s %8.3f ms\n", what, std::chrono::duration<float, std::milli>(t1 - t_lap).count());
		t_lap = t1;
	};
	out = FlatScene();
	Flattener fl{s, out};
	fl.items.reserve(s.objects.size()); fl.prim_boxes.reserve(s.objects.size()); fl.recs.reserve(s.objects.size()); fl.rec_type.reserve(s.objects.size());
	{ const char* e = getenv("RTB_BOX_AS_QUADS"); fl.box_as_quads = e && e[0] == '1'; }
	Xf ident;
	int rc = fl.walk(s.root, ident, 0);
	if (rc) return rc;
	lap("walk");
	if (fl.items.empty()) return fail(RTB_ERR_INVALID, "scene has no primitives");
	if (fl.items.size() >= (1u << 26)) return fail(RTB_ERR_UNSUPPORTED, "too many primitives");

	// Participating media are tested BEFORE the BVH walk (at most 8, the largest first): a ray inside a
	// medium then starts traversal with a tight t bound instead of wading through every box that
	// happens to contain its origin.  Closest-hit results do not depend on the test order.
	{
		std::vector<int> media;
		for (size_t i = 0; i < fl.items.size(); ++i) if (fl.items[i].type == PRIM_MEDIUM_SPHERE || fl.items[i].type == PRIM_MEDIUM_BOX) media.push_back((int)i);
		std::stable_sort(media.begin(), media.end(), [&](int a, int b) { return surface_area(fl.prim_boxes[a]) > surface_area(fl.prim_boxes[b]); });
		if (media.size() > 8) media.resize(8);
		if (!media.empty()) {
		std::vector<char> is_pre(fl.items.size(), 0);
		for (int m : media) is_pre[m] = 1;
		std::vector<Flattener::Item> rest; std::vector<Box3> rest_boxes;
		for (int m : media) {
			const Flattener::Item& it = fl.items[m];
			out.pre_list.push_back((int32_t)(((int)out.prims.size() << RTB_LEAF_TYPE_BITS) | it.type));
			for (int k = 0; k < it.nrec; ++k) { out.prims.push_back(fl.recs[it.first + k]); out.prim_info.push_back(it.info); out.prim_type.push_back(fl.rec_type[it.first + k]); }
		}
		rest.reserve(fl.items.size()); rest_boxes.reserve(fl.items.size());
		for (size_t i = 0; i < fl.items.size(); ++i) if (!is_pre[i]) { rest.push_back(fl.items[i]); rest_boxes.push_back(fl.prim_boxes[i]); }
		fl.items.swap(rest); fl.prim_boxes.swap(rest_boxes);
		}
	}
	if (fl.items.empty()) {   // nothing but pre-tested media: no BVH at all
		out.bvh_empty = 1; out.root_ref = 0; out.max_depth_nodes = 0;
		s.world_nodes.clear(); s.world_root = -1;
	}

	// World BVH: a quality SAH tree by default; with RTB_WORLD_BVH_AS_BUILT a root that is a reference BVH keeps the
	// reference builder (and therefore its exact node / primitive order).  Closest hits are the same either way.

	const rtbs_object& root = s.objects[s.root];
	if (!out.bvh_empty) {
	std::vector<rtb_bvh_node> nodes; std::vector<int> order; int root_idx = -1;
	const int STACK_LIMIT = RTB_TREE_DEPTH_NORMAL;
	bool built = false;
	int depth = 0;
	lap("media");
	const auto t_build = std::chrono::steady_clock::now();
	if (root.kind == RTB_OBJ_BVH && s.world_bvh_mode == RTB_WORLD_BVH_AS_BUILT) {
		rc = build_bvh(fl.prim_boxes, root.aux, nodes, order, root_idx);
		if (rc < 0) return rc;
		depth = bvh_depth(nodes, root_idx);
		built = depth <= STACK_LIMIT;
		out.builder = RTB_WORLD_BVH_AS_BUILT;
	} else if (s.world_bvh_mode == RTB_WORLD_BVH_GPU_LBVH) {
		rc = build_bvh_lbvh_gpu(fl.prim_boxes, nodes, order, root_idx, *gpu);
		if (rc < 0) return rc;
		depth = bvh_depth(nodes, root_idx);
		built = depth <= RTB_TREE_DEPTH_MAX;
		out.builder = RTB_WORLD_BVH_GPU_LBVH;
	}
	if (!built) {
		rc = build_bvh_world_sah(fl.prim_boxes, nodes, order, root_idx);
		if (rc < 0) return rc;
		out.builder = RTB_WORLD_BVH_QUALITY;
		depth = bvh_depth(nodes, root_idx);
		if (depth > STACK_LIMIT) {
			rc = build_bvh(fl.prim_boxes, RTB_BVH_TOPDOWN_MEDIAN, nodes, order, root_idx);
			if (rc < 0) return rc;
			out.builder = RTB_BUILDER_MEDIAN_FALLBACK;
			depth = bvh_depth(nodes, root_idx);
		}
	}
	out.bvh_build_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_build).count();
	out.max_depth_nodes = depth;
	out.n_items = (int32_t)order.size();
	lap("bvh");

	// Lay the records out in BVH leaf order (Factory::hittables, BVH.cu:174-177); a leaf refers to
	// the first record slot of its item.
	std::vector<int> slot_of(order.size()), type_of(order.size());
	{
		size_t slots = out.prims.size();
		for (size_t i = 0; i < order.size(); ++i) { const Flattener::Item& it = fl.items[order[i]]; slot_of[i] = (int)slots; type_of[i] = it.type; slots += it.nrec; }
		out.prims.resize(slots); out.prim_info.resize(slots); out.prim_type.resize(slots);
	}
	parallel_for(order.size(), [&](size_t a, size_t b) {
		for (size_t i = a; i < b; ++i) {
			const Flattener::Item& it = fl.items[order[i]];
			for (int k = 0; k < it.nrec; ++k) { out.prims[slot_of[i] + k] = fl.recs[it.first + k]; out.prim_info[slot_of[i] + k] = it.info; out.prim_type[slot_of[i] + k] = fl.rec_type[it.first + k]; }
		}
	});
	if (out.prims.size() >= (1u << (31 - RTB_LEAF_TYPE_BITS))) return fail(RTB_ERR_UNSUPPORTED, "too many primitive record slots for a leaf reference (2^27)");
	// Triangle attributes (DESIGN.md §5e): the records, and per slot the index of its record (-1: none).  The primitive
	// records and the tree stay those of the same scene without attributes.
	if (!s.tri_attrs.empty()) {
		out.attr_slot.assign(out.prims.size(), -1);
		for (size_t i = 0; i < order.size(); ++i) out.attr_slot[slot_of[i]] = fl.items[order[i]].attr;
		out.tri_attr.resize(s.tri_attrs.size());
		for (size_t k = 0; k < s.tri_attrs.size(); ++k) {
			const rtbs_tri_attr& a = s.tri_attrs[k]; float* q = out.tri_attr[k].q;
			for (int c = 0; c < 3; ++c) { q[4 * c] = a.n[c][0]; q[4 * c + 1] = a.n[c][1]; q[4 * c + 2] = a.n[c][2]; }
			q[3] = a.uv[0][0]; q[7] = a.uv[0][1]; q[11] = a.uv[1][0];
			q[12] = a.uv[1][1]; q[13] = a.uv[2][0]; q[14] = a.uv[2][1]; q[15] = rt::u2f((uint32_t)a.flags);
		}
	}
	lap("layout");

	// Wide layout: one 64-byte record per inner node carrying both children's boxes, numbered in
	// depth-first pre-order (root = 0) so the near part of a subtree is contiguous.
	auto leaf_ref = [&](int node) { int item = nodes[node].right_child_hittable_idx; return make_leaf_ref(slot_of[item], type_of[item]); };
	if (nodes[root_idx].left_child_idx == -1) {
		out.root_ref = leaf_ref(root_idx);
	} else {
		std::vector<int> dev_index(nodes.size(), -1);
		std::vector<int> stack; stack.push_back(root_idx); int next = 0;
		std::vector<int> inner_order;
		while (!stack.empty()) {
			int i = stack.back(); stack.pop_back();
			if (nodes[i].left_child_idx == -1) continue;
			dev_index[i] = next++; inner_order.push_back(i);
			stack.push_back(nodes[i].right_child_hittable_idx);
			stack.push_back(nodes[i].left_child_idx);
		}
		out.nodes.resize(inner_order.size());
		auto ref_of = [&](int i) { return nodes[i].left_child_idx == -1 ? leaf_ref(i) : dev_index[i]; };
		parallel_for(inner_order.size(), [&](size_t a, size_t b) {
		for (size_t at = a; at < b; ++at) {
			const int i = inner_order[at];
			const rtb_bvh_node& l = nodes[nodes[i].left_child_idx];
			const rtb_bvh_node& r = nodes[nodes[i].right_child_hittable_idx];
			DevNode& d = out.nodes[dev_index[i]];
			// each child box as (min, extent): the kernel forms both slab planes with FMAs, near/far chosen by
			// the ray's direction signs.  The extent is rounded up (and min + extent >= max re-checked) so the
			// box the kernel sees always contains the exact one.
			auto put_box = [](float* f, const rtb_bvh_node& b) {
				for (int k = 0; k < 3; ++k) {
					float mn = b.bmin[k], ext = (b.bmax[k] - mn) * 1.000001f;
					if (!(ext >= 0.0f)) ext = 0.0f;
					while (mn + ext < b.bmax[k]) ext = std::nextafter(ext * 1.000001f + 1e-30f, INFINITY);
					f[k] = mn; f[3 + k] = ext;
				}
			};
#if RTB_NODE_PAIRED
			float lb[6], rb[6]; put_box(lb, l); put_box(rb, r);
			d.f[0] = lb[0]; d.f[1] = lb[1]; d.f[2] = lb[3]; d.f[3] = lb[4];
			d.f[4] = rb[0]; d.f[5] = rb[1]; d.f[6] = rb[3]; d.f[7] = rb[4];
			d.f[8] = lb[2]; d.f[9] = rb[2]; d.f[10] = lb[5]; d.f[11] = rb[5];
#else
			put_box(d.f, l); put_box(d.f + 6, r);
#endif
			d.left = ref_of(nodes[i].left_child_idx); d.right = ref_of(nodes[i].right_child_hittable_idx); d.pad0 = d.pad1 = 0;
		}
		});
		out.root_ref = 0;
	}
	for (int k = 0; k < 3; ++k) { out.world_min[k] = nodes[root_idx].bmin[k]; out.world_max[k] = nodes[root_idx].bmax[k]; }
	// The ray-binning grid spans the centres of the primitives' boxes, not their extents: one huge primitive (a
	// 1000-unit ground sphere under a scene a few units wide) must not decide the cell size.
	for (int k = 0; k < 3; ++k) { out.bin_min[k] = INFINITY; out.bin_max[k] = -INFINITY; }
	for (const Box3& b : fl.prim_boxes)
		for (int k = 0; k < 3; ++k) { const float c = 0.5f * (b.mn[k] + b.mx[k]); out.bin_min[k] = std::min(out.bin_min[k], c); out.bin_max[k] = std::max(out.bin_max[k], c); }
	for (int k = 0; k < 3; ++k) {   // a margin of 5 %, and never thinner than a thousandth of the largest side
		const float ext = out.bin_max[k] - out.bin_min[k];
		out.bin_min[k] -= 0.05f * ext; out.bin_max[k] += 0.05f * ext;
	}
	{
		const float widest = std::max(std::max(out.bin_max[0] - out.bin_min[0], out.bin_max[1] - out.bin_min[1]), out.bin_max[2] - out.bin_min[2]);
		for (int k = 0; k < 3; ++k) if (out.bin_max[k] - out.bin_min[k] < 1e-3f * widest || !(out.bin_max[k] > out.bin_min[k])) { out.bin_min[k] -= 0.5e-3f * widest + 1e-6f; out.bin_max[k] += 0.5e-3f * widest + 1e-6f; }
	}
	s.world_nodes = std::move(nodes); s.world_root = root_idx;

	}

	lap("wide");
	// Materials / textures.
	out.materials.resize(s.materials.size());
	for (size_t i = 0; i < s.materials.size(); ++i) {
		const rtbs_material& m = s.materials[i]; DevMaterial& d = out.materials[i];
		d.kind = m.kind; d.tex = m.tex; d.param = m.param; d.pad = s.mat_alpha[i];   // the GGX width (0 unless rough)
		d.albedo[0] = m.albedo[0]; d.albedo[1] = m.albedo[1]; d.albedo[2] = m.albedo[2]; d.albedo[3] = 0.0f;
	}
	out.textures.resize(s.textures.size());
	for (size_t i = 0; i < s.textures.size(); ++i) {
		const rtbs_texture& t = s.textures[i]; DevTexture& d = out.textures[i];
		d.kind = t.kind; d.even = t.even; d.odd = t.odd;
		d.scale = (t.kind == RTB_TEX_CHECKER) ? 1.0f / t.scale : t.scale;  // checker_texture ctor: inv_scale(1.0f/scale)
		d.rgb[0] = t.rgb[0]; d.rgb[1] = t.rgb[1]; d.rgb[2] = t.rgb[2]; d.rgb[3] = 0.0f;
		d.width = t.width; d.height = t.height; d.blob_offset = t.blob_offset; d.pad = 0;
	}
	out.blob = s.blob;
	for (int id : s.sampled_lights) {
		DevPrim rec; DevLightInfo info;
		rc = light_record(s, id, rec, info);
		if (rc) return rc;
		out.lights.push_back(rec); out.light_info.push_back(info);
	}
	if (s.env_width > 0) {
		build_env_tables(s.env_rgb.data(), s.env_width, s.env_height, out.env, out.env_cdf);
		out.env_width = s.env_width; out.env_height = s.env_height; out.env_sample = (s.env_flags & RTB_ENV_SAMPLE) ? 1 : 0;
	}
	out.background_mode = s.background_mode;
	memcpy(out.background, s.background, 12);
	out.flatten_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_start).count();
	return RTB_OK;
}

}  // namespace rtb

extern "C" int rtb_scene_flatten_stats(rtb_scene* s, int32_t out4[4]) {
	if (!s || !out4) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_flatten_stats: null argument");
	rtb::FlatScene fs;
	int rc = rtb::flatten(*s, fs);
	if (rc) return rc;
	out4[0] = (int32_t)((s->world_nodes.size() + 1) / 2); out4[1] = (int32_t)fs.prims.size();
	out4[2] = (int32_t)fs.nodes.size(); out4[3] = fs.max_depth_nodes;
	return RTB_OK;
}

extern "C" int rtb_scene_flatten_hash(rtb_scene* s, uint64_t* hash_out) {
	if (!s || !hash_out) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_flatten_hash: null argument");
	rtb::FlatScene fs;
	int rc = rtb::flatten(*s, fs);
	if (rc) return rc;
	uint64_t h = 1469598103934665603ull;
	auto mix = [&h](const void* p, size_t n) { const uint8_t* b = static_cast<const uint8_t*>(p); for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; } };
	if (!fs.nodes.empty()) mix(fs.nodes.data(), fs.nodes.size() * sizeof(rtb::DevNode));
	if (!fs.prims.empty()) mix(fs.prims.data(), fs.prims.size() * sizeof(rtb::DevPrim));
	if (!fs.prim_info.empty()) mix(fs.prim_info.data(), fs.prim_info.size() * sizeof(rtb::DevPrimInfo));
	if (!fs.prim_type.empty()) mix(fs.prim_type.data(), fs.prim_type.size() * sizeof(fs.prim_type[0]));
	if (!fs.pre_list.empty()) mix(fs.pre_list.data(), fs.pre_list.size() * sizeof(fs.pre_list[0]));
	mix(&fs.root_ref, sizeof fs.root_ref);
	if (!fs.lights.empty()) {   // (only then: the hashes of scenes without sampled lights stay what they were)
		mix(fs.lights.data(), fs.lights.size() * sizeof(rtb::DevPrim));
		mix(fs.light_info.data(), fs.light_info.size() * sizeof(rtb::DevLightInfo));
	}
	if (!fs.env.empty()) {      // (likewise for the environment map)
		const int32_t dims[3] = {fs.env_width, fs.env_height, fs.env_sample};
		mix(dims, sizeof dims);
		mix(fs.env.data(), fs.env.size() * sizeof(rtb::DevEnvTexel));
		mix(fs.env_cdf.data(), fs.env_cdf.size() * sizeof(float));
	}
	if (!fs.tri_attr.empty()) { // (likewise for triangle attributes)
		mix(fs.tri_attr.data(), fs.tri_attr.size() * sizeof(rtb::DevTriAttr));
		mix(fs.attr_slot.data(), fs.attr_slot.size() * sizeof(int32_t));
	}
	if (s->has_rough()) {       // (likewise for the GGX widths)
		for (const rtb::DevMaterial& m : fs.materials) mix(&m.pad, sizeof m.pad);
	}
	*hash_out = h;
	return RTB_OK;
}

extern "C" int rtb_scene_set_sampled_lights(rtb_scene* s, const int* objects, int n) {
	if (!s) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_sampled_lights: null scene");
	if (n < 0 || n > RTB_MAX_SAMPLED_LIGHTS) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_sampled_lights: n must be in [0, " + std::to_string(RTB_MAX_SAMPLED_LIGHTS) + "]");
	if (n > 0 && !objects) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_sampled_lights: null object list");
	for (int i = 0; i < n; ++i) {   // validate everything first: a refused list leaves the scene as it was
		rtb::DevPrim rec; rtb::DevLightInfo info;
		const int rc = rtb::light_record(*s, objects[i], rec, info);
		if (rc) return rc;
	}
	s->sampled_lights.assign(objects, objects + n);
	s->version++;
	return RTB_OK;
}

// Environment map (DESIGN.md §5d, "Sampling").  Weights luminance(texel) * sin(theta of the row centre) in double; the CDFs
// are prefix sums over the total (marginal) or the row sum (conditional), stored as float with the last entry exactly 1.
// A texel's probability is defined from the stored floats, so that the sampler and the pdf agree.
namespace {
double env_row_sin(int j, int H) { return std::sin(3.14159265358979323846 * (j + 0.5) / H); }
double env_luminance(const float* px) { return 0.2126 * px[0] + 0.7152 * px[1] + 0.0722 * px[2]; }
}  // namespace

double rtb::env_weight_sum(const float* rgb, int W, int H) {
	double total = 0.0;
	for (int j = 0; j < H; ++j) {
		const double st = env_row_sin(j, H);
		const float* px = rgb + (size_t)j * W * 3;
		double acc = 0.0;
		for (int i = 0; i < W; ++i) acc += env_luminance(px + 3 * i) * st;
		total += acc;
	}
	return total;
}

void rtb::build_env_tables(const float* rgb, int W, int H, std::vector<DevEnvTexel>& texels, std::vector<float>& cdf) {
	const double kPi = 3.14159265358979323846;
	std::vector<double> row(H, 0.0), pre(W);
	texels.assign((size_t)W * H, DevEnvTexel{});
	cdf.assign((size_t)(H + 1) + (size_t)H * (W + 1), 0.0f);
	float* cm = cdf.data();
	for (int j = 0; j < H; ++j) {
		const double st = env_row_sin(j, H);
		const float* px = rgb + (size_t)j * W * 3;
		double acc = 0.0;
		for (int i = 0; i < W; ++i) { acc += env_luminance(px + 3 * i) * st; pre[i] = acc; }
		row[j] = acc;
		float* cc = cm + (H + 1) + (size_t)j * (W + 1);
		for (int i = 0; i + 1 < W; ++i) cc[i + 1] = acc > 0.0 ? (float)(pre[i] / acc) : (float)((double)(i + 1) / W);   // (a row of weight 0 is never sampled)
		cc[0] = 0.0f; cc[W] = 1.0f;
	}
	double total = 0.0;
	for (int j = 0; j < H; ++j) total += row[j];
	if (total > 0.0) {
		double acc = 0.0;
		for (int j = 0; j + 1 < H; ++j) { acc += row[j]; cm[j + 1] = (float)(acc / total); }
	} else {
		for (int j = 0; j + 1 < H; ++j) cm[j + 1] = (float)((double)(j + 1) / H);
	}
	cm[0] = 0.0f; cm[H] = 1.0f;
	const double norm = (double)W * (double)H / (2.0 * kPi * kPi);
	for (int j = 0; j < H; ++j) {
		const double pj = total > 0.0 ? (double)cm[j + 1] - (double)cm[j] : 0.0;
		const float* cc = cm + (H + 1) + (size_t)j * (W + 1);
		for (int i = 0; i < W; ++i) {
			DevEnvTexel& t = texels[(size_t)j * W + i];
			const float* px = rgb + ((size_t)j * W + i) * 3;
			t.r = px[0]; t.g = px[1]; t.b = px[2];
			t.pdf = (float)(pj * ((double)cc[i + 1] - (double)cc[i]) * norm);
		}
	}
}

extern "C" int rtb_scene_set_environment(rtb_scene* s, const float* rgb, int width, int height, const float scale[3], int flags) {
	if (!s) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: null scene");
	if ((flags & ~RTB_ENV_SAMPLE) != 0) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: unknown flags");
	if (!rgb && width == 0 && height == 0) {   // clear: the background applies again
		s->env_rgb.clear(); s->env_rgb.shrink_to_fit();
		s->env_width = s->env_height = s->env_flags = 0;
		s->env_scale[0] = s->env_scale[1] = s->env_scale[2] = 1.0f;
		s->version++;
		return RTB_OK;
	}
	if (!rgb) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: null texels (clear with width = height = 0)");
	if (width < 1 || width > RTB_ENV_MAX_SIZE || height < 1 || height > RTB_ENV_MAX_SIZE || (int64_t)width * height > (int64_t(1) << 24))
		return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: width and height must be in [1, 16384] with width x height <= 2^24");
	const float one[3] = {1.0f, 1.0f, 1.0f};
	const float* sc = scale ? scale : one;
	for (int c = 0; c < 3; ++c)
		if (!(sc[c] >= 0.0f) || !std::isfinite(sc[c])) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: scale must be finite and >= 0");
	const size_t n = (size_t)width * height * 3;
	std::vector<float> scaled(n);
	for (size_t k = 0; k < n; ++k) {
		const float v = rgb[k];
		if (!(v >= 0.0f) || !std::isfinite(v))
			return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: texel " + std::to_string(k / 3) + " is negative, NaN or infinite");
		scaled[k] = v * sc[k % 3];
		if (!std::isfinite(scaled[k])) return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: texel " + std::to_string(k / 3) + " overflows when scaled");
	}
	if ((flags & RTB_ENV_SAMPLE) && !(rtb::env_weight_sum(scaled.data(), width, height) > 0.0))   // (the total the flattener's tables divide by)
			return rtb::fail(RTB_ERR_INVALID, "rtb_scene_set_environment: RTB_ENV_SAMPLE on a map whose sampling weights are all zero");
	s->env_rgb.swap(scaled);
	s->env_width = width; s->env_height = height; s->env_flags = flags;
	memcpy(s->env_scale, sc, 12);
	s->version++;
	return RTB_OK;
}

// ============================================================== cameras (cu_Cameras.cuh ctors restated, host arithmetic)

namespace {
struct H3 { float x, y, z; };
H3 hsub(H3 a, H3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
H3 hmul(H3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
H3 hcross(H3 x, H3 y) { return {x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y}; }  // glm::cross
H3 hnormalize(H3 v) { float d = v.x * v.x + v.y * v.y + v.z * v.z; return hmul(v, 1.0f / std::sqrt(d)); }   // glm::normalize
void put3(float* d, H3 v) { d[0] = v.x; d[1] = v.y; d[2] = v.z; }
H3 get3(const float* p) { return {p[0], p[1], p[2]}; }
}  // namespace

extern "C" {

int rtb_camera_pinhole(rtb_camera* c, const float lf[3], const float la[3], const float up[3], float vfov, float aspect) {
	int rc = rtb_camera_motion(c, lf, la, up, vfov, aspect, 0.0f, 0.0f);
	if (rc) return rc;
	c->kind = RTB_CAM_PINHOLE;
	return RTB_OK;
}
int rtb_camera_motion(rtb_camera* c, const float lf[3], const float la[3], const float up[3], float vfov, float aspect, float t0, float t1) {
	if (!c || !lf || !la || !up) return fail(RTB_ERR_INVALID, "rtb_camera_motion: null argument");
	memset(c, 0, sizeof *c);
	c->kind = RTB_CAM_MOTION; c->t0 = t0; c->t1 = t1;
	float theta = vfov * 0.01745329251994329576923690768489f;
	float vh = tanf(theta * 0.5f), vw = vh * aspect;
	H3 w = hnormalize(hsub(get3(la), get3(lf)));
	H3 u = hmul(hnormalize(hcross(get3(up), w)), vw);
	H3 v = hmul(hnormalize(hcross(w, u)), vh);
	put3(c->o, get3(lf)); put3(c->u, u); put3(c->v, v); put3(c->w, w);
	c->viewport_width = vw; c->viewport_height = vh; c->focus_dist = 1.0f;
	return RTB_OK;
}
int rtb_camera_defocus(rtb_camera* c, const float lf[3], const float la[3], const float up[3], float vfov, float aspect,
                       float aperture, float focus_dist, float t0, float t1) {
	if (!c || !lf || !la || !up) return fail(RTB_ERR_INVALID, "rtb_camera_defocus: null argument");
	memset(c, 0, sizeof *c);
	c->kind = RTB_CAM_DEFOCUS; c->t0 = t0; c->t1 = t1;
	float theta = vfov * 0.01745329251994329576923690768489f;
	c->viewport_height = tanf(theta * 0.5f); c->viewport_width = c->viewport_height * aspect;
	H3 w = hnormalize(hsub(get3(la), get3(lf)));
	H3 u = hnormalize(hcross(get3(up), w));
	H3 v = hnormalize(hcross(w, u));
	put3(c->o, get3(lf)); put3(c->u, u); put3(c->v, v); put3(c->w, w);
	c->lens_radius = aperture * 0.5f; c->focus_dist = focus_dist;
	return RTB_OK;
}

}  // extern "C"
