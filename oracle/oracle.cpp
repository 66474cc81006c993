// oracle/oracle.cpp — TEST INFRASTRUCTURE: CPU restatement of the reference's path-tracing hot path.
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
// this library.  It evaluates the scene object graph recursively, the way the reference's device
// object model does, and shares nothing with the product but the RTBS scene blob format.
//
// Reference code followed (paths relative to the reference checkout):
//   integrator        sample_world / render_kernel            main/src/Renderer.cu:139-217
//   flat BVH          BVH::ClosestIntersection                main/src/rt_engine/geometry/BVH.cu:54-106
//   BVH builders      BVH_Handle::Factory                     main/src/rt_engine/geometry/BVH.cu:166-383
//   slab test         aabb::intersects                        main/src/rt_engine/geometry/aabb.cuh:30-44
//   spheres           _sphere_closest_intersection            main/src/rt_engine/geometry/SphereHittable.cuh:15-33
//                     Sphere/MovingSphereHittable             main/src/rt_engine/geometry/SphereHittable.cu:43-102
//   list              HittableList::ClosestIntersection       main/src/rt_engine/geometry/HittableList.cuh:21-34
//   materials         Lambertian/Metal/Dielectric             main/src/rt_engine/shaders/cu_materials.cuh:17-144
//   textures          solid / checker                         main/src/rt_engine/shaders/cu_Textures.cuh:9-40
//   cameras           sample_ray                              main/src/rt_engine/shaders/cu_Cameras.cuh:27-30,54-64,87-89
//   samplers          cuRandomInUnit / cuRandomOnUnit         main/src/utilities/glm_utils.h:84-98
//   XORWOW            curand_init / curand / curand_uniform   /usr/local/cuda/include/curand_kernel.h:800-826,863-874
// Quads, boxes, translate, rotate_y, constant_medium, diffuse_light, isotropic, image and noise
// textures are NOT in the reference; they follow "Ray Tracing: The Next Week" (SURVEY.md App. B) in
// the reference's idiom (un-normalised directions, t >= 0, origin offset by d*0.001).
#include "oracle.h"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cstdio>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../include/rtb_scene_format.h"
#include "omath.h"

using namespace orc;

namespace {

thread_local std::string g_err;

const float MISS_DIST = 3.402823466e+38F;  // _MISS_DIST  ray_data.cuh:17

struct Ray {
	V3 o, d; float time;
	Ray() : o(), d(0, 0, 1), time(0) {}
	Ray(V3 o_, V3 d_, float t_ = 0.0f) : o(o_), d(d_), time(t_) {}
	V3 at(float t) const { return fma3(d, t, o); }
};

struct Box {
	V3 mn, mx;
	Box() : mn(1e9f, 1e9f, 1e9f), mx(-1e9f, -1e9f, -1e9f) {}     // aabb()  aabb.cuh:17
	Box(V3 a, V3 b) : mn(a), mx(b) {}
	void grow(const Box& b) {                                      // operator+=  aabb.cuh:24 (glm::min / glm::max)
		mn = V3(b.mn.x < mn.x ? b.mn.x : mn.x, b.mn.y < mn.y ? b.mn.y : mn.y, b.mn.z < mn.z ? b.mn.z : mn.z);
		mx = V3(mx.x < b.mx.x ? b.mx.x : mx.x, mx.y < b.mx.y ? b.mx.y : mx.y, mx.z < b.mx.z ? b.mx.z : mx.z);
	}
	// aabb::intersects  aabb.cuh:30-44 — literal: divides by d per call, glm::min/max component selects
	bool intersects(const Ray& r, float ray_max, float& dist) const {
		float bmin[3] = {(mn.x - r.o.x) / r.d.x, (mn.y - r.o.y) / r.d.y, (mn.z - r.o.z) / r.d.z};
		float bmax[3] = {(mx.x - r.o.x) / r.d.x, (mx.y - r.o.y) / r.d.y, (mx.z - r.o.z) / r.d.z};
		float lo[3], hi[3];
		for (int i = 0; i < 3; ++i) {
			lo[i] = (bmax[i] < bmin[i]) ? bmax[i] : bmin[i];   // glm::min(x,y) = (y < x) ? y : x
			hi[i] = (bmin[i] < bmax[i]) ? bmax[i] : bmin[i];   // glm::max(x,y) = (x < y) ? y : x
		}
		float tmin = std::max(std::max(lo[0], lo[1]), lo[2]);  // compMax  gtx/component_wise.inl
		float tmax = std::min(std::min(hi[0], hi[1]), hi[2]);  // compMin
		bool hit = tmin <= tmax && tmin < ray_max && tmax > 0;
		if (hit) dist = tmin;
		return hit;
	}
	bool intersects(const Ray& r, float ray_max) const { float d; return intersects(r, ray_max, d); }
	int longest_axis() const {                                     // aabb.cuh:46-53
		float sx = std::fabs(mx.x - mn.x), sy = std::fabs(mx.y - mn.y), sz = std::fabs(mx.z - mn.z);
		if (sx > sy) return sx > sz ? 0 : 2;
		return sy > sz ? 1 : 2;
	}
	float surface_area() const {                                   // aabb.cuh:55-64
		float sx = mx.x - mn.x, sy = mx.y - mn.y, sz = mx.z - mn.z;
		if (sx < 0 || sy < 0 || sz < 0) return 0.0f;
		float cost = 0.0f; cost += sx * sy; cost += sx * sz; cost += sy * sz;
		return 2.0f * cost;
	}
	float centroid(int a) const { return (mx[a] + mn[a]) * 0.5f; } // centeroid  aabb.cuh:66-68
};

void pad_box(Box& b) {   // book aabb::pad_to_minimums
	const float delta = 0.0001f;
	float mn[3] = {b.mn.x, b.mn.y, b.mn.z}, mx[3] = {b.mx.x, b.mx.y, b.mx.z};
	for (int i = 0; i < 3; ++i) if (mx[i] - mn[i] < delta) { mn[i] -= delta * 0.5f; mx[i] += delta * 0.5f; }
	b.mn = V3(mn[0], mn[1], mn[2]); b.mx = V3(mx[0], mx[1], mx[2]);
}

// ---------------------------------------------------------------- BVH builders (independent restatement)

struct BItem { Box box; int idx; };

struct BvhBuild {
	std::vector<BItem> arr;
	std::vector<rtb_bvh_node> nodes;
	Box range_bounds(int s, int e) const { Box b; for (int i = s; i < e; ++i) b.grow(arr[i].box); return b; }   // BVH.cu:306-312
	int emit(const Box& b, int l, int r) {
		rtb_bvh_node n;
		n.bmin[0] = b.mn.x; n.bmin[1] = b.mn.y; n.bmin[2] = b.mn.z; n.bmax[0] = b.mx.x; n.bmax[1] = b.mx.y; n.bmax[2] = b.mx.z;
		n.left_child_idx = l; n.right_child_hittable_idx = r;
		nodes.push_back(n);
		return (int)nodes.size() - 1;
	}
	void sort_range(int s, int e, int axis) {   // BVH.cu:195-199: std::sort by aabb.min[axis] with operator<
		std::sort(arr.begin() + s, arr.begin() + e, [axis](const BItem& a, const BItem& b) { return a.box.mn[axis] < b.box.mn[axis]; });
	}
	int topdown_median(int s, int e) {          // _build_bvh_rec1  BVH.cu:180-210
		Box b = range_bounds(s, e);
		int axis = b.longest_axis();
		if (e - s == 1) return emit(b, -1, s);
		sort_range(s, e, axis);
		int mid = (s + e) / 2;
		int l = topdown_median(s, mid);
		int r = topdown_median(mid, e);
		return emit(b, l, r);
	}
	int topdown_sah(int s, int e) {             // _build_bvh_rec2  BVH.cu:212-304
		Box b = range_bounds(s, e);
		if (e - s == 1) return emit(b, -1, s);
		int best_axis = 0; float best_split = 0.0f, best_cost = FLT_MAX;
		for (int axis = 0; axis < 3; ++axis) for (int k = 0; k < 16; ++k) {
			float pos = (k + 1.0f) / (16 + 1.0f);
			pos = b.mn[axis] * (1.0f - pos) + b.mx[axis] * pos;
			Box lb, rb; int lc = 0, rc = 0;
			for (int i = s; i < e; ++i) {
				if (arr[i].box.centroid(axis) < pos) { lb.grow(arr[i].box); lc++; } else { rb.grow(arr[i].box); rc++; }
			}
			float cost = lb.surface_area() * lc + rb.surface_area() * rc;
			if (cost < best_cost) { best_cost = cost; best_axis = axis; best_split = pos; }
		}
		int i = s, j = e;
		while (i < j) { if (arr[i].box.centroid(best_axis) < best_split) i++; else std::swap(arr[i], arr[--j]); }
		int mid = i;
		if (mid == s || mid == e) {             // the reference would recurse forever here; median fallback
			sort_range(s, e, b.longest_axis());
			mid = (s + e) / 2;
		}
		int l = topdown_sah(s, mid);
		int r = topdown_sah(mid, e);
		return emit(b, l, r);
	}
};

int bvh_build_impl(const std::vector<Box>& boxes, int builder, std::vector<rtb_bvh_node>& nodes, std::vector<int>& order, int& root) {
	int n = (int)boxes.size();
	if (builder == RTB_BVH_BOTTOMUP) {          // BuildBVH_BottomUp  BVH.cu:315-383
		struct W { Box box; int count, node; };
		std::vector<W> work; nodes.clear(); order.clear();
		BvhBuild bb;
		for (int i = 0; i < n; ++i) { order.push_back(i); int id = bb.emit(boxes[i], -1, i); work.push_back({boxes[i], 1, id}); }
		while (work.size() > 1) {
			float best = FLT_MAX; int ai = 0, bi = 1;
			for (size_t a = 0; a < work.size(); ++a) for (size_t b = a + 1; b < work.size(); ++b) {
				Box u = work[a].box; u.grow(work[b].box);
				float cost = u.surface_area() * (work[a].count + work[b].count);
				if (cost < best) { ai = (int)a; bi = (int)b; best = cost; }
			}
			Box u = work[ai].box; u.grow(work[bi].box);
			int id = bb.emit(u, work[ai].node, work[bi].node);
			W m{u, work[ai].count + work[bi].count, id};
			work.erase(work.begin() + bi); work.erase(work.begin() + ai);
			work.push_back(m);
		}
		root = work[0].node; nodes.swap(bb.nodes);
		return (int)nodes.size();
	}
	BvhBuild bb; bb.arr.resize(n);
	for (int i = 0; i < n; ++i) { bb.arr[i].box = boxes[i]; bb.arr[i].idx = i; }
	if (builder == RTB_BVH_TOPDOWN_MEDIAN) root = bb.topdown_median(0, n);
	else if (builder == RTB_BVH_TOPDOWN_SAH) root = bb.topdown_sah(0, n);
	else return -1;
	nodes.swap(bb.nodes);
	order.resize(n);
	for (int i = 0; i < n; ++i) order[i] = bb.arr[i].idx;
	return (int)nodes.size();
}

// ---------------------------------------------------------------- scene graph (instantiated as a tree)

struct Rec {                      // RayPayload (ray_data.cuh:33-42) widened to what the extended materials need
	float distance = MISS_DIST;
	int material = -1;
	int object = -1;
	V3 normal;                    // what G::getNormal returns (spheres: outward; quads: facing the ray)
	V3 n_geom;                    // geometric normal (front_face / dielectric)
	float u = 0.0f, v = 0.0f;
};

struct Node;
struct Ctx;
bool hit(const Node* n, const Ray& r, Rec& rec, Ctx& ctx);

struct Node {
	int kind = 0, mat = -1, id = -1;
	float f[11] = {0};
	std::vector<std::unique_ptr<Node>> kids;
	Box bounds;
	std::vector<rtb_bvh_node> bvh_nodes; std::vector<const Node*> bvh_hittables; int bvh_root = -1;
	int medium_index = -1;
	// quads: derived constants (book quad ctor)
	V3 Q, U, Vv, W, N; float D = 0.0f;
};

struct Texture { rtbs_texture t; };

struct Scene {
	std::vector<rtbs_texture> textures;
	std::vector<rtbs_material> materials;
	std::vector<uint8_t> blob;
	std::unique_ptr<Node> root;
	int background_mode = 0; V3 background;
	int n_media = 0;
	bool any_uv_texture = false;
};

void init_quad(Node& n, V3 Q, V3 u, V3 v) {
	n.Q = Q; n.U = u; n.Vv = v;
	V3 nn = cross(u, v);
	n.N = normalize(nn);
	n.D = dot(n.N, Q);
	n.W = nn / dot(nn, nn);
	V3 c[4] = {Q, Q + u, Q + v, Q + u + v};
	int cnt = n.kind == RTB_OBJ_TRIANGLE ? 3 : 4;
	Box b(c[0], c[0]);
	for (int i = 1; i < cnt; ++i) {
		b.mn = V3(std::min(b.mn.x, c[i].x), std::min(b.mn.y, c[i].y), std::min(b.mn.z, c[i].z));
		b.mx = V3(std::max(b.mx.x, c[i].x), std::max(b.mx.y, c[i].y), std::max(b.mx.z, c[i].z));
	}
	pad_box(b); n.bounds = b;
}

std::unique_ptr<Node> make_quad_child(int id, int mat, V3 Q, V3 u, V3 v) {
	auto q = std::make_unique<Node>(); q->kind = RTB_OBJ_QUAD; q->id = id; q->mat = mat; init_quad(*q, Q, u, v); return q;
}

struct Loader {
	const rtbs_object* objs; const int32_t* children; uint32_t n_objects, n_children; Scene* sc;
	std::unique_ptr<Node> build(int id, int depth) {
		if (id < 0 || (uint32_t)id >= n_objects || depth > 64) { g_err = "bad object id / graph too deep"; return nullptr; }
		const rtbs_object& o = objs[id];
		auto n = std::make_unique<Node>();
		n->kind = o.kind; n->mat = o.mat; n->id = id; memcpy(n->f, o.f, sizeof o.f);
		auto child = [&](int k) -> std::unique_ptr<Node> {
			if (o.child_begin < 0 || (uint32_t)(o.child_begin + k) >= n_children) { g_err = "child index out of range"; return nullptr; }
			return build(children[o.child_begin + k], depth + 1);
		};
		switch (o.kind) {
		case RTB_OBJ_SPHERE: {   // getSphereBounds  SphereHittable.cu:52-54
			V3 c(o.f[0], o.f[1], o.f[2]); float r = o.f[3];
			n->bounds = Box(c - V3(r, r, r), c + V3(r, r, r));
			break;
		}
		case RTB_OBJ_MOVING_SPHERE: {   // getMovingSphereBounds  SphereHittable.cu:85-89
			V3 c0(o.f[0], o.f[1], o.f[2]), c1(o.f[4], o.f[5], o.f[6]); float r = o.f[3];
			Box b0(c0 - V3(r, r, r), c0 + V3(r, r, r)), b1(c1 - V3(r, r, r), c1 + V3(r, r, r));
			Box u = b0;
			u.mn = V3(b1.mn.x < b0.mn.x ? b1.mn.x : b0.mn.x, b1.mn.y < b0.mn.y ? b1.mn.y : b0.mn.y, b1.mn.z < b0.mn.z ? b1.mn.z : b0.mn.z);
			u.mx = V3(b0.mx.x < b1.mx.x ? b1.mx.x : b0.mx.x, b0.mx.y < b1.mx.y ? b1.mx.y : b0.mx.y, b0.mx.z < b1.mx.z ? b1.mx.z : b0.mx.z);
			n->bounds = u;
			break;
		}
		case RTB_OBJ_QUAD: case RTB_OBJ_TRIANGLE:
			init_quad(*n, V3(o.f[0], o.f[1], o.f[2]), V3(o.f[3], o.f[4], o.f[5]), V3(o.f[6], o.f[7], o.f[8]));
			break;
		case RTB_OBJ_BOX: {   // book box(a,b): front, right, back, left, top, bottom
			V3 mn(o.f[0], o.f[1], o.f[2]), mx(o.f[3], o.f[4], o.f[5]);
			V3 dx(mx.x - mn.x, 0, 0), dy(0, mx.y - mn.y, 0), dz(0, 0, mx.z - mn.z);
			n->kids.push_back(make_quad_child(id, o.mat, V3(mn.x, mn.y, mx.z), dx, dy));
			n->kids.push_back(make_quad_child(id, o.mat, V3(mx.x, mn.y, mx.z), -dz, dy));
			n->kids.push_back(make_quad_child(id, o.mat, V3(mx.x, mn.y, mn.z), -dx, dy));
			n->kids.push_back(make_quad_child(id, o.mat, V3(mn.x, mn.y, mn.z), dz, dy));
			n->kids.push_back(make_quad_child(id, o.mat, V3(mn.x, mx.y, mx.z), dx, -dz));
			n->kids.push_back(make_quad_child(id, o.mat, V3(mn.x, mn.y, mn.z), dx, dz));
			Box b; for (auto& k : n->kids) b.grow(k->bounds);
			n->bounds = b;
			break;
		}
		case RTB_OBJ_LIST: case RTB_OBJ_BVH: {
			Box b;
			for (int k = 0; k < o.child_count; ++k) { auto c = child(k); if (!c) return nullptr; b.grow(c->bounds); n->kids.push_back(std::move(c)); }
			n->bounds = b;
			if (o.kind == RTB_OBJ_BVH) {
				if (n->kids.empty()) { g_err = "empty BVH"; return nullptr; }
				std::vector<Box> boxes; for (auto& k : n->kids) boxes.push_back(k->bounds);
				std::vector<int> order;
				if (bvh_build_impl(boxes, o.aux, n->bvh_nodes, order, n->bvh_root) < 0) { g_err = "bad BVH builder"; return nullptr; }
				for (int idx : order) n->bvh_hittables.push_back(n->kids[idx].get());
				const rtb_bvh_node& rn = n->bvh_nodes[n->bvh_root];
				n->bounds = Box(V3(rn.bmin[0], rn.bmin[1], rn.bmin[2]), V3(rn.bmax[0], rn.bmax[1], rn.bmax[2]));
			}
			break;
		}
		case RTB_OBJ_TRANSLATE: {
			auto c = child(0); if (!c) return nullptr;
			V3 off(o.f[0], o.f[1], o.f[2]);
			n->bounds = Box(c->bounds.mn + off, c->bounds.mx + off);
			n->kids.push_back(std::move(c));
			break;
		}
		case RTB_OBJ_ROTATE_Y: {   // book rotate_y ctor
			auto c = child(0); if (!c) return nullptr;
			float sn = o.f[1], cs = o.f[2];
			float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
			for (int i = 0; i < 2; ++i) for (int j = 0; j < 2; ++j) for (int k = 0; k < 2; ++k) {
				float x = i ? c->bounds.mx.x : c->bounds.mn.x, y = j ? c->bounds.mx.y : c->bounds.mn.y, z = k ? c->bounds.mx.z : c->bounds.mn.z;
				float t[3] = {cs * x + sn * z, y, -sn * x + cs * z};
				for (int a = 0; a < 3; ++a) { mn[a] = std::fmin(mn[a], t[a]); mx[a] = std::fmax(mx[a], t[a]); }
			}
			n->bounds = Box(V3(mn[0], mn[1], mn[2]), V3(mx[0], mx[1], mx[2]));
			n->kids.push_back(std::move(c));
			break;
		}
		case RTB_OBJ_CONSTANT_MEDIUM: {
			n->medium_index = sc->n_media++;   // depth-first instance order, as the flattener numbers them
			auto c = child(0); if (!c) return nullptr;
			n->bounds = c->bounds;
			n->kids.push_back(std::move(c));
			break;
		}
		default: g_err = "unknown object kind"; return nullptr;
		}
		return n;
	}
};

// ---------------------------------------------------------------- RNG policies

struct Ctx {
	int mode = ORC_RNG_PHILOX;
	bool skip_media = false;
	bool want_uv = false;         // some texture in the scene reads (u,v): spheres then evaluate get_sphere_uv
	// philox
	uint32_t seed = 0, pixel = 0, sample = 0, bounce = 0;
	F4 r{0, 0, 0, 0};
	// xorwow
	Xorwow* xw = nullptr;
	uint64_t rays = 0;

	void begin(uint32_t b) { bounce = b; if (mode == ORC_RNG_PHILOX) r = rng4(seed, pixel, sample, b, STREAM_SCATTER); }
	float uniform() { return mode == ORC_RNG_PHILOX ? r.z : xw->next(); }
	V3 on_unit_sphere() {
		if (mode == ORC_RNG_PHILOX) return unit_sphere(r.x, r.y);
		for (;;) {   // cuRandomOnUnit<3>  glm_utils.h:92-98
			float a = xw->next(), b = xw->next(), c = xw->next();
			V3 v(a * 2.0f - 1.0f, b * 2.0f - 1.0f, c * 2.0f - 1.0f);
			if (!near_zero(v) && dot(v, v) < 1.0f) return normalize(v);
		}
	}
	void in_unit_disc(float& dx, float& dy, bool lens) {
		if (mode == ORC_RNG_PHILOX) {
			F4 q = lens ? rng4(seed, pixel, sample, bounce, STREAM_LENS) : r;
			unit_disc(q.x, q.y, dx, dy); return;
		}
		for (;;) {   // cuRandomInUnit<2>  glm_utils.h:84-90
			float a = xw->next(), b = xw->next();
			float x = a * 2.0f - 1.0f, y = b * 2.0f - 1.0f;
			if (std::fmaf(y, y, x * x) < 1.0f) { dx = x; dy = y; return; }
		}
	}
	float medium_u(int medium_index) {
		if (mode == ORC_RNG_PHILOX) {   // medium m: component (m & 3) of stream STREAM_MEDIUM0 + (m >> 2)
			F4 q = rng4(seed, pixel, sample, bounce, STREAM_MEDIUM0 + ((uint32_t)medium_index >> 2));
			int c = medium_index & 3;
			return c == 0 ? q.x : (c == 1 ? q.y : (c == 2 ? q.z : q.w));
		}
		return xw->next();
	}
};

// ---------------------------------------------------------------- intersection

// book sphere::get_sphere_uv on the outward unit normal in the sphere's own frame
void sphere_uv(V3 n, float& u, float& v) {
	float theta = acosf(-n.y);
	float phi = atan2f(-n.z, n.x) + 3.14159265358979323846f;
	u = phi / 6.28318530717958647692f; v = theta / 3.14159265358979323846f;
}

// _sphere_closest_intersection  SphereHittable.cuh:15-33 in the spec's operation order
float sphere_closest(const Ray& r, V3 center, float radius) {
	V3 oc = r.o - center;
	float a = dot(r.d, r.d);
	float hb = dot(r.d, oc);
	float c = std::fmaf(-radius, radius, dot(oc, oc));
	float d = std::fmaf(hb, hb, -(a * c));
	if (!(d > 0.0f)) return MISS_DIST;
	d = std::sqrt(d);
	float t = (-hb - d) / a;
	if (t < 0.0f) {
		t = (-hb + d) / a;
		if (t < 0.0f) return MISS_DIST;
	}
	return t;
}

// Book quad::hit; returns t or MISS_DIST. `lo <= t <= hi` is the book's interval::contains.
float planar_t(const Node& q, const Ray& r, float lo, float hi, bool strict_hi, float* alpha_out = nullptr, float* beta_out = nullptr) {
	float denom = dot(q.N, r.d);
	if (std::fabs(denom) < 1e-8f) return MISS_DIST;
	float t = (q.D - dot(q.N, r.o)) / denom;
	if (!(t >= lo)) return MISS_DIST;
	if (strict_hi ? !(t < hi) : !(t <= hi)) return MISS_DIST;
	V3 P = r.at(t);
	V3 planar = P - q.Q;
	float alpha = dot(q.W, cross(planar, q.Vv));
	float beta = dot(q.W, cross(q.U, planar));
	if (q.kind == RTB_OBJ_TRIANGLE) { if (alpha < 0.0f || beta < 0.0f || alpha + beta > 1.0f) return MISS_DIST; }
	else { if (alpha < 0.0f || alpha > 1.0f || beta < 0.0f || beta > 1.0f) return MISS_DIST; }
	if (alpha_out) *alpha_out = alpha;
	if (beta_out) *beta_out = beta;
	return t;
}

Ray to_rotated(const Node& n, const Ray& r) {   // book rotate_y::hit: world -> object
	float sn = n.f[1], cs = n.f[2];
	V3 o(std::fmaf(cs, r.o.x, -(sn * r.o.z)), r.o.y, std::fmaf(sn, r.o.x, cs * r.o.z));
	V3 d(std::fmaf(cs, r.d.x, -(sn * r.d.z)), r.d.y, std::fmaf(sn, r.d.x, cs * r.d.z));
	return Ray(o, d, r.time);
}
V3 from_rotated(const Node& n, V3 v) {          // object -> world
	float sn = n.f[1], cs = n.f[2];
	return V3(std::fmaf(cs, v.x, sn * v.z), v.y, std::fmaf(-sn, v.x, cs * v.z));
}

// Boundary query of constant_medium: closest t with lo < t < hi (spheres: surrounds) / lo <= t <= hi (quads: contains).
float boundary_t(const Node* n, const Ray& r, float lo, float hi) {
	switch (n->kind) {
	case RTB_OBJ_SPHERE: case RTB_OBJ_MOVING_SPHERE: {   // book sphere::hit root selection, reference sign convention
		V3 c(n->f[0], n->f[1], n->f[2]);
		if (n->kind == RTB_OBJ_MOVING_SPHERE) c = mix(c, V3(n->f[4], n->f[5], n->f[6]), r.time);
		V3 oc = r.o - c; float a = dot(r.d, r.d), hb = dot(r.d, oc);
		float cc = std::fmaf(-n->f[3], n->f[3], dot(oc, oc));
		float disc = std::fmaf(hb, hb, -(a * cc));
		if (!(disc > 0.0f)) return MISS_DIST;
		float sq = std::sqrt(disc);
		float root = (-hb - sq) / a;
		if (!(lo < root && root < hi)) { root = (-hb + sq) / a; if (!(lo < root && root < hi)) return MISS_DIST; }
		return root;
	}
	case RTB_OBJ_QUAD: case RTB_OBJ_TRIANGLE: return planar_t(*n, r, lo, hi, false);
	case RTB_OBJ_BOX: case RTB_OBJ_LIST: case RTB_OBJ_BVH: {
		float best = MISS_DIST;
		for (auto& k : n->kids) { float t = boundary_t(k.get(), r, lo, best < hi ? best : hi); if (t < best) best = t; }
		return best;
	}
	case RTB_OBJ_TRANSLATE: return boundary_t(n->kids[0].get(), Ray(r.o - V3(n->f[0], n->f[1], n->f[2]), r.d, r.time), lo, hi);
	case RTB_OBJ_ROTATE_Y: return boundary_t(n->kids[0].get(), to_rotated(*n, r), lo, hi);
	default: return MISS_DIST;
	}
}

bool hit(const Node* n, const Ray& r, Rec& rec, Ctx& ctx) {
	switch (n->kind) {
	case RTB_OBJ_SPHERE: {   // SphereHittable::ClosestIntersection  SphereHittable.cu:56-66
		V3 c(n->f[0], n->f[1], n->f[2]);
		float t = sphere_closest(r, c, n->f[3]);
		if (!(t < rec.distance)) return false;
		rec.material = n->mat; rec.distance = t; rec.object = n->id;
		rec.normal = (r.at(t) - c) / n->f[3]; rec.n_geom = rec.normal;
		if (ctx.want_uv) sphere_uv(rec.normal, rec.u, rec.v);
		return true;
	}
	case RTB_OBJ_MOVING_SPHERE: {   // MovingSphereHittable::ClosestIntersection  SphereHittable.cu:91-102
		V3 c = mix(V3(n->f[0], n->f[1], n->f[2]), V3(n->f[4], n->f[5], n->f[6]), r.time);
		float t = sphere_closest(r, c, n->f[3]);
		if (!(t < rec.distance)) return false;
		rec.material = n->mat; rec.distance = t; rec.object = n->id;
		rec.normal = (r.at(t) - c) / n->f[3]; rec.n_geom = rec.normal;
		if (ctx.want_uv) sphere_uv(rec.normal, rec.u, rec.v);
		return true;
	}
	case RTB_OBJ_QUAD: case RTB_OBJ_TRIANGLE: {
		float a, b;
		float t = planar_t(*n, r, 0.0f, rec.distance, true, &a, &b);
		if (!(t < rec.distance)) return false;
		rec.material = n->mat; rec.distance = t; rec.object = n->id;
		rec.n_geom = n->N;
		rec.normal = dot(r.d, n->N) > 0.0f ? -n->N : n->N;   // book set_face_normal
		rec.u = a; rec.v = b;
		return true;
	}
	case RTB_OBJ_BOX: {
		bool any = false;
		for (auto& k : n->kids) any |= hit(k.get(), r, rec, ctx);
		return any;
	}
	case RTB_OBJ_LIST: {   // HittableList::ClosestIntersection  HittableList.cuh:21-34
		if (!n->bounds.intersects(r, rec.distance)) return false;
		bool any = false;
		for (auto& k : n->kids) if (hit(k.get(), r, rec, ctx)) any = true;
		return any;
	}
	case RTB_OBJ_BVH: {    // BVH::ClosestIntersection  BVH.cu:54-106 (LIFO mode, _USE_PRIO_QUEUE false)
		auto node_box = [&](int i) { const rtb_bvh_node& b = n->bvh_nodes[i]; return Box(V3(b.bmin[0], b.bmin[1], b.bmin[2]), V3(b.bmax[0], b.bmax[1], b.bmax[2])); };
		int stack[64]; int head = 0;
		float root_dist;
		if (!node_box(n->bvh_root).intersects(r, rec.distance, root_dist)) return false;
		stack[head++] = n->bvh_root;
		bool any = false;
		while (head != 0) {
			int idx = stack[--head];
			const rtb_bvh_node& nd = n->bvh_nodes[idx];
			if (nd.left_child_idx == -1) { any |= hit(n->bvh_hittables[nd.right_child_hittable_idx], r, rec, ctx); continue; }
			float ld = MISS_DIST, rd = MISS_DIST;
			int li = nd.left_child_idx, ri = nd.right_child_hittable_idx;
			node_box(li).intersects(r, rec.distance, ld);
			node_box(ri).intersects(r, rec.distance, rd);
			if (ld > rd) { std::swap(li, ri); std::swap(ld, rd); }
			if (rd < rec.distance && head < 64) stack[head++] = ri;
			if (ld < rec.distance && head < 64) stack[head++] = li;
		}
		return any;
	}
	case RTB_OBJ_TRANSLATE: {   // book translate::hit (the hit point is recomputed from the world ray by the integrator)
		Ray moved(r.o - V3(n->f[0], n->f[1], n->f[2]), r.d, r.time);
		return hit(n->kids[0].get(), moved, rec, ctx);
	}
	case RTB_OBJ_ROTATE_Y: {    // book rotate_y::hit
		if (!hit(n->kids[0].get(), to_rotated(*n, r), rec, ctx)) return false;
		rec.normal = from_rotated(*n, rec.normal);
		rec.n_geom = from_rotated(*n, rec.n_geom);
		return true;
	}
	case RTB_OBJ_CONSTANT_MEDIUM: {   // book constant_medium::hit, ray_t = [0, closest so far)
		if (ctx.skip_media) return false;
		const Node* b = n->kids[0].get();
		float t1 = boundary_t(b, r, -INFINITY, INFINITY);
		if (!(t1 < MISS_DIST)) return false;
		float t2 = boundary_t(b, r, t1 + 0.0001f, INFINITY);
		if (!(t2 < MISS_DIST)) return false;
		float u = ctx.medium_u(n->medium_index);
		if (t1 < 0.0f) t1 = 0.0f;
		if (t2 > rec.distance) t2 = rec.distance;
		if (t1 >= t2) return false;
		float len = std::sqrt(dot(r.d, r.d));
		float dist_inside = (t2 - t1) * len;
		float hit_distance = n->f[1] * logpos(u);
		if (hit_distance > dist_inside) return false;
		float t = t1 + hit_distance / len;
		if (!(t < rec.distance)) return false;
		rec.distance = t; rec.material = n->mat; rec.object = n->id;
		rec.normal = V3(1, 0, 0); rec.n_geom = rec.normal; rec.u = rec.v = 0.0f;
		return true;
	}
	}
	return false;
}

// ---------------------------------------------------------------- textures and materials

float perlin_noise(const float* grad, const int32_t* perm, V3 p) {   // book perlin::noise / perlin_interp
	float fx = std::floor(p.x), fy = std::floor(p.y), fz = std::floor(p.z);
	float u = p.x - fx, v = p.y - fy, w = p.z - fz;
	int i = (int)fx, j = (int)fy, k = (int)fz;
	float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
	float accum = 0.0f;
	for (int di = 0; di < 2; ++di) for (int dj = 0; dj < 2; ++dj) for (int dk = 0; dk < 2; ++dk) {
		int g = perm[(i + di) & 255] ^ perm[256 + ((j + dj) & 255)] ^ perm[512 + ((k + dk) & 255)];
		V3 c(grad[3 * g], grad[3 * g + 1], grad[3 * g + 2]);
		V3 wv(u - (float)di, v - (float)dj, w - (float)dk);
		float wi = di ? uu : 1.0f - uu, wj = dj ? vv : 1.0f - vv, wk = dk ? ww : 1.0f - ww;
		accum = std::fmaf(wi * wj * wk, dot(c, wv), accum);
	}
	return accum;
}

V3 texture_value(const Scene& sc, int tex, float u, float v, V3 p) {
	for (int guard = 0; guard < 16; ++guard) {
		const rtbs_texture& t = sc.textures[tex];
		if (t.kind == RTB_TEX_SOLID) return V3(t.rgb[0], t.rgb[1], t.rgb[2]);          // solid_texture::value  cu_Textures.cuh:16-18
		if (t.kind == RTB_TEX_CHECKER) {                                                  // checker_texture::value  cu_Textures.cuh:32-39
			float inv = 1.0f / t.scale;
			int sum = (int)(p.x * inv) + (int)(p.y * inv) + (int)(p.z * inv);               // ivec3(pos * inv_scale): truncation; compAdd
			tex = (sum % 2 == 0) ? t.even : t.odd;
			continue;
		}
		if (t.kind == RTB_TEX_IMAGE) {                                                    // book image_texture::value
			float uc = std::fmin(std::fmax(u, 0.0f), 1.0f), vc = 1.0f - std::fmin(std::fmax(v, 0.0f), 1.0f);
			int i = (int)(uc * (float)t.width), j = (int)(vc * (float)t.height);
			i = i < t.width - 1 ? i : t.width - 1; j = j < t.height - 1 ? j : t.height - 1;
			const uint8_t* px = sc.blob.data() + t.blob_offset + 3 * ((size_t)j * t.width + i);
			const float s = 1.0f / 255.0f;
			return V3(s * (float)px[0], s * (float)px[1], s * (float)px[2]);
		}
		const float* grad = reinterpret_cast<const float*>(sc.blob.data() + t.blob_offset);   // book noise_texture::value (marble)
		const int32_t* perm = reinterpret_cast<const int32_t*>(sc.blob.data() + t.blob_offset + 256 * 3 * 4);
		float accum = 0.0f, weight = 1.0f; V3 tp = p;
		for (int k = 0; k < 7; ++k) { accum = std::fmaf(weight, perlin_noise(grad, perm, tp), accum); weight *= 0.5f; tp = tp * 2.0f; }
		float val = 0.5f * (1.0f + sin_any(std::fmaf(t.scale, p.z, 10.0f * std::fabs(accum))));
		return V3(val, val, val);
	}
	return V3();
}

// 0 absorbed, 1 scattered, 2 emitted
int scatter(const Scene& sc, const Ray& in, const Rec& rec, V3 p, Ctx& ctx, V3& dir, V3& att) {
	const rtbs_material& m = sc.materials[rec.material];
	V3 albedo = m.tex >= 0 ? texture_value(sc, m.tex, rec.u, rec.v, p) : V3(m.albedo[0], m.albedo[1], m.albedo[2]);
	switch (m.kind) {
	case RTB_MAT_LAMBERTIAN: {   // cu_materials.cuh:52-64 (and LambertianTexture :26-40)
		dir = rec.normal + ctx.on_unit_sphere();
		if (near_zero(dir)) return 0;
		att = albedo; return 1;
	}
	case RTB_MAT_METAL: {        // cu_materials.cuh:77-95
		V3 refl = reflect(in.d, rec.normal);
		dir = fma3(ctx.on_unit_sphere(), m.param, refl);
		if (dot(dir, rec.normal) < 0.0f || near_zero(dir)) return 0;
		att = albedo; return 1;
	}
	case RTB_MAT_DIELECTRIC: {   // cu_materials.cuh:115-143; reflectance :99-104 with (1-cos)^5 as exact products
		V3 n = rec.n_geom;
		bool back = dot(in.d, n) > 0.0f;
		if (back) n = -n;
		float ratio = back ? m.param : 1.0f / m.param;
		V3 ud = normalize(in.d);
		float cos_theta = std::fmin(dot(-ud, n), 1.0f);
		float sin_theta = std::sqrt(std::fmaf(-cos_theta, cos_theta, 1.0f));
		float r0 = (1.0f - ratio) / (1.0f + ratio); r0 = r0 * r0;
		float x = 1.0f - cos_theta, x2 = x * x;
		float prob = std::fmaf(1.0f - r0, x2 * x2 * x, r0);
		if (ratio * sin_theta > 1.0f || prob > ctx.uniform()) {   // the uniform is drawn only when not TIR (short-circuit)
			dir = reflect(ud, n);
		} else {   // glm::refract  func_geometric.inl:113-124
			float dv = dot(n, ud);
			float k = std::fmaf(-(ratio * ratio), std::fmaf(-dv, dv, 1.0f), 1.0f);
			if (k < 0.0f) return 0;
			float coef = std::fmaf(ratio, dv, std::sqrt(k));
			dir = V3(std::fmaf(-coef, n.x, ratio * ud.x), std::fmaf(-coef, n.y, ratio * ud.y), std::fmaf(-coef, n.z, ratio * ud.z));
		}
		if (dir.x == 0.0f && dir.y == 0.0f && dir.z == 0.0f) return 0;
		att = albedo; return 1;
	}
	case RTB_MAT_ISOTROPIC: dir = ctx.on_unit_sphere(); att = albedo; return 1;   // book isotropic::scatter
	default: att = albedo; return 2;                                              // book diffuse_light::emitted, no scatter
	}
}

V3 background(const Scene& sc, V3 d) {
	if (sc.background_mode == RTB_BG_CONSTANT) return sc.background;
	float ny = d.y * (1.0f / std::sqrt(dot(d, d)));   // Renderer.cu:149-151
	float t = std::fmaf(ny, 0.5f, 0.5f);
	return V3(std::fmaf(0.9f - 0.1f, t, 0.1f), std::fmaf(0.9f - 0.2f, t, 0.2f), std::fmaf(0.99f - 0.4f, t, 0.4f));
}

// sample_world  Renderer.cu:139-181 (+ emission at the terminating hit, book ray_color)
V3 sample_world(const Scene& sc, Ray ray, uint32_t max_depth, Ctx& ctx) {
	V3 thr(1, 1, 1);
	for (uint32_t i = 0; i < max_depth; ++i) {
		Rec rec;
		ctx.begin(i);
		ctx.rays++;
		if (!hit(sc.root.get(), ray, rec, ctx)) return thr * background(sc, ray.d);
		V3 p = ray.at(rec.distance);
		V3 dir, att;
		int res = scatter(sc, ray, rec, p, ctx, dir, att);
		if (res == 2) return thr * att;
		if (res == 0) return V3();
		thr = thr * att;
		ray = Ray(fma3(dir, 0.001f, p), dir, ray.time);   // Renderer.cu:168-175
	}
	return V3();
}

Ray camera_ray(const rtb_camera& cam, float s, float t, Ctx& ctx) {
	V3 o(cam.o[0], cam.o[1], cam.o[2]), cu(cam.u[0], cam.u[1], cam.u[2]), cv(cam.v[0], cam.v[1], cam.v[2]), cw(cam.w[0], cam.w[1], cam.w[2]);
	if (cam.kind == RTB_CAM_DEFOCUS) {   // cu_Cameras.cuh:54-64
		float lx, ly; ctx.in_unit_disc(lx, ly, true);
		V3 off = V3(std::fmaf(cv.x, ly, cu.x * lx), std::fmaf(cv.y, ly, cu.y * lx), std::fmaf(cv.z, ly, cu.z * lx)) * cam.lens_radius;
		V3 fwd = cw * cam.focus_dist, hori = (cu * cam.viewport_width) * cam.focus_dist, vert = (cv * cam.viewport_height) * cam.focus_dist;
		float time = mixf(cam.t0, cam.t1, ctx.uniform());
		return Ray(o + off, fma3(vert, t, fma3(hori, s, fwd)) - off, time);
	}
	V3 d = fma3(cv, t, fma3(cu, s, cw));   // cu_Cameras.cuh:27-30
	float time = 0.0f;
	if (cam.kind == RTB_CAM_MOTION) time = mixf(cam.t0, cam.t1, ctx.uniform());   // cu_Cameras.cuh:87-89
	return Ray(o, d, time);
}

// Renders samples [s0, s1) of every pixel, rows handed out to `threads` workers; ADDS into sum (and sum2), and stores the
// number of traced segments in *rays_out.  trace(ray, ctx) is the integrator: it returns the sample's radiance.
template <class Trace>
void render_rows(const rtb_camera& cam, uint32_t W, uint32_t H, uint32_t s0, uint32_t s1, uint32_t seed, int mode, int threads,
                 bool want_uv, float* sum, float* sum2, uint64_t* rays_out, const Trace& trace) {
	if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
	if (threads <= 0) threads = 1;
	std::atomic<uint32_t> next_row{0};
	std::atomic<uint64_t> total_rays{0};
	const float px = 1.0f / (float)W, py = 1.0f / (float)H;   // pixel_size  Renderer.cu:188
	auto worker = [&]() {
		uint64_t rays = 0;
		for (;;) {
			uint32_t y = next_row.fetch_add(1);
			if (y >= H) break;
			for (uint32_t x = 0; x < W; ++x) {
				uint32_t gid = y * W + x;
				Xorwow xw((uint64_t)seed + gid);             // init_random_states: cuRandom(seed + gid, 0, 0)  Renderer.cu:22-29
				Ctx ctx; ctx.mode = mode; ctx.seed = seed; ctx.pixel = gid; ctx.xw = &xw; ctx.want_uv = want_uv;
				float ndcx = std::fmaf(((float)x + 0.5f) * px, 2.0f, -1.0f);   // Renderer.cu:192
				float ndcy = std::fmaf(((float)y + 0.5f) * py, 2.0f, -1.0f);
				float ax = 0, ay = 0, az = 0, qx = 0, qy = 0, qz = 0;
				for (uint32_t smp = s0; smp < s1; ++smp) {
					ctx.sample = smp;
					ctx.begin(CAMERA_BOUNCE);
					float jx, jy; ctx.in_unit_disc(jx, jy, false);          // Renderer.cu:199
					Ray ray = camera_ray(cam, std::fmaf(jx, px, ndcx), std::fmaf(jy, py, ndcy), ctx);
					V3 c = trace(ray, ctx);
					ax += c.x; ay += c.y; az += c.z;
					qx = std::fmaf(c.x, c.x, qx); qy = std::fmaf(c.y, c.y, qy); qz = std::fmaf(c.z, c.z, qz);
				}
				float* o = sum + 4 * (size_t)gid;
				o[0] += ax; o[1] += ay; o[2] += az; o[3] += (float)(s1 - s0);
				if (sum2) { float* q = sum2 + 4 * (size_t)gid; q[0] += qx; q[1] += qy; q[2] += qz; q[3] += (float)(s1 - s0); }
				rays += ctx.rays;
			}
		}
		total_rays += rays;
	};
	std::vector<std::thread> pool;
	for (int t = 1; t < threads; ++t) pool.emplace_back(worker);
	worker();
	for (auto& t : pool) t.join();
	if (rays_out) *rays_out = total_rays.load();
}

}  // namespace

// ================================================================= C API

struct orc_scene { Scene sc; };

extern "C" {

const char* orc_last_error(void) { return g_err.c_str(); }

orc_scene* orc_scene_load(const void* blob, size_t size) {
	if (!blob || size < sizeof(rtbs_header)) { g_err = "blob too small"; return nullptr; }
	const uint8_t* p = static_cast<const uint8_t*>(blob);
	rtbs_header h; memcpy(&h, p, sizeof h);
	if (h.magic != RTBS_MAGIC || h.version != RTBS_VERSION) { g_err = "bad magic/version"; return nullptr; }
	size_t need = sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) + (size_t)h.n_materials * sizeof(rtbs_material) +
	              (size_t)h.n_objects * sizeof(rtbs_object) + (size_t)h.n_children * 4 + h.n_blob_bytes;
	if (size < need) { g_err = "blob truncated"; return nullptr; }
	auto s = std::make_unique<orc_scene>();
	p += sizeof h;
	s->sc.textures.resize(h.n_textures); memcpy(s->sc.textures.data(), p, h.n_textures * sizeof(rtbs_texture)); p += h.n_textures * sizeof(rtbs_texture);
	s->sc.materials.resize(h.n_materials); memcpy(s->sc.materials.data(), p, h.n_materials * sizeof(rtbs_material)); p += h.n_materials * sizeof(rtbs_material);
	std::vector<rtbs_object> objs(h.n_objects); memcpy(objs.data(), p, h.n_objects * sizeof(rtbs_object)); p += h.n_objects * sizeof(rtbs_object);
	std::vector<int32_t> children(h.n_children); memcpy(children.data(), p, h.n_children * 4); p += h.n_children * 4;
	s->sc.blob.assign(p, p + h.n_blob_bytes);
	s->sc.background_mode = h.background_mode; s->sc.background = V3(h.background[0], h.background[1], h.background[2]);
	for (const rtbs_texture& t : s->sc.textures) if (t.kind == RTB_TEX_IMAGE) s->sc.any_uv_texture = true;
	Loader ld{objs.data(), children.data(), h.n_objects, h.n_children, &s->sc};
	s->sc.root = ld.build(h.root_object, 0);
	if (!s->sc.root) return nullptr;
	return s.release();
}
void orc_scene_free(orc_scene* s) { delete s; }

int orc_render(const orc_scene* s, const rtb_camera* cam, uint32_t W, uint32_t H, uint32_t s0, uint32_t s1, uint32_t max_depth,
               uint32_t seed, int mode, int threads, float* sum, float* sum2, uint64_t* rays_out) {
	if (!s || !cam || !sum || W == 0 || H == 0) { g_err = "orc_render: bad argument"; return -1; }
	if (mode == ORC_RNG_XORWOW && s0 != 0) { g_err = "orc_render: XORWOW mode renders from sample 0 (per-pixel sequential streams)"; return -1; }
	const Scene& sc = s->sc;
	render_rows(*cam, W, H, s0, s1, seed, mode, threads, sc.any_uv_texture, sum, sum2, rays_out,
	            [&](const Ray& ray, Ctx& ctx) { return sample_world(sc, ray, max_depth, ctx); });
	return 0;
}

int orc_trace_rays(const orc_scene* s, const rtb_ray* rays, size_t n, rtb_hit* out) {
	if (!s || (n && (!rays || !out))) { g_err = "orc_trace_rays: bad argument"; return -1; }
	const Scene& sc = s->sc;
	for (size_t i = 0; i < n; ++i) {
		Ray r(V3(rays[i].o[0], rays[i].o[1], rays[i].o[2]), V3(rays[i].d[0], rays[i].d[1], rays[i].d[2]), rays[i].time);
		Ctx ctx; ctx.skip_media = true; ctx.want_uv = true;
		Rec rec;
		rtb_hit h; memset(&h, 0, sizeof h);
		if (!hit(sc.root.get(), r, rec, ctx)) { h.t = MISS_DIST; h.prim = -1; h.object = -1; h.material = -1; out[i] = h; continue; }
		V3 p = r.at(rec.distance);
		h.t = rec.distance; h.prim = -1; h.object = rec.object; h.material = rec.material;
		h.p[0] = p.x; h.p[1] = p.y; h.p[2] = p.z;
		h.n[0] = rec.normal.x; h.n[1] = rec.normal.y; h.n[2] = rec.normal.z;
		h.front_face = dot(r.d, rec.n_geom) > 0.0f ? 0 : 1;   // isBackfacing  ray_data.cuh:44-46
		h.u = rec.u; h.v = rec.v;
		out[i] = h;
	}
	return 0;
}

int orc_sphere_index_image(const float* sp, int n, const rtb_camera* cam, int W, int H, int32_t* out) {
	if (!sp || !cam || !out || n < 0) return -1;
	V3 o(cam->o[0], cam->o[1], cam->o[2]), cu(cam->u[0], cam->u[1], cam->u[2]), cv(cam->v[0], cam->v[1], cam->v[2]), cw(cam->w[0], cam->w[1], cam->w[2]);
	for (int y = 0; y < H; ++y) for (int x = 0; x < W; ++x) {   // test.cpp:87-106
		float u = x / (W - 1.0f) * 2 - 1, v = y / (H - 1.0f) * 2 - 1;
		Ray ray(o, fma3(cv, v, fma3(cu, u, cw)));
		float best = MISS_DIST; int idx = -1;
		for (int i = 0; i < n; ++i) {
			float d = sphere_closest(ray, V3(sp[4 * i], sp[4 * i + 1], sp[4 * i + 2]), sp[4 * i + 3]);
			if (d < best) { idx = i; best = d; }
		}
		out[(size_t)y * W + x] = idx;
	}
	return 0;
}

int orc_bvh_build(const float* aabbs, int n, int builder, rtb_bvh_node* nodes_out, int* order_out, int* root_out) {
	if (!aabbs || n <= 0 || !nodes_out || !order_out || !root_out) return -1;
	std::vector<Box> boxes(n);
	for (int i = 0; i < n; ++i) boxes[i] = Box(V3(aabbs[6 * i], aabbs[6 * i + 1], aabbs[6 * i + 2]), V3(aabbs[6 * i + 3], aabbs[6 * i + 4], aabbs[6 * i + 5]));
	std::vector<rtb_bvh_node> nodes; std::vector<int> order; int root = -1;
	int rc = bvh_build_impl(boxes, builder, nodes, order, root);
	if (rc < 0) return rc;
	memcpy(nodes_out, nodes.data(), nodes.size() * sizeof(rtb_bvh_node));
	memcpy(order_out, order.data(), order.size() * sizeof(int));
	*root_out = root;
	return rc;
}

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
	U4 c; for (int i = 0; i < 4; ++i) c.v[i] = ctr[i];
	U4 r = philox4x32_10(c, key[0], key[1]);
	for (int i = 0; i < 4; ++i) out[i] = r.v[i];
}
void orc_xorwow_uniforms(uint64_t seed, int n, float* out) { Xorwow x(seed); for (int i = 0; i < n; ++i) out[i] = x.next(); }
void orc_sincos2pi(float u, float* s, float* c) { sincos2pi(u, *s, *c); }
float orc_logpos(float x) { return logpos(x); }

}  // extern "C"
