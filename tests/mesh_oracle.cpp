// tests/mesh_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's integrator with per-vertex normals and texture coordinates
// of mesh triangles.
//
// An independent CPU restatement of DESIGN.md §5e ("Triangle attributes"), built on top of the environment-map oracle: this
// file includes tests/env_oracle.cpp (and through it tests/light_oracle.cpp and oracle/oracle.cpp) unchanged and reuses its
// scene, lights, map, materials and Philox streams.  The oracle's hit() sets a triangle's record inside its recursive walk
// and rotate_y turns the normal on the way back, so the interpolation has to happen at the leaf, in the triangle's own
// frame: this file restates the walk (hit_attr below, case for case the oracle's hit()) instead of adding a hook to
// oracle.cpp, whose behaviour therefore stays exactly what it was.  What it adds is the attribute table read from an RTBS v4
// blob, the interpolation at triangle leaves, the dielectric about the interpolated normal, and the integrator that uses
// them.  tests/mesh_oracle.py compiles it (g++ -ffp-contract=off, like the oracle) into a temporary directory on first use.
#include "env_oracle.cpp"

namespace {

// The attribute table and, per object id, its record index + 1 (the objects' `aux`; 0: none).
struct Attrs {
	std::vector<rtbs_tri_attr> rec;
	std::vector<int32_t> aux;
};

// Rec widened with m: the shading normal on the geometric normal's side (the geometric normal without attributes).
struct MRec : Rec { V3 m; };

bool hit_attr(const Node* n, const Ray& r, MRec& rec, Ctx& ctx, const Attrs& at) {
	switch (n->kind) {
	case RTB_OBJ_SPHERE: case RTB_OBJ_MOVING_SPHERE: case RTB_OBJ_CONSTANT_MEDIUM: {
		if (!hit(n, r, rec, ctx)) return false;
		rec.m = rec.n_geom;
		return true;
	}
	case RTB_OBJ_QUAD: case RTB_OBJ_TRIANGLE: {
		float a, b;
		float t = planar_t(*n, r, 0.0f, rec.distance, true, &a, &b);
		if (!(t < rec.distance)) return false;
		rec.material = n->mat; rec.distance = t; rec.object = n->id;
		rec.n_geom = n->N;
		V3 m = n->N;
		rec.u = a; rec.v = b;
		const int k = n->kind == RTB_OBJ_TRIANGLE && n->id >= 0 && (size_t)n->id < at.aux.size() ? at.aux[n->id] : 0;
		if (k > 0) {   // §5e: w = (1 - alpha) - beta; x interpolates as fma(x2, beta, fma(x1, alpha, x0 * w))
			const rtbs_tri_attr& A = at.rec[k - 1];
			const float w = (1.0f - a) - b;
			auto interp = [&](float x0, float x1, float x2) { return std::fmaf(x2, b, std::fmaf(x1, a, x0 * w)); };
			if (A.flags & RTBS_ATTR_NORMALS) {
				m = V3(interp(A.n[0][0], A.n[1][0], A.n[2][0]), interp(A.n[0][1], A.n[1][1], A.n[2][1]), interp(A.n[0][2], A.n[1][2], A.n[2][2]));
				m = dot(m, m) > 0.0f ? normalize(m) : n->N;
				if (dot(m, n->N) < 0.0f) m = -m;
			}
			if (A.flags & RTBS_ATTR_UVS) { rec.u = interp(A.uv[0][0], A.uv[1][0], A.uv[2][0]); rec.v = interp(A.uv[0][1], A.uv[1][1], A.uv[2][1]); }
		}
		rec.normal = dot(r.d, n->N) > 0.0f ? -m : m;   // book set_face_normal with m in place of N
		rec.m = m;
		return true;
	}
	case RTB_OBJ_BOX: {
		bool any = false;
		for (auto& k : n->kids) any |= hit_attr(k.get(), r, rec, ctx, at);
		return any;
	}
	case RTB_OBJ_LIST: {
		if (!n->bounds.intersects(r, rec.distance)) return false;
		bool any = false;
		for (auto& k : n->kids) if (hit_attr(k.get(), r, rec, ctx, at)) any = true;
		return any;
	}
	case RTB_OBJ_BVH: {
		auto node_box = [&](int i) { const rtb_bvh_node& b = n->bvh_nodes[i]; return Box(V3(b.bmin[0], b.bmin[1], b.bmin[2]), V3(b.bmax[0], b.bmax[1], b.bmax[2])); };
		int stack[64]; int head = 0;
		float root_dist;
		if (!node_box(n->bvh_root).intersects(r, rec.distance, root_dist)) return false;
		stack[head++] = n->bvh_root;
		bool any = false;
		while (head != 0) {
			int idx = stack[--head];
			const rtb_bvh_node& nd = n->bvh_nodes[idx];
			if (nd.left_child_idx == -1) { any |= hit_attr(n->bvh_hittables[nd.right_child_hittable_idx], r, rec, ctx, at); continue; }
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
	case RTB_OBJ_TRANSLATE: {
		Ray moved(r.o - V3(n->f[0], n->f[1], n->f[2]), r.d, r.time);
		return hit_attr(n->kids[0].get(), moved, rec, ctx, at);
	}
	case RTB_OBJ_ROTATE_Y: {
		if (!hit_attr(n->kids[0].get(), to_rotated(*n, r), rec, ctx, at)) return false;
		rec.normal = from_rotated(*n, rec.normal);
		rec.n_geom = from_rotated(*n, rec.n_geom);
		rec.m = from_rotated(*n, rec.m);
		return true;
	}
	}
	return false;
}

// scatter() of the oracle, with the dielectric refracting and reflecting about m (negated on the back, the back decided
// by the geometric normal).
int scatter_attr(const Scene& sc, const Ray& in, const MRec& rec, V3 p, Ctx& ctx, V3& dir, V3& att) {
	const rtbs_material& m = sc.materials[rec.material];
	if (m.kind != RTB_MAT_DIELECTRIC) return scatter(sc, in, rec, p, ctx, dir, att);
	V3 albedo = m.tex >= 0 ? texture_value(sc, m.tex, rec.u, rec.v, p) : V3(m.albedo[0], m.albedo[1], m.albedo[2]);
	bool back = dot(in.d, rec.n_geom) > 0.0f;
	V3 n = back ? -rec.m : rec.m;
	float ratio = back ? m.param : 1.0f / m.param;
	V3 ud = normalize(in.d);
	float cos_theta = std::fmin(dot(-ud, n), 1.0f);
	float sin_theta = std::sqrt(std::fmaf(-cos_theta, cos_theta, 1.0f));
	float r0 = (1.0f - ratio) / (1.0f + ratio); r0 = r0 * r0;
	float x = 1.0f - cos_theta, x2 = x * x;
	float prob = std::fmaf(1.0f - r0, x2 * x2 * x, r0);
	if (ratio * sin_theta > 1.0f || prob > ctx.uniform()) {
		dir = reflect(ud, n);
	} else {
		float dv = dot(n, ud);
		float k = std::fmaf(-(ratio * ratio), std::fmaf(-dv, dv, 1.0f), 1.0f);
		if (k < 0.0f) return 0;
		float coef = std::fmaf(ratio, dv, std::sqrt(k));
		dir = V3(std::fmaf(-coef, n.x, ratio * ud.x), std::fmaf(-coef, n.y, ratio * ud.y), std::fmaf(-coef, n.z, ratio * ud.z));
	}
	if (dir.x == 0.0f && dir.y == 0.0f && dir.z == 0.0f) return 0;
	att = albedo; return 1;
}

// sample_world_env of tests/env_oracle.cpp with the attribute walk and scatter.
V3 sample_world_attr(const Scene& sc, const std::vector<Light>& lights, const Env* env, const Attrs& at, Ray ray, uint32_t max_depth, Ctx& ctx) {
	V3 thr(1, 1, 1);
	const bool mix = !lights.empty() || (env && env->sample);
	for (uint32_t i = 0; i < max_depth; ++i) {
		MRec rec;
		ctx.begin(i);
		ctx.rays++;
		if (!hit_attr(sc.root.get(), ray, rec, ctx, at)) return thr * (env ? env_radiance(*env, ray.d) : background(sc, ray.d));
		V3 p = ray.at(rec.distance);
		V3 dir, att;
		const rtbs_material& m = sc.materials[rec.material];
		if (mix && (m.kind == RTB_MAT_LAMBERTIAN || m.kind == RTB_MAT_ISOTROPIC)) {
			att = m.tex >= 0 ? texture_value(sc, m.tex, rec.u, rec.v, p) : V3(m.albedo[0], m.albedo[1], m.albedo[2]);
			float w;
			if (!env_light_mix(lights, env, m.kind == RTB_MAT_ISOTROPIC, p, rec.normal, ctx, dir, w)) return V3();
			thr = (thr * w) * att;
		} else {
			int res = scatter_attr(sc, ray, rec, p, ctx, dir, att);
			if (res == 2) return thr * att;
			if (res == 0) return V3();
			thr = thr * att;
		}
		ray = Ray(fma3(dir, 0.001f, p), dir, ray.time);
	}
	return V3();
}

}  // namespace

struct omesh_scene { oenv_scene* base = nullptr; Attrs at; };

extern "C" {

// Loads an RTBS v1 - v4 blob: the scene, lights and map through oenv_scene_load, the attributes of a v4 blob.
omesh_scene* omesh_scene_load(const void* blob, size_t size) {
	if (!blob || size < sizeof(rtbs_header)) { g_err = "blob too small"; return nullptr; }
	const uint8_t* p = static_cast<const uint8_t*>(blob);
	rtbs_header h; memcpy(&h, p, sizeof h);
	if (h.magic != RTBS_MAGIC || h.version < 1u || h.version > 4u) { g_err = "bad magic/version"; return nullptr; }
	auto s = std::make_unique<omesh_scene>();
	const size_t v1 = sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) + (size_t)h.n_materials * sizeof(rtbs_material) +
	                  (size_t)h.n_objects * sizeof(rtbs_object) + (size_t)h.n_children * 4 + h.n_blob_bytes;
	if (size < v1) { g_err = "blob truncated"; return nullptr; }
	s->at.aux.assign(h.n_objects, 0);
	if (h.version < 4u) {
		s->base = oenv_scene_load(blob, size);
		return s->base ? s.release() : nullptr;
	}
	int32_t nl = 0;
	if (size < v1 + 4) { g_err = "blob truncated (light list)"; return nullptr; }
	memcpy(&nl, p + v1, 4);
	if (nl < 0 || nl > RTB_MAX_SAMPLED_LIGHTS) { g_err = "bad light list"; return nullptr; }
	const size_t v2 = v1 + 4 + 4 * (size_t)nl;
	rtbs_env eh;
	if (size < v2 + sizeof eh) { g_err = "blob truncated (environment map)"; return nullptr; }
	memcpy(&eh, p + v2, sizeof eh);
	const bool has_env = eh.width > 0 || eh.height > 0;
	if (has_env && (eh.width < 1 || eh.height < 1 || eh.width > RTB_ENV_MAX_SIZE || eh.height > RTB_ENV_MAX_SIZE)) { g_err = "bad environment map"; return nullptr; }
	const size_t v3 = v2 + sizeof eh + (has_env ? (size_t)eh.width * eh.height * 12 : 0);
	uint32_t na = 0;
	if (size < v3 + 4) { g_err = "blob truncated (triangle attributes)"; return nullptr; }
	memcpy(&na, p + v3, 4);
	if (size < v3 + 4 + (size_t)na * sizeof(rtbs_tri_attr)) { g_err = "blob truncated (triangle attributes)"; return nullptr; }
	s->at.rec.resize(na);
	if (na) memcpy(s->at.rec.data(), p + v3 + 4, (size_t)na * sizeof(rtbs_tri_attr));
	for (uint32_t k = 0; k < h.n_objects; ++k) {
		rtbs_object o; memcpy(&o, p + sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) + (size_t)h.n_materials * sizeof(rtbs_material) + (size_t)k * sizeof o, sizeof o);
		if (o.kind != RTB_OBJ_TRIANGLE || o.aux == 0) continue;
		if (o.aux < 0 || (uint32_t)o.aux > na) { g_err = "bad triangle attribute index"; return nullptr; }
		s->at.aux[k] = o.aux;
	}
	// the scene part as the blob a v1 - v3 reader expects
	std::vector<uint8_t> b(p, p + (has_env ? v3 : nl > 0 ? v2 : v1));
	const uint32_t ver = has_env ? 3u : nl > 0 ? 2u : 1u; memcpy(b.data() + 4, &ver, 4);
	s->base = oenv_scene_load(b.data(), b.size());
	return s->base ? s.release() : nullptr;
}
void omesh_scene_free(omesh_scene* s) { if (s) { oenv_scene_free(s->base); delete s; } }

// The attribute table as read (n records of 16 floats: normals, UVs, flags as a float-sized int), and the count.
int omesh_attr_count(const omesh_scene* s) { return s ? (int)s->at.rec.size() : -1; }
void omesh_attrs(const omesh_scene* s, rtbs_tri_attr* out) { if (!s->at.rec.empty()) memcpy(out, s->at.rec.data(), s->at.rec.size() * sizeof(rtbs_tri_attr)); }

// orc_trace_rays with the attribute walk: n is the shading normal, (u, v) the interpolated coordinates.
int omesh_trace_rays(const omesh_scene* s, const rtb_ray* rays, size_t n, rtb_hit* out) {
	if (!s || (n && (!rays || !out))) { g_err = "omesh_trace_rays: bad argument"; return -1; }
	const Scene& sc = s->base->base->base->sc;
	for (size_t i = 0; i < n; ++i) {
		Ray r(V3(rays[i].o[0], rays[i].o[1], rays[i].o[2]), V3(rays[i].d[0], rays[i].d[1], rays[i].d[2]), rays[i].time);
		Ctx ctx; ctx.skip_media = true; ctx.want_uv = true;
		MRec rec;
		rtb_hit h; memset(&h, 0, sizeof h);
		if (!hit_attr(sc.root.get(), r, rec, ctx, s->at)) { h.t = MISS_DIST; h.prim = -1; h.object = -1; h.material = -1; out[i] = h; continue; }
		V3 p = r.at(rec.distance);
		h.t = rec.distance; h.prim = -1; h.object = rec.object; h.material = rec.material;
		h.p[0] = p.x; h.p[1] = p.y; h.p[2] = p.z;
		h.n[0] = rec.normal.x; h.n[1] = rec.normal.y; h.n[2] = rec.normal.z;
		h.front_face = dot(r.d, rec.n_geom) > 0.0f ? 0 : 1;
		h.u = rec.u; h.v = rec.v;
		out[i] = h;
	}
	return 0;
}

// oenv_render with the attributes (Philox streams only).
int omesh_render(const omesh_scene* s, const rtb_camera* cam, uint32_t W, uint32_t H, uint32_t s0, uint32_t s1, uint32_t max_depth,
                 uint32_t seed, int mode, int threads, float* sum, float* sum2, uint64_t* rays_out) {
	if (!s || !cam || !sum || W == 0 || H == 0) { g_err = "omesh_render: bad argument"; return -1; }
	if (mode != ORC_RNG_PHILOX) { g_err = "omesh_render: render in Philox mode"; return -1; }
	if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
	if (threads <= 0) threads = 1;
	const Scene& sc = s->base->base->base->sc;
	const std::vector<Light>& lights = s->base->base->lights;
	const Env* env = s->base->has_env ? &s->base->env : nullptr;
	std::atomic<uint32_t> next_row{0};
	std::atomic<uint64_t> total_rays{0};
	const float px = 1.0f / (float)W, py = 1.0f / (float)H;
	auto worker = [&]() {
		uint64_t rays = 0;
		for (;;) {
			uint32_t y = next_row.fetch_add(1);
			if (y >= H) break;
			for (uint32_t x = 0; x < W; ++x) {
				uint32_t gid = y * W + x;
				Ctx ctx; ctx.mode = ORC_RNG_PHILOX; ctx.seed = seed; ctx.pixel = gid; ctx.want_uv = sc.any_uv_texture;
				float ndcx = std::fmaf(((float)x + 0.5f) * px, 2.0f, -1.0f);
				float ndcy = std::fmaf(((float)y + 0.5f) * py, 2.0f, -1.0f);
				float ax = 0, ay = 0, az = 0, qx = 0, qy = 0, qz = 0;
				for (uint32_t smp = s0; smp < s1; ++smp) {
					ctx.sample = smp;
					ctx.begin(CAMERA_BOUNCE);
					float jx, jy; ctx.in_unit_disc(jx, jy, false);
					Ray ray = camera_ray(*cam, std::fmaf(jx, px, ndcx), std::fmaf(jy, py, ndcy), ctx);
					V3 c = sample_world_attr(sc, lights, env, s->at, ray, max_depth, ctx);
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
	return 0;
}

}  // extern "C"
