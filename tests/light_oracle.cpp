// tests/light_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's integrator with light importance sampling.
//
// An independent CPU restatement of DESIGN.md §5b ("Light sampling"), built on top of the CPU oracle: this file includes
// oracle/oracle.cpp unchanged and reuses its scene graph, intersection, materials, textures, camera and Philox streams;
// what it adds is the light table (from an RTBS v2 blob's light list), the mixture scatter and the integrator that uses it.
// tests/light_oracle.py compiles it (g++ -ffp-contract=off, like the oracle) into a temporary directory on first use.
#include "../oracle/oracle.cpp"

namespace {

// A sampled light in world space: a sphere (c, R) or a quad node (the book's quad constants) with its area.
struct Light {
	bool quad = false;
	V3 c; float R = 0.0f;
	Node q; float area = 0.0f;
};

// The world-from-object transform of a translate / rotate_y chain, composed from the listed object down.
struct ChainXf {
	float c = 1.0f, s = 0.0f; V3 off; bool rot = false, tr = false;
	V3 vec(V3 p) const {
		if (!rot) return p;
		return V3(std::fmaf(c, p.x, s * p.z), p.y, std::fmaf(c, p.z, -(s * p.x)));
	}
	V3 point(V3 p) const { V3 r = vec(p); return tr ? r + off : r; }
};

bool build_light(const rtbs_object* objs, const int32_t* children, uint32_t n_objects, uint32_t n_children, int id, Light& L) {
	ChainXf x;
	int cur = id;
	for (int guard = 0; guard < 64; ++guard) {
		if (cur < 0 || (uint32_t)cur >= n_objects) { g_err = "sampled light: bad object id"; return false; }
		const rtbs_object& o = objs[cur];
		if (o.kind == RTB_OBJ_TRANSLATE || o.kind == RTB_OBJ_ROTATE_Y) {
			if (o.child_begin < 0 || (uint32_t)o.child_begin >= n_children) { g_err = "sampled light: bad child index"; return false; }
			if (o.kind == RTB_OBJ_TRANSLATE) { x.off = x.point(V3(o.f[0], o.f[1], o.f[2])); x.tr = true; }
			else {
				float sn = o.f[1], cs = o.f[2];
				if (x.rot) { float c = x.c * cs - x.s * sn, s = x.s * cs + x.c * sn; x.c = c; x.s = s; }
				else { x.c = cs; x.s = sn; }
				x.rot = true;
			}
			cur = children[o.child_begin];
			continue;
		}
		if (o.kind == RTB_OBJ_SPHERE) {
			L.quad = false; L.c = x.point(V3(o.f[0], o.f[1], o.f[2])); L.R = std::fabs(o.f[3]);
			if (!(L.R > 0.0f)) { g_err = "sampled light: sphere without radius"; return false; }
			return true;
		}
		if (o.kind == RTB_OBJ_QUAD) {
			V3 Q = x.point(V3(o.f[0], o.f[1], o.f[2])), u = x.vec(V3(o.f[3], o.f[4], o.f[5])), v = x.vec(V3(o.f[6], o.f[7], o.f[8]));
			L.quad = true; L.q.kind = RTB_OBJ_QUAD; init_quad(L.q, Q, u, v);
			V3 nn = cross(u, v);
			L.area = std::sqrt(dot(nn, nn));
			if (!(L.area > 0.0f)) { g_err = "sampled light: quad without area"; return false; }
			return true;
		}
		g_err = "sampled light: only spheres and quads (under translate / rotate_y) can be sampled";
		return false;
	}
	g_err = "sampled light: chain too deep";
	return false;
}

// book 3 sphere::pdf_value / random_to_sphere, in the spec's operation order
float cone_cos_max(float d2, float R2) { return std::sqrt(1.0f - R2 / d2); }
float cone_pdf(float cmax) { return 1.0f / (6.28318530717958647692f * (1.0f - cmax)); }
V3 cone_direction(V3 e, float cmax, float u0, float u1) {
	float z = std::fmaf(u1, cmax - 1.0f, 1.0f);
	float z2 = std::fmaf(-z, z, 1.0f);
	float sz = std::sqrt(z2 < 0.0f ? 0.0f : z2);
	float sn, cs; sincos2pi(u0, sn, cs);
	float x = cs * sz, y = sn * sz;
	V3 W = normalize(e);
	V3 A = std::fabs(W.x) > 0.9f ? V3(0, 1, 0) : V3(1, 0, 0);
	V3 Vb = normalize(cross(W, A));
	V3 U = cross(W, Vb);
	return normalize(V3(std::fmaf(z, W.x, std::fmaf(y, Vb.x, x * U.x)), std::fmaf(z, W.y, std::fmaf(y, Vb.y, x * U.y)),
	                    std::fmaf(z, W.z, std::fmaf(y, Vb.z, x * U.z))));
}

const uint32_t STREAM_LIGHT = 2;

// pdf of light L's own sampling for the unit direction u from p (step 5)
float light_pdf(const Light& L, V3 p, V3 u) {
	Ray r(p, u);
	if (L.quad) {
		float t = planar_t(L.q, r, 0.0f, MISS_DIST, true);
		if (!(t > 0.0f) || !(t < MISS_DIST)) return 0.0f;
		return (t * t) / (std::fabs(dot(u, L.q.N)) * L.area);
	}
	V3 e = L.c - p;
	float d2 = dot(e, e), R2 = L.R * L.R;
	if (!(d2 > R2)) return 0.0f;
	if (!(sphere_closest(r, L.c, L.R) < MISS_DIST)) return 0.0f;
	return cone_pdf(cone_cos_max(d2, R2));
}

// The mixture of the material's directions and directions towards the sampled lights (steps 1-6).
bool light_mix(const std::vector<Light>& lights, bool iso, V3 p, V3 n, Ctx& ctx, V3& dir, float& w) {
	F4 l = rng4(ctx.seed, ctx.pixel, ctx.sample, ctx.bounce, STREAM_LIGHT);
	const int nl = (int)lights.size();
	if (l.x < 0.5f) {
		int k = (int)(l.y * (float)nl); if (k > nl - 1) k = nl - 1;
		const Light& L = lights[k];
		if (L.quad) {
			V3 e = fma3(L.q.Vv, l.w, fma3(L.q.U, l.z, L.q.Q)) - p;
			if (!(dot(e, e) > 0.0f)) return false;
			dir = normalize(e);
		} else {
			V3 e = L.c - p;
			float d2 = dot(e, e), R2 = L.R * L.R;
			if (!(d2 > R2)) return false;
			dir = cone_direction(e, cone_cos_max(d2, R2), l.z, l.w);
		}
	} else if (iso) {
		dir = ctx.on_unit_sphere();
	} else {
		dir = n + ctx.on_unit_sphere();
		if (near_zero(dir)) return false;
	}
	V3 u = normalize(dir);
	float spdf = iso ? 0.07957747154594767f : std::fmax(0.0f, dot(n, u)) * 0.31830988618379067f;
	if (!(spdf > 0.0f)) return false;
	float sum = 0.0f;
	for (const Light& L : lights) sum += light_pdf(L, p, u);
	float mixture = std::fmaf(0.5f, sum / (float)nl, 0.5f * spdf);
	if (!(mixture > 0.0f)) return false;
	w = spdf / mixture;
	return w > 0.0f;
}

// sample_world with the mixture at Lambertian and isotropic scatters when there are lights to sample (step 7: throughput
// (thr * w) * albedo); every other material goes through the oracle's own scatter.
V3 sample_world_lit(const Scene& sc, const std::vector<Light>& lights, Ray ray, uint32_t max_depth, Ctx& ctx) {
	V3 thr(1, 1, 1);
	for (uint32_t i = 0; i < max_depth; ++i) {
		Rec rec;
		ctx.begin(i);
		ctx.rays++;
		if (!hit(sc.root.get(), ray, rec, ctx)) return thr * background(sc, ray.d);
		V3 p = ray.at(rec.distance);
		V3 dir, att;
		const rtbs_material& m = sc.materials[rec.material];
		if (!lights.empty() && (m.kind == RTB_MAT_LAMBERTIAN || m.kind == RTB_MAT_ISOTROPIC)) {
			att = m.tex >= 0 ? texture_value(sc, m.tex, rec.u, rec.v, p) : V3(m.albedo[0], m.albedo[1], m.albedo[2]);
			float w;
			if (!light_mix(lights, m.kind == RTB_MAT_ISOTROPIC, p, rec.normal, ctx, dir, w)) return V3();
			thr = (thr * w) * att;
		} else {
			int res = scatter(sc, ray, rec, p, ctx, dir, att);
			if (res == 2) return thr * att;
			if (res == 0) return V3();
			thr = thr * att;
		}
		ray = Ray(fma3(dir, 0.001f, p), dir, ray.time);
	}
	return V3();
}

}  // namespace

struct orl_scene { orc_scene* base = nullptr; std::vector<Light> lights; };

extern "C" {

// Loads an RTBS v1 or v2 blob: the scene through orc_scene_load (as v1), the light list of a v2 blob into world space.
orl_scene* orl_scene_load(const void* blob, size_t size) {
	if (!blob || size < sizeof(rtbs_header)) { g_err = "blob too small"; return nullptr; }
	const uint8_t* p = static_cast<const uint8_t*>(blob);
	rtbs_header h; memcpy(&h, p, sizeof h);
	if (h.magic != RTBS_MAGIC || (h.version != 1u && h.version != 2u)) { g_err = "bad magic/version"; return nullptr; }
	const size_t v1 = sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) + (size_t)h.n_materials * sizeof(rtbs_material) +
	                  (size_t)h.n_objects * sizeof(rtbs_object) + (size_t)h.n_children * 4 + h.n_blob_bytes;
	if (size < v1) { g_err = "blob truncated"; return nullptr; }
	std::vector<int32_t> ids;
	if (h.version == 2u) {   // int32 n_lights, int32 objects[n_lights] after the v1 blob
		int32_t nl = 0;
		if (size < v1 + 4) { g_err = "blob truncated (light list)"; return nullptr; }
		memcpy(&nl, p + v1, 4);
		if (nl < 1 || nl > RTB_MAX_SAMPLED_LIGHTS || size < v1 + 4 + 4 * (size_t)nl) { g_err = "bad light list"; return nullptr; }
		ids.resize(nl); memcpy(ids.data(), p + v1 + 4, 4 * (size_t)nl);
	}
	std::vector<uint8_t> b(p, p + v1);
	const uint32_t one = 1u; memcpy(b.data() + 4, &one, 4);
	auto s = std::make_unique<orl_scene>();
	s->base = orc_scene_load(b.data(), b.size());
	if (!s->base) return nullptr;
	const rtbs_object* objs = reinterpret_cast<const rtbs_object*>(b.data() + sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) +
	                                                                (size_t)h.n_materials * sizeof(rtbs_material));
	const int32_t* children = reinterpret_cast<const int32_t*>(reinterpret_cast<const uint8_t*>(objs) + (size_t)h.n_objects * sizeof(rtbs_object));
	for (int32_t id : ids) {
		Light L;
		if (!build_light(objs, children, h.n_objects, h.n_children, id, L)) { orc_scene_free(s->base); return nullptr; }
		s->lights.push_back(std::move(L));
	}
	return s.release();
}
void orl_scene_free(orl_scene* s) { if (s) { orc_scene_free(s->base); delete s; } }
int orl_num_lights(const orl_scene* s) { return s ? (int)s->lights.size() : -1; }

// orc_render with the light mixture; Philox streams only (XORWOW is the reference's mode, and the reference has no
// light sampling).
int orl_render(const orl_scene* s, const rtb_camera* cam, uint32_t W, uint32_t H, uint32_t s0, uint32_t s1, uint32_t max_depth,
               uint32_t seed, int mode, int threads, float* sum, float* sum2, uint64_t* rays_out) {
	if (!s || !cam || !sum || W == 0 || H == 0) { g_err = "orl_render: bad argument"; return -1; }
	if (mode != ORC_RNG_PHILOX) { g_err = "orl_render: XORWOW mode reproduces the reference, which has no light sampling: render in Philox mode"; return -1; }
	if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
	if (threads <= 0) threads = 1;
	const Scene& sc = s->base->sc;
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
					V3 c = sample_world_lit(sc, s->lights, ray, max_depth, ctx);
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
