// tests/rough_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's integrator with the GGX microfacet materials
// (rough metal, rough dielectric).
//
// An independent CPU restatement of DESIGN.md §5f ("Rough metal and rough glass"), built on top of the triangle-attribute
// oracle: this file includes tests/mesh_oracle.cpp (and through it the environment-map, light and plain oracles) unchanged
// and reuses its scene, lights, map, attribute walk, materials and Philox streams.  What it adds is the table of GGX widths
// read from an RTBS v5 blob, the two scatters, and the integrator that uses them.  tests/rough_oracle.py compiles it
// (g++ -ffp-contract=off, like the oracle) into a temporary directory on first use.
#include "mesh_oracle.cpp"

namespace {

// Smith Lambda of a local direction, a2 = alpha^2 (§5f step 3)
float ggx_lambda(V3 w, float a2) {
	const float t = std::fmaf(w.y, w.y, w.x * w.x) / (w.z * w.z);
	return (std::sqrt(std::fmaf(a2, t, 1.0f)) - 1.0f) * 0.5f;
}

// §5f steps 1-6 for one scatter.  n = the frame normal, ratio = the dielectric's ior ratio (unused for the metal),
// r = the bounce's STREAM_SCATTER block.  0 = black, 1 = scattered.
int rough_scatter(bool diel, V3 n, V3 d, F4 r, float alpha, float ratio, V3 albedo, V3& dir, V3& att) {
	const V3 wo_w = -normalize(d);
	const V3 A = std::fabs(n.x) > 0.9f ? V3(0.0f, 1.0f, 0.0f) : V3(1.0f, 0.0f, 0.0f);
	const V3 Vb = normalize(cross(n, A));
	const V3 Ub = cross(n, Vb);
	const V3 wo(dot(wo_w, Ub), dot(wo_w, Vb), dot(wo_w, n));
	if (!(wo.z > 0.0f)) return 0;
	const V3 wh = normalize(V3(alpha * wo.x, alpha * wo.y, wo.z));
	float sn, cs; sincos2pi(r.x, sn, cs);
	const float z = std::fmaf(1.0f - r.y, 1.0f + wh.z, -wh.z);
	const float st = std::sqrt(std::fmax(0.0f, std::fmaf(-z, z, 1.0f)));
	const V3 h(st * cs + wh.x, st * sn + wh.y, z + wh.z);
	if (!(dot(h, h) > 0.0f)) return 0;
	const V3 wm = normalize(V3(alpha * h.x, alpha * h.y, h.z));
	const float cos_om = dot(wo, wm);
	if (!(cos_om > 0.0f)) return 0;
	V3 wi;
	if (!diel) {
		wi = reflect(-wo, wm);
		if (!(wi.z > 0.0f)) return 0;
	} else {
		const V3 ui = -wo;
		const float cos_theta = std::fmin(cos_om, 1.0f);
		const float sin_theta = std::sqrt(std::fmaf(-cos_theta, cos_theta, 1.0f));
		float r0 = (1.0f - ratio) / (1.0f + ratio); r0 = r0 * r0;
		const float x = 1.0f - cos_theta, x2 = x * x;
		const float prob = std::fmaf(1.0f - r0, x2 * x2 * x, r0);
		if (ratio * sin_theta > 1.0f || prob > r.z) {
			wi = reflect(ui, wm);
			if (!(wi.z > 0.0f)) return 0;
		} else {
			const float dv = dot(wm, ui);
			const float k = std::fmaf(-(ratio * ratio), std::fmaf(-dv, dv, 1.0f), 1.0f);
			if (k < 0.0f) return 0;
			const float coef = std::fmaf(ratio, dv, std::sqrt(k));
			wi = V3(std::fmaf(-coef, wm.x, ratio * ui.x), std::fmaf(-coef, wm.y, ratio * ui.y), std::fmaf(-coef, wm.z, ratio * ui.z));
			if (!(wi.z < 0.0f)) return 0;
		}
	}
	const float a2 = alpha * alpha;
	const float lo = 1.0f + ggx_lambda(wo, a2);
	const float g = lo / (lo + ggx_lambda(wi, a2));
	if (!diel) {
		const float x = 1.0f - cos_om, x2 = x * x, x5 = x2 * x2 * x;
		att = V3(std::fmaf(1.0f - albedo.x, x5, albedo.x) * g, std::fmaf(1.0f - albedo.y, x5, albedo.y) * g, std::fmaf(1.0f - albedo.z, x5, albedo.z) * g);
	} else {
		att = albedo * g;
	}
	dir = V3(std::fmaf(wi.z, n.x, std::fmaf(wi.y, Vb.x, wi.x * Ub.x)), std::fmaf(wi.z, n.y, std::fmaf(wi.y, Vb.y, wi.x * Ub.y)),
	         std::fmaf(wi.z, n.z, std::fmaf(wi.y, Vb.z, wi.x * Ub.z)));
	return 1;
}

// sample_world_attr of tests/mesh_oracle.cpp with the two GGX kinds, which stay out of the light mixture.
V3 sample_world_rough(const Scene& sc, const std::vector<Light>& lights, const Env* env, const Attrs& at, const std::vector<float>& alpha,
                      Ray ray, uint32_t max_depth, Ctx& ctx) {
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
		if (m.kind == RTB_MAT_ROUGH_METAL || m.kind == RTB_MAT_ROUGH_DIELECTRIC) {
			const V3 albedo(m.albedo[0], m.albedo[1], m.albedo[2]);
			int res;
			if (m.kind == RTB_MAT_ROUGH_METAL) {
				res = rough_scatter(false, rec.normal, ray.d, ctx.r, alpha[rec.material], 0.0f, albedo, dir, att);
			} else {
				const bool back = dot(ray.d, rec.n_geom) > 0.0f;
				res = rough_scatter(true, back ? -rec.m : rec.m, ray.d, ctx.r, alpha[rec.material], back ? m.param : 1.0f / m.param, albedo, dir, att);
			}
			if (res == 0) return V3();
			thr = thr * att;
		} else if (mix && (m.kind == RTB_MAT_LAMBERTIAN || m.kind == RTB_MAT_ISOTROPIC)) {
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

struct orough_scene { omesh_scene* base = nullptr; std::vector<float> alpha; };

extern "C" {

// Loads an RTBS v1 - v5 blob: everything but the widths through omesh_scene_load, the widths of a v5 blob.
orough_scene* orough_scene_load(const void* blob, size_t size) {
	if (!blob || size < sizeof(rtbs_header)) { g_err = "blob too small"; return nullptr; }
	const uint8_t* p = static_cast<const uint8_t*>(blob);
	rtbs_header h; memcpy(&h, p, sizeof h);
	if (h.magic != RTBS_MAGIC || h.version < 1u || h.version > 5u) { g_err = "bad magic/version"; return nullptr; }
	auto s = std::make_unique<orough_scene>();
	s->alpha.assign(h.n_materials, 0.0f);
	if (h.version < 5u) {
		s->base = omesh_scene_load(blob, size);
		return s->base ? s.release() : nullptr;
	}
	// the v4 part: v1 content, light list, map record and texels, attribute table
	size_t off = sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) + (size_t)h.n_materials * sizeof(rtbs_material) +
	             (size_t)h.n_objects * sizeof(rtbs_object) + (size_t)h.n_children * 4 + h.n_blob_bytes;
	int32_t nl = 0;
	if (size < off + 4) { g_err = "blob truncated (light list)"; return nullptr; }
	memcpy(&nl, p + off, 4);
	if (nl < 0 || nl > RTB_MAX_SAMPLED_LIGHTS) { g_err = "bad light list"; return nullptr; }
	off += 4 + 4 * (size_t)nl;
	rtbs_env eh;
	if (size < off + sizeof eh) { g_err = "blob truncated (environment map)"; return nullptr; }
	memcpy(&eh, p + off, sizeof eh);
	if (eh.width < 0 || eh.height < 0 || eh.width > RTB_ENV_MAX_SIZE || eh.height > RTB_ENV_MAX_SIZE) { g_err = "bad environment map"; return nullptr; }
	off += sizeof eh + (size_t)eh.width * eh.height * 12;
	uint32_t na = 0;
	if (size < off + 4) { g_err = "blob truncated (triangle attributes)"; return nullptr; }
	memcpy(&na, p + off, 4);
	off += 4 + (size_t)na * sizeof(rtbs_tri_attr);
	uint32_t nm = 0;
	if (size < off + 4) { g_err = "blob truncated (GGX widths)"; return nullptr; }
	memcpy(&nm, p + off, 4);
	if (nm != h.n_materials || size != off + 4 + 4 * (size_t)nm) { g_err = "bad GGX width table"; return nullptr; }
	if (nm) memcpy(s->alpha.data(), p + off + 4, 4 * (size_t)nm);
	for (uint32_t k = 0; k < nm; ++k) {
		rtbs_material m; memcpy(&m, p + sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) + (size_t)k * sizeof m, sizeof m);
		const bool rough = m.kind == RTB_MAT_ROUGH_METAL || m.kind == RTB_MAT_ROUGH_DIELECTRIC;
		if (rough && !(s->alpha[k] >= 0.001f && s->alpha[k] <= 1.0f)) { g_err = "bad GGX width"; return nullptr; }
	}
	// the rest as the v4 blob omesh_scene_load reads
	std::vector<uint8_t> b(p, p + off);
	const uint32_t ver = 4u; memcpy(b.data() + 4, &ver, 4);
	s->base = omesh_scene_load(b.data(), b.size());
	return s->base ? s.release() : nullptr;
}
void orough_scene_free(orough_scene* s) { if (s) { omesh_scene_free(s->base); delete s; } }

// The widths as read (one per material), and their count.
int orough_alpha_count(const orough_scene* s) { return s ? (int)s->alpha.size() : -1; }
void orough_alphas(const orough_scene* s, float* out) { if (!s->alpha.empty()) memcpy(out, s->alpha.data(), s->alpha.size() * 4); }

// omesh_render with the GGX materials (Philox streams only).
int orough_render(const orough_scene* s, const rtb_camera* cam, uint32_t W, uint32_t H, uint32_t s0, uint32_t s1, uint32_t max_depth,
                  uint32_t seed, int mode, int threads, float* sum, float* sum2, uint64_t* rays_out) {
	if (!s || !cam || !sum || W == 0 || H == 0) { g_err = "orough_render: bad argument"; return -1; }
	if (mode != ORC_RNG_PHILOX) { g_err = "orough_render: render in Philox mode"; return -1; }
	if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
	if (threads <= 0) threads = 1;
	const Scene& sc = s->base->base->base->base->sc;
	const std::vector<Light>& lights = s->base->base->base->lights;
	const Env* env = s->base->base->has_env ? &s->base->base->env : nullptr;
	const Attrs& at = s->base->at;
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
					V3 c = sample_world_rough(sc, lights, env, at, s->alpha, ray, max_depth, ctx);
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
