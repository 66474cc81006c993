// tests/env_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's integrator with an HDR environment map.
//
// An independent CPU restatement of DESIGN.md §5d ("Environment map"), built on top of the light-sampling oracle: this file
// includes tests/light_oracle.cpp (and through it oracle/oracle.cpp) unchanged and reuses its scene, lights, light pdfs and
// Philox streams; what it adds is the map read from an RTBS v3 blob, its sampling tables, lookup, sampler and pdf, the
// mixture with the map as one more strategy, and the integrator that uses them.  tests/env_oracle.py compiles it
// (g++ -ffp-contract=off, like the oracle) into a temporary directory on first use.
#include "light_oracle.cpp"

namespace {

// The map: scaled texels (row 0 = top), the pdf numerator per texel and the CDFs, built as §5d "Sampling" states.
struct Env {
	int W = 0, H = 0;
	bool sample = false;
	std::vector<float> rgb;    // H x W x 3
	std::vector<float> pdf;    // H x W: p_ij * W * H / (2 pi^2)
	std::vector<float> cm;     // H + 1
	std::vector<float> cc;     // H x (W + 1)
	double total = 0.0;
};

void env_build(Env& e) {
	const double kPi = 3.14159265358979323846;
	const int W = e.W, H = e.H;
	e.cm.assign(H + 1, 0.0f); e.cc.assign((size_t)H * (W + 1), 0.0f); e.pdf.assign((size_t)W * H, 0.0f);
	std::vector<double> row(H, 0.0);
	for (int j = 0; j < H; ++j) {
		const double st = std::sin(kPi * (j + 0.5) / H);
		std::vector<double> pre(W);
		double acc = 0.0;
		for (int i = 0; i < W; ++i) {
			const float* t = &e.rgb[((size_t)j * W + i) * 3];
			acc += (0.2126 * t[0] + 0.7152 * t[1] + 0.0722 * t[2]) * st;
			pre[i] = acc;
		}
		row[j] = acc;
		float* c = &e.cc[(size_t)j * (W + 1)];
		c[0] = 0.0f;
		for (int i = 1; i < W; ++i) c[i] = acc > 0.0 ? (float)(pre[i - 1] / acc) : (float)((double)i / W);
		c[W] = 1.0f;
	}
	double total = 0.0;
	for (int j = 0; j < H; ++j) total += row[j];
	e.total = total;
	double acc = 0.0;
	for (int j = 1; j < H; ++j) { acc += row[j - 1]; e.cm[j] = total > 0.0 ? (float)(acc / total) : (float)((double)j / H); }
	e.cm[0] = 0.0f; e.cm[H] = 1.0f;
	for (int j = 0; j < H; ++j) {
		const double pj = total > 0.0 ? (double)e.cm[j + 1] - (double)e.cm[j] : 0.0;
		const float* c = &e.cc[(size_t)j * (W + 1)];
		for (int i = 0; i < W; ++i)
			e.pdf[(size_t)j * W + i] = (float)(pj * ((double)c[i + 1] - (double)c[i]) * ((double)W * (double)H / (2.0 * kPi * kPi)));
	}
}

// Lookup (§5d "Lookup"): texel index of direction d and sin(theta) of its unit vector.
size_t env_index(const Env& e, V3 d, float& sin_theta) {
	const float inv = 1.0f / std::sqrt(dot(d, d));
	const V3 n(d.x * inv, d.y * inv, d.z * inv);
	float u, v; sphere_uv(n, u, v);
	int i = (int)(u * (float)e.W), j = (int)((1.0f - v) * (float)e.H);
	if (i > e.W - 1) i = e.W - 1;
	if (j > e.H - 1) j = e.H - 1;
	sin_theta = std::sqrt(std::fmaf(n.x, n.x, n.z * n.z));
	return (size_t)j * e.W + i;
}
V3 env_radiance(const Env& e, V3 d) {
	float st; const float* t = &e.rgb[3 * env_index(e, d, st)];
	return V3(t[0], t[1], t[2]);
}
float env_pdf(const Env& e, V3 u) {
	float st; const float num = e.pdf[env_index(e, u, st)];
	return st > 0.0f ? num / st : 0.0f;
}
int cdf_invert(const float* c, int n, float x, float& frac) {
	x = std::fmin(x, 0.99999994f);
	int lo = 0, hi = n;
	while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (c[mid] <= x) lo = mid; else hi = mid; }
	frac = (x - c[lo]) / (c[lo + 1] - c[lo]);
	return lo;
}
V3 env_direction(const Env& e, float zr, float zc) {
	float fr, fc;
	const int j = cdf_invert(e.cm.data(), e.H, zr, fr);
	const int i = cdf_invert(&e.cc[(size_t)j * (e.W + 1)], e.W, zc, fc);
	const float v = 1.0f - ((float)j + fr) / (float)e.H;
	const float u = ((float)i + fc) / (float)e.W;
	float st, ct, sp, cp;
	sincos2pi(0.5f * v, st, ct);
	sincos2pi(u, sp, cp);
	return V3(-(st * cp), -ct, st * sp);
}

// light_mix of tests/light_oracle.cpp with the map as strategy n of n + 1 when it is sampled.
bool env_light_mix(const std::vector<Light>& lights, const Env* env, bool iso, V3 p, V3 n, Ctx& ctx, V3& dir, float& w) {
	F4 l = rng4(ctx.seed, ctx.pixel, ctx.sample, ctx.bounce, STREAM_LIGHT);
	const int nl = (int)lights.size();
	const bool es = env && env->sample;
	const int m = es ? nl + 1 : nl;
	if (l.x < 0.5f) {
		int k = (int)(l.y * (float)m); if (k > m - 1) k = m - 1;
		if (es && k == nl) {
			dir = env_direction(*env, l.z, l.w);
		} else {
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
	if (es) sum += env_pdf(*env, u);
	float mixture = std::fmaf(0.5f, sum / (float)m, 0.5f * spdf);
	if (!(mixture > 0.0f)) return false;
	w = spdf / mixture;
	return w > 0.0f;
}

// sample_world_lit of tests/light_oracle.cpp with the map: a miss returns thr * texel; the mixture runs when there are
// lights or a sampled map.
V3 sample_world_env(const Scene& sc, const std::vector<Light>& lights, const Env* env, Ray ray, uint32_t max_depth, Ctx& ctx) {
	V3 thr(1, 1, 1);
	const bool mix = !lights.empty() || (env && env->sample);
	for (uint32_t i = 0; i < max_depth; ++i) {
		Rec rec;
		ctx.begin(i);
		ctx.rays++;
		if (!hit(sc.root.get(), ray, rec, ctx)) return thr * (env ? env_radiance(*env, ray.d) : background(sc, ray.d));
		V3 p = ray.at(rec.distance);
		V3 dir, att;
		const rtbs_material& m = sc.materials[rec.material];
		if (mix && (m.kind == RTB_MAT_LAMBERTIAN || m.kind == RTB_MAT_ISOTROPIC)) {
			att = m.tex >= 0 ? texture_value(sc, m.tex, rec.u, rec.v, p) : V3(m.albedo[0], m.albedo[1], m.albedo[2]);
			float w;
			if (!env_light_mix(lights, env, m.kind == RTB_MAT_ISOTROPIC, p, rec.normal, ctx, dir, w)) return V3();
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

struct oenv_scene { orl_scene* base = nullptr; bool has_env = false; Env env; };

extern "C" {

// Loads an RTBS v1, v2 or v3 blob: the scene and its light list through orl_scene_load (as v1 / v2), the map of a v3 blob.
oenv_scene* oenv_scene_load(const void* blob, size_t size) {
	if (!blob || size < sizeof(rtbs_header)) { g_err = "blob too small"; return nullptr; }
	const uint8_t* p = static_cast<const uint8_t*>(blob);
	rtbs_header h; memcpy(&h, p, sizeof h);
	if (h.magic != RTBS_MAGIC || h.version < 1u || h.version > 3u) { g_err = "bad magic/version"; return nullptr; }
	auto s = std::make_unique<oenv_scene>();
	if (h.version < 3u) {
		s->base = orl_scene_load(blob, size);
		return s->base ? s.release() : nullptr;
	}
	const size_t v1 = sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture) + (size_t)h.n_materials * sizeof(rtbs_material) +
	                  (size_t)h.n_objects * sizeof(rtbs_object) + (size_t)h.n_children * 4 + h.n_blob_bytes;
	int32_t nl = 0;
	if (size < v1 + 4) { g_err = "blob truncated (light list)"; return nullptr; }
	memcpy(&nl, p + v1, 4);
	if (nl < 0 || nl > RTB_MAX_SAMPLED_LIGHTS) { g_err = "bad light list"; return nullptr; }
	const size_t v2 = v1 + 4 + 4 * (size_t)nl;
	rtbs_env eh;
	if (size < v2 + sizeof eh) { g_err = "blob truncated (environment map)"; return nullptr; }
	memcpy(&eh, p + v2, sizeof eh);
	if (eh.width < 1 || eh.height < 1 || eh.width > RTB_ENV_MAX_SIZE || eh.height > RTB_ENV_MAX_SIZE ||
	    size < v2 + sizeof eh + (size_t)eh.width * eh.height * 12) { g_err = "bad environment map"; return nullptr; }
	// the scene part as the blob a v1 (no lights) or v2 reader expects
	std::vector<uint8_t> b(p, p + (nl > 0 ? v2 : v1));
	const uint32_t ver = nl > 0 ? 2u : 1u; memcpy(b.data() + 4, &ver, 4);
	s->base = orl_scene_load(b.data(), b.size());
	if (!s->base) return nullptr;
	s->has_env = true;
	s->env.W = eh.width; s->env.H = eh.height; s->env.sample = (eh.flags & RTB_ENV_SAMPLE) != 0;
	s->env.rgb.resize((size_t)eh.width * eh.height * 3);
	memcpy(s->env.rgb.data(), p + v2 + sizeof eh, s->env.rgb.size() * 4);
	env_build(s->env);
	return s.release();
}
void oenv_scene_free(oenv_scene* s) { if (s) { orl_scene_free(s->base); delete s; } }

// The map's pieces, for the sampler tests (the scene must carry a map).
int oenv_dims(const oenv_scene* s, int* wh) { if (!s || !s->has_env) return -1; wh[0] = s->env.W; wh[1] = s->env.H; return 0; }
void oenv_tables(const oenv_scene* s, float* pdf_num, float* cm, float* cc) {
	memcpy(pdf_num, s->env.pdf.data(), s->env.pdf.size() * 4);
	memcpy(cm, s->env.cm.data(), s->env.cm.size() * 4);
	memcpy(cc, s->env.cc.data(), s->env.cc.size() * 4);
}
// n directions drawn with the uniforms z[2k], z[2k + 1]; dir[3k..], their texel index and pdf
void oenv_sample(const oenv_scene* s, const float* z, int n, float* dir, int64_t* texel, float* pdf) {
	for (int k = 0; k < n; ++k) {
		V3 d = env_direction(s->env, z[2 * k], z[2 * k + 1]);
		dir[3 * k] = d.x; dir[3 * k + 1] = d.y; dir[3 * k + 2] = d.z;
		float st; texel[k] = (int64_t)env_index(s->env, d, st);
		pdf[k] = env_pdf(s->env, d);
	}
}
// texel index and pdf of n given directions
void oenv_lookup(const oenv_scene* s, const float* dir, int n, int64_t* texel, float* pdf) {
	for (int k = 0; k < n; ++k) {
		V3 d(dir[3 * k], dir[3 * k + 1], dir[3 * k + 2]);
		float st; texel[k] = (int64_t)env_index(s->env, d, st);
		pdf[k] = env_pdf(s->env, d);
	}
}

// orl_render with the map (Philox streams only).
int oenv_render(const oenv_scene* s, const rtb_camera* cam, uint32_t W, uint32_t H, uint32_t s0, uint32_t s1, uint32_t max_depth,
                uint32_t seed, int mode, int threads, float* sum, float* sum2, uint64_t* rays_out) {
	if (!s || !cam || !sum || W == 0 || H == 0) { g_err = "oenv_render: bad argument"; return -1; }
	if (mode != ORC_RNG_PHILOX) { g_err = "oenv_render: render in Philox mode"; return -1; }
	if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
	if (threads <= 0) threads = 1;
	const Scene& sc = s->base->base->sc;
	const std::vector<Light>& lights = s->base->lights;
	const Env* env = s->has_env ? &s->env : nullptr;
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
					V3 c = sample_world_env(sc, lights, env, ray, max_depth, ctx);
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
