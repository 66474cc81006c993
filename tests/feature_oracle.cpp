// tests/feature_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's integrator with every feature the plain oracle lacks.
//
// An independent CPU restatement of DESIGN.md §5b (light sampling), §5d (environment map), §5e (triangle attributes) and
// §5f (rough metal and rough glass), built on top of the CPU oracle: this file includes oracle/oracle.cpp unchanged and
// reuses its scene graph, intersection, materials, textures, camera, Philox streams and render loop.  What it adds is one
// loader for RTBS v1 - v5 (the light list, the map, the attribute table and the GGX widths), the light and map mixture,
// the attribute walk, the GGX scatters, and the one integrator that uses them.  A new feature extends this loader and this
// integrator; the plain oracle keeps refusing any version above 1.  tests/feature_oracle.py compiles it
// (g++ -ffp-contract=off, like the oracle) into a temporary directory on first use.
#include "../oracle/oracle.cpp"

namespace {

// ---------------------------------------------------------------- sampled lights (§5b)

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

// pdf of light L's own sampling for the unit direction u from p (§5b step 5)
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

// ---------------------------------------------------------------- environment map (§5d)

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

// The mixture of the material's directions and directions towards the sampled lights (§5b steps 1-6), with the map as
// strategy n of n + 1 when it is sampled (§5d).
bool light_mix(const std::vector<Light>& lights, const Env* env, bool iso, V3 p, V3 n, Ctx& ctx, V3& dir, float& w) {
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

// ---------------------------------------------------------------- triangle attributes (§5e)

// The attribute table and, per object id, its record index + 1 (the objects' `aux`; 0: none).
struct Attrs {
	std::vector<rtbs_tri_attr> rec;
	std::vector<int32_t> aux;
};

// Rec widened with m: the shading normal on the geometric normal's side (the geometric normal without attributes).
struct MRec : Rec { V3 m; };

// The oracle's hit() sets a triangle's record inside its recursive walk and rotate_y turns the normal on the way back, so
// the interpolation has to happen at the leaf, in the triangle's own frame: hit_attr restates the walk, case for case the
// oracle's hit(), instead of adding a hook to oracle.cpp, whose behaviour therefore stays exactly what it was.
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

// ---------------------------------------------------------------- rough metal and rough glass (§5f)

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

// ---------------------------------------------------------------- the scene and its integrator

struct FeatureScene {
	Scene sc;                    // what orc_scene_load reads from the v1 body
	std::vector<Light> lights;   // the light list (v2 and later), in world space
	bool has_env = false; Env env;
	Attrs at;                    // the attribute table (v4 and later); empty before
	std::vector<float> alpha;    // one GGX width per material (v5); zeros before
};

// sample_world of the oracle with every feature: a miss returns thr * texel when there is a map; the two GGX kinds scatter
// on their own; Lambertian and isotropic scatters go through the mixture when there are lights or a sampled map (§5b step
// 7: throughput (thr * w) * albedo); every other material goes through the oracle's scatter, the dielectric about m.
V3 sample_world_features(const FeatureScene& s, Ray ray, uint32_t max_depth, Ctx& ctx) {
	const Scene& sc = s.sc;
	const Env* env = s.has_env ? &s.env : nullptr;
	V3 thr(1, 1, 1);
	const bool mix = !s.lights.empty() || (env && env->sample);
	for (uint32_t i = 0; i < max_depth; ++i) {
		MRec rec;
		ctx.begin(i);
		ctx.rays++;
		if (!hit_attr(sc.root.get(), ray, rec, ctx, s.at)) return thr * (env ? env_radiance(*env, ray.d) : background(sc, ray.d));
		V3 p = ray.at(rec.distance);
		V3 dir, att;
		const rtbs_material& m = sc.materials[rec.material];
		if (m.kind == RTB_MAT_ROUGH_METAL || m.kind == RTB_MAT_ROUGH_DIELECTRIC) {
			const V3 albedo(m.albedo[0], m.albedo[1], m.albedo[2]);
			int res;
			if (m.kind == RTB_MAT_ROUGH_METAL) {
				res = rough_scatter(false, rec.normal, ray.d, ctx.r, s.alpha[rec.material], 0.0f, albedo, dir, att);
			} else {
				const bool back = dot(ray.d, rec.n_geom) > 0.0f;
				res = rough_scatter(true, back ? -rec.m : rec.m, ray.d, ctx.r, s.alpha[rec.material], back ? m.param : 1.0f / m.param, albedo, dir, att);
			}
			if (res == 0) return V3();
			thr = thr * att;
		} else if (mix && (m.kind == RTB_MAT_LAMBERTIAN || m.kind == RTB_MAT_ISOTROPIC)) {
			att = m.tex >= 0 ? texture_value(sc, m.tex, rec.u, rec.v, p) : V3(m.albedo[0], m.albedo[1], m.albedo[2]);
			float w;
			if (!light_mix(s.lights, env, m.kind == RTB_MAT_ISOTROPIC, p, rec.normal, ctx, dir, w)) return V3();
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

struct ofeat_scene : FeatureScene {};   // the C API's handle

extern "C" {

// Loads an RTBS v1 - v5 blob, one section after the other: the v1 body (through orc_scene_load, as v1), the light list
// (v2 and later), the map record and its texels (v3 and later), the attribute table (v4 and later) and the GGX widths (v5).
// The refusals and their order are those of the loaders this one replaced, which each read one more section than the one
// below and handed it the rest; where the versions differ, the comments say how.
ofeat_scene* ofeat_scene_load(const void* blob, size_t size) {
	if (!blob || size < sizeof(rtbs_header)) { g_err = "blob too small"; return nullptr; }
	const uint8_t* p = static_cast<const uint8_t*>(blob);
	rtbs_header h; memcpy(&h, p, sizeof h);
	const uint32_t ver = h.version;
	if (h.magic != RTBS_MAGIC || ver < RTBS_VERSION || ver > RTBS_VERSION_ROUGH) { g_err = "bad magic/version"; return nullptr; }
	const size_t mats_off = sizeof h + (size_t)h.n_textures * sizeof(rtbs_texture);
	const size_t objs_off = mats_off + (size_t)h.n_materials * sizeof(rtbs_material);
	const size_t v1 = objs_off + (size_t)h.n_objects * sizeof(rtbs_object) + (size_t)h.n_children * 4 + h.n_blob_bytes;
	size_t off = v1;
	if (ver < RTBS_VERSION_ROUGH && size < off) { g_err = "blob truncated"; return nullptr; }   // v5: a truncated light list
	auto s = std::make_unique<ofeat_scene>();
	int32_t nl = 0;
	size_t lights_off = 0;
	if (ver >= RTBS_VERSION_LIGHTS) {   // int32 n_lights, int32 objects[n_lights]
		if (size < off + 4) { g_err = "blob truncated (light list)"; return nullptr; }
		memcpy(&nl, p + off, 4);
		// v2 lists at least one light and is checked for the ids here; from v3 on the list may be empty, and the next
		// section's check covers the ids
		const bool v2 = ver == RTBS_VERSION_LIGHTS;
		if (nl < (v2 ? 1 : 0) || nl > RTB_MAX_SAMPLED_LIGHTS || (v2 && size < off + 4 + 4 * (size_t)nl)) { g_err = "bad light list"; return nullptr; }
		lights_off = off + 4;
		off += 4 + 4 * (size_t)nl;
	}
	rtbs_env eh{};
	bool map_ok = true;
	size_t env_off = 0;
	if (ver >= RTBS_VERSION_ENV) {   // rtbs_env, then its texels
		if (size < off + sizeof eh) { g_err = "blob truncated (environment map)"; return nullptr; }
		memcpy(&eh, p + off, sizeof eh);
		// v3 always carries a map; v4 and v5 write a 0 x 0 record without one (and v4 reads any record of no positive size
		// as none)
		s->has_env = ver == RTBS_VERSION_ENV || eh.width > 0 || eh.height > 0;
		const bool in_range = eh.width >= 0 && eh.height >= 0 && eh.width <= RTB_ENV_MAX_SIZE && eh.height <= RTB_ENV_MAX_SIZE;
		map_ok = in_range && eh.width > 0 && eh.height > 0;
		// v5 refuses an N x 0 map only after its width table
		const bool bad = ver == RTBS_VERSION_ROUGH ? !in_range : s->has_env && !map_ok;
		if (bad) { g_err = "bad environment map"; return nullptr; }
		env_off = off + sizeof eh;
		off = env_off + (s->has_env ? (size_t)eh.width * eh.height * 12 : 0);
		if (ver == RTBS_VERSION_ENV && size < off) { g_err = "bad environment map"; return nullptr; }
	}
	uint32_t na = 0;
	size_t attrs_off = 0;
	if (ver >= RTBS_VERSION_ATTR) {   // uint32 n, rtbs_tri_attr[n]
		if (size < off + 4) { g_err = "blob truncated (triangle attributes)"; return nullptr; }
		memcpy(&na, p + off, 4);
		attrs_off = off + 4;
		off = attrs_off + (size_t)na * sizeof(rtbs_tri_attr);
		// v5: the width table's check covers the records
		if (ver == RTBS_VERSION_ATTR && size < off) { g_err = "blob truncated (triangle attributes)"; return nullptr; }
	}
	s->alpha.assign(h.n_materials, 0.0f);
	if (ver >= RTBS_VERSION_ROUGH) {   // uint32 n_materials, float alpha[n_materials], and nothing after it
		uint32_t nm = 0;
		if (size < off + 4) { g_err = "blob truncated (GGX widths)"; return nullptr; }
		memcpy(&nm, p + off, 4);
		if (nm != h.n_materials || size != off + 4 + 4 * (size_t)nm) { g_err = "bad GGX width table"; return nullptr; }
		if (nm) memcpy(s->alpha.data(), p + off + 4, 4 * (size_t)nm);
		for (uint32_t k = 0; k < nm; ++k) {
			rtbs_material m; memcpy(&m, p + mats_off + (size_t)k * sizeof m, sizeof m);
			const bool rough = m.kind == RTB_MAT_ROUGH_METAL || m.kind == RTB_MAT_ROUGH_DIELECTRIC;
			if (rough && !(s->alpha[k] >= 0.001f && s->alpha[k] <= 1.0f)) { g_err = "bad GGX width"; return nullptr; }
		}
		if (s->has_env && !map_ok) { g_err = "bad environment map"; return nullptr; }
	}
	s->at.aux.assign(h.n_objects, 0);
	s->at.rec.resize(na);
	if (na) memcpy(s->at.rec.data(), p + attrs_off, (size_t)na * sizeof(rtbs_tri_attr));
	if (ver >= RTBS_VERSION_ATTR) {
		for (uint32_t k = 0; k < h.n_objects; ++k) {
			rtbs_object o; memcpy(&o, p + objs_off + (size_t)k * sizeof o, sizeof o);
			if (o.kind != RTB_OBJ_TRIANGLE || o.aux == 0) continue;
			if (o.aux < 0 || (uint32_t)o.aux > na) { g_err = "bad triangle attribute index"; return nullptr; }
			s->at.aux[k] = o.aux;
		}
	}
	// the v1 body as the plain oracle reads it
	std::vector<uint8_t> b(p, p + v1);
	const uint32_t one = RTBS_VERSION; memcpy(b.data() + 4, &one, 4);
	std::unique_ptr<orc_scene> plain(orc_scene_load(b.data(), b.size()));
	if (!plain) return nullptr;
	s->sc = std::move(plain->sc);
	const rtbs_object* objs = reinterpret_cast<const rtbs_object*>(b.data() + objs_off);
	const int32_t* children = reinterpret_cast<const int32_t*>(b.data() + objs_off + (size_t)h.n_objects * sizeof(rtbs_object));
	for (int32_t k = 0; k < nl; ++k) {
		int32_t id; memcpy(&id, p + lights_off + 4 * (size_t)k, 4);
		Light L;
		if (!build_light(objs, children, h.n_objects, h.n_children, id, L)) return nullptr;
		s->lights.push_back(std::move(L));
	}
	if (s->has_env) {
		s->env.W = eh.width; s->env.H = eh.height; s->env.sample = (eh.flags & RTB_ENV_SAMPLE) != 0;
		s->env.rgb.resize((size_t)eh.width * eh.height * 3);
		memcpy(s->env.rgb.data(), p + env_off, s->env.rgb.size() * 4);
		env_build(s->env);
	}
	return s.release();
}
void ofeat_scene_free(ofeat_scene* s) { delete s; }
int ofeat_num_lights(const ofeat_scene* s) { return s ? (int)s->lights.size() : -1; }

// The map's pieces, for the sampler tests (the scene must carry a map).
int ofeat_env_dims(const ofeat_scene* s, int* wh) { if (!s || !s->has_env) return -1; wh[0] = s->env.W; wh[1] = s->env.H; return 0; }
void ofeat_env_tables(const ofeat_scene* s, float* pdf_num, float* cm, float* cc) {
	memcpy(pdf_num, s->env.pdf.data(), s->env.pdf.size() * 4);
	memcpy(cm, s->env.cm.data(), s->env.cm.size() * 4);
	memcpy(cc, s->env.cc.data(), s->env.cc.size() * 4);
}
// n directions drawn with the uniforms z[2k], z[2k + 1]; dir[3k..], their texel index and pdf
void ofeat_env_sample(const ofeat_scene* s, const float* z, int n, float* dir, int64_t* texel, float* pdf) {
	for (int k = 0; k < n; ++k) {
		V3 d = env_direction(s->env, z[2 * k], z[2 * k + 1]);
		dir[3 * k] = d.x; dir[3 * k + 1] = d.y; dir[3 * k + 2] = d.z;
		float st; texel[k] = (int64_t)env_index(s->env, d, st);
		pdf[k] = env_pdf(s->env, d);
	}
}
// texel index and pdf of n given directions
void ofeat_env_lookup(const ofeat_scene* s, const float* dir, int n, int64_t* texel, float* pdf) {
	for (int k = 0; k < n; ++k) {
		V3 d(dir[3 * k], dir[3 * k + 1], dir[3 * k + 2]);
		float st; texel[k] = (int64_t)env_index(s->env, d, st);
		pdf[k] = env_pdf(s->env, d);
	}
}

// The attribute table as read (n records of 16 floats: normals, UVs, flags as a float-sized int), and the count.
int ofeat_attr_count(const ofeat_scene* s) { return s ? (int)s->at.rec.size() : -1; }
void ofeat_attrs(const ofeat_scene* s, rtbs_tri_attr* out) { if (!s->at.rec.empty()) memcpy(out, s->at.rec.data(), s->at.rec.size() * sizeof(rtbs_tri_attr)); }

// The widths as read (one per material), and their count.
int ofeat_alpha_count(const ofeat_scene* s) { return s ? (int)s->alpha.size() : -1; }
void ofeat_alphas(const ofeat_scene* s, float* out) { if (!s->alpha.empty()) memcpy(out, s->alpha.data(), s->alpha.size() * 4); }

// orc_trace_rays with the attribute walk: n is the shading normal, (u, v) the interpolated coordinates.
int ofeat_trace_rays(const ofeat_scene* s, const rtb_ray* rays, size_t n, rtb_hit* out) {
	if (!s || (n && (!rays || !out))) { g_err = "ofeat_trace_rays: bad argument"; return -1; }
	for (size_t i = 0; i < n; ++i) {
		Ray r(V3(rays[i].o[0], rays[i].o[1], rays[i].o[2]), V3(rays[i].d[0], rays[i].d[1], rays[i].d[2]), rays[i].time);
		Ctx ctx; ctx.skip_media = true; ctx.want_uv = true;
		MRec rec;
		rtb_hit h; memset(&h, 0, sizeof h);
		if (!hit_attr(s->sc.root.get(), r, rec, ctx, s->at)) { h.t = MISS_DIST; h.prim = -1; h.object = -1; h.material = -1; out[i] = h; continue; }
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

// orc_render with every feature; Philox streams only (XORWOW is the reference's mode, and the reference has none of them).
int ofeat_render(const ofeat_scene* s, const rtb_camera* cam, uint32_t W, uint32_t H, uint32_t s0, uint32_t s1, uint32_t max_depth,
                 uint32_t seed, int mode, int threads, float* sum, float* sum2, uint64_t* rays_out) {
	if (!s || !cam || !sum || W == 0 || H == 0) { g_err = "ofeat_render: bad argument"; return -1; }
	if (mode != ORC_RNG_PHILOX) { g_err = "ofeat_render: XORWOW mode reproduces the reference, which has none of these features: render in Philox mode"; return -1; }
	render_rows(*cam, W, H, s0, s1, seed, mode, threads, s->sc.any_uv_texture, sum, sum2, rays_out,
	            [&](const Ray& ray, Ctx& ctx) { return sample_world_features(*s, ray, max_depth, ctx); });
	return 0;
}

}  // extern "C"
