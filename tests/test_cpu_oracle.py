"""CPU tests: the oracle pinned against the reference's own outputs (tests/golden/, produced by the
reference's sources compiled unmodified — see tests/golden/make_golden.py) and against known answers."""
import math
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from helpers import camera_rays, parse_blob, psnr, random_rays, tonemap


# ---------------------------------------------------------------- arithmetic spec kernels

def test_philox_known_answers(orc):
    """Random123 kat_vectors for philox4x32-10."""
    assert [hex(x) for x in orc.philox([0, 0, 0, 0], [0, 0])] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    assert [hex(x) for x in orc.philox([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2)] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    assert [hex(x) for x in orc.philox([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0])] == \
        ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_sincos_and_log_kernels(orc):
    us = np.concatenate([np.linspace(1e-7, 1.0, 4001), [2.0 ** -33, 0.125, 0.25, 0.5, 0.75, 1.0]])
    err = 0.0
    for u in us:
        s, c = orc.sincos2pi(float(np.float32(u)))
        a = 2 * math.pi * float(np.float32(u))
        err = max(err, abs(s - math.sin(a)), abs(c - math.cos(a)))
    assert err < 5e-7
    assert orc.sincos2pi(1.0) == (0.0, 1.0) and orc.sincos2pi(0.25) == (1.0, 0.0)
    for x in np.geomspace(2.0 ** -33, 1.0, 2000):
        x = float(np.float32(x))
        assert abs(orc.logpos(x) - math.log(x)) <= 1e-6 * max(1.0, abs(math.log(x)))


def test_xorwow_matches_device_curand(orc):
    """curand_init(seed,0,0) + curand_uniform streams dumped on a B200 (oracle/_ref/ref_render rng)."""
    d = np.fromfile(GOLDEN / "ref_rng.bin", dtype=np.float32)
    dev = d[4608:].reshape(4, 64)
    for i, seed in enumerate((1984, 1985, 1984 + 45000, 1984 + 89999)):
        assert np.array_equal(orc.xorwow_uniforms(seed, 64), dev[i])
    assert d[:4608].min() > 0.0 and d[:4608].max() <= 1.0      # (0,1]


# ---------------------------------------------------------------- scene + BVH against the reference

def test_scene_equals_reference_scene(rtb):
    """The host mirror's SceneBook2BVH == what the reference's own Scenes.cu built (cuRAND stream, argument
    evaluation order, sphere and material parameters), dumped from device memory on the GPU box."""
    raw = np.fromfile(GOLDEN / "ref_scene_book2_bouncing.bin", dtype=np.uint8)
    n = int(np.frombuffer(raw[:4], dtype=np.int32)[0])
    rec = np.frombuffer(raw[4:], dtype=np.float32).reshape(n, 16)
    s = rtb.Scene.named("book2_bouncing")
    _, mats, objs, _ = parse_blob(s.serialize())
    assert n == 488 and s.num_objects() == 489
    kinds = {0: 0, 1: 0, 2: 0}
    for i in range(n):
        o, m = objs[i], mats[objs[i]["mat"]]
        if rec[i, 0] == 1.0:
            assert o["kind"] == 1 and np.array_equal(rec[i, 1:4], o["f"][:3]) and np.array_equal(rec[i, 4:7], o["f"][4:7]) and rec[i, 7] == o["f"][3]
        else:
            assert o["kind"] == 0 and np.array_equal(rec[i, 1:5], o["f"][:4])
        assert np.array_equal(rec[i, 8:11], m["albedo"])
        if m["kind"] in (1, 2):
            assert rec[i, 11] == m["param"]
        kinds[int(m["kind"])] += 1
    assert kinds == {0: 396, 1: 63, 2: 29}      # 394 moving + ground + left; 62 + right; 28 + centre (SURVEY App. C)


def _read_ref_bvh(path, rtb):
    d = open(path, "rb").read()
    nn, root = struct.unpack("ii", d[:8])
    nodes = np.frombuffer(d[8:8 + 32 * nn], dtype=rtb.BVH_NODE_DTYPE)
    order = np.frombuffer(d[8 + 32 * nn:], dtype=np.int32)
    return nodes, order, root


def test_bvh_bit_exact_vs_reference_golden(rtb, orc):
    """Node array + primitive order of the reference's BuildBVH_TopDown (BVH.cu:166-210) on config 1/2's boxes."""
    s = rtb.Scene.named("book2_bouncing")
    boxes = np.array([s.bounds(i) for i in range(488)], dtype=np.float32)
    gn, go, gr = _read_ref_bvh(GOLDEN / "ref_bvh_book2_bouncing.bin", rtb)
    assert len(gn) == 975 and gr == 974 and gn[gr]["left_child_idx"] == 486 and gn[gr]["right_child_hittable_idx"] == 973
    for build in (lambda: rtb.bvh_build(boxes, rtb.BVH_TOPDOWN_MEDIAN), lambda: orc.bvh_build(boxes, rtb.BVH_TOPDOWN_MEDIAN, rtb.BVH_NODE_DTYPE)):
        n, o, r = build()
        assert np.array_equal(n.view(np.uint8), gn.view(np.uint8)) and np.array_equal(o, go) and r == gr
    # asked to walk the tree as built, the renderer traverses that same tree
    s.set_world_bvh(rtb.WORLD_BVH_AS_BUILT)
    s.flatten_stats()
    wn, wr = s.world_bvh()
    assert np.array_equal(wn.view(np.uint8), gn.view(np.uint8)) and wr == gr


BVH_CASES = [(0, 3000), (0, 1), (0, 2), (0, 37), (2, 120)]


def _duplicate_key_boxes(builder, n):
    """Seeded random boxes with duplicate sort keys (the reference uses an unstable std::sort)."""
    rng = np.random.default_rng(n + builder)
    c = rng.uniform(-50, 50, (n, 3)).astype(np.float32); r = rng.uniform(0.1, 3, (n, 1)).astype(np.float32)
    c[::3, 0] = np.round(c[::3, 0]); c[::5] = c[0]
    return np.concatenate([c - r, c + r], 1)


@pytest.mark.parametrize("builder,n", BVH_CASES)
def test_bvh_builders_product_equals_oracle(rtb, orc, builder, n):
    """The product's builders and the oracle's restatement give the same node array, primitive order and root on the
    boxes of test_bvh_bit_exact_vs_reference_live, which needs the reference-derived checker."""
    boxes = _duplicate_key_boxes(builder, n)
    gn, go, gr = orc.bvh_build(boxes, builder, rtb.BVH_NODE_DTYPE)
    got = rtb.bvh_build(boxes, builder)
    assert len(gn) == 2 * n - 1 and sorted(go.tolist()) == list(range(n))
    assert np.array_equal(got[0].view(np.uint8), gn.view(np.uint8)) and np.array_equal(got[1], go) and got[2] == gr


@pytest.mark.skipif(not (ROOT / "oracle" / "_ref" / "ref_bvh").exists(), reason="reference-derived checker not built (make -C oracle ref with a checkout of the reference)")
@pytest.mark.parametrize("builder,n", BVH_CASES)
def test_bvh_bit_exact_vs_reference_live(rtb, orc, builder, n, tmp_path):
    """Random boxes with duplicate sort keys (the reference uses an unstable std::sort) through the reference's own BVH.cu."""
    boxes = _duplicate_key_boxes(builder, n)
    fin, fout = tmp_path / "in.bin", tmp_path / "out.bin"
    fin.write_bytes(struct.pack("i", n) + boxes.tobytes())
    subprocess.run([str(ROOT / "oracle" / "_ref" / "ref_bvh"), str(fin), str(fout), str(builder)], check=True)
    gn, go, gr = _read_ref_bvh(fout, rtb)
    for got in (rtb.bvh_build(boxes, builder), orc.bvh_build(boxes, builder, rtb.BVH_NODE_DTYPE)):
        assert np.array_equal(got[0].view(np.uint8), gn.view(np.uint8)) and np.array_equal(got[1], go) and got[2] == gr


# ---------------------------------------------------------------- integrator against the reference megakernel

def test_oracle_matches_reference_megakernel_per_pixel(rtb, orc):
    """XORWOW mode = the reference's own streams: same image as render_kernel compiled for sm_100a, up to
    paths whose branch flips on nvcc's FMA contraction (they also shift that pixel's stream)."""
    ref = np.fromfile(GOLDEN / "ref_megakernel_200x112_4spp_d50.bin", dtype=np.float32).reshape(112, 200, 4)
    s = rtb.Scene.named("book2_bouncing")
    cam = rtb.make_camera("motion", (13, 2, 3), (0, 0, 0), (0, 1, 0), 30.0, 200 / 112.0, t0=0.1, t1=1.0)
    osum, _, _ = orc.OracleScene(s.serialize()).render(cam, 200, 112, 0, 4, 50, seed=1984, mode=orc.RNG_XORWOW)
    img = tonemap(osum)
    assert np.array_equal(ref[..., 3], np.ones((112, 200), dtype=np.float32))
    diff = np.abs(img - ref[..., :3]).max(axis=2)
    assert (diff <= 1e-4).mean() > 0.95, f"only {(diff <= 1e-4).mean():.4f} of pixels agree to 1e-4"
    assert psnr(img, ref[..., :3]) > 35.0


def test_oracle_matches_reference_megakernel_config2(rtb, orc):
    """Config 2 at full size (400x225, 100 spp, depth 50): PSNR and per-channel mean vs the reference's image."""
    ref = np.load(GOLDEN / "ref_megakernel_400x225_100spp_d50_f16.npy").astype(np.float32)
    s = rtb.Scene.named("book2_bouncing")
    cam = s.info.camera
    o = orc.OracleScene(s.serialize())
    xs, _, _ = o.render(cam, 400, 225, 0, 100, 50, seed=1984, mode=orc.RNG_XORWOW)
    assert psnr(tonemap(xs), ref) > 45.0
    # the new path's own streams (Philox): a different sample set of the same estimator
    ps, ps2, _ = o.render(cam, 400, 225, 0, 100, 50, seed=1984, mode=orc.RNG_PHILOX, want_sum2=True)
    p = psnr(tonemap(ps), ref)
    assert p > 30.0, f"PSNR {p:.1f} dB"
    mean_p = (ps[..., :3] / 100.0); mean_x = (xs[..., :3] / 100.0)
    var = np.maximum(ps2[..., :3] / 100.0 - mean_p ** 2, 0.0) / 100.0          # variance of each pixel mean
    for c in range(3):
        bias = float((mean_p[..., c] - mean_x[..., c]).mean())
        sigma = float(np.sqrt(2.0 * var[..., c].sum()) / var[..., c].size)
        assert abs(bias) <= 3.0 * sigma + 1e-4, f"channel {c}: mean error {bias:.2e} vs 3 sigma {3 * sigma:.2e}"


# ---------------------------------------------------------------- oracle self-consistency / edge cases

def test_traversal_order_does_not_change_hits(rtb, orc):
    """Closest hit through the reference's BVH walk (BVH.cu:54-106) == linear HittableList scan == brute force index."""
    src = rtb.Scene.named("book2_bouncing")
    _, mats, objs, _ = parse_blob(src.serialize())
    def build(kind):
        s = rtb.Scene(); ids = []
        for o in objs[:488]:
            m = s.lambertian(albedo=(0.5, 0.5, 0.5))
            ids.append(s.moving_sphere(o["f"][:3], o["f"][4:7], float(o["f"][3]), m) if o["kind"] == 1 else s.sphere(o["f"][:3], float(o["f"][3]), m))
        s.set_root(s.bvh(ids) if kind == "bvh" else s.list(ids))
        return s
    rays = np.concatenate([camera_rays(rtb, src.info.camera, 160, 90, "renderer"), random_rays(rtb, 20000, -12, 12, seed=5)])
    a = orc.OracleScene(build("bvh").serialize()).trace_rays(rays, rtb.HIT_DTYPE)
    b = orc.OracleScene(build("list").serialize()).trace_rays(rays, rtb.HIT_DTYPE)
    assert np.array_equal(a["object"], b["object"]) and np.array_equal(a["t"].view(np.uint32), b["t"].view(np.uint32))
    assert (a["object"] >= 0).sum() > 5000


def test_sphere_index_recipe_cpu(rtb, orc):
    """google_testing/test.cpp:87-106 recipe on the CPU side: brute force over raw spheres == oracle BVH trace."""
    src = rtb.Scene.named("book2_bouncing")
    _, _, objs, _ = parse_blob(src.serialize())
    sp = np.array([[*o["f"][:3], o["f"][3]] for o in objs[:488]], dtype=np.float32)
    W, H = 320, 180
    cam = rtb.make_camera("pinhole", (0, 1, -4), (0, 1, 0), (0, 1, 0), 90.0, 1280 / 720)
    truth = orc.sphere_index_image(sp, cam, W, H)
    assert (truth >= 0).mean() > 0.5 and truth.max() < 488
    s = rtb.Scene(); m = s.lambertian(albedo=(0.5, 0.5, 0.5))
    s.set_root(s.bvh([s.sphere(c[:3], float(c[3]), m) for c in sp]))
    hits = orc.OracleScene(s.serialize()).trace_rays(camera_rays(rtb, cam, W, H, "test"), rtb.HIT_DTYPE)
    assert (hits["object"].reshape(H, W) == truth).mean() > 0.9999


def test_sphere_index_recipe_reference_functions(rtb, orc, tmp_path):
    """The reference's own unit test (google_testing/test.cpp:87-106), with the reference's own functions as the truth:
    _sphere_closest_intersection (SphereHittable.cuh:15-33) and PinholeCamera (cu_Cameras.cuh:12-31) compiled from the
    reference's headers (oracle/_ref/ref_sphere_index host).  The committed golden is that binary's output (run live as
    well when the binary is present, and then the rays numpy builds must be the reference's, bit for bit); the camera
    the product's rtb_camera_pinhole builds is the reference's, bit for bit; and the
    oracle's BVH trace names the reference's sphere on all 921,600 pixels but the handful where a sphere is grazed
    within float32 rounding (the reference's host code does not contract multiply-adds, the arithmetic spec does)."""
    from helpers import grazing_only, reference_sphere_index, test_spheres
    W, H = 1280, 720
    gold = np.load(GOLDEN / "ref_sphere_index_host_1280x720.npz")
    idx, cam12 = gold["index"].reshape(-1).astype(np.int32), gold["camera"]
    cam = rtb.make_camera("pinhole", (0, 1, -4), (0, 1, 0), (0, 1, 0), 90.0, W / H)
    assert np.array_equal(np.array([*cam.o, *cam.u, *cam.v, *cam.w], dtype=np.float32), cam12)
    rays = camera_rays(rtb, cam, W, H, "test")
    if (ROOT / "oracle" / "_ref" / "ref_sphere_index").exists():
        live, live_cam12, ref_rays = reference_sphere_index(rtb, "host", tmp_path, W, H)
        assert np.array_equal(live, idx) and np.array_equal(live_cam12, cam12)
        assert np.array_equal(rays["d"].view(np.uint32), ref_rays["d"].view(np.uint32)) and np.array_equal(rays["o"], ref_rays["o"])
    sp = test_spheres(rtb)
    s = rtb.Scene(); m = s.lambertian(albedo=(0.5, 0.5, 0.5))
    s.set_root(s.bvh([s.sphere(c[:3], float(c[3]), m) for c in sp]))
    got = orc.OracleScene(s.serialize()).trace_rays(rays, rtb.HIT_DTYPE)["object"]
    bad = np.nonzero(got != idx)[0]
    assert len(bad) <= 16, f"{len(bad)} pixels differ"
    assert grazing_only(rays[bad], sp, got[bad], idx[bad]).all(), "a differing pixel is not a grazing tie"
    brute = orc.sphere_index_image(sp, cam, W, H).reshape(-1)      # the restated recipe follows the same arithmetic spec
    assert np.array_equal(brute, got)


def test_oracle_hit_records_match_reference_device(rtb, orc):
    """Per-ray hit records against the reference's own DEVICE code: world->ClosestIntersection (BVH.cu:54-106,
    SphereHittable.cu:56-66,91-102) and getNormal (:43-50,75-83) run on a B200 over 102,400 rays of config 1-2's scene
    (camera rays with shutter times, random segments, grazing rays; moving spheres at many times) by
    `oracle/_ref/ref_render trace` - tests/golden/ref_trace_book2_bouncing.npz.  The sphere hit is the same one; t, point and
    normal lie inside the binary32 rounding bound of the reference's formula (see helpers.check_against_reference_trace)."""
    from helpers import check_against_reference_trace, load_reference_trace, reference_trace_rays
    rays = reference_trace_rays(rtb)
    s = rtb.Scene.named("book2_bouncing")
    got = orc.OracleScene(s.serialize()).trace_rays(rays, rtb.HIT_DTYPE)
    print(check_against_reference_trace(rtb, rays, got, load_reference_trace(rays, GOLDEN / "ref_trace_book2_bouncing.npz")))


def test_medium_transmission_known_answer(rtb, orc):
    """Beer-Lambert: an absorbing slab (isotropic albedo 0) of density s and thickness L in front of a white
    background transmits exp(-s L)."""
    s = rtb.Scene()
    black = s.isotropic(s.solid((0, 0, 0)))
    slab = s.box((-50, -50, 0), (50, 50, 4), s.lambertian(albedo=(1, 1, 1)))
    s.set_root(s.list([s.constant_medium(slab, 0.25, black)]))
    s.set_background(rtb.BG_CONSTANT, (1, 1, 1))
    cam = rtb.make_camera("pinhole", (0, 0, -10), (0, 0, 0), (0, 1, 0), 2.0, 1.0)
    acc, _, _ = orc.OracleScene(s.serialize()).render(cam, 32, 32, 0, 256, 8, seed=7)
    mean = float((acc[..., 0] / acc[..., 3]).mean())
    assert abs(mean - math.exp(-1.0)) < 0.004, mean


def test_edge_cases(rtb, orc):
    s = rtb.Scene.named("book2_checker")
    o = orc.OracleScene(s.serialize())
    cam = s.info.camera
    acc, _, rays = o.render(cam, 8, 4, 5, 5, 10)                 # empty sample range
    assert not acc.any() and rays == 0
    acc, _, rays = o.render(cam, 1, 1, 0, 3, 1)                  # 1x1 image, a single segment per path
    assert acc[0, 0, 3] == 3 and rays == 3
    rays_in = np.zeros(4, dtype=rtb.RAY_DTYPE)                   # axis-aligned rays (zero direction components)
    rays_in["o"] = [(0, 30, 0), (0, -30, 0), (50, 0, 0), (0, -10, 0)]
    rays_in["d"] = [(0, -1, 0), (0, 1, 0), (0, 1, 0), (0, 1, 0)]
    h = o.trace_rays(rays_in, rtb.HIT_DTYPE)
    assert h["object"][0] >= 0 and h["object"][1] >= 0 and h["object"][2] == -1
    assert h["t"][0] == 10.0 and h["t"][3] == 10.0               # from the centre of the lower sphere: near root < 0, far root taken
    with pytest.raises(RuntimeError):
        orc.OracleScene(b"not a scene")


def test_oracle_has_not_drifted(rtb, orc):
    """The oracle is the checker of every GPU test, so it gets a tripwire of its own: its Philox renders of every
    registered scene (32x18, 2 spp, depth 8) against the committed copies (tests/golden/make_golden.py oracle)."""
    from conftest import ROOT
    gold = np.load(ROOT / "tests" / "golden" / "oracle_images_32x18.npz")
    names = rtb.scene_names()
    assert sorted(k for k in gold.files if not k.endswith("__rays")) == sorted(names)
    for name in names:
        s = rtb.Scene.named(name)
        acc, _, rays = orc.OracleScene(s.serialize()).render(s.info.camera, 32, 18, 0, 2, 8, seed=1984)
        assert rays == int(gold[name + "__rays"][0]), name
        np.testing.assert_allclose(acc, gold[name], rtol=1e-6, atol=1e-6, err_msg=name)


# ---------------------------------------------------------------- analytic pins for features the reference does not contain

def _oracle_trace(rtb, orc):
    return lambda scene, rays: orc.OracleScene(scene.serialize()).trace_rays(rays, rtb.HIT_DTYPE)


def _oracle_render(orc):
    return lambda scene, cam, w, h, spp, depth: orc.OracleScene(scene.serialize()).render(cam, w, h, 0, spp, depth, seed=5)[0]


def test_analytic_quad_alpha_beta(rtb, orc):
    import analytic
    analytic.check_quad_alpha_beta(rtb, _oracle_trace(rtb, orc))


def test_analytic_rotate_y_quarter_turn(rtb, orc):
    import analytic
    analytic.check_rotate_y_quarter_turn(rtb, _oracle_trace(rtb, orc))


def test_analytic_sphere_uv(rtb, orc):
    import analytic
    analytic.check_sphere_uv(rtb, _oracle_trace(rtb, orc))


def test_analytic_checker_truncation(rtb, orc):
    import analytic
    analytic.check_checker_at_negative_coordinates(rtb, _oracle_trace(rtb, orc), _oracle_render(orc))


def test_analytic_image_texture(rtb, orc):
    import analytic
    analytic.check_image_texture_lookup(rtb, _oracle_render(orc))


def test_analytic_box_faces(rtb, orc):
    import analytic
    analytic.check_box_faces(rtb, _oracle_trace(rtb, orc))


def test_analytic_triangle(rtb, orc):
    import analytic
    analytic.check_triangle_barycentric(rtb, _oracle_trace(rtb, orc))


def test_analytic_emitter_and_mirror(rtb, orc):
    import analytic
    analytic.check_emitter_and_mirror(rtb, _oracle_render(orc))


def test_analytic_white_furnace(rtb, orc):
    import analytic
    analytic.check_white_furnace(rtb, _oracle_render(orc))


def test_analytic_beer_lambert(rtb, orc):
    import analytic
    analytic.check_beer_lambert(rtb, _oracle_render(orc))


def test_analytic_perlin_lattice(rtb, orc):
    import analytic
    analytic.check_perlin_lattice(rtb, _oracle_render(orc))


def test_committed_headline_scene_is_current(rtb, orc):
    """tests/golden/book2_final.rtbs.xz + .json (what `bench.py --impl reference` renders without touching the product) is
    what the host mirror builds today, byte for byte, camera included."""
    import json
    import lzma
    s = rtb.Scene.named("book2_final")
    blob = lzma.decompress((GOLDEN / "book2_final.rtbs.xz").read_bytes())
    assert blob == s.serialize()
    meta = json.loads((GOLDEN / "book2_final.json").read_text())
    assert (meta["width"], meta["height"], meta["max_depth"]) == (s.info.width, s.info.height, s.info.max_depth)
    cam = orc.camera_from_dict(meta["camera"])
    assert bytes(cam) == bytes(s.info.camera)
    a, _, ra = orc.OracleScene(blob).render(cam, 24, 24, 0, 2, 12, seed=3)
    b, _, rb = orc.OracleScene(s.serialize()).render(s.info.camera, 24, 24, 0, 2, 12, seed=3)
    assert np.array_equal(a, b) and ra == rb
