"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs.  Geometry is specified to be bit-exact (explicit-FMA arithmetic spec); images agree
per pixel up to the rare path whose branch flips on a last-ulp difference of a libm function."""
import numpy as np
import pytest

from helpers import camera_rays, parse_blob, psnr, random_rays, tonemap

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def renderer(rtb):
    return rtb.Renderer(0)


def _oracle_scene(orc, scene):
    return orc.OracleScene(scene.serialize())


def _compare_hits(rtb, g, o, exact=True, rtol=1e-5, max_tie_frac=0.01):
    miss_g = g["object"] < 0; miss_o = o["object"] < 0
    assert np.array_equal(miss_g, miss_o), f"hit/miss differs on {(miss_g != miss_o).sum()} rays"
    hit = ~miss_g
    # Two primitives hit at exactly the same t (coplanar faces of adjacent boxes, a box standing on the
    # floor) are a tie: which one "t < rec.distance" keeps depends on traversal order.  Everything else
    # must name the same object.
    diff_obj = hit & (g["object"] != o["object"])
    assert np.array_equal(g["t"][diff_obj].view(np.uint32), o["t"][diff_obj].view(np.uint32)), "different object at a different t"
    assert diff_obj.sum() <= max_tie_frac * hit.sum(), f"{diff_obj.sum()} ties out of {hit.sum()} hits"
    same = hit & ~diff_obj
    assert np.array_equal(g["material"][same], o["material"][same])
    assert np.array_equal(g["front_face"][same], o["front_face"][same])
    if exact:
        assert np.array_equal(g["t"][hit].view(np.uint32), o["t"][hit].view(np.uint32)), "t not bit-exact"
        assert np.array_equal(g["p"][hit].view(np.uint32), o["p"][hit].view(np.uint32)), "p not bit-exact"
        assert np.array_equal(g["n"][same].view(np.uint32), o["n"][same].view(np.uint32)), "n not bit-exact"
    else:
        np.testing.assert_allclose(g["t"][hit], o["t"][hit], rtol=rtol)
        np.testing.assert_allclose(g["p"][hit], o["p"][hit], rtol=rtol, atol=rtol * 10)
        np.testing.assert_allclose(g["n"][same], o["n"][same], rtol=0, atol=2e-5)
    return int(hit.sum())


def test_sphere_index_recipe(rtb, orc, renderer, tmp_path):
    """google_testing/test.cpp (SphereTest.DeviceSphereIndexTest) extended to the new path: scene recipe of the test (488
    static spheres), its camera and pixel mapping (u = x/(W-1)*2-1), closest-sphere index per pixel.  The truth is what the
    REFERENCE's own _sphere_closest_intersection + PinholeCamera::sample_ray give (compiled from the reference's headers:
    oracle/_ref/ref_sphere_index, golden tests/golden/ref_sphere_index_host_1280x720.npz; run live - host and, as the
    reference's test does, device - when the binary travelled with the repo).  The GPU traces the very rays the reference
    built, through its BVH: equal on all 921,600 pixels, except where a sphere is grazed within float32 rounding (the
    reference's host code, its device code and the arithmetic spec contract multiply-adds differently; the reference's own
    host-vs-device EXPECT_EQ is subject to the same handful of pixels)."""
    from conftest import GOLDEN, ROOT
    from helpers import grazing_only, reference_sphere_index, test_spheres
    W, H = 1280, 720
    sp = test_spheres(rtb)
    s = rtb.Scene(); m = s.lambertian(albedo=(0.5, 0.5, 0.5))
    s.set_root(s.bvh([s.sphere(c[:3], float(c[3]), m) for c in sp]))
    renderer.set_scene(s)
    cam = rtb.make_camera("pinhole", (0, 1, -4), (0, 1, 0), (0, 1, 0), 90.0, W / H)
    gold = np.load(GOLDEN / "ref_sphere_index_host_1280x720.npz")
    assert np.array_equal(np.array([*cam.o, *cam.u, *cam.v, *cam.w], dtype=np.float32), gold["camera"])
    rays = camera_rays(rtb, cam, W, H, "test")
    truths = {"golden(host)": gold["index"].reshape(-1).astype(np.int32)}
    if (ROOT / "oracle" / "_ref" / "ref_sphere_index").exists():
        for mode in ("host", "device"):
            idx, cam12, ref_rays = reference_sphere_index(rtb, mode, tmp_path, W, H)
            assert np.array_equal(cam12, gold["camera"])
            if mode == "host":
                assert np.array_equal(ref_rays["d"].view(np.uint32), rays["d"].view(np.uint32)) and np.array_equal(ref_rays["o"], rays["o"])
                assert np.array_equal(idx, truths["golden(host)"])
            truths[mode] = idx
    hits = renderer.trace_rays(rays)
    got = hits["object"]
    assert np.array_equal(got, _oracle_scene(orc, s).trace_rays(rays, rtb.HIT_DTYPE)["object"])     # GPU == oracle, all pixels
    for name, truth in truths.items():
        bad = np.nonzero(got != truth)[0]
        print(f"sphere index vs reference {name}: {len(bad)} of {W * H} pixels differ")
        assert len(bad) <= 16
        assert grazing_only(rays[bad], sp, got[bad], truth[bad]).all(), f"{name}: a differing pixel is not a grazing tie"
    if "device" in truths:   # the reference's own test on this box, for the record
        own = np.nonzero(truths["host"] != truths["device"])[0]
        print(f"reference host vs reference device (its own EXPECT_EQ): {len(own)} pixels differ")
        assert grazing_only(rays[own], sp, truths["host"][own], truths["device"][own]).all()


def test_hit_records_match_reference_device(rtb, renderer):
    """Per-ray hit records against the reference's own DEVICE code - world->ClosestIntersection (BVH.cu:54-106 ->
    SphereHittable.cu:56-66,91-102) and getNormal, run on a B200 over 102,400 rays (oracle/_ref/ref_render trace;
    tests/golden/ref_trace_book2_bouncing.npz): rtb_trace_rays on the same rays must name the same sphere, with t, point
    and normal inside the binary32 rounding bound of the reference's formula (helpers.check_against_reference_trace says
    why north_star's flat 1e-5 cannot be the bar on the r = 1000 sphere, and checks it where it can)."""
    from conftest import GOLDEN
    from helpers import check_against_reference_trace, load_reference_trace, reference_trace_rays
    rays = reference_trace_rays(rtb)
    scene = rtb.Scene.named("book2_bouncing")
    renderer.set_scene(scene)
    got = renderer.trace_rays(rays)
    gold = load_reference_trace(rays, GOLDEN / "ref_trace_book2_bouncing.npz")
    print("reference device hit records:", check_against_reference_trace(rtb, rays, got, gold))


@pytest.mark.parametrize("name,lo,hi", [("book2_bouncing", -12, 12), ("book1_final", -12, 12), ("book2_quads", -6, 9)])
def test_hit_records_bit_exact(rtb, orc, renderer, name, lo, hi):
    scene = rtb.Scene.named(name)
    renderer.set_scene(scene)
    rays = np.concatenate([camera_rays(rtb, scene.info.camera, 320, 180, "renderer"), random_rays(rtb, 200_000, lo, hi, seed=7)])
    g = renderer.trace_rays(rays)
    o = _oracle_scene(orc, scene).trace_rays(rays, rtb.HIT_DTYPE)
    n = _compare_hits(rtb, g, o, exact=True)
    assert n > 10_000


@pytest.mark.parametrize("name,lo,hi", [("book2_cornell", 0, 555), ("book2_final", -200, 600), ("mesh_icospheres", -4, 4)])
def test_hit_records_instanced_bit_exact(rtb, orc, renderer, name, lo, hi):
    """translate(rotate_y(x)) instances: the kernels take the ray into the primitive's frame with the
    same operations as the book's translate::hit / rotate_y::hit, so hits stay bit-exact."""
    scene = rtb.Scene.named(name)
    renderer.set_scene(scene)
    rays = np.concatenate([camera_rays(rtb, scene.info.camera, 200, 200, "renderer"), random_rays(rtb, 100_000, lo, hi, seed=11)])
    g = renderer.trace_rays(rays)
    o = _oracle_scene(orc, scene).trace_rays(rays, rtb.HIT_DTYPE)
    assert _compare_hits(rtb, g, o, exact=True) > 10_000


def test_hit_records_nested_instances(rtb, orc, renderer):
    """Deeper chains (rotate(translate(rotate(...)))) are composed into one transform by the flattener
    while the oracle applies them one by one: same geometry, different rounding."""
    s = rtb.Scene()
    m = s.lambertian(albedo=(0.5, 0.5, 0.5))
    box = s.box((0, 0, 0), (30, 60, 30), m)
    sph = s.sphere((10, 70, 10), 12.0, m)
    tri = s.triangle((0, 0, 40), (30, 0, 0), (0, 30, 0), m)
    grp = s.list([box, sph, tri])
    inst = s.rotate_y(s.translate(s.rotate_y(grp, 25.0), (40, 5, -20)), -40.0)
    inst2 = s.translate(s.rotate_y(grp, 200.0), (-60, 0, 30))
    s.set_root(s.list([inst, inst2, s.quad((-200, -1, -200), (400, 0, 0), (0, 0, 400), m)]))
    renderer.set_scene(s)
    rays = random_rays(rtb, 200_000, -120, 120, seed=3)
    g = renderer.trace_rays(rays)
    o = _oracle_scene(orc, s).trace_rays(rays, rtb.HIT_DTYPE)
    same = g["object"] == o["object"]
    assert same.mean() > 0.9995, f"closest object agrees on {same.mean():.6f}"
    hit = same & (g["object"] >= 0)
    assert hit.sum() > 20_000
    rel = np.abs(g["t"][hit] - o["t"][hit]) / np.abs(o["t"][hit])
    print(f"nested instances: t rel err median {np.median(rel):.2e} q99 {np.quantile(rel, 0.99):.2e} q99.9 {np.quantile(rel, 0.999):.2e} max {rel.max():.2e}")
    assert np.quantile(rel, 0.99) < 1e-5
    assert np.abs(g["n"][hit] - o["n"][hit]).max() < 1e-3
    assert np.array_equal(g["front_face"][hit], o["front_face"][hit]) or (g["front_face"][hit] != o["front_face"][hit]).mean() < 1e-4


def test_world_bvh_choice_does_not_change_hits(rtb, renderer):
    """The renderer walks a SAH tree by default; walking the tree exactly as the reference's builder made it
    (RTB_WORLD_BVH_AS_BUILT) gives bit-identical hit records and images."""
    rays = None; results = []
    for mode in (rtb.WORLD_BVH_QUALITY, rtb.WORLD_BVH_AS_BUILT):
        scene = rtb.Scene.named("book2_bouncing"); scene.set_world_bvh(mode)
        renderer.set_scene(scene); renderer.set_camera(scene.info.camera)
        if rays is None:
            rays = np.concatenate([camera_rays(rtb, scene.info.camera, 320, 180, "renderer"), random_rays(rtb, 100_000, -12, 12, seed=2)])
        h = renderer.trace_rays(rays)
        renderer.render(160, 90, 0, 4, 50); img = renderer.download_accum()
        results.append((h, img))
    (h0, i0), (h1, i1) = results
    for f in ("t", "object", "p", "n", "front_face"):
        assert np.array_equal(h0[f], h1[f]), f
    assert np.array_equal(i0, i1)
    assert h1["nodes_visited"].mean() > 1.5 * h0["nodes_visited"].mean()    # and the SAH tree is the cheaper walk


IMAGE_CASES = [
    # name, W, H, spp, depth, max mismatching pixel fraction
    ("book2_bouncing", 200, 112, 4, 50, 0.01),
    ("book1_final", 160, 90, 4, 50, 0.01),
    ("book2_checker", 160, 90, 4, 50, 0.01),
    ("book2_earth", 160, 90, 4, 50, 0.01),
    ("book2_perlin", 160, 90, 4, 50, 0.01),
    ("book2_quads", 120, 120, 4, 50, 0.01),
    ("book2_simple_light", 160, 90, 8, 50, 0.01),
    ("book2_cornell", 100, 100, 8, 50, 0.01),
    ("book2_cornell_smoke", 100, 100, 8, 50, 0.02),
    ("book2_final", 100, 100, 8, 40, 0.02),
    ("mesh_icospheres", 160, 90, 4, 50, 0.01),     # 2 x 1,280 OBJ triangles, instanced, glass and metal
]


@pytest.mark.parametrize("name,W,H,spp,depth,tol_frac", IMAGE_CASES)
def test_image_matches_oracle(rtb, orc, renderer, name, W, H, spp, depth, tol_frac):
    """Same Philox streams on both sides => the same paths: compare radiance sums per pixel."""
    scene = rtb.Scene.named(name)
    cam = scene.info.camera
    renderer.set_scene(scene); renderer.set_camera(cam)
    renderer.reset_counters()
    renderer.render(W, H, 0, spp, depth, seed=1984)
    renderer.synchronize()
    gpu = renderer.download_accum()
    cnt = renderer.counters()
    ref, _, rays = _oracle_scene(orc, scene).render(cam, W, H, 0, spp, depth, seed=1984)
    assert np.array_equal(gpu[..., 3], ref[..., 3])
    assert np.isfinite(gpu).all()
    diff = np.abs(gpu[..., :3] - ref[..., :3]).max(axis=2)
    scale = np.maximum(np.abs(ref[..., :3]).max(axis=2), 1.0)
    bad = float((diff > 1e-4 * scale).mean())
    p = psnr(tonemap(gpu), tonemap(ref))
    print(f"{name}: mismatching pixels {bad * 100:.3f}%  PSNR(same streams) {p:.1f} dB  rays gpu {cnt.rays} oracle {rays}")
    assert bad <= tol_frac
    assert cnt.paths == W * H * spp
    assert abs(int(cnt.rays) - int(rays)) <= 0.002 * rays + 8


def test_sample_ranges_and_batches_compose(rtb, renderer):
    """[0,8) in one call == [0,3)+[3,8) accumulated == any batch size; rows split too (multi-GPU partitions)."""
    scene = rtb.Scene.named("book2_bouncing")
    cam = scene.info.camera
    renderer.set_scene(scene); renderer.set_camera(cam)
    W, H, D = 128, 72, 20
    renderer.render(W, H, 0, 8, D); whole = renderer.download_accum()
    renderer.render(W, H, 0, 8, D); again = renderer.download_accum()
    assert np.array_equal(whole, again), "render is not deterministic"
    renderer.render(W, H, 0, 3, D); renderer.render(W, H, 3, 8, D, clear=False); split = renderer.download_accum()
    np.testing.assert_allclose(split, whole, rtol=1e-5, atol=1e-5)
    renderer.render(W, H, 0, 8, D, samples_per_batch=3); b3 = renderer.download_accum()
    np.testing.assert_allclose(b3, whole, rtol=1e-5, atol=1e-5)
    renderer.render(W, H, 0, 8, D, rows=(0, 30)); renderer.render(W, H, 0, 8, D, rows=(30, 72), clear=False); rows = renderer.download_accum()
    assert np.array_equal(rows, whole), "row partition changes the image"


def test_full_size_properties(rtb, renderer):
    """BASELINE's headline configuration (Book 2 final scene, 800x800, depth 40) is too large for the oracle, so it is
    checked through properties that do not depend on size: sample ranges and row ranges compose, the image does not
    depend on which world BVH is walked or on the batch size, the ray count is the same every time, and the output
    is a finite image in [0, 1] with alpha 1."""
    scene = rtb.Scene.named("book2_final"); cam = scene.info.camera
    W, H, D, SPP = scene.info.width, scene.info.height, scene.info.max_depth, 6
    assert (W, H, D) == (800, 800, 40)
    renderer.set_scene(scene); renderer.set_camera(cam)
    renderer.reset_counters(); renderer.render(W, H, 0, SPP, D, seed=1984); whole = renderer.download_accum(); c0 = renderer.counters()
    assert c0.paths == W * H * SPP and c0.rays > 4 * c0.paths
    assert np.isfinite(whole).all() and np.array_equal(whole[..., 3], np.full((H, W), SPP, dtype=np.float32)) and (whole[..., :3] >= 0).all()
    out = renderer.download()
    assert np.isfinite(out).all() and out[..., :3].min() >= 0.0 and out[..., :3].max() <= 1.0 and (out[..., 3] == 1.0).all()
    # sample ranges add up (float addition order differs: allclose), rows partition exactly
    renderer.render(W, H, 0, 2, D, seed=1984); renderer.render(W, H, 2, SPP, D, seed=1984, clear=False)
    np.testing.assert_allclose(renderer.download_accum(), whole, rtol=1e-5, atol=1e-5)
    renderer.reset_counters()
    renderer.render(W, H, 0, SPP, D, seed=1984, rows=(0, 333)); renderer.render(W, H, 0, SPP, D, seed=1984, rows=(333, H), clear=False)
    assert np.array_equal(renderer.download_accum(), whole) and renderer.counters().rays == c0.rays
    # batch size (1.28 M-path batches instead of one 3.84 M-path batch): same paths, same sums per pixel
    renderer.reset_counters(); renderer.render(W, H, 0, SPP, D, seed=1984, samples_per_batch=2)
    np.testing.assert_allclose(renderer.download_accum(), whole, rtol=1e-5, atol=1e-5)     # (per-pixel sums associate differently)
    assert renderer.counters().rays == c0.rays
    # the tree does not matter: the GPU-built linear BVH gives the same image, path for path
    scene.set_world_bvh(rtb.WORLD_BVH_GPU_LBVH); renderer.set_scene(scene)
    assert renderer.scene_stats()["builder"] == "gpu_lbvh"
    renderer.reset_counters(); renderer.render(W, H, 0, SPP, D, seed=1984); lb = renderer.download_accum()
    scene.set_world_bvh(rtb.WORLD_BVH_QUALITY)
    differing = (np.abs(lb[..., :3] - whole[..., :3]).max(axis=2) > 1e-4 * np.maximum(whole[..., :3].max(axis=2), 1.0)).mean()
    assert differing < 1e-4 and abs(int(renderer.counters().rays) - int(c0.rays)) <= 1e-5 * c0.rays
    # another seed is another image
    renderer.set_scene(scene); renderer.render(W, H, 0, SPP, D, seed=7)
    assert not np.array_equal(renderer.download_accum(), whole)


def test_furnace_energy_is_conserved(rtb, renderer):
    """White Lambertian boxes, spheres and an instanced box under a constant white background: every path carries
    throughput exactly 1 until it escapes (radiance 1) or runs out of depth (radiance 0), so every accumulated sample is 0
    or 1 exactly, whatever the geometry does — at the headline image size."""
    s = rtb.Scene(); white = s.lambertian(albedo=(1.0, 1.0, 1.0))
    rng = np.random.default_rng(5)
    objs = [s.box((-30.0, -1.0, -30.0), (30.0, 0.0, 30.0), white)]
    objs += [s.box((float(x), 0.0, float(z)), (float(x) + 1.5, float(rng.uniform(0.5, 3.0)), float(z) + 1.5), white) for x in range(-8, 8, 3) for z in range(-8, 8, 3)]
    objs += [s.sphere((float(rng.uniform(-8, 8)), float(rng.uniform(0.5, 4)), float(rng.uniform(-8, 8))), float(rng.uniform(0.3, 1.0)), white) for _ in range(40)]
    objs.append(s.translate(s.rotate_y(s.box((0.0, 0.0, 0.0), (2.0, 5.0, 2.0), white), 25.0), (3.0, 0.0, -2.0)))
    s.set_root(s.list(objs)); s.set_background(rtb.BG_CONSTANT, (1.0, 1.0, 1.0))
    cam = rtb.make_camera("pinhole", (14, 9, 16), (0, 1, 0), (0, 1, 0), 40.0, 1.0)
    renderer.set_scene(s); renderer.set_camera(cam)
    W = H = 800; SPP = 5
    renderer.render(W, H, 0, SPP, 40, seed=3); acc = renderer.download_accum()
    assert np.array_equal(acc[..., 3], np.full((H, W), SPP, dtype=np.float32))
    rgb = acc[..., :3]
    assert np.array_equal(rgb, np.round(rgb)) and rgb.min() >= 0 and rgb.max() <= SPP          # whole numbers of escaped paths
    assert np.array_equal(rgb[..., 0], rgb[..., 1]) and np.array_equal(rgb[..., 0], rgb[..., 2])
    assert 0.9 < rgb.mean() / SPP <= 1.0                                                        # nearly everything escapes within 40 bounces


def test_download_matches_reference_tonemap(rtb, renderer):
    scene = rtb.Scene.named("book2_checker")
    renderer.set_scene(scene); renderer.set_camera(scene.info.camera)
    renderer.render(64, 36, 0, 4, 10)
    out = renderer.download(); acc = renderer.download_accum()
    assert np.array_equal(out[..., 3], np.ones((36, 64), dtype=np.float32))
    np.testing.assert_allclose(out[..., :3], tonemap(acc), rtol=2e-7, atol=1e-7)


def test_errors_are_loud(rtb):
    r = rtb.Renderer(0)
    with pytest.raises(rtb.RtbError):
        r.render(8, 8, 0, 1, 4)            # no scene
    s = rtb.Scene()
    with pytest.raises(rtb.RtbError):
        r.set_scene(s)                      # no root
    with pytest.raises(rtb.RtbError):
        s.sphere((0, 0, 0), 1.0, 5)         # bad material id


def test_cli_app_matches_the_library(rtb, renderer, tmp_path):
    """rtb_app book2_bouncing goes through the host mirror exactly like FirstApp::MakeApp/Run
    (MotionBlurCamera -> SceneBook2BVH::Factory -> Renderer::MakeRenderer -> Render -> DownloadRenderbuffer)
    and writes the 8-bit image the way write_renderbuffer does (x*255.999, rows flipped)."""
    import subprocess
    from conftest import ROOT
    out = tmp_path / "img.ppm"
    W, H, SPP, D = 160, 90, 4, 12
    subprocess.run([str(ROOT / "ray-tracing-v06_b200" / "rtb_app"), "book2_bouncing", "--width", str(W), "--height", str(H), "--spp", str(SPP),
                    "--depth", str(D), "--out", str(out)], check=True, capture_output=True)
    raw = out.read_bytes()
    header = f"P6\n{W} {H}\n255\n".encode()
    assert raw.startswith(header)
    img = np.frombuffer(raw[len(header):], dtype=np.uint8).reshape(H, W, 3)
    scene = rtb.Scene.named("book2_bouncing")
    cam = rtb.make_camera("motion", (13, 2, 3), (0, 0, 0), (0, 1, 0), 30.0, W / H, t0=0.1, t1=1.0)
    renderer.set_scene(scene); renderer.set_camera(cam)
    renderer.render(W, H, 0, SPP, D, seed=1984)
    ref = (renderer.download()[::-1, :, :3] * np.float32(255.999)).astype(np.uint8)
    assert np.array_equal(img, ref)


def _check_tree(nodes, root, n_prims):
    """Structure of a world BVH in the reference node layout: 2n-1 nodes, every primitive in exactly one leaf,
    every inner box the exact union of its children's."""
    assert len(nodes) == 2 * n_prims - 1
    leaf = nodes["left_child_idx"] == -1
    assert sorted(nodes["right_child_hittable_idx"][leaf].tolist()) == list(range(n_prims))
    inner = np.nonzero(~leaf)[0]
    l = nodes[nodes["left_child_idx"][inner]]; r = nodes[nodes["right_child_hittable_idx"][inner]]
    assert np.array_equal(nodes["bmin"][inner], np.minimum(l["bmin"], r["bmin"]))
    assert np.array_equal(nodes["bmax"][inner], np.maximum(l["bmax"], r["bmax"]))
    seen = np.zeros(len(nodes), dtype=np.int32)           # a tree: every node but the root has exactly one parent
    np.add.at(seen, nodes["left_child_idx"][inner], 1); np.add.at(seen, nodes["right_child_hittable_idx"][inner], 1)
    assert seen[root] == 0 and (np.delete(seen, root) == 1).all()


@pytest.mark.parametrize("name,lo,hi", [("book2_bouncing", -12, 12), ("book2_final", -200, 600), ("mesh_icospheres", -4, 4), ("book2_cornell_smoke", 0, 555)])
def test_gpu_lbvh_world_bvh(rtb, orc, renderer, name, lo, hi):
    """RTB_WORLD_BVH_GPU_LBVH: the tree built on the device (Morton codes, radix sort, one-pass hierarchy, bottom-up
    fit) is a valid BVH over the same primitives, and closest hits through it are bit-identical to the oracle's
    (which walks the scene graph as the reference would)."""
    scene = rtb.Scene.named(name)
    scene.set_world_bvh(rtb.WORLD_BVH_GPU_LBVH)
    renderer.set_scene(scene)
    st = renderer.scene_stats()
    assert st["builder"] == "gpu_lbvh" and st["depth"] <= 30
    nodes, root = scene.world_bvh()
    _check_tree(nodes, root, st["primitives"])
    rays = np.concatenate([camera_rays(rtb, scene.info.camera, 160, 160, "renderer"), random_rays(rtb, 100_000, lo, hi, seed=5)])
    if name != "book2_cornell_smoke":                       # (a medium's hit distance is random: the image below covers that scene)
        g = renderer.trace_rays(rays)
        o = _oracle_scene(orc, scene).trace_rays(rays, rtb.HIT_DTYPE)
        assert _compare_hits(rtb, g, o, exact=True) > 10_000
    # and the same image, path for path
    cam = scene.info.camera; renderer.set_camera(cam)
    renderer.render(96, 96, 0, 4, 20, seed=1984); gpu = renderer.download_accum()
    ref, _, _ = _oracle_scene(orc, scene).render(cam, 96, 96, 0, 4, 20, seed=1984)
    diff = np.abs(gpu[..., :3] - ref[..., :3]).max(axis=2)
    assert float((diff > 1e-4 * np.maximum(np.abs(ref[..., :3]).max(axis=2), 1.0)).mean()) <= 0.02


def test_gpu_lbvh_degenerate_inputs(rtb, orc, renderer):
    """One primitive, two primitives, and many primitives with identical boxes (equal Morton codes are split by
    sorted position; a run that would make the tree deeper than the traversal stack falls back to the host builder)."""
    for count, same in [(1, False), (2, False), (3, False), (700, True), (5000, True)]:
        s = rtb.Scene(); m = s.lambertian(albedo=(0.5, 0.5, 0.5))
        ids = [s.sphere((1.0, 2.0, 3.0) if same else (2.5 * k, 0.0, 0.0), 0.5 + (0.001 * k if same else 0.0), m) for k in range(count)]
        s.set_root(s.list(ids)); s.set_world_bvh(rtb.WORLD_BVH_GPU_LBVH)
        renderer.set_scene(s)
        st = renderer.scene_stats()
        assert st["primitives"] == count and st["depth"] <= 30 and st["builder"] in ("gpu_lbvh", "host_sah", "host_median_fallback")
        if count <= 700:
            assert st["builder"] == "gpu_lbvh"
        nodes, root = s.world_bvh(); _check_tree(nodes, root, count)
        rays = random_rays(rtb, 20_000, -6, 9, seed=count)
        g = renderer.trace_rays(rays); o = _oracle_scene(orc, s).trace_rays(rays, rtb.HIT_DTYPE)
        _compare_hits(rtb, g, o, exact=True)


def test_gpu_lbvh_deep_tree_uses_the_deep_stack(rtb, orc, renderer):
    """A linear BVH can be much deeper than a SAH tree: centres at 1000 * 2^-k peel off one Morton bit per level,
    and 4,000 primitives sharing one cell add their own levels.  Past 30 levels the kernels switch to the 64-entry
    stack; hits and the image stay identical to the oracle's."""
    s = rtb.Scene(); m = s.lambertian(albedo=(0.5, 0.5, 0.5)); g = s.dielectric(1.5)
    ids = [s.sphere((1000.0 * 2.0 ** -k, 0.0, 0.0), 0.2 * 1000.0 * 2.0 ** -k, m if k % 2 else g) for k in range(21)]
    ids += [s.sphere((0.0, 0.0, 0.0), 0.05 * (1 + k / 4000.0), m) for k in range(4000)]
    s.set_root(s.list(ids)); s.set_world_bvh(rtb.WORLD_BVH_GPU_LBVH)
    renderer.set_scene(s)
    st = renderer.scene_stats()
    assert st["builder"] == "gpu_lbvh" and 30 < st["depth"] <= 62, st
    nodes, root = s.world_bvh(); _check_tree(nodes, root, len(ids))
    cam = rtb.make_camera("pinhole", (400, 300, 900), (300, 0, 0), (0, 1, 0), 60.0, 1.0)
    rays = np.concatenate([camera_rays(rtb, cam, 128, 128, "renderer"), random_rays(rtb, 20_000, -50, 1100, seed=3), random_rays(rtb, 10_000, -3, 3, seed=4)])
    rays["d"][-10_000:] = -rays["o"][-10_000:] + rays["d"][-10_000:] * np.float32(0.01)   # the last third aims at the crowded cell
    g_hits = renderer.trace_rays(rays); o = _oracle_scene(orc, s); o_hits = o.trace_rays(rays, rtb.HIT_DTYPE)
    assert _compare_hits(rtb, g_hits, o_hits, exact=True) > 5_000
    renderer.set_camera(cam); renderer.render(64, 64, 0, 4, 12, seed=5); gpu = renderer.download_accum()
    ref, _, _ = o.render(cam, 64, 64, 0, 4, 12, seed=5)
    np.testing.assert_allclose(gpu[..., :3], ref[..., :3], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("name", ["book2_final", "book2_cornell"])
def test_box_leaf_equals_six_quad_leaves(rtb, orc, renderer, name, monkeypatch):
    """A box is one BVH leaf whose slab test picks the faces to run the exact quad test on (PRIM_BOX); with
    RTB_BOX_AS_QUADS=1 its six quads are independent leaves as in the book.  Both must give the same hit records, bit for
    bit, including for rays aimed exactly at box edges and corners (where two faces meet, or none is hit) — and both
    equal the oracle, which evaluates the six quads of every box in list order."""
    scene = rtb.Scene.named(name)
    _, _, objs, _ = parse_blob(scene.serialize())
    boxes = np.array([o["f"][:6] for o in objs if o["kind"] == 4], dtype=np.float32)
    assert len(boxes) >= 2
    rng = np.random.default_rng(17)
    n = 60_000
    b = boxes[rng.integers(0, len(boxes), n)]
    # a point on the box surface with 1, 2 or 3 coordinates pinned to a face: faces, edges, corners
    u = rng.random((n, 3), dtype=np.float32)
    target = b[:, :3] + (b[:, 3:] - b[:, :3]) * u
    pin = rng.integers(1, 8, n)
    for k in range(3):
        side = rng.integers(0, 2, n).astype(bool)
        pinned = ((pin >> k) & 1).astype(bool)
        target[pinned, k] = np.where(side[pinned], b[pinned, 3 + k], b[pinned, k])
    rays = random_rays(rtb, n, float(boxes.min()) - 50, float(boxes.max()) + 50, seed=23)
    if name == "book2_cornell":      # the boxes are instanced (rotate_y + translate): aim in world space at the rotated target
        rays = np.concatenate([camera_rays(rtb, scene.info.camera, 200, 200, "renderer"), rays])
    else:
        rays["d"] = target - rays["o"]
        rays = np.concatenate([camera_rays(rtb, scene.info.camera, 200, 200, "renderer"), rays, random_rays(rtb, 40_000, -200, 600, seed=29)])
    hits = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("RTB_BOX_AS_QUADS", mode)
        scene.set_world_bvh(rtb.WORLD_BVH_QUALITY)           # bumps the scene version: forces a re-flatten under the new mode
        renderer.set_scene(scene)
        hits[mode] = renderer.trace_rays(rays)
    monkeypatch.delenv("RTB_BOX_AS_QUADS")
    assert renderer.scene_stats()["primitives"] > 0
    g, q = hits["0"], hits["1"]
    # Independent quad leaves are flat boxes padded by 1e-4 in the BVH: a ray aimed exactly at an edge or a corner can
    # lose them to the rounding of the slab test (about 6e-8 |o/d|).  The box leaf selects its faces with a tolerance
    # and finds those hits, as the oracle (which has no BVH inside a box) does.  So: the quad-leaf run may miss a few
    # of the aimed rays, never the other way round; everywhere else the two runs agree bit for bit.
    same_t = g["t"].view(np.uint32) == q["t"].view(np.uint32)
    assert (~same_t).mean() < 0.005 and (g["t"][~same_t] < q["t"][~same_t]).all()
    assert np.array_equal(g["p"][same_t].view(np.uint32), q["p"][same_t].view(np.uint32))
    # Two surfaces met at the same t, bit for bit (two faces of one box at an edge; the wall two neighbouring boxes
    # share): the box leaf keeps the first face in list order, as the oracle's hittable_list does; between leaves,
    # whichever the walk met first stays.
    tie = same_t & ((g["n"].view(np.uint32) != q["n"].view(np.uint32)).any(axis=1) | (g["object"] != q["object"]))
    assert tie.mean() < 0.10
    ok = same_t & ~tie
    for field in ("object", "material", "front_face", "u", "v"):
        assert np.array_equal(g[field][ok], q[field][ok]), field
    assert (g["prims_tested"].sum() < q["prims_tested"].sum()) and (g["nodes_visited"].sum() < q["nodes_visited"].sum())
    # Against the oracle: identical, except that the oracle walks the scene's own bvh_node trees with the reference's
    # slab test and can itself lose an edge-on hit to a box cull (at most a handful of the 60,000 aimed rays).
    o = _oracle_scene(orc, scene).trace_rays(rays, rtb.HIT_DTYPE)
    agree = g["t"].view(np.uint32) == o["t"].view(np.uint32)
    assert (~agree).sum() <= 8, f"{(~agree).sum()} rays differ from the oracle"
    assert _compare_hits(rtb, g[agree], o[agree], exact=True, max_tie_frac=0.10) > 10_000     # (rays aimed at edges: many shared-wall ties)


def test_cli_app_renders_an_obj_mesh(tmp_path):
    """rtb_app --obj: MeshHandle::LoadObj -> MakeMesh -> HittableList -> Renderer::MakeRenderer.  An octahedron of grey
    clay on the checkered floor under the sky: the centre of the image is the mesh (grey, r == g == b up to noise),
    the top row is sky (blue-ish), the bottom rows are floor."""
    import subprocess
    from conftest import ROOT
    (tmp_path / "octa.obj").write_text("v 1 0 0\nv -1 0 0\nv 0 1 0\nv 0 -1 0\nv 0 0 1\nv 0 0 -1\n"
                                       "f 1 3 5\nf 3 2 5\nf 2 4 5\nf 4 1 5\nf 3 1 6\nf 2 3 6\nf 4 2 6\nf 1 4 6\n")
    out = tmp_path / "octa.ppm"
    W, H = 120, 90
    log = subprocess.run([str(ROOT / "ray-tracing-v06_b200" / "rtb_app"), "--obj", str(tmp_path / "octa.obj"), "--width", str(W), "--height", str(H),
                          "--spp", "64", "--depth", "8", "--out", str(out)], check=True, capture_output=True, text=True).stdout
    assert "8 triangles" in log
    raw = out.read_bytes(); header = f"P6\n{W} {H}\n255\n".encode()
    assert raw.startswith(header)
    img = np.frombuffer(raw[len(header):], dtype=np.uint8).reshape(H, W, 3).astype(np.int32)
    centre = img[H // 2 - 3:H // 2 + 3, W // 2 - 3:W // 2 + 3].reshape(-1, 3).mean(axis=0)
    sky = img[0].mean(axis=0)
    assert sky[2] > sky[0] + 20                                     # sky gradient: blue over red at the top
    assert abs(centre[0] - centre[2]) < 25 and 40 < centre.mean() < 250   # grey clay lit by the sky
    assert img.std() > 10


def test_edge_cases_gpu(rtb, orc, renderer):
    """Empty and ragged inputs: empty sample range, 1x1 and odd-sized images, depth 1, depth 200, reallocation."""
    scene = rtb.Scene.named("book2_checker"); cam = scene.info.camera
    renderer.set_scene(scene); renderer.set_camera(cam)
    o = _oracle_scene(orc, scene)
    renderer.render(8, 4, 5, 5, 10)                                 # empty sample range: accumulators stay zero
    assert not renderer.download_accum().any()
    for (W, H, s0, s1, D) in [(1, 1, 0, 3, 1), (33, 17, 2, 9, 3), (257, 3, 0, 2, 200), (5, 129, 0, 1, 50)]:
        renderer.render(W, H, s0, s1, D, seed=11)
        g = renderer.download_accum()
        ref, _, rays = o.render(cam, W, H, s0, s1, D, seed=11)
        assert g.shape == (H, W, 4) and np.array_equal(g[..., 3], ref[..., 3])
        np.testing.assert_allclose(g[..., :3], ref[..., :3], rtol=1e-5, atol=1e-5)
    assert renderer.trace_rays(np.zeros(0, dtype=rtb.RAY_DTYPE)).shape == (0,)
    with pytest.raises(rtb.RtbError):
        renderer.render(0, 4, 0, 1, 4)
    with pytest.raises(rtb.RtbError):
        renderer.render(4, 4, 3, 1, 4)                              # sample_end < sample_begin
    with pytest.raises(rtb.RtbError):
        renderer.render(4, 4, 0, 1, 4, rows=(3, 9))


def test_media_only_and_many_media(rtb, orc, renderer):
    """A scene that is nothing but a medium (no BVH at all), and one with more media than the pre-test list holds
    (the rest become BVH leaves): both must follow the oracle sample for sample."""
    s = rtb.Scene()
    s.set_root(s.constant_medium(s.sphere((0, 0, 0), 2.0, s.dielectric(1.5)), 0.8, s.isotropic(s.solid((0.8, 0.6, 0.3)))))
    s.set_background(rtb.BG_CONSTANT, (0.7, 0.8, 1.0))
    many = rtb.Scene(); objs = []
    white = many.lambertian(albedo=(0.7, 0.7, 0.7))
    objs.append(many.quad((-20, -1, -20), (40, 0, 0), (0, 0, 40), white))
    for k in range(11):
        iso = many.isotropic(many.solid((0.2 + 0.07 * k, 0.9 - 0.06 * k, 0.5)))
        if k % 2:
            b = many.translate(many.rotate_y(many.box((-0.6, 0, -0.6), (0.6, 1.5, 0.6), white), 10.0 * k), (-7.5 + 1.5 * k, -1, 0.5 * k))
        else:
            b = many.sphere((-7.5 + 1.5 * k, 0.0, 0.3 * k), 0.7, white)
        objs.append(many.constant_medium(b, 0.9, iso))
    many.set_root(many.list(objs))
    cam = rtb.make_camera("pinhole", (0, 1.5, -14), (0, 0, 0), (0, 1, 0), 40.0, 2.0)
    for sc, name in ((s, "medium only"), (many, "11 media")):
        renderer.set_scene(sc); renderer.set_camera(cam)
        renderer.render(96, 48, 0, 8, 30, seed=5)
        g = renderer.download_accum()
        ref, _, rays = _oracle_scene(orc, sc).render(cam, 96, 48, 0, 8, 30, seed=5)
        diff = np.abs(g[..., :3] - ref[..., :3]).max(axis=2)
        bad = float((diff > 1e-4 * np.maximum(ref[..., :3].max(axis=2), 1.0)).mean())
        print(f"{name}: mismatching pixels {bad * 100:.3f}%  rays gpu {renderer.counters().rays}")
        assert bad <= 0.02 and g[..., :3].sum() > 0


def test_scene_and_size_switching(rtb, renderer):
    """One renderer, several scenes and framebuffer sizes back to back (arena / queue reallocation, graph rebuild)."""
    ref = {}
    for name, W, H in [("book2_quads", 64, 64), ("book2_final", 80, 80), ("book2_quads", 64, 64), ("book2_final", 40, 120), ("book2_final", 80, 80)]:
        scene = rtb.Scene.named(name)
        renderer.set_scene(scene); renderer.set_camera(scene.info.camera)
        renderer.render(W, H, 0, 4, 20, seed=3)
        img = renderer.download_accum()
        key = (name, W, H)
        if key in ref:
            assert np.array_equal(ref[key], img), key
        ref[key] = img


def test_signed_zero_and_axis_parallel_directions(rtb, orc, renderer):
    """Direction components of exactly +0.0 and -0.0 (numpy's `-np.array([0, 0, 1])` is (-0, -0, -1)): the slab test takes
    every sign decision from the value it took the reciprocal of, so such rays - from inside and outside the boxes - walk
    the tree like any other (aabb::intersects, aabb.cuh:30-44, gives -inf..+inf on such an axis)."""
    for name, lo, hi in (("book2_bouncing", -8.0, 8.0), ("book2_final", -100.0, 500.0), ("book2_cornell", 50.0, 500.0)):
        scene = rtb.Scene.named(name)
        renderer.set_scene(scene)
        rng = np.random.default_rng(99)
        n = 30_000
        rays = np.zeros(n, dtype=rtb.RAY_DTYPE)
        rays["o"] = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
        if name == "book2_bouncing":
            rays["o"][:, 1] = rng.uniform(0.05, 3.0, n).astype(np.float32)
        d = rng.normal(size=(n, 3)).astype(np.float32)
        zero = rng.integers(0, 7, n)                      # which components are zeroed (never all three)
        sign = rng.integers(0, 2, (n, 3)).astype(bool)
        for k in range(3):
            z = ((zero >> k) & 1).astype(bool)
            d[z, k] = np.where(sign[z, k], np.float32(-0.0), np.float32(0.0))
        rays["d"] = d; rays["time"] = rng.random(n).astype(np.float32)
        assert (np.signbit(rays["d"]) & (rays["d"] == 0)).sum() > 1000
        g = renderer.trace_rays(rays)
        o = _oracle_scene(orc, scene).trace_rays(rays, rtb.HIT_DTYPE)
        assert _compare_hits(rtb, g, o, exact=True, max_tie_frac=0.02) > 3_000


def test_thin_far_geometry_is_never_culled(rtb, orc, renderer):
    """Quads (zero thickness; 1e-4 of padding in the BVH, which vanishes in float32 beyond 1,000 units) and 1e-4-thick boxes
    1,000 to 10,000 units from the rays' origins, seen face-on, obliquely and edge-on: the reference's slab test
    ((min - o) / d, aabb.cuh:30-44) keeps such boxes, and the product's reciprocal form widens the far distance by its
    rounding bound so that it does too.  The oracle scans the list without any BVH: every hit must be found, bit for bit."""
    rng = np.random.default_rng(4)
    s = rtb.Scene(); m = s.lambertian(albedo=(0.5, 0.5, 0.5))
    objs = []; targets = []
    for k in range(300):
        dist = float(rng.uniform(1000.0, 10000.0))
        dirn = rng.normal(size=3); dirn /= np.linalg.norm(dirn)
        c = (dirn * dist).astype(np.float32)
        axis = int(rng.integers(0, 3))
        u = np.zeros(3, dtype=np.float32); v = np.zeros(3, dtype=np.float32)
        u[(axis + 1) % 3] = rng.uniform(0.5, 4.0); v[(axis + 2) % 3] = rng.uniform(0.5, 4.0)
        if k % 3 == 2:      # a 1e-4-thick slab
            a = c.copy(); b = c + u + v; b[axis] = a[axis] + np.float32(1e-4)
            objs.append(s.box(a, b, m))
        else:
            objs.append(s.quad(c, u, v, m))
        targets.append((c, u, v))
    s.set_root(s.list(objs))
    renderer.set_scene(s)
    n_per = 200
    rays = np.zeros(len(targets) * n_per, dtype=rtb.RAY_DTYPE)
    for k, (c, u, v) in enumerate(targets):
        a = rng.random((n_per, 1)).astype(np.float32); b = rng.random((n_per, 1)).astype(np.float32)
        tgt = c[None, :] + u[None, :] * a + v[None, :] * b
        o = rng.uniform(-5.0, 5.0, (n_per, 3)).astype(np.float32)
        scale = rng.choice(np.array([1.0, 1e-3, 37.0], dtype=np.float32), (n_per, 1))     # un-normalised directions of several lengths
        rays["o"][k * n_per:(k + 1) * n_per] = o
        rays["d"][k * n_per:(k + 1) * n_per] = (tgt - o) * scale
    g = renderer.trace_rays(rays)
    o_hits = _oracle_scene(orc, s).trace_rays(rays, rtb.HIT_DTYPE)
    assert (o_hits["object"] >= 0).mean() > 0.5
    lost = (o_hits["object"] >= 0) & (g["object"] < 0)
    assert not lost.any(), f"{lost.sum()} hits of the oracle were culled by the slab test"
    assert _compare_hits(rtb, g, o_hits, exact=True, max_tie_frac=0.02) > 20_000


# ---------------------------------------------------------------- analytic pins (tests/analytic.py) through the CUDA path

def _gpu_trace(renderer):
    def trace(scene, rays):
        renderer.set_scene(scene)
        return renderer.trace_rays(rays)
    return trace


def _gpu_render(renderer):
    def render(scene, cam, w, h, spp, depth):
        renderer.set_scene(scene); renderer.set_camera(cam)
        renderer.render(w, h, 0, spp, depth, seed=5)
        return renderer.download_accum()
    return render


def test_analytic_pins_gpu(rtb, renderer):
    """The hand-derived known answers for the features the reference lacks (quad alpha/beta and (u,v), rotate_y at 90
    degrees, sphere (u,v) at the poles and the seam, the reference's truncating checker at negative coordinates, image
    texel lookup, box faces, triangle barycentrics, emitter and mirror radiance, the white furnace, Beer-Lambert transmission, Perlin noise at lattice points), through rtb_trace_rays /
    rtb_render."""
    import analytic
    analytic.check_quad_alpha_beta(rtb, _gpu_trace(renderer))
    analytic.check_rotate_y_quarter_turn(rtb, _gpu_trace(renderer))
    analytic.check_sphere_uv(rtb, _gpu_trace(renderer))
    analytic.check_checker_at_negative_coordinates(rtb, _gpu_trace(renderer), _gpu_render(renderer))
    analytic.check_image_texture_lookup(rtb, _gpu_render(renderer))
    analytic.check_box_faces(rtb, _gpu_trace(renderer))
    analytic.check_triangle_barycentric(rtb, _gpu_trace(renderer))
    analytic.check_emitter_and_mirror(rtb, _gpu_render(renderer))
    analytic.check_white_furnace(rtb, _gpu_render(renderer))
    analytic.check_beer_lambert(rtb, _gpu_render(renderer))
    analytic.check_perlin_lattice(rtb, _gpu_render(renderer))
