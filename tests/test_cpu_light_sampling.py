"""CPU tests of light importance sampling (DESIGN.md §5b): the rtb_scene_set_sampled_lights API, the RTBS v2 blob, the
flatten hash, and the estimator of the CPU oracle - known answers worked out in float64, unbiasedness against the plain
estimator on independent seeds, and the variance it removes on the Cornell box."""
import ctypes as C

import numpy as np
import pytest

from helpers import parse_blob
from feature_oracle import RNG_XORWOW, FeatureOracleScene

ERR_INVALID, ERR_UNSUPPORTED = -1, -5


def _set(rtb, scene, ids):
    arr = (C.c_int * max(len(ids), 1))(*ids)
    return rtb.lib().rtb_scene_set_sampled_lights(scene.handle, arr, len(ids))


def _kinds_scene(rtb):
    """One object of every kind, and the ids of the ones light sampling must refuse / accept."""
    s = rtb.Scene()
    white = s.lambertian((0.7, 0.7, 0.7)); lamp = s.diffuse_light(s.solid((4, 4, 4))); fog = s.isotropic(s.solid((1, 1, 1)))
    ids = {
        "sphere": s.sphere((0, 2, 0), 0.5, lamp),
        "quad": s.quad((-1, 3, -1), (2, 0, 0), (0, 0, 2), lamp),
        "moving_sphere": s.moving_sphere((0, 1, 0), (0, 1.5, 0), 0.3, lamp),
        "triangle": s.triangle((0, 0, 0), (1, 0, 0), (0, 1, 0), lamp),
        "box": s.box((2, 0, 2), (3, 1, 3), white),
        "flat_quad": s.quad((0, 5, 0), (1, 0, 0), (2, 0, 0), lamp),       # u parallel to v: no area
    }
    ids["medium"] = s.constant_medium(s.sphere((5, 1, 5), 1.0, white), 0.5, fog)
    ids["translated_quad"] = s.translate(s.rotate_y(ids["quad"], 30.0), (1, 0, 0))
    ids["translated_box"] = s.translate(ids["box"], (1, 0, 0))
    ids["list"] = s.list([ids["sphere"], ids["quad"]])
    ids["bvh"] = s.bvh([ids["sphere"], ids["quad"]])
    floor = s.quad((-10, 0, -10), (20, 0, 0), (0, 0, 20), white)
    s.set_root(s.list([floor, ids["sphere"], ids["quad"], ids["box"]]))
    return s, ids


def test_api_validation(rtb):
    s, ids = _kinds_scene(rtb)
    for k in ("moving_sphere", "triangle", "box", "translated_box", "medium", "list", "bvh"):
        assert _set(rtb, s, [ids[k]]) == ERR_UNSUPPORTED, k
    for bad in (-1, s.num_objects(), 10 ** 6):
        assert _set(rtb, s, [bad]) == ERR_INVALID, bad
    assert _set(rtb, s, [ids["flat_quad"]]) == ERR_INVALID
    assert _set(rtb, s, [ids["sphere"]] * (rtb.MAX_SAMPLED_LIGHTS + 1)) == ERR_INVALID
    assert rtb.lib().rtb_scene_set_sampled_lights(s.handle, None, 1) == ERR_INVALID
    assert rtb.lib().rtb_scene_set_sampled_lights(s.handle, None, -1) == ERR_INVALID
    before = s.serialize()
    assert _set(rtb, s, [ids["sphere"], ids["box"]]) == ERR_UNSUPPORTED     # a refused list changes nothing
    assert s.serialize() == before
    assert _set(rtb, s, [ids["sphere"]] * rtb.MAX_SAMPLED_LIGHTS) == 0
    s.sample_lights([ids["sphere"], ids["quad"], ids["translated_quad"]])
    assert parse_blob(s.serialize())[0]["version"] == 2
    s.sample_lights([])                                                   # n = 0 clears
    assert s.serialize() == before
    with pytest.raises(rtb.RtbError, match="sampled light"):
        s.sample_lights([ids["triangle"]])


def test_blob_round_trips(rtb, orc):
    """A scene without lights writes RTBS v1 byte for byte (set-then-cleared included); with lights, v2 = the v1 blob with
    the version word changed and (n, ids) appended, and the oracle loads it."""
    s = rtb.Scene.named("book2_final")
    v1 = s.serialize()
    assert parse_blob(v1)[0]["version"] == 1
    s.sample_lights(s.info.light_ids)
    v2 = s.serialize()
    assert parse_blob(v2)[0]["version"] == 2
    n = len(s.info.light_ids)
    assert len(v2) == len(v1) + 4 + 4 * n
    assert v2[8:len(v1)] == v1[8:] and v2[:4] == v1[:4]
    assert np.array_equal(np.frombuffer(v2[len(v1):], dtype=np.int32), np.array([n, *s.info.light_ids], dtype=np.int32))
    assert FeatureOracleScene(v2).num_lights == n and FeatureOracleScene(v1).num_lights == 0
    with pytest.raises(RuntimeError, match="version"):
        orc.OracleScene(v2)                      # the plain oracle cannot drop a light list silently: it refuses the blob
    s.sample_lights([])
    assert s.serialize() == v1
    with pytest.raises(RuntimeError, match="bad light list"):
        FeatureOracleScene(v2[:len(v1)] + np.array([0], dtype=np.int32).tobytes())


def test_named_scenes_list_their_lights_without_setting_them(rtb):
    want = {"book2_simple_light": 2, "book2_cornell": 1, "book2_cornell_smoke": 1, "book2_final": 1}
    for name in rtb.scene_names():
        s = rtb.Scene.named(name)
        assert len(s.info.light_ids) == want.get(name, 0), name
        assert parse_blob(s.serialize())[0]["version"] == 1, name
        _, mats, objs, _ = parse_blob(s.serialize())
        for i in s.info.light_ids:
            assert objs[i]["kind"] in (0, 2) and mats[objs[i]["mat"]]["kind"] == 3, (name, i)   # a sphere / quad emitter


def test_flatten_hash(rtb):
    s = rtb.Scene.named("book2_cornell")
    h0 = s.flatten_hash()
    s.sample_lights(s.info.light_ids)
    h1 = s.flatten_hash()
    s.sample_lights([])
    assert s.flatten_hash() == h0 and h1 != h0
    s.sample_lights([s.info.light_ids[0], s.info.light_ids[0]])
    assert s.flatten_hash() not in (h0, h1)


def test_xorwow_mode_refuses_light_sampling(rtb, orc):
    s = rtb.Scene.named("book2_cornell"); cam = s.info.camera
    s.sample_lights(s.info.light_ids)
    with pytest.raises(RuntimeError, match="XORWOW"):
        FeatureOracleScene(s.serialize()).render(cam, 8, 8, 0, 2, 4, seed=1, mode=RNG_XORWOW)


@pytest.mark.parametrize("name", ["book2_simple_light", "book2_cornell_smoke"])
def test_light_oracle_without_lights_is_the_oracle(rtb, orc, name):
    """tests/feature_oracle.cpp on a blob without a light list renders exactly what the oracle renders: same sums, same rays."""
    s = rtb.Scene.named(name); cam = s.info.camera
    a, a2, ra = orc.OracleScene(s.serialize()).render(cam, 24, 16, 0, 8, 20, seed=5, want_sum2=True)
    b, b2, rb = FeatureOracleScene(s.serialize()).render(cam, 24, 16, 0, 8, 20, seed=5, want_sum2=True)
    assert np.array_equal(a, b) and np.array_equal(a2, b2) and ra == rb


# ------------------------------------------------------------------------------------------------ known answers
#
# A white Lambertian floor (y = 0, albedo A) under one emitter of radiance E, black background, max_depth = 2: a camera path
# hits the floor, scatters once, and carries A * E when that segment meets the emitter.  The pixel's expectation is
# A * E * F, F the form factor from the floor point to the emitter; the camera looks straight down from below the emitter.

A, E = 0.6, 5.0
KW = KH = 8


def lambert_form_factor(x, poly):
    """Point-to-polygon form factor (Lambert's formula) at point x with normal +y, float64."""
    R = [np.asarray(v, dtype=np.float64) - x for v in poly]
    f = 0.0
    for i in range(len(R)):
        a, b = R[i], R[(i + 1) % len(R)]
        c = np.cross(a, b)
        gamma = np.arccos(np.clip(np.dot(a, b) / (np.linalg.norm(a) * np.linalg.norm(b)), -1.0, 1.0))
        f += gamma * c[1] / np.linalg.norm(c)
    return abs(f) / (2.0 * np.pi)


def floor_points(cam, W, H, height):
    """Where the pixel centres' camera rays meet y = 0 (pinhole camera of rtb_camera_pinhole), float64."""
    o = np.array(cam.o[:], dtype=np.float64); u = np.array(cam.u[:]); v = np.array(cam.v[:]); w = np.array(cam.w[:])
    pts = np.zeros((H, W, 3))
    for y in range(H):
        for x in range(W):
            s = ((x + 0.5) / W) * 2 - 1; t = ((y + 0.5) / H) * 2 - 1
            d = w + u * s + v * t
            pts[y, x] = o + d * (-o[1] / d[1])
    return pts


def known_answer_scene(rtb, kind):
    s = rtb.Scene()
    floor_mat = s.lambertian((A, A, A)); lamp = s.diffuse_light(s.solid((E, E, E)))
    floor = s.quad((-50, 0, -50), (100, 0, 0), (0, 0, 100), floor_mat)
    if kind == "quad":
        light = s.quad((-1.0, 2.0, -0.75), (2.0, 0, 0), (0, 0, 1.5), lamp)
        poly = [(-1.0, 2.0, -0.75), (1.0, 2.0, -0.75), (1.0, 2.0, 0.75), (-1.0, 2.0, 0.75)]
        expect = lambda p: lambert_form_factor(p, poly)
        cam_y = 1.0
    else:
        c, R = np.array([0.3, 3.0, -0.2]), 0.8
        light = s.sphere(tuple(c), R, lamp)
        def expect(p):
            e = c - p; d = np.linalg.norm(e)
            return (R / d) ** 2 * (e[1] / d)
        cam_y = 1.5
    s.set_root(s.list([floor, light]))
    s.set_background(rtb.BG_CONSTANT, (0, 0, 0))
    cam = rtb.make_camera("pinhole", (0, cam_y, 0), (0, 0, 0), (0, 0, 1), 40.0, 1.0)
    pts = floor_points(cam, KW, KH, cam_y)
    want = A * E * np.array([[expect(pts[y, x]) for x in range(KW)] for y in range(KH)])
    return s, cam, light, want


def check_known_answer(sums, sums2, spp, want, label):
    n = float(spp)
    m = sums[..., 0].astype(np.float64) / n
    var = np.maximum(sums2[..., 0].astype(np.float64) / n - m ** 2, 0.0) / n
    err = float((m - want).mean()); sigma = float(np.sqrt(var.sum()) / var.size)
    print(f"{label}: mean {m.mean():.5f} expected {want.mean():.5f} error/sigma {err / sigma:+.2f}")
    assert abs(err) <= 4.0 * sigma, (label, err, sigma)
    assert np.array_equal(sums[..., 0], sums[..., 1]) and np.array_equal(sums[..., 0], sums[..., 2])   # white: grey
    return float(var.mean())


@pytest.mark.parametrize("kind", ["quad", "sphere"])
def test_known_answer_on_the_oracle(rtb, orc, kind):
    s, cam, light, want = known_answer_scene(rtb, kind)
    spp = 4096
    variances = {}
    for lights in (False, True):
        s.sample_lights([light] if lights else [])
        a, a2, _ = FeatureOracleScene(s.serialize()).render(cam, KW, KH, 0, spp, 2, seed=11 + lights, want_sum2=True)
        variances[lights] = check_known_answer(a, a2, spp, want, f"oracle {kind} lights={lights}")
    assert variances[True] < 0.5 * variances[False]


# ------------------------------------------------------------------------------------------------ unbiasedness, variance

def mean_error_sigmas(a, a2, b, b2, n):
    """Per channel: (mean of the per-pixel difference of the two estimates, its standard error)."""
    ma, mb = a[..., :3].astype(np.float64) / n, b[..., :3].astype(np.float64) / n
    va = np.maximum(a2[..., :3].astype(np.float64) / n - ma ** 2, 0.0) / n
    vb = np.maximum(b2[..., :3].astype(np.float64) / n - mb ** 2, 0.0) / n
    return [(float((ma[..., c] - mb[..., c]).mean()), float(np.sqrt((va[..., c] + vb[..., c]).sum()) / va[..., c].size)) for c in range(3)]


@pytest.mark.parametrize("name", ["book2_cornell", "book2_cornell_smoke"])
def test_oracle_light_sampling_is_unbiased(rtb, orc, name):
    s = rtb.Scene.named(name); cam = s.info.camera
    W = H = 24; spp = 512
    a, a2, _ = orc.OracleScene(s.serialize()).render(cam, W, H, 0, spp, 50, seed=21, want_sum2=True)
    s.sample_lights(s.info.light_ids)
    b, b2, _ = FeatureOracleScene(s.serialize()).render(cam, W, H, 0, spp, 50, seed=22, want_sum2=True)
    for c, (bias, sigma) in enumerate(mean_error_sigmas(b, b2, a, a2, spp)):
        print(f"{name} channel {c}: error / sigma {bias / sigma:+.2f}")
        assert abs(bias) <= 3.0 * sigma, (name, c, bias, sigma)


# Calibrated on the oracle (book2_cornell, 48x48, depth 50, 256 spp, seed 7): the mean per-pixel variance with the light
# sampled is 0.40 of the variance without (median over pixels 0.055; what is left is mostly the edge of the emitter seen
# directly by the camera, which light sampling cannot help).
VARIANCE_RATIO_BAR = 0.5


def pixel_variance(sums, sums2, n):
    m = sums[..., :3].astype(np.float64) / n
    return np.maximum(sums2[..., :3].astype(np.float64) / n - m ** 2, 0.0)


def test_oracle_variance_reduction_on_the_cornell_box(rtb, orc):
    s = rtb.Scene.named("book2_cornell"); cam = s.info.camera
    W = H = 48; spp = 256
    a, a2, _ = orc.OracleScene(s.serialize()).render(cam, W, H, 0, spp, 50, seed=7, want_sum2=True)
    s.sample_lights(s.info.light_ids)
    b, b2, _ = FeatureOracleScene(s.serialize()).render(cam, W, H, 0, spp, 50, seed=7, want_sum2=True)
    ratio = pixel_variance(b, b2, spp).mean() / pixel_variance(a, a2, spp).mean()
    print(f"book2_cornell 48x48x{spp}: variance with / without light sampling {ratio:.3f}")
    assert ratio <= VARIANCE_RATIO_BAR


def test_cli_refuses_sample_lights_for_scenes_without_lights(rtb):
    import subprocess
    from conftest import ROOT
    app = ROOT / "ray-tracing-v06_b200" / "rtb_app"
    for scene in ("book2_quads", "book2_bouncing"):
        out = subprocess.run([str(app), scene, "--sample-lights", "--spp", "1"], capture_output=True, text=True)
        assert out.returncode != 0 and "lists no lights" in out.stderr, out.stderr
