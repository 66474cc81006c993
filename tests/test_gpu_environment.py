"""GPU tests of the HDR environment map (DESIGN.md §5d): the known answers of tests/test_cpu_environment.py through
rtb_render, the CUDA path against the CPU restatement (tests/env_oracle.cpp) on the same Philox streams, unbiasedness of
the sampled map against the oracle's plain one, and the invariances a map must keep (specular-only paths, progressive,
resumed and adaptive renders, two GPUs, the bounds-checked build, rtb_app)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import env_scenes as es
from conftest import ROOT
from env_oracle import EnvOracleScene
from helpers import psnr, tonemap
from test_cpu_environment import SMALL_OBJ, check_mean, write_pfm
from test_cpu_light_sampling import mean_error_sigmas
from test_gpu_adaptive import _dense_snapshots, _expect_per_pixel

pytestmark = pytest.mark.gpu


def _render(rtb, s, cam, W, H, spp, D, seed, **kw):
    r = rtb.Renderer(0); r.set_scene(s); r.set_camera(cam)
    r.render(W, H, 0, spp, D, seed=seed, variance=True, **kw)
    return r.download_accum(want_sum2=True)


# ------------------------------------------------------------------------------------------------ known answers

def test_one_by_one_map_is_the_constant_background(rtb):
    s, cam = es.sky_scene(rtb)
    a, a2 = _render(rtb, s, cam, 96, 64, 8, 12, 3)
    s.set_environment(np.float32(es.SKY).reshape(1, 1, 3))
    b, b2 = _render(rtb, s, cam, 96, 64, 8, 12, 3)
    assert np.array_equal(a, b) and np.array_equal(a2, b2)


def test_orientation(rtb):
    want = es.orientation_map()
    for sample in (False, True):
        s = es.orientation_scene(rtb, sample)
        for axis, (i, j) in es.axis_texels().items():
            a, _ = _render(rtb, s, es.orientation_camera(rtb, axis), 1, 1, 16, 4, 1)
            assert np.array_equal(a[0, 0, :3] / 16, want[j, i]), (axis, sample, a[0, 0], want[j, i])


def test_one_texel_irradiance(rtb):
    want = es.one_texel_expected()
    var = {}
    for sample in (False, True):
        s, cam = es.one_texel_scene(rtb, sample)
        a, a2 = _render(rtb, s, cam, 16, 16, 8192, 2, 41 + sample)
        var[sample] = check_mean(a, a2, 8192, want, f"gpu one texel sample={sample}")
    print(f"gpu one texel: variance sampled / unsampled {var[True] / var[False]:.4f}")
    assert var[True] <= 0.25 * var[False]


def test_furnace(rtb):
    s, cam = es.furnace_scene(rtb, False)
    a, _ = _render(rtb, s, cam, 32, 32, 64, 8, 7)
    assert np.array_equal(a[..., :3], np.full((32, 32, 3), 64.0, np.float32))
    s, cam = es.furnace_scene(rtb, True)
    a, a2 = _render(rtb, s, cam, 32, 32, 2048, 8, 7)
    check_mean(a, a2, 2048, 1.0, "gpu furnace sampled", k=3.0)


# ------------------------------------------------------------------------------------------------ same streams as the oracle

def sun_scene(rtb, W=256, H=128, seed=3, sample=False, sun_deg=4.0):
    """Diffuse, metal and glass spheres on a diffuse ground quad under a procedural sun and sky."""
    s = rtb.Scene()
    ground = s.quad((-30, 0, -30), (60, 0, 0), (0, 0, 60), s.lambertian((0.55, 0.5, 0.45)))
    a = s.sphere((-2.2, 1, 0), 1.0, s.lambertian((0.7, 0.25, 0.2)))
    b = s.sphere((0, 1, 0), 1.0, s.metal((0.8, 0.8, 0.85), 0.1))
    c = s.sphere((2.2, 1, 0), 1.0, s.dielectric(1.5))
    s.set_root(s.list([ground, a, b, c]))
    m, _ = es.sun_sky_map(W, H, seed=seed, sun_deg=sun_deg)
    s.set_environment(m, sample=sample)
    cam = rtb.make_camera("pinhole", (0, 2.5, 8), (0, 0.8, 0), (0, 1, 0), 40.0, 1.5)
    return s, cam


def _with_map(rtb, name, lights, sample):
    s = rtb.Scene.named(name)
    if lights:
        s.sample_lights(s.info.light_ids)
    m, _ = es.sun_sky_map(128, 64, seed=5, sun_deg=6.0)
    s.set_environment(m, scale=(0.5, 0.5, 0.5), sample=sample)
    return s, s.info.camera


def media_scene(rtb):
    """Lights, media and a sampled map together, in the open: a fog sphere and a fog slab (isotropic phase), a diffuse sphere
    and ground, a listed quad light above, under the sun and sky.  (The media are not instanced: the Cornell box with smoke
    rotates and translates its fog boxes, where the device's world-space and the oracle's object-space boundary distances
    already round apart on a few paths without any map - DESIGN.md §4.)"""
    s = rtb.Scene()
    ground = s.quad((-30, 0, -30), (60, 0, 0), (0, 0, 60), s.lambertian((0.55, 0.5, 0.45)))
    ball = s.sphere((-2.2, 1, 0), 1.0, s.lambertian((0.7, 0.25, 0.2)))
    fog = s.constant_medium(s.sphere((0.3, 1.2, 0.2), 1.2, s.lambertian((1, 1, 1))), 0.8, s.isotropic(s.solid((0.8, 0.8, 0.9))))
    slab = s.constant_medium(s.box((1.6, 0.0, -1.0), (3.4, 1.5, 1.0), s.lambertian((1, 1, 1))), 1.5, s.isotropic(s.solid((0.9, 0.7, 0.5))))
    light = s.quad((-1, 4, -1), (2, 0, 0), (0, 0, 2), s.diffuse_light(s.solid((6, 6, 6))))
    s.set_root(s.list([ground, ball, fog, slab, light]))
    s.sample_lights([light])
    m, _ = es.sun_sky_map(128, 64, seed=5, sun_deg=6.0)
    s.set_environment(m, scale=(0.5, 0.5, 0.5), sample=True)
    return s, rtb.make_camera("pinhole", (0, 2.5, 8), (0.5, 1, 0), (0, 1, 0), 40.0, 1.0)


CASES = {
    "map_only": lambda rtb: sun_scene(rtb, sample=False),
    "map_sampled": lambda rtb: sun_scene(rtb, sample=True),
    "map_lights_media": lambda rtb: media_scene(rtb),                                     # isotropic scatters
    "map_deferred_texture": lambda rtb: _with_map(rtb, "book2_simple_light", False, True),  # Perlin albedo: texture_kernel
    "book2_final_800": lambda rtb: _with_map(rtb, "book2_final", True, True),            # binned queues, tail kernel
}


@pytest.mark.parametrize("case,W,H,S,D", [("map_only", 192, 128, 8, 20), ("map_sampled", 192, 128, 8, 20),
                                          ("map_lights_media", 160, 160, 8, 50), ("map_deferred_texture", 200, 112, 8, 50),
                                          ("book2_final_800", 800, 800, 16, 40)])
def test_same_streams_as_the_oracle(rtb, case, W, H, S, D):
    """The bars of test_gpu_light_sampling.py::test_same_streams_as_the_oracle: at most 1e-4 of the pixels differ, ray
    counts within 5e-6."""
    scene, cam = CASES[case](rtb)
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.reset_counters(); r.render(W, H, 0, S, D, seed=1984); g = r.download_accum(); cnt = r.counters()
    ref, _, rays = EnvOracleScene(scene.serialize()).render(cam, W, H, 0, S, D, seed=1984)
    diff = np.abs(g[..., :3] - ref[..., :3]).max(axis=2)
    bad = float((diff > 1e-4 * np.maximum(np.abs(ref[..., :3]).max(axis=2), 1.0)).mean())
    print(f"{case} {W}x{H}x{S}: {bad * 100:.4f} % of pixels differ, rays gpu {cnt.rays} oracle {rays}, PSNR {psnr(tonemap(g), tonemap(ref)):.1f} dB")
    assert bad <= 1e-4
    assert abs(int(cnt.rays) - int(rays)) <= max(5e-6 * rays, 4)


def test_sampled_map_agrees_with_the_oracle_unsampled(rtb):
    """Sampling changes the noise only: the GPU with the sampled map against the oracle's unsampled map on independent
    streams, per channel within 3 sigma."""
    W, H, SPP, D = 48, 32, 2048, 12
    plain, cam = sun_scene(rtb, 64, 32, sample=False, sun_deg=8.0)
    a, a2, _ = EnvOracleScene(plain.serialize()).render(cam, W, H, 0, SPP, D, seed=202, want_sum2=True)
    sampled, _ = sun_scene(rtb, 64, 32, sample=True, sun_deg=8.0)
    g, g2 = _render(rtb, sampled, cam, W, H, SPP, D, 101)
    for c, (bias, sigma) in enumerate(mean_error_sigmas(g, g2, a, a2, SPP)):
        print(f"channel {c}: error / sigma {bias / sigma:+.2f}")
        assert abs(bias) <= 3.0 * sigma + 1e-6, (c, bias, sigma)


# ------------------------------------------------------------------------------------------------ invariances

def test_specular_only_scenes_ignore_sampling(rtb):
    """Metal and glass only: no Lambertian or isotropic scatter, so sampling the map changes nothing."""
    s = rtb.Scene()
    mirror = s.sphere((0, 1, 0), 1.0, s.metal((0.9, 0.9, 0.9), 0.0))
    fuzzy = s.sphere((-2.2, 1, 0), 1.0, s.metal((0.8, 0.6, 0.5), 0.3))
    glass = s.sphere((2.2, 0.8, 0.5), 0.8, s.dielectric(1.5))
    floor = s.quad((-20, 0, -20), (40, 0, 0), (0, 0, 40), s.metal((0.7, 0.6, 0.5), 0.0))
    s.set_root(s.list([mirror, fuzzy, glass, floor]))
    m, _ = es.sun_sky_map(128, 64, seed=9, sun_deg=5.0)
    cam = rtb.make_camera("pinhole", (0, 2, 7), (0, 1, 0), (0, 1, 0), 45.0, 1.5)
    r = rtb.Renderer(0); r.set_camera(cam)
    out = []
    for sample in (False, True):
        s.set_environment(m, sample=sample); r.set_scene(s)
        r.reset_counters(); r.render(120, 80, 0, 16, 20, seed=5, variance=True)
        out.append((*r.download_accum(want_sum2=True), r.counters().rays))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1]) and out[0][2] == out[1][2]
    assert out[0][0][..., :3].max() > 1.0


def test_progressive_and_resumed_renders_are_bit_exact(rtb, tmp_path):
    scene, cam = _with_map(rtb, "book2_cornell_smoke", True, True)
    W, H, D = 96, 80, 24
    a = rtb.Renderer(0); a.set_scene(scene); a.set_camera(cam)
    a.render(W, H, 0, 8, D, seed=11, variance=True, samples_per_batch=1)
    want, want2 = a.download_accum(want_sum2=True)
    a.render(W, H, 0, 3, D, seed=11, variance=True, samples_per_batch=1)
    ck = tmp_path / "env.rtba"
    a.save_accum(ck)
    a.render(W, H, 3, 8, D, seed=11, clear=False, variance=True, samples_per_batch=1)
    got, got2 = a.download_accum(want_sum2=True)
    assert np.array_equal(got, want) and np.array_equal(got2, want2)
    b = rtb.Renderer(0); b.set_scene(scene); b.set_camera(cam)
    assert b.load_accum(ck) == 3
    b.render(W, H, 3, 8, D, seed=11, clear=False, variance=True, samples_per_batch=1)
    got, got2 = b.download_accum(want_sum2=True)
    assert np.array_equal(got, want) and np.array_equal(got2, want2)


@pytest.mark.parametrize("sample", [False, True])
def test_adaptive_render_with_a_map(rtb, sample):
    """Every pixel of an adaptive render holds the dense render's sums at its own count (the LIST x ENV kernels)."""
    scene, cam = sun_scene(rtb, sample=sample)
    W, H, D, seed, spb = 64, 48, 20, 77, 8
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    cursors, c = [0], 0
    while True:
        st = r.render_adaptive(W, H, 128, D, tolerance=0.03, min_spp=8, max_rounds=1, seed=seed, clear=(c == 0), samples_per_batch=spb)
        if st["cursor"] == c:
            break
        c = st["cursor"]; cursors.append(c)
        if st["active_pixels"] == 0:
            break
    a, q = r.download_accum(want_sum2=True)
    print(f"sample={sample}: cursors {cursors}, mean spp {a[..., 3].mean():.1f}")
    assert len(cursors) >= 3 and 0 < (a[..., 3] < cursors[-1]).mean()
    d = rtb.Renderer(0); d.set_scene(scene); d.set_camera(cam)
    _expect_per_pixel(_dense_snapshots(rtb, d, W, H, D, seed, cursors, (0, 0), spb), a, q, (0, 0), H)


def test_two_gpus_with_a_map(rtb):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    scene, cam = _with_map(rtb, "book2_final", True, True)
    W, H, D = 96, 96, 20
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, 5, D, seed=1984, variance=True); a0, q0 = r.download_accum(want_sum2=True)
    r.render(W, H, 5, 10, D, seed=1984, variance=True); a1, q1 = r.download_accum(want_sum2=True)
    m = rtb.MultiRenderer([0, 1], reduce=rtb.REDUCE_P2P)
    m.set_scene(scene); m.set_camera(cam)
    m.render(W, H, 0, 10, D, seed=1984, variance=True); m.synchronize()
    got, got2 = m.download_accum(want_sum2=True)
    assert np.array_equal(got, a0 + a1) and np.array_equal(got2, q0 + q1)


def test_debug_bounds_build_with_a_map(rtb):
    """librtb200_debug.so on map scenes, sampled and not, binning forced: no index out of range (texel and CDF indices are
    checked under the "texture" class)."""
    if not rtb.DEBUG_LIB_PATH.exists():
        pytest.skip("librtb200_debug.so not built")
    code = r'''
import importlib, json, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
rtb = importlib.import_module("ray-tracing-v06_b200")
import env_scenes as es
r = rtb.Renderer(0); n = 0
for name in ("book2_cornell_smoke", "book2_simple_light", "book2_final"):
    for sample in (False, True):
        s = rtb.Scene.named(name)
        s.sample_lights(s.info.light_ids)
        m, _ = es.sun_sky_map(96, 48, seed=n, sun_deg=6.0)
        s.set_environment(m, sample=sample); r.set_scene(s); r.set_camera(s.info.camera); n += 1
        r.render(72, 56, 0, 6, 40, seed=9, samples_per_batch=4, variance=True)
        r.render_adaptive(40, 40, 32, 8, tolerance=0.05, min_spp=4, seed=9)
        r.synchronize()
print("REPORT " + json.dumps(dict(r.debug_bounds_report(), scenes=n)))
''' % (str(ROOT), str(ROOT / "tests"))
    env = dict(os.environ, RTB_LIB=str(rtb.DEBUG_LIB_PATH), RTB_BIN_MASK="116")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    rep = json.loads([l for l in out.stdout.splitlines() if l.startswith("REPORT ")][-1][7:])
    print("bounds report with a map:", rep)
    assert rep.pop("scenes") == 6
    assert rep.pop("rays_checked") > 10_000
    assert all(v == 0 for v in rep.values()), rep


def read_pfm_raw(path):
    with open(path, "rb") as f:
        data = f.read()
    parts = data.split(b"\n", 3)
    W, H = map(int, parts[1].split())
    return np.frombuffer(parts[3], dtype="<f4").reshape(H, W, 3)


def test_rtb_app_env_matches_the_python_render(rtb, tmp_path):
    m, _ = es.sun_sky_map(96, 48, seed=4, sun_deg=6.0)
    write_pfm(tmp_path / "sky.pfm", m)
    W, H, SPP, S = 120, 90, 4, 0.75
    out = tmp_path / "y.pfm"
    res = subprocess.run([str(ROOT / "ray-tracing-v06_b200" / "rtb_app"), "book2_simple_light", "--width", str(W), "--height", str(H),
                          "--spp", str(SPP), "--env", str(tmp_path / "sky.pfm"), "--env-scale", str(S), "--sample-env",
                          "--out", str(out)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    assert "48" in res.stdout and "sampled" in res.stdout
    s = rtb.Scene.named("book2_simple_light")
    s.set_environment(m, scale=(S, S, S), sample=True)
    r = rtb.Renderer(0); r.set_scene(s); r.set_camera(s.info.camera)
    r.render(W, H, 0, SPP, s.info.max_depth, seed=1984)
    want = r.download()[..., :3]
    assert np.array_equal(read_pfm_raw(out), want)


@pytest.mark.parametrize("which", ["obj", "book2_bouncing"])
def test_rtb_app_env_reaches_mirror_built_scenes(tmp_path, which):
    """--obj and the default scene build their world through the host mirror (Renderer::MakeRenderer): --env must reach that
    scene.  A map scaled to 0 leaves only black (neither scene emits), a lit map gives an image other than the default sky's."""
    (tmp_path / "m.obj").write_text(SMALL_OBJ)
    m, _ = es.sun_sky_map(64, 32, seed=2, sun_deg=8.0)
    write_pfm(tmp_path / "sky.pfm", m)
    base = [str(ROOT / "ray-tracing-v06_b200" / "rtb_app")] + (["--obj", str(tmp_path / "m.obj")] if which == "obj" else [])
    base += ["--width", "64", "--height", "48", "--spp", "4", "--depth", "8"]
    imgs = {}
    for label, extra in (("sky", []), ("zero", ["--env", str(tmp_path / "sky.pfm"), "--env-scale", "0"]),
                         ("map", ["--env", str(tmp_path / "sky.pfm"), "--sample-env"])):
        out = tmp_path / f"{label}.pfm"
        res = subprocess.run(base + extra + ["--out", str(out)], capture_output=True, text=True)
        assert res.returncode == 0, (label, res.stderr)
        imgs[label] = read_pfm_raw(out)
    assert (imgs["sky"] > 0).any() and not imgs["zero"].any()
    assert not np.array_equal(imgs["map"], imgs["sky"]) and (imgs["map"] > 0).any()
