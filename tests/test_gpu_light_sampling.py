"""GPU tests of light importance sampling (DESIGN.md §5b): the CUDA path against the CPU oracle path for path on the same
Philox streams, the known answers of tests/test_cpu_light_sampling.py through rtb_render, unbiasedness against the plain
estimator, the variance bar, and the invariances light sampling must keep (specular-only paths, progressive and resumed
renders, two GPUs, the bounds-checked build)."""
import numpy as np
import pytest

from helpers import psnr, tonemap
from light_oracle import LightOracleScene
from test_cpu_light_sampling import (KH, KW, VARIANCE_RATIO_BAR, check_known_answer, known_answer_scene, mean_error_sigmas,
                                     pixel_variance)

pytestmark = pytest.mark.gpu


def _lit(rtb, name):
    s = rtb.Scene.named(name)
    s.sample_lights(s.info.light_ids)
    return s, s.info.camera


@pytest.mark.parametrize("name,W,H,S,D", [("book2_simple_light", 200, 112, 8, 50),    # sphere + quad light, Perlin albedo (deferred texture path)
                                          ("book2_cornell", 160, 160, 8, 50),          # instanced boxes
                                          ("book2_cornell_smoke", 160, 160, 8, 50),    # media: isotropic scatters
                                          ("book2_final", 800, 800, 16, 40)])          # binned queues, tail kernel
def test_same_streams_as_the_oracle(rtb, name, W, H, S, D):
    """Same Philox streams on both sides: the bars of test_gpu_statistics.py::test_headline_config_full_size_same_streams
    (at most 1e-4 of the pixels differ, ray counts within 5e-6)."""
    scene, cam = _lit(rtb, name)
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.reset_counters(); r.render(W, H, 0, S, D, seed=1984); g = r.download_accum(); cnt = r.counters()
    ref, _, rays = LightOracleScene(scene.serialize()).render(cam, W, H, 0, S, D, seed=1984)
    diff = np.abs(g[..., :3] - ref[..., :3]).max(axis=2)
    bad = float((diff > 1e-4 * np.maximum(np.abs(ref[..., :3]).max(axis=2), 1.0)).mean())
    print(f"{name} {W}x{H}x{S} with lights: {bad * 100:.4f} % of pixels differ, rays gpu {cnt.rays} oracle {rays}, PSNR {psnr(tonemap(g), tonemap(ref)):.1f} dB")
    assert bad <= 1e-4
    assert abs(int(cnt.rays) - int(rays)) <= max(5e-6 * rays, 4)
    assert psnr(tonemap(g), tonemap(ref)) > 60.0


@pytest.mark.parametrize("kind", ["quad", "sphere"])
def test_known_answer_on_the_gpu(rtb, kind):
    s, cam, light, want = known_answer_scene(rtb, kind)
    spp = 16384
    r = rtb.Renderer(0); r.set_camera(cam)
    variances = {}
    for lights in (False, True):
        s.sample_lights([light] if lights else [])
        r.set_scene(s); r.render(KW, KH, 0, spp, 2, seed=31 + lights, variance=True)
        a, a2 = r.download_accum(want_sum2=True)
        variances[lights] = check_known_answer(a, a2, spp, want, f"gpu {kind} lights={lights}")
    assert variances[True] < 0.5 * variances[False]


@pytest.mark.parametrize("cfg,name,W,H,D", [("cfg4", "book2_cornell_smoke", 72, 72, 50), ("cfg5", "book2_final", 72, 72, 40)])
def test_lights_on_gpu_agree_with_the_oracle_without_lights(rtb, orc, cfg, name, W, H, D):
    """The expected image does not depend on the light list: the GPU with light sampling against the oracle's plain estimator
    on independent streams, per channel within 3 sigma (the method of test_gpu_statistics.py, its reduced sizes)."""
    SPP = 1024
    plain = rtb.Scene.named(name); cam = plain.info.camera
    a, a2, _ = orc.OracleScene(plain.serialize()).render(cam, W, H, 0, SPP, D, seed=202, want_sum2=True)
    scene, _ = _lit(rtb, name)
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, SPP, D, seed=101, variance=True)
    g, g2 = r.download_accum(want_sum2=True)
    for c, (bias, sigma) in enumerate(mean_error_sigmas(g, g2, a, a2, SPP)):
        print(f"{cfg} channel {c}: error / sigma {bias / sigma:+.2f}")
        assert abs(bias) <= 3.0 * sigma + 1e-6, (cfg, c, bias, sigma)


def test_gpu_variance_reduction_on_the_cornell_box(rtb):
    scene = rtb.Scene.named("book2_cornell"); cam = scene.info.camera
    W = H = 48; spp = 256
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, spp, 50, seed=7, variance=True); a, a2 = r.download_accum(want_sum2=True)
    scene.sample_lights(scene.info.light_ids); r.set_scene(scene)
    r.render(W, H, 0, spp, 50, seed=7, variance=True); b, b2 = r.download_accum(want_sum2=True)
    ratio = pixel_variance(b, b2, spp).mean() / pixel_variance(a, a2, spp).mean()
    print(f"gpu book2_cornell 48x48x{spp}: variance with / without light sampling {ratio:.3f}")
    assert ratio <= VARIANCE_RATIO_BAR


def test_specular_only_paths_ignore_the_light_list(rtb):
    """An emitter and a fuzz-0 mirror (plus glass) under the sky: no Lambertian or isotropic scatter anywhere, so the light
    list changes nothing - bit-identical sums and ray counts."""
    s = rtb.Scene()
    lamp = s.diffuse_light(s.solid((6, 5, 4)))
    light = s.quad((-1, 3, -1), (2, 0, 0), (0, 0, 2), lamp)
    mirror = s.sphere((0, 1, 0), 1.0, s.metal((0.9, 0.9, 0.9), 0.0))
    glass = s.sphere((2.2, 0.8, 0.5), 0.8, s.dielectric(1.5))
    floor = s.quad((-20, 0, -20), (40, 0, 0), (0, 0, 40), s.metal((0.7, 0.6, 0.5), 0.0))
    s.set_root(s.list([light, mirror, glass, floor]))
    cam = rtb.make_camera("pinhole", (0, 2, 7), (0, 1, 0), (0, 1, 0), 45.0, 1.5)
    r = rtb.Renderer(0); r.set_camera(cam)
    out = []
    for lights in ([], [light, mirror]):
        s.sample_lights(lights); r.set_scene(s)
        r.reset_counters(); r.render(120, 80, 0, 16, 20, seed=5, variance=True)
        out.append((*r.download_accum(want_sum2=True), r.counters().rays))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1]) and out[0][2] == out[1][2]
    assert out[0][0][..., :3].max() > 1.0


def test_progressive_and_resumed_renders_are_bit_exact(rtb, tmp_path):
    """With lights: [0,3) + [3,8) (progressive) and [0,3) -> checkpoint -> another renderer -> [3,8) both equal the
    uninterrupted [0,8), bit for bit (one sample per batch, so every sum is formed in the same order)."""
    scene, cam = _lit(rtb, "book2_cornell_smoke")
    W, H, D = 96, 80, 24
    a = rtb.Renderer(0); a.set_scene(scene); a.set_camera(cam)
    a.render(W, H, 0, 8, D, seed=11, variance=True, samples_per_batch=1)
    want, want2 = a.download_accum(want_sum2=True)
    a.render(W, H, 0, 3, D, seed=11, variance=True, samples_per_batch=1)
    ck = tmp_path / "lit.rtba"
    a.save_accum(ck)
    a.render(W, H, 3, 8, D, seed=11, clear=False, variance=True, samples_per_batch=1)
    got, got2 = a.download_accum(want_sum2=True)
    assert np.array_equal(got, want) and np.array_equal(got2, want2)
    b = rtb.Renderer(0); b.set_scene(scene); b.set_camera(cam)
    assert b.load_accum(ck) == 3
    b.render(W, H, 3, 8, D, seed=11, clear=False, variance=True, samples_per_batch=1)
    got, got2 = b.download_accum(want_sum2=True)
    assert np.array_equal(got, want) and np.array_equal(got2, want2)


def test_two_gpus_with_lights(rtb):
    """rtb_multi_render on two GPUs with a light list == the sum of the two sample sub-ranges rendered on one GPU (the light
    table travels with the shared scene arena)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    scene, cam = _lit(rtb, "book2_final")
    W, H, D = 96, 96, 20
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, 5, D, seed=1984, variance=True); a0, q0 = r.download_accum(want_sum2=True)
    r.render(W, H, 5, 10, D, seed=1984, variance=True); a1, q1 = r.download_accum(want_sum2=True)
    m = rtb.MultiRenderer([0, 1], reduce=rtb.REDUCE_P2P)
    m.set_scene(scene); m.set_camera(cam)
    m.render(W, H, 0, 10, D, seed=1984, variance=True); m.synchronize()
    got, got2 = m.download_accum(want_sum2=True)
    assert np.array_equal(got, a0 + a1) and np.array_equal(got2, q0 + q1)


def test_debug_bounds_build_with_lights(rtb):
    """librtb200_debug.so on every scene that lists lights, with light sampling on: no index out of range (the light index
    is checked under the "primitive" class)."""
    import json
    import os
    import subprocess
    import sys
    from conftest import ROOT
    if not rtb.DEBUG_LIB_PATH.exists():
        pytest.skip("librtb200_debug.so not built")
    code = r'''
import importlib, json, sys
sys.path.insert(0, %r)
rtb = importlib.import_module("ray-tracing-v06_b200")
r = rtb.Renderer(0); lit = 0
for name in rtb.scene_names():
    s = rtb.Scene.named(name)
    if not s.info.light_ids:
        continue
    s.sample_lights(s.info.light_ids); r.set_scene(s); r.set_camera(s.info.camera); lit += 1
    r.render(72, 56, 0, 6, 60, seed=9, samples_per_batch=4, variance=True)
    r.render(40, 40, 6, 9, 8, seed=9)
    r.synchronize()
print("REPORT " + json.dumps(dict(r.debug_bounds_report(), lit=lit)))
''' % (str(ROOT),)
    env = dict(os.environ, RTB_LIB=str(rtb.DEBUG_LIB_PATH), RTB_BIN_MASK="116")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    rep = json.loads([l for l in out.stdout.splitlines() if l.startswith("REPORT ")][-1][7:])
    print("bounds report with lights:", rep)
    assert rep.pop("lit") == 4
    assert rep.pop("rays_checked") > 10_000
    assert all(v == 0 for v in rep.values()), rep
