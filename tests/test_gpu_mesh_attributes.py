"""GPU tests of per-vertex shading normals and texture coordinates of mesh triangles (DESIGN.md §5e): the known answers of
tests/test_cpu_mesh_attributes.py through rtb_trace_rays and rtb_render, the CUDA path against the CPU restatement
(tests/feature_oracle.cpp) on the same Philox streams, adaptive rounds, light sampling, what smooth shading buys against an
analytic sphere, two GPUs, the bounds-checked build and rtb_app."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import mesh_scenes as ms
from conftest import ROOT
from helpers import psnr, tonemap
from feature_oracle import FeatureOracleScene
from test_cpu_light_sampling import mean_error_sigmas
from test_cpu_mesh_attributes import _check_hits
from test_gpu_adaptive import _dense_snapshots, _expect_per_pixel

pytestmark = pytest.mark.gpu

HIT_FIELDS = ("t", "object", "material", "p", "n", "front_face", "u", "v")


def _render(rtb, s, cam, W, H, spp, D, seed, **kw):
    r = rtb.Renderer(0); r.set_scene(s); r.set_camera(cam)
    r.reset_counters(); r.render(W, H, 0, spp, D, seed=seed, variance=True, **kw)
    a, a2 = r.download_accum(want_sum2=True)
    return a, a2, r.counters().rays


def _same_hits(got, want):
    for k in HIT_FIELDS:
        assert np.array_equal(got[k], want[k]), k


# ------------------------------------------------------------------------------------------------ known answers

@pytest.mark.parametrize("instanced", [False, True])
@pytest.mark.parametrize("flip", [False, True])
@pytest.mark.parametrize("normals,uvs", [(True, True), (True, False), (False, True)])
def test_triangle_known_answers_trace_rays(rtb, instanced, flip, normals, uvs):
    """rtb_trace_rays reports the interpolated shading normal and UVs: float64 within 1e-6, and the oracle's records bit for
    bit."""
    if flip and not normals:
        pytest.skip("flip negates normals")
    s = ms.triangle_scene(rtb, normals=normals, flip=flip, uvs=uvs, instanced=instanced)
    rays, ab, back = ms.triangle_rays(rtb, instanced=instanced)
    r = rtb.Renderer(0); r.set_scene(s)
    got = r.trace_rays(rays)
    _check_hits(got, rays, ab, back, normals, uvs, instanced)
    _same_hits(got, FeatureOracleScene(s.serialize()).trace(rays, rtb.HIT_DTYPE))


def test_canonical_uvs_reproduce_the_plain_mesh(rtb):
    """Canonical UVs on unshared faces: the GPU's accumulators equal the plain mesh's and the oracle's bit for bit."""
    (a, cam), (b, _) = ms.canonical_uv_scene(rtb, False), ms.canonical_uv_scene(rtb, True)
    W, H, S, D = 96, 64, 8, 12
    ga, ga2, ra = _render(rtb, a, cam, W, H, S, D, 5)
    gb, gb2, rb = _render(rtb, b, cam, W, H, S, D, 5)
    assert np.array_equal(ga, gb) and np.array_equal(ga2, gb2) and ra == rb
    ref, _, rays = FeatureOracleScene(b.serialize()).render(cam, W, H, 0, S, D, seed=5)
    assert np.array_equal(gb, ref) and rays == rb


def test_white_furnace_smooth_icosphere(rtb):
    """The oracle's furnace on the GPU: integer sums, at most spp, equal to the oracle's per pixel."""
    s, cam = ms.furnace_scene(rtb, smooth=True)
    spp = 32
    g, _, _ = _render(rtb, s, cam, 48, 48, spp, 20, 7)
    rgb = g[..., :3]
    assert np.all(rgb == np.round(rgb)) and np.all(rgb <= spp)
    ref, _, _ = FeatureOracleScene(s.serialize()).render(cam, 48, 48, 0, spp, 20, seed=7)
    assert np.array_equal(g, ref)


# ------------------------------------------------------------------------------------------------ parity with the oracle

@pytest.mark.parametrize("kind", list(ms.PARITY_KINDS) + ["binned_tail"])
def test_same_streams_as_the_oracle(rtb, kind, monkeypatch):
    """Path for path on the same Philox streams: at most 1e-4 of the pixels differ (a tie between two hits at one t may
    resolve differently), ray counts within 5e-6.  binned_tail: the glass and metal scene with every binned bounce forced
    and the fused tail kernel taking over early."""
    if kind == "binned_tail":
        monkeypatch.setenv("RTB_BIN_MASK", "116"); monkeypatch.setenv("RTB_TAIL_THRESHOLD", "40000")
    scene, cam = ms.parity_scene(rtb, "glass_metal" if kind == "binned_tail" else kind)
    W, H, S, D = 192, 128, 8, 30
    g, _, rays_g = _render(rtb, scene, cam, W, H, S, D, 1984)
    ref, _, rays = FeatureOracleScene(scene.serialize()).render(cam, W, H, 0, S, D, seed=1984)
    diff = np.abs(g[..., :3] - ref[..., :3]).max(axis=2)
    bad = float((diff > 1e-4 * np.maximum(np.abs(ref[..., :3]).max(axis=2), 1.0)).mean())
    print(f"{kind} {W}x{H}x{S}: {bad * 100:.4f} % of pixels differ, exact {np.array_equal(g, ref)}, rays gpu {rays_g} oracle {rays}, "
          f"PSNR {psnr(tonemap(g), tonemap(ref)):.1f} dB")
    assert bad <= 1e-4
    assert abs(int(rays_g) - int(rays)) <= max(5e-6 * rays, 4)


def test_adaptive_rounds_on_a_smooth_mesh(rtb):
    """Every pixel of an adaptive render holds the dense render's sums at its own count (the LIST x ATTR kernels)."""
    scene, cam = ms.parity_scene(rtb, "textured")
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
    print(f"cursors {cursors}, mean spp {a[..., 3].mean():.1f}")
    assert len(cursors) >= 3 and 0 < (a[..., 3] < cursors[-1]).mean()
    d = rtb.Renderer(0); d.set_scene(scene); d.set_camera(cam)
    _expect_per_pixel(_dense_snapshots(rtb, d, W, H, D, seed, cursors, (0, 0), spb), a, q, (0, 0), H)


def test_trace_rays_on_a_deep_gpu_lbvh(rtb):
    """rtb_trace_rays on a smooth, UV-mapped 1024 x 1024 height field under the GPU linear BVH, a tree deep enough for the
    64-entry stack: the oracle's hit records.  (Triangle hits bit for bit; on the glass ball the sphere (u, v) goes through
    acosf / atan2f, which the device and the host round differently in the last bit.)"""
    scene, cam = ms.height_field_scene(rtb, 1024, "textured")
    scene.set_world_bvh(rtb.WORLD_BVH_GPU_LBVH)
    r = rtb.Renderer(0); r.set_scene(scene)
    st = r.scene_stats()
    print("height field 1024 GPU LBVH:", st)
    assert st["builder"] == "gpu_lbvh" and st["depth"] > 30
    from helpers import camera_rays
    rays = camera_rays(rtb, cam, 160, 160)
    got = r.trace_rays(rays)
    want = FeatureOracleScene(scene.serialize()).trace(rays, rtb.HIT_DTYPE)
    assert (got["t"] < 1e30).mean() > 0.5
    tri = got["material"] == 0                                  # the mesh's material (the ball's is 1)
    assert tri.mean() > 0.3
    for k in ("t", "object", "material", "p", "n", "front_face"):
        assert np.array_equal(got[k], want[k]), k
    for k in ("u", "v"):
        assert np.array_equal(got[k][tri], want[k][tri]), k
        assert np.allclose(got[k][~tri], want[k][~tri], rtol=0, atol=1e-6), k


def test_light_sampling_on_a_smooth_mesh_is_unbiased(rtb):
    """Sampling the quad light changes the noise only: the images with and without it agree within 3 sigma per channel."""
    W, H, SPP, D = 48, 32, 1024, 12
    scene, cam = ms.parity_scene(rtb, "lights")
    a, a2, _ = _render(rtb, scene, cam, W, H, SPP, D, 202)
    scene.sample_lights([])
    b, b2, _ = _render(rtb, scene, cam, W, H, SPP, D, 101)
    for c, (bias, sigma) in enumerate(mean_error_sigmas(a, a2, b, b2, SPP)):
        print(f"channel {c}: error / sigma {bias / sigma:+.2f}")
        assert abs(bias) <= 3.0 * sigma + 1e-6, (c, bias, sigma)


# Measured on a B200 (1,000 W): RMS against the sphere 0.00268 smooth, 0.00624 flat, ratio 0.43 (sphere against itself on
# another seed: 0.00031, so the ratio is geometry, not noise).  The bar leaves 0.17 of margin.
SMOOTH_OVER_FLAT_MAX = 0.6


def test_smooth_icosphere_approaches_the_analytic_sphere(rtb):
    """A subdivision-3 icosphere with analytic vertex normals against rtb_add_sphere of the same radius, a mirror reflecting
    the sky gradient (the reflected direction, and so the colour, follows the normal), at equal spp on independent seeds:
    the smooth mesh's RMS difference from the sphere's image is a fraction of the flat mesh's."""
    W, H, SPP, D = 96, 96, 256, 4
    v, f = ms.icosphere(3)

    def scene(kind):
        s = rtb.Scene()
        mat = s.metal((0.9, 0.9, 0.9), 0.0)
        s.set_root(s.sphere((0, 0, 0), 1.0, mat) if kind == "sphere" else s.mesh(v, f, mat, normals=v if kind == "smooth" else None))
        return s
    cam = rtb.make_camera("pinhole", (0.0, 0.6, 3.2), (0, 0, 0), (0, 1, 0), 40.0, 1.0)
    img = {k: tonemap(_render(rtb, scene(kind), cam, W, H, SPP, D, seed)[0])
           for k, kind, seed in (("sphere", "sphere", 1), ("smooth", "smooth", 2), ("flat", "flat", 3), ("sphere2", "sphere", 4))}
    rms = {k: float(np.sqrt(((img[k] - img["sphere"]) ** 2).mean())) for k in ("smooth", "flat", "sphere2")}
    ratio = rms["smooth"] / rms["flat"]
    print(f"RMS against the analytic sphere: smooth {rms['smooth']:.5f} flat {rms['flat']:.5f} (noise floor, sphere vs sphere: "
          f"{rms['sphere2']:.5f}) ratio {ratio:.3f}")
    assert ratio <= SMOOTH_OVER_FLAT_MAX


def test_two_gpus_with_a_smooth_mesh(rtb):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    scene, cam = ms.parity_scene(rtb, "textured")
    W, H, D = 96, 96, 20
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, 5, D, seed=1984, variance=True); a0, q0 = r.download_accum(want_sum2=True)
    r.render(W, H, 5, 10, D, seed=1984, variance=True); a1, q1 = r.download_accum(want_sum2=True)
    m = rtb.MultiRenderer([0, 1], reduce=rtb.REDUCE_P2P)
    m.set_scene(scene); m.set_camera(cam)
    m.render(W, H, 0, 10, D, seed=1984, variance=True); m.synchronize()
    got, got2 = m.download_accum(want_sum2=True)
    assert np.array_equal(got, a0 + a1) and np.array_equal(got2, q0 + q1)


def test_debug_bounds_build_with_attributes(rtb):
    """librtb200_debug.so on every new scene, binning forced, dense and adaptive: no index out of range (the attribute
    index and record are checked under the "primitive" class)."""
    if not rtb.DEBUG_LIB_PATH.exists():
        pytest.skip("librtb200_debug.so not built")
    code = r'''
import importlib, json, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
rtb = importlib.import_module("ray-tracing-v06_b200")
import mesh_scenes as ms
r = rtb.Renderer(0); n = 0
scenes = [ms.parity_scene(rtb, k) for k in ms.PARITY_KINDS] + [ms.canonical_uv_scene(rtb, True), ms.furnace_scene(rtb)]
for s, cam in scenes:
    r.set_scene(s); r.set_camera(cam); n += 1
    r.render(72, 56, 0, 6, 30, seed=9, samples_per_batch=4, variance=True)
    r.render_adaptive(40, 40, 32, 8, tolerance=0.05, min_spp=4, seed=9)
    r.synchronize()
print("REPORT " + json.dumps(dict(r.debug_bounds_report(), scenes=n)))
''' % (str(ROOT), str(ROOT / "tests"))
    env = dict(os.environ, RTB_LIB=str(rtb.DEBUG_LIB_PATH), RTB_BIN_MASK="116")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    rep = json.loads([l for l in out.stdout.splitlines() if l.startswith("REPORT ")][-1][7:])
    print("bounds report with attributes:", rep)
    assert rep.pop("scenes") == len(ms.PARITY_KINDS) + 2
    assert rep.pop("rays_checked") > 10_000
    assert all(v == 0 for v in rep.values()), rep


def test_rtb_app_smooth_textured_obj(rtb, tmp_path):
    """rtb_app --obj ... --smooth --obj-texture ...: a picture in which the textured model shows the image's colours, and
    one that differs from the flat, untextured render."""
    v, f = ms.icosphere(2)
    uv = ms.sphere_uvs(v)
    text = "".join(f"v {x:.9g} {y:.9g} {z:.9g}\n" for x, y, z in v) + "".join(f"vt {a:.9g} {b:.9g}\n" for a, b in uv)
    text += "".join(f"f {a + 1}/{a + 1} {b + 1}/{b + 1} {c + 1}/{c + 1}\n" for a, b, c in f)
    (tmp_path / "ball.obj").write_text(text)
    img = np.zeros((8, 16, 3), np.uint8); img[..., 0] = 230; img[..., 2] = 20          # red
    (tmp_path / "red.ppm").write_bytes(b"P6\n16 8\n255\n" + img.tobytes())
    app = str(ROOT / "ray-tracing-v06_b200" / "rtb_app")
    base = [app, "--obj", str(tmp_path / "ball.obj"), "--width", "64", "--height", "48", "--spp", "16", "--depth", "8"]
    outs = {}
    for label, extra in (("flat", []), ("smooth", ["--smooth"]), ("textured", ["--smooth", "--obj-texture", str(tmp_path / "red.ppm")])):
        out = tmp_path / f"{label}.pfm"
        res = subprocess.run(base + extra + ["--out", str(out)], capture_output=True, text=True)
        assert res.returncode == 0, (label, res.stderr)
        data = out.read_bytes().split(b"\n", 3)
        Wp, Hp = map(int, data[1].split())
        outs[label] = np.frombuffer(data[3], "<f4").reshape(Hp, Wp, 3)
    assert not np.array_equal(outs["flat"], outs["smooth"])
    centre = outs["textured"][18:30, 26:38]
    assert (centre[..., 0] > 2 * centre[..., 2]).mean() > 0.8                      # the red skin shows where the model is
    assert not (outs["smooth"][18:30, 26:38, 0] > 2 * outs["smooth"][18:30, 26:38, 2]).any()
