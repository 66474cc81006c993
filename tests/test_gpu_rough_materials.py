"""GPU tests of the GGX microfacet materials (DESIGN.md §5f): directional albedo against the float64 integral of the BSDF
(tests/microfacet_reference.py), path for path against the CPU restatement (tests/rough_oracle.cpp) on every case of
tests/feature_scenes.py with rough objects added, the smooth limits and the white furnace, schedule invariance of the
ROUGH instantiations, checkpoints, two GPUs, rtb_app and the bounds-checked build."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import feature_scenes as fs
import microfacet_reference as mr
from conftest import ROOT
from helpers import psnr, tonemap
from rough_oracle import RoughOracleScene
from test_cpu_rough_materials import half_sky, mean_and_error, plane_scene
from test_gpu_schedules import SCHEDULES, schedule

pytestmark = pytest.mark.gpu

ALPHAS = (0.05, 0.2, 0.5, 1.0)
THETAS = (0.0, 45.0, 75.0)


def _render(rtb, scene, cam, W, H, spp, depth, seed, **kw):
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, spp, depth, seed=seed, variance=True, **kw)
    return r.download_accum(want_sum2=True)


def _albedo(rtb, scene, cam, seed=7):
    a, a2 = _render(rtb, scene, cam, 64, 64, 256, 2, seed)
    return mean_and_error(a, a2)


# ------------------------------------------------------------------------------------------------ 1. albedo vs the integral
@pytest.mark.parametrize("theta", THETAS)
@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("f0", [(1.0, 1.0, 1.0), (0.95, 0.64, 0.1)])
def test_rough_metal_albedo(rtb, f0, alpha, theta):
    s, cam = plane_scene(rtb, "metal", theta, alpha, f0=f0)
    m, e = _albedo(rtb, s, cam)
    want = np.array([mr.albedo(theta, alpha, "R", f0=c) for c in f0])
    print(f"F0 {f0} alpha {alpha} theta {theta}: {m} +- {e}, integral {want}")
    assert np.all(np.abs(m - want) <= 4 * e + 2e-5), (m, e, want)


@pytest.mark.parametrize("theta", THETAS)
@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("back", [False, True], ids=["eta1.5", "eta0.667"])
def test_rough_glass_albedo(rtb, back, alpha, theta):
    """White sky: E_R + E_T.  A map white above the horizon: E_R; below: E_T."""
    eta = 1 / 1.5 if back else 1.5
    R, T = mr.albedo(theta, alpha, "R", eta=eta), mr.albedo(theta, alpha, "T", eta=eta)
    for sky, want in ((None, R + T), (half_sky(36, 18), R), (half_sky(36, 18, below=True), T)):
        s, cam = plane_scene(rtb, "glass", theta, alpha, back=back, sky=sky)
        m, e = _albedo(rtb, s, cam)
        assert np.all(np.abs(m - want) <= 4 * e + 2e-5), (sky is None, m, e, want)


@pytest.mark.parametrize("white_rows,zmin", [(6, 0.8660254037844387), (12, 0.5)])   # elevation 60 / 30 degrees
@pytest.mark.parametrize("kind,alpha,theta", [("metal", 0.2, 45.0), ("metal", 0.5, 0.0), ("glass", 0.5, 45.0)])
def test_lobe_shape(rtb, kind, alpha, theta, white_rows, zmin):
    """A map white only above elevation beta: where the lobe puts its energy, not only how much."""
    s, cam = plane_scene(rtb, kind, theta, alpha, sky=half_sky(36, white_rows))
    m, e = _albedo(rtb, s, cam)
    kw = dict(f0=1.0) if kind == "metal" else dict(eta=1.5)
    want, err = mr.converged(theta, alpha, "R", zmin=zmin, n=48, **kw)
    print(f"{kind} alpha {alpha} theta {theta} beta row {white_rows}: {m} +- {e}, integral {want} (+- {err:.1e})")
    assert np.all(np.abs(m - want) <= 4 * e + err + 2e-5)


# ------------------------------------------------------------------------------------------------ 2. path for path
def rough_case(rtb, case):
    """The feature scene of a case with a rough metal sphere, a rough glass sphere, an instanced rough glass quad and a
    smooth (ATTR cases) or plain rough-metal icosphere added to its root list."""
    s, cam = fs.build(rtb, case)
    import mesh_scenes as ms
    root = s.num_objects() - 1
    rm, rg = s.rough_metal((0.95, 0.64, 0.54), 0.3), s.rough_dielectric(1.5, 0.15, (0.95, 0.95, 1.0))
    v, f = ms.icosphere(2)
    ball = s.mesh(v * np.float32(0.35), f, s.rough_metal((0.8, 0.8, 0.85), 0.6), normals=v if case.attr else None)
    objs = [root, s.sphere((0.2, -0.65, 1.6), 0.35, rm), s.sphere((-0.9, -0.7, 1.9), 0.3, rg),
            s.translate(s.rotate_y(s.quad((-0.4, -1.0, 0.0), (0.8, 0, 0), (0, 0.9, 0), rg), 30.0), (0.6, 0.0, 1.0)),
            s.translate(s.rotate_y(ball, 15.0), (-1.2, -0.4, 0.2))]
    s.set_root(s.list(objs))
    return s, cam


CASES = [pytest.param(c, id=c.id) for c in fs.CASES]
ROUGH_SHADE = {k + (True,) for k in fs.ALL_SHADE}
ROUGH_TAIL = {k + (True,) for k in fs.ALL_TAIL}


def test_rough_coverage():
    """Every case has rough materials, so the ROUGH flag is set in all of them: with fs.check_coverage, the cases select
    every ROUGH shade (16) and tail (64) instantiation."""
    t = fs.check_coverage()
    shade = {k + (True,) for k in t["shade"]}
    tail = {k + (True,) for k in t["tail"]}
    assert shade == ROUGH_SHADE and len(shade) == 16
    assert tail == ROUGH_TAIL and len(tail) == 64


@pytest.mark.parametrize("case", CASES)
def test_same_streams_as_the_rough_oracle(rtb, monkeypatch, case):
    """Schedules B (every bounce in the wavefront), A (the tail kernel) and D (every bounce binned) against the CPU oracle on
    the same Philox streams: at most 1e-4 of the pixels differ, ray counts within 5e-6."""
    scene, cam = rough_case(rtb, case)
    assert scene.serialize()[4] == 5
    W, H, S, D = 128, 96, 6, 24
    ref, _, rays = RoughOracleScene(scene.serialize()).render(cam, W, H, 0, S, D, seed=1984)
    for name in ("B", "A", "D"):
        with schedule(monkeypatch, name):
            r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam); r.reset_counters()
            r.render(W, H, 0, S, D, seed=1984)
            g = r.download_accum(); rays_g = int(r.counters().rays)
        diff = np.abs(g[..., :3] - ref[..., :3]).max(axis=2)
        bad = float((diff > 1e-4 * np.maximum(np.abs(ref[..., :3]).max(axis=2), 1.0)).mean())
        print(f"{case.id} schedule {name}: {bad * 100:.4f} % of pixels differ, rays gpu {rays_g} oracle {rays}")
        assert bad <= 1e-4
        assert abs(rays_g - int(rays)) <= max(5e-6 * rays, 4)


# ------------------------------------------------------------------------------------------------ 3. limits and energy
def _limit_scene(rtb, kind, rough):
    s = rtb.Scene()
    ground = s.lambertian(tex=s.checker(0.5, s.solid((0.2, 0.3, 0.1)), s.solid((0.9, 0.9, 0.9))))
    if kind == "metal":
        m = s.rough_metal((1, 1, 1), 0.001) if rough else s.metal((1, 1, 1), 0.0)
    else:
        m = s.rough_dielectric(1.5, 0.001) if rough else s.dielectric(1.5)
    s.set_root(s.list([s.quad((-8, -1, -8), (16, 0, 0), (0, 0, 16), ground), s.sphere((0, 0, 0), 1.0, m),
                       s.sphere((1.8, -0.5, -1.0), 0.5, m)]))
    return s, rtb.make_camera("pinhole", (0.5, 1.2, 4.0), (0, -0.2, 0), (0, 1, 0), 40.0, 1.5)


@pytest.mark.parametrize("kind", ["metal", "glass"])
def test_small_alpha_tends_to_the_smooth_material(rtb, kind):
    W, H, SPP, D = 72, 48, 1024, 16
    a, a2 = _render(rtb, *_limit_scene(rtb, kind, True), W, H, SPP, D, 101)
    b, b2 = _render(rtb, *_limit_scene(rtb, kind, False), W, H, SPP, D, 202)
    c, _ = _render(rtb, *_limit_scene(rtb, kind, False), W, H, SPP, D, 303)
    ma, ea = mean_and_error(a, a2); mb, eb = mean_and_error(b, b2)
    assert np.all(np.abs(ma - mb) <= 3 * np.hypot(ea, eb)), (ma, mb, ea, eb)
    p_rough, p_floor = psnr(tonemap(a), tonemap(b)), psnr(tonemap(c), tonemap(b))
    print(f"{kind}: PSNR rough vs smooth {p_rough:.2f} dB, smooth vs smooth {p_floor:.2f} dB")
    assert p_rough >= p_floor - 0.5


def test_white_furnace(rtb):
    """Uniform white sky, white rough spheres of both kinds at alpha = 1: no pixel gains energy, and the metal loses some."""
    s = rtb.Scene()
    s.set_root(s.list([s.sphere((-1.1, 0, 0), 1.0, s.rough_metal((1, 1, 1), 1.0)), s.sphere((1.1, 0, 0), 1.0, s.rough_dielectric(1.5, 1.0))]))
    s.set_background(rtb.BG_CONSTANT, (1, 1, 1))
    cam = rtb.make_camera("pinhole", (0, 0, 6), (0, 0, 0), (0, 1, 0), 50.0, 2.0)
    W, H, SPP = 96, 48, 256
    a, _ = _render(rtb, s, cam, W, H, SPP, 64, 5)
    assert np.all(a[..., :3] <= SPP * (1 + 1e-6))
    # the metal sphere (x = -1.1: columns 30-47 of 96, rows 15-32 of 48) around its centre: strictly below
    metal = a[21:27, 35:42, :3]
    assert np.all(metal < SPP * 0.999), metal.min()


# ------------------------------------------------------------------------------------------------ 4. schedules
W_S, H_S, SPB, D_S = 640, 400, 9, 16


@pytest.mark.parametrize("case", CASES)
def test_dense_and_adaptive_schedules_are_bit_identical(rtb, monkeypatch, case):
    scene, cam = rough_case(rtb, case)
    dense, adapt = {}, {}
    for name in SCHEDULES:
        with schedule(monkeypatch, name):
            r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam); r.reset_counters()
            r.render(W_S, H_S, 0, 3 * SPB, D_S, seed=29, variance=True, samples_per_batch=SPB)
            dense[name] = r.download_accum(want_sum2=True) + (int(r.counters().rays),)
            if name in "ABCD":
                r2 = rtb.Renderer(0); r2.set_scene(scene); r2.set_camera(cam)
                st = r2.render_adaptive(W_S, H_S, 256, D_S, tolerance=0.02, min_spp=SPB, max_rounds=3, seed=31, samples_per_batch=SPB)
                adapt[name] = r2.download_accum(want_sum2=True) + (st, int(r2.counters().rays))
                del r2
            del r
    for name, g in dense.items():
        assert all(np.array_equal(x, y) for x, y in zip(g[:2], dense["A"][:2])) and g[2] == dense["A"][2], f"dense schedule {name}"
    assert adapt["A"][2]["rounds"] == 3
    for name, g in adapt.items():
        assert all(np.array_equal(x, y) for x, y in zip(g[:2], adapt["A"][:2])) and g[2:] == adapt["A"][2:], f"adaptive schedule {name}"


# ------------------------------------------------------------------------------------------------ 5. carried features
def test_checkpoint_resume_is_bit_exact(rtb, tmp_path):
    scene, cam = rough_case(rtb, fs.Case("pre", "shallow", True, "sampled", True))
    W, H, D = 96, 80, 24
    a = rtb.Renderer(0); a.set_scene(scene); a.set_camera(cam)
    a.render(W, H, 0, 8, D, seed=11, variance=True, samples_per_batch=1)
    want, want2 = a.download_accum(want_sum2=True)
    a.render(W, H, 0, 3, D, seed=11, variance=True, samples_per_batch=1)
    ck = tmp_path / "rough.rtba"
    a.save_accum(ck)
    b = rtb.Renderer(0); b.set_scene(scene); b.set_camera(cam)
    assert b.load_accum(ck) == 3
    b.render(W, H, 3, 8, D, seed=11, clear=False, variance=True, samples_per_batch=1)
    got, got2 = b.download_accum(want_sum2=True)
    assert np.array_equal(got, want) and np.array_equal(got2, want2)


def test_two_gpus_with_rough_materials(rtb):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    scene, cam = rough_case(rtb, fs.Case("none", "shallow", False, "unsampled", True))
    W, H, D = 96, 96, 20
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, 5, D, seed=1984, variance=True); a0, q0 = r.download_accum(want_sum2=True)
    r.render(W, H, 5, 10, D, seed=1984, variance=True); a1, q1 = r.download_accum(want_sum2=True)
    m = rtb.MultiRenderer([0, 1], reduce=rtb.REDUCE_P2P)
    m.set_scene(scene); m.set_camera(cam)
    m.render(W, H, 0, 10, D, seed=1984, variance=True); m.synchronize()
    got, got2 = m.download_accum(want_sum2=True)
    assert np.array_equal(got, a0 + a1) and np.array_equal(got2, q0 + q1)


def test_rtb_app_rough_obj(rtb, tmp_path):
    import mesh_scenes as ms
    v, f = ms.icosphere(2)
    text = "".join(f"v {x:.9g} {y:.9g} {z:.9g}\n" for x, y, z in v) + "".join(f"f {a + 1} {b + 1} {c + 1}\n" for a, b, c in f)
    (tmp_path / "ball.obj").write_text(text)
    app = str(ROOT / "ray-tracing-v06_b200" / "rtb_app")
    outs = {}
    for label, extra in (("clay", []), ("metal", ["--obj-material", "rough-metal", "--alpha", "0.3"]), ("glass", ["--obj-material", "rough-glass"])):
        out = tmp_path / f"{label}.pfm"
        res = subprocess.run([app, "--obj", str(tmp_path / "ball.obj"), "--width", "48", "--height", "32", "--spp", "8", "--depth", "8",
                              "--out", str(out)] + extra, capture_output=True, text=True)
        assert res.returncode == 0, (label, res.stderr)
        data = out.read_bytes().split(b"\n", 3)
        outs[label] = np.frombuffer(data[3], "<f4")
        assert np.all(np.isfinite(outs[label]))
    assert not np.array_equal(outs["clay"], outs["metal"]) and not np.array_equal(outs["metal"], outs["glass"])


def test_debug_bounds_build_with_rough_materials(rtb):
    if not rtb.DEBUG_LIB_PATH.exists():
        pytest.skip("librtb200_debug.so not built")
    code = r'''
import importlib, json, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
rtb = importlib.import_module("ray-tracing-v06_b200")
import feature_scenes as fs
from test_gpu_rough_materials import rough_case, plane_scene
from test_cpu_rough_materials import half_sky
r = rtb.Renderer(0); n = 0
scenes = [rough_case(rtb, c) for c in fs.CASES[::3]] + [plane_scene(rtb, "glass", 45.0, 0.3, sky=half_sky(36, 18))]
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
    print("bounds report with rough materials:", rep)
    assert rep.pop("scenes") == len(fs.CASES[::3]) + 1
    assert rep.pop("rays_checked") > 10_000
    assert all(v == 0 for v in rep.values()), rep
