"""GPU tests of the Book-1 / Book-2 materials, camera samplers and media against the float64 references of
tests/scatter_reference.py, which are derived from DESIGN.md §5, §5d, §6 and the books, not from the kernels: a slip that
the kernels and the CPU oracle share (both restate the same Philox-mode spec) passes every same-stream test, but not
these.  Every measured quantity takes at least 2^20 paths and must lie within 4 standard errors (from the sums of
squares) plus the quadrature bound plus 2e-5 of its reference.  The cameras look through a periscope of two lossless
mirrors, so the measured interaction happens at bounce 2, and every case is rendered under schedule B (no tail: the
traverse and shade kernels run every bounce) and schedule C (the tail kernel takes every batch over from bounce 2), so
that the shade and the tail instantiations are both measured; each render checks from the launch profile that the tail
ran under C and not under B.  The exception is the 90-degree metal field, which no periscope passes: it is measured at
bounce 0, by the shade kernel only, and so are the metal lobes of fuzz 1 and 1.5 (see metal_periscope in the scene
file).  The scenes are built in tests/test_cpu_scatter_distributions.py, where the same
references are checked against the CPU oracle."""
import math

import numpy as np
import pytest

import feature_scenes as fs
import scatter_reference as sr
import test_cpu_scatter_distributions as sd
from test_cpu_rough_materials import mean_and_error
from test_gpu_schedules import schedule

pytestmark = pytest.mark.gpu

SCHEDS = ["B", "C"]         # test_gpu_schedules.SCHEDULES: no tail / the tail kernel from bounce 2
PATHS = 1 << 20


def render(rtb, monkeypatch, sched, scene, cam, W, H, spp, depth=sd.DEPTH, seed=11):
    with schedule(monkeypatch, sched):
        r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
        r.set_profiling(True)
        r.render(W, H, 0, spp, depth, seed=seed, variance=True)
        a, a2 = r.download_accum(want_sum2=True)
        tails = int(r.profile().tail_launches); r.set_profiling(False)
        del r
    assert (tails > 0) == (sched == "C" and depth > 2), (sched, depth, tails)
    return a, a2


def image_mean(rtb, monkeypatch, sched, scene, cam, depth=sd.DEPTH, seed=11):
    """Mean and standard error over a 64 x 64 x 256 render (2^20 paths), per channel."""
    return mean_and_error(*render(rtb, monkeypatch, sched, scene, cam, 64, 64, 256, depth=depth, seed=seed))


def pixel_mean(a, a2):
    """Per pixel and channel: mean and standard error."""
    n = a[..., 3:4].astype(np.float64)
    m = a[..., :3] / n
    return m, np.sqrt(np.maximum(a2[..., :3] / n - m * m, 0.0) / n)


def check(m, e, want, bound=0.0, what=""):
    m, e, want = np.asarray(m), np.asarray(e), np.asarray(want)
    print(f"{what}: {m} +- {e}, reference {want} (+- {np.max(bound):.1e})")
    assert np.all(np.abs(m - want) <= 4 * e + bound + 2e-5), (what, m, e, want)


# ------------------------------------------------------------------------------------------------ Lambertian
@pytest.mark.parametrize("sched", SCHEDS)
@pytest.mark.parametrize("mix", ["plain", "lamp", "env_sampled"])
@pytest.mark.parametrize("target", ["front", "back", "sphere"])
def test_lambertian_lobe(rtb, monkeypatch, target, mix, sched):
    """The cosine lobe per texel band and on a checkerboard of the hemisphere.  With a sampled lamp (which emits exactly
    the texels it hides) or with the map sampled, the LIGHTS / ENV mixture draws other directions and reweights them:
    the expectation must not move."""
    sky = sd.lambert_map()
    scene, cam = sd.lambert_scene(rtb, target, sky, lamp=(mix == "lamp"), sample_env=(mix == "env_sampled"))
    m, e = image_mean(rtb, monkeypatch, sched, scene, cam)
    check(m, e, sr.expected(sr.lambert_masses(sd.LW, sd.LH), sky), what=f"lambertian {target} {mix} {sched}")


# ------------------------------------------------------------------------------------------------ metal
METAL = [(f, sched) for f in (0.1, 0.5) for sched in SCHEDS] + [(1.0, "B"), (1.5, "B")]


@pytest.mark.parametrize("fuzz,sched", METAL)
def test_metal_fuzz_lobe(rtb, monkeypatch, fuzz, sched):
    """Normal incidence, |d| = 1: 1 - absorbed, and the mass in two polar bands (fuzz is not clamped, so 1.5 is valid).
    Fuzz 0.1 and 0.5 through the periscope under both schedules; fuzz 1 and 1.5, whose lobes reach the horizon, straight
    from the camera at depth 2 (test_cpu_scatter_distributions.metal_periscope says why), by the shade kernel."""
    sky = sd.metal_map()
    scene, cam = sd.metal_scene(rtb, fuzz, sky)
    d = np.array(cam.w, np.float64)
    m, e = image_mean(rtb, monkeypatch, sched, scene, cam, depth=sd.metal_depth(fuzz))
    check(m, e, sr.expected(sr.metal_masses(sd.MW, sd.MH, fuzz, float(np.linalg.norm(d))), sky), what=f"metal fuzz {fuzz} {sched}")


@pytest.mark.parametrize("sched", ["B"])
def test_metal_wide_field(rtb, monkeypatch, sched):
    """A 90-degree field, fuzz 1: per pixel, 1 - absorbed = 1 - clip((1 - |d . n|) / 2, 0, 1) over the pixel filter, where
    d is the pixel's un-normalised camera direction.  Fuzz added to a normalised reflection would absorb more where
    |d| > 1, toward the corners.  Depth 2, the plane at bounce 0: the tail kernel cannot run, so one schedule."""
    W = H = 12
    scene, cam = sd.metal_scene(rtb, 1.0, wide=True)
    m, e = pixel_mean(*render(rtb, monkeypatch, sched, scene, cam, W, H, PATHS, depth=2))
    want, err = sd.metal_wide_reference(cam, W, H, 1.0)
    worst = np.abs(m[..., 0] - want) / (4 * e[..., 0] + err + 2e-5)
    print(f"wide-field metal {sched}: reference {want.min():.4f}-{want.max():.4f}, worst |diff| / tolerance {worst.max():.2f}")
    assert np.all(np.abs(m - want[..., None]) <= 4 * e + err[..., None] + 2e-5), worst


# ------------------------------------------------------------------------------------------------ dielectric
DIELECTRIC = [(th, False) for th in (0.0, 30.0, 60.0, 85.0)] + [(th, True) for th in (0.0, 30.0, 41.0, 42.0, 60.0, 85.0)]


@pytest.mark.parametrize("sched", SCHEDS)
@pytest.mark.parametrize("theta,back", DIELECTRIC, ids=[f"{'back' if b else 'front'}{t:g}" for t, b in DIELECTRIC])
def test_dielectric_split_and_directions(rtb, monkeypatch, theta, back, sched):
    """eta = 1.5: R (upper half-map) and T (lower half-map) from Schlick, 1 past the 41.81-degree critical angle of the
    back face; then the one-degree rows of the mirror and the Snell directions hold R and T, and no other row holds
    anything."""
    for sky, want in sd.dielectric_maps(math.radians(theta), back):
        scene, cam = sd.dielectric_scene(rtb, theta, back, sky)
        m, e = image_mean(rtb, monkeypatch, sched, scene, cam, depth=sd.DEPTH_RETRO)
        check(m, e, want, what=f"dielectric {'back' if back else 'front'} {theta} map {sky.shape[0]} rows {sched}")


# ------------------------------------------------------------------------------------------------ isotropic media
@pytest.mark.parametrize("sched", SCHEDS)
@pytest.mark.parametrize("sigma", [0.1, 1.0, 3.0])
@pytest.mark.parametrize("b", [0.0, 0.5, 0.9])
def test_isotropic_medium_sphere(rtb, monkeypatch, b, sigma, sched):
    """R = 1, the medium at bounce 2 and depth 4 (one scatter, as at depth 2 without the periscope): transmission plus one isotropic scatter that escapes (free flight, phase function, truncation)."""
    want, err = sr.medium_pixel(1.0, sigma, sd.MEDIUM_ALBEDO, b)
    m, e = image_mean(rtb, monkeypatch, sched, *sd.medium_scene(rtb, 1.0, sigma, b))
    check(m, e, [want] * 3, err, what=f"medium b {b} sigma {sigma} {sched}")


@pytest.mark.parametrize("sched", SCHEDS)
def test_media_beyond_the_pre_list(rtb, monkeypatch, sched):
    """Ten media: number 5 is in the pre-test list of the eight largest and draws from stream 17; number 9 is a BVH leaf
    (the MEDIA = 2 traverse and tail) and draws from stream 18."""
    for target in (5, 9):
        R = 1.0 + 0.01 * (9 - target)
        scene, cam = sd.medium_scene(rtb, R, 1.0, 0.5, others=9, target_index=target)
        info = fs.scene_features(scene.serialize())
        assert info["n_media"] == 10 and info["n_media"] > fs.PRE_LIST_MAX
        radii = sorted((1.0 + 0.01 * (9 - k) if k != target else R, k) for k in range(10))
        pre = {k for _, k in radii[-fs.PRE_LIST_MAX:]}
        assert (target in pre) == (target == 5) and len({r for r, _ in radii}) == 10
        want, err = sr.medium_pixel(R, 1.0, sd.MEDIUM_ALBEDO, 0.5)
        m, e = image_mean(rtb, monkeypatch, sched, scene, cam)
        check(m, e, [want] * 3, err, what=f"medium {target} of 10 {sched}")


@pytest.mark.parametrize("sched", SCHEDS)
def test_medium_with_a_sampled_light(rtb, monkeypatch, sched):
    """The isotropic light mixture: a sampled lamp emitting the sky's white leaves the expectation where it was."""
    scene, cam = sd.medium_scene(rtb, 1.0, 1.0, 0.5, lamp=True)
    assert fs.scene_features(scene.serialize())["n_lights"] == 1
    want, err = sr.medium_pixel(1.0, 1.0, sd.MEDIUM_ALBEDO, 0.5)
    m, e = image_mean(rtb, monkeypatch, sched, scene, cam)
    check(m, e, [want] * 3, err, what=f"medium with lamp {sched}")


# ------------------------------------------------------------------------------------------------ camera samplers
EDGE_OFFSETS = [round(-0.6 + 0.1 * k, 1) for k in range(13)]


def _edge_check(rtb, monkeypatch, sched, scene, cam, geom, what):
    m, e = pixel_mean(*render(rtb, monkeypatch, sched, scene, cam, sd.EDGE_W, sd.EDGE_H, PATHS))
    want, err = sd.edge_reference(cam, geom)
    print(f"{what}: {m[..., 0].ravel()} reference {want.ravel()}")
    assert np.all(np.abs(m[..., 0] - want) <= 4 * e[..., 0] + err + 2e-5), (what, m[..., 0], e[..., 0], want)


@pytest.mark.parametrize("sched", SCHEDS)
@pytest.mark.parametrize("alpha", [0.0, 30.0])
def test_pixel_filter_disc(rtb, monkeypatch, alpha, sched):
    """An emitting half-plane whose edge (horizontal or tilted 30 degrees) is moved across the pixels in steps of 0.1
    pixel: each pixel's lit fraction is the circular segment of a disc of radius 1/2 pixel."""
    for off in EDGE_OFFSETS:
        _edge_check(rtb, monkeypatch, sched, *sd.edge_scene(rtb, alpha, off), what=f"edge {alpha} offset {off} {sched}")


@pytest.mark.parametrize("sched", SCHEDS)
@pytest.mark.parametrize("ratio", [1.0, 0.8, 1.5])
def test_defocus_lens_disc(rtb, monkeypatch, ratio, sched):
    """The edge at distance D with the lens focused at F = D / ratio: the jitter (radius 1/2 pixel x D / F) and the lens
    (radius lens_radius |1 - D / F|, 0.8 pixel here) are independent discs, so the lit fraction is their convolution;
    at D = F it is the pixel filter's."""
    for off in (-0.9, -0.5, -0.2, 0.0, 0.3, 0.7):
        s, cam, geom = sd.edge_scene(rtb, 0.0, off, kind="defocus", focus_ratio=ratio)
        if ratio == 1.0:
            assert np.allclose(sd.edge_reference(cam, geom)[0], sd.edge_reference(*sd.edge_scene(rtb, 0.0, off)[1:])[0], atol=1e-6)
        _edge_check(rtb, monkeypatch, sched, s, cam, geom, what=f"defocus D/F {ratio} offset {off} {sched}")


@pytest.mark.parametrize("sched", SCHEDS)
@pytest.mark.parametrize("shutter", [(0.2, 0.7), (0.0, 1.0)], ids=["shutter0.2-0.7", "shutter0-1"])
@pytest.mark.parametrize("path", [0, 1])
def test_motion_blur_shutter(rtb, monkeypatch, path, shutter, sched):
    """A moving emitter crossing the view axis: the hit fraction is the share of the raw shutter [t0, t1] during which the
    centre mix(c0, c1, time) is within R of the ray."""
    scene, cam = sd.motion_scene(rtb, *sd.MOTION_PATHS[path], *shutter)
    m, e = image_mean(rtb, monkeypatch, sched, scene, cam)
    check(m, e, [sd.motion_reference(cam, *sd.MOTION_PATHS[path])] * 3, what=f"motion path {path} shutter {shutter} {sched}")
