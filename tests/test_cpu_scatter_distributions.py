"""The float64 references of tests/scatter_reference.py - cosine lobe, fuzzy metal, Schlick dielectric, isotropic medium
sphere, pixel filter, defocus and motion blur - checked on their own and against the CPU restatement of the Philox-mode
spec (tests/feature_oracle.cpp) on the scenes that tests/test_gpu_scatter_distributions.py renders on the GPU.  Nothing
here needs a GPU.  The scene builders below are shared with the GPU file."""
import math

import numpy as np
import pytest

import scatter_reference as sr
from feature_oracle import FeatureOracleScene
from test_cpu_rough_materials import mean_and_error

NARROW = 0.05           # degrees: the field of the single-direction scenes (every pixel sees the same incidence)


# ------------------------------------------------------------------------------------------------ detector masks
def row_mask(H: int, W: int, rows) -> np.ndarray:
    m = np.zeros((H, W), np.float32)
    m[list(rows)] = 1.0
    return m


def stack(*channels) -> np.ndarray:
    """An [H, W, 3] map from three [H, W] masks."""
    return np.ascontiguousarray(np.stack(channels, -1), np.float32)


LW, LH = 16, 18         # Lambertian detector: 10-degree rows, 22.5-degree columns


def lambert_map() -> np.ndarray:
    """R: polar 0-30 degrees from +y; G: 30-60; B: a checkerboard of the upper hemisphere (azimuth and elevation)."""
    j, i = np.mgrid[0:LH, 0:LW]
    checker = ((i + j) % 2 == 0) & (j < LH // 2)
    return stack(row_mask(LH, LW, range(0, 3)), row_mask(LH, LW, range(3, 6)), checker.astype(np.float32))


MW, MH = 8, 36          # metal detector: 5-degree rows


def metal_map() -> np.ndarray:
    """R: the upper hemisphere (1 - absorbed); G: polar 0-10 degrees; B: 10-25 degrees.  No band edge lies on the rim of
    a fuzz cone (asin(fuzz): 5.7 and 30 degrees), where the density has an integrable singularity and the pixel jitter's
    tilt of the cone would move mass across the edge."""
    return stack(row_mask(MH, MW, range(0, MH // 2)), row_mask(MH, MW, range(0, 2)), row_mask(MH, MW, range(2, 5)))


# ------------------------------------------------------------------------------------------------ periscope
# Every scene but the wide-field metal one is seen through two parallel white fuzz-0 metal mirrors, so that the measured
# interaction happens at bounce 2, where a schedule with the tail kernel (tail from bounce 2) hands the batch to it.
PERISCOPE_L, PERISCOPE_E = 0.3, 0.2
DEPTH = 4           # mirrors at bounces 0 and 1, the measured interaction at bounce 2, its scattered ray at bounce 3
DEPTH_RETRO = 6     # ... and bounces 3-5 for a ray scattered straight back through the periscope (metal, dielectric)
RETRO_FOV = 0.002   # degrees: the field of those scenes.  A ray reflected near the way it came deviates from the incoming
                    # line by twice the jitter's angle; at this field it stays well inside both mirrors on the way back


def _unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v)


def periscope_camera(rtb, s, objs, kind, lookfrom, lookat, up, *args, size=0.004, **kw):
    """make_camera(kind, lookfrom, lookat, up, ...) moved by L (a + p) (a: the view axis, p: the camera's u axis) and seen
    through two parallel mirrors appended to objs: the first e ahead of the moved camera, with normal (a + p) / sqrt 2,
    turns the rays to -p; the second, on the original line of sight L + e ahead of lookfrom, turns them back.  Two
    reflections in parallel planes are a translation, here by -L (a + p): every ray, of any direction and lens offset,
    leaves the second mirror on the line, with the direction and |d|, of the camera at lookfrom (to float32 rounding),
    and keeps its time; albedo 1 and fuzz 0 lose nothing.  size: the mirrors' side, small enough that a scattered ray
    meets them with a probability far below the tolerances."""
    cam = rtb.make_camera(kind, lookfrom, lookat, up, *args, **kw)
    C, a, p = np.asarray(lookfrom, np.float64), _unit(np.subtract(lookat, lookfrom)), _unit(cam.u)
    q, tv = np.cross(a, p), (a - p) / math.sqrt(2.0)
    shift = PERISCOPE_L * (a + p)
    mirror = s.metal((1.0, 1.0, 1.0), 0.0)
    for M in (C + shift + PERISCOPE_E * a, C + (PERISCOPE_L + PERISCOPE_E) * a):
        objs.append(s.quad(tuple(M - 0.5 * size * (q + tv)), tuple(size * q), tuple(size * tv), mirror))
    return rtb.make_camera(kind, tuple(C + shift), tuple(np.asarray(lookat, np.float64) + shift), up, *args, **kw)


def virtual_origin(cam) -> np.ndarray:
    """The position of the camera whose rays a periscope camera reproduces."""
    return np.array(cam.o, np.float64) - PERISCOPE_L * (_unit(cam.w) + _unit(cam.u))


# ------------------------------------------------------------------------------------------------ scenes
def _plane(s, mat, normal_down=False):
    """A 2000 x 2000 quad in y = 0 with normal +y (or -y)."""
    u, v = ((2000, 0, 0), (0, 0, 2000)) if normal_down else ((0, 0, 2000), (2000, 0, 0))
    return s.quad((-1000, 0, -1000), u, v, mat)


def _incident_camera(rtb, s, objs, theta_deg, dist=10.0, fov=NARROW):
    th = math.radians(theta_deg)
    up = (0, 0, 1) if theta_deg == 0 else (0, 1, 0)
    return periscope_camera(rtb, s, objs, "pinhole", (dist * math.sin(th), dist * math.cos(th), 0.0), (0, 0, 0), up, fov, 1.0)


LAMP_POLAR, LAMP_U, LAMP_DIST, LAMP_SIZE = math.radians(45.0), 0.1, 20.0, 1.0


def lamp_corners():
    c = LAMP_DIST * sr.direction(LAMP_POLAR, LAMP_U)
    a = np.cross(c, (0.0, 1.0, 0.0)); a /= np.linalg.norm(a)
    b = np.cross(c, a); b /= np.linalg.norm(b)
    Q = c - 0.5 * LAMP_SIZE * (a + b)
    return Q, LAMP_SIZE * a, LAMP_SIZE * b


def lambert_scene(rtb, target: str, sky: np.ndarray, lamp: bool = False, sample_env: bool = False):
    """A white Lambertian quad seen on its front ("front") or back ("back") face at 45 degrees, or the top of a white
    Lambertian sphere seen from straight above ("sphere"); the shading normal is +y in all three (quads face the ray).
    lamp: a small sampled quad light in the sky, emitting exactly the map texels it covers, so the expectation is the
    map's; sample_env: the map is importance-sampled in the light mixture."""
    s = rtb.Scene()
    white = s.lambertian((1.0, 1.0, 1.0))
    if target == "sphere":
        objs = [s.sphere((0.0, -1.0, 0.0), 1.0, white)]
        cam = _incident_camera(rtb, s, objs, 0.0)
    else:
        objs = [_plane(s, white, normal_down=(target == "back"))]
        cam = _incident_camera(rtb, s, objs, 45.0)
    if lamp:
        Q, u, v = lamp_corners()
        corners = np.array([Q, Q + u, Q + v, Q + u + v, Q + 0.5 * (u + v)])
        ci, cj = sr.texel_of(corners, sky.shape[1], sky.shape[0])
        assert len(set(ci)) == 1 and len(set(cj)) == 1, "the lamp must lie inside one texel"
        lamp_id = s.quad(tuple(Q), tuple(u), tuple(v), s.diffuse_light(s.solid(tuple(float(x) for x in sky[cj[0], ci[0]]))))
        objs.append(lamp_id)
    s.set_root(s.list(objs))
    if lamp:
        s.sample_lights([lamp_id])
    s.set_environment(sky, sample=sample_env)
    return s, cam


def metal_scene(rtb, fuzz: float, sky=None, wide=False):
    """A white metal quad with the given fuzz.  Narrow: seen from straight above (reflect(d, n) = +y, |d| = 1 to 1e-7)
    with a RETRO_FOV field, measured through the map; through the periscope at DEPTH_RETRO when metal_periscope(fuzz),
    else directly at depth 2.  Wide: a 90-degree camera 3 units up, tilted 30 degrees, under a white sky, so that |d| and
    d . n vary from pixel to pixel; no periscope passes a 90-degree field, so it is rendered at depth 2, the plane at
    bounce 0."""
    s = rtb.Scene()
    objs = [_plane(s, s.metal((1.0, 1.0, 1.0), fuzz))]
    if wide:
        s.set_root(objs[0])
        s.set_background(rtb.BG_CONSTANT, (1.0, 1.0, 1.0))
        return s, rtb.make_camera("pinhole", (0.0, 3.0, 0.0), (3.0 * math.tan(math.radians(30.0)), 0.0, 0.0), (0, 1, 0), 90.0, 1.0)
    if metal_periscope(fuzz):
        cam = _incident_camera(rtb, s, objs, 0.0, fov=RETRO_FOV)
    else:
        cam = rtb.make_camera("pinhole", (0.0, 10.0, 0.0), (0, 0, 0), (0, 0, 1), RETRO_FOV, 1.0)
    s.set_root(s.list(objs))
    s.set_environment(sky)
    return s, cam


def metal_periscope(fuzz: float) -> bool:
    """Whether the narrow metal scene is seen through the periscope.  Not for fuzz >= |d| = 1: there dir = reflect(d, n) +
    fuzz s reaches the horizon with a length near 0, so the next ray's origin p + 0.001 dir (§6) lies within float32
    rounding of the hit point.  Straight from the camera the hit distance (10) and so the hit point are exact; behind the
    mirrors the last leg's distance is not, the point lands up to half an ulp of it (5e-7) below the plane on half the
    paths, and every scatter with 0.001 dir . n below that re-hits the plane from behind: about 2e-4 of the paths at
    fuzz 1, an effect of the book's offset that the reference does not model.  Fuzz 0.1 and 0.5 keep dir . n >= 0.5."""
    return fuzz < 1.0


def metal_depth(fuzz: float) -> int:
    return DEPTH_RETRO if metal_periscope(fuzz) else 2


def metal_wide_reference(cam, W, H, fuzz, n=12):
    """Per pixel: 1 - absorbed fraction averaged over the pixel filter (a disc of radius 1/2 pixel), from each jittered
    camera direction d = w + s u + t v; polar Gauss-Legendre over the disc, (value [H, W], error bound)."""
    u, v, w = (np.array(x, np.float64) for x in (cam.u, cam.v, cam.w))

    def value(m):
        r, wr = np.polynomial.legendre.leggauss(m)
        r, wr = 0.5 * (r + 1.0), 0.5 * wr                 # radius on [0, 1], weight r dr
        ph, wp = np.polynomial.legendre.leggauss(2 * m)
        ph, wp = np.pi * (ph + 1.0), np.pi * wp
        jx = (r[:, None] * np.cos(ph)[None, :]).ravel(); jy = (r[:, None] * np.sin(ph)[None, :]).ravel()
        wt = ((wr * r)[:, None] * wp[None, :]).ravel() / np.pi
        y, x = np.mgrid[0:H, 0:W]
        s = ((x + 0.5) / W * 2.0 - 1.0)[..., None] + jx / W
        t = ((y + 0.5) / H * 2.0 - 1.0)[..., None] + jy / H
        d = w + s[..., None] * u + t[..., None] * v
        return np.einsum("hwk,k->hw", 1.0 - sr.metal_absorbed(d, (0.0, 1.0, 0.0), fuzz), wt)
    a, b = value(n), value(2 * n)
    return b, np.abs(b - a)


def dielectric_scene(rtb, theta_deg: float, back: bool, sky, ior=1.5):
    """A clear dielectric quad in y = 0 seen from above at theta_deg; back=True gives the quad the normal -y, so that the
    ray meets its back face (refraction ratio ior, as if leaving the glass)."""
    s = rtb.Scene()
    objs = [_plane(s, s.dielectric(ior), normal_down=back)]
    cam = _incident_camera(rtb, s, objs, theta_deg, fov=RETRO_FOV)
    s.set_root(s.list(objs))
    s.set_environment(sky)
    return s, cam


def band_rows(theta: float, back: bool, candidates=range(181, 121, -2)):
    """(H, mirror row, Snell row or None): the first odd row count whose rows hold both directions with a margin of
    twice their spread over the pixel (0.01 degree of incidence, magnified by ratio cos(theta) / cos(theta_t) after
    refraction) from the row edges."""
    ratio = 1.5 if back else 1 / 1.5
    dirs = [(sr.mirror_polar(theta), 0.01)]
    tir = ratio * math.sin(theta) > 1.0
    if not tir:
        tt = math.asin(ratio * math.sin(theta))
        dirs.append((sr.snell_polar(theta, 1.5, back), 0.01 * ratio * math.cos(theta) / math.cos(tt)))
    for H in candidates:
        ok = True
        for polar, spread_deg in dirs:
            p, margin = sr.row_position(polar, H), 2 * spread_deg * H / 180.0 + 0.02
            ok &= p < margin or p > H - margin or min(p - math.floor(p), math.ceil(p) - p) >= margin
        if ok:
            rows = [min(int(sr.row_position(p, H)), H - 1) for p, _ in dirs]
            return H, rows[0], (None if tir else rows[1])
    raise AssertionError("no row count keeps the directions inside their rows")


def dielectric_maps(theta: float, back: bool):
    """Two maps: (upper half = R, lower half = T) and (mirror row, Snell row, every other row) with their expectations."""
    R = sr.dielectric_reflect_probability(theta, 1.5, back)
    H2 = 36
    halves = stack(row_mask(H2, 8, range(0, H2 // 2)), row_mask(H2, 8, range(H2 // 2, H2)), np.zeros((H2, 8), np.float32))
    H, rm, rt_ = band_rows(theta, back)
    rest = [j for j in range(H) if j not in (rm, rt_)]
    bands = stack(row_mask(H, 8, [rm]), row_mask(H, 8, [] if rt_ is None else [rt_]), row_mask(H, 8, rest))
    return [(halves, np.array([R, 1.0 - R, 0.0])), (bands, np.array([R, 1.0 - R, 0.0]))]


MEDIUM_ALBEDO = 0.7


def medium_scene(rtb, R: float, sigma: float, b: float, lamp=False, others: int = 0, target_index: int = 0):
    """A sphere of isotropic medium (albedo 0.7) at the origin under a white sky, seen along a chord at impact parameter
    b.  others > 0: the scene holds others + 1 media in creation order (medium numbers), the one at the origin being
    number target_index; the rest lie 300 units away in the x-y plane, radius 1 + 0.01 (9 - k) for medium k, so that the
    eight largest - the pre-test list - are media 0-7.  lamp: a sampled quad light emitting the sky's white, off to the
    side, so the expectation is unchanged."""
    s = rtb.Scene()
    objs = []
    for k in range(others + 1):
        c = (0.0, 0.0, 0.0) if k == target_index else (300.0 * math.cos(0.5 * k + 0.3), 300.0 * math.sin(0.5 * k + 0.3), 0.0)
        radius = R if k == target_index else (1.0 + 0.01 * (9 - k))
        iso = s.isotropic(s.solid((MEDIUM_ALBEDO,) * 3))
        objs.append(s.constant_medium(s.sphere(c, radius, s.lambertian((1, 1, 1))), sigma, iso))
    lamp_id = None
    if lamp:
        lamp_id = s.quad((-1.0, 3.0, -1.0), (2.0, 0.0, 0.0), (0.0, 0.0, 2.0), s.diffuse_light(s.solid((1.0, 1.0, 1.0))))
        objs.append(lamp_id)
    cam = periscope_camera(rtb, s, objs, "pinhole", (b, 0.0, 10.0), (b, 0.0, 0.0), (0, 1, 0), 0.02, 1.0)
    s.set_root(s.list(objs))
    if lamp:
        s.sample_lights([lamp_id])
    s.set_background(rtb.BG_CONSTANT, (1.0, 1.0, 1.0))
    return s, cam


EDGE_W, EDGE_H, EDGE_D, EDGE_PIXEL = 2, 2, 1.0, 0.001      # a 2 x 2 image of 1 mm pixels, one unit away


def edge_scene(rtb, alpha_deg: float, offset_px: float, kind="pinhole", focus_ratio=1.0, lens_px=0.8):
    """A white emitting half-plane in z = 0 under a black sky, its edge through the image centre shifted by offset_px
    pixels along the edge normal and tilted alpha_deg from horizontal, seen from z = EDGE_D.  kind "defocus": a lens
    focused at EDGE_D / focus_ratio whose blur at the plane has radius lens_px pixels.  Returns the scene, the camera and
    the geometry (edge normal, a point of the edge) for the reference."""
    a = math.radians(alpha_deg)
    t, m = np.array([math.cos(a), math.sin(a), 0.0]), np.array([-math.sin(a), math.cos(a), 0.0])
    P = -offset_px * EDGE_PIXEL * m
    s = rtb.Scene()
    # 100 x 50 pixels: a few pixels would do; a larger quad would put its corner Q where a float32 ulp is a sizeable
    # fraction of a pixel, and a tilted edge through it would move by that much
    Q = P - 0.05 * t
    objs = [s.quad(tuple(Q), tuple(0.1 * t), tuple(0.05 * m), s.diffuse_light(s.solid((1.0, 1.0, 1.0))))]
    s.set_background(rtb.BG_CONSTANT, (0.0, 0.0, 0.0))
    vfov = math.degrees(2.0 * math.atan(0.5 * EDGE_H * EDGE_PIXEL / EDGE_D))
    if kind == "pinhole":
        cam = periscope_camera(rtb, s, objs, "pinhole", (0, 0, EDGE_D), (0, 0, 0), (0, 1, 0), vfov, EDGE_W / EDGE_H, size=0.05)
    else:
        F = EDGE_D / focus_ratio
        lens = 0.0 if focus_ratio == 1.0 else lens_px * EDGE_PIXEL / abs(1.0 - focus_ratio)
        cam = periscope_camera(rtb, s, objs, "defocus", (0, 0, EDGE_D), (0, 0, 0), (0, 1, 0), vfov, EDGE_W / EDGE_H, aperture=2.0 * lens,
                               focus_dist=F, size=0.05)
    s.set_root(s.list(objs))
    return s, cam, (m, P)


def edge_reference(cam, geom, W=EDGE_W, H=EDGE_H, n=64):
    """Per pixel (value [H, W], error bound [H, W]) of an edge scene: the pixel-centre ray's point on z = 0 and its signed
    distance inside the lit side; pixel filter (pinhole) or the defocus convolution.  The rays are those of the camera
    the periscope reproduces."""
    m, P = geom
    u, v, w = (np.array(x, np.float64) for x in (cam.u, cam.v, cam.w))
    o = virtual_origin(cam)
    val, err = np.zeros((H, W)), np.zeros((H, W))
    for y in range(H):
        for x in range(W):
            s, t = (x + 0.5) / W * 2.0 - 1.0, (y + 0.5) / H * 2.0 - 1.0
            if cam.kind == 1:            # defocus (RTB_CAM_DEFOCUS): hori = u vw F, ...; the point at depth D is o + D (w + vw s u + vh t v)
                d = w + cam.viewport_width * s * u + cam.viewport_height * t * v
                ratio = EDGE_D / cam.focus_dist
                rj = EDGE_D * cam.viewport_width / W
                rl = cam.lens_radius * abs(1.0 - ratio)
            else:
                d = w + s * u + t * v
                rj = EDGE_D * np.linalg.norm(u) / W
                rl = 0.0
            p = o + d * (-o[2] / d[2])
            delta = float(m @ (p - P))
            val[y, x], err[y, x] = sr.defocus_lit(delta, rj, rl, n) if rl > 0 else (float(sr.pixel_filter_lit(delta / (2 * rj))), 0.0)
    return val, err


MOTION_PATHS = [((-1.0, 0.0, 0.0), (1.0, 0.0, 0.0)), ((-1.6, 0.0, 0.0), (0.4, 0.0, 0.0))]


def motion_scene(rtb, c0, c1, t0, t1, R=0.3):
    """A white emitting sphere of radius R moving from c0 (time 0) to c1 (time 1) across the view axis, black sky, a
    motion camera with shutter [t0, t1] looking down -z at the origin with a 0.01-degree field."""
    s = rtb.Scene()
    objs = [s.moving_sphere(c0, c1, R, s.diffuse_light(s.solid((1.0, 1.0, 1.0))))]
    cam = periscope_camera(rtb, s, objs, "motion", (0, 0, 10), (0, 0, 0), (0, 1, 0), 0.01, 1.0, t0=t0, t1=t1)
    s.set_root(s.list(objs))
    s.set_background(rtb.BG_CONSTANT, (0.0, 0.0, 0.0))
    return s, cam


def motion_reference(cam, c0, c1, R=0.3):
    return sr.motion_hit_fraction(virtual_origin(cam), cam.w, c0, c1, R, cam.t0, cam.t1)


# ------------------------------------------------------------------------------------------------ reference self-tests
def test_detector_map_convention():
    """+y is row 0, -y the last row, -x column 0 (u = 0), +z at u = 1/4, +x at 1/2, -z at 3/4 (DESIGN.md §5d)."""
    W, H = 8, 9
    dirs = np.array([[0, 1, 0], [0, -1, 0], [-1, 0, 1e-9], [0, 0, 1], [1, 0, 0], [0, 0, -1]], np.float64)
    i, j = sr.texel_of(dirs, W, H)
    assert list(j) == [0, H - 1, 4, 4, 4, 4]
    assert list(i) == [W // 2, W // 2, 0, W // 4, W // 2, 3 * W // 4]
    for polar in (0.3, 1.2, 2.9):
        for u in (0.05, 0.4, 0.9):
            ii, jj = sr.texel_of(sr.direction(polar, u), W, H)
            assert ii == int(u * W) and jj == int(polar / np.pi * H)


def test_mass_tables_sum_to_one_minus_absorbed():
    lam = sr.lambert_masses(LW, LH)
    assert abs(lam.sum() - 1.0) < 1e-12 and np.all(lam[LH // 2:] == 0)
    assert np.allclose(sr.lambert_masses(LW, LH, -1), lam[::-1])
    # above elevation asin(zmin) the cosine lobe holds 1 - zmin^2
    for rows, zmin in ((3, math.cos(math.radians(30))), (6, math.cos(math.radians(60)))):
        assert abs(lam[:rows].sum() - (1 - zmin ** 2)) < 1e-12
    for fuzz in (0.1, 0.5, 1.0, 1.5):
        for dlen in (1.0, 1.3):
            m = sr.metal_masses(MW, MH, fuzz, dlen)
            absorbed = float(sr.metal_absorbed(np.array([0.0, -dlen, 0.0]), (0, 1, 0), fuzz))
            assert abs(m.sum() - (1.0 - absorbed)) < 1e-12, (fuzz, dlen, m.sum(), absorbed)
            assert abs(sr.metal_cdf(np.pi, fuzz / dlen) - 1.0) < 1e-12


def test_metal_cdf_known_values():
    """g < 1: the fuzz sphere subtends a cone of half-angle asin g, all mass inside; g -> 0: a point; g large: nearly
    uniform (P(angle <= pi/2) -> 1/2); and against the closed form P(angle <= x) at g = 1, where p = r + s makes the
    angle beta / 2 with r for s at angle beta: (1 - cos 2x) / 2."""
    for g in (0.1, 0.5, 0.9):
        assert sr.metal_cdf(math.asin(g) + 1e-9, g) == 1.0
        assert sr.metal_cdf(math.asin(g) * 0.999, g) < 1.0
    assert sr.metal_cdf(1e-3, 1e-6) == 1.0
    assert abs(sr.metal_cdf(np.pi / 2, 1e6) - 0.5) < 1e-5
    for x in (0.1, 0.7, 1.4):
        assert abs(sr.metal_cdf(x, 1.0) - 0.5 * (1 - math.cos(2 * x))) < 1e-12
    # a uniform-sphere check at g = 1.5 against direct 1-D quadrature of the angle over u = s . r
    g, x = 1.5, 1.0
    u = np.linspace(-1, 1, 2_000_001)
    ang = np.arctan2(g * np.sqrt(1 - u * u), 1 + g * u)
    assert abs(sr.metal_cdf(x, g) - np.mean(ang <= x)) < 2e-6


def test_schlick_and_critical_angle():
    assert abs(sr.schlick(1.0, 1 / 1.5) - 0.04) < 1e-15 and abs(sr.schlick(1.0, 1.5) - 0.04) < 1e-15
    assert sr.schlick(0.0, 1.5) == 1.0
    crit = math.asin(1 / 1.5)
    assert abs(math.degrees(crit) - 41.8103149) < 1e-6
    assert sr.dielectric_reflect_probability(math.radians(41.0), 1.5, True) < 0.5
    assert sr.dielectric_reflect_probability(math.radians(42.0), 1.5, True) == 1.0
    assert sr.dielectric_reflect_probability(math.radians(85.0), 1.5, False) < 1.0
    # Snell: sin of the refracted angle is ratio x sin of the incident one
    th = math.radians(30.0)
    assert abs(math.sin(np.pi - sr.snell_polar(th, 1.5, False)) - math.sin(th) / 1.5) < 1e-15


def test_medium_limits():
    """albedo -> 0: the transmission e^(-2 R sigma) through the centre; sigma -> 0: the white furnace (1); and the error
    bound of the rule is below 1e-7 at every case the GPU file uses."""
    for sigma in (0.1, 1.0, 3.0):
        v, e = sr.medium_pixel(1.0, sigma, 0.0, 0.0)
        assert abs(v - math.exp(-2 * sigma)) < 1e-14
    v, e = sr.medium_pixel(1.0, 1e-7, 1.0, 0.3)
    assert abs(v - 1.0) < 1e-6
    for sigma in (0.1, 1.0, 3.0):
        for b in (0.0, 0.5, 0.9):
            v, e = sr.medium_pixel(1.0, sigma, MEDIUM_ALBEDO, b)
            assert e < 1e-7 and 0 < v < 1, (sigma, b, v, e)
    # with albedo 1, depth 2 loses the twice-scattered paths: the value stays below 1 (the 0.001 offset included)
    assert sr.medium_pixel(1.0, 3.0, 1.0, 0.0)[0] < 1.0


def test_pixel_filter_and_defocus_reference():
    assert sr.pixel_filter_lit(0.0) == 0.5
    assert sr.pixel_filter_lit(0.5) == 1.0 and sr.pixel_filter_lit(-0.5) == 0.0
    assert abs(sr.pixel_filter_lit(0.2) + sr.pixel_filter_lit(-0.2) - 1.0) < 1e-15
    for delta in (-0.3, 0.0, 0.1, 0.45):
        # no lens blur: the pixel filter itself; a tiny lens: continuous in rl
        v0, _ = sr.defocus_lit(delta, 0.5, 0.0)
        assert abs(v0 - sr.pixel_filter_lit(delta)) < 1e-15
        v1, e1 = sr.defocus_lit(delta, 0.5, 1e-6)
        assert abs(v1 - v0) < 1e-5 and e1 < 1e-9
        # symmetric in the two radii (the sum of two independent projections), and odd about 1/2
        a, ea = sr.defocus_lit(delta, 0.5, 0.8)
        b, eb = sr.defocus_lit(delta, 0.8, 0.5)
        c, _ = sr.defocus_lit(-delta, 0.5, 0.8)
        assert abs(a - b) < 1e-9 and abs(a + c - 1.0) < 1e-9 and ea < 1e-9 and eb < 1e-9


def test_motion_reference():
    o, d = (0, 0, 10), (0, 0, -1)
    assert abs(sr.motion_hit_fraction(o, d, *MOTION_PATHS[0], 0.3, 0.2, 0.7) - 0.6) < 1e-12
    assert abs(sr.motion_hit_fraction(o, d, *MOTION_PATHS[0], 0.3, 0.0, 1.0) - 0.3) < 1e-12
    assert abs(sr.motion_hit_fraction(o, d, *MOTION_PATHS[1], 0.3, 0.2, 0.7) - 0.1) < 1e-12
    assert abs(sr.motion_hit_fraction(o, d, *MOTION_PATHS[1], 0.3, 0.0, 1.0) - 0.3) < 1e-12


# ------------------------------------------------------------------------------------------------ the oracle against the references
def oracle_mean(scene, cam, W, H, spp, depth=DEPTH, seed=5):
    sum_, sum2, _ = FeatureOracleScene(scene.serialize()).render(cam, W, H, 0, spp, depth, seed=seed, want_sum2=True)
    return mean_and_error(sum_, sum2)


def within(m, e, want, bound=0.0):
    return np.all(np.abs(np.asarray(m) - np.asarray(want)) <= 4 * np.asarray(e) + bound + 2e-5)


@pytest.mark.parametrize("target", ["front", "back", "sphere"])
def test_oracle_lambertian(rtb, target):
    sky = lambert_map()
    want = sr.expected(sr.lambert_masses(LW, LH), sky)
    for lamp, sample_env in ((False, False), (True, False), (False, True)):
        m, e = oracle_mean(*lambert_scene(rtb, target, sky, lamp, sample_env), 16, 16, 128)
        assert within(m, e, want), (lamp, sample_env, m, e, want)


@pytest.mark.parametrize("fuzz", [0.1, 0.5, 1.0, 1.5])
def test_oracle_metal(rtb, fuzz):
    sky = metal_map()
    m, e = oracle_mean(*metal_scene(rtb, fuzz, sky), 16, 16, 128, depth=metal_depth(fuzz))
    assert within(m, e, sr.expected(sr.metal_masses(MW, MH, fuzz), sky)), (m, e)


def test_oracle_metal_wide_field(rtb):
    W = H = 4
    s, cam = metal_scene(rtb, 1.0, wide=True)
    sum_, sum2, _ = FeatureOracleScene(s.serialize()).render(cam, W, H, 0, 8192, 2, seed=9, want_sum2=True)
    n = sum_[..., 3:4].astype(np.float64)
    m = sum_[..., :3] / n
    e = np.sqrt(np.maximum(sum2[..., :3] / n - m * m, 0) / n)
    want, err = metal_wide_reference(cam, W, H, 1.0)
    assert np.all(np.abs(m - want[..., None]) <= 4 * e + err[..., None] + 2e-5), (m[..., 0], want)
    assert want.min() < 0.8 and want.max() > 0.95            # the absorbed fraction varies across the field


@pytest.mark.parametrize("theta,back", [(0.0, False), (60.0, False), (30.0, True), (41.0, True), (42.0, True)])
def test_oracle_dielectric(rtb, theta, back):
    for sky, want in dielectric_maps(math.radians(theta), back):
        m, e = oracle_mean(*dielectric_scene(rtb, theta, back, sky), 16, 16, 64, depth=DEPTH_RETRO)
        assert within(m, e, want), (m, e, want)


@pytest.mark.parametrize("sigma,b", [(1.0, 0.0), (3.0, 0.5), (0.1, 0.9)])
def test_oracle_medium(rtb, sigma, b):
    want, err = sr.medium_pixel(1.0, sigma, MEDIUM_ALBEDO, b)
    m, e = oracle_mean(*medium_scene(rtb, 1.0, sigma, b), 16, 16, 128)
    assert within(m, e, [want] * 3, err), (m, e, want)


def test_oracle_media_beyond_the_pre_list(rtb):
    """Medium 5 (uniform from stream 17, pre-tested) and medium 9 (a BVH leaf) of ten."""
    for target in (5, 9):
        R = 1.0 + 0.01 * (9 - target)
        want, err = sr.medium_pixel(R, 1.0, MEDIUM_ALBEDO, 0.5)
        m, e = oracle_mean(*medium_scene(rtb, R, 1.0, 0.5, others=9, target_index=target), 16, 16, 128)
        assert within(m, e, [want] * 3, err), (target, m, e, want)


@pytest.mark.parametrize("alpha", [0.0, 30.0])
def test_oracle_pixel_filter(rtb, alpha):
    for off in (-0.6, -0.2, 0.1, 0.5):
        s, cam, geom = edge_scene(rtb, alpha, off)
        sum_, _, _ = FeatureOracleScene(s.serialize()).render(cam, EDGE_W, EDGE_H, 0, 4096, DEPTH, seed=3)
        m = sum_[..., 0] / sum_[..., 3]
        want, _ = edge_reference(cam, geom)
        assert np.all(np.abs(m - want) <= 4 * np.sqrt(want * (1 - want) / 4096) + 2e-5), (off, m, want)


@pytest.mark.parametrize("ratio", [1.0, 0.8, 1.5])
def test_oracle_defocus(rtb, ratio):
    for off in (-0.6, 0.0, 0.4):
        s, cam, geom = edge_scene(rtb, 0.0, off, kind="defocus", focus_ratio=ratio)
        sum_, _, _ = FeatureOracleScene(s.serialize()).render(cam, EDGE_W, EDGE_H, 0, 4096, DEPTH, seed=4)
        m = sum_[..., 0] / sum_[..., 3]
        want, err = edge_reference(cam, geom)
        if ratio == 1.0:
            pin = edge_reference(*edge_scene(rtb, 0.0, off)[1:])[0]
            assert np.allclose(want, pin, atol=1e-6)
        assert np.all(np.abs(m - want) <= 4 * np.sqrt(want * (1 - want) / 4096) + err + 2e-5), (off, m, want)


@pytest.mark.parametrize("shutter", [(0.2, 0.7), (0.0, 1.0)])
@pytest.mark.parametrize("path", [0, 1])
def test_oracle_motion_blur(rtb, shutter, path):
    s, cam = motion_scene(rtb, *MOTION_PATHS[path], *shutter)
    m, e = oracle_mean(s, cam, 8, 8, 256)
    want = motion_reference(cam, *MOTION_PATHS[path])
    assert within(m, e, [want] * 3), (m, e, want)
