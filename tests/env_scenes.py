"""TEST INFRASTRUCTURE: the environment-map scenes and hand-derived answers shared by tests/test_cpu_environment.py and
tests/test_gpu_environment.py (DESIGN.md §5d).  Nothing here renders: the tests render these scenes on the CPU oracle
(tests/feature_oracle.py) and on the GPU."""
from __future__ import annotations

import numpy as np

# ------------------------------------------------------------------------------------------------ orientation
# Which texel (column i, row j; row 0 = top) each axis direction reads on a W x H map, from §5d "Lookup" with W and H odd
# (so that no axis falls on a texel edge; -x lies on the seam between the last column and column 0 and reads column 0).
OW, OH = 5, 3


def axis_texels(W=OW, H=OH):
    return {"+x": (W // 2, H // 2), "-x": (0, H // 2), "+y": (W // 2, 0), "-y": (W // 2, H - 1),
            "+z": (W // 4, H // 2), "-z": ((3 * W) // 4, H // 2)}


AXES = {"+x": (1, 0, 0), "-x": (-1, 0, 0), "+y": (0, 1, 0), "-y": (0, -1, 0), "+z": (0, 0, 1), "-z": (0, 0, -1)}


def distinct_map(W, H):
    """Every texel a different colour: (1 + i, 1 + j, 1 + i + W j)."""
    j, i = np.mgrid[0:H, 0:W]
    return np.stack([1.0 + i, 1.0 + j, 1.0 + i + W * j], axis=-1).astype(np.float32)


def orientation_map():
    """distinct_map with the top and bottom rows constant: a camera along +-y sees the pole, where every column meets."""
    m = distinct_map(OW, OH)
    m[0, :] = (50.0, 60.0, 70.0)
    m[-1, :] = (80.0, 90.0, 100.0)
    return m


def orientation_scene(rtb, sample=False):
    """No geometry in view: one tiny sphere off every axis, the orientation map as the sky."""
    s = rtb.Scene()
    s.set_root(s.sphere((40.0, 30.0, 20.0), 0.01, s.lambertian((0.5, 0.5, 0.5))))
    s.set_environment(orientation_map(), sample=sample)
    return s


def orientation_camera(rtb, axis):
    """A 1 x 1 pixel camera at the origin with a 0.01 degree field looking along `axis`.  (-x looks 0.01 rad towards +z:
    exactly along -x half of the jittered rays would cross the seam into the last column.)"""
    d = list(AXES[axis])
    if axis == "-x":
        d[2] = 0.01
    up = (0, 0, 1) if axis in ("+y", "-y") else (0, 1, 0)
    return rtb.make_camera("pinhole", (0, 0, 0), tuple(d), up, 0.01, 1.0)


# ------------------------------------------------------------------------------------------------ one texel
# A Lambertian quad of albedo RHO in the plane y = 0 facing +y, seen from above, max_depth 2: the camera ray hits it, the
# scattered ray leaves the scene and reads the map, which is black except texel (TI, TJ) of radiance L.  Expected
# radiance (rho / pi) L (2 pi / W) (sin^2 b - sin^2 a) / 2 with [a, b] the texel's angles from +y.
RHO, L = 0.6, 7.0
TW, TH, TI, TJ = 8, 6, 3, 1


def one_texel_map():
    m = np.zeros((TH, TW, 3), np.float32)
    m[TJ, TI] = L
    return m


def one_texel_expected():
    a, b = np.pi * TJ / TH, np.pi * (TJ + 1) / TH
    return RHO / np.pi * L * (2 * np.pi / TW) * (np.sin(b) ** 2 - np.sin(a) ** 2) / 2


def one_texel_scene(rtb, sample):
    s = rtb.Scene()
    s.set_root(s.quad((-100, 0, -100), (200, 0, 0), (0, 0, 200), s.lambertian((RHO, RHO, RHO))))
    s.set_environment(one_texel_map(), sample=sample)
    cam = rtb.make_camera("pinhole", (0, 2, 0), (0, 0, 0), (0, 0, 1), 30.0, 1.0)
    return s, cam


# ------------------------------------------------------------------------------------------------ furnace, 1x1 map

def furnace_scene(rtb, sample):
    """A white Lambertian sphere under a white 1 x 1 map: every path returns exactly 1 without sampling."""
    s = rtb.Scene()
    s.set_root(s.sphere((0, 0, 0), 1.0, s.lambertian((1.0, 1.0, 1.0))))
    s.set_environment(np.ones((1, 1, 3), np.float32), sample=sample)
    cam = rtb.make_camera("pinhole", (0, 0, 4), (0, 0, 0), (0, 1, 0), 40.0, 1.0)
    return s, cam


SKY = (0.3, 0.5, 0.9)


def sky_scene(rtb):
    """Ground, a diffuse and a glass sphere, a camera that sees the sky: background constant SKY."""
    s = rtb.Scene()
    ground = s.quad((-20, 0, -20), (40, 0, 0), (0, 0, 40), s.lambertian((0.5, 0.6, 0.4)))
    ball = s.sphere((0, 1, 0), 1.0, s.lambertian((0.7, 0.3, 0.2)))
    glass = s.sphere((2.2, 1, 0.5), 1.0, s.dielectric(1.5))
    s.set_root(s.list([ground, ball, glass]))
    s.set_background(rtb.BG_CONSTANT, SKY)
    cam = rtb.make_camera("pinhole", (0, 2, 7), (0.5, 1, 0), (0, 1, 0), 50.0, 1.5)
    return s, cam


def sun_sky_map(W, H, seed=0, sun_deg=0.5, sun_radiance=None):
    """Procedural sun and sky: a gradient sky (blue above, pale at the horizon, dim ground) plus a disc of angular diameter
    `sun_deg` that carries most of the irradiance, its direction drawn from `seed`."""
    rng = np.random.default_rng(seed)
    j, i = np.mgrid[0:H, 0:W]
    theta = np.pi * (j + 0.5) / H                      # from +y
    phi = 2 * np.pi * (i + 0.5) / W
    y = np.cos(theta)
    sky = np.where(y[..., None] > 0, np.array([0.25, 0.45, 0.9]) * (0.4 + 0.6 * y[..., None]) + np.array([0.6, 0.6, 0.55]) * (1 - y[..., None]) ** 4,
                   np.array([0.15, 0.13, 0.1]))
    el = np.deg2rad(rng.uniform(25, 60)); az = rng.uniform(0, 2 * np.pi)
    # direction of texel (i, j) with the lookup's convention: u = phi / 2 pi, v = 1 - theta / pi (book v from -y)
    u = phi / (2 * np.pi); v = 1 - theta / np.pi
    dirs = np.stack([-np.sin(np.pi * v) * np.cos(2 * np.pi * u), -np.cos(np.pi * v), np.sin(np.pi * v) * np.sin(2 * np.pi * u)], -1)
    sun = np.array([np.cos(el) * np.cos(az), np.sin(el), np.cos(el) * np.sin(az)])
    r = np.deg2rad(sun_deg) / 2
    disc = (dirs @ sun) > np.cos(r)
    if not disc.any():                                 # a map too coarse for the disc: the nearest texel
        disc.reshape(-1)[np.argmax((dirs @ sun).reshape(-1))] = True
    if sun_radiance is None:                           # ~90 % of the irradiance on a plane facing the sun
        sun_radiance = 9.0 * np.pi * 0.6 / (2 * np.pi * (1 - np.cos(r)))
    out = sky.copy()
    out[disc] = np.array([1.0, 0.95, 0.85]) * sun_radiance
    return out.astype(np.float32), sun
