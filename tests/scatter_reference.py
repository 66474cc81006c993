"""TEST INFRASTRUCTURE: float64 references for the materials, camera samplers and media of Books 1 and 2 in the Philox-mode
spec (DESIGN.md §5, §5d, §6), written from that text and the books, not from the kernels.  Nothing here is Monte Carlo:
each value is closed form, or Gauss-Legendre quadrature returned with an error bound (the change when the rule is doubled).

Conventions shared with the scenes of tests/test_cpu_scatter_distributions.py and tests/test_gpu_scatter_distributions.py:
  * A detector map is an equirectangular environment map (§5d): row j of H covers polar angles [pi j / H, pi (j + 1) / H]
    measured from +y, column i of W covers u = (atan2(-z, x) + pi) / 2 pi in [i / W, (i + 1) / W].  A render under a map
    whose texels are 0 / 1 masks measures the probability that the scattered direction lands in the masked texels.
  * Angles are radians unless a name ends in _deg.
"""
from __future__ import annotations

import math

import numpy as np

SCATTER_OFFSET = 0.001      # a scattered ray leaves from p + 0.001 dir (§6, Renderer.cu:168-175)


# ------------------------------------------------------------------------------------------------ detector maps
def row_edges(H: int) -> np.ndarray:
    """Polar angles (from +y) of the H + 1 row edges."""
    return np.pi * np.arange(H + 1) / H


def texel_of(d, W: int, H: int):
    """(column, row) of unit or un-normalised directions d [..., 3] on a W x H map (float64, §5d steps 1-3)."""
    d = np.asarray(d, np.float64)
    n = d / np.linalg.norm(d, axis=-1, keepdims=True)
    u = (np.arctan2(-n[..., 2], n[..., 0]) + np.pi) / (2 * np.pi)
    v = np.arccos(np.clip(-n[..., 1], -1.0, 1.0)) / np.pi
    return np.minimum((u * W).astype(int), W - 1), np.minimum(((1.0 - v) * H).astype(int), H - 1)


def direction(polar: float, u: float) -> np.ndarray:
    """The unit direction at polar angle `polar` from +y and map coordinate u (the inverse of the lookup)."""
    phi = 2 * np.pi * u
    return np.array([-math.sin(polar) * math.cos(phi), math.cos(polar), math.sin(polar) * math.sin(phi)])


def row_position(polar: float, H: int) -> float:
    """Fractional row coordinate of a polar angle: row j holds [j, j + 1)."""
    return polar / np.pi * H


def band_masses(cdf, H: int, flip: bool = False) -> np.ndarray:
    """Per-row masses of an azimuthally symmetric distribution about +y (about -y with flip), from the CDF of its polar
    angle.  Mass that is not in any row (absorbed) is simply missing from the sum."""
    e = row_edges(H)
    F = np.array([cdf(x) for x in e])
    m = np.diff(F)
    return m[::-1].copy() if flip else m


def texel_masses(rows: np.ndarray, W: int) -> np.ndarray:
    """[H, W] texel masses of a distribution whose azimuth about the y axis is uniform."""
    return np.repeat(rows[:, None] / W, W, axis=1)


def expected(masses: np.ndarray, mask: np.ndarray) -> np.ndarray:
    """The pixel value a render measures under a map: sum of texel mass x texel value, per channel (mask [H, W, 3])."""
    return np.einsum("hw,hwc->c", masses, np.asarray(mask, np.float64))


# ------------------------------------------------------------------------------------------------ Lambertian
def lambert_cdf(x: float) -> float:
    """P(polar angle from the normal <= x) of the direction of n + s, s uniform on the unit sphere: the cosine lobe,
    sin^2 x up to the horizon."""
    return math.sin(min(x, np.pi / 2)) ** 2


def lambert_masses(W: int, H: int, normal_sign: int = 1) -> np.ndarray:
    """Texel masses of a Lambertian scatter about the normal (0, normal_sign, 0)."""
    return texel_masses(band_masses(lambert_cdf, H, flip=normal_sign < 0), W)


# ------------------------------------------------------------------------------------------------ metal with fuzz
def metal_cdf(x: float, g: float) -> float:
    """P(angle between r + g s and r <= x) for a unit vector r and s uniform on the unit sphere (g = fuzz / |d|: the book
    reflects the un-normalised d, so reflect(d, n) has length |d|, and the fuzz sphere of radius fuzz is relative to it).

    With u = s.r uniform on [-1, 1] (Archimedes), p = r + g s has p.r = 1 + g u and |p|^2 = 1 + 2 g u + g^2; the event
    p.r >= cos x |p| changes truth only at the roots of (1 + g u)^2 = cos^2 x (1 + 2 g u + g^2), u = (-sin^2 x +- cos x
    sqrt(g^2 - sin^2 x)) / g, and where 1 + g u changes sign.  Between those points it is tested directly: the measure is
    exact up to float64 rounding."""
    if x <= 0.0:
        return 0.0
    if x >= np.pi:
        return 1.0
    c, s2 = math.cos(x), math.sin(x) ** 2
    pts = {-1.0, 1.0}
    if g > 0:
        pts.add(-1.0 / g)
        if g * g >= s2:
            r = abs(c) * math.sqrt(g * g - s2)
            pts.update(((-s2 + r) / g, (-s2 - r) / g))
    pts = sorted(p for p in pts if -1.0 <= p <= 1.0)
    inside = 0.0
    for a, b in zip(pts[:-1], pts[1:]):
        u = 0.5 * (a + b)
        if 1.0 + g * u >= c * math.sqrt(max(1.0 + 2.0 * g * u + g * g, 0.0)):
            inside += b - a
    return 0.5 * inside


def metal_absorbed(d, n, fuzz: float) -> np.ndarray:
    """P(dir . n < 0) for dir = reflect(d, n) + fuzz s: reflect(d, n) . n = -d . n, and s . n is uniform on [-1, 1], so the
    fraction is clip((1 - |d . n| / fuzz) / 2, 0, 1).  d [..., 3] un-normalised camera directions, n the unit normal."""
    dn = np.abs(np.asarray(d, np.float64) @ np.asarray(n, np.float64))
    if fuzz == 0:
        return np.zeros_like(dn)
    return np.clip(0.5 * (1.0 - dn / fuzz), 0.0, 1.0)


def metal_masses(W: int, H: int, fuzz: float, dlen: float = 1.0) -> np.ndarray:
    """Texel masses at normal incidence on a plane with normal +y (reflect(d, n) along +y): rows of the lower hemisphere
    are absorbed and left out, so the table sums to 1 - absorbed (H even: the horizon is a row edge)."""
    assert H % 2 == 0
    rows = band_masses(lambda x: metal_cdf(x, fuzz / dlen), H)
    rows[H // 2:] = 0.0
    return texel_masses(rows, W)


# ------------------------------------------------------------------------------------------------ dielectric
def schlick(cos: float, ratio: float) -> float:
    r0 = ((1.0 - ratio) / (1.0 + ratio)) ** 2
    return r0 + (1.0 - r0) * (1.0 - cos) ** 5


def dielectric_reflect_probability(theta: float, ior: float, back: bool) -> float:
    """P(reflect) of the book's dielectric at incidence theta: the refraction ratio is 1 / ior on a front face and ior on a
    back face; Schlick with the incident cosine, and 1 past the critical angle."""
    ratio = ior if back else 1.0 / ior
    if ratio * math.sin(theta) > 1.0:
        return 1.0
    return schlick(math.cos(theta), ratio)


def mirror_polar(theta: float) -> float:
    """Polar angle from +y of the mirror direction off a plane with normal +y (the ray arrives from above)."""
    return theta


def snell_polar(theta: float, ior: float, back: bool) -> float:
    """Polar angle from +y of the refracted direction (the ray arrives from above and continues below)."""
    ratio = ior if back else 1.0 / ior
    return np.pi - math.asin(ratio * math.sin(theta))


# ------------------------------------------------------------------------------------------------ isotropic medium sphere
def _gl(a: float, b: float, n: int):
    x, w = np.polynomial.legendre.leggauss(n)
    return 0.5 * (b - a) * x + 0.5 * (b + a), 0.5 * (b - a) * w


def medium_pixel(R: float, sigma: float, albedo: float, b: float, n: int = 96):
    """(value, error bound) of a camera ray along a chord at impact parameter b through a sphere of isotropic medium
    (radius R, density sigma, albedo) under a constant white background, at max_depth = 2:

        e^(-sigma L) + albedo * int_0^L sigma e^(-sigma s) E(r(s)) ds,   E(r) = 1/2 int_-1^1 e^(-sigma l(r, mu)) dmu,

    L = 2 sqrt(R^2 - b^2) the chord, r(s) the distance of the scatter point from the centre, mu the cosine between the
    scattered direction and the outward radius, l = -r mu + sqrt(R^2 - r^2 (1 - mu^2)) - 0.001 the distance the scattered
    ray travels inside (it leaves 0.001 along its direction).  A second scatter ends the path black at this depth."""
    def value(m):
        L = 2.0 * math.sqrt(R * R - b * b)
        s, ws = _gl(0.0, L, m)
        mu, wm = _gl(-1.0, 1.0, m)
        r = np.sqrt(b * b + (s - 0.5 * L) ** 2)[:, None]
        ell = -r * mu[None, :] + np.sqrt(np.maximum(R * R - r * r * (1.0 - mu[None, :] ** 2), 0.0))
        ell = np.maximum(ell - SCATTER_OFFSET, 0.0)
        E = 0.5 * (np.exp(-sigma * ell) @ wm)
        once = float(np.sum(ws * sigma * np.exp(-sigma * s) * E))
        return math.exp(-sigma * L) + albedo * once
    v, v2 = value(n), value(2 * n)
    return v2, abs(v2 - v)


# ------------------------------------------------------------------------------------------------ pixel filter and defocus
def disc_below(h):
    """Fraction of a disc on the side x <= h r of a chord (h in units of the radius, clipped to [-1, 1])."""
    h = np.clip(np.asarray(h, np.float64), -1.0, 1.0)
    return (h * np.sqrt(1.0 - h * h) + np.arcsin(h) + 0.5 * np.pi) / np.pi


def pixel_filter_lit(delta):
    """Lit fraction of a pixel whose centre lies delta pixels inside an emitting half-plane: the filter is a uniform disc
    of radius 1/2 pixel (§6), so this is the circular segment beyond the edge."""
    return disc_below(np.asarray(delta, np.float64) / 0.5)


def defocus_lit(delta: float, rj: float, rl: float, n: int = 64):
    """(lit fraction, error bound) of a defocused pixel: the hit point on the edge's plane is the pixel-centre point plus
    the jitter (a uniform disc of radius rj) plus the lens offset (a uniform disc of radius rl = lens_radius |1 - D / F|),
    independent; along the edge's normal each projects to a semicircle law, and the point is lit when the sum exceeds
    -delta (delta: signed distance of the pixel-centre point inside the lit side, same units).  A 1-D convolution: the
    jitter's projection rj cos(phi) has density (2 / pi) sin^2(phi) on [0, pi]; the rule is split where the lens term
    has its kinks."""
    if rl == 0.0:
        return float(disc_below(delta / rj)), 0.0

    def lens_above(y):                  # P(lens projection > y)
        return 1.0 - disc_below(y / rl)

    def value(m):
        cuts = {0.0, np.pi}
        for k in (-delta - rl, -delta + rl):
            if abs(k) < rj:
                cuts.add(math.acos(k / rj))
        cuts = sorted(cuts)
        tot = 0.0
        for a, b in zip(cuts[:-1], cuts[1:]):
            phi, w = _gl(a, b, m)
            tot += float(np.sum(w * (2.0 / np.pi) * np.sin(phi) ** 2 * lens_above(-delta - rj * np.cos(phi))))
        return tot
    v, v2 = value(n), value(2 * n)
    return v2, abs(v2 - v)


# ------------------------------------------------------------------------------------------------ motion blur
def motion_hit_fraction(o, d, c0, c1, R: float, t0: float, t1: float) -> float:
    """Fraction of shutter samples at which the ray (o, d) meets a sphere of radius R centred at mix(c0, c1, time), with
    time = mix(t0, t1, u) on the raw shutter (§6) and u uniform.  The squared distance from the centre to the ray's line
    is a quadratic in time; the hit times are where it is below R^2 (the sphere lies in front of the ray)."""
    o, d, c0, c1 = (np.asarray(v, np.float64) for v in (o, d, c0, c1))
    e = d / np.linalg.norm(d)

    def perp(v):
        return v - (v @ e) * e
    p0, dp = perp(c0 - o), perp(c1 - c0)            # perpendicular offset at time 0 and its rate
    A, B, C = dp @ dp, 2 * (p0 @ dp), p0 @ p0 - R * R
    disc = B * B - 4 * A * C
    if A == 0.0:
        return 1.0 if C < 0 else 0.0
    if disc <= 0:
        return 0.0
    lo, hi = (-B - math.sqrt(disc)) / (2 * A), (-B + math.sqrt(disc)) / (2 * A)
    a, b = max(lo, min(t0, t1)), min(hi, max(t0, t1))
    return max(b - a, 0.0) / abs(t1 - t0)
