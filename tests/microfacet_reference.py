"""TEST INFRASTRUCTURE: float64 directional albedo of the GGX materials of DESIGN.md §5f, by quadrature of the BSDF.

Independent of the renderer's sampler: nothing here draws a visible normal or uses G2 / G1.  The integrand is the BSDF of
Walter et al. 2007 - the GGX distribution D, the height-correlated Smith G2 = 1 / (1 + Lambda(o) + Lambda(i)), Schlick's
Fresnel term F (for the dielectric with total internal reflection, F = 1 where ratio * sin > 1, ratio = 1 / eta) - times
|i.z|, integrated over the outgoing hemisphere (reflection) or the lower one (transmission):

    E_R(o) = int f_r(o, i) |i.z| d(omega_i),   f_r = D G2 F / (4 |o.z| |i.z|)
    E_T(o) = int f_t(o, i) |i.z| d(omega_i),   f_t = |o.h| |i.h| eta^2 (1 - F) D G2 / (|o.z| |i.z| (o.h + eta i.h)^2)

with eta = n_inside / n_outside of the side o is on (the outside).  The dielectric of §5f has no 1 / eta^2 radiance factor,
which is f_t above as Walter writes it for flux.  The integrals are taken over half-vector coordinates: d(omega_i) =
J d(omega_h), J = 4 |o.h| (reflection) or (o.h + eta i.h)^2 / (eta^2 |i.h|) (refraction), and h is parametrised by
(u, phi) with D cos(theta_h) d(omega_h) = du dphi / (2 pi) - so a narrow lobe (alpha = 0.05) is spread evenly over u - and
u = 1 - t^2, which removes the 1 / sqrt(1 - u) of grazing half vectors.  Along each phi the t-range is split where the
integrand is discontinuous or has a kink (o.h = 0, i.z = 0, total internal reflection, the restriction i.z > z_min), and
Gauss-Legendre rules are used on every piece, so the result converges fast; albedo() with n and 2n shows by how much.
Frame: the normal is +z, o = (sin theta_o, 0, cos theta_o)."""
from __future__ import annotations

import numpy as np

np.seterr(divide="ignore", invalid="ignore")   # masked out below: grazing and non-existent directions

PI = np.pi


# ------------------------------------------------------------------ BSDF in direction space
def _dot(a, b):
    return np.sum(a * b, axis=-1)


def _normalize(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def ggx_d(h, alpha):
    c2 = h[..., 2] ** 2
    tan2 = (1.0 - c2) / c2
    return 1.0 / (PI * alpha * alpha * c2 * c2 * (1.0 + tan2 / (alpha * alpha)) ** 2)


def smith_lambda(w, alpha):
    tan2 = (w[..., 0] ** 2 + w[..., 1] ** 2) / w[..., 2] ** 2
    return (np.sqrt(1.0 + alpha * alpha * tan2) - 1.0) * 0.5


def smith_g2(o, i, alpha):
    return 1.0 / (1.0 + smith_lambda(o, alpha) + smith_lambda(i, alpha))


def schlick(cos, r0):
    return r0 + (1.0 - r0) * (1.0 - cos) ** 5


def dielectric_fresnel(cos, eta):
    """The Fresnel term of §5f's dielectric at cos = o.h: Schlick with r0 of ratio = 1 / eta, and 1 under total internal
    reflection (ratio * sin > 1)."""
    ratio = 1.0 / eta
    r0 = ((1.0 - ratio) / (1.0 + ratio)) ** 2
    sin = np.sqrt(np.maximum(0.0, 1.0 - cos * cos))
    return np.where(ratio * sin > 1.0, 1.0, schlick(cos, r0))


def f_reflect(o, i, alpha, fresnel):
    """Reflection BSDF (fresnel: a function of o.h), 0 unless both directions are above the surface."""
    h = _normalize(o + i)
    ok = (o[..., 2] > 0) & (i[..., 2] > 0)
    val = ggx_d(h, alpha) * smith_g2(o, i, alpha) * fresnel(np.abs(_dot(o, h))) / (4.0 * np.abs(o[..., 2]) * np.abs(i[..., 2]))
    return np.where(ok, val, 0.0)


def f_transmit(o, i, alpha, eta, fresnel=True):
    """Walter's refraction BSDF from o (outside, o.z > 0) to i (i.z < 0, inside, index ratio eta); fresnel=False leaves
    out the (1 - F) factor (the rest is reciprocal up to eta^2)."""
    h = o + eta * i
    h = _normalize(np.where(h[..., 2:3] < 0, -h, h))
    oh, ih = _dot(o, h), _dot(i, h)
    ok = (o[..., 2] > 0) & (i[..., 2] < 0) & (oh > 0) & (ih < 0)
    den = oh + eta * ih
    val = np.abs(oh) * np.abs(ih) * eta * eta * ggx_d(h, alpha) * smith_g2(o, i, alpha) / (np.abs(o[..., 2]) * np.abs(i[..., 2]) * den * den)
    if fresnel:
        val = val * (1.0 - dielectric_fresnel(np.abs(oh), eta))
    return np.where(ok, val, 0.0)


# ------------------------------------------------------------------ half-vector quadrature
def _half(t, phi, alpha):
    """h(t, phi) and the factor du dphi / (2 pi D cos theta_h) per dt dphi."""
    t2 = t * t
    s = np.sqrt(t2 + alpha * alpha * (1.0 - t2))
    cos, sin = t / s, alpha * np.sqrt(1.0 - t2) / s
    h = np.stack([sin * np.cos(phi), sin * np.sin(phi), cos], -1)
    return h, h


def _reflect_dir(o, h):
    return 2.0 * _dot(o, h)[..., None] * h - o


def _refract_dir(o, h, eta):
    """The sampler's refraction of -o about h with ratio = 1 / eta; NaN where it does not exist."""
    ratio = 1.0 / eta
    ud = -o
    dv = _dot(h, ud)
    k = 1.0 - ratio * ratio * (1.0 - dv * dv)
    coef = ratio * dv + np.sqrt(np.where(k >= 0, k, np.nan))
    return ratio * ud - coef[..., None] * h


def _integrand(t, phi, o, alpha, part, fresnel, eta, zmin):
    """The BSDF x |i.z| x Jacobian / (D cos theta_h) x du/dt / (2 pi), per dt dphi."""
    h, _ = _half(t, phi, alpha)
    oh = _dot(o, h)
    dn = ggx_d(h, alpha) * h[..., 2]
    w = 2.0 * t / (2.0 * PI) / dn
    if part == "R":
        i = _reflect_dir(o, h)
        f = f_reflect(o, i, alpha, fresnel)
        val = f * np.abs(i[..., 2]) * 4.0 * np.abs(oh) * w
        keep = (oh > 0) & (i[..., 2] > zmin)
    else:
        i = _refract_dir(o, h, eta)
        ih = _dot(i, h)
        f = f_transmit(o, i, alpha, eta)
        den = oh + eta * ih
        val = f * np.abs(i[..., 2]) * den * den / (eta * eta * np.abs(ih)) * w
        keep = (oh > 0) & (-i[..., 2] > zmin)
    return np.where(keep & np.isfinite(val), val, 0.0)


def _breaks(phi, o, alpha, part, eta, zmin, m=512):
    """Per phi, the t in (0, 1) where a piece of the integrand starts or ends, sorted, padded with 1."""
    t = (np.arange(m) + 0.5) / m
    T, P = np.meshgrid(t, phi)

    def funcs(T, P):
        h, _ = _half(T, P, alpha)
        oh = _dot(o, h)
        out = [oh]
        ir = _reflect_dir(o, h)
        out += [ir[..., 2], ir[..., 2] - zmin]
        if eta is not None:
            c = np.clip(oh, -1, 1)
            out.append((1.0 / eta) * np.sqrt(np.maximum(0.0, 1.0 - c * c)) - 1.0)
            it = _refract_dir(o, h, eta)
            out += [np.nan_to_num(it[..., 2], nan=1.0), np.nan_to_num(-it[..., 2] - zmin, nan=-1.0)]
        return out

    found = [[] for _ in phi]
    for k, f in enumerate(funcs(T, P)):
        sc = (np.sign(f[:, :-1]) * np.sign(f[:, 1:])) < 0
        rows, cols = np.nonzero(sc)
        if len(rows) == 0:
            continue
        lo, hi = t[cols].copy(), t[cols + 1].copy()
        flo = f[rows, cols]
        for _ in range(45):   # bisection, all crossings at once
            mid = 0.5 * (lo + hi)
            fm = funcs(mid, phi[rows])[k]
            same = np.sign(fm) == np.sign(flo)
            lo = np.where(same, mid, lo); hi = np.where(same, hi, mid); flo = np.where(same, fm, flo)
        for r, b in zip(rows, 0.5 * (lo + hi)):
            found[r].append(b)
    K = max(len(x) for x in found)
    B = np.ones((len(phi), K))
    for r, x in enumerate(found):
        B[r, :len(x)] = sorted(x)
    return B


def albedo(theta_o_deg: float, alpha: float, part: str = "R", f0: float | None = None, eta: float | None = None,
           zmin: float = 0.0, n: int = 48) -> float:
    """Directional albedo of GGX width alpha seen from theta_o: part "R" (reflected) or "T" (transmitted), restricted to
    outgoing directions with |i.z| > zmin.  Metal: f0 (Schlick, no refraction); dielectric: eta (Schlick with total
    internal reflection).  n = Gauss-Legendre nodes per piece in t; 12 n nodes in phi over (0, pi), doubled by symmetry."""
    assert (f0 is None) != (eta is None) and part in ("R", "T") and (part == "R" or eta is not None)
    th = np.radians(theta_o_deg)
    o = np.array([np.sin(th), 0.0, np.cos(th)])
    fresnel = (lambda c: schlick(c, f0)) if f0 is not None else (lambda c: dielectric_fresnel(c, eta))
    xp, wp = np.polynomial.legendre.leggauss(12 * n)
    phi, wphi = 0.5 * PI * (xp + 1.0), 0.5 * PI * wp
    B = _breaks(phi, o, alpha, part, eta, zmin)
    edges = np.concatenate([np.zeros((len(phi), 1)), B, np.ones((len(phi), 1))], 1)   # (nphi, K + 2)
    xt, wt = np.polynomial.legendre.leggauss(n)
    a, b = edges[:, :-1, None], edges[:, 1:, None]                                       # pieces
    T = a + (b - a) * 0.5 * (xt + 1.0)
    W = (b - a) * 0.5 * wt
    P = np.broadcast_to(phi[:, None, None], T.shape)
    val = _integrand(T, P, o, alpha, part, fresnel, eta, zmin)
    return float(2.0 * np.sum(wphi[:, None, None] * W * val))


def converged(theta_o_deg, alpha, part="R", f0=None, eta=None, zmin=0.0, n=48):
    """(albedo at n, |albedo(2n) - albedo(n)|)."""
    a = albedo(theta_o_deg, alpha, part, f0, eta, zmin, n)
    return a, abs(albedo(theta_o_deg, alpha, part, f0, eta, zmin, 2 * n) - a)
