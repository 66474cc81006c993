"""TEST INFRASTRUCTURE: the mesh scenes and hand-derived answers shared by tests/test_cpu_mesh_attributes.py and
tests/test_gpu_mesh_attributes.py (DESIGN.md §5e).  Nothing here renders: the tests render these scenes on the CPU oracle
(tests/mesh_oracle.py) and on the GPU."""
from __future__ import annotations

import numpy as np

# ------------------------------------------------------------------------------------------------ one triangle
# v0 = (-1, -1, 0), v1 = (1, -1, 0), v2 = (-1, 1, 0): u = v1 - v0 and v = v2 - v0 are (2, 0, 0) and (0, 2, 0), the face
# normal N is +z, and the point of planar coordinates (alpha, beta) is v0 + alpha u + beta v.
TRI_V = np.float32([[-1, -1, 0], [1, -1, 0], [-1, 1, 0]])
TRI_N = np.float32([[0.3, 0.2, 1.0], [-0.2, 0.1, 1.0], [0.1, -0.4, 1.0]])      # leaning normals on N's side (not unit)
TRI_UV = np.float32([[0.1, 0.2], [0.9, 0.3], [0.2, 0.8]])
# vertices, edge midpoints, centroid
POINTS = [(0.0, 0.0), (1.0, 0.0), (0.0, 1.0), (0.5, 0.0), (0.0, 0.5), (0.5, 0.5), (1 / 3, 1 / 3)]
ROT_DEG, OFFSET = 90.0, (1.0, 2.0, 3.0)


def triangle_scene(rtb, normals=True, flip=False, uvs=True, instanced=False):
    """The triangle with its attributes (flip: every vertex normal negated, so they disagree with the winding), optionally
    under rotate_y(90) + translate(OFFSET)."""
    s = rtb.Scene()
    n = None if not normals else (-TRI_N if flip else TRI_N)
    m = s.mesh(TRI_V, np.int32([[0, 1, 2]]), s.lambertian((0.5, 0.5, 0.5)), normals=n, uvs=TRI_UV if uvs else None)
    if instanced:
        m = s.translate(s.rotate_y(m, ROT_DEG), OFFSET)
    s.set_root(m)
    return s


def _rot(v):
    """World from object of rotate_y(90): (x, y, z) -> (z, y, -x)."""
    v = np.asarray(v, np.float64)
    return np.stack([v[..., 2], v[..., 1], -v[..., 0]], -1)


def triangle_rays(rtb, instanced=False, inset=1e-4):
    """Rays along -z (front) and +z (back) of the object frame through every point of POINTS, moved the fraction `inset`
    towards the centroid (a ray exactly on the edge of the box may miss it); returns (rays, the (alpha, beta) of each, and whether it comes from the back)."""
    pts = [(a + inset * (1 / 3 - a), b + inset * (1 / 3 - b)) for a, b in POINTS]
    rays = np.zeros(2 * len(pts), rtb.RAY_DTYPE)
    ab, back = [], []
    for k, (a, b) in enumerate(pts):
        p = TRI_V[0].astype(np.float64) + a * (TRI_V[1] - TRI_V[0]) + b * (TRI_V[2] - TRI_V[0])
        for side, (z, dz) in enumerate(((3.0, -1.0), (-3.0, 1.0))):
            o, d = np.array([p[0], p[1], z]), np.array([0.0, 0.0, dz])
            if instanced:
                o, d = _rot(o) + np.array(OFFSET), _rot(d)
            rays[2 * k + side]["o"] = o; rays[2 * k + side]["d"] = d
            ab.append((a, b)); back.append(side == 1)
    return rays, np.array(ab), np.array(back)


def expected_attributes(ab, back, normals=True, uvs=True, instanced=False):
    """§5e in float64: the shading normal (facing the ray) and the (u, v) at planar coordinates ab."""
    a, b = ab[:, 0], ab[:, 1]
    w = 1.0 - a - b
    N = np.array([0.0, 0.0, 1.0])
    if normals:
        n = TRI_N.astype(np.float64) / np.linalg.norm(TRI_N.astype(np.float64), axis=1, keepdims=True)
        m = w[:, None] * n[0] + a[:, None] * n[1] + b[:, None] * n[2]
        m /= np.linalg.norm(m, axis=1, keepdims=True)
        m[(m @ N) < 0] *= -1
    else:
        m = np.tile(N, (len(a), 1))
    ns = np.where(back[:, None], -m, m)
    uv = (w[:, None] * TRI_UV[0] + a[:, None] * TRI_UV[1] + b[:, None] * TRI_UV[2]) if uvs else np.stack([a, b], -1)
    return (_rot(ns) if instanced else ns), uv


# ------------------------------------------------------------------------------------------------ icospheres

def icosphere(subdivisions):
    """Unit icosphere (the registry's construction): vertices on the sphere, faces wound outwards."""
    t = (1 + 5 ** 0.5) / 2
    v = [np.array(p, np.float64) / np.linalg.norm(p) for p in
         [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t), (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6), (7, 1, 8),
         (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    for _ in range(subdivisions):
        mid, nf = {}, []

        def midpoint(a, b):
            key = (min(a, b), max(a, b))
            if key not in mid:
                p = (v[a] + v[b]) / 2
                v.append(p / np.linalg.norm(p)); mid[key] = len(v) - 1
            return mid[key]
        for a, b, c in f:
            ab, bc, ca = midpoint(a, b), midpoint(b, c), midpoint(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    return np.array(v, np.float32), np.array(f, np.int32)


def sphere_uvs(v):
    """The sphere-texture (u, v) of unit positions (book get_sphere_uv)."""
    theta = np.arccos(np.clip(-v[:, 1], -1, 1)); phi = np.arctan2(-v[:, 2], v[:, 0]) + np.pi
    return np.stack([phi / (2 * np.pi), theta / np.pi], -1).astype(np.float32)


def unshared(v, f):
    """Every face with vertices of its own (so that per-face attributes can differ)."""
    return v[f.reshape(-1)], np.arange(f.size, dtype=np.int32).reshape(-1, 3)


def checker_image(w=16, h=8):
    j, i = np.mgrid[0:h, 0:w]
    img = np.zeros((h, w, 3), np.uint8)
    img[..., 0] = 40 + 200 * ((i + j) % 2); img[..., 1] = 10 * i; img[..., 2] = 255 - 20 * j
    return img


def furnace_scene(rtb, smooth=True, subdivisions=2):
    """A white Lambertian icosphere under a uniform white sky: every path that leaves returns exactly 1."""
    s = rtb.Scene()
    v, f = icosphere(subdivisions)
    s.set_root(s.mesh(v, f, s.lambertian((1.0, 1.0, 1.0)), normals=v if smooth else None))
    s.set_background(rtb.BG_CONSTANT, (1.0, 1.0, 1.0))
    cam = rtb.make_camera("pinhole", (0, 0.5, 3.5), (0, 0, 0), (0, 1, 0), 40.0, 1.0)
    return s, cam


def canonical_uv_scene(rtb, with_uvs):
    """An image-textured icosphere with unshared faces; with_uvs: every face carries (0,0), (1,0), (0,1), which §5e maps to
    exactly (alpha, beta) - the image then reads what the plain mesh reads."""
    s = rtb.Scene()
    v, f = unshared(*icosphere(1))
    uvs = np.tile(np.float32([[0, 0], [1, 0], [0, 1]]), (len(f), 1)) if with_uvs else None
    s.set_root(s.list([s.mesh(v, f, s.lambertian(tex=s.image(checker_image())), uvs=uvs),
                       s.quad((-4, -1, -4), (8, 0, 0), (0, 0, 8), s.lambertian((0.4, 0.5, 0.3)))]))
    cam = rtb.make_camera("pinhole", (0.4, 0.8, 3.2), (0, 0, 0), (0, 1, 0), 40.0, 1.5)
    return s, cam


def parity_scene(rtb, kind):
    """Scenes for path-for-path parity with the oracle.
      textured     smooth, UV-mapped image-textured icosphere on a ground (the deferred-texture path)
      glass_metal  smooth dielectric and metal icospheres, instanced (rotate_y + translate), a noise-textured ground
      lights       a smooth icosphere under a sampled quad light (LIGHTS x ATTR)
      env          a smooth icosphere under a sampled environment map (ENV x ATTR)
      media        a smooth icosphere next to a constant medium (MEDIA x ATTR)"""
    s = rtb.Scene()
    v, f = icosphere(2)
    ground = s.quad((-6, -1, -6), (12, 0, 0), (0, 0, 12), s.lambertian((0.5, 0.55, 0.45)))
    cam = rtb.make_camera("pinhole", (0.3, 1.0, 4.2), (0, 0, 0), (0, 1, 0), 45.0, 1.5)
    if kind == "textured":
        m = s.mesh(v, f, s.lambertian(tex=s.image(checker_image())), normals=v, uvs=sphere_uvs(v))
        s.set_root(s.list([ground, m]))
    elif kind == "glass_metal":
        g = s.mesh(v, f, s.dielectric(1.5), normals=v)
        mt = s.mesh(v, f, s.metal((0.8, 0.7, 0.6), 0.05), normals=v)
        noise_ground = s.quad((-6, -1, -6), (12, 0, 0), (0, 0, 12), s.lambertian(tex=s.noise(2.0)))
        s.set_root(s.list([noise_ground, s.translate(s.rotate_y(g, 30.0), (-0.9, 0, 0)), s.translate(s.rotate_y(mt, -50.0), (1.2, 0, -0.5))]))
    elif kind == "lights":
        m = s.mesh(v, f, s.lambertian((0.7, 0.6, 0.5)), normals=v)
        lamp = s.quad((-0.5, 2.5, -0.5), (1, 0, 0), (0, 0, 1), s.diffuse_light(s.solid((8, 8, 8))))
        s.set_root(s.list([ground, m, lamp]))
        s.set_background(rtb.BG_CONSTANT, (0.05, 0.05, 0.08))
        s.sample_lights([lamp])
    elif kind == "env":
        m = s.mesh(v, f, s.lambertian((0.7, 0.6, 0.5)), normals=v)
        s.set_root(s.list([ground, m]))
        j, i = np.mgrid[0:16, 0:32]
        sky = np.stack([0.3 + 0.02 * i, 0.4 + 0.01 * j, np.where(j < 8, 1.2, 0.2)], -1).astype(np.float32)
        sky[3, 5] = 40.0
        s.set_environment(sky, sample=True)
    elif kind == "media":
        m = s.mesh(v, f, s.lambertian((0.7, 0.6, 0.5)), normals=v)
        fog = s.constant_medium(s.sphere((1.6, 0, 0.3), 0.7, s.lambertian((1, 1, 1))), 1.5, s.isotropic(s.solid((0.9, 0.9, 0.9))))
        s.set_root(s.list([ground, m, fog]))
    else:
        raise ValueError(kind)
    return s, cam


PARITY_KINDS = ("textured", "glass_metal", "lights", "env", "media")


def height_field(rtb, n, smooth=True):
    """tools/bvh_build_bench.py's height field (2 n^2 triangles over [-1, 1]^2) with its analytic normals."""
    s = rtb.Scene()
    xs = np.linspace(-1, 1, n + 1, dtype=np.float32)
    X, Z = np.meshgrid(xs, xs, indexing="ij")
    Y = (0.08 * np.sin(9 * X) * np.cos(7 * Z) + 0.03 * np.sin(31 * X + 17 * Z)).astype(np.float32)
    dX = 0.72 * np.cos(9 * X) * np.cos(7 * Z) + 0.93 * np.cos(31 * X + 17 * Z)
    dZ = -0.56 * np.sin(9 * X) * np.sin(7 * Z) + 0.51 * np.cos(31 * X + 17 * Z)
    P = np.stack([X, Y, Z], axis=-1).reshape(-1, 3)
    N = np.stack([-dX, np.ones_like(dX), -dZ], axis=-1).reshape(-1, 3).astype(np.float32)
    uv = np.stack([(X + 1) / 2, (Z + 1) / 2], axis=-1).reshape(-1, 2).astype(np.float32)
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    v00 = (i * (n + 1) + j).ravel(); v10 = v00 + (n + 1); v01 = v00 + 1; v11 = v10 + 1
    tris = np.concatenate([np.stack([v00, v10, v01], axis=1), np.stack([v11, v10, v01], axis=1)]).astype(np.int32)
    return s, P, tris, (N if smooth else None), uv


def height_field_scene(rtb, n, variant):
    """variant: flat, smooth, or textured (smooth + an image mapped through the UVs)."""
    s, P, tris, N, uv = height_field(rtb, n, smooth=variant != "flat")
    mat = s.lambertian(tex=s.image(checker_image(64, 64))) if variant == "textured" else s.lambertian((0.6, 0.55, 0.5))
    ids = [s.mesh(P, tris, mat, normals=N, uvs=uv if variant == "textured" else None), s.sphere((0.0, 0.35, 0.0), 0.25, s.dielectric(1.5))]
    s.set_root(s.list(ids))
    cam = rtb.make_camera("pinhole", (1.6, 1.1, 1.9), (0, 0, 0), (0, 1, 0), 40.0, 1.0)
    return s, cam
