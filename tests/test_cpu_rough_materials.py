"""CPU tests of the GGX microfacet materials (DESIGN.md §5f): the rtb_add_rough_metal / rtb_add_rough_dielectric API, the
RTBS v5 blob and flatten hash, the plain oracle's refusal of v5, rtb_app's --obj-material / --alpha refusals, the float64
reference integral's own checks (tests/microfacet_reference.py), and the CPU restatement (tests/feature_oracle.cpp) against
that integral on the plane scenes the GPU tests use."""
import ctypes as C
import math
import subprocess
from pathlib import Path

import numpy as np
import pytest

import microfacet_reference as mr
from feature_oracle import FeatureOracleScene
from helpers import parse_blob

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "ray-tracing-v06_b200"
ERR_INVALID = -1
RTB_MAT_ROUGH_METAL, RTB_MAT_ROUGH_DIELECTRIC = 5, 6


# ------------------------------------------------------------------------------------------------ plane scenes
def half_sky(rows: int, white_rows: int, below: bool = False) -> np.ndarray:
    """An equirectangular map, 4 texels wide, whose first `white_rows` rows (from the top, +y) are white and the rest black
    (below=True: the other way round).  Row j ends at elevation 90 - 180 (j + 1) / rows degrees."""
    m = np.zeros((rows, 4, 3), np.float32)
    if below:
        m[rows - white_rows:] = 1.0
    else:
        m[:white_rows] = 1.0
    return m


def plane_scene(rtb, kind: str, theta_deg: float, alpha: float, f0=(1.0, 1.0, 1.0), ior=1.5, back=False, sky=None):
    """A 2000 x 2000 quad in y = 0 (normal +y, or -y with back=True, so that a ray from above meets its back face) of rough
    metal ("metal", F0 = f0) or rough glass ("glass"), seen at theta_deg from the normal by a camera 10 units away with a
    0.05-degree field: every pixel measures the directional albedo at theta.  sky: None = constant white background, else
    an environment map (unsampled)."""
    s = rtb.Scene()
    mat = s.rough_metal(f0, alpha) if kind == "metal" else s.rough_dielectric(ior, alpha)
    u, v = ((2000, 0, 0), (0, 0, 2000)) if back else ((0, 0, 2000), (2000, 0, 0))   # normal = cross(u, v) / |..|
    s.set_root(s.quad((-1000, 0, -1000), u, v, mat))
    if sky is None:
        s.set_background(rtb.BG_CONSTANT, (1.0, 1.0, 1.0))
    else:
        s.set_environment(sky)
    th = math.radians(theta_deg)
    cam = rtb.make_camera("pinhole", (10 * math.sin(th), 10 * math.cos(th), 0.0), (0, 0, 0), (0, 0, 1), 0.05, 1.0)
    return s, cam


def mean_and_error(sum_, sum2):
    """Per channel: the mean over every sample of the image, and one standard error of it (float64)."""
    n = float(sum_[..., 3].sum())
    s = sum_[..., :3].reshape(-1, 3).astype(np.float64).sum(0)
    q = sum2[..., :3].reshape(-1, 3).astype(np.float64).sum(0)
    m = s / n
    return m, np.sqrt(np.maximum(q / n - m * m, 0.0) / n)


# ------------------------------------------------------------------------------------------------ API and format
def test_api_refusals_leave_the_scene_unchanged(rtb):
    s = rtb.Scene()
    s.set_root(s.sphere((0, 0, 0), 1, s.lambertian((0.5, 0.5, 0.5))))
    before, h0, n0 = s.serialize(), s.flatten_hash(), len(parse_blob(s.serialize())[1])
    L = rtb.lib()
    f3 = lambda v: (C.c_float * 3)(*v)
    for bad in (np.nan, np.inf, -np.inf):
        assert L.rtb_add_rough_metal(s.handle, f3((0.5, bad, 0.5)), 0.3) == ERR_INVALID
        assert L.rtb_add_rough_metal(s.handle, f3((0.5, 0.5, 0.5)), bad) == ERR_INVALID
        assert L.rtb_add_rough_dielectric(s.handle, f3((1, 1, bad)), 1.5, 0.3) == ERR_INVALID
        assert L.rtb_add_rough_dielectric(s.handle, f3((1, 1, 1)), bad, 0.3) == ERR_INVALID
        assert L.rtb_add_rough_dielectric(s.handle, f3((1, 1, 1)), 1.5, bad) == ERR_INVALID
    for a in (0.0, 0.0009, -0.5, 1.0001, 2.0):
        assert L.rtb_add_rough_metal(s.handle, f3((1, 1, 1)), a) == ERR_INVALID
        assert L.rtb_add_rough_dielectric(s.handle, f3((1, 1, 1)), 1.5, a) == ERR_INVALID
    for ior in (0.0, -1.5):
        assert L.rtb_add_rough_dielectric(s.handle, f3((1, 1, 1)), ior, 0.3) == ERR_INVALID
    assert L.rtb_add_rough_metal(s.handle, None, 0.3) == ERR_INVALID
    assert L.rtb_add_rough_dielectric(s.handle, None, 1.5, 0.3) == ERR_INVALID
    assert L.rtb_add_rough_metal(None, f3((1, 1, 1)), 0.3) == ERR_INVALID
    assert s.serialize() == before and s.flatten_hash() == h0 and len(parse_blob(s.serialize())[1]) == n0
    with pytest.raises(rtb.RtbError):
        s.rough_metal((1, 1, 1), 1.5)
    assert s.serialize() == before
    # the ends of the range are accepted
    assert s.rough_metal((1, 1, 1), 0.001) >= 0 and s.rough_dielectric(1.5, 1.0) >= 0


def test_v5_blob_round_trip(rtb, orc):
    """v5 = the v4 content (empty light list, empty map record, no attributes), then n_materials and one width per material
    (0 for the other kinds).  The plain oracle refuses it; the feature oracle reads it back."""
    def build(rough):
        s = rtb.Scene()
        lam = s.lambertian((0.5, 0.5, 0.5))
        mats = [lam, s.metal((0.8, 0.8, 0.8), 0.1)]
        if rough:
            mats += [s.rough_metal((0.9, 0.6, 0.5), 0.25), s.rough_dielectric(1.33, 0.7, (1.0, 0.9, 0.9))]
        s.set_root(s.list([s.sphere((k, 0, 0), 0.4, m) for k, m in enumerate(mats)]))
        return s
    s, p = build(True), build(False)
    blob, plain = s.serialize(), p.serialize()
    h, mats, objs, _ = parse_blob(blob)
    assert h["version"] == 5 and parse_blob(plain)[0]["version"] == 1
    assert list(mats["kind"][2:]) == [RTB_MAT_ROUGH_METAL, RTB_MAT_ROUGH_DIELECTRIC]
    assert np.isclose(mats["param"][3], 1.33) and np.allclose(mats["albedo"][2], (0.9, 0.6, 0.5))
    body = 48 + 48 * int(h["n_textures"]) + 24 * int(h["n_materials"]) + 64 * int(h["n_objects"]) + 4 * int(h["n_children"]) + int(h["n_blob_bytes"])
    tail = blob[body:]
    assert len(tail) == 4 + 24 + 4 + 4 + 4 * 4
    assert np.frombuffer(tail[:4], np.int32)[0] == 0 and list(np.frombuffer(tail[4:16], np.int32)) == [0, 0, 0]
    assert np.frombuffer(tail[28:32], np.uint32)[0] == 0 and np.frombuffer(tail[32:36], np.uint32)[0] == 4
    assert np.array_equal(np.frombuffer(tail[36:], np.float32), np.float32([0, 0, 0.25, 0.7]))
    assert np.array_equal(FeatureOracleScene(blob).alphas(), np.float32([0, 0, 0.25, 0.7]))
    with pytest.raises(RuntimeError, match="version"):
        orc.OracleScene(blob)
    # the same geometry without the rough materials hashes differently only through them
    assert s.flatten_hash() != p.flatten_hash()
    # with a map, a light list and attributes too: the v4 content in full, then the widths
    s.set_environment(np.ones((2, 4, 3), np.float32))
    blob2 = s.serialize()
    assert parse_blob(blob2)[0]["version"] == 5 and len(blob2) == len(blob) + 2 * 4 * 3 * 4
    assert np.array_equal(FeatureOracleScene(blob2).alphas(), np.float32([0, 0, 0.25, 0.7]))


def test_alpha_changes_the_hash(rtb):
    hs = []
    for a in (0.2, 0.3):
        s = rtb.Scene(); s.set_root(s.sphere((0, 0, 0), 1, s.rough_metal((1, 1, 1), a))); hs.append(s.flatten_hash())
    assert hs[0] != hs[1]


@pytest.mark.parametrize("name", ["book2_bouncing", "book2_final", "mesh_icospheres"])
def test_scenes_without_rough_materials_keep_their_bytes(rtb, name):
    """Registry scenes serialise as before (v1) and are read by the feature oracle's loader; adding a material of another
    kind keeps v1."""
    s = rtb.Scene.named(name)
    blob = s.serialize()
    assert parse_blob(blob)[0]["version"] == 1
    assert np.all(FeatureOracleScene(blob).alphas() == 0)


def test_app_option_refusals(rtb, tmp_path):
    app = str(PKG / "rtb_app")
    obj = tmp_path / "m.obj"
    obj.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    (tmp_path / "t.ppm").write_bytes(b"P6\n2 1\n255\n" + bytes(6))
    cases = [
        (["--obj-material", "rough-metal"], "--obj"),
        (["--alpha", "0.3"], "--obj"),
        (["--obj", str(obj), "--alpha", "0.3"], "--alpha"),
        (["--obj", str(obj), "--obj-material", "clay", "--alpha", "0.3"], "--alpha"),
        (["--obj", str(obj), "--obj-material", "gold"], "--obj-material"),
        (["--obj", str(obj), "--obj-material", "rough-glass", "--alpha", "0"], "--alpha"),
        (["--obj", str(obj), "--obj-material", "rough-glass", "--alpha", "1.5"], "--alpha"),
        (["--obj", str(obj), "--smooth", "--obj-texture", str(tmp_path / "t.ppm"), "--obj-material", "rough-metal"], "--obj-texture"),
    ]
    for args, word in cases:
        r = subprocess.run([app] + args, capture_output=True, text=True)
        assert r.returncode == 1 and word in r.stderr, (args, r.stderr)


# ------------------------------------------------------------------------------------------------ the reference integral
def test_reference_smooth_limits():
    """E_R(alpha -> 0, F0 = 1) -> 1; for the dielectric E_R + E_T -> 1 as alpha -> 0 (no 1 / eta^2 factor)."""
    for th in (0.0, 45.0, 75.0):
        assert abs(mr.albedo(th, 0.001, "R", f0=1.0) - 1.0) < 1e-5
        for eta in (1.5, 1 / 1.5):
            tot = mr.albedo(th, 0.001, "R", eta=eta) + mr.albedo(th, 0.001, "T", eta=eta)
            assert abs(tot - 1.0) < 1e-5, (th, eta, tot)


def test_reference_known_value():
    """alpha = 1, F0 = 1, normal incidence: D = 1 / pi, G2 = 2 cos / (1 + cos), E_R = int_0^1 c / (1 + c) dc = 1 - ln 2."""
    assert abs(mr.albedo(0.0, 1.0, "R", f0=1.0) - (1.0 - math.log(2.0))) < 1e-9


def test_reference_reciprocity():
    rng = np.random.default_rng(5)
    def dirs(n, up):
        v = rng.normal(size=(n, 3)); v /= np.linalg.norm(v, axis=1, keepdims=True)
        v[:, 2] = np.abs(v[:, 2]) * (1 if up else -1)
        return v
    o, i, d = dirs(500, True), dirs(500, True), dirs(500, False)
    for a in (0.05, 0.3, 1.0):
        f = lambda c: mr.schlick(c, 0.3)
        assert np.allclose(mr.f_reflect(o, i, a, f), mr.f_reflect(i, o, a, f), rtol=1e-12)
        for eta in (1.5, 1 / 1.5):
            # radiance form: f_t(o -> d) / eta_d^2 = f_t(d -> o) / eta_o^2, the Fresnel factor aside (Schlick is not symmetric)
            fwd = mr.f_transmit(o, d, a, eta, fresnel=False) / eta ** 2
            bwd = mr.f_transmit(-d, -o, a, 1 / eta, fresnel=False)
            assert np.allclose(fwd, bwd, rtol=1e-10), (a, eta)


@pytest.mark.parametrize("theta", [0.0, 45.0, 75.0])
@pytest.mark.parametrize("alpha", [0.05, 0.2, 0.5, 1.0])
def test_reference_converges(theta, alpha):
    """Doubling the rule changes E_R, E_T by less than 1e-5; restricted to |i.z| > z_min (a jump across the lobe) by less
    than 5e-4."""
    for kw in (dict(part="R", f0=1.0), dict(part="R", eta=1.5), dict(part="T", eta=1.5), dict(part="T", eta=1 / 1.5)):
        _, err = mr.converged(theta, alpha, n=48, **kw)
        assert err < 1e-5, (kw, err)
    _, err = mr.converged(theta, alpha, part="R", f0=1.0, zmin=0.5, n=48)
    assert err < 5e-4


# ------------------------------------------------------------------------------------------------ oracle against the integral
@pytest.mark.parametrize("kind,alpha,theta,back", [("metal", 0.3, 45.0, False), ("metal", 1.0, 0.0, False),
                                                   ("glass", 0.3, 45.0, False), ("glass", 0.5, 30.0, True)])
def test_oracle_matches_the_integral(rtb, kind, alpha, theta, back):
    """The CPU restatement on the white-sky plane (E_R for the metal, E_R + E_T for the glass) within 4 sigma."""
    s, cam = plane_scene(rtb, kind, theta, alpha, back=back)
    W, S = 8, 512
    sum_, sum2, _ = FeatureOracleScene(s.serialize()).render(cam, W, W, 0, S, 2, seed=3, want_sum2=True)
    m, e = mean_and_error(sum_, sum2)
    if kind == "metal":
        want = mr.albedo(theta, alpha, "R", f0=1.0)
    else:
        eta = 1 / 1.5 if back else 1.5
        want = mr.albedo(theta, alpha, "R", eta=eta) + mr.albedo(theta, alpha, "T", eta=eta)
    assert np.all(np.abs(m - want) <= 4 * e + 1e-5), (m, e, want)
