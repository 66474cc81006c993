"""CPU tests of the HDR environment map (DESIGN.md §5d): the rtb_scene_set_environment API, the RTBS v3 blob, the flatten
hash, the map's sampler and pdf on the CPU restatement (tests/env_oracle.cpp), and the hand-derived answers rendered on
that restatement: a 1 x 1 map is the constant background, the axis directions read the tabulated texels, one lit texel
gives its irradiance integral, and the white furnace returns exactly 1."""
import ctypes as C

import numpy as np
import pytest
from scipy import stats

import env_scenes as es
from env_oracle import EnvOracleScene
from helpers import parse_blob
from light_oracle import LightOracleScene

ERR_INVALID = -1


def _set(rtb, s, rgb, w, h, scale=(1, 1, 1), flags=0):
    ptr = None if rgb is None else np.ascontiguousarray(rgb, np.float32).ctypes.data
    return rtb.lib().rtb_scene_set_environment(s.handle, ptr, w, h, (C.c_float * 3)(*scale), flags)


def test_api_validation(rtb):
    s, _ = es.sky_scene(rtb)
    before, h0 = s.serialize(), s.flatten_hash()
    good = np.ones((2, 4, 3), np.float32)
    refused = [
        (good, 0, 2, (1, 1, 1), 0), (good, 4, 0, (1, 1, 1), 0), (good, -4, 2, (1, 1, 1), 0),
        (np.ones((1, 16385, 3), np.float32), 16385, 1, (1, 1, 1), 0),
        (None, 4, 2, (1, 1, 1), 0),
        (good, 4, 2, (1, 1, 1), 2), (good, 4, 2, (1, 1, 1), -1),                         # unknown flags
        (good, 4, 2, (1, -1, 1), 0), (good, 4, 2, (1, float("nan"), 1), 0), (good, 4, 2, (float("inf"), 1, 1), 0),
        (np.zeros((2, 4, 3), np.float32), 4, 2, (1, 1, 1), rtb.ENV_SAMPLE),              # nothing to sample
        (good, 4, 2, (0, 0, 0), rtb.ENV_SAMPLE),
        (None, 0, 0, (1, 1, 1), 4),
    ]
    for bad in (-1.0, float("nan"), float("inf")):
        m = good.copy(); m[1, 2, 1] = bad
        refused.append((m, 4, 2, (1, 1, 1), 0))
    for rgb, w, h, scale, flags in refused:
        assert _set(rtb, s, rgb, w, h, scale, flags) == ERR_INVALID, (w, h, scale, flags)
        assert s.serialize() == before and s.flatten_hash() == h0
    # the size bound: 2^24 texels pass the size check (a 16384 x 1024 map), one row more does not
    assert _set(rtb, s, None, 16384, 1025, (1, 1, 1), 0) == ERR_INVALID
    big = np.zeros((1024, 16384, 3), np.float32)
    assert _set(rtb, s, big, 16384, 1024) == 0
    assert _set(rtb, s, None, 0, 0) == 0
    # zero weights are fine without sampling; a black map with the sampling flag is not
    assert _set(rtb, s, np.zeros((2, 4, 3), np.float32), 4, 2) == 0
    with pytest.raises(rtb.RtbError, match="all zero"):
        s.set_environment(np.zeros((2, 4, 3), np.float32), sample=True)
    with pytest.raises(ValueError):
        s.set_environment(np.ones((4, 3), np.float32))
    s.set_environment(None)
    assert s.serialize() == before and s.flatten_hash() == h0


def test_blob_round_trips(rtb, orc):
    """Without a map: v1 / v2 byte for byte.  With one: v3 = the v1 body, the light list (n may be 0), rtbs_env and the
    scaled texels; setting then clearing restores the bytes and the flatten hash; the plain and light oracles refuse v3."""
    s = rtb.Scene.named("book2_final")
    v1, h1 = s.serialize(), s.flatten_hash()
    m = es.distinct_map(6, 4)
    s.set_environment(m, scale=(2.0, 0.5, 1.0), sample=True)
    v3 = s.serialize()
    assert parse_blob(v3)[0]["version"] == 3
    assert v3[:4] == v1[:4] and v3[8:len(v1)] == v1[8:]
    tail = v3[len(v1):]
    assert np.frombuffer(tail[:4], np.int32)[0] == 0
    env = np.frombuffer(tail[4:16], np.int32)
    assert list(env) == [6, 4, rtb.ENV_SAMPLE]
    assert np.array_equal(np.frombuffer(tail[16:28], np.float32), np.float32([2.0, 0.5, 1.0]))
    texels = np.frombuffer(tail[28:], np.float32).reshape(4, 6, 3)
    assert np.array_equal(texels, m * np.float32([2.0, 0.5, 1.0]))
    h3 = s.flatten_hash()
    assert h3 != h1
    s.set_environment(m, scale=(2.0, 0.5, 1.0), sample=False)
    assert s.flatten_hash() not in (h1, h3)                     # the sampling flag is part of the flattened scene
    for oracle in (orc.OracleScene, LightOracleScene):
        with pytest.raises(RuntimeError, match="version"):
            oracle(v3)
    assert EnvOracleScene(v3).dims() == (6, 4)
    s.sample_lights(s.info.light_ids)                           # lights and a map: the list, then the map
    v3l = s.serialize()
    n = len(s.info.light_ids)
    assert np.array_equal(np.frombuffer(v3l[len(v1):len(v1) + 4 + 4 * n], np.int32), np.int32([n, *s.info.light_ids]))
    s.set_environment(None)
    assert parse_blob(s.serialize())[0]["version"] == 2
    s.sample_lights([])
    assert s.serialize() == v1 and s.flatten_hash() == h1


# ------------------------------------------------------------------------------------------------ the sampler

def _sampling_map(rng, W=8, H=5):
    m = rng.uniform(0.0, 2.0, size=(H, W, 3)).astype(np.float32)
    m[1, 2] = 0.0                                               # a black texel is never drawn
    m[3, :] *= 5.0
    return m


def _env(rtb, m, sample=True, scale=(1, 1, 1)):
    s = rtb.Scene()
    s.set_root(s.sphere((0, 0, 0), 1.0, s.lambertian((0.5, 0.5, 0.5))))
    s.set_environment(m, scale=scale, sample=sample)
    return EnvOracleScene(s.serialize())


def test_tables(rtb):
    """The CDFs start at 0 and end at exactly 1, are non-decreasing, and a texel's probability follows its weight
    luminance x sin(theta of the row centre)."""
    rng = np.random.default_rng(1)
    m = _sampling_map(rng)
    H, W = m.shape[:2]
    num, cm, cc = _env(rtb, m, scale=(1.0, 2.0, 0.5)).tables()
    assert cm[0] == 0 and cm[-1] == 1 and np.all(np.diff(cm) >= 0)
    assert np.all(cc[:, 0] == 0) and np.all(cc[:, -1] == 1) and np.all(np.diff(cc, axis=1) >= 0)
    p = (np.diff(cm.astype(np.float64))[:, None] * np.diff(cc.astype(np.float64), axis=1))
    assert np.allclose(num, p * W * H / (2 * np.pi ** 2), rtol=1e-6, atol=0)
    ms = m.astype(np.float64) * np.float32([1.0, 2.0, 0.5]).astype(np.float32)
    w = (0.2126 * ms[..., 0] + 0.7152 * ms[..., 1] + 0.0722 * ms[..., 2]) * np.sin(np.pi * (np.arange(H) + 0.5) / H)[:, None]
    assert np.allclose(p, w / w.sum(), rtol=1e-5, atol=1e-7)
    assert p[1, 2] == 0


def test_sampled_texels_follow_their_probabilities(rtb):
    """chi-square: the texels of many drawn directions against p_ij."""
    rng = np.random.default_rng(2)
    m = _sampling_map(rng)
    H, W = m.shape[:2]
    e = _env(rtb, m)
    num, cm, cc = e.tables()
    p = (np.diff(cm.astype(np.float64))[:, None] * np.diff(cc.astype(np.float64), axis=1)).reshape(-1)
    N = 400_000
    _, texel, _ = e.sample(rng.random((N, 2), dtype=np.float32))
    counts = np.bincount(texel, minlength=W * H)
    assert counts[np.flatnonzero(p == 0)].sum() == 0
    nz = p > 0
    chi2 = float((((counts[nz] - N * p[nz]) ** 2) / (N * p[nz])).sum())
    pval = float(stats.chi2.sf(chi2, nz.sum() - 1))
    print(f"chi2 {chi2:.1f} on {nz.sum() - 1} dof, p = {pval:.3f}")
    assert pval > 1e-3


def test_pdf_of_a_sample_is_its_texel_density(rtb):
    """pdf(sample(z)) = p_ij W H / (2 pi^2 sin theta), (i, j) the lookup's texel, theta of the direction."""
    rng = np.random.default_rng(3)
    m = _sampling_map(rng)
    H, W = m.shape[:2]
    e = _env(rtb, m)
    num, cm, cc = e.tables()
    d, texel, pdf = e.sample(rng.random((20_000, 2), dtype=np.float32))
    assert np.allclose(np.linalg.norm(d.astype(np.float64), axis=1), 1.0, atol=1e-6)
    p = (np.diff(cm.astype(np.float64))[:, None] * np.diff(cc.astype(np.float64), axis=1)).reshape(-1)
    sin_t = np.sqrt(d[:, 0].astype(np.float64) ** 2 + d[:, 2].astype(np.float64) ** 2)
    want = p[texel] * W * H / (2 * np.pi ** 2 * sin_t)
    assert np.allclose(pdf, want, rtol=1e-5)
    t2, p2 = e.lookup(d)                                          # the lookup of the same direction agrees
    assert np.array_equal(t2, texel) and np.array_equal(p2, pdf)


def test_pdf_integrates_to_one(rtb):
    rng = np.random.default_rng(4)
    m = _sampling_map(rng, 16, 9)
    e = _env(rtb, m)
    N = 400_000
    d = rng.normal(size=(N, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    _, pdf = e.lookup(d.astype(np.float32))
    vals = 4 * np.pi * pdf.astype(np.float64)
    mean, sigma = vals.mean(), vals.std() / np.sqrt(N)
    print(f"integral of the pdf {mean:.5f} +- {sigma:.5f}")
    assert abs(mean - 1.0) <= 3 * sigma


def test_axis_directions_read_the_tabulated_texels(rtb):
    for W, H in ((es.OW, es.OH), (7, 5), (33, 17)):
        e = _env(rtb, es.distinct_map(W, H), sample=False)
        tex, _ = e.lookup(np.float32([es.AXES[a] for a in es.AXES]))
        for a, t in zip(es.AXES, tex):
            i, j = es.axis_texels(W, H)[a]
            assert t == j * W + i, (W, H, a, divmod(int(t), W), (j, i))


# ------------------------------------------------------------------------------------------------ known answers (oracle)

def test_one_by_one_map_is_the_constant_background(rtb):
    s, cam = es.sky_scene(rtb)
    a, a2, ra = EnvOracleScene(s.serialize()).render(cam, 24, 16, 0, 8, 12, seed=3, want_sum2=True)
    s.set_environment(np.float32(es.SKY).reshape(1, 1, 3))
    b, b2, rb = EnvOracleScene(s.serialize()).render(cam, 24, 16, 0, 8, 12, seed=3, want_sum2=True)
    assert np.array_equal(a, b) and np.array_equal(a2, b2) and ra == rb
    assert (a[..., 2] > 0).all()


def test_orientation_on_the_oracle(rtb):
    want = es.orientation_map()
    s = es.orientation_scene(rtb)
    o = EnvOracleScene(s.serialize())
    for axis, (i, j) in es.axis_texels().items():
        a, _, _ = o.render(es.orientation_camera(rtb, axis), 1, 1, 0, 16, 4, seed=1)
        assert np.array_equal(a[0, 0, :3] / 16, want[j, i]), (axis, a[0, 0], want[j, i])


def check_mean(sums, sums2, spp, want, label, k=4.0):
    n = float(spp)
    m = sums[..., :3].astype(np.float64) / n
    var = np.maximum(sums2[..., :3].astype(np.float64) / n - m ** 2, 0.0) / n
    err = float((m - want).mean()); sigma = float(np.sqrt(var.sum()) / var.size)
    print(f"{label}: mean {m.mean():.6f} expected {np.mean(want):.6f} error/sigma {err / max(sigma, 1e-30):+.2f}")
    assert abs(err) <= k * sigma, (label, err, sigma)
    return float(var.mean() * n)


def test_one_texel_irradiance_on_the_oracle(rtb):
    want = es.one_texel_expected()
    var = {}
    for sample in (False, True):
        s, cam = es.one_texel_scene(rtb, sample)
        a, a2, _ = EnvOracleScene(s.serialize()).render(cam, 8, 8, 0, 2048, 2, seed=5 + sample, want_sum2=True)
        var[sample] = check_mean(a, a2, 2048, want, f"oracle one texel sample={sample}")
    print(f"variance sampled / unsampled {var[True] / var[False]:.3f}")
    assert var[True] <= 0.25 * var[False]


def test_furnace_on_the_oracle(rtb):
    s, cam = es.furnace_scene(rtb, False)
    a, _, _ = EnvOracleScene(s.serialize()).render(cam, 16, 16, 0, 64, 8, seed=7)
    assert np.array_equal(a[..., :3], np.full((16, 16, 3), 64.0, np.float32))
    s, cam = es.furnace_scene(rtb, True)
    a, a2, _ = EnvOracleScene(s.serialize()).render(cam, 16, 16, 0, 1024, 8, seed=7, want_sum2=True)
    check_mean(a, a2, 1024, 1.0, "oracle furnace sampled", k=3.0)


def test_rtb_app_refuses_bad_env_arguments(tmp_path):
    """rtb_app --env: a missing file, a file that is not a PFM, a truncated PFM and --sample-env without a map all exit 1
    before anything is rendered."""
    import subprocess
    from conftest import ROOT
    app = str(ROOT / "ray-tracing-v06_b200" / "rtb_app")
    (tmp_path / "junk.pfm").write_bytes(b"P6\n2 2\n255\n" + bytes(12))
    (tmp_path / "short.pfm").write_bytes(b"PF\n4 2\n-1.0\n" + bytes(40))
    for args, msg in ((["--env", str(tmp_path / "none.pfm")], "cannot open"), (["--env", str(tmp_path / "junk.pfm")], "not a PFM"),
                      (["--env", str(tmp_path / "short.pfm")], "truncated"), (["--sample-env"], "needs --env")):
        out = subprocess.run([app, "book2_cornell", *args], capture_output=True, text=True)
        assert out.returncode == 1 and msg in out.stderr, (args, out.stderr)


SMALL_OBJ = "v 0 0 0\nv 1 0 0\nv 0 1 0\nv 0 0 1\nf 1 3 2\nf 1 2 4\nf 1 4 3\nf 2 3 4\n"


def write_pfm(path, rgb):
    """rgb (H, W, 3), row 0 = top -> a little-endian PFM (rows bottom-up)."""
    H, W = rgb.shape[:2]
    with open(path, "wb") as f:
        f.write(f"PF\n{W} {H}\n-1.0\n".encode())
        f.write(np.ascontiguousarray(np.flipud(rgb), dtype="<f4").tobytes())


def test_rtb_app_applies_env_to_obj_scenes(tmp_path):
    """--obj builds its world through the host mirror: the map reaches that scene too (a black map with --sample-env is
    refused there, before anything is rendered)."""
    import subprocess
    from conftest import ROOT
    app = str(ROOT / "ray-tracing-v06_b200" / "rtb_app")
    (tmp_path / "m.obj").write_text(SMALL_OBJ)
    write_pfm(tmp_path / "black.pfm", np.zeros((4, 8, 3), np.float32))
    out = subprocess.run([app, "--obj", str(tmp_path / "m.obj"), "--env", str(tmp_path / "black.pfm"), "--sample-env"],
                         capture_output=True, text=True)
    assert out.returncode == 1 and "all zero" in out.stderr, out.stderr
