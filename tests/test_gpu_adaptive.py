"""GPU tests of adaptive sampling (rtb_render_adaptive, DESIGN.md §5c).  The uniform renders are pinned to the CPU oracle
elsewhere; here every adaptive result is pinned to them: a pixel that stopped after n samples must hold, bit for bit, the
sums a dense progressive render holds after n samples, and the pixels each round renders must be exactly the ones the
float32 restatement in tests/adaptive_rule.py predicts from the accumulators."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import adaptive_rule as ar
from conftest import ROOT
from helpers import psnr, tonemap

pytestmark = pytest.mark.gpu

BUDGET = 64 << 20   # the default batch path budget (RTB_BATCH_PATHS unset, a B200 has the memory for it)


def _renderer(rtb, name, lights=False):
    s = rtb.Scene.named(name)
    if lights:
        s.sample_lights(s.info.light_ids)
    r = rtb.Renderer(0); r.set_scene(s); r.set_camera(s.info.camera)
    return r, s


def _dense_snapshots(rtb, r, W, H, D, seed, cursors, rows, spb):
    """Dense progressive renders over [cursors[i], cursors[i + 1]): {cursor: (accum, accum2)} after each call."""
    snaps = {0: (np.zeros((H, W, 4), np.float32), np.zeros((H, W, 4), np.float32))}
    for c0, c1 in zip(cursors[:-1], cursors[1:]):
        r.render(W, H, c0, c1, D, seed=seed, clear=(c0 == 0), variance=True, rows=rows, samples_per_batch=spb)
        snaps[c1] = r.download_accum(want_sum2=True)
    return snaps


def _expect_per_pixel(snaps, a, q, rows, H):
    """Every pixel of the row range holds the dense values at its own count; rows outside are untouched (zero)."""
    r0, r1 = (0, H) if tuple(rows) == (0, 0) else rows
    counts = a[..., 3]
    for c in np.unique(counts[r0:r1]):
        assert int(c) in snaps, f"count {c} is not a round boundary"
        sel = np.zeros(counts.shape, bool); sel[r0:r1] = counts[r0:r1] == c
        da, dq = snaps[int(c)]
        assert np.array_equal(a[sel], da[sel]) and np.array_equal(q[sel], dq[sel]), f"pixels with {c} samples differ from the dense render"
    assert not a[:r0].any() and not a[r1:].any()


def _run_rounds(rtb, r, W, H, D, seed, tol, min_spp, cap, rows=(0, 0), spb=0):
    """One round per call; before each, the active set is predicted from the accumulators.  Returns the cursors."""
    a = np.zeros((H, W, 4), np.float32); q = np.zeros_like(a)
    cursors, c, partial = [0], 0, 0
    while True:
        want = ar.active_mask(a, q, c, tol, min_spp, cap, rows)
        if not want.any():
            break
        st = r.render_adaptive(W, H, cap, D, tolerance=tol, min_spp=min_spp, max_rounds=1, seed=seed, clear=(c == 0), rows=rows,
                               samples_per_batch=spb)
        a2, q2 = r.download_accum(want_sum2=True)
        grew = a2[..., 3] > a[..., 3]
        assert st["rounds"] == 1
        assert np.array_equal(grew, want), f"round at cursor {c}: {int((grew != want).sum())} pixels differ from the prediction"
        k = ar.round_size(c, int(want.sum()), BUDGET, min_spp, cap)
        assert st["cursor"] == c + k and st["samples"] == int(want.sum()) * k
        partial += 0 < want.sum() < want[(slice(None) if tuple(rows) == (0, 0) else slice(*rows))].size
        a, q, c = a2, q2, c + k
        cursors.append(c)
        assert st["active_pixels"] == int(ar.active_mask(a, q, c, tol, min_spp, cap, rows).sum())
    return a, q, cursors, partial


@pytest.mark.parametrize("name,lights,W,H,D,rows,bin_mask", [
    ("book2_cornell_smoke", False, 48, 48, 50, (0, 0), None),    # media: the list gather in the media RNG
    ("book2_simple_light", True, 64, 40, 50, (0, 0), None),      # LIGHTS x list, the deferred Perlin texture
    ("book2_cornell", False, 48, 48, 50, (10, 37), None),        # a row range
    ("book2_final", False, 64, 64, 40, (0, 0), "116"),           # binning forced, the tail kernel, media, textures
])
def test_rounds_match_the_rule_and_the_dense_render(rtb, monkeypatch, name, lights, W, H, D, rows, bin_mask):
    if bin_mask:
        monkeypatch.setenv("RTB_BIN_MASK", bin_mask)
    r, _ = _renderer(rtb, name, lights)
    tol, min_spp, cap, spb, seed = 0.02, 8, 128, 8, 77
    a, q, cursors, partial = _run_rounds(rtb, r, W, H, D, seed, tol, min_spp, cap, rows, spb)
    print(f"{name}: cursors {cursors}, mean spp {a[..., 3].mean():.1f}, rounds with some pixels stopped {partial}")
    assert partial >= 1, "every round rendered every pixel or none: the list was not exercised"
    d, _ = _renderer(rtb, name, lights)
    _expect_per_pixel(_dense_snapshots(rtb, d, W, H, D, seed, cursors, rows, spb), a, q, rows, H)


def test_tolerance_zero_is_the_uniform_render(rtb):
    """Tolerance 0 stops only pixels whose whole 3x3 neighbourhood has an error of exactly 0 (black, or saturated beyond
    one standard error: the emitter seen directly); every other pixel runs to the cap with the dense render's sums."""
    W = H = 64
    r, _ = _renderer(rtb, "book2_cornell_smoke")
    st = r.render_adaptive(W, H, 256, 50, tolerance=0.0, min_spp=16, seed=5, samples_per_batch=16)
    a, q = r.download_accum(want_sum2=True)
    cursors = [0, 16, 32, 64, 128, 256]
    assert st["cursor"] == 256 and st["rounds"] == 5 and st["active_pixels"] == 0
    assert st["samples"] == int(a[..., 3].astype(np.int64).sum())
    d, _ = _renderer(rtb, "book2_cornell_smoke")
    snaps = _dense_snapshots(rtb, d, W, H, 50, 5, cursors, (0, 0), 16)
    _expect_per_pixel(snaps, a, q, (0, 0), H)
    stopped = a[..., 3] < 256
    print(f"tolerance 0: {int(stopped.sum())} of {W * H} pixels stopped early")
    assert stopped.mean() < 0.25
    for c in cursors[1:-1]:   # a pixel stopped at c had a zero window there
        sel = a[..., 3] == c
        if sel.any():
            assert (ar.window_max(ar.pixel_error(*snaps[c]))[sel] == 0).all()


def test_resume_from_a_checkpoint_is_bit_exact(rtb, tmp_path):
    W = H = 48
    kw = dict(tolerance=0.02, min_spp=8, seed=3, samples_per_batch=8)
    r, s = _renderer(rtb, "book2_cornell_smoke")
    full = r.render_adaptive(W, H, 256, 50, **kw)
    want, want2 = r.download_accum(want_sum2=True)
    r.render_adaptive(W, H, 256, 50, max_rounds=2, **kw)
    ck = tmp_path / "adaptive.rtba"
    r.save_accum(ck)
    b = rtb.Renderer(0); b.set_scene(s); b.set_camera(s.info.camera)
    assert b.load_accum(ck) == 16
    rest = b.render_adaptive(W, H, 256, 50, clear=False, **kw)
    got, got2 = b.download_accum(want_sum2=True)
    assert rest["cursor"] == full["cursor"] and rest["rounds"] == full["rounds"] - 2
    assert np.array_equal(got, want) and np.array_equal(got2, want2)


def test_quality_at_30_db(rtb):
    W = H = 120
    r, _ = _renderer(rtb, "book2_cornell_smoke")
    st = r.render_adaptive(W, H, 4096, 50, target_db=30, min_spp=64, seed=11)
    a = r.download_accum()
    r.render(W, H, 0, 16384, 50, seed=12)
    ref = r.download_accum()
    p = psnr(tonemap(a), tonemap(ref))
    print(f"30 dB target: {st}, mean spp {a[..., 3].mean():.1f}, PSNR against 16,384 spp {p:.2f} dB")
    assert p >= 29.0
    assert a[..., 3].mean() < 4096
    # every camera path the call reports started landed in the accumulator (a round whose queues were reallocated once
    # rendered nothing: the zeroing of the new queues was not ordered before the round's sample range)
    assert st["samples"] == int(a[..., 3].astype(np.int64).sum())


def test_validation(rtb):
    r, _ = _renderer(rtb, "book2_cornell")
    lib = rtb.lib()
    def call(width=32, height=32, sample_begin=0, sample_end=64, flags=rtb.RENDER_CLEAR, tol=0.01, min_spp=8):
        p = rtb.RenderParams(width, height, sample_begin, sample_end, 0, 0, 20, 1, flags, 0)
        a = rtb.AdaptiveParams(tol, min_spp, 0, 0)
        return lib.rtb_render_adaptive(r.handle, p, a, None, None)
    assert call() == 0
    for kw in (dict(min_spp=1), dict(min_spp=0), dict(sample_end=4), dict(sample_end=(1 << 24) + 1), dict(tol=-0.01),
               dict(tol=float("nan")), dict(tol=float("inf")), dict(sample_begin=1)):
        assert call(**kw) == -1, kw
    # continuing an accumulator without sums of squares: the first round (up to min_spp) has candidates without them
    r.render(32, 32, 0, 4, 20, seed=1)
    assert call(flags=0, min_spp=8) == -4
    assert "sums of squares" in lib.rtb_last_error().decode()
    # ... and past min_spp, where without sums of squares every error would read as 0 and the render would look converged
    r.render(32, 32, 0, 16, 20, seed=1)
    before = r.download_accum()
    assert call(flags=0, min_spp=8) == -4
    assert "sums of squares" in lib.rtb_last_error().decode()
    assert np.array_equal(r.download_accum(), before) and r.sample_cursor() == 16
    assert call(flags=0, min_spp=8, sample_end=16) == -4            # at the cap too
    # continuing an accumulator of another size
    r.render(32, 32, 0, 8, 20, seed=1, variance=True)
    assert call(width=48, height=48, flags=0) == -4
    with pytest.raises(ValueError):
        r.render_adaptive(32, 32, 64, 20)
    with pytest.raises(ValueError):
        r.render_adaptive(32, 32, 64, 20, tolerance=0.1, target_db=20)


def test_counters_cover_the_whole_call(rtb):
    """The path and ray totals of rtb_get_counters survive the queue enlargements of later rounds (the first round is
    min_spp x every pixel; later ones fill a whole batch), so they count every camera path the call started."""
    r, _ = _renderer(rtb, "book2_cornell_smoke")
    r.reset_counters()
    st = r.render_adaptive(160, 160, 2048, 50, tolerance=0.01, min_spp=16, seed=4)
    k = r.counters()
    a = r.download_accum()
    print(f"counters: {st}, paths {k.paths}, rays {k.rays}")
    assert st["rounds"] >= 3 and k.paths == st["samples"] == int(a[..., 3].astype(np.int64).sum())
    assert k.rays >= k.paths


def test_rtb_app_target_db(tmp_path):
    app = str(ROOT / "ray-tracing-v06_b200" / "rtb_app")
    out = tmp_path / "adaptive.ppm"
    res = subprocess.run([app, "book2_cornell_smoke", "--width", "64", "--height", "64", "--target-db", "30", "--spp", "256",
                          "--min-spp", "16", "--out", str(out)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    m = re.search(r"(\d+) rounds, mean ([0-9.]+) spp", res.stdout)
    assert m, res.stdout
    print(res.stdout.strip().splitlines()[-3:])
    assert int(m.group(1)) >= 1 and float(m.group(2)) < 256
    assert out.exists() and out.stat().st_size > 64 * 64 * 3
    res = subprocess.run([app, "book2_cornell_smoke", "--gpus", "2", "--target-db", "30"], capture_output=True, text=True)
    assert res.returncode == 1 and "one GPU" in res.stderr
    # resuming a uniform checkpoint (no sums of squares) adaptively fails instead of reporting the image converged
    ck = tmp_path / "uniform.rtba"
    base = ["book2_cornell_smoke", "--width", "64", "--height", "64", "--out", str(tmp_path / "u.ppm")]
    assert subprocess.run([app, *base, "--spp", "128", "--checkpoint", str(ck)], capture_output=True, text=True).returncode == 0
    res = subprocess.run([app, *base, "--resume", str(ck), "--target-db", "40", "--spp", "1024"], capture_output=True, text=True)
    assert res.returncode == 1 and "sums of squares" in res.stderr, (res.stdout, res.stderr)


def test_debug_bounds_build_adaptive(rtb):
    """librtb200_debug.so: an adaptive render of every registered scene (and, where it lists lights, with light sampling),
    binning forced: no index out of range (list entries and list indices are checked as path indices)."""
    if not rtb.DEBUG_LIB_PATH.exists():
        pytest.skip("librtb200_debug.so not built")
    code = r'''
import importlib, json, sys
sys.path.insert(0, %r)
rtb = importlib.import_module("ray-tracing-v06_b200")
r = rtb.Renderer(0); n = 0
for name in rtb.scene_names():
    for lights in (False, True):
        s = rtb.Scene.named(name)
        if lights:
            if not s.info.light_ids:
                continue
            s.sample_lights(s.info.light_ids)
        r.set_scene(s); r.set_camera(s.info.camera); n += 1
        r.render_adaptive(72, 56, 32, 40, tolerance=0.05, min_spp=4, seed=9, samples_per_batch=4)
        r.render_adaptive(72, 56, 32, 40, tolerance=0.05, min_spp=4, seed=9, rows=(10, 41))
        r.synchronize()
print("REPORT " + json.dumps(dict(r.debug_bounds_report(), renders=n)))
''' % (str(ROOT),)
    env = dict(os.environ, RTB_LIB=str(rtb.DEBUG_LIB_PATH), RTB_BIN_MASK="116")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    rep = json.loads([l for l in out.stdout.splitlines() if l.startswith("REPORT ")][-1][7:])
    print("bounds report, adaptive:", rep)
    assert rep.pop("renders") >= len(rtb.scene_names())
    assert rep.pop("rays_checked") > 10_000
    assert all(v == 0 for v in rep.values()), rep
