"""Schedule invariance of the wavefront at production queue sizes, and oracle parity with the wavefront running every bounce.

Which kernels run depends on sizes and switches: the fused tail kernel takes a batch over once its live queue is shorter than
sms x 768 rays (checked from bounce 2); traverse and shade pull chunks beyond their static grid span (blocks x 128 rays)
through the work counters; binning runs where RTB_BIN_MASK or the automatic rule says.  A schedule only decides which rays
share a warp and which launch does the work - never what a path computes - so every schedule below must give the same
sums, bit for bit, for every case of tests/feature_scenes.py, whose cases together select every traverse, shade and tail
instantiation (in dense renders and in adaptive rounds)."""
import json
import os
import subprocess
import sys
import time
from contextlib import contextmanager

import numpy as np
import pytest

import feature_scenes as fs
from conftest import ROOT
from feature_oracle import FeatureOracleScene

pytestmark = pytest.mark.gpu

SWITCHES = ("RTB_TAIL_THRESHOLD", "RTB_BIN_MASK", "RTB_BIN_BITS", "RTB_LANES", "RTB_NO_GRAPH", "RTB_BATCH_PATHS")
NO_TAIL = "0"
TAIL_FROM_2 = "4294967295"
SCHEDULES = {
    "A": {},                                                              # default
    "B": {"RTB_TAIL_THRESHOLD": NO_TAIL},                                  # the wavefront runs every bounce
    "C": {"RTB_TAIL_THRESHOLD": TAIL_FROM_2},                              # the tail kernel from bounce 2
    "D": {"RTB_TAIL_THRESHOLD": NO_TAIL, "RTB_BIN_MASK": "fffffffffffffffe"},   # ... and every bounce binned
    "E": {"RTB_LANES": "2"},                                               # two lanes (three batches)
    "F": {"RTB_NO_GRAPH": "1"},                                            # launches without the batch graph
}
# dense: three batches of 640 x 400 x 9 = 2.3 M paths
W, H, SPB, D = 640, 400, 9, 16
SPP = 3 * SPB
CASES = [pytest.param(c, id=c.id) for c in fs.CASES]


@contextmanager
def schedule(monkeypatch, name, **extra):
    """The environment of a schedule (every switch not named is unset).  The switches are read when a Renderer is created,
    RTB_NO_GRAPH and RTB_BATCH_PATHS also when it renders: create and render inside."""
    with monkeypatch.context() as m:
        for k in SWITCHES:
            m.delenv(k, raising=False)
        for k, v in {**SCHEDULES[name], **extra}.items():
            m.setenv(k, v)
        yield


def _renderer(rtb, scene, cam):
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam); r.reset_counters()
    return r


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_coverage_table():
    print("\n" + fs.format_coverage(fs.check_coverage()))


@pytest.mark.parametrize("case", CASES)
def test_dense_schedules_are_bit_identical(rtb, monkeypatch, case):
    """Schedules A-F on batches of 2.3 M paths: the accumulators, sums of squares, path and ray counts are identical."""
    sms = _sms()
    assert W * H * SPB > 4 * sms * 16 * 128, "a batch must outgrow the static grid span of traverse several times"
    assert W * H * SPB > sms * 768, "a batch must start above the tail threshold"
    scene, cam = fs.build(rtb, case)
    got = {}
    for name in SCHEDULES:
        with schedule(monkeypatch, name):
            r = _renderer(rtb, scene, cam)
            if name == "A":
                fs.check_selection(case, scene, r.scene_stats())
            r.render(W, H, 0, SPP, D, seed=29, variance=True, samples_per_batch=SPB)
            a, a2 = r.download_accum(want_sum2=True); k = r.counters()
            assert k.batches == 3
            got[name] = (a, a2, int(k.paths), int(k.rays))
            del r
    base = got["A"]
    assert base[2] == W * H * SPP and base[3] > base[2]
    for name, g in got.items():
        assert np.array_equal(g[0], base[0]), f"schedule {name}: radiance sums differ from schedule A"
        assert np.array_equal(g[1], base[1]), f"schedule {name}: sums of squares differ from schedule A"
        assert g[2:] == base[2:], f"schedule {name}: paths / rays {g[2:]} against {base[2:]}"
    print(f"{case.id}: {base[3]} rays, schedules A-F identical")


@pytest.mark.parametrize("case", CASES)
def test_adaptive_schedules_are_bit_identical(rtb, monkeypatch, case):
    """Three adaptive rounds (list-mode kernels) of 640 x 400 pixels, the first 2.3 M paths in one batch, the third in two
    batches: schedules A-D give the same accumulators and the same stats."""
    scene, cam = fs.build(rtb, case)
    got = {}
    for name in "ABCD":
        with schedule(monkeypatch, name):
            r = _renderer(rtb, scene, cam)
            st = r.render_adaptive(W, H, 256, D, tolerance=0.02, min_spp=SPB, max_rounds=3, seed=31, samples_per_batch=SPB)
            a, a2 = r.download_accum(want_sum2=True)
            got[name] = (a, a2, st, int(r.counters().rays))
            del r
    base = got["A"]
    assert base[2]["rounds"] == 3 and base[2]["cursor"] == 4 * SPB and base[2]["samples"] > W * H * SPB
    for name, g in got.items():
        assert np.array_equal(g[0], base[0]) and np.array_equal(g[1], base[1]), f"schedule {name}: accumulators differ from schedule A"
        assert g[2] == base[2] and g[3] == base[3], f"schedule {name}: {g[2]}, {g[3]} rays against {base[2]}, {base[3]}"
    print(f"{case.id}: {base[2]}")


OW, OH, OS, OD = 192, 128, 8, 24


@pytest.mark.parametrize("case", CASES)
def test_wavefront_every_bounce_matches_the_oracle(rtb, monkeypatch, case):
    """Schedule B (no tail: traverse, shade and texture run every bounce) against the CPU oracle on the same Philox streams:
    at most 1e-4 of the pixels differ (a tie between two hits at one t may resolve differently), ray counts within 5e-6.
    With the dense invariance above, every schedule is then pinned to the oracle."""
    scene, cam = fs.build(rtb, case)
    with schedule(monkeypatch, "B"):
        r = _renderer(rtb, scene, cam)
        r.render(OW, OH, 0, OS, OD, seed=1984)
        g = r.download_accum(); rays_g = int(r.counters().rays)
    t = time.time()
    ref, _, rays = FeatureOracleScene(scene.serialize()).render(cam, OW, OH, 0, OS, OD, seed=1984)
    t = time.time() - t
    diff = np.abs(g[..., :3] - ref[..., :3]).max(axis=2)
    bad = float((diff > 1e-4 * np.maximum(np.abs(ref[..., :3]).max(axis=2), 1.0)).mean())
    print(f"{case.id}: {bad * 100:.4f} % of pixels differ, rays gpu {rays_g} oracle {rays}, oracle {t:.2f} s")
    assert np.array_equal(g[..., 3], ref[..., 3])
    assert bad <= 1e-4
    assert abs(rays_g - int(rays)) <= max(5e-6 * rays, 4)


def test_the_wavefront_runs_every_bounce_without_the_tail(rtb):
    """librtb200_debug.so counts the rays entering traverse_kernel (process-global).  Under schedule B that count grows by
    exactly the rays the renders report, so traverse ran every bounce of every case; under schedule C (tail from bounce 2)
    it grows by less.  No bounds class may count a violation."""
    if not rtb.DEBUG_LIB_PATH.exists():
        pytest.skip("librtb200_debug.so not built")
    code = r'''
import importlib, json, os, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
rtb = importlib.import_module("ray-tracing-v06_b200")
import feature_scenes as fs
out = []
for case in fs.CASES:
    s, cam = fs.build(rtb, case)
    row = {"case": case.id}
    for name, thr in (("B", "0"), ("C", "4294967295")):
        os.environ["RTB_TAIL_THRESHOLD"] = thr
        r = rtb.Renderer(0); r.set_scene(s); r.set_camera(cam)
        for mode in ("dense", "list"):
            before = r.debug_bounds_report()["rays_checked"]; r.reset_counters()
            if mode == "dense":
                r.render(96, 64, 0, 6, 16, seed=7, samples_per_batch=3)
            else:
                r.render_adaptive(96, 64, 64, 16, tolerance=0.05, min_spp=4, max_rounds=3, seed=7)
            r.synchronize()
            row[name + " " + mode] = (r.debug_bounds_report()["rays_checked"] - before, int(r.counters().rays))
    out.append(row)
print("REPORT " + json.dumps({"rows": out, "bounds": r.debug_bounds_report()}))
''' % (str(ROOT), str(ROOT / "tests"))
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env["RTB_LIB"] = str(rtb.DEBUG_LIB_PATH)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert res.returncode == 0, res.stderr[-3000:]
    rep = json.loads([l for l in res.stdout.splitlines() if l.startswith("REPORT ")][-1][7:])
    for row in rep["rows"]:
        print(row)
        for mode in ("dense", "list"):
            checked, rays = row["B " + mode]
            assert checked == rays > 0, f"{row['case']} {mode}: schedule B traversed {checked} of {rays} rays"
            checked, rays = row["C " + mode]
            assert 0 < checked < rays, f"{row['case']} {mode}: schedule C traversed {checked} of {rays} rays"
    bounds = rep["bounds"]
    print("bounds report:", bounds)
    assert bounds.pop("rays_checked") > 0
    assert all(v == 0 for v in bounds.values()), bounds


BIN_CASE = fs.Case("bvh", "normal", True, "sampled", True)


@pytest.mark.parametrize("bits,mask", [("0,1", None), ("1,0", None), ("5,4", None), ("8,1", "2")])
def test_bin_grid_extremes(rtb, monkeypatch, bits, mask):
    """Binning every bounce (schedule D) at the smallest grids - 4 bins, where one thread of the single scan block holds
    them all, and 8 bins - and at 2^23 bins (2,048 scan blocks; nearly every key of a tile distinct, so the count table
    flushes every tile): the image is the unbinned one, bit for bit.  2^26 bins, the largest grid accepted, bins bounce 1
    only: its scan re-reads every earlier count per block (O(bins^2 / 4096)), and the time is printed."""
    scene, cam = fs.build(rtb, BIN_CASE)
    Wb, Hb, S = 640, 400, 4
    with schedule(monkeypatch, "B"):
        r = _renderer(rtb, scene, cam)
        r.render(Wb, Hb, 0, S, D, seed=41, variance=True, samples_per_batch=S)
        want = r.download_accum(want_sum2=True) + (int(r.counters().rays),)
        del r
    extra = {"RTB_BIN_BITS": bits}
    if mask:
        extra["RTB_BIN_MASK"] = mask
    with schedule(monkeypatch, "D", **extra):
        r = _renderer(rtb, scene, cam)
        r.render(Wb, Hb, 0, S, D, seed=41, samples_per_batch=S)   # warm-up (queues, graph)
        r.synchronize(); r.reset_counters()
        t = time.time()
        r.render(Wb, Hb, 0, S, D, seed=41, variance=True, samples_per_batch=S)
        r.synchronize(); t = time.time() - t
        got = r.download_accum(want_sum2=True) + (int(r.counters().rays),)
        launches = int(r.counters().launches)
        del r
    print(f"RTB_BIN_BITS={bits} RTB_BIN_MASK={mask or 'fffffffffffffffe'}: {Wb}x{Hb}x{S} in one batch, {t * 1e3:.1f} ms, {launches} launches")
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]
