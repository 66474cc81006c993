"""Adaptive rounds beyond a million pixels (rtb_render_adaptive, DESIGN.md §5c).  At 1920 x 1080 the select step has 2,025
blocks of 1,024 pixels, so adaptive_scan_kernel scans their counts in two chunks with a carry; a row range of (7, 1075)
starts and ends inside a block.  With the batch budget pinned (RTB_BATCH_PATHS), the rounds take every shape the host
code gives them: split into several batches, a sample count bound by the budget, automatic binning on and off.  Every round
must render exactly the pixels tests/adaptive_rule.py predicts, and every pixel must end with the dense render's sums at its
own count, bit for bit."""
import time

import numpy as np
import pytest

import adaptive_rule as ar
import feature_scenes as fs
from test_gpu_schedules import SWITCHES

pytestmark = pytest.mark.gpu

W, H = 1920, 1080
BUDGET = 16 << 20        # RTB_BATCH_PATHS: 8 samples of every pixel per batch
MIN_SPP, CAP, TOL, D, SEED = 16, 32, 0.01, 40, 91   # (the cap makes the last round small enough to go unbinned)
BIN_MIN_PATHS, BIN_MIN_NODES = 8 << 20, 512    # the automatic binning rule of rtb_render / rtb_render_adaptive
TAIL_CHECKPOINTS = (2, 3, 4, 5, 6, 8, 10, 12, 15, 18, 22, 27, 33, 40, 48)    # tail_checkpoint() below bounce 50
DEFAULT_BIN_BOUNCES = (1, 2, 4, 8)                                             # the default RTB_BIN_MASK 0x116


def _scene(rtb, name):
    if name == "feature":
        case = fs.Case("pre", "normal", False, "sampled", True)
        return fs.build(rtb, case)
    s = rtb.Scene.named(name)
    if name == "book2_cornell_smoke":
        s.sample_lights(s.info.light_ids)
    return s, s.info.camera


def _launches_per_batch(deferred_tex, binned):
    """rtb_render_adaptive's launch count of one batch (enqueue_batch) with the default tail threshold and bin mask."""
    return (3 + 2 * D + sum(b < D for b in TAIL_CHECKPOINTS) + (D - 1 if deferred_tex else 0)
            + (3 * sum(b < D for b in DEFAULT_BIN_BOUNCES) if binned else 0))


def _rounds(rtb, r, rows, n_nodes, deferred_tex):
    """One round per call.  Before each, the active set and the round's shape are predicted from the accumulators; after it,
    the pixels that grew, the stats and the launches are checked.  Returns the final accumulators and the rounds."""
    a = np.zeros((H, W, 4), np.float32); q = np.zeros_like(a)
    c, rounds = 0, []
    while True:
        want = ar.active_mask(a, q, c, TOL, MIN_SPP, CAP, rows)
        n = int(want.sum())
        if n == 0:
            break
        k = ar.round_size(c, n, BUDGET, MIN_SPP, CAP)
        S = ar.batch_samples(BUDGET, n, k)
        nb = -(-k // S)
        binned = n_nodes >= BIN_MIN_NODES and n * S >= BIN_MIN_PATHS
        l0 = int(r.counters().launches)
        st = r.render_adaptive(W, H, CAP, D, tolerance=TOL, min_spp=MIN_SPP, max_rounds=1, seed=SEED, clear=(c == 0), rows=rows)
        launches = int(r.counters().launches) - l0
        a2, q2 = r.download_accum(want_sum2=True)
        grew = a2[..., 3] > a[..., 3]
        assert np.array_equal(grew, want), f"round at cursor {c}: {int((grew != want).sum())} pixels differ from the prediction"
        assert st["rounds"] == 1 and st["cursor"] == c + k and st["samples"] == n * k, (st, c, k, n)
        # the launches show the batch count and whether the round was binned (plus the select steps before and after it)
        select = (4 if c >= MIN_SPP else 3) + (4 if c + k >= MIN_SPP else 3)
        assert launches == select + nb * _launches_per_batch(deferred_tex, binned), (launches, nb, binned)
        a, q, c = a2, q2, c + k
        assert st["active_pixels"] == int(ar.active_mask(a, q, c, TOL, MIN_SPP, CAP, rows).sum())
        rounds.append(dict(cursor=c - k, active=n, k=k, S=S, batches=nb, budget_bound=k == BUDGET // n < c - k,
                           binned=binned))
    return a, q, rounds


def _expect_dense(rtb, scene, cam, a, q, rounds, rows):
    """A dense progressive render over the same sample ranges with the same batch sizes: after each range, the pixels whose
    count is the new cursor hold its sums bit for bit.  One snapshot at a time."""
    d = rtb.Renderer(0); d.set_scene(scene); d.set_camera(cam)
    r0, r1 = rows
    counts = a[..., 3]
    seen = 0
    for rd in rounds:
        c0, c1 = rd["cursor"], rd["cursor"] + rd["k"]
        d.render(W, H, c0, c1, D, seed=SEED, clear=(c0 == 0), variance=True, rows=rows, samples_per_batch=rd["S"])
        da, dq = d.download_accum(want_sum2=True)
        sel = np.zeros(counts.shape, bool); sel[r0:r1] = counts[r0:r1] == c1
        assert np.array_equal(a[sel], da[sel]) and np.array_equal(q[sel], dq[sel]), f"pixels with {c1} samples differ from the dense render"
        seen += int(sel.sum())
    assert seen == (r1 - r0) * W, "a pixel's count is not a round boundary"
    assert not a[:r0].any() and not a[r1:].any()


@pytest.mark.parametrize("rows", [(0, H), (7, 1075)], ids=["full", "rows_7_1075"])
@pytest.mark.parametrize("name", ["book2_final", "book2_cornell_smoke", "feature"])
def test_rounds_at_1080p(rtb, monkeypatch, name, rows):
    t0 = time.time()
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("RTB_BATCH_PATHS", str(BUDGET))
    scene, cam = _scene(rtb, name)
    r = rtb.Renderer(0); r.set_scene(scene); r.set_camera(cam)
    stats = r.scene_stats()
    deferred_tex = name != "book2_cornell_smoke"
    a, q, rounds = _rounds(rtb, r, rows, stats["inner_nodes"], deferred_tex)
    print(f"\n{name} rows {rows}: {stats['inner_nodes']} inner nodes; predicted and observed rounds:")
    for rd in rounds:
        kinds = [s for s, on in (("several batches", rd["batches"] > 1), ("k bound by the budget", rd["budget_bound"]),
                                 ("binned", rd["binned"]), ("not binned", not rd["binned"])) if on]
        print(f"  cursor {rd['cursor']:3d}: {rd['active']:8d} pixels, k {rd['k']:2d}, {rd['batches']} x {rd['S']} samples  [{', '.join(kinds)}]")
    assert any(rd["batches"] > 1 for rd in rounds) and any(rd["budget_bound"] for rd in rounds)
    if name == "book2_final":
        assert any(rd["binned"] for rd in rounds) and any(not rd["binned"] for rd in rounds)
    assert max(rd["active"] for rd in rounds) > 1024 * 1024, "the select step must run more than one chunk of blocks"
    _expect_dense(rtb, scene, cam, a, q, rounds, rows)
    if name == "book2_final" and rows == (0, H):
        # the same rounds with the tail off (schedule B of tests/test_gpu_schedules.py): the wavefront runs every bounce
        monkeypatch.setenv("RTB_TAIL_THRESHOLD", "0")
        b = rtb.Renderer(0); b.set_scene(scene); b.set_camera(cam)
        st = b.render_adaptive(W, H, CAP, D, tolerance=TOL, min_spp=MIN_SPP, seed=SEED, rows=rows)
        ba, bq = b.download_accum(want_sum2=True)
        assert st["rounds"] == len(rounds) and np.array_equal(ba, a) and np.array_equal(bq, q)
    print(f"{name} rows {rows}: {time.time() - t0:.1f} s")
