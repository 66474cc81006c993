"""CPU tests of the adaptive stopping rule's restatement (tests/adaptive_rule.py, DESIGN.md §5c) against hand-derived
answers: the per-pixel error, the window, the candidate test, the PSNR-target conversion and the round schedule."""
import numpy as np

import adaptive_rule as ar

F = np.float32


def _accum(samples):
    """(sums, count), (sums of squares, count) of one grey pixel, summed in float32 in sample order as accumulate does."""
    s = F(0); q = F(0)
    for x in np.asarray(samples, dtype=F):
        s = F(s + x); q = F(q + F(x * x))
    n = F(len(samples))
    return np.array([s, s, s, n], dtype=F), np.array([q, q, q, n], dtype=F)


def _grid(H, W, count, value=0.0):
    a = np.zeros((H, W, 4), dtype=F); q = np.zeros((H, W, 4), dtype=F)
    a[..., :3] = F(value) * F(count); q[..., :3] = F(value) * F(value) * F(count)
    a[..., 3] = count; q[..., 3] = count
    return a, q


def _make_noisy(a, q, y, x):
    """Pixel (y, x): half its samples 0.2, half 0.6 (error well above 1e-3)."""
    n = int(a[y, x, 3])
    pa, pq = _accum([0.2] * (n // 2) + [0.6] * (n - n // 2))
    a[y, x] = pa; q[y, x] = pq


def test_constant_samples_have_zero_error():
    for v in (0.0, 0.25, 0.5, 3.0):                       # black, exactly representable greys, saturated
        a, q = _accum([v] * 16)
        assert ar.pixel_error(a, q) == 0.0, v


def test_mean_above_one_by_more_than_one_standard_error_is_zero():
    # samples 1.5 and 3.5, 8 of each: mean 2.5, standard error sqrt((16/15) / 16) = 0.258; m - s = 2.24 > 1, both ends clamp to 1
    a, q = _accum([1.5, 3.5] * 8)
    assert ar.pixel_error(a, q) == 0.0
    # ... but within one standard error of 1 it is not
    a, q = _accum([0.5, 1.6] * 8)
    assert ar.pixel_error(a, q) > 0.0


def test_two_valued_samples_closed_form():
    for lo_v, hi_v, nlo, nhi in ((0.1, 0.4, 8, 8), (0.0, 0.9, 30, 2), (0.05, 0.07, 100, 156)):
        a, q = _accum([lo_v] * nlo + [hi_v] * nhi)
        n = nlo + nhi
        m = (nlo * lo_v + nhi * hi_v) / n
        var = nlo * nhi * (hi_v - lo_v) ** 2 / (n * (n - 1))          # unbiased sample variance of the two values
        s = np.sqrt(var / n)
        want = (np.sqrt(np.clip(m + s, 0, 1)) - np.sqrt(np.clip(m - s, 0, 1))) / 2
        got = float(ar.pixel_error(a, q))
        assert abs(got - want) <= 2e-4 * want, (lo_v, hi_v, got, want)


def test_window_dilates_to_the_neighbours():
    H, W, c = 6, 5, 8
    a, q = _grid(H, W, c)
    _make_noisy(a, q, 2, 3)
    act = ar.active_mask(a, q, c, 1e-3, 4, 64)
    want = np.zeros((H, W), bool); want[1:4, 2:5] = True
    assert np.array_equal(act, want)
    # a NaN error (sums that overflowed) counts as +inf: it keeps itself and its neighbours active
    a2, q2 = _grid(H, W, c)
    a2[0, 0, :3] = np.inf; q2[0, 0, :3] = np.inf
    assert np.isnan(ar.pixel_error(a2, q2)[0, 0])
    want = np.zeros((H, W), bool); want[0:2, 0:2] = True
    assert np.array_equal(ar.active_mask(a2, q2, c, 1e-3, 4, 64), want)


def test_window_is_clipped_to_the_row_range():
    H, W, c = 6, 5, 8
    a, q = _grid(H, W, c)
    _make_noisy(a, q, 3, 1)
    # rows [1, 3): the noisy pixel is outside, so nothing inside sees it, and rows outside are never active
    assert not ar.active_mask(a, q, c, 1e-3, 4, 64, rows=(1, 3)).any()
    # rows [1, 4): row 3 is inside; the window loses row 4
    act = ar.active_mask(a, q, c, 1e-3, 4, 64, rows=(1, 4))
    want = np.zeros((H, W), bool); want[2:4, 0:3] = True
    assert np.array_equal(act, want)


def test_min_spp_forces_pixels_and_stopped_pixels_never_return():
    H, W = 4, 4
    a, q = _grid(H, W, 4)                                  # zero error everywhere
    assert ar.active_mask(a, q, 4, 0.5, 8, 64).all()       # cursor 4 < min_spp 8: every candidate is active
    assert not ar.active_mask(a, q, 4, 0.5, 4, 64).any()   # from min_spp on, zero error stops them
    # pixels with fewer samples than the cursor missed a round: never active, however noisy
    a, q = _grid(H, W, 16)
    a[1, 1, 3] = q[1, 1, 3] = 8
    _make_noisy(a, q, 1, 1)                                # 8 samples, very noisy
    a[0, 0, 3] = q[0, 0, 3] = 8
    act = ar.active_mask(a, q, 16, 1e-3, 4, 64)
    assert not act[1, 1] and not act[0, 0]
    assert act[2, 2] and act[0, 1]                         # neighbours of the noisy pixel still are
    assert not ar.active_mask(a, q, 8, 1e-3, 4, 8).any()   # at the cap nothing is active
    # a pixel holding the cursor without sums of squares is detected, before the window: with Q = 0 its error reads as 0
    a, q = _grid(H, W, 16)
    _make_noisy(a, q, 1, 1)
    q[..., :] = 0
    assert not ar.active_mask(a, q, 16, 1e-3, 8, 64).any()      # the window test alone would call it converged
    assert ar.missing_squares(a, q, 16)
    assert not ar.missing_squares(a, q, 8)                      # no pixel holds cursor 8
    a2, q2 = _grid(H, W, 16)
    assert not ar.missing_squares(a2, q2, 16)


def test_tolerance_for_db(rtb):
    assert abs(ar.tolerance_for_db(40) - 0.01) < 1e-12
    assert abs(ar.tolerance_for_db(20) - 0.1) < 1e-12
    assert abs(ar.tolerance_for_db(0) - 1.0) < 1e-12
    for db in (30, 37, 43):
        assert rtb.tolerance_for_db(db) == ar.tolerance_for_db(db)


def test_round_size_sequence():
    P = 64 << 20
    # 800 x 800: the first round up to min_spp, then one doubling per round while a batch holds it
    sched = ar.round_schedule([640000, 640000, 300000, 100000, 1000, 10, 0], P, 64, 4096)
    assert sched == [(0, 64), (64, 64), (128, 128), (256, 256), (512, 512), (1024, 1024)]
    # many active pixels: a round is at most one batch of P paths
    sched = ar.round_schedule([8_000_000, 8_000_000, 4_000_000, 4_000_000], P, 16, 1024)
    assert sched == [(0, 16), (16, 8), (24, 16), (40, 16)]
    # the cap clamps the last round; a round of one sample when the budget is smaller than the active count
    assert ar.round_size(1000, 10, P, 64, 1024) == 24
    assert ar.round_size(100, P + 1, P, 64, 4096) == 1
    # batches of a round: equal-sized, as rtb_render splits its range; an explicit size is honoured
    assert ar.batch_samples(P, 8_000_000, 16) == 8
    assert ar.batch_samples(P, 10_000_000, 64) == 6        # 6 per batch fits, 11 batches, evened out to ceil(64 / 11) = 6
    assert ar.batch_samples(P, 640000, 64) == 64
    assert ar.batch_samples(P, 640000, 64, samples_per_batch=16) == 16
