"""float32 restatement of the adaptive stopping rule and round schedule (DESIGN.md §5c), written from that text
independently of the CUDA code: the per-pixel display-space error, the 3x3 window, the candidate test and the round size.
Every operation is a binary32 operation in the order DESIGN.md writes it (numpy rounds each float32 operation exactly once,
as the kernels built with -fmad=false do), and maxima / minima propagate NaN, so the GPU's decisions can be predicted
pixel for pixel."""
import numpy as np

F = np.float32


def tolerance_for_db(db):
    """tol = 10^(-D/20)."""
    return float(10.0 ** (-float(db) / 20.0))


def channel_error(S, Q, n):
    """One standard error of the mean, through clamp and sqrt, halved: (hi - lo) / 2 per channel (float32 arrays)."""
    S, Q, n = (np.asarray(x, dtype=F) for x in (S, Q, n))
    with np.errstate(all="ignore"):
        m = S / n
        v = np.maximum((Q - S * m) / (n - F(1)), F(0))
        s = np.sqrt(v / n)
        hi = np.sqrt(np.minimum(np.maximum(m + s, F(0)), F(1)))
        lo = np.sqrt(np.minimum(np.maximum(m - s, F(0)), F(1)))
        return (hi - lo) * F(0.5)


def pixel_error(accum, accum2):
    """e_p = max over r, g, b of the channel error, for (..., 4) accumulators (sums, count) and (sums of squares, count)."""
    a = np.asarray(accum, dtype=F); q = np.asarray(accum2, dtype=F)
    n = a[..., 3]
    e = [channel_error(a[..., c], q[..., c], n) for c in range(3)]
    return np.maximum(np.maximum(e[0], e[1]), e[2])


def window_max(e):
    """Maximum of e over the 3x3 neighbourhood, clipped to the array (the row range); NaN counts as +inf."""
    x = np.where(np.isnan(e), F(np.inf), e).astype(F)
    p = np.pad(x, 1, constant_values=F(-np.inf))
    H, W = x.shape
    out = np.full_like(x, F(-np.inf))
    for dy in range(3):
        for dx in range(3):
            out = np.maximum(out, p[dy:dy + H, dx:dx + W])
    return out


def _row_range(height, rows):
    r0, r1 = rows if rows is not None else (0, 0)
    return (0, height) if (r0, r1) == (0, 0) else (r0, r1)


def active_mask(accum, accum2, cursor, tolerance, min_spp, max_spp, rows=None):
    """(H, W) bool: the pixels the next round renders."""
    a = np.asarray(accum, dtype=F); q = np.asarray(accum2, dtype=F)
    H, W = a.shape[:2]
    r0, r1 = _row_range(H, rows)
    act = np.zeros((H, W), dtype=bool)
    if cursor >= max_spp:
        return act
    cand = a[r0:r1, :, 3] == F(cursor)
    if cursor >= min_spp:
        w = window_max(pixel_error(a[r0:r1], q[r0:r1]))
        cand &= ~(w <= F(tolerance))
    act[r0:r1] = cand
    return act


def missing_squares(accum, accum2, cursor, rows=None):
    """True when a pixel of the row range that holds the cursor's samples has no sums of squares (its count in accum2
    differs), whatever its error and the cap: the call fails then.  (Without sums of squares every error reads as 0.)"""
    a = np.asarray(accum, dtype=F); q = np.asarray(accum2, dtype=F)
    r0, r1 = _row_range(a.shape[0], rows)
    held = a[r0:r1, :, 3] == F(cursor)
    return bool(np.any(q[r0:r1, :, 3][held] != a[r0:r1, :, 3][held]))


def round_size(cursor, n_active, budget, min_spp, max_spp):
    """k = min(max_spp - c, c < min_spp ? min_spp - c : min(c, max(1, P / n_active)))."""
    k = min_spp - cursor if cursor < min_spp else min(cursor, max(1, budget // n_active))
    return min(max_spp - cursor, k)


def batch_samples(budget, n_active, k, samples_per_batch=0):
    """Samples per batch of a round of k samples, as rtb_render splits its sample range (equal batches when automatic)."""
    S = samples_per_batch if samples_per_batch else budget // n_active
    S = max(S, 1)
    S = min(S, k) if k else 1
    if not samples_per_batch and k:
        nb = -(-k // S)
        S = -(-k // nb)
    return S


def round_schedule(active_counts, budget, min_spp, max_spp, cursor=0):
    """Cursors before each round for a history of active-pixel counts (one per select step): [(cursor, k), ...] up to the
    first count of 0 or the cap."""
    out = []
    for n in active_counts:
        if n == 0 or cursor >= max_spp:
            break
        k = round_size(cursor, n, budget, min_spp, max_spp)
        out.append((cursor, k))
        cursor += k
    return out
