"""numpy restatements for the f0 labels: K12b's frame labels (sgb_rows_f0_frames) and the frame count of K9, and the
float32 tolerance the f0 track is held to."""
import math

import numpy as np


def frame_count(length, wl, overlap):
    """nc = length(seq(1, max(1, len - wl), h)), 0 for an empty row (sgb_spec_frames)."""
    if length <= 0:
        return 0
    h = wl - overlap * wl / 100.0
    to = max(1.0, float(length - wl))
    if to == 1.0:
        return 1
    return int(math.floor((to - 1.0) / h + 1e-10)) + 1


def frame_labels(x, length, wl, overlap, cap=None):
    """[cap, 2] float32: label k = [x at s_k + wl/2 (0 at or past length), nonzero samples in [s_k, s_k + wl) within
    [0, length) / wl], s_k = floor(1 + k h) - 1; zeros past the row's frames."""
    nc = frame_count(length, wl, overlap)
    cap = nc if cap is None else cap
    h = wl - overlap * wl / 100.0
    x = np.asarray(x, dtype=np.float32)[:length]
    P = np.concatenate(([0], np.cumsum(x != 0)))
    out = np.zeros((cap, 2), dtype=np.float32)
    m = min(nc, cap)
    k = np.arange(m, dtype=np.float64)
    s = np.floor(1.0 + k * h).astype(np.int64) - 1
    e = np.minimum(s + wl, length)
    c = s + wl // 2
    xp = np.concatenate((x, np.zeros(wl, dtype=np.float32)))
    out[:m, 0] = np.where(c < length, xp[np.minimum(c, xp.size - 1)], 0)
    out[:m, 1] = (P[e] - P[s]).astype(np.float32) / np.float32(wl)
    return out


def within_ulp(dev, ref, n_ulp=2):
    """|dev - ref| <= n_ulp float32 ulps of ref (ref in FP64), elementwise."""
    ref = np.asarray(ref, dtype=np.float64)
    ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
    return np.abs(np.asarray(dev, dtype=np.float64) - ref) <= n_ulp * ulp
