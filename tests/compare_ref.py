"""Float64 restatement of the similarity scores of sgb_rows_compare (include/soundgen_b200.h).  The parity target of
tests/test_gpu_compare.py."""
from __future__ import annotations

import numpy as np


def padded(a, b, pad):
    """a [n_a, F], b [n_b, F] as [N, F] each, N = max(n_a, n_b), the missing frames filled with pad."""
    N = max(a.shape[0], b.shape[0])
    A = np.full((N, a.shape[1]), float(pad))
    B = np.full((N, b.shape[1]), float(pad))
    A[:a.shape[0]] = a
    B[:b.shape[0]] = b
    return A.ravel(), B.ravel()


def dtw_plain(a, b):
    """symmetric2 DTW distance D(n_a, n_b) by the plain double loop: D(1,1) = d(1,1) as dtw's globalCostMatrix starts
    it, then D(i,j) = min(D(i-1,j-1) + 2d, D(i-1,j) + d, D(i,j-1) + d), d = Euclidean distance of the frames."""
    d = np.sqrt(((a[:, None, :] - b[None, :, :]) ** 2).sum(axis=2))
    D = np.full(d.shape, np.inf)
    for i in range(d.shape[0]):
        for j in range(d.shape[1]):
            if i == 0 and j == 0:
                D[i, j] = d[i, j]
                continue
            c = np.inf
            if i > 0 and j > 0:
                c = D[i - 1, j - 1] + 2 * d[i, j]
            if i > 0:
                c = min(c, D[i - 1, j] + d[i, j])
            if j > 0:
                c = min(c, D[i, j - 1] + d[i, j])
            D[i, j] = c
    return D[-1, -1]


def dtw(a, b):
    """dtw_plain's distance, one anti-diagonal at a time (for rows of thousands of frames)."""
    na, nb = a.shape[0], b.shape[0]
    prev2 = prev1 = None
    for k in range(na + nb - 1):
        i = np.arange(max(0, k - nb + 1), min(k, na - 1) + 1)
        j = k - i
        d = np.sqrt(((a[i] - b[j]) ** 2).sum(axis=1))
        if k == 0:
            cur = d.copy()
        else:
            cur = np.full(i.size, np.inf)
            lo1 = max(0, k - nb)                 # first i of diagonal k-1
            lo2 = max(0, k - 1 - nb)             # first i of diagonal k-2
            m = (i > 0) & (j > 0)
            if m.any():
                cur[m] = prev2[i[m] - 1 - lo2] + 2 * d[m]
            m = i > 0
            cur[m] = np.minimum(cur[m], prev1[i[m] - 1 - lo1] + d[m])
            m = j > 0
            cur[m] = np.minimum(cur[m], prev1[i[m] - lo1] + d[m])
        prev2, prev1 = prev1, cur
    return prev1[-1]


def score(a, b, method, pad=0.0):
    """The score of rows a [n_a, n_feat] and b [n_b, n_feat]: 'cor', 'cosine' (both over the padded cells) or 'dtw'
    (-D / (n_a + n_b), no padding); NaN for an empty row, a constant side (cor) or an all-zero side (cosine)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if a.shape[0] == 0 or b.shape[0] == 0:
        return float('nan')
    if method == 'dtw':
        return -dtw(a, b) / (a.shape[0] + b.shape[0])
    x, y = padded(a, b, pad)
    if method == 'cor':
        if np.all(x == x[0]) or np.all(y == y[0]):
            return float('nan')
        x = x - x.mean()
        y = y - y.mean()
    with np.errstate(invalid='ignore'):
        return float(np.dot(x, y) / (np.sqrt(np.dot(x, x)) * np.sqrt(np.dot(y, y))))
