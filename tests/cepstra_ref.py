"""Float64 restatement of the device cepstra (sgb_rows_cepstra, include/soundgen_b200.h): the DCT-II matrix of
mfcc_device, the projection, and deltas of order 1 and 2 with the row's edge frames replicated.  The parity target of
tests/test_gpu_cepstra.py."""
from __future__ import annotations

import numpy as np


def dct(n_mfcc, n_mels, include_c0=True):
    """Orthonormal DCT-II rows k = 0 .. n_mfcc - 1 (or 1 .. n_mfcc without c0) over n_mels bands, [n_mfcc, n_mels]."""
    k0 = 0 if include_c0 else 1
    k = np.arange(k0, k0 + n_mfcc, dtype=np.float64)[:, None]
    b = np.arange(n_mels, dtype=np.float64)[None, :]
    scale = np.where(k == 0, np.sqrt(1.0 / n_mels), np.sqrt(2.0 / n_mels))
    return scale * np.cos(np.pi * k * (2 * b + 1) / (2 * n_mels))


def deltas(c, n):
    """d_t = sum_{j=1..n} j (c[min(t + j, nc - 1)] - c[max(t - j, 0)]) / (2 sum j^2) over the rows of c [nc, k]."""
    c = np.asarray(c, dtype=np.float64)
    nc = c.shape[0]
    d = np.zeros_like(c)
    t = np.arange(nc)
    for j in range(1, n + 1):
        d += j * (c[np.minimum(t + j, nc - 1)] - c[np.maximum(t - j, 0)])
    return d / (2 * sum(j * j for j in range(1, n + 1)))


def cepstra(x, M, order=0, n=2):
    """[c | d | dd] of the frames x [nc, n_in] for the matrix M [n_ceps, n_in]: [nc, n_ceps (1 + order)]."""
    c = np.asarray(x, dtype=np.float64) @ np.asarray(M, dtype=np.float64).T
    out = [c]
    for _ in range(order):
        out.append(deltas(out[-1], n))
    return np.concatenate(out, axis=1)
