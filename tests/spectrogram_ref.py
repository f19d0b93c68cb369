"""Float64 restatement of the device spectrogram (sgb_rows_spectrogram, include/soundgen_b200.h), built on the
oracle's frame rule and seewave windows.  The parity target of tests/test_gpu_spectrogram.py."""
from __future__ import annotations

import numpy as np

from oracle.rprims import hamming_w, hanning_w
from oracle.soundgen_oracle import frame_starts

WINDOWS = {'hamming': hamming_w, 'hanning': hanning_w}


def stft_complex(wave, wl, step, window='hamming'):
    """seewave stft(complex = TRUE, wn = window, zp = 0) as the filter block calls it (the oracle's stft_complex with
    the window as a parameter): frame k starts at the truncated index step[k]; bins 0..wl/2-1; divided by wl."""
    W = WINDOWS[window](wl)
    half = wl // 2
    z = np.zeros((half, step.size), dtype=np.complex128)
    for k, x in enumerate(step):
        s = int(x)  # R truncates fractional indices
        z[:, k] = np.fft.fft(wave[s - 1:s - 1 + wl] * W)[:half]
    return z / wl


def spectrogram(x, wl, overlap, window='hamming', bands=None, db_floor=None):
    """Frames at frame_starts(len(x), wl, overlap) (none when len(x) = 0), samples past the end read as 0,
    X = stft_complex(x, wl, step, window), F = |X|^2 [nc, wl/2], or F @ bands.T for a [n_bands, wl/2] bank;
    db_floor given: 10 log10(max(F, db_floor))."""
    x = np.asarray(x, dtype=np.float64)
    if x.size == 0:
        F = np.zeros((0, wl // 2))
    else:
        step = frame_starts(x.size, wl, overlap)
        xp = np.concatenate((x, np.zeros(wl)))
        F = np.abs(stft_complex(xp, wl, step, window).T) ** 2
    if bands is not None:
        F = F @ np.asarray(bands, dtype=np.float64).T
    if db_floor is not None:
        F = 10 * np.log10(np.maximum(F, db_floor))
    return F
