"""Synthetic, seeded parameter sets for the BASELINE.json configs (SURVEY.md 8d).

Each generator returns a list of keyword dicts for `soundgen()` / `BatchBuilder.add_soundgen`.
cfg1-3 (temperature 0): host-drawn random buffers ride along as `z` (list of normal streams, one per
voiced syllable) and `u` (list of uniform buffers, one per noise segment), numpy PCG64 with
seed = 20260000 + cfg (+ rank offset).  cfg0 and cfg4 carry `seed`: the call draws everything from R's
own stream after set.seed(seed), as the reference would.
"""
from __future__ import annotations

import numpy as np

from . import host


def _lu(r, lo, hi, n=None):
    return np.exp(r.uniform(np.log(lo), np.log(hi), n))


def _pitch_anchors(r, lo, hi):
    n = 2 if r.random() < 0.5 else 12
    return (host.seq_len(0, 1, n), _lu(r, lo, hi, n))


def _formants(r, moving):
    nf = int(r.integers(3, 6))
    freqs = np.sort(r.uniform(300, 5000, nf))
    out = []
    for f in freqs:
        amp, width = r.uniform(20, 50), r.uniform(50, 300)
        if moving:
            f2 = float(np.clip(f * r.uniform(0.8, 1.25), 300, 5000))
            out.append(np.array([[0, f, amp, width], [1, f2, r.uniform(20, 50), r.uniform(50, 300)]]))
        else:
            out.append(np.array([[0, f, amp, width]]))
    return out


def noise_uniform_count(length, wl, overlap=75):
    h = wl - (overlap * wl / 100)
    return (wl // 2) * host.seq_by_count(1.0, float(length) + wl, h)


def config0(n=1, seed=1):
    """The literal reference call `set.seed(k); soundgen(sylLen = 1000)`: every default, i.e. the
    4-anchor loess pitch contour, temperature 0.025, vowel 'a' formants, 16 kHz."""
    return [dict(sylLen=1000, seed=seed + i) for i in range(n)]


def config1(n=1024, seed=20260001):
    """1024 voiced syllables x 500 ms at 44.1 kHz, randomised pitch, rolloff and formants."""
    r = np.random.default_rng(seed)
    out = []
    for i in range(n):
        out.append(dict(
            sylLen=500, samplingRate=44100, temperature=0, nonlinBalance=0,
            pitchAnchors=_pitch_anchors(r, 80, 800), contour_method='spline',
            rolloff=r.uniform(-24, -6), rolloffOct=r.uniform(-12, 0), rolloffKHz=r.uniform(-12, 0),
            rolloffParab=r.uniform(-20, 20), rolloffParabHarm=int(r.integers(1, 11)),
            formants=_formants(r, moving=(i % 2 == 1))))
    return out


def config2(n=4096, seed=20260002):
    """noise-heavy: n x 2 s at 22.05 kHz with noiseAnchors, breathing / separately filtered
    turbulence and spectral-envelope filtering; weak voiced part."""
    r = np.random.default_rng(seed)
    sr, wl = 22050, 1102
    out = []
    for i in range(n):
        na = 2 if r.random() < 0.5 else 12
        t = np.sort(r.uniform(-100, 2200, na))
        t[0] = -100 + r.uniform(0, 50)
        anchors = (t, r.uniform(-60, 20, na))
        tpos = t.copy()   # sylLen == dur_syl, so the rescale at soundgen.R:647-649 is the identity
        ulen = int(np.rint((np.max(tpos) - np.min(tpos)) * sr / 1000))
        kw = dict(sylLen=2000, samplingRate=sr, temperature=0, nonlinBalance=0,
                  pitchAnchors=_pitch_anchors(r, 100, 400), contour_method='spline',
                  rolloff=-24, noiseAnchors=anchors, rolloffNoise=r.uniform(-14, 0),
                  u=[r.random(noise_uniform_count(ulen, wl))])
        if i % 2 == 1:
            kw['formantsNoise'] = _formants(r, moving=True)[:3]
        out.append(kw)
    return out


def config3(n=8192, seed=20260003):
    """harmonic-rich: n x 1 s at 48 kHz, low pitch, jitter, shimmer, vibrato, subharmonics."""
    r = np.random.default_rng(seed)
    out = []
    for i in range(n):
        out.append(dict(
            sylLen=1000, samplingRate=48000, invalidArgAction='ignore', temperature=0,
            pitchAnchors=_pitch_anchors(r, 50, 120), contour_method='spline',
            rolloff=r.uniform(-6, -1), rolloffOct=0, rolloffKHz=0, nonlinBalance=100,
            jitterDep=r.uniform(0.5, 3), jitterLen=r.uniform(1, 20), shimmerDep=r.uniform(5, 30),
            vibratoFreq=r.uniform(3, 8), vibratoDep=r.uniform(0.25, 2), subFreq=r.uniform(25, 60),
            subDep=r.uniform(20, 150), shortestEpoch=300, z=[r.standard_normal(1024)]))
    return out


def config4(n=65536, seed=0):
    """datagen sweep: call i = `set.seed(seed + i); eval(parse(text = preset[i mod 33]))` in the order of
    R/presets.R:156-410, each preset with its own temperature, loess contours, stochastic formants."""
    from . import presets
    ps = presets.load()
    out = []
    for i in range(n):
        _, _, kw = ps[i % len(ps)]
        kw = dict(kw)
        kw.update(seed=seed + i)
        out.append(kw)
    return out


def _smooth(r, n, lo, hi, log=False):
    """n points of a slow random walk (a measured track, say) rescaled into a random sub-range of [lo, hi],
    log-uniformly when `log`"""
    w = np.cumsum(r.standard_normal(n))
    w = np.convolve(np.pad(w, 4, mode='edge'), np.ones(9) / 9, mode='valid')
    w = (w - w.min()) / max(float(np.ptp(w)), 1e-9)
    a, b = np.sort(r.uniform(0, 1, 2))
    f = a + (b - a) * w
    if log:
        return np.exp(np.log(lo) + (np.log(hi) - np.log(lo)) * f)
    return lo + (hi - lo) * f


def resynthesis(n=4096, seed=20260005, points=101):
    """resynthesis from measured tracks: n x 2 s at 22.05 kHz, temperature 0, one anchor per 20 ms (`points`)
    for pitchAnchors (80-600 Hz), amplAnchors, noiseAnchors, mouthAnchors and amplAnchorsGlobal, and 4 formants
    that move through `points` time points."""
    r = np.random.default_rng(seed)
    sr, wl, dur = 22050, 1102, 2000
    t01 = host.seq_len(0, 1, points)
    out = []
    for i in range(n):
        tms = t01 * dur
        ulen = int(np.rint((tms[-1] - tms[0]) * sr / 1000))
        fm = []
        for f0 in np.sort(r.uniform(400, 4500, 4)):
            fm.append(np.column_stack([t01, _smooth(r, points, 0.8 * f0, 1.25 * f0), _smooth(r, points, 20, 50),
                                       _smooth(r, points, 80, 300)]))
        out.append(dict(
            sylLen=dur, samplingRate=sr, temperature=0, nonlinBalance=0, contour_method='spline',
            pitchAnchors=(t01, _smooth(r, points, 80, 600, log=True)),
            amplAnchors=(t01, _smooth(r, points, 40, 120)),
            noiseAnchors=(tms, _smooth(r, points, -60, 10)),
            mouthAnchors=(t01, _smooth(r, points, 0, 1)),
            amplAnchorsGlobal=(t01, _smooth(r, points, 60, 120)),
            formants=fm, rolloffNoise=-8,
            u=[r.random(noise_uniform_count(ulen, wl))]))
    return out


def thinned(calls, points=60):
    """the same calls with every contour and formant track resampled (linearly) to `points` points"""
    def rs(t, v):
        t = np.asarray(t, dtype=np.float64)
        tn = host.seq_len(float(t[0]), float(t[-1]), points)
        return tn, np.interp(tn, t, np.asarray(v, dtype=np.float64))
    out = []
    for kw in calls:
        kw = dict(kw)
        for k in ('pitchAnchors', 'amplAnchors', 'noiseAnchors', 'mouthAnchors', 'amplAnchorsGlobal'):
            if k in kw:
                kw[k] = rs(*kw[k])
        if 'formants' in kw:
            fm = []
            for f in kw['formants']:
                tn = rs(f[:, 0], f[:, 1])[0]
                fm.append(np.column_stack([tn] + [rs(f[:, 0], f[:, j])[1] for j in (1, 2, 3)]))
            kw['formants'] = fm
        out.append(kw)
    return out


def amp_paths(seed=20260010):
    """One call per code path of the amplitude kernel K3, 400 ms each at 48 kHz: epochs without sub-harmonics on both
    sides of the tensor-core row threshold (224) and with more than 1024 kept rows, dense sub-harmonic epochs up to
    more than 2560 rows, sub-harmonic epochs of fewer than 512 rows, and untabled epochs (more than 16 sub-harmonics,
    or more than 1024 kept rows with sub-harmonics)."""
    r = np.random.default_rng(seed)
    cases = [(60, 90, 35, 60),      # dense: 600-1900 rows, several epochs
             (50, 55, 9, 100),      # n = 5 on up to 479 kept rows: more than 2560 rows
             (100, 110, 40, 0),     # no sub-harmonics, > 224 rows
             (400, 420, 40, 0),     # no sub-harmonics, < 224 rows
             (300, 320, 150, 80),   # n = 1, < 512 rows (and < 224)
             (180, 200, 90, 80),    # n = 1, 224-512 rows
             (80, 160, 60, 80),     # epochs without and with sub-harmonics in one syllable
             (400, 410, 20, 100),   # n > 16: untabled
             (21, 22, 40, 0),       # > 1024 kept rows, no sub-harmonics
             (21, 22, 10, 100)]     # > 1024 kept rows with sub-harmonics: untabled
    out = []
    for lo, hi, sub_freq, sub_dep in cases:
        out.append(dict(
            sylLen=400, samplingRate=48000, invalidArgAction='ignore', temperature=0, pitchFloor=1,
            pitchAnchors=(host.seq_len(0, 1, 2), [lo, hi]), contour_method='spline',
            rolloff=r.uniform(-6, -1), rolloffOct=0, rolloffKHz=0, nonlinBalance=100,
            jitterDep=r.uniform(0.5, 2), jitterLen=r.uniform(1, 20), shimmerDep=r.uniform(5, 30),
            subFreq=sub_freq, subDep=sub_dep, shortestEpoch=100, z=[r.standard_normal(1024)]))
    return out


CONFIGS = {0: config0, 1: config1, 2: config2, 3: config3, 4: config4}
NAMES = {0: 'cfg0 soundgen() defaults, 1 x 1000 ms @ 16 kHz',
         1: 'cfg1 voiced batch, 1024 x 500 ms @ 44.1 kHz',
         2: 'cfg2 noise-heavy batch, 4096 x 2 s @ 22.05 kHz',
         3: 'cfg3 harmonic-rich batch, 8192 x 1 s @ 48 kHz',
         4: 'cfg4 datagen sweep over the 33 bundled presets, set.seed(i) each'}
SAMPLING_RATE = {0: 16000, 1: 44100, 2: 22050, 3: 48000, 4: None}   # cfg4: per call
