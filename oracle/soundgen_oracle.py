"""CPU restatement of soundgen's source-filter synthesis path.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) -- PARITY UNPINNED: no golden
vectors exist in the reference and R is not available here, so this file is the
parity target for the CUDA path, itself pinned only by SURVEY.md Appendix B.

Every function cites the reference lines it restates (paths relative to
/root/reference; `seewave.r` = R/seewave.r inside
packrat/src/seewave/seewave_2.0.5.tar.gz).  All arithmetic is IEEE double like
R's; indices are kept 1-based where the reference's results are indices, so the
integer artefacts can be compared directly.

Random draws are never made here: every stochastic component takes its draws
from an `RStream`, which hands out pre-drawn standard normals / uniforms in the
order R would consume them (SURVEY.md 8a "RNG ledger").
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

from .rprims import (fmm_coef, fmm_eval, hamming_w, hanning_w, r_approx,
                     r_cumsum, r_mean, r_round, r_seq_by, r_seq_len_out,
                     r_spline, r_sum)

# --------------------------------------------------------------------------
# tables (R/presets.R:22-79; data-raw/noiseThresholdsDict.R:4-18)
# --------------------------------------------------------------------------
PERMITTED = {  # name: (default, low, high, step)
    'repeatBout': (1, 1, 20, 1), 'nSyl': (1, 1, 10, 1),
    'sylLen': (300, 20, 5000, 10), 'pauseLen': (200, 20, 1000, 10),
    'temperature': (.025, 0, 1, .025), 'maleFemale': (0, -1, 1, 0.1),
    'creakyBreathy': (0, -1, 1, 0.1), 'nonlinBalance': (0, 0, 100, 1),
    'nonlinDep': (50, 0, 100, 1), 'jitterDep': (3, 0, 24, 0.1),
    'jitterLen': (1, 1, 100, 1), 'vibratoFreq': (5, 3, 10, .5),
    'vibratoDep': (0, 0, 3, 0.125), 'shimmerDep': (0, 0, 100, 1),
    'attackLen': (50, 0, 200, 10), 'rolloff': (-12, -60, 0, 1),
    'rolloffOct': (-12, -30, 10, 1), 'rolloffParab': (0, -50, 50, 5),
    'rolloffParabHarm': (3, 1, 20, 1), 'rolloffKHz': (-6, -20, 0, 1),
    'rolloffLip': (6, 0, 20, 1), 'formantDep': (1, 0, 5, .1),
    'formantDepStoch': (30, 0, 60, 10), 'vocalTract': (15.5, 2, 100, .5),
    'subFreq': (100, 10, 1000, 10), 'subDep': (100, 0, 500, 10),
    'shortestEpoch': (300, 50, 500, 25), 'amDep': (0, 0, 100, 5),
    'amFreq': (30, 10, 100, 5), 'amShape': (0, -1, 1, .025),
    'samplingRate': (16000, 8000, 44100, 100),
    'windowLength': (40, 5, 100, 2.5), 'rolloffNoise': (-14, -20, 20, 1),
    'overlap': (50, 0, 99, 1), 'addSilence': (100, 0, 1000, 50),
    'pitchFloor': (50, 1, 1000, 1), 'pitchCeiling': (3500, 10, 100000, 10),
    'pitchSamplingRate': (3500, 10, 100000, 10),
    'throwaway': (-120, -200, -10, 10),
    'specWindowLength': (40, 5, 100, 2.5), 'specContrast': (.2, -1, 1, .05),
    'specBrightness': (0, -1, 1, .05), 'mouthOpening': (.5, 0, 1, .05),
    'pitch': (100, 25, 3500, 1), 'pitchDeltas': (0, -24, 24, 1),
    'time': (0, 0, 5000, 1), 'noiseAmpl': (0, -120, 40, 1),
}
CHECKED_PARS = list(PERMITTED)[:list(PERMITTED).index('rolloffNoise') + 1]


def noise_thresholds(nonlinBalance):
    """noiseThresholdsDict$q1/q2[nonlinBalance + 1]; a fractional nonlinBalance is
    truncated by R's indexing (utilities_math.R:361-363)."""
    a = float(int(nonlinBalance + 1) - 1)
    q1 = 100.0 / (1.0 + math.exp(0.1 * (a - 33.0)))
    q2 = 100.0 / (1.0 + math.exp(0.1 * (a - 66.0)))
    return q1, q2


class RStream:
    """Pre-drawn random numbers handed out in R's consumption order.
    `z`: standard normals (R `norm_rand()` values); `u`: uniforms."""

    def __init__(self, z=None, u=None):
        self.z = np.zeros(0) if z is None else np.asarray(z, dtype=np.float64)
        self.u = np.zeros(0) if u is None else np.asarray(u, dtype=np.float64)
        self.zi = 0
        self.ui = 0

    def rnorm(self, n, mean=0.0, sd=1.0):
        n = int(n)
        if self.zi + n > self.z.size:
            raise IndexError('normal stream exhausted')
        z = self.z[self.zi:self.zi + n]
        self.zi += n
        mean = np.resize(np.asarray(mean, dtype=np.float64), n)  # R recycles
        return mean + sd * z

    def runif(self, n):
        n = int(n)
        if self.ui + n > self.u.size:
            raise IndexError('uniform stream exhausted')
        u = self.u[self.ui:self.ui + n]
        self.ui += n
        return u


# --------------------------------------------------------------------------
# small utilities (R/utilities_math.R, R/utilities_soundgen.R)
# --------------------------------------------------------------------------
def HzToSemitones(h):  # utilities_math.R:16-18
    return np.log2(np.asarray(h, dtype=np.float64) / 16.3516) * 12


def semitonesToHz(s):  # utilities_math.R:25-27
    return 16.3516 * 2 ** (np.asarray(s, dtype=np.float64) / 12)


def zeroOne(x):  # utilities_math.R:58-61
    x = x - np.min(x)
    return x / np.max(x)


def matchLengths(myseq, length, padWith=0.0):
    """utilities_math.R:413-444, padDir = 'central'."""
    myseq = np.asarray(myseq, dtype=np.float64)
    length = int(length)
    if myseq.size == length:
        return myseq
    if myseq.size < length:
        pad = np.full(length, padWith)
        myseq = np.concatenate((pad, myseq, pad))
    halflen = length / 2
    center = (1 + myseq.size) / 2
    start = int(math.ceil(center - halflen))
    return myseq[start - 1:start - 1 + length]


def addVectors(v1, v2, insertionPoint):
    """utilities_math.R:500-526, including the `insertionPoint` (not -1) zero
    padding of v2 (:507-509)."""
    v1 = np.nan_to_num(np.asarray(v1, dtype=np.float64), nan=0.0)
    v2 = np.nan_to_num(np.asarray(v2, dtype=np.float64), nan=0.0)
    insertionPoint = int(insertionPoint)
    if insertionPoint > 1:
        v2 = np.concatenate((np.zeros(insertionPoint), v2))
    elif insertionPoint < 1:
        v1 = np.concatenate((np.zeros(1 - insertionPoint), v1))
    d = v2.size - v1.size
    if d > 0:
        v1 = np.concatenate((v1, np.zeros(d)))
    elif d < 0:
        v2 = np.concatenate((v2, np.zeros(-d)))
    return v1 + v2


def clumper(s, minLength):
    """utilities_math.R:555-600."""
    s = np.array(s, dtype=np.float64)
    minLength = np.atleast_1d(np.asarray(minLength, dtype=np.float64))
    if np.max(minLength) < 2:
        return s
    minLength = r_round(minLength)
    n = s.size
    if (np.unique(s).size < 2 or (minLength.size == 1 and n < minLength[0])
            or n < minLength[0]):
        return np.full(n, r_round(np.median(s)))
    if minLength.size == 1 or minLength.size != n:
        minLength = np.resize(minLength, n)
    c = 0
    for i in range(1, n):  # R: i in 2:length(s)
        if s[i - 1] == s[i]:
            c += 1
        else:
            if c < minLength[i]:
                s[i] = s[i - 1]
                c += 1
            else:
                c = 1
    ml = int(minLength[-1])
    lo = max(n - ml + 1, 2)
    idx_min = np.arange(lo, n + 1)  # 1-based
    if np.sum(s[idx_min - 1] == s[-1]) < ml:
        idx = idx_min[::-1]
        c = 1
        i = 2
        while i <= idx.size and s[idx[i - 1] - 1] == s[idx[i - 1] - 2] and i < idx.size:
            c += 1
            i += 1
        if c < ml:
            s[idx - 1] = s[idx_min.min() - 1]
    return s


def getRandomWalk(length, rng, rw_range=1.0, rw_smoothing=.2, method='spline',
                  trend=0.0):
    """utilities_math.R:289-326.  `trend` may be a callable: R passes `trend = rnorm(1)` as a
    promise, which is only forced (drawn) once `length(trend)` is looked at, i.e. when len >= 2."""
    length = int(length)
    if length < 2:
        return np.array([rng.rgamma(1, 1 / rw_range ** 2, 1 / rw_range ** 2)[0]])
    if callable(trend):
        trend = trend()
    with np.errstate(over='ignore', divide='ignore'):
        p = 2.0 ** (1.0 / rw_smoothing) if rw_smoothing != 0 else np.inf
    n = math.floor(max(2.0, p)) if np.isfinite(p) else np.inf
    trend = np.atleast_1d(np.asarray(trend, dtype=np.float64))
    if trend.size > 1:
        n = r_round(n / 2) * 2
        n = int(n) if np.isfinite(n) else n
        trend_short = np.repeat(trend, int(n // trend.size)) if np.isfinite(n) else trend
    else:
        trend_short = trend
    if n > length:
        rw_long = r_cumsum(rng.rnorm(length, trend_short))
    else:
        n = int(n)
        rw_short = r_cumsum(rng.rnorm(n, trend_short))
        if method == 'linear':
            rw_long = r_approx(rw_short, length)
        else:
            rw_long = r_spline(rw_short, length)
    rw_normalized = rw_long - np.min(rw_long)
    rw_normalized = rw_normalized / np.max(np.abs(rw_normalized)) * rw_range
    return rw_normalized


def getIntegerRandomWalk(rw, nonlinBalance=50, minLength=50):
    """utilities_math.R:352-387."""
    n = rw.size
    if nonlinBalance == 0:
        return np.zeros(n)
    if nonlinBalance == 100:
        return np.full(n, 2.0)
    q1, q2 = noise_thresholds(nonlinBalance)
    rw_bin = np.zeros(n)
    rw_bin[rw > q1] = 1
    rw_bin[rw > q2] = 2
    return clumper(rw_bin, minLength)


def getSigmoid(length, samplingRate=16000, freq=5, shape=0, spikiness=1):
    """utilities_math.R:639-653."""
    frm = -math.exp(-shape * spikiness)
    to = math.exp(shape * spikiness)
    slope = math.exp(abs(shape)) * 5
    a = r_seq_len_out(frm, to, samplingRate / freq / 2)
    b = 1 / (1 + np.exp(-a * slope))
    b = zeroOne(b)
    return np.resize(np.concatenate((b, b[::-1])), int(length))


def getGlottalCycles(pitch, samplingRate):
    """utilities_soundgen.R:477-486.  Returns 1-based indices."""
    gc = []
    i = 1
    n = len(pitch)
    while i < n:
        gc.append(i)
        i = i + max(2, math.floor(samplingRate / pitch[i - 1]))
    return np.array(gc, dtype=np.int64)


def upsample(pitch_per_gc, samplingRate=16000):
    """utilities_soundgen.R:392-416.  Returns (pitch_upsampled, gc_upsampled)."""
    p = np.asarray(pitch_per_gc, dtype=np.float64)
    l = p.size
    gclen = r_round(samplingRate / p)
    c = r_cumsum(gclen)
    gc_up = np.concatenate(([1.0], c)).astype(np.int64)
    if l == 1:
        pu = np.repeat(p, int(gclen[0]))
    elif l == 2:
        pu = r_seq_len_out(p[0], p[1], r_sum(gclen))
    else:
        t = np.ones(l)
        t[l - 1] = r_sum(gclen)
        for i in range(2, l):  # R i = 2..l-1
            t[i - 1] = c[i - 2] + r_round(gclen[i - 1] / 2)
        pu = r_spline(p, int(c[-1]), x=t)
    return pu, gc_up


def findZeroCrossing(ampl, location):
    """utilities_soundgen.R:255-295 (1-based in/out; None = NA)."""
    n = len(ampl)
    if n < 1 or location < 1 or location > n:
        return None
    if n == 1 and location == 1:
        return location
    zc_left = zc_right = None
    i = 1  # R leaves `i` undefined only when location == 1 == len (handled above)
    if location > 1:
        i = location
        while i > 1:
            if ampl[i - 1] > 0 and ampl[i - 2] < 0:
                zc_left = i - 1
                break
            i -= 1
    if location < n:
        i = location
    while i < n - 1:
        if ampl[i] > 0 and ampl[i - 1] < 0:
            zc_right = i
            break
        i += 1
    if zc_left is None and zc_right is None:
        return None
    if zc_left is None:
        return zc_right
    if zc_right is None:
        return zc_left
    return zc_left if abs(zc_left - location) <= abs(zc_right - location) else zc_right


def crossFade(ampl1, ampl2, samplingRate, crossLen=15, crossLenPoints=None):
    """utilities_soundgen.R:328-375.  Also returns (zc1, zc2) for artefact checks."""
    ampl1 = np.atleast_1d(np.asarray(ampl1, dtype=np.float64))
    ampl2 = np.atleast_1d(np.asarray(ampl2, dtype=np.float64))
    zc1 = findZeroCrossing(ampl1, len(ampl1))
    if zc1 is not None:
        ampl1 = np.concatenate((ampl1[:zc1], [0.0]))
    zc2 = findZeroCrossing(ampl2, 1)
    if zc2 is not None:
        ampl2 = ampl2[zc2:]
    if crossLenPoints is None:
        crossLenPoints = min(math.floor(crossLen * samplingRate / 1000),
                             len(ampl1) - 1, len(ampl2) - 1)
    else:
        crossLenPoints = min(crossLenPoints, len(ampl1) - 1, len(ampl2) - 1)
    if crossLenPoints < 2:
        out = np.concatenate((ampl1, ampl2))
    else:
        multipl = r_seq_len_out(0, 1, crossLenPoints)
        idx1 = len(ampl1) - crossLenPoints
        cross = multipl[::-1] * ampl1[idx1:] + multipl * ampl2[:crossLenPoints]
        out = np.concatenate((ampl1[:idx1], cross, ampl2[crossLenPoints:]))
    return out, zc1, zc2


def fadeInOut(ampl, do_fadeIn=True, do_fadeOut=True, length_fade=1000):
    """utilities_soundgen.R:440-459."""
    ampl = np.array(ampl, dtype=np.float64)
    if (not do_fadeIn and not do_fadeOut) or length_fade < 2:
        return ampl
    length_fade = int(min(length_fade, ampl.size))
    fadeIn = r_seq_len_out(0, 1, length_fade)
    if do_fadeIn:
        ampl[:length_fade] = ampl[:length_fade] * fadeIn
    if do_fadeOut:
        ampl[ampl.size - length_fade:] = ampl[ampl.size - length_fade:] * fadeIn[::-1]
    return ampl


# --------------------------------------------------------------------------
# contours (R/smoothContours.R)
# --------------------------------------------------------------------------
def getSmoothContour(anchors, length=None, thisIsPitch=False, method='loess',
                     valueFloor=None, valueCeiling=None, samplingRate=16000):
    """smoothContours.R:53-227.  `anchors` = (time[], value[]).  The loess branch
    (3-10 anchors, the R default) goes through oracle/rloess.py."""
    if anchors is None:
        return None
    time = np.array(anchors[0], dtype=np.float64)
    value = np.array(anchors[1], dtype=np.float64)
    n = time.size
    if n > 10 and method == 'loess':
        method = 'spline'
    if valueFloor is not None:
        value[value < valueFloor] = valueFloor
    if valueCeiling is not None:
        value[value > valueCeiling] = valueCeiling
    if thisIsPitch:
        value = HzToSemitones(value)
        if valueFloor is not None:
            valueFloor = float(HzToSemitones(valueFloor))
        if valueCeiling is not None:
            valueCeiling = float(HzToSemitones(valueCeiling))
    if length is None:
        duration_ms = np.max(time) - np.min(time)
        length = math.floor(duration_ms * samplingRate / 1000)
    else:
        time = time - np.min(time)
        with np.errstate(invalid='ignore', divide='ignore'):
            time = time / np.max(time)
        duration_ms = length / samplingRate * 1000
    length = int(length)
    if duration_ms == 0 or length == 0:
        return None
    if n == 1:
        sc = np.full(length, value[0])
    elif n == 2:
        sc = r_seq_len_out(value[0], value[1], length)
    else:
        if method == 'spline':
            sc = r_spline(value, length, x=time)
        else:
            from .rloess import smooth_contour_loess
            sc, _ = smooth_contour_loess(time, value, length, duration_ms, n, valueFloor)
        with np.errstate(invalid='ignore'):
            if valueFloor is not None:
                sc[sc < valueFloor] = valueFloor
            if valueCeiling is not None:
                sc[sc > valueCeiling] = valueCeiling
    sc = np.nan_to_num(sc, nan=0.0)
    if thisIsPitch:
        sc = semitonesToHz(sc)
    return sc


# --------------------------------------------------------------------------
# spectral shaping (R/sourceSpectrum.R, R/subharmonics.R)
# --------------------------------------------------------------------------
def getRolloff(pitch_per_gc, nHarmonics=100, rolloff=-12, rolloffOct=-2,
               rolloffParab=0, rolloffParabHarm=2, rolloffParabCeiling=None,
               rolloffKHz=-6, baseline=200, throwaway=-120, samplingRate=16000):
    """sourceSpectrum.R:71-186.  Returns (matrix rows x G, rownames 1..rows)."""
    p = np.atleast_1d(np.asarray(pitch_per_gc, dtype=np.float64))
    G = p.size
    nH = int(nHarmonics)
    rolloff = np.resize(np.atleast_1d(np.asarray(rolloff, dtype=np.float64)), G)
    rolloffOct = np.resize(np.atleast_1d(np.asarray(rolloffOct, dtype=np.float64)), G)
    rolloffKHz = np.resize(np.atleast_1d(np.asarray(rolloffKHz, dtype=np.float64)), G)
    h = np.arange(1, nH + 1, dtype=np.float64)[:, None]
    deltas = np.zeros((nH, G))
    if np.sum(rolloffOct != 0) > 0:
        deltas[1:, :] = (rolloffOct[None, :] * (p[None, :] * h[1:] - baseline) / 1000)
    r = ((rolloff + rolloffKHz * (p - baseline) / 1000)[None, :] * np.log2(h)) + deltas
    r[h * p[None, :] >= samplingRate / 2] = -np.inf
    if rolloffParab != 0:
        if rolloffParabCeiling is not None:
            PH = r_round(rolloffParabCeiling / p)
        else:
            PH = np.full(G, float(r_round(rolloffParabHarm)))
        PH[PH == 2] = 3
        with np.errstate(divide='ignore'):
            a = -4 * rolloffParab / (PH - 1) ** 2
        b = -a * (1 + PH)
        c = a * PH
        sel = PH < 3
        r[0, sel] = r[0, sel] + rolloffParab
        for i in np.nonzero(PH >= 3)[0]:
            k = int(PH[i])
            rows = np.arange(1, k + 1, dtype=np.float64)
            r[:k, i] = r[:k, i] + a[i] * rows ** 2 + b[i] * rows + c[i]
    if throwaway is not None:
        r[r < throwaway] = -np.inf
    r = r - np.max(r, axis=0)[None, :]
    r = 2 ** (r / 10)
    keep = np.array([r_sum(r[k, :]) > 0 for k in range(nH)])
    r = r[keep, :]
    return r, np.arange(1, r.shape[0] + 1, dtype=np.float64)


def _r_name_roundtrip(v):
    """as.numeric(as.character(v)): rownames keep 15 significant digits
    (subharmonics.R:39 -> source.R:401)."""
    return float('%.15g' % v)


def getVocalFry_per_epoch(rolloff, names, pitch_per_gc, nSubharm, sideband_width_vector,
                          throwaway01):
    """subharmonics.R:25-86 incl. the scalar-index quirk at :76-77
    (`rolloff_new[row_lwr]` = column 1 of that row)."""
    nSubharm = int(nSubharm)
    if nSubharm < 1:
        return rolloff, names
    H, G = rolloff.shape
    by = 1 / (nSubharm + 1)
    g_seq = r_seq_by(0, H + 1, by)
    R = np.full((g_seq.size, G), np.nan)
    R[0, :] = 0
    R[-1, :] = 0
    for k in range(1, H + 1):
        R[k * (nSubharm + 1), :] = rolloff[k - 1, :]
    sw = np.asarray(sideband_width_vector, dtype=np.float64)

    def dnorm0(d):  # dnorm(d, 0, sw) / dnorm(0, 0, sw); sd == 0, d > 0 -> 0
        with np.errstate(divide='ignore', invalid='ignore'):
            out = np.exp(-0.5 * (d / sw) ** 2)
        return np.where(sw == 0, np.where(d == 0, np.nan, 0.0), out)

    multipl_lwr = [dnorm0(pitch_per_gc * s / (nSubharm + 1)) for s in range(1, nSubharm + 1)]
    multipl_upr = multipl_lwr[::-1]
    for block in range(1, H + 2):
        row_lwr = 1 + (block - 1) * (nSubharm + 1)
        row_upr = row_lwr + nSubharm + 1
        for g in range(1, nSubharm + 1):
            harm_g = R[row_lwr - 1, 0] * multipl_lwr[g - 1] + R[row_upr - 1, 0] * multipl_upr[g - 1]
            R[row_lwr + g - 1, :] = harm_g
    R[R < throwaway01] = 0
    keep = np.array([r_sum(R[k, :]) > 0 for k in range(R.shape[0])])
    nm = np.array([_r_name_roundtrip(v) for v in g_seq])
    return R[keep, :], nm[keep]


def getVocalFry(rolloff, names, pitch_per_gc, subFreq=100, subDep=100, throwaway=-120,
                shortestEpoch=300):
    """subharmonics.R:108-163.  Returns (list of (matrix, rownames), epochs (start,end) 1-based,
    nSubharm per gc after clumping)."""
    p = np.asarray(pitch_per_gc, dtype=np.float64)
    G = p.size
    subFreq = np.resize(np.atleast_1d(np.asarray(subFreq, dtype=np.float64)), G)
    nSubharm = r_round(p / subFreq) - 1
    nSubharm[nSubharm < 0] = 0
    if np.max(nSubharm) < 1:
        return [(rolloff, names)], np.array([[1, G]]), nSubharm
    subDep = np.atleast_1d(np.asarray(subDep, dtype=np.float64))
    if subDep.size < G:
        subDep = np.full(G, subDep[0])
    throwaway01 = 2 ** (throwaway / 10)
    period_ms = 1000 / p
    min_epoch_length_points = r_round(shortestEpoch / period_ms)
    if G > 1:
        nSubharm = clumper(nSubharm, min_epoch_length_points)
    change = np.nonzero(np.diff(nSubharm) != 0)[0] + 1  # 1-based last idx before change
    starts = np.concatenate(([1], change + 1))
    ends = np.concatenate((change, [G]))
    per_epoch = nSubharm[np.concatenate((change, [G])) - 1]
    out = []
    for e in range(starts.size):
        sl = slice(starts[e] - 1, ends[e])
        out.append(getVocalFry_per_epoch(rolloff[:, sl], names, p[sl], per_epoch[e],
                                         subDep[sl], throwaway01))
    return out, np.stack((starts, ends), axis=1), nSubharm


# --------------------------------------------------------------------------
# generateHarmonics (R/source.R:173-471)
# --------------------------------------------------------------------------
@dataclass
class HarmonicsArtefacts:
    gc: np.ndarray = None              # glottal cycle starts on the pitch grid (1-based)
    gc_upsampled: np.ndarray = None    # 1-based, length G+1
    pitch_per_gc: np.ndarray = None    # after jitter/drift/clamp
    nHarmonics: int = 0
    rows_kept: int = 0
    epochs: np.ndarray = None          # (E,2) 1-based gc indices
    nSubharm: np.ndarray = None
    rw_bin: np.ndarray = None
    jitter_idx: np.ndarray = None
    zc: list = field(default_factory=list)   # (zc1, zc2) per epoch
    epoch_rows: list = field(default_factory=list)
    n_upsampled: int = 0
    z_used: int = 0
    raw_max: float = 0.0               # max(waveform) before normalisation
    mats: list = None                  # per-epoch (matrix, rownames)
    integr: np.ndarray = None          # cumsum(pitch_upsampled) / samplingRate
    epoch_waves: list = field(default_factory=list)
    ampl_gain: np.ndarray = None       # 2^(amplEnvelope / 10) per sample of the joined waveform, or None
    drift_upsampled: np.ndarray = None # drift gain per sample of the output (temperature > 0), or None


def generateHarmonics(pitch, attackLen=50, nonlinBalance=0, nonlinDep=0, jitterDep=0,
                      jitterLen=1, vibratoFreq=100, vibratoDep=0, shimmerDep=0,
                      creakyBreathy=0, rolloff=-18, rolloffOct=-2, rolloffKHz=-6,
                      rolloffParab=0, rolloffParabHarm=3, rolloffLip=6, rolloff_perAmpl=12,
                      temperature=0, pitchDriftDep=.5, pitchDriftFreq=.125,
                      randomWalk_trendStrength=.5, shortestEpoch=300, subFreq=100, subDep=0,
                      amDep=0, amFreq=30, amplAnchors=None, overlap=75, samplingRate=16000,
                      pitchFloor=75, pitchCeiling=3500, pitchSamplingRate=3500,
                      throwaway=-120, rng=None, contour_method='loess', want_artefacts=False):
    """R/source.R:173-471.  `rng` supplies the normal stream; `amplAnchors` =
    (time[], value[]) or None."""
    rng = rng or RStream()
    art = HarmonicsArtefacts()
    pitch = np.array(pitch, dtype=np.float64)
    if vibratoDep > 0:  # :208-213
        k = np.arange(1, pitch.size + 1, dtype=np.float64)
        vibrato = 2 ** (np.sin(2 * np.pi * k * vibratoFreq / pitchSamplingRate) * vibratoDep / 12)
        pitch = pitch * vibrato
    gc = getGlottalCycles(pitch, pitchSamplingRate)  # :216
    pitch_per_gc = pitch[gc - 1]
    nGC = pitch_per_gc.size
    art.gc = gc

    use_ampl = amplAnchors is not None and np.sum(np.asarray(amplAnchors[1]) < -throwaway) > 0
    if use_ampl:  # :221-235
        amplContour = getSmoothContour(amplAnchors, length=nGC, valueFloor=0,
                                       valueCeiling=-throwaway, samplingRate=samplingRate,
                                       method=contour_method)
        amplContour = amplContour / abs(throwaway) - 1
        rolloffAmpl = amplContour * rolloff_perAmpl
    else:
        rolloffAmpl = 0.0

    if temperature > 0:  # :238-258
        rw = getRandomWalk(nGC, rng, rw_range=temperature,
                           trend=[randomWalk_trendStrength, -randomWalk_trendStrength],
                           rw_smoothing=.3)
        rw_0_100 = zeroOne(rw) * 100
        rw_bin = getIntegerRandomWalk(rw_0_100, nonlinBalance=nonlinBalance,
                                      minLength=np.ceil(shortestEpoch / 1000 * pitch_per_gc))
        rw = rw - r_mean(rw) + 1
        vocalFry_on = (rw_bin > 0).astype(np.float64)
        jitter_on = shimmer_on = (rw_bin == 2).astype(np.float64)
        art.rw_bin = rw_bin
    else:
        rw = np.ones(nGC)
        vocalFry_on = jitter_on = shimmer_on = np.ones(nGC)

    if jitterDep > 0 and nonlinBalance > 0:  # :265-290
        ratio = pitch_per_gc * jitterLen / 1000
        idx = [1.0]
        i = 1.0
        while i < nGC:
            i = idx[-1] + ratio[int(i) - 1]
            idx.append(i)
        idx = r_round(np.array(idx))
        idx = idx[idx <= nGC]
        _, first = np.unique(idx, return_index=True)
        idx = idx[np.sort(first)].astype(np.int64)
        art.jitter_idx = idx
        jitter = 2 ** (rng.rnorm(idx.size, 0, jitterDep / 12) * rw[idx - 1] * jitter_on[idx - 1])
        jitter_per_gc = r_spline(jitter, nGC, x=idx.astype(np.float64))
        pitch_per_gc = pitch_per_gc * jitter_per_gc

    drift = None
    if temperature > 0:  # :293-320
        rw_smoothing = .9 - temperature * pitchDriftFreq - 1.2 / (1 + math.exp(-.008 * (nGC - 10))) + .6
        rw_range = temperature * pitchDriftDep + nGC / 1000 / 12
        drift = getRandomWalk(nGC, rng, rw_range=rw_range, rw_smoothing=rw_smoothing,
                              method='spline')
        drift = 2 ** (drift - r_mean(drift))
        pitch_per_gc = pitch_per_gc * drift

    pitch_per_gc = np.minimum(pitch_per_gc, pitchCeiling)  # :324-325
    pitch_per_gc = np.maximum(pitch_per_gc, pitchFloor)
    art.pitch_per_gc = pitch_per_gc

    pmin = np.min(pitch_per_gc)
    nHarmonics = int(math.ceil((samplingRate / 2 - pmin) / pmin))  # :329
    art.nHarmonics = nHarmonics
    rolloff_source, names = getRolloff(  # :331-341
        pitch_per_gc, nHarmonics, rolloff=(rolloff + rolloffAmpl) * rw ** 3,
        rolloffOct=rolloffOct * rw ** 3, rolloffKHz=rolloffKHz * rw,
        rolloffParab=rolloffParab, rolloffParabHarm=rolloffParabHarm,
        samplingRate=samplingRate, throwaway=throwaway)
    art.rows_kept = rolloff_source.shape[0]

    if shimmerDep > 0 and nonlinBalance > 0:  # :348-357
        shimmer = 2 ** (rng.rnorm(nGC, 0, shimmerDep / 100) * rw * shimmer_on)
        rolloff_source = rolloff_source * shimmer[None, :]

    if subDep > 0 and nonlinBalance > 0:  # :360-375
        mats, epochs, nSub = getVocalFry(rolloff_source, names, pitch_per_gc,
                                         subFreq=subFreq * rw ** 4,
                                         subDep=subDep * rw ** 4 * vocalFry_on,
                                         shortestEpoch=shortestEpoch, throwaway=throwaway)
        art.nSubharm = nSub
    else:
        mats = [(rolloff_source, names)]
        epochs = np.array([[1, nGC]])
    art.epochs = epochs
    art.epoch_rows = [m[1] for m in mats]
    art.mats = mats

    pitch_upsampled, gc_upsampled = upsample(pitch_per_gc, samplingRate)  # :382
    art.gc_upsampled = gc_upsampled
    art.n_upsampled = pitch_upsampled.size
    integr = r_cumsum(pitch_upsampled) / samplingRate  # :385
    art.integr = integr
    waveform = np.zeros(1)  # `waveform = 0`

    for e in range(epochs.shape[0]):  # :389-427
        idx_gc_up = gc_upsampled[epochs[e, 0] - 1:epochs[e, 1] + 1]
        lo, hi = int(idx_gc_up.min()), int(idx_gc_up.max())
        n_e = hi - lo + 1
        integr_epoch = integr[lo - 1:hi]
        mat, nm = mats[e]
        waveform_epoch = np.zeros(n_e)
        xk = idx_gc_up[:-1].astype(np.float64)
        two_pi_integr = 2 * np.pi * integr_epoch
        for h in range(mat.shape[0]):
            am_upsampled = r_approx(mat[h, :], n_e, x=xk)
            waveform_epoch = waveform_epoch + np.sin(two_pi_integr * nm[h]) * am_upsampled
        if want_artefacts:
            art.epoch_waves.append(waveform_epoch)
        waveform, zc1, zc2 = crossFade(waveform, waveform_epoch, samplingRate, crossLen=15)
        art.zc.append((zc1, zc2))

    if use_ampl:  # :436-448
        amplEnvelope = getSmoothContour(amplAnchors, length=waveform.size, valueFloor=0,
                                        samplingRate=samplingRate, method=contour_method)
        art.ampl_gain = 2 ** (amplEnvelope / 10)
        waveform = waveform * art.ampl_gain
    art.raw_max = float(np.max(waveform))
    waveform = waveform / np.max(waveform)  # :449 signed max
    if attackLen > 0:  # :452-456
        waveform = fadeInOut(waveform, length_fade=math.floor(attackLen * samplingRate / 1000))
    if temperature > 0:  # :459-467
        drift_upsampled = r_approx(drift, waveform.size, x=gc_upsampled[:-1].astype(np.float64))
        art.drift_upsampled = drift_upsampled
        waveform = waveform * drift_upsampled
    art.z_used = getattr(rng, "zi", None)
    return (waveform, art) if want_artefacts else waveform


# --------------------------------------------------------------------------
# getSpectralEnvelope (R/sourceSpectrum.R:261-566), deterministic part.
# --------------------------------------------------------------------------
def upsample_formants(formants, nc, smoothLinearFactor=1):
    """sourceSpectrum.R:321-344.  `formants` = list of arrays (k,4) with columns
    time, freq, amp, width.  Returns list of (nc,4) arrays."""
    nPoints = max(f.shape[0] for f in formants)
    out = []
    for f in formants:
        f = np.asarray(f, dtype=np.float64)
        cols = []
        for j in range(4):
            y = f[:, j]
            if f.shape[0] > 1:
                a = r_approx(y, nPoints + 2 ** smoothLinearFactor, x=f[:, 0])
                cols.append(r_spline(a, nc))
            else:
                cols.append(np.full(nc, y[0]))
        out.append(np.stack(cols, axis=1))
    return out


def getSpectralEnvelope(nr, nc, formants=None, formantDep=1, rolloffLip=6, mouthAnchors=None,
                        mouthOpenThres=0, openMouthBoost=0, vocalTract=None, temperature=0,
                        smoothLinearFactor=1, samplingRate=16000, speedSound=35400,
                        formants_upsampled=None, contour_method='loess', formDrift=.3, formDisp=.2,
                        formantDepStoch=30, rng=None, terms=None):
    """sourceSpectrum.R:261-566 with temperature == 0 (the stochastic block
    :346-415 draws rgamma/rnorm on the host; pass its result via
    `formants_upsampled`).  `formants`: list of (k,4) arrays or None.
    `terms` (a dict) receives the intermediates an error bound needs: 'tracks' (the formant tracks in Hz after
    the stochastic block), 'smoothed' (the tracks or the mouth opening come from a contour), 'bins' (the (nc, 4) rows of every gamma bump in bins, nasal pole and zero included),
    'mouth_open', 'mouth_bin', 'formantDep', 'rolloffLip', 'openMouthBoost'."""
    nr = int(nr)
    nc = int(nc)
    if formants is not None and not (isinstance(vocalTract, (int, float))) and formants[0].shape[1] > 2:
        freqs = np.concatenate([np.asarray(f)[:, 1] for f in formants])  # :294-303
        formantDispersion = float(np.mean(np.diff(freqs)))
        vocalTract = speedSound / 2 / formantDispersion
    if formants is None and isinstance(vocalTract, (int, float)):  # :304-315 schwa
        freq = speedSound / 4 / vocalTract
        formants = [np.array([[0, freq, 30, 50 * (1 + freq ** 2 / 6 / 10 ** 6)]])]
    env = np.zeros((nr, nc))
    mouthOpen_binary = np.ones(nc)
    mouthOpening_upsampled = np.full(nc, 0.5)
    if formants is not None:
        fu = formants_upsampled if formants_upsampled is not None else \
            upsample_formants(formants, nc, smoothLinearFactor)
        fu = [np.array(f, dtype=np.float64) for f in fu]
        if temperature > 0 and formants_upsampled is None:  # :346-415
            if rng is None:
                raise ValueError('temperature > 0 needs an R random stream')
            if vocalTract is None and len(formants) > 1:
                ff = np.array([np.asarray(f)[0, 1] for f in formants])
                formantDispersion = float(np.mean(np.concatenate(([ff[0]], np.diff(ff)))))
            elif vocalTract is not None:
                formantDispersion = 2 * speedSound / (4 * vocalTract)
            else:
                formantDispersion = float('nan')
            sdG = formantDispersion * temperature * formDisp
            freq_max = np.max(fu[-1][:, 1])
            if not np.isnan(sdG) and formantDepStoch > 0:
                while freq_max < (samplingRate / 2 - 1000):
                    rw = getRandomWalk(nc, rng, rw_range=temperature * formDrift, rw_smoothing=0, trend=0)
                    if rw.size > 1:
                        rw = rw - r_mean(rw) + 1
                    new = np.zeros((nc, 4))
                    new[:, 0] = fu[0][:, 0]
                    new[:, 1] = fu[-1][:, 1] + r_round(
                        rng.rgamma(1, formantDispersion ** 2 / sdG ** 2, formantDispersion / sdG ** 2)[0] * rw)
                    new[:, 2] = r_round(rng.rgamma(
                        1, (formantDep / temperature) ** 2,
                        formantDepStoch * formantDep / (formantDepStoch * temperature) ** 2)[0] * rw)
                    new[:, 3] = 50 + (np.log2(new[:, 1]) - 5) * 20
                    fu.append(new)
                    freq_max = np.max(new[:, 1])
            for f in fu:
                for c in (1, 2, 3):
                    rw = getRandomWalk(nc, rng, rw_range=temperature * formDrift, rw_smoothing=0.3,
                                       trend=lambda: rng.rnorm(1)[0])
                    if rw.size > 1:
                        rw = rw - r_mean(rw) + 1
                    f[:, c] = f[:, c] * rw
        if terms is not None:
            terms['tracks'] = [f.copy() for f in fu]
            # tracks that a device evaluates (splines) or draws (temperature > 0) on its own, or a mouth contour
            terms['smoothed'] = (mouthAnchors is not None or temperature > 0 or
                                 (formants_upsampled is None and max(np.asarray(f).shape[0] for f in formants) > 1))
        bin_width = samplingRate / 2 / nr  # :419
        for f in fu:
            f[:, 1] = (f[:, 1] - bin_width / 2) / bin_width + 1
            f[:, 3] = f[:, 3] / bin_width
        if mouthAnchors is not None:  # :431-445
            mouthOpening_upsampled = getSmoothContour(
                mouthAnchors, length=nc, valueFloor=PERMITTED['mouthOpening'][1],
                valueCeiling=PERMITTED['mouthOpening'][2], method=contour_method)
            mouthOpening_upsampled = np.array(mouthOpening_upsampled)
            mouthOpening_upsampled[mouthOpening_upsampled < mouthOpenThres] = 0
            mouthOpen_binary = np.where(mouthOpening_upsampled > 0, 1.0, 0.0)
        if vocalTract is not None and np.isfinite(vocalTract):  # :449-459
            adjustment_hz = (mouthOpening_upsampled - 0.5) * speedSound / (4 * vocalTract)
            adjustment_bins = (adjustment_hz - bin_width / 2) / bin_width + 1
        else:
            adjustment_bins = 0.0
        for f in fu:
            f[:, 1] = f[:, 1] + adjustment_bins
            f[f[:, 1] < 1, 1] = 1
        nas = np.nonzero(mouthOpen_binary == 0)[0]  # :469-504
        if nas.size > 0:
            f1 = fu[0]
            fnp = f1.copy()
            fnp[:, 2] = 0
            fnp[nas, 2] = f1[nas, 2] * 2 / 3
            fnp[nas, 3] = f1[nas, 3] * 2 / 3
            fnp[nas, 1] = np.where(f1[nas, 1] > 550 / bin_width, f1[nas, 1] - 250 / bin_width,
                                   f1[nas, 1] + 250 / bin_width)
            fnz = f1.copy()
            fnz[:, 2] = 0
            fnz[nas, 2] = -f1[nas, 2] * 2 / 3
            fnz[nas, 1] = (fnp[nas, 1] + f1[nas, 1]) / 2
            fnz[nas, 3] = fnp[nas, 3]
            f1[nas, 2] = f1[nas, 2] * 4 / 5
            f1[nas, 3] = f1[nas, 3] * 5 / 4
            fu = fu + [fnp, fnz]
        x = np.arange(1, nr + 1, dtype=np.float64)
        lx = np.log(x)
        for f in fu:  # :507-522
            mg = f[:, 1]
            sdg = f[:, 3].copy()
            sdg[sdg == 0] = 1
            shape = mg ** 2 / sdg ** 2
            rate = mg / sdg ** 2
            for c in range(nc):
                logd = (shape[c] - 1) * lx - rate[c] * x  # dgamma up to a constant
                env[:, c] += np.exp(logd - np.max(logd)) * f[c, 2]
        env = env * formantDep
        if terms is not None:
            terms['bins'] = fu
    lip_dB = rolloffLip * np.log2(np.arange(1, nr + 1, dtype=np.float64))  # :532-537
    for c in range(nc):
        env[:, c] = (env[:, c] + lip_dB * mouthOpen_binary[c]) * \
            2 ** (mouthOpening_upsampled[c] * openMouthBoost / 10)
    if terms is not None:
        terms.setdefault('bins', [])
        terms.setdefault('smoothed', mouthAnchors is not None)
        terms.update(mouth_open=mouthOpening_upsampled, mouth_bin=mouthOpen_binary, formantDep=formantDep,
                     rolloffLip=rolloffLip, openMouthBoost=openMouthBoost)
    return 2 ** (env / 10)  # :540


# --------------------------------------------------------------------------
# seewave stft / istft (seewave.r:7782-7818, :3447-3487) and the filter block
# --------------------------------------------------------------------------
def frame_starts(length, wl, overlap):
    """soundgen.R:744-746: step = seq(1, max(1, len - wl), wl - overlap*wl/100)."""
    return r_seq_by(1, max(1, length - wl), wl - (overlap * wl / 100))


def stft_complex(wave, wl, step):
    """seewave stft(complex = TRUE, wn = 'hamming', zp = 0): frame k starts at
    the truncated index step[k]; keeps bins 0..wl/2-1; divides by wl."""
    W = hamming_w(wl)
    half = wl // 2
    z = np.zeros((half, step.size), dtype=np.complex128)
    for k, x in enumerate(step):
        s = int(x)  # R truncates fractional indices
        z[:, k] = np.fft.fft(wave[s - 1:s - 1 + wl] * W)[:half]
    return z / wl


def istft(z, wl, ovlp=75):
    """seewave istft (wn = 'hanning'): Hermitian rebuild with Nyquist :=
    Re(last bin), fft(inverse)/wl, weighted OLA at b = k*h, scale h/sum(win^2)."""
    h = wl * (100 - ovlp) / 100
    coln = z.shape[1]
    xlen = int(wl + (coln - 1) * h)  # numeric(xlen) truncates
    x = np.zeros(xlen)
    win = hanning_w(wl)
    for k in range(coln):
        b = k * h
        X = z[:, k]
        mirror = np.conj(X[1:][::-1])
        Xf = np.concatenate((X, [complex(X[-1].real, 0.0)], mirror))
        xprim = np.real(np.fft.ifft(Xf))  # fft(inverse)/length(X)
        s = int(b + 1)
        x[s - 1:s - 1 + wl] += xprim * win
    return x * h / r_sum(win ** 2)


def filter_sound(sound, spectralEnvelope, wl, overlap=75):
    """soundgen.R:743-807 given the envelope (nr x nInt, nInt in {1, nc}).
    `wl` must already be clamped (soundgen.R:743)."""
    step = frame_starts(sound.size, wl, overlap)
    z = stft_complex(sound, wl, step)
    if spectralEnvelope.shape[1] == 1:
        z = z * spectralEnvelope[:, [0]]
    else:
        z = z * spectralEnvelope
    y = istft(z, wl, overlap)
    return y / np.max(y)


# --------------------------------------------------------------------------
# generateNoise (R/source.R:57-138)
# --------------------------------------------------------------------------
def generateNoise(length, noiseAnchors=((0, 300), (-120, -120)), rolloffNoise=-6, attackLen=10,
                  windowLength_points=1024, samplingRate=16000, overlap=75, throwaway=-120,
                  filterNoise=None, rng=None, contour_method='loess', strength=None):
    """source.R:57-138.  `filterNoise`: None or (nr x k) array.  `strength`:
    optional pre-evaluated dB contour (stands in for a host-side loess)."""
    length = int(length)
    wl = int(windowLength_points)
    if strength is None:
        strength = getSmoothContour(noiseAnchors, length=length,
                                    valueFloor=PERMITTED['noiseAmpl'][1],
                                    valueCeiling=PERMITTED['noiseAmpl'][2],
                                    samplingRate=samplingRate, method=contour_method)
    if strength is None:
        return np.zeros(length)
    breathingStrength = 2 ** (np.asarray(strength, dtype=np.float64) / 10)
    step = r_seq_by(1, length + wl, wl - (overlap * wl / 100))
    nr = wl // 2
    nc = step.size
    rolloff_vec = 2 ** (rolloffNoise / 10 * np.log2(np.arange(1, nr + 1, dtype=np.float64)))
    if filterNoise is None:
        # 1 x nr matrix -> apply() -> nr x nr; column 1 = rolloff vector (source.R:96-105,113)
        filt = rolloff_vec[:, None]
        filterRowIdx = np.ones(nc, dtype=np.int64)
    else:
        filterNoise = np.asarray(filterNoise, dtype=np.float64)
        filterRowIdx = r_round(r_seq_len_out(1, filterNoise.shape[1], nc)).astype(np.int64)
        filt = filterNoise * rolloff_vec[:, None]
    u = rng.runif(nr * nc)
    z1 = u.reshape((nc, nr)).T  # column-major fill
    z1_filtered = (z1 * filt[:, filterRowIdx - 1]).astype(np.complex128)
    breathing = istft(z1_filtered, wl, overlap)
    breathing = matchLengths(breathing, length)
    breathing = breathing / np.max(breathing) * breathingStrength
    return fadeInOut(breathing, length_fade=math.floor(attackLen * samplingRate / 1000))


def savewav_pcm16(x):
    """The 16-bit samples seewave::savewav(x, f) writes (seewave.r:5192-5229 with rescale = NULL):
    level = max(x) if max(x) <= 1 else 1, then tuneR::normalize(unit = "16", centre = TRUE, level)
    (tuneR normalize.R): x - mean(x); level * x / max|x|; round(x * 32767)."""
    x = np.asarray(x, dtype=np.float64)
    mx = float(np.max(x))
    level = mx if mx <= 1 else 1.0
    xc = x - np.mean(x)
    m = float(np.max(np.abs(xc)))
    if abs(m) > 1.5e-8:                      # !isTRUE(all.equal(m, 0))
        xc = level * xc / m
    return np.rint(xc * 32767).astype(np.int64)
