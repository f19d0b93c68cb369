"""Contours and formant tracks of any length on the host side: sgb_smooth_contour against the oracle around and far
past the old 64-knot table, R's stream after seeded calls with long contours, and descriptions of long-contour
calls for every entry point."""
import ctypes as C

import numpy as np
import pytest

import soundgen_beta_b200 as sg
from soundgen_beta_b200 import _abi, host
from oracle import soundgen_oracle as so
from oracle.rrng import RRng
from oracle.soundgen_call import soundgen as osg

NS = [11, 63, 64, 65, 200, 1000, 5000]


def contour(t, v, n, sr, lo, hi, pitch):
    t = np.ascontiguousarray(t, dtype=np.float64)
    v = np.ascontiguousarray(v, dtype=np.float64)
    out = np.zeros(n)
    rc = _abi.load().sgb_smooth_contour(t.ctypes.data, v.ctypes.data, v.size, n, float(sr), 1, float(lo), 1,
                                        float(hi), int(pitch), _abi.SGB_CONTOUR_SPLINE, out.ctypes.data)
    return rc, out


def anchors(r, n, pitch):
    t = np.sort(r.uniform(0, 1, n))
    t[0], t[-1] = 0, 1
    while np.any(np.diff(t) <= 0):          # distinct times
        t = np.sort(r.uniform(0, 1, n))
        t[0], t[-1] = 0, 1
    return t, (r.uniform(60, 800, n) if pitch else r.uniform(-100, 30, n))


@pytest.mark.parametrize('n', NS)
@pytest.mark.parametrize('pitch', [False, True])
def test_smooth_contour_any_length_vs_oracle(n, pitch):
    r = np.random.default_rng(n * 2 + pitch)
    lo, hi = (50, 3500) if pitch else (-120, 40)
    worst = 0.0
    for length in (7, 50, 350, 1050, 3500, 17500):
        t, v = anchors(r, n, pitch)
        ref = so.getSmoothContour((t, v), length=length, samplingRate=3500, valueFloor=lo, valueCeiling=hi,
                                  thisIsPitch=pitch, method='spline')
        rc, out = contour(t, v, length, 3500, lo, hi, pitch)
        assert rc == 0
        worst = max(worst, float(np.max(np.abs(out - ref) / np.maximum(1, np.abs(ref)))))
    assert worst < 1e-10, worst


def _long(r, n, lo, hi, t_hi=1.0):
    return (host.seq_len(0, t_hi, n), r.uniform(lo, hi, n))


@pytest.mark.parametrize('seed', [3, 8])
def test_front_end_stream_after_long_contours(seed):
    """Seeded calls with 100+ pitch, noise and amplitude anchors at temperature > 0: the host evaluates the pitch
    contour to count the draws, and R's stream must stand where the oracle's does after the whole call."""
    r = np.random.default_rng(seed)
    kw = dict(sylLen=400, temperature=0.1, nonlinBalance=50, jitterDep=1, shimmerDep=5, contour_method='spline',
              pitchAnchors=_long(r, 120, 90, 400), amplAnchors=_long(r, 130, 60, 120),
              noiseAnchors=_long(r, 110, -50, -10, 400))
    fe = sg.FrontEnd()
    fe.add(seed=seed, **kw)
    fe.round_begin()
    state, status = fe.rng_state(0), fe.status()[0]
    rng = RRng(seed)
    osg(rng=rng, **kw)
    assert status == 0
    assert np.array_equal(np.array(rng.state(), dtype=np.uint32).astype(np.int32), state)


def _tables(d):
    def arr(p, n, T):
        q = C.cast(p, C.POINTER(T))
        return [q[i] for i in range(n)]
    return dict(syls=arr(d.syllables, d.n_syllables, _abi.Syllable), noises=arr(d.noises, d.n_noises, _abi.Noise),
                bouts=arr(d.bouts, d.n_bouts, _abi.Bout), envs=arr(d.envelopes, d.n_envelopes, _abi.Envelope),
                frefs=arr(d.formant_index, d.n_formant_refs, _abi.FormantRef))


def long_calls(n):
    """one call per row of what used to be capped at 64 knots, each with n points"""
    r = np.random.default_rng(n)
    fm = [np.column_stack([host.seq_len(0, 1, n), r.uniform(700, 900, n), np.full(n, 30.), np.full(n, 100.)]),
          np.column_stack([host.seq_len(0, 1, n), r.uniform(1500, 1900, n), np.full(n, 25.), np.full(n, 150.)])]
    base = dict(sylLen=300, temperature=0, contour_method='spline', pitchAnchors=[150, 200])
    return {
        'pitch_device': dict(base, pitchAnchors=_long(r, n, 100, 300)),
        'pitch_host': dict(base, pitchAnchors=_long(r, n, 100, 300), temperature=0.05, seed=4),
        'ampl': dict(base, amplAnchors=_long(r, n, 40, 120)),
        'noise': dict(base, noiseAnchors=_long(r, n, -50, 0, 300), seed=5),
        'mouth': dict(base, mouthAnchors=_long(r, n, 0, 1)),
        'aglobal': dict(base, amplAnchorsGlobal=_long(r, n, 60, 120)),
        'formants': dict(base, formants=fm),
        'pitch_global': dict(base, nSyl=3, pauseLen=50, pitchAnchorsGlobal=_long(r, n, -3, 3)),
    }


@pytest.mark.parametrize('n', [64, 65, 200])
def test_front_end_describes_long_contours(n):
    for name, kw in long_calls(n).items():
        fe = sg.FrontEnd()
        fe.add(**kw)
        d, _ = fe.round_begin()
        assert fe.status()[0] == 0, name
        t = _tables(d)
        y = t['syls'][0]
        if name == 'pitch_device':
            assert y.pitch_anchor_n == n
        if name == 'pitch_host':
            assert y.pitch_anchor_n == 0 and d.n_pitch >= y.pitch_len
        if name == 'ampl':
            assert y.ampl_n == n
        if name == 'noise':
            assert t['noises'][0].anchor_n == n
        if name == 'mouth':
            assert max(e.mouth_n for e in t['envs']) == n
        if name == 'aglobal':
            assert t['bouts'][0].aglobal_n == n
        if name == 'formants':
            assert max(f.n for f in t['frefs']) == n


def test_mirrors_accept_loess_anchor_counts():
    bb = sg.BatchBuilder()
    s = bb.add_syllable(np.full(500, 150.), amplAnchors=((0, .3, .5, .7, 1), (120, 80, 100, 60, 120)))
    assert bb.syls[s].ampl_n == 5 and bb.syls[s].ampl_method == _abi.SGB_CONTOUR_LOESS
    n = bb.add_noise(3000, ((0, 50, 100, 150, 200), (-30, -10, -20, -5, -40)), np.zeros(10000), contour_method='spline')
    assert bb.noises[n].anchor_n == 5 and bb.noises[n].anchor_method == _abi.SGB_CONTOUR_SPLINE
    e = bb.add_envelope([np.array([[0, 800, 30, 100.]])], mouthAnchors=((0, .25, .5, .75, 1), (0, .8, .3, .9, .5)))
    assert bb.envs[e].mouth_n == 5 and bb.envs[e].mouth_method == _abi.SGB_CONTOUR_LOESS
