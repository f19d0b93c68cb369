"""Contours and formant tracks of any length on a B200: every entry point that used to stop at 64 knots, against the
oracle (waveforms within 1e-4 of peak, integer artefacts bit-exact), in batches mixed with other calls, and the
Python single-call mirrors with loess anchor counts."""
import numpy as np
import pytest

import soundgen_beta_b200 as sg
from soundgen_beta_b200 import _abi, host, workloads
from oracle import soundgen_oracle as so
from oracle.rrng import RRng
from oracle.soundgen_call import soundgen as osg

from test_long_contours_host import long_calls

pytestmark = pytest.mark.gpu
TOL = 1e-4


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(b)))


def oracle_call(kw):
    kw = dict(kw)
    z, u = kw.pop('z', None), kw.pop('u', None)
    if 'seed' in kw:
        return osg(rng=RRng(kw.pop('seed')), **kw)
    return osg(rng=so.RStream(z=np.concatenate(z) if z else None, u=np.concatenate(u) if u else None), **kw)


@pytest.mark.parametrize('n', [64, 65, 200])
def test_every_entry_point_with_long_contours(n):
    calls = long_calls(n)
    for name, kw in calls.items():
        y = sg.soundgen(**kw)
        ref = oracle_call(kw)
        assert y.size == ref.size and rel(y, ref) < TOL, name
    # the same calls in one batch: each gives what it gives alone
    outs, st = sg.soundgen_batch(list(calls.values()), out_dtype=np.float64)
    assert np.all(st == 0)
    for (name, kw), y in zip(calls.items(), outs):
        assert rel(y, oracle_call(kw)) < TOL, name


def test_pitch_contour_of_5000_points_artefacts_bit_exact():
    r = np.random.default_rng(5000)
    t = host.seq_len(0, 1, 5000)
    v = np.exp(np.log(120) + 0.6 * np.sin(np.linspace(0, 40, 5000)) + 0.05 * r.standard_normal(5000))
    pitch = so.getSmoothContour((t, v), length=3500, samplingRate=3500, valueFloor=75, valueCeiling=3500,
                                thisIsPitch=True, method='spline')
    amp = (host.seq_len(0, 1, 300), r.uniform(40, 120, 300))
    z = r.standard_normal(40000)
    pars = dict(samplingRate=22050, nonlinBalance=100, jitterDep=1.0, jitterLen=5, shimmerDep=10, subFreq=90,
                subDep=40, temperature=0.2)
    ref, art = so.generateHarmonics(pitch, rng=so.RStream(z=z), amplAnchors=amp, want_artefacts=True,
                                    contour_method='spline', **pars)
    y, a = sg.generateHarmonics(pitch, z=z, amplAnchors=amp, want_artefacts=True, contour_method='spline', **pars)
    assert np.array_equal(a['gc'], art.gc) and np.array_equal(a['gc_upsampled'], art.gc_upsampled)
    assert np.array_equal(a['epochs'], art.epochs) and a['z_used'] == art.z_used
    assert [tuple(int(v or 0) for v in zz) for zz in art.zc] == [tuple(q) for q in a['zc'].tolist()]
    assert y.size == ref.size and rel(y, ref) < TOL
    # the device evaluates the 5000-anchor contour itself (soundgen() with pitchAnchors)
    kw = dict(sylLen=1000, temperature=0, pitchAnchors=(t, v), contour_method='spline', samplingRate=22050,
              invalidArgAction='ignore')
    yb, bt = sg.soundgen(return_batch=True, **kw)
    ref, arts, _ = osg(rng=RRng(1), want_artefacts=True, **kw)
    ab = bt.artefacts(0)
    assert np.array_equal(ab['gc'], arts[0].gc) and np.array_equal(ab['epochs'], arts[0].epochs)
    assert yb.size == ref.size and rel(yb, ref) < TOL


@pytest.mark.parametrize('npoints', [62, 63, 200])
@pytest.mark.parametrize('slf', [1, 3])
def test_formant_tracks_any_length(npoints, slf):
    r = np.random.default_rng(npoints + slf)
    t = host.seq_len(0, 1, npoints)
    fm = [np.column_stack([t, r.uniform(lo, lo * 1.3, npoints), r.uniform(20, 40, npoints), r.uniform(60, 200, npoints)])
          for lo in (500, 1400, 2600)]
    mouth = (host.seq_len(0, 1, 80), r.uniform(0, 1, 80))
    for nc in (5, 77, 400):
        a = sg.getSpectralEnvelope(256, nc, formants=fm, smoothLinearFactor=slf, mouthAnchors=mouth,
                                   contour_method='spline')
        b = so.getSpectralEnvelope(256, nc, formants=fm, smoothLinearFactor=slf, mouthAnchors=mouth)
        assert rel(a, b) < 1e-10, nc


def _mixed_calls():
    calls = list(workloads.resynthesis(n=6, seed=11)) + workloads.config3(n=4) + workloads.config4(n=6, seed=40)
    for n in (65, 200):
        calls += list(long_calls(n).values())
    return calls


def test_mixed_batch_gives_each_call_its_own_result_and_is_reproducible():
    L = _abi.load()
    calls = _mixed_calls()
    outs, st = sg.soundgen_batch(calls, out_dtype=np.float64)
    assert np.all(st == 0)
    for i, kw in enumerate(calls):
        alone = sg.soundgen_batch([kw], out_dtype=np.float64)[0][0]
        assert np.array_equal(alone, outs[i]), i
        if i < 6 or i >= 16:       # the long-contour calls against the oracle (cfg3 / cfg4 have their own tests)
            assert rel(outs[i], oracle_call(kw)) < TOL, i
    sums = []
    for _ in range(2):
        bb = sg.BatchBuilder(u_dtype=np.float32)
        for kw in calls:
            bb.add_soundgen(**kw)
        bt = sg.Batch()
        bt.upload(bb.build())
        bt.run()
        cs = np.zeros(9, dtype=np.uint64)
        assert L.sgb_batch_checksums(bt.h, cs.ctypes.data, 9) == 0
        sums.append(cs)
        bt.close()
    assert np.array_equal(sums[0], sums[1])


@pytest.mark.parametrize('nanch', [3, 5, 10])
def test_single_call_mirrors_fit_loess(nanch):
    r = np.random.default_rng(nanch)
    t = np.sort(r.uniform(0, 1, nanch)); t[0], t[-1] = 0, 1
    pitch = np.exp(np.linspace(np.log(140), np.log(220), 1200))
    amp = (t, r.uniform(40, 120, nanch))
    y = sg.generateHarmonics(pitch, amplAnchors=amp, samplingRate=16000)
    ref = so.generateHarmonics(pitch, rng=so.RStream(), amplAnchors=amp, samplingRate=16000)
    assert y.size == ref.size and rel(y, ref) < TOL
    L, wl = 6000, 1024
    u = np.random.default_rng(1).random(workloads.noise_uniform_count(L, wl))
    na = (np.sort(r.uniform(0, 370, nanch)), r.uniform(-40, 0, nanch))
    na[0][0] = 0
    y = sg.generateNoise(L, noiseAnchors=na, u=u)
    ref = so.generateNoise(L, noiseAnchors=na, rng=so.RStream(u=u))
    assert y.size == ref.size and rel(y, ref) < TOL
    mouth = (t, r.uniform(0, 1, nanch))
    fm = [np.array([[0, 700, 30, 100.], [1, 900, 25, 120.]]), np.array([[0, 1500, 25, 150.]])]
    a = sg.getSpectralEnvelope(256, 40, formants=fm, mouthAnchors=mouth)
    b = so.getSpectralEnvelope(256, 40, formants=fm, mouthAnchors=mouth)
    assert rel(a, b) < 1e-10
