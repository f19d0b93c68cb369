"""K4 (kernels_env.cu) on its own: the FP32 envelope table every filter reads (read back with sgb_batch_envelope)
against the float64 oracle within the per-element bound of envelope_bound.py, on the edges of the kernel (formant
count and its 32-lane loop, widths, frequencies, mouth, track kinds, sizes), inside a batch of more than a thousand
instances, and through soundgen() calls; the stand-alone FP64 path within the same bound with FP64 roundings."""
import ctypes as C

import numpy as np
import pytest

import soundgen_beta_b200 as sg
from envelope_bound import CASES, bound, capture, reference
from oracle.rrng import RRng
from oracle.soundgen_call import soundgen as osg
from soundgen_beta_b200 import _abi

pytestmark = pytest.mark.gpu
NOISE_AN = (np.array([0., 300.]), np.array([-10., -10.]))
SR = {80: 16000, 301: 16000, 400: 16000, 551: 22050, 600: 24000, 1102: 44100, 1200: 48000}
ENV_ARGS = ('formants', 'formantDep', 'rolloffLip', 'mouthAnchors', 'mouthOpenThres', 'openMouthBoost', 'vocalTract',
            'samplingRate', 'smoothLinearFactor')


def env_batch(specs, seed=0):
    """One batch whose noises are filtered by the envelopes `specs` = [(nr, nc, getSpectralEnvelope arguments)]
    (noise i: window 2 nr, envelope nr x nc), under one bout filtered by lip radiation only (nr 80).  Returns the
    batch handle and the device envelopes, noise by noise."""
    r = np.random.default_rng(seed)
    bb = sg.BatchBuilder()
    bb.add_silent_syllable(8)
    main = bb.add_envelope(None)
    for nr, nc, kw in specs:
        ek = {k: v for k, v in kw.items() if k in ENV_ARGS}
        env = bb.add_envelope(ek.pop('formants', None), nc_fixed=nc, tracks=kw.get('formants_upsampled'), **ek)
        wl = 2 * nr
        n = 3 * wl
        bb.add_noise(n, NOISE_AN, r.random(bb.noise_uniform_count(n, wl)), windowLength_points=wl,
                     samplingRate=kw.get('samplingRate', 16000), env_id=env)
    bb.add_bout(0, 1, 0, len(specs), main, False, 160)
    bb.add_call(0, 1)
    bt = sg.Batch()
    bt.upload(bb.build())
    bt.run()
    assert np.all(bt.status() == 0)
    return bt, [bt.envelope(1, i) for i in range(len(specs))]


def check(got, ref, terms, what):
    assert got is not None and got.shape == ref.shape, (what, None if got is None else got.shape, ref.shape)
    b = bound(terms, ref.shape[0])
    err = np.abs(got.astype(np.float64) - ref) / ref
    assert np.all(err <= b), (what, float(np.max(err / b)))
    return float(np.max(err / b))


def test_batch_path_within_bound():
    bt, got = env_batch([(nr, nc, kw) for _, nr, nc, kw in CASES])
    worst = 0.0
    for (name, nr, nc, kw), g in zip(CASES, got):
        ref, terms = reference(nr, nc, **kw)
        worst = max(worst, check(g, ref, terms, name))
        assert float(np.max(bound(terms, nr))) <= 3e-5, name
    main = bt.envelope(0, 0)                        # the bout's filter: no formants, lip radiation only (F = 0)
    ref, terms = reference(80, 1)
    check(main, ref, terms, 'bout')
    bt.close()
    print('worst FP32 error / bound: %.3f' % worst)


def test_standalone_fp64_within_bound():
    worst = 0.0
    for name, nr, nc, kw in CASES:
        ref, terms = reference(nr, nc, **kw)
        got = sg.getSpectralEnvelope(nr, nc, **kw)
        b = bound(terms, nr, fp32=False)
        err = np.abs(got - ref) / ref
        assert np.all(err <= b), (name, float(np.max(err / b)))
        worst = max(worst, float(np.max(err / b)))
    print('worst FP64 error / bound: %.3f' % worst)


def test_literal_filter_matrix_is_cast_exactly():
    r = np.random.default_rng(5)
    bb = sg.BatchBuilder()
    bb.add_silent_syllable(8)
    main = bb.add_envelope(None)
    mats = [r.uniform(0.01, 50, (400, 1)), r.uniform(0.01, 50, (400, 37)), r.uniform(1e-3, 1e3, (551, 5))]
    for i, m in enumerate(mats):
        wl = 2 * m.shape[0]
        e = bb.add_envelope_matrix(m)
        bb.add_noise(4000, NOISE_AN, r.random(bb.noise_uniform_count(4000, wl)), windowLength_points=wl, env_id=e)
    bb.add_noise(4000, NOISE_AN, r.random(bb.noise_uniform_count(4000, 800)), windowLength_points=800)   # unfiltered
    bb.add_bout(0, 1, 0, len(mats) + 1, main, False, 160)
    bb.add_call(0, 1)
    bt = sg.Batch()
    bt.upload(bb.build())
    bt.run()
    for i, m in enumerate(mats):
        got = bt.envelope(1, i)
        assert np.array_equal(got.view(np.uint32), m.astype(np.float32).view(np.uint32)), i
    assert bt.envelope(1, len(mats)) is None
    bt.close()


def _instance(i):
    nr = (80, 301, 400, 551)[i % 4]
    fm = [np.array([[0, 500. + i, 30, 100]]), np.array([[0, 1500. + 0.5 * i, 20, 150]])]
    if i % 7 == 3:      # a few filters of 40 formants: the launch's table stride is set by them
        fm += [np.array([[0, 1700. + 150 * k + 0.1 * i, 10, 120]]) for k in range(38)]
    kw = dict(formants=fm, vocalTract=16., samplingRate=SR[nr])
    if i % 5 == 0:
        kw['mouthAnchors'] = (np.array([0., 1]), np.array([0.1 + i / 5000, 0.9]))
        kw['mouthOpenThres'] = 0.3
    return nr, 1 + i % 3, kw


def test_thousand_instances():
    """1100 envelopes of mixed nr, nc and formant count (2 or 40) in one launch (the instance of a work item is found
    by bisection over col0, the shared-memory tables are strided by the largest count): each within the bound of its
    own reference, and a sample (the first, the last, instances spread over the list, both formant counts) bit for
    bit what it is in a batch of its own."""
    specs = [_instance(i) for i in range(1100)]
    sample = sorted(set(range(0, 15)) | set(range(0, 1100, 97)) | set(range(1085, 1100)) | {3, 10, 507, 1095})
    alone = {}
    for i in sample:
        bt, got = env_batch([specs[i]])
        bt.close()
        alone[i] = got[0]
    bt, big = env_batch(specs)
    bt.close()
    for i, (nr, nc, kw) in enumerate(specs):
        ref, terms = reference(nr, nc, **kw)
        check(big[i], ref, terms, i)
    for i in sample:
        assert np.array_equal(alone[i].view(np.uint32), big[i].view(np.uint32)), i


def run_calls(calls):
    """Every call through the front-end's rounds on one batch handle.  Returns (waveforms, device envelopes per call
    in the oracle's order: per bout its filtered noises, then its main filter), statuses, the front-end."""
    fe = sg.FrontEnd()
    for kw in calls:
        fe.add(**kw)
    bt = sg.Batch()
    parts, envs = [[] for _ in calls], [[] for _ in calls]
    while True:
        desc, n = fe.round_begin()
        if n == 0:
            break
        cl = C.cast(desc.calls, C.POINTER(_abi.Call))
        bo = C.cast(desc.bouts, C.POINTER(_abi.Bout))
        ranges = [[(b, bo[b].noise_begin, bo[b].noise_end) for b in range(cl[k].bout_begin, cl[k].bout_end)]
                  for k in range(n)]
        bt.upload(desc)
        bt.run()
        segs = bt.fetch(np.float64)
        for k, ci in enumerate(fe.round_calls()):
            parts[ci].append(segs[k].copy())
            for b, q0, q1 in ranges[k]:
                for e in [bt.envelope(1, q) for q in range(q0, q1)] + [bt.envelope(0, b)]:
                    if e is not None:
                        envs[ci].append(e)
    bt.close()
    return [np.concatenate(p) for p in parts], envs, fe.status(), fe


def check_calls(calls, rng_state=False, parity=False):
    """Every envelope of every call within the bound of the one the oracle's soundgen() built at that point;
    (rng_state) R's stream after each call where the oracle's stands; (parity) the waveform within 1e-4 of peak of
    the oracle's.  Without `parity` the waveforms are only held to the oracle's length."""
    outs, envs, st, fe = run_calls(calls)
    assert np.all(st == 0), st
    for ci, kw in enumerate(calls):
        okw = dict(kw)
        rng = RRng(okw.pop('seed'))
        with capture() as rec:
            ref = osg(rng=rng, **okw)
        assert outs[ci].shape == ref.shape, ci
        if parity:
            err = float(np.max(np.abs(outs[ci] - ref)) / np.max(np.abs(ref)))
            assert err <= 1e-4, (ci, err)
        assert len(envs[ci]) == len(rec), (ci, len(envs[ci]), len(rec))
        for j, (g, r) in enumerate(zip(envs[ci], rec)):
            check(g, r['env'], r['terms'], (ci, j))
        if rng_state:
            assert np.array_equal(np.array(rng.state(), dtype=np.uint32).astype(np.int32), fe.rng_state(ci)), ci
    fe.close()


FM2 = [np.array([[0, 860, 30, 120.], [1, 500, 35, 100]]), np.array([[0, 1280, 40, 120.], [1, 2000, 20, 150]])]
SOUNDGEN = [
    dict(sylLen=250, formants=FM2, temperature=0, seed=11),                                # moving tracks
    dict(sylLen=250, temperature=0.2, seed=12),                                            # stochastic, static
    dict(sylLen=250, temperature=0.2, mouthAnchors=[0.3, 0.9], seed=13),                   # stochastic, set_tracks
    dict(sylLen=200, nSyl=2, pauseLen=80, noiseAnchors=((0., 250.), (-20., -10.)), formantsNoise=FM2,
         temperature=0.1, seed=14),                                                        # noise envelopes
    dict(sylLen=200, repeatBout=2, pauseLen=100, temperature=0, mouthAnchors=[0, 0.7, 0], seed=15),  # closed mouth
    dict(sylLen=300, samplingRate=44100, temperature=0, seed=16),                          # nr 1102
    dict(sylLen=300, samplingRate=48000, invalidArgAction='ignore', temperature=0, seed=17),  # nr 1200
    dict(sylLen=300, windowLength=10, temperature=0, seed=18),                             # nr 80
    dict(sylLen=300, samplingRate=24000, temperature=0, seed=19),                          # nr 600
    dict(sylLen=200, repeatBout=2, pauseLen=60, temperature=0.1, mouthAnchors=[.2, .8], seed=20),  # rounds
]


def test_soundgen_envelopes_within_bound():
    check_calls(SOUNDGEN)


def test_stochastic_formants_past_62():
    """vocalTract = 100 cm: R draws pseudo-formants 177 Hz apart up to Nyquist - 1000 Hz, 106 at 44.1 kHz and 72 at
    32 kHz (43 at 22.05 kHz; at 16 kHz only 26, under the old cap of 62, so that rate does not test it).  R's stream
    after the call and the device envelope with all of them match."""
    calls = [dict(sylLen=300, vocalTract=100, temperature=0.1, samplingRate=sr, seed=s)
             for sr in (44100, 32000, 22050) for s in (1, 2, 3, 4)]
    check_calls(calls, rng_state=True)


def test_stochastic_formants_past_62_sound_like_r():
    """The same calls with formantDepStoch = 10 (the same 106 and 72 formants; pseudo-formants of 10 dB instead of
    30): waveform within 1e-4 of peak of the oracle's, as well as stream and envelope.  With the default 30 dB the
    pseudo-formants pile up to gains of up to 1.5e8 (82 dB) in the top band, where the source lies ~80 dB below its
    peak: rounding the oracle's own unfiltered sound to float32 and filtering it in float64 already moves the result
    by up to 1.5e-3 of peak, so no FP32 sound reaches 1e-4 there."""
    calls = [dict(sylLen=300, vocalTract=100, temperature=0.1, formantDepStoch=10, samplingRate=sr, seed=s)
             for sr in (44100, 32000) for s in (1, 2, 3, 4)]
    check_calls(calls, rng_state=True, parity=True)
