"""The f0 labels without a device: the f0 track the device is checked against (tests/f0_oracle.py), the numpy
restatement of K12b's frames, the refusals that need no GPU and the no-device path of the new entry points."""
import os
import subprocess
import sys

import numpy as np
import pytest

from f0_oracle import soundgen_f0, syllable_epoch_map, syllable_track
from f0_ref import frame_count, frame_labels
from oracle import soundgen_oracle as so
from oracle.rrng import RRng
from oracle.soundgen_call import soundgen as osg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_epoch_map_places_the_epoch_samples():
    """Outside cross-fades, joined position q holds sample k of epoch e exactly: with no envelope, fade or drift the
    output is the joined waveform over its maximum.  A vocal-fry syllable: several epochs, several crossings."""
    kw = dict(pitch=np.linspace(300, 80, 2000), samplingRate=16000, temperature=0, attackLen=0, nonlinBalance=100,
              subDep=150, subFreq=60, shortestEpoch=50)
    y, art = so.generateHarmonics(want_artefacts=True, **kw)
    assert art.epochs.shape[0] >= 3
    ep, kk = syllable_epoch_map(art, 16000)
    assert ep.size == y.size and np.all(np.diff(ep) >= 0)
    joined = y * art.raw_max
    skip = np.zeros(y.size, dtype=bool)
    skip[:2] = True
    for j in np.flatnonzero(np.diff(ep)) + 1:     # the zero after a crossing and the cross-fade that follows
        skip[max(j - 1, 0):j + 15 * 16] = True
    want = np.array([art.epoch_waves[e][k] for e, k in zip(ep, kk)])
    ok = np.abs(joined - want) <= 1e-12 * np.max(np.abs(want))
    assert np.all(ok | skip) and np.mean(~skip) > 0.8


def test_track_of_one_syllable_is_pitch_upsampled():
    """A single-epoch syllable: after the two leading samples, the track is pitch_upsampled from zc2 on."""
    y, art = so.generateHarmonics(pitch=np.linspace(150, 210, 1000), samplingRate=16000, temperature=0, attackLen=0,
                                  want_artefacts=True)
    assert art.epochs.shape[0] == 1
    pu, _ = so.upsample(art.pitch_per_gc, 16000)
    zc2 = art.zc[0][1] or 0
    f0 = syllable_track(art, 16000)
    assert f0.size == y.size
    assert np.array_equal(f0[2:], pu[zc2:]) and np.all(f0[:2] == pu[zc2])


CALLS = [dict(sylLen=300, pitchAnchors=[120, 180], temperature=0, addSilence=50),
         dict(sylLen=1000, seed=1),
         dict(sylLen=400, nSyl=2, repeatBout=2, pauseLen=120, pitchAnchors=[300, 500, 250], seed=11),
         dict(sylLen=500, noiseAnchors=((-150, 500), (-20, -30)), pitchAnchors=[200, 260], seed=13),
         dict(sylLen=500, noiseAnchors=((-80, 300), (-25, -25)), formantsNoise=[[[0, 4000, 20, 400]]],
              pitchAnchors=[150, 180], seed=14),
         dict(sylLen=700, nonlinBalance=100, subDep=150, subFreq=60, jitterDep=2, shortestEpoch=50,
              pitchAnchors=[110, 90], seed=16)]


def rng_of(kw):
    kw = dict(kw)
    return (RRng(kw.pop('seed')) if 'seed' in kw else None), kw


@pytest.mark.parametrize('i', range(len(CALLS)))
def test_soundgen_f0(i):
    rng, kw = rng_of(CALLS[i])
    y0 = osg(rng=rng, **kw)
    rng, kw = rng_of(CALLS[i])
    y, f0 = soundgen_f0(rng=rng, **kw)
    assert np.array_equal(y, y0)                            # the oracle's samples, bit for bit: its layout
    assert f0.size == y.size and f0.any()
    v = f0[f0 != 0]
    assert np.all(v >= 50) and np.all(v <= 3500)            # pitchFloor, pitchCeiling
    # voiced runs sit inside the sound: never in the leading or trailing silence
    n = int(round(16000 / 1000 * CALLS[i].get('addSilence', 100)))
    assert not f0[:n].any() and not f0[f0.size - n:].any()


def test_frame_restatement(built_lib):
    for length in (0, 1, 5, 799, 800, 801, 1600, 44100, 123457):
        for wl, overlap in ((800, 75), (1102, 75), (64, 90), (1000, 0), (4, 50)):
            assert frame_count(length, wl, overlap) == built_lib.sgb_spec_frames(length, wl, float(overlap))
    x = np.zeros(5000, dtype=np.float32)
    x[1000:3000] = np.linspace(100, 200, 2000)
    lab = frame_labels(x, 5000, 800, 75)
    assert lab.shape == (frame_count(5000, 800, 75), 2)
    k = np.arange(lab.shape[0])
    s = np.floor(1 + k * 200.0).astype(int) - 1
    want = np.array([np.count_nonzero(x[a:a + 800]) / 800 for a in s], dtype=np.float32)
    assert np.array_equal(lab[:, 1], want) and np.array_equal(lab[:, 0], x[s + 400])
    assert np.array_equal(frame_labels(x, 300, 800, 75), [[x[400] * 0, 0.0]])    # one frame, centre past len


def test_refusals_before_device_work(built_lib):
    import ctypes as C
    from soundgen_beta_b200 import _abi
    o = _abi.DeviceOut()
    off, ln = np.zeros(1, dtype=np.int64), np.full(1, 4, dtype=np.int64)
    o.dst_off, o.cap, o.dst_elems = off.ctypes.data, ln.ctypes.data, 8
    buf = np.zeros(4, dtype=np.float32)
    args = lambda wl, ov, src_elems=4: (0, buf.ctypes.data, src_elems, off.ctypes.data, ln.ctypes.data, 1, wl, ov,
                                        C.byref(o))
    for wl, ov in ((5, 75.0), (2, 75.0), (800, 100.0), (800, -1.0), (4, 90.0)):
        assert built_lib.sgb_rows_f0_frames(*args(wl, ov)) == _abi.SGB_ERR_INVALID
    assert built_lib.sgb_rows_f0_frames(*args(800, 75.0, src_elems=3)) == _abi.SGB_ERR_INVALID   # row past src
    o.format = _abi.SGB_OUT_PCM16
    assert built_lib.sgb_rows_f0_frames(*args(800, 75.0)) == _abi.SGB_ERR_INVALID
    assert built_lib.sgb_batch_f0(None, C.byref(o)) == _abi.SGB_ERR_INVALID


NO_DEVICE_CHECK = '''
import ctypes as C
import numpy as np
import pytest
import soundgen_beta_b200 as sg
from soundgen_beta_b200 import _abi
L = _abi.load()
assert L.sgb_device_count() == 0
o = _abi.DeviceOut()
off, ln = np.zeros(1, dtype=np.int64), np.full(1, 4, dtype=np.int64)
o.dst_off, o.cap, o.dst_elems, o.format = off.ctypes.data, ln.ctypes.data, 8, _abi.SGB_OUT_F32
buf = np.zeros(4, dtype=np.float32)
assert L.sgb_rows_f0_frames(0, buf.ctypes.data, 4, off.ctypes.data, ln.ctypes.data, 1, 800, 75.0,
                            C.byref(o)) == _abi.SGB_ERR_CUDA
with pytest.raises(sg.SoundgenError) as ei:
    sg.soundgen_batch_device([dict(sylLen=100, pitchAnchors=[100, 150], temperature=0)], f0=True)
assert ei.value.code == _abi.SGB_ERR_CUDA
'''


def test_no_device_path(built_lib):
    pytest.importorskip('torch')
    code = 'import sys; sys.path.insert(0, %r)\n' % ROOT + NO_DEVICE_CHECK
    r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_entry_points_are_declared(built_lib):
    from soundgen_beta_b200 import _abi
    hdr = open(os.path.join(ROOT, 'include', 'soundgen_b200.h')).read()
    for name in ('sgb_batch_f0', 'sgb_rows_f0_frames'):
        assert name in _abi.EXPORTS and ('int %s(' % name) in hdr
        assert getattr(built_lib, name) is not None
