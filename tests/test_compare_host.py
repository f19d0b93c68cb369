"""Spectrogram comparison and the parameter search without a device: the float64 reference on cases worked by hand,
sgb_param_range against the oracle's permittedValues, the 12-entry struct mirror, argument refusals made before any
device work, wiggle_pars, and the no-device path of sgb_rows_compare (no host fallback: SGB_ERR_CUDA)."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from compare_ref import dtw, dtw_plain, score
from oracle import soundgen_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_identical_rows():
    a = np.random.default_rng(3).standard_normal((5, 4))
    assert score(a, a, 'cor') == pytest.approx(1.0, abs=1e-15)
    assert score(a, a, 'cosine') == pytest.approx(1.0, abs=1e-15)
    assert score(a, a, 'dtw') == 0.0


def test_reference_worked_by_hand():
    # a = (0, 1, 2), b = (0, 2), one feature: d = [[0, 2], [1, 1], [2, 0]];
    # D = [[0, 2], [1, min(0 + 2, 2 + 1, 1 + 1) = 2], [3, min(1 + 0, 2 + 0, 3 + 0) = 1]]; score -1 / (3 + 2)
    a, b = np.array([[0.0], [1.0], [2.0]]), np.array([[0.0], [2.0]])
    assert dtw_plain(a, b) == dtw(a, b) == dtw(b, a) == 1.0
    assert score(a, b, 'dtw') == -0.2
    # cosine with padding: a = (1, 2) then pad 0, b = (1, 2), (3, 4): 5 / (sqrt(5) sqrt(30))
    a, b = np.array([[1.0, 2.0]]), np.array([[1.0, 2.0], [3.0, 4.0]])
    assert score(a, b, 'cosine') == pytest.approx(5 / math.sqrt(150), abs=1e-15)
    # the pad value changes cor and cosine, never DTW
    assert score(a, b, 'cosine', pad=1.0) == pytest.approx(12 / math.sqrt(7 * 30), abs=1e-15)
    assert score(a, b, 'cor', pad=1.0) == pytest.approx(np.corrcoef([1, 2, 1, 1], [1, 2, 3, 4])[0, 1], abs=1e-15)
    assert score(a, b, 'dtw', pad=5.0) == score(a, b, 'dtw') == -(0.0 + math.sqrt(8)) / 3


def test_reference_dtw_forms_agree():
    r = np.random.default_rng(7)
    for na, nb in [(1, 1), (1, 6), (6, 1), (9, 4), (13, 13), (3, 21)]:
        a, b = r.standard_normal((na, 3)), r.standard_normal((nb, 3))
        assert dtw(a, b) == pytest.approx(dtw_plain(a, b), rel=1e-14)
        assert dtw(a, b) == dtw(b, a)


def test_reference_nan_cases():
    a = np.ones((3, 2))
    for m in ('cor', 'cosine', 'dtw'):
        assert math.isnan(score(np.zeros((0, 2)), a, m)) and math.isnan(score(a, np.zeros((0, 2)), m))
    assert math.isnan(score(a, np.arange(6.0).reshape(3, 2), 'cor'))              # constant side
    assert math.isnan(score(a, a, 'cor', pad=1.0))
    assert not math.isnan(score(a[:2], np.arange(6.0).reshape(3, 2), 'cor'))     # the pad breaks the constant
    assert math.isnan(score(np.zeros((2, 2)), a, 'cosine'))                        # all-zero side
    assert math.isnan(score(np.zeros((1, 2)), np.zeros((4, 2)), 'cosine', pad=0.0))


def test_param_range_is_the_front_ends_table(built_lib):
    from soundgen_beta_b200 import api
    for name in so.CHECKED_PARS:
        out = np.zeros(3)
        assert built_lib.sgb_param_range(name.encode(), out.ctypes.data) == 0, name
        assert tuple(out) == tuple(float(v) for v in so.PERMITTED[name][:3]), name
        assert api.param_range(name) == tuple(out)
    out = np.zeros(3)
    for bad in (b'noSuchPar', b'', None):
        assert built_lib.sgb_param_range(bad, out.ctypes.data) == -1
    assert built_lib.sgb_param_range(b'rolloff', None) == -1
    with pytest.raises(ValueError):
        api.param_range('addSilence')                     # in permittedValues, but not range-checked by soundgen()


def test_compare_params_struct_mirror(built_lib):
    from soundgen_beta_b200 import _abi
    sizes = (C.c_int32 * 12)()
    assert built_lib.sgb_abi_sizes(sizes, 12) == 0
    assert sizes[11] == C.sizeof(_abi.CompareParams) == 16
    assert sizes[10] == C.sizeof(_abi.SpecParams)
    for k in (9, 10, 11):                                  # callers that know fewer structs keep working
        short = (C.c_int32 * k)()
        assert built_lib.sgb_abi_sizes(short, k) == 0 and list(short) == list(sizes)[:k]


def _compare(L, n=1, method=0, n_feat=4, pad=0.0, a_elems=400, b_elems=400, a_off=0, a_frames=10, b_off=0,
             b_frames=10, dst_elems=None, p=True):
    from soundgen_beta_b200 import _abi
    q = _abi.CompareParams()
    q.method, q.n_feat, q.pad = method, n_feat, pad
    tabs = [np.full(max(n, 1), v, dtype=np.int64) for v in (a_off, a_frames, b_off, b_frames)]
    return L.sgb_rows_compare(0, None, a_elems, None, b_elems, *(t.ctypes.data for t in tabs), n,
                              C.byref(q) if p else None, None, n if dst_elems is None else dst_elems, None)


BAD = [  # (arguments, code): refused from the arguments alone, before the device is looked at
    (dict(method=3), -1), (dict(method=-1), -1), (dict(n_feat=0), -1), (dict(pad=float('nan')), -1),
    (dict(pad=float('inf')), -1), (dict(p=False), -1), (dict(n=-1), -1), (dict(a_off=-1), -1), (dict(b_frames=-1), -1),
    (dict(a_frames=101), -1), (dict(a_off=361), -1), (dict(b_off=1, b_frames=100), -1), (dict(a_elems=-4), -1),
    (dict(dst_elems=0), -1),
    (dict(method=2, a_frames=4097, a_elems=4 * 4097), -3), (dict(method=2, b_frames=4097, b_elems=4 * 4097), -3),
]


def test_abi_refuses_bad_arguments_before_device_work(built_lib):
    for kw, code in BAD:
        assert _compare(built_lib, **kw) == code, kw
    # at the DTW limit and for cor / cosine over it the arguments are fine: what is left is the device (none here,
    # or no pointers at all)
    for kw in (dict(method=2, a_frames=4096, b_frames=4096, a_elems=4 * 4096, b_elems=4 * 4096),
               dict(method=0, a_frames=5000, a_elems=4 * 5000)):
        assert _compare(built_lib, **kw) not in (-3,), kw


def test_python_refusals_before_device_work(built_lib, monkeypatch):
    pytest.importorskip('torch')
    from soundgen_beta_b200 import api

    def no_call(*a, **k):
        raise AssertionError('device work before the argument check')
    for nm in ('soundgen_batch_device', 'spectrogram_device', 'compare_spectrograms'):
        monkeypatch.setattr(api, nm, no_call)
    x = np.zeros(16000, dtype=np.float32)
    for pars in (['samplingRate'], ['windowLength'], ['temperature'], ['repeatBout'], ['nSyl'], ['noSuchPar'],
                 ['overlap'], [], ['rolloff', 'rolloff']):
        with pytest.raises(ValueError):
            api.match_pars(x, 16000, pars)
    with pytest.raises(ValueError):
        api.match_pars(x, 16000, ['rolloff'], method='euclid')
    with pytest.raises(ValueError):
        api.match_pars(x, 16000, ['rolloff'], n_candidates=0)
    with pytest.raises(ValueError):                       # the front-end's 'adjust' would reset 48 kHz to 16 kHz
        api.match_pars(x, 48000, ['rolloff'])
    with pytest.raises(ValueError):
        api.match_pars(x, 48000, ['rolloff'], base=dict(invalidArgAction='abort'))
    with pytest.raises(ValueError):
        api.match_pars(x, 16000, ['rolloff'], base=dict(samplingRate=22050))


def test_wiggle_pars(built_lib):
    from soundgen_beta_b200 import api
    pars = ['rolloff', 'rolloffOct', 'jitterDep', 'vocalTract']
    start = dict(rolloff=-59.0, rolloffOct=9.5, jitterDep=3.0, vocalTract=15.5, sylLen=300, pitchAnchors=[100, 150])
    r = np.random.default_rng(11)
    seen = {nm: [] for nm in pars}
    for _ in range(400):
        w = api.wiggle_pars(start, pars, 0.25, 0.3, r)
        assert w['sylLen'] == 300 and w['pitchAnchors'] is start['pitchAnchors']
        assert any(w[nm] != start[nm] for nm in pars)      # at least one changes
        for nm in pars:
            _, lo, hi = api.param_range(nm)
            assert lo <= w[nm] <= hi, (nm, w[nm])
            seen[nm].append(w[nm])
    for nm in pars:                                        # each changes about a quarter of the time (or more)
        assert 60 <= sum(v != start[nm] for v in seen[nm]) <= 200, nm
    assert start['rolloff'] == -59.0                       # the input is not modified
    # the same seed gives the same draws; another seed others
    a = [api.wiggle_pars(start, pars, rng=np.random.default_rng(5)) for _ in range(3)]
    b = [api.wiggle_pars(start, pars, rng=np.random.default_rng(5)) for _ in range(3)]
    assert a == b and a[0] != api.wiggle_pars(start, pars, rng=np.random.default_rng(6))
    # prob_mutation 1: everything moves; 0: exactly one
    assert all(api.wiggle_pars(start, pars, 1.0, rng=1)[nm] != start[nm] for nm in pars)
    assert sum(api.wiggle_pars(start, pars, 0.0, rng=2)[nm] != start[nm] for nm in pars) == 1
    for bad in (['samplingRate'], ['nSyl'], ['noSuchPar'], []):
        with pytest.raises(ValueError):
            api.wiggle_pars(start, bad, rng=0)
    with pytest.raises(ValueError):
        api.wiggle_pars(start, pars, step_variance=0.0, rng=0)


NO_DEVICE_CHECK = '''
import ctypes as C
import numpy as np
from soundgen_beta_b200 import _abi
L = _abi.load()
assert L.sgb_device_count() == 0
p = _abi.CompareParams()
p.method, p.n_feat, p.pad = 0, 4, 0.0
t = np.array([0, 10], dtype=np.int64)
buf = np.zeros(40, dtype=np.float32)
dst = np.zeros(1)
for m in (0, 1, 2):
    p.method = m
    assert L.sgb_rows_compare(0, buf.ctypes.data, 40, buf.ctypes.data, 40, t.ctypes.data, t[1:].ctypes.data,
                              t.ctypes.data, t[1:].ctypes.data, 1, C.byref(p), dst.ctypes.data, 1, None) == -2
'''


def test_no_device_path(built_lib):
    code = 'import sys; sys.path.insert(0, %r)\n' % ROOT + NO_DEVICE_CHECK
    r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
