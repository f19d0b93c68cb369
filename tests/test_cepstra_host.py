"""Cepstra without a device: dct_matrix against scipy, the float64 reference on cases worked by hand and against
torchaudio, the 13-entry struct mirror, argument refusals made before any device work, Python argument errors, and
the no-device path of sgb_rows_cepstra (no host fallback: SGB_ERR_CUDA)."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from cepstra_ref import cepstra, dct, deltas

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('n_mels', [1, 2, 13, 24, 40, 64, 128])
def test_dct_matrix_against_scipy(n_mels):
    from scipy.fft import dct as sdct
    from soundgen_beta_b200 import api
    full = sdct(np.eye(n_mels), type=2, norm='ortho', axis=0)
    D = api.dct_matrix(n_mels, n_mels)
    assert D.dtype == np.float64 and D.shape == (n_mels, n_mels)
    assert np.max(np.abs(D - full)) <= 1e-15
    assert np.max(np.abs(D @ D.T - np.eye(n_mels))) <= 1e-13                  # orthonormal
    assert np.array_equal(api.dct_matrix(min(13, n_mels), n_mels), D[:min(13, n_mels)])
    assert np.max(np.abs(D - dct(n_mels, n_mels))) <= 2e-14              # the angle not reduced: larger rounding
    if n_mels > 1:
        m = min(13, n_mels - 1)
        no_c0 = api.dct_matrix(m, n_mels, include_c0=False)
        assert np.array_equal(no_c0, D[1:m + 1])
        assert np.max(np.abs(no_c0.sum(axis=1))) <= 1e-13                      # rows k >= 1 sum to zero
        assert np.max(np.abs(no_c0 @ np.full(n_mels, -100.0))) <= 1e-11        # silence at the dB floor -> 0


def test_reference_deltas_worked_by_hand():
    # a linear ramp: the interior has the slope, the edges are replicated frames
    c = (3.0 * np.arange(6) + 1.0)[:, None]
    assert np.allclose(deltas(c, 2)[:, 0], 3.0 * np.array([0.5, 0.8, 1.0, 1.0, 0.8, 0.5]), rtol=0, atol=1e-15)
    assert np.allclose(deltas(c, 1)[:, 0], 3.0 * np.array([0.5, 1, 1, 1, 1, 0.5]), rtol=0, atol=1e-15)
    ramp = np.arange(40.0)[:, None] * np.array([[1.0, -2.0, 0.25]])
    for n in (1, 2, 4, 8):
        d = deltas(ramp, n)
        assert np.allclose(d[n:40 - n], [[1.0, -2.0, 0.25]], rtol=0, atol=1e-13), n
        assert np.all(np.abs(d[0]) < np.abs(d[n])) and np.all(np.abs(d[-1]) < np.abs(d[-1 - n]))
        assert np.allclose(deltas(d, n)[2 * n:40 - 2 * n], 0.0, atol=1e-13)   # the slope is constant
    # one frame: every delta is 0; two frames (0, 1) at n = 2: (1 (1 - 0) + 2 (1 - 0)) / 10 at both
    assert np.array_equal(deltas(np.array([[5.0, -7.0]]), 3), np.zeros((1, 2)))
    assert np.allclose(deltas(np.array([[0.0], [1.0]]), 2)[:, 0], [0.3, 0.3], rtol=0, atol=1e-16)
    # the layout of the reference: [c | d | dd]
    x = np.random.default_rng(1).standard_normal((7, 5))
    M = np.random.default_rng(2).standard_normal((3, 5))
    out = cepstra(x, M, 2, 2)
    assert out.shape == (7, 9)
    assert np.allclose(out[:, :3], x @ M.T) and np.allclose(out[:, 3:6], deltas(x @ M.T, 2))
    assert np.allclose(out[:, 6:], deltas(deltas(x @ M.T, 2), 2))
    assert cepstra(x[:0], M, 2, 2).shape == (0, 9)


@pytest.mark.parametrize('n', [1, 2, 4, 8])
@pytest.mark.parametrize('nc', [1, 2, 3, 5, 97])
def test_reference_against_torchaudio(nc, n):
    torch = pytest.importorskip('torch')
    F = pytest.importorskip('torchaudio.functional')
    c = np.random.default_rng(nc * 10 + n).standard_normal((nc, 13))
    ct = torch.tensor(c.T[None])                                     # torchaudio: [..., coefficient, time], float64
    d1 = F.compute_deltas(ct, win_length=2 * n + 1)
    d2 = F.compute_deltas(d1, win_length=2 * n + 1)
    assert np.max(np.abs(deltas(c, n) - d1[0].numpy().T)) <= 1e-13
    assert np.max(np.abs(deltas(deltas(c, n), n) - d2[0].numpy().T)) <= 1e-13


def test_dct_against_torchaudio():
    torch = pytest.importorskip('torch')
    F = pytest.importorskip('torchaudio.functional')
    from soundgen_beta_b200 import api
    for n_mfcc, n_mels in ((13, 40), (20, 64), (13, 128), (40, 40)):
        ta = F.create_dct(n_mfcc, n_mels, 'ortho').T.double().numpy()
        # torchaudio evaluates the angles, up to pi n_mfcc, in float32: each is off by up to half an ulp of its size
        assert np.max(np.abs(api.dct_matrix(n_mfcc, n_mels) - ta)) <= 2 ** -24 * math.pi * n_mfcc + 2 ** -24


def test_ceps_params_struct_mirror(built_lib):
    from soundgen_beta_b200 import _abi
    sizes = (C.c_int32 * 13)()
    assert built_lib.sgb_abi_sizes(sizes, 13) == 0
    assert sizes[12] == C.sizeof(_abi.CepsParams) == 24
    assert sizes[11] == C.sizeof(_abi.CompareParams)
    for k in (9, 10, 11, 12):                              # callers that know fewer structs keep working
        short = (C.c_int32 * k)()
        assert built_lib.sgb_abi_sizes(short, k) == 0 and list(short) == list(sizes)[:k]


def _ceps(L, n=1, n_in=8, n_ceps=3, order=2, dn=2, matrix='ok', src_elems=800, src_off=0, frames=10, p=True,
          device=0):
    from soundgen_beta_b200 import _abi
    M = np.ones((max(n_ceps, 1), max(n_in, 1)), dtype=np.float32)
    if matrix == 'nan':
        M[-1, -1] = np.nan
    elif matrix == 'inf':
        M[0, 0] = -np.inf
    q = _abi.CepsParams()
    q.n_in, q.n_ceps, q.delta_order, q.delta_n = n_in, n_ceps, order, dn
    q.matrix = None if matrix is None else M.ctypes.data
    so = np.full(max(n, 1), src_off, dtype=np.int64)
    fr = np.full(max(n, 1), frames, dtype=np.int64)
    return L.sgb_rows_cepstra(device, None, src_elems, so.ctypes.data, fr.ctypes.data, n, C.byref(q) if p else None,
                              None)


BAD = [  # refused from the arguments alone, before the device is looked at
    dict(p=False), dict(n_in=0), dict(n_ceps=0), dict(n_in=-3), dict(matrix=None), dict(matrix='nan'),
    dict(matrix='inf'), dict(order=3), dict(order=-1), dict(dn=0), dict(dn=9), dict(n=-1), dict(src_off=-1),
    dict(frames=-1), dict(src_elems=-1), dict(frames=101), dict(src_off=721), dict(src_off=801, frames=0),
    dict(frames=2 ** 31, src_elems=2 ** 40),
]


def test_abi_refuses_bad_arguments_before_device_work(built_lib):
    for kw in BAD:
        assert _ceps(built_lib, **kw) == -1, kw
    # the shared-memory limit: UNSUPPORTED, also before the device
    assert _ceps(built_lib, n_in=4096, n_ceps=64) == -3
    assert _ceps(built_lib, n_in=512, n_ceps=64, order=2, dn=4, src_elems=5120) == -3
    # the typical sizes fit: what is left is the device (none here, or no pointers at all)
    for kw in (dict(n_in=256, n_ceps=64, order=2, dn=4, src_elems=2560), dict(n_in=256, n_ceps=64, order=2, dn=8,
                                                                                src_elems=2560),
               dict(n_in=40, n_ceps=13, order=0, dn=8),
               dict(frames=100), dict(src_off=800, frames=0)):
        assert _ceps(built_lib, **kw) not in (-3,), kw


def test_python_argument_errors(built_lib, monkeypatch):
    torch = pytest.importorskip('torch')
    from soundgen_beta_b200 import api
    for args in ((0, 40), (13, 0), (41, 40), (40, 40, False), (-1, 40)):
        with pytest.raises(ValueError):
            api.dct_matrix(*args)
    src = torch.zeros(8)
    dst = torch.zeros(8)
    for kw in (dict(src=np.zeros(8, np.float32)), dict(src=torch.zeros(8, dtype=torch.float64)),
               dict(src_off=[0, 0]), dict(matrix=np.zeros((0, 4))), dict(matrix=np.zeros(4))):
        a = dict(device=0, src=src, src_off=[0], frames=[1], dst=dst, dst_off=[0], cap=[1], matrix=np.ones((2, 4)))
        a.update(kw)
        with pytest.raises(ValueError):
            api.rows_cepstra(**a)

    def no_call(*a, **k):
        raise AssertionError('device work before the argument check')
    mfcc = api.mfcc_device
    for nm in ('soundgen_batch_device', 'spectrogram_device', '_spectrogram_device', 'compare_spectrograms',
               'mfcc_device', 'rows_cepstra'):
        monkeypatch.setattr(api, nm, no_call)
    for kw in (dict(deltas=3), dict(deltas=-1), dict(delta_n=0), dict(delta_n=9), dict(n_mfcc=41), dict(n_mfcc=0),
               dict(n_mfcc=40, include_c0=False), dict(max_frames=-1), dict(n_mels=None)):
        with pytest.raises(ValueError):
            mfcc(torch.zeros((1, 16)), [16], 16000, **kw)
    x = np.zeros(16000, dtype=np.float32)
    for kw in (dict(features='lpc'), dict(features='mfcc', n_mfcc=64), dict(features='mfcc', deltas=3),
               dict(features='mfcc', n_mfcc=0)):
        with pytest.raises(ValueError):
            api.match_pars(x, 16000, ['rolloff'], **kw)


NO_DEVICE_CHECK = '''
import ctypes as C
import numpy as np
from soundgen_beta_b200 import _abi
L = _abi.load()
assert L.sgb_device_count() == 0
M = np.ones((3, 8), dtype=np.float32)
p = _abi.CepsParams()
p.n_in, p.n_ceps, p.matrix, p.delta_order, p.delta_n = 8, 3, M.ctypes.data, 2, 2
so, fr, cap = np.array([0], dtype=np.int64), np.array([10], dtype=np.int64), np.array([10], dtype=np.int64)
src, dst = np.zeros(80, dtype=np.float32), np.zeros(90, dtype=np.float32)
o = _abi.DeviceOut()
o.dst, o.dst_elems, o.dst_off, o.cap, o.format = dst.ctypes.data, 90, so.ctypes.data, cap.ctypes.data, 0
for order in (0, 1, 2):
    p.delta_order = order
    assert L.sgb_rows_cepstra(0, src.ctypes.data, 80, so.ctypes.data, fr.ctypes.data, 1, C.byref(p), C.byref(o)) == -2
'''


def test_no_device_path(built_lib):
    code = 'import sys; sys.path.insert(0, %r)\n' % ROOT + NO_DEVICE_CHECK
    r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
