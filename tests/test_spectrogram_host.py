"""Spectrograms without a device: the frame count of the library against the oracle's frame rule, the oracle against
torch.stft, mel_filterbank against torchaudio's bank, argument refusals that need no GPU, the 11-entry struct
mirror, and the no-device path of the two entries (no host fallback: SGB_ERR_CUDA)."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import soundgen_oracle as so
from spectrogram_ref import spectrogram as ref_spectrogram

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('wl,overlap', [(800, 75), (1102, 75), (2400, 50), (160, 70), (592, 75), (2204, 90), (4, 0)])
def test_frame_count_equals_the_oracle(built_lib, wl, overlap):       # 1102 at 75 %: hop 275.5
    for L in sorted({0, 1, 5, wl // 2, wl - 1, wl, wl + 1, wl + 2, 3 * wl + 7, 44100, 57000, 57001}):
        want = 0 if L == 0 else so.frame_starts(L, wl, overlap).size
        assert built_lib.sgb_spec_frames(L, wl, overlap) == want, (L, wl, overlap)


def test_frame_count_refuses_bad_geometry(built_lib):
    assert built_lib.sgb_spec_frames(1000, 801, 75) == -1      # odd
    assert built_lib.sgb_spec_frames(1000, 2, 0) == -1         # < 4
    assert built_lib.sgb_spec_frames(1000, 800, 100) == -1     # no hop
    assert built_lib.sgb_spec_frames(1000, 800, 99.9) == -1    # hop 0.8 < 1
    assert built_lib.sgb_spec_frames(-1, 800, 75) == -1


@pytest.mark.parametrize('window', ['hamming', 'hanning'])
@pytest.mark.parametrize('wl,overlap', [(800, 75), (2400, 50), (160, 70), (592, 75)])
def test_oracle_equals_torch_stft_on_the_shared_frames(wl, overlap, window):
    torch = pytest.importorskip('torch')
    hop = wl - overlap * wl / 100
    assert hop == int(hop)
    x = np.random.default_rng(wl).standard_normal(20 * wl + 3 * int(hop))
    F = ref_spectrogram(x, wl, overlap, window)
    w = {'hamming': so.hamming_w, 'hanning': so.hanning_w}[window](wl)
    S = torch.stft(torch.tensor(x), wl, int(hop), wl, window=torch.tensor(w), center=False,
                   return_complex=True).numpy()
    P = np.abs(S[:wl // 2].T / wl) ** 2
    assert P.shape[0] >= F.shape[0] >= P.shape[0] - 1        # torch.stft may have one frame more
    assert np.max(np.abs(F - P[:F.shape[0]])) <= 1e-12 * np.max(F)
    # the one-frame difference: len - wl a multiple of the hop
    x = x[:wl + 4 * int(hop)]
    S = torch.stft(torch.tensor(x), wl, int(hop), wl, window=torch.tensor(w), center=False, return_complex=True)
    assert ref_spectrogram(x, wl, overlap, window).shape[0] == S.shape[1] - 1


def test_oracle_short_rows_are_zero_padded():
    x = np.random.default_rng(1).standard_normal(300)
    F = ref_spectrogram(x, 800, 75)
    assert F.shape == (1, 400)
    want = np.abs(np.fft.fft(np.concatenate((x, np.zeros(500))) * so.hamming_w(800))[:400] / 800) ** 2
    assert np.allclose(F[0], want, rtol=1e-12, atol=0)
    assert ref_spectrogram(np.zeros(0), 800, 75).shape == (0, 400)


def _torchaudio_bank(n_freqs, f_min, f_max, n_mels, sample_rate, norm, mel_scale):
    """torchaudio.functional.melscale_fbanks; restated (in float32 torch, as torchaudio computes it) where
    torchaudio is not installed."""
    try:
        import torchaudio
        return torchaudio.functional.melscale_fbanks(n_freqs, f_min, f_max, n_mels, sample_rate, norm, mel_scale)
    except ImportError:
        pass
    import torch

    def hz_to_mel(f):
        if mel_scale == 'htk':
            return 2595.0 * math.log10(1.0 + f / 700.0)
        f_sp = 200.0 / 3
        m = f / f_sp
        if f >= 1000.0:
            m = 1000.0 / f_sp + math.log(f / 1000.0) / (math.log(6.4) / 27.0)
        return m

    def mel_to_hz(m):
        if mel_scale == 'htk':
            return 700.0 * (10.0 ** (m / 2595.0) - 1.0)
        f_sp = 200.0 / 3
        f = f_sp * m
        t = m >= 1000.0 / f_sp
        f[t] = 1000.0 * torch.exp(math.log(6.4) / 27.0 * (m[t] - 1000.0 / f_sp))
        return f
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    f_pts = mel_to_hz(torch.linspace(hz_to_mel(f_min), hz_to_mel(f_max), n_mels + 2))
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    down = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up = slopes[:, 2:] / f_diff[1:]
    fb = torch.max(torch.zeros(1), torch.min(down, up))
    if norm == 'slaney':
        fb *= (2.0 / (f_pts[2:n_mels + 2] - f_pts[:n_mels])).unsqueeze(0)
    return fb


@pytest.mark.parametrize('norm', [None, 'slaney'])
@pytest.mark.parametrize('mel_scale', ['htk', 'slaney'])
@pytest.mark.parametrize('sr,wl', [(16000, 800), (22050, 1102), (44100, 2204), (48000, 2400)])
def test_mel_filterbank_equals_torchaudio(sr, wl, mel_scale, norm):
    pytest.importorskip('torch')
    from soundgen_beta_b200 import api
    for n_mels, fmin, fmax in ((128, 0.0, None), (40, 60.0, 7600.0)):
        got = api.mel_filterbank(sr, wl, n_mels, fmin, fmax, mel_scale, norm)
        ref = _torchaudio_bank(wl // 2 + 1, fmin, float(sr // 2) if fmax is None else fmax, n_mels, sr, norm,
                               mel_scale)[:wl // 2].T.double().numpy()
        assert got.shape == ref.shape == (n_mels, wl // 2)
        # torchaudio's bank is float32: its slopes (f_pts - f) / f_diff carry float32 rounding of frequencies in Hz
        assert np.max(np.abs(got - ref)) <= 1e-4 * ref.max(), np.max(np.abs(got - ref))
        api.bands_csr(got, wl // 2)                       # every band has contiguous support


def test_bands_csr_and_non_contiguous_bands():
    from soundgen_beta_b200 import api
    B = np.zeros((3, 8))
    B[0, 2:5] = [1, 2, 3]
    B[2, 7] = 0.5
    lo, ln, w = api.bands_csr(B, 8)
    assert list(lo) == [2, 0, 7] and list(ln) == [3, 0, 1] and list(w) == [1, 2, 3, 0.5]
    B[1, [1, 3]] = 1.0
    with pytest.raises(ValueError):
        api.bands_csr(B, 8)
    with pytest.raises(ValueError):
        api.bands_csr(np.ones((2, 7)), 8)
    with pytest.raises(ValueError):
        api.bands_csr(np.ones((0, 8)), 8)


def test_python_refusals_before_device_work(built_lib, monkeypatch):
    torch = pytest.importorskip('torch')
    from soundgen_beta_b200 import api

    def no_call(*a, **k):
        raise AssertionError('library called before the argument check')
    monkeypatch.setattr(built_lib, 'sgb_rows_spectrogram', no_call)
    src = torch.zeros(1600)
    dst = torch.zeros(4000)
    B = np.zeros((2, 400))
    B[0, [3, 9]] = 1
    for kw in (dict(bands=B), dict(window='blackman'), dict(bands=np.ones((2, 300)))):
        with pytest.raises(ValueError):
            api.rows_spectrogram(0, src, [0], [1600], dst, [0], [4], 800, **kw)
    with pytest.raises(ValueError):                      # float64 source
        api.rows_spectrogram(0, src.double(), [0], [1600], dst, [0], [4], 800)
    with pytest.raises(ValueError):
        api.mel_filterbank(16000, 800, 40, mel_scale='bark')
    with pytest.raises(ValueError):
        api.mel_filterbank(16000, 800, 40, norm='area')


def _params(**kw):
    from soundgen_beta_b200 import _abi
    p = _abi.SpecParams()
    p.wl, p.window, p.overlap, p.db, p.db_floor = 800, 0, 75.0, 0, 1e-10
    keep = []
    if 'bands' in kw:
        lo, ln, w = (np.ascontiguousarray(a) for a in kw.pop('bands'))
        keep += [lo, ln, w]
        p.n_bands, p.band_lo, p.band_len, p.band_w = lo.size, lo.ctypes.data, ln.ctypes.data, w.ctypes.data
    for k, v in kw.items():
        setattr(p, k, v)
    return p, keep


BAD_PARAMS = [  # (fields, code): refused from the parameters alone, before the device is looked at
    (dict(wl=801), -3), (dict(wl=2), -3), (dict(wl=20000), -3),
    (dict(overlap=100.0), -1), (dict(overlap=-1.0), -1), (dict(overlap=99.9), -1), (dict(overlap=float('nan')), -1),
    (dict(window=2), -1), (dict(db=1, db_floor=0.0), -1), (dict(db=1, db_floor=-1.0), -1), (dict(db=2), -1),
    (dict(bands=(np.int32([398]), np.int32([3]), np.float32([1, 1, 1]))), -1),        # past wl / 2
    (dict(bands=(np.int32([-1]), np.int32([2]), np.float32([1, 1]))), -1),
    (dict(bands=(np.int32([0]), np.int32([2]), np.float32([1, np.inf]))), -1),
    (dict(bands=(np.int32([0]), np.int32([2]), np.float32([np.nan, 1]))), -1),
    (dict(n_bands=-1), -1),
]


def test_abi_refuses_bad_parameters(built_lib):
    from soundgen_beta_b200 import _abi
    o = _abi.DeviceOut()
    for fields, code in BAD_PARAMS:
        p, keep = _params(**dict(fields))
        assert built_lib.sgb_rows_spectrogram(0, None, None, None, 0, C.byref(p), C.byref(o)) == code, fields
        assert built_lib.sgb_batch_spectrogram(None, C.byref(p), C.byref(o)) == code, fields
    assert built_lib.sgb_rows_spectrogram(0, None, None, None, 0, None, C.byref(o)) == -1


def test_spec_params_struct_mirror(built_lib):
    from soundgen_beta_b200 import _abi
    sizes = (C.c_int32 * 11)()
    assert built_lib.sgb_abi_sizes(sizes, 11) == 0
    assert sizes[10] == C.sizeof(_abi.SpecParams) == 56
    assert sizes[9] == C.sizeof(_abi.DeviceOut)
    ten = (C.c_int32 * 10)()                       # callers that know ten structs keep working
    assert built_lib.sgb_abi_sizes(ten, 10) == 0 and list(ten) == list(sizes)[:10]


NO_DEVICE_CHECK = '''
import ctypes as C
import numpy as np
from soundgen_beta_b200 import _abi
L = _abi.load()
assert L.sgb_device_count() == 0
p = _abi.SpecParams()
p.wl, p.window, p.overlap = 800, 0, 75.0
o = _abi.DeviceOut()
o.dst_elems = 4000
off, ln, cap = np.zeros(1, dtype=np.int64), np.full(1, 1600, dtype=np.int64), np.full(1, 10, dtype=np.int64)
o.dst_off, o.cap = off.ctypes.data, cap.ctypes.data
buf = np.zeros(1600, dtype=np.float32)
assert L.sgb_rows_spectrogram(0, buf.ctypes.data, off.ctypes.data, ln.ctypes.data, 1, C.byref(p), C.byref(o)) == -2
assert L.sgb_batch_spectrogram(None, C.byref(p), C.byref(o)) == -2
'''


def test_no_device_path(built_lib):
    code = 'import sys; sys.path.insert(0, %r)\n' % ROOT + NO_DEVICE_CHECK
    r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
