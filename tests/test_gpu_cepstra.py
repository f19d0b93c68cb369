"""Cepstra on the device (k_cepstra through sgb_rows_cepstra, rows_cepstra and mfcc_device) against the float64
reference on K9's own log-mel output, their layout in caller memory, bit identity across runs, row orders, batch sizes
and crops, stream order, the refusals, and match_pars on MFCC features."""
import ctypes as C
import math

import numpy as np
import pytest

import soundgen_beta_b200 as sg
from cepstra_ref import cepstra as ref_cepstra, dct as ref_dct
from spectrogram_ref import spectrogram as ref_spectrogram
from soundgen_beta_b200 import _abi
from test_gpu_compare import BASE, target
from test_gpu_device_out import mixed_calls
from test_gpu_spectrogram import batch_rates

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

SR, WL_MS = 16000, 50                    # wl 800, hop 200 at 75 % overlap
FRAMES = [0, 1, 2, 3, 5, 97, 400]
LENS = [0] + [801 + (f - 1) * 200 for f in FRAMES[1:]]     # rows of exactly FRAMES frames
U = 2.0 ** -23
_cache = {}


def logmel(n_in):
    """K9 log-mel rows of n_in bands, packed [rows, F, n_in] with every value past a row's frames set to NaN."""
    if n_in not in _cache:
        r = np.random.default_rng(n_in)
        w = np.zeros((len(LENS), max(LENS)), dtype=np.float32)
        for c, L in enumerate(LENS):
            t = np.arange(L)
            x = 0.01 * r.standard_normal(L)
            for h in range(1, 8):
                x += np.sin(2 * np.pi * h * r.uniform(0.004, 0.02) * t * (1 + 0.2 * t / max(L, 1))) / h
            w[c, :L] = x * (1 + np.sin(2 * np.pi * t / 3000))
        spec, fr = sg.spectrogram_device(torch.tensor(w, device='cuda'), LENS, SR, windowLength=WL_MS, n_mels=n_in,
                                         db=True)
        assert fr.cpu().tolist() == FRAMES
        for c, f in enumerate(FRAMES):
            spec[c, f:] = float('nan')
        _cache[n_in] = spec
    return _cache[n_in]


def run(src, frames, M, order, dn, cap=None, stride_pad=0, stream=None):
    """rows_cepstra over the rows of src [n, F, n_in] into a NaN-filled destination; returns (out [n, S], written)."""
    n, F, n_in = src.shape
    n_out = M.shape[0] * (1 + order)
    cap = np.full(n, F) if cap is None else np.asarray(cap)
    S = int(cap.max(initial=0)) * n_out + stride_pad
    dst = torch.full((n * S,), float('nan'), dtype=torch.float32, device='cuda')
    w = sg.rows_cepstra(src.device.index, src, np.arange(n) * F * n_in, frames, dst, np.arange(n) * S, cap, M, order,
                        dn, stream)
    return dst.view(n, S), w


def bound(x, M, order, dn):
    """Per-value error bound of K11 against the float64 reference: the FP32 dot product n_in 2^-23 sum_b |M_kb x_b|,
    carried through the delta weights, plus (dn + 2) 2^-23 of the delta's own terms for its sums and division."""
    x, M = np.asarray(x, dtype=np.float64), np.asarray(M, dtype=np.float64)
    c = x @ M.T
    err = [M.shape[1] * U * (np.abs(x) @ np.abs(M).T)]
    mag = [np.abs(c)]
    nc, t = c.shape[0], np.arange(c.shape[0])
    den = 2 * sum(j * j for j in range(1, dn + 1))
    for _ in range(order):
        e, a = err[-1], mag[-1]
        ne, na = np.zeros_like(e), np.zeros_like(a)
        for j in range(1, dn + 1):
            hi, lo = np.minimum(t + j, nc - 1), np.maximum(t - j, 0)
            ne += j * (e[hi] + e[lo])
            na += j * (a[hi] + a[lo])
        err.append(ne / den + (dn + 2) * U * na / den)
        mag.append(na / den)
    return np.concatenate(err, axis=1)


@pytest.mark.parametrize('n_in', [24, 40, 64, 128])
def test_reference_parity_layout_and_crop(n_in):
    src = logmel(n_in)
    F = src.shape[1]
    X = src.double().cpu().numpy()
    worst = 0.0
    for n_ceps in (13, 20):
        for c0 in (True, False):
            M = sg.dct_matrix(n_ceps, n_in, c0).astype(np.float32)
            for order in (0, 1, 2):
                for dn in (1, 2, 4):
                    n_out = n_ceps * (1 + order)
                    out, w = run(src, FRAMES, M, order, dn, stride_pad=37)      # odd stride: no row is aligned
                    crop, wc = run(src, FRAMES, M, order, dn, cap=np.full(len(FRAMES), 5), stride_pad=3)
                    torch.cuda.synchronize()
                    out, crop = out.cpu().numpy(), crop.cpu().numpy()
                    assert list(w) == FRAMES and list(wc) == list(np.minimum(FRAMES, 5))
                    for c, nc in enumerate(FRAMES):
                        row = out[c, :F * n_out].reshape(F, n_out)
                        assert not np.isnan(row).any(), (c, n_ceps, c0, order, dn)   # NaN input past nc is not read
                        assert np.all(row[nc:] == 0) and np.all(np.isnan(out[c, F * n_out:]))
                        assert np.array_equal(crop[c, :5 * n_out].view(np.int32), out[c, :5 * n_out].view(np.int32))
                        assert np.all(np.isnan(crop[c, 5 * n_out:]))
                        if nc == 0:
                            continue
                        want = ref_cepstra(X[c, :nc], M, order, dn)
                        b = bound(X[c, :nc], M, order, dn)
                        ratio = np.abs(row[:nc] - want) / b
                        assert np.all(ratio <= 1.0), (c, n_ceps, c0, order, dn, ratio.max())
                        worst = max(worst, float(ratio.max()))
    print('n_in %d: worst |K11 - reference| / bound = %.3g' % (n_in, worst))


def test_bit_identity_runs_permutation_and_batch_size():
    src = logmel(64)
    n, F, n_in = src.shape
    M = sg.dct_matrix(13, n_in).astype(np.float32)
    r = np.random.default_rng(9)
    idx = r.integers(0, n, 2048)
    big = src[torch.as_tensor(idx, device='cuda')].contiguous()
    fr = np.asarray(FRAMES)[idx]
    a, _ = run(big, fr, M, 2, 2)
    b, _ = run(big, fr, M, 2, 2)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))                        # across runs
    perm = r.permutation(2048)
    p, _ = run(big[torch.as_tensor(perm, device='cuda')].contiguous(), fr[perm], M, 2, 2)
    assert torch.equal(p.view(torch.int32), a[torch.as_tensor(perm, device='cuda')].view(torch.int32))
    for c in range(n):                                                                  # one row against 2048
        one, _ = run(src[c:c + 1].contiguous(), FRAMES[c:c + 1], M, 2, 2)
        j = int(np.flatnonzero(idx == c)[-1])
        assert torch.equal(one[0].view(torch.int32), a[j].view(torch.int32)), c


def test_stream_order_without_host_sync():
    src = logmel(40)
    n, F, n_in = src.shape
    M = sg.dct_matrix(13, n_in).astype(np.float32)
    ref, _ = run(src, FRAMES, M, 2, 2)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        x = torch.zeros_like(src)
        torch.cuda._sleep(50_000_000)                  # keep the stream busy: the copy and K11 wait behind it
        x.copy_(src)
        got, _ = run(x, FRAMES, M, 2, 2, stream=s)
        sums = torch.nan_to_num(got.double(), nan=0.0).sum(dim=1)     # queued at once, no synchronise in between
    s.synchronize()
    assert torch.equal(got.view(torch.int32), ref.view(torch.int32))
    assert torch.equal(sums, torch.nan_to_num(ref.double(), nan=0.0).sum(dim=1))


def _raw(src, src_elems, dst, dst_elems, n_in=8, n_ceps=3, frames=4, cap=4, dst_off=0, device=None):
    M = np.ones((n_ceps, n_in), dtype=np.float32)
    p = _abi.CepsParams()
    p.n_in, p.n_ceps, p.matrix, p.delta_order, p.delta_n = n_in, n_ceps, M.ctypes.data, 2, 2
    so, fr = np.zeros(1, dtype=np.int64), np.full(1, frames, dtype=np.int64)
    off, cp, wr = np.full(1, dst_off, dtype=np.int64), np.full(1, cap, dtype=np.int64), np.zeros(1, dtype=np.int64)
    o = _abi.DeviceOut()
    o.dst, o.dst_elems, o.dst_off, o.cap, o.out_written, o.format = dst, dst_elems, off.ctypes.data, cp.ctypes.data, \
        wr.ctypes.data, _abi.SGB_OUT_F32
    dev = torch.cuda.current_device() if device is None else device
    return _abi.load().sgb_rows_cepstra(dev, src, src_elems, so.ctypes.data, fr.ctypes.data, 1, C.byref(p), C.byref(o))


def test_refusals():
    src = torch.randn(32, device='cuda')
    dst = torch.full((36,), float('nan'), device='cuda')
    host = np.zeros(36, dtype=np.float32)
    pinned = torch.zeros(36).pin_memory()
    big = torch.zeros(600 * 64, device='cuda')
    INV, UNS = _abi.SGB_ERR_INVALID, _abi.SGB_ERR_UNSUPPORTED
    assert _raw(src.data_ptr(), 32, host.ctypes.data, 36) == INV                          # host dst
    assert _raw(src.data_ptr(), 32, pinned.data_ptr(), 36) == INV                         # pinned dst
    assert _raw(pinned.data_ptr(), 32, dst.data_ptr(), 36) == INV                         # pinned src
    both = torch.zeros(100, device='cuda')
    assert _raw(both.data_ptr(), 32, both.data_ptr() + 4 * 20, 36) == INV                 # dst overlaps src
    assert _raw(both.data_ptr() + 4 * 60, 32, both.data_ptr(), 61) == INV                 # its end overlaps src
    assert _raw(src.data_ptr(), 31, dst.data_ptr(), 36) == INV                            # the row ends past src
    assert _raw(src.data_ptr(), 32, dst.data_ptr(), 35) == INV                            # the row ends past dst
    assert _raw(src.data_ptr(), 32, dst.data_ptr(), 36, dst_off=-1) == INV
    assert _raw(src.data_ptr(), 32, dst.data_ptr(), 36, device=torch.cuda.device_count()) == INV
    assert _raw(big.data_ptr(), big.numel(), dst.data_ptr(), 36, n_in=600, n_ceps=64) == UNS   # shared memory
    torch.cuda.synchronize()
    assert torch.isnan(dst).all()                                                          # nothing was queued
    assert _raw(both.data_ptr() + 4 * 60, 32, both.data_ptr(), 60) == 0                    # adjacent is fine
    assert _raw(src.data_ptr(), 32, dst.data_ptr(), 36) == 0
    torch.cuda.synchronize()
    x = src.double().cpu().numpy().reshape(4, 8)
    want = ref_cepstra(x, np.ones((3, 8)), 2, 2)
    assert np.allclose(dst.cpu().numpy().reshape(4, 9), want, rtol=1e-5, atol=1e-5)
    with pytest.raises(sg.SoundgenError) as ei:
        sg.rows_cepstra(0, src, [0], [4], dst, [0], [4], np.ones((3, 8)), deltas=3)
    assert ei.value.code == INV


def test_mfcc_device_end_to_end():
    calls = mixed_calls()
    wave, lengths, st = sg.soundgen_batch_device(calls)
    rates = batch_rates(calls)
    assert len(set(rates)) > 1 and np.any(st != 0)
    n_mels, n_mfcc, order, dn = 40, 13, 2, 2
    feat, frames = sg.mfcc_device(wave, lengths, rates, n_mfcc=n_mfcc, deltas=order, delta_n=dn, n_mels=n_mels)
    assert feat.dtype == torch.float32 and feat.is_cuda and frames.is_cuda and feat.shape[2] == n_mfcc * 3
    w, ln, fr, ft = wave.cpu().numpy(), lengths.cpu().numpy(), frames.cpu().numpy(), feat.cpu().numpy()
    D = ref_dct(n_mfcc, n_mels)
    tol, H, checked = 0.01 * math.sqrt(n_mels), order * dn, 0
    for i in range(len(calls)):
        if ln[i] == 0:
            assert fr[i] == 0 and np.all(ft[i] == 0)
            continue
        wl = int(np.floor(50 / 1000 * rates[i] / 2) * 2)
        P = ref_spectrogram(w[i, :ln[i]].astype(np.float64), wl, 75, 'hamming', sg.mel_filterbank(rates[i], wl, n_mels))
        nc = P.shape[0]
        assert fr[i] == nc and np.all(ft[i, nc:] == 0)
        want = ref_cepstra(10 * np.log10(np.maximum(P, 1e-10)), D, order, dn)
        loud = np.all(P >= 1e-6 * P.max(), axis=1)
        t = np.arange(nc)
        keep = np.ones(nc, dtype=bool)
        for j in range(-H, H + 1):
            keep &= loud[np.clip(t + j, 0, nc - 1)]
        if keep.any():
            assert np.max(np.abs(ft[i, :nc][keep] - want[keep])) <= tol, i
            checked += int(keep.sum())
    assert checked > 100
    # a crop is a bit-exact prefix: the last deltas before max_frames read the log-mel frames past it
    Fc = int(fr.max()) // 2
    cut, fc = sg.mfcc_device(wave, lengths, rates, n_mfcc=n_mfcc, deltas=order, delta_n=dn, n_mels=n_mels,
                             max_frames=Fc)
    assert cut.shape[1] == Fc and np.array_equal(fc.cpu().numpy(), np.minimum(fr, Fc))
    assert torch.equal(cut.view(torch.int32), feat[:, :Fc].contiguous().view(torch.int32))
    # on a stream that is not the current one
    s = torch.cuda.Stream()
    got, _ = sg.mfcc_device(wave, lengths, rates, n_mfcc=n_mfcc, deltas=order, delta_n=dn, n_mels=n_mels, stream=s)
    s.synchronize()
    assert torch.equal(got.view(torch.int32), feat.view(torch.int32))


@pytest.mark.parametrize('method', ['cor', 'dtw'])
def test_match_pars_on_mfcc(method):
    x = target()
    kw = dict(base=dict(BASE, rolloff=-25), n_candidates=16, max_iter=6, seed=3, method=method, features='mfcc',
              deltas=1)
    best_kw, best, hist = sg.match_pars(x, SR, ['rolloff', 'rolloffOct'], **kw)
    cur = [h['best'] for h in hist]
    assert len(hist) == 7 and all(c1 >= c0 for c0, c1 in zip(cur, cur[1:])) and best == cur[-1]
    assert math.isfinite(cur[0])
    print('match_pars mfcc %s: initial %.6f final %.6f' % (method, cur[0], best))
    _, best2, hist2 = sg.match_pars(x, SR, ['rolloff', 'rolloffOct'], **kw)
    assert best2 == best
    for h, h2 in zip(hist, hist2):
        assert h['score'] == h2['score'] and h['accepted'] == h2['accepted'] and h['best'] == h2['best']
        assert np.array_equal(h['values'], h2['values'])
