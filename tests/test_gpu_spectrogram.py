"""Spectrograms on the device (k_spectrogram through sgb_rows_spectrogram / sgb_batch_spectrogram, Batch.spectrogram,
rows_spectrogram, spectrogram_device) against the float64 oracle, their layout in caller memory, bit identity across
entries, segmentations and runs, stream order, and the refusals."""
import ctypes as C

import numpy as np
import pytest

import soundgen_beta_b200 as sg
from spectrogram_ref import spectrogram as ref_spectrogram
from soundgen_beta_b200 import _abi, api, workloads
from test_gpu_device_out import built, built_desc, mixed_calls

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu


def signal_rows(wl, seed):
    """Rows of several lengths (empty, shorter than the window, one window, many frames): harmonics + noise."""
    r = np.random.default_rng(seed)
    lens = [0, wl // 3, wl, wl + 1, 9 * wl + 13, 57000]
    rows = []
    for L in lens:
        t = np.arange(L)
        x = 0.3 * r.standard_normal(L) * 0.05
        for h in range(1, 12):
            x += np.sin(2 * np.pi * (h * 0.011 + r.uniform(0, 0.002)) * t + r.uniform(0, 6)) / h
        rows.append(x.astype(np.float32))
    return rows


def run_rows(rows, wl, overlap, window='hamming', bands=None, db=False, db_floor=1e-10, F=None, stride_pad=0):
    """rows_spectrogram over `rows` packed into one tensor; returns (spec [n, F, n_feat] as numpy, written)."""
    n = len(rows)
    lens = np.array([r.size for r in rows], dtype=np.int64)
    src_off = np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.int64)
    src = torch.tensor(np.concatenate(rows + [np.zeros(1, np.float32)]), device='cuda')
    nc = [sg_frames(L, wl, overlap) for L in lens]
    F = max(nc) if F is None else F
    nf = wl // 2 if bands is None else bands.shape[0]
    S = F * nf + stride_pad
    dst = torch.full((n * S,), float('nan'), dtype=torch.float32, device='cuda')
    w = api.rows_spectrogram(torch.cuda.current_device(), src, src_off, lens, dst, np.arange(n) * S, np.full(n, F),
                             wl, overlap, window, bands, db, db_floor)
    torch.cuda.synchronize()
    return dst.view(n, S).cpu().numpy(), w, F, nf


def sg_frames(L, wl, overlap):
    return int(_abi.load().sgb_spec_frames(int(L), int(wl), float(overlap)))


@pytest.mark.parametrize('window', ['hamming', 'hanning'])
@pytest.mark.parametrize('overlap', [50, 70, 75])
@pytest.mark.parametrize('wl', [160, 800, 1102, 1200, 2204, 2400, 592])
def test_oracle_parity(wl, overlap, window):
    rows = signal_rows(wl, wl + overlap)
    sr = wl * 20                                           # 50 ms windows
    bank = api.mel_filterbank(sr, wl, 64 if wl > 200 else 24)
    for mode in ('power', 'mel', 'db'):
        bands = bank if mode == 'mel' else None
        out, written, F, nf = run_rows(rows, wl, overlap, window, bands, db=(mode == 'db'), stride_pad=3)
        for i, x in enumerate(rows):
            ref = ref_spectrogram(x.astype(np.float64), wl, overlap, window, bank if mode == 'mel' else None)
            nc = ref.shape[0]
            assert written[i] == nc == sg_frames(x.size, wl, overlap), (i, written[i], nc)
            got = out[i, :F * nf].reshape(F, nf)
            assert np.all(got[nc:] == 0) and not np.isnan(got).any()
            assert np.all(np.isnan(out[i, F * nf:]))      # the gap between rows is not written
            if nc == 0:
                continue
            g = got[:nc]
            if mode == 'db':
                keep = ref >= 1e-6 * ref.max()
                want = 10 * np.log10(np.maximum(ref, 1e-10))
                assert np.max(np.abs(g[keep] - want[keep])) <= 0.01, (i, mode)
                assert np.all(g >= -100.0 - 1e-4)
            else:
                assert np.max(np.abs(g - ref)) <= 1e-5 * ref.max(), (i, mode, np.max(np.abs(g - ref)) / ref.max())


def batch_rates(calls):
    """Each call's sampling rate as its bout in the front-end's description has it (the front-end may reset it)."""
    fe = api.FrontEnd()
    for kw in calls:
        fe.add(**kw)
    desc, m = fe.round_begin()
    cl = C.cast(desc.calls, C.POINTER(_abi.Call))
    bouts = C.cast(desc.bouts, C.POINTER(_abi.Bout))
    ids = fe.round_calls()
    rates = np.full(len(calls), 16000.0)
    for i in range(m):
        rates[ids[i]] = bouts[cl[i].bout_begin].samplingRate
    fe.close()
    return rates


def test_mixed_batch_through_spectrogram_device():
    calls = mixed_calls()
    wave, lengths, st = sg.soundgen_batch_device(calls)
    rates = batch_rates(calls)
    assert len(set(rates)) > 1
    with pytest.raises(ValueError):                         # a linear spectrogram needs one window length
        sg.spectrogram_device(wave, lengths, rates)
    for kw in (dict(n_mels=40), dict(n_mels=40, mel_scale='slaney', norm='slaney', db=True, window='hanning')):
        spec, frames = sg.spectrogram_device(wave, lengths, rates, **kw)
        assert spec.dtype == torch.float32 and spec.is_cuda and frames.dtype == torch.int64 and frames.is_cuda
        w, ln, fr, sp = wave.cpu().numpy(), lengths.cpu().numpy(), frames.cpu().numpy(), spec.cpu().numpy()
        assert sp.shape[0] == len(calls) and sp.shape[2] == 40
        failed = np.flatnonzero(st != 0)
        assert failed.size
        # an empty row (here: the failed call's row cut to 0 samples) has no frames and is all zeros; the other rows
        # keep their bits
        ln0 = lengths.clone()
        ln0[torch.as_tensor(failed, device=ln0.device)] = 0
        sp0, fr0 = sg.spectrogram_device(wave, ln0, rates, max_frames=sp.shape[1], **kw)
        sp0, fr0 = sp0.cpu().numpy(), fr0.cpu().numpy()
        ok = np.setdiff1d(np.arange(len(calls)), failed)
        assert np.all(fr0[failed] == 0) and np.all(sp0[failed] == 0)
        assert np.array_equal(fr0[ok], fr[ok]) and np.array_equal(sp0[ok].view(np.int32), sp[ok].view(np.int32))
        for i in range(len(calls)):
            wl = int(np.floor(50 / 1000 * rates[i] / 2) * 2)
            assert fr[i] == sg_frames(ln[i], wl, 75), (i, ln[i], fr[i])
            if ln[i] == 0:
                assert np.all(sp[i] == 0)
                continue
            bank = sg.mel_filterbank(rates[i], wl, 40, mel_scale=kw.get('mel_scale', 'htk'), norm=kw.get('norm'))
            ref = ref_spectrogram(w[i, :ln[i]].astype(np.float64), wl, 75, kw.get('window', 'hamming'), bank)
            assert fr[i] == ref.shape[0] and np.all(sp[i, fr[i]:] == 0)
            g = sp[i, :fr[i]]
            if kw.get('db'):
                keep = ref >= 1e-6 * ref.max()
                want = 10 * np.log10(np.maximum(ref, 1e-10))                # the default db_floor
                assert np.max(np.abs(g[keep] - want[keep])) <= 0.01, i
            else:
                assert np.max(np.abs(g - ref)) <= 1e-5 * ref.max(), i


def test_nan_destination_odd_stride_and_crop():
    calls = workloads.config1(n=2) + workloads.config0()
    bt = built(calls)
    host = bt.fetch(np.float32)
    n, wl = len(calls), 800
    nc = np.array([sg_frames(h.size, wl, 75) for h in host])
    F, nf = int(nc.max()) + 3, wl // 2
    S = F * nf + 37                                        # odd row stride: no row is aligned
    dst = torch.full((n * S,), float('nan'), dtype=torch.float32, device='cuda')
    written = bt.spectrogram(dst, np.arange(n) * S, np.full(n, F), wl)
    crop = torch.full((n * S,), float('nan'), dtype=torch.float32, device='cuda')
    written_c = bt.spectrogram(crop, np.arange(n) * S, np.full(n, 5), wl)
    torch.cuda.synchronize()
    assert np.array_equal(written, nc) and np.array_equal(written_c, np.minimum(nc, 5))
    a, c = dst.view(n, S).cpu().numpy(), crop.view(n, S).cpu().numpy()
    for i in range(n):
        row = a[i, :F * nf].reshape(F, nf)
        assert not np.isnan(row).any() and np.all(row[nc[i]:] == 0) and np.all(np.isnan(a[i, F * nf:]))
        assert np.array_equal(c[i, :5 * nf].view(np.int32), a[i, :5 * nf].view(np.int32))   # bit for bit
        assert np.all(np.isnan(c[i, 5 * nf:]))
    bt.close()


def test_bit_identity_across_entries_segmentations_and_runs():
    calls = workloads.config3(n=2) + workloads.config1(n=2)
    bt = built(calls)
    host = bt.fetch(np.float32)
    n, wl, ov = len(calls), 2400, 75
    lens = np.array([h.size for h in host], dtype=np.int64)
    F, nf = max(sg_frames(L, wl, ov) for L in lens), 128
    bank = sg.mel_filterbank(48000, wl, nf)
    outs = []
    for _ in range(2):                                     # two runs of the batch entry
        d = torch.empty((n, F, nf), dtype=torch.float32, device='cuda')
        bt.spectrogram(d, np.arange(n) * F * nf, np.full(n, F), wl, ov, bands=bank)
        outs.append(d)
    # the rows entry over the same samples, each row alone and among 640 rows
    src = torch.tensor(np.concatenate(host), device='cuda')
    offs = np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.int64)
    d = torch.empty((n, F, nf), dtype=torch.float32, device='cuda')
    sg.rows_spectrogram(src.device.index, src, offs, lens, d,
                        np.arange(n) * F * nf, np.full(n, F), wl, ov, bands=bank)
    outs.append(d)
    big = 640
    pick = np.arange(big) % n
    d = torch.empty((big, F, nf), dtype=torch.float32, device='cuda')
    sg.rows_spectrogram(src.device.index, src, offs[pick], lens[pick], d, np.arange(big) * F * nf, np.full(big, F), wl,
                        ov, bands=bank)
    for i in range(n):
        alone = torch.empty((1, F, nf), dtype=torch.float32, device='cuda')
        sg.rows_spectrogram(src.device.index, src, offs[i:i + 1], lens[i:i + 1], alone, [0], [F], wl, ov, bands=bank)
        torch.cuda.synchronize()
        assert torch.equal(alone[0].view(torch.int32), outs[0][i].view(torch.int32)), i
        for j in np.flatnonzero(pick == i)[[0, -1]]:
            assert torch.equal(d[j].view(torch.int32), alone[0].view(torch.int32)), (i, j)
    for o in outs[1:]:
        assert torch.equal(o.view(torch.int32), outs[0].view(torch.int32))
    bt.close()


def test_stream_order_without_host_sync():
    calls = workloads.config3(n=64)
    bt = built(calls)
    n, wl, F = len(calls), 2400, 100
    ref = torch.empty((n, F, wl // 2), dtype=torch.float32, device='cuda')
    bt.spectrogram(ref, np.arange(n) * F * (wl // 2), np.full(n, F), wl)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dst = torch.empty((n, F, wl // 2), dtype=torch.float32, device='cuda')
        torch.cuda._sleep(50_000_000)                      # keep the stream busy: the spectrogram must wait behind it
        bt.spectrogram(dst, np.arange(n) * F * (wl // 2), np.full(n, F), wl, stream=s)
        sums = dst.double().sum(dim=(1, 2))                # queued at once, no synchronise in between
    # the same handle takes another batch at once: its run must not overwrite the rows before they are read
    bt.upload(built_desc(workloads.config1(n=4)))
    bt.run()
    s.synchronize()
    assert torch.equal(dst.view(torch.int32), ref.view(torch.int32))
    assert torch.allclose(sums, ref.double().sum(dim=(1, 2)), rtol=1e-12, atol=0)
    bt.close()


def test_refusals():
    calls = workloads.config1(n=2)
    bt = sg.Batch()
    bt.upload(built_desc(calls))
    n, wl, F = len(calls), 800, 200
    dst = torch.empty((n, F, wl // 2), dtype=torch.float32, device='cuda')
    ok_off, ok_cap = np.arange(n) * F * (wl // 2), np.full(n, F)
    with pytest.raises(sg.SoundgenError) as ei:            # uploaded, never run
        bt.spectrogram(dst, ok_off, ok_cap, wl)
    assert ei.value.code == _abi.SGB_ERR_STATE
    bt.run()
    pinned = torch.empty((n, F, wl // 2), dtype=torch.float32).pin_memory()
    bad = [(dict(dst=pinned), _abi.SGB_ERR_INVALID), (dict(dst=torch.empty_like(pinned)), _abi.SGB_ERR_INVALID),
           (dict(off=np.zeros(n, dtype=np.int64)), _abi.SGB_ERR_INVALID),          # rows overlap
           (dict(off=ok_off + 1), _abi.SGB_ERR_INVALID),                             # the last row ends past dst
           (dict(cap=ok_cap + 1), _abi.SGB_ERR_INVALID),
           (dict(off=ok_off - 1), _abi.SGB_ERR_INVALID),
           (dict(overlap=100), _abi.SGB_ERR_INVALID), (dict(overlap=99.95), _abi.SGB_ERR_INVALID),
           (dict(db=True, db_floor=0.0), _abi.SGB_ERR_INVALID),
           (dict(bands=np.full((2, wl // 2), np.nan)), _abi.SGB_ERR_INVALID),
           (dict(wl=801), _abi.SGB_ERR_UNSUPPORTED), (dict(wl=12000), _abi.SGB_ERR_UNSUPPORTED)]
    for kw, code in bad:
        kw = dict(kw)
        d, off, cap = kw.pop('dst', dst), kw.pop('off', ok_off), kw.pop('cap', ok_cap)
        w = kw.pop('wl', wl)
        with pytest.raises(sg.SoundgenError) as ei:
            bt.spectrogram(d, off, cap, w, **kw)
        assert ei.value.code == code, kw
    # PCM16 is not a spectrogram format; a host or foreign source is refused by the rows entry
    L = _abi.load()
    p, _ = api._spec_params(wl, 75, 'hamming', None, False, 1e-10)
    o = _abi.DeviceOut()
    offs, caps = np.ascontiguousarray(ok_off, dtype=np.int64), np.ascontiguousarray(ok_cap, dtype=np.int64)
    o.dst, o.dst_elems, o.dst_off, o.cap, o.format = dst.data_ptr(), dst.numel(), offs.ctypes.data, caps.ctypes.data, 1
    assert L.sgb_batch_spectrogram(bt.h, C.byref(p), C.byref(o)) == _abi.SGB_ERR_INVALID
    host = bt.fetch(np.float32)
    lens = np.array([h.size for h in host], dtype=np.int64)
    so_ = np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.int64)
    cpu_src = torch.tensor(np.concatenate(host))
    with pytest.raises(sg.SoundgenError) as ei:
        sg.rows_spectrogram(0, cpu_src, so_, lens, dst, ok_off, ok_cap, wl)
    assert ei.value.code == _abi.SGB_ERR_INVALID
    # the refusals queued nothing and left the handle usable
    bt.spectrogram(dst, ok_off, ok_cap, wl)
    torch.cuda.synchronize()
    for i, h in enumerate(host):
        ref = ref_spectrogram(h.astype(np.float64), wl, 75)
        g = dst[i, :ref.shape[0]].cpu().numpy()
        assert np.max(np.abs(g - ref)) <= 1e-5 * ref.max()
    bt.close()
    fresh = sg.Batch()                                     # never uploaded
    with pytest.raises(sg.SoundgenError) as ei:
        fresh.spectrogram(dst[:0], np.zeros(0), np.zeros(0), wl)
    assert ei.value.code == _abi.SGB_ERR_STATE
    fresh.close()
