"""The f0 labels on the GPU: K12a (Batch.f0, soundgen_batch_device(..., f0=True)) against the f0 track of tests/f0_oracle.py, K12b
(rows_f0_frames, f0_frames_device) against a numpy restatement, the track against an autocorrelation estimate of
the waveform, and the export contract (determinism, stream order, failed calls, refusals)."""
import ctypes as C

import numpy as np
import pytest

import soundgen_beta_b200 as sg
from f0_oracle import soundgen_f0
from f0_ref import frame_labels, within_ulp
from oracle import soundgen_oracle as so
from oracle.rrng import RRng
from soundgen_beta_b200 import _abi, presets, workloads

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

PS = {(s, n): kw for s, n, kw in presets.load()}


def oracle_f0(kw):
    kw = dict(kw)
    z, u = kw.pop('z', None), kw.pop('u', None)
    if 'seed' in kw:
        rng = RRng(kw.pop('seed'))
    else:
        rng = so.RStream(z=np.concatenate(z) if z else None, u=np.concatenate(u) if u else None)
    return soundgen_f0(rng=rng, **kw)


def corpus():
    calls = workloads.config0() + workloads.config1(n=3) + workloads.config2(n=3) + workloads.config3(n=3)
    calls += [dict(kw, seed=i) for i, (_, _, kw) in enumerate(presets.load())]        # set.seed(i), own temperature
    calls += [
        dict(sylLen=400, nSyl=2, repeatBout=3, pauseLen=120, pitchAnchors=[300, 500, 250], seed=11),   # multi-bout
        dict(PS[('Cat', 'Scream')], seed=904),                  # 2 bouts, the second in a second round
        dict(sylLen=300, noiseAnchors=((0, 300), (40, 40)), seed=12),                                  # noise only
        dict(sylLen=500, noiseAnchors=((-150, 500), (-20, -30)), pitchAnchors=[200, 260], seed=13),    # breathing first
        dict(sylLen=500, noiseAnchors=((-80, 300), (-25, -25)), formantsNoise=[[[0, 4000, 20, 400]]],  # post-filter
             pitchAnchors=[150, 180], seed=14),
        dict(sylLen=600, amplAnchors=((0, .3, 1), (120, 60, 110)), amplAnchorsGlobal=((0, 1), (120, 80)),
             pitchAnchors=[220, 330, 200], seed=15),
        dict(sylLen=700, nonlinBalance=100, subDep=150, subFreq=60, jitterDep=2, shortestEpoch=50,   # vocal fry
             pitchAnchors=[110, 90], seed=16),
        dict(sylLen=800, samplingRate=22050, windowLength=50, pitchAnchors=[180, 240, 160], seed=17),  # hop 275.5
    ]
    return calls


def check_track(f0, ln, kw):
    y, ref = oracle_f0(kw)
    assert ln == y.size and ref.size == y.size
    got = f0[:ln]
    assert np.array_equal(got != 0, ref != 0), np.flatnonzero((got != 0) != (ref != 0))[:10]
    v = ref != 0
    ok = within_ulp(got[v], ref[v])
    assert ok.all(), (np.flatnonzero(v)[~ok][:5], got[v][~ok][:5], ref[v][~ok][:5])
    return int(v.sum())


def test_track_matches_the_oracle():
    calls = corpus()
    wave, lengths, st, f0 = sg.soundgen_batch_device(calls, f0=True)
    _, _, st2 = sg.soundgen_batch_device(calls)
    assert np.array_equal(st, st2)
    f, ln = f0.cpu().numpy(), lengths.cpu().numpy()
    assert f.shape == tuple(wave.shape) and f0.dtype == torch.float32
    voiced, refused = 0, []
    for i, kw in enumerate(calls):
        if st[i] == _abi.SGB_ERR_UNSUPPORTED:     # the odd clamped windows test_gpu_presets also finds refused
            refused.append(i)
            assert not f[i].any()
            continue
        assert st[i] == 0, (i, st[i])
        voiced += check_track(f[i], int(ln[i]), kw)
        assert not f[i, ln[i]:].any()
    assert len(refused) <= 2 and voiced > 0, refused


def test_fixed_batch_and_crop_is_a_prefix():
    calls = workloads.config1(n=2) + workloads.config3(n=2) + workloads.config0()
    bb = sg.BatchBuilder()
    for kw in calls:
        bb.add_soundgen(**kw)
    bt = sg.Batch()
    bt.upload(bb.build())
    bt.run()
    lens = bt.lengths()
    n, T = len(calls), int(lens.max())
    S = T + 37                                           # odd row stride
    full = torch.full((n * S,), float('nan'), dtype=torch.float32, device='cuda')
    assert np.array_equal(bt.f0(full, np.arange(n) * S, np.full(n, S)), lens)
    crop = torch.full((n * 1001,), float('nan'), dtype=torch.float32, device='cuda')
    bt.f0(crop, np.arange(n) * 1001, np.full(n, 1001))
    again = torch.empty_like(full)
    bt.f0(again, np.arange(n) * S, np.full(n, S))
    torch.cuda.synchronize()
    a, c = full.view(n, S).cpu().numpy(), crop.view(n, 1001).cpu().numpy()
    assert not np.isnan(a).any() and not np.isnan(c).any()
    assert torch.equal(full.view(torch.int32), again.view(torch.int32))       # two exports: the same bits
    for i, kw in enumerate(calls):
        check_track(a[i], int(lens[i]), kw)
        assert not a[i, lens[i]:].any()
        assert np.array_equal(c[i].view(np.int32), a[i, :1001].view(np.int32))
    bt.close()


def test_two_runs_are_bit_identical():
    calls = workloads.config3(n=4) + [dict(PS[('Cat', 'Hiss')], seed=900)] + workloads.config0()
    a = sg.soundgen_batch_device(calls, f0=True)[3]
    b = sg.soundgen_batch_device(calls, f0=True)[3]
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_failed_calls_give_zero_rows():
    calls = workloads.config1(n=1) + [dict(sylLen=300, pitchAnchors=[100, 150], temperature=0,
                                           noiseAnchors=((0, 300), (-10, -10)))]      # no uniforms: SGB_ERR_STREAM
    wave, lengths, st, f0 = sg.soundgen_batch_device(calls, f0=True)
    assert st[0] == 0 and st[1] != 0
    f = f0.cpu().numpy()
    assert f[0].any() and not f[1].any()


def test_stream_ordering_without_host_sync():
    calls = workloads.config3(n=32)
    bb = sg.BatchBuilder()
    for kw in calls:
        bb.add_soundgen(**kw)
    bt = sg.Batch()
    bt.upload(bb.build())
    bt.run()
    n, T = len(calls), int(bt.lengths().max())
    ref = torch.empty((n, T), dtype=torch.float32, device='cuda')
    bt.f0(ref, np.arange(n) * T, np.full(n, T))
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dst = torch.empty((n, T), dtype=torch.float32, device='cuda')
        torch.cuda._sleep(50_000_000)                  # keep the stream busy: the export must wait behind this
        bt.f0(dst, np.arange(n) * T, np.full(n, T), stream=s)
        sums = dst.double().sum(dim=1)                 # queued right away, no synchronise in between
    bb2 = sg.BatchBuilder()                            # the next run of the handle is queued behind the export
    for kw in workloads.config1(n=2):
        bb2.add_soundgen(**kw)
    bt.upload(bb2.build())
    bt.run()
    s.synchronize()
    assert torch.equal(dst.view(torch.int32), ref.view(torch.int32))
    assert torch.allclose(sums, ref.double().sum(dim=1), rtol=0, atol=0)
    bt.close()


def test_refusals():
    calls = workloads.config1(n=2)
    bb = sg.BatchBuilder()
    for kw in calls:
        bb.add_soundgen(**kw)
    bt = sg.Batch()
    bt.upload(bb.build())
    n = len(calls)
    dst = torch.empty((n, 30000), dtype=torch.float32, device='cuda')
    with pytest.raises(sg.SoundgenError) as ei:         # uploaded, never run
        bt.f0(dst, np.arange(n) * 30000, np.full(n, 30000))
    assert ei.value.code == _abi.SGB_ERR_STATE
    bt.run()
    T = int(bt.lengths().max())
    dst = torch.empty((n, T), dtype=torch.float32, device='cuda')
    ok_off, ok_cap = np.arange(n) * T, np.full(n, T)
    bad = [(torch.empty((n, T), dtype=torch.float32).pin_memory(), ok_off, ok_cap),
           (torch.empty((n, T), dtype=torch.float32), ok_off, ok_cap),
           (dst, np.zeros(n, dtype=np.int64), ok_cap),                 # rows overlap
           (dst, ok_off + 1, ok_cap),                                  # last row ends past dst
           (dst, ok_off - 1, ok_cap)]                                  # negative offset
    for d, off, cap in bad:
        with pytest.raises(sg.SoundgenError) as ei:
            bt.f0(d, off, cap)
        assert ei.value.code == _abi.SGB_ERR_INVALID
    L = _abi.load()
    o = _abi.DeviceOut()
    off, cp = np.ascontiguousarray(ok_off, dtype=np.int64), np.ascontiguousarray(ok_cap, dtype=np.int64)
    o.dst, o.dst_elems, o.dst_off, o.cap = dst.data_ptr(), dst.numel(), off.ctypes.data, cp.ctypes.data
    o.format = _abi.SGB_OUT_PCM16                                      # the track is float32 only
    assert L.sgb_batch_f0(bt.h, C.byref(o)) == _abi.SGB_ERR_INVALID
    bt.f0(dst, ok_off, ok_cap)                          # the refusals queued nothing and left the handle usable
    torch.cuda.synchronize()
    assert dst.abs().sum().item() > 0
    bt.close()

    src = torch.rand(4096, device='cuda')
    lab = torch.empty(64, device='cuda')
    one = np.zeros(1, dtype=np.int64)
    good = dict(src=src, src_off=one, lens=[4096], dst=lab, dst_off=one, cap=[8], wl=800, overlap=75)
    sg.rows_f0_frames(0, **good)
    for change in (dict(wl=801), dict(wl=2), dict(overlap=100), dict(overlap=-1), dict(wl=4, overlap=90),
                   dict(lens=[4097]), dict(src_off=[1]), dict(dst=src), dict(dst=torch.empty(64)),
                   dict(src=torch.rand(4096)), dict(cap=[33]), dict(dst_off=[-1])):
        with pytest.raises(sg.SoundgenError) as ei:
            sg.rows_f0_frames(0, **dict(good, **change))
        assert ei.value.code == _abi.SGB_ERR_INVALID, change


def test_frame_labels_equal_the_numpy_restatement():
    calls = workloads.config1(n=2) + workloads.config2(n=2) + [dict(PS[('Cat', 'Hiss')], seed=900)] + \
        workloads.config0() + [dict(sylLen=30, pitchAnchors=[300], temperature=0, addSilence=0)]   # shorter than wl
    wave, lengths, st, f0 = sg.soundgen_batch_device(calls, f0=True)
    f, ln = f0.cpu().numpy(), lengths.cpu().numpy()
    n, T = f.shape
    for wl, overlap in ((800, 75), (1102, 75), (2400, 75), (512, 50), (1000, 0), (64, 90)):
        S = T + 37                                      # odd strides on both sides
        src = torch.zeros(n * S, dtype=torch.float32, device='cuda')
        src.view(n, S)[:, :T] = f0
        nc = np.array([sg.api._abi.load().sgb_spec_frames(int(l), wl, float(overlap)) for l in ln])
        F = int(nc.max()) + 3
        D = 2 * F + 5
        dst = torch.full((n * D,), float('nan'), dtype=torch.float32, device='cuda')
        written = sg.rows_f0_frames(0, src, np.arange(n) * S, ln, dst, np.arange(n) * D, np.full(n, F), wl, overlap)
        assert np.array_equal(written, np.minimum(nc, F))
        crop = torch.full((n * D,), float('nan'), dtype=torch.float32, device='cuda')
        sg.rows_f0_frames(0, src, np.arange(n) * S, ln, crop, np.arange(n) * D, np.maximum(nc // 2, 1), wl, overlap)
        torch.cuda.synchronize()
        d, c = dst.view(n, D).cpu().numpy(), crop.view(n, D).cpu().numpy()
        for i in range(n):
            ref = frame_labels(f[i], int(ln[i]), wl, overlap, F)
            got = d[i, :2 * F].reshape(F, 2)
            assert np.array_equal(got.view(np.int32), ref.view(np.int32)), (wl, overlap, i)
            assert np.isnan(d[i, 2 * F:]).all()                         # nothing past the row
            k = max(nc[i] // 2, 1)
            assert np.array_equal(c[i, :2 * k].view(np.int32), d[i, :2 * k].view(np.int32))


def test_f0_frames_device_aligns_with_spectrogram_device():
    calls = workloads.config1(n=2) + workloads.config2(n=2) + workloads.config0()     # 44.1, 22.05 and 16 kHz
    sr = np.array([kw.get('samplingRate', 16000) for kw in calls], dtype=np.float64)
    wave, lengths, st, f0 = sg.soundgen_batch_device(calls, f0=True)
    spec, frames = sg.spectrogram_device(wave, lengths, sr, n_mels=40)
    labels, fr = sg.f0_frames_device(f0, lengths, sr)
    assert torch.equal(fr, frames) and labels.shape[:2] == spec.shape[:2] and labels.shape[2] == 2
    f, ln, lab = f0.cpu().numpy(), lengths.cpu().numpy(), labels.cpu().numpy()
    for i in range(len(calls)):
        wl = int(np.floor(50 / 1000 * sr[i] / 2) * 2)
        ref = frame_labels(f[i], int(ln[i]), wl, 75, lab.shape[1])
        assert np.array_equal(lab[i].view(np.int32), ref.view(np.int32)), i


def acf_f0(x, sr, lo=60.0, hi=600.0):
    """f0 of a frame from its normalised autocorrelation: the first lag whose peak reaches 0.9 of the highest one in
    [sr / hi, sr / lo], refined by a parabola through the peak."""
    x = x - x.mean()
    n = x.size
    r = np.fft.irfft(np.abs(np.fft.rfft(x, 2 * n)) ** 2)[:n]
    r = r / (r[0] * (n - np.arange(n)) / n)               # unbiased, normalised
    a, b = int(sr / hi), int(sr / lo) + 1
    seg = r[a:b]
    peaks = [j for j in range(1, seg.size - 1) if seg[j] >= seg[j - 1] and seg[j] > seg[j + 1]]
    top = max(seg[j] for j in peaks)
    j = next(j for j in peaks if seg[j] >= 0.9 * top)
    y0, y1, y2 = seg[j - 1], seg[j], seg[j + 1]
    lag = a + j + 0.5 * (y0 - y2) / (y0 - 2 * y1 + y2)
    return sr / lag


def test_labels_agree_with_the_waveform():
    """Clean calls (temperature 0, no noise, jitter or sub-harmonics): where a frame is fully voiced, the label's f0
    is within 1 % of an autocorrelation estimate of the waveform itself."""
    contours = [[150, 150], [320, 320], [110, 160], [400, 300, 420], [90, 95]]
    calls = [dict(sylLen=1200, pitchAnchors=p, temperature=0, subDep=0, jitterDep=0, shimmerDep=0, vibratoDep=0,
                  nonlinBalance=0, samplingRate=sr, invalidArgAction='ignore')
             for p in contours for sr in (16000, 44100)]
    wave, lengths, st, f0 = sg.soundgen_batch_device(calls, f0=True)
    assert np.all(st == 0)
    sr = np.array([kw['samplingRate'] for kw in calls], dtype=np.float64)
    labels, frames = sg.f0_frames_device(f0, lengths, sr, windowLength=40)
    w, lab, fr = wave.cpu().numpy(), labels.cpu().numpy(), frames.cpu().numpy()
    checked, worst = 0, 0.0
    for i in range(len(calls)):
        wl = int(np.floor(40 / 1000 * sr[i] / 2) * 2)
        h = wl - 75 * wl / 100
        for k in range(int(fr[i])):
            if lab[i, k, 1] != 1.0:
                continue
            s = int(np.floor(1 + k * h)) - 1
            est = acf_f0(w[i, s:s + wl].astype(np.float64), sr[i])
            err = abs(est / lab[i, k, 0] - 1)
            worst = max(worst, err)
            assert err < 0.01, (i, k, est, lab[i, k, 0])
            checked += 1
    assert checked > 200
    print('%d fully voiced frames, worst relative error %.2e' % (checked, worst))
