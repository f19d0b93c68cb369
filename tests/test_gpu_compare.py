"""Spectrogram comparison on the device (k_spec_compare through sgb_rows_compare and compare_spectrograms) against the
float64 reference on K9 features, its bit identity across runs, pair orders and batch sizes, stream order, the DTW
frame limit and the refusals; and match_pars end to end."""
import ctypes as C
import math

import numpy as np
import pytest

import soundgen_beta_b200 as sg
from compare_ref import score as ref_score
from soundgen_beta_b200 import _abi

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

SR, WL_MS = 16000, 50                    # wl 800, hop 200 at 75 % overlap
FRAMES = [0, 1, 2, 97, 400]
LENS = [0, 700, 1001, 800 + 1 + 96 * 200, 800 + 1 + 399 * 200]     # rows of exactly FRAMES frames


def signal_rows(seed):
    r = np.random.default_rng(seed)
    rows = np.zeros((len(LENS), max(LENS)), dtype=np.float32)
    for c, L in enumerate(LENS):
        t = np.arange(L)
        f0 = r.uniform(0.005, 0.02)
        x = 0.02 * r.standard_normal(L)
        for h in range(1, 10):
            x += np.sin(2 * np.pi * h * f0 * t * (1 + 0.3 * t / max(L, 1)) + r.uniform(0, 6)) / h
        rows[c, :L] = x * np.hanning(L + 2)[1:-1] if L else x
    return rows


def features(seed, kind):
    """K9 features of signal_rows(seed): 'mel' (64-band log-mel) or 'power' (400 bins)."""
    w = torch.tensor(signal_rows(seed), device='cuda')
    kw = dict(n_mels=64, db=True) if kind == 'mel' else {}
    spec, frames = sg.spectrogram_device(w, LENS, SR, windowLength=WL_MS, **kw)
    assert frames.cpu().tolist() == FRAMES
    return spec, frames


def check(got, a, af, b, bf, pairs, method, pad):
    A, B = a.double().cpu().numpy(), b.double().cpu().numpy()
    afh, bfh = np.asarray(af.cpu() if torch.is_tensor(af) else af), np.asarray(bf.cpu() if torch.is_tensor(bf) else bf)
    g = got.cpu().numpy()
    for c, p in enumerate(pairs):
        want = ref_score(A[c, :afh[c]], B[p, :bfh[p]], method, pad)
        if math.isnan(want):
            assert math.isnan(g[c]), (c, p, g[c])
        elif method == 'dtw':
            assert abs(g[c] - want) <= 2e-5 * abs(want) + 1e-300, (c, p, g[c], want)
        else:
            assert abs(g[c] - want) <= 1e-9, (c, p, g[c], want)


@pytest.mark.parametrize('kind', ['mel', 'power'])
@pytest.mark.parametrize('method', ['cor', 'cosine', 'dtw'])
def test_reference_parity(method, kind):
    a, af = features(1, kind)
    b, bf = features(2, kind)
    pad = -100.0 if kind == 'mel' else 1e-7
    n = len(FRAMES)
    # every row of a against every row of b (equal and unequal lengths, empty rows)
    ai = np.repeat(np.arange(n), n)
    pairs = np.tile(np.arange(n), n)
    aa, aaf = a[torch.as_tensor(ai, device='cuda')].contiguous(), af[torch.as_tensor(ai, device='cuda')]
    for pd in (0.0, pad):
        got = sg.compare_spectrograms(aa, aaf, b, bf, method, pairs=pairs, pad=pd)
        assert got.dtype == torch.float64 and got.is_cuda and got.shape == (n * n,)
        check(got, aa, aaf, b, bf, pairs, method, pd)
    # many candidates against one target row, b aliased (m = 1), and a row against itself
    tgt, tf = a[3:4].contiguous(), af[3:4]
    got = sg.compare_spectrograms(a, af, tgt, tf, method, pad=pad)
    check(got, a, af, tgt, tf, [0] * n, method, pad)
    same = sg.compare_spectrograms(tgt, tf, tgt, tf, method).item()
    assert same == (0.0 if method == 'dtw' else pytest.approx(1.0, abs=1e-9))


def test_nan_rules_on_the_device():
    F = 6
    a = torch.zeros((4, F, 3), device='cuda')
    a[1] = 2.5                                                  # constant
    a[2, :3] = torch.arange(9.0, device='cuda').view(3, 3)
    a[3, 0, 0] = 1.0
    af = torch.tensor([F, F, 3, 1])
    for method, want_nan in (('cor', [True, True, False, False]), ('cosine', [True, False, False, False])):
        s = sg.compare_spectrograms(a, af, a[2:3].contiguous(), af[2:3], method).cpu().numpy()
        assert list(np.isnan(s)) == want_nan, (method, s)
    for method in ('cor', 'cosine', 'dtw'):
        s = sg.compare_spectrograms(a, [0, F, 3, 1], a[2:3].contiguous(), [3], method).cpu().numpy()
        assert np.isnan(s[0]) and (method != 'dtw' or not np.isnan(s[1:]).any())
        s = sg.compare_spectrograms(a, af, a[2:3].contiguous(), [0], method).cpu().numpy()
        assert np.isnan(s).all()


@pytest.mark.parametrize('method', ['cor', 'cosine', 'dtw'])
def test_bit_identity(method):
    a, af = features(3, 'mel')
    tgt, tf = a[3:4].contiguous(), af[3:4]
    r = np.random.default_rng(4)
    # 2048 rows: the five rows over and over, plus random rows of random lengths
    idx = r.integers(0, len(FRAMES), 2048)
    big = a[torch.as_tensor(idx, device='cuda')].contiguous()
    bf = af[torch.as_tensor(idx, device='cuda')].clone()
    big[1000:] += torch.randn(big[1000:].shape, generator=torch.Generator('cuda').manual_seed(5), device='cuda')
    bf[1000:] = torch.as_tensor(r.integers(1, 401, 1048), device='cuda')
    s1 = sg.compare_spectrograms(big, bf, tgt, tf, method, pad=-100.0)
    s2 = sg.compare_spectrograms(big, bf, tgt, tf, method, pad=-100.0)
    assert torch.equal(s1.view(torch.int64), s2.view(torch.int64))                         # across runs
    perm = torch.as_tensor(r.permutation(2048), device='cuda')
    sp = sg.compare_spectrograms(big[perm].contiguous(), bf[perm], tgt, tf, method, pad=-100.0)
    assert torch.equal(sp.view(torch.int64), s1[perm].view(torch.int64))                  # across pair orders
    for c in (0, 3, 1500, 2047):                                                         # n = 1 against n = 2048
        one = sg.compare_spectrograms(big[c:c + 1].contiguous(), bf[c:c + 1], tgt, tf, method, pad=-100.0)
        assert one.view(torch.int64).item() == s1[c:c + 1].view(torch.int64).item()


def test_stream_order_without_host_sync():
    a, af = features(5, 'mel')
    tgt, tf = a[4:5].contiguous(), af[4:5]
    ref = sg.compare_spectrograms(a, af, tgt, tf, 'dtw')
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        x = torch.zeros_like(a)
        torch.cuda._sleep(50_000_000)                 # keep the stream busy: the copy and the comparison wait behind it
        x.copy_(a)
        got = sg.compare_spectrograms(x, af, tgt, tf, 'dtw', stream=s)
        got2 = got * 2                                # queued at once, no synchronise in between
    s.synchronize()
    assert torch.equal(got.view(torch.int64), ref.view(torch.int64))
    assert torch.allclose(got2, ref * 2, rtol=0, atol=0, equal_nan=True)     # row 0 has no frames: NaN


def test_dtw_frame_limit():
    M = _abi.SGB_CMP_DTW_MAX_FRAMES
    g = torch.Generator('cuda').manual_seed(6)
    a = torch.randn((1, M + 1, 8), generator=g, device='cuda')
    b = torch.randn((1, M, 8), generator=g, device='cuda')
    got = sg.compare_spectrograms(a, [M], b, [M], 'dtw').item()
    want = ref_score(a[0, :M].double().cpu().numpy(), b[0].double().cpu().numpy(), 'dtw')
    assert abs(got - want) <= 2e-5 * abs(want)
    with pytest.raises(sg.SoundgenError) as ei:
        sg.compare_spectrograms(a, [M + 1], b, [M], 'dtw')
    assert ei.value.code == _abi.SGB_ERR_UNSUPPORTED
    assert not math.isnan(sg.compare_spectrograms(a, [M + 1], b, [M], 'cor').item())    # no limit for cor


def _raw(a, a_elems, b, b_elems, dst, dst_elems, n=1, device=None, frames=2):
    p = _abi.CompareParams()
    p.method, p.n_feat, p.pad = 0, 4, 0.0
    off, fr = np.zeros(n, dtype=np.int64), np.full(n, frames, dtype=np.int64)
    L = _abi.load()
    return L.sgb_rows_compare(torch.cuda.current_device() if device is None else device, a, a_elems, b, b_elems,
                              off.ctypes.data, fr.ctypes.data, off.ctypes.data, fr.ctypes.data, n, C.byref(p), dst,
                              dst_elems, None)


def test_refusals():
    a = torch.randn(64, device='cuda')
    dst = torch.zeros(4, dtype=torch.float64, device='cuda')
    ok = _raw(a.data_ptr(), 64, a.data_ptr(), 64, dst.data_ptr(), 4)
    torch.cuda.synchronize()
    assert ok == 0 and dst[0].item() == pytest.approx(1.0, abs=1e-12)
    host = np.zeros(4)
    assert _raw(a.data_ptr(), 64, a.data_ptr(), 64, host.ctypes.data, 4) == _abi.SGB_ERR_INVALID      # host dst
    pinned = torch.zeros(64).pin_memory()
    assert _raw(pinned.data_ptr(), 64, a.data_ptr(), 64, dst.data_ptr(), 4) == _abi.SGB_ERR_INVALID   # host a
    assert _raw(a.data_ptr(), 64, host.ctypes.data, 64, dst.data_ptr(), 4) == _abi.SGB_ERR_INVALID   # host b
    assert _raw(a.data_ptr(), 64, a.data_ptr(), 64, dst.data_ptr() + 4, 3) == _abi.SGB_ERR_INVALID   # misaligned
    assert _raw(a.data_ptr(), 7, a.data_ptr(), 64, dst.data_ptr(), 4) == _abi.SGB_ERR_INVALID        # a row past a
    assert _raw(a.data_ptr(), 64, a.data_ptr(), 64, dst.data_ptr(), 1, n=2) == _abi.SGB_ERR_INVALID  # dst too short
    assert _raw(a.data_ptr(), 64, a.data_ptr(), 64, dst.data_ptr(), 4, device=torch.cuda.device_count()) \
        == _abi.SGB_ERR_INVALID                                                                      # no such device
    if torch.cuda.device_count() > 1:
        other = torch.zeros(4, dtype=torch.float64, device='cuda:1')
        assert _raw(a.data_ptr(), 64, a.data_ptr(), 64, other.data_ptr(), 4) == _abi.SGB_ERR_INVALID
    with pytest.raises(ValueError):
        sg.compare_spectrograms(a.view(1, 16, 4), [17], a.view(1, 16, 4), [16])                    # frames > F
    with pytest.raises(ValueError):
        sg.compare_spectrograms(a.view(2, 8, 4), [8, 8], a.view(4, 4, 4), [4] * 4)                 # n_feat ok, m != n
    with pytest.raises(ValueError):
        sg.compare_spectrograms(a.view(1, 16, 4), [16], a.view(1, 16, 4), [16], 'euclid')


# ---- match_pars ----
BASE = dict(sylLen=400, pitchAnchors=[150, 220, 170], jitterDep=0, shimmerDep=0, addSilence=50,
            formants=[dict(time=0, freq=700, amp=30, width=100), dict(time=0, freq=1300, amp=30, width=120),
                      dict(time=0, freq=2600, amp=20, width=200)])


def target():
    return sg.soundgen(**BASE, temperature=0, rolloff=-8, rolloffOct=-4).astype(np.float32)


def test_target_scores_one_against_itself():
    x = torch.tensor(target(), device='cuda').view(1, -1)
    spec, fr = sg.spectrogram_device(x, [x.shape[1]], SR, windowLength=40, overlap=50, n_mels=64, db=True)
    assert sg.compare_spectrograms(spec, fr, spec, fr, 'cor').item() == pytest.approx(1.0, abs=1e-9)


def test_match_pars_end_to_end():
    x = target()
    kw = dict(base=dict(BASE, rolloff=-25), n_candidates=32, max_iter=15, seed=7)
    best_kw, best, hist = sg.match_pars(x, SR, ['rolloff', 'rolloffOct'], **kw)
    assert len(hist) == 16 and hist[0]['values'].shape == (1, 2) and hist[1]['values'].shape == (32, 2)
    cur = [h['best'] for h in hist]
    assert all(c1 >= c0 for c0, c1 in zip(cur, cur[1:]))             # each step keeps or improves the score
    assert best == cur[-1] and any(h['accepted'] for h in hist[1:])
    print('match_pars: initial %.6f final %.6f rolloff %.3f rolloffOct %.3f' % (cur[0], best, best_kw['rolloff'],
                                                                               best_kw['rolloffOct']))
    assert best >= cur[0] + 0.002                                    # the margin: 0.002 of correlation
    assert abs(best_kw['rolloff'] + 8) < 17 - 4                      # closer to the target's -8 than -25 was, by 4 dB
    assert best_kw['samplingRate'] == SR and best_kw['temperature'] == 0
    # the same seed gives the same history, bit for bit
    _, best2, hist2 = sg.match_pars(x, SR, ['rolloff', 'rolloffOct'], **kw)
    assert best2 == best and len(hist2) == len(hist)
    for h, h2 in zip(hist, hist2):
        assert h['score'] == h2['score'] and h['accepted'] == h2['accepted'] and h['best'] == h2['best']
        assert np.array_equal(h['values'], h2['values'])


def test_match_pars_all_candidates_fail():
    x = target()
    # a noise segment without the uniforms it draws from: every candidate gets SGB_ERR_STREAM
    base = dict(sylLen=300, pitchAnchors=[100, 150], noiseAnchors=((0, 300), (-10, -10)))
    best_kw, best, hist = sg.match_pars(x, SR, ['rolloff'], base=base, n_candidates=4, max_iter=2, method='dtw')
    assert best == -math.inf and len(hist) == 3
    assert all(h['score'] == -math.inf and h['best'] == -math.inf for h in hist)
    assert not any(h['accepted'] for h in hist[1:])
