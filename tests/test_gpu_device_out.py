"""Device output: waveforms exported straight into caller-owned CUDA memory (sgb_batch_export / sgb_rows_export,
Batch.export, soundgen_batch_device, PipelinedBatches(device_out=...)) equal what the host fetches return, bit for
bit, and are ordered on the caller's stream without a host synchronisation."""
import numpy as np
import pytest

import soundgen_beta_b200 as sg
from oracle import soundgen_oracle as so
from oracle.rrng import RRng
from oracle.soundgen_call import soundgen as osg
from soundgen_beta_b200 import _abi, api, presets, workloads

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

PS = {(s, n): kw for s, n, kw in presets.load()}
SCREAM = dict(PS[('Cat', 'Scream')], seed=904)      # 2 bouts; the moving stochastic main filter defers the second


def mixed_calls():
    calls = workloads.config0() + workloads.config1(n=2) + workloads.config3(n=1)
    calls += [dict(PS[('Cat', 'Hiss')], seed=900), dict(PS[('Misc', 'Seagull')], seed=901), SCREAM]
    # a noise segment without the uniform buffer it draws from: the front-end marks the call SGB_ERR_STREAM
    calls.append(dict(sylLen=300, pitchAnchors=[100, 150], temperature=0, noiseAnchors=((0, 300), (-10, -10))))
    return calls


def built(calls):
    bb = sg.BatchBuilder()
    for kw in calls:
        bb.add_soundgen(**kw)
    bt = sg.Batch()
    bt.upload(bb.build())
    bt.run()
    return bt


def test_equals_host_path_bit_for_bit(monkeypatch):
    calls = mixed_calls()
    ref, st_ref = sg.soundgen_batch(calls, out_dtype=np.float32)
    rounds = []
    orig = api.FrontEnd.round_begin

    def counting(self):
        d, n = orig(self)
        if n:
            rounds.append(n)
        return d, n
    monkeypatch.setattr(api.FrontEnd, 'round_begin', counting)
    wave, lengths, st = sg.soundgen_batch_device(calls)
    assert len(rounds) == 2, rounds                  # Scream really ran a second round
    assert np.array_equal(st, st_ref) and np.any(st != 0), st
    assert wave.dtype == torch.float32 and wave.is_cuda and lengths.dtype == torch.int64 and lengths.is_cuda
    w, ln = wave.cpu().numpy(), lengths.cpu().numpy()
    assert w.shape == (len(calls), max(r.size for r in ref))
    for i, r in enumerate(ref):
        assert ln[i] == r.size
        assert np.array_equal(w[i, :r.size], r), i
        assert np.all(w[i, r.size:] == 0), i


def test_zero_fill_is_the_kernels():
    calls = workloads.config1(n=2) + workloads.config0()
    bt = built(calls)
    host = bt.fetch(np.float32)
    n, T = len(calls), max(h.size for h in host)
    S = T + 37                                       # odd row stride: no row is aligned
    dst = torch.full((n * S,), float('nan'), dtype=torch.float32, device='cuda')
    written = bt.export(dst, np.arange(n) * S, np.full(n, S))
    torch.cuda.synchronize()
    assert np.array_equal(written, [h.size for h in host])
    w = dst.view(n, S).cpu().numpy()
    assert not np.isnan(w).any()
    for i, h in enumerate(host):
        assert np.array_equal(w[i, :h.size], h) and np.all(w[i, h.size:] == 0)
    bt.close()


def test_crop():
    calls = workloads.config0() + workloads.config1(n=2) + [dict(PS[('Cat', 'Hiss')], seed=900)]
    ref, _ = sg.soundgen_batch(calls, out_dtype=np.float32)
    T = int(np.median([r.size for r in ref]))
    assert min(r.size for r in ref) < T < max(r.size for r in ref)
    wave, lengths, _ = sg.soundgen_batch_device(calls, max_len=T)
    w, ln = wave.cpu().numpy(), lengths.cpu().numpy()
    assert w.shape == (len(calls), T)
    for i, r in enumerate(ref):
        k = min(r.size, T)
        assert ln[i] == k and np.array_equal(w[i, :k], r[:k]) and np.all(w[i, k:] == 0)


def test_pcm16_single_round_equals_host_fetch():
    calls = workloads.config1(n=3) + workloads.config0()
    bt = built(calls)
    host = bt.fetch(np.int16)
    n, T = len(calls), max(h.size for h in host)
    dst = torch.empty((n, T), dtype=torch.int16, device='cuda')
    bt.export(dst, np.arange(n) * T, np.full(n, T), fmt='pcm16')
    wave, lengths, _ = sg.soundgen_batch_device(calls, dtype=torch.int16)
    a, b = dst.cpu().numpy(), wave.cpu().numpy()
    for i, h in enumerate(host):
        assert np.array_equal(a[i, :h.size], h) and np.all(a[i, h.size:] == 0), i
        assert np.array_equal(b[i, :h.size], h) and np.all(b[i, h.size:] == 0), i
    bt.close()


def test_pcm16_multi_round_call_is_normalised_over_the_whole_call():
    wave, lengths, st = sg.soundgen_batch_device([SCREAM], dtype=torch.int16)
    assert st[0] == 0
    kw = dict(SCREAM)
    ref = so.savewav_pcm16(osg(rng=RRng(kw.pop('seed')), **kw))
    q = wave[0, :int(lengths[0])].cpu().numpy()
    assert q.size == ref.size
    d = np.abs(q.astype(np.int64) - ref)
    assert d.max() <= 1 and np.mean(d > 0) < 0.2
    assert np.max(np.abs(ref)) >= 32700


def test_stream_ordering_without_host_sync():
    calls = workloads.config3(n=64)
    bt = built(calls)
    host = bt.fetch(np.float32)
    n, T = len(calls), max(h.size for h in host)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dst = torch.empty((n, T), dtype=torch.float32, device='cuda')
        torch.cuda._sleep(50_000_000)            # keep the stream busy: the export must wait behind this
        bt.export(dst, np.arange(n) * T, np.full(n, T), stream=s)
        sums = dst.double().sum(dim=1)           # queued right away, no synchronise in between
    # the same handle takes a different batch at once: its run must not overwrite the rows before they are read
    bt.upload(built_desc(workloads.config1(n=4)))
    bt.run()
    s.synchronize()
    want = np.array([np.sum(h.astype(np.float64)) for h in host])
    assert np.allclose(sums.cpu().numpy(), want, rtol=1e-12, atol=1e-9)
    w = dst.cpu().numpy()
    for i, h in enumerate(host):
        assert np.array_equal(w[i, :h.size], h)
    bt.close()


def built_desc(calls):
    bb = sg.BatchBuilder()
    for kw in calls:
        bb.add_soundgen(**kw)
    return bb.build()


@pytest.mark.parametrize('dtype', ['float32', 'int16'])
def test_pipelined_batches_device_out(dtype):
    calls = workloads.config1(n=3) + workloads.config0(n=2)
    subs = [calls[:2], calls[2:]]
    descs = [built_desc(c) for c in subs]
    pipe = sg.PipelinedBatches(descs, device_out=dict(dtype=getattr(torch, dtype)))
    pipe.run_steps(2)
    got = [(w, ln) for w, ln in pipe.results]
    for s in pipe.streams:
        s.synchronize()
    pipe.close()
    for (w, ln), c in zip(got, subs):
        bt = built(c)
        host = bt.fetch(np.int16 if dtype == 'int16' else np.float32)
        bt.close()
        w, ln = w.cpu().numpy(), ln.cpu().numpy()
        assert w.shape == (len(c), max(h.size for h in host))
        for i, h in enumerate(host):
            assert ln[i] == h.size and np.array_equal(w[i, :h.size], h) and np.all(w[i, h.size:] == 0)


def test_refusals():
    calls = workloads.config1(n=2)
    desc = built_desc(calls)
    bt = sg.Batch()
    bt.upload(desc)
    n = len(calls)
    dst = torch.empty((n, 30000), dtype=torch.float32, device='cuda')
    with pytest.raises(sg.SoundgenError) as ei:         # uploaded, never run
        bt.export(dst, np.arange(n) * 30000, np.full(n, 30000))
    assert ei.value.code == _abi.SGB_ERR_STATE
    bt.run()
    T = int(bt.lengths().max())
    dst = torch.empty((n, T), dtype=torch.float32, device='cuda')
    ok_off, ok_cap = np.arange(n) * T, np.full(n, T)
    pinned = torch.empty((n, T), dtype=torch.float32).pin_memory()
    pageable = torch.empty((n, T), dtype=torch.float32)
    bad = [(pinned, ok_off, ok_cap), (pageable, ok_off, ok_cap),
           (dst, np.zeros(n, dtype=np.int64), ok_cap),                 # rows overlap
           (dst, ok_off + 1, ok_cap),                                  # last row ends past dst
           (dst, ok_off, ok_cap + 1),                                  # rows overlap and run past dst
           (dst, ok_off - 1, ok_cap)]                                  # negative offset
    for d, off, cap in bad:
        with pytest.raises(sg.SoundgenError) as ei:
            bt.export(d, off, cap)
        assert ei.value.code == _abi.SGB_ERR_INVALID
    bt.export(dst, ok_off, ok_cap)                      # the refusals queued nothing and left the handle usable
    torch.cuda.synchronize()
    host = bt.fetch(np.float32)
    assert all(np.array_equal(dst[i, :h.size].cpu().numpy(), h) for i, h in enumerate(host))
    bt.close()
    fresh = sg.Batch()                                  # never uploaded
    with pytest.raises(sg.SoundgenError) as ei:
        fresh.export(dst[:0], np.zeros(0), np.zeros(0))
    assert ei.value.code == _abi.SGB_ERR_STATE
    fresh.close()


def test_refusal_on_a_second_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two CUDA devices')
    bt = built(workloads.config0())
    T = int(bt.lengths()[0])
    other = torch.empty(T, dtype=torch.float32, device='cuda:1')
    with pytest.raises(sg.SoundgenError) as ei:
        bt.export(other, [0], [T])
    assert ei.value.code == _abi.SGB_ERR_INVALID
    bt.close()


def test_exports_are_deterministic():
    calls = workloads.config1(n=2) + [dict(PS[('Cat', 'Hiss')], seed=900)]
    bt = built(calls)
    n, T = len(calls), int(bt.lengths().max())
    out = []
    for fmt, dt in (('f32', torch.float32), ('f32', torch.float32), ('pcm16', torch.int16), ('pcm16', torch.int16)):
        d = torch.empty((n, T), dtype=dt, device='cuda')
        bt.export(d, np.arange(n) * T, np.full(n, T), fmt=fmt)
        out.append(d)
    torch.cuda.synchronize()
    assert torch.equal(out[0].view(torch.int32), out[1].view(torch.int32))
    assert torch.equal(out[2], out[3])
    bt.close()
