"""Spectrograms of the resident cfg3 batch on one GPU: one JSON line.

    python scripts/bench_spectrogram.py [--batch 8192] [--steps 5] [--reps 3] [--mels 128] [--out FILE]

Measured in one process on the same resident batch (inputs uploaded once, outputs left on the device):
  step            one resident run (Batch.run: synthesis through the K2 filter and finalisation);
  step_linear     the run plus Batch.spectrogram of every call: power, wl 2400 (50 ms at 48 kHz), 75 % overlap,
                  into one [calls, F, 1200] float32 tensor;
  step_logmel     the run plus a `--mels`-band HTK mel bank in dB into [calls, F, mels].
The three modes alternate `--reps` times, `--steps` steps each; each reports its best per-step time (host clock
around the steps, ended by a synchronise).  filter_ms: K2's time in the same runs (sgb_run_info.ms[filter]), best.
kernel: k_spectrogram alone, from torch.profiler's CUDA activity in a separate profiled pass, and from CUDA events
around `--iters` calls on one stream (row tables staged and the stream hand-offs included).  Algorithmic bytes: 4 B
per input sample read (the sum of the call lengths) + 4 B per output value written (calls x F x n_feat, zero tails
included); GB/s against the 7.7 TB/s HBM3e data-sheet figure of one B200.  FFT flops: 5 N log2 N per complex FFT of
N = wl points, one per frame pair.  The card name and power limit are read in the same run.  Writes nothing but
`--out`.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HBM_DATASHEET_GBS = 7700.0


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(',')[:2]]
        return name, power
    except Exception as e:
        return None, 'unknown (%s)' % type(e).__name__


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--batch', type=int, default=8192)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--mels', type=int, default=128)
    ap.add_argument('--out', default=None, help='also append the JSON line here')
    args = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    import torch
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi, workloads
    if not torch.cuda.is_available():
        sys.exit('bench_spectrogram: no CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    L = _abi.load()
    assert L.sgb_set_device(0) == 0

    calls = workloads.config3(n=args.batch)
    bb = sg.BatchBuilder(u_dtype=np.float32)
    for kw in calls:
        bb.add_soundgen(**kw)
    desc = bb.build()
    sg.pin_desc(desc)
    bt = sg.Batch()
    bt.upload(desc)
    for _ in range(max(1, args.warmup)):
        bt.run()
    lens = bt.lengths()
    n, wl, ov, sr = len(calls), 2400, 75, 48000
    nc = np.array([L.sgb_spec_frames(int(x), wl, float(ov)) for x in lens], dtype=np.int64)
    F = int(nc.max())
    bank = sg.mel_filterbank(sr, wl, args.mels)
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        lin = torch.empty((n, F, wl // 2), dtype=torch.float32, device=dev)
        mel = torch.empty((n, F, args.mels), dtype=torch.float32, device=dev)
    modes = {
        'step': None,
        'step_linear': lambda: bt.spectrogram(lin, np.arange(n) * F * (wl // 2), np.full(n, F), wl, ov, stream=stream),
        'step_logmel': lambda: bt.spectrogram(mel, np.arange(n) * F * args.mels, np.full(n, F), wl, ov, bands=bank,
                                              db=True, stream=stream),
    }
    filt = []

    def timed(mode):
        f = modes[mode]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            filt.append(bt.run().ms[_abi.T_NAMES.index('filter')])
            if f is not None:
                f()
        stream.synchronize()
        return (time.perf_counter() - t0) / args.steps * 1e3

    for m in modes:
        timed(m)                                           # warms every shape
    best = {m: math.inf for m in modes}
    for _ in range(args.reps):
        for m in modes:
            best[m] = min(best[m], timed(m))

    samples = int(lens.sum())
    pairs = int(np.sum((nc + 1) // 2))
    flops = pairs * 5.0 * wl * math.log2(wl)
    kern = {}
    for m, nf in (('step_linear', wl // 2), ('step_logmel', args.mels)):
        f = modes[m]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.iters):
            f()
        e1.record(stream)
        e1.synchronize()
        ev_ms = e0.elapsed_time(e1) / args.iters
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                f()
            stream.synchronize()
        kt = [e.device_time_total / max(1, e.count) for e in prof.key_averages() if e.key.startswith('k_spectrogram')]
        k_ms = kt[0] * 1e-3 if kt else None
        algo = 4 * samples + 4 * n * F * nf
        kern[m] = {'n_feat': nf, 'bytes': algo, 'out_bytes': 4 * n * F * nf, 'event_ms': ev_ms,
                   'event_gbs': algo / (ev_ms * 1e-3) / 1e9, 'kernel_ms': k_ms,
                   'kernel_gbs': algo / (k_ms * 1e-3) / 1e9 if k_ms else None,
                   'frac_of_datasheet_hbm': algo / (k_ms * 1e-3) / 1e9 / HBM_DATASHEET_GBS if k_ms else None,
                   'fft_gflops': flops / (k_ms * 1e-3) / 1e9 if k_ms else None}
        if k_ms is None:
            kern[m]['kernel_note'] = 'the profiler listed no k_spectrogram launch: kernel time not measured'
    bt.close()
    name, power = gpu_info()
    line = {'config': workloads.NAMES[3], 'calls': n, 'steps': args.steps, 'reps': args.reps,
            'gpu': name or torch.cuda.get_device_name(dev), 'power_limit': power, 'wl': wl, 'overlap': ov,
            'frames_per_call_max': F, 'frames_per_call_mean': float(nc.mean()), 'samples': samples,
            'frame_pairs': pairs, 'fft_flops': flops,
            'ms_per_step': best, 'added_ms': {m: best[m] - best['step'] for m in ('step_linear', 'step_logmel')},
            'filter_ms_best': min(filt), 'k_spectrogram': kern, 'hbm_datasheet_gbs': HBM_DATASHEET_GBS}
    js = json.dumps(line)
    print(js, flush=True)
    if args.out:
        with open(args.out, 'a') as f:
            f.write(js + '\n')


if __name__ == '__main__':
    main()
