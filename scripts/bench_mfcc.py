"""MFCCs of the resident cfg3 batch on one GPU (K9 log-mel, then K11), and match_pars on mel and MFCC features: one
JSON line.

    python scripts/bench_mfcc.py [--batch 8192] [--steps 5] [--reps 3] [--candidates 512] [--out FILE]

Measured in one process on the same resident batch (inputs uploaded once, outputs left on the device):
  step            one resident run (Batch.run);
  step_logmel     the run plus Batch.spectrogram of every call: 64-band HTK log-mel, wl 2400 (50 ms at 48 kHz), 75 %
                  overlap, into [calls, F, 64];
  step_mfcc       the same plus rows_cepstra over it (K11): 13 coefficients of the DCT-II with c0, delta and
                  delta-delta over 5 frames (delta_n 2), into [calls, F, 39].
The three modes alternate --reps times, --steps steps each; each reports its best per-step time (host clock around
the steps, ended by a synchronise).
k_cepstra alone: torch.profiler's CUDA activity in a profiled pass of its own, --iters (K9, K11) pairs, so K11 reads
features K9 has just written (about 205 MB, more than the 126 MB of L2: mostly not L2-resident); and CUDA events
around --iters K11 calls back to back (row tables staged and stream hand-offs included).  Algorithmic bytes,
computed from the tiling: 4 B per input value of every tile's staged frames (the halo re-reads included) + 4 B per
output value (zero tails included) + the matrix once per tile; against the 7.7 TB/s HBM3e data-sheet figure.
FLOPs: 2 n_in n_ceps per staged frame (the halo's cepstra are recomputed per tile) + 3 delta_n + 1 per delta value.
match_pars: per-step time of match_pars with --candidates candidates (difference of a 4-step and a 1-step search
after a warm-up, best of 2), features 'mel' against 'mfcc' (13 coefficients without c0, deltas=1), cor and dtw.
The card name and power limit are read in the same run.  Writes nothing but --out.
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
TILE = 64                    # CEPS_TILE of csrc/engine.cuh


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(',')[:2]]
        return name, power
    except Exception as e:
        return None, 'unknown (%s)' % type(e).__name__


def k11_counts(nc, cap, n_in, n_ceps, order, dn):
    """Algorithmic bytes and FLOPs of one K11 call, tile by tile as the host builds them."""
    H, n_out = order * dn, n_ceps * (1 + order)
    staged = deltas = tiles = 0
    for f, c in zip(nc.tolist(), cap.tolist()):
        m = min(f, c)
        for t0 in range(0, m, TILE):
            t1 = min(m, t0 + TILE)
            staged += min(t1 + H, f) - max(t0 - H, 0)
            if order >= 1:                 # the tile's last order
                deltas += (t1 - t0) * n_ceps
            if order == 2:                 # the first order over the tile and its halo
                deltas += (min(t1 + dn, f) - max(t0 - dn, 0)) * n_ceps
            tiles += 1
    out = int(np.sum(cap)) * n_out
    byts = 4 * staged * n_in + 4 * out + 4 * tiles * n_in * n_ceps
    flops = 2.0 * n_in * n_ceps * staged + (3 * dn + 1) * deltas
    return byts, flops, staged, tiles


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--batch', type=int, default=8192)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--candidates', type=int, default=512)
    ap.add_argument('--out', default=None, help='also append the JSON line here')
    args = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    import torch
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi, workloads
    if not torch.cuda.is_available():
        sys.exit('bench_mfcc: no CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    L = _abi.load()
    assert L.sgb_set_device(0) == 0
    name, power = gpu_info()

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
    n, wl, ov, sr, nm, nk, order, dn = len(calls), 2400, 75, 48000, 64, 13, 2, 2
    n_out = nk * (1 + order)
    nc = np.array([L.sgb_spec_frames(int(x), wl, float(ov)) for x in lens], dtype=np.int64)
    F = int(nc.max())
    bank = sg.mel_filterbank(sr, wl, nm)
    M = sg.dct_matrix(nk, nm).astype(np.float32)
    rows = np.arange(n, dtype=np.int64)
    cap = np.full(n, F, dtype=np.int64)
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        mel = torch.empty((n, F, nm), dtype=torch.float32, device=dev)
        feat = torch.empty((n, F, n_out), dtype=torch.float32, device=dev)

    def logmel():
        bt.spectrogram(mel, rows * F * nm, cap, wl, ov, bands=bank, db=True, stream=stream)

    def k11():
        sg.rows_cepstra(0, mel, rows * F * nm, nc, feat, rows * F * n_out, cap, M, order, dn, stream)

    modes = {'step': [], 'step_logmel': [logmel], 'step_mfcc': [logmel, k11]}

    def timed(mode):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            bt.run()
            for f in modes[mode]:
                f()
        stream.synchronize()
        return (time.perf_counter() - t0) / args.steps * 1e3

    for m in modes:
        timed(m)                                           # warms every shape
    best = {m: math.inf for m in modes}
    for _ in range(args.reps):
        for m in modes:
            best[m] = min(best[m], timed(m))

    # k_cepstra alone
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.iters):
        k11()
    e1.record(stream)
    e1.synchronize()
    ev_ms = e0.elapsed_time(e1) / args.iters
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.iters):
            logmel()
            k11()
        stream.synchronize()
    kt = [e.device_time_total / max(1, e.count) for e in prof.key_averages() if e.key.startswith('k_cepstra')]
    k_ms = kt[0] * 1e-3 if kt else None
    sp = [e.device_time_total / max(1, e.count) for e in prof.key_averages() if e.key.startswith('k_spectrogram')]
    byts, flops, staged, tiles = k11_counts(nc, cap, nm, nk, order, dn)
    kern = {'n_in': nm, 'n_ceps': nk, 'delta_order': order, 'delta_n': dn, 'tiles': tiles,
            'staged_frames': staged, 'frames': int(nc.sum()), 'input_bytes_k9_wrote': 4 * n * F * nm,
            'bytes': byts, 'flops': flops, 'event_ms': ev_ms, 'kernel_ms': k_ms,
            'k_spectrogram_ms_same_pass': sp[0] * 1e-3 if sp else None}
    if k_ms:
        kern.update(kernel_gbs=byts / (k_ms * 1e-3) / 1e9, frac_of_datasheet_hbm=byts / (k_ms * 1e-3) / 1e9 /
                    HBM_DATASHEET_GBS, gflops=flops / (k_ms * 1e-3) / 1e9)
    else:
        kern['kernel_note'] = 'the profiler listed no k_cepstra launch: kernel time not measured'
    # the features agree with a torch restatement on a few rows (a guard that the timed call computes MFCCs)
    torch.cuda.synchronize()
    ref = mel[:4].double() @ torch.tensor(M, dtype=torch.float64, device=dev).T
    got = feat[:4, :, :nk].double()
    kern['check_max_abs_err_c'] = float(torch.max(torch.abs(got - ref) * (torch.arange(F, device=dev)[None, :, None] <
                                                  torch.as_tensor(nc[:4], device=dev)[:, None, None])).item())
    bt.close()
    del mel, feat
    torch.cuda.empty_cache()

    # match_pars on mel and MFCC features
    call = workloads.config3(n=1)[0]
    base = dict(call, rolloff=-20.0)
    x = sg.soundgen(**dict(call, rolloff=-3.0)).astype(np.float32)
    mp = {}
    for features in ('mel', 'mfcc'):
        for method in ('cor', 'dtw'):
            kw = dict(base=base, n_candidates=args.candidates, method=method, windowLength=40, overlap=50,
                      features=features, deltas=1, seed=1)
            sg.match_pars(x, sr, ['rolloff', 'jitterDep', 'vibratoDep'], max_iter=1, **kw)     # warm-up
            tt = {}
            for it in (1, 4):
                tt[it] = math.inf
                for _ in range(2):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    _, sc, _ = sg.match_pars(x, sr, ['rolloff', 'jitterDep', 'vibratoDep'], max_iter=it, **kw)
                    tt[it] = min(tt[it], (time.perf_counter() - t0) * 1e3)
            mp['%s_%s' % (features, method)] = {'step_ms': (tt[4] - tt[1]) / 3, 'best_score_4_steps': sc}
    line = {'config': workloads.NAMES[3], 'calls': n, 'steps': args.steps, 'reps': args.reps,
            'gpu': name or torch.cuda.get_device_name(dev), 'power_limit': power, 'wl': wl, 'overlap': ov,
            'n_mels': nm, 'frames_per_call_max': F, 'frames_per_call_mean': float(nc.mean()),
            'ms_per_step': best, 'added_ms': {m: best[m] - best['step'] for m in ('step_logmel', 'step_mfcc')},
            'k11_added_ms': best['step_mfcc'] - best['step_logmel'], 'k_cepstra': kern,
            'match_pars_candidates': args.candidates, 'match_pars': mp, 'hbm_datasheet_gbs': HBM_DATASHEET_GBS}
    js = json.dumps(line)
    print(js, flush=True)
    if args.out:
        with open(args.out, 'a') as f:
            f.write(js + '\n')


if __name__ == '__main__':
    main()
