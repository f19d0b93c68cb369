"""match_pars steps on one GPU: one JSON line.

    python scripts/bench_match_pars.py [--candidates 64 512 4096] [--methods cor cosine dtw] [--steps 3] [--out FILE]

Workload: a 1 s target at 48 kHz synthesised from the first call of workloads.config3 (cfg3: low pitch, jitter,
shimmer, vibrato, subharmonics) with rolloff -3; the search starts from the same call at rolloff -20 and searches
rolloff, jitterDep and vibratoDep; features: 64-band log-mel, windowLength 40 ms (wl 1920), overlap 50 %.
For each candidate count and method:
  step_ms       one search step as match_pars runs it (wiggle_pars for every candidate, soundgen_batch_device,
                spectrogram_device, compare_spectrograms, the argmax read back), host clock, best of --steps after
                one warm-up step; candidates_per_s = candidates / step_ms.
  split_ms      the same step with a synchronise after each stage: host = wiggle_pars; synth = soundgen_batch_device
                (front-end, upload, synthesis, export); k9 = spectrogram_device; k10 = compare_spectrograms (CUDA
                events around the call: row-table staging and stream hand-offs included).  Best of --steps each.
  k10           k_spec_compare alone from torch.profiler's CUDA activity, in a separate profiled pass over --iters
                calls on the last step's features; its share of step_ms.  Bytes (cor, cosine): 4 B per feature of
                each row of a pair read once (candidate + target), against the 7.7 TB/s HBM3e data-sheet figure.
                DTW: cells = sum of n_a * n_b over the pairs, per second of kernel time.
The card name and power limit are read in the same run.  Writes nothing but --out.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HBM_DATASHEET_GBS = 7700.0
SR = 48000
PARS = ['rolloff', 'jitterDep', 'vibratoDep']
SPEC = dict(windowLength=40, overlap=50, n_mels=64, db=True, db_floor=1e-10)


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
    ap.add_argument('--candidates', type=int, nargs='+', default=[64, 512, 4096])
    ap.add_argument('--methods', nargs='+', default=['cor', 'cosine', 'dtw'])
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--out', default=None, help='also append the JSON line here')
    args = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    import torch
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import workloads
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: nothing here is measured without one')
    name, power = gpu_info()
    call = workloads.config3(n=1)[0]
    base = dict(call, rolloff=-20.0)
    x = sg.soundgen(**dict(call, rolloff=-3.0)).astype(np.float32)
    dev = torch.device('cuda', torch.cuda.current_device())
    xt = torch.tensor(x, device=dev).view(1, -1)
    tgt, tf = sg.spectrogram_device(xt, [x.size], SR, **SPEC)
    pad = -100.0
    cur = {nm: float(base[nm]) for nm in PARS}
    res = dict(gpu=name, power_limit=power, target_samples=int(x.size), target_frames=int(tf.item()),
               n_feat=SPEC['n_mels'], pars=PARS, runs={})

    def step(n, method, rng, split=False):
        t = [time.perf_counter()]
        cands = [sg.wiggle_pars(cur, PARS, 0.25, 0.1, rng) for _ in range(n)]
        t.append(time.perf_counter())
        wave, lengths, status = sg.soundgen_batch_device([dict(base, **c) for c in cands], device=dev.index)
        if split:
            torch.cuda.synchronize()
        t.append(time.perf_counter())
        spec, frames = sg.spectrogram_device(wave, lengths, SR, **SPEC)
        if split:
            torch.cuda.synchronize()
        t.append(time.perf_counter())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s = sg.compare_spectrograms(spec, frames, tgt, tf, method, pad=pad)
        e1.record()
        bad = torch.as_tensor(np.asarray(status) != 0, device=dev) | torch.isnan(s)
        s = torch.where(bad, torch.full_like(s, -np.inf), s)
        i = torch.argmax(s)
        got = torch.stack((s[i], i.to(torch.float64))).cpu()
        t.append(time.perf_counter())
        ms = np.diff(t) * 1e3
        return dict(total=float(sum(ms)), host=float(ms[0]), synth=float(ms[1]), k9=float(ms[2]),
                    k10=float(e0.elapsed_time(e1))), spec, frames, int(np.sum(status != 0)), float(got[0])

    for n in args.candidates:
        for method in args.methods:
            rng = np.random.default_rng(1)
            step(n, method, rng)                                            # warm-up
            e2e = [step(n, method, rng)[0]['total'] for _ in range(args.steps)]
            splits = [step(n, method, rng, split=True) for _ in range(args.steps)]
            _, spec, frames, failed, best = splits[-1]
            split = {k: min(s[0][k] for s in splits) for k in ('host', 'synth', 'k9', 'k10')}
            # k_spec_compare alone under torch.profiler (a pass of its own)
            from torch.profiler import ProfilerActivity, profile
            sg.compare_spectrograms(spec, frames, tgt, tf, method, pad=pad)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.iters):
                    sg.compare_spectrograms(spec, frames, tgt, tf, method, pad=pad)
                torch.cuda.synchronize()
            ks = [e for e in prof.key_averages() if 'k_spec_compare' in e.key]
            k_ms = (sum(getattr(e, 'device_time_total', getattr(e, 'cuda_time_total', 0)) for e in ks)
                    / max(1, sum(e.count for e in ks)) / 1e3) if ks else None
            fr = frames.cpu().numpy()
            step_ms = min(e2e)
            r = dict(step_ms=step_ms, candidates_per_s=n / step_ms * 1e3, split_ms=split, failed=failed,
                     best_score=best, frames_mean=float(fr.mean()), k10_kernel_ms=k_ms,
                     k10_share_of_step=(k_ms / step_ms) if k_ms else None)
            if k_ms:
                if method == 'dtw':
                    cells = float(np.sum(fr.astype(np.float64) * float(tf.item())))
                    r.update(dtw_cells=cells, dtw_gcells_per_s=cells / k_ms / 1e6)
                else:
                    nbytes = float(4 * SPEC['n_mels'] * np.sum(fr + int(tf.item())))
                    r.update(bytes=nbytes, gbs=nbytes / k_ms / 1e6,
                             frac_of_datasheet_hbm=nbytes / k_ms / 1e6 / HBM_DATASHEET_GBS)
            res['runs']['%d_%s' % (n, method)] = r
            print('%5d %-6s step %8.2f ms  %9.0f cand/s  split %s  k10 %s ms' % (
                n, method, step_ms, r['candidates_per_s'], {k: round(v, 3) for k, v in split.items()}, k_ms),
                flush=True)
    res['hbm_datasheet_gbs'] = HBM_DATASHEET_GBS
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'a') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
