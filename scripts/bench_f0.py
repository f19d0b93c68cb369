"""The f0 labels of the resident cfg3 batch on one GPU (K12a track, K12b frame labels): one JSON line.

    python scripts/bench_f0.py [--batch 8192] [--steps 5] [--reps 3] [--iters 10] [--out FILE]

Measured in one process on the same resident batch (inputs uploaded once, outputs left on the device):
  step              one resident run (Batch.run);
  step_export       the run plus Batch.export of every call into a [calls, T] float32 tensor;
  step_export_f0    the same plus Batch.f0 (K12a) into a second [calls, T] tensor;
  step_f0_frames    the same plus rows_f0_frames (K12b) over the track, wl 2400 (50 ms at 48 kHz), 75 % overlap,
                    into [calls, F, 2].
The modes alternate --reps times, --steps steps each; each reports its best per-step time (host clock around the
steps, ended by a synchronise).
Kernel times: torch.profiler's CUDA activity in a profiled pass of its own (--iters export + track + labels).
Algorithmic bytes, from the shapes: K12a writes 4 B per output sample (its reads -- row and span tables, one
F0Epochs header per span, the spline pieces -- are small against that); K12b reads 4 B per sample of every segment's
range (the wl - h overlap between segments included) and writes 8 B per frame (zero tails included).  Against the
7.7 TB/s HBM3e data-sheet figure.  The card name and power limit are read in the same run.  Writes nothing but --out.
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
SEG_FRAMES = 256             # F0F_FRAMES of csrc/engine.cuh


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(',')[:2]]
        return name, power
    except Exception as e:
        return None, 'unknown (%s)' % type(e).__name__


def k12b_bytes(lens, nc, cap, wl, h):
    """Samples K12b reads (every segment's [s_first, min(s_last + wl, len))) and bytes it moves."""
    read = 0
    for ln, f, c in zip(lens.tolist(), nc.tolist(), cap.tolist()):
        m = min(f, c)
        for ka in range(0, m, SEG_FRAMES):
            kb = min(m, ka + SEG_FRAMES)
            a = int(math.floor(1 + ka * h)) - 1
            b = min(int(math.floor(1 + (kb - 1) * h)) - 1 + wl, ln)
            read += b - a
    return 4 * read + 8 * int(np.sum(cap)), read


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--batch', type=int, default=8192)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--out', default=None, help='also append the JSON line here')
    args = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    import torch
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi, workloads
    if not torch.cuda.is_available():
        sys.exit('bench_f0: no CUDA device')
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
    n, T, wl, ov = len(calls), int(lens.max()), 2400, 75
    h = wl - ov * wl / 100
    nc = np.array([L.sgb_spec_frames(int(x), wl, float(ov)) for x in lens], dtype=np.int64)
    F = int(nc.max())
    rows = np.arange(n, dtype=np.int64)
    cap_t, cap_f = np.full(n, T, dtype=np.int64), np.full(n, F, dtype=np.int64)
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        wave = torch.empty((n, T), dtype=torch.float32, device=dev)
        track = torch.empty((n, T), dtype=torch.float32, device=dev)
        labels = torch.empty((n, F, 2), dtype=torch.float32, device=dev)

    def export():
        bt.export(wave, rows * T, cap_t, stream)

    def k12a():
        bt.f0(track, rows * T, cap_t, stream)

    def k12b():
        sg.rows_f0_frames(0, track, rows * T, lens, labels, rows * F * 2, cap_f, wl, ov, stream)

    modes = {'step': [], 'step_export': [export], 'step_export_f0': [export, k12a],
             'step_f0_frames': [export, k12a, k12b]}

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

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.iters):
            export()
            k12a()
            k12b()
        stream.synchronize()
    kt = {}
    for e in prof.key_averages():
        for k in ('k_f0_epochs', 'k_f0_track', 'k_f0_frames', 'k_export_f32'):
            if e.key.startswith(k):
                kt[k] = e.device_time_total / max(1, e.count) * 1e-3
    samples = int(np.sum(cap_t))
    a_bytes = 4 * samples
    b_bytes, b_read = k12b_bytes(lens, nc, cap_f, wl, h)
    kern = {'samples_written': samples, 'voiced_fraction': None, 'k12a_bytes': a_bytes, 'k12b_bytes': b_bytes,
            'k12b_samples_read': b_read, 'kernel_ms': kt}
    for k, byts in (('k_f0_track', a_bytes), ('k_f0_frames', b_bytes), ('k_export_f32', 2 * a_bytes)):
        if kt.get(k):
            kern[k] = {'gbs': byts / (kt[k] * 1e-3) / 1e9, 'frac_of_datasheet_hbm': byts / (kt[k] * 1e-3) / 1e9 /
                       HBM_DATASHEET_GBS, 'floor_ms': byts / (HBM_DATASHEET_GBS * 1e9) * 1e3}
        else:
            kern[k] = 'the profiler listed no launch: kernel time not measured'
    torch.cuda.synchronize()
    kern['voiced_fraction'] = float((track != 0).sum().item()) / float(lens.sum())
    # a guard that the timed calls compute labels: row 0's labels against its track
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from f0_ref import frame_labels
    ref = frame_labels(track[0].cpu().numpy(), int(lens[0]), wl, ov, F)
    kern['check_row0_labels_equal'] = bool(np.array_equal(ref.view(np.int32), labels[0].cpu().numpy().view(np.int32)))
    bt.close()
    line = {'config': workloads.NAMES[3], 'calls': n, 'steps': args.steps, 'reps': args.reps,
            'gpu': name or torch.cuda.get_device_name(dev), 'power_limit': power, 'wl': wl, 'overlap': ov,
            'T': T, 'frames_per_call_max': F, 'ms_per_step': best,
            'added_ms': {'export': best['step_export'] - best['step'],
                         'f0_track': best['step_export_f0'] - best['step_export'],
                         'f0_frames': best['step_f0_frames'] - best['step_export_f0']},
            'kernels': kern, 'hbm_datasheet_gbs': HBM_DATASHEET_GBS}
    js = json.dumps(line)
    print(js, flush=True)
    if args.out:
        with open(args.out, 'a') as f:
            f.write(js + '\n')


if __name__ == '__main__':
    main()
