"""Device output against the host fetch: one rank per GPU (torchrun, like bench.py), one JSON line from rank 0.

    python scripts/bench_device_out.py [--config 3|4] [--steps 5] [--warmup 2] [--reps 3] [--pipeline 8] [--out FILE]
    torchrun --nproc_per_node 8 scripts/bench_device_out.py --config 4

Measured in the same process, on the same prebuilt batch descriptions:
  value          the resident step (inputs uploaded once, outputs left on the device), as bench.py's `value`;
  host_pcm16     PipelinedBatches with the host PCM16 fetch (bench.py's `e2e_prebuilt`);
  device_f32     the same pipeline with device_out=dict(dtype=torch.float32): every sub-batch exported into a
                 [calls, T] CUDA tensor on its consumer stream instead of crossing PCIe;
  device_pcm16   the same with dtype=torch.int16.
The three pipelines run in turn, `--reps` times, alternating; each reports its best and median.  A pipeline step
ends when every consumer stream has the rows (the timer stops after a synchronise of those streams).
export_kernel: sgb_batch_export of the whole resident batch into one tensor (rows packed back to back), timed with
CUDA events on the caller's stream over `--export-iters` exports (row table upload and the two stream hand-offs
included), and the kernel alone (k_export_f32 / k_pcm16) from torch.profiler's CUDA activity.  GB/s = algorithmic
bytes (every sample read once and written once, from the lengths) over that time, against the 7.7 TB/s HBM3e
data-sheet figure of one B200.  The card name and power limit are read in the same run.  Writes nothing but `--out`.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HBM_DATASHEET_GBS = 7700.0


def gpu_info(local):
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', str(local)],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(',')[:2]]
        return name, power
    except Exception as e:
        return None, 'unknown (%s)' % type(e).__name__


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--config', type=int, default=3, choices=[3, 4])
    ap.add_argument('--batch', type=int, default=0, help='calls per GPU (default 8192)')
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--pipeline', type=int, default=8)
    ap.add_argument('--runners', type=int, default=0)
    ap.add_argument('--export-iters', type=int, default=20)
    ap.add_argument('--max-len', type=int, default=-1,
                    help='T of the device pipelines (-1: the longest call for cfg3, the 99th percentile of the call '
                         'lengths for cfg4, whose longest presets would make the padded tensors needlessly large)')
    ap.add_argument('--out', default=None, help='also append the JSON line here')
    args = ap.parse_args()
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.runners <= 0:
        args.runners = 4 if (os.cpu_count() or 8) // max(1, world) >= 8 else 3
    os.environ.setdefault('SGB_FRONTEND_THREADS', str(max(1, min(16, (os.cpu_count() or 16) // max(1, world)))))
    import __graft_entry__
    __graft_entry__.build()
    import torch
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi, sharding, workloads
    if not torch.cuda.is_available():
        sys.exit('bench_device_out: no CUDA device')
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    L = _abi.load()
    assert L.sgb_set_device(local) == 0
    if world > 1:
        sharding.bind_to_gpu_numa(L, local)
    dev = torch.device('cuda', local)

    def barrier():
        if dist is not None:
            dist.barrier()

    n = args.batch or 8192     # cfg4: bench.py's 65 536-call sweep is 8192 per GPU on 8 GPUs; the three pipelines'
                               # handles of a whole sweep on one GPU do not fit in its memory
    calls = workloads.CONFIGS[args.config](n=n, seed=sharding.shard_seed(args.config, rank))
    srs = np.array([float(kw.get('samplingRate', 16000)) for kw in calls])

    def desc_of(some):
        bb = sg.BatchBuilder(u_dtype=np.float32)
        for kw in some:
            bb.add_soundgen(**kw)
        d = bb.build()
        sg.pin_desc(d)
        return d, bb

    # ---- resident step ----
    desc, bb = desc_of(calls)
    bt = sg.Batch()
    bt.upload(desc)
    for _ in range(max(1, args.warmup)):
        bt.run()
    barrier()
    ms = 0.0
    for _ in range(args.steps):
        ms += bt.run().ms[_abi.T_NAMES.index('total')]
    lens = bt.lengths()
    audio_s = float(np.sum(lens / srs))

    # ---- the export kernel on the resident batch ----
    rows, cap = (np.cumsum(lens) - lens).astype(np.int64), lens.astype(np.int64)    # packed rows: a pure copy
    total = int(lens.sum())
    s = torch.cuda.Stream(dev)
    kern = {}
    for fmt, dt, kname in (('f32', torch.float32, 'k_export_f32'), ('pcm16', torch.int16, 'k_pcm16')):
        with torch.cuda.stream(s):
            dst = torch.empty(max(total, 1), dtype=dt, device=dev)
        for _ in range(3):
            bt.export(dst, rows, cap, s, fmt)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(args.export_iters):
            bt.export(dst, rows, cap, s, fmt)
        e1.record(s)
        e1.synchronize()
        ev_ms = e0.elapsed_time(e1) / args.export_iters
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                bt.export(dst, rows, cap, s, fmt)
            s.synchronize()
        kt = [e.device_time_total / max(1, e.count) for e in prof.key_averages() if e.key.startswith(kname)]
        k_ms = kt[0] * 1e-3 if kt else None
        esz = 4 if fmt == 'f32' else 2
        algo = (4 + esz) * total                         # every sample read once and written once
        kern[fmt] = {'kernel': kname, 'bytes_per_export': algo, 'samples': total,
                     'event_ms': ev_ms, 'event_gbs': algo / (ev_ms * 1e-3) / 1e9,
                     'kernel_ms': k_ms, 'kernel_gbs': (algo / (k_ms * 1e-3) / 1e9) if k_ms else None,
                     'frac_of_datasheet_hbm': (algo / (k_ms * 1e-3) / 1e9 / HBM_DATASHEET_GBS) if k_ms else None}
        if k_ms is None:
            kern[fmt]['kernel_note'] = 'the profiler listed no %s launch: kernel time not measured' % kname
        del dst
    bt.close()

    # ---- pipelines from prebuilt descriptions ----
    max_len = args.max_len if args.max_len >= 0 else (None if args.config == 3 else int(np.percentile(lens, 99)))
    npipe = max(1, min(args.pipeline, n))
    subs = []
    for i in range(npipe):
        lo, hi = sharding.shard_range(n, i, npipe)
        subs.append(desc_of(calls[lo:hi])[0])
    pipes = {'host_pcm16': sg.PipelinedBatches(subs, runners=args.runners),
             'device_f32': sg.PipelinedBatches(subs, runners=args.runners,
                                               device_out=dict(dtype=torch.float32, device=local, max_len=max_len)),
             'device_pcm16': sg.PipelinedBatches(subs, runners=args.runners,
                                                 device_out=dict(dtype=torch.int16, device=local, max_len=max_len))}

    def timed(name, steps):
        p = pipes[name]
        barrier()
        t0 = time.perf_counter()
        p.run_steps(steps, dtype=np.int16)
        if p.device_out is not None:
            for st in p.streams:
                st.synchronize()
        barrier()
        return time.perf_counter() - t0

    for name in pipes:
        timed(name, 2)                 # sizes every handle's pools and allocates the outputs
    times = {name: [] for name in pipes}
    for _ in range(args.reps):
        for name in pipes:
            times[name].append(timed(name, args.steps))
    out_bytes = {name: (sum(o.nbytes for o in p.outs if o is not None) if p.device_out is None
                        else sum(w.numel() * w.element_size() for w in p.waves)) for name, p in pipes.items()}
    for p in pipes.values():
        p.close()

    # ---- over ranks: max of the times, sum of the audio ----
    keys = sorted(times)
    vec = [ms * 1e-3] + [t for k in keys for t in (min(times[k]), statistics.median(times[k]))]
    if dist is not None:
        tv = torch.tensor(vec, dtype=torch.float64, device=dev)
        av = torch.tensor([audio_s], dtype=torch.float64, device=dev)
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        dist.all_reduce(av, op=dist.ReduceOp.SUM)
        vec, audio_total = tv.tolist(), float(av[0])
    else:
        audio_total = audio_s
    if rank == 0:
        name, power = gpu_info(local)
        line = {'config': workloads.NAMES[args.config], 'n_gpus': world, 'calls_per_gpu': n, 'steps': args.steps,
                'reps': args.reps, 'pipeline': npipe, 'runners': args.runners,
                'gpu': name or torch.cuda.get_device_name(dev), 'power_limit': power, 'unit': 'audio-s/s',
                'value': audio_total * args.steps / vec[0], 'ms_per_step': vec[0] / args.steps * 1e3,
                'h2d_bytes_per_gpu_step': int(bb.h2d_bytes()), 'device_out_max_len': max_len}
        for j, k in enumerate(keys):
            best, med = vec[1 + 2 * j], vec[2 + 2 * j]
            line[k] = {'value': audio_total * args.steps / best, 'median': audio_total * args.steps / med,
                       'ms_per_step': best / args.steps * 1e3, 'out_bytes_per_gpu_step': int(out_bytes[k])}
        line['export_kernel'] = kern
        line['export_kernel']['hbm_datasheet_gbs'] = HBM_DATASHEET_GBS
        js = json.dumps(line)
        print(js, flush=True)
        if args.out:
            with open(args.out, 'a') as f:
                f.write(js + '\n')
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
