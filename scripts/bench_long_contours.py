"""Resident throughput of calls with long contours (workloads.resynthesis: 101 anchors per contour, 4 formants with
101 time points) and of the same calls thinned to 60 points per contour, with the per-stage device times and the
max error against the oracle on a seeded sample of calls.  Prints one JSON line per workload.

    python scripts/bench_long_contours.py [--batch 4096] [--steps 5] [--warmup 2] [--only thinned] [--out FILE]

Timing as in bench.py: the batch is uploaded once, `--warmup` runs size the pools, then `--steps` runs are timed
with the library's stage events (sgb_run_info.ms).  Needs a GPU; it writes nothing but `--out`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(',')[:2]]
        return name, power
    except Exception as e:      # the device name still comes from the runtime below
        return None, 'unknown (%s)' % type(e).__name__


def oracle_call(kw):
    from oracle import soundgen_oracle as so
    from oracle.soundgen_call import soundgen as osg
    kw = dict(kw)
    z, u = kw.pop('z', None), kw.pop('u', None)
    rng = so.RStream(z=np.concatenate(z) if z else None, u=np.concatenate(u) if u else None)
    return osg(rng=rng, **kw)


def run(name, calls, args):
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi
    srs = np.array([float(kw['samplingRate']) for kw in calls])
    bb = sg.BatchBuilder(u_dtype=np.float32)
    for kw in calls:
        bb.add_soundgen(**kw)
    bt = sg.Batch()
    bt.upload(bb.build())
    for _ in range(max(args.warmup, 1)):
        bt.run()
    stage = np.zeros(len(_abi.T_NAMES))
    for _ in range(args.steps):
        info = bt.run()
        stage += np.array(list(info.ms))
    stage /= args.steps
    lens = bt.lengths()
    status = bt.status()
    outs = bt.fetch(np.float32)
    audio_s = float(np.sum(lens / srs))
    ms = {nm: float(v) for nm, v in zip(_abi.T_NAMES, stage)}
    sample = np.random.default_rng(7).choice(len(calls), size=min(8, len(calls)), replace=False)
    err = 0.0
    for i in sample:
        ref = oracle_call(calls[int(i)])
        y = outs[int(i)].astype(np.float64)
        assert y.size == ref.size, (name, int(i), y.size, ref.size)
        err = max(err, float(np.max(np.abs(y - ref)) / np.max(np.abs(ref))))
    bt.close()
    return {'workload': name, 'calls': len(calls), 'failed': int(np.sum(status != 0)), 'audio_s': audio_s,
            'audio_s_per_s': audio_s / (ms['total'] * 1e-3), 'total_ms': ms['total'],
            'K0_control_ms': ms['control'], 'K4_envelope_ms': ms['envelope'], 'K6_compose_ms': ms['compose'],
            'K7_mix_finalize_ms': ms['assemble'] + ms['finalize'], 'stage_ms': ms,
            'max_err_of_peak_vs_oracle': err, 'oracle_sample': sorted(int(i) for i in sample)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--batch', type=int, default=4096)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--only', choices=['long', 'thinned'], default=None)
    ap.add_argument('--out', default=None, help='also write the JSON lines here')
    args = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    import torch
    from soundgen_beta_b200 import workloads
    if not torch.cuda.is_available():
        sys.exit('bench_long_contours: no CUDA device')
    smi_name, power = gpu_info()
    gpu = {'gpu': smi_name or torch.cuda.get_device_name(0), 'power_limit': power}
    calls = workloads.resynthesis(n=args.batch)
    todo = [('long', calls), ('thinned', workloads.thinned(calls))]
    lines = []
    for name, cs in todo:
        if args.only and name != args.only:
            continue
        r = run(name, cs, args)
        r.update(gpu)
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
