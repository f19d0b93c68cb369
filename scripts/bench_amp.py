"""The amplitude kernel K3 (`k_amp`) in the resident step: its stage time and the step time on cfg3 (8192 calls, the
seed bench.py uses) and cfg4 (8192 preset calls), the bytes K3 must write and the share of HBM bandwidth that is, and
the checksums of the tables K3 writes and of what is computed from them.

    python scripts/bench_amp.py [--parent DIR] [--reps 3] [--out FILE]

--parent DIR: a built copy of another revision of this tree.  Each repetition then runs this tree and DIR one after the
other, each in a process of its own (both import the package `soundgen_beta_b200`), so that the two builds are
compared in turns on the same GPU.  Timing as in bench.py: the batch is uploaded once, two runs warm up, then the
library's CUDA-event stage timers (sgb_run_info.ms) are averaged over the timed runs.  K3 writes its tables once per
run and reads almost nothing, so the least time it can take is the bytes it writes over the HBM bandwidth: the FP64
matrix (8 B per element) and the FP32 table (8 B per element, {Y, dY}, for epochs of the tensor-core synthesis kernel;
16 B, {Y, Y, dY, dY}, for the others).  Needs a GPU; it writes nothing but --out.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBM_GBS = 7700.0          # NVIDIA's data-sheet HBM3e bandwidth of one B200
CHECK_SLOTS = {3: 'amp32', 4: 'amp64', 5: 'wave', 8: 'out'}


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(',')[:2]]
        return name, power
    except Exception as e:      # noqa: BLE001 - reported in the output
        return 'unknown', 'unknown (%s)' % type(e).__name__


def worker(tree, steps3, steps4):
    sys.path.insert(0, tree)
    import numpy as np
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi, sharding, workloads
    L = _abi.load()
    if not hasattr(workloads, 'amp_paths'):     # an older tree: this tree's workload module, on the tree's package
        import importlib.util
        spec = importlib.util.spec_from_file_location('soundgen_beta_b200.workloads_amp',
                                                      os.path.join(ROOT, 'soundgen_beta_b200', 'workloads.py'))
        workloads = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(workloads)

    def batch(calls, min_rows=-1):
        assert L.sgb_synth_min_rows_set(min_rows) == 0
        bb = sg.BatchBuilder(u_dtype=np.float32)
        for kw in calls:
            bb.add_soundgen(**kw)
        bt = sg.Batch()
        bt.upload(bb.build())
        return bt

    def checksums(bt):
        cs = np.zeros(9, dtype=np.uint64)
        assert L.sgb_batch_checksums(bt.h, cs.ctypes.data, 9) == 0
        return {nm: '%016x' % int(cs[k]) for k, nm in CHECK_SLOTS.items()}

    def k3_bytes(bt):
        """Bytes K3 writes, from the epoch shapes of the last run."""
        if not hasattr(L, 'sgb_batch_amp_tables'):
            return None
        total = 0
        shape = np.zeros(3, dtype=np.int32)
        for s in range(bt.desc.n_syllables):
            a = bt.artefacts(s)
            if a['status'] != 0 or a['nGC'] == 0:
                continue
            for e in range(a['nEpochs']):
                assert L.sgb_batch_amp_tables(bt.h, s, e, None, None, 0, shape.ctypes.data) == 0
                rows, cols, pairs = (int(v) for v in shape)
                total += 8 * rows * cols + (8 if pairs else 16) * rows * (cols - 1)
        return total

    res = {'tree': tree, 'timed': {}, 'checksums': {}}
    for cfg, steps in ((3, steps3), (4, steps4)):
        calls = workloads.CONFIGS[cfg](n=8192, seed=sharding.shard_seed(cfg, 0))
        bt = batch(calls)
        for _ in range(2):
            bt.run()
        ms = np.zeros(len(_abi.T_NAMES))
        per_step = []
        for _ in range(steps):
            info = bt.run()
            ms += np.array(list(info.ms))
            per_step.append(float(info.ms[_abi.T_NAMES.index('ampl')]))
        ms /= steps
        stage = {nm: round(float(v), 4) for nm, v in zip(_abi.T_NAMES, ms)}
        srs = np.array([float(kw.get('samplingRate', 16000)) for kw in calls])
        audio_s = float(np.sum(bt.lengths() / srs))
        r = {'steps': steps, 'ampl_ms': stage['ampl'], 'ampl_ms_min': min(per_step), 'ampl_ms_max': max(per_step),
             'total_ms': stage['total'], 'audio_s_per_s': audio_s / (stage['total'] * 1e-3),
             'failed_calls': int(np.sum(bt.status() != 0)), 'stage_ms': stage}
        nb = k3_bytes(bt)
        if nb is not None:
            gbs = nb / (stage['ampl'] * 1e-3) / 1e9
            r.update(k3_bytes_written=nb, k3_GBps=round(gbs, 1), k3_share_of_hbm=round(gbs / HBM_GBS, 3),
                     k3_write_floor_ms=round(nb / (HBM_GBS * 1e9) * 1e3, 3))
        res['timed']['cfg%d' % cfg] = r
        res['checksums']['cfg%d' % cfg] = checksums(bt)
        if cfg == 3:
            bt.close()
            bt = batch(calls, min_rows=1 << 30)      # as SGB_SYNTH=ffma: every epoch on the FP32-pipe kernel
            bt.run()
            res['checksums']['cfg3_ffma'] = checksums(bt)
        bt.close()
    for name, calls in (('cfg1', workloads.config1(n=1024)), ('cfg2', workloads.config2(n=4096)),
                        ('amp_paths', workloads.amp_paths())):
        bt = batch(calls)
        bt.run()
        res['checksums'][name] = checksums(bt)
        bt.close()
    L.sgb_synth_min_rows_set(-1)
    print('RESULT ' + json.dumps(res), flush=True)


def dumps_identical(trees):
    """Runs each tree's bench.py with --dump-outputs into a temporary directory and compares the files byte for
    byte."""
    import filecmp
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        dirs = []
        for label, tree in trees:
            d = os.path.join(tmp, label)
            subprocess.run([sys.executable, 'bench.py', '--gpus', '1', '--steps', '2', '--warmup', '1',
                            '--no-cpu-baseline', '--no-parity', '--dump-outputs', d], cwd=tree, check=True,
                           capture_output=True)
            dirs.append(d)
        names = [sorted(os.listdir(d)) for d in dirs]
        if not names[0] or any(n != names[0] for n in names):
            return False
        return all(filecmp.cmp(os.path.join(dirs[0], f), os.path.join(d, f), shallow=False)
                   for f in names[0] for d in dirs[1:])


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--parent', default=None, help='a built copy of another revision, run in turns with this tree')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--steps3', type=int, default=80, help='timed cfg3 runs (about 45 ms each)')
    ap.add_argument('--steps4', type=int, default=30, help='timed cfg4 runs')
    ap.add_argument('--out', default=None, help='also write the report here')
    ap.add_argument('--worker', default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        worker(args.worker, args.steps3, args.steps4)
        return
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    name, power = gpu_info()
    trees = [('this', ROOT)] + ([('parent', os.path.abspath(args.parent))] if args.parent else [])
    lines = ['GPU: %s, power limit %s' % (name, power)]
    print(lines[0], flush=True)
    runs = {label: [] for label, _ in trees}
    for rep in range(args.reps):
        for label, tree in trees:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), '--worker', tree, '--steps3',
                                str(args.steps3), '--steps4', str(args.steps4)], capture_output=True, text=True)
            res = [json.loads(ln[7:]) for ln in p.stdout.splitlines() if ln.startswith('RESULT ')]
            if p.returncode != 0 or not res:
                sys.exit('bench_amp: %s failed:\n%s\n%s' % (tree, p.stdout[-3000:], p.stderr[-3000:]))
            res = res[0]
            runs[label].append(res)
            for cfg, r in res['timed'].items():
                ln = '%-6s rep %d %s: ampl %.3f ms (per run %.3f-%.3f), step %.2f ms, %.0f audio-s/s, failed %d' % (
                    label, rep, cfg, r['ampl_ms'], r['ampl_ms_min'], r['ampl_ms_max'], r['total_ms'],
                    r['audio_s_per_s'], r['failed_calls'])
                if 'k3_bytes_written' in r:
                    ln += '; K3 writes %.2f GB: %.0f GB/s = %.3f of %.0f GB/s (write floor %.2f ms)' % (
                        r['k3_bytes_written'] / 1e9, r['k3_GBps'], r['k3_share_of_hbm'], HBM_GBS,
                        r['k3_write_floor_ms'])
                lines.append(ln)
                print(ln, flush=True)
            lines.append('%-6s rep %d stage_ms: %s' % (label, rep, json.dumps(
                {c: r['stage_ms'] for c, r in res['timed'].items()})))
    lines.append('checksums (slots 3 amp32, 4 amp64, 5 wave, 8 out):')
    for label, _ in trees:
        for wl, cs in runs[label][0]['checksums'].items():
            lines.append('  %-6s %-10s %s' % (label, wl, ' '.join('%s=%s' % kv for kv in cs.items())))
    same_runs = all(r['checksums'] == runs[label][0]['checksums'] for label, _ in trees for r in runs[label])
    lines.append('checksums equal over the repetitions: %s' % same_runs)
    if args.parent:
        lines.append('checksums equal to the parent: %s' % (runs['this'][0]['checksums'] ==
                                                           runs['parent'][0]['checksums']))
        lines.append('bench.py --dump-outputs (cfg3) byte-identical to the parent: %s' % dumps_identical(trees))
    for cfg in ('cfg3', 'cfg4'):
        for key in ('ampl_ms', 'total_ms'):
            lines.append('%s %s: ' % (cfg, key) + ', '.join(
                '%s %s' % (label, ' '.join('%.3f' % r['timed'][cfg][key] for r in runs[label])) for label, _ in trees))
            if args.parent:
                med = {label: sorted(r['timed'][cfg][key] for r in runs[label])[len(runs[label]) // 2]
                       for label, _ in trees}
                lines.append('  median this / parent %.3f, parent - this %.3f ms' % (
                    med['this'] / med['parent'], med['parent'] - med['this']))
    for ln in lines[-(13 if args.parent else 5):]:
        print(ln, flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
