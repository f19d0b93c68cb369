"""The tensor-core synthesis kernel K1 (`k_synth_tc`) in the resident step: `stage_ms` (synth and the rest) and the
step time on cfg3 (8192 calls, the seed bench.py uses), cfg1 (1024), cfg2 (4096) and cfg4 (8192 preset calls), and
the work K1 skips above each unit's live top row, counted on the CPU.

    python scripts/bench_synth_tc.py [--parent DIR] [--reps 3] [--out FILE]

--parent DIR: a built copy of another revision of this tree.  Each repetition then runs this tree and DIR one after the
other, each in a process of its own, so that the two builds are compared in turns on the same GPU.  Timing as in
bench.py: the batch is uploaded once, two runs warm up, then the library's CUDA-event stage timers (sgb_run_info.ms)
are averaged over the timed runs.  With --parent it also checks that both builds compute the same samples: each
tree's `bench.py --dump-outputs` for configs 3, 1, 2 and 4 (cfg4 at 8192 calls), compared with np.array_equal, and
`workloads.amp_paths()` and the corpus of tests/synth_bound.py with every epoch on `k_synth_tc`.  The cfg3 bench.py
run also gives each tree's `value` (audio-s/s).

The CPU count takes 10 cfg3 calls of the same batch through the oracle and weights every unit (one glottal cycle of
one epoch) by its samples.  A unit's live top is its highest row with Y != 0 or dY != 0.  "now" is what the parent
kernel synthesises per super-pass of 1152 rows (blocks of 16 rows padded to a multiple of 8); "live" stops at the live
top: block pairs up to the top pair, passes of 24 blocks up to the top block (padded to 8).  Needs a GPU except with
--count-only; it writes nothing but --out.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_amp import gpu_info  # noqa: E402

SIZES = {3: 8192, 1: 1024, 2: 4096, 4: 8192}
TC_KR, TC_PASS_BLOCKS, TC_MAX_ROWS = 16, 24, 1152


def worker(tree, steps, dump):
    sys.path.insert(0, tree)
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi, sharding, workloads
    L = _abi.load()
    res = {'tree': tree, 'timed': {}}
    for cfg, n in SIZES.items():
        calls = workloads.CONFIGS[cfg](n=n, seed=sharding.shard_seed(cfg, 0))
        bb = sg.BatchBuilder(u_dtype=np.float32)
        for kw in calls:
            bb.add_soundgen(**kw)
        bt = sg.Batch()
        bt.upload(bb.build())
        for _ in range(2):
            bt.run()
        ms = np.zeros(len(_abi.T_NAMES))
        per = []
        for _ in range(steps[cfg]):
            info = bt.run()
            ms += np.array(list(info.ms))
            per.append(float(info.ms[_abi.T_NAMES.index('synth')]))
        ms /= steps[cfg]
        stage = {nm: round(float(v), 4) for nm, v in zip(_abi.T_NAMES, ms)}
        srs = np.array([float(kw.get('samplingRate', 16000)) for kw in calls])
        res['timed']['cfg%d' % cfg] = {
            'steps': steps[cfg], 'synth_ms': stage['synth'], 'synth_ms_min': min(per), 'synth_ms_max': max(per),
            'total_ms': stage['total'], 'audio_s_per_s': float(np.sum(bt.lengths() / srs)) / (stage['total'] * 1e-3),
            'failed_calls': int(np.sum(bt.status() != 0)), 'stage_ms': stage}
        bt.close()
    # every epoch on k_synth_tc: the K3 path workload and the float64-bound corpus
    sys.path.insert(1, os.path.join(ROOT, 'tests'))
    import synth_bound as sb
    out = {}
    assert L.sgb_synth_min_rows_set(0) == 0
    try:
        bb = sg.BatchBuilder(u_dtype=np.float32)
        for kw in workloads.amp_paths():
            bb.add_soundgen(**kw)
        bt = sg.Batch()
        bt.upload(bb.build())
        bt.run()
        lens = bt.lengths()
        y = np.zeros(int(lens.sum()), dtype=np.float32)
        bt.fetch(np.float32, out=y)
        out['amp_paths/lengths'] = lens
        out['amp_paths/status'] = bt.status()
        out['amp_paths/samples'] = y
        bt.close()
        for nm in sb.CASE_NAMES:
            pitch, z, anchors, pars = sb.case_inputs(nm)
            out['corpus/' + nm] = np.asarray(sg.generateHarmonics(pitch, z=z, amplAnchors=anchors, **pars))
    finally:
        L.sgb_synth_min_rows_set(-1)
    np.savez(dump, **out)
    print('RESULT ' + json.dumps(res), flush=True)


def bench_dump(tree, cfg, d):
    """bench.py of `tree` with --dump-outputs d; returns its JSON result line."""
    args = ['--config', str(cfg), '--no-cpu-baseline', '--no-parity', '--dump-outputs', d]
    args += ['--steps', '20', '--warmup', '3'] if cfg == 3 else ['--steps', '2', '--warmup', '1']
    if cfg == 4:
        args += ['--batch', str(SIZES[4])]
    p = subprocess.run([sys.executable, 'bench.py', '--gpus', '1'] + args, cwd=tree, capture_output=True, text=True)
    if p.returncode != 0:
        sys.exit('bench.py failed in %s:\n%s' % (tree, p.stderr[-3000:]))
    return json.loads([ln for ln in p.stdout.splitlines() if ln.startswith('{')][-1])


def same_arrays(files):
    a, b = (dict(np.load(f)) if f.endswith('.npz') else {'': np.load(f)} for f in files)
    return sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)


def count_live(ncalls=10):
    """Block pairs and passes per sample, now and stopping at the live top, over `ncalls` cfg3 calls."""
    sys.path.insert(0, ROOT)
    from oracle import soundgen_oracle as so
    from oracle.soundgen_call import soundgen as osg
    from soundgen_beta_b200 import sharding, workloads
    calls = workloads.config3(n=SIZES[3], seed=sharding.shard_seed(3, 0))
    pick = np.sort(np.random.default_rng(7).choice(len(calls), ncalls, replace=False))
    c = dict(pairs_now=0, pairs_live=0, passes_now=0, passes_live=0, units=0, units_dead=0)
    for ci in pick:
        kw = dict(calls[ci])
        z = kw.pop('z')
        _, arts, _ = osg(rng=so.RStream(z=np.concatenate(z)), want_artefacts=True, **kw)
        for a in arts:
            gu = np.asarray(a.gc_upsampled)
            for e, (st, en) in enumerate(np.asarray(a.epochs).reshape(-1, 2)):
                ref, names = a.mats[e]
                n = int(a.nSubharm[st - 1]) if a.nSubharm is not None else 0
                J = a.rows_kept * (n + 1) + n if n > 0 else a.rows_kept
                if J < 224:                  # the FP32-pipe kernel's epoch
                    continue
                M = np.zeros((J + 1, np.shape(ref)[1]))          # dense rows j = 0 (zero) .. J
                M[np.rint(np.asarray(names) * (n + 1)).astype(int)] = np.asarray(ref)
                for i, L in enumerate(np.diff(gu[st - 1:en + 1])):
                    if i + 1 >= M.shape[1] or L <= 0:
                        continue
                    nz = np.nonzero((M[:, i] != 0) | (M[:, i + 1] != 0))[0]
                    top = int(nz.max()) if nz.size else -1
                    c['units'] += 1
                    c['units_dead'] += top < 0
                    for row0 in range(0, J + 1, TC_MAX_ROWS):
                        here = min(J + 1 - row0, TC_MAX_ROWS)
                        b_now = (-(-here // TC_KR) + 7) & ~7
                        lb = max(0, min(top - row0 + 1, here) + TC_KR - 1) // TC_KR if top >= row0 else 0
                        c['pairs_now'] += L * (b_now // 2)
                        c['passes_now'] += L * -(-b_now // TC_PASS_BLOCKS)
                        c['pairs_live'] += L * -(-lb // 2)
                        c['passes_live'] += L * -(-((lb + 7) & ~7) // TC_PASS_BLOCKS)
    return ('CPU count, %d cfg3 calls of the timed batch (%d units, %d without a live row), sample-weighted: '
            'block pairs live/now %.3f (%d / %d), passes live/now %.3f (%d / %d)' % (
                ncalls, c['units'], c['units_dead'], c['pairs_live'] / c['pairs_now'], c['pairs_live'],
                c['pairs_now'], c['passes_live'] / c['passes_now'], c['passes_live'], c['passes_now']))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--parent', default=None, help='a built copy of another revision, run in turns with this tree')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--steps3', type=int, default=60, help='timed cfg3 runs (about 40 ms each)')
    ap.add_argument('--steps', type=int, default=20, help='timed runs of cfg1, cfg2 and cfg4')
    ap.add_argument('--count-only', action='store_true', help='only the CPU count (no GPU)')
    ap.add_argument('--out', default=None, help='also write the report here')
    ap.add_argument('--worker', default=None, help=argparse.SUPPRESS)
    ap.add_argument('--dump', default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    steps = {3: args.steps3, 1: args.steps, 2: args.steps, 4: args.steps}
    if args.worker:
        worker(args.worker, steps, args.dump)
        return
    if args.count_only:
        print(count_live())
        return
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    name, power = gpu_info()
    trees = [('this', ROOT)] + ([('parent', os.path.abspath(args.parent))] if args.parent else [])
    lines = ['GPU: %s, power limit %s' % (name, power)]
    print(lines[0], flush=True)
    runs = {label: [] for label, _ in trees}
    with tempfile.TemporaryDirectory() as tmp:
        for rep in range(args.reps):
            for label, tree in trees:
                dump = os.path.join(tmp, '%s_tc.npz' % label)
                p = subprocess.run([sys.executable, os.path.abspath(__file__), '--worker', tree, '--dump', dump,
                                    '--steps3', str(args.steps3), '--steps', str(args.steps)],
                                   capture_output=True, text=True)
                res = [json.loads(ln[7:]) for ln in p.stdout.splitlines() if ln.startswith('RESULT ')]
                if p.returncode != 0 or not res:
                    sys.exit('bench_synth_tc: %s failed:\n%s\n%s' % (tree, p.stdout[-3000:], p.stderr[-3000:]))
                runs[label].append(res[0])
                for cfg, r in res[0]['timed'].items():
                    ln = '%-6s rep %d %s: synth %.3f ms (per run %.3f-%.3f), step %.2f ms, %.0f audio-s/s, failed %d' % (
                        label, rep, cfg, r['synth_ms'], r['synth_ms_min'], r['synth_ms_max'], r['total_ms'],
                        r['audio_s_per_s'], r['failed_calls'])
                    lines.append(ln)
                    print(ln, flush=True)
                lines.append('%-6s rep %d stage_ms: %s' % (label, rep, json.dumps(
                    {c: r['stage_ms'] for c, r in res[0]['timed'].items()})))
        if args.parent:
            lines.append('every epoch on k_synth_tc (amp_paths, synth_bound corpus) equal to the parent: %s' % same_arrays(
                [os.path.join(tmp, 'this_tc.npz'), os.path.join(tmp, 'parent_tc.npz')]))
            for cfg in SIZES:
                val = {}
                for label, tree in trees:
                    val[label] = bench_dump(tree, cfg, os.path.join(tmp, '%s_cfg%d' % (label, cfg)))['value']
                eq = {f: same_arrays([os.path.join(tmp, '%s_cfg%d' % (label, cfg), f) for label, _ in trees])
                      for f in ('lengths.npy', 'status.npy', 'sample_waveforms.npy')}
                lines.append('bench.py --config %d --dump-outputs: np.array_equal to the parent %s; value this %.0f, '
                             'parent %.0f audio-s/s' % (cfg, eq, val['this'], val['parent']))
                print(lines[-1], flush=True)
    for cfg in ('cfg%d' % c for c in SIZES):
        for key in ('synth_ms', 'total_ms'):
            lines.append('%s %s: ' % (cfg, key) + ', '.join(
                '%s %s' % (label, ' '.join('%.3f' % r['timed'][cfg][key] for r in runs[label])) for label, _ in trees))
            if args.parent:
                med = {label: sorted(r['timed'][cfg][key] for r in runs[label])[len(runs[label]) // 2]
                       for label, _ in trees}
                lines.append('  median this / parent %.3f, parent - this %.3f ms' % (
                    med['this'] / med['parent'], med['parent'] - med['this']))
    lines.append(count_live())
    for ln in lines[-(26 if args.parent else 9):]:
        print(ln, flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
