#!/usr/bin/env python
"""Benchmark of the soundgen source-filter synthesis path on B200.

  python bench.py --gpus N --steps K --warmup W [--config 3] [--batch B] [--dump-outputs DIR]
  python bench.py --impl reference ...      (the reference algorithm on the host cores)

A "step" is one pass of the whole hot path (control stage, amplitude matrices, additive
synthesis, epoch joining, envelopes, noise, fused STFT filter, mixing) over one batch of
synthetic soundgen() calls of the chosen BASELINE.json config.  `value` is audio seconds
synthesised per second with inputs resident in HBM; `e2e` includes the H2D copy of the
step's inputs from pinned host memory and the D2H read of every waveform.
One JSON line is printed by rank 0.

The inputs are seeded: the same arguments give the same calls on every run, and
`--dump-outputs DIR` writes what the last timed step returned (see `dump_outputs`), so two
builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import faulthandler
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # a benchmark run leaves the tree as it found it: no __pycache__ beside the sources

T_START = time.perf_counter()
METRIC = 'audio_seconds_synthesised_per_second'
UNIT = 'audio-s/s'


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(',')])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for i, nm in enumerate(names):
                    if r[3 + i].lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                continue
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def find_r():
    """Rscript with the reference package installed (baseline/_ref as an R library, or the site library)?
    Returns (rscript, lib) or None.  Probed at run time: the build image has no R, a GPU box may."""
    import shutil
    rs = shutil.which('Rscript')
    if not rs:
        return None
    lib = os.path.join(ROOT, 'baseline', '_ref')
    code = ('.libPaths(c("%s", .libPaths())); suppressMessages(library(soundgen)); cat(R.version.string)' % lib)
    try:
        out = subprocess.run([rs, '-e', code], capture_output=True, text=True, timeout=120)
        if out.returncode == 0 and 'R version' in out.stdout:
            return rs, lib, out.stdout.strip()
    except Exception:
        pass
    return None


def r_value(v):
    if v is None:
        return 'NA'
    if isinstance(v, str):
        return "'%s'" % v
    if isinstance(v, (tuple, list)) and len(v) == 2 and np.ndim(v[0]) == 1 and np.ndim(v[1]) == 1 and not np.isscalar(v[0]):
        return 'list(time = c(%s), value = c(%s))' % (', '.join(repr(float(x)) for x in v[0]),
                                                       ', '.join(repr(float(x)) for x in v[1]))
    if isinstance(v, (list, tuple)) and len(v) and np.ndim(v[0]) == 2:      # formants: list of (k, 4) arrays
        fs = []
        for i, f in enumerate(v):
            f = np.asarray(f, dtype=np.float64)
            cols = ['%s = c(%s)' % (nm, ', '.join(repr(float(x)) for x in f[:, j]))
                    for j, nm in enumerate(('time', 'freq', 'amp', 'width'))]
            fs.append('f%d = list(%s)' % (i + 1, ', '.join(cols)))
        return 'list(%s)' % ', '.join(fs)
    if np.ndim(v) == 1:
        return 'c(%s)' % ', '.join(repr(float(x)) for x in v)
    return repr(float(v)) if not isinstance(v, (bool, np.bool_)) else ('TRUE' if v else 'FALSE')


def r_call_string(kw):
    """The soundgen() call of one workload item as R source (the reference draws its own random numbers)."""
    kw = {k: v for k, v in kw.items() if k not in ('z', 'u', 'contour_method', 'device_pitch')}
    seed = kw.pop('seed', None)
    args = ', '.join('%s = %s' % (k, r_value(v)) for k, v in kw.items())
    return ('{set.seed(%d); ' % seed if seed is not None else '{') + 'length(soundgen(%s, play = FALSE))}' % args


def run_r_reference(rinfo, calls, cores, srs):
    """Times the reference's own soundgen() over `calls` with mclapply on `cores` cores."""
    rs, lib, version = rinfo
    import tempfile
    src = ['.libPaths(c("%s", .libPaths()))' % lib, 'suppressMessages(library(soundgen))', 'library(parallel)',
           'calls <- list(' + ',\n'.join('function() %s' % r_call_string(kw) for kw in calls) + ')',
           't0 <- proc.time()[["elapsed"]]',
           'n <- unlist(mclapply(calls, function(f) suppressWarnings(f()), mc.cores = %d))' % cores,
           'cat(proc.time()[["elapsed"]] - t0, paste(n, collapse = " "))']
    with tempfile.NamedTemporaryFile('w', suffix='.R', delete=False) as f:
        f.write('\n'.join(src))
    out = subprocess.run([rs, f.name], capture_output=True, text=True, timeout=1500)
    if out.returncode != 0:
        raise RuntimeError(out.stderr[-500:])
    tok = out.stdout.split()
    secs = float(tok[0])
    lens = np.array([float(x) for x in tok[1:]])
    return float(np.sum(lens / srs[:lens.size])) / secs, version


def oracle_arts_partials(arts):
    """(reference, dense) partial-samples of one call from the oracle's artefacts: rows the reference keeps
    per epoch (all-zero rows dropped, R/subharmonics.R:83-84) vs the dense rows_kept (n + 1) + n the device sums."""
    ref = dense = 0
    for a in arts:
        gu = a.gc_upsampled
        for e, (st, en) in enumerate(np.asarray(a.epochs).reshape(-1, 2)):
            ne = int(gu[en] - gu[st - 1] + 1)
            n = int(a.nSubharm[st - 1]) if a.nSubharm is not None else 0
            ref += ne * len(a.epoch_rows[e])
            dense += ne * (a.rows_kept * (n + 1) + n if n > 0 else a.rows_kept)
    return ref, dense


def parity_sample(calls, outs, idx):
    """Checks the calls `idx` of the timed batch against the CPU oracle: max |err| / peak, SNR in dB and the
    ratio dense / reference partial-samples (for the K1 roofline numerator)."""
    from oracle import soundgen_oracle as so
    from oracle.soundgen_call import soundgen as osg
    worst, snr_min, pref, pdense, bad_len = 0.0, float('inf'), 0, 0, 0
    for i in idx:
        kw = dict(calls[i])
        z, u = kw.pop('z', None), kw.pop('u', None)
        kw.pop('device_pitch', None)
        if 'seed' in kw:
            from oracle.rrng import RRng
            rng = RRng(kw.pop('seed'))
        else:
            rng = so.RStream(z=np.concatenate(z) if z else None, u=np.concatenate(u) if u else None)
        ref, arts, _ = osg(rng=rng, want_artefacts=True, **kw)
        y = np.asarray(outs[i], dtype=np.float64)
        if y.size != ref.size:
            bad_len += 1
            continue
        err = y - ref
        worst = max(worst, float(np.max(np.abs(err)) / np.max(np.abs(ref))))
        snr_min = min(snr_min, float(10 * np.log10(np.sum(ref ** 2) / max(np.sum(err ** 2), 1e-300))))
        a, b = oracle_arts_partials(arts)
        pref += a
        pdense += b
    return {'calls_checked': len(idx), 'length_mismatches': bad_len, 'max_err_of_peak': worst,
            'snr_db_min': snr_min, 'checker': 'numpy restatement of the R reference (parity unpinned: no R here)',
            'dense_over_reference_partials': (pdense / pref) if pref else None}


DUMP_BYTES = 64_000_000


def dump_outputs(path, out, lens, status):
    """Writes what the timed path returned in its last step as .npy files under `path`:
      lengths.npy           float64, the waveform length of every call of the batch
      status.npy            float64, the status code of every call (0 = ok)
      sample_calls.npy      float64, indices of the sampled calls, ascending
      sample_waveforms.npy  float32, the waveforms of those calls, concatenated in that order
    Every call is sampled when the files fit in DUMP_BYTES.  Otherwise the calls are visited in an order
    drawn with a fixed seed from the batch size alone, and each one is kept while its waveform still fits."""
    os.makedirs(path, exist_ok=True)
    offs = np.concatenate(([0], np.cumsum(lens)))
    budget = DUMP_BYTES - 24 * lens.size - 4 * 128     # the three float64 arrays and the four .npy headers
    pick, used = [], 0
    for i in np.random.default_rng(2026).permutation(lens.size):
        if used + 4 * int(lens[i]) <= budget:
            pick.append(int(i))
            used += 4 * int(lens[i])
    pick.sort()
    np.save(os.path.join(path, 'lengths.npy'), lens.astype(np.float64))
    np.save(os.path.join(path, 'status.npy'), status.astype(np.float64))
    np.save(os.path.join(path, 'sample_calls.npy'), np.array(pick, dtype=np.float64))
    np.save(os.path.join(path, 'sample_waveforms.npy'),
            np.concatenate([out[offs[i]:offs[i + 1]] for i in pick] + [np.zeros(0, np.float32)]).astype(np.float32))


def oracle_one(kw):
    """One soundgen() call through the CPU oracle; returns (seconds of audio, samples)."""
    from oracle import soundgen_oracle as so
    from oracle.soundgen_call import soundgen as osg
    kw = dict(kw)
    z = kw.pop('z', None)
    u = kw.pop('u', None)
    if 'seed' in kw:      # cfg0 / cfg4: R's own stream after set.seed(seed)
        from oracle.rrng import RRng
        rng = RRng(kw.pop('seed'))
    else:
        rng = so.RStream(z=np.concatenate(z) if z else None, u=np.concatenate(u) if u else None)
    y = osg(rng=rng, **kw)
    return y.size / float(kw.get('samplingRate', 16000))


def run_reference(args, rank, world):
    """The reference algorithm (CPU restatement under oracle/) on all host cores, bounded sample."""
    if rank != 0:
        return
    import multiprocessing as mp
    from soundgen_beta_b200 import workloads
    cores = os.cpu_count() or 1
    per_step = max(cores, 2 * cores if args.config in (1,) else cores)
    if args.config == 4:
        per_step = max(per_step, 33)
    calls = workloads.CONFIGS[args.config](n=per_step)
    rinfo = find_r()
    if rinfo is not None:
        try:
            srs = np.array([float(kw.get('samplingRate', 16000)) for kw in calls])
            t0 = time.perf_counter()
            vals = [run_r_reference(rinfo, calls, cores, srs) for _ in range(max(1, args.steps))]
            dt = time.perf_counter() - t0
            val = float(np.mean([v for v, _ in vals]))
            line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus,
                    'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / max(1, args.steps) * 1e3,
                    'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
                    'data': 'synthetic', 'gpu_launches': 0,
                    'config': {'workload': workloads.NAMES[args.config], 'calls_per_step': len(calls)},
                    'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'reference',
                                     'sample': '%d calls per step through the R package itself (%s), mclapply'
                                               % (len(calls), vals[0][1])},
                    'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
            print(json.dumps(line), flush=True)
            return
        except Exception as e:      # fall back to the port, saying why
            print('R reference failed (%s); timing the numpy restatement instead' % str(e)[:200], file=sys.stderr)
    with mp.Pool(cores) as pool:
        for _ in range(args.warmup):
            pool.map(oracle_one, calls[:cores])
        t0 = time.perf_counter()
        audio = 0.0
        for _ in range(args.steps):
            audio += sum(pool.map(oracle_one, calls))
        dt = time.perf_counter() - t0
    val = audio / dt
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
            'data': 'synthetic', 'gpu_launches': 0,
            'config': {'workload': workloads.NAMES[args.config], 'calls_per_step': len(calls)},
            'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                             'sample': '%d calls of %s per step (numpy restatement of the R reference; '
                                       'R itself is not installed)' % (len(calls), workloads.NAMES[args.config])},
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200')
    ap.add_argument('--config', type=int, default=3)
    ap.add_argument('--batch', type=int, default=0, help='calls per GPU per step (default: the config size)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-parity', action='store_true', help='skip the oracle check of a sample of the timed batch')
    ap.add_argument('--parity-calls', type=int, default=16)
    ap.add_argument('--pipeline', type=int, default=8,
                    help='sub-batches (handles / CUDA streams) of the end-to-end measurement')
    ap.add_argument('--fe-threads', type=int, default=3, help='host front-end threads of the from-arguments pipeline')
    ap.add_argument('--runners', type=int, default=0,
                    help='host threads that run kernels in the end-to-end pipeline (plus one uploader, one fetcher); '
                         '0 = 4 when the rank has at least 8 host cores to itself, else 3')
    ap.add_argument('--watchdog', type=int, default=1500, help='seconds after which a stuck run dumps its stacks and exits')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step (rank 0) as DIR/<name>.npy, see dump_outputs()')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU path; --impl reference has none')
    faulthandler.dump_traceback_later(args.watchdog, exit=True)   # a stuck run reports where, instead of hanging the box
    rank, world, local = env_int('RANK', 0), env_int('WORLD_SIZE', 1), env_int('LOCAL_RANK', 0)
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    if args.runners <= 0:
        args.runners = 4 if (os.cpu_count() or 8) // max(1, world) >= 8 else 3
    # worker threads of the library's host stage: the ranks of one box share its cores
    os.environ.setdefault('SGB_FRONTEND_THREADS', str(max(1, min(16, (os.cpu_count() or 16) // max(1, world)))))
    import __graft_entry__ as ge
    ge.build()
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import _abi, workloads
    L = _abi.load()
    if L.sgb_device_count() < 1:
        raise SystemExit('bench.py: no CUDA device (the product path has no CPU fallback)')
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    assert L.sgb_set_device(local) == 0
    from soundgen_beta_b200 import sharding
    numa_cpus = sharding.bind_to_gpu_numa(L, local) if world > 1 else []

    sizes = {0: 1, 1: 1024, 2: 4096, 3: 8192, 4: max(1, 65536 // world)}   # cfg4: one sweep shared by the ranks
    n = args.batch or sizes[args.config]
    gen = workloads.CONFIGS[args.config]
    from soundgen_beta_b200 import sharding
    calls = gen(n=n, seed=sharding.shard_seed(args.config, rank))
    srs = np.array([float(kw.get('samplingRate', 16000)) for kw in calls])

    def add_calls(builder, some):
        for kw in some:
            builder.add_soundgen(**kw)

    bb = sg.BatchBuilder(u_dtype=np.float32)   # uniforms travel as float32 (halves the PCIe bytes)
    t_fe = time.perf_counter()
    add_calls(bb, calls)
    desc = bb.build()
    fe_ms = (time.perf_counter() - t_fe) * 1e3
    sg.pin_desc(desc)   # page-lock the host pools
    bt = sg.Batch()
    bt.upload(desc)

    def barrier():
        if dist is not None:
            dist.barrier()

    # ---- warm-up (also sizes the device pools) ----
    info = None
    for _ in range(max(args.warmup, 1)):
        info = bt.run()
    lens = bt.lengths()
    audio_s = float(np.sum(lens / srs))
    out = np.zeros(int(lens.sum()), dtype=np.float32)
    L.sgb_pin(out.ctypes.data, out.nbytes)
    bt.fetch(np.float32, out=out)

    # ---- timed: inputs resident in HBM ----
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    barrier()
    stage_ms = np.zeros(len(_abi.T_NAMES))
    t0 = time.perf_counter()
    launches = 0
    for _ in range(args.steps):
        info = bt.run()   # ends with a stream synchronise
        stage_ms += np.array(list(info.ms))
        launches += info.kernel_launches
    barrier()
    dt_wall = time.perf_counter() - t0
    # device time of the K steps: CUDA events recorded on the launching stream around every step
    # (first launch to last kernel, host-side layout between the stages included)
    dt = float(stage_ms[_abi.T_NAMES.index('total')]) * 1e-3
    # ---- timed: end to end through the public batch API (H2D + run + D2H of every waveform) ----
    # the batch is cut into `--pipeline` sub-batches that flow through an upload / run / fetch software
    # pipeline (one uploader, `--runners` kernel threads, one fetcher), so the transfers of one
    # sub-batch overlap the kernels of others (no work is skipped)
    npipe = max(1, min(args.pipeline, len(calls)))
    subs = []
    for i in range(npipe):
        lo, hi = sharding.shard_range(len(calls), i, npipe)
        sb = sg.BatchBuilder(u_dtype=np.float32)
        add_calls(sb, calls[lo:hi])
        sd = sb.build()
        sg.pin_desc(sd)
        subs.append(sd)
    pipe = sg.PipelinedBatches(subs, runners=args.runners)

    def report_stuck():   # fires shortly before the watchdog: where is every handle waiting?
        for i, hb in enumerate([bt] + pipe.batches):
            st = np.zeros(12, dtype=np.int32)
            L.sgb_batch_debug_state(hb.h, st.ctypes.data, 12)
            print('handle %d: wait %d, stage events done %s' % (i, st[0], st[1:].tolist()), file=sys.stderr, flush=True)
    stuck = threading.Timer(max(3, args.watchdog - 8 - (time.perf_counter() - T_START)), report_stuck)
    stuck.daemon = True
    stuck.start()
    pipe.run_steps(2)    # warm-up: sizes the pools of every handle, pins the outputs
    barrier()
    t1 = time.perf_counter()
    pipe.run_steps(args.steps)
    barrier()
    dt_e2e = time.perf_counter() - t1
    d2h_f32 = sum(o.nbytes for o in pipe.outs)
    # the same end to end, fetching 16-bit PCM (what the reference's savePath branch writes): half the D2H bytes
    pipe.run_steps(1, dtype=np.int16)
    barrier()
    t2 = time.perf_counter()
    pipe.run_steps(args.steps, dtype=np.int16)
    barrier()
    dt_wav = time.perf_counter() - t2
    d2h_i16 = sum(o.nbytes for o in pipe.outs)
    pipe.close()
    # the same again, but every step starts from the ARGUMENT LISTS (one sgb_soundgen_args struct per call, the
    # form a binding such as r/src/rshim.c produces): `--fe-threads` threads run the library's host front-end
    # (validation, R's RNG stream, contour set-up, description) for a sub-batch before it is uploaded
    srcs = []
    for i in range(npipe):
        lo, hi = sharding.shard_range(len(calls), i, npipe)
        srcs.append(sg.ArgArray(calls[lo:hi], np.float32))
    pipe_a = sg.PipelinedBatches(sources=srcs, runners=args.runners, fe_threads=args.fe_threads)
    pipe_a.run_steps(2, dtype=np.int16)
    barrier()
    t3 = time.perf_counter()
    pipe_a.run_steps(args.steps, dtype=np.int16)
    barrier()
    dt_args = time.perf_counter() - t3
    h2d_args = int(sum(fe.h2d_bytes() for fe in pipe_a.fes))
    pipe_a.close()
    stuck.cancel()
    d2h_bytes = d2h_f32
    clocks = sampler.stop()
    stage_ms /= args.steps
    # ---- the waveforms of the last timed step (bt ran nothing since) ----
    if (not args.no_parity or args.dump_outputs) and rank == 0:
        bt.fetch(np.float32, out=out)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, bt.lengths(), bt.status())
    # ---- parity of the timed batch itself: a random sample of its calls against the CPU oracle ----
    parity = None
    if not args.no_parity and rank == 0:
        offs = np.concatenate(([0], np.cumsum(lens)))
        pick = np.random.default_rng(7).choice(len(calls), size=min(args.parity_calls, len(calls)), replace=False)
        outs_pick = {int(i): out[offs[i]:offs[i + 1]] for i in pick}
        parity = parity_sample(calls, outs_pick, [int(i) for i in pick])

    dt, dt_e2e, audio_total, dt_wav, dt_args = sharding.aggregate(dist, dt, dt_e2e, audio_s,
                                                                  device='cuda' if dist is not None else None,
                                                                  extra=(dt_wav, dt_args))
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    value = audio_total * args.steps / dt
    e2e_f32 = audio_total * args.steps / dt_e2e
    e2e = audio_total * args.steps / dt_wav
    # ---- roofline of the dominant kernel: K1 additive synthesis ----
    # Default build: k_synth_tc, the harmonic sum as an FP16 x FP16 -> FP32 contraction on tcgen05 (two-term
    # split of both operands, three products): bound "tensor".  SGB_SYNTH=ffma selects the round-1 FP32-pipe
    # kernel (blocked Clenshaw on FFMA2), whose roofline is the FP32 pipe.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    import ctypes
    fp32 = ctypes.c_double(0)
    L.sgb_measure_fp32_peak(ctypes.byref(fp32))
    use_tc = os.environ.get('SGB_SYNTH', 'tc') != 'ffma'
    kname = 'k_synth_tc' if use_tc else 'k_synth'
    ms_synth = float(stage_ms[_abi.T_NAMES.index('synth')])
    ms_filter = float(stage_ms[_abi.T_NAMES.index('filter')])
    ms_noise = float(stage_ms[_abi.T_NAMES.index('noise')])
    traffic, traffic_f = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')))
        key = 'cfg%d_%d' % (args.config, len(calls))
        traffic = tj.get(key, {}).get(kname, {}).get('dram_bytes_per_launch')
        traffic_f = tj.get(key, {}).get('k_stft_filter', {}).get('dram_bytes_per_launch')
    except Exception:
        pass
    # K1's algorithmic work: 6 flop per partial-sample the REFERENCE sums (rows that survive the all-zero
    # pruning of R/subharmonics.R:83-84).  The device sums dense rows (harmonics and sub-harmonics share one
    # index, dead rows included); the ratio dense / reference is measured on the parity sample of this batch.
    nominal_fp32 = 148 * 128 * 2 * 1.965e9 / 1e12          # 74.4 TFLOP/s: SMs x FP32 lanes x FMA x max clock
    ratio = (parity or {}).get('dense_over_reference_partials') or None
    roofline = None
    if ms_synth > 0 and info.synth_partials > 0:
        dense = 6.0 * info.synth_partials / (ms_synth * 1e-3) / 1e12
        ach = dense / ratio if ratio else dense
        algo = ('6 flop per partial-sample x %d dense partial-samples per launch / %s (dense / reference rows, '
                'from the parity sample)' % (info.synth_partials, ('%.3f' % ratio) if ratio else 'n/a'))
        if use_tc:
            tpeak = peaks.get('bf16_tflops_sustained', 1400.0)      # timed inside a long step: the sustained figure
            # executed on the tensor cores: {cos, sin} x {hi hi, lo hi, hi lo} x {Y, dY} = 12 MAC per dense
            # partial-sample (row padding to 128 rows and sample padding to 128 per tile not counted)
            executed = 24.0 * info.synth_partials / (ms_synth * 1e-3) / 1e12
            roofline = {'kernel': kname, 'bound': 'tensor', 'achieved': ach, 'peak': tpeak, 'unit': 'TFLOP/s',
                        'frac': ach / tpeak, 'traffic': traffic,
                        'peak_source': ('MEASURED_PEAKS.json bf16_tflops_sustained (of measured)' if 'bf16_tflops_sustained' in peaks
                                        else 'fallback 1400 TFLOP/s sustained (of fallback)'),
                        'executed_tensor_tflops': executed, 'frac_executed': executed / tpeak,
                        'fp32_pipe_peak': fp32.value, 'frac_of_fp32_pipe': ach / fp32.value if fp32.value else None,
                        'achieved_dense_rows': dense, 'dense_over_reference_partials': ratio, 'algorithmic': algo,
                        'note': 'achieved = the reference\'s 6 flop per partial-sample over the kernel time; the kernel '
                                'executes 4x that on the tensor cores (executed_tensor_tflops) and is bound by the '
                                'issue -> commit -> wait round trip of its small MMAs (about 500 cycles per 384-row '
                                'pass, profiles/r02_mma_rate_micro.txt), not by tensor throughput; frac_of_fp32_pipe '
                                '> 1 is why it left the FP32 pipe (round-1 kernel: SGB_SYNTH=ffma, 0.62 of that peak)'}
        else:
            roofline = {'kernel': kname, 'bound': 'fp32', 'achieved': ach, 'peak': fp32.value,
                        'unit': 'TFLOP/s', 'frac': ach / fp32.value if fp32.value else None, 'traffic': traffic,
                        'peak_source': 'measured in this run: sgb_measure_fp32_peak (FFMA2 dependency chains); '
                                       'MEASURED_PEAKS.json has no FP32 figure',
                        'peak_nominal': nominal_fp32, 'frac_of_nominal': ach / nominal_fp32,
                        'achieved_dense_rows': dense, 'frac_dense_rows': dense / fp32.value if fp32.value else None,
                        'dense_over_reference_partials': ratio, 'algorithmic': algo}
    hbm = peaks.get('hbm_gbs', 6650.0)
    roof_filter = None
    if ms_filter > 0 and info.filter_samples > 0:
        ach = 8.0 * info.filter_samples / (ms_filter * 1e-3) / 1e9
        roof_filter = {'kernel': 'k_stft_reg<filter>', 'bound': 'hbm', 'achieved': ach, 'peak': hbm, 'unit': 'GB/s',
                       'frac': ach / hbm, 'traffic': traffic_f,
                       'peak_source': 'MEASURED_PEAKS.json' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s',
                       'algorithmic': '8 B per output sample x %d samples per launch' % info.filter_samples,
                       # the roofline that actually binds it: shared-memory traffic of the FFT passes.  Tuned plans
                       # (800 / 1200 / 2400 / 160 points): 3 forward + 3 inverse passes with the middle two fused = 5
                       # read + write sweeps of 8 B per complex point; a complex FFT carries two real frames and the
                       # hop is a quarter window: 5 x 16 B x wl / (2 x wl / 4) = 160 B per output sample
                       'smem': {'algorithmic_bytes_per_sample': 160,
                                'achieved': 160.0 * info.filter_samples / (ms_filter * 1e-3) / 1e9,
                                'peak': 148 * 128 * 1.965, 'unit': 'GB/s',
                                'frac': 160.0 * info.filter_samples / (ms_filter * 1e-3) / 1e9 / (148 * 128 * 1.965),
                                'peak_source': 'nominal: 148 SMs x 128 B per clock x 1965 MHz'},
                       'note': 'the kernel is bound by its shared-memory FFT passes, not by HBM: see '
                               'profiles/r02_ncu_k_stft_summary.txt (shared-memory wavefronts, issue slots)'}
    if roofline is None:
        roofline = roof_filter

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        m = {0: 8, 1: 24, 2: 4, 3: 6, 4: 33}[args.config]
        sample = (calls * m)[:m]
        tc = time.perf_counter()
        a = sum(oracle_one(kw) for kw in sample)
        tc = time.perf_counter() - tc
        cpu = {'value': a / tc, 'unit': UNIT, 'cores': 1, 'kind': 'port',
               'sample': 'first %d calls of the workload, numpy restatement of the R reference '
                         '(Rscript + the soundgen package probed at run time: %s)'
                         % (len(sample), 'found, see --impl reference' if find_r() else 'not found')}
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3, 'wall_ms_per_step': dt_wall / args.steps * 1e3,
            'timing': 'cuda events on the launching stream, max over ranks', 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32 (f64 phase / control; K1 products as FP16 hi + lo pairs, FP32 accumulate)', 'data': 'synthetic',
            'config': {'workload': workloads.NAMES[args.config], 'calls_per_gpu': len(calls),
                       'audio_seconds_per_gpu_step': audio_s, 'l2': 'inputs and intermediates larger than L2',
                       'uniforms': 'float32'},
            # End to end through the public batch API with HOST buffers.  The result every step reads back is the
            # waveform of every call as the 16-bit PCM samples the reference's savePath branch writes
            # (R/soundgen.R:855-857 -> seewave::savewav), normalised and packed on the device; `e2e_f32` is the same
            # pipeline fetching FP32 samples (what soundgen() returns in memory): twice the bytes, and on an
            # 8-GPU box it runs at the bare pinned-copy ceiling of the host (profiles/r02_copy_ceiling_8gpu.json).
            'e2e': {'value': audio_total * args.steps / dt_args, 'unit': UNIT, 'h2d_bytes_per_step': h2d_args,
                    'd2h_bytes_per_step': int(d2h_i16), 'ms_per_step': dt_args / args.steps * 1e3,
                    'result_format': 'int16 PCM (savePath / WAV sample format)', 'pipeline': npipe, 'runners': args.runners,
                    'fe_threads': args.fe_threads, 'cpus_bound': len(numa_cpus),
                    'note': 'every step starts from the ARGUMENT LISTS (one sgb_soundgen_args struct per call, the form a '
                            'binding such as r/src/rshim.c produces): library front-end (validation, R RNG stream, contour '
                            'set-up, description) -> pinned H2D -> kernels -> PCM16 D2H, sub-batches pipelined'},
            'e2e_prebuilt': {'value': e2e, 'unit': UNIT, 'h2d_bytes_per_step': int(bb.h2d_bytes()),
                             'd2h_bytes_per_step': int(d2h_i16), 'ms_per_step': dt_wav / args.steps * 1e3,
                             'front_end_ms_per_step': fe_ms,
                             'note': 'the same pipeline timed from prebuilt batch descriptions (round-1 definition); '
                                     'front_end_ms_per_step = argument lists -> description on ONE thread through the Python '
                                     'mirror, per-call Python marshalling included'},
            'e2e_f32': {'value': e2e_f32, 'unit': UNIT, 'ms_per_step': dt_e2e / args.steps * 1e3,
                        'd2h_bytes_per_step': int(d2h_bytes),
                        'note': 'same pipeline, waveforms fetched as FP32 samples'},
            'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roofline,
            'roofline_filter': roof_filter, 'cpu_baseline': cpu, 'parity_sample': parity,
            'parity_sample_max_err': (parity or {}).get('max_err_of_peak'), 'snr_db': (parity or {}).get('snr_db_min'),
            'stage_ms': {nm: float(v) for nm, v in zip(_abi.T_NAMES, stage_ms)},
            'failed_calls': int(info.n_failed)}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
