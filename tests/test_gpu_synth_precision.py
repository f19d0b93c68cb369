"""K1 against its float64 error bound, sample by sample (tests/synth_bound.py), on a B200: every corpus case under
every K1 dispatch (tensor cores only, FP32 pipe only, the default split) and with k_synth's per-lane Reinsch form
forced on every warp (SGB_SYNTH_MODE=0, read once per process: run in a child process)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import soundgen_beta_b200 as sg
import synth_bound as sb

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DISPATCH = {'tc': 0, 'ffma': 1 << 30, 'default': -1}


def _device_run(rows):
    from soundgen_beta_b200 import _abi
    L = _abi.load()
    out = {}
    try:
        assert L.sgb_synth_min_rows_set(rows) == 0
        for n in sb.CASE_NAMES:
            pitch, z, anchors, pars = sb.case_inputs(n)
            y, a = sg.generateHarmonics(pitch, z=z, amplAnchors=anchors, want_artefacts=True, **pars)
            out[n] = (np.asarray(y, dtype=np.float64), a)
    finally:
        L.sgb_synth_min_rows_set(-1)
    return out


def _sample_map(art, pars):
    """Output sample -> (epoch, sample of that epoch) of the epoch with the largest weight there."""
    sr = pars['samplingRate']
    E = len(art.epoch_waves)
    share = [sb.join([np.full(w.size, float(f == e)) for f, w in enumerate(art.epoch_waves)], art.zc, sr)
             for e in range(E)]
    idx = [sb.join([np.arange(w.size, dtype=np.float64) * (f == e) for f, w in enumerate(art.epoch_waves)],
                   art.zc, sr) for e in range(E)]
    ep = np.argmax(np.stack(share), axis=0)
    k = np.array([idx[e][i] / share[e][i] if share[e][i] > 0 else -1 for i, e in enumerate(ep)])
    return ep, np.rint(k).astype(int)


def _check(n, label, y, a, rows, force_mode, worst):
    ref, art = sb.oracle_case(n)
    pars = sb.case_inputs(n)[3]
    assert y.size == ref.size, (n, label)
    assert np.array_equal(a['gc_upsampled'], art.gc_upsampled) and np.array_equal(a['epochs'], art.epochs), (n, label)
    assert [tuple(int(v or 0) for v in zz) for zz in art.zc] == [tuple(r) for r in a['zc'].tolist()], (n, label)
    eps = sb.epochs_of(art)
    kernels = [sb.kernel_of(ep, rows) for ep in eps]
    B, _ = sb.output_bound(n, kernels, force_mode)
    err = np.abs(y - ref)
    emap, kmap = _sample_map(art, pars)
    # the path of every output sample: kernel, and for k_synth the warp's mode (or the fix-up of a straddling pair)
    path = []
    for e, ep in enumerate(eps):
        if kernels[e] == 'tc':
            path.append(np.array(['tc'] * ep.Ne, dtype=object))
            continue
        p = np.empty(ep.Ne, dtype=object)
        for w in sb.synth_warps(ep):
            m = w['mode'] if force_mode is None else force_mode
            p[w['kw']:w['kw'] + w['n']] = 'ffma mode %d%s' % (m, '' if force_mode is None else ' (forced)')
            p[w['straddle']] = 'ffma straddle fix-up'
        path.append(p)
    bad = np.nonzero(err > B)[0]
    if bad.size:
        i = int(bad[np.argmax(err[bad] / np.maximum(B[bad], 1e-300))])
        raise AssertionError('%s [%s]: %d samples over the bound; worst: output sample %d = epoch %d sample %d, '
                             'path %s, |err| %.3e > B %.3e' % (n, label, bad.size, i, emap[i], kmap[i],
                                                               path[emap[i]][kmap[i]], err[i], B[i]))
    ok = B > 0
    r = np.where(ok, err / np.where(ok, B, 1.0), 0.0)
    keys = np.array([path[e][k] for e, k in zip(emap, kmap)], dtype=object)
    for key in set(keys):
        rk = float(np.max(r[keys == key]))
        if rk >= worst.get(key, (0.0,))[0]:
            worst[key] = (rk, n, label)


def test_k1_within_float64_bound(tmp_path):
    worst = {}
    for label, rows in DISPATCH.items():
        for n, (y, a) in _device_run(rows).items():
            _check(n, label, y, a, rows, None, worst)
    # k_synth with its per-lane Reinsch form on every warp: SGB_SYNTH_MODE is read once per process
    out = tmp_path / 'mode0.npz'
    code = ('import sys, numpy as np; sys.path[:0] = [%r, %r]\n'
            'import test_gpu_synth_precision as t\n'
            'res = t._device_run(1 << 30)\n'
            'd = {}\n'
            'for n, (y, a) in res.items():\n'
            '    d[n] = y; d[n + "/gc_upsampled"] = a["gc_upsampled"]; d[n + "/epochs"] = a["epochs"]; d[n + "/zc"] = a["zc"]\n'
            'np.savez(%r, **d)\n') % (ROOT, os.path.join(ROOT, 'tests'), str(out))
    env = dict(os.environ, SGB_SYNTH_MODE='0')
    p = subprocess.run([sys.executable, '-c', code], env=env, cwd=ROOT, timeout=900, capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    ys = np.load(out)
    for n in sb.CASE_NAMES:
        a = {k: ys[n + '/' + k] for k in ('gc_upsampled', 'epochs', 'zc')}
        _check(n, 'ffma, SGB_SYNTH_MODE=0', ys[n], a, 1 << 30, 0, worst)
    print('\nK1 worst |err| / B per path:')
    for k in sorted(worst):
        print('  %-32s %.4f  (%s, %s)' % (k, *worst[k]))
