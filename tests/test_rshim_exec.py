"""The R .Call shim (r/src/rshim.c) EXECUTED without R: it is compiled against a miniature functional R
runtime (tests/rstub/fake_r.c: heap SEXPs, attributes, PROTECT counter, Rf_error by longjmp) and linked to
the real libsoundgen_b200.so.  CPU part: the error paths (Rf_error before and after native resources exist,
PROTECT balance, "no device" -- there is no CPU fallback).  GPU part: all six entry points, outputs compared
with the ctypes path on the same inputs, R's .Random.seed handed in and back."""
import atexit
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUB = os.path.join(ROOT, 'tests', 'rstub')
_exe = []


def build():
    """Compile the shim driver once per process into a temporary directory (the checkout may be read-only)."""
    if not _exe:
        d = tempfile.mkdtemp(prefix='sgb_rshim_')
        atexit.register(shutil.rmtree, d, True)
        exe = os.path.join(d, 'run_shim')
        lib = os.path.join(ROOT, 'soundgen_beta_b200')
        srcs = [os.path.join(STUB, 'fake_r.c'), os.path.join(STUB, 'run_shim.c'), os.path.join(ROOT, 'r', 'src', 'rshim.c')]
        subprocess.check_call(['gcc', '-O1', '-Wall', '-Werror', '-I', STUB, '-I', os.path.join(ROOT, 'include'), '-o', exe] +
                              srcs + ['-L', lib, '-lsoundgen_b200', '-Wl,-rpath,' + lib, '-lm'])
        _exe.append(exe)
    return _exe[0]


def inputs():
    from oracle.rrng import RRng
    r = np.random.default_rng(5)
    rec = {'rolloff_pitch': [100., 150., 130.],
           'filter_sound': np.sin(np.arange(4000) * 0.05) * np.linspace(0.2, 1, 4000), 'filter_env': np.ones(400),
           'harm_pitch': np.linspace(120, 180, 1050), 'harm_z': r.standard_normal(2200),
           'noise_u': r.random(400 * 19),
           # .Random.seed after set.seed(1): kind code 403 (Mersenne-Twister + Inversion), then mti and mt[] as R
           # stores them: signed 32-bit integers
           'seed': [403] + list(np.array(RRng(1).state(), dtype=np.uint32).astype(np.int32))}
    return rec


def write(path, rec):
    with open(path, 'w') as f:
        for k, v in rec.items():
            v = np.atleast_1d(np.asarray(v, dtype=np.float64))
            f.write('%s %d %s\n' % (k, v.size, ' '.join(repr(float(x)) for x in v)))


def read(path):
    out = {}
    for line in open(path):
        tok = line.split()
        out[tok[0]] = tok[2:]
    return out


def run(mode, tmp_path, env=None):
    exe = build()
    inp, outp = str(tmp_path / 'in.txt'), str(tmp_path / 'out.txt')
    write(inp, inputs())
    r = subprocess.run([exe, mode, inp, outp], capture_output=True, text=True, timeout=600, env=env)
    return r, read(outp)


def test_shim_error_paths_without_a_device(tmp_path):
    # every device is hidden from the shim's process, so the no-device path runs on GPU machines too
    r, _ = run('cpu', tmp_path, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))
    assert r.returncode == 0, r.stdout + r.stderr
    assert 'SHIM TEST PASSED' in r.stdout
    assert 'noise_badfilter: Rf_error: filterNoise must have windowLength_points / 2 rows; protect depth 0' in r.stdout
    assert 'rolloff_nodevice: Rf_error: soundgen_b200: no CUDA device' in r.stdout
    assert 'soundgen_nodevice: Rf_error: soundgen_b200: no CUDA device' in r.stdout


@pytest.mark.gpu
def test_shim_entry_points_match_the_ctypes_path(tmp_path):
    import soundgen_beta_b200 as sg
    r, out = run('gpu', tmp_path)
    assert r.returncode == 0 and 'SHIM TEST PASSED' in r.stdout, r.stdout + r.stderr
    assert 'harmonics_fail: Rf_error: Failed to generate the new syllable!; protect depth 0' in r.stdout
    rec = inputs()
    f = lambda k: np.array(out[k], dtype=np.float64)
    # getRolloff: matrix + dim + rownames
    m = sg.getRolloff(rec['rolloff_pitch'], nHarmonics=20, rolloff=-12, rolloffOct=-2, rolloffKHz=-6, rolloffParab=0,
                      rolloffParabHarm=3)
    assert [int(x) for x in out['rolloff_dim']] == list(m.shape) and out['rolloff_lastname'] == [str(m.shape[0])]
    assert np.array_equal(f('rolloff'), m.ravel(order='F'))
    assert np.array_equal(f('filter'), sg.filter_sound(rec['filter_sound'], rec['filter_env'], 800))
    y, art = sg.generateHarmonics(rec['harm_pitch'], nonlinBalance=100, jitterDep=1.0, shimmerDep=5.0, subDep=60, subFreq=80,
                                  z=rec['harm_z'], want_artefacts=True)
    assert np.array_equal(f('harm_wave'), y) and int(out['harm_z_used'][0]) == art['z_used']
    assert np.array_equal(np.array(out['harm_gc'], dtype=np.int64), art['gc'])
    assert np.array_equal(f('noise'), sg.generateNoise(3000, ((0, 300), (-20, -10)), rolloffNoise=-6, attackLen=10,
                                                       windowLength_points=800, u=rec['noise_u']))
    env = sg.getSpectralEnvelope(400, 5, formants=sg.api.DEFAULT_FORMANTS, vocalTract=15.5)
    assert np.array_equal(f('env'), env.ravel(order='F'))
    # soundgen(): R's stream goes in as .Random.seed and comes back advanced exactly as far as the call drew
    y = sg.soundgen(sylLen=300, seed=1)
    assert np.array_equal(f('soundgen_wave'), y) and out['soundgen_status'] == ['0']
    fe = sg.FrontEnd()
    fe.add(sylLen=300, seed=1)
    fe.round_begin()
    assert np.array_equal(np.array(out['soundgen_seed'][1:], dtype=np.int64), fe.rng_state(0))
    assert np.array_equal(f('batch_wave_1'), y) and np.array_equal(f('batch_wave_2'), sg.soundgen(sylLen=300, seed=2))
