"""The K4 error bound (envelope_bound.py) on the host: k_envelope<float>'s operation order emulated in numpy stays
inside the bound on every case of the corpus, and the bound itself stays tight; the front-end draws R's stochastic
formants without a cap (no GPU needed)."""
import ctypes as C

import numpy as np
import pytest

import soundgen_beta_b200 as sg
from envelope_bound import CASES, bound, capture, kernel_f32, reference
from oracle.rrng import RRng
from oracle.soundgen_call import soundgen as osg
from soundgen_beta_b200 import _abi


@pytest.mark.parametrize('name,nr,nc,kw', CASES, ids=[c[0] for c in CASES])
def test_emulated_kernel_within_bound(name, nr, nc, kw):
    env, terms = reference(nr, nc, **kw)
    b = bound(terms, nr)
    got = kernel_f32(terms, nr).astype(np.float64)
    err = np.abs(got - env) / env
    assert np.all(err <= b), (name, float(np.max(err / b)))
    assert float(np.max(b)) <= 3e-5, name            # a loose bound would hide errors
    assert float(np.max(err / b)) >= 0.05, name      # and a bound this far above the emulated error would be loose


FP64_CEILING = {'very narrow': 1e-6, 'F62 closed': 2e-8, 'F200': 2e-8, 'F1024 closed': 2e-8}


@pytest.mark.parametrize('name,nr,nc,kw', CASES, ids=[c[0] for c in CASES])
def test_fp64_bound_stays_small(name, nr, nc, kw):
    """The FP64 path's bound is set by the cancellation of the two log-density terms: it stays below 1e-9 except
    for a very narrow formant (0.2 Hz: shape ~4e7) and for filters of 62 formants and more."""
    env, terms = reference(nr, nc, **kw)
    assert float(np.max(bound(terms, nr, fp32=False))) <= FP64_CEILING.get(name, 1e-9), name


def test_filter_past_the_formant_limit_is_refused():
    """A vocal tract of a kilometre puts R's pseudo-formants 0.18 Hz apart: each draw rounds to a 0 Hz step and R's
    loop would never reach Nyquist - 1000 Hz.  The front-end stops at SGB_MAX_FORMANTS and refuses the call."""
    fe = sg.FrontEnd()
    fe.add(sylLen=300, vocalTract=1e5, temperature=0.1, invalidArgAction='ignore', seed=1)
    desc, _ = fe.round_begin()
    assert fe.status()[0] == _abi.SGB_ERR_UNSUPPORTED
    assert 'formants per filter' in fe.warnings(0)
    bout = C.cast(desc.bouts, C.POINTER(_abi.Bout))[0]
    assert C.cast(desc.envelopes, C.POINTER(_abi.Envelope))[bout.env_id].n_formants == 1024
    fe.close()


def _table_call(sr, seed):
    return dict(sylLen=300, vocalTract=100, temperature=0.1, samplingRate=sr, seed=seed)


@pytest.mark.parametrize('sr,seed', [(sr, s) for sr in (44100, 32000, 22050) for s in (1, 2, 3, 4)])
def test_stochastic_formants_are_not_truncated(sr, seed):
    """vocalTract = 100 cm puts R's pseudo-formants 177 Hz apart up to Nyquist - 1000 Hz: 106 formants at 44.1 kHz
    and 72 at 32 kHz under set.seed(1) (past the old cap of 62), 43 at 22.05 kHz.  (At 16 kHz the same call has 26,
    with vocalTract = 60 17: under the cap, so those rates do not test it.)  R's stream after the call, and the
    number of formants of the main filter, must be the oracle's."""
    kw = _table_call(sr, seed)
    fe = sg.FrontEnd()
    fe.add(**kw)
    desc, _ = fe.round_begin()
    state, status = fe.rng_state(0), fe.status()[0]
    okw = dict(kw)
    rng = RRng(okw.pop('seed'))
    with capture() as rec:
        osg(rng=rng, **okw)
    assert status == 0
    assert np.array_equal(np.array(rng.state(), dtype=np.uint32).astype(np.int32), state)
    bout = C.cast(desc.bouts, C.POINTER(_abi.Bout))[0]
    env = C.cast(desc.envelopes, C.POINTER(_abi.Envelope))[bout.env_id]
    assert env.n_formants == len(rec[-1]['terms']['tracks'])
    fe.close()
