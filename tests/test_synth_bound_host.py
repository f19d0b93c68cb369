"""The float64 bound of K1 (tests/synth_bound.py) on CPU: the corpus reaches every path it is meant to reach, the
bound covers what it claims to cover, and its propagation through the steps after K1 is sound."""
import numpy as np
import pytest

import synth_bound as sb


def _all():
    for n in sb.CASE_NAMES:
        y, art = sb.oracle_case(n)
        yield n, y, art, sb.case_inputs(n)[3], sb.epochs_of(art)


def test_corpus_covers_every_feature():
    srs, nsubs, rows, warps, spans = set(), set(), [], [], []
    feats = dict(shimmer=False, high=False, flat=False, steep=False, long=False, temp=False, anchors=False, attack=False,
                 ne_odd=False)
    for n, y, art, pars, eps in _all():
        srs.add(pars['samplingRate'])
        for e, ep in enumerate(eps):
            nsubs.add(min(ep.nsub, 3))
            rows.append(ep.J)
            feats['ne_odd'] |= ep.Ne % 4 != 0
            ws = sb.synth_warps(ep)
            warps += ws
            feats['high'] |= any(w['ncolw'] > 16 for w in ws)
            spans += sb.tc_piece_spans(art, e, pars['samplingRate'])
            mat = ep.mat
            if mat.shape[1] > 1:     # amplitudes that jump by a factor of 1.5 or more between adjacent cycles
                r = mat[:, 1:] / np.maximum(mat[:, :-1], 1e-300)
                feats['shimmer'] |= bool(np.any((mat[:, :-1] > 1e-3 * mat.max()) & ((r > 1.5) | (r < 1 / 1.5))))
            feats['flat'] |= bool(ep.J >= 100 and np.median(mat.max(axis=1)) > 0.3 * mat.max())
            feats['steep'] |= bool(np.min(mat[mat > 0]) < 2 ** -11.5 * mat.max())
        feats['long'] |= float(art.integr.max()) > 2000
        feats['temp'] |= pars.get('temperature', 0) > 0 and art.drift_upsampled is not None
        feats['anchors'] |= art.ampl_gain is not None
        feats['attack'] |= sb.attack_points(pars) > 0
    assert srs == {16000.0, 22050.0, 44100.0, 48000.0}
    assert nsubs == {0, 1, 2, 3}
    for b in (224, 384, 768, 1152, 2304):
        assert any(b - 8 <= J < b for J in rows) and any(b < J <= b + 8 for J in rows), b
    assert max(rows) > 2304
    assert all(feats.values()), feats
    # k_synth's per-warp selections (kernels_synth.cu:147-168, :201-207)
    assert {w['mode'] for w in warps} == {0, 1, 2, 3}
    assert {w['staged'] for w in warps} == {True, False}
    assert {w['K'] for w in warps} >= {128, 64, 32}
    assert sum(w['straddle'].size for w in warps) > 0
    # k_synth_tc's piece fallback (kernels_synth_tc.cu:273): an interval that reaches a fourth spline piece
    assert max(spans) >= 4


@pytest.mark.parametrize('name', ['sr16k_sub1', 'sr44k_sub3', 'rows385', 'shimmer_jitter', 'high16k', 'long_phase'])
def test_bound_covers_table_and_phase_rounding(name):
    """Each perturbation of the oracle itself in float64 stays inside the term of B that accounts for it."""
    y, art = sb.oracle_case(name)
    # slack 1e-10 of peak: the oracle's own float64 sine arguments (up to ~1e6 rad) carry ~1e-10 of noise
    for e, ep in enumerate(sb.epochs_of(art)):
        ref = ep.wave()
        assert np.allclose(ref, art.epoch_waves[e], rtol=0, atol=1e-12 * np.max(np.abs(ref)))
        d_tab = np.abs(ep.wave(mat=ep.mat.astype(np.float32).astype(np.float64)) - ref)
        assert np.all(d_tab <= sb.table_term(ep) * (1 + 1e-9) + 1e-10 * np.max(np.abs(ref))), (name, e)
        # every float angle of k_synth_tc off by 2^-25 cycles in the same direction
        d_ph = np.abs(ep.wave(dphi=2.0 ** -25 * sb.tc_angle_roundings(ep.j)) - ref)
        assert np.all(d_ph <= sb.float_phase_term(ep) * (1 + 1e-9) + 1e-10 * np.max(np.abs(ref))), (name, e)
        # both sit inside k_synth_tc's bound; k_synth rounds its phase finer (2^-27 cycles) and carries the table
        assert np.all(sb.table_term(ep) + sb.float_phase_term(ep) <= sb.epoch_bound(ep, 'tc')), (name, e)
        assert np.all(sb.table_term(ep) <= sb.epoch_bound(ep, 'ffma')), (name, e)


@pytest.mark.parametrize('name', ['shimmer_jitter', 'temperature', 'ampl_anchors', 'sr44k_sub3'])
def test_propagation_is_sound(name):
    """Perturbing every epoch by at most B_e changes the joined, normalised output by at most the propagated bound
    (zero crossings fixed at the oracle's)."""
    y, art = sb.oracle_case(name)
    pars = sb.case_inputs(name)[3]
    assert np.array_equal(sb.compose(art.epoch_waves, art, pars), y)
    r = np.random.default_rng(3)
    pk = max(np.max(np.abs(w)) for w in art.epoch_waves)
    for scale in (1e-6, 1e-3):
        Bs = [scale * pk * r.random(w.size) for w in art.epoch_waves]
        prop = sb.propagate(Bs, art, pars, k6=False)
        for trial in range(4):
            if trial == 0:
                sg = [np.ones(w.size) for w in art.epoch_waves]          # every sample pushed up: moves the maximum
            else:
                sg = [r.choice([-1.0, 1.0], w.size) * r.random(w.size) ** 0.1 for w in art.epoch_waves]
            yp = sb.compose([w + s * b for w, s, b in zip(art.epoch_waves, sg, Bs)], art, pars)
            assert np.all(np.abs(yp - y) <= prop * (1 + 1e-9)), (name, scale, trial)
