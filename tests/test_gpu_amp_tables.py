"""The amplitude kernel K3 on its own: its FP64 matrices against the oracle's, its FP32 table against the FP64 matrix,
and both unchanged by the batch a call runs in (which sets how K3 splits a syllable's columns over CTAs)."""
import numpy as np
import pytest

import soundgen_beta_b200 as sg
from soundgen_beta_b200 import _abi, workloads
from oracle import soundgen_oracle as so
from oracle.soundgen_call import soundgen as oracle_soundgen

pytestmark = pytest.mark.gpu


def run_batch(calls, min_rows=-1):
    L = _abi.load()
    assert L.sgb_synth_min_rows_set(min_rows) == 0
    try:
        bb = sg.BatchBuilder(u_dtype=np.float32)
        for kw in calls:
            bb.add_soundgen(**kw)
        bt = sg.Batch()
        bt.upload(bb.build())
        bt.run()
    finally:
        L.sgb_synth_min_rows_set(-1)
    assert np.all(bt.status() == 0)
    return bt


def tables(bt, syl):
    """[(n, rows, pairs, f64 rows x columns, f32 region columns x rows x 4)] for the epochs of syllable `syl`."""
    L = _abi.load()
    art = bt.artefacts(syl)
    out = []
    for e in range(art['nEpochs']):
        shape = np.zeros(3, dtype=np.int32)
        assert L.sgb_batch_amp_tables(bt.h, syl, e, None, None, 0, shape.ctypes.data) == 0
        rows, cols, pairs = (int(v) for v in shape)
        f64 = np.zeros(rows * cols)
        f32 = np.zeros(4 * rows * cols, dtype=np.float32)
        assert L.sgb_batch_amp_tables(bt.h, syl, e, f64.ctypes.data, f32.ctypes.data, f64.size,
                                      shape.ctypes.data) == 0
        n = (rows + 1) // (art['rows_kept'] + 1) - 1          # rows = Hk (n + 1) + n
        out.append((n, rows, bool(pairs), f64.reshape(cols, rows).T.copy(), f32.reshape(cols, rows, 4)))
    return out


def check_f32(f64, f32, pairs):
    """The FP32 table is (float)Y_g and (float)(Y_{g+1} - Y_g), bit for bit, in the layout K1 reads."""
    rows, cols = f64.shape
    y = f64[:, :-1].T.astype(np.float32)
    dy = (f64[:, 1:] - f64[:, :-1]).T.astype(np.float32)
    if pairs:
        flat = f32.reshape(-1)
        got = flat[:2 * rows * (cols - 1)].reshape(cols - 1, rows, 2)
        assert np.array_equal(got[..., 0].view(np.uint32), y.view(np.uint32))
        assert np.array_equal(got[..., 1].view(np.uint32), dy.view(np.uint32))
        assert not np.any(flat[2 * rows * (cols - 1):])      # the memset half stays zero
    else:
        got = f32[:cols - 1]
        for c, ref in ((0, y), (1, y), (2, dy), (3, dy)):
            assert np.array_equal(got[..., c].view(np.uint32), ref.view(np.uint32))


@pytest.fixture(scope='module')
def paths():
    calls = workloads.amp_paths()
    bt = run_batch(calls)
    yield calls, bt
    bt.close()


def test_f64_matches_oracle_on_every_path(paths):
    calls, bt = paths
    seen = set()
    for i, kw in enumerate(calls):
        kw = dict(kw)
        z = kw.pop('z')
        _, arts, _ = oracle_soundgen(rng=so.RStream(z=np.concatenate(z)), want_artefacts=True, **kw)
        assert len(arts) == 1
        ref_mats = arts[0].mats
        got = tables(bt, i)
        assert len(got) == len(ref_mats), i
        hk = arts[0].rows_kept
        for e, ((n, rows, pairs, f64, f32), (ref, names)) in enumerate(zip(got, ref_mats)):
            j = np.rint(np.asarray(names) * (n + 1)).astype(np.int64)
            assert f64.shape[1] == ref.shape[1] and np.all((j >= 1) & (j <= rows)), (i, e)
            dense = np.zeros_like(f64)
            dense[j - 1, :] = ref
            tol = 1e-13 * np.max(np.abs(ref), axis=0, keepdims=True)
            err = np.abs(f64 - dense)
            assert np.all(err <= tol), (i, e, float(np.max(err / np.maximum(tol, 1e-300))))
            missing = np.ones(rows, dtype=bool)
            missing[j - 1] = False
            assert not np.any(f64[missing, :]), (i, e)
            check_f32(f64, f32, pairs)
            seen.add('n0' if n == 0 else ('untabled' if hk > 1024 or n > 16 else
                                          ('dense' if rows >= 512 else 'sub<512')))
            if n == 0 and hk > 1024:
                seen.add('n0 Hk>1024')
            if rows > 2560:
                seen.add('>2560')
            seen.add('tc' if pairs else 'fp32')
    assert seen >= {'n0', 'dense', 'sub<512', 'untabled', 'n0 Hk>1024', '>2560', 'tc', 'fp32'}, seen


def test_f32_layout_of_the_fp32_pipe(paths):
    calls, _ = paths
    bt = run_batch(calls, min_rows=1 << 30)      # as SGB_SYNTH=ffma: every epoch on the FP32-pipe kernel
    for i in range(len(calls)):
        for n, rows, pairs, f64, f32 in tables(bt, i):
            assert not pairs
            check_f32(f64, f32, pairs)
    bt.close()


def test_tables_do_not_depend_on_the_batch():
    """A syllable alone (16 column ranges per syllable), in a 300-call batch (4) and in a 2048-call batch (1)."""
    probe = workloads.amp_paths()
    filler = workloads.config3(n=2048)
    ref = None
    for calls in (probe, probe + filler[:300 - len(probe)], probe + filler[:2048 - len(probe)]):
        bt = run_batch(calls)
        got = [tables(bt, i) for i in range(len(probe))]
        bt.close()
        if ref is None:
            ref = got
            continue
        for i, (a, b) in enumerate(zip(ref, got)):
            assert len(a) == len(b)
            for ea, eb in zip(a, b):
                assert ea[:3] == eb[:3]
                assert np.array_equal(ea[3].view(np.uint64), eb[3].view(np.uint64)), i
                assert np.array_equal(ea[4].view(np.uint32), eb[4].view(np.uint32)), i
