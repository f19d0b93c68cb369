"""Python mirror of soundgen's R shells over the C ABI (libsoundgen_b200.so).

Same function names and argument meaning as the reference
(R/soundgen.R:208-277, R/source.R:57-68, :173-205, R/sourceSpectrum.R:71-82, :261-283);
all sample-rate work is done by the CUDA library -- there is no CPU path here.
R is absent from the build image, so this mirror stands in for the R shells of `r/R/`
(which call the same entry points through `.Call`, see INTEGRATION.md).

Random draws: the library never draws.  `z` = standard normals (R `rnorm` stream) per
voiced syllable, `u` = uniforms (`runif`) per noise segment, drawn by the caller in the
reference's order.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _abi, host
from ._abi import (BatchDesc, Bout, Call, Envelope, FormantRef, Noise, RunInfo, SylArtefacts,
                   Syllable)


class SoundgenError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('%s (code %d)' % (msg, code))
        self.code = code


def _check(rc):
    if rc < 0:
        raise SoundgenError(rc, _abi.load().sgb_last_error().decode())
    return rc


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


DEFAULT_FORMANTS = [dict(time=0, freq=860, amp=30, width=120),
                    dict(time=0, freq=1280, amp=40, width=120),
                    dict(time=0, freq=2900, amp=25, width=200)]


def _formant_rows(f):
    """one formant (dict/list/array) -> (k,4) array time, freq, amp, width"""
    if isinstance(f, np.ndarray) and f.ndim == 2 and f.shape[1] == 4 and f.dtype == np.float64:
        return f
    if isinstance(f, dict):
        cols = [np.atleast_1d(np.asarray(f[k], dtype=np.float64)) for k in ('time', 'freq', 'amp', 'width')]
        n = max(c.size for c in cols)
        return np.stack([np.resize(c, n) for c in cols], axis=1)
    a = np.asarray(f, dtype=np.float64)
    return a.reshape(-1, 4)


def _formant_list(formants):
    if formants is None:
        return None
    if isinstance(formants, str):
        raise NotImplementedError('phoneme strings need the presets dictionary (convertStringToFormants, '
                                  'R/utilities_soundgen.R:135-222): pass a list of formants')
    if isinstance(formants, dict):
        formants = list(formants.values())
    return [_formant_rows(f) for f in formants]


def _anchor_arg(a, keep):
    """None / numeric vector / (time, value) / dict -> sgb_anchor_arg"""
    A = _abi.AnchorArg()
    if a is None:
        return A
    if isinstance(a, dict):
        t, v = a['time'], a['value']
    elif isinstance(a, (tuple, list)) and len(a) == 2 and np.ndim(a[0]) == 1 and np.ndim(a[1]) == 1 \
            and len(a[0]) == len(a[1]) and not np.isscalar(a[0]):
        t, v = a
    else:
        t, v = None, a
    v = np.ascontiguousarray(v, dtype=np.float64).reshape(-1)
    if v.size == 0 or (v[0] != v[0] and np.all(np.isnan(v))):
        return A
    keep.append(v)
    A.value, A.n = v.ctypes.data, v.size
    if t is not None:
        t = np.ascontiguousarray(t, dtype=np.float64).reshape(-1)
        keep.append(t)
        A.time = t.ctypes.data
    return A


def _formant_args(fl, keep):
    arr = (_abi.FormantArg * max(1, len(fl)))()
    for i, f in enumerate(fl):
        cols = np.ascontiguousarray(f.T, dtype=np.float64)     # 4 x k
        keep.append(cols)
        k = cols.shape[1]
        for j, nm in enumerate(('time', 'freq', 'amp', 'width')):
            setattr(arr[i], nm, cols[j].ctypes.data)
            setattr(arr[i], 'n_' + nm, k)
    keep.append(arr)
    return arr


SOUNDGEN_DEFAULTS = dict(
    repeatBout=1, nSyl=1, sylLen=300, pauseLen=200, temperature=0.025, maleFemale=0, creakyBreathy=0,
    nonlinBalance=0, nonlinDep=50, jitterLen=1, jitterDep=3, vibratoFreq=5, vibratoDep=0, shimmerDep=0,
    attackLen=50, rolloff=-12, rolloffOct=-12, rolloffKHz=-6, rolloffParab=0, rolloffParabHarm=3, rolloffLip=6,
    formantDep=1, formantDepStoch=30, vocalTract=15.5, subFreq=100, subDep=100, shortestEpoch=300, amDep=0,
    amFreq=30, amShape=0, rolloffNoise=-14, samplingRate=16000, windowLength=50, overlap=75, addSilence=100,
    pitchFloor=50, pitchCeiling=3500, pitchSamplingRate=3500, throwaway=-120)     # R/soundgen.R:208-277
_ANCHOR_DEFAULTS = dict(pitchAnchors=((0, .1, .9, 1), (100, 150, 135, 100)), pitchAnchorsGlobal=None,
                        noiseAnchors=((0, 300), (-120, -120)), mouthAnchors=((0, 1), (.5, .5)), amplAnchors=None,
                        amplAnchorsGlobal=None)
_ACTIONS = {'adjust': 0, 'abort': 1, 'ignore': 2}
_DEFAULT_FORMANT_ARGS = None
_METHODS = {'loess': _abi.SGB_CONTOUR_LOESS, 'spline': _abi.SGB_CONTOUR_SPLINE}


class ArgArray:
    """soundgen() argument lists marshalled once into a contiguous array of `sgb_soundgen_args` -- the form in which
    a binding hands its calls to the library (`sgb_frontend_add_many`)."""

    def __init__(self, calls, u_dtype=np.float64):
        fe = FrontEnd(u_dtype)
        pairs = [fe.marshal(**dict(kw)) for kw in calls]
        fe.close()
        self.n = len(pairs)
        self.u_dtype = np.dtype(u_dtype)
        self.arr = (_abi.SoundgenArgs * max(1, self.n))(*[p[0] for p in pairs])
        self.keep = [p[1] for p in pairs]


class FrontEnd:
    """Handle of the library's host front-end: soundgen() argument lists in, batch descriptions out."""

    def __init__(self, u_dtype=np.float64):
        self.L = _abi.load()
        self.u_dtype = np.dtype(u_dtype)
        self.h = C.c_void_p()
        _check(self.L.sgb_frontend_create(C.byref(self.h), 1 if self.u_dtype == np.float32 else 0))
        self.n_calls = 0
        self.n_sub = 0
        self._keep_alive = []

    def close(self):
        if self.h:
            self.L.sgb_frontend_destroy(self.h)
            self.h = C.c_void_p()
        self._keep_alive = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add(self, warn=None, seeds=None, **kw):
        """One soundgen() call; with `seeds` (a sequence) the same argument list once per seed."""
        A, keep = self.marshal(**kw)
        self._keep_alive.append(keep)      # the library references the caller-drawn z / u buffers until the rounds end
        if seeds is not None:
            sd = np.ascontiguousarray(np.asarray(seeds, dtype=np.int64) & 0xFFFFFFFF, dtype=np.uint32)
            A.rng_mode = 0
            rc = self.L.sgb_frontend_add_seeded(self.h, C.byref(A), sd.ctypes.data, sd.size)
        else:
            rc = self.L.sgb_frontend_add(self.h, C.byref(A))
        self._raise(rc)
        self.n_calls = rc + (1 if seeds is None else len(seeds))
        if warn is not None:
            w = self.L.sgb_frontend_warnings(self.h, rc).decode()
            if w:
                warn.extend(w.split('\n'))
        return rc

    def _raise(self, rc):
        if rc < 0:
            msg = self.L.sgb_last_error().decode()
            if rc == _abi.SGB_ERR_INVALID and 'must be between' in msg:
                raise ValueError(msg)
            if rc == _abi.SGB_ERR_UNSUPPORTED:
                raise NotImplementedError(msg)
            raise SoundgenError(rc, msg)

    def add_many(self, args):
        """Every call of an `ArgArray` (argument lists already in the library's struct form) in one library call."""
        rc = self.L.sgb_frontend_add_many(self.h, args.arr, args.n)
        self._keep_alive.append(args)
        self._raise(rc)
        self.n_calls = rc + args.n
        return rc

    def clear(self):
        _check(self.L.sgb_frontend_clear(self.h))
        self._keep_alive = []
        self.n_calls = 0
        self.n_sub = 0

    def marshal(self, seed=None, z=None, u=None, contour_method='loess', invalidArgAction='adjust',
                formants='default', formantsNoise=None, tempEffects=None, device_pitch=True, rng_state=None,
                sample_kind='Rounding', **kw):
        """A soundgen() argument list as the library's `sgb_soundgen_args` struct (+ the arrays it points to)."""
        keep = []
        A = _abi.SoundgenArgs()
        for k, d in SOUNDGEN_DEFAULTS.items():
            v = kw.pop(k, d) if k in kw else d
            if v is None:
                v = float('nan')
            try:
                setattr(A, k, v)
            except TypeError:
                raise TypeError('%s must be numeric' % k)
        for k, d in _ANCHOR_DEFAULTS.items():
            setattr(A, k, _anchor_arg(kw.pop(k, d), keep))
        if kw:
            raise TypeError('soundgen() got unexpected arguments: %s' % ', '.join(sorted(kw)))
        te = dict(sylLenDep=.02)
        te.update(tempEffects or {})
        for i, k in enumerate(_abi.TEMP_EFFECTS):
            A.tempEffects[i] = float(te.get(k, float('nan')))
        if isinstance(formants, str) and formants == 'default':
            global _DEFAULT_FORMANT_ARGS
            if _DEFAULT_FORMANT_ARGS is None:
                k0 = []
                _DEFAULT_FORMANT_ARGS = (_formant_args(_formant_list(DEFAULT_FORMANTS), k0), k0)
            A.formants = C.cast(_DEFAULT_FORMANT_ARGS[0], C.c_void_p)
            A.n_formants = len(DEFAULT_FORMANTS)
            fl = None
        else:
            if isinstance(formants, str):
                formants = host.convert_string_to_formants(formants)     # soundgen.R:384-386
            fl = _formant_list(formants)
        if fl:
            A.formants = C.cast(_formant_args(fl, keep), C.c_void_p)
            A.n_formants = len(fl)
        fn = _formant_list(formantsNoise)
        if fn:
            A.formantsNoise = C.cast(_formant_args(fn, keep), C.c_void_p)
            A.n_formantsNoise = len(fn)
        A.invalidArgAction = _ACTIONS[invalidArgAction]
        A.contour_method = _METHODS[contour_method]
        A.device_pitch = 1 if device_pitch else 0
        A.sample_rejection = 1 if sample_kind == 'Rejection' else 0
        if rng_state is not None:
            st = np.ascontiguousarray(rng_state, dtype=np.int32)
            keep.append(st)
            A.rng_mode, A.rng_state = 1, st.ctypes.data
        elif seed is not None:
            A.rng_mode, A.seed = 0, int(seed) & 0xFFFFFFFF
        else:
            A.rng_mode = 2
            zl = [] if z is None else (list(z) if isinstance(z, (list, tuple)) else [z])
            ul = [] if u is None else (list(u) if isinstance(u, (list, tuple)) else [u])
            if zl:
                zc = np.ascontiguousarray(np.concatenate([np.ravel(q) for q in zl]), dtype=np.float64)
                zn = np.array([np.size(q) for q in zl], dtype=np.int64)
                keep += [zc, zn]
                A.z, A.z_len, A.n_z = zc.ctypes.data, zn.ctypes.data, len(zl)
            if ul:
                uc = np.ascontiguousarray(np.concatenate([np.ravel(q) for q in ul]), dtype=self.u_dtype)
                un = np.array([np.size(q) for q in ul], dtype=np.int64)
                keep += [uc, un]
                A.u, A.u_len, A.n_u = uc.ctypes.data, un.ctypes.data, len(ul)
        return A, keep

    def round_begin(self):
        d = BatchDesc()
        n = C.c_int32()
        _check(self.L.sgb_frontend_round_begin(self.h, C.byref(d), C.byref(n)))
        self.n_sub = n.value
        esz = 4 if self.u_dtype == np.float32 else 8
        d._keep = {'pitch': _Raw(d.pitch, 8 * d.n_pitch), 'anchors': _Raw(d.anchors, 16 * d.n_anchors),
                   'formants': _Raw(d.formants, 32 * d.n_formants), 'z': _Raw(d.z, 8 * d.n_z),
                   'u': _Raw(d.u, esz * d.n_u), 'pre': _Raw(d.pre, 8 * d.n_pre)}
        d._fe = self
        return d, n.value

    def resolve(self, batch):
        _check(self.L.sgb_frontend_resolve(self.h, batch.h))

    def round_end(self, batch):
        _check(self.L.sgb_frontend_round_end(self.h, batch.h))

    def round_calls(self):
        out = np.zeros(max(1, self.n_sub), dtype=np.int32)
        _check(self.L.sgb_frontend_round_calls(self.h, _ptr(out)))
        return out[:self.n_sub]

    def status(self):
        out = np.zeros(max(1, self.n_calls), dtype=np.int32)
        _check(self.L.sgb_frontend_status(self.h, _ptr(out)))
        return out[:self.n_calls]

    def warnings(self, call):
        return self.L.sgb_frontend_warnings(self.h, call).decode()

    def rng_state(self, call):
        out = np.zeros(625, dtype=np.int32)
        _check(self.L.sgb_frontend_rng_state(self.h, call, _ptr(out)))
        return out

    def h2d_bytes(self):
        return int(self.L.sgb_frontend_h2d_bytes(self.h))


class _Raw:
    """A library-owned host buffer (pointer + bytes) in the shape pin_desc expects."""

    def __init__(self, ptr, nbytes):
        self.ptr, self.nbytes, self.size = ptr or 0, int(nbytes), int(nbytes)

    @property
    def ctypes(self):
        return self

    @property
    def data(self):
        return self.ptr


def run_rounds(fe, batch=None, out_dtype=np.float32, copy=True):
    """Drives every round of a front-end through one batch handle: upload, run_begin, draw the
    deferred formant tracks, run_finish, fetch.  Returns (waveforms per call, statuses)."""
    own = batch is None
    bt = batch or Batch()
    parts = [[] for _ in range(fe.n_calls)]
    while True:
        desc, n = fe.round_begin()
        if n == 0:
            break
        bt.upload(desc)
        bt.run()
        segs = bt.fetch(out_dtype)
        for k, ci in enumerate(fe.round_calls()):
            parts[ci].append(segs[k].copy() if copy else segs[k])
    st = fe.status()
    if own:
        bt.close()
    outs = [(np.concatenate(p) if len(p) > 1 else (p[0] if p else np.zeros(0, dtype=out_dtype))) for p in parts]
    return outs, st


class BatchBuilder:
    """Accumulates soundgen() calls into the flat pools of an sgb_batch_desc."""

    def __init__(self, u_dtype=np.float64):
        self.calls, self.bouts, self.syls, self.noises, self.envs, self.frefs = [], [], [], [], [], []
        self.pitch, self.anchors, self.formants, self.z, self.u, self.pre = [], [], [], [], [], []
        self.n_pitch = self.n_anchors = self.n_formants = self.n_z = self.n_u = self.n_pre = 0
        self.u_dtype = np.dtype(u_dtype)
        self._keep = []
        self._fe = None

    # ---- pools ----
    def _add_pitch(self, p):
        p = np.ascontiguousarray(p, dtype=np.float64)
        off = self.n_pitch
        self.pitch.append(p)
        self.n_pitch += p.size
        return off

    def _add_anchors(self, an):
        t, v = an
        a = np.stack([np.asarray(t, dtype=np.float64), np.asarray(v, dtype=np.float64)], axis=1)
        off = self.n_anchors
        self.anchors.append(a.ravel())
        self.n_anchors += a.shape[0]
        return off, a.shape[0]

    def _add_z(self, z):
        z = np.zeros(0) if z is None else np.ascontiguousarray(z, dtype=np.float64)
        off = self.n_z
        self.z.append(z)
        self.n_z += z.size
        return off, z.size

    def _add_u(self, u):
        u = np.ascontiguousarray(u, dtype=self.u_dtype)
        off = self.n_u
        self.u.append(u)
        self.n_u += u.size
        return off

    def _add_pre(self, c):
        c = np.ascontiguousarray(c, dtype=np.float64)
        off = self.n_pre
        self.pre.append(c)
        self.n_pre += c.size
        return off

    def add_envelope(self, formants, formantDep=1, rolloffLip=6, mouthAnchors=None, mouthOpenThres=0,
                     openMouthBoost=0, vocalTract=None, samplingRate=16000, speedSound=35400,
                     smoothLinearFactor=1, nc_fixed=0, tracks=None, contour_method='loess'):
        """Registers one getSpectralEnvelope() specification; resolves the vocalTract /
        schwa defaults of R/sourceSpectrum.R:294-315 (argument munging, host side)."""
        fl = _formant_list(formants)
        if fl is not None and vocalTract is None and fl[0].shape[1] > 2:
            freqs = np.concatenate([f[:, 1] for f in fl])
            if freqs.size > 1:
                vocalTract = speedSound / 2 / float(np.mean(np.diff(freqs)))
            else:
                vocalTract = speedSound / 4 / float(fl[0][0, 1])
        if fl is None and vocalTract is not None:
            freq = speedSound / 4 / vocalTract
            fl = [np.array([[0, freq, 30, 50 * (1 + freq ** 2 / 6 / 10 ** 6)]])]
        e = Envelope()
        e.n_formants = 0 if fl is None else len(fl)
        e.tracks_given = 0
        e.formant_off = len(self.frefs)
        if tracks is not None:
            fl = [np.asarray(t, dtype=np.float64).reshape(-1, 4) for t in tracks]
            e.n_formants = len(fl)
            e.tracks_given = 1
        if fl is not None:
            for f in fl:
                r = FormantRef()
                r.off = self.n_formants
                r.n = f.shape[0]
                self.frefs.append(r)
                self.formants.append(np.ascontiguousarray(f, dtype=np.float64).ravel())
                self.n_formants += f.shape[0]
        ma = host.as_anchors(mouthAnchors)
        if ma is not None and not np.any(np.isnan(ma[1])):
            e.mouth_off, e.mouth_n = self._add_anchors(ma)
            e.mouth_method = _METHODS[contour_method]
        else:
            e.mouth_n = 0
        e.nc_fixed = int(nc_fixed)
        e.formantDep, e.rolloffLip = float(formantDep), float(rolloffLip)
        e.mouthOpenThres, e.openMouthBoost = float(mouthOpenThres), float(openMouthBoost)
        e.vocalTract = float('nan') if vocalTract is None else float(vocalTract)
        e.samplingRate, e.speedSound = float(samplingRate), float(speedSound)
        e.smoothLinearFactor = float(smoothLinearFactor)
        self.envs.append(e)
        return len(self.envs) - 1

    def add_envelope_matrix(self, m, samplingRate=16000):
        """Registers a literal (nr x nc) filter matrix, e.g. generateNoise()'s filterNoise."""
        m = np.asarray(m, dtype=np.float64)
        if m.ndim == 1:
            m = m[:, None]
        e = Envelope()
        e.n_formants, e.tracks_given = 0, 2
        e.formant_off = self._add_pre(np.asfortranarray(m).ravel(order='F'))
        e.mouth_n, e.nc_fixed = 0, int(m.shape[1])
        e.formantDep, e.rolloffLip, e.mouthOpenThres, e.openMouthBoost = 1.0, 0.0, 0.0, 0.0
        e.vocalTract, e.samplingRate, e.speedSound, e.smoothLinearFactor = float('nan'), float(samplingRate), 35400.0, 1.0
        self.envs.append(e)
        return len(self.envs) - 1

    def add_syllable(self, pitch, z=None, amplAnchors=None, pause_after=0, contour_method='loess', **pars):
        s = Syllable()
        s.kind = 1
        s.pitch_off = self._add_pitch(pitch)
        s.pitch_len = int(np.size(pitch))
        s.pause_after = int(pause_after)
        s.z_off, s.z_cap = self._add_z(z)
        an = host.as_anchors(amplAnchors)
        if an is not None:
            s.ampl_off, s.ampl_n = self._add_anchors(an)
            s.ampl_method = _METHODS[contour_method]
        d = dict(attackLen=50, nonlinBalance=0, jitterDep=0, jitterLen=1, vibratoFreq=100, vibratoDep=0,
                 shimmerDep=0, rolloff=-18, rolloffOct=-2, rolloffKHz=-6, rolloffParab=0,
                 rolloffParabHarm=3, rolloff_perAmpl=12, temperature=0, pitchDriftDep=.5,
                 pitchDriftFreq=.125, randomWalk_trendStrength=.5, shortestEpoch=300, subFreq=100,
                 subDep=0, samplingRate=16000, pitchFloor=75, pitchCeiling=3500, pitchSamplingRate=3500,
                 throwaway=-120)
        for k, v in pars.items():
            if k in d:
                d[k] = v
        for k in _abi.SYL_DOUBLES:
            setattr(s, k, float(d[k]))
        self.syls.append(s)
        return len(self.syls) - 1

    def add_silent_syllable(self, n, pause_after=0):
        s = Syllable()
        s.kind = 0
        s.silent_len = int(n)
        s.pause_after = int(pause_after)
        self.syls.append(s)
        return len(self.syls) - 1

    def add_noise(self, length, noiseAnchors, u, rolloffNoise=-6, attackLen=10, windowLength_points=1024,
                  samplingRate=16000, overlap=75, env_id=-1, insertion=1, mix=0, strength=None,
                  contour_method='loess'):
        n = Noise()
        n.len = int(length)
        n.insertion = int(insertion)
        n.mix = int(mix)
        n.wl = int(windowLength_points)
        n.u_off = self._add_u(u)
        an = host.as_anchors(noiseAnchors)
        n.strength_pre_off = -1
        if strength is not None:
            n.strength_pre_off = self._add_pre(strength)
            n.anchor_n = 0
        else:
            n.anchor_off, n.anchor_n = self._add_anchors(an)
            n.anchor_method = _METHODS[contour_method]
        n.env_id = int(env_id)
        n.rolloffNoise, n.attackLen = float(rolloffNoise), float(attackLen)
        n.samplingRate, n.overlap = float(samplingRate), float(overlap)
        self.noises.append(n)
        return len(self.noises) - 1

    def add_bout(self, syl_begin, syl_end, noise_begin, noise_end, env_id, moving, wl, overlap=75,
                 lead_silence=0, tail_silence=0, amplAnchorsGlobal=None, amDep=0, amFreq=30, amShape=0,
                 samplingRate=16000, throwaway=-120, contour_method='loess'):
        b = Bout()
        b.syl_begin, b.syl_end, b.noise_begin, b.noise_end = syl_begin, syl_end, noise_begin, noise_end
        b.env_id, b.moving, b.wl = int(env_id), int(bool(moving)), int(wl)
        b.lead_silence, b.tail_silence = int(lead_silence), int(tail_silence)
        if amplAnchorsGlobal is not None:
            b.aglobal_off, b.aglobal_n = self._add_anchors(amplAnchorsGlobal)
            b.aglobal_method = _METHODS[contour_method]
        b.overlap, b.amDep, b.amFreq, b.amShape = float(overlap), float(amDep), float(amFreq), float(amShape)
        b.samplingRate, b.throwaway = float(samplingRate), float(throwaway)
        self.bouts.append(b)
        return len(self.bouts) - 1

    def add_call(self, bout_begin, bout_end):
        c = Call()
        c.bout_begin, c.bout_end = bout_begin, bout_end
        self.calls.append(c)
        return len(self.calls) - 1

    # ---- the bout orchestrator's host stage (R/soundgen.R:279-733): C front-end ----
    def add_soundgen(self, **kw):
        """Adds one soundgen() call through the library's host front-end (csrc/frontend.cu).
        Besides soundgen()'s own arguments: `seed` (R's set.seed; every draw of the call then comes
        from R's stream in the reference's order), or `z` / `u` (lists of caller-drawn normal /
        uniform buffers, one per voiced syllable / noise segment; temperature must be 0),
        `contour_method` ('loess' = reference, 'spline'), `warn` (list receiving the warnings),
        `device_pitch` (evaluate the pitch contour on the device when no draw count depends on it).
        Returns the call index."""
        if self.syls or self.bouts:
            raise ValueError('add_soundgen cannot be mixed with the low-level add_* calls in one builder')
        if self._fe is None:
            self._fe = FrontEnd(self.u_dtype)
        return self._fe.add(**kw)

    def noise_uniform_count(self, length, windowLength_points, overlap=75):
        """number of runif() draws generateNoise makes (R/source.R:88-111)."""
        wl = int(windowLength_points)
        h = wl - (overlap * wl / 100)
        return (wl // 2) * host.seq_by_count(1.0, float(length) + wl, h)

    # ---- finalise ----
    def build(self):
        if self._fe is not None:
            desc, _ = self._fe.round_begin()
            return desc

        def arr(T, items):
            a = (T * max(1, len(items)))()
            for i, it in enumerate(items):
                a[i] = it
            return a

        def cat(parts, dtype):
            return np.ascontiguousarray(np.concatenate(parts), dtype=dtype) if parts else np.zeros(0, dtype=dtype)
        d = BatchDesc()
        keep = dict(calls=arr(Call, self.calls), bouts=arr(Bout, self.bouts), syls=arr(Syllable, self.syls),
                    noises=arr(Noise, self.noises), envs=arr(Envelope, self.envs),
                    frefs=arr(FormantRef, self.frefs), pitch=cat(self.pitch, np.float64),
                    anchors=cat(self.anchors, np.float64), formants=cat(self.formants, np.float64),
                    z=cat(self.z, np.float64), u=cat(self.u, self.u_dtype), pre=cat(self.pre, np.float64))
        d.n_calls, d.n_bouts, d.n_syllables = len(self.calls), len(self.bouts), len(self.syls)
        d.n_noises, d.n_envelopes, d.n_formant_refs = len(self.noises), len(self.envs), len(self.frefs)
        for k in ('calls', 'bouts', 'noises'):
            setattr(d, k, C.cast(keep[k], C.c_void_p))
        d.syllables = C.cast(keep['syls'], C.c_void_p)
        d.envelopes = C.cast(keep['envs'], C.c_void_p)
        d.formant_index = C.cast(keep['frefs'], C.c_void_p)
        d.pitch, d.n_pitch = _ptr(keep['pitch']), self.n_pitch
        d.anchors, d.n_anchors = _ptr(keep['anchors']), self.n_anchors
        d.formants, d.n_formants = _ptr(keep['formants']), self.n_formants
        d.z, d.n_z = _ptr(keep['z']), self.n_z
        d.u, d.n_u = _ptr(keep['u']), self.n_u
        d.u_is_float = 1 if self.u_dtype == np.float32 else 0
        d.pre, d.n_pre = _ptr(keep['pre']), self.n_pre
        d._keep = keep
        return d

    def h2d_bytes(self):
        if self._fe is not None:
            return self._fe.h2d_bytes()
        return (8 * (self.n_pitch + 2 * self.n_anchors + 4 * self.n_formants + self.n_z + self.n_pre) +
                self.u_dtype.itemsize * self.n_u + C.sizeof(Syllable) * len(self.syls) +
                C.sizeof(Bout) * len(self.bouts) + C.sizeof(Noise) * len(self.noises) +
                C.sizeof(Envelope) * len(self.envs) + C.sizeof(FormantRef) * len(self.frefs))


class Batch:
    """Owner of one sgb_batch handle."""

    def __init__(self):
        self.L = _abi.load()
        self.h = C.c_void_p()
        _check(self.L.sgb_batch_create(C.byref(self.h)))
        self.desc = None
        self.info = None

    def close(self):
        if self.h:
            self.L.sgb_batch_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, desc):
        self.desc = desc
        _check(self.L.sgb_batch_upload(self.h, C.byref(desc)))

    def run(self):
        """One pass of the whole path over the uploaded batch.  A description that came from the host
        front-end may hold main filters whose stochastic tracks can only be drawn once the device knows
        the number of STFT frames: those are resolved between the two phases of the run."""
        info = RunInfo()
        fe = getattr(self.desc, '_fe', None)
        if fe is None:
            _check(self.L.sgb_batch_run(self.h, C.byref(info)))
        else:
            _check(self.L.sgb_batch_run_begin(self.h))
            fe.resolve(self)
            _check(self.L.sgb_batch_run_finish(self.h, C.byref(info)))
            fe.round_end(self)
        self.info = info
        return info

    def lengths(self):
        n = self.desc.n_calls
        out = np.zeros(n, dtype=np.int64)
        _check(self.L.sgb_batch_lengths(self.h, _ptr(out)))
        return out

    def status(self):
        out = np.zeros(self.desc.n_calls, dtype=np.int32)
        _check(self.L.sgb_batch_status(self.h, _ptr(out)))
        return out

    def fetch(self, dtype=np.float64, out=None):
        lens = self.lengths()
        total = int(lens.sum())
        if out is None:
            out = np.zeros(max(total, 1), dtype=dtype)
        if np.dtype(dtype) == np.int16:     # WAV samples as the reference's savePath branch writes them
            _check(self.L.sgb_batch_fetch_pcm16(self.h, _ptr(out), out.size))
        elif np.dtype(dtype) == np.float32:
            _check(self.L.sgb_batch_fetch_f32(self.h, _ptr(out), out.size))
        else:
            _check(self.L.sgb_batch_fetch_f64(self.h, _ptr(out), out.size))
        offs = np.concatenate(([0], np.cumsum(lens)))
        return [out[offs[i]:offs[i + 1]] for i in range(lens.size)]

    def export(self, dst, dst_off, cap, stream=None, fmt='f32'):
        """Writes every call of the last run into the CUDA tensor `dst` (float32 for fmt 'f32', int16 for 'pcm16'):
        call c fills exactly cap[c] elements from element dst_off[c] of the flattened tensor, its first
        min(len, cap) samples and then zeros.  Ordered on `stream` (a torch.cuda.Stream or a raw cudaStream_t; default
        the current stream of dst's device) with no host synchronisation.  Returns the samples written per call."""
        n = self.desc.n_calls if self.desc is not None else 0
        return _export(lambda o: self.L.sgb_batch_export(self.h, C.byref(o)), n, dst, dst_off, cap, stream, fmt)

    def spectrogram(self, dst, dst_off, cap, wl, overlap=75, window='hamming', bands=None, db=False, db_floor=1e-10,
                    stream=None):
        """Spectrogram of every call of the last run (row c = call c) into the float32 CUDA tensor `dst`: call c fills
        exactly cap[c] frames of n_feat floats from element dst_off[c] of the flattened tensor, its first min(nc, cap)
        frames and then zeros (see sgb_batch_spectrogram for the frame and spectrum definitions).  bands: None (power,
        n_feat = wl / 2) or a dense [n_bands, wl / 2] filterbank whose rows each have contiguous support (n_feat =
        n_bands), e.g. mel_filterbank(); db: 10 log10(max(F, db_floor)).  Ordered on `stream` like export().
        Returns the frames written per call."""
        n = self.desc.n_calls if self.desc is not None else 0
        return _spectrogram(lambda p, o: self.L.sgb_batch_spectrogram(self.h, C.byref(p), C.byref(o)), n, dst, dst_off,
                            cap, wl, overlap, window, bands, db, db_floor, stream)

    def f0(self, dst, dst_off, cap, stream=None):
        """The f0 track of every call of the last run (K12a, sgb_batch_f0) into the float32 CUDA tensor `dst`, laid out
        as export() lays out the samples: call c fills exactly cap[c] elements from element dst_off[c], the f0 in Hz of
        each of its first min(len, cap) samples (0 where unvoiced) and then zeros.  With sub-harmonics the partials
        are multiples of f0 / (nSubharm + 1); the track still reports f0.  Ordered on `stream` like export().
        Returns the samples written per call."""
        n = self.desc.n_calls if self.desc is not None else 0
        return _export(lambda o: self.L.sgb_batch_f0(self.h, C.byref(o)), n, dst, dst_off, cap, stream, 'f32')

    def syllable(self, s):
        n = C.c_int64()
        _check(self.L.sgb_batch_syllable_len(self.h, s, C.byref(n)))
        out = np.zeros(max(n.value, 1))
        _check(self.L.sgb_batch_syllable_fetch(self.h, s, _ptr(out), out.size))
        return out[:n.value]

    def noise(self, n, length):
        out = np.zeros(max(int(length), 1))
        _check(self.L.sgb_batch_noise_fetch(self.h, n, _ptr(out), out.size))
        return out[:int(length)]

    def envelope(self, kind, index):
        """The FP32 spectral envelope (nr x nint) the last run filtered with: kind 0 the main filter of bout `index`,
        kind 1 the filter of noise `index`; None for a bypassed bout or an unfiltered noise."""
        shape = np.zeros(2, dtype=np.int32)
        _check(self.L.sgb_batch_envelope(self.h, kind, index, None, 0, _ptr(shape)))
        nr, nint = (int(v) for v in shape)
        if nr * nint == 0:
            return None
        out = np.zeros(nr * nint, dtype=np.float32)
        _check(self.L.sgb_batch_envelope(self.h, kind, index, _ptr(out), out.size, _ptr(shape)))
        return out.reshape(nint, nr).T.copy()

    def artefacts(self, s):
        a = SylArtefacts()
        _check(self.L.sgb_batch_artefacts(self.h, s, C.byref(a)))
        res = dict(nGC=a.nGC, nHarmonics=a.nHarmonics, rows_kept=a.rows_kept, nEpochs=a.nEpochs,
                   n_upsampled=a.n_upsampled, z_used=a.z_used, status=a.status, raw_max=a.raw_max)
        cap = max(a.nGC + 2, 2 * a.nEpochs + 2, a.n_jitter_idx + 2)
        names = ['gc', 'gc_upsampled', 'nSubharm', 'rw_bin', 'jitter_idx', 'epochs', 'zc']
        for w, nm in enumerate(names):
            buf = np.zeros(cap, dtype=np.int32)
            n = _check(self.L.sgb_batch_artefact_ints(self.h, s, w, _ptr(buf), cap))
            res[nm] = buf[:n].copy()
        res['epochs'] = res['epochs'].reshape(-1, 2)
        res['zc'] = res['zc'].reshape(-1, 2)
        p = np.zeros(max(a.nGC, 1))
        _check(self.L.sgb_batch_pitch_per_gc(self.h, s, _ptr(p), p.size))
        res['pitch_per_gc'] = p[:a.nGC]
        return res


# ------------------------------------------------------------------------------
# R-named entry points
# ------------------------------------------------------------------------------
def soundgen(*args, return_batch=False, **kwargs):
    """soundgen() (R/soundgen.R:208-277): returns the synthesised waveform (float64).
    `seed` plays the role of set.seed() before the call; without it the call must not need host
    draws (temperature = 0) and takes its jitter / shimmer normals `z` and noise uniforms `u` from the
    caller.  Raises SoundgenError('Failed to generate the new syllable!') where the reference stops."""
    names = ['repeatBout', 'nSyl', 'sylLen', 'pauseLen', 'pitchAnchors', 'pitchAnchorsGlobal', 'temperature']
    kwargs.update(dict(zip(names, args)))
    kwargs.pop('pitchContours', None)
    fe = FrontEnd()
    fe.add(**kwargs)
    bt = Batch()
    try:
        outs, st = run_rounds(fe, bt, np.float64)
    except SoundgenError as e:
        if e.code == _abi.SGB_ERR_STREAM:
            raise ValueError('soundgen(): a uniform buffer `u` is needed for each noise segment (%s)' % e)
        raise
    if st[0] == _abi.SGB_ERR_SYNTH:
        raise SoundgenError(st[0], 'Failed to generate the new syllable!')
    if st[0] == _abi.SGB_ERR_STREAM and kwargs.get('seed') is None:
        raise ValueError('soundgen(): the `z` / `u` buffers are shorter than the draws needed')
    if st[0] != 0:
        raise SoundgenError(int(st[0]), 'soundgen failed: %s' % fe.warnings(0))
    y = outs[0]
    if return_batch:
        return y, bt
    bt.close()
    fe.close()
    return y


def soundgen_batch(list_of_kwargs, out_dtype=np.float32, u_dtype=np.float64):
    """Many soundgen() calls in one pass (the batched entry the reference lacks)."""
    fe = FrontEnd(u_dtype)
    for kw in list_of_kwargs:
        fe.add(**kw)
    outs, st = run_rounds(fe, None, out_dtype)
    fe.close()
    return outs, st


_OUT_FORMATS = {'f32': (_abi.SGB_OUT_F32, 'float32'), 'pcm16': (_abi.SGB_OUT_PCM16, 'int16')}


def _stream_handle(stream, dst):
    import torch
    if stream is None:
        return torch.cuda.current_stream(dst.device).cuda_stream if dst.is_cuda else 0
    return stream.cuda_stream if hasattr(stream, 'cuda_stream') else int(stream)


def _export(call, n, dst, dst_off, cap, stream, fmt):
    """Fills an sgb_device_out for the tensor `dst` and runs `call` on it; the library checks where dst lives."""
    import torch
    if fmt not in _OUT_FORMATS:
        raise ValueError("fmt must be 'f32' or 'pcm16', not %r" % (fmt,))
    code, tname = _OUT_FORMATS[fmt]
    if dst.dtype != getattr(torch, tname):
        raise ValueError('fmt %r writes %s, dst is %s' % (fmt, tname, dst.dtype))
    if not dst.is_contiguous():
        raise ValueError('dst must be contiguous')
    off = np.ascontiguousarray(dst_off, dtype=np.int64)
    cp = np.ascontiguousarray(cap, dtype=np.int64)
    if off.shape != (n,) or cp.shape != (n,):
        raise ValueError('dst_off and cap need one entry per row (%d)' % n)
    written = np.zeros(n, dtype=np.int64)
    o = _abi.DeviceOut()
    o.dst, o.dst_elems = dst.data_ptr() or None, dst.numel()
    o.dst_off, o.cap, o.out_written = _ptr(off), _ptr(cp), _ptr(written)
    o.stream = _stream_handle(stream, dst) or None
    o.format = code
    _check(call(o))
    return written


def rows_export(device, src, src_off, lens, dst, dst_off, cap, stream=None, fmt='pcm16'):
    """sgb_rows_export: the export over float32 rows the caller holds in the CUDA tensor `src` (row c = lens[c]
    samples from element src_off[c]); with fmt 'pcm16' every row is normalised over its lens[c] samples."""
    so = np.ascontiguousarray(src_off, dtype=np.int64)
    ln = np.ascontiguousarray(lens, dtype=np.int64)
    if not src.is_contiguous() or so.shape != ln.shape:
        raise ValueError('src must be contiguous, src_off and lens of one length')
    L = _abi.load()
    return _export(lambda o: L.sgb_rows_export(int(device), src.data_ptr() or None, _ptr(so), _ptr(ln), ln.size,
                                               C.byref(o)), ln.size, dst, dst_off, cap, stream, fmt)


_WINDOWS = {'hamming': _abi.SGB_WIN_HAMMING, 'hanning': _abi.SGB_WIN_HANNING}


def bands_csr(bands, n_bins):
    """A dense filterbank [n_bands, n_bins] as the library takes it: (lo, len, weights), row b's weights on the
    contiguous bins [lo[b], lo[b] + len[b]).  A row whose nonzero weights are not contiguous raises ValueError."""
    B = np.asarray(bands, dtype=np.float32)
    if B.ndim != 2 or B.shape[0] < 1 or B.shape[1] != n_bins:
        raise ValueError('bands must be a [n_bands >= 1, %d] array, not %r' % (n_bins, B.shape))
    lo = np.zeros(B.shape[0], dtype=np.int32)
    ln = np.zeros(B.shape[0], dtype=np.int32)
    w = []
    for b, row in enumerate(B):
        nz = np.flatnonzero(row)
        if nz.size == 0:
            continue
        a, e = int(nz[0]), int(nz[-1]) + 1
        if nz.size != e - a:
            raise ValueError('band %d: weights on non-contiguous bins (%d nonzero in [%d, %d))' % (b, nz.size, a, e))
        lo[b], ln[b] = a, e - a
        w.append(row[a:e])
    return lo, ln, (np.concatenate(w) if w else np.zeros(1, dtype=np.float32))


def _spec_params(wl, overlap, window, bands, db, db_floor):
    """sgb_spec_params for the arguments; also returns the arrays it points into (keep them alive)."""
    if window not in _WINDOWS:
        raise ValueError("window must be 'hamming' or 'hanning', not %r" % (window,))
    p = _abi.SpecParams()
    p.wl, p.window, p.overlap = int(wl), _WINDOWS[window], float(overlap)
    p.db, p.db_floor = int(bool(db)), float(db_floor)
    keep = None
    if bands is not None:
        keep = bands_csr(bands, int(wl) // 2)
        p.n_bands = keep[0].size
        p.band_lo, p.band_len, p.band_w = (_ptr(a) for a in keep)
    return p, keep


def _spectrogram(call, n, dst, dst_off, cap, wl, overlap, window, bands, db, db_floor, stream):
    p, keep = _spec_params(wl, overlap, window, bands, db, db_floor)
    written = _export(lambda o: call(p, o), n, dst, dst_off, cap, stream, 'f32')
    del keep
    return written


def rows_spectrogram(device, src, src_off, lens, dst, dst_off, cap, wl, overlap=75, window='hamming', bands=None,
                     db=False, db_floor=1e-10, stream=None):
    """sgb_rows_spectrogram: Batch.spectrogram over float32 rows the caller holds in the CUDA tensor `src` (row c =
    lens[c] samples from element src_off[c]).  Returns the frames written per row."""
    import torch
    so = np.ascontiguousarray(src_off, dtype=np.int64)
    ln = np.ascontiguousarray(lens, dtype=np.int64)
    if not src.is_contiguous() or src.dtype != torch.float32 or so.shape != ln.shape or so.ndim != 1:
        raise ValueError('src must be a contiguous float32 tensor, src_off and lens of one length')
    L = _abi.load()
    return _spectrogram(lambda p, o: L.sgb_rows_spectrogram(int(device), src.data_ptr() or None, _ptr(so), _ptr(ln),
                                                            ln.size, C.byref(p), C.byref(o)),
                        ln.size, dst, dst_off, cap, wl, overlap, window, bands, db, db_floor, stream)


def rows_f0_frames(device, src, src_off, lens, dst, dst_off, cap, wl, overlap=75, stream=None):
    """sgb_rows_f0_frames (K12b): frame labels of float32 rows the caller holds in the CUDA tensor `src` (row c =
    lens[c] samples from element src_off[c]), typically f0 tracks.  Frame k of a row is K9's frame k at the same wl
    and overlap; its label is [f0 at the frame's centre sample, fraction of the frame's wl samples that are nonzero
    (voiced)].  Row c fills exactly cap[c] labels (2 cap[c] floats) of the float32 CUDA tensor `dst` from element
    dst_off[c], zeros past the row's frames.  Ordered on `stream` like export().  Returns the frames written per row."""
    import torch
    so = np.ascontiguousarray(src_off, dtype=np.int64)
    ln = np.ascontiguousarray(lens, dtype=np.int64)
    if not (torch.is_tensor(src) and src.is_contiguous() and src.dtype == torch.float32) or so.shape != ln.shape \
            or so.ndim != 1:
        raise ValueError('src must be a contiguous float32 tensor, src_off and lens of one length')
    L = _abi.load()
    return _export(lambda o: L.sgb_rows_f0_frames(int(device), src.data_ptr() or None, src.numel(), _ptr(so), _ptr(ln),
                                                  ln.size, int(wl), float(overlap), C.byref(o)), ln.size, dst, dst_off,
                   cap, stream, 'f32')


def f0_frames_device(f0, lengths, samplingRate, windowLength=50, overlap=75):
    """Frame labels of the [n, T] float32 f0 tracks that soundgen_batch_device(..., f0=True) returns, aligned frame
    for frame with spectrogram_device(wave, lengths, samplingRate, windowLength, overlap): the same per-row window
    wl = floor(windowLength / 1000 * sr / 2) * 2 at the row's rate (samplingRate: one value or one per row; one
    library call per window length) and the same frames.  Returns (labels, frames): labels [n, F, 2] float32 on the
    same device, labels[c, k] = [f0 at frame k's centre sample, voiced fraction of its wl samples], zeros past the
    row's frames, F = the most frames of any row; frames: int64 CUDA tensor, equal to spectrogram_device's.  Ordered
    on the device's current torch stream; a CUDA `lengths` is read back once."""
    import torch
    if not (torch.is_tensor(f0) and f0.is_cuda and f0.dtype == torch.float32 and f0.dim() == 2):
        raise ValueError('f0 must be a 2-D float32 CUDA tensor')
    n, T = f0.shape
    lens = (lengths.cpu().numpy() if torch.is_tensor(lengths) else np.asarray(lengths)).astype(np.int64).reshape(-1)
    if lens.shape != (n,) or np.any(lens < 0) or np.any(lens > T):
        raise ValueError('lengths needs one value in [0, %d] per row (%d)' % (T, n))
    sr = np.broadcast_to(np.asarray(samplingRate, dtype=np.float64).reshape(-1), (n,)) if n else np.zeros(0)
    if not np.all(np.isfinite(sr) & (sr > 0)):
        raise ValueError('samplingRate must be positive')
    wl = (np.floor(windowLength / 1000 * sr / 2) * 2).astype(np.int64)
    L = _abi.load()
    nc = np.array([L.sgb_spec_frames(int(l), int(w), float(overlap)) for l, w in zip(lens, wl)], dtype=np.int64)
    if np.any(nc < 0):
        raise SoundgenError(_abi.SGB_ERR_UNSUPPORTED, 'window of %s points / overlap %r cannot be analysed'
                            % (np.unique(wl[nc < 0]), overlap))
    F = int(nc.max(initial=0))
    labels = torch.empty((n, F, 2), dtype=torch.float32, device=f0.device)
    if n and F:
        src = f0.contiguous()
        rows = np.arange(n, dtype=np.int64)
        for w in np.unique(wl):
            cap = np.where(wl == w, F, 0).astype(np.int64)
            rows_f0_frames(f0.device.index, src, rows * T, lens, labels, rows * F * 2, cap, int(w), overlap)
    return labels, torch.as_tensor(nc, dtype=torch.int64).to(f0.device)


def _hz_to_mel(f, mel_scale):
    f = np.asarray(f, dtype=np.float64)
    if mel_scale == 'htk':
        return 2595.0 * np.log10(1.0 + f / 700.0)
    f_sp, min_log_hz = 200.0 / 3, 1000.0
    min_log_mel, logstep = min_log_hz / f_sp, math.log(6.4) / 27.0
    return np.where(f >= min_log_hz, min_log_mel + np.log(np.maximum(f, min_log_hz) / min_log_hz) / logstep, f / f_sp)


def _mel_to_hz(m, mel_scale):
    m = np.asarray(m, dtype=np.float64)
    if mel_scale == 'htk':
        return 700.0 * (10.0 ** (m / 2595.0) - 1.0)
    f_sp, min_log_hz = 200.0 / 3, 1000.0
    min_log_mel, logstep = min_log_hz / f_sp, math.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), f_sp * m)


def mel_filterbank(samplingRate, wl, n_mels, fmin=0, fmax=None, mel_scale='htk', norm=None):
    """Triangular mel filterbank over the wl / 2 bins of a wl-point spectrum (bin j at j * samplingRate / wl), as a
    [n_mels, wl / 2] float64 array: torchaudio.functional.melscale_fbanks(wl // 2 + 1, fmin, fmax, n_mels,
    samplingRate, norm, mel_scale)[:wl // 2].T, without the dependency.  fmax defaults to samplingRate // 2.
    mel_scale: 'htk' or 'slaney'; norm: None or 'slaney' (each band scaled to unit area in Hz)."""
    if mel_scale not in ('htk', 'slaney'):
        raise ValueError("mel_scale must be 'htk' or 'slaney', not %r" % (mel_scale,))
    if norm not in (None, 'slaney'):
        raise ValueError("norm must be None or 'slaney', not %r" % (norm,))
    wl, n_mels = int(wl), int(n_mels)
    if wl < 4 or wl % 2 or n_mels < 1 or not samplingRate > 0:
        raise ValueError('need an even wl >= 4, n_mels >= 1 and a positive samplingRate')
    fmax = float(samplingRate // 2) if fmax is None else float(fmax)
    if not 0 <= fmin < fmax:
        raise ValueError('need 0 <= fmin < fmax (%r, %r)' % (fmin, fmax))
    freqs = np.arange(wl // 2, dtype=np.float64) * float(samplingRate) / wl
    m = np.linspace(_hz_to_mel(float(fmin), mel_scale), _hz_to_mel(fmax, mel_scale), n_mels + 2)
    f_pts = _mel_to_hz(m, mel_scale)
    f_diff = np.diff(f_pts)
    slopes = f_pts[None, :] - freqs[:, None]
    down = -slopes[:, :-2] / f_diff[:-1]
    up = slopes[:, 2:] / f_diff[1:]
    fb = np.maximum(0.0, np.minimum(down, up))
    if norm == 'slaney':
        fb = fb * (2.0 / (f_pts[2:n_mels + 2] - f_pts[:n_mels]))[None, :]
    return np.ascontiguousarray(fb.T)


def spectrogram_device(wave, lengths, samplingRate, windowLength=50, overlap=75, window='hamming', n_mels=None, fmin=0,
                       fmax=None, mel_scale='htk', norm=None, db=False, db_floor=1e-10, max_frames=None, stream=None):
    """Power (n_mels None) or mel spectrograms of the [n, T] float32 CUDA tensor `wave` that soundgen_batch_device
    returns, row c = its first lengths[c] samples.  Returns (spec, frames): spec [n, F, n_feat] float32 on the same
    device, frame k of row c at spec[c, k] (zeros past the row's frames), F = max_frames or the most frames of any
    row; frames: int64 CUDA tensor of the frames present per row.  n_feat = wl / 2 bins, or n_mels.
    Each row's window is wl = floor(windowLength / 1000 * sr / 2) * 2 points (soundgen.R:317) at its sampling rate
    sr: samplingRate is one value or one per row, and must be the rate the row was synthesised at.  A linear
    spectrogram needs one wl for all rows; mel features may mix rates (one library call per rate).
    lengths may be host or CUDA; a CUDA tensor is read back once, which synchronises with its stream.
    The result is ordered on `stream` (default: the device's current torch stream), with no other host wait."""
    import torch
    spec, frames = _spectrogram_device(wave, lengths, samplingRate, windowLength, overlap, window, n_mels, fmin, fmax,
                                       mel_scale, norm, db, db_floor, max_frames, stream)
    return spec, torch.as_tensor(frames, dtype=torch.int64).to(wave.device)


def _spectrogram_device(wave, lengths, samplingRate, windowLength, overlap, window, n_mels, fmin, fmax, mel_scale, norm,
                        db, db_floor, max_frames, stream):
    """spectrogram_device with the frames per row as a host array."""
    import torch
    if not (torch.is_tensor(wave) and wave.is_cuda and wave.dtype == torch.float32 and wave.dim() == 2):
        raise ValueError('wave must be a 2-D float32 CUDA tensor')
    if window not in _WINDOWS:
        raise ValueError("window must be 'hamming' or 'hanning', not %r" % (window,))
    n, T = wave.shape
    lens = (lengths.cpu().numpy() if torch.is_tensor(lengths) else np.asarray(lengths)).astype(np.int64).reshape(-1)
    if lens.shape != (n,) or np.any(lens < 0) or np.any(lens > T):
        raise ValueError('lengths needs one value in [0, %d] per row (%d)' % (T, n))
    sr = np.broadcast_to(np.asarray(samplingRate, dtype=np.float64).reshape(-1), (n,)) if n else np.zeros(0)
    if not np.all(np.isfinite(sr) & (sr > 0)):
        raise ValueError('samplingRate must be positive')
    wl = (np.floor(windowLength / 1000 * sr / 2) * 2).astype(np.int64)
    if max_frames is not None and int(max_frames) < 0:
        raise ValueError('max_frames must be non-negative')
    if n_mels is None:
        if np.unique(wl).size > 1:
            raise ValueError('a linear spectrogram needs one window length for all rows, not %s' % np.unique(wl))
        groups = [(np.arange(n), None)]
        n_feat = int(wl[0]) // 2 if n else 0
    else:
        if int(n_mels) < 1:
            raise ValueError('n_mels must be positive')
        groups = [(np.flatnonzero(sr == r), r) for r in np.unique(sr)]
        n_feat = int(n_mels)
    L = _abi.load()
    nc = np.array([L.sgb_spec_frames(int(l), int(w), float(overlap)) for l, w in zip(lens, wl)], dtype=np.int64)
    if np.any(nc < 0):
        raise SoundgenError(_abi.SGB_ERR_UNSUPPORTED, 'window of %s points / overlap %r cannot be analysed'
                            % (np.unique(wl[nc < 0]), overlap))
    F = int(max_frames) if max_frames is not None else int(nc.max(initial=0))
    spec = torch.empty((n, F, n_feat), dtype=torch.float32, device=wave.device)
    if n and F and n_feat:
        src = wave.contiguous()
        rows = np.arange(n, dtype=np.int64)
        for idx, r in groups:
            w = int(wl[idx[0]])
            bands = None if r is None else mel_filterbank(r, w, n_feat, fmin, fmax, mel_scale, norm)
            cap = np.zeros(n, dtype=np.int64)
            cap[idx] = F
            rows_spectrogram(wave.device.index, src, rows * T, lens, spec, rows * F * n_feat, cap, w, overlap, window,
                             bands, db, db_floor, stream)
    return spec, np.minimum(nc, F)



def dct_matrix(n_mfcc, n_mels, include_c0=True):
    """The orthonormal DCT-II that turns log-mel frames into MFCCs, as a float64 [n_mfcc, n_mels] array:
    D[k, b] = sqrt((2 - delta_k0) / n_mels) cos(pi k (2 b + 1) / (2 n_mels)) for k = 0 .. n_mfcc - 1, or for
    k = 1 .. n_mfcc with include_c0=False.  These are rows of scipy.fft.dct(eye(n_mels), type=2, norm='ortho',
    axis=0), and with c0 the matrix is torchaudio.functional.create_dct(n_mfcc, n_mels, 'ortho').T.  The rows
    k >= 1 sum to zero, so a constant frame (silence at the dB floor) has 0 in every coefficient but c0."""
    n_mfcc, n_mels, k0 = int(n_mfcc), int(n_mels), 0 if include_c0 else 1
    if n_mfcc < 1 or n_mels < 1 or k0 + n_mfcc > n_mels:
        raise ValueError('need 1 <= n_mfcc <= n_mels%s (%d, %d)' % ('' if include_c0 else ' - 1 without c0', n_mfcc,
                                                                    n_mels))
    k = np.arange(k0, k0 + n_mfcc, dtype=np.int64)[:, None]
    b = np.arange(n_mels, dtype=np.int64)[None, :]
    # the angle reduced exactly, in integers, to [0, 2 pi): k (2b + 1) mod 4 n_mels quarter-turns of pi / (2 n_mels)
    D = math.sqrt(2.0 / n_mels) * np.cos(math.pi * ((k * (2 * b + 1)) % (4 * n_mels)) / (2 * n_mels))
    if include_c0:
        D[0] = math.sqrt(1.0 / n_mels)
    return D


def rows_cepstra(device, src, src_off, frames, dst, dst_off, cap, matrix, deltas=0, delta_n=2, stream=None):
    """sgb_rows_cepstra (K11): cepstra c = matrix @ x of the frames the caller holds in the float32 CUDA tensor `src`
    (row c = frames[c] frames of n_in = matrix.shape[1] floats from element src_off[c], as rows_spectrogram writes
    them), followed by `deltas` (0, 1 or 2) orders of deltas over 2 delta_n + 1 frames with the row's edge frames
    replicated (torchaudio's compute_deltas over the row's own frames).  Row c of dst gets cap[c] frames of
    n_ceps (1 + deltas) floats, [c | delta | delta-delta], from element dst_off[c] on, zeros past the row's frames.
    Returns the frames written per row."""
    import torch
    so = np.ascontiguousarray(src_off, dtype=np.int64)
    fr = np.ascontiguousarray(frames, dtype=np.int64)
    if not (torch.is_tensor(src) and src.is_contiguous() and src.dtype == torch.float32) or so.shape != fr.shape \
            or so.ndim != 1:
        raise ValueError('src must be a contiguous float32 tensor, src_off and frames of one length')
    M = np.ascontiguousarray(matrix, dtype=np.float32)
    if M.ndim != 2 or M.size == 0:
        raise ValueError('matrix must be a non-empty [n_ceps, n_in] array, not %r' % (M.shape,))
    p = _abi.CepsParams()
    p.n_ceps, p.n_in, p.matrix = M.shape[0], M.shape[1], _ptr(M)
    p.delta_order, p.delta_n = int(deltas), int(delta_n)
    L = _abi.load()
    return _export(lambda o: L.sgb_rows_cepstra(int(device), src.data_ptr() or None, src.numel(), _ptr(so), _ptr(fr),
                                                fr.size, C.byref(p), C.byref(o)), fr.size, dst, dst_off, cap, stream,
                   'f32')


def mfcc_device(wave, lengths, samplingRate, n_mfcc=13, include_c0=True, deltas=0, delta_n=2, windowLength=50,
                overlap=75, window='hamming', n_mels=40, fmin=0, fmax=None, mel_scale='htk', norm=None, db_floor=1e-10,
                max_frames=None, stream=None):
    """MFCCs and their deltas of the [n, T] float32 CUDA tensor `wave` that soundgen_batch_device returns: the
    log-mel spectrogram of spectrogram_device(..., n_mels, db=True) (mixed sampling rates as there), projected on
    dct_matrix(n_mfcc, n_mels, include_c0) with `deltas` (0, 1 or 2) orders of deltas over 2 delta_n + 1 frames, in
    one call of K11 (rows_cepstra) over all rows.  Returns (feat, frames): feat [n, F, n_mfcc (1 + deltas)] float32,
    frame k of row c = [c | delta | delta-delta] at feat[c, k], zeros past the row's frames, F = max_frames or the
    most frames of any row; frames: int64 CUDA tensor of the frames present per row.  A row cut at max_frames is a
    bit-exact prefix of the whole row: its last deltas read the log-mel frames past the cut.  Ordered on `stream`
    (default: the device's current torch stream), with no host wait besides reading back a CUDA `lengths`."""
    import torch
    if int(deltas) not in (0, 1, 2) or not 1 <= int(delta_n) <= 8:
        raise ValueError('need deltas in 0, 1, 2 and delta_n in 1..8, not %r, %r' % (deltas, delta_n))
    if max_frames is not None and int(max_frames) < 0:
        raise ValueError('max_frames must be non-negative')
    if n_mels is None:
        raise ValueError('n_mels must be given')
    M = dct_matrix(n_mfcc, n_mels, include_c0).astype(np.float32)
    H = int(deltas) * int(delta_n)           # frames past the cut that the deltas before it read
    spec, nc = _spectrogram_device(wave, lengths, samplingRate, windowLength, overlap, window, int(n_mels), fmin, fmax,
                                   mel_scale, norm, True, db_floor, None if max_frames is None else int(max_frames) + H,
                                   stream)
    n, Fs, nm = spec.shape
    F = int(max_frames) if max_frames is not None else Fs
    n_out = M.shape[0] * (1 + int(deltas))
    feat = torch.empty((n, F, n_out), dtype=torch.float32, device=wave.device)
    if n and F:
        rows = np.arange(n, dtype=np.int64)
        rows_cepstra(wave.device.index, spec, rows * Fs * nm, nc, feat, rows * F * n_out, np.full(n, F, dtype=np.int64),
                     M, deltas, delta_n, stream)
        h = _stream_handle(stream, spec)
        if h != torch.cuda.current_stream(spec.device).cuda_stream:
            # spec goes back to the allocator here, on the current stream: keep it until K11 has read it on `stream`
            spec.record_stream(stream if isinstance(stream, torch.cuda.Stream)
                               else torch.cuda.ExternalStream(h, device=spec.device))
    return feat, torch.as_tensor(np.minimum(nc, F), dtype=torch.int64).to(wave.device)

def _torch_out_dtype(dtype):
    import torch
    if dtype == torch.float32:
        return 'f32'
    if dtype == torch.int16:
        return 'pcm16'
    raise ValueError('dtype must be torch.float32 or torch.int16 (PCM16), not %r' % (dtype,))


def soundgen_batch_device(calls, dtype=None, device=None, max_len=None, u_dtype=np.float64, f0=False):
    """soundgen_batch with the waveforms delivered on the GPU: returns (wave, lengths, status).
    wave: [n_calls, T] tensor on the device, rows padded with zeros, T = max_len (longer calls are cropped) or else
    the longest call; lengths: int64 CUDA tensor of the samples present per row; status: as soundgen_batch returns it.
    dtype: torch.float32 (the samples soundgen() returns) or torch.int16 (16-bit PCM as seewave::savewav writes it,
    normalised over the whole call, before any cropping).  device: CUDA device index (default: torch's current one).
    f0=True also returns the exact f0 track of every call (Batch.f0, K12a) as a fourth element: a [n_calls, T]
    float32 tensor aligned sample for sample with wave (same rounds, offsets and crop), f0 in Hz, 0 where unvoiced and
    in every row whose status is not 0.  The result is ordered on the device's current torch stream."""
    import torch
    fmt = _torch_out_dtype(torch.float32 if dtype is None else dtype)
    if max_len is not None and int(max_len) < 0:
        raise ValueError('max_len must be non-negative')
    L = _abi.load()
    if isinstance(device, (str, torch.device)):
        device = torch.device(device).index
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    device = int(device)
    _check(L.sgb_set_device(device))       # the handles below are made on this thread's current device
    fe = FrontEnd(u_dtype)
    rounds = []
    try:
        for kw in calls:
            fe.add(**kw)
        n = fe.n_calls
        # one handle per round: the next round would overwrite a handle's output, and T is known after the last one
        while True:
            desc, m = fe.round_begin()
            if m == 0:
                break
            bt = Batch()
            rounds.append(bt)
            bt.upload(desc)
            bt.run()
            bt.round_calls = fe.round_calls().copy()
            bt.seg_len = bt.lengths()
        status = fe.status()
    finally:
        fe.close()
    try:
        total = np.zeros(n, dtype=np.int64)
        for bt in rounds:
            np.add.at(total, bt.round_calls, bt.seg_len)
        T = int(max_len) if max_len is not None else int(total.max(initial=0))
        dev = torch.device('cuda', device)
        stream = torch.cuda.current_stream(dev)
        rows = np.arange(n, dtype=np.int64)
        last = np.full(n, -1)              # the last round each call took part in
        for r, bt in enumerate(rounds):
            last[bt.round_calls] = r
        if fmt == 'f32':
            wave = torch.empty((n, T), dtype=torch.float32, device=dev)
            if np.any(last < 0):           # a call that never reached the device: its row is written by nobody
                wave.zero_()
            tgt, base, width = wave, rows * T, np.full(n, T, dtype=np.int64)
        else:   # whole calls in float32 first (packed): PCM16 is normalised over the whole call
            wave = torch.empty((n, T), dtype=torch.int16, device=dev)
            base = (np.cumsum(total) - total).astype(np.int64)
            tgt, width = torch.empty(int(total.sum()), dtype=torch.float32, device=dev), total
        # a call's segment of round r lands behind its earlier segments; its last segment also writes the zero tail
        done = np.zeros(n, dtype=np.int64)
        for r, bt in enumerate(rounds):
            ci = bt.round_calls
            room = np.maximum(width[ci] - done[ci], 0)
            cap = np.where(last[ci] == r, room, np.minimum(bt.seg_len, room))
            bt.export(tgt, base[ci] + np.minimum(done[ci], width[ci]), cap, stream, 'f32')
            done[ci] += bt.seg_len
        if fmt == 'pcm16':
            rows_export(device, tgt, base, total, wave, rows * T, np.full(n, T, dtype=np.int64), stream, 'pcm16')
        if f0:                             # the f32 layout of wave: the same segments at the same places
            track = torch.empty((n, T), dtype=torch.float32, device=dev)
            if np.any(last < 0):
                track.zero_()
            done = np.zeros(n, dtype=np.int64)
            for r, bt in enumerate(rounds):
                ci = bt.round_calls
                room = np.maximum(T - done[ci], 0)
                cap = np.where(last[ci] == r, room, np.minimum(bt.seg_len, room))
                bt.f0(track, rows[ci] * T + np.minimum(done[ci], T), cap, stream)
                done[ci] += bt.seg_len
            failed = np.flatnonzero(np.asarray(status) != 0)    # also the calls the front-end failed: no voiced sample
            if failed.size:
                with torch.cuda.stream(stream):
                    track.index_fill_(0, torch.as_tensor(failed, device=dev), 0.0)
        lengths = torch.as_tensor(np.minimum(total, T), dtype=torch.int64).to(dev)
    finally:
        for bt in rounds:      # destroying a handle waits for its stream, i.e. for the export queued on it
            bt.close()
    return (wave, lengths, status, track) if f0 else (wave, lengths, status)


_CMP_METHODS = {'cor': _abi.SGB_CMP_COR, 'cosine': _abi.SGB_CMP_COSINE, 'dtw': _abi.SGB_CMP_DTW}


def _host_counts(x, n, hi, what):
    import torch
    v = (x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)).astype(np.int64).reshape(-1)
    if v.shape != (n,) or np.any(v < 0) or np.any(v > hi):
        raise ValueError('%s needs one value in [0, %d] per row (%d)' % (what, hi, n))
    return v


def compare_spectrograms(a, a_frames, b, b_frames, method='cor', pairs=None, pad=0.0, stream=None):
    """Similarity of spectrogram rows on the device (K10, sgb_rows_compare): a [n, F, n_feat] and b [m, F', n_feat]
    are float32 CUDA tensors as spectrogram_device returns them, a_frames / b_frames the frames present per row (host
    or CUDA; a CUDA tensor is read back once).  Row c of a is scored against row pairs[c] of b (default: row 0 when
    m == 1, else row c).  method: 'cor' (Pearson correlation), 'cosine' or 'dtw' (minus the normalised symmetric2 DTW
    distance); for cor and cosine the frames past the shorter row of a pair read as `pad`.  Higher is more similar;
    NaN for a row without frames, a constant side (cor) or an all-zero side (cosine).  Returns a float64 CUDA
    tensor [n], ordered on `stream` (default: the device's current torch stream) with no host wait."""
    import torch
    if method not in _CMP_METHODS:
        raise ValueError("method must be 'cor', 'cosine' or 'dtw', not %r" % (method,))
    for t, nm in ((a, 'a'), (b, 'b')):
        if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32 and t.dim() == 3 and t.is_contiguous()):
            raise ValueError('%s must be a contiguous [rows, frames, n_feat] float32 CUDA tensor' % nm)
    if a.device != b.device:
        raise ValueError('a and b must be on one device')
    n, Fa, nf = a.shape
    m, Fb, nfb = b.shape
    if nf != nfb or nf < 1:
        raise ValueError('a and b need the same n_feat >= 1, not %d and %d' % (nf, nfb))
    af = _host_counts(a_frames, n, Fa, 'a_frames')
    bf = _host_counts(b_frames, m, Fb, 'b_frames')
    if pairs is None:
        if m != 1 and m != n:
            raise ValueError('pairs is needed when b has neither one row nor one row per row of a')
        pairs = np.zeros(n) if m == 1 else np.arange(n)
    pr = np.asarray(pairs).reshape(-1)
    if pr.shape != (n,) or not np.all((pr >= 0) & (pr < m) & (pr == np.floor(pr))):
        raise ValueError('pairs needs one row index of b in [0, %d) per row of a (%d)' % (m, n))
    pr = pr.astype(np.int64)
    p = _abi.CompareParams()
    p.method, p.n_feat, p.pad = _CMP_METHODS[method], nf, float(pad)
    a_off = np.arange(n, dtype=np.int64) * Fa * nf
    b_off = np.ascontiguousarray(pr * Fb * nf)
    b_fr = np.ascontiguousarray(bf[pr])
    dst = torch.empty(n, dtype=torch.float64, device=a.device)
    L = _abi.load()
    _check(L.sgb_rows_compare(a.device.index, a.data_ptr() or None, a.numel(), b.data_ptr() or None, b.numel(),
                              _ptr(a_off), _ptr(af), _ptr(b_off), _ptr(b_fr), n, C.byref(p), dst.data_ptr() or None,
                              n, _stream_handle(stream, dst) or None))
    return dst


def param_range(name):
    """(default, low, high) of a scalar soundgen() argument as the front-end range-checks it (permittedValues,
    R/presets.R:22-79).  ValueError for a name it does not check."""
    out = np.zeros(3)
    if not isinstance(name, str) or _abi.load().sgb_param_range(name.encode(), _ptr(out)) != _abi.SGB_OK:
        raise ValueError('%r is not a range-checked scalar argument of soundgen()' % (name,))
    return float(out[0]), float(out[1]), float(out[2])


# arguments match_pars does not search: the sampling rate and window set the analysis, temperature the draws, and
# the counts of bouts and syllables change the structure of the call
_NOT_SEARCHED = ('samplingRate', 'windowLength', 'temperature', 'repeatBout', 'nSyl')


def _searched(pars):
    pars = [pars] if isinstance(pars, str) else list(pars)
    if not pars or len(set(pars)) != len(pars):
        raise ValueError('pars must name one or more distinct arguments')
    for nm in pars:
        if nm in _NOT_SEARCHED:
            raise ValueError('%s cannot be searched (not one of %s)' % (nm, ', '.join(_NOT_SEARCHED)))
        param_range(nm)
    return pars


def wiggle_pars(values, pars, prob_mutation=0.25, step_variance=0.1, rng=None):
    """One mutation of `values` (a dict holding every name of `pars`), drawn from the numpy Generator `rng` (or a
    seed): each name of pars changes with probability prob_mutation, and one chosen at random when none did, to a
    normal draw with mean its value and sd step_variance * (high - low), redrawn up to 100 times until it falls in
    [low, high] of param_range, then clipped.  Returns a new dict; the other entries are copied unchanged."""
    pars = _searched(pars)
    if not 0.0 <= float(prob_mutation) <= 1.0 or not float(step_variance) > 0.0:
        raise ValueError('need 0 <= prob_mutation <= 1 and step_variance > 0')
    rng = rng if isinstance(rng, np.random.Generator) else np.random.default_rng(rng)
    out = dict(values)
    mutate = rng.random(len(pars)) < float(prob_mutation)
    if not mutate.any():
        mutate[rng.integers(len(pars))] = True
    for nm, mu in zip(pars, mutate):
        if not mu:
            continue
        _, lo, hi = param_range(nm)
        mean, sd = float(values[nm]), float(step_variance) * (hi - lo)
        for _ in range(100):
            v = float(rng.normal(mean, sd))
            if lo <= v <= hi:
                break
        out[nm] = min(max(v, lo), hi)
    return out


_DB_FLOOR = 1e-10


def match_pars(target, samplingRate, pars, base=None, n_candidates=64, max_iter=50, prob_mutation=0.25,
               step_variance=0.1, method='cor', min_delta=0.0, windowLength=40, overlap=50, n_mels=64, seed=0,
               features='mel', n_mfcc=13, deltas=0):
    """Searches soundgen() arguments for a call that sounds like `target` (a 1-D float32 waveform, numpy or CUDA, at
    samplingRate): a hill-climb in the manner of the reference's matchPars that tries n_candidates mutations of the
    current best per step on the GPU.  base: the fixed arguments (temperature defaults to 0); pars: the scalar
    arguments searched, starting from their values in base (or soundgen()'s defaults).  Each step draws the
    candidates with wiggle_pars, synthesises them at samplingRate (soundgen_batch_device), takes their log-mel
    spectrograms as the target's (spectrogram_device with windowLength, overlap, n_mels, db=True) and scores them
    against it (compare_spectrograms with `method`; missing frames read as the dB floor, i.e. silence).  A candidate
    with a non-zero status or a NaN score counts as -inf.  The best candidate replaces the current one when its score
    beats the current score by more than min_delta.
    Returns (best_kwargs, best_score, history): history[0] is the starting point, history[k] step k, each a dict with
    'score' (the step's best), 'accepted', 'values' ([candidates, len(pars)] array of the values tried) and 'best'
    (the current score after the step).  The same seed, inputs and n_candidates give the same history, bit for bit.
    features='mfcc' scores MFCCs instead: mfcc_device with the same windowLength, overlap and n_mels, n_mfcc
    coefficients without c0 and `deltas` orders of deltas, missing frames read as 0 (silence: the DCT rows without
    c0 sum to zero, so a frame at the dB floor has 0 in every coefficient and delta).
    This is not R's matchPars: the draws come from numpy's generator, not R's stream, and the features are this
    library's log-mel spectrograms or MFCCs, not tuneR::melfcc."""
    import torch
    pars = _searched(pars)
    if method not in _CMP_METHODS:
        raise ValueError("method must be 'cor', 'cosine' or 'dtw', not %r" % (method,))
    if int(n_candidates) < 1 or int(max_iter) < 0:
        raise ValueError('need n_candidates >= 1 and max_iter >= 0')
    if features not in ('mel', 'mfcc'):
        raise ValueError("features must be 'mel' or 'mfcc', not %r" % (features,))
    if features == 'mfcc':
        dct_matrix(n_mfcc, n_mels, include_c0=False)
        if int(deltas) not in (0, 1, 2):
            raise ValueError('deltas must be 0, 1 or 2, not %r' % (deltas,))
    sr = float(samplingRate)
    kw = dict(temperature=0)
    kw.update(base or {})
    if kw.get('samplingRate', sr) != sr:
        raise ValueError('base sets samplingRate %r, the target is at %r' % (kw['samplingRate'], sr))
    kw['samplingRate'] = sr
    _, lo, hi = param_range('samplingRate')
    if not lo <= sr <= hi and kw.get('invalidArgAction', 'adjust') != 'ignore':
        raise ValueError("samplingRate %g is outside [%g, %g]: the front-end would not synthesise at it unless base "
                         "sets invalidArgAction='ignore'" % (sr, lo, hi))
    if torch.is_tensor(target):
        dev = target.device if target.is_cuda else torch.device('cuda', torch.cuda.current_device())
        x = target.to(dev, torch.float32)
    else:
        dev = torch.device('cuda', torch.cuda.current_device())
        x = torch.as_tensor(np.asarray(target, dtype=np.float32), device=dev)
    if x.dim() != 1:
        raise ValueError('target must be a 1-D waveform')
    if features == 'mel':
        spec_kw = dict(windowLength=windowLength, overlap=overlap, n_mels=int(n_mels), db=True, db_floor=_DB_FLOOR)
        feats, pad = spectrogram_device, 10.0 * math.log10(_DB_FLOOR)
    else:
        spec_kw = dict(windowLength=windowLength, overlap=overlap, n_mels=int(n_mels), n_mfcc=int(n_mfcc),
                       include_c0=False, deltas=int(deltas), db_floor=_DB_FLOOR)
        feats, pad = mfcc_device, 0.0
    tgt, tgt_frames = feats(x.reshape(1, -1).contiguous(), [x.numel()], sr, **spec_kw)

    def best_of(cands):
        wave, lengths, status = soundgen_batch_device([dict(kw, **c) for c in cands], device=dev.index)
        spec, frames = feats(wave, lengths, sr, **spec_kw)
        s = compare_spectrograms(spec, frames, tgt, tgt_frames, method, pad=pad)
        bad = torch.as_tensor(np.asarray(status) != 0, device=dev) | torch.isnan(s)
        s = torch.where(bad, torch.full_like(s, -math.inf), s)
        i = torch.argmax(s)                       # the first of equal maxima
        got = torch.stack((s[i], i.to(torch.float64))).cpu()
        return float(got[0]), int(got[1])

    cur = {nm: float(kw.get(nm, SOUNDGEN_DEFAULTS[nm])) for nm in pars}
    best = best_of([cur])[0]
    history = [dict(score=best, accepted=True, values=np.array([[cur[nm] for nm in pars]]), best=best)]
    rng = np.random.default_rng(seed)
    for _ in range(int(max_iter)):
        cands = [wiggle_pars(cur, pars, prob_mutation, step_variance, rng) for _ in range(int(n_candidates))]
        s, i = best_of(cands)
        accepted = s > best + min_delta
        if accepted:
            cur, best = cands[i], s
        history.append(dict(score=s, accepted=accepted, values=np.array([[c[nm] for nm in pars] for c in cands]),
                            best=best))
    return dict(kw, **cur), best, history


class PipelinedBatches:
    """Several sub-batches, each with its own handle / CUDA stream, driven as a three-stage software
    pipeline: one thread uploads (H2D copy engine), `runners` threads run the kernels (two, so that the
    latency-bound control / joining stages of one sub-batch overlap the FMA-bound synthesis of another
    and the host-side layout of one overlaps the kernels of the other), one thread fetches (D2H copy
    engine).  ctypes releases the GIL during the library calls.  Independent sounds need no ordering,
    so no work is skipped and nothing is shared between the sub-batches."""

    def __init__(self, descs=None, runners=2, sources=None, fe_threads=2, device_out=None):
        """`descs`: prebuilt batch descriptions, one per sub-batch -- or `sources`: one `ArgArray` per sub-batch, in
        which case every step starts from the argument lists: `fe_threads` threads run the library's host
        front-end (`sgb_frontend_add_many` + `round_begin`) for a sub-batch before it is uploaded.
        `device_out`: None (results are fetched to host memory) or dict(dtype=torch.float32 | torch.int16,
        max_len=None | T, device=None | index): the fetch stage exports every sub-batch into CUDA tensors allocated
        once, `results[i] = (wave [n_i, T], lengths)`, ordered on `streams[i]` (one consumer stream per sub-batch).
        A step overwrites the tensors of the step before: consume them on `streams[i]` (or copy them) first."""
        self.sources = list(sources) if sources is not None else None
        if self.sources is not None:
            self.fes = [FrontEnd(src.u_dtype) for src in self.sources]
            descs = [None] * len(self.sources)
            self._pinned = [dict() for _ in self.sources]
        self.fe_threads = max(1, int(fe_threads))
        self.descs = list(descs)
        self.batches = [Batch() for _ in self.descs]
        self.outs = [None] * len(self.descs)
        self.runners = max(1, int(runners))
        self.results = [None] * len(self.descs)
        self.device_out = None
        if device_out is not None:
            import torch
            do = dict(device_out)
            self.device_out = dict(fmt=_torch_out_dtype(do.pop('dtype', torch.float32)), max_len=do.pop('max_len', None),
                                   device=do.pop('device', None))
            if do:
                raise TypeError('device_out: unknown keys %s' % sorted(do))
            if self.device_out['device'] is None:
                self.device_out['device'] = torch.cuda.current_device()
            dev = torch.device('cuda', int(self.device_out['device']))
            self.streams = [torch.cuda.Stream(dev) for _ in self.descs]
            self.waves = [None] * len(self.descs)

    def _export(self, i):
        """device_out: sub-batch i -> its [n_i, T] tensor, ordered on streams[i]"""
        import torch
        bt, s, do = self.batches[i], self.streams[i], self.device_out
        lens = bt.lengths()
        T = int(do['max_len']) if do['max_len'] is not None else int(lens.max(initial=0))
        w = self.waves[i]
        with torch.cuda.stream(s):
            if w is None or w.shape != (lens.size, T):      # allocated once (again only if a longer call appears)
                w = torch.empty((lens.size, T), dtype=torch.float32 if do['fmt'] == 'f32' else torch.int16,
                                device=s.device)
                self.waves[i] = w
            n = lens.size
            bt.export(w, np.arange(n, dtype=np.int64) * T, np.full(n, T, dtype=np.int64), s, do['fmt'])
            lengths = torch.as_tensor(np.minimum(lens, T), dtype=torch.int64).to(s.device, non_blocking=True)
        return w, lengths

    def _fetch(self, i, dtype):
        bt = self.batches[i]
        if self.outs[i] is not None and self.outs[i].dtype != np.dtype(dtype):
            _abi.load().sgb_unpin(self.outs[i].ctypes.data)     # a registration must not outlive its array
            self.outs[i] = None
        if self.outs[i] is None:
            n = int(bt.lengths().sum())
            self.outs[i] = np.zeros(max(n, 1), dtype=dtype)
            _abi.load().sgb_pin(self.outs[i].ctypes.data, self.outs[i].nbytes)
        return bt.fetch(dtype, out=self.outs[i])

    def run_steps(self, nsteps=1, dtype=np.float32, transfer=True):
        """`nsteps` passes over all sub-batches.  transfer=True: every pass uploads the inputs and
        fetches every waveform (end to end); False: inputs stay resident, outputs stay on the device.
        A sub-batch is re-uploaded for the next pass only after its previous results were fetched."""
        import queue
        import threading
        n = len(self.descs)
        q_run, q_fetch = queue.Queue(), queue.Queue()
        free = [threading.Semaphore(1) for _ in range(n)]     # handle i is idle
        err = []
        abort = threading.Event()

        class _Abort(Exception):
            pass

        def q_get(q):
            while True:
                try:
                    return q.get(timeout=0.2)
                except queue.Empty:
                    if abort.is_set():
                        raise _Abort()

        def acquire(sem):
            while not sem.acquire(timeout=0.2):
                if abort.is_set():
                    raise _Abort()

        def guard(f):
            def g():
                try:
                    f()
                except _Abort:
                    pass
                except Exception as e:   # surfaced to the caller below; the other stages stop waiting
                    err.append(e)
                    abort.set()
            return g

        q_fe, q_up = queue.Queue(), queue.Queue()

        def front_end():
            while True:
                i = q_get(q_fe)
                if i is None:
                    q_up.put(None)
                    return
                acquire(free[i])
                fe = self.fes[i]
                fe.clear()
                fe.add_many(self.sources[i])
                d, _ = fe.round_begin()
                self._pin_pools(i, d)
                self.descs[i] = d
                q_up.put(i)

        def uploader():
            if self.sources is not None:
                done = 0
                while done < self.fe_threads:
                    i = q_get(q_up)
                    if i is None:
                        done += 1
                        continue
                    self.batches[i].upload(self.descs[i])
                    q_run.put(i)
            else:
                for s in range(nsteps):
                    for i in range(n):
                        acquire(free[i])
                        if transfer or self.batches[i].desc is None:
                            self.batches[i].upload(self.descs[i])
                        q_run.put(i)
            for _ in range(self.runners):
                q_run.put(None)

        def runner():
            while True:
                i = q_get(q_run)
                if i is None:
                    q_fetch.put(None)
                    return
                self.batches[i].run()
                q_fetch.put(i)

        def fetcher():
            done = 0
            while done < self.runners:
                i = q_get(q_fetch)
                if i is None:
                    done += 1
                    continue
                if transfer:
                    self.results[i] = self._export(i) if self.device_out is not None else self._fetch(i, dtype)
                free[i].release()

        th = [threading.Thread(target=guard(uploader))] + \
             [threading.Thread(target=guard(runner)) for _ in range(self.runners)] + \
             [threading.Thread(target=guard(fetcher))]
        if self.sources is not None:
            for s_ in range(nsteps):
                for i in range(n):
                    q_fe.put(i)
            for _ in range(self.fe_threads):
                q_fe.put(None)
            th += [threading.Thread(target=guard(front_end)) for _ in range(self.fe_threads)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if err:
            raise err[0]

    def _pin_pools(self, i, d):
        """Page-locks the pools of a description the front-end just rebuilt, unless they sit where they sat last
        time (cleared vectors keep their storage, so from the second step on this is a dictionary lookup)."""
        L = _abi.load()
        cur = {}
        for k, a in d._keep.items():
            if a.size:
                cur[k] = (a.ctypes.data, a.nbytes)
        old = self._pinned[i]
        for k, v in old.items():
            if cur.get(k) != v:
                L.sgb_unpin(v[0])
        for k, v in cur.items():
            if old.get(k) != v:
                _check(L.sgb_pin(v[0], v[1]))
        self._pinned[i] = cur

    def step(self, dtype=np.float32):
        """upload + run + fetch of every sub-batch; returns the per-call waveforms in order."""
        self.run_steps(1, dtype=dtype, transfer=True)
        return [w for r in self.results for w in r]

    def close(self):
        for b in self.batches:
            b.close()
        for o in self.outs:            # a registration must not outlive the array it covers
            if o is not None:
                _abi.load().sgb_unpin(o.ctypes.data)
        self.outs = [None] * len(self.descs)
        if self.sources is not None:
            for pm in self._pinned:
                for v in pm.values():
                    _abi.load().sgb_unpin(v[0])
            self._pinned = [dict() for _ in self.sources]
            for fe in self.fes:
                fe.close()


def pin_desc(desc, pin=True):
    """Page-locks (or releases) the host pools of a built batch description so that its uploads are
    truly asynchronous.  Unpin before the description is garbage-collected."""
    L = _abi.load()
    for k in ('pitch', 'anchors', 'formants', 'z', 'u', 'pre'):
        a = desc._keep[k]
        if a.size:
            _check(L.sgb_pin(a.ctypes.data, a.nbytes) if pin else L.sgb_unpin(a.ctypes.data))


def generateHarmonics(pitch, attackLen=50, nonlinBalance=0, nonlinDep=0, jitterDep=0, jitterLen=1,
                      vibratoFreq=100, vibratoDep=0, shimmerDep=0, creakyBreathy=0, rolloff=-18,
                      rolloffOct=-2, rolloffKHz=-6, rolloffParab=0, rolloffParabHarm=3, rolloffLip=6,
                      rolloff_perAmpl=12, temperature=0, pitchDriftDep=.5, pitchDriftFreq=.125,
                      randomWalk_trendStrength=.5, shortestEpoch=300, subFreq=100, subDep=0, amDep=0,
                      amFreq=30, amplAnchors=None, overlap=75, samplingRate=16000, pitchFloor=75,
                      pitchCeiling=3500, pitchSamplingRate=3500, throwaway=-120, z=None,
                      contour_method='loess', want_artefacts=False):
    """generateHarmonics() (R/source.R:173-205).  `z`: the syllable's normal stream."""
    pars = dict(locals())
    for k in ('pitch', 'z', 'amplAnchors', 'contour_method', 'want_artefacts', 'nonlinDep', 'creakyBreathy',
              'rolloffLip', 'amDep', 'amFreq', 'overlap'):
        pars.pop(k)
    bb = BatchBuilder()
    bb.add_syllable(pitch, z=z, amplAnchors=amplAnchors, contour_method=contour_method, **pars)
    env = bb.add_envelope(None, samplingRate=samplingRate)
    wl = int(math.floor(50 / 1000 * samplingRate / 2) * 2)
    bb.add_bout(0, 1, 0, 0, env, False, wl, samplingRate=samplingRate, throwaway=throwaway)
    bb.add_call(0, 1)
    bt = Batch()
    bt.upload(bb.build())
    bt.run()
    art = bt.artefacts(0)
    if art['status'] == _abi.SGB_ERR_SYNTH:
        raise SoundgenError(art['status'], 'Failed to generate the new syllable!')
    if art['status'] != 0:
        raise SoundgenError(art['status'], 'generateHarmonics failed')
    y = bt.syllable(0).copy()
    bt.close()
    return (y, art) if want_artefacts else y


def generateNoise(len, noiseAnchors=((0, 300), (-120, -120)), rolloffNoise=-6, attackLen=10,
                  windowLength_points=1024, samplingRate=16000, overlap=75, throwaway=-120, filterNoise=None,
                  u=None, strength=None, contour_method='loess'):
    """generateNoise() (R/source.R:57-68).  `u`: the runif(nr * nc) draws; filterNoise:
    None or an (nr x k) matrix (as returned by getSpectralEnvelope).  `contour_method` smooths noiseAnchors."""
    bb = BatchBuilder()
    bb.add_silent_syllable(8)
    env = bb.add_envelope(None, samplingRate=samplingRate)
    env_n = -1
    if filterNoise is not None:
        fm = np.asarray(filterNoise, dtype=np.float64)
        if fm.shape[0] != int(windowLength_points) // 2:
            raise ValueError('filterNoise must have windowLength_points / 2 rows')
        env_n = bb.add_envelope_matrix(fm, samplingRate=samplingRate)
    bb.add_noise(len, noiseAnchors, u, rolloffNoise=rolloffNoise, attackLen=attackLen,
                 windowLength_points=windowLength_points, samplingRate=samplingRate, overlap=overlap,
                 insertion=1, mix=0, strength=strength, env_id=env_n, contour_method=contour_method)
    bb.add_bout(0, 1, 0, 1, env, False, max(4, int(windowLength_points)), samplingRate=samplingRate,
                throwaway=throwaway)
    bb.add_call(0, 1)
    bt = Batch()
    bt.upload(bb.build())
    bt.run()
    y = bt.noise(0, len).copy()
    bt.close()
    return y


def getRolloff(pitch_per_gc=(440,), nHarmonics=100, rolloff=-12, rolloffOct=-2, rolloffParab=0,
               rolloffParabHarm=2, rolloffParabCeiling=None, rolloffKHz=-6, baseline=200, throwaway=-120,
               samplingRate=16000, plot=False):
    """getRolloff() (R/sourceSpectrum.R:71-82): matrix rows x nGC, rownames 1..rows."""
    L = _abi.load()
    p = np.ascontiguousarray(np.atleast_1d(pitch_per_gc), dtype=np.float64)
    v = lambda a: np.ascontiguousarray(np.atleast_1d(a), dtype=np.float64)
    ro, roct, rk = v(rolloff), v(rolloffOct), v(rolloffKHz)
    out = np.zeros(int(nHarmonics) * p.size)
    rows = C.c_int32()
    _check(L.sgb_get_rolloff(_ptr(p), p.size, int(nHarmonics), _ptr(ro), ro.size, _ptr(roct), roct.size,
                             _ptr(rk), rk.size, float(rolloffParab), float(rolloffParabHarm),
                             -1.0 if rolloffParabCeiling is None else float(rolloffParabCeiling),
                             float(baseline), float(throwaway), float(samplingRate), _ptr(out), C.byref(rows)))
    m = out.reshape(p.size, int(nHarmonics)).T
    return m[:rows.value, :].copy()


def getSpectralEnvelope(nr, nc, formants=None, formantDep=1, rolloffLip=6, mouthAnchors=None,
                        mouthOpenThres=0, openMouthBoost=0, vocalTract=None, temperature=0, formDrift=.3,
                        formDisp=.2, formantDepStoch=30, smoothLinearFactor=1, samplingRate=16000,
                        speedSound=35400, plot=False, formants_upsampled=None, contour_method='loess'):
    """getSpectralEnvelope() (R/sourceSpectrum.R:261-283), deterministic part; with
    temperature > 0 pass the host-drawn tracks as `formants_upsampled`.  `contour_method` smooths mouthAnchors."""
    if temperature > 0 and formants_upsampled is None:
        raise NotImplementedError('stochastic formants are drawn on the host from R\'s RNG')
    L = _abi.load()
    bb = BatchBuilder()
    eid = bb.add_envelope(formants, formantDep=formantDep, rolloffLip=rolloffLip, mouthAnchors=mouthAnchors,
                          mouthOpenThres=mouthOpenThres, openMouthBoost=openMouthBoost, vocalTract=vocalTract,
                          samplingRate=samplingRate, speedSound=speedSound,
                          smoothLinearFactor=smoothLinearFactor, tracks=formants_upsampled,
                          contour_method=contour_method)
    e = bb.envs[eid]
    fm = np.ascontiguousarray(np.concatenate(bb.formants)) if bb.formants else np.zeros(4)
    fn = np.array([r.n for r in bb.frefs], dtype=np.int32) if bb.frefs else np.zeros(1, dtype=np.int32)
    an = np.ascontiguousarray(np.concatenate(bb.anchors)) if bb.anchors else np.zeros(2)
    out = np.zeros(int(nr) * int(nc))
    _check(L.sgb_get_spectral_envelope(int(nr), int(nc), C.byref(e), _ptr(fm), _ptr(fn), _ptr(an), _ptr(out)))
    return out.reshape(int(nc), int(nr)).T.copy()


def filter_sound(sound, spectralEnvelope, windowLength_points, overlap=75):
    """The STFT -> envelope -> ISTFT -> /max block of soundgen() (R/soundgen.R:743-807)."""
    L = _abi.load()
    s = np.ascontiguousarray(sound, dtype=np.float64)
    env = np.asarray(spectralEnvelope, dtype=np.float64)
    if env.ndim == 1:
        env = env[:, None]
    e = np.ascontiguousarray(env.T).ravel()   # column-major
    n = L.sgb_filter_len(s.size, int(windowLength_points), float(overlap))
    if n < 0:
        raise SoundgenError(-1, 'sound too short')
    out = np.zeros(n)
    _check(L.sgb_filter(_ptr(s), s.size, _ptr(e), env.shape[1], int(windowLength_points), float(overlap),
                        _ptr(out), out.size))
    return out
