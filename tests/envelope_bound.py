"""Float64 reference and per-element error bound of K4, the spectral envelope of getSpectralEnvelope
(R/sourceSpectrum.R:261-566), as k_envelope (kernels_env.cu) computes it.  Test infrastructure only.

The reference is the oracle's so.getSpectralEnvelope in float64, which also reports (`terms`) every gamma bump of
every column in bins (formant f: mode mg, width sdg, amplitude a), the mouth opening and its binary mask.  For bin
x = r + 1 of column c, with shape = mg^2 / sdg^2, rate = mg / sdg^2 and ref = the log-density at the integer arg-max,

    ld_f = (shape - 1) log x - rate x - ref,    t_f = a_f e^{ld_f}  (ld_f <= 0),
    v = formantDep sum_f t_f,   L = rolloffLip mouth_bin log2 x,   W = (v + L) boost,   y = 2^(W / 10),

boost = 2^(mouth_open openMouthBoost / 10).  An error dW in W is a relative error (ln 2 / 10) dW of y.

The bound (u = 2^-24, e = 2^-53; S = sum_f |t_f|; n = the column's bump count: the formants, plus the nasal pole and
zero in a closed-mouth column):

* ld_f in FP64, in the kernel and the reference alike: the two log-density terms cancel near the mode, so the error
  scales with their size M_f = |shape - 1| (log x + log x_ref) + rate (x + x_ref): the products, the differences,
  the 1-ulp log of either side and the FP64 shape / rate each add a few e M_f; the inputs (device spline tracks,
  device mouth contour, host-drawn stochastic tracks) agree with the oracle's to D = 64 e relatively, which moves mg
  and sdg and so ld by <= 4 D M_f (shape is quadratic in them) and a by D; D = 0 where the kernel reads the given
  values themselves.  dld_f <= (6 e + 4 D) M_f + e |ld_f| + D.
* FP32 path (k_envelope<float>): (float)ld_f rounds once (u |ld_f|), expf has <= 2 ulp (4u), (float)a_f one rounding
  (u).  The fmaf chain: step k rounds P_k = P_{k-1} + t_k, an error <= min(u |P_k|, |t_k|), so the chain adds
  A = sum_k min(u |P_k|, |t_k|) (<= n u S, far less where most bumps are negligible at the bin).
  dv <= |formantDep| (sum_f |t_f| (dld_f + u |ld_f| + 5u) + A) + 2u |v|; L from (float)rolloffLip and (float)(log x log2 e): <= 3u |L|; the sum, (float)boost and the
  product: 3u |W|, and the division by 10: u |W| / 10.  exp2f: <= 2 ulp of y (4u relative).
      rel32 = (ln 2 / 10) (boost (dv + 3u |L|) + 3.1u |W|) + 4u   (to first order; the second order is added)
* FP64 path (k_envelope<double>, the stand-alone getSpectralEnvelope): the same with e for u (no FMA, -fmad=false:
  the product's rounding joins the 5e per term) and 1-ulp exp / exp2 on both sides.

The bound is element by element; the tests hold it tight as well (bound32 <= 3e-5 over the corpus: filters of 62
and more formants reach 1.8e-5 and 2.5e-5) so that a loose bound cannot hide an error.  The FP64 bound is dominated by
the cancellation term 6e M_f: below 1e-9 where no formant is very narrow and there are at most a few dozen formants,
up to 2e-8 with hundreds of formants, and 6e-7 for the 0.2 Hz formant of the corpus; the host test holds it to those
ceilings.
"""
import contextlib
import math

import numpy as np

from oracle import soundgen_oracle as so

U32 = 2.0 ** -24
U64 = 2.0 ** -53
D_IN = 64 * U64         # relative agreement of the inputs (device tracks and mouth contour) with the oracle's


@contextlib.contextmanager
def capture():
    """Records every so.getSpectralEnvelope call (the oracle's soundgen calls it for each filtered noise and then
    for the main filter of each bout that is not bypassed) as dict(args, kwargs, env, terms), in call order."""
    records = []
    orig = so.getSpectralEnvelope

    def wrapped(*a, **kw):
        terms = {}
        env = orig(*a, terms=terms, **kw)
        records.append(dict(args=a, kwargs=kw, env=env, terms=terms))
        return env
    so.getSpectralEnvelope = wrapped
    try:
        yield records
    finally:
        so.getSpectralEnvelope = orig


def reference(nr, nc, **kw):
    """(envelope, terms) of so.getSpectralEnvelope."""
    terms = {}
    env = so.getSpectralEnvelope(nr, nc, terms=terms, **kw)
    return env, terms


def _parts(terms, nr, u):
    """Per element (nr x nc): S, sum |t| dld, sum |t| |ld|, the accumulation bound A, v, L, W, boost."""
    d_in = D_IN if terms['smoothed'] else 0.0
    bins = terms['bins']
    mb = np.asarray(terms['mouth_bin'], dtype=np.float64)
    mo = np.asarray(terms['mouth_open'], dtype=np.float64)
    nc = mb.size
    x = np.arange(1, nr + 1, dtype=np.float64)[:, None]
    lx = np.log(x)
    S = np.zeros((nr, nc))
    Td = np.zeros((nr, nc))
    Tl = np.zeros((nr, nc))
    A = np.zeros((nr, nc))
    v = np.zeros((nr, nc))
    nasal = bool(np.any(mb == 0))
    F = len(bins) - (2 if nasal else 0)
    for k, f in enumerate(bins):
        mg = f[:, 1]
        sdg = f[:, 3].copy()
        sdg[sdg == 0] = 1
        shape = mg ** 2 / sdg ** 2
        rate = mg / sdg ** 2
        logd = (shape - 1) * lx - rate * x
        iref = np.argmax(logd, axis=0)
        xr = (iref + 1).astype(np.float64)
        ld = logd - logd[iref, np.arange(nc)]
        a = f[:, 2]
        if k >= F:       # the nasal pole and zero exist in closed-mouth columns only
            a = np.where(mb == 0, a, 0.0)
        t = np.abs(a) * np.exp(ld)
        M = np.abs(shape - 1) * (lx + np.log(xr)) + rate * (x + xr)
        dld = (6 * U64 + 4 * d_in) * M + U64 * np.abs(ld) + d_in
        S += t
        Td += t * dld
        Tl += t * np.abs(ld)
        v += a * np.exp(ld)
        A += np.minimum(u * np.abs(v), t)        # rounding P + t errs by <= u |P + t| and by <= |t|
    fd = float(terms['formantDep'])
    v = v * fd
    L = float(terms['rolloffLip']) * np.log2(x) * mb
    boost = 2.0 ** (mo * float(terms['openMouthBoost']) / 10)
    W = (v + L) * boost
    return dict(S=S, Td=Td, Tl=Tl, A=A, v=v, L=L, W=W, boost=boost, fd=abs(fd),
                dboost=d_in * np.abs(mo * float(terms['openMouthBoost'])) * math.log(2) / 10)


def bound(terms, nr, fp32=True):
    """Per-element bound (nr x nc) of |y_kernel - y_ref| / y_ref for the FP32 (or FP64) path."""
    u = U32 if fp32 else U64
    p = _parts(terms, nr, u)
    if fp32:
        dv = p['fd'] * (p['Td'] + u * p['Tl'] + 5 * u * p['S'] + p['A']) + 2 * u * np.abs(p['v'])
    else:
        dv = p['fd'] * (p['Td'] + 5 * u * p['S'] + p['A']) + 2 * u * np.abs(p['v'])
    dW = p['boost'] * (dv + 3 * u * np.abs(p['L'])) + (3.1 * u + p['dboost']) * np.abs(p['W'])
    g = math.log(2) / 10 * dW
    return np.expm1(g) + (4 * u if fp32 else 4 * U64) * (1 + g)


def kernel_f32(terms, nr):
    """k_envelope<float>'s arithmetic in numpy, operation by operation (host check of the bound): FP64 ld, then FP32
    expf, fmaf chain, formantDep, lip term, boost and exp2f."""
    bins = terms['bins']
    mb = np.asarray(terms['mouth_bin'], dtype=np.float64)
    mo = np.asarray(terms['mouth_open'], dtype=np.float64)
    nc = mb.size
    nasal = bool(np.any(mb == 0))
    F = len(bins) - (2 if nasal else 0)
    x = np.arange(1, nr + 1, dtype=np.float64)
    lx = np.log(x)
    out = np.zeros((nr, nc), dtype=np.float32)
    for c in range(nc):
        n = F + (2 if mb[c] == 0 else 0)
        v = np.zeros(nr, dtype=np.float32)
        for f in bins[:n]:
            mg, sdg, a = f[c, 1], f[c, 3], f[c, 2]
            sdg = 1.0 if sdg == 0 else sdg
            shape, rate = mg * mg / (sdg * sdg), mg / (sdg * sdg)
            xs = 1.0
            if shape > 1:
                mode = (shape - 1) / rate
                lo, hi = min(max(math.floor(mode), 1.0), nr), min(max(math.ceil(mode), 1.0), nr)
                la, lb = (shape - 1) * math.log(lo) - rate * lo, (shape - 1) * math.log(hi) - rate * hi
                xs = hi if lb > la else lo
            ref = (shape - 1) * math.log(xs) - rate * xs
            ld = (shape - 1) * lx - rate * x - ref
            e = np.exp(ld.astype(np.float32))
            v = (e.astype(np.float64) * np.float64(np.float32(a)) + v.astype(np.float64)).astype(np.float32)   # fmaf
        v = v * np.float32(terms['formantDep'])
        lip = np.float32(float(terms['rolloffLip']) * mb[c])
        fboost = np.float32(2.0 ** (mo[c] * float(terms['openMouthBoost']) / 10))
        v = (v + lip * (lx * 1.4426950408889634).astype(np.float32)) * fboost
        out[:, c] = np.exp2(v / np.float32(10))
    return out


def _formants(n, seed, lo=300.0, hi=7500.0, amp=1.0):
    r = np.random.default_rng(seed)
    fr = np.sort(r.uniform(lo, hi, n))
    return [np.array([[0, f, amp * r.uniform(10, 40), r.uniform(50, 300)]]) for f in fr]


def _moving(points, seed):
    r = np.random.default_rng(seed)
    out = []
    for k, n in enumerate(points):
        t = np.linspace(0, 1, n)
        out.append(np.column_stack([t, r.uniform(400 + 900 * k, 900 + 900 * k, n), r.uniform(10, 40, n),
                                    r.uniform(60, 250, n)]))
    return out


def _tracks(nf, nc, seed):
    """stochastic-looking formant tracks (nc rows of time, freq, amp, width each), given literally"""
    r = np.random.default_rng(seed)
    out = []
    for k in range(nf):
        walk = 1 + 0.05 * np.cumsum(r.standard_normal(nc)) / np.sqrt(nc)
        out.append(np.column_stack([np.zeros(nc), (600 + 1100 * k) * walk, 30 * walk, 120 * walk]))
    return out


CLOSED = (np.array([0., 1]), np.array([0., 0]))
# (name, nr, nc, getSpectralEnvelope arguments): the edges of K4 (formant count and its 32-lane loop, widths,
# frequencies, mouth, track kinds, sizes)
CASES = [
    ('F0 lip only', 400, 1, dict(formants=None)),
    ('schwa', 400, 1, dict(formants=None, vocalTract=15.5)),
    ('F1', 400, 1, dict(formants=_formants(1, 1), vocalTract=16.)),
    ('F31', 400, 2, dict(formants=_formants(31, 31), vocalTract=16.)),
    ('F32', 400, 1, dict(formants=_formants(32, 32), vocalTract=16.)),
    ('F33', 551, 1, dict(formants=_formants(33, 33, hi=10000), vocalTract=16., samplingRate=22050)),
    ('F62 closed', 400, 3, dict(formants=_formants(62, 62), vocalTract=16., mouthAnchors=CLOSED)),
    ('F200', 1200, 1, dict(formants=_formants(200, 200, hi=23000, amp=.3), vocalTract=100., samplingRate=48000)),
    ('F1024 closed', 400, 1, dict(formants=_formants(1024, 1024, amp=.02), vocalTract=16., mouthAnchors=CLOSED)),
    ('width 0', 400, 1, dict(formants=[np.array([[0, 1000, 30, 0.]]), np.array([[0, 2500, 20, 0.]])], vocalTract=15.)),
    ('very wide', 400, 1, dict(formants=[np.array([[0, 500, 30, 5000.]]), np.array([[0, 2000, 20, 3000.]])],
                               vocalTract=15.)),
    ('very narrow', 400, 1, dict(formants=[np.array([[0, 3000, 30, 0.5]]), np.array([[0, 1234.5, 25, 0.2]])],
                                 vocalTract=15.)),
    ('below bin 1', 400, 1, dict(formants=[np.array([[0, 3, 30, 80.]]), np.array([[0, 900, 20, 100.]])],
                                 vocalTract=float('nan'))),
    ('above Nyquist', 400, 1, dict(formants=[np.array([[0, 1200, 30, 100.]]), np.array([[0, 9500, 30, 200.]])],
                                   vocalTract=15.)),
    ('negative amplitude', 400, 1, dict(formants=[np.array([[0, 800, -25, 100.]]), np.array([[0, 1800, 30, 150.]])],
                                        vocalTract=15.)),
    ('closed below 550 Hz', 400, 24, dict(formants=[np.array([[0, 400, 30, 90.]]), np.array([[0, 1900, 25, 150.]])],
                                          vocalTract=17., mouthAnchors=(np.array([0., .5, 1]), np.array([0., .6, .1])),
                                          mouthOpenThres=.3, openMouthBoost=10)),
    ('closed above 550 Hz', 400, 24, dict(formants=[np.array([[0, 700, 30, 90.]]), np.array([[0, 1900, 25, 150.]])],
                                          vocalTract=17., mouthAnchors=(np.array([0., .5, 1]), np.array([.9, 0., .4])),
                                          mouthOpenThres=.2, openMouthBoost=-6)),
    ('vocalTract NA', 400, 1, dict(formants=_formants(4, 4), vocalTract=float('nan'))),
    ('formantDep 0', 400, 1, dict(formants=_formants(5, 5), vocalTract=16., formantDep=0)),
    ('formantDep 5', 400, 1, dict(formants=_formants(5, 6), vocalTract=16., formantDep=5)),
    ('rolloffLip 0', 400, 1, dict(formants=_formants(5, 7), vocalTract=16., rolloffLip=0)),
    ('moving 3/5/1 points slf 0', 400, 40, dict(formants=_moving([3, 5, 1], 0), vocalTract=16., smoothLinearFactor=0)),
    ('moving 2/7 points slf 1', 600, 37, dict(formants=_moving([2, 7], 1), vocalTract=16., samplingRate=24000)),
    ('moving 4/4/9 points slf 10', 80, 50, dict(formants=_moving([4, 4, 9], 2), vocalTract=16., samplingRate=16000)),
    ('given tracks', 400, 30, dict(formants_upsampled=_tracks(5, 30, 3), formants=_formants(5, 3), vocalTract=16.)),
    ('nr 301', 301, 1, dict(formants=_formants(4, 8), vocalTract=16.)),
    ('nr 1102', 1102, 1, dict(formants=_formants(6, 9, hi=20000), vocalTract=16., samplingRate=44100)),
    ('nint 300', 400, 300, dict(formants=_moving([6, 3], 4), vocalTract=16., mouthAnchors=(np.array([0., .3, 1]),
                                                                                            np.array([.2, .9, .5])))),
]
