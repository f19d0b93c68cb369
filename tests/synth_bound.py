"""Float64 reference and per-sample error bound of K1, the harmonic sum of generateHarmonics
(R/source.R:389-419), for both kernels that compute it: k_synth (FP32 pipe, kernels_synth.cu) and k_synth_tc
(tensor cores, kernels_synth_tc.cu).  Test infrastructure only.

Notation.  u = 2^-24 (FP32 unit roundoff).  For sample k of epoch e, lying in interval i of approx() with weight
w (source.R:403-405), row h of the epoch's matrix has the knot values Y_h = mat[h, i], Y'_h = mat[h, i+1], the
interpolant a_h = Y_h + w (Y'_h - Y_h) and the integer multiple j_h = name_h (nSubharm + 1) of
theta' = 2 pi integr / (nSubharm + 1).  The oracle's matrices are non-negative (2^(dB/10) rolloffs, shimmer
factors 2^N, Gaussian side bands), so |a_h| = a_h and |Y' - Y| <= max(Y, Y').  The bound uses

    A1[k]  = sum_h max(Y_h, Y'_h)          the magnitudes the FP32 lerp Y + w dY carries (>= sum_h |a_h|: a lerp
                                           rounds on its knot values, not on their interpolant);
    Aj[k]  = sum_h j_h |a_h(u_k)|;
    AjK[k] = sum_h rho_K(j_h) |a_h(u_k)|,  rho_K(j) = ((j - 1) mod K) + 1, the row's index inside its block of K
                                           rows (k_synth's Clenshaw blocks);
    An[k]  = sum_h name_h |a_h(u_k)| = Aj / (nSubharm + 1).

and has the form  B_e[k] = u (c_a A1 + c_phi 2 pi Aj  [+ the k_synth terms in AjK]) + 2 pi eps_K0 An, except that
k_synth_tc's phase roundings depend on a row's place in its block and pass, not on j (rho_tc below).

Common to both kernels
----------------------
* FP32 table (K3, kernels_ctrl.cu `amp32`): Y and dY = Y' - Y rounded from FP64, u Y and u |dY| <= u max(Y, Y').
* weight w = (float)(v - xg) * rcp((float)(xn - xg)) (kernels_synth.cu:136, kernels_synth_tc.cu:266): three
  roundings, 3u w |dY| <= 3u max(Y, Y').
* lerp FMA Y + w dY (kernels_synth.cu:50, the Cc / Ss FFMA2 of kernels_synth_tc.cu:364-365): u |a| <= u max.
  With the table this is 6 u A1 (k_synth) or 5 u A1 + the Cc rounding (k_synth_tc, below).
* FP32 store of the epoch sample (kernels_synth.cu:323, kernels_synth_tc.cu:387): u |w_e| <= u A1.
* K0's phase: integr from the quartic of each spline piece (kernels_ctrl.cu:89, evaluated at
  kernels_synth.cu:141 and kernels_synth_tc.cu:280) agrees with R's long-double cumsum to eps_K0 = 1e-9 cycles
  (DESIGN.md section 4, "Phase").  Row h's phase is 2 pi integr name_h: error <= 2 pi eps_K0 An.
* FP64 reduction x = frac(integr / (nSubharm + 1)) is exact to ~1e-16 cycles: not a term.

k_synth (kernels_synth.cu), per warp of 128 samples: block length K (:147-153), recurrence mode (:155-170)
--------------------------------------------------------------------------------------------------------
Let Lam = min(K, 1 / |sin theta'|).  Inside a block, b_r = sum_{m >= r} a_m U_{m-r}(cos theta') with
|U_n| = |sin((n+1) theta') / sin theta'| <= Lam, so |b_r| <= Lam A_r (A_r = the block's sum_{m >= r} |a_m|); the
sum over r of A_r is AjK.
* Mode 3, standard Clenshaw (SYNTH_STEP3, :69-74).  All lanes are >= 0.03 cycles from both poles (:163), so
  Lam = 1 / |sin theta'| <= 1 / sin(2 pi 0.03) = 5.34.  Clenshaw is backward stable in its coefficients: an error
  injected into b_r acts as a change of a_r.  FFMA + FADD per step: u (2 Lam A_{r+1} + |a_r|) + u Lam A_r
  -> u (3 Lam AjK + A1).  The coefficient k0 = 2 (1 - 2 sh^2) from sincospif of xr = (float)(x - q/2) (:179-189;
  rounding |xr| <= 1/4 costs <= 2^-27 cycles = 0.8 u rad, sincospif 1 ulp = 2u relative) has an absolute error
  <= 9u, an angle error dth <= u (0.8 + 9 Lam), whose effect on the block sum (b_1 sin theta', b_1 cos theta' -
  b_2 with the separately rounded sin / cos) is <= 2 dth (AjK + Lam A1).  Epilogue (:247-258): Cs, Ss from
  b_1, b_2 with cos / sin errors <= 9u / 5u: (2 + 14 Lam) u per block -> (2 + 14 Lam) u A1.
* Modes 0, 1, 2, Reinsch's form around the pole sigma (:51-68): state (b_r, d_r = b_r - sigma b_{r+1}),
  d_r = a_r + delta b_{r+1} + sigma d_{r+1}, b_r = sigma b_{r+1} + d_r, delta = 2 cos theta' - 2 sigma.  Let
  theta_s be the angle to sigma (mode 0: to the lane's nearer pole, <= pi / 2; modes 1, 2: <= 3/4 pi, the lanes
  are within 3/8 cycle of it), s = sin(theta_s / 2), c = cos(theta_s / 2).  Then |d_r| <= A_r / c (its kernel is
  cos((2n+1) theta_s / 2) / cos(theta_s / 2)), and an error in d_r acts as a change of a_r.  An error e in b_r
  (with d_r kept) acts as e on a_r and (delta - sigma) e on a_{r-1}: it reaches the block sum with a factor
  |1 - e^{-i theta_s}| + |delta| = 2s + 4s^2, and with |b_r| <= Lam A_r, Lam 2s + 4s^2 <= g = min(K (2s + 4s^2),
  (1 + 2s) / c): the b rounding never sees the 1 / sin theta' growth.  Two roundings into d, on |d_{r+1}| + |a_r|
  and |d_r|, <= u (2 A_r / c + |a_r|) <= u (5.3 A_r + |a_r|) with c >= cos(3 pi / 8); one into b:
  -> u ((5.3 + g) AjK + A1).  k0 = -4 sh^2 (or
  4 ch^2, :186-188) carries <= 6u relative error: an angle error 6u tan(theta_s / 2) = 6u s / c, plus 0.8u,
  effect 2 dth AjK; the epilogue (Cs = b_1 k0 / 2 + sigma d_1, Ss = b_1 es, and es against the recurrence's
  angle) <= 24 u A1.
* Per block, both: the acc FFMA2 pair: 2u |acc| per block -> 2 u nb A1 (nb = ceil(J / K) blocks).
* Base rotation e^{i K theta'} (:191-193, :254-256): xk reduced in FP64, rounded to float (<= 2^-26 cycles =
  1.6u rad), sincospif 1 ulp, two roundings per component per step: <= 8u per block, block b = floor((j-1)/K)
  <= j / K rows: 8 u Aj / K.
* Straddling pairs (:201-237; the second sample of a pair in the next cycle, evaluated by the whole warp):
  lerp / table / store 7 u A1; the start rotation e^{i ja theta'} from an FP64-reduced phase (<= 5 u A1); the
  float rotator e^{i theta'} (xs rounded to 2^-26 cycles, sincospif, two roundings): <= 8u per row step, fewer
  steps than j: 8 u Aj; the per-lane running sum of at most chunk = ceil(J / 32) rows: chunk u A1; the warp
  reduction: 5 u A1.  Those samples take  u ((18 + chunk) A1 + 8 Aj)  instead of the block bound.

A warp's mode is decided in float (:161-168), so where a lane sits within 1e-6 cycles of a threshold the bound
takes the larger of the candidate modes' bounds.

k_synth_tc (kernels_synth_tc.cu), per unit = interval of approx()
------------------------------------------------------------------
* Amplitude operand (:228-256): Y, dY scaled by a power of two so that the largest of the super-pass, mx, sits
  in [2^14, 2^15), then hi + lo in FP16: <= 2^-22 |value| + 2^-39 mx each (lo may be subnormal); two values per
  row: 8 u A1 + J 2^-38 mx <= (8 + J / 2^14) u A1.
* Trig operand (:297-313): (float)x with x in [0, 1): <= 2^-25 cycles = pi u rad on theta', i.e. m pi u on row
  m of the block; e^{i theta'} from sincospif (2u), e^{2 i theta'} (<= 7u), the packed chain (<= 10u per step,
  rows m <= 15): <= (2 + 5 m) u <= 77 u per trig value; its FP16 split: <= (2^-22 + 2^-25) per component, 6.4u
  for the pair; the dropped lo * lo products of the three MMAs (:169-171): <= 2^-22 (|cos| + |sin|) |a| = 5.7u.
  With Y and w dY each <= max(Y, Y'): 2 (77 + 6.4 + 5.7) u A1 = 178 u A1, the m pi u part in the phase term.
* MMA accumulation in FP32 (:169-171): the tensor cores' accumulation order and rounding are not specified;
  one ulp (2u) per addition of sequential summation is assumed: 16 products + 2 accumulator adds of the
  dominant hi * hi chain, on sum |t| |Y| and sum |t| |dY| for C and S separately: 2 * 18 * sqrt(2) * 2 u A1 = 102 u A1.
* Epilogue (:350-386): Cc / Ss FFMA2 rounding 2u A1 (the lerp, above); Horner in z^2 over <= 12 block pairs per
  pass: the step for block pair q rounds twice on values <= the pass's partial sum above it: <= 6 u (A1 + Aj / 32);
  z from (float)(16 x mod 1): pi u on 16 theta' per block (phase term), sincospif and squaring <= 8u per block
  pair: 4u per block b <= j / 16 -> 0.25 u Aj; the even / odd combination and acc update <= 6 u A1; the pass
  rotation e^{i 384 theta'} ((float)(384 x mod 1): pi u, sincospif and the rotation product <= 5u) per pass
  p <= j / 384; the super-pass rotation e^{i row0 theta'} (pi u + 2u, once) and the read-back add
  `fmaf(acc, unscale, prev)` (:386): u A1 per super-pass.
* Per-row terms.  Row j sits in super-pass sp = j // 1152, pass p, block b (< 24) and block row m (< 16) of it
  (:232, :248).  x, 16 x, 384 x and row0 x are each reduced in FP64 and rounded to float separately (:299, :324,
  :329, :332), so row j's angle carries m + b + p + [sp > 0] roundings of <= pi u, not j of them.  With the
  z^2 chain (4u per block b), Horner (6u per step the row's block pair takes: b // 2 + 1), the pass rotation
  (5u per pass p) and the super-pass rotation (2u):
      rho_tc(j) = pi (m + b + p + [sp > 0]) + 4 b + 6 (b // 2 + 1) + 5 p + 2 [sp > 0]   (<= 320),
  and the bound carries u sum_h rho_tc(j_h) |a_h| in place of a c_phi 2 pi Aj term.
* c_a = 5 (table, weight) + 2 (Cc) + 8 + J / 2^14 (operand split) + 178 (trig) + 102 (MMA) + 6 (combination) +
  nsuper (read-back) + 1 (store).

k_build_units_tc (:86-110) gives every interval of approx() of an epoch one unit; its samples reach from the
stretched coordinate of one knot to that of the next: u-length (x_{i+1} - x_i) / by with
by = (x_last - x_first) / (Ne - 1) <= 1.  The spline pieces of pitch_upsampled change at the middle of every
glottal cycle, so an interval spans two or three pieces unless 1 / by stretches it over further cycles, which
needs an epoch whose last cycle is longer than the cycles before it together (a pitch drop by a factor of
several within the epoch: strong jitter in a short epoch).  `tc_piece_spans` counts the pieces per unit from
the oracle's knots, and the corpus holds a case that reaches the fourth piece (the fallback at :273).

After K1 (K6, kernels_compose.cu)
---------------------------------
Every later step is linear with non-negative weights, so the bound goes through it like the signal
(`propagate`): crossFade at the oracle's zero crossings (the inserted 0 is exact), the amplitude envelope,
division by the signed maximum (plus |y[k]| dmax / max for the error dmax of the maximum itself, where dmax is the
largest bound of any sample that can compete for the maximum), fadeInOut and the drift gain.  K6's own
arithmetic: the FP32 stores of the cross-fade (kernels_compose.cu:263) and of the envelope product (:296), each
u of the magnitude carried there, and the final FP32 store (:365), u |y|; its FP64 products are far below that.
"""
import functools
import math

import numpy as np

from oracle import soundgen_oracle as so
from oracle.rprims import r_seq_len_out

U = 2.0 ** -24
EPS_K0 = 1e-9           # cycles: K0's quartic phase against R's long-double cumsum (DESIGN.md section 4)
MIN_ROWS_DEFAULT = 224  # K1 dispatch: epochs with at least this many rows go to k_synth_tc (engine.cu)
WARP = 128              # samples per warp of k_synth (32 lanes x 4)
MODE_THR = (0.03, 0.375)


# ----------------------------------------------------------------------------------------------------------------
# corpus: each case aims at one place where an implementation of the sum goes wrong
# ----------------------------------------------------------------------------------------------------------------
def _flat(f0, sr, ms):
    return np.full(int(round(ms * 3.5)), float(f0))


def _rows_case(rows, nsub=0):
    """flat pitch at 48 kHz whose epoch has `rows` rows (every harmonic below Nyquist kept, rolloff ~flat)."""
    harm = (rows - nsub) // (nsub + 1)
    assert harm * (nsub + 1) + nsub == rows
    f0 = 24000.0 / (harm + 0.5)
    pars = dict(samplingRate=48000.0, pitchFloor=1, temperature=0, rolloff=-1, rolloffOct=0, rolloffKHz=0,
                attackLen=10, nonlinBalance=0)
    if nsub:
        pars.update(nonlinBalance=100, subDep=100, subFreq=f0 / (nsub + 1), shortestEpoch=50)
    ms = max(120.0, 4000.0 / f0)
    return dict(pitch=_flat(f0, 48000, ms) * np.linspace(1, 1.0001, int(round(ms * 3.5))), pars=pars)


def _glide(f0a, f0b, ms):
    P = int(round(ms * 3.5))
    return np.exp(np.linspace(np.log(f0a), np.log(f0b), P))


CORPUS = {
    # sampling rates, nSubharm 1 / 2 / >= 3 (vocal-fry epochs next to plain ones), moderate shimmer and jitter
    'sr16k_sub1': dict(pitch=_glide(140, 190, 400), pars=dict(
        samplingRate=16000.0, nonlinBalance=100, subDep=80, subFreq=85, shortestEpoch=50, jitterDep=0.5,
        shimmerDep=10, rolloff=-12, attackLen=20)),
    'sr22k_sub2': dict(pitch=_glide(230, 260, 350), pars=dict(
        samplingRate=22050.0, nonlinBalance=100, subDep=120, subFreq=82, shortestEpoch=50, rolloff=-9,
        attackLen=0)),
    'sr44k_sub3': dict(pitch=_glide(160, 260, 500), pars=dict(
        samplingRate=44100.0, nonlinBalance=100, subDep=150, subFreq=45, shortestEpoch=50, rolloff=-8,
        rolloffOct=-1, attackLen=10)),
    # the K1 dispatch (224 rows), pass (384), resident group (1152) and 2 x 1152 boundaries
    'rows223': _rows_case(223), 'rows225': _rows_case(225),
    'rows383': _rows_case(383), 'rows385': _rows_case(385),
    'rows767': _rows_case(767), 'rows769': _rows_case(769),
    'rows1151': _rows_case(1151), 'rows1153': _rows_case(1153),
    'rows2303': _rows_case(2303, nsub=1), 'rows2305': _rows_case(2305, nsub=1), 'rows2401': _rows_case(2401, nsub=1),
    # strong shimmer and jitter: amplitudes jump between cycles; short epochs, long last cycles
    'shimmer_jitter': dict(pitch=_glide(90, 140, 400), pars=dict(
        samplingRate=48000.0, nonlinBalance=100, shimmerDep=60, jitterDep=3, jitterLen=1, subDep=60, subFreq=60,
        shortestEpoch=20, rolloff=-6, attackLen=10)),
    'jitter_wide': dict(pitch=_glide(120, 150, 300), pars=dict(
        samplingRate=22050.0, nonlinBalance=100, jitterDep=12, jitterLen=1, subDep=100, subFreq=50,
        shortestEpoch=40, pitchFloor=20, rolloff=-10, attackLen=0)),
    # high pitch at 16 kHz: more than 16 cycles per 128 samples (k_synth's direct path)
    'high16k': dict(pitch=_glide(2400, 3300, 300), pars=dict(
        samplingRate=16000.0, pitchCeiling=3500, rolloff=-6, rolloffOct=-1, attackLen=10)),
    # flat rolloff (A1 largest next to the peak) and a steep one down to the -120 dB throwaway
    'flat_rolloff': dict(pitch=_glide(110, 125, 300), pars=dict(
        samplingRate=44100.0, rolloff=0, rolloffOct=0, rolloffKHz=0, attackLen=0)),
    'steep_rolloff': dict(pitch=_glide(95, 105, 300), pars=dict(
        samplingRate=44100.0, rolloff=-30, rolloffOct=-12, rolloffKHz=-12, attackLen=10)),
    # a phase beyond 2000 cycles
    'long_phase': dict(pitch=_glide(480, 520, 4500), pars=dict(
        samplingRate=22050.0, rolloff=-12, attackLen=50)),
    # temperature > 0 (random walks, drift gain), amplitude anchors and an attack
    'temperature': dict(pitch=_glide(150, 220, 500), pars=dict(
        samplingRate=16000.0, temperature=0.3, nonlinBalance=100, jitterDep=1, shimmerDep=20, subDep=50,
        subFreq=80, rolloff=-10, attackLen=50)),
    'ampl_anchors': dict(pitch=_glide(200, 170, 400), anchors=(np.array([0., 0.4, 1.]), np.array([60., 110., 80.])),
                         pars=dict(samplingRate=48000.0, rolloff=-9, attackLen=50)),
}
CASE_NAMES = sorted(CORPUS)


def case_inputs(name):
    c = CORPUS[name]
    z = np.random.default_rng(sum(map(ord, name))).standard_normal(20000)
    return c['pitch'], z, c.get('anchors'), dict(c['pars'])


@functools.lru_cache(maxsize=None)
def oracle_case(name):
    pitch, z, anchors, pars = case_inputs(name)
    y, art = so.generateHarmonics(pitch, rng=so.RStream(z=z), amplAnchors=anchors, want_artefacts=True, **pars)
    return y, art


def attack_points(pars):
    a = pars.get('attackLen', 50)
    return int(math.floor(a * pars.get('samplingRate', 16000) / 1000)) if a > 0 else 0


# ----------------------------------------------------------------------------------------------------------------
# per-epoch inputs of the sum, and the float64 restatement
# ----------------------------------------------------------------------------------------------------------------
class Epoch:
    """The inputs of epoch e's sum (source.R:389-409) as the kernels see them."""

    def __init__(self, art, e):
        ep = art.epochs[e]
        idx = art.gc_upsampled[ep[0] - 1:ep[1] + 1]
        lo, hi = int(idx.min()), int(idx.max())
        self.Ne = hi - lo + 1
        self.x_first_i = lo
        self.nsub = int(art.nSubharm[ep[1] - 1]) if art.nSubharm is not None else 0
        mat, nm = art.mats[e]
        assert np.all(mat >= 0), 'the bound assumes non-negative amplitude matrices'
        self.mat, self.names = mat, np.asarray(nm, dtype=np.float64)
        self.j = np.rint(self.names * (self.nsub + 1)).astype(np.int64)
        self.J = int(self.j.max())
        xk = idx[:-1].astype(np.float64)
        self.xk = xk
        v = r_seq_len_out(xk[0], xk[-1], self.Ne)
        i = np.clip(np.searchsorted(xk, v, side='right') - 1, 0, xk.size - 2)
        self.iv = i
        self.w = (v - xk[i]) / (xk[i + 1] - xk[i])
        self.integr = art.integr[lo - 1:hi]
        self.x = np.mod(self.integr / (self.nsub + 1), 1.0)   # theta' / 2 pi, cycles

    def weighted(self, f):
        """sum_h f_h |a_h(u_k)| per sample (a >= 0, linear in w)."""
        s = f @ self.mat
        return (1.0 - self.w) * s[self.iv] + self.w * s[self.iv + 1]

    def A1(self):
        m = np.maximum(self.mat[:, :-1], self.mat[:, 1:]).sum(axis=0)
        return m[self.iv]

    def Aj(self):
        return self.weighted(self.j.astype(np.float64))

    def An(self):
        return self.weighted(self.names)

    def AjK(self, K):
        return self.weighted(((self.j - 1) % K + 1).astype(np.float64))

    def wave(self, mat=None, dphi=None):
        """sum_h a_h sin(2 pi integr name_h) as the oracle computes it; `mat`, `dphi` (per-row phase offsets in
        cycles): perturbed."""
        mat = self.mat if mat is None else mat
        out = np.zeros(self.Ne)
        a_lo, a_hi = mat[:, self.iv], mat[:, self.iv + 1]
        two_pi_integr = 2 * np.pi * self.integr          # the oracle's association (source.R:397)
        for h in range(mat.shape[0]):
            am = a_lo[h] + (a_hi[h] - a_lo[h]) * self.w
            off = 0.0 if dphi is None else 2 * np.pi * dphi[h]
            out += np.sin(two_pi_integr * self.names[h] + off) * am
        return out


def epochs_of(art):
    return [Epoch(art, e) for e in range(art.epochs.shape[0])]


# ----------------------------------------------------------------------------------------------------------------
# host mirror of k_synth's per-warp choices (kernels_synth.cu:110-170, :201-207)
# ----------------------------------------------------------------------------------------------------------------
def _mode_of(xf, thr_a, thr_p):
    d0 = np.minimum(xf, np.float32(1) - xf)
    dpi = np.abs(xf - np.float32(0.5))
    if np.all((d0 >= np.float32(thr_a)) & (dpi >= np.float32(thr_a))):
        return 3
    if np.all(d0 <= np.float32(thr_p)):
        return 1
    if np.all(dpi <= np.float32(thr_p)):
        return 2
    return 0


def synth_warps(ep):
    """One record per warp: first sample, K, staged, the set of modes it may pick (two when a lane sits within
    1e-6 cycles of a threshold) and the samples that are straddling second samples of a pair."""
    out = []
    for kw in range(0, ep.Ne, WARP):
        k = np.minimum(kw + np.arange(WARP), ep.Ne - 1)
        gi = ep.iv[k] - ep.iv[kw]
        ncolw = int(gi[-1]) + 1
        staged = ncolw <= 16
        if staged:
            ks = 7
            cap = 1
            while cap < ncolw:
                cap <<= 1
                ks -= 1
        else:
            ks = 6
        K = min(1 << ks, 128)
        xf = ep.x[k].astype(np.float32)
        modes = {_mode_of(xf, a, p) for a in (MODE_THR[0] - 1e-6, MODE_THR[0] + 1e-6)
                 for p in (MODE_THR[1] - 1e-6, MODE_THR[1] + 1e-6)}
        ks_ = kw + np.arange(WARP)
        pair0 = ks_[0::2]
        need = staged & (gi[1::2] != gi[0::2]) & (pair0 + 1 < ep.Ne)
        strad = (pair0 + 1)[need]
        out.append(dict(kw=kw, n=min(WARP, ep.Ne - kw), K=K, staged=staged, ncolw=ncolw,
                        mode=_mode_of(xf, *MODE_THR), modes=modes, straddle=strad))
    return out


def tc_piece_spans(art, ep_idx, sr):
    """Spline pieces of pitch_upsampled (knots: utilities_soundgen.R:405-413) that each tensor-core unit of the
    epoch touches (k_synth_tc stages four, kernels_synth_tc.cu:123, :273)."""
    p = art.pitch_per_gc
    gclen = np.rint(sr / p)     # r_round: the knots only need to be right to the sample
    c = np.cumsum(gclen)
    l = p.size
    if l < 3:
        return [1]
    t = np.ones(l)
    t[l - 1] = c[-1]
    for i in range(2, l):
        t[i - 1] = c[i - 2] + so.r_round(gclen[i - 1] / 2)
    ep = Epoch(art, ep_idx)
    u = ep.x_first_i + np.arange(ep.Ne, dtype=np.float64)
    piece = np.searchsorted(t, u, side='right') - 1
    spans = []
    for i in np.unique(ep.iv):
        pc = piece[ep.iv == i]
        spans.append(int(pc.max() - pc.min() + 1))
    return spans


# ----------------------------------------------------------------------------------------------------------------
# the bounds
# ----------------------------------------------------------------------------------------------------------------
def k0_term(ep):
    return 2 * np.pi * EPS_K0 * ep.An()


def synth_block_bound(ep, K, mode, A1, Aj, AjK, x):
    """k_synth: u (...) of the module docstring for one recurrence mode and block length K (no K0 term)."""
    nb = math.ceil(ep.J / K)
    if mode == 3:
        lam = 1.0 / np.maximum(np.abs(np.sin(2 * np.pi * x)), 1e-300)
        dth = 0.8 + 9 * lam
        body = (3 * lam * AjK + A1) + 2 * dth * (AjK + lam * A1) + (2 + 14 * lam) * A1
    else:
        # angle to the pole the form is built around: the lane's own (mode 0), theta = 0 (1) or pi (2)
        d = np.minimum(x, 1 - x) if mode == 1 else (np.abs(x - 0.5) if mode == 2 else
                                                     np.minimum(np.minimum(x, 1 - x), np.abs(x - 0.5)))
        s, c = np.sin(np.pi * d), np.cos(np.pi * d)          # sin, cos of theta_sigma / 2
        g = np.minimum(K * (2 * s + 4 * s * s), (1 + 2 * s) / c)
        dth = 0.8 + 6 * s / c
        body = ((5.3 + g) * AjK + A1) + 2 * dth * AjK + 24 * A1
    return U * (7 * A1 + body + 2 * nb * A1 + 8 * Aj / K)


def synth_fixup_bound(ep, A1, Aj):
    chunk = (ep.J + 31) // 32
    return U * ((18 + chunk) * A1 + 8 * Aj)


def synth_bound(ep, force_mode=None):
    """Per-sample bound of epoch `ep` computed by k_synth (force_mode=0: SGB_SYNTH_MODE=0)."""
    A1, Aj = ep.A1(), ep.Aj()
    AjK = {}
    B = np.zeros(ep.Ne)
    for wr in synth_warps(ep):
        K = wr['K']
        if K not in AjK:
            AjK[K] = ep.AjK(K)
        sl = slice(wr['kw'], wr['kw'] + wr['n'])
        modes = {force_mode} if force_mode is not None else wr['modes']
        B[sl] = np.max([synth_block_bound(ep, K, m, A1[sl], Aj[sl], AjK[K][sl], ep.x[sl]) for m in modes], axis=0)
        if wr['straddle'].size:
            B[wr['straddle']] = synth_fixup_bound(ep, A1, Aj)[wr['straddle']]
    return B + k0_term(ep)


def tc_row_place(j):
    """(super-pass, pass, block, block row) of row j in k_synth_tc (rows 0 .. J, 1152 per super-pass)."""
    sp, r = np.divmod(j, 1152)
    return sp, r // 384, (r % 384) // 16, r % 16


def tc_angle_roundings(j):
    """m + b + p + [sp > 0]: the float-rounded angles that make up row j's phase."""
    sp, p, b, m = tc_row_place(j)
    return m + b + p + (sp > 0)


def tc_c_a(J):
    nsuper = (J + 1 + 1151) // 1152
    return 5 + 2 + 8 + J / 2.0 ** 14 + 178 + 102 + 6 + nsuper + 1


def tc_rho(j):
    sp, p, b, m = tc_row_place(j)
    return np.pi * tc_angle_roundings(j) + 4 * b + 6 * (b // 2 + 1) + 5 * p + 2 * (sp > 0)


def tc_bound(ep):
    return U * (tc_c_a(ep.J) * ep.A1() + ep.weighted(tc_rho(ep.j).astype(np.float64))) + k0_term(ep)


def table_term(ep):
    """The FP32 table's share of either bound (u A1): what rounding the matrices to float32 may cause."""
    return U * ep.A1()


def float_phase_term(ep):
    """k_synth_tc's share of its float angles: pi u per rounding, tc_angle_roundings(j) of them on row j."""
    return U * np.pi * ep.weighted(tc_angle_roundings(ep.j).astype(np.float64))


def epoch_bound(ep, kernel, force_mode=None):
    return tc_bound(ep) if kernel == 'tc' else synth_bound(ep, force_mode)


def kernel_of(ep, min_rows):
    """Which kernel runs the epoch under sgb_synth_min_rows_set(min_rows)."""
    m = MIN_ROWS_DEFAULT if min_rows < 0 else min_rows
    return 'tc' if ep.J >= m else 'ffma'


# ----------------------------------------------------------------------------------------------------------------
# the steps after K1 (source.R:427-467), with the oracle's own zero crossings
# ----------------------------------------------------------------------------------------------------------------
def cross_fade_at(ampl1, ampl2, sr, zc1, zc2, crossLen=15):
    """crossFade (utilities_soundgen.R:328-375) at given 1-based zero crossings (None or 0: none found); the
    sample at zc1 becomes an exact 0 as in the reference."""
    if zc1:
        ampl1 = np.concatenate((ampl1[:zc1], [0.0]))
    if zc2:
        ampl2 = ampl2[zc2:]
    cl = min(math.floor(crossLen * sr / 1000), len(ampl1) - 1, len(ampl2) - 1)
    if cl < 2:
        return np.concatenate((ampl1, ampl2))
    mu = r_seq_len_out(0, 1, cl)
    idx1 = len(ampl1) - cl
    return np.concatenate((ampl1[:idx1], mu[::-1] * ampl1[idx1:] + mu * ampl2[:cl], ampl2[cl:]))


def join(waves, zc, sr):
    out = np.zeros(1)
    for wv, (z1, z2) in zip(waves, zc):
        out = cross_fade_at(out, wv, sr, z1, z2)
    return out


def compose(waves, art, pars):
    """The oracle's output from (possibly perturbed) epoch waves, with the oracle's zero crossings."""
    c = join(waves, art.zc, pars['samplingRate'])
    if art.ampl_gain is not None:
        c = c * art.ampl_gain
    y = c / np.max(c)
    lf = attack_points(pars)
    if lf > 0:
        y = so.fadeInOut(y, length_fade=lf)
    if art.drift_upsampled is not None:
        y = y * art.drift_upsampled
    return y


def propagate(bounds, art, pars, waves=None, k6=True):
    """Carry per-epoch bounds through crossFade, envelope, signed-max normalisation, fade and drift.  `waves`:
    the reference epoch waves (default: the oracle's)."""
    sr = pars['samplingRate']
    waves = art.epoch_waves if waves is None else waves
    Bj = join(bounds, art.zc, sr)
    c = join(waves, art.zc, sr)
    M = join([np.abs(w) + b for w, b in zip(waves, bounds)], art.zc, sr)
    if art.ampl_gain is not None:
        if k6:
            Bj = Bj + U * M
        Bj, c, M = Bj * art.ampl_gain, c * art.ampl_gain, M * art.ampl_gain
    im = int(np.argmax(c))
    mx = c[im]
    # the device's maximum is that of some sample that can reach at least the reference maximum's lower end
    cand = c + Bj >= mx - Bj[im]
    dmax = float(np.max(Bj[cand]))
    den = mx - dmax
    assert den > 0
    yb = (Bj + np.abs(c) * dmax / mx) / den
    if k6:
        yb = yb + U * 2 * M / den
    lf = attack_points(pars)
    if lf > 0:
        yb = so.fadeInOut(yb, length_fade=lf)
    if art.drift_upsampled is not None:
        yb = yb * np.abs(art.drift_upsampled)
    if k6:
        y = compose(waves, art, pars)
        yb = yb + U * (np.abs(y) + yb)
    return yb


def output_bound(name, kernels, force_mode=None):
    """Per-sample bound of the final output of corpus case `name`, and per epoch: the kernel and its bound."""
    y, art = oracle_case(name)
    pars = case_inputs(name)[3]
    eps = epochs_of(art)
    Bs = [epoch_bound(ep, k, force_mode) for ep, k in zip(eps, kernels)]
    return propagate(Bs, art, pars), Bs


def epoch_of_output(art, pars):
    """For every output sample: the epoch whose wave it comes from (cross-fades: the later epoch)."""
    E = len(art.epoch_waves)
    share = [join([np.full(w.size, float(f == e)) for f, w in enumerate(art.epoch_waves)], art.zc,
                  pars['samplingRate']) for e in range(E)]
    return np.argmax(np.stack(share), axis=0)
