// K0: control-rate prologue of generateHarmonics (R/source.R:206-385), one
// syllable per call, scalar IEEE-double code (see common.cuh).  Emits the integer
// artefacts (glottal cycles, epochs, nSubharm, rw_bin, jitter idx, gc_upsampled)
// and the per-glottal-cycle arrays the sample-rate kernels consume.
#pragma once
#include "contour.cuh"
#if !defined(__CUDACC__)
#include <vector>
#endif

// ---------------------------------------------------------------- helpers ---
// noiseThresholdsDict (data-raw/noiseThresholdsDict.R:4-18); a fractional
// nonlinBalance is truncated by R's indexing (utilities_math.R:361-363).
SGB_HD void noise_thresholds(double nonlinBalance, double *q1, double *q2) {
  double a = (double)((int)(nonlinBalance + 1.0) - 1);
  *q1 = 100.0 / (1.0 + exp(0.1 * (a - 33.0)));
  *q2 = 100.0 / (1.0 + exp(0.1 * (a - 66.0)));
}

// round(median(s)) for the degenerate branch of clumper (utilities_math.R:561).
SGB_HD double median_round(const int32_t *s, int n, double *tmp) {
  for (int i = 0; i < n; i++) {   // insertion sort (rare path, small n)
    double v = (double)s[i];
    int j = i - 1;
    while (j >= 0 && tmp[j] > v) { tmp[j + 1] = tmp[j]; j--; }
    tmp[j + 1] = v;
  }
  double m = (n & 1) ? tmp[n / 2] : (tmp[n / 2 - 1] + tmp[n / 2]) / 2.0;
  return rint(m);
}

// clumper (R/utilities_math.R:555-600).  s: in/out, n values; minLength: per-element
// vector (already the caller's values, rounded here), tmp: scratch of n doubles.
SGB_HD void clumper(int32_t *s, int n, const double *minLength, double *tmp) {
  double mx = minLength[0];
  for (int i = 1; i < n; i++) mx = fmax(mx, minLength[i]);
  if (mx < 2.0) return;
  bool all_same = true;
  for (int i = 1; i < n; i++) if (s[i] != s[0]) { all_same = false; break; }
  if (all_same || (double)n < rint(minLength[0])) {
    int32_t m = (int32_t)median_round(s, n, tmp);
    for (int i = 0; i < n; i++) s[i] = m;
    return;
  }
  int c = 0;
  for (int i = 1; i < n; i++) {
    if (s[i - 1] == s[i]) {
      c++;
    } else {
      if ((double)c < rint(minLength[i])) { s[i] = s[i - 1]; c++; } else { c = 1; }
    }
  }
  int ml = (int)rint(minLength[n - 1]);
  int lo = n - ml + 1; if (lo < 2) lo = 2;            // 1-based
  int cnt = 0;
  for (int p = lo; p <= n; p++) if (s[p - 1] == s[n - 1]) cnt++;
  if (cnt < ml) {
    int len_idx = n - lo + 1;                          // idx = rev(lo:n): idx[i] = n - i + 1
    int cc = 1, i = 2;
    while (i <= len_idx) {
      int pos = n - i + 1;                             // idx[i], 1-based
      bool same = (s[pos - 1] == s[pos - 2]);
      if (!(same && i < len_idx)) break;
      cc++; i++;
    }
    if (cc < ml) {
      int32_t v = s[lo - 1];
      for (int p = lo; p <= n; p++) s[p - 1] = v;
    }
  }
}

// getRandomWalk (R/utilities_math.R:289-326) for len >= 2.  Draws come from the
// syllable's normal stream z (cursor *zi, capacity zcap).  trend2: nonzero when
// trend = c(+t, -t).  out: len values; work arrays w0..w4: >= max(len, knots).
// Returns false if the stream is exhausted.
SGB_HD bool random_walk(int len, double rw_range, double rw_smoothing, bool trend2, double trend,
                        const double *z, int zcap, int *zi, double *out,
                        double *w0, double *w1, double *w2, double *w3, double *w4) {
  double p = (rw_smoothing != 0.0) ? exp2(1.0 / rw_smoothing) : INFINITY;
  double nf = floor(fmax(2.0, p));
  if (trend2) nf = rint(nf / 2.0) * 2.0;
  bool direct = !(nf <= (double)len);        // n > len
  int n = direct ? len : (int)nf;
  if (*zi + n > zcap) return false;
  // cumsum(rnorm(n, trend_short)): mean + 1 * z
  const int period = trend2 ? (int)nf : 1;   // trend_short = rep(c(t, -t), each = nf/2)
  CompSum acc;
  for (int i = 0; i < n; i++) {
    double m = trend;
    if (trend2) m = ((i % period) < period / 2) ? trend : -trend;
    acc.add(m + 1.0 * z[*zi + i]);
    w0[i] = acc.value();
  }
  *zi += n;
  if (direct) {
    for (int i = 0; i < len; i++) out[i] = w0[i];
  } else {
    for (int i = 0; i < n; i++) w1[i] = (double)(i + 1);
    fmm_coef(n, w1, w0, w2, w3, w4);
    const double by = r_seq_by_step(w1[0], w1[n - 1], len);
    for (int k = 0; k < len; k++) out[k] = r_spline_at_by(n, w1, w0, w2, w3, w4, by, len, k);
  }
  double mn = out[0];
  for (int i = 1; i < len; i++) mn = fmin(mn, out[i]);
  double mxabs = 0.0;
  for (int i = 0; i < len; i++) { out[i] = out[i] - mn; mxabs = fmax(mxabs, fabs(out[i])); }
  for (int i = 0; i < len; i++) out[i] = out[i] / mxabs * rw_range;
  return true;
}

// r[h, g] of getRolloff before normalisation (R/sourceSpectrum.R:84-143), in dB;
// -INFINITY for discarded entries.  h is the ORIGINAL harmonic number (1-based).
// rolloff_db_l with the per-cycle slope (ro + rk * (p - baseline) / 1000) supplied by the caller
// (K3 evaluates it once per column): the same operations in the same order.
SGB_HD double rolloff_db_s(int h, double lg2h, double p, double slope, double roct, bool any_oct,
                           double rolloffParab, int parab_harm, double pa, double pb, double pc,
                           double baseline, double throwaway, double samplingRate) {
  double hd = (double)h;
  double delta = 0.0;
  if (any_oct && h >= 2) delta = roct * (p * hd - baseline) / 1000.0;
  double r = (slope * lg2h) + delta;
  if (hd * p >= samplingRate / 2.0) r = -INFINITY;
  if (rolloffParab != 0.0) {
    if (parab_harm < 3) {
      if (h == 1) r = r + rolloffParab;
    } else if (h <= parab_harm) {
      r = r + pa * (hd * hd) + pb * hd + pc;
    }
  }
  if (r < throwaway) r = -INFINITY;
  return r;
}
SGB_HD double rolloff_db_l(int h, double lg2h, double p, double ro, double roct, double rk, bool any_oct,
                           double rolloffParab, int parab_harm, double pa, double pb, double pc,
                           double baseline, double throwaway, double samplingRate) {
  return rolloff_db_s(h, lg2h, p, ro + rk * (p - baseline) / 1000.0, roct, any_oct, rolloffParab, parab_harm,
                      pa, pb, pc, baseline, throwaway, samplingRate);
}

SGB_HD double rolloff_db(int h, double p, double ro, double roct, double rk, bool any_oct,
                         double rolloffParab, int parab_harm, double pa, double pb, double pc,
                         double baseline, double throwaway, double samplingRate) {
  return rolloff_db_l(h, log2((double)h), p, ro, roct, rk, any_oct, rolloffParab, parab_harm, pa, pb, pc,
                      baseline, throwaway, samplingRate);
}

// vibrato (R/source.R:208-213): element i (1-based) of the pitch contour.
SGB_HD double ctrl_vibrato(const sgb_syllable &sp, int i, double p) {
  if (!(sp.vibratoDep > 0.0)) return p;
  const double two_pi = 2.0 * 3.141592653589793;   // R: 2 * pi
  double v = exp2(sin(two_pi * (double)i * sp.vibratoFreq / sp.pitchSamplingRate) * sp.vibratoDep / 12.0);
  return p * v;
}

// ------------------------------------------------------- sequential stage ---
// Everything of generateHarmonics between the vibrato and the harmonic loop that is
// inherently sequential per syllable.  A.pitch must already hold the vibrato'd
// pitch contour.  ampl_contour: getSmoothContour(amplAnchors, len = nGC) is
// evaluated from atab / aknots, prepared with contour_prepare(len = 0, valueFloor = 0,
// valueCeiling = -throwaway); a loess fit is done here for len = nGC.
SGB_HD void ctrl_sequential(const sgb_syllable &sp, const double *anchors, const ContourTab *atab,
                            const double *aknots, const double *zpool, SylArrays &A, SylCtrl &C) {
  const int P = sp.pitch_len;
  const double psr = sp.pitchSamplingRate, sr = sp.samplingRate;
  const double *z = zpool + sp.z_off;
  int zi = 0;
  C.status = SGB_OK;
  C.nEpochs = 0; C.n_jidx = 0; C.vf_active = 0; C.rows_kept = 0; C.nHarmonics = 0;
  C.n_up = 0; C.out_len = 0; C.tiles = 0; C.tiles_tc = 0; C.pad_tc = 0; C.amp_elems = 0; C.wave_elems = 0; C.raw_max = 0.0;

  // getGlottalCycles (R/utilities_soundgen.R:477-486)
  int G = 0;
  {
    int i = 1;
    while (i < P) {
      if (G >= A.cap) { C.status = SGB_ERR_INVALID; return; }
      A.gc[G++] = i;
      double st = floor(psr / A.pitch[i - 1]);
      if (!(st >= 2.0)) st = 2.0;
      if (st > (double)P) st = (double)P;
      i = i + (int)st;
    }
  }
  C.nGC = G;
  if (G < 2) { C.status = SGB_ERR_SYNTH; return; }   // approx() needs two points (source.R:403)
  for (int g = 0; g < G; g++) A.ppg[g] = A.pitch[A.gc[g] - 1];

  // amplitude contour -> rolloffAmpl (source.R:221-235); t4 holds rolloffAmpl
  C.use_ampl = 0;
  if (sp.ampl_n > 0) {
    const double *an = anchors + 2 * sp.ampl_off;
    int cnt = 0;
    for (int i = 0; i < sp.ampl_n; i++) if (an[2 * i + 1] < -sp.throwaway) cnt++;
    if (cnt > 0) C.use_ampl = 1;
  }
  double *rolloffAmpl = A.t4;
  if (C.use_ampl) {
    // getSmoothContour(len = nGC, valueFloor = 0, valueCeiling = -throwaway, samplingRate)
    ContourTab T = *atab;
    contour_fit_len(&T, aknots, G, sp.samplingRate);
    if (T.status != SGB_OK) { C.status = T.status; return; }
    for (int g = 0; g < G; g++) {
      double v = contour_eval(&T, aknots, G, g);
      rolloffAmpl[g] = (v / fabs(sp.throwaway) - 1.0) * sp.rolloff_perAmpl;
    }
  } else {
    for (int g = 0; g < G; g++) rolloffAmpl[g] = 0.0;
  }

  // random walk for intra-syllable variation (source.R:238-262)
  const bool temp_on = sp.temperature > 0.0;
  double *vf_on = A.t1, *js_on = A.t2;    // vocalFry_on, jitter_on == shimmer_on
  if (temp_on) {
    if (!random_walk(G, sp.temperature, 0.3, true, sp.randomWalk_trendStrength, z, sp.z_cap, &zi,
                     A.rw, A.sb, A.sc, A.sd, A.phi, A.kt)) { C.status = SGB_ERR_STREAM; return; }
    // rw_0_100 = zeroOne(rw) * 100
    double mn = A.rw[0];
    for (int g = 1; g < G; g++) mn = fmin(mn, A.rw[g]);
    double mx = 0.0;
    for (int g = 0; g < G; g++) { A.t3[g] = A.rw[g] - mn; }
    mx = A.t3[0];
    for (int g = 1; g < G; g++) mx = fmax(mx, A.t3[g]);
    // getIntegerRandomWalk (utilities_math.R:352-387)
    if (sp.nonlinBalance == 0.0) {
      for (int g = 0; g < G; g++) A.rwbin[g] = 0;
    } else if (sp.nonlinBalance == 100.0) {
      for (int g = 0; g < G; g++) A.rwbin[g] = 2;
    } else {
      double q1, q2;
      noise_thresholds(sp.nonlinBalance, &q1, &q2);
      for (int g = 0; g < G; g++) {
        double v = A.t3[g] / mx * 100.0;
        A.rwbin[g] = (v > q2) ? 2 : ((v > q1) ? 1 : 0);
        A.sb[g] = ceil(sp.shortestEpoch / 1000.0 * A.ppg[g]);   // minLength
      }
      clumper(A.rwbin, G, A.sb, A.sc);
    }
    double m = r_mean(A.rw, G);
    for (int g = 0; g < G; g++) {
      A.rw[g] = A.rw[g] - m + 1.0;
      vf_on[g] = (A.rwbin[g] > 0) ? 1.0 : 0.0;
      js_on[g] = (A.rwbin[g] == 2) ? 1.0 : 0.0;
    }
  } else {
    for (int g = 0; g < G; g++) { A.rw[g] = 1.0; vf_on[g] = 1.0; js_on[g] = 1.0; A.rwbin[g] = 0; }
  }

  // jitter (source.R:265-290)
  if (sp.jitterDep > 0.0 && sp.nonlinBalance > 0.0) {
    int nj = 0;
    double cur = 1.0;     // tail(idx, 1), unrounded
    A.jidx[nj++] = 1;
    double i = 1.0;
    long guard = 0;
    double *ratio_g = A.t3;      // ratio = pitch_per_gc * jitterLen / 1000, one division per cycle
    for (int g = 0; g < G; g++) ratio_g[g] = A.ppg[g] * sp.jitterLen / 1000.0;
    while (i < (double)G) {
      double ratio = ratio_g[(int)i - 1];
      i = cur + ratio;
      cur = i;
      double r = rint(i);
      if (r <= (double)G) {
        int ri = (int)r;
        if (ri != A.jidx[nj - 1]) A.jidx[nj++] = ri;
      }
      if (++guard > 100000000L) { C.status = SGB_ERR_INVALID; return; }
    }
    C.n_jidx = nj;
    if (zi + nj > sp.z_cap) { C.status = SGB_ERR_STREAM; return; }
    // jitter = 2 ^ (rnorm(n, 0, jitterDep / 12) * rw[idx] * jitter_on[idx])
    double *jx = A.kt, *jy = A.phi;
    const double sd = sp.jitterDep / 12.0;
    for (int k = 0; k < nj; k++) {
      int gi = A.jidx[k] - 1;
      jx[k] = (double)A.jidx[k];
      jy[k] = exp2((0.0 + sd * z[zi + k]) * A.rw[gi] * js_on[gi]);
    }
    zi += nj;
    fmm_coef(nj, jx, jy, A.sb, A.sc, A.sd);
    const double jby = r_seq_by_step(jx[0], jx[nj - 1], G);
    for (int g = 0; g < G; g++) {
      double jg = r_spline_at_by(nj, jx, jy, A.sb, A.sc, A.sd, jby, G, g);
      A.ppg[g] = A.ppg[g] * jg;
    }
  }

  // slow random drift of f0 (source.R:293-320)
  if (temp_on) {
    double rw_smoothing = 0.9 - sp.temperature * sp.pitchDriftFreq -
                          1.2 / (1.0 + exp(-0.008 * ((double)G - 10.0))) + 0.6;
    double rw_range = sp.temperature * sp.pitchDriftDep + (double)G / 1000.0 / 12.0;
    if (!random_walk(G, rw_range, rw_smoothing, false, 0.0, z, sp.z_cap, &zi, A.drift,
                     A.sb, A.sc, A.sd, A.phi, A.kt)) { C.status = SGB_ERR_STREAM; return; }
    double m = r_mean(A.drift, G);
    for (int g = 0; g < G; g++) {
      A.drift[g] = exp2(A.drift[g] - m);
      A.ppg[g] = A.ppg[g] * A.drift[g];
    }
  } else {
    for (int g = 0; g < G; g++) A.drift[g] = 1.0;
  }

  // clamp (source.R:324-325)
  double pmin = INFINITY;
  for (int g = 0; g < G; g++) {
    if (A.ppg[g] > sp.pitchCeiling) A.ppg[g] = sp.pitchCeiling;
    if (A.ppg[g] < sp.pitchFloor) A.ppg[g] = sp.pitchFloor;
    pmin = fmin(pmin, A.ppg[g]);
  }
  C.nHarmonics = (int)ceil((sr / 2.0 - pmin) / pmin);    // source.R:329
  if (C.nHarmonics < 2) { C.status = SGB_ERR_SYNTH; return; }
  if (C.nHarmonics > A.hcap) { C.status = SGB_ERR_INVALID; return; }

  // per-gc arguments of getRolloff (source.R:331-341)
  C.any_oct = 0;
  for (int g = 0; g < G; g++) {
    double rw3 = (A.rw[g] == 1.0) ? 1.0 : pow(A.rw[g], 3.0);
    A.ro[g] = (sp.rolloff + rolloffAmpl[g]) * rw3;
    A.roct[g] = sp.rolloffOct * rw3;
    A.rk[g] = sp.rolloffKHz * A.rw[g];
    if (A.roct[g] != 0.0) C.any_oct = 1;
  }
  {
    double ph = rint(sp.rolloffParabHarm);
    if (ph == 2.0) ph = 3.0;
    C.parab_harm = (int)ph;
    if (C.parab_harm > C.nHarmonics) C.parab_harm = C.nHarmonics;  // R would fail: subscript out of bounds
    C.parab_a = -4.0 * sp.rolloffParab / ((ph - 1.0) * (ph - 1.0));
    C.parab_b = -C.parab_a * (1.0 + ph);
    C.parab_c = C.parab_a * ph;
  }

  // shimmer (source.R:348-357): drawn after getRolloff in the reference; the stream
  // order (jitter, drift, shimmer) is what matters.
  if (sp.shimmerDep > 0.0 && sp.nonlinBalance > 0.0) {
    if (zi + G > sp.z_cap) { C.status = SGB_ERR_STREAM; return; }
    const double sd = sp.shimmerDep / 100.0;
    for (int g = 0; g < G; g++)
      A.shimmer[g] = exp2((0.0 + sd * z[zi + g]) * A.rw[g] * js_on[g]);
    zi += G;
  } else {
    for (int g = 0; g < G; g++) A.shimmer[g] = 1.0;
  }
  C.z_used = zi;

  // vocal fry epochs (subharmonics.R:108-163)
  bool fry = (sp.subDep > 0.0 && sp.nonlinBalance > 0.0);
  int maxsub = 0;
  if (fry) {
    for (int g = 0; g < G; g++) {
      double rw4 = (A.rw[g] == 1.0) ? 1.0 : pow(A.rw[g], 4.0);
      double subFreq = sp.subFreq * rw4;
      A.subdep[g] = sp.subDep * rw4 * vf_on[g];
      double ns = rint(A.ppg[g] / subFreq) - 1.0;
      if (ns < 0.0) ns = 0.0;
      if (ns > 1.0e6) ns = 1.0e6;
      A.nsub[g] = (int)ns;
      if (A.nsub[g] > maxsub) maxsub = A.nsub[g];
    }
  }
  if (!fry || maxsub < 1) {
    for (int g = 0; g < G; g++) { A.nsub[g] = 0; }
    C.vf_active = 0;
    C.nEpochs = 1;
    C.ep_start[0] = 1; C.ep_end[0] = G; C.ep_nsub[0] = 0;
  } else {
    C.vf_active = 1;
    for (int g = 0; g < G; g++) A.sb[g] = rint(sp.shortestEpoch / (1000.0 / A.ppg[g]));
    if (G > 1) clumper(A.nsub, G, A.sb, A.sc);
    int ne = 0;
    int start = 1;
    for (int g = 1; g <= G; g++) {
      bool last = (g == G);
      if (last || A.nsub[g] != A.nsub[g - 1]) {
        if (ne >= SGB_MAX_EPOCHS) { C.status = SGB_ERR_UNSUPPORTED; return; }
        C.ep_start[ne] = start; C.ep_end[ne] = g; C.ep_nsub[ne] = A.nsub[g - 1];
        ne++;
        start = g + 1;
      }
    }
    C.nEpochs = ne;
  }
  for (int e = 0; e < C.nEpochs; e++)
    if (C.ep_end[e] - C.ep_start[e] + 1 < 2) { C.status = SGB_ERR_SYNTH; return; }  // approx needs 2 gcs

  // upsample (R/utilities_soundgen.R:392-416)
  {
    double c = 0.0;
    A.gcup[0] = 1;
    for (int g = 0; g < G; g++) {
      double len = rint(sr / A.ppg[g]);
      if (len < 4.0) { C.status = SGB_ERR_UNSUPPORTED; return; }   // glottal cycles shorter than 4 samples (f0 > sr/4)
      A.t3[g] = len;
      c += len;
      if (c > 2.0e9) { C.status = SGB_ERR_INVALID; return; }
      A.gcup[g + 1] = (int32_t)c;
    }
    int N = A.gcup[G];
    C.n_up = N;
    if (G == 2) {
      A.kt[0] = 1.0; A.kt[1] = (double)N;
      A.sb[0] = (A.ppg[1] - A.ppg[0]) / (double)(N - 1);   // seq(p1, p2, length.out = N)
      A.sb[1] = A.sb[0];
      A.sc[0] = A.sc[1] = A.sd[0] = A.sd[1] = 0.0;
      A.kt[1] = 2.0e9;   // single interval: every sample uses knot 0
    } else {
      A.kt[0] = 1.0;
      A.kt[G - 1] = (double)N;
      for (int g = 1; g < G - 1; g++) A.kt[g] = (double)A.gcup[g] + rint(A.t3[g] / 2.0);
      fmm_coef(G, A.kt, A.ppg, A.sb, A.sc, A.sd);
    }
    // phi[i] = sum_{v < kt[i]} pitch_upsampled[v]  (closed-form sums of the cubic pieces)
    CompSum acc;
    for (int i = 0; i < G; i++) {
      A.phi[i] = acc.value();
      if (i < G - 1 && A.kt[i + 1] < 1.9e9) {
        double M = A.kt[i + 1] - A.kt[i] - 1.0;     // last offset inside the piece
        double s1 = M * (M + 1.0) / 2.0;
        double s2 = M * (M + 1.0) * (2.0 * M + 1.0) / 6.0;
        double s3 = s1 * s1;
        acc.add(A.ppg[i] * (M + 1.0));
        acc.add(A.sb[i] * s1);
        acc.add(A.sc[i] * s2);
        acc.add(A.sd[i] * s3);
      }
    }
  }
}

#if !defined(__CUDACC__)
// Host builds of the scalar code: the same stage with the amplitude contour prepared here from the anchors,
// as k_syl_contours prepares it for K0 (no length: a loess fit is done above for len = nGC).
SGB_HD void ctrl_sequential(const sgb_syllable &sp, const double *anchors, const double *zpool, SylArrays &A,
                            SylCtrl &C) {
  ContourTab T{};
  std::vector<double> K((size_t)contour_knot_doubles(sp.ampl_n > 0 ? sp.ampl_n : 1));
  if (sp.ampl_n > 0)
    contour_prepare(&T, K.data(), anchors + 2 * sp.ampl_off, sp.ampl_n, 0, sp.samplingRate, true, 0.0, true,
                    -sp.throwaway, false, sp.ampl_method);
  ctrl_sequential(sp, anchors, &T, K.data(), zpool, A, C);
}
#endif

// column maximum of r[, g] (R/sourceSpectrum.R:146): one glottal cycle.
SGB_HD double ctrl_colmax(const sgb_syllable &sp, const SylArrays &A, const SylCtrl &C, int g) {
  double m = -INFINITY;
  for (int h = 1; h <= C.nHarmonics; h++) {
    double r = rolloff_db(h, A.ppg[g], A.ro[g], A.roct[g], A.rk[g], C.any_oct != 0,
                          sp.rolloffParab, C.parab_harm, C.parab_a, C.parab_b, C.parab_c,
                          200.0, sp.throwaway, sp.samplingRate);
    if (r > m) m = r;
  }
  return m;
}

// is harmonic h non-zero anywhere?  (R/sourceSpectrum.R:182)
SGB_HD bool ctrl_rowkept(const sgb_syllable &sp, const SylArrays &A, const SylCtrl &C, int h) {
  for (int g = 0; g < C.nGC; g++) {
    double r = rolloff_db(h, A.ppg[g], A.ro[g], A.roct[g], A.rk[g], C.any_oct != 0,
                          sp.rolloffParab, C.parab_harm, C.parab_a, C.parab_b, C.parab_c,
                          200.0, sp.throwaway, sp.samplingRate);
    if (r > -INFINITY) return true;
  }
  return false;
}

// sizes of the dense per-epoch amplitude matrices and of the K1 work list
// tc_min_rows: epochs with at least that many rows are synthesised by the tensor-core kernel (work list: one unit
// per interval of approx()), the others by the FP32-pipe kernel (work list: tiles of `tile` samples)
SGB_HD void ctrl_sizes(SylArrays &A, SylCtrl &C, int tile, int tc_min_rows = 1 << 30) {
  int64_t amp = 0, wave = 0;
  int tiles = 0;
  for (int e = 0; e < C.nEpochs; e++) {
    int n = C.ep_nsub[e];
    int rows = C.rows_kept * (n + 1) + n;        // multiples of f0/(n+1): j = 1..rows
    if (!C.vf_active || n == 0) rows = C.rows_kept;
    C.ep_rows[e] = rows;
    int Ge = C.ep_end[e] - C.ep_start[e] + 1;
    int Ne = A.gcup[C.ep_end[e]] - A.gcup[C.ep_start[e] - 1] + 1;
    C.ep_amp_off[e] = amp;
    C.ep_wave_off[e] = wave;
    amp += (int64_t)rows * Ge;
    wave += ((int64_t)Ne + 3) & ~(int64_t)3;
    if (rows < tc_min_rows) tiles += (Ne + tile - 1) / tile;
  }
  C.amp_elems = amp;
  C.wave_elems = wave;
  C.tiles = tiles;
  // tensor-core work list: one unit per interval of approx() of every epoch
  int tc = 0;
  for (int e = 0; e < C.nEpochs; e++)
    if (C.ep_rows[e] >= tc_min_rows) tc += C.ep_end[e] - C.ep_start[e];
  C.tiles_tc = tc;
}

// Exact (double) amplitude of dense row j (1-based multiple of f0/(nsub+1)) at
// glottal cycle g (0-based, absolute) of epoch e: rolloff matrix after shimmer and
// vocal fry (R/source.R:331-375, R/subharmonics.R:25-86 incl. the scalar-index
// quirk at :76-77: sub-harmonic amplitudes use column 1 of the epoch).
SGB_HD double ampl_exact(const sgb_syllable &sp, const SylArrays &A, const SylCtrl &C, int e,
                         int j, int g) {
  const int n = (C.vf_active ? C.ep_nsub[e] : 0);
  const double thr01 = exp2(sp.throwaway / 10.0);
  auto fh = [&](int k, int gg) -> double {      // f-harmonic k (kept-row index, 1-based)
    if (k < 1 || k > C.rows_kept) return 0.0;
    int h = A.rowmap[k - 1];
    double r = rolloff_db(h, A.ppg[gg], A.ro[gg], A.roct[gg], A.rk[gg], C.any_oct != 0,
                          sp.rolloffParab, C.parab_harm, C.parab_a, C.parab_b, C.parab_c,
                          200.0, sp.throwaway, sp.samplingRate);
    double v = exp2((r - A.colmax[gg]) / 10.0);
    return v * A.shimmer[gg];
  };
  if (n == 0) return fh(j, g);
  int k = j / (n + 1), s = j % (n + 1);
  double v;
  if (s == 0) {
    v = fh(k, g);
  } else {
    int g0 = C.ep_start[e] - 1;                  // first column of the epoch
    double lwr = fh(k, g0), upr = fh(k + 1, g0);
    double sw = A.subdep[g];
    double dl = A.ppg[g] * (double)s / (double)(n + 1);
    double du = A.ppg[g] * (double)(n + 1 - s) / (double)(n + 1);
    double ml, mu;
    if (sw == 0.0) { ml = 0.0; mu = 0.0; }
    else { ml = exp(-0.5 * (dl / sw) * (dl / sw)); mu = exp(-0.5 * (du / sw) * (du / sw)); }
    v = lwr * ml + upr * mu;
  }
  if (v < thr01) v = 0.0;
  return v;
}
