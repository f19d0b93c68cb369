// Host front-end: the host stage of soundgen() (R/soundgen.R:279-733) behind the C ABI.
//
// What stays on the host in north_star: argument checks, hyper-parameters, syllable segmentation
// and every draw from R's RNG stream -- consumed here in the reference's order (SURVEY.md 8a "RNG
// ledger"): rbinom for fractional nSyl / repeatBout (soundgen.R:394-400); per bout rnorm_bounded for
// the syllable and pause durations (:485-506) and divideIntoSyllables (utilities_soundgen.R:515-551);
// per syllable nine rnorm_bounded draws (:549-562), wiggleAnchors for pitch / noise / amplitude
// (:563-590, utilities_soundgen.R:634-735), the normals generateHarmonics consumes (random walk,
// jitter, drift, shimmer: source.R:239-353 -- counted here, consumed on the device), stochastic
// noise formants + runif(nr * nc) (:659-696, source.R:111), and after the syllables the stochastic
// formants of the main filter (sourceSpectrum.R:346-415).  Nothing here computes samples.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <chrono>

#include "ctrl.cuh"
#include "rrng.h"
#include "hostpar.h"

int sgb_fail_msg(int code, const char *msg);   // engine.cu: sets the thread-local error string

namespace {

int ffail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  return sgb_fail_msg(code, buf);
}

// permittedValues (R/presets.R:22-79): default, low, high
struct Perm { const char *name; double dflt, lo, hi; };
const Perm PERM[] = {
    {"repeatBout", 1, 1, 20}, {"nSyl", 1, 1, 10}, {"sylLen", 300, 20, 5000}, {"pauseLen", 200, 20, 1000},
    {"temperature", .025, 0, 1}, {"maleFemale", 0, -1, 1}, {"creakyBreathy", 0, -1, 1},
    {"nonlinBalance", 0, 0, 100}, {"nonlinDep", 50, 0, 100}, {"jitterDep", 3, 0, 24}, {"jitterLen", 1, 1, 100},
    {"vibratoFreq", 5, 3, 10}, {"vibratoDep", 0, 0, 3}, {"shimmerDep", 0, 0, 100}, {"attackLen", 50, 0, 200},
    {"rolloff", -12, -60, 0}, {"rolloffOct", -12, -30, 10}, {"rolloffParab", 0, -50, 50},
    {"rolloffParabHarm", 3, 1, 20}, {"rolloffKHz", -6, -20, 0}, {"rolloffLip", 6, 0, 20},
    {"formantDep", 1, 0, 5}, {"formantDepStoch", 30, 0, 60}, {"vocalTract", 15.5, 2, 100},
    {"subFreq", 100, 10, 1000}, {"subDep", 100, 0, 500}, {"shortestEpoch", 300, 50, 500}, {"amDep", 0, 0, 100},
    {"amFreq", 30, 10, 100}, {"amShape", 0, -1, 1}, {"samplingRate", 16000, 8000, 44100},
    {"windowLength", 40, 5, 100}, {"rolloffNoise", -14, -20, 20}};
const int N_PERM = (int)(sizeof(PERM) / sizeof(PERM[0]));
const double PITCH_LO = 25, PITCH_HI = 3500, NOISE_LO = -120, NOISE_HI = 40, SYL_LO = 20, SYL_HI = 5000,
             PAUSE_LO = 20, PAUSE_HI = 1000;

const Perm *perm(const char *n) {
  for (int i = 0; i < N_PERM; i++) if (!strcmp(PERM[i].name, n)) return &PERM[i];
  return nullptr;
}

double r_round0(double x) { return std::nearbyint(x); }     // round half even (R < 4.0 fround(x, 0))

struct Anchors {
  std::vector<double> t, v;
  bool na() const { return v.empty(); }
  int n() const { return (int)v.size(); }
};

struct Formant { std::vector<double> time, freq, amp, width; int n() const { return (int)time.size(); } };

// rnorm_bounded (R/utilities_math.R:187-231), n values with per-element mean / sd, scalar bounds
void rnorm_bounded(RRng &g, int n, std::vector<double> mean, std::vector<double> sd, double low, double high,
                   bool roundToInteger, std::vector<double> &out) {
  for (auto &m : mean) { if (m < low) m = low; if (m > high) m = high; }     // with a warning in R
  if ((int)mean.size() < n) mean.assign(n, mean[0]);
  if ((int)sd.size() < n) sd.assign(n, sd[0]);
  bool any_sd = false;
  for (int i = 0; i < n; i++) if (sd[i] != 0) any_sd = true;
  out.assign(mean.begin(), mean.begin() + n);
  if (!any_sd) {
    if (roundToInteger) for (auto &o : out) o = r_round0(o);
    return;
  }
  for (int i = 0; i < n; i++) out[i] = g.rnorm(mean[i], sd[i]);
  if (roundToInteger) for (auto &o : out) o = r_round0(o);
  for (int i = 0; i < n; i++) {
    int guard = 0;
    while (out[i] < low || out[i] > high) {
      out[i] = g.rnorm(mean[i], sd[i]);
      if (roundToInteger) for (auto &o : out) o = r_round0(o);
      if (++guard > 100000000) break;
    }
  }
}
double rnorm_bounded1(RRng &g, double mean, double sd, double low, double high, bool roundToInteger) {
  std::vector<double> o;
  rnorm_bounded(g, 1, {mean}, {sd}, low, high, roundToInteger, o);
  return o[0];
}

// wiggleAnchors (R/utilities_soundgen.R:634-735) for a two-column data.frame (time, value)
void wiggle_anchors(RRng &g, Anchors &df, double temperature, double temp_coef, const double low[2],
                    const double high[2], bool wiggleAllRows) {
  if (df.na()) return;
  for (int i = 0; i < df.n(); i++) if (std::isnan(df.t[i]) || std::isnan(df.v[i])) return;
  const double pr[3] = {1 - temperature, temperature / 2, temperature / 2};
  int action = g.sample_prob1(pr, 3);          // 1 nothing, 2 remove, 3 add
  int nrow = df.n();
  if (action == 3) {
    if (nrow == 1) {
      std::vector<double> nw;
      rnorm_bounded(g, 1, {df.v[0]}, {df.v[0] * temperature * temp_coef}, low[1], high[1], false, nw);
      df.t.push_back(1.0); df.v.push_back(nw[0]);
      df.t[0] = 0.0;
    } else {
      int a1 = g.sample_int1(nrow);
      int direction = (g.sample_int1(2) == 1) ? -1 : 1;
      int a2 = (a1 + direction < 1 || a1 + direction > nrow) ? a1 - direction : a1 + direction;
      int i1 = std::min(a1, a2), i2 = std::max(a1, a2);
      // colMeans(df[i1:i2, ]) -- i1 and i2 are neighbours
      double nt = (df.t[i1 - 1] + df.t[i2 - 1]) / 2.0, nv = (df.v[i1 - 1] + df.v[i2 - 1]) / 2.0;
      df.t.insert(df.t.begin() + i1, nt);
      df.v.insert(df.v.begin() + i1, nv);
    }
  } else if (action == 2) {
    if (wiggleAllRows) {
      int idx = g.sample_int1(nrow);
      df.t.erase(df.t.begin() + (idx - 1)); df.v.erase(df.v.begin() + (idx - 1));
    } else if (nrow > 2) {
      int idx = 1 + g.sample_int1(nrow - 2);          // sampleModif(2:(nrow - 1), 1)
      df.t.erase(df.t.begin() + (idx - 1)); df.v.erase(df.v.begin() + (idx - 1));
    }
  }
  nrow = df.n();
  if (nrow < 1) return;
  const double orig0 = df.t[0], orig1 = df.t[nrow - 1];
  double ranges[2];
  if (nrow == 1) { ranges[0] = df.t[0]; ranges[1] = df.v[0]; }
  else {
    for (int c = 0; c < 2; c++) {
      const std::vector<double> &x = c ? df.v : df.t;
      double mn = x[0], mx = x[0];
      for (double e : x) { mn = std::fmin(mn, e); mx = std::fmax(mx, e); }
      ranges[c] = std::fabs(mx - mn);
      if (ranges[c] == 0) ranges[c] = std::fabs(x[0]);
    }
  }
  for (int c = 0; c < 2; c++) {
    std::vector<double> &x = c ? df.v : df.t;
    std::vector<double> w;
    rnorm_bounded(g, nrow, x, {ranges[c] * temperature * temp_coef}, low[c], high[c], false, w);
    x = w;
  }
  if (!wiggleAllRows) { df.t[0] = orig0; df.t[nrow - 1] = orig1; }
}

// getRandomWalk (R/utilities_math.R:289-326) with a scalar trend given lazily (R forces the promise
// `trend = rnorm(1)` only when len >= 2)
template <typename TrendFn>
void random_walk_host(RRng &g, int len, double rw_range, double rw_smoothing, TrendFn trend_fn, std::vector<double> &out) {
  if (len < 2) { out.assign(1, g.rgamma(1 / (rw_range * rw_range), 1.0 / (1 / (rw_range * rw_range)))); return; }
  double nf = std::floor(std::fmax(2.0, (rw_smoothing != 0.0) ? std::exp2(1.0 / rw_smoothing) : INFINITY));
  const double trend = trend_fn();
  out.resize(len);
  if (nf > (double)len) {
    CompSum acc;
    for (int i = 0; i < len; i++) { acc.add(g.rnorm(trend, 1.0)); out[i] = acc.value(); }
  } else {
    const int n = (int)nf;
    std::vector<double> x(n), y(n), b(n), c(n), d(n);
    CompSum acc;
    for (int i = 0; i < n; i++) { acc.add(g.rnorm(trend, 1.0)); y[i] = acc.value(); x[i] = (double)(i + 1); }
    fmm_coef(n, x.data(), y.data(), b.data(), c.data(), d.data());
    for (int k = 0; k < len; k++) out[k] = r_spline_at(n, x.data(), y.data(), b.data(), c.data(), d.data(), len, k);
  }
  double mn = out[0];
  for (double e : out) mn = std::fmin(mn, e);
  double mxabs = 0;
  for (auto &e : out) { e = e - mn; mxabs = std::fmax(mxabs, std::fabs(e)); }
  for (auto &e : out) e = e / mxabs * rw_range;
}

struct SylPars {   // pars_list / pars_syllable of soundgen.R:416-446
  double nonlinDep, attackLen, jitterDep, shimmerDep, rolloff, rolloffOct, shortestEpoch, subFreq, subDep;
};

struct CallState {
  sgb_soundgen_args a;          // scalars (pointers inside are not used after add)
  Anchors pitchAnchors, pitchAnchorsGlobal, noiseAnchors, mouthAnchors, amplAnchors, amplAnchorsGlobal;
  std::vector<Formant> formants, formantsNoise;
  bool has_formants = false, has_formantsNoise = false;
  RRng rng;
  bool use_rng = true;
  // rng_mode 2: the caller's buffers, by reference (they stay valid until the calls' last round has ended)
  struct Span { const void *p; int64_t n; };
  std::vector<Span> zbuf;                  // one stream of normals per voiced syllable
  std::vector<Span> ubuf;                  // one buffer of uniforms per noise (float or double: the handle's u type)
  size_t zi = 0, ui = 0;
  // derived by the host stage before the bout loop
  int nSyl = 1, repeatBout = 1, wl_points = 0;
  double jitterDep, shimmerDep, subDep, subFreq, rolloff, rolloffOct, nonlinBalance, vocalTract;
  std::vector<double> pitchDeltas;
  bool wiggleNoise = false, wiggleAmpl = false;
  int next_bout = 0;
  int status = SGB_OK;
  std::string warnings;
  int wl_running = -1;          // soundgen.R:743 persists across bouts
  // deferred main filter of the last bout emitted in the current round
  bool deferred = false;
  int deferred_env = -1, deferred_bout = -1;
  // a round may be run more than once (a bench step, a retry): every resolve of the same round restarts from the
  // stream position the first one found, so the same description always yields the same tracks
  bool resolved = false;
  RRng rng_pre;
};

struct Round {
  std::vector<sgb_call> calls;
  std::vector<sgb_bout> bouts;
  std::vector<sgb_syllable> syls;
  std::vector<sgb_noise> noises;
  std::vector<sgb_envelope> envs;
  std::vector<sgb_formant_ref> frefs;
  std::vector<double> pitch, anchors, formants, z, pre, u64;
  std::vector<float> u32;
  std::vector<int> sub_call;        // sub-call -> original call
  std::vector<int> syl_z_drawn;     // normals handed to each syllable (exact count in rng modes 0 / 1)
  std::vector<int> syl_call;
  int64_t virt_pitch = 0;           // doubles of device-evaluated pitch contours (work pool only)
  void clear() {
    virt_pitch = 0;
    calls.clear(); bouts.clear(); syls.clear(); noises.clear(); envs.clear(); frefs.clear(); pitch.clear();
    anchors.clear(); formants.clear(); z.clear(); pre.clear(); u64.clear(); u32.clear(); sub_call.clear();
    syl_z_drawn.clear(); syl_call.clear();
  }
};

// round_begin emits the calls on worker threads: every thread fills its own shard of the round (contiguous calls),
// the shards are concatenated in call order afterwards.  While a thread emits, this points at its shard.
static thread_local Round *tl_round = nullptr;

}  // namespace

struct sgb_frontend {
  int u_is_float = 0;
  std::vector<CallState> calls;
  Round R;
  std::vector<Round> shards;       // kept between rounds: their vectors keep their storage
  Round &round() { return tl_round ? *tl_round : R; }
  int64_t add_anchors(const Anchors &a, int32_t *n) {
    Round &R = round();
    int64_t off = (int64_t)(R.anchors.size() / 2);
    for (int i = 0; i < a.n(); i++) { R.anchors.push_back(a.t[i]); R.anchors.push_back(a.v[i]); }
    *n = a.n();
    return off;
  }
};

namespace {

void warn(CallState &C, const char *fmt, ...) {
  char buf[256];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (!C.warnings.empty()) C.warnings += "\n";
  C.warnings += buf;
}

Anchors take_anchors(const sgb_anchor_arg &A, double t_hi) {
  Anchors r;
  if (A.n <= 0 || !A.value) return r;
  r.v.assign(A.value, A.value + A.n);
  if (A.time) r.t.assign(A.time, A.time + A.n);
  else {       // numeric vector: time = seq(0, t_hi, length.out = n) (soundgen.R:305-315)
    r.t.resize(A.n);
    for (int i = 0; i < A.n; i++) r.t[i] = r_seq_at(0.0, t_hi, A.n, i);
  }
  return r;
}

std::vector<Formant> take_formants(const sgb_formant_arg *F, int n) {
  std::vector<Formant> out;
  for (int f = 0; f < n; f++) {
    const sgb_formant_arg &A = F[f];
    int rows = std::max(std::max(A.n_time, A.n_freq), std::max(A.n_amp, A.n_width));
    Formant fm;
    for (int i = 0; i < rows; i++) {      // as.data.frame recycles the shorter columns
      fm.time.push_back(A.time[i % A.n_time]); fm.freq.push_back(A.freq[i % A.n_freq]);
      fm.amp.push_back(A.amp[i % A.n_amp]); fm.width.push_back(A.width[i % A.n_width]);
    }
    out.push_back(fm);
  }
  return out;
}

// formants_upsampled of getSpectralEnvelope (sourceSpectrum.R:321-344): per formant nc rows of
// (time, freq, amp, width)
void upsample_formants(const std::vector<Formant> &fl, int nc, double smoothLinearFactor,
                       std::vector<std::vector<double>> &up /* [f][4 * nc] */) {
  int nPoints = 0;
  for (auto &f : fl) nPoints = std::max(nPoints, f.n());
  const int na = (int)std::ceil((double)nPoints + std::exp2(smoothLinearFactor));
  up.assign(fl.size(), std::vector<double>());
  for (size_t f = 0; f < fl.size(); f++) {
    const Formant &F = fl[f];
    up[f].resize(4 * (size_t)nc);
    const std::vector<double> *cols[4] = {&F.time, &F.freq, &F.amp, &F.width};
    for (int j = 0; j < 4; j++) {
      if (F.n() > 1) {
        std::vector<double> ax(na), ay(na), b(na), c(na), d(na);
        for (int i = 0; i < na; i++) { ax[i] = (double)(i + 1); ay[i] = r_approx_at(F.n(), F.time.data(), cols[j]->data(), na, i); }
        fmm_coef(na, ax.data(), ay.data(), b.data(), c.data(), d.data());
        for (int k = 0; k < nc; k++) up[f][4 * k + j] = r_spline_at(na, ax.data(), ay.data(), b.data(), c.data(), d.data(), nc, k);
      } else {
        for (int k = 0; k < nc; k++) up[f][4 * k + j] = (*cols[j])[0];
      }
    }
  }
}

// Stochastic block of getSpectralEnvelope (sourceSpectrum.R:346-415): extra pseudo-formants up to
// Nyquist - 1000 Hz, then a random-walk wiggle of every formant's freq / amp / width.
void stochastic_formants(RRng &g, std::vector<std::vector<double>> &up, int nc, double temperature, double formDrift,
                         double formDisp, double formantDep, double formantDepStoch, double vocalTract,
                         double samplingRate, double speedSound) {
  const double formantDispersion = 2 * speedSound / (4 * vocalTract);    // vocalTract is numeric in soundgen()
  const double sdG = formantDispersion * temperature * formDisp;
  int nF = (int)up.size();
  auto col_max = [&](int f, int j) { double m = -INFINITY; for (int k = 0; k < nc; k++) m = std::fmax(m, up[f][4 * k + j]); return m; };
  double freq_max = col_max(nF - 1, 1);
  const double rr = temperature * formDrift;
  if (!std::isnan(sdG) && formantDepStoch > 0) {
    while (freq_max < (samplingRate / 2 - 1000)) {
      if (nF >= 62) break;
      std::vector<double> rw;
      random_walk_host(g, nc, rr, 0.0, [] { return 0.0; }, rw);
      if (rw.size() > 1) { double m = r_mean(rw.data(), (int)rw.size()); for (auto &e : rw) e = e - m + 1; }
      std::vector<double> nw(4 * (size_t)nc);
      const double gf = g.rgamma(formantDispersion * formantDispersion / (sdG * sdG), 1.0 / (formantDispersion / (sdG * sdG)));
      for (int k = 0; k < nc; k++) {
        nw[4 * k] = up[0][4 * k];
        nw[4 * k + 1] = up[nF - 1][4 * k + 1] + r_round0(gf * rw[rw.size() > 1 ? k : 0]);
      }
      const double sh = (formantDep / temperature) * (formantDep / temperature);
      const double rate = formantDepStoch * formantDep / ((formantDepStoch * temperature) * (formantDepStoch * temperature));
      const double ga = g.rgamma(sh, 1.0 / rate);
      for (int k = 0; k < nc; k++) {
        nw[4 * k + 2] = r_round0(ga * rw[rw.size() > 1 ? k : 0]);
        nw[4 * k + 3] = 50 + (std::log2(nw[4 * k + 1]) - 5) * 20;
      }
      up.push_back(nw);
      nF++;
      freq_max = col_max(nF - 1, 1);
    }
  }
  for (int f = 0; f < nF; f++)
    for (int j = 1; j <= 3; j++) {
      std::vector<double> rw;
      random_walk_host(g, nc, rr, 0.3, [&] { return g.rnorm(0.0, 1.0); }, rw);
      if (rw.size() > 1) { double m = r_mean(rw.data(), (int)rw.size()); for (auto &e : rw) e = e - m + 1; }
      for (int k = 0; k < nc; k++) up[f][4 * k + j] = up[f][4 * k + j] * rw[rw.size() > 1 ? k : 0];
    }
}

// number of normals generateHarmonics will consume for this syllable (source.R:239-353), from the
// control-rate logic that determines it: glottal cycles of the vibrato'd contour and the jitter walk
int count_syllable_normals(const sgb_syllable &sp, const double *pitch, int P, int *nGC_out) {
  std::vector<double> pv(P);
  for (int i = 0; i < P; i++) pv[i] = ctrl_vibrato(sp, i + 1, pitch[i]);
  std::vector<int> gc;
  {
    int i = 1;
    while (i < P) {
      gc.push_back(i);
      double st = std::floor(sp.pitchSamplingRate / pv[i - 1]);
      if (!(st >= 2.0)) st = 2.0;
      if (st > (double)P) st = (double)P;
      i = i + (int)st;
    }
  }
  const int G = (int)gc.size();
  *nGC_out = G;
  if (G < 2) return 0;
  int n = 0;
  const bool temp_on = sp.temperature > 0.0;
  auto rw_count = [&](double smoothing, bool trend2) {
    double p = (smoothing != 0.0) ? std::exp2(1.0 / smoothing) : INFINITY;
    double nf = std::floor(std::fmax(2.0, p));
    if (trend2) nf = std::nearbyint(nf / 2.0) * 2.0;
    return (!(nf <= (double)G)) ? G : (int)nf;
  };
  if (temp_on) n += rw_count(0.3, true);
  if (sp.jitterDep > 0.0 && sp.nonlinBalance > 0.0) {
    int nj = 1, last = 1;
    double cur = 1.0, i = 1.0;
    long guard = 0;
    while (i < (double)G) {
      double ratio = pv[gc[(int)i - 1] - 1] * sp.jitterLen / 1000.0;
      i = cur + ratio;
      cur = i;
      double r = std::nearbyint(i);
      if (r <= (double)G) { int ri = (int)r; if (ri != last) { nj++; last = ri; } }
      if (++guard > 100000000L) break;
    }
    n += nj;
  }
  if (temp_on) {
    double sm = 0.9 - sp.temperature * sp.pitchDriftFreq - 1.2 / (1.0 + std::exp(-0.008 * ((double)G - 10.0))) + 0.6;
    n += rw_count(sm, false);
  }
  if (sp.shimmerDep > 0.0 && sp.nonlinBalance > 0.0) n += G;
  return n;
}

int seq_by_count(double from, double to, double by) {
  if (from == to) return 1;
  return (int)std::floor((to - from) / by + 1e-10) + 1;
}

}  // namespace

extern "C" {

int sgb_frontend_create(sgb_frontend **out, int32_t u_is_float) {
  if (!out) return ffail(SGB_ERR_INVALID, "null out pointer");
  sgb_frontend *fe = new sgb_frontend();
  fe->u_is_float = u_is_float ? 1 : 0;
  *out = fe;
  return SGB_OK;
}

void sgb_frontend_destroy(sgb_frontend *fe) { delete fe; }

// Parses one argument list into `C` (validation, defaults, copies of every table it points to); 0 or an error.
static int build_call(const sgb_frontend *fe, const sgb_soundgen_args *args, CallState &C) {
  C.a = *args;
  sgb_soundgen_args &a = C.a;
  // ---- range check against permittedValues (soundgen.R:279-302) ----
  double *vals[] = {&a.repeatBout, &a.nSyl, &a.sylLen, &a.pauseLen, &a.temperature, &a.maleFemale, &a.creakyBreathy,
                    &a.nonlinBalance, &a.nonlinDep, &a.jitterDep, &a.jitterLen, &a.vibratoFreq, &a.vibratoDep,
                    &a.shimmerDep, &a.attackLen, &a.rolloff, &a.rolloffOct, &a.rolloffParab, &a.rolloffParabHarm,
                    &a.rolloffKHz, &a.rolloffLip, &a.formantDep, &a.formantDepStoch, &a.vocalTract, &a.subFreq, &a.subDep,
                    &a.shortestEpoch, &a.amDep, &a.amFreq, &a.amShape, &a.samplingRate, &a.windowLength, &a.rolloffNoise};
  for (int i = 0; i < N_PERM; i++) {
    double v = *vals[i];
    if (std::isnan(v) || v < PERM[i].lo || v > PERM[i].hi) {
      if (a.invalidArgAction == 1) {
        return ffail(SGB_ERR_INVALID, "%s must be between %g and %g", PERM[i].name, PERM[i].lo, PERM[i].hi);
      } else if (a.invalidArgAction == 2) {
        warn(C, "%s outside its range in 'permittedValues'", PERM[i].name);
      } else {
        *vals[i] = PERM[i].dflt;
        warn(C, "%s outside permitted range, reset to %g", PERM[i].name, PERM[i].dflt);
      }
    }
  }
  if (!(a.samplingRate > 0) || !(a.pitchSamplingRate > 0) || !(a.pitchFloor > 0) || !(a.throwaway < 0)) {
    return ffail(SGB_ERR_INVALID, "samplingRate, pitchSamplingRate, pitchFloor must be positive and throwaway negative");
  }
  C.pitchAnchors = take_anchors(a.pitchAnchors, 1.0);
  C.pitchAnchorsGlobal = take_anchors(a.pitchAnchorsGlobal, 1.0);
  C.amplAnchors = take_anchors(a.amplAnchors, 1.0);
  C.amplAnchorsGlobal = take_anchors(a.amplAnchorsGlobal, 1.0);
  C.mouthAnchors = take_anchors(a.mouthAnchors, 1.0);
  C.noiseAnchors = take_anchors(a.noiseAnchors, a.sylLen);
  C.has_formants = a.n_formants > 0 && a.formants;
  C.has_formantsNoise = a.n_formantsNoise > 0 && a.formantsNoise;
  if (C.has_formants) C.formants = take_formants(a.formants, a.n_formants);
  if (C.has_formantsNoise) C.formantsNoise = take_formants(a.formantsNoise, a.n_formantsNoise);
  // tempEffects defaults (soundgen.R:320-326; sylLenDep has none: the signature's .02 must come from the caller)
  const double te_dflt[8] = {.02, .3, .2, .5, .125, .05, .1, .1};
  for (int i = 0; i < 8; i++) if (std::isnan(a.tempEffects[i])) a.tempEffects[i] = te_dflt[i];
  // random stream
  C.use_rng = (a.rng_mode != 2);
  C.rng.rejection_sampling = a.sample_rejection != 0;
  if (a.rng_mode == 0) C.rng.set_seed(a.seed);
  else if (a.rng_mode == 1) {
    if (!a.rng_state) { return ffail(SGB_ERR_INVALID, "rng_mode 1 needs rng_state"); }
    C.rng.set_state(a.rng_state);
  } else {
    if (a.temperature > 0) {
      return ffail(SGB_ERR_UNSUPPORTED, "temperature > 0 draws from R's stream on the host: use rng_mode 0 / 1 (a seed), "
                                        "caller buffers only cover the device draws");
    }
    const double *zp = a.z;
    for (int i = 0; i < a.n_z; i++) { C.zbuf.push_back(CallState::Span{zp, a.z_len[i]}); zp += a.z_len[i]; }
    if (fe->u_is_float) {
      const float *up = (const float *)a.u;
      for (int i = 0; i < a.n_u; i++) { C.ubuf.push_back(CallState::Span{up, a.u_len[i]}); up += a.u_len[i]; }
    } else {
      const double *up = (const double *)a.u;
      for (int i = 0; i < a.n_u; i++) { C.ubuf.push_back(CallState::Span{up, a.u_len[i]}); up += a.u_len[i]; }
    }
  }
  C.wl_points = (int)(std::floor(a.windowLength / 1000 * a.samplingRate / 2) * 2);      // :317
  // ---- hyper-parameters (:337-379) ----
  C.nonlinBalance = a.nonlinBalance; C.jitterDep = a.jitterDep; C.shimmerDep = a.shimmerDep; C.subDep = a.subDep;
  if (a.creakyBreathy < 0) {
    C.nonlinBalance = std::fmin(100, C.nonlinBalance - a.creakyBreathy * 50);
    C.jitterDep = std::fmax(0, C.jitterDep - a.creakyBreathy / 2);
    C.shimmerDep = std::fmax(0, C.shimmerDep - a.creakyBreathy * 5);
    C.subDep = C.subDep * std::pow(2.0, -a.creakyBreathy);
  } else if (a.creakyBreathy > 0) {
    C.noiseAnchors.t = {0.0, a.sylLen + 100};
    double v = -120 + a.creakyBreathy * 160;
    if (v > NOISE_HI) v = NOISE_HI;
    C.noiseAnchors.v = {v, v};
  }
  C.rolloff = a.rolloff - a.creakyBreathy * 10;
  C.rolloffOct = a.rolloffOct - a.creakyBreathy * 5;
  C.subFreq = 2 * (a.subFreq - 50) / (1 + std::exp(-.1 * (50 - a.nonlinDep))) + 50;
  C.jitterDep = 2 * C.jitterDep / (1 + std::exp(.1 * (50 - a.nonlinDep)));
  C.vocalTract = a.vocalTract;
  if (a.maleFemale != 0) {
    const double k2 = std::pow(2.0, a.maleFemale), k125 = std::pow(1.25, a.maleFemale);
    for (auto &v : C.pitchAnchors.v) v = v * k2;
    for (auto &f : C.formants) for (auto &q : f.freq) q = q * k125;
    C.vocalTract = C.vocalTract * (1 - .25 * a.maleFemale);
  }
  // ---- stochastic rounding of nSyl / repeatBout (:394-400) ----
  {
    double fl = std::floor(a.nSyl);
    C.nSyl = (int)(fl + (C.use_rng ? C.rng.rbinom(1, a.nSyl - fl) : 0.0));
    fl = std::floor(a.repeatBout);
    C.repeatBout = (int)(fl + (C.use_rng ? C.rng.rbinom(1, a.repeatBout - fl) : 0.0));
  }
  if (C.nSyl < 1 || C.repeatBout < 1) { return ffail(SGB_ERR_INVALID, "nSyl and repeatBout must be at least 1"); }
  // ---- pitchDeltas (:448-462): getDiscreteContour(len = nSyl, method = 'spline') ----
  C.pitchDeltas.assign(C.nSyl, 1.0);
  {
    bool any_nz = false;
    for (double v : C.pitchAnchorsGlobal.v) if (v != 0) any_nz = true;
    if (!C.pitchAnchorsGlobal.na() && any_nz && C.nSyl > 1) {
      std::vector<double> an;
      for (int i = 0; i < C.pitchAnchorsGlobal.n(); i++) { an.push_back(C.pitchAnchorsGlobal.t[i]); an.push_back(C.pitchAnchorsGlobal.v[i]); }
      ContourTab T;
      std::vector<double> K((size_t)contour_knot_doubles(C.pitchAnchorsGlobal.n()));
      contour_prepare(&T, K.data(), an.data(), C.pitchAnchorsGlobal.n(), C.nSyl, 16000.0, false, 0, false, 0, false,
                      SGB_CONTOUR_SPLINE);
      if (T.status != SGB_OK) { return ffail(T.status, "pitchAnchorsGlobal: no anchors"); }
      for (int s = 0; s < C.nSyl; s++) C.pitchDeltas[s] = std::pow(2.0, contour_eval(&T, K.data(), C.nSyl, s) / 12);
    }
  }
  // ---- pitchAnchors$time to 0..1 (:465-472) ----
  if (!C.pitchAnchors.na()) {
    double mn = C.pitchAnchors.t[0], mx;
    for (double t : C.pitchAnchors.t) mn = std::fmin(mn, t);
    if (mn < 0) for (auto &t : C.pitchAnchors.t) t = t - mn;
    mx = C.pitchAnchors.t[0];
    for (double t : C.pitchAnchors.t) mx = std::fmax(mx, t);
    if (mx > 1) for (auto &t : C.pitchAnchors.t) t = t / mx;
  }
  {
    int cnt = 0;
    for (double v : C.noiseAnchors.v) if (v > a.throwaway) cnt++;
    C.wiggleNoise = a.temperature > 0 && !C.noiseAnchors.na() && cnt > 0;
    cnt = 0;
    for (double v : C.amplAnchors.v) if (v < -a.throwaway) cnt++;
    C.wiggleAmpl = a.temperature > 0 && !C.amplAnchors.na() && cnt > 0;
  }
  return SGB_OK;
}

int sgb_frontend_add(sgb_frontend *fe, const sgb_soundgen_args *args) {
  if (!fe || !args) return ffail(SGB_ERR_INVALID, "null argument");
  fe->calls.emplace_back();
  int rc = build_call(fe, args, fe->calls.back());
  if (rc < 0) { fe->calls.pop_back(); return rc; }
  return (int)fe->calls.size() - 1;
}

/* n calls that differ only in their seed (call i = set.seed(seeds[i]); soundgen(<args>)): the data-generation
 * sweep registers one preset a few thousand times without crossing the binding once per call. */
int sgb_frontend_add_seeded(sgb_frontend *fe, const sgb_soundgen_args *args, const uint32_t *seeds, int32_t n) {
  if (!fe || !args || !seeds || n < 1) return ffail(SGB_ERR_INVALID, "bad argument");
  if (args->rng_mode != 0) return ffail(SGB_ERR_INVALID, "sgb_frontend_add_seeded needs rng_mode 0");
  int first = -1;
  for (int i = 0; i < n; i++) {
    sgb_soundgen_args a = *args;
    a.seed = seeds[i];
    int rc = sgb_frontend_add(fe, &a);
    if (rc < 0) return rc;
    if (i == 0) first = rc;
  }
  return first;
}

// n argument lists at once (one library call instead of n: a binding marshals its calls into an array once).
int sgb_frontend_add_many(sgb_frontend *fe, const sgb_soundgen_args *args, int32_t n) {
  if (!fe || !args || n < 1) return ffail(SGB_ERR_INVALID, "bad argument");
  const size_t base = fe->calls.size();
  fe->calls.resize(base + (size_t)n);
  std::vector<int> rcs((size_t)n, 0);
  parallel_for(n, [&](int i) { rcs[i] = build_call(fe, &args[i], fe->calls[base + i]); });
  for (int i = 0; i < n; i++)
    if (rcs[i] < 0) {                       // the message belongs to a worker thread: produce it again on this one
      CallState tmp;
      int rc = build_call(fe, &args[i], tmp);
      fe->calls.resize(base);
      return rc < 0 ? rc : rcs[i];
    }
  return (int)base;
}

// Forget every registered call (the handle and its buffers are reused for the next batch).
int sgb_frontend_clear(sgb_frontend *fe) {
  if (!fe) return ffail(SGB_ERR_INVALID, "null argument");
  fe->calls.clear();
  fe->R.clear();
  return SGB_OK;
}

}  // extern "C"

namespace {

// One envelope specification (the argument munging of sourceSpectrum.R:294-315 happens here).
// tracks: host-drawn formants_upsampled (stochastic) or nullptr; deferred: tracks come after run_begin.
int add_envelope(sgb_frontend *fe, CallState &C, const std::vector<Formant> *fl, bool has_f, int nc_fixed,
                 const std::vector<std::vector<double>> *tracks, int tracks_nc, bool deferred) {
  Round &R = fe->round();
  const sgb_soundgen_args &a = C.a;
  sgb_envelope e;
  memset(&e, 0, sizeof e);
  std::vector<Formant> schwa;
  double vocalTract = C.vocalTract;
  if (!has_f) {       // formants NA: schwa from vocalTract (sourceSpectrum.R:303-315)
    double freq = 35400.0 / 4 / vocalTract;
    Formant f;
    f.time = {0}; f.freq = {freq}; f.amp = {30}; f.width = {50 * (1 + freq * freq / 6 / 1e6)};
    schwa.push_back(f);
    fl = &schwa;
  }
  e.formant_off = (int64_t)R.frefs.size();
  e.tracks_given = 0;
  if (deferred) {
    e.tracks_given = 3; e.n_formants = 0;
  } else if (tracks) {
    e.tracks_given = 1;
    e.n_formants = (int)tracks->size();
    for (auto &t : *tracks) {
      sgb_formant_ref r; r.off = (int64_t)(R.formants.size() / 4); r.n = tracks_nc; r.pad = 0;
      R.frefs.push_back(r);
      R.formants.insert(R.formants.end(), t.begin(), t.end());
    }
  } else {
    e.n_formants = (int)fl->size();
    for (auto &f : *fl) {
      sgb_formant_ref r; r.off = (int64_t)(R.formants.size() / 4); r.n = f.n(); r.pad = 0;
      R.frefs.push_back(r);
      for (int i = 0; i < f.n(); i++) { R.formants.push_back(f.time[i]); R.formants.push_back(f.freq[i]); R.formants.push_back(f.amp[i]); R.formants.push_back(f.width[i]); }
    }
  }
  bool mouth_ok = !C.mouthAnchors.na();
  for (double v : C.mouthAnchors.v) if (std::isnan(v)) mouth_ok = false;
  if (mouth_ok) e.mouth_off = fe->add_anchors(C.mouthAnchors, &e.mouth_n);
  e.mouth_method = a.contour_method;
  e.nc_fixed = nc_fixed;
  e.formantDep = a.formantDep; e.rolloffLip = a.rolloffLip; e.mouthOpenThres = 0; e.openMouthBoost = 0;
  e.vocalTract = vocalTract; e.samplingRate = a.samplingRate; e.speedSound = 35400; e.smoothLinearFactor = 1;
  R.envs.push_back(e);
  return (int)R.envs.size() - 1;
}

bool formants_moving(const std::vector<Formant> &fl) {
  for (auto &f : fl) if (f.n() > 1) return true;
  return false;
}

// Emits bout `b` of call C into the round.  Returns false when the round must stop after this bout
// (its main filter is deferred and later bouts draw after it).
bool emit_bout(sgb_frontend *fe, int ci, int b) {
  CallState &C = fe->calls[ci];
  Round &R = fe->round();
  const sgb_soundgen_args &a = C.a;
  RRng &g = C.rng;
  const double T = a.temperature, sr = a.samplingRate;
  const double sylLenDep = a.tempEffects[0];
  // ---- syllable segmentation (:483-516) ----
  double sylDur_s = a.sylLen;
  if (a.sylLen >= SYL_LO && a.sylLen <= SYL_HI)
    sylDur_s = rnorm_bounded1(g, a.sylLen, (SYL_HI - SYL_LO) * T * sylLenDep, SYL_LO, SYL_HI, false);
  double pauseDur_s = rnorm_bounded1(g, a.pauseLen, (PAUSE_HI - PAUSE_LO) * T * sylLenDep, PAUSE_LO, PAUSE_HI, false);
  std::vector<double> st, en;
  if (C.nSyl == 1) { st.push_back(0.0); en.push_back(sylDur_s); }
  else {
    const double Td = T * sylLenDep;
    double c = 0;
    while ((int)st.size() < C.nSyl) {
      double dur = rnorm_bounded1(g, sylDur_s, sylDur_s * Td, SYL_LO, SYL_HI, false);
      double pau = rnorm_bounded1(g, pauseDur_s, pauseDur_s * Td, PAUSE_LO, PAUSE_HI, false);
      double s0 = 1 + c, e0 = s0 + dur;
      st.push_back(s0); en.push_back(e0);
      c = e0 + pau;
    }
  }
  const int ns = (int)st.size();
  std::vector<double> startIdx(ns);
  for (int s = 0; s < ns; s++) startIdx[s] = r_round0(st[s] * sr / 1000);     // :517-532
  startIdx[0] = 1;
  if (!C.noiseAnchors.na() && C.noiseAnchors.t[0] != 0) {
    double shift = -r_round0(C.noiseAnchors.t[0] * sr / 1000);
    if (C.noiseAnchors.t[0] < 0) startIdx[0] = startIdx[0] - shift;
    else for (auto &v : startIdx) v = v - shift;
  }
  const int syl_begin = (int)R.syls.size(), noise_begin = (int)R.noises.size();
  bool has_noise = false;
  { int cnt = 0; for (double v : C.noiseAnchors.v) if (v > a.throwaway) cnt++; has_noise = !C.noiseAnchors.na() && cnt > 0; }
  const SylPars base = {a.nonlinDep, a.attackLen, C.jitterDep, C.shimmerDep, C.rolloff, C.rolloffOct, a.shortestEpoch, C.subFreq, C.subDep};
  for (int s = 0; s < ns; s++) {          // :540
    SylPars ps = base;
    Anchors pitchA = C.pitchAnchors, amplA = C.amplAnchors;
    if (T > 0) {                          // :546-591
      struct { const char *nm; double *dst; double mean; bool rnd; } pv[9] = {
          {"nonlinDep", &ps.nonlinDep, base.nonlinDep, false}, {"attackLen", &ps.attackLen, base.attackLen, true},
          {"jitterDep", &ps.jitterDep, base.jitterDep, false}, {"shimmerDep", &ps.shimmerDep, base.shimmerDep, false},
          {"rolloff", &ps.rolloff, base.rolloff, false}, {"rolloffOct", &ps.rolloffOct, base.rolloffOct, false},
          {"shortestEpoch", &ps.shortestEpoch, base.shortestEpoch, false}, {"subFreq", &ps.subFreq, base.subFreq, true},
          {"subDep", &ps.subDep, base.subDep, true}};
      for (int p = 0; p < 9; p++) {
        const Perm *pm = perm(pv[p].nm);
        *pv[p].dst = rnorm_bounded1(g, pv[p].mean, (pm->hi - pm->lo) * T / 10, pm->lo, pm->hi, pv[p].rnd);
      }
      if (!pitchA.na()) {
        const double lo[2] = {0, PITCH_LO}, hi[2] = {1, PITCH_HI};
        wiggle_anchors(g, pitchA, T, a.tempEffects[5], lo, hi, false);
      }
      if (C.wiggleNoise) {                 // result is overwritten at :646, the draws are consumed
        Anchors tmp = C.noiseAnchors;
        const double lo[2] = {-INFINITY, NOISE_LO}, hi[2] = {INFINITY, NOISE_HI};
        wiggle_anchors(g, tmp, T, a.tempEffects[6], lo, hi, true);
      }
      if (C.wiggleAmpl) {
        const double lo[2] = {0, 0}, hi[2] = {1, -a.throwaway};
        wiggle_anchors(g, amplA, T, a.tempEffects[7], lo, hi, false);
      }
    }
    const double dur_syl = en[s] - st[s];
    int pause = 0;
    if (s < ns - 1) pause = (int)std::floor((st[s + 1] - en[s]) * sr / 1000);
    double noise_min = INFINITY;
    for (double v : C.noiseAnchors.v) noise_min = std::fmin(noise_min, v);
    const bool silent = dur_syl < SYL_LO || (!C.noiseAnchors.na() && noise_min >= 40) || pitchA.na();
    sgb_syllable y;
    memset(&y, 0, sizeof y);
    y.pause_after = pause;
    if (silent) {
      y.kind = 0;
      y.silent_len = (int)r_round0(dur_syl * sr / 1000);
      R.syls.push_back(y); R.syl_z_drawn.push_back(0); R.syl_call.push_back(ci);
    } else {
      y.kind = 1;
      y.pitch_len = (int)r_round0(dur_syl * a.pitchSamplingRate / 1000);
      if (y.pitch_len < 3) { C.status = SGB_ERR_SYNTH; y.kind = 0; y.silent_len = 0; R.syls.push_back(y); R.syl_z_drawn.push_back(0); R.syl_call.push_back(ci); continue; }
      y.pitch_off = (int64_t)R.pitch.size();
      y.pitch_scale = C.pitchDeltas[s];
      y.pitch_method = a.contour_method;
      y.ampl_method = a.contour_method;
      int32_t npa = 0;
      y.pitch_anchor_off = fe->add_anchors(pitchA, &npa);
      y.reserved0 = 1;                    // pitch_anchor_off is set (merge_shard rebases it)
      if (!amplA.na()) y.ampl_off = fe->add_anchors(amplA, &y.ampl_n);
      y.attackLen = ps.attackLen; y.nonlinBalance = C.nonlinBalance; y.jitterDep = ps.jitterDep; y.jitterLen = a.jitterLen;
      y.vibratoFreq = a.vibratoFreq; y.vibratoDep = a.vibratoDep; y.shimmerDep = ps.shimmerDep; y.rolloff = ps.rolloff;
      y.rolloffOct = ps.rolloffOct; y.rolloffKHz = a.rolloffKHz; y.rolloffParab = a.rolloffParab;
      y.rolloffParabHarm = a.rolloffParabHarm; y.rolloff_perAmpl = 12; y.temperature = T;
      y.pitchDriftDep = a.tempEffects[3]; y.pitchDriftFreq = a.tempEffects[4]; y.randomWalk_trendStrength = .5;
      y.shortestEpoch = ps.shortestEpoch; y.subFreq = ps.subFreq; y.subDep = ps.subDep; y.samplingRate = sr;
      y.pitchFloor = a.pitchFloor; y.pitchCeiling = a.pitchCeiling; y.pitchSamplingRate = a.pitchSamplingRate;
      y.throwaway = a.throwaway;
      // does the device need a host count of the normals?  (any draw at all?)
      const bool draws = (T > 0) || (C.nonlinBalance > 0 && (ps.jitterDep > 0 || ps.shimmerDep > 0));
      const bool need_host_pitch = (C.use_rng && draws) || !a.device_pitch;
      int zdrawn = 0;
      if (need_host_pitch) {
        // pitchContour_syl = getSmoothContour(...) * pitchDeltas[s]  (:596-603)
        std::vector<double> an;
        for (int i = 0; i < pitchA.n(); i++) { an.push_back(pitchA.t[i]); an.push_back(pitchA.v[i]); }
        ContourTab Tb;
        std::vector<double> Kb((size_t)contour_knot_doubles(pitchA.n()));
        contour_prepare(&Tb, Kb.data(), an.data(), pitchA.n(), y.pitch_len, a.pitchSamplingRate, true, a.pitchFloor, true,
                        a.pitchCeiling, true, a.contour_method);
        if (Tb.status != SGB_OK) { C.status = Tb.status; y.kind = 0; y.silent_len = 0; R.syls.push_back(y); R.syl_z_drawn.push_back(0); R.syl_call.push_back(ci); continue; }
        R.pitch.resize(R.pitch.size() + y.pitch_len);
        double *pc = R.pitch.data() + y.pitch_off;
        for (int i = 0; i < y.pitch_len; i++) pc[i] = contour_eval(&Tb, Kb.data(), y.pitch_len, i) * C.pitchDeltas[s];
        y.pitch_anchor_n = 0;             // the device reads the contour the host evaluated
        if (C.use_rng && draws) {
          int nGC = 0;
          zdrawn = count_syllable_normals(y, pc, y.pitch_len, &nGC);
          y.z_off = (int64_t)R.z.size();
          y.z_cap = zdrawn;
          for (int i = 0; i < zdrawn; i++) R.z.push_back(g.norm_rand());
        }
      } else {
        y.pitch_anchor_n = npa;           // evaluated on the device: its slot lies behind the host pool in the
        y.pitch_off = -1 - R.virt_pitch;  // device's work pool (offset fixed up once the host pool is complete)
        R.virt_pitch += y.pitch_len;
      }
      if (!C.use_rng) {
        if (C.zi < C.zbuf.size()) {
          const double *zp = (const double *)C.zbuf[C.zi].p;
          y.z_off = (int64_t)R.z.size(); y.z_cap = (int)C.zbuf[C.zi].n;
          R.z.insert(R.z.end(), zp, zp + C.zbuf[C.zi].n);
        }
        C.zi++;
        zdrawn = -1;
      }
      R.syls.push_back(y); R.syl_z_drawn.push_back(zdrawn); R.syl_call.push_back(ci);
    }
    if (has_noise) {                       // :643-698
      Anchors na = C.noiseAnchors;
      double tmin = INFINITY, tmax = -INFINITY;
      for (auto &t : na.t) { if (t > 0) t = t * dur_syl / a.sylLen; tmin = std::fmin(tmin, t); tmax = std::fmax(tmax, t); }
      const double rng_t = tmax - tmin;
      sgb_noise N;
      memset(&N, 0, sizeof N);
      N.len = (int)r_round0(rng_t * sr / 1000);
      N.insertion = (int)startIdx[s];
      N.mix = C.has_formantsNoise ? 1 : 0;
      N.wl = C.wl_points;
      N.env_id = -1;
      N.strength_pre_off = -1;
      N.anchor_method = a.contour_method;
      N.rolloffNoise = a.rolloffNoise; N.attackLen = a.attackLen; N.samplingRate = sr; N.overlap = a.overlap;
      if (N.len < 1 || N.wl < 4 || (N.wl & 1)) { C.status = SGB_ERR_UNSUPPORTED; continue; }
      if (C.has_formantsNoise) {
        // :662: max(unlist(lapply(formantsNoise, length))) > 1 is TRUE for any formant list (length of a
        // data.frame is its number of columns), so the noise filter always has one column per 10 ms
        int nInt = (int)r_round0(rng_t / 10);
        if (nInt < 1) { C.status = SGB_ERR_SYNTH; continue; }
        if (T > 0) {
          std::vector<std::vector<double>> up;
          upsample_formants(C.formantsNoise, nInt, 1.0, up);
          stochastic_formants(g, up, nInt, T, a.tempEffects[1], a.tempEffects[2], a.formantDep, a.formantDepStoch,
                              C.vocalTract, sr, 35400.0);
          N.env_id = add_envelope(fe, C, &C.formantsNoise, true, nInt, &up, nInt, false);
        } else {
          N.env_id = add_envelope(fe, C, &C.formantsNoise, true, nInt, nullptr, 0, false);
        }
      }
      N.anchor_off = fe->add_anchors(na, &N.anchor_n);
      const double h = N.wl - (a.overlap * N.wl / 100.0);
      const int64_t nu = (int64_t)(N.wl / 2) * seq_by_count(1.0, (double)N.len + N.wl, h);
      N.u_off = fe->u_is_float ? (int64_t)R.u32.size() : (int64_t)R.u64.size();
      if (C.use_rng) {
        // (no reserve(size + nu) here: an exact-size reserve per segment would re-copy the whole pool every time)
        if (fe->u_is_float) {
          const size_t o = R.u32.size();
          R.u32.resize(o + (size_t)nu);           // geometric growth; filled in place
          float *dst = R.u32.data() + o;
          for (int64_t i = 0; i < nu; i++) dst[i] = (float)g.unif_rand();
        } else {
          const size_t o = R.u64.size();
          R.u64.resize(o + (size_t)nu);
          double *dst = R.u64.data() + o;
          for (int64_t i = 0; i < nu; i++) dst[i] = g.unif_rand();
        }
      } else {
        bool ok = C.ui < C.ubuf.size() && C.ubuf[C.ui].n >= nu;
        if (!ok) { C.status = SGB_ERR_STREAM; C.ui++; continue; }
        if (fe->u_is_float) { const float *up = (const float *)C.ubuf[C.ui].p; R.u32.insert(R.u32.end(), up, up + nu); }
        else { const double *up = (const double *)C.ubuf[C.ui].p; R.u64.insert(R.u64.end(), up, up + nu); }
        C.ui++;
      }
      R.noises.push_back(N);
    }
  }
  // ---- amplAnchorsGlobal (:721-724: converted in place, so a later bout sees converted values) ----
  sgb_bout B;
  memset(&B, 0, sizeof B);
  {
    int cnt = 0;
    for (double v : C.amplAnchorsGlobal.v) if (v < -a.throwaway) cnt++;
    if (!C.amplAnchorsGlobal.na() && cnt > 0) {
      for (auto &v : C.amplAnchorsGlobal.v) v = std::pow(2.0, v / 10);
      B.aglobal_off = fe->add_anchors(C.amplAnchorsGlobal, &B.aglobal_n);
    }
  }
  B.aglobal_method = a.contour_method;
  // ---- main filter (:751-775) ----
  bool moving = C.has_formants && formants_moving(C.formants);
  { int cnt = 0; for (double v : C.mouthAnchors.v) if (v != .5) cnt++; if (!C.mouthAnchors.na() && cnt > 0) moving = true; }
  bool deferred = false;
  int env_main;
  if (T > 0 && C.use_rng) {                 // stochastic formants: getSpectralEnvelope draws at :762
    if (moving) {
      env_main = add_envelope(fe, C, &C.formants, C.has_formants, 0, nullptr, 0, true);   // nc is the device's
      deferred = true;
    } else {
      std::vector<std::vector<double>> up;
      std::vector<Formant> schwa;
      const std::vector<Formant> *fl = &C.formants;
      if (!C.has_formants) {
        double freq = 35400.0 / 4 / C.vocalTract;
        Formant f; f.time = {0}; f.freq = {freq}; f.amp = {30}; f.width = {50 * (1 + freq * freq / 6 / 1e6)};
        schwa.push_back(f); fl = &schwa;
      }
      upsample_formants(*fl, 1, 1.0, up);
      stochastic_formants(g, up, 1, T, a.tempEffects[1], a.tempEffects[2], a.formantDep, a.formantDepStoch, C.vocalTract, sr, 35400.0);
      env_main = add_envelope(fe, C, fl, true, 0, &up, 1, false);
    }
  } else {
    env_main = add_envelope(fe, C, &C.formants, C.has_formants, 0, nullptr, 0, false);
  }
  const int n_sil = std::isnan(a.addSilence) ? 0 : (int)r_round0(sr / 1000 * a.addSilence);
  B.syl_begin = syl_begin; B.syl_end = (int)R.syls.size();
  B.noise_begin = noise_begin; B.noise_end = (int)R.noises.size();
  B.env_id = env_main; B.moving = moving ? 1 : 0;
  B.wl = (C.wl_running > 0) ? C.wl_running : C.wl_points;
  B.lead_silence = (b == 0) ? n_sil : (int)(a.pauseLen * sr / 1000);       // :836-849
  B.tail_silence = (b == C.repeatBout - 1) ? n_sil : 0;
  B.overlap = a.overlap; B.amDep = a.amDep; B.amFreq = a.amFreq; B.amShape = a.amShape; B.samplingRate = sr;
  B.throwaway = a.throwaway;
  R.bouts.push_back(B);
  C.deferred = deferred;
  if (deferred) { C.deferred_env = env_main; C.deferred_bout = (int)R.bouts.size() - 1; }
  return !(deferred && b < C.repeatBout - 1);
}

// One call's share of a round: its next bouts into the current round (fe->round()).
static void emit_call(sgb_frontend *fe, int ci) {
  Round &R = fe->round();
  CallState &C = fe->calls[ci];
  C.deferred = false;
  C.resolved = false;
  if (C.next_bout >= C.repeatBout || C.status != SGB_OK) return;
  sgb_call cl;
  cl.bout_begin = (int)R.bouts.size();
  while (C.next_bout < C.repeatBout) {
    bool go_on = emit_bout(fe, ci, C.next_bout);
    C.next_bout++;
    if (!go_on) break;
  }
  cl.bout_end = (int)R.bouts.size();
  R.calls.push_back(cl);
  R.sub_call.push_back(ci);
}

template <typename T>
static void append(std::vector<T> &dst, const std::vector<T> &src) { dst.insert(dst.end(), src.begin(), src.end()); }

// Appends shard S to R: every index and pool offset of S is relative to S and is rebased.
static void merge_shard(sgb_frontend *fe, Round &R, const Round &S) {
  const int b_bout = (int)R.bouts.size(), b_syl = (int)R.syls.size(), b_noise = (int)R.noises.size(), b_env = (int)R.envs.size();
  const int64_t b_fref = (int64_t)R.frefs.size(), b_pitch = (int64_t)R.pitch.size(), b_anchor = (int64_t)(R.anchors.size() / 2);
  const int64_t b_formant = (int64_t)(R.formants.size() / 4), b_z = (int64_t)R.z.size(), b_pre = (int64_t)R.pre.size();
  const int64_t b_u = fe->u_is_float ? (int64_t)R.u32.size() : (int64_t)R.u64.size(), b_virt = R.virt_pitch;
  for (sgb_call c : S.calls) { c.bout_begin += b_bout; c.bout_end += b_bout; R.calls.push_back(c); }
  for (sgb_bout b : S.bouts) {
    b.syl_begin += b_syl; b.syl_end += b_syl; b.noise_begin += b_noise; b.noise_end += b_noise;
    if (b.env_id >= 0) b.env_id += b_env;
    if (b.aglobal_n > 0) b.aglobal_off += b_anchor;     // unused offsets stay what the serial loop writes (0)
    R.bouts.push_back(b);
  }
  for (sgb_syllable y : S.syls) {
    if (y.pitch_off < 0) y.pitch_off -= b_virt;                    // virtual: -1 - offset
    else if (y.pitch_len > 0) y.pitch_off += b_pitch;
    if (y.z_cap > 0) y.z_off += b_z;
    if (y.ampl_n > 0) y.ampl_off += b_anchor;
    if (y.reserved0 & 1) y.pitch_anchor_off += b_anchor;
    R.syls.push_back(y);
  }
  for (sgb_noise n : S.noises) {
    n.u_off += b_u;
    if (n.anchor_n > 0) n.anchor_off += b_anchor;
    if (n.env_id >= 0) n.env_id += b_env;
    if (n.strength_pre_off >= 0) n.strength_pre_off += b_pre;
    R.noises.push_back(n);
  }
  for (sgb_envelope e : S.envs) {
    e.formant_off += (e.tracks_given == 2) ? b_pre : b_fref;
    if (e.mouth_n > 0) e.mouth_off += b_anchor;
    R.envs.push_back(e);
  }
  for (sgb_formant_ref r : S.frefs) { r.off += b_formant; R.frefs.push_back(r); }
  for (int ci : S.sub_call) {
    CallState &C = fe->calls[ci];
    if (C.deferred) { C.deferred_env += b_env; C.deferred_bout += b_bout; }
  }
  append(R.pitch, S.pitch); append(R.anchors, S.anchors); append(R.formants, S.formants); append(R.z, S.z);
  append(R.pre, S.pre); append(R.u64, S.u64); append(R.u32, S.u32);
  append(R.sub_call, S.sub_call); append(R.syl_z_drawn, S.syl_z_drawn); append(R.syl_call, S.syl_call);
  R.virt_pitch += S.virt_pitch;
}

}  // namespace

extern "C" {

int sgb_param_range(const char *name, double out3[3]) {
  const Perm *q = name ? perm(name) : nullptr;
  if (!q) return ffail(SGB_ERR_INVALID, "no permitted range for %s", name ? name : "(null)");
  if (!out3) return ffail(SGB_ERR_INVALID, "null out3");
  out3[0] = q->dflt; out3[1] = q->lo; out3[2] = q->hi;
  return SGB_OK;
}

// test hook: worker threads of the host stage (0 = SGB_FRONTEND_THREADS / the default)
int sgb_host_set_threads(int32_t n) { sgb_host_threads_override().store(n > 0 ? n : 0); return SGB_OK; }

int sgb_frontend_round_begin(sgb_frontend *fe, sgb_batch_desc *D, int32_t *n_subcalls) {
  if (!fe || !D || !n_subcalls) return ffail(SGB_ERR_INVALID, "null argument");
  Round &R = fe->R;
  R.clear();
  const int ncall = (int)fe->calls.size();
  const int ov = sgb_host_threads_override().load();
  const int T = std::min(ov > 0 ? ov : sgb_host_threads(), ncall / 16);
  if (T <= 1) {
    for (int ci = 0; ci < ncall; ci++) emit_call(fe, ci);
  } else {
    // contiguous shards of calls, one thread each, concatenated in call order: the description is the one the
    // serial loop builds, byte for byte (tests/test_host_api.py)
    if ((int)fe->shards.size() < T) fe->shards.resize(T);
    parallel_for(T, [&](int t) {
      Round &S = fe->shards[t];
      S.clear();
      tl_round = &S;
      const int lo = (int)((int64_t)ncall * t / T), hi = (int)((int64_t)ncall * (t + 1) / T);
      for (int ci = lo; ci < hi; ci++) emit_call(fe, ci);
      tl_round = nullptr;
    }, 1);
    for (int t = 0; t < T; t++) merge_shard(fe, R, fe->shards[t]);
  }
  for (auto &y : R.syls)
    if (y.kind == 1 && y.pitch_off < 0) y.pitch_off = (int64_t)R.pitch.size() + (-1 - y.pitch_off);
  *n_subcalls = (int)R.calls.size();
  memset(D, 0, sizeof *D);
  if (R.calls.empty()) return SGB_OK;
  if (R.anchors.empty()) R.anchors.assign(2, 0.0);
  D->n_calls = (int)R.calls.size(); D->n_bouts = (int)R.bouts.size(); D->n_syllables = (int)R.syls.size();
  D->n_noises = (int)R.noises.size(); D->n_envelopes = (int)R.envs.size(); D->n_formant_refs = (int)R.frefs.size();
  D->calls = R.calls.data(); D->bouts = R.bouts.data(); D->syllables = R.syls.data(); D->noises = R.noises.data();
  D->envelopes = R.envs.data(); D->formant_index = R.frefs.data();
  D->pitch = R.pitch.data(); D->n_pitch = (int64_t)R.pitch.size();
  D->anchors = R.anchors.data(); D->n_anchors = (int64_t)(R.anchors.size() / 2);
  D->formants = R.formants.data(); D->n_formants = (int64_t)(R.formants.size() / 4);
  D->z = R.z.data(); D->n_z = (int64_t)R.z.size();
  if (fe->u_is_float) { D->u = R.u32.data(); D->n_u = (int64_t)R.u32.size(); }
  else { D->u = R.u64.data(); D->n_u = (int64_t)R.u64.size(); }
  D->u_is_float = fe->u_is_float;
  D->pre = R.pre.data(); D->n_pre = (int64_t)R.pre.size();
  return SGB_OK;
}

int sgb_frontend_resolve(sgb_frontend *fe, sgb_batch *b) {
  if (!fe || !b) return ffail(SGB_ERR_INVALID, "null argument");
  struct Job { CallState *C; int ncol, nint; std::vector<double> rows; int nf; };
  std::vector<Job> jobs;
  for (auto &C : fe->calls) {
    if (!C.deferred) continue;
    if (C.resolved) C.rng = C.rng_pre;
    else { C.rng_pre = C.rng; C.resolved = true; }
    int32_t nc = 0, nint = 0, wl = 0, slen = 0;
    int rc = sgb_batch_bout_geometry(b, C.deferred_bout, &nc, &nint, &wl, &slen);
    if (rc != SGB_OK) return rc;
    Job j; j.C = &C; j.nint = nint; j.nf = 0;
    j.ncol = std::max(1, nint);        // a bypassed bout has no filter: draw as for one column
    jobs.push_back(std::move(j));
  }
  const bool trace = getenv("SGB_TRACE_HOST") != nullptr;
  auto t0 = std::chrono::steady_clock::now();
  parallel_for((int)jobs.size(), [&](int i) {
    Job &J = jobs[i];
    CallState &C = *J.C;
    const sgb_soundgen_args &a = C.a;
    std::vector<Formant> schwa;
    const std::vector<Formant> *fl = &C.formants;
    if (!C.has_formants) {
      double freq = 35400.0 / 4 / C.vocalTract;
      Formant f; f.time = {0}; f.freq = {freq}; f.amp = {30}; f.width = {50 * (1 + freq * freq / 6 / 1e6)};
      schwa.push_back(f); fl = &schwa;
    }
    std::vector<std::vector<double>> up;
    upsample_formants(*fl, J.ncol, 1.0, up);
    if (J.nint >= 1)    // sum(sound) == 0 skips the filter block, and with it the draws (soundgen.R:736-739)
      stochastic_formants(C.rng, up, J.ncol, a.temperature, a.tempEffects[1], a.tempEffects[2], a.formantDep,
                          a.formantDepStoch, C.vocalTract, a.samplingRate, 35400.0);
    for (auto &t : up) J.rows.insert(J.rows.end(), t.begin(), t.end());
    J.nf = (int)up.size();
  });
  auto t1 = std::chrono::steady_clock::now();
  for (auto &J : jobs) {
    int rc = sgb_batch_set_tracks(b, J.C->deferred_env, J.rows.data(), J.nf, J.ncol);
    if (rc != SGB_OK) return rc;
  }
  if (trace) {
    auto t2 = std::chrono::steady_clock::now();
    size_t bytes = 0;
    for (auto &J : jobs) bytes += J.rows.size() * 8;
    fprintf(stderr, "resolve: %zu calls, draw %.1f ms (parallel), set_tracks %.1f ms, %.1f MB of tracks\n", jobs.size(),
            std::chrono::duration<double, std::milli>(t1 - t0).count(), std::chrono::duration<double, std::milli>(t2 - t1).count(),
            bytes / 1e6);
  }
  return SGB_OK;
}

int sgb_frontend_round_end(sgb_frontend *fe, sgb_batch *b) {
  if (!fe || !b) return ffail(SGB_ERR_INVALID, "null argument");
  Round &R = fe->round();
  std::vector<int32_t> st(R.calls.size()), zu(R.syls.size());
  int rc = sgb_batch_status(b, st.data());
  if (rc != SGB_OK) return rc;
  rc = sgb_batch_z_used(b, zu.data());
  if (rc != SGB_OK) return rc;
  for (size_t k = 0; k < R.calls.size(); k++) {
    CallState &C = fe->calls[R.sub_call[k]];
    if (st[k] != SGB_OK && C.status == SGB_OK) C.status = st[k];
    // soundgen.R:743 mutates windowLength_points for the later bouts too
    int32_t nc, nint, wl, slen;
    for (int bi = R.calls[k].bout_begin; bi < R.calls[k].bout_end; bi++)
      if (sgb_batch_bout_geometry(b, bi, &nc, &nint, &wl, &slen) == SGB_OK && wl > 0) C.wl_running = wl;
  }
  for (size_t s = 0; s < R.syls.size(); s++) {
    if (R.syl_z_drawn[s] < 0 || R.syls[s].kind != 1) continue;
    CallState &C = fe->calls[R.syl_call[s]];
    if (C.status == SGB_OK && zu[s] != R.syl_z_drawn[s]) {
      C.status = SGB_ERR_STREAM;     // host and device disagree on the draw count: the stream is off
      warn(C, "syllable %d: the device consumed %d normals, the host had counted %d", (int)s, zu[s], R.syl_z_drawn[s]);
    }
  }
  return SGB_OK;
}

int sgb_frontend_round_calls(sgb_frontend *fe, int32_t *out) {
  if (!fe || !out) return ffail(SGB_ERR_INVALID, "null argument");
  for (size_t k = 0; k < fe->R.sub_call.size(); k++) out[k] = fe->R.sub_call[k];
  return SGB_OK;
}

int sgb_frontend_status(sgb_frontend *fe, int32_t *out) {
  if (!fe || !out) return ffail(SGB_ERR_INVALID, "null argument");
  for (size_t c = 0; c < fe->calls.size(); c++) out[c] = fe->calls[c].status;
  return SGB_OK;
}

const char *sgb_frontend_warnings(sgb_frontend *fe, int32_t call) {
  if (!fe || call < 0 || call >= (int)fe->calls.size()) return "";
  return fe->calls[call].warnings.c_str();
}

int sgb_frontend_rng_state(sgb_frontend *fe, int32_t call, int32_t *out625) {
  if (!fe || !out625 || call < 0 || call >= (int)fe->calls.size()) return ffail(SGB_ERR_INVALID, "bad argument");
  fe->calls[call].rng.get_state(out625);
  return SGB_OK;
}

int64_t sgb_frontend_h2d_bytes(sgb_frontend *fe) {
  if (!fe) return 0;
  const Round &R = fe->R;
  return (int64_t)(8 * (R.pitch.size() + R.anchors.size() + R.formants.size() + R.z.size() + R.pre.size() + R.u64.size()) +
                   4 * R.u32.size() + sizeof(sgb_syllable) * R.syls.size() + sizeof(sgb_bout) * R.bouts.size() +
                   sizeof(sgb_noise) * R.noises.size() + sizeof(sgb_envelope) * R.envs.size() +
                   sizeof(sgb_formant_ref) * R.frefs.size());
}

int sgb_rng_draw(uint32_t seed, int32_t kind, double p1, double p2, int32_t skip_uniforms, double *out, int32_t n) {
  if (!out || n < 0) return ffail(SGB_ERR_INVALID, "bad argument");
  RRng g;
  g.set_seed(seed);
  for (int i = 0; i < skip_uniforms; i++) g.unif_rand();
  for (int i = 0; i < n; i++) {
    switch (kind) {
      case 0: out[i] = g.unif_rand(); break;
      case 1: out[i] = g.norm_rand(); break;
      case 2: out[i] = g.exp_rand(); break;
      case 3: out[i] = g.rgamma(p1, 1.0 / p2); break;
      case 4: out[i] = g.rbinom(p1, p2); break;
      case 5: out[i] = (double)g.sample_int1((int)p1); break;
      default: return ffail(SGB_ERR_INVALID, "unknown kind");
    }
  }
  return SGB_OK;
}

int sgb_smooth_contour(const double *time, const double *value, int32_t n, int32_t len, double samplingRate,
                       int32_t has_floor, double valueFloor, int32_t has_ceiling, double valueCeiling,
                       int32_t thisIsPitch, int32_t method, double *out) {
  if (!value || !out || n < 1 || len < 1) return ffail(SGB_ERR_INVALID, "bad argument");
  std::vector<double> an(2 * (size_t)n);
  for (int i = 0; i < n; i++) { an[2 * i] = time ? time[i] : r_seq_at(0.0, 1.0, n, i); an[2 * i + 1] = value[i]; }
  ContourTab T;
  std::vector<double> K((size_t)contour_knot_doubles(n));
  contour_prepare(&T, K.data(), an.data(), n, len, samplingRate, has_floor != 0, valueFloor, has_ceiling != 0, valueCeiling,
                  thisIsPitch != 0, method);
  if (T.status != SGB_OK) return ffail(T.status, "getSmoothContour: loess() stops (span is too small)");
  for (int k = 0; k < len; k++) out[k] = contour_eval(&T, K.data(), len, k);
  return SGB_OK;
}

}  // extern "C"
