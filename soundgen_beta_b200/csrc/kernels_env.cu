// K4: spectral envelope -- getSpectralEnvelope (R/sourceSpectrum.R:261-566), the
// deterministic part: formant tracks -> gamma-density bumps + lip radiation + mouth
// opening + nasalisation -> 2^(dB/10).  One WARP per (column, instance) (four per CTA): the per-column
// set-up runs on a few lanes, so a whole CTA per column would leave most of its threads waiting for it.
#include "engine.cuh"
#include "contour.cuh"

#define ENV_THREADS 128
#define ENV_WARPS (ENV_THREADS / 32)
#define ENV_MAXF 64        // formants per filter (incl. stochastic extras and the nasal pole / zero)

template <typename OutT>
__global__ void __launch_bounds__(ENV_THREADS, 6)
k_envelope(const EnvInst *__restrict__ inst, const sgb_envelope *__restrict__ envs,
           const sgb_formant_ref *__restrict__ fidx, const double *__restrict__ formants,
           const double *__restrict__ formants_late, const double *__restrict__ trk,
           const double *__restrict__ mouth, const double *__restrict__ pre,
           OutT *__restrict__ out, int n_flat, int n_items) {
  // work item -> (instance, column): flat list (one item per warp; the instance is found by bisection
  // over col0) or the plain 2-D grid of the stand-alone API call (blockIdx.y = instance)
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int ii = blockIdx.y, c = (int)blockIdx.x * ENV_WARPS + wid;
  if (n_flat > 0) {
    const int item = c;
    if (item >= n_items) return;
    int lo = 0, hi = n_flat - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (inst[mid].col0 <= item) lo = mid; else hi = mid - 1;
    }
    ii = lo;
    c = item - inst[lo].col0;
  }
  const EnvInst I = inst[ii];
  if (c >= I.nc) return;
  const sgb_envelope E = envs[I.env_id];
  const int nr = I.nr, nc = I.nc;
  if (E.tracks_given == 2) {   // literal nr x nc matrix supplied by the caller (generateNoise's filterNoise)
    const double *m = pre + E.formant_off + (int64_t)c * nr;
    OutT *colL = out + I.out_off + (int64_t)c * nr;
    for (int r = lane; r < nr; r += 32) colL[r] = (OutT)m[r];
    return;
  }
  __shared__ double sf_freq[ENV_WARPS][ENV_MAXF], sf_amp[ENV_WARPS][ENV_MAXF], sf_width[ENV_WARPS][ENV_MAXF];
  __shared__ double sg_shape[ENV_WARPS][ENV_MAXF], sg_rate[ENV_WARPS][ENV_MAXF], sg_ref[ENV_WARPS][ENV_MAXF],
      sg_amp[ENV_WARPS][ENV_MAXF];
  __shared__ int s_nF[ENV_WARPS];
  __shared__ double s_mouth_open[ENV_WARPS], s_mouth_bin[ENV_WARPS];
  double *f_freq = sf_freq[wid], *f_amp = sf_amp[wid], *f_width = sf_width[wid];
  double *g_shape = sg_shape[wid], *g_rate = sg_rate[wid], *g_ref = sg_ref[wid], *g_amp = sg_amp[wid];
  const int F = E.n_formants;     // <= ENV_MAXF - 2, checked at upload

  // ---- formant values at column c (sourceSpectrum.R:321-344) ----
  for (int fl = lane; fl < F; fl += 32) {
    const sgb_formant_ref R = fidx[E.formant_off + fl];
    const double *rows = (R.pad ? formants_late : formants) + 4 * R.off;
    double val[3];
    if (E.tracks_given) {
      for (int j = 0; j < 3; j++) val[j] = rows[4 * c + 1 + j];
    } else if (R.n <= 1) {
      for (int j = 0; j < 3; j++) val[j] = rows[1 + j];
    } else {   // moving formant: evaluated once per instance by k_env_tracks
      const double *tv = trk + I.trk_off + ((int64_t)c * E.n_formants + fl) * 3;
      for (int j = 0; j < 3; j++) val[j] = tv[j];
    }
    f_freq[fl] = val[0]; f_amp[fl] = val[1]; f_width[fl] = val[2];
  }
  __syncwarp();

  // ---- Hz -> bins, mouth opening, nasalisation (sourceSpectrum.R:417-504) ----
  if (lane == 0) {
    double mo = 0.5, mb = 1.0;
    int n = 0;
    if (F > 0) {
      const double bin_width = E.samplingRate / 2.0 / (double)nr;
      if (E.mouth_n > 0) {
        mo = mouth[I.col0 + c];
        if (mo < E.mouthOpenThres) mo = 0.0;
        mb = (mo > 0.0) ? 1.0 : 0.0;
      }
      double adj = 0.0;
      if (isfinite(E.vocalTract)) {
        double adj_hz = (mo - 0.5) * E.speedSound / (4.0 * E.vocalTract);
        adj = (adj_hz - bin_width / 2.0) / bin_width + 1.0;
      }
      for (int f = 0; f < F; f++) {
        double fr = (f_freq[f] - bin_width / 2.0) / bin_width + 1.0;
        fr = fr + adj;
        if (fr < 1.0) fr = 1.0;
        f_freq[f] = fr;
        f_width[f] = f_width[f] / bin_width;
      }
      n = F;
      if (mb == 0.0) {   // nasalise: pole + zero, modified f1
        double f1f = f_freq[0], f1a = f_amp[0], f1w = f_width[0];
        double pf = (f1f > 550.0 / bin_width) ? f1f - 250.0 / bin_width : f1f + 250.0 / bin_width;
        f_freq[n] = pf; f_amp[n] = f1a * 2.0 / 3.0; f_width[n] = f1w * 2.0 / 3.0; n++;
        f_freq[n] = (pf + f1f) / 2.0; f_amp[n] = -f1a * 2.0 / 3.0; f_width[n] = f1w * 2.0 / 3.0; n++;
        f_amp[0] = f1a * 4.0 / 5.0; f_width[0] = f1w * 5.0 / 4.0;
      }
      for (int f = 0; f < n; f++) {   // gamma bumps (sourceSpectrum.R:507-520)
        double mg = f_freq[f], sdg = f_width[f];
        if (sdg == 0.0) sdg = 1.0;
        double shape = (mg * mg) / (sdg * sdg);
        double rate = mg / (sdg * sdg);
        // arg-max of dgamma over the integer bins 1..nr
        double xs = 1.0;
        if (shape > 1.0) {
          double mode = (shape - 1.0) / rate;
          double a = fmin(fmax(floor(mode), 1.0), (double)nr), b = fmin(fmax(ceil(mode), 1.0), (double)nr);
          double la = (shape - 1.0) * log(a) - rate * a, lb = (shape - 1.0) * log(b) - rate * b;
          xs = (lb > la) ? b : a;
        }
        g_shape[f] = shape; g_rate[f] = rate; g_amp[f] = f_amp[f];
        g_ref[f] = (shape - 1.0) * log(xs) - rate * xs;
      }
    }
    s_nF[wid] = n; s_mouth_open[wid] = mo; s_mouth_bin[wid] = mb;
  }
  __syncwarp();

  const int n = s_nF[wid];
  const double mouth_open = s_mouth_open[wid], mouth_bin = s_mouth_bin[wid];
  const double boost = exp2(mouth_open * E.openMouthBoost / 10.0);
  OutT *col = out + I.out_off + (int64_t)c * nr;
  if constexpr (sizeof(OutT) == 4) {
    // FP32 table for the filter kernels: the log-density difference stays in double (its terms cancel),
    // the exponentials and the dB sum run in FP32 (relative error of the result ~1e-6)
    const float fdep = (float)E.formantDep, lip = (float)(E.rolloffLip * mouth_bin), fboost = (float)boost;
    for (int r = lane; r < nr; r += 32) {
      const double x = (double)(r + 1), lx = log(x);
      float v = 0.0f;
      for (int f = 0; f < n; f++) {
        const double ld = (g_shape[f] - 1.0) * lx - g_rate[f] * x - g_ref[f];
        v = fmaf(expf((float)ld), (float)g_amp[f], v);
      }
      v = v * fdep;
      v = (v + lip * (float)(lx * 1.4426950408889634)) * fboost;
      col[r] = (OutT)exp2f(v / 10.0f);
    }
    return;
  }
  for (int r = lane; r < nr; r += 32) {
    double x = (double)(r + 1), lx = log(x);
    double v = 0.0;
    for (int f = 0; f < n; f++) {
      double ld = (g_shape[f] - 1.0) * lx - g_rate[f] * x - g_ref[f];
      v += exp(ld) * g_amp[f];
    }
    v = v * E.formantDep;
    v = (v + E.rolloffLip * log2(x) * mouth_bin) * boost;
    col[r] = (OutT)exp2(v / 10.0);
  }
}

// Pre-pass, one CTA per envelope instance: the formant tracks (sourceSpectrum.R:321-344:
// spline(approx(y, n = nPoints + 2^smoothLinearFactor, x = time)$y, n = nc)) and the mouth-opening
// contour (:436-443) depend on the column only through the evaluation point, so their coefficients
// are solved once per instance here and k_envelope just reads the per-column values.
// The mouth-opening contour's fit (a loess fit is a millisecond of FP64 on one thread): one thread per instance
// here, instead of thread 0 of every 128-thread CTA of k_env_tracks while the other 127 wait.
__global__ void k_mouth_tabs(const EnvInst *__restrict__ inst, int n_inst, const sgb_envelope *__restrict__ envs,
                             const double *__restrict__ anchors, ContourTab *__restrict__ tabs,
                             double *__restrict__ knots) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_inst) return;
  const EnvInst I = inst[i];
  const sgb_envelope E = envs[I.env_id];
  if (E.mouth_n > 0 && E.n_formants > 0 && E.tracks_given != 2) {
    // getSmoothContour(len = nc, mouthAnchors, valueFloor = 0, valueCeiling = 1): samplingRate is
    // not passed, so the span heuristic sees getSmoothContour's own default of 16000
    contour_prepare(&tabs[i], knots + I.mouth_koff, anchors + 2 * E.mouth_off, E.mouth_n, I.nc, 16000.0, true, 0.0,
                    true, 1.0, false, E.mouth_method);       // a failing fit is reported by the host (contour_fits)
  }
}

// knots: the envelope knot pool, written here (the mouth knots by k_mouth_tabs, the tracks' scratch below): plain
// loads, not the read-only path
__global__ void __launch_bounds__(ENV_THREADS)
k_env_tracks(const EnvInst *__restrict__ inst, const sgb_envelope *__restrict__ envs,
             const sgb_formant_ref *__restrict__ fidx, const double *__restrict__ formants,
             const ContourTab *__restrict__ tabs, double *knots, double *__restrict__ trk, double *__restrict__ mouth) {
  const EnvInst I = inst[blockIdx.x];
  const sgb_envelope E = envs[I.env_id];
  const int nc = I.nc, F = E.n_formants;
  __shared__ ContourTab T;
  if (E.mouth_n > 0 && F > 0 && E.tracks_given != 2) {
    contour_tab_load(&T, &tabs[blockIdx.x]);
    __syncthreads();
    const double *K = knots + I.mouth_koff;
    for (int c = threadIdx.x; c < nc; c += blockDim.x) mouth[I.col0 + c] = (T.status == SGB_OK) ? contour_eval(&T, K, nc, c) : 0.5;
  }
  if (I.trk_off < 0 || E.tracks_given) return;
  int nPoints = 0;
  for (int f = 0; f < F; f++) nPoints = max(nPoints, fidx[E.formant_off + f].n);
  const int na = (int)ceil((double)nPoints + exp2(E.smoothLinearFactor));
  const int64_t per = 2 * (int64_t)nPoints + 5 * (int64_t)na;     // scratch doubles per track
  // the coefficients: one thread per moving track, sequential FMM solve (tx, ty: the time points; ax, ay: approx())
  for (int t = threadIdx.x; t < 3 * F; t += blockDim.x) {
    const int f = t / 3, j = t % 3;
    const sgb_formant_ref R = fidx[E.formant_off + f];
    if (R.n <= 1) continue;
    const double *rows = formants + 4 * R.off;
    double *tx = knots + I.fit_off + t * per, *ty = tx + nPoints, *ax = ty + nPoints, *ay = ax + na;
    const int n = R.n;
    for (int i = 0; i < n; i++) { tx[i] = rows[4 * i]; ty[i] = rows[4 * i + 1 + j]; }
    for (int i = 0; i < na; i++) { ax[i] = (double)(i + 1); ay[i] = r_approx_at(n, tx, ty, na, i); }
    fmm_coef(na, ax, ay, ay + na, ay + 2 * na, ay + 3 * na);
  }
  __syncthreads();
  // the values: (column, track) pairs across the CTA, in the order of trk
  for (int64_t q = threadIdx.x; q < (int64_t)nc * 3 * F; q += blockDim.x) {
    const int c = (int)(q / (3 * F)), t = (int)(q - (int64_t)c * 3 * F);
    const int f = t / 3, j = t % 3;
    const sgb_formant_ref R = fidx[E.formant_off + f];
    double v;
    if (R.n <= 1) {
      v = formants[4 * R.off + 1 + j];
    } else {
      const double *ax = knots + I.fit_off + t * per + 2 * nPoints, *ay = ax + na;
      v = r_spline_at(na, ax, ay, ay + na, ay + 2 * na, ay + 3 * na, nc, c);
    }
    trk[I.trk_off + q] = v;
  }
}

void launch_env_tracks(const EnvInst *inst, int n_inst, const sgb_envelope *envs, const sgb_formant_ref *fidx,
                       const double *formants, const double *anchors, double *trk, double *mouth, void *tabs,
                       double *knots, cudaStream_t st) {
  if (n_inst <= 0) return;
  k_mouth_tabs<<<(n_inst + 31) / 32, 32, 0, st>>>(inst, n_inst, envs, anchors, (ContourTab *)tabs, knots);
  k_env_tracks<<<n_inst, ENV_THREADS, 0, st>>>(inst, envs, fidx, formants, (const ContourTab *)tabs, knots, trk, mouth);
}

void launch_envelope_f32(const EnvInst *inst, int n_inst, int max_nc, const sgb_envelope *envs,
                         const sgb_formant_ref *fidx, const double *formants, const double *formants_late,
                         const double *trk, const double *mouth, const double *pre, float *out, cudaStream_t st) {
  if (n_inst <= 0 || max_nc <= 0) return;
  // max_nc carries the TOTAL number of (instance, column) work items here: one warp each
  k_envelope<float><<<(max_nc + ENV_WARPS - 1) / ENV_WARPS, ENV_THREADS, 0, st>>>(inst, envs, fidx, formants, formants_late, trk, mouth, pre,
                                                                           out, n_inst, max_nc);
}
void launch_envelope_f64(const EnvInst *inst, int n_inst, int max_nc, const sgb_envelope *envs,
                         const sgb_formant_ref *fidx, const double *formants, const double *formants_late,
                         const double *trk, const double *mouth, const double *pre, double *out, cudaStream_t st) {
  if (n_inst <= 0 || max_nc <= 0) return;
  dim3 g((max_nc + ENV_WARPS - 1) / ENV_WARPS, n_inst);
  k_envelope<double><<<g, ENV_THREADS, 0, st>>>(inst, envs, fidx, formants, formants_late, trk, mouth, pre, out, 0, 0);
}
