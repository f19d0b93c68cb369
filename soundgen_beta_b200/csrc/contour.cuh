// getSmoothContour (R/smoothContours.R:53-227) as a two-step scalar host/device routine:
// contour_prepare() turns the anchors into a small header plus knot storage once (one thread, or the host
// front-end), contour_eval() evaluates element k of the contour from them (any thread).
//   1 anchor: flat; 2 anchors: seq(); 3-10 anchors: loess (rloess.cuh) unless method 'spline';
//   more than 10 anchors: FMM spline, any number of knots.
// The knots live in storage the caller provides, contour_knot_doubles(na) doubles laid out x | y | b | c | d
// (n each): the host passes a vector, the device a slice of the batch's knot pool.  A spline's knots are
// normalised to [0, 1] and do not depend on the evaluation length; a loess fit does (contour_fit_len()).
#pragma once
#include "rloess.cuh"

#define SGB_CONTOUR_LOESS 0    // the reference's default method
#define SGB_CONTOUR_SPLINE 1

struct ContourTab {
  int kind;        // 0 flat, 1 seq between two anchors, 2 FMM spline, 3 loess
  int n;           // spline knots (kind 2), anchors (kind 3)
  int pitch;       // thisIsPitch: smooth on the semitone scale, return Hz
  int status;      // SGB_OK or SGB_ERR_*
  int has_lo, has_hi;
  double lo, hi;   // valueFloor / valueCeiling on the smoothing scale
  double v0, v1;
  double x0, x1;   // first and last knot (kind 2): the ends of the evaluation grid
  LoessFit L;
};

SGB_HD int64_t contour_knot_doubles(int na) { return 5 * (int64_t)na; }

SGB_HD double hz_to_semitones(double h) { return log2(h / 16.3516) * 12.0; }       // utilities_math.R:16-18
SGB_HD double semitones_to_hz(double s) { return 16.3516 * exp2(s / 12.0); }       // utilities_math.R:25-27

// The loess branch only: fits the anchors kept in K (x | y) for a contour of len points.
SGB_HD void contour_fit_len(ContourTab *T, const double *K, int len, double samplingRate) {
  if (T->kind != 3 || T->status != SGB_OK) return;
  const double duration_ms = (double)len / samplingRate * 1000.0;
  contour_loess_fit(T->n, K, K + T->n, len, duration_ms, T->has_lo != 0, T->lo, &T->L);
  if (T->L.status != 0) T->status = SGB_ERR_SYNTH;        // loess() stops: the reference call fails
}

// an: interleaved (time, value) anchors.  K: contour_knot_doubles(na) doubles.  len: points of the contour;
// samplingRate only enters the loess span heuristic (duration_ms = len / samplingRate * 1000,
// smoothContours.R:99,127).  len < 1 prepares everything but the loess fit, which contour_fit_len() then
// does for the length of each use.
SGB_HD void contour_prepare(ContourTab *T, double *K, const double *an, int na, int len, double samplingRate,
                            bool has_lo, double lo, bool has_hi, double hi, bool pitch, int method) {
  T->status = SGB_OK; T->pitch = pitch ? 1 : 0; T->n = 0; T->kind = 0;
  T->has_lo = has_lo ? 1 : 0; T->has_hi = has_hi ? 1 : 0;
  T->v0 = T->v1 = 0.0; T->x0 = T->x1 = 0.0;
  T->L.status = 0; T->L.nv = 0;
  if (na < 1) { T->status = SGB_ERR_INVALID; return; }
  if (na > 10 && method == SGB_CONTOUR_LOESS) method = SGB_CONTOUR_SPLINE;          // :73-76
  double *x = K, *y = K + na;
  double tmin = an[0];
  for (int i = 1; i < na; i++) tmin = fmin(tmin, an[2 * i]);
  double tmax = an[0] - tmin;
  for (int i = 1; i < na; i++) tmax = fmax(tmax, an[2 * i] - tmin);
  for (int i = 0; i < na; i++) {
    double v = an[2 * i + 1];
    if (has_lo && v < lo) v = lo;                                                    // :78-83
    if (has_hi && v > hi) v = hi;
    if (pitch) v = hz_to_semitones(v);
    y[i] = v;
    x[i] = (an[2 * i] - tmin) / tmax;                                                // :96-98
  }
  if (pitch) { if (has_lo) lo = hz_to_semitones(lo); if (has_hi) hi = hz_to_semitones(hi); }
  T->lo = lo; T->hi = hi;
  if (na == 1) { T->kind = 0; T->v0 = y[0]; return; }
  if (na == 2) { T->kind = 1; T->v0 = y[0]; T->v1 = y[1]; return; }
  if (method == SGB_CONTOUR_SPLINE) {
    // spline() sorts its knots by x (insertion sort: O(n) on anchors that arrive in order)
    for (int i = 1; i < na; i++) {
      double xi = x[i], yi = y[i];
      int j = i - 1;
      while (j >= 0 && x[j] > xi) { x[j + 1] = x[j]; y[j + 1] = y[j]; j--; }
      x[j + 1] = xi; y[j + 1] = yi;
    }
    T->kind = 2; T->n = na;
    T->x0 = x[0]; T->x1 = x[na - 1];
    fmm_coef(na, x, y, K + 2 * na, K + 3 * na, K + 4 * na);
    return;
  }
  T->kind = 3; T->n = na;
  if (len >= 1) contour_fit_len(T, K, len, samplingRate);
}

// clamps and unit of a smoothed value v (kinds 2, 3)
SGB_HD double contour_finish(const ContourTab *T, double v) {
  if (T->has_lo && v < T->lo) v = T->lo;                                             // :155-156
  if (T->has_hi && v > T->hi) v = T->hi;
  if (v != v) v = 0.0;                                                               // NA -> 0 (:224)
  return T->pitch ? semitones_to_hz(v) : v;
}

// element k (0-based) of the contour of length len
SGB_HD double contour_eval(const ContourTab *T, const double *K, int len, int k) {
  double v;
  if (T->kind == 0) v = T->v0;
  else if (T->kind == 1) v = r_seq_at(T->v0, T->v1, len, k);
  else {
    const int n = T->n;
    if (T->kind == 2) v = r_spline_at(n, K, K + n, K + 2 * n, K + 3 * n, K + 4 * n, len, k);
    else v = loess_eval(&T->L, (double)(k + 1));
    return contour_finish(T, v);
  }
  return T->pitch ? semitones_to_hz(v) : v;
}

#if defined(__CUDACC__)
#include <cuda_pipeline.h>
// ---- per-sample evaluation in a CTA: contiguous windows of knots staged in shared memory ----
// The CTA evaluates the monotone run of grid points [k0, k1).  A window holds the knots [i0, i0 + CONTOUR_WIN)
// from the interval i0 of the first point not yet evaluated; it serves every point up to the first one at or past
// knot i0 + CONTOUR_WIN (found by bisection over the points: the grid is arithmetic, no memory is read).  Bisection
// inside the window finds the same interval as bisection over all knots (for sorted knots the largest i with
// x[i] <= u is unique), so the values are bit-identical to contour_eval().
#define CONTOUR_WIN 48          // knots per window: 5 x 48 doubles = 1.9 KB of shared memory

// copy a prepared header into shared memory, all threads of the CTA (the caller synchronises)
__device__ __forceinline__ void contour_tab_load(ContourTab *dst, const ContourTab *src) {
  static_assert(sizeof(ContourTab) % 8 == 0, "ContourTab is copied as doubles");
  const double *g = reinterpret_cast<const double *>(src);
  double *d = reinterpret_cast<double *>(dst);
  for (int i = threadIdx.x; i < (int)(sizeof(ContourTab) / 8); i += blockDim.x) d[i] = g[i];
}

// Called by every thread of the CTA with the same arguments; f(k, value) for each k in [k0, k1), each k once.
// sh: 5 * CONTOUR_WIN doubles and shi: 3 ints of shared memory.  T may live in shared memory; it is not written.
template <typename F>
__device__ void contour_eval_run(const ContourTab &T, const double *K, double *sh, int *shi, int len, int k0, int k1,
                                 F &&f) {
  if (T.kind != 2) {
    for (int k = k0 + (int)threadIdx.x; k < k1; k += blockDim.x) f(k, contour_eval(&T, K, len, k));
    return;
  }
  const int n = T.n;
  const double x0 = T.x0, x1 = T.x1;
  for (int k = k0; k < k1;) {
    __syncthreads();                    // the previous window has been read
    if (threadIdx.x == 0) {
      const int i0 = upper_interval(n, K, r_seq_at(x0, x1, len, k));
      int wn = n - i0, kend = k1;
      if (wn > CONTOUR_WIN) {
        wn = CONTOUR_WIN;
        const double xe = K[i0 + CONTOUR_WIN];
        int lo = k, hi = k1;            // u(lo) < xe; hi == k1 or u(hi) >= xe
        while (hi > lo + 1) {
          const int mid = (lo + hi) >> 1;
          if (r_seq_at(x0, x1, len, mid) >= xe) hi = mid; else lo = mid;
        }
        kend = hi;
      }
      shi[0] = i0; shi[1] = wn; shi[2] = kend;
    }
    __syncthreads();
    const int i0 = shi[0], wn = shi[1], kend = shi[2];
    for (int t = threadIdx.x; t < 5 * wn; t += blockDim.x) {
      const int a = t / wn, i = t - a * wn;
      __pipeline_memcpy_async(sh + a * CONTOUR_WIN + i, K + (int64_t)a * n + i0 + i, sizeof(double));
    }
    __pipeline_commit();
    __pipeline_wait_prior(0);
    __syncthreads();
    const double *x = sh, *y = sh + CONTOUR_WIN, *b = sh + 2 * CONTOUR_WIN, *c = sh + 3 * CONTOUR_WIN,
                 *d = sh + 4 * CONTOUR_WIN;
    for (int kk = k + (int)threadIdx.x; kk < kend; kk += blockDim.x) {
      const double u = r_seq_at(x0, x1, len, kk);
      const int i = upper_interval(wn, x, u);
      const double dx = u - x[i];
      f(kk, contour_finish(&T, y[i] + dx * (b[i] + dx * (c[i] + dx * d[i]))));
    }
    k = kend;
  }
}
#endif
