// K6: epoch joining and post-synthesis effects of generateHarmonics
// (R/source.R:386-467): crossFade at upward zero crossings
// (R/utilities_soundgen.R:255-375), amplitude envelope, signed-max normalisation,
// attack fade, drift amplitude.  One CTA per syllable, epochs in sequence.
//
// The zero-crossing searches decide the syllable's LENGTH, so a sign flip from FP32
// rounding would shift the whole waveform.  K1's float samples are therefore only
// trusted when |w| is well above their error bound; samples closer to zero are
// re-evaluated in FP64 with the reference's own formula (exact_epoch_sample).
#include "engine.cuh"
#include <cstring>
#include <cstdio>

// (512-thread CTAs are no faster.  They did expose, as rare irreproducible joins and hangs with several
// batches in flight, the write-after-read race that the barrier after the zc1 search now closes;
// tests/test_gpu_determinism.py keeps watching.)
#define COMPOSE_THREADS 256
#define ZC_REL_TOL 2e-4f

// Diagnostics of a non-terminating search: records land in mapped host memory, readable after a trap.
__device__ int *g_dbg = nullptr;
static int *h_dbg = nullptr;
int *compose_debug_buffer() {
  if (!h_dbg) {
    if (cudaHostAlloc((void **)&h_dbg, 4096 * sizeof(int), cudaHostAllocMapped) != cudaSuccess) return nullptr;
    memset(h_dbg, 0, 4096 * sizeof(int));
    int *d = nullptr;
    cudaHostGetDevicePointer((void **)&d, h_dbg, 0);
    cudaMemcpyToSymbol(g_dbg, &d, sizeof d);
  }
  return h_dbg;
}
__device__ __noinline__ void dbg_record(int loop, int s, int e, int a, int b, int c, int d2, int e2) {
  if (!g_dbg) return;
  int slot = atomicAdd(&g_dbg[0], 1);
  if (slot < 400) {
    int *r = g_dbg + 8 + slot * 10;
    r[0] = loop; r[1] = s; r[2] = e; r[3] = (int)threadIdx.x; r[4] = a; r[5] = b; r[6] = c; r[7] = d2; r[8] = e2; r[9] = 1;
  }
  __threadfence_system();
}

struct SylView {
  const int32_t *gcup;
  const double *kt, *py, *sb, *sc, *sd, *phi;
  const SylCtrl *C;
  const double *amp;     // syllable's amplitude block
  double sr;
  int G;
};

// waveform_epoch[k] (0-based k) exactly as R/source.R:403-409 computes it, in double.
// Cooperative: every thread of the CTA calls it with the same (e, k); the rows are split
// across the threads and the partial sums are combined in a fixed order.
__device__ double exact_epoch_sample(const SylView &V, int e, int k, double *red) {
  const SylCtrl &C = *V.C;
  const int g_first = C.ep_start[e] - 1, g_lastStart = C.ep_end[e] - 1;
  const int nsub = C.vf_active ? C.ep_nsub[e] : 0;
  const int J = C.ep_rows[e];
  const int x_first_i = V.gcup[g_first];
  const double x_first = (double)x_first_i, x_last = (double)V.gcup[g_lastStart];
  const int Ne = V.gcup[C.ep_end[e]] - x_first_i + 1;
  const double by = (x_last - x_first) / (double)(Ne - 1);
  const int nk = g_lastStart - g_first + 1;
  double v = (k >= Ne - 1) ? x_last : (x_first + (double)k * by);
  int lo = 0, hi = nk - 1;
  while (hi > lo + 1) {
    int mid = (lo + hi) >> 1;
    if (v < (double)V.gcup[g_first + mid]) hi = mid; else lo = mid;
  }
  double xg = (double)V.gcup[g_first + lo], xn = (double)V.gcup[g_first + lo + 1];
  double wfrac = (v - xg) / (xn - xg);
  double u = (double)(x_first_i + k);
  int a = 0, b = V.G;
  while (b > a + 1) {
    int mid = (a + b) >> 1;
    if (u < V.kt[mid]) b = mid; else a = mid;
  }
  double M = u - V.kt[a];
  double s1 = M * (M + 1.0) * 0.5, s2 = M * (M + 1.0) * (2.0 * M + 1.0) / 6.0, s3 = s1 * s1;
  double integr = (V.phi[a] + V.py[a] * (M + 1.0) + V.sb[a] * s1 + V.sc[a] * s2 + V.sd[a] * s3) / V.sr;
  const double *col = V.amp + C.ep_amp_off[e] + (int64_t)lo * J;
  double sum = 0.0;
  for (int j = 1 + threadIdx.x; j <= J; j += blockDim.x) {
    double y0 = col[j - 1], y1 = col[J + j - 1];
    if (y0 == 0.0 && y1 == 0.0) continue;
    double am = y0 + (y1 - y0) * wfrac;
    double x = integr * ((double)j / (double)(nsub + 1));
    x -= floor(x);
    sum += sinpi(2.0 * x) * am;
  }
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  double tot = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); i++) tot += red[i];
  __syncthreads();
  return tot;
}

// three-valued sign of a float sample: -1 / +1 when |v| >= tol, 0 = too close to call
__device__ __forceinline__ int sign3(float v, float tol) {
  return (fabsf(v) >= tol) ? (v > 0.0f ? 1 : -1) : 0;
}

// the loess fit of the amplitude envelope (3-10 anchors) for the composed length, kept out of line: one thread runs
// it, and inlined it would take registers from the cross-fade loops
__device__ __noinline__ void compose_ampl_fit(ContourTab *T, const double *K, int len, double samplingRate) {
  contour_fit_len(T, K, len, samplingRate);
}

#ifndef COMPOSE_MIN_CTAS
#define COMPOSE_MIN_CTAS 4     // one CTA per syllable, bound by memory latency: four resident CTAs (64 registers, some spills) beat two (cfg3: 2.9 -> 2.0 ms)
#endif
__global__ void __launch_bounds__(COMPOSE_THREADS, COMPOSE_MIN_CTAS)
k_compose(const sgb_syllable *__restrict__ syl, int S, SylCtrl *__restrict__ ctrl,
          const SylLayout *__restrict__ lay, Pools P, const double *__restrict__ amp,
          const float *__restrict__ wave, float *__restrict__ raw, const double *__restrict__ anchors,
          const double *__restrict__ pitch_pool, const int *__restrict__ epmax) {
  const int s = blockIdx.x;
  if (s >= S) return;
  SylCtrl &C = ctrl[s];
  const sgb_syllable sp = syl[s];
  float *comp = raw + lay[s].raw_off;
  __shared__ float red[32];
  __shared__ double redd[32];
  __shared__ int sh_found;
  __shared__ int red_i[32];

  if (sp.kind == 2) {   // raw samples supplied by the caller (sgb_filter)
    const double *src = pitch_pool + sp.pitch_off;
    for (int i = threadIdx.x; i < sp.pitch_len; i += blockDim.x) comp[i] = (float)src[i];
    return;
  }
  if (sp.kind != 1) return;
  if (C.status != SGB_OK) { if (threadIdx.x == 0) C.out_len = 0; return; }

  SylView V;
  const int64_t o = P.gc_off[s];
  V.gcup = P.gcup + o; V.kt = P.kt + o; V.py = P.ppg + o; V.sb = P.sb + o; V.sc = P.sc + o;
  V.sd = P.sd + o; V.phi = P.phi + o; V.C = &C; V.amp = amp + lay[s].amp_off;
  V.sr = sp.samplingRate; V.G = C.nGC;

  int Lc = 1;                 // `waveform = 0` (source.R:386)
  if (threadIdx.x == 0) comp[0] = 0.0f;
  int tail_e = -1, tail_start = 0, tail_koff = 0;   // comp[pos] == epoch_tail_e[pos - tail_koff] for pos >= tail_start
  float tail_tol = 0.0f;
  const int crossMax = (int)floor(15.0 * sp.samplingRate / 1000.0);
  __syncthreads();

  for (int e = 0; e < C.nEpochs; e++) {
    const float *w2 = wave + lay[s].wave_off + C.ep_wave_off[e];
    const int Ne = V.gcup[C.ep_end[e]] - V.gcup[C.ep_start[e] - 1] + 1;
    const float tol2 = ZC_REL_TOL * ordered_to_float(epmax[(int64_t)s * SGB_MAX_EPOCHS + e]);

    // ---- zc1: last upward zero crossing of the sound so far (findZeroCrossing(ampl1, len)) ----
    int Lc1;
    int zc1 = 0;
    if (Lc == 1) {
      zc1 = 1; Lc1 = 2;
      if (threadIdx.x == 0) comp[1] = 0.0f;
    } else {
      // largest p in [0, Lc-2] with comp[p] < 0 && comp[p+1] > 0.  Candidates are pairs that are,
      // or could be (a value within tol of zero), an upward crossing; each candidate is then
      // settled in FP64.  Only samples of the tail epoch (not yet cross-faded) are re-evaluated.
      int found = -1;
      int top = Lc - 2;
      int guard1 = 0;
      while (top >= 0 && found < 0) {
        if (++guard1 > (1 << 22)) { dbg_record(1, s, e, top, found, Lc, tail_start, sh_found); __trap(); }
        int p = top - (int)threadIdx.x;
        int hit = -1;
        if (p >= 0) {
          float t0 = (p >= tail_start) ? tail_tol : 0.0f, t1 = (p + 1 >= tail_start) ? tail_tol : 0.0f;
          float v0 = comp[p], v1 = comp[p + 1];
          bool neg0 = (t0 > 0.0f) ? (sign3(v0, t0) <= 0) : (v0 < 0.0f);
          bool pos1 = (t1 > 0.0f) ? (sign3(v1, t1) >= 0) : (v1 > 0.0f);
          if (neg0 && pos1) hit = p;
        }
        for (int of = 16; of > 0; of >>= 1) hit = max(hit, __shfl_xor_sync(0xffffffffu, hit, of));
        if ((threadIdx.x & 31) == 0) red_i[threadIdx.x >> 5] = hit;
        __syncthreads();
        if (threadIdx.x == 0) {
          int m = -1;
          for (int i = 0; i < (COMPOSE_THREADS >> 5); i++) m = max(m, red_i[i]);
          sh_found = m;
        }
        __syncthreads();
        int cand = sh_found;
        __syncthreads();
        if (cand < 0) { top -= COMPOSE_THREADS; continue; }
        float v0 = comp[cand], v1 = comp[cand + 1];
        bool ok0, ok1;
        if (cand >= tail_start && fabsf(v0) < tail_tol) ok0 = exact_epoch_sample(V, tail_e, cand - tail_koff, redd) < 0.0;
        else ok0 = v0 < 0.0f;
        if (cand + 1 >= tail_start && fabsf(v1) < tail_tol) ok1 = exact_epoch_sample(V, tail_e, cand + 1 - tail_koff, redd) > 0.0;
        else ok1 = v1 > 0.0f;
        if (ok0 && ok1) found = cand; else top = cand - 1;
      }
      // every thread has read comp[cand], comp[cand + 1] for its own copy of the decision: only now may
      // the sample after the crossing be overwritten (without this barrier a slow warp could read the
      // new zero, reject the crossing the others accepted, and search on alone, forever)
      __syncthreads();
      if (found >= 0) {
        zc1 = found + 1;
        Lc1 = found + 2;
        if (threadIdx.x == 0) comp[found + 1] = 0.0f;
      } else {
        Lc1 = Lc;
      }
    }

    // ---- zc2: first upward zero crossing of the new epoch (findZeroCrossing(ampl2, 1)) ----
    int zc2 = 0;
    {
      int found = -1;
      int base = 0;
      int guard2 = 0;
      while (base <= Ne - 3 && found < 0) {
        if (++guard2 > (1 << 22)) { dbg_record(2, s, e, base, found, Ne, Lc, sh_found); __trap(); }
        int p = base + (int)threadIdx.x;
        int hit = 0x7fffffff;
        if (p <= Ne - 3) {
          int s0 = sign3(w2[p], tol2), s1 = sign3(w2[p + 1], tol2);
          if (s0 <= 0 && s1 >= 0) hit = p;
        }
        for (int of = 16; of > 0; of >>= 1) hit = min(hit, __shfl_xor_sync(0xffffffffu, hit, of));
        if ((threadIdx.x & 31) == 0) red_i[threadIdx.x >> 5] = hit;
        __syncthreads();
        if (threadIdx.x == 0) {
          int m = 0x7fffffff;
          for (int i = 0; i < (COMPOSE_THREADS >> 5); i++) m = min(m, red_i[i]);
          sh_found = (m == 0x7fffffff) ? -1 : m;
        }
        __syncthreads();
        int cand = sh_found;
        __syncthreads();
        if (cand < 0) { base += COMPOSE_THREADS; continue; }
        float v0 = w2[cand], v1 = w2[cand + 1];
        bool ok0 = (fabsf(v0) < tol2) ? (exact_epoch_sample(V, e, cand, redd) < 0.0) : (v0 < 0.0f);
        bool ok1 = (fabsf(v1) < tol2) ? (exact_epoch_sample(V, e, cand + 1, redd) > 0.0) : (v1 > 0.0f);
        if (ok0 && ok1) found = cand; else base = cand + 1;
      }
      if (found >= 0) zc2 = found + 1;
    }
    const int L2 = Ne - zc2;                 // ampl2 = ampl2[(zc2 + 1):length(ampl2)]
    const float *a2 = w2 + zc2;
    int cl = min(crossMax, min(Lc1 - 1, L2 - 1));
    __syncthreads();
    int Lnew;
    if (cl < 2) {
#pragma unroll 8
      for (int i = threadIdx.x; i < L2; i += COMPOSE_THREADS) comp[Lc1 + i] = a2[i];
      Lnew = Lc1 + L2;
    } else {
      const int idx1 = Lc1 - cl;
      const double byc = 1.0 / (double)(cl - 1);     // multipl = seq(0, 1, length.out = cl)
      for (int i = threadIdx.x; i < cl; i += blockDim.x) {
        double mu = (i == cl - 1) ? 1.0 : (double)i * byc;
        int ir = cl - 1 - i;
        double mr = (ir == cl - 1) ? 1.0 : (double)ir * byc;   // rev(multipl)[i]
        comp[idx1 + i] = (float)(mr * (double)comp[idx1 + i] + mu * (double)a2[i]);
      }
#pragma unroll 8
      for (int i = cl + threadIdx.x; i < L2; i += COMPOSE_THREADS) comp[idx1 + i] = a2[i];
      Lnew = idx1 + L2;
    }
    if (threadIdx.x == 0) { C.ep_zc1[e] = zc1; C.ep_zc2[e] = zc2; }
    tail_e = e;
    tail_koff = Lnew - Ne;
    tail_start = Lnew - L2 + max(cl, 0);
    if (cl < 2) tail_start = Lnew - L2;
    tail_tol = tol2;
    Lc = Lnew;
    __syncthreads();
  }

  // ---- amplitude envelope (source.R:436-448) ----
  if (C.use_ampl) {
    // getSmoothContour(amplAnchors, len = length(waveform), valueFloor = 0, samplingRate): no ceiling
    // (prepared by k_syl_contours; a loess fit depends on the length and is done here)
    __shared__ ContourTab T;
    __shared__ double win[5 * CONTOUR_WIN];
    __shared__ int wi[3];
    const double *K = P.knots + P.koff[3 * s + 2];
    contour_tab_load(&T, P.ctab + 3 * s + 2);
    __syncthreads();
    if (threadIdx.x == 0) compose_ampl_fit(&T, K, Lc, sp.samplingRate);
    __syncthreads();
    if (T.status != SGB_OK) {
      if (threadIdx.x == 0) { C.status = T.status; C.out_len = 0; C.raw_max = 1.0; }
      return;
    }
    contour_eval_run(T, K, win, wi, Lc, 0, Lc,
                     [&](int k, double v) { comp[k] = (float)((double)comp[k] * exp2(v / 10.0)); });
    __syncthreads();
  }

  // ---- signed maximum (source.R:449: max(waveform), not max|.|) ----
  float m = -INFINITY;
#pragma unroll 8
  for (int i = threadIdx.x; i < Lc; i += COMPOSE_THREADS) m = fmaxf(m, comp[i]);
  for (int of = 16; of > 0; of >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, of));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    float v = red[0];
    for (int i = 1; i < (COMPOSE_THREADS >> 5); i++) v = fmaxf(v, red[i]);
    C.raw_max = (double)v;
    C.out_len = Lc;
  }
}

// Normalised, faded syllables placed into their bout's `sound` buffer
// (source.R:449-467 and the concatenation soundgen.R:632-640).  grid: (chunks, S).
__global__ void __launch_bounds__(256)
k_place_voiced(const sgb_syllable *__restrict__ syl, int S, const SylCtrl *__restrict__ ctrl,
               const SylLayout *__restrict__ lay, const SylPlace *__restrict__ place, Pools P,
               const float *__restrict__ raw, float *__restrict__ sound) {
  const int s = blockIdx.x;
  const SylCtrl &C = ctrl[s];
  const sgb_syllable &sp = syl[s];
  const int L = place[s].len;
  float *dst = sound + place[s].dst_off;
  const float *src = raw + lay[s].raw_off;
  if (sp.kind == 0 || C.status != SGB_OK) {
    for (int k = blockIdx.y * blockDim.x + threadIdx.x; k < L; k += gridDim.y * blockDim.x) dst[k] = 0.0f;
    return;
  }
  if (sp.kind == 2) {
    for (int k = blockIdx.y * blockDim.x + threadIdx.x; k < L; k += gridDim.y * blockDim.x) dst[k] = src[k];
    return;
  }
  const double inv_max = C.raw_max;
  const double rcp_max = 1.0 / inv_max;     // one division per syllable: x * (1 / max) is within an ulp of x / max in
                                            // double, far below the FP32 the sample is stored in
  int lf = 0;
  if (sp.attackLen > 0.0) {
    lf = (int)floor(sp.attackLen * sp.samplingRate / 1000.0);
    if (lf < 2) lf = 0;
    if (lf > L) lf = L;
  }
  const bool drift_on = sp.temperature > 0.0;
  const int64_t o = P.gc_off[s];
  const int32_t *gcup = P.gcup + o;
  const double *drift = P.drift + o;
  const int G = C.nGC;
#pragma unroll 4
  for (int k = blockIdx.y * blockDim.x + threadIdx.x; k < L; k += gridDim.y * blockDim.x) {
    double v = (double)src[k] * rcp_max;
    if (lf > 0) {
      if (k < lf) v = v * r_seq_at(0.0, 1.0, lf, k);                        // fade-in
      if (k >= L - lf) v = v * r_seq_at(0.0, 1.0, lf, (L - 1) - k);         // fade-out = rev(fadeIn)
    }
    if (drift_on) {
      // approx(drift, n = L, x = gc_upsampled[-length(gc_upsampled)]) (source.R:460-462)
      double xv = r_seq_at((double)gcup[0], (double)gcup[G - 1], L, k);
      int lo = 0, hi = G - 1;
      while (hi > lo + 1) { int mid = (lo + hi) >> 1; if (xv < (double)gcup[mid]) hi = mid; else lo = mid; }
      double xi = (double)gcup[lo], xj = (double)gcup[lo + 1];
      double d = drift[lo] + (drift[lo + 1] - drift[lo]) * ((xv - xi) / (xj - xi));
      v = v * d;
    }
    dst[k] = (float)v;
  }
}

void launch_compose(const sgb_syllable *syl, int S, SylCtrl *ctrl, const SylLayout *lay, const Pools &P,
                    const double *amp, const float *wave, float *raw, const double *anchors,
                    const double *pitch_pool, const int *epmax, cudaStream_t st) {
  if (S <= 0) return;
  k_compose<<<S, COMPOSE_THREADS, 0, st>>>(syl, S, ctrl, lay, P, amp, wave, raw, anchors, pitch_pool, epmax);
}

void launch_place_voiced(const sgb_syllable *syl, int S, const SylCtrl *ctrl, const SylLayout *lay,
                         const SylPlace *place, const Pools &P, const float *raw, float *sound,
                         int chunks, cudaStream_t st) {
  if (S <= 0) return;
  dim3 g(S, chunks);   // objects on x: more than 65535 syllables are routine in a preset sweep
  k_place_voiced<<<g, 256, 0, st>>>(syl, S, ctrl, lay, place, P, raw, sound);
}
