// K0 (control-rate prologue), size scan, K1 work list, K3 (amplitude matrices).
#include "engine.cuh"

// The syllables' contours, one thread each (index 3 s + role, see Pools): the sequential FMM solve (or the sort and
// loess fit) once per contour, ahead of K0.  The amplitude envelopes' lengths (glottal cycles, composed samples) are
// only known later: their loess fits (3-10 anchors) are done where they are used, for the length of the use.
__global__ void k_syl_contours(const sgb_syllable *__restrict__ syl, int S, const double *__restrict__ anchors, Pools P) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 3 * S) return;
  const int s = t / 3, role = t - 3 * s;
  const sgb_syllable &sp = syl[s];
  if (sp.kind != 1) return;
  double *K = P.knots + P.koff[t];
  if (role == 0) {
    if (sp.pitch_anchor_n > 0)
      contour_prepare(P.ctab + t, K, anchors + 2 * sp.pitch_anchor_off, sp.pitch_anchor_n, sp.pitch_len,
                      sp.pitchSamplingRate, true, sp.pitchFloor, true, sp.pitchCeiling, true, sp.pitch_method);
  } else if (sp.ampl_n > 0) {
    // getSmoothContour(amplAnchors, valueFloor = 0, samplingRate): K0 adds valueCeiling = -throwaway (source.R:221-235),
    // K6 passes no ceiling (source.R:436-448)
    contour_prepare(P.ctab + t, K, anchors + 2 * sp.ampl_off, sp.ampl_n, 0, sp.samplingRate, true, 0.0, role == 1,
                    -sp.throwaway, false, sp.ampl_method);
  }
}

// One CTA per syllable.  Parallel: vibrato, column maxima, row pruning.
// Sequential (thread 0): glottal cycles, random walks, jitter, drift, epochs,
// upsampling knots -- R/source.R:206-385.
#define CTRL_THREADS 32   // one warp per syllable: the stage is bound by the latency of its sequential
                          // part, so what matters is how many syllables are resident per SM
// MINB: resident syllables per SM.  16 (128 registers) when the batch has long outliers -- the kernel then ends with its
// longest lane-0 chain, which spills would stretch; 32 (64 registers, some spills) when the syllables are alike and
// the stage is a matter of how many of them are in flight (cfg3: 4.4 -> 3.7 ms).  launch_control() picks.
template <int MINB>
__global__ void __launch_bounds__(CTRL_THREADS, MINB)
k_control(const sgb_syllable *syl, int S, const int32_t *__restrict__ order, const double *pitch, const double *anchors,
          const double *z, Pools P, SylCtrl *ctrl, int tc_min_rows) {
  if ((int)blockIdx.x >= S) return;
  const int s = order[blockIdx.x];        // longest pitch contours first
  const sgb_syllable sp = syl[s];
  SylCtrl &C = ctrl[s];
  __shared__ int sh_status;
  if (sp.kind != 1) {
    if (threadIdx.x == 0) {
      C.status = SGB_OK; C.nGC = 0; C.nEpochs = 0; C.tiles = 0; C.amp_elems = 0; C.wave_elems = 0;
      C.n_up = 0; C.rows_kept = 0; C.nHarmonics = 0; C.n_jidx = 0; C.z_used = 0; C.use_ampl = 0;
      C.out_len = (sp.kind == 0) ? sp.silent_len : sp.pitch_len;
      C.raw_max = 1.0;
    }
    return;
  }
  SylArrays A = make_arrays(P, sp, s);
  if (sp.pitch_anchor_n > 0) {
    // pitchContour_syl = getSmoothContour(pitchAnchors, len, samplingRate = pitchSamplingRate, pitchFloor,
    //                                     pitchCeiling, thisIsPitch = TRUE) * pitchDeltas[s]  (soundgen.R:596-603),
    // prepared by k_syl_contours
    __shared__ ContourTab T;
    __shared__ double win[5 * CONTOUR_WIN];
    __shared__ int wi[3];
    contour_tab_load(&T, P.ctab + 3 * s);
    __syncthreads();
    if (T.status != SGB_OK) {
      if (threadIdx.x == 0) {
        C.status = T.status; C.nGC = 0; C.nEpochs = 0; C.tiles = 0; C.amp_elems = 0; C.wave_elems = 0; C.n_up = 0;
        C.rows_kept = 0; C.nHarmonics = 0; C.n_jidx = 0; C.z_used = 0; C.use_ampl = 0; C.out_len = 0; C.raw_max = 1.0;
      }
      return;
    }
    contour_eval_run(T, P.knots + P.koff[3 * s], win, wi, sp.pitch_len, 0, sp.pitch_len,
                     [&](int i, double v) { A.pitch[i] = ctrl_vibrato(sp, i + 1, v * sp.pitch_scale); });
  } else {
    const double *pin = pitch + sp.pitch_off;
    for (int i = threadIdx.x; i < sp.pitch_len; i += blockDim.x) A.pitch[i] = ctrl_vibrato(sp, i + 1, pin[i]);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    ctrl_sequential(sp, anchors, P.ctab + 3 * s + 1, P.knots + P.koff[3 * s + 1], z, A, C);
    sh_status = C.status;
  }
  __syncthreads();
  if (sh_status != SGB_OK) return;
  const int G = C.nGC, nH = C.nHarmonics;
  // K1's view of pitch_upsampled: per spline piece the knot and the quartic in M = u - kt of
  //   sum_{v <= u} pitch_upsampled[v] = phi + y (M+1) + b S1(M) + c S2(M) + d S3(M)   (Faulhaber sums)
  {
    double *pc = P.pc + SYNTH_PC * P.gc_off[s];
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
      const double y = A.ppg[g], b = A.sb[g], c = A.sc[g], d = A.sd[g];
      pc[SYNTH_PC * g + 0] = A.kt[g];
      pc[SYNTH_PC * g + 1] = A.phi[g] + y;
      pc[SYNTH_PC * g + 2] = y + b / 2.0 + c / 6.0;
      pc[SYNTH_PC * g + 3] = b / 2.0 + c / 2.0 + d / 4.0;
      pc[SYNTH_PC * g + 4] = c / 3.0 + d / 2.0;
      pc[SYNTH_PC * g + 5] = d / 4.0;
    }
  }
  const bool use_tab = nH <= 1024;       // (the name is historical: log2(h) used to sit in a shared table, whose 8 KB
                                         // would cap the resident CTAs per SM; it is recomputed where needed)
  __syncthreads();
  const bool ao = C.any_oct != 0;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    if (!use_tab) { A.colmax[g] = ctrl_colmax(sp, A, C, g); continue; }
    // max over h of r(h, g) (sourceSpectrum.R:146).  Past the parabola r is slope*log2(h) + oct*h + const:
    // monotone or with a single stationary point, so the maximum sits at the first harmonics, at the
    // last harmonic below Nyquist or next to the stationary point; those candidates are evaluated
    // with the exact expression (dead entries are -Inf and never win).
    double m = -INFINITY;
    const double pg = A.ppg[g], rog = A.ro[g], roctg = A.roct[g], rkg = A.rk[g];
    auto probe = [&](int h) {
      if (h < 1 || h > nH) return;
      double r = rolloff_db_l(h, log2((double)h), pg, rog, roctg, rkg, ao, sp.rolloffParab, C.parab_harm, C.parab_a,
                              C.parab_b, C.parab_c, 200.0, sp.throwaway, sp.samplingRate);
      if (r > m) m = r;
    };
    const int hhead = min(nH, max(C.parab_harm, 2) + 1);
    for (int h = 1; h <= hhead; h++) probe(h);
    int hl = (int)fmin((double)nH, floor(sp.samplingRate / 2.0 / pg)) + 1;      // last harmonic below Nyquist
    while (hl > 1 && (double)hl * pg >= sp.samplingRate / 2.0) hl--;
    probe(hl); probe(hl - 1);
    if (ao && roctg != 0.0) {
      const double slope = rog + rkg * (pg - 200.0) / 1000.0;
      const double hs = -slope * 1000.0 / (roctg * pg * 0.6931471805599453);    // d/dh = 0
      if (hs > 1.0 && hs < (double)nH + 1.0) {
        const int h0 = (int)floor(hs);
        for (int h = h0 - 1; h <= h0 + 2; h++) probe(h);
      }
    }
    A.colmax[g] = m;
  }
  for (int h = 1 + threadIdx.x; h <= nH; h += blockDim.x) {
    if (!use_tab) { A.rowmap[h - 1] = ctrl_rowkept(sp, A, C, h) ? 1 : 0; continue; }
    int kept = 0;
    const double lh = log2((double)h);
    for (int g = 0; g < G && !kept; g++) {
      double r = rolloff_db_l(h, lh, A.ppg[g], A.ro[g], A.roct[g], A.rk[g], ao, sp.rolloffParab, C.parab_harm,
                              C.parab_a, C.parab_b, C.parab_c, 200.0, sp.throwaway, sp.samplingRate);
      if (r > -INFINITY) kept = 1;
    }
    A.rowmap[h - 1] = kept;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int kept = 0;
    for (int h = 1; h <= nH; h++) if (A.rowmap[h - 1]) A.rowmap[kept++] = h;
    C.rows_kept = kept;
    if (kept < 1) C.status = SGB_ERR_SYNTH;
    ctrl_sizes(A, C, SYNTH_TILE, tc_min_rows);
    if (C.status != SGB_OK) { C.tiles = 0; C.tiles_tc = 0; C.amp_elems = 0; C.wave_elems = 0; }
  }
}

// Exclusive prefix sums of the per-syllable scratch sizes (single CTA).
// totals: [0] amp doubles, [1] wave floats, [2] tiles, [3] raw floats, [4] synth partials,
//         [5] synth samples (4,5 filled by k_build_tiles), [6] failed syllables
__device__ inline int64_t raw_cap(const SylCtrl &C) {
  return (((int64_t)(C.nGC > 0 ? C.n_up + 2 : C.out_len)) + 3) & ~(int64_t)3;
}
__global__ void __launch_bounds__(1024)
k_scan_sizes(const SylCtrl *ctrl, int S, SylLayout *lay, int64_t *totals) {
  __shared__ int64_t part[6][1024];
  const int t = threadIdx.x, nt = blockDim.x;
  const int per = (S + nt - 1) / nt;
  const int lo = min(S, t * per), hi = min(S, lo + per);
  int64_t a = 0, w = 0, tl = 0, r = 0, failed = 0, tc = 0;
  for (int s = lo; s < hi; s++) {
    const SylCtrl &C = ctrl[s];
    bool ok = (C.status == SGB_OK);
    if (!ok) failed++;
    a += ok ? C.amp_elems : 0; w += ok ? C.wave_elems : 0; tl += ok ? C.tiles : 0; tc += ok ? C.tiles_tc : 0;
    r += raw_cap(C);
  }
  part[5][t] = tc;
  part[0][t] = a; part[1][t] = w; part[2][t] = tl; part[3][t] = r; part[4][t] = failed;
  __syncthreads();
  if (t < 6) {   // serial scan of <= 1024 partials per quantity: negligible
    int64_t run = 0;
    for (int i = 0; i < nt; i++) { int64_t v = part[t][i]; part[t][i] = run; run += v; }
    totals[t == 4 ? 6 : (t == 5 ? 7 : t)] = run;
  }
  __syncthreads();
  a = part[0][t]; w = part[1][t]; tl = part[2][t]; r = part[3][t]; tc = part[5][t];
  for (int s = lo; s < hi; s++) {
    const SylCtrl &C = ctrl[s];
    bool ok = (C.status == SGB_OK);
    lay[s].amp_off = a; lay[s].wave_off = w; lay[s].tile_off = (int32_t)tl; lay[s].raw_off = r;
    lay[s].pad = (int32_t)tc;
    a += ok ? C.amp_elems : 0; w += ok ? C.wave_elems : 0; tl += ok ? C.tiles : 0; tc += ok ? C.tiles_tc : 0;
    r += raw_cap(C);
  }
}

// K1 work list: one thread per syllable writes its (epoch, k0) tiles; also accumulates the
// algorithmic work counters (rows x samples) used for the K1 roofline.
__global__ void k_build_tiles(const SylCtrl *ctrl, int S, const SylLayout *lay, const Pools P,
                              SynthTile *tiles, int64_t *totals, int tc_min_rows) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const SylCtrl &C = ctrl[s];
  if (C.status != SGB_OK || C.nGC == 0) return;
  const int32_t *gcup = P.gcup + P.gc_off[s];
  const double *kt = P.kt + P.gc_off[s];
  const int G = C.nGC;
  int t = lay[s].tile_off;
  int64_t partials = 0, samples = 0;
  int a = 0;                                    // spline piece: largest a with kt[a] <= u (monotone over the syllable)
  for (int e = 0; e < C.nEpochs; e++) {
    const int g_first = C.ep_start[e] - 1, g_last = C.ep_end[e] - 1;
    const int x_first_i = gcup[g_first];
    const double x_first = (double)x_first_i, x_last = (double)gcup[g_last];
    const int Ne = gcup[C.ep_end[e]] - x_first_i + 1;
    const double by = (x_last - x_first) / (double)(Ne - 1);
    const int nknots = g_last - g_first + 1;
    int lo = 0;                                 // amplitude interval of approx(): largest lo <= nknots-2 with knot <= v
    for (int k0 = 0; k0 < Ne && C.ep_rows[e] < tc_min_rows; k0 += SYNTH_TILE) {     // the other epochs: k_synth_tc
      const double v = (k0 >= Ne - 1) ? x_last : (x_first + (double)k0 * by);
      while (lo < nknots - 2 && v >= (double)gcup[g_first + lo + 1]) lo++;
      const double u = (double)(x_first_i + k0);
      while (a < G - 1 && u >= kt[a + 1]) a++;
      SynthTile T; T.syl = s; T.epoch = e; T.k0 = k0; T.gi_lo = lo; T.a_lo = a; T.pad[0] = T.pad[1] = T.pad[2] = 0;
      tiles[t++] = T;
    }
    // epochs overlap by one cycle (the next one starts at this one's last cycle): rewind the piece index
    while (a > 0 && (double)gcup[g_last] < kt[a]) a--;
    partials += (int64_t)Ne * C.ep_rows[e];
    samples += Ne;
  }
  atomicAdd((unsigned long long *)&totals[4], (unsigned long long)partials);
  atomicAdd((unsigned long long *)&totals[5], (unsigned long long)samples);
}

// K3: dense per-epoch amplitude matrices A[e][g][j] (column per glottal cycle, rows =
// multiples of f0/(nSubharm+1)), exact doubles: getRolloff + shimmer + getVocalFry
// (R/sourceSpectrum.R:71-186, R/source.R:348-375, R/subharmonics.R:25-163).
// grid (S, chunks of glottal cycles).  Per epoch the CTA tabulates what the reference's
// quirk makes column-independent -- the f-harmonic amplitudes of the epoch's FIRST cycle
// (subharmonics.R:76-77) -- and the per-(s, cycle) sideband multipliers, so that an f row
// costs one exp2 and a g row two FMAs.
#define AMP_MAXH 1024
#define AMP_MAXS 16
#define AMP_CG 32
#ifndef AMP_MIN_CTAS
#define AMP_MIN_CTAS 4      // resident CTAs per SM (64 registers): measured 2 / 3 / 4 / 5 / 6 -> cfg3 6.0 / 5.8 / 5.9 / 6.7 / 7.0 ms, preset sweep 17.7 / 15.3 / 14.3 / 14.7 / 16.9 ms
#endif
#define AMP_RPT 4
#define AMP_VF 1024      // f-harmonics per column the dense variant keeps in shared memory
#define AMP_DR 10        // rows per thread of the dense variant (rows <= 2560)
__global__ void __launch_bounds__(256, AMP_MIN_CTAS)
k_amp(const sgb_syllable *syl, int S, const SylCtrl *ctrl, const SylLayout *lay, Pools P, double *amp,
      float4 *amp32, int tc_min_rows) {
  int s = blockIdx.x;
  if (s >= S) return;
  const SylCtrl &C = ctrl[s];
  if (C.status != SGB_OK || C.nGC == 0) return;
  const sgb_syllable sp = syl[s];
  SylArrays A = make_arrays(P, sp, s);
  double *out = amp + lay[s].amp_off;
  float4 *out32 = amp32 + lay[s].amp_off;
  __shared__ double A0[AMP_MAXH + 2];
  __shared__ double ML[AMP_MAXS * (AMP_CG + 1)], MU[AMP_MAXS * (AMP_CG + 1)];
  __shared__ double VF[2][AMP_VF + 2];
  const int G = C.nGC, Hk = C.rows_kept;
  const double thr01 = exp2(sp.throwaway / 10.0);
  for (int c0 = blockIdx.y * AMP_CG; c0 < G; c0 += gridDim.y * AMP_CG) {
    const int c1 = min(G, c0 + AMP_CG);
    for (int e = 0; e < C.nEpochs; e++) {
      const int ga = max(c0, C.ep_start[e] - 1), gb = min(c1, C.ep_end[e]);   // [ga, gb) 0-based
      if (ga >= gb) continue;
      const int gx = min(gb + 1, C.ep_end[e]);     // one extra column for the differences
      const int n = C.vf_active ? C.ep_nsub[e] : 0;
      const int rows = C.ep_rows[e];
      const int g0 = C.ep_start[e] - 1;
      double *oe = out + C.ep_amp_off[e];
      float4 *oe32 = out32 + C.ep_amp_off[e];
      // the tensor-core kernel reads {Y, dY} pairs (8 B per element, packed at the start of the epoch's region); the
      // FP32-pipe kernel wants {Y, Y, dY, dY} (one broadcast LDS.128 feeds both packed lanes)
      const bool tc_ep = rows >= tc_min_rows;
      const bool tabled = (n == 0) || (Hk <= AMP_MAXH && n <= AMP_MAXS);
      __syncthreads();
      if (tabled && n > 0) {
        for (int k = threadIdx.x; k <= Hk + 1; k += blockDim.x) {   // A0[k], k = 0..Hk+1 (ends are 0)
          double v = 0.0;
          if (k >= 1 && k <= Hk) {
            int h = A.rowmap[k - 1];
            double r = rolloff_db(h, A.ppg[g0], A.ro[g0], A.roct[g0], A.rk[g0], C.any_oct != 0, sp.rolloffParab,
                                  C.parab_harm, C.parab_a, C.parab_b, C.parab_c, 200.0, sp.throwaway, sp.samplingRate);
            v = exp2((r - A.colmax[g0]) / 10.0) * A.shimmer[g0];
          }
          A0[k] = v;
        }
        const int ncol = gx - ga;
        for (int idx = threadIdx.x; idx < n * ncol; idx += blockDim.x) {
          int si = idx / ncol, gi = idx - si * ncol;
          int g = ga + gi, sidx = si + 1;
          double sw = A.subdep[g];
          double dl = A.ppg[g] * (double)sidx / (double)(n + 1);
          double du = A.ppg[g] * (double)(n + 1 - sidx) / (double)(n + 1);
          double ml = 0.0, mu = 0.0;
          if (sw != 0.0) { ml = exp(-0.5 * (dl / sw) * (dl / sw)); mu = exp(-0.5 * (du / sw) * (du / sw)); }
          ML[si * (AMP_CG + 1) + gi] = ml; MU[si * (AMP_CG + 1) + gi] = mu;
        }
      }
      __syncthreads();
      if (tabled && n > 0 && rows >= 512 && Hk <= AMP_VF && rows <= 256 * AMP_DR) {
        // Dense variant (epochs with sub-harmonics).  Only every (n+1)-th row is an f-harmonic (rolloff + exp2, the
        // expensive rows); evaluated row by row they would keep 1/(n+1) of a warp's lanes busy.  So per
        // column the f-harmonics are first computed densely over the threads into shared memory
        // (double-buffered: one barrier per column), then every thread writes the rows it owns.
        double prev[AMP_DR], lgk[AMP_VF / 256];
        int hk[AMP_VF / 256];
#pragma unroll
        for (int i = 0; i < AMP_VF / 256; i++) {
          const int k = (int)threadIdx.x + 1 + 256 * i;
          hk[i] = 1; lgk[i] = 0.0;
          if (k <= Hk) { hk[i] = A.rowmap[k - 1]; lgk[i] = log2((double)hk[i]); }
        }
#pragma unroll
        for (int i = 0; i < AMP_DR; i++) prev[i] = 0.0;
        for (int g = ga; g < gx; g++) {
          const int gi = g - ga;
          const double pg = A.ppg[g], roctg = A.roct[g], cmg = A.colmax[g], shg = A.shimmer[g];
          const double slope = A.ro[g] + A.rk[g] * (pg - 200.0) / 1000.0;   // column term of rolloff_db_l
          double *vf = VF[gi & 1];
#pragma unroll
          for (int i = 0; i < AMP_VF / 256; i++) {
            const int k = (int)threadIdx.x + 1 + 256 * i;
            if (k > Hk) continue;
            double r = rolloff_db_s(hk[i], lgk[i], pg, slope, roctg, C.any_oct != 0, sp.rolloffParab, C.parab_harm,
                                    C.parab_a, C.parab_b, C.parab_c, 200.0, sp.throwaway, sp.samplingRate);
            vf[k] = exp2((r - cmg) / 10.0) * shg;
          }
          __syncthreads();
          double *oc = oe + (int64_t)(g - g0) * rows;
          float4 *oc32 = oe32 + (int64_t)(g - 1 - g0) * rows;
#pragma unroll
          for (int i = 0; i < AMP_DR; i++) {
            const int j = i * 256 + (int)threadIdx.x + 1;
            if (j > rows) continue;
            double v;
            if (n == 0) {
              v = vf[j];
            } else {
              const int k = j / (n + 1), si = j - k * (n + 1);
              if (si == 0) v = vf[k];
              else v = A0[k] * ML[(si - 1) * (AMP_CG + 1) + gi] + A0[k + 1] * MU[(si - 1) * (AMP_CG + 1) + gi];
              if (v < thr01) v = 0.0;
            }
            if (g < gb) oc[j - 1] = v;
            if (g > ga) {   // {Y, Y, dY, dY}: one 16-byte load gives K1 both packed FFMA2 operands
              const float y = (float)prev[i], dy = (float)(v - prev[i]);
              if (tc_ep) reinterpret_cast<float2 *>(oe32)[(int64_t)(g - 1 - g0) * rows + (j - 1)] = make_float2(y, dy);
              else oc32[j - 1] = make_float4(y, y, dy, dy);
            }
            prev[i] = v;
          }
        }
        continue;
      }
      // General variant: each thread owns rows j = rb + tid + i*256 and walks the columns, so that the
      // FP32 {Y_g, Y_{g+1} - Y_g} table K1 consumes falls out of the same pass
      for (int rb = 0; rb < rows; rb += 256 * AMP_RPT) {
        double prev[AMP_RPT], lg[AMP_RPT];
        int rk_[AMP_RPT], rs_[AMP_RPT], rh_[AMP_RPT];     // per owned row: f index k, sub index s, harmonic h
#pragma unroll
        for (int i = 0; i < AMP_RPT; i++) {
          const int j = rb + i * 256 + (int)threadIdx.x + 1;
          rk_[i] = 0; rs_[i] = 0; rh_[i] = 1; lg[i] = 0.0; prev[i] = 0.0;
          if (j <= rows) {
            rk_[i] = (n == 0) ? j : j / (n + 1);
            rs_[i] = (n == 0) ? 0 : j % (n + 1);
            if (rs_[i] == 0) { rh_[i] = A.rowmap[rk_[i] - 1]; lg[i] = log2((double)rh_[i]); }
          }
        }
        for (int g = ga; g < gx; g++) {
          const int gi = g - ga;
          const double pg = A.ppg[g], roctg = A.roct[g], cmg = A.colmax[g], shg = A.shimmer[g];
          const double slope = A.ro[g] + A.rk[g] * (pg - 200.0) / 1000.0;   // column term of rolloff_db_l
          double *oc = oe + (int64_t)(g - g0) * rows;
          float4 *oc32 = oe32 + (int64_t)(g - 1 - g0) * rows;
#pragma unroll
          for (int i = 0; i < AMP_RPT; i++) {
            const int j = rb + i * 256 + (int)threadIdx.x + 1;
            if (j > rows) continue;
            double v;
            if (!tabled) {
              v = ampl_exact(sp, A, C, e, j, g);
            } else {
              if (rs_[i] == 0) {
                double r = rolloff_db_s(rh_[i], lg[i], pg, slope, roctg, C.any_oct != 0, sp.rolloffParab,
                                        C.parab_harm, C.parab_a, C.parab_b, C.parab_c, 200.0, sp.throwaway,
                                        sp.samplingRate);
                v = exp2((r - cmg) / 10.0) * shg;
              } else {
                v = A0[rk_[i]] * ML[(rs_[i] - 1) * (AMP_CG + 1) + gi] + A0[rk_[i] + 1] * MU[(rs_[i] - 1) * (AMP_CG + 1) + gi];
              }
              if (n > 0 && v < thr01) v = 0.0;
            }
            if (g < gb) oc[j - 1] = v;
            if (g > ga) {   // {Y, Y, dY, dY}: one 16-byte load gives K1 both packed FFMA2 operands
              const float y = (float)prev[i], dy = (float)(v - prev[i]);
              if (tc_ep) reinterpret_cast<float2 *>(oe32)[(int64_t)(g - 1 - g0) * rows + (j - 1)] = make_float2(y, dy);
              else oc32[j - 1] = make_float4(y, y, dy, dy);
            }
            prev[i] = v;
          }
        }
      }
    }
  }
}

// getRolloff as a stand-alone call (R/sourceSpectrum.R:71-186).  Single CTA; out is
// nHarmonics x nGC column-major with the kept rows compacted to the top; scratch:
// colmax[nGC] doubles, kept[nHarmonics] ints.
__global__ void __launch_bounds__(256)
k_rolloff_api(const double *p, int G, int nH, const double *ro, int n_ro, const double *roct, int n_roct,
              const double *rk, int n_rk, double rolloffParab, double rolloffParabHarm, double parabCeiling,
              double baseline, double throwaway, double sr, double *out, int *out_rows, double *colmax,
              int *kept) {
  __shared__ int any_oct;
  if (threadIdx.x == 0) any_oct = 0;
  __syncthreads();
  for (int g = threadIdx.x; g < G; g += blockDim.x) if (roct[n_roct == 1 ? 0 : g] != 0.0) any_oct = 1;
  __syncthreads();
  const bool ao = any_oct != 0;
  auto rdb = [&](int h, int g) -> double {
    double ph = (parabCeiling >= 0.0) ? rint(parabCeiling / p[g]) : rint(rolloffParabHarm);
    if (ph == 2.0) ph = 3.0;
    int phi = (int)fmin(ph, (double)nH);
    double a = -4.0 * rolloffParab / ((ph - 1.0) * (ph - 1.0));
    double b = -a * (1.0 + ph), c = a * ph;
    return rolloff_db(h, p[g], ro[n_ro == 1 ? 0 : g], roct[n_roct == 1 ? 0 : g], rk[n_rk == 1 ? 0 : g], ao,
                      rolloffParab, phi, a, b, c, baseline, throwaway, sr);
  };
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    double m = -INFINITY;
    for (int h = 1; h <= nH; h++) m = fmax(m, rdb(h, g));
    colmax[g] = m;
  }
  for (int h = 1 + threadIdx.x; h <= nH; h += blockDim.x) {
    int k = 0;
    for (int g = 0; g < G && !k; g++) if (rdb(h, g) > -INFINITY) k = 1;
    kept[h - 1] = k;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int n = 0;
    for (int h = 1; h <= nH; h++) if (kept[h - 1]) kept[n++] = h;
    *out_rows = n;
    for (int i = n; i < nH; i++) kept[i] = 0;
  }
  __syncthreads();
  const int n = *out_rows;
  for (int idx = threadIdx.x; idx < nH * G; idx += blockDim.x) {
    int g = idx / nH, k = idx - g * nH;
    out[idx] = (k < n) ? exp2((rdb(kept[k], g) - colmax[g]) / 10.0) : 0.0;
  }
}

// ---- host launchers (kernels stay private to this translation unit) ----
static int g_tc_min_rows = 1 << 30;      // K1 dispatch (engine.cu): epochs with >= this many rows go to k_synth_tc
void synth_min_rows_set(int v) { g_tc_min_rows = v; }
int synth_min_rows() { return g_tc_min_rows; }
void launch_control(const sgb_syllable *syl, int S, bool dense, const int32_t *order, const double *pitch, const double *anchors, const double *z,
                    const Pools &P, SylCtrl *ctrl, SylLayout *lay, int64_t *totals, cudaStream_t st) {
  k_syl_contours<<<(3 * S + 127) / 128, 128, 0, st>>>(syl, S, anchors, P);
  if (dense) k_control<32><<<S, CTRL_THREADS, 0, st>>>(syl, S, order, pitch, anchors, z, P, ctrl, g_tc_min_rows);
  else k_control<16><<<S, CTRL_THREADS, 0, st>>>(syl, S, order, pitch, anchors, z, P, ctrl, g_tc_min_rows);
  k_scan_sizes<<<1, 1024, 0, st>>>(ctrl, S, lay, totals);
}
void launch_tiles_amp(const sgb_syllable *syl, int S, const SylCtrl *ctrl, const SylLayout *lay, const Pools &P,
                      SynthTile *tiles, int64_t *totals, double *amp, float4 *amp32, cudaStream_t st) {
  k_build_tiles<<<(S + 127) / 128, 128, 0, st>>>(ctrl, S, lay, P, tiles, totals, g_tc_min_rows);
  dim3 g(S, S >= 2048 ? 1 : (S >= 256 ? 4 : 16));
  k_amp<<<g, 256, 0, st>>>(syl, S, ctrl, lay, P, amp, amp32, g_tc_min_rows);
}
void launch_rolloff_api(const double *p, int G, int nH, const double *ro, int n_ro, const double *roct, int n_roct,
                        const double *rk, int n_rk, double rolloffParab, double rolloffParabHarm,
                        double parabCeiling, double baseline, double throwaway, double sr, double *out,
                        int *out_rows, double *colmax, int *kept) {
  k_rolloff_api<<<1, 256>>>(p, G, nH, ro, n_ro, roct, n_roct, rk, n_rk, rolloffParab, rolloffParabHarm, parabCeiling,
                            baseline, throwaway, sr, out, out_rows, colmax, kept);
}
