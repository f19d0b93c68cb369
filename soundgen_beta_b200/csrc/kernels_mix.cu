// Sample-rate glue of the bout orchestrator (R/soundgen.R:700-849): noise
// normalisation (source.R:125-131), mixing with addVectors (utilities_math.R:500-526),
// global amplitude envelope, normalisation after the filter, AM trill, silences.
#include "engine.cuh"
#include "contour.cuh"

// breathingStrength = getSmoothContour(len, noiseAnchors, floor -120, ceiling 40, samplingRate): the fit (FMM
// spline or loess: a millisecond of FP64 on one thread) once per noise, one thread each, instead of once per CTA of
// k_noise_final with 255 threads waiting.  The knots go to the noise's slice of the batch's knot pool.
__global__ void k_noise_tabs(const sgb_noise *__restrict__ noises, int n_noise, const double *__restrict__ anchors,
                             ContourTab *__restrict__ tabs, double *__restrict__ knots, const int64_t *__restrict__ koff) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_noise) return;
  const sgb_noise N = noises[n];
  if (N.strength_pre_off < 0)
    contour_prepare(&tabs[n], knots + koff[n], anchors + 2 * N.anchor_off, N.anchor_n, N.len, N.samplingRate, true,
                    -120.0, true, 40.0, false, N.anchor_method);
}

// [k0, k1): the contiguous share of chunk `part` of `parts` in L points
__device__ __forceinline__ void chunk_range(int L, int part, int parts, int *k0, int *k1) {
  const int per = (L + parts - 1) / parts;
  *k0 = min(L, part * per);
  *k1 = min(L, *k0 + per);
}

// generateNoise tail (R/source.R:70-81,125-131):
// breathing / max(breathing) * 2^(contour/10), then fadeInOut.  grid (noises, chunks): each CTA a contiguous run.
__global__ void __launch_bounds__(256)
k_noise_final(const sgb_noise *__restrict__ noises, const NoiseLayout *__restrict__ nl,
              const ContourTab *__restrict__ tabs, const double *__restrict__ knots, const int64_t *__restrict__ koff,
              const double *__restrict__ pre, const int *__restrict__ maxpool, int max_base,
              const float *__restrict__ raw, float *__restrict__ fin) {
  const int n = blockIdx.x;
  const sgb_noise N = noises[n];
  const int L = N.len;
  const float mx = ordered_to_float(maxpool[max_base + n]);
  const double rcp_mx = 1.0 / (double)mx;     // x * (1 / max): within an ulp of x / max in double, stored as FP32
  const float *src = raw + nl[n].raw_off;
  float *dst = fin + nl[n].raw_off;
  int lf = (int)floor(N.attackLen * N.samplingRate / 1000.0);
  if (lf < 2) lf = 0;
  if (lf > L) lf = L;
  auto emit = [&](int k, double c) {
    double v = (double)src[k] * rcp_mx * exp2(c / 10.0);
    if (lf > 0) {
      if (k < lf) v = v * r_seq_at(0.0, 1.0, lf, k);
      if (k >= L - lf) v = v * r_seq_at(0.0, 1.0, lf, (L - 1) - k);
    }
    dst[k] = (float)v;
  };
  int k0, k1;
  chunk_range(L, blockIdx.y, gridDim.y, &k0, &k1);
  if (N.strength_pre_off >= 0) {
    for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) emit(k, pre[N.strength_pre_off + k]);
    return;
  }
  __shared__ ContourTab T;
  __shared__ double win[5 * CONTOUR_WIN];
  __shared__ int wi[3];
  contour_tab_load(&T, &tabs[n]);
  __syncthreads();
  contour_eval_run(T, knots + koff[n], win, wi, L, k0, k1, emit);
}

// amplEnvelope = getSmoothContour(amplAnchorsGlobal, len = length(sound), 0, -throwaway, samplingRate), once per
// bout (one thread each) now that length(sound) is known
__global__ void k_aglobal_tabs(const sgb_bout *__restrict__ bouts, int n_bouts, const BoutLayout *__restrict__ bl,
                               const double *__restrict__ anchors, ContourTab *__restrict__ tabs,
                               double *__restrict__ knots, const int64_t *__restrict__ koff) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_bouts) return;
  const sgb_bout &B = bouts[b];
  if (B.aglobal_n > 0)
    contour_prepare(&tabs[b], knots + koff[b], anchors + 2 * B.aglobal_off, B.aglobal_n, bl[b].sound_len,
                    B.samplingRate, true, 0.0, true, -B.throwaway, false, B.aglobal_method);
}

// sound = voiced (+ breathing noise added BEFORE filtering, soundgen.R:708-714), then the
// global amplitude envelope (soundgen.R:721-733).  The voiced syllables are already in
// place; this pass adds the noises in call order and applies the envelope.
// grid (bouts, chunks): each CTA a contiguous run.
__global__ void __launch_bounds__(256)
k_sound_mix(const sgb_bout *__restrict__ bouts, const BoutLayout *__restrict__ bl,
            const sgb_noise *__restrict__ noises, const NoiseLayout *__restrict__ nl,
            const ContourTab *__restrict__ tabs, const double *__restrict__ knots, const int64_t *__restrict__ koff,
            const float *__restrict__ noise_fin, float *__restrict__ sound) {
  const int b = blockIdx.x;
  const sgb_bout B = bouts[b];
  const BoutLayout L = bl[b];
  float *snd = sound + L.sound_off;
  const bool has_env = (B.aglobal_n > 0);
  bool any_noise = false;
  for (int n = B.noise_begin; n < B.noise_end; n++) if (noises[n].mix == 0) any_noise = true;
  if (!any_noise && !has_env) return;
  auto mix = [&](int k) {
    float v = snd[k];
    for (int n = B.noise_begin; n < B.noise_end; n++) {
      if (noises[n].mix != 0) continue;
      int64_t rel = (L.sound_off + k) - nl[n].dst_off;
      if (rel >= 0 && rel < noises[n].len) v = v + noise_fin[nl[n].raw_off + rel];
    }
    return v;
  };
  int k0, k1;
  chunk_range(L.sound_len, blockIdx.y, gridDim.y, &k0, &k1);
  if (!has_env) {
    for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) snd[k] = mix(k);
    return;
  }
  __shared__ ContourTab T;
  __shared__ double win[5 * CONTOUR_WIN];
  __shared__ int wi[3];
  contour_tab_load(&T, &tabs[b]);
  __syncthreads();
  contour_eval_run(T, knots + koff[b], win, wi, L.sound_len, k0, k1,
                   [&](int k, double e) { snd[k] = (float)((double)mix(k) * e); });
}

// soundFiltered / max, + separately filtered noise (soundgen.R:807-818), AM trill
// (soundgen.R:821-833, getSigmoid utilities_math.R:639-653), written at the bout's place in
// the call's output (silences were zero-filled).  grid (chunks, bouts).
template <typename OutT>
__global__ void __launch_bounds__(256)
k_finalize(const sgb_bout *__restrict__ bouts, const BoutLayout *__restrict__ bl,
           const sgb_noise *__restrict__ noises, const NoiseLayout *__restrict__ nl,
           const float *__restrict__ sound, const float *__restrict__ filt,
           const float *__restrict__ noise_fin, const int *__restrict__ maxpool,
           OutT *__restrict__ out) {
  const int b = blockIdx.x;
  const sgb_bout B = bouts[b];
  const BoutLayout L = bl[b];
  const float *src = L.bypass ? (sound + L.sound_off) : (filt + L.filt_off);
  const double mx = L.bypass ? 1.0 : (double)ordered_to_float(maxpool[b]);
  const double rcp_mx = 1.0 / mx;
  OutT *dst = out + L.out_off;
  // AM pattern
  const bool am = B.amDep > 0.0;
  int nb = 1;
  double from = 0, to = 0, slope = 0, bmin = 0, bmax = 1;
  if (am) {
    from = -exp(-B.amShape * 1.0);
    to = exp(B.amShape * 1.0);
    slope = exp(fabs(B.amShape)) * 5.0;
    nb = (int)ceil(B.samplingRate / B.amFreq / 2.0);
    if (nb < 1) nb = 1;
    bmin = 1.0 / (1.0 + exp(-from * slope));
    bmax = 1.0 / (1.0 + exp(-to * slope));
  }
#pragma unroll 4
  for (int k = blockIdx.y * blockDim.x + threadIdx.x; k < L.final_len; k += gridDim.y * blockDim.x) {
    double v = 0.0;
    int rel = k - L.final_shift;
    if (rel >= 0 && rel < L.filt_len) v = (double)src[rel] * rcp_mx;
    for (int n = B.noise_begin; n < B.noise_end; n++) {
      if (noises[n].mix != 1) continue;
      int64_t r2 = (L.out_off + k) - nl[n].dst_off;
      if (r2 >= 0 && r2 < noises[n].len) v = v + (double)noise_fin[nl[n].raw_off + r2];
    }
    if (am) {
      int ph = k % (2 * nb);
      int i = (ph < nb) ? ph : (2 * nb - 1 - ph);
      double a = r_seq_at(from, to, nb, i);
      double bb = 1.0 / (1.0 + exp(-a * slope));
      double sig = (bb - bmin) / (bmax - bmin);
      v = v * (1.0 - sig * B.amDep / 100.0);
    }
    dst[k] = (OutT)v;
  }
}

void launch_noise_final(const sgb_noise *noises, int n_noise, const NoiseLayout *nl, const double *anchors,
                        const double *pre, const int *maxpool, int max_base, const float *raw, float *fin,
                        void *tabs, double *knots, const int64_t *koff, int chunks, cudaStream_t st) {
  if (n_noise <= 0) return;
  k_noise_tabs<<<(n_noise + 31) / 32, 32, 0, st>>>(noises, n_noise, anchors, (ContourTab *)tabs, knots, koff);
  dim3 g(n_noise, chunks);
  k_noise_final<<<g, 256, 0, st>>>(noises, nl, (const ContourTab *)tabs, knots, koff, pre, maxpool, max_base, raw, fin);
}
size_t contour_tab_bytes() { return sizeof(ContourTab); }

void launch_sound_mix(const sgb_bout *bouts, int n_bouts, const BoutLayout *bl, const sgb_noise *noises,
                      const NoiseLayout *nl, const double *anchors, const float *noise_fin, float *sound,
                      void *tabs, double *knots, const int64_t *koff, bool any_env, int chunks, cudaStream_t st) {
  if (n_bouts <= 0) return;
  if (any_env)
    k_aglobal_tabs<<<(n_bouts + 31) / 32, 32, 0, st>>>(bouts, n_bouts, bl, anchors, (ContourTab *)tabs, knots, koff);
  dim3 g(n_bouts, chunks);
  k_sound_mix<<<g, 256, 0, st>>>(bouts, bl, noises, nl, (const ContourTab *)tabs, knots, koff, noise_fin, sound);
}

void launch_finalize(int f64, const sgb_bout *bouts, int n_bouts, const BoutLayout *bl,
                     const sgb_noise *noises, const NoiseLayout *nl, const float *sound, const float *filt,
                     const float *noise_fin, const int *maxpool, void *out, int chunks, cudaStream_t st) {
  if (n_bouts <= 0) return;
  dim3 g(n_bouts, chunks);
  if (f64) k_finalize<double><<<g, 256, 0, st>>>(bouts, bl, noises, nl, sound, filt, noise_fin, maxpool, (double *)out);
  else k_finalize<float><<<g, 256, 0, st>>>(bouts, bl, noises, nl, sound, filt, noise_fin, maxpool, (float *)out);
}
