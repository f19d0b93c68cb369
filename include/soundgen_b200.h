/*
 * soundgen_b200.h -- C ABI of libsoundgen_b200.so
 *
 * B200 (sm_100a) implementation of soundgen's per-frame source-filter synthesis
 * path.  The reference (nemochina2008/soundgen_beta) is pure R and has no FFI for
 * this path, so each entry point below replaces an R function (file:line under
 * the reference tree) and is what the package's `.Call` shim binds
 * (r/src/rshim.c, see INTEGRATION.md).
 *
 * Conventions
 *   - plain C, POD structs, pointers + sizes; no C++ / torch types.
 *   - all host buffers are caller-owned and read-only unless named `out_*`.
 *   - matrices are column-major (R layout); indices returned as artefacts are
 *     1-based like R's.
 *   - every function returns SGB_OK (0) or a negative error code; the message is
 *     available from sgb_last_error() (thread-local).
 *   - there is NO CPU fallback: without a usable CUDA device every compute
 *     entry point fails with SGB_ERR_CUDA.
 *   - random draws are never made inside the library: normals / uniforms are
 *     drawn by the caller from R's set.seed stream in the reference's order and
 *     passed in as buffers ("z" = standard normals, "u" = uniforms).
 */
#ifndef SOUNDGEN_B200_H
#define SOUNDGEN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGB_OK                 0
#define SGB_ERR_INVALID       -1   /* bad argument                                   */
#define SGB_ERR_CUDA          -2   /* CUDA runtime failure / no device               */
#define SGB_ERR_UNSUPPORTED   -3   /* valid in the reference, not in this library     */
#define SGB_ERR_SYNTH         -4   /* the reference would stop() ("Failed to generate
                                      the new syllable!", soundgen.R:624-626)          */
#define SGB_ERR_STREAM        -5   /* a z/u stream was shorter than the draws needed  */
#define SGB_ERR_STATE         -6   /* call sequence error on a batch handle           */

#define SGB_VERSION 200

int         sgb_version(void);
const char *sgb_last_error(void);
int         sgb_device_count(void);
int         sgb_set_device(int device);

/* Page-locks / unlocks a caller-owned host buffer so that the library's
 * cudaMemcpyAsync calls on it are true DMA transfers (optional). */
/* PCI bus id ("0000:1b:00.0") of a CUDA device: lets a one-process-per-GPU launcher bind the process to
 * the GPU's NUMA node before it allocates its pinned buffers. */
int sgb_device_pci_bus_id(int device, char *out, int cap);
int sgb_pin(void *ptr, int64_t bytes);
int sgb_unpin(void *ptr);
/* Measures the FP32 FMA throughput of the current device with a dependent-chain
 * FFMA2 kernel (TFLOP/s, FMA = 2 flop); used as the roofline denominator of the
 * additive-synthesis kernel, which is bound by the FP32 pipe, not by HBM. */
int sgb_measure_fp32_peak(double *out_tflops);

/* ------------------------------------------------------------------------- */
/* Batched whole-path interface: replaces the bout loop of soundgen()         */
/* (R/soundgen.R:482-849) for many calls at once.                             */
/* ------------------------------------------------------------------------- */

/* Anchors are (time, value) pairs stored interleaved in the `anchors` pool;
 * contour evaluation follows getSmoothContour (R/smoothContours.R:53-227): 1
 * anchor flat, 2 anchors seq(), 3-10 anchors loess (the reference's default
 * method, fitted on the device where the contour length is only known there),
 * more than 10 anchors or method 'spline': FMM spline. */
#define SGB_CONTOUR_LOESS  0
#define SGB_CONTOUR_SPLINE 1

/* One voiced syllable = one generateHarmonics() call (R/source.R:173-205). */
typedef struct sgb_syllable {
  int32_t kind;          /* 1 = synthesise; 0 = `silent_len` zeros (soundgen.R:608-613);
                            2 = raw samples given in `pitch` pool (used by sgb_filter)  */
  int32_t silent_len;
  int64_t pitch_off;     /* offset into `pitch` pool (doubles)                        */
  int32_t pitch_len;     /* P = round(dur * pitchSamplingRate / 1000)                 */
  int32_t pause_after;   /* zeros appended after the syllable (soundgen.R:632-640)    */
  int64_t z_off;         /* offset into `z` pool: this syllable's normal stream       */
  int32_t z_cap;         /* normals available                                         */
  int32_t ampl_n;        /* amplAnchors: number of anchors, 0 = NA                    */
  int64_t ampl_off;      /* offset (in pairs) into `anchors`                          */
  int32_t ampl_method;   /* SGB_CONTOUR_LOESS (reference default) or SGB_CONTOUR_SPLINE */
  int32_t pitch_anchor_n;/* > 0: the pitch contour is evaluated on the device from these
                            pitchAnchors (getSmoothContour, thisIsPitch = TRUE, len =
                            pitch_len, soundgen.R:596-603) and `pitch` is not read      */
  int64_t pitch_anchor_off; /* offset (pairs) into `anchors`                          */
  int32_t pitch_method;  /* contour method of the pitch anchors                       */
  int32_t reserved0;
  double pitch_scale;    /* pitchDeltas[s] (soundgen.R:603); used with pitch anchors  */
  double attackLen, nonlinBalance, jitterDep, jitterLen, vibratoFreq, vibratoDep,
         shimmerDep, rolloff, rolloffOct, rolloffKHz, rolloffParab, rolloffParabHarm,
         rolloff_perAmpl, temperature, pitchDriftDep, pitchDriftFreq,
         randomWalk_trendStrength, shortestEpoch, subFreq, subDep, samplingRate,
         pitchFloor, pitchCeiling, pitchSamplingRate, throwaway;
} sgb_syllable;

/* One formant filter = one getSpectralEnvelope() call (R/sourceSpectrum.R:261-283). */
typedef struct sgb_envelope {
  int32_t n_formants;    /* 0 = formants NA and vocalTract NULL (lip radiation only)  */
  int32_t tracks_given;  /* 1: `formants` holds nc pre-upsampled rows per formant (the
                            host ran the stochastic block sourceSpectrum.R:346-415);
                            2: a literal filter matrix (wl/2 x nc_fixed doubles, column-major)
                            at offset `formant_off` of the `pre` pool, e.g. generateNoise's
                            filterNoise argument (R/source.R:66-68, :95-101);
                            3: deferred -- the tracks need the bout's STFT frame count, which
                            the device decides: they arrive through sgb_batch_set_tracks()
                            between sgb_batch_run_begin() and sgb_batch_run_finish()     */
  int64_t formant_off;   /* offset into `formant_index` (one {off,n} entry per formant) */
  int32_t mouth_n;       /* mouthAnchors: number of anchors, 0 = NA                   */
  int32_t nc_fixed;      /* >0: number of columns; 0: one column per STFT frame       */
  int64_t mouth_off;     /* offset (pairs) into `anchors`                             */
  int32_t mouth_method;  /* contour method of the mouth anchors                       */
  int32_t reserved0;
  double formantDep, rolloffLip, mouthOpenThres, openMouthBoost,
         vocalTract /* NaN = NULL */, samplingRate, speedSound, smoothLinearFactor;
} sgb_envelope;

/* One unvoiced segment = one generateNoise() call (R/source.R:57-68). */
typedef struct sgb_noise {
  int32_t len;           /* unvoicedDur_syl                                           */
  int32_t insertion;     /* syllableStartIdx[s] (1-based, may be < 1)                 */
  int32_t mix;           /* 0: added before filtering (soundgen.R:708-714);
                            1: added after filtering (soundgen.R:813-818)             */
  int32_t wl;            /* windowLength_points                                       */
  int64_t u_off;         /* offset into `u` pool (nr*nc uniforms, column-major)       */
  int64_t anchor_off;    /* noise anchors (time ms, value dB), offset in pairs        */
  int32_t anchor_n;
  int32_t env_id;        /* index into envelopes[], -1 = no filterNoise               */
  int64_t strength_pre_off; /* >= 0: pre-evaluated dB contour (len doubles) in `pre`  */
  int32_t anchor_method; /* contour method of the noise anchors                       */
  int32_t reserved0;
  double rolloffNoise, attackLen, samplingRate, overlap;
} sgb_noise;

/* One bout (R/soundgen.R:482-843). */
typedef struct sgb_bout {
  int32_t syl_begin, syl_end;       /* [begin, end) in syllables[]                    */
  int32_t noise_begin, noise_end;   /* [begin, end) in noises[]                       */
  int32_t env_id;                   /* main vocal-tract filter                        */
  int32_t moving;                   /* movingFormants (soundgen.R:751-759)            */
  int32_t wl;                       /* windowLength_points before the clamp at :743   */
  int32_t lead_silence;             /* zeros before this bout in the call's output    */
  int32_t tail_silence;             /* zeros after it (addSilence on the last bout)   */
  int32_t aglobal_n;                /* amplAnchorsGlobal anchors (values already
                                       2^(dB/10), soundgen.R:724), 0 = NA             */
  int64_t aglobal_off;
  int32_t aglobal_method;           /* contour method of amplAnchorsGlobal            */
  int32_t reserved0;
  double overlap, amDep, amFreq, amShape, samplingRate, throwaway;
} sgb_bout;

/* One soundgen() call = consecutive bouts. */
typedef struct sgb_call {
  int32_t bout_begin, bout_end;
} sgb_call;

typedef struct sgb_formant_ref { int64_t off; int32_t n; int32_t pad; } sgb_formant_ref;

typedef struct sgb_batch_desc {
  int32_t n_calls, n_bouts, n_syllables, n_noises, n_envelopes, n_formant_refs;
  const sgb_call        *calls;
  const sgb_bout        *bouts;
  const sgb_syllable    *syllables;
  const sgb_noise       *noises;
  const sgb_envelope    *envelopes;
  const sgb_formant_ref *formant_index;
  const double *pitch;    int64_t n_pitch;     /* pitch contours                       */
  const double *anchors;  int64_t n_anchors;   /* (time, value) pairs: 2*n doubles     */
  const double *formants; int64_t n_formants;  /* rows of (time, freq, amp, width)     */
  const double *z;        int64_t n_z;         /* standard normals                     */
  const void   *u;        int64_t n_u;         /* uniforms, double or float            */
  int32_t       u_is_float;
  int32_t       reserved;
  const double *pre;      int64_t n_pre;       /* pre-evaluated contours               */
} sgb_batch_desc;

typedef struct sgb_batch sgb_batch;   /* opaque */

/* Stage timings of the last sgb_batch_run (CUDA events on the library's stream). */
enum { SGB_T_H2D = 0, SGB_T_CONTROL, SGB_T_AMPL, SGB_T_SYNTH, SGB_T_COMPOSE,
       SGB_T_NOISE, SGB_T_ASSEMBLE, SGB_T_ENVELOPE, SGB_T_FILTER, SGB_T_FINALIZE,
       SGB_T_D2H, SGB_T_TOTAL, SGB_T_COUNT };

typedef struct sgb_run_info {
  int64_t total_samples;      /* sum of output lengths over calls                     */
  int64_t synth_partials;     /* sum over epochs of rows * samples (K1 work units)    */
  int64_t synth_samples;      /* samples produced by K1                               */
  int64_t filter_samples;     /* samples emitted by K2                                */
  int64_t filter_frames;      /* STFT frames processed by K2 (incl. warm-up)          */
  int64_t noise_samples;      /* samples emitted by K5                                */
  int32_t kernel_launches;    /* kernels launched by this run                         */
  int32_t n_failed;           /* syllables/bouts whose reference call would stop()    */
  float   ms[SGB_T_COUNT];
} sgb_run_info;

int sgb_batch_create(sgb_batch **out);
void sgb_batch_destroy(sgb_batch *b);

/* Copies the description to the device (pinned staging + cudaMemcpyAsync). */
int sgb_batch_upload(sgb_batch *b, const sgb_batch_desc *desc);
/* Runs the whole path on data already resident on the device. */
int sgb_batch_run(sgb_batch *b, sgb_run_info *info);
/* Per-call output lengths (valid after run). */
int sgb_batch_lengths(sgb_batch *b, int64_t *out_len /* n_calls */);
/* Concatenated outputs of all calls, call c at sum(len[0..c)). */
int sgb_batch_fetch_f32(sgb_batch *b, float *out, int64_t n);
int sgb_batch_fetch_f64(sgb_batch *b, double *out, int64_t n);
/* The same, as the 16-bit PCM samples the reference's savePath branch writes (R/soundgen.R:855-857 ->
 * seewave::savewav -> tuneR::normalize(unit = "16")): centred, largest magnitude scaled to
 * min(1, max(x)), round(x * 32767).  Halves the device -> host bytes. */
int sgb_batch_fetch_pcm16(sgb_batch *b, int16_t *out, int64_t n);
/* Per-call failure flags (0 = ok, else an SGB_ERR_* code). */
int sgb_batch_status(sgb_batch *b, int32_t *out_status /* n_calls */);

/* Device output: results written straight into caller-owned device memory (for a consumer on the same GPU,
 * e.g. a model trained with PyTorch), with no trip through host memory.
 *
 * Row c is written from element dst_off[c] on: exactly cap[c] elements, the first min(len_c, cap_c) samples of the
 * row and then zeros (a padded [rows, T] tensor needs no separate clearing pass).  SGB_OUT_F32 copies the samples
 * bit for bit as sgb_batch_fetch_f32 returns them; SGB_OUT_PCM16 writes the 16-bit PCM of sgb_batch_fetch_pcm16,
 * normalised over the row's len_c source samples (same kernel, same bits), so cropping keeps the normalisation of
 * the whole row.
 *
 * Stream contract: nothing here waits on the host.  The library records an event on the caller's stream and
 * makes its own stream wait for it (the destination is free), runs the copy, records an event and makes the
 * caller's stream wait for that: work the caller queues on `stream` afterwards sees the rows.  Later runs of the
 * same handle are queued behind the export on the handle's stream, so they cannot overwrite the source first.
 * `stream` may come from another CUDA runtime in the process (torch's: torch.cuda.Stream.cuda_stream): both use
 * the device's primary context.
 *
 * Every argument is checked before anything is queued (SGB_ERR_INVALID): `dst` must be device (or managed)
 * memory of the batch's device, aligned to its element type; offsets and capacities non-negative, every row
 * inside [0, dst_elems), no two rows overlapping.  A handle without a completed run gives SGB_ERR_STATE.
 * There is no host path: without a device both calls return SGB_ERR_CUDA. */
#define SGB_OUT_F32    0
#define SGB_OUT_PCM16  1
typedef struct sgb_device_out {
  void          *dst;         /* device memory on the batch's device (float * or int16_t *)       */
  int64_t        dst_elems;   /* elements available at dst (bounds check)                         */
  const int64_t *dst_off;     /* host, n: first element of row c in dst                           */
  const int64_t *cap;         /* host, n: elements written for row c (samples, then zeros)        */
  int64_t       *out_written; /* host, n (may be NULL): min(len_c, cap_c)                         */
  void          *stream;      /* caller's cudaStream_t (NULL = the legacy default stream)         */
  int32_t        format;      /* SGB_OUT_F32 / SGB_OUT_PCM16                                      */
  int32_t        reserved;
} sgb_device_out;
/* Every call of the last run (n = n_calls rows, row c = call c) -> caller-owned device memory. */
int sgb_batch_export(sgb_batch *b, const sgb_device_out *o);
/* The same over n float32 rows the caller already holds on `device` (row c = len[c] samples at src + src_off[c]):
 * used to normalise to PCM16 a call assembled from several rounds, over the whole call. */
int sgb_rows_export(int32_t device, const float *src, const int64_t *src_off, const int64_t *len, int32_t n,
                    const sgb_device_out *o);

/* Spectrograms on the device, into caller-owned device memory (K9).  For a row x of L samples, window length wl
 * and hop h = wl - overlap*wl/100 (may be fractional):
 *   frames   k = 0 .. nc-1 start at the 1-based sample floor(1 + k*h), nc = length(seq(1, max(1, L - wl), h))
 *            (soundgen.R:744-746), nc = 0 when L = 0; samples past L read as 0 (one zero-padded frame when L <= wl);
 *   spectrum X_k(j) = (1/wl) sum_n x[s_k - 1 + n] w(n) exp(-2 pi i n j / wl), j = 0 .. wl/2 - 1 (seewave's stft as
 *            soundgen's filter calls it), w = seewave's symmetric hamming.w or hanning.w;
 *   power    P_k(j) = |X_k(j)|^2;  bands (optional): F_k(b) = sum_j B_b(j) P_k(j) over the contiguous bins
 *            [band_lo[b], band_lo[b] + band_len[b]) inside [0, wl/2), weights band_w in that order, row after row;
 *            without bands F = P and n_feat = wl/2, else n_feat = n_bands;
 *   dB       (optional) 10 log10(max(F, db_floor)).
 * Layout as sgb_device_out describes it, with cap counted in frames: row c gets exactly cap[c] frames of n_feat
 * floats from element dst_off[c] on, frame after frame; frames >= nc are zeros; out_written[c] = min(nc, cap[c]);
 * a row with cap[c] = 0 is left alone (one call per sampling-rate group of a batch).  format must be SGB_OUT_F32.
 * Frames 2m and 2m+1 share one complex FFT, always: a row's values do not depend on cap or on the other rows.
 * Stream contract, pinned staging and argument checks are those of the exports.  A wl that cannot be planned or
 * whose working set does not fit in shared memory gives SGB_ERR_UNSUPPORTED; a bad overlap (hop < 1), window,
 * band, weight or db_floor gives SGB_ERR_INVALID. */
#define SGB_WIN_HAMMING 0
#define SGB_WIN_HANNING 1
typedef struct sgb_spec_params {
  int32_t wl, window;            /* even, >= 4; SGB_WIN_*                                           */
  double  overlap;               /* percent; hop = wl - overlap*wl/100 must be >= 1                 */
  int32_t n_bands, db;           /* n_bands = 0: no filterbank; db: 0 power, 1 10*log10             */
  double  db_floor;              /* > 0 when db                                                     */
  const int32_t *band_lo, *band_len;  const float *band_w;   /* host, n_bands rows (CSR)            */
} sgb_spec_params;
/* nc of a row of `len` samples (0 when len = 0), or -1 for a bad wl / overlap. */
int64_t sgb_spec_frames(int64_t len, int32_t wl, double overlap);
/* Every call of the last run (row c = call c). */
int sgb_batch_spectrogram(sgb_batch *b, const sgb_spec_params *p, const sgb_device_out *o);
/* n float32 rows the caller holds on `device` (row c = len[c] samples at src + src_off[c]). */
int sgb_rows_spectrogram(int32_t device, const float *src, const int64_t *src_off, const int64_t *len,
                         int32_t n, const sgb_spec_params *p, const sgb_device_out *o);

/* Similarity of spectrogram rows on the device (K10), one float64 score per pair into caller-owned device memory.
 * Pair c compares row a_c (a_frames[c] frames of n_feat floats, frame after frame, from element a_off[c] of a) with
 * row b_c (likewise in b); pairs may share rows.  With N = max(n_a, n_b), the frames past the shorter row read as
 * `pad` in every feature:
 *   SGB_CMP_COR     Pearson correlation over the N * n_feat cells (two-pass, FP64);
 *   SGB_CMP_COSINE  <a, b> / (|a| |b|) over the same cells (FP64);
 *   SGB_CMP_DTW     -D(n_a, n_b) / (n_a + n_b), no padding: cell cost d(i, j) = |a_i - b_j|_2 over the features (FP32),
 *                   step pattern symmetric2 of R's dtw package, D(1, 1) = d(1, 1) and
 *                   D(i, j) = min(D(i-1, j-1) + 2 d, D(i-1, j) + d, D(i, j-1) + d) (FP64).
 * Higher is more similar.  A row with 0 frames gives NaN, and so does a constant side (cor) or an all-zero side
 * (cosine), as 0/0 does.  A pair's score does not depend on the other pairs, their order or their number.
 * dst gets n scores (8-byte aligned device memory of `device`, dst_elems >= n); a and b must be device memory of
 * `device` (checked when a row of that side has frames).  The stream contract and pinned staging are those of the
 * exports: ordered after the work queued on `stream` so far, and the caller's later work on `stream` sees dst, with
 * no host wait.  Refused before anything is queued: an unknown method, n_feat < 1, a non-finite pad, negative
 * offsets or frames, a row outside a_elems / b_elems, or bad pointers give SGB_ERR_INVALID; a DTW row of more than
 * SGB_CMP_DTW_MAX_FRAMES frames gives SGB_ERR_UNSUPPORTED (its wavefront lives in shared memory). */
#define SGB_CMP_COR    0
#define SGB_CMP_COSINE 1
#define SGB_CMP_DTW    2
#define SGB_CMP_DTW_MAX_FRAMES 4096
typedef struct sgb_compare_params {
  int32_t method, n_feat;        /* SGB_CMP_*; floats per frame                                     */
  double  pad;                   /* value of the frames past the shorter row (cor, cosine)          */
} sgb_compare_params;
int sgb_rows_compare(int32_t device, const float *a, int64_t a_elems, const float *b, int64_t b_elems,
                     const int64_t *a_off, const int64_t *a_frames, const int64_t *b_off, const int64_t *b_frames,
                     int32_t n, const sgb_compare_params *p, double *dst, int64_t dst_elems, void *stream);
/* Cepstra and their deltas of spectrogram rows on the device (K11), into caller-owned device memory.  Row c has
 * frames[c] = nc frames of n_in floats, frame after frame, from element src_off[c] of src (rows as
 * sgb_rows_spectrogram writes them, typically log-mel).  With the caller's matrix M [n_ceps, n_in] (row-major,
 * e.g. an orthonormal DCT-II for MFCCs), for frame t of a row:
 *   cepstra  c_t[k] = sum_b M[k, b] x_t[b], FP32 in a fixed order of b;
 *   deltas   order 1, N = delta_n in 1..8:
 *            d_t = (sum_{j=1..N} j (c_{min(t+j, nc-1)} - c_{max(t-j, 0)})) / (2 sum_{j=1..N} j^2),
 *            the row's first and last frames replicated at its edges (torchaudio's compute_deltas with
 *            win_length 2N + 1 over the row's nc frames alone); order 2 adds the same formula over the d_t;
 *   output   frame t = [c_t | d_t | dd_t], n_out = n_ceps (1 + delta_order) floats.
 * Layout as sgb_device_out describes it, with cap counted in frames: row c gets exactly cap[c] frames of n_out
 * floats from element dst_off[c] on; frames >= nc are zeros; out_written[c] = min(nc, cap[c]); a row with
 * cap[c] = 0 is left alone.  format must be SGB_OUT_F32.  Frames at or past nc are never read, and the deltas near
 * cap read the input past cap (up to nc): a row's values do not depend on cap or on the other rows, so a cropped
 * row is a bit-exact prefix of the whole one.  Stream contract and pinned staging are those of the exports.
 * Refused before anything is queued: n_in or n_ceps < 1, a null or non-finite matrix, delta_order not in {0, 1, 2},
 * delta_n not in 1..8, negative offsets or frames, a row outside src_elems, frames[c] or cap[c] above 2^31 - 1,
 * the export's checks on dst, a dst range [dst, dst + dst_elems) that intersects [src, src + src_elems), or src not
 * device memory of `device` give SGB_ERR_INVALID.  A working set over 226 KB of shared memory gives
 * SGB_ERR_UNSUPPORTED: with ld = n_in | 1, S = 64 + 2 delta_order delta_n, it is
 *   4 (n_ceps ld + S ld + S n_ceps + (delta_order == 2 ? (64 + 2 delta_n) n_ceps : 0)) <= 226 * 1024 bytes,
 * which holds for every delta_order and delta_n up to n_in 256 and n_ceps 64 (205 KB at the largest). */
typedef struct sgb_ceps_params {
  int32_t n_in, n_ceps;          /* floats per input frame; cepstra per frame                       */
  const float *matrix;           /* host, n_ceps * n_in, row-major                                  */
  int32_t delta_order, delta_n;  /* 0, 1 or 2; 1..8                                                 */
} sgb_ceps_params;
int sgb_rows_cepstra(int32_t device, const float *src, int64_t src_elems, const int64_t *src_off,
                     const int64_t *frames, int32_t n, const sgb_ceps_params *p, const sgb_device_out *o);
/* The f0 track of every call of the last run (K12a), aligned sample for sample with the rows sgb_batch_export
 * writes: the fundamental frequency in Hz of the contour the harmonics of that sample were built on, 0 where the
 * sample is unvoiced.  A sample is voiced when it lies in the span of a voiced syllable (not a pause, a silence, a
 * noise-only stretch, a filter tail past the last syllable, or any sample of a failed call).  Its value is
 * pitch_upsampled of the reference (source.R:382, after vibrato, jitter, drift and pitchAnchorsGlobal) at the
 * sample's position in the epoch that produced it -- the incoming epoch inside a cross-fade, the first epoch's
 * first sample for the two leading zeros of a syllable -- evaluated in FP64 from the spline piece K1's phase
 * integrates, rounded to float once.  With sub-harmonics (nSubharm > 0) the partials are multiples of
 * f0 / (nSubharm + 1); the track still reports f0.
 * Layout, capacity, zero tail, crop, argument checks and stream contract are those of sgb_batch_export (row c gets
 * exactly cap[c] floats, out_written[c] = min(len_c, cap_c)); format must be SGB_OUT_F32. */
int sgb_batch_f0(sgb_batch *b, const sgb_device_out *o);
/* Frame labels of n float32 rows on `device` (K12b), typically f0 tracks of sgb_batch_f0: row c = len[c] samples
 * at src + src_off[c], inside [src, src + src_elems).  Frames k = 0 .. nc-1 are K9's for the same wl and overlap
 * (start s_k = floor(1 + k h), nc = sgb_spec_frames(len, wl, overlap)); label k is two floats:
 *   [x[s_k - 1 + wl/2] (0 at or past len),  (nonzero samples in [s_k - 1, s_k - 1 + wl) ∩ [0, len)) / wl],
 * the count exact in integers and divided once.  Row c gets exactly cap[c] labels (2 cap[c] floats) from element
 * dst_off[c] on, zeros past nc; out_written[c] = min(nc, cap[c]); a label does not depend on cap or on other rows.
 * Refused before anything is queued with SGB_ERR_INVALID: wl odd or < 4, overlap outside [0, 100) or a hop below
 * one sample, a format other than SGB_OUT_F32, a row outside src_elems, the export's checks on dst, a dst range
 * that intersects [src, src + src_elems), src or dst not device memory of `device`.  No device: SGB_ERR_CUDA.
 * Stream contract and pinned staging are those of the exports. */
int sgb_rows_f0_frames(int32_t device, const float *src, int64_t src_elems, const int64_t *src_off,
                       const int64_t *len, int32_t n, int32_t wl, double overlap, const sgb_device_out *o);
/* default, low and high of a scalar argument of soundgen() as the front-end checks it (permittedValues,
 * R/presets.R:22-79); SGB_ERR_INVALID for a name the front-end does not range-check. */
int sgb_param_range(const char *name, double out3[3]);

/* Intermediate results (valid after run).  Sizes via the *_len calls. */
int sgb_batch_syllable_len(sgb_batch *b, int32_t syl, int64_t *out_len);
int sgb_batch_syllable_fetch(sgb_batch *b, int32_t syl, double *out, int64_t n);
int sgb_batch_noise_fetch(sgb_batch *b, int32_t noise, double *out, int64_t n);

/* Integer artefacts of one voiced syllable (bit-exact contract, SURVEY.md 8c). */
typedef struct sgb_syl_artefacts {
  int32_t nGC, nHarmonics, rows_kept, nEpochs, n_upsampled, n_jitter_idx, z_used, status;
  double  raw_max;
} sgb_syl_artefacts;
int sgb_batch_artefacts(sgb_batch *b, int32_t syl, sgb_syl_artefacts *out);
/* which: 0 gc (nGC), 1 gc_upsampled (nGC+1), 2 nSubharm (nGC), 3 rw_bin (nGC),
 *        4 jitter idx, 5 epochs (2*nEpochs: start,end), 6 zero crossings
 *        (2*nEpochs: zc1, zc2; 0 = NA) */
int sgb_batch_artefact_ints(sgb_batch *b, int32_t syl, int which, int32_t *out, int32_t cap);
int sgb_batch_pitch_per_gc(sgb_batch *b, int32_t syl, double *out, int32_t cap);
/* Diagnostic: the amplitude tables of epoch `epoch` of syllable `syl` of the last run.  shape[3] receives
 * {rows, columns, pairs}.  f64 (cap >= rows * columns doubles) receives the FP64 matrix, column by column;
 * f32 (4 * cap floats) the epoch's FP32 table region, 16 bytes per element: with pairs, {Y_g, Y_{g+1} - Y_g}
 * float pairs for columns 0..columns-2 at its start and zeros after; otherwise {Y, Y, dY, dY} per element.
 * Null f64 and f32 report the shape only. */
int sgb_batch_amp_tables(sgb_batch *b, int32_t syl, int32_t epoch, double *f64, float *f32, int64_t cap,
                         int32_t *shape);
/* Diagnostic: the FP32 spectral envelope the last run filtered with.  kind 0: the main filter of bout `index`;
 * kind 1: the filter of noise `index`.  shape[2] receives {nr, nint}; out (cap >= nr * nint floats) the table
 * column by column, copied on the handle's stream (the call returns once it has arrived).  A bypassed bout or an
 * unfiltered noise has shape {0, 0}; a null out reports the shape only.  SGB_ERR_STATE before the first run. */
int sgb_batch_envelope(sgb_batch *b, int32_t kind, int32_t index, float *out, int64_t cap, int32_t *shape);
/* Diagnostic: nine position-weighted checksums of the last run's intermediates (see engine.cu);
 * identical inputs must give identical checksums on every run. */
int sgb_batch_checksums(sgb_batch *b, uint64_t *out, int32_t cap);
/* Diagnostic for a stuck run, callable from another thread: out[0] = the wait the handle's host thread is
 * in, out[1..11] = completion of the stage events of the current run (see engine.cu). */
int sgb_batch_debug_state(sgb_batch *b, int32_t *out, int32_t cap);

/* Two-phase run: sgb_batch_run == sgb_batch_run_begin + sgb_batch_run_finish.  Between the two the
 * lengths that only the device can know (syllables after their zero-crossing joins, hence STFT
 * frames per bout) are available, which is what the host needs to draw the stochastic formant
 * tracks of a moving main filter in R's order (getRandomWalk(len = nc), sourceSpectrum.R:346-415). */
int sgb_batch_run_begin(sgb_batch *b);
int sgb_batch_run_finish(sgb_batch *b, sgb_run_info *info);
/* After run_begin: geometry of one bout (STFT frames, envelope columns, clamped window, length(sound)). */
int sgb_batch_bout_geometry(sgb_batch *b, int32_t bout, int32_t *nc, int32_t *nint, int32_t *wl, int32_t *sound_len);
/* Between begin and finish: replaces envelope `env` by host-drawn tracks (tracks_given = 1):
 * rows = n_formants blocks of nc rows (time, freq, amp, width). */
int sgb_batch_set_tracks(sgb_batch *b, int32_t env, const double *rows, int32_t n_formants, int32_t nc);
/* Normal draws each voiced syllable consumed (valid after run_begin); n_syllables values. */
int sgb_batch_z_used(sgb_batch *b, int32_t *out);
/* sizeof() of the ABI structs, for bindings to verify their mirrors:
 * syllable, envelope, noise, bout, call, formant_ref, batch_desc, run_info, soundgen_args, device_out, spec_params,
 * compare_params, ceps_params (cap >= 9; the 10th to 13th are written when cap allows). */
int sgb_abi_sizes(int32_t *out, int32_t cap);
/* The additive synthesis has two kernels: epochs with at least `rows` rows run on the tensor cores, the others on the
   FP32 pipe (default 224, or SGB_SYNTH / SGB_SYNTH_MIN_ROWS from the environment).  0 = tensor cores only, a huge value =
   FP32 pipe only, -1 = back to the default.  Applies to batches that run after the call; meant for tests and A/B runs. */
int sgb_synth_min_rows_set(int32_t rows);
/* Worker threads of the library's host stage (front-end registration, round_begin, resolve, layout checks):
   0 = SGB_FRONTEND_THREADS from the environment, else the hardware's, at most 16. */
int sgb_host_set_threads(int32_t n);

/* ------------------------------------------------------------------------- */
/* Host front-end: the host stage of soundgen() (R/soundgen.R:279-733)         */
/* ------------------------------------------------------------------------- */
/* Argument validation against permittedValues, hyper-parameters, syllable segmentation and -- with
 * temperature > 0 -- every draw the reference makes from R's RNG stream, in the reference's order
 * ("RNG ledger", SURVEY.md 8a): rbinom (fractional nSyl / repeatBout), rnorm_bounded, divideIntoSyllables,
 * wiggleAnchors, the normals generateHarmonics consumes, stochastic formants, runif for the noise.
 * The stream is R's: Mersenne-Twister seeded like set.seed(seed) (or continued from a caller-supplied
 * .Random.seed), inversion normals, R < 3.6 sample().  The result is an sgb_batch_desc for
 * sgb_batch_upload; nothing here computes samples. */

typedef struct sgb_anchor_arg {      /* a data.frame(time, value); n = 0: NA                    */
  const double *time;                /* NULL: plain numeric vector (soundgen.R:305-315)         */
  const double *value;
  int32_t n, reserved;
} sgb_anchor_arg;

typedef struct sgb_formant_arg {     /* one formant: list(time, freq, amp, width), each recycled */
  const double *time, *freq, *amp, *width;
  int32_t n_time, n_freq, n_amp, n_width;
} sgb_formant_arg;

typedef struct sgb_soundgen_args {   /* arguments of soundgen(), R/soundgen.R:208-277 */
  double repeatBout, nSyl, sylLen, pauseLen, temperature, maleFemale, creakyBreathy, nonlinBalance,
         nonlinDep, jitterLen, jitterDep, vibratoFreq, vibratoDep, shimmerDep, attackLen, rolloff,
         rolloffOct, rolloffKHz, rolloffParab, rolloffParabHarm, rolloffLip, formantDep,
         formantDepStoch, vocalTract, subFreq, subDep, shortestEpoch, amDep, amFreq, amShape,
         rolloffNoise, samplingRate, windowLength, overlap, addSilence /* NaN = NULL */, pitchFloor,
         pitchCeiling, pitchSamplingRate, throwaway;
  /* tempEffects: sylLenDep, formDrift, formDisp, pitchDriftDep, pitchDriftFreq, pitchAnchorsDep,
   * noiseAnchorsDep, amplAnchorsDep (NaN = missing; all but sylLenDep then get their defaults) */
  double tempEffects[8];
  sgb_anchor_arg pitchAnchors, pitchAnchorsGlobal, noiseAnchors, mouthAnchors, amplAnchors, amplAnchorsGlobal;
  const sgb_formant_arg *formants;      int32_t n_formants;       /* 0 = NA */
  int32_t reserved0;
  const sgb_formant_arg *formantsNoise; int32_t n_formantsNoise;  /* 0 = NA */
  int32_t invalidArgAction;             /* 0 adjust, 1 abort, 2 ignore (soundgen.R:285-300)     */
  int32_t contour_method;               /* SGB_CONTOUR_LOESS (reference) / SGB_CONTOUR_SPLINE   */
  int32_t rng_mode;                     /* 0: R stream from `seed`; 1: continue `rng_state`;
                                           2: caller buffers z / u (temperature must be 0)       */
  uint32_t seed;
  int32_t sample_rejection;             /* 1: R >= 3.6 sample() ("Rejection")                   */
  const int32_t *rng_state;             /* rng_mode 1: .Random.seed[2:626]                      */
  /* rng_mode 2: one normal buffer per voiced syllable / one uniform buffer per noise segment    */
  const double *z; const int64_t *z_len; int32_t n_z; int32_t device_pitch;
  const void *u;   const int64_t *u_len; int32_t n_u; int32_t reserved1;
} sgb_soundgen_args;

typedef struct sgb_frontend sgb_frontend;   /* opaque */
int  sgb_frontend_create(sgb_frontend **out, int32_t u_is_float);
void sgb_frontend_destroy(sgb_frontend *fe);
/* Registers one soundgen() call; returns the call index or an error.  Scalars and tables are copied; the
 * caller-drawn buffers `z` and `u` (rng_mode 2) are referenced and must stay valid until the call's last round ended.
 * The host stage up to the bout loop (validation, hyper-parameters, rbinom draws) runs here. */
int  sgb_frontend_add(sgb_frontend *fe, const sgb_soundgen_args *args);
/* n calls that differ only in their seed (rng_mode 0): returns the index of the first. */
int  sgb_frontend_add_seeded(sgb_frontend *fe, const sgb_soundgen_args *args, const uint32_t *seeds, int32_t n);
/* `n` argument lists in one call (index of the first, or an error); the pointers inside every element must stay
   valid until the last round of these calls has ended */
int  sgb_frontend_add_many(sgb_frontend *fe, const sgb_soundgen_args *args, int32_t n);
/* forget every registered call; the handle and its buffers are reused */
int  sgb_frontend_clear(sgb_frontend *fe);
/* Builds the description of the next round.  One round covers every call that still has bouts
 * to generate, up to and including the first bout whose main filter has to be drawn after the
 * device has run (stochastic moving formants): most batches need exactly one round.
 * *n_subcalls = 0 when every call is complete. */
int  sgb_frontend_round_begin(sgb_frontend *fe, sgb_batch_desc *desc, int32_t *n_subcalls);
/* Call between sgb_batch_run_begin and sgb_batch_run_finish: draws the deferred formant tracks. */
int  sgb_frontend_resolve(sgb_frontend *fe, sgb_batch *b);
/* After sgb_batch_run_finish: records statuses / lengths, checks the draw counts against the device. */
int  sgb_frontend_round_end(sgb_frontend *fe, sgb_batch *b);
/* Which original call each sub-call of the current round belongs to (n_subcalls values). */
int  sgb_frontend_round_calls(sgb_frontend *fe, int32_t *out);
/* Status of every registered call so far (SGB_OK or the first error), warnings text of a call. */
int  sgb_frontend_status(sgb_frontend *fe, int32_t *out);
const char *sgb_frontend_warnings(sgb_frontend *fe, int32_t call);
/* rng_mode 0/1: the call's stream state after everything drawn so far (.Random.seed[2:626]). */
int  sgb_frontend_rng_state(sgb_frontend *fe, int32_t call, int32_t *out625);
/* Bytes the current round's description uploads. */
int64_t sgb_frontend_h2d_bytes(sgb_frontend *fe);

/* R's stream by itself (set.seed(seed); runif / rnorm / rexp / rgamma / rbinom / sample): used by the
 * bindings and by the tests that pin the stream to published R answers.
 * kind: 0 runif, 1 rnorm, 2 rexp, 3 rgamma(shape = p1, rate = p2), 4 rbinom(size = p1, prob = p2),
 *       5 sample.int(p1, 1). */
int sgb_rng_draw(uint32_t seed, int32_t kind, double p1, double p2, int32_t skip_uniforms, double *out, int32_t n);
/* getSmoothContour on the host (same scalar code the kernels run): out[len]. */
int sgb_smooth_contour(const double *time, const double *value, int32_t n, int32_t len, double samplingRate,
                       int32_t has_floor, double valueFloor, int32_t has_ceiling, double valueCeiling,
                       int32_t thisIsPitch, int32_t method, double *out);

/* ------------------------------------------------------------------------- */
/* Single-call interfaces                                                     */
/* ------------------------------------------------------------------------- */

/* getRolloff (R/sourceSpectrum.R:71-186).  rolloff / rolloffOct / rolloffKHz are
 * vectors of length 1 or nGC (n_* gives which).  out: nHarmonics x nGC doubles,
 * column-major, of which the first *out_rows rows per column are valid after
 * compaction (leading dimension stays nHarmonics); rownames are 1..*out_rows.
 * rolloffParabCeiling < 0 means NULL. */
int sgb_get_rolloff(const double *pitch_per_gc, int32_t nGC, int32_t nHarmonics,
                    const double *rolloff, int32_t n_rolloff,
                    const double *rolloffOct, int32_t n_rolloffOct,
                    const double *rolloffKHz, int32_t n_rolloffKHz,
                    double rolloffParab, double rolloffParabHarm,
                    double rolloffParabCeiling, double baseline, double throwaway,
                    double samplingRate, double *out, int32_t *out_rows);

/* getSpectralEnvelope (R/sourceSpectrum.R:261-566), deterministic part.
 * formants: n_formants blocks, block f has formant_n[f] rows of
 * (time, freq, amp, width).  out: nr x nc doubles, column-major. */
int sgb_get_spectral_envelope(int32_t nr, int32_t nc, const sgb_envelope *env,
                              const double *formants, const int32_t *formant_n,
                              const double *mouth_anchors, double *out);

/* STFT -> envelope multiply -> ISTFT -> /max (R/soundgen.R:743-807 with
 * seewave::stft / istft, seewave.r:7782-7818, :3447-3487).  envelope: nr x nInt,
 * nInt in {1, nc}.  out must hold sgb_filter_len() doubles. */
int64_t sgb_filter_len(int64_t len, int32_t wl, double overlap);
int sgb_filter(const double *sound, int64_t len, const double *envelope, int32_t nInt,
               int32_t wl, double overlap, double *out, int64_t out_cap);

#ifdef __cplusplus
}
#endif
#endif /* SOUNDGEN_B200_H */
