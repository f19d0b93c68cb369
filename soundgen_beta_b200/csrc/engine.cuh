// Device-side data model shared by the kernels and the host engine.
#pragma once
#include <cuda_runtime.h>
#include "ctrl.cuh"

#define SYNTH_THREADS 128
#define SYNTH_SPT 4                         // samples per thread
#define SYNTH_TILE (SYNTH_THREADS * SYNTH_SPT)
#define SYNTH_KMAX 128                      // rows per Clenshaw block when a warp sees one glottal cycle
#define SYNTH_STAGE 128                     // float4 entries per warp stage: columns x rows per block
#define SYNTH_PC 6                          // doubles per spline piece {kt, c0..c4}

// Formants per filter: the given ones, the stochastic pseudo-formants and host-drawn tracks together (K4 adds the
// nasal pole and zero on top).  K4 keeps 7 FP64 values per formant for each of its 4 warps in dynamic shared memory,
// sized by the launch's largest count: 224 B x (1024 + 2) = 229,824 B, inside the 232,448 B a block may opt in to.
#define SGB_MAX_FORMANTS 1024

// Pooled per-glottal-cycle scratch: syllable s owns [gc_off[s], gc_off[s+1]) of every array.
struct Pools {
  double *pitch_w;      // vibrato'd pitch, same layout as the pitch pool
  int32_t *gc, *nsub, *rwbin, *jidx, *gcup, *rowmap;
  double *ppg, *rw, *ro, *roct, *rk, *shimmer, *drift, *subdep, *colmax, *kt, *sb, *sc, *sd, *phi,
      *t1, *t2, *t3, *t4;
  double *pc;              // [6 * cap] per spline piece: knot, quartic phase polynomial (K1)
  const int64_t *gc_off;   // [S+1] prefix of (cap+1)
  const int64_t *h_off;    // [S+1] prefix of hcap
  // per syllable three contours, index 3 s + role: 0 the pitch, 1 the amplitude envelope over the glottal cycles
  // (K0), 2 the amplitude envelope over the composed syllable (K6); they differ in their ceiling
  ContourTab *ctab;        // [3 S] headers (k_syl_contours)
  double *knots;           // the batch's knot pool (contour.cuh)
  const int64_t *koff;     // [3 S + noises + bouts] first knot of each contour in the pool
};

__device__ inline SylArrays make_arrays(const Pools &P, const sgb_syllable &sp, int s) {
  SylArrays A;
  int64_t o = P.gc_off[s];
  A.pitch = P.pitch_w + sp.pitch_off;
  A.gc = P.gc + o; A.nsub = P.nsub + o; A.rwbin = P.rwbin + o; A.jidx = P.jidx + o; A.gcup = P.gcup + o;
  A.ppg = P.ppg + o; A.rw = P.rw + o; A.ro = P.ro + o; A.roct = P.roct + o; A.rk = P.rk + o;
  A.shimmer = P.shimmer + o; A.drift = P.drift + o; A.subdep = P.subdep + o; A.colmax = P.colmax + o;
  A.kt = P.kt + o; A.sb = P.sb + o; A.sc = P.sc + o; A.sd = P.sd + o; A.phi = P.phi + o;
  A.t1 = P.t1 + o; A.t2 = P.t2 + o; A.t3 = P.t3 + o; A.t4 = P.t4 + o;
  A.rowmap = P.rowmap + P.h_off[s];
  A.cap = (int32_t)(P.gc_off[s + 1] - o - 1);
  A.hcap = (int32_t)(P.h_off[s + 1] - P.h_off[s]);
  return A;
}

// Per-syllable offsets produced by the size scan (device) and the layout (host).
struct SylLayout {
  int64_t amp_off;     // doubles, into the amplitude pool
  int64_t wave_off;    // floats, into the epoch-waveform pool
  int64_t raw_off;     // floats, into the composed-syllable pool (capacity n_up + 2)
  int32_t tile_off;    // first K1 tile
  int32_t pad;         // first tile slot of the tensor-core K1 work list
};

// One K1 tile: SYNTH_TILE samples of one epoch.  gi_lo / a_lo are the amplitude interval and the
// spline piece of the tile's first sample (the warps scan forward from there).
struct SynthTile { int32_t syl; int32_t epoch; int32_t k0; int32_t gi_lo; int32_t a_lo; int32_t pad[3]; };
// One unit of the tensor-core K1: the samples [kbeg, kend) of one epoch that lie in ONE interval of approx()
// (one amplitude column), with everything the kernel needs so that it never touches SylCtrl.
struct TcUnit {
  int64_t col_off;      // first {Y, dY} pair (float2) of the interval's column in the amplitude table (row j - 1)
  int64_t wave_off;     // sample 0 of the epoch in the wave buffer
  int64_t pc_off;       // the syllable's first spline piece
  double x_first, by, x_last, inv_sr_np1;
  int32_t Ne, kbeg, kend, xg, xn, a_lo, G, J, epmax_idx, pad;
};

// Host-computed layout of one bout (after syllable lengths are known).
struct BoutLayout {
  int64_t sound_off;     // floats into the sound pool (16-byte aligned)
  int64_t filt_off;      // floats into the filtered pool
  int64_t env_off;       // floats into the envelope pool
  int64_t out_off;       // position of this bout's first sample in the output pool
  int32_t sound_len;     // length(sound) before filtering
  int32_t voiced_shift;  // index of the first voiced sample inside `sound`
  int32_t wl;            // clamped window (soundgen.R:743)
  int32_t nc;            // STFT frames
  int32_t nint;          // envelope columns (1 or nc)
  int32_t filt_len;      // length(soundFiltered) (= sound_len when bypassed)
  int32_t final_len;     // after post-filter noise insertion
  int32_t final_shift;   // index of filtered[0] inside the final bout
  int32_t bypass;        // sum(sound) == 0 -> no filtering
  int32_t fft_plan;      // index into the FFT plan table
  int32_t pad0, pad1;
};

struct SylPlace {        // where a syllable's samples go inside its bout's `sound`
  int64_t dst_off;       // absolute float offset in the sound pool
  int32_t len;
  int32_t bout;
};

struct NoiseLayout {
  int64_t raw_off;       // floats into the noise pool (len samples)
  int64_t env_off;       // floats into the envelope pool (nr x nc), -1 none
  int64_t dst_off;       // absolute float offset of noise[0] in the sound / output pool
  int32_t nc_env;        // envelope columns
  int32_t nc;            // ISTFT frames
  int32_t xlen;          // ISTFT output length
  int32_t trim_start;    // 0-based index into the (virtually padded) ISTFT output of noise[0]
  int32_t pad_len;       // zeros virtually prepended by matchLengths (0 or len)
  int32_t fft_plan;
  int32_t bout;
  int32_t pad;
};

struct EnvInst {
  int64_t out_off;      // floats (or doubles) into the envelope pool
  int32_t env_id;
  int32_t nr;
  int32_t nc;
  int32_t col0;         // first column of this instance in the flat (instance, column) work list
  int64_t trk_off;      // doubles into the formant-track scratch (nc x F x 3), -1: formants do not move
  int64_t mouth_koff;   // doubles into the envelope knot pool: the mouth-opening contour's knots, -1 none
  int64_t fit_off;      // doubles into the envelope knot pool: per moving track 2 nPoints + 5 na (k_env_tracks)
};


#define FFT_THREADS 512
#define FFT_MAX_PASS 16

struct FftPlan {
  int32_t n;                 // FFT length = window length (even)
  int32_t npass;
  int32_t radix[FFT_MAX_PASS];
  int64_t tw_off;            // float2[n]: exp(-2*pi*i*t/n)
  int64_t wa_off;            // float[n]: analysis window (Hamming) / n
  int64_t ws_off;            // float[n]: synthesis window (Hanning) * h / (sum(win^2) * n)
  int64_t wh_off;            // float[n]: Hanning analysis window / n (K9)
  double h_in;               // wl - overlap*wl/100  (frame starts 1 + k*h_in)
  double h_out;              // wl*(100-overlap)/100 (OLA offsets k*h_out)
};

struct FftJob {              // one sound (bout to filter, or noise segment to generate)
  int64_t in_off;            // filter: floats into the sound pool; noise: offset into the u pool
  int64_t out_off;           // floats into the output pool
  int64_t env_off;           // floats into the envelope pool (nr x nint), -1: none
  int32_t plan;
  int32_t nc;                // frames
  int32_t nint;              // envelope columns
  int32_t xlen;              // ISTFT output length
  int32_t out_len;           // filter: xlen; noise: len
  int32_t shift;             // noise: out index = t - shift (matchLengths trim), filter: 0
  int32_t max_slot;          // index into the per-job signed-max array
  int32_t pad;
  double rolloffNoise;       // noise only
};

struct FftSeg { int32_t job, ka, kb, pad; };

struct SpecRow {             // one row of a spectrogram (K9); nc and cap count frames
  int64_t src_off;           // floats into the source
  int64_t dst_off;           // floats into the destination
  int64_t len;               // samples
  int64_t nc;                // frames of the row
  int64_t cap;               // frames written (the first min(nc, cap) computed, the rest zeros)
};

struct CepsRow {             // one row of cepstra (K11); nc counts input frames, cap output frames
  int64_t src_off;           // floats into the source
  int64_t dst_off;           // floats into the destination
  int32_t nc, cap;
};
struct CepsTile { int32_t row, t0, t1, zero; };   // output frames [t0, t1) of a row; zero: the tail past nc
constexpr int CEPS_TILE = 64;                     // most frames of a compute tile (the choice: kernels_ceps.cu)

// f0 track (K12a).  A voiced span: n output samples of a row from sample t0 on, the composed samples [0, n) of
// syllable syl.  A row's spans are sorted and disjoint; everything outside them is unvoiced.
struct F0Span { int64_t t0; int32_t n, syl; };
// one CTA of K12a: samples [chunk * F0_CHUNK, (chunk + 1) * F0_CHUNK) of a row, whose spans are [s_lo, s_hi)
struct F0Chunk { int32_t row, chunk, s_lo, s_hi; };
// K6's epoch spans of one syllable, replayed by k_f0_epochs: epoch e covers the composed positions q >= ep[e].x
// (up to the next epoch's), where pitch_upsampled is read at the 1-based index u = ep[e].y + q
struct F0Epochs { int32_t nE, G; int2 ep[SGB_MAX_EPOCHS]; };
constexpr int F0_THREADS = 256, F0_PER_THREAD = 32, F0_CHUNK = F0_THREADS * F0_PER_THREAD;
// K12b: frames [ka, kb) of a row (zero: frames at or past nc, written as zeros)
struct F0Row { int64_t src_off, dst_off, len, nc, cap; };
struct F0Seg { int32_t row, ka, kb, zero; };
constexpr int F0F_THREADS = 256, F0F_FRAMES = 256;  // frames per segment: at most one per thread


// Ordered-int encoding so that atomicMax on int implements a signed float max.
__device__ __forceinline__ int float_to_ordered(float f) {
  int i = __float_as_int(f);
  return (i >= 0) ? i : (i ^ 0x7FFFFFFF);
}
__device__ __forceinline__ float ordered_to_float(int i) {
  return __int_as_float((i >= 0) ? i : (i ^ 0x7FFFFFFF));
}
#define ORDERED_NEG_INF ((int)0x80000000)
