// Shared declarations for the soundgen B200 kernels.
//
// Functions marked SGB_HD are plain scalar code that runs in one device thread
// (or in a host test harness built from tests/hostsim, never in the product
// library's compute path).  They restate control-rate pieces of the reference
// (file:line cited at each) in IEEE double with the reference's operation order;
// the translation units that include them are compiled with -fmad=false so that
// integer artefacts (glottal-cycle boundaries, epoch tables) come out bit-exact.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define SGB_HD __host__ __device__ inline
#else
#define SGB_HD inline
#endif

#include "../../include/soundgen_b200.h"

#define SGB_MAX_EPOCHS 128     // sub-harmonic epochs per syllable

// Per-syllable results of the control-rate stage (K0), device resident.
struct SylCtrl {
  int32_t status;        // SGB_OK or error
  int32_t nGC;
  int32_t nHarmonics;    // nominal (source.R:329)
  int32_t rows_kept;     // rows of the rolloff matrix after pruning (sourceSpectrum.R:182)
  int32_t nEpochs;
  int32_t n_up;          // length(pitch_upsampled)
  int32_t n_jidx;
  int32_t z_used;
  int32_t parab_harm;    // rolloffParabHarm after rounding / 2 -> 3
  int32_t any_oct;       // sum(rolloffOct != 0) > 0
  int32_t vf_active;     // getVocalFry took the epoch path (max(nSubharm) >= 1)
  int32_t use_ampl;      // amplAnchors active
  int32_t out_len;       // length of the composed syllable (after cross-fades)
  int32_t tiles;         // K1 tiles
  int32_t tiles_tc;      // units of the tensor-core K1 (intervals of approx() over all epochs)
  int32_t pad_tc;
  int64_t amp_elems;     // doubles in the amplitude matrices
  int64_t wave_elems;    // floats of epoch waveform scratch
  double  parab_a, parab_b, parab_c;
  double  raw_max;       // signed max before normalisation (source.R:449)
  int32_t ep_start[SGB_MAX_EPOCHS];   // 1-based gc index
  int32_t ep_end[SGB_MAX_EPOCHS];
  int32_t ep_nsub[SGB_MAX_EPOCHS];
  int32_t ep_rows[SGB_MAX_EPOCHS];    // dense row count J_e (multiples of f0/(nsub+1))
  int32_t ep_zc1[SGB_MAX_EPOCHS];     // zero crossings found by crossFade, 0 = NA
  int32_t ep_zc2[SGB_MAX_EPOCHS];
  int64_t ep_amp_off[SGB_MAX_EPOCHS]; // offset of the epoch's matrix inside the syllable's block
  int64_t ep_wave_off[SGB_MAX_EPOCHS];
};

// Per-glottal-cycle arrays of one syllable (views into pooled device scratch).
struct SylArrays {
  double *pitch;       // [P] working copy (vibrato applied)
  int32_t *gc;         // [cap]
  double *ppg;         // [cap] pitch_per_gc (final)
  double *rw;          // [cap]
  double *ro, *roct, *rk;  // [cap] per-gc rolloff / rolloffOct / rolloffKHz passed to getRolloff
  double *shimmer;     // [cap] multiplicative factor (1 when off)
  double *drift;       // [cap] 2^(drift - mean) (1 when temperature == 0)
  double *subdep;      // [cap] sideband width per gc
  double *colmax;      // [cap] max over harmonics of r[, g]
  int32_t *nsub;       // [cap]
  int32_t *rwbin;      // [cap]
  int32_t *jidx;       // [cap]
  int32_t *gcup;       // [cap+1]
  double *kt;          // [cap] spline knots (sample index, 1-based)
  double *sb, *sc, *sd;    // [cap] FMM coefficients of pitch_upsampled
  double *phi;         // [cap] sum of pitch_upsampled before knot i
  double *t1, *t2, *t3, *t4;  // [cap] scratch
  int32_t *rowmap;     // [nHcap] kept row -> original harmonic number
  int32_t cap;
  int32_t hcap;
};
