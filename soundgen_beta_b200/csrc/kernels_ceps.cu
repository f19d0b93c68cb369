// K11 k_cepstra: cepstra c = M x of spectrogram frames and their deltas (sgb_rows_cepstra, include/soundgen_b200.h).
//
// Grid: a host-built table of tiles, each output frames [t0, t1) of one row: at most CEPS_TILE frames below
// min(nc, cap), then the frames from nc to cap as zero tiles of about 8192 floats that read nothing.  A compute
// tile stages in shared memory
//   M   n_ceps x n_in, stride ld = n_in | 1: odd, so the lanes of a warp read 32 different k (or frames) of one
//       column b from 32 different banks;
//   X   the input frames [lo, hi) = [t0 - H, t1 + H) clipped to [0, nc), H = delta_order * delta_n, stride ld (one
//       contiguous span of the row, loaded coalesced);
//   C   their cepstra, stride n_ceps;
//   D   (order 2) the deltas of the frames [t0 - N, t1 + N) clipped to [0, nc), N = delta_n,
// and reads frame p of a row as frame min(max(p, 0), nc - 1): the replicated edges of the delta formula, and no
// frame at or past nc.  Every output value is one fixed sequence of FP32 operations on its row's input (the dot
// product in b order from 0, the delta sums in k order), so a row's bits do not depend on cap, on the tiling or on
// the other rows.
//
// CEPS_TILE = 64: the halo re-read 2H / 64 is 12.5 % at the default order 2, N = 2 (25 % at N = 4), and the
// working set of the typical shapes stays inside the 226 KB a CTA may use: 29 KB for 64 bands, 13 coefficients,
// order 2, N = 2 (seven CTAs per SM), 183 KB for 256 inputs, 64 coefficients, order 2, N = 4 (one CTA per SM).
#include <cstdint>
#include <cuda_runtime.h>

#include "engine.cuh"

namespace {

constexpr int CEPS_THREADS = 256, CEPS_R = 4;      // CEPS_R frames per thread in the dot product: M read once per 4 FMAs

// (sum_{j=1..N} j (s[min(p + j, nc - 1)] - s[max(p - j, 0)])) / den for coefficient k; s holds frames from `base` on
__device__ __forceinline__ float delta_at(const float *s, int base, int p, int k, int stride, int nc, int dn, float den) {
  float a = 0.0f;
  for (int j = 1; j <= dn; j++) {
    const int u = min(p + j, nc - 1) - base, v = max(p - j, 0) - base;
    a = fmaf((float)j, s[u * stride + k] - s[v * stride + k], a);
  }
  return a / den;
}

}  // namespace

// outside the anonymous namespace: the profiler lists it as k_cepstra
__global__ void __launch_bounds__(CEPS_THREADS)
k_cepstra(const CepsTile *__restrict__ tiles, const CepsRow *__restrict__ rows, const float *__restrict__ mat,
          const float *__restrict__ src, float *__restrict__ dst, int n_in, int n_ceps, int order, int dn) {
  extern __shared__ float ceps_smem[];
  const CepsTile t = tiles[blockIdx.x];
  const CepsRow R = rows[t.row];
  const int n_out = n_ceps * (1 + order), n_y = (t.t1 - t.t0) * n_out;
  float *y = dst + R.dst_off + (int64_t)t.t0 * n_out;
  if (t.zero) {
    for (int i = threadIdx.x; i < n_y; i += CEPS_THREADS) y[i] = 0.0f;
    return;
  }
  const int ld = n_in | 1, H = order * dn, nc = R.nc, span = CEPS_TILE + 2 * H;
  const int lo = max(t.t0 - H, 0), nl = min(t.t1 + H, nc) - lo;
  const int dlo = max(t.t0 - dn, 0), nd = min(t.t1 + dn, nc) - dlo;
  float *sM = ceps_smem, *sX = sM + n_ceps * ld, *sC = sX + span * ld, *sD = sC + span * n_ceps;

  for (int i = threadIdx.x; i < n_ceps * n_in; i += CEPS_THREADS) sM[(i / n_in) * ld + i % n_in] = mat[i];
  const float *x = src + R.src_off + (int64_t)lo * n_in;
  const int n_x = nl * n_in;
  for (int i0 = 0; i0 < n_x; i0 += 8 * CEPS_THREADS) {      // 8 loads in flight per thread before the stores
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int i = i0 + k * CEPS_THREADS + threadIdx.x;
      v[k] = i < n_x ? __ldg(x + i) : 0.0f;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int i = i0 + k * CEPS_THREADS + threadIdx.x;
      if (i < n_x) sX[(i / n_in) * ld + i % n_in] = v[k];
    }
  }
  __syncthreads();

  // cepstra of the nl staged frames: thread item (frame group g, coefficient k), CEPS_R frames per group
  const int ng = (nl + CEPS_R - 1) / CEPS_R;
  for (int o = threadIdx.x; o < ng * n_ceps; o += CEPS_THREADS) {
    const int k = o % n_ceps, g = o / n_ceps;
    const float *m = sM + k * ld;
    const float *xr[CEPS_R];
    float acc[CEPS_R];
#pragma unroll
    for (int r = 0; r < CEPS_R; r++) {
      xr[r] = sX + min(g * CEPS_R + r, nl - 1) * ld;      // the last group repeats its last frame (not stored)
      acc[r] = 0.0f;
    }
    for (int b = 0; b < n_in; b++) {
      const float mb = m[b];
#pragma unroll
      for (int r = 0; r < CEPS_R; r++) acc[r] = fmaf(mb, xr[r][b], acc[r]);
    }
#pragma unroll
    for (int r = 0; r < CEPS_R; r++)
      if (g * CEPS_R + r < nl) sC[(g * CEPS_R + r) * n_ceps + k] = acc[r];
  }
  __syncthreads();

  int den = 0;
  for (int j = 1; j <= dn; j++) den += 2 * j * j;
  const float fden = (float)den;
  if (order == 2) {
    for (int o = threadIdx.x; o < nd * n_ceps; o += CEPS_THREADS) {
      const int f = o / n_ceps, k = o - f * n_ceps;
      sD[o] = delta_at(sC, lo, dlo + f, k, n_ceps, nc, dn, fden);
    }
    __syncthreads();
  }

  // [c | delta | delta-delta] of each frame, stored coalesced
  for (int i = threadIdx.x; i < n_y; i += CEPS_THREADS) {
    const int f = i / n_out, j = i - f * n_out, w = j / n_ceps, k = j - w * n_ceps, p = t.t0 + f;
    float v;
    if (w == 0)
      v = sC[(p - lo) * n_ceps + k];
    else if (w == 1)
      v = order == 1 ? delta_at(sC, lo, p, k, n_ceps, nc, dn, fden) : sD[(p - dlo) * n_ceps + k];
    else
      v = delta_at(sD, dlo, p, k, n_ceps, nc, dn, fden);
    y[i] = v;
  }
}

// Shared memory of a compute tile: M, X, C and (order 2) D at their largest.
size_t cepstra_smem_bytes(int n_in, int n_ceps, int order, int dn) {
  const size_t ld = (size_t)(n_in | 1), nk = (size_t)n_ceps, span = CEPS_TILE + 2 * (size_t)order * dn;
  return sizeof(float) * (nk * ld + span * ld + span * nk + (order == 2 ? (CEPS_TILE + 2 * (size_t)dn) * nk : 0));
}

cudaError_t launch_cepstra(const CepsTile *tiles, int n_tiles, const CepsRow *rows, const float *mat, const float *src,
                           float *dst, int n_in, int n_ceps, int order, int dn, cudaStream_t st) {
  if (n_tiles <= 0) return cudaSuccess;
  const size_t smem = cepstra_smem_bytes(n_in, n_ceps, order, dn);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k_cepstra, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  k_cepstra<<<(unsigned)n_tiles, CEPS_THREADS, smem, st>>>(tiles, rows, mat, src, dst, n_in, n_ceps, order, dn);
  return cudaGetLastError();
}
