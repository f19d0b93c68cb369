// K10 k_spec_compare: one similarity score per pair of spectrogram rows (sgb_rows_compare, include/soundgen_b200.h).
//
// One CTA per pair, CMP_THREADS threads whatever the launch: a pair's cells go to the same threads in the same order
// and its partial sums are reduced in the same fixed tree, so its score does not depend on the other pairs, their
// order or their number.  No atomics.
//   cor / cosine: FP64 sums over the N * n_feat cells (N = the longer row, missing frames read as `pad`); cor is
//                 two-pass (means first, then centred products), cosine one pass (a float product is exact in FP64).
//   DTW:          wavefront over the anti-diagonals of the (short side) x (long side) grid, three diagonals of FP64
//                 sums in shared memory indexed by the short side's frame; each cell's distance is computed on the
//                 fly in FP32 by one thread.  No cost matrix leaves the CTA.
#include <cstdint>
#include <cuda_runtime.h>

#include "engine.cuh"

namespace {

constexpr int CMP_THREADS = 256;

struct Pair {             // element offsets and frame counts of a_c and b_c
  int64_t a_off, a_frames, b_off, b_frames;
};

// Sums of CMP_THREADS threads in a fixed order: butterfly within each warp, then warp 0 adds the warps in order.
// Every thread gets the total.
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double *red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; k++)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
  __syncthreads();                       // `red` may still be read from an earlier call
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < K; k++) red[w * K + k] = v[k];
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; k++) {
    double s = 0.0;
    for (int i = 0; i < CMP_THREADS / 32; i++) s += red[i * K + k];
    v[k] = s;
  }
}

__device__ void corcos(const float *__restrict__ a, const float *__restrict__ b, const Pair &P, int n_feat, double pad,
                       int method, double *red, double *out) {
  const int64_t na = P.a_frames * n_feat, nb = P.b_frames * n_feat;
  const int64_t cells = (P.a_frames > P.b_frames ? P.a_frames : P.b_frames) * n_feat;
  const float *A = a + P.a_off, *B = b + P.b_off;
  double v[3] = {0.0, 0.0, 0.0};             // ab, aa, bb
  double ma = 0.0, mb = 0.0;
  bool constant = false;
  if (method == SGB_CMP_COR) {
    // means, and whether a side is constant (its variance is then exactly 0 and the score NaN): every thread
    // compares its cells with cell 0
    const double a0 = A[0], b0 = B[0];
    double m[4] = {0.0, 0.0, 0.0, 0.0};      // sum a, sum b, cells != a0, cells != b0
    for (int64_t i = threadIdx.x; i < cells; i += CMP_THREADS) {
      const double x = i < na ? (double)A[i] : pad, y = i < nb ? (double)B[i] : pad;
      m[0] += x; m[1] += y;
      m[2] += (double)(x != a0); m[3] += (double)(y != b0);
    }
    block_sum(m, red);
    ma = m[0] / (double)cells; mb = m[1] / (double)cells;
    constant = m[2] == 0.0 || m[3] == 0.0;
  }
  for (int64_t i = threadIdx.x; i < cells; i += CMP_THREADS) {
    const double x = (i < na ? (double)A[i] : pad) - ma, y = (i < nb ? (double)B[i] : pad) - mb;
    v[0] = fma(x, y, v[0]); v[1] = fma(x, x, v[1]); v[2] = fma(y, y, v[2]);
  }
  block_sum(v, red);
  if (threadIdx.x == 0) *out = constant ? __longlong_as_double(0x7ff8000000000000LL) : v[0] / (sqrt(v[1]) * sqrt(v[2]));
}

// symmetric2: D(0,0) = d(0,0); D(i,j) = min(D(i-1,j-1) + 2d, D(i-1,j) + d, D(i,j-1) + d); -D(n_a-1,n_b-1)/(n_a+n_b).
// The grid is walked as (s, l) over the short and the long row: d and the recurrence are symmetric in the two rows, so
// the result is the same bits as over (a, b).
__device__ void dtw(const float *__restrict__ a, const float *__restrict__ b, const Pair &P, int n_feat, double *diag,
                    double *out) {
  const bool a_short = P.a_frames <= P.b_frames;
  const float *S = a_short ? a + P.a_off : b + P.b_off, *L = a_short ? b + P.b_off : a + P.a_off;
  const int ns = (int)(a_short ? P.a_frames : P.b_frames), nl = (int)(a_short ? P.b_frames : P.a_frames);
  double *d0 = diag, *d1 = diag + ns, *d2 = diag + 2 * ns;   // diagonals k-2, k-1, k
  for (int k = 0; k <= ns + nl - 2; k++) {
    const int lo = k - (nl - 1) > 0 ? k - (nl - 1) : 0, hi = k < ns - 1 ? k : ns - 1;
    for (int i = lo + (int)threadIdx.x; i <= hi; i += CMP_THREADS) {
      const int j = k - i;
      const float *x = S + (int64_t)i * n_feat, *y = L + (int64_t)j * n_feat;
      float s = 0.0f;
      for (int f = 0; f < n_feat; f++) {
        const float t = x[f] - y[f];
        s = fmaf(t, t, s);
      }
      const double d = (double)sqrtf(s);
      double D;
      if (k == 0) {
        D = d;
      } else {
        D = INFINITY;
        if (i > 0 && j > 0) D = d0[i - 1] + 2.0 * d;
        if (i > 0) D = fmin(D, d1[i - 1] + d);
        if (j > 0) D = fmin(D, d1[i] + d);
      }
      d2[i] = D;
    }
    __syncthreads();
    double *t = d0; d0 = d1; d1 = d2; d2 = t;
  }
  if (threadIdx.x == 0) *out = -d1[ns - 1] / (double)(ns + nl);
}

}  // namespace

// outside the anonymous namespace: the profiler lists it as k_spec_compare
__global__ void __launch_bounds__(CMP_THREADS) k_spec_compare(const float *__restrict__ a, const float *__restrict__ b,
                                                              const int64_t *__restrict__ tab, int method, int n_feat,
                                                              double pad, double *__restrict__ dst) {
  extern __shared__ double cmp_smem[];
  const int64_t *t = tab + 4 * (size_t)blockIdx.x;       // the host's table: a_off, a_frames, b_off, b_frames
  const Pair P = {t[0], t[1], t[2], t[3]};
  if (P.a_frames == 0 || P.b_frames == 0) {
    if (threadIdx.x == 0) dst[blockIdx.x] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  if (method == SGB_CMP_DTW)
    dtw(a, b, P, n_feat, cmp_smem, dst + blockIdx.x);
  else
    corcos(a, b, P, n_feat, pad, method, cmp_smem, dst + blockIdx.x);
}

// Shared memory of a launch: the reduction scratch, or three diagonals of the longest short side for DTW.
size_t spec_compare_smem_bytes(int method, int64_t max_short) {
  const size_t red = sizeof(double) * 4 * (CMP_THREADS / 32);
  const size_t dg = method == SGB_CMP_DTW ? sizeof(double) * 3 * (size_t)max_short : 0;
  return dg > red ? dg : red;
}

cudaError_t launch_spec_compare(const float *a, const float *b, const void *pairs, int n, int method, int n_feat,
                                double pad, int64_t max_short, double *dst, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  const size_t smem = spec_compare_smem_bytes(method, max_short);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k_spec_compare, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  k_spec_compare<<<(unsigned)n, CMP_THREADS, smem, st>>>(a, b, reinterpret_cast<const int64_t *>(pairs), method, n_feat,
                                                         pad, dst);
  return cudaGetLastError();
}
