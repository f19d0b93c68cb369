// K12: the exact f0 contour of every generated call, per output sample (K12a, sgb_batch_f0) and per analysis frame
// (K12b, sgb_rows_f0_frames).
//
// K12a reads what a run leaves on the device: the spline of pitch_upsampled (Pools kt / ppg / sb / sc / sd, one
// cubic piece per glottal cycle, built by K0 and read by K1's phase), the epochs and the zero crossings K6 chose
// (SylCtrl), and the host's placement of syllables and bouts (as F0Span rows).  Nothing after K6 writes those
// arrays, so the track describes the handle's last run as long as the next run is queued behind it (same stream).
#include "engine.cuh"

// K6's composition (kernels_compose.cu, k_compose) replayed from the recorded crossings, one thread per syllable:
// epoch e starts at idx1_e in the composed syllable, and there its sample k sits at position k + koff_e with
// koff_e = idx1_e - zc2_e.  Stored as (idx1_e, gc_upsampled[ep_start_e - 1] - koff_e): the 1-based index of
// pitch_upsampled at composed position q >= idx1_e is that second value + q.
__global__ void __launch_bounds__(128)
k_f0_epochs(const sgb_syllable *__restrict__ syl, int S, const SylCtrl *__restrict__ ctrl, Pools P,
            F0Epochs *__restrict__ out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  F0Epochs &T = out[s];
  const SylCtrl &C = ctrl[s];
  if (syl[s].kind != 1 || C.status != SGB_OK) { T.nE = 0; T.G = 0; return; }
  const int32_t *gcup = P.gcup + P.gc_off[s];
  const int crossMax = (int)floor(15.0 * syl[s].samplingRate / 1000.0);
  int Lc = 1;                                          // `waveform = 0`
  for (int e = 0; e < C.nEpochs; e++) {
    const int u0 = gcup[C.ep_start[e] - 1];
    const int Ne = gcup[C.ep_end[e]] - u0 + 1;
    const int zc1 = C.ep_zc1[e], zc2 = C.ep_zc2[e];
    const int Lc1 = zc1 > 0 ? zc1 + 1 : Lc;            // ampl1 = c(ampl1[1:zc1], 0), or unchanged without a crossing
    const int L2 = Ne - zc2;
    const int cl = min(crossMax, min(Lc1 - 1, L2 - 1));
    const int idx1 = cl < 2 ? Lc1 : Lc1 - cl;
    T.ep[e] = make_int2(idx1, u0 - (idx1 - zc2));
    Lc = idx1 + L2;
  }
  T.nE = C.nEpochs;
  T.G = C.nGC;
}

// largest a in [0, G) with kt[a] <= u (kt[0] = 1 <= u): the piece R's spline_eval picks
__device__ __forceinline__ int f0_piece(const double *kt, int G, double u) {
  int a = 0, b = G;
  while (b > a + 1) {
    const int mid = (a + b) >> 1;
    if (u < kt[mid]) b = mid; else a = mid;
  }
  return a;
}

// K12a: every sample of every row, voiced spans and zeros.  Grid: host-built (row, chunk) pairs of F0_CHUNK samples,
// as the f32 export.  Thread j evaluates the 32 consecutive samples [32 j, 32 j + 32) of the chunk, so it finds its
// span, epoch and spline piece once and then mostly stays in them with the piece's coefficients in registers (a
// lookup per sample would be a chain of dependent loads); the values go through shared memory (row stride 33: no
// bank conflicts either way) and leave in coalesced stores.  The value is the FP64 spline of pitch_upsampled
// evaluated as R's spline_eval does (y + d (b + d (c + d e)), no contraction: -fmad=false), rounded to float once.
static_assert(F0_PER_THREAD == 32, "k_f0_track maps chunk position r to thread r >> 5, slot r & 31");
__global__ void __launch_bounds__(F0_THREADS)
k_f0_track(const F0Chunk *__restrict__ chunks, const int64_t *__restrict__ dst_off, const int64_t *__restrict__ cap,
           const F0Span *__restrict__ spans, const F0Epochs *__restrict__ ept, Pools P, float *__restrict__ dst) {
  __shared__ float buf[F0_THREADS * (F0_PER_THREAD + 1)];
  const F0Chunk ch = chunks[blockIdx.x];
  const int64_t c = cap[ch.row];
  const int64_t base = (int64_t)ch.chunk * F0_CHUNK;
  float *out = buf + threadIdx.x * (F0_PER_THREAD + 1);
  int sp = ch.s_lo, cur = -1;
  int64_t t0 = 0, t1 = 0;                              // [t0, t1): the span sp
  int nE = 0, G = 0, e = 0, a = -1;
  const int2 *ep = nullptr;
  const double *kt = nullptr, *py = nullptr, *sb = nullptr, *sc = nullptr, *sd = nullptr;
  double k_lo = 0.0, k_hi = 0.0, cy = 0.0, cb = 0.0, cc = 0.0, cd = 0.0;   // piece a: [k_lo, k_hi), coefficients
  if (sp < ch.s_hi) { t0 = spans[sp].t0; t1 = t0 + spans[sp].n; }
  for (int k = 0; k < F0_PER_THREAD; k++) {
    const int64_t i = base + (int64_t)threadIdx.x * F0_PER_THREAD + k;
    while (sp < ch.s_hi && t1 <= i) {
      if (++sp < ch.s_hi) { t0 = spans[sp].t0; t1 = t0 + spans[sp].n; }
    }
    float v = 0.0f;
    if (i < c && sp < ch.s_hi && i >= t0) {
      if (sp != cur) {
        cur = sp;
        const int s = spans[sp].syl;
        const F0Epochs *T = ept + s;
        nE = T->nE; G = T->G; ep = T->ep;
        const int64_t o = P.gc_off[s];
        kt = P.kt + o; py = P.ppg + o; sb = P.sb + o; sc = P.sc + o; sd = P.sd + o;
        e = 0; a = -1;
      }
      const int q = (int)(i - t0);
      while (e + 1 < nE && ep[e + 1].x <= q) e++;
      const int2 E = ep[e];
      const double u = (double)(E.y + max(q, E.x));   // before the first epoch: its first sample (the leading zeros)
      if (a < 0 || u < k_lo || u >= k_hi) {
        a = (a >= 0 && u >= k_hi && a + 2 < G && u < kt[a + 2]) ? a + 1 : f0_piece(kt, G, u);
        k_lo = kt[a]; k_hi = a + 1 < G ? kt[a + 1] : INFINITY;
        cy = py[a]; cb = sb[a]; cc = sc[a]; cd = sd[a];
      }
      const double M = u - k_lo;
      v = (float)(cy + M * (cb + M * (cc + M * cd)));
    }
    out[k] = v;
  }
  __syncthreads();
  float *y = dst + dst_off[ch.row];
#pragma unroll 4
  for (int r = threadIdx.x; r < F0_CHUNK; r += F0_THREADS) {
    const int64_t i = base + r;
    if (i < c) y[i] = buf[(r >> 5) * (F0_PER_THREAD + 1) + (r & 31)];
  }
}

cudaError_t launch_f0_track(const sgb_syllable *syl, int S, const SylCtrl *ctrl, const Pools &P, F0Epochs *ept,
                            const F0Chunk *chunks, int n_chunks, const int64_t *dst_off, const int64_t *cap,
                            const F0Span *spans, float *dst, cudaStream_t st) {
  if (S > 0) k_f0_epochs<<<(S + 127) / 128, 128, 0, st>>>(syl, S, ctrl, P, ept);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || n_chunks <= 0) return e;
  k_f0_track<<<n_chunks, F0_THREADS, 0, st>>>(chunks, dst_off, cap, spans, ept, P, dst);
  return cudaGetLastError();
}

// 0-based start of frame k: K9's frame_in_start (R's truncated 1 + k h), in 64 bits
__device__ __forceinline__ int64_t f0_frame_start(int k, double h) { return (int64_t)floor(1.0 + (double)k * h) - 1; }

// K12b: frame labels of float32 rows.  Frame k of a row of len samples covers [s_k, s_k + wl) ∩ [0, len) with
// s_k = f0_frame_start(k); its label is {x[s_k + wl/2] (0 at or past len), nonzero samples of the frame / wl}.
// A CTA takes a segment of at most F0F_FRAMES frames, one per thread, and sweeps the samples the segment covers
// once, F0F_TILE at a time: each warp ballots the nonzero flags of 256 consecutive samples (8 coalesced loads per
// lane), the CTA turns them into running counts, and a thread whose frame starts or ends inside the tile records
// the count there.  Every sample is read once per segment (plus the wl - h overlap between segments), not wl / h
// times.  Counts are exact integers, divided once.
constexpr int F0F_TILE = 8 * 256;
__global__ void __launch_bounds__(F0F_THREADS)
k_f0_frames(const F0Seg *__restrict__ segs, const F0Row *__restrict__ rows, const float *__restrict__ src, int wl,
            double h, float *__restrict__ dst) {
  __shared__ uint32_t msk[F0F_TILE / 32];
  __shared__ int wpre[F0F_TILE / 32], wtot[F0F_THREADS / 32];
  const F0Seg sg = segs[blockIdx.x];
  const F0Row R = rows[sg.row];
  float *out = dst + R.dst_off;
  if (sg.zero) {
    for (int64_t i = 2 * (int64_t)sg.ka + threadIdx.x; i < 2 * (int64_t)sg.kb; i += F0F_THREADS) out[i] = 0.0f;
    return;
  }
  const float *x = src + R.src_off;
  const int64_t len = R.len;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = sg.ka + (int)threadIdx.x;
  const bool mine = k < sg.kb;
  const int64_t s_k = mine ? f0_frame_start(k, h) : 0, e_k = mine ? min(s_k + wl, len) : 0;
  const int64_t A = f0_frame_start(sg.ka, h), B = min(f0_frame_start(sg.kb - 1, h) + wl, len);
  int64_t base = 0;
  int64_t cs = 0, ce = 0;                              // running counts at s_k and e_k
  for (int64_t lo = A; lo <= B; lo += F0F_TILE) {
    // warp w: samples [lo + 256 w, lo + 256 w + 256), ballot j of them [.. + 32 j, .. + 32 j + 32)
    int tot = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int64_t p = lo + 256 * warp + 32 * j + lane;
      const uint32_t m = __ballot_sync(0xffffffffu, p < B && x[p] != 0.0f);
      if (lane == 0) { msk[8 * warp + j] = m; wpre[8 * warp + j] = tot; }
      tot += __popc(m);
    }
    if (lane == 0) wtot[warp] = tot;
    __syncthreads();
    int64_t wbase[F0F_THREADS / 32];
    int64_t acc = base;
#pragma unroll
    for (int w = 0; w < F0F_THREADS / 32; w++) { wbase[w] = acc; acc += wtot[w]; }
    auto count_at = [&](int64_t pos) -> int64_t {          // nonzero samples in [A, pos), pos in [lo, lo + tile)
      const int d = (int)(pos - lo), w = d >> 8, j = (d >> 5) & 7, r = d & 31;
      int64_t wb = 0;
#pragma unroll
      for (int ww = 0; ww < F0F_THREADS / 32; ww++) if (ww == w) wb = wbase[ww];
      return wb + wpre[8 * w + j] + __popc(msk[8 * w + j] & ((1u << r) - 1u));
    };
    if (mine) {
      if (s_k >= lo && s_k < lo + F0F_TILE) cs = count_at(s_k);
      if (e_k >= lo && e_k < lo + F0F_TILE) ce = count_at(e_k);
    }
    base = acc;
    __syncthreads();
  }
  if (mine) {
    const int64_t ci = s_k + wl / 2;
    out[2 * (int64_t)k] = ci < len ? x[ci] : 0.0f;
    out[2 * (int64_t)k + 1] = (float)(ce - cs) / (float)wl;
  }
}

cudaError_t launch_f0_frames(const F0Seg *segs, int n_segs, const F0Row *rows, const float *src, int wl, double h,
                             float *dst, cudaStream_t st) {
  if (n_segs <= 0) return cudaSuccess;
  k_f0_frames<<<n_segs, F0F_THREADS, 0, st>>>(segs, rows, src, wl, h, dst);
  return cudaGetLastError();
}
