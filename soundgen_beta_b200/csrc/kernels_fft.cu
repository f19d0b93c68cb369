// K2: fused STFT -> envelope multiply -> ISTFT overlap-add (R/soundgen.R:743-806 with
// seewave::stft / istft, seewave.r:7782-7818 and :3447-3487), and
// K5: noise spectrum -> ISTFT overlap-add (R/source.R:88-124).
//
// One CTA walks a run of consecutive frames of one sound.  Two real frames share one
// complex FFT (A + iB); the FFT is a hand-written shared-memory Stockham autosort with
// radix-4 / radix-2 register butterflies and a table-driven generic radix for the odd
// factors soundgen's window sizes need (3, 5, 19, 29, or any prime after the clamp at
// soundgen.R:743).  Frame inputs are staged by TMA bulk copies (cp.async.bulk +
// mbarrier) into a double buffer while the previous pair is transformed; the weighted
// overlap-add lives in a shared-memory ring and every output sample is written once.
//
// Round 2: the tuned window sizes run REGISTER-RESIDENT passes -- radix 16 / 15 / 10 / 8 butterflies
// generated as straight-line code (fft_radix_gen.cuh), e.g. 2400 = 16 * 15 * 10 -- and the last forward
// pass, the spectrum split / envelope multiply / Hermitian rebuild and the first inverse pass are ONE
// pass: the thread that holds the outputs q + S j of forward butterfly q (and of its mirror S - q) holds
// exactly the inputs of inverse butterflies q and S - q.  A frame pair costs 5 shared-memory passes
// (4 for noise) instead of 12.  Prime radices (19, 29: 22.05 / 44.1 kHz) pair k with r - k and produce
// outputs j and r - j together (half the loads and multiplies of a plain DFT).
#include "engine.cuh"
#include <cstdio>
#include "fft_radix_gen.cuh"

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ int g_stft_timeout = 0;   // set when a staged frame load never completed (checked by the host)
int stft_timeout_flag() { int v = 0; cudaMemcpyFromSymbol(&v, g_stft_timeout, sizeof v); return v; }
__device__ __forceinline__ bool mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok = 0;
  unsigned long long polls = 0;
  while (!ok) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
                 " selp.b32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    if (!ok && ++polls > (1ull << 26)) {   // seconds: a staged load that never lands must fail loudly, not hang
      g_stft_timeout = 1;
      return false;
    }
  }
  return true;
}

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }

// Input of the first forward pass: two real frames read straight from the TMA staging buffer, multiplied by
// the analysis window and packed as A + iB (no separate windowing pass).
struct WinIn {
  const float *a, *b, *w;
  int off;
  bool hasB;
  __device__ __forceinline__ WinIn operator+(int o) const { WinIn r = *this; r.off += o; return r; }
  __device__ __forceinline__ float2 operator[](int i) const {
    const int k = off + i;
    const float wv = w[k];
    return make_float2(a[k] * wv, hasB ? b[k] * wv : 0.0f);
  }
};
// Input of the first inverse pass of the noise generator: the real, zero-phase spectrum u * rolloff * filter
// of two frames (R/source.R:103-114), Hermitian-extended with Nyquist := last kept bin (seewave.r:3470-3474),
// generated on the fly from the uniforms in global memory.
template <typename UT>
struct NoiseIn {
  const UT *uA, *uB;
  const float *ro, *fA, *fB;
  int off, N, nr;
  bool hasB;
  __device__ __forceinline__ NoiseIn operator+(int o) const { NoiseIn r = *this; r.off += o; return r; }
  __device__ __forceinline__ float2 operator[](int i) const {
    int kk = off + i;
    if (kk > nr) kk = N - kk;
    if (kk == nr) kk = nr - 1;
    const float r0 = ro[kk];
    const float va = (float)uA[kk] * r0 * (fA ? fA[kk] : 1.0f);
    const float vb = hasB ? (float)uB[kk] * r0 * (fB ? fB[kk] : 1.0f) : 0.0f;
    return make_float2(va, vb);
  }
};
// Output of the last inverse pass: weighted overlap-add straight into the rings (frame A of a pair into
// ring A, frame B into ring B, so no two threads of a pass touch the same slot).
struct OlaOut {
  float *ra, *rb;
  const float *ws;
  int oA, oB, ring;
  bool hasB;
  __device__ __forceinline__ void add(int o, float2 v) const {
    const float wv = ws[o];
    int sa = oA + o;
    if (sa >= ring) sa -= ring;
    ra[sa] += v.x * wv;
    if (hasB) {
      int sb = oB + o;
      if (sb >= ring) sb -= ring;
      rb[sb] += v.y * wv;
    }
  }
};

// Odd (prime) radix r: X_j = x_0 + sum_{k=1..(r-1)/2} [(x_k + x_{r-k}) cos(2 pi jk / r) -/+ i (x_k - x_{r-k}) sin(2 pi jk / r)],
// so one work item produces outputs j and r - j from (r-1)/2 complex sums and differences.
template <int DIR, class XIn, bool LAST>
__device__ __forceinline__ void pass_prime(XIn x, float2 *__restrict__ y, int N, int s, int r,
                                           const float2 *__restrict__ tw, const OlaOut &O) {
  auto put = [&](int o, float2 v) { if (LAST) O.add(o, v); else y[o] = v; };
  const int nb = N / r, m = nb / s, half = (r - 1) >> 1, wstep = N / r;
  const int items = (half + 1) * nb;
  for (int idx = threadIdx.x; idx < items; idx += (int)blockDim.x) {
    const int jj = idx / nb, b = idx - jj * nb;
    const int p = b / s, q = b - p * s;
    const XIn xi = x + (q + s * p);
    const int sm = s * m;
    const float2 a0 = xi[0];
    const int yo = q + s * r * p;
    if (jj == 0) {
      float2 acc = a0;
      for (int k = 1; k < r; k++) { const float2 a = xi[k * sm]; acc.x += a.x; acc.y += a.y; }
      put(yo, acc);
      continue;
    }
    float2 P = a0, Q = make_float2(0.0f, 0.0f);
    int t = 0;
    const int st = jj * wstep;
    for (int k = 1; k <= half; k++) {
      t += st;
      if (t >= N) t -= N;
      const float2 w = tw[t];                 // (cos, -sin) of 2 pi jj k / r
      const float2 a = xi[k * sm], c = xi[(r - k) * sm];
      P.x = fmaf(a.x + c.x, w.x, P.x); P.y = fmaf(a.y + c.y, w.x, P.y);
      Q.x = fmaf(a.x - c.x, -w.y, Q.x); Q.y = fmaf(a.y - c.y, -w.y, Q.y);
    }
    // forward: X_j = P - i Q, X_{r-j} = P + i Q; inverse: the other way round
    const float2 lo = make_float2(P.x + Q.y, P.y - Q.x), hi = make_float2(P.x - Q.y, P.y + Q.x);
    const float2 Xj = (DIR < 0) ? lo : hi, Xr = (DIR < 0) ? hi : lo;
    const int t1 = p * s * jj, t2 = p * s * (r - jj);      // p s < N / r, so both stay below N
    float2 w1 = tw[t1], w2 = tw[t2];
    if (DIR > 0) { w1.y = -w1.y; w2.y = -w2.y; }
    put(yo + jj * s, cmul(Xj, w1));
    put(yo + (r - jj) * s, cmul(Xr, w2));
  }
}

template <int R> __device__ __forceinline__ void dft_r(float2 *a) {
  if constexpr (R == 2) dft2(a);
  else if constexpr (R == 3) dft3(a);
  else if constexpr (R == 4) dft4(a);
  else if constexpr (R == 5) dft5(a);
  else if constexpr (R == 8) dft8(a);
  else if constexpr (R == 10) dft10(a);
  else if constexpr (R == 15) dft15(a);
  else dft16(a);
}
// inverse DFT = swap(re, im) . forward DFT . swap(re, im): the swaps are register renames
template <int DIR, int R> __device__ __forceinline__ void bfly(float2 *a) {
  if constexpr (DIR > 0) {
#pragma unroll
    for (int k = 0; k < R; k++) a[k] = make_float2(a[k].y, a[k].x);
  }
  dft_r<R>(a);
  if constexpr (DIR > 0) {
#pragma unroll
    for (int k = 0; k < R; k++) a[k] = make_float2(a[k].y, a[k].x);
  }
}
__host__ __device__ constexpr bool reg_radix(int r) { return r == 2 || r == 3 || r == 4 || r == 5 || r == 8 || r == 10 || r == 15 || r == 16; }

// Register-resident Stockham pass with everything known at compile time.
template <int DIR, int N, int S, int R, class XIn, bool LAST>
__device__ __forceinline__ void pass_ct(XIn x, float2 *__restrict__ y, const float2 *__restrict__ tw, const OlaOut &O) {
  if constexpr (!reg_radix(R)) {
    pass_prime<DIR, XIn, LAST>(x, y, N, S, R, tw, O);
  } else {
    constexpr int nb = N / R, m = nb / S, sm = S * m;
    for (int b = threadIdx.x; b < nb; b += (int)blockDim.x) {
      const int p = b / S, q = b - p * S;
      const XIn xi = x + (q + S * p);
      float2 a[R];
#pragma unroll
      for (int k = 0; k < R; k++) a[k] = xi[k * sm];
      bfly<DIR, R>(a);
      const int yo = q + S * R * p, ti = p * S;
      if (LAST) O.add(yo, a[0]); else y[yo] = a[0];
#pragma unroll
      for (int j = 1; j < R; j++) {
        float2 w = tw[j * ti];
        if (DIR > 0) w.y = -w.y;
        const float2 v = cmul(a[j], w);
        if (LAST) O.add(yo + j * S, v); else y[yo + j * S] = v;
      }
    }
  }
}

// Bin kk of each of the two real frames packed as Z = A + iB: zk = Z[kk], zm = Z[(N - kk) mod N].
__device__ __forceinline__ void pair_split(float2 zk, float2 zm, float2 *XA, float2 *XB) {
  *XA = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));      // (zk + conj(zm)) / 2
  *XB = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));     // (zk - conj(zm)) / (2i)
}

// Spectrum of one bin pair of the two packed frames (seewave.r:7806, soundgen.R:790-795, seewave.r:3470-3474):
// zk = Z[kk], zm = Z[N - kk], 0 < kk < N/2.  Returns the packed filtered pair for the inverse transform.
__device__ __forceinline__ void spec_pair(float2 zk, float2 zm, float ea, float eb, float2 *outk, float2 *outm,
                                          float *nyqA, float *nyqB) {
  float2 XA, XB;
  pair_split(zk, zm, &XA, &XB);
  const float2 FA = make_float2(ea * XA.x, ea * XA.y), FB = make_float2(eb * XB.x, eb * XB.y);
  *outk = make_float2(FA.x - FB.y, FA.y + FB.x);            // FA + i FB
  *outm = make_float2(FA.x + FB.y, FB.x - FA.y);            // conj(FA) + i conj(FB)
  *nyqA = FA.x; *nyqB = FB.x;
}

// Last forward pass (radix R, stride S = N / R) + spectrum + first inverse pass (radix R, stride 1) in registers.
template <int N, int R>
__device__ __forceinline__ void fused_mid(const float2 *__restrict__ x, float2 *__restrict__ y,
                                          const float2 *__restrict__ tw, const float *__restrict__ eA,
                                          const float *__restrict__ eB) {
  constexpr int S = N / R, nr = N / 2;
  static_assert(R % 2 == 0, "the middle radix must be even (the Nyquist bin belongs to butterfly 0)");
  for (int t = threadIdx.x; t <= S / 2; t += (int)blockDim.x) {
    const int q1 = t, q2 = (t == 0) ? 0 : S - t;
    const bool self = (q2 == q1);            // butterflies 0 and S/2 mirror onto themselves
    float2 a1[R], a2[R];
#pragma unroll
    for (int k = 0; k < R; k++) { a1[k] = x[q1 + S * k]; a2[k] = self ? a1[k] : x[q2 + S * k]; }
    dft_r<R>(a1);
    if (!self) dft_r<R>(a2);
    float na, nb;
    if (t == 0) {
      // indices S j: DC (j = 0), pairs (j, R - j), Nyquist slot at j = R / 2
      a1[0] = make_float2(eA[0] * a1[0].x, eB[0] * a1[0].y);
#pragma unroll
      for (int j = 1; j < R / 2; j++) spec_pair(a1[j], a1[R - j], eA[S * j], eB[S * j], &a1[j], &a1[R - j], &na, &nb);
      // Nyquist := Re(last kept bin nr - 1): that bin and its mirror live in other threads' registers, so
      // their two forward outputs are recomputed here (2 R multiply-adds)
      constexpr int qa = (nr - 1) % S, ja = (nr - 1) / S, qb = (nr + 1) % S, jb = (nr + 1) / S;
      float2 zk = make_float2(0.f, 0.f), zm = make_float2(0.f, 0.f);
#pragma unroll
      for (int k = 0; k < R; k++) {
        const float2 wa = tw[((ja * k) % R) * S], wb = tw[((jb * k) % R) * S];
        zk = cadd(zk, cmul(x[qa + S * k], wa));
        zm = cadd(zm, cmul(x[qb + S * k], wb));
      }
      float2 d0, d1;
      spec_pair(zk, zm, eA[nr - 1], eB[nr - 1], &d0, &d1, &na, &nb);
      a1[R / 2] = make_float2(na, nb);
    } else if (self) {
      // q = S / 2: index S/2 + S j mirrors onto S/2 + S (R - 1 - j)
#pragma unroll
      for (int j = 0; j < R / 2; j++) spec_pair(a1[j], a1[R - 1 - j], eA[q1 + S * j], eB[q1 + S * j], &a1[j], &a1[R - 1 - j], &na, &nb);
    } else {
      // index q1 + S j (butterfly q1) mirrors onto q2 + S (R - 1 - j) (butterfly q2); kk = the smaller index
#pragma unroll
      for (int j = 0; j < R; j++) {
        const int i1 = q1 + S * j;
        if (i1 < nr) spec_pair(a1[j], a2[R - 1 - j], eA[i1], eB[i1], &a1[j], &a2[R - 1 - j], &na, &nb);
        else spec_pair(a2[R - 1 - j], a1[j], eA[N - i1], eB[N - i1], &a2[R - 1 - j], &a1[j], &na, &nb);
      }
    }
    // first inverse pass: butterfly p = q reads x'[q + S k], writes y[R p + j] * conj(tw[j p])
    bfly<+1, R>(a1);
    y[R * q1] = a1[0];
#pragma unroll
    for (int j = 1; j < R; j++) { float2 w = tw[j * q1]; w.y = -w.y; y[R * q1 + j] = cmul(a1[j], w); }
    if (!self) {
      bfly<+1, R>(a2);
      y[R * q2] = a2[0];
#pragma unroll
      for (int j = 1; j < R; j++) { float2 w = tw[j * q2]; w.y = -w.y; y[R * q2 + j] = cmul(a2[j], w); }
    }
  }
}

// One Stockham pass (decimation in frequency): N points, stride s (product of the
// radices already done), radix r.  DIR = -1 forward, +1 inverse (conjugated twiddles).
// XIn: plain pointer or WinIn; LAST: the outputs go to the overlap-add rings instead of y.
template <int DIR, class XIn, bool LAST>
__device__ __forceinline__ void fft_pass(XIn x, float2 *__restrict__ y, int N, int s, int r,
                                         const float2 *__restrict__ tw, const OlaOut &O) {
  auto put = [&](int o, float2 v) { if (LAST) O.add(o, v); else y[o] = v; };
  const int nb = N / r;             // butterflies
  const int m = nb / s;             // N / (s * r)
  if (r == 4) {
    for (int b = threadIdx.x; b < nb; b += (int)blockDim.x) {
      int p = b / s, q = b - p * s;
      const XIn xi = x + (q + s * p);
      float2 a0 = xi[0], a1 = xi[s * m], a2 = xi[2 * s * m], a3 = xi[3 * s * m];
      float2 t0 = make_float2(a0.x + a2.x, a0.y + a2.y), t1 = make_float2(a0.x - a2.x, a0.y - a2.y);
      float2 t2 = make_float2(a1.x + a3.x, a1.y + a3.y), t3 = make_float2(a1.x - a3.x, a1.y - a3.y);
      // forward: b1 = t1 - i t3, b3 = t1 + i t3 ; inverse swaps them
      float2 mi = (DIR < 0) ? make_float2(t3.y, -t3.x) : make_float2(-t3.y, t3.x);   // (-i or +i) * t3
      float2 b0 = make_float2(t0.x + t2.x, t0.y + t2.y);
      float2 b2 = make_float2(t0.x - t2.x, t0.y - t2.y);
      float2 b1 = make_float2(t1.x + mi.x, t1.y + mi.y);
      float2 b3 = make_float2(t1.x - mi.x, t1.y - mi.y);
      const int yo = q + s * 4 * p;
      int ti = p * s;
      float2 w1 = tw[ti], w2 = tw[2 * ti], w3 = tw[3 * ti];
      if (DIR > 0) { w1.y = -w1.y; w2.y = -w2.y; w3.y = -w3.y; }
      put(yo, b0); put(yo + s, cmul(b1, w1)); put(yo + 2 * s, cmul(b2, w2)); put(yo + 3 * s, cmul(b3, w3));
    }
  } else if (r == 3) {
    const float c3 = 0.86602540378443864676f;   // sin(2 pi / 3)
    for (int b = threadIdx.x; b < nb; b += (int)blockDim.x) {
      int p = b / s, q = b - p * s;
      const XIn xi = x + (q + s * p);
      const int sm = s * m;
      float2 a0 = xi[0], a1 = xi[sm], a2 = xi[2 * sm];
      float2 t = make_float2(a1.x + a2.x, a1.y + a2.y), u = make_float2(a1.x - a2.x, a1.y - a2.y);
      float2 mm = make_float2(fmaf(-0.5f, t.x, a0.x), fmaf(-0.5f, t.y, a0.y));
      // forward: -i * c3 * u ; inverse: +i * c3 * u
      float2 v = (DIR < 0) ? make_float2(c3 * u.y, -c3 * u.x) : make_float2(-c3 * u.y, c3 * u.x);
      const int yo = q + s * 3 * p;
      int ti = p * s;
      float2 w1 = tw[ti], w2 = tw[2 * ti];
      if (DIR > 0) { w1.y = -w1.y; w2.y = -w2.y; }
      put(yo, make_float2(a0.x + t.x, a0.y + t.y));
      put(yo + s, cmul(make_float2(mm.x + v.x, mm.y + v.y), w1));
      put(yo + 2 * s, cmul(make_float2(mm.x - v.x, mm.y - v.y), w2));
    }
  } else if (r == 5) {
    const float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;
    const float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;
    for (int b = threadIdx.x; b < nb; b += (int)blockDim.x) {
      int p = b / s, q = b - p * s;
      const XIn xi = x + (q + s * p);
      const int sm = s * m;
      float2 a0 = xi[0], a1 = xi[sm], a2 = xi[2 * sm], a3 = xi[3 * sm], a4 = xi[4 * sm];
      float2 t1 = make_float2(a1.x + a4.x, a1.y + a4.y), t2 = make_float2(a2.x + a3.x, a2.y + a3.y);
      float2 t3 = make_float2(a1.x - a4.x, a1.y - a4.y), t4 = make_float2(a2.x - a3.x, a2.y - a3.y);
      float2 m1 = make_float2(fmaf(c1, t1.x, fmaf(c2, t2.x, a0.x)), fmaf(c1, t1.y, fmaf(c2, t2.y, a0.y)));
      float2 m2 = make_float2(fmaf(c2, t1.x, fmaf(c1, t2.x, a0.x)), fmaf(c2, t1.y, fmaf(c1, t2.y, a0.y)));
      float2 n1 = make_float2(fmaf(s1, t3.x, s2 * t4.x), fmaf(s1, t3.y, s2 * t4.y));
      float2 n2 = make_float2(fmaf(s2, t3.x, -s1 * t4.x), fmaf(s2, t3.y, -s1 * t4.y));
      // forward: b1 = m1 - i n1, b4 = m1 + i n1, b2 = m2 - i n2, b3 = m2 + i n2 (inverse: conjugate)
      float2 i1 = (DIR < 0) ? make_float2(n1.y, -n1.x) : make_float2(-n1.y, n1.x);
      float2 i2 = (DIR < 0) ? make_float2(n2.y, -n2.x) : make_float2(-n2.y, n2.x);
      const int yo = q + s * 5 * p;
      int ti = p * s;
      float2 w1 = tw[ti], w2 = tw[2 * ti], w3 = tw[3 * ti], w4 = tw[4 * ti];
      if (DIR > 0) { w1.y = -w1.y; w2.y = -w2.y; w3.y = -w3.y; w4.y = -w4.y; }
      put(yo, make_float2(a0.x + t1.x + t2.x, a0.y + t1.y + t2.y));
      put(yo + s, cmul(make_float2(m1.x + i1.x, m1.y + i1.y), w1));
      put(yo + 2 * s, cmul(make_float2(m2.x + i2.x, m2.y + i2.y), w2));
      put(yo + 3 * s, cmul(make_float2(m2.x - i2.x, m2.y - i2.y), w3));
      put(yo + 4 * s, cmul(make_float2(m1.x - i1.x, m1.y - i1.y), w4));
    }
  } else if (r == 8) {
    const float h = 0.70710678118654752440f;
    for (int b = threadIdx.x; b < nb; b += (int)blockDim.x) {
      int p = b / s, q = b - p * s;
      const XIn xi = x + (q + s * p);
      const int sm = s * m;
      float2 a[8];
#pragma unroll
      for (int k = 0; k < 8; k++) a[k] = xi[k * sm];
      // radix-2 stage: u_k = a_k + a_{k+4}; v_k = (a_k - a_{k+4}) w8^k  (w8 = e^{DIR i pi/4})
      float2 u[4], v[4];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        u[k] = make_float2(a[k].x + a[k + 4].x, a[k].y + a[k + 4].y);
        v[k] = make_float2(a[k].x - a[k + 4].x, a[k].y - a[k + 4].y);
      }
      // forward w8^1 = (1 - i) h, w8^2 = -i, w8^3 = (-1 - i) h; inverse: conjugates
      if (DIR < 0) {
        v[1] = make_float2(h * (v[1].x + v[1].y), h * (v[1].y - v[1].x));
        v[2] = make_float2(v[2].y, -v[2].x);
        v[3] = make_float2(h * (v[3].y - v[3].x), -h * (v[3].x + v[3].y));
      } else {
        v[1] = make_float2(h * (v[1].x - v[1].y), h * (v[1].x + v[1].y));
        v[2] = make_float2(-v[2].y, v[2].x);
        v[3] = make_float2(-h * (v[3].x + v[3].y), h * (v[3].x - v[3].y));
      }
      // two radix-4 butterflies: even outputs from u, odd outputs from v
      float2 X[8];
#pragma unroll
      for (int par = 0; par < 2; par++) {
        const float2 *c = par ? v : u;
        float2 t0 = make_float2(c[0].x + c[2].x, c[0].y + c[2].y), t1 = make_float2(c[0].x - c[2].x, c[0].y - c[2].y);
        float2 t2 = make_float2(c[1].x + c[3].x, c[1].y + c[3].y), t3 = make_float2(c[1].x - c[3].x, c[1].y - c[3].y);
        float2 mi = (DIR < 0) ? make_float2(t3.y, -t3.x) : make_float2(-t3.y, t3.x);
        X[par] = make_float2(t0.x + t2.x, t0.y + t2.y);
        X[4 + par] = make_float2(t0.x - t2.x, t0.y - t2.y);
        X[2 + par] = make_float2(t1.x + mi.x, t1.y + mi.y);
        X[6 + par] = make_float2(t1.x - mi.x, t1.y - mi.y);
      }
      const int yo = q + s * 8 * p;
      const int ti = p * s;
      put(yo, X[0]);
#pragma unroll
      for (int j = 1; j < 8; j++) {
        float2 w = tw[j * ti];
        if (DIR > 0) w.y = -w.y;
        put(yo + j * s, cmul(X[j], w));
      }
    }
  } else if (r == 2) {
    for (int b = threadIdx.x; b < nb; b += (int)blockDim.x) {
      int p = b / s, q = b - p * s;
      float2 a0 = x[q + s * p], a1 = x[q + s * (p + m)];
      float2 w1 = tw[p * s];
      if (DIR > 0) w1.y = -w1.y;
      put(q + s * 2 * p, make_float2(a0.x + a1.x, a0.y + a1.y));
      put(q + s * (2 * p + 1), cmul(make_float2(a0.x - a1.x, a0.y - a1.y), w1));
    }
  } else {
    pass_prime<DIR, XIn, LAST>(x, y, N, s, r, tw, O);
  }
}

// full transform; returns the buffer holding the result.  FIN: the first pass reads the windowed staging
// buffer (W); FOUT: the last pass adds into the overlap-add rings (O) and nothing is written to the buffer.
template <int DIR, bool FIN, bool FOUT>
__device__ float2 *fft_run(float2 *a, float2 *b, const FftPlan &pl, const float2 *tw, const WinIn &W, const OlaOut &O) {
  int s = 1;
  float2 *src = a, *dst = b;
  for (int i = 0; i < pl.npass; i++) {
    const int r = pl.radix[i];
    const bool first = FIN && i == 0, last = FOUT && i == pl.npass - 1;
    if (first && last) fft_pass<DIR, WinIn, true>(W, dst, pl.n, s, r, tw, O);
    else if (first) fft_pass<DIR, WinIn, false>(W, dst, pl.n, s, r, tw, O);
    else if (last) fft_pass<DIR, const float2 *, true>(src, dst, pl.n, s, r, tw, O);
    else fft_pass<DIR, const float2 *, false>(src, dst, pl.n, s, r, tw, O);
    __syncthreads();
    s *= r;
    float2 *t = src; src = dst; dst = t;
  }
  return src;
}

// Compile-time plans for soundgen's usual windows (50 ms at 16 / 22.05 / 24 / 44.1 / 48 kHz and the 10 ms
// presets): forward radices F1, F2, MID; inverse radices MID, F2, F1.  SPEC 0 = run-time plan (any even length).
template <int SPEC> struct CtPlan;
template <> struct CtPlan<1> { static constexpr int N = 800, F1 = 16, F2 = 5, MID = 10; };
template <> struct CtPlan<2> { static constexpr int N = 1102, F1 = 29, F2 = 19, MID = 2; };
template <> struct CtPlan<3> { static constexpr int N = 1200, F1 = 8, F2 = 15, MID = 10; };
template <> struct CtPlan<4> { static constexpr int N = 2204, F1 = 29, F2 = 19, MID = 4; };
template <> struct CtPlan<5> { static constexpr int N = 2400, F1 = 16, F2 = 15, MID = 10; };
template <> struct CtPlan<6> { static constexpr int N = 160, F1 = 16, F2 = 1, MID = 10; };

// K2, tuned sizes: windowed frames (W) -> filtered, synthesis-windowed frames added into the rings (O).
// bufA / bufB: two N-point work buffers.
template <int SPEC>
__device__ __forceinline__ void filter_pair_ct(float2 *bufA, float2 *bufB, const float2 *tw, const WinIn &W,
                                               const OlaOut &O, const float *eA, const float *eB) {
  using P = CtPlan<SPEC>;
  constexpr int N = P::N, F1 = P::F1, F2 = P::F2, MID = P::MID;
  OlaOut O0 = {};
  if constexpr (reg_radix(F1)) {
    pass_ct<-1, N, 1, F1, WinIn, false>(W, bufB, tw, O0);           // window + A + iB packing fused in
  } else {
    // a prime first radix reads every input (r + 1) / 2 times: window the frames once, in a pass of its own
    for (int i = threadIdx.x; i < N; i += (int)blockDim.x) bufA[i] = W[i];
    __syncthreads();
    pass_ct<-1, N, 1, F1, const float2 *, false>(bufA, bufB, tw, O0);
  }
  __syncthreads();
  float2 *src = bufB, *dst = bufA;
  if constexpr (F2 > 1) {
    pass_ct<-1, N, F1, F2, const float2 *, false>(bufB, bufA, tw, O0);
    __syncthreads();
    src = bufA; dst = bufB;
  }
  fused_mid<N, MID>(src, dst, tw, eA, eB);
  __syncthreads();
  if constexpr (F2 > 1) {
    pass_ct<+1, N, MID, F2, const float2 *, false>(dst, src, tw, O0);
    __syncthreads();
    pass_ct<+1, N, MID * F2, F1, const float2 *, true>(src, dst, tw, O);
  } else {
    pass_ct<+1, N, MID, F1, const float2 *, true>(dst, src, tw, O);
  }
  __syncthreads();
}

// K5, tuned sizes: the real zero-phase spectrum is generated on the fly by the first inverse pass.
template <int SPEC, class NIn>
__device__ __forceinline__ void noise_pair_ct(float2 *bufA, float2 *bufB, const float2 *tw, const NIn &X, const OlaOut &O) {
  using P = CtPlan<SPEC>;
  constexpr int N = P::N, F1 = P::F1, F2 = P::F2, MID = P::MID;
  OlaOut O0 = {};
  pass_ct<+1, N, 1, MID, NIn, false>(X, bufA, tw, O0);
  __syncthreads();
  if constexpr (F2 > 1) {
    pass_ct<+1, N, MID, F2, const float2 *, false>(bufA, bufB, tw, O0);
    __syncthreads();
    pass_ct<+1, N, MID * F2, F1, const float2 *, true>(bufB, bufA, tw, O);
  } else {
    pass_ct<+1, N, MID, F1, const float2 *, true>(bufA, bufB, tw, O);
  }
  __syncthreads();
}

__device__ __forceinline__ int frame_in_start(const FftPlan &pl, int k) {   // 0-based
  return (int)floor(1.0 + (double)k * pl.h_in) - 1;
}
__device__ __forceinline__ int frame_out_start(const FftPlan &pl, int k) {
  return (int)floor((double)k * pl.h_out + 1.0) - 1;
}

// MODE 0: filter (K2).  MODE 1: noise (K5), UT = uniform dtype.
template <int MODE, typename UT, int SPEC>
__global__ void __launch_bounds__(256, 4)
k_stft(const FftSeg *__restrict__ segs, const FftJob *__restrict__ jobs, const FftPlan *__restrict__ plans,
       const float2 *__restrict__ twpool, const float *__restrict__ winpool,
       const float *__restrict__ in_f, const UT *__restrict__ in_u, const float *__restrict__ envpool,
       float *__restrict__ outpool, int *__restrict__ maxpool) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t bars[2];
  __shared__ float red[FFT_THREADS / 32];

  const FftSeg sg = segs[blockIdx.x];
  const FftJob jb = jobs[sg.job];
  const FftPlan pl = plans[jb.plan];
  const int N = pl.n, nr = N / 2;
  const int hceil = (int)ceil(pl.h_out) + 2;
  const int ring = N + 2 * hceil + 4;
  const int stage_len = (N + (int)ceil(pl.h_in) + 12) & ~3;     // floats per staging buffer

  float2 *bufA = reinterpret_cast<float2 *>(smem_raw);
  float2 *bufB = bufA + N;
  float2 *tw = bufB + N;
  float *ola = reinterpret_cast<float *>(tw + N);      // ring A: even frames of the pairs
  float *olb = ola + ((ring + 3) & ~3);                // ring B: odd frames
  float *stage0 = olb + ((ring + 3) & ~3);
  float *stage1 = stage0 + stage_len;
  float *vec = stage1 + ((MODE == 0) ? stage_len : 0);           // noise: rolloff vector [nr]

  const float2 *twg = twpool + pl.tw_off;
  const float *wa = winpool + pl.wa_off;
  const float *ws = winpool + pl.ws_off;
  for (int i = threadIdx.x; i < N; i += (int)blockDim.x) tw[i] = twg[i];
  for (int i = threadIdx.x; i < ring; i += (int)blockDim.x) { ola[i] = 0.0f; olb[i] = 0.0f; }
  if (MODE == 1) {
    // rolloff vector 2^(rolloffNoise/10 * log2(1:nr)) (source.R:103-105)
    for (int i = threadIdx.x; i < nr; i += (int)blockDim.x)
      vec[i] = (float)exp2(jb.rolloffNoise / 10.0 * log2((double)(i + 1)));
  }
  if (MODE == 0 && threadIdx.x == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const int nwarm = (int)ceil((double)N / pl.h_out) - 1;
  const int kstart = max(0, sg.ka - nwarm);
  const int flush_lo = (sg.ka == 0) ? 0 : frame_out_start(pl, sg.ka);
  const int flush_hi = (sg.kb >= jb.nc) ? jb.xlen : frame_out_start(pl, sg.kb);
  int flushed = frame_out_start(pl, kstart);      // ring position accounted so far
  if (sg.ka == 0) flushed = 0;
  const float *src_f = (MODE == 0) ? (in_f + jb.in_off) : nullptr;
  float vmax = -INFINITY;

  // TMA prefetch of the first pair
  uint32_t phase[2] = {0u, 0u};
  auto issue_load = [&](int k, int buf) {
    // frames k, k+1 need input [s_k, s_{k+1} + N)
    int sA = frame_in_start(pl, k);
    int kB = min(k + 1, jb.nc - 1);
    int sB = frame_in_start(pl, kB);
    int a0 = sA & ~3;
    int cnt = ((sB + N - a0) + 3) & ~3;
    if (cnt > stage_len) cnt = stage_len;
    uint32_t bytes = (uint32_t)cnt * 4u;
    mbar_expect_tx(&bars[buf], bytes);
    tma_load_1d(buf ? stage1 : stage0, src_f + a0, bytes, &bars[buf]);
  };
  if (MODE == 0 && threadIdx.x == 0 && kstart < sg.kb) issue_load(kstart, 0);

  int cur = 0;
  for (int k = kstart; k < sg.kb; k += 2) {
    const bool hasB = (k + 1 < sg.kb) && (k + 1 < jb.nc);
    float2 *spec;
    if (MODE == 0) {
      // ---- wait for the staged input, prefetch the next pair ----
      if (!mbar_wait(&bars[cur], phase[cur])) return;   // the host reports it (stft_timeout_flag)
      phase[cur] ^= 1u;
      if (threadIdx.x == 0 && k + 2 < sg.kb) issue_load(k + 2, cur ^ 1);
      const float *st = cur ? stage1 : stage0;
      const int sA = frame_in_start(pl, k);
      const int a0 = sA & ~3;
      WinIn W;
      W.a = st + (sA - a0); W.b = st + (hasB ? (frame_in_start(pl, k + 1) - a0) : 0); W.w = wa; W.off = 0; W.hasB = hasB;
      const float *eA = envpool + jb.env_off + (int64_t)((jb.nint > 1) ? k : 0) * nr;
      const float *eB = envpool + jb.env_off + (int64_t)((jb.nint > 1 && hasB) ? (k + 1) : 0) * nr;
      if constexpr (SPEC != 0) {
        OlaOut O;
        O.ra = ola; O.rb = olb; O.ws = ws; O.ring = ring; O.hasB = hasB;
        O.oA = frame_out_start(pl, k) % ring;
        O.oB = hasB ? frame_out_start(pl, k + 1) % ring : 0;
        filter_pair_ct<SPEC>(bufA, bufB, tw, W, O, eA, eB);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        spec = nullptr;
      } else {
      OlaOut O0 = {};
      const bool fuse_rt = (pl.radix[0] <= 5 || pl.radix[0] == 8);
      float2 *Z;
      if (fuse_rt) {
        Z = fft_run<-1, true, false>(bufA, bufB, pl, tw, W, O0);
      } else {
        for (int i = threadIdx.x; i < N; i += (int)blockDim.x) bufA[i] = W[i];
        __syncthreads();
        Z = fft_run<-1, false, false>(bufA, bufB, pl, tw, W, O0);
      }
      // all generic-proxy reads of this staging buffer are done: make it safe for the next TMA write
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      // ---- split the two spectra, multiply by the envelope, rebuild Hermitian halves ----
      for (int kk = threadIdx.x; kk < nr; kk += (int)blockDim.x) {
        if (kk == 0) {
          float2 z0 = Z[0];
          Z[0] = make_float2(eA[0] * z0.x, eB[0] * z0.y);
        } else {
          float2 ok, om;
          float na, nb;
          spec_pair(Z[kk], Z[N - kk], eA[kk], eB[kk], &ok, &om, &na, &nb);
          Z[kk] = ok; Z[N - kk] = om;
          if (kk == nr - 1) Z[nr] = make_float2(na, nb);        // Nyquist := Re(last bin) (seewave.r:3474)
        }
      }
      __syncthreads();
      spec = Z;
      }
    } else {
      // ---- noise: real, zero-phase spectrum u * filter (source.R:111-114) ----
      const UT *uA = in_u + jb.in_off + (int64_t)k * nr;
      const UT *uB = in_u + jb.in_off + (int64_t)(k + 1) * nr;
      const float *fA = nullptr, *fB = nullptr;
      if (jb.env_off >= 0) {
        // filterRowIdx = round(seq(1, ncol, length.out = nc)) (source.R:99)
        int cA = (int)rint(r_seq_at(1.0, (double)jb.nint, jb.nc, k)) - 1;
        int cB = hasB ? (int)rint(r_seq_at(1.0, (double)jb.nint, jb.nc, k + 1)) - 1 : 0;
        fA = envpool + jb.env_off + (int64_t)cA * nr;
        fB = envpool + jb.env_off + (int64_t)cB * nr;
      }
      if constexpr (SPEC != 0) {
        NoiseIn<UT> X;
        X.uA = uA; X.uB = uB; X.ro = vec; X.fA = fA; X.fB = fB; X.off = 0; X.N = N; X.nr = nr; X.hasB = hasB;
        OlaOut O;
        O.ra = ola; O.rb = olb; O.ws = ws; O.ring = ring; O.hasB = hasB;
        O.oA = frame_out_start(pl, k) % ring;
        O.oB = hasB ? frame_out_start(pl, k + 1) % ring : 0;
        noise_pair_ct<SPEC>(bufA, bufB, tw, X, O);
        spec = nullptr;
      } else {
      for (int kk = threadIdx.x; kk < nr; kk += (int)blockDim.x) {
        float ro = vec[kk];
        float va = (float)uA[kk] * ro * (fA ? fA[kk] : 1.0f);
        float vb = hasB ? (float)uB[kk] * ro * (fB ? fB[kk] : 1.0f) : 0.0f;
        float2 v = make_float2(va, vb);
        bufA[kk] = v;
        if (kk > 0) bufA[N - kk] = v;
        if (kk == nr - 1) bufA[nr] = v;
      }
      __syncthreads();
      spec = bufA;
      }
    }
    if (spec != nullptr) {
      float2 *other = (spec == bufA) ? bufB : bufA;
      // the last inverse pass adds the synthesis-windowed frames straight into the two rings
      OlaOut O;
      O.ra = ola; O.rb = olb; O.ws = ws; O.ring = ring; O.hasB = hasB;
      O.oA = frame_out_start(pl, k) % ring;
      O.oB = hasB ? frame_out_start(pl, k + 1) % ring : 0;
      WinIn W0 = {};
      fft_run<+1, false, true>(spec, other, pl, tw, W0, O);
    }
    // ---- samples before the next frame's start are final: write them out once ----
    int knext = k + 2;
    int done_to = (knext < sg.kb) ? frame_out_start(pl, knext) : ((sg.kb >= jb.nc) ? jb.xlen : frame_out_start(pl, sg.kb));
    if (knext >= sg.kb && sg.kb < jb.nc) done_to = flush_hi;
    const int fbase = flushed % ring;
    for (int t = flushed + threadIdx.x; t < done_to; t += (int)blockDim.x) {
      int slot = fbase + (t - flushed);
      if (slot >= ring) slot -= ring;
      float v = ola[slot] + olb[slot];
      ola[slot] = 0.0f; olb[slot] = 0.0f;
      if (t >= flush_lo && t < flush_hi) {
        int oi = t - jb.shift;
        if (oi >= 0 && oi < jb.out_len) {
          outpool[jb.out_off + oi] = v;
          vmax = fmaxf(vmax, v);
        }
      }
    }
    flushed = max(flushed, done_to);
    __syncthreads();
    cur ^= 1;
  }

  // ---- signed maximum of what this CTA emitted ----
  for (int of = 16; of > 0; of >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, of));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = vmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float v = red[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); i++) v = fmaxf(v, red[i]);
    if (v > -INFINITY) atomicMax(&maxpool[jb.max_slot], float_to_ordered(v));
  }
}

size_t stft_smem_bytes(int n, double h_in, double h_out, int mode) {
  int hceil = (int)ceil(h_out) + 2;
  int ring = n + 2 * hceil + 4;
  int stage_len = (n + (int)ceil(h_in) + 12) & ~3;
  size_t floats = (size_t)6 * n + 2 * (size_t)((ring + 3) & ~3) + (mode == 0 ? 2 * (size_t)stage_len : (size_t)stage_len + n / 2 + 4);
  return floats * 4 + 64;
}

// ---------------------------------------------------------------------------------------------------
// Tuned sizes whose radices are all register butterflies (800, 1200, 2400, 160): the same passes, laid
// out for residency.  Every pass has at most one butterfly per thread, so a pass can run IN PLACE
// (load + compute, barrier, store) in a single N-point buffer; the two frames of a pair are added to
// ONE overlap-add ring in two barrier-separated steps; the staging buffer is single (it is only read by
// the first pass, so the next pair's TMA load is issued right after it and overlaps the other four
// passes); twiddles come from global memory through L1.  46 KB per CTA at N = 2400: four CTAs per SM.
// The work buffer is padded by one element per 16 (index i lives at i + i / 16): a first-pass thread
// stores its 16 outputs at 16 p + j, a stride of 128 bytes between lanes that would put a whole half-warp
// on one bank pair; with the pad every pass of the tuned plans stores and loads without conflicts worth
// speaking of (ncu: 4.7e7 store conflicts per 1024 sounds before, see profiles/).
#define STFT_REG_THREADS 160                 // = the largest butterfly count of any tuned pass (2400 / 15)
#ifndef STFT_PAD_DIV
#define STFT_PAD_DIV 16
#endif
__device__ __forceinline__ int pad16(int i) { return i + i / STFT_PAD_DIV; }
struct PadIn {
  const float2 *b;
  int off;
  __device__ __forceinline__ PadIn operator+(int o) const { PadIn r = *this; r.off += o; return r; }
  __device__ __forceinline__ float2 operator[](int i) const { return b[pad16(off + i)]; }
};

template <int DIR, int N, int S, int R, class XIn>
__device__ __forceinline__ bool pass_lc(XIn x, const float2 *__restrict__ tw, float2 *a, int *yo, int b = -1) {
  constexpr int nb = N / R, m = nb / S, sm = S * m;
  if (b < 0) {       // in-place passes: one butterfly per thread
    static_assert(nb <= STFT_REG_THREADS || S == 1, "one butterfly per thread");
    b = threadIdx.x;
  }
  if (b >= nb) return false;
  const int p = b / S, q = b - p * S;
  const XIn xi = x + (q + S * p);
#pragma unroll
  for (int k = 0; k < R; k++) a[k] = xi[k * sm];
  bfly<DIR, R>(a);
  const int ti = p * S;
  if (S > 1 || true) {
#pragma unroll
    for (int j = 1; j < R; j++) {
      float2 w = __ldg(&tw[j * ti]);
      if (DIR > 0) w.y = -w.y;
      a[j] = cmul(a[j], w);
    }
  }
  *yo = q + S * R * p;
  return true;
}

template <int N, int R>
__device__ __forceinline__ bool fused_mid_lc(const PadIn x, const float2 *__restrict__ tw,
                                             const float *__restrict__ eA, const float *__restrict__ eB, float2 *a1,
                                             float2 *a2, int *q1o, int *q2o) {
  constexpr int S = N / R, nr = N / 2;
  const int t = threadIdx.x;
  if (t > S / 2) return false;
  const int q1 = t, q2 = (t == 0) ? 0 : S - t;
  const bool self = (q2 == q1);
#pragma unroll
  for (int k = 0; k < R; k++) { a1[k] = x[q1 + S * k]; a2[k] = self ? a1[k] : x[q2 + S * k]; }
  dft_r<R>(a1);
  if (!self) dft_r<R>(a2);
  float na, nb;
  if (t == 0) {
    a1[0] = make_float2(eA[0] * a1[0].x, eB[0] * a1[0].y);
#pragma unroll
    for (int j = 1; j < R / 2; j++) spec_pair(a1[j], a1[R - j], eA[S * j], eB[S * j], &a1[j], &a1[R - j], &na, &nb);
    constexpr int qa = (nr - 1) % S, ja = (nr - 1) / S, qb = (nr + 1) % S, jb = (nr + 1) / S;
    float2 zk = make_float2(0.f, 0.f), zm = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < R; k++) {
      const float2 wa = __ldg(&tw[((ja * k) % R) * S]), wb = __ldg(&tw[((jb * k) % R) * S]);
      zk = cadd(zk, cmul(x[qa + S * k], wa));
      zm = cadd(zm, cmul(x[qb + S * k], wb));
    }
    float2 d0, d1;
    spec_pair(zk, zm, eA[nr - 1], eB[nr - 1], &d0, &d1, &na, &nb);
    a1[R / 2] = make_float2(na, nb);
  } else if (self) {
#pragma unroll
    for (int j = 0; j < R / 2; j++) spec_pair(a1[j], a1[R - 1 - j], eA[q1 + S * j], eB[q1 + S * j], &a1[j], &a1[R - 1 - j], &na, &nb);
  } else {
#pragma unroll
    for (int j = 0; j < R; j++) {
      const int i1 = q1 + S * j;
      if (i1 < nr) spec_pair(a1[j], a2[R - 1 - j], eA[i1], eB[i1], &a1[j], &a2[R - 1 - j], &na, &nb);
      else spec_pair(a2[R - 1 - j], a1[j], eA[N - i1], eB[N - i1], &a2[R - 1 - j], &a1[j], &na, &nb);
    }
  }
  bfly<+1, R>(a1);
#pragma unroll
  for (int j = 1; j < R; j++) { float2 w = __ldg(&tw[j * q1]); w.y = -w.y; a1[j] = cmul(a1[j], w); }
  if (!self) {
    bfly<+1, R>(a2);
#pragma unroll
    for (int j = 1; j < R; j++) { float2 w = __ldg(&tw[j * q2]); w.y = -w.y; a2[j] = cmul(a2[j], w); }
  }
  *q1o = q1; *q2o = self ? -1 : q2;
  return true;
}

template <int MODE, typename UT, int SPEC>
#ifndef STFT_REG_OCC
#define STFT_REG_OCC 4
#endif
__global__ void __launch_bounds__(STFT_REG_THREADS, STFT_REG_OCC)
k_stft_reg(const FftSeg *__restrict__ segs, const FftJob *__restrict__ jobs, const FftPlan *__restrict__ plans,
           const float2 *__restrict__ twpool, const float *__restrict__ winpool,
           const float *__restrict__ in_f, const UT *__restrict__ in_u, const float *__restrict__ envpool,
           float *__restrict__ outpool, int *__restrict__ maxpool) {
  using P = CtPlan<SPEC>;
  constexpr int N = P::N, F1 = P::F1, F2 = P::F2, MID = P::MID, nr = N / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t bar;
  __shared__ float red[8];

  const FftSeg sg = segs[blockIdx.x];
  const FftJob jb = jobs[sg.job];
  const FftPlan pl = plans[jb.plan];
  const int hceil = (int)ceil(pl.h_out) + 2;
  const int ring = N + 2 * hceil + 4;
  const int stage_len = (N + (int)ceil(pl.h_in) + 12) & ~3;

  float2 *buf = reinterpret_cast<float2 *>(smem_raw);
  float *ola = reinterpret_cast<float *>(buf + ((N + N / 8 + 3) & ~1));      // keeps the TMA target 16-byte aligned
  const PadIn pbuf = {buf, 0};
  float *stage = ola + ((ring + 3) & ~3);                         // filter: staged input; noise: rolloff vector
  const float2 *tw = twpool + pl.tw_off;
  const float *wa = winpool + pl.wa_off;
  const float *ws = winpool + pl.ws_off;
  for (int i = threadIdx.x; i < ring; i += STFT_REG_THREADS) ola[i] = 0.0f;
  if (MODE == 1) {
    for (int i = threadIdx.x; i < nr; i += STFT_REG_THREADS) stage[i] = (float)exp2(jb.rolloffNoise / 10.0 * log2((double)(i + 1)));
  }
  if (MODE == 0 && threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const int nwarm = (int)ceil((double)N / pl.h_out) - 1;
  const int kstart = max(0, sg.ka - nwarm);
  const int flush_lo = (sg.ka == 0) ? 0 : frame_out_start(pl, sg.ka);
  const int flush_hi = (sg.kb >= jb.nc) ? jb.xlen : frame_out_start(pl, sg.kb);
  int flushed = frame_out_start(pl, kstart);
  if (sg.ka == 0) flushed = 0;
  const float *src_f = (MODE == 0) ? (in_f + jb.in_off) : nullptr;
  float vmax = -INFINITY;
  uint32_t phase = 0u;
  auto issue_load = [&](int k) {
    int sA = frame_in_start(pl, k);
    int kB = min(k + 1, jb.nc - 1);
    int sB = frame_in_start(pl, kB);
    int a0 = sA & ~3;
    int cnt = ((sB + N - a0) + 3) & ~3;
    if (cnt > stage_len) cnt = stage_len;
    uint32_t bytes = (uint32_t)cnt * 4u;
    mbar_expect_tx(&bar, bytes);
    tma_load_1d(stage, src_f + a0, bytes, &bar);
  };
  if (MODE == 0 && threadIdx.x == 0 && kstart < sg.kb) issue_load(kstart);

  for (int k = kstart; k < sg.kb; k += 2) {
    const bool hasB = (k + 1 < sg.kb) && (k + 1 < jb.nc);
    constexpr int RMAX = (F1 > MID) ? ((F1 > F2) ? F1 : F2) : ((MID > F2) ? MID : F2);
    float2 a[RMAX], a2[MID];
    int yo = 0;
    bool act;
    if (MODE == 0) {
      if (!mbar_wait(&bar, phase)) return;
      phase ^= 1u;
      const int sA = frame_in_start(pl, k);
      const int a0 = sA & ~3;
      WinIn W;
      W.a = stage + (sA - a0); W.b = stage + (hasB ? (frame_in_start(pl, k + 1) - a0) : 0); W.w = wa; W.off = 0; W.hasB = hasB;
      const float *eA = envpool + jb.env_off + (int64_t)((jb.nint > 1) ? k : 0) * nr;
      const float *eB = envpool + jb.env_off + (int64_t)((jb.nint > 1 && hasB) ? (k + 1) : 0) * nr;
      // forward pass 1: staged frames (window + A + iB packing fused in) -> buf
      act = pass_lc<-1, N, 1, F1, WinIn>(W, tw, a, &yo);
      if (act) {
#pragma unroll
        for (int j = 0; j < F1; j++) buf[pad16(yo + j)] = a[j];
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncthreads();
      if (threadIdx.x == 0 && k + 2 < sg.kb) issue_load(k + 2);      // overlaps the remaining passes
      if constexpr (F2 > 1) {                                          // forward pass 2, in place
        act = pass_lc<-1, N, F1, F2, PadIn>(pbuf, tw, a, &yo);
        __syncthreads();
        if (act) {
#pragma unroll
          for (int j = 0; j < F2; j++) buf[pad16(yo + j * F1)] = a[j];
        }
        __syncthreads();
      }
      // last forward pass + spectrum + first inverse pass, in place
      int q1, q2;
      act = fused_mid_lc<N, MID>(pbuf, tw, eA, eB, a, a2, &q1, &q2);
      __syncthreads();
      if (act) {
#pragma unroll
        for (int j = 0; j < MID; j++) buf[pad16(MID * q1 + j)] = a[j];
        if (q2 >= 0) {
#pragma unroll
          for (int j = 0; j < MID; j++) buf[pad16(MID * q2 + j)] = a2[j];
        }
      }
      __syncthreads();
    } else {
      const UT *uA = in_u + jb.in_off + (int64_t)k * nr;
      const UT *uB = in_u + jb.in_off + (int64_t)(k + 1) * nr;
      NoiseIn<UT> X;
      X.uA = uA; X.uB = uB; X.ro = stage; X.fA = nullptr; X.fB = nullptr; X.off = 0; X.N = N; X.nr = nr; X.hasB = hasB;
      if (jb.env_off >= 0) {
        int cA = (int)rint(r_seq_at(1.0, (double)jb.nint, jb.nc, k)) - 1;
        int cB = hasB ? (int)rint(r_seq_at(1.0, (double)jb.nint, jb.nc, k + 1)) - 1 : 0;
        X.fA = envpool + jb.env_off + (int64_t)cA * nr;
        X.fB = envpool + jb.env_off + (int64_t)cB * nr;
      }
      for (int b = threadIdx.x; b < N / MID; b += STFT_REG_THREADS) {      // global -> buf: no in-place hazard
        pass_lc<+1, N, 1, MID, NoiseIn<UT>>(X, tw, a, &yo, b);
#pragma unroll
        for (int j = 0; j < MID; j++) buf[pad16(yo + j)] = a[j];
      }
      __syncthreads();
    }
    if constexpr (F2 > 1) {                                            // inverse pass 2, in place
      act = pass_lc<+1, N, MID, F2, PadIn>(pbuf, tw, a, &yo);
      __syncthreads();
      if (act) {
#pragma unroll
        for (int j = 0; j < F2; j++) buf[pad16(yo + j * MID)] = a[j];
      }
      __syncthreads();
    }
    // last inverse pass: synthesis window + overlap-add, frame A then frame B into the one ring
    constexpr int SL = MID * F2;
    act = pass_lc<+1, N, SL, F1, PadIn>(pbuf, tw, a, &yo);
    const int oA = frame_out_start(pl, k) % ring;
    const int oB = hasB ? frame_out_start(pl, k + 1) % ring : 0;
    if (act) {
#pragma unroll
      for (int j = 0; j < F1; j++) {
        const int o = yo + j * SL;
        int sa = oA + o;
        if (sa >= ring) sa -= ring;
        ola[sa] += a[j].x * __ldg(&ws[o]);
      }
    }
    __syncthreads();
    if (act && hasB) {
#pragma unroll
      for (int j = 0; j < F1; j++) {
        const int o = yo + j * SL;
        int sb = oB + o;
        if (sb >= ring) sb -= ring;
        ola[sb] += a[j].y * __ldg(&ws[o]);
      }
    }
    __syncthreads();
    // ---- samples before the next frame's start are final: write them out once ----
    int knext = k + 2;
    int done_to = (knext < sg.kb) ? frame_out_start(pl, knext) : ((sg.kb >= jb.nc) ? jb.xlen : frame_out_start(pl, sg.kb));
    if (knext >= sg.kb && sg.kb < jb.nc) done_to = flush_hi;
    const int fbase = flushed % ring;
    for (int t = flushed + threadIdx.x; t < done_to; t += STFT_REG_THREADS) {
      int slot = fbase + (t - flushed);
      if (slot >= ring) slot -= ring;
      float v = ola[slot];
      ola[slot] = 0.0f;
      if (t >= flush_lo && t < flush_hi) {
        int oi = t - jb.shift;
        if (oi >= 0 && oi < jb.out_len) {
          outpool[jb.out_off + oi] = v;
          vmax = fmaxf(vmax, v);
        }
      }
    }
    flushed = max(flushed, done_to);
    __syncthreads();
  }
  for (int of = 16; of > 0; of >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, of));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = vmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float v = red[0];
    for (int i = 1; i < STFT_REG_THREADS / 32; i++) v = fmaxf(v, red[i]);
    if (v > -INFINITY) atomicMax(&maxpool[jb.max_slot], float_to_ordered(v));
  }
}

static bool spec_is_reg(int spec) { return spec == 1 || spec == 3 || spec == 5 || spec == 6; }

size_t stft_smem_bytes_spec(int n, double h_in, double h_out, int mode, int spec) {
  if (!spec_is_reg(spec)) return stft_smem_bytes(n, h_in, h_out, mode);
  int hceil = (int)ceil(h_out) + 2;
  int ring = n + 2 * hceil + 4;
  int stage_len = (n + (int)ceil(h_in) + 12) & ~3;
  size_t floats = (size_t)2 * ((n + n / 8 + 3) & ~1) + (size_t)((ring + 3) & ~3) + (mode == 0 ? (size_t)stage_len : (size_t)(n / 2 + 4));
  return floats * 4 + 64;
}

#define N_SPEC 7
#define STFT_THREADS 256
static size_t attr_smem[3][N_SPEC];   // kept for the call sites; the opt-in itself is per device and serialised

// The dynamic shared-memory opt-in is a per-device function attribute.  Several host threads launch through
// here at once (PipelinedBatches) and a process may drive more than one device, so the attribute is set to the
// device's opt-in maximum once per (device, kernel), under a lock, instead of racing towards a running maximum.
#include <mutex>
#include <set>
#include <utility>
template <typename K>
static cudaError_t ensure_smem(K kf, size_t *slot, size_t smem) {
  (void)slot;
  if (smem <= 48 * 1024) return cudaSuccess;
  static std::mutex mu;
  static std::set<std::pair<int, const void *>> done;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lk(mu);
  auto key = std::make_pair(dev, (const void *)kf);
  if (done.count(key)) return cudaSuccess;
  int optin = 0;
  e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (e != cudaSuccess) return e;
  cudaFuncAttributes fa;
  e = cudaFuncGetAttributes(&fa, kf);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
  if (e == cudaSuccess) done.insert(key);
  return e;
}

int stft_spec_of(int n, const int *radix, int npass) {
  (void)radix; (void)npass;
  static const int sizes[N_SPEC] = {0, 800, 1102, 1200, 2204, 2400, 160};
  for (int sp = 1; sp < N_SPEC; sp++) if (sizes[sp] == n) return sp;
  return 0;
}

template <int SPEC>
static cudaError_t launch_spec(int mode, int u_is_float, const FftSeg *segs, int n_segs, const FftJob *jobs,
                               const FftPlan *plans, const float2 *tw, const float *win, const float *in_f,
                               const void *in_u, const float *env, float *out, int *maxpool, size_t smem,
                               cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  if constexpr (SPEC == 1 || SPEC == 3 || SPEC == 5 || SPEC == 6) {
    if (mode == 0) {
      auto kf = k_stft_reg<0, float, SPEC>;
      if ((e = ensure_smem(kf, &attr_smem[0][SPEC], smem)) != cudaSuccess) return e;
      kf<<<n_segs, STFT_REG_THREADS, smem, st>>>(segs, jobs, plans, tw, win, in_f, nullptr, env, out, maxpool);
    } else if (u_is_float) {
      auto kf = k_stft_reg<1, float, SPEC>;
      if ((e = ensure_smem(kf, &attr_smem[1][SPEC], smem)) != cudaSuccess) return e;
      kf<<<n_segs, STFT_REG_THREADS, smem, st>>>(segs, jobs, plans, tw, win, nullptr, (const float *)in_u, env, out, maxpool);
    } else {
      auto kf = k_stft_reg<1, double, SPEC>;
      if ((e = ensure_smem(kf, &attr_smem[2][SPEC], smem)) != cudaSuccess) return e;
      kf<<<n_segs, STFT_REG_THREADS, smem, st>>>(segs, jobs, plans, tw, win, nullptr, (const double *)in_u, env, out, maxpool);
    }
    return cudaGetLastError();
  }
  if (mode == 0) {
    auto kf = k_stft<0, float, SPEC>;
    if ((e = ensure_smem(kf, &attr_smem[0][SPEC], smem)) != cudaSuccess) return e;
    kf<<<n_segs, STFT_THREADS, smem, st>>>(segs, jobs, plans, tw, win, in_f, nullptr, env, out, maxpool);
  } else if (u_is_float) {
    auto kf = k_stft<1, float, SPEC>;
    if ((e = ensure_smem(kf, &attr_smem[1][SPEC], smem)) != cudaSuccess) return e;
    kf<<<n_segs, STFT_THREADS, smem, st>>>(segs, jobs, plans, tw, win, nullptr, (const float *)in_u, env, out, maxpool);
  } else {
    auto kf = k_stft<1, double, SPEC>;
    if ((e = ensure_smem(kf, &attr_smem[2][SPEC], smem)) != cudaSuccess) return e;
    kf<<<n_segs, STFT_THREADS, smem, st>>>(segs, jobs, plans, tw, win, nullptr, (const double *)in_u, env, out, maxpool);
  }
  return cudaGetLastError();
}

// all segments of one launch share `spec` (0 = run-time plan)
cudaError_t launch_stft(int mode, int u_is_float, int spec, const FftSeg *segs, int n_segs, const FftJob *jobs,
                        const FftPlan *plans, const float2 *tw, const float *win, const float *in_f,
                        const void *in_u, const float *env, float *out, int *maxpool, size_t smem,
                        cudaStream_t st) {
  if (n_segs <= 0) return cudaSuccess;
#define SGB_CASE(SP) case SP: return launch_spec<SP>(mode, u_is_float, segs, n_segs, jobs, plans, tw, win, in_f, in_u, env, out, maxpool, smem, st);
  switch (spec) {
    SGB_CASE(1) SGB_CASE(2) SGB_CASE(3) SGB_CASE(4) SGB_CASE(5) SGB_CASE(6)
    default: return launch_spec<0>(mode, u_is_float, segs, n_segs, jobs, plans, tw, win, in_f, in_u, env, out, maxpool, smem, st);
  }
#undef SGB_CASE
}

// ---------------------------------------------------------------------------------------------------
// K9: power / banded / dB spectrogram of float32 rows into caller-owned memory (sgb_batch_spectrogram,
// sgb_rows_spectrogram).  The forward half of K2: frames start at R's truncated 1 + k h (frame_in_start), two real
// frames share one complex FFT, a pair's input is staged by one TMA bulk copy into a double buffer while the
// previous pair is transformed.  Epilogue: split the two spectra, |X|^2, optional projection onto contiguous bands
// (weights staged in shared memory), optional 10 log10(max(F, floor)), coalesced stores at any dst alignment.
// A CTA walks one segment: frames [ka, kb) of one row (ka even), or, when ka >= nc, the zero tail [ka, kb).
// Frame 2m is always transformed together with frame 2m + 1 (when that frame exists, whether or not it is stored),
// so a row's bits do not depend on its segmentation, on its capacity or on the other rows of the launch.
__global__ void __launch_bounds__(STFT_THREADS)
k_spectrogram(const FftSeg *__restrict__ segs, const SpecRow *__restrict__ rows, const FftPlan pl,
              const float2 *__restrict__ twg, const float *__restrict__ win, const float *__restrict__ src,
              int n_bands, const int32_t *__restrict__ band_tab, const float *__restrict__ band_w, int n_w, int db,
              float db_floor, float *__restrict__ dst) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t bars[2];
  const FftSeg sg = segs[blockIdx.x];
  const SpecRow R = rows[sg.job];
  const int N = pl.n, nr = N / 2, nf = n_bands ? n_bands : nr;
  float *out = dst + R.dst_off;
  if (sg.ka >= R.nc) {                      // zero tail: frames [ka, kb) of the row, no transform
    const int64_t a = (int64_t)sg.ka * nf, e = (int64_t)sg.kb * nf;
    for (int64_t i = a + threadIdx.x; i < e; i += STFT_THREADS) __stcs(out + i, 0.0f);
    return;
  }
  const int stage_len = (N + (int)ceil(pl.h_in) + 12) & ~3;
  float2 *bufA = reinterpret_cast<float2 *>(smem_raw);
  float2 *bufB = bufA + N;
  float2 *tw = bufB + N;
  float *stage0 = reinterpret_cast<float *>(tw + N);
  float *stage1 = stage0 + stage_len;
  int32_t *blo = reinterpret_cast<int32_t *>(stage1 + stage_len), *blen = blo + n_bands, *boff = blen + n_bands;
  float *bw = reinterpret_cast<float *>(boff + n_bands);
  for (int i = threadIdx.x; i < N; i += STFT_THREADS) tw[i] = twg[i];
  for (int i = threadIdx.x; i < 3 * n_bands; i += STFT_THREADS) blo[i] = band_tab[i];
  for (int i = threadIdx.x; i < n_w; i += STFT_THREADS) bw[i] = band_w[i];
  const float *x = src + R.src_off;
  // a row shorter than the window has one frame, read past the row's end as zeros: plain loads, no TMA
  const bool short_row = R.len < N;
  if (short_row) {
    for (int i = threadIdx.x; i < N; i += STFT_THREADS) stage0[i] = (i < R.len) ? x[i] : 0.0f;
  } else if (threadIdx.x == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // frames k, k+1 need input [s_k, s_{k+1} + N); the copy is widened to 16-byte boundaries of the address, which
  // stay inside the allocation (allocations are aligned far coarser than that)
  uint32_t phase[2] = {0u, 0u};
  auto stage_shift = [&](int k) { return (int)(((uintptr_t)(x + frame_in_start(pl, k)) & 15u) >> 2); };
  auto issue_load = [&](int k, int buf) {
    const int sA = frame_in_start(pl, k), sB = frame_in_start(pl, min(k + 1, (int)R.nc - 1));
    const int d = stage_shift(k);
    int cnt = (d + sB - sA + N + 3) & ~3;
    if (cnt > stage_len) cnt = stage_len;
    const uint32_t bytes = (uint32_t)cnt * 4u;
    mbar_expect_tx(&bars[buf], bytes);
    tma_load_1d(buf ? stage1 : stage0, x + sA - d, bytes, &bars[buf]);
  };
  if (!short_row && threadIdx.x == 0) issue_load(sg.ka, 0);

  int cur = 0;
  for (int k = sg.ka; k < sg.kb; k += 2) {
    const bool hasB = k + 1 < R.nc;
    const bool keepA = k < R.cap, keepB = hasB && k + 1 < R.cap;
    const float *st = stage0;
    int d = 0;
    if (!short_row) {
      if (!mbar_wait(&bars[cur], phase[cur])) return;   // sets g_stft_timeout
      phase[cur] ^= 1u;
      if (threadIdx.x == 0 && k + 2 < sg.kb) issue_load(k + 2, cur ^ 1);
      st = cur ? stage1 : stage0;
      d = stage_shift(k);
    }
    WinIn W;
    W.a = st + d; W.b = st + d + (hasB ? frame_in_start(pl, k + 1) - frame_in_start(pl, k) : 0);
    W.w = win; W.off = 0; W.hasB = hasB;
    OlaOut O0 = {};
    float2 *Z;
    if (pl.radix[0] <= 5 || pl.radix[0] == 8) {
      Z = fft_run<-1, true, false>(bufA, bufB, pl, tw, W, O0);
    } else {   // a large prime first radix reads every input (r + 1) / 2 times: window the frames once
      for (int i = threadIdx.x; i < N; i += STFT_THREADS) bufA[i] = W[i];
      __syncthreads();
      Z = fft_run<-1, false, false>(bufA, bufB, pl, tw, W, O0);
    }
    // all generic-proxy reads of this staging buffer are done: make it safe for the next TMA write
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    float *oA = out + (int64_t)k * nf, *oB = oA + nf;
    float *P = reinterpret_cast<float *>(Z == bufA ? bufB : bufA);      // power of frame A, then of frame B
    for (int kk = threadIdx.x; kk < nr; kk += STFT_THREADS) {
      float2 XA, XB;
      pair_split(Z[kk], Z[kk ? N - kk : 0], &XA, &XB);
      const float pa = XA.x * XA.x + XA.y * XA.y, pb = XB.x * XB.x + XB.y * XB.y;
      if (n_bands) {
        P[kk] = pa; P[nr + kk] = pb;
      } else {
        if (keepA) __stcs(oA + kk, db ? 10.0f * log10f(fmaxf(pa, db_floor)) : pa);
        if (keepB) __stcs(oB + kk, db ? 10.0f * log10f(fmaxf(pb, db_floor)) : pb);
      }
    }
    if (n_bands) {
      __syncthreads();
      for (int i = threadIdx.x; i < 2 * n_bands; i += STFT_THREADS) {
        const int f = i >= n_bands, b = i - f * n_bands;
        if (!(f ? keepB : keepA)) continue;
        const float *pp = P + f * nr + blo[b], *ww = bw + boff[b];
        float acc = 0.0f;
        for (int j = 0; j < blen[b]; j++) acc = fmaf(ww[j], pp[j], acc);
        __stcs((f ? oB : oA) + b, db ? 10.0f * log10f(fmaxf(acc, db_floor)) : acc);
      }
    }
    __syncthreads();
    cur ^= 1;
  }
}

size_t spectrogram_smem_bytes(int n, double h_in, int n_bands, int64_t n_w) {
  const int stage_len = (n + (int)ceil(h_in) + 12) & ~3;
  return (size_t)24 * n + 8 * (size_t)stage_len + 12 * (size_t)n_bands + 4 * (size_t)n_w;
}

cudaError_t launch_spectrogram(const FftSeg *segs, int n_segs, const SpecRow *rows, const FftPlan &pl, const float2 *tw,
                               const float *win, const float *src, int n_bands, const int32_t *band_tab,
                               const float *band_w, int n_w, int db, float db_floor, float *dst, size_t smem,
                               cudaStream_t st) {
  if (n_segs <= 0) return cudaSuccess;
  cudaError_t e = ensure_smem(k_spectrogram, nullptr, smem);
  if (e != cudaSuccess) return e;
  k_spectrogram<<<n_segs, STFT_THREADS, smem, st>>>(segs, rows, pl, tw, win, src, n_bands, band_tab, band_w, n_w, db,
                                                    db_floor, dst);
  return cudaGetLastError();
}
