// K1 on the 5th-generation tensor cores (tcgen05 + TMEM): the harmonic loop of generateHarmonics
// (R/source.R:389-419) as a contraction.
//
// The rows of an epoch are integer multiples j of theta' = 2 pi integr / (nSubharm + 1).  With j = KR b + m,
//   sum_j a_j(u) sin(j theta'_u) = Re sum_b e^{i KR b theta'_u} [ S_b(u) - i C_b(u) ],
//   C_b(u) = sum_m a_{KR b + m}(u) cos(m theta'_u),   S_b(u) = sum_m a_{KR b + m}(u) sin(m theta'_u),
// and a_j(u) = Y_j + w(u) dY_j inside one interval of approx() (source.R:403-405), so for the samples of one
// interval C and S are small GEMMs  [128 samples x KR] . [KR x 2 blocks]  of a trig matrix (KR values per sample,
// one complex rotation each) against the interval's amplitude column -- instead of one recurrence step per
// (row, sample) on the FMA pipe.  A CTA (128 threads, four per SM, persistent) takes one interval of approx() (one
// glottal cycle of one epoch, a "unit") at a time:
//   * it stages the amplitude operand of the interval ONCE: Y | dY of up to 1152 rows from K3's FP32 table, scaled by
//     a power of two and split hi + lo in FP16 (22 significant bits), in shared memory in the canonical K-major
//     core-matrix layout, one image per pass of 384 rows; the rows arrive by cp.async while the unit before runs,
//     and rows above the highest nonzero one (they add exactly 0) are skipped in whole block pairs;
//   * per tile of 128 samples (thread = sample = TMEM lane) every thread writes its trig row cos / sin(m theta'),
//     m < KR, hi + lo in FP16, into TMEM with tcgen05.st: the A operand of the MMAs never touches shared memory;
//   * per pass two threads issue three tcgen05.mma kind::f16 each (M 128, N = 2 x blocks <= 48, K 16: hi hi + lo hi +
//     hi lo, one chain for C and one for S), FP32 accumulators in TMEM (128 columns per CTA: 32 of A, 96 of C | S);
//   * tcgen05.ld hands every thread its own lane: C_b, S_b (Y and dY parts) of the pass for ITS sample, reduced
//     in registers by a complex Horner recurrence in e^{2 i KR theta'} on packed FP32 pairs (even | odd blocks); the
//     pass offset e^{i 384 p theta'} is a rotation seeded from the FP64 phase.
// Phase: as in the FMA kernel, FP64 closed form per spline piece (K0's quartic), re-anchored at every knot.
// Why it looks like this (operands in TMEM, FP16, two issuers, pass size): scripts/micro/mma_rate.cu and
// profiles/README.md.  Epochs with few rows are left to the FP32-pipe kernel (kernels_synth.cu; engine.cu decides).
#include "engine.cuh"
#include <cuda_fp16.h>
#include <cstdlib>
#include <cstdio>

#define TC_KR 16                         // rows per block = K of the contraction
#define TC_TILE 128                      // samples per tile = M of the MMAs = TMEM lanes

__device__ __forceinline__ uint32_t tc_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// -DTC_PROF: wall-clock shares of the kernel's phases as one worker warp sees them (printed per launch)
#ifdef TC_PROF
__device__ unsigned long long g_tc_prof[16];
#define TP_DECL long long prof[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long t0_ = clock64();
#define TP(i) { long long t_ = clock64(); if (tid == 64) prof[i] += t_ - t0_; t0_ = t_; }
#define TP_END if (tid == 64) for (int i = 0; i < 10; i++) atomicAdd(&g_tc_prof[i], (unsigned long long)prof[i]);
#else
#define TP_DECL
#define TP(i)
#define TP_END
#endif
__device__ int g_tc_timeout = 0;          // an MMA completion barrier that never flipped (reported by the host)
int synth_tc_timeout_flag() { int v = 0; cudaMemcpyFromSymbol(&v, g_tc_timeout, sizeof v); return v; }

// tcgen05.ld 32x32b.x16: 16 consecutive columns of this thread's lane
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float *v) {
  uint32_t *r = reinterpret_cast<uint32_t *>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                 "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr));
}

// Work list: one unit per interval of approx() of every epoch.  One thread per syllable; intervals without
// samples get kbeg == kend.
__global__ void k_build_units_tc(const sgb_syllable *syl, const SylCtrl *ctrl, int S, const SylLayout *lay, const Pools P, TcUnit *units,
                                 int min_rows) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const SylCtrl &C = ctrl[s];
  if (C.status != SGB_OK || C.nGC == 0) return;
  const int64_t o = P.gc_off[s];
  const int32_t *gcup = P.gcup + o;
  const double *kt = P.kt + o;
  const int G = C.nGC;
  int t = lay[s].pad;                     // first unit of this syllable
  const int t_end = t + C.tiles_tc;
  int a = 0;
  for (int e = 0; e < C.nEpochs; e++) {
    const int g_first = C.ep_start[e] - 1, g_last = C.ep_end[e] - 1;
    const int x_first_i = gcup[g_first];
    const double x_first = (double)x_first_i, x_last = (double)gcup[g_last];
    const int Ne = gcup[C.ep_end[e]] - x_first_i + 1;
    const double by = (x_last - x_first) / (double)(Ne - 1);
    const int nknots = g_last - g_first + 1;
    const int nsub = C.vf_active ? C.ep_nsub[e] : 0;
    const int J = C.ep_rows[e];
    if (J < min_rows) {                    // few rows: the FP32-pipe kernel's epoch (no units were reserved for it)
      while (a > 0 && (double)gcup[g_last] < kt[a]) a--;
      continue;
    }
    auto vfun = [&](int k) { return (k >= Ne - 1) ? x_last : (x_first + (double)k * by); };
    int kcur = 0;
    for (int i = 0; i <= nknots - 2; i++) {
      int kend = Ne;
      if (i < nknots - 2) {               // first sample whose coordinate reaches the next knot
        const double X = (double)gcup[g_first + i + 1];
        int k = (int)ceil((X - x_first) / by);
        k = max(kcur, min(k, Ne));
        while (k > kcur && vfun(k - 1) >= X) k--;
        while (k < Ne && vfun(k) < X) k++;
        kend = k;
      }
      const double u = (double)(x_first_i + kcur);
      while (a < G - 1 && u >= kt[a + 1]) a++;
      TcUnit U;
      U.col_off = 2 * (lay[s].amp_off + C.ep_amp_off[e]) + (int64_t)i * J;      // in {Y, dY} pairs (8 B)
      U.wave_off = lay[s].wave_off + C.ep_wave_off[e];
      U.pc_off = o;
      U.x_first = x_first; U.by = by; U.x_last = x_last;
      U.inv_sr_np1 = 1.0 / (syl[s].samplingRate * (double)(nsub + 1));
      U.Ne = Ne; U.kbeg = kcur; U.kend = kend;
      U.xg = gcup[g_first + i]; U.xn = gcup[g_first + i + 1];
      U.a_lo = a; U.G = G; U.J = J; U.epmax_idx = s * SGB_MAX_EPOCHS + e; U.pad = 0;
      if (t < t_end) units[t++] = U;
      kcur = kend;
    }
    while (a > 0 && (double)gcup[g_last] < kt[a]) a--;     // epochs overlap by one cycle
  }
  TcUnit Z = {};
  while (t < t_end) units[t++] = Z;
}

#define TC_PASS_BLOCKS 24                         // blocks of one pass: N = 48 accumulator columns for C and for S
#define TC_PASS_ROWS (TC_PASS_BLOCKS * TC_KR)     // 384 rows
#define TC_B_PASSES 3                             // passes whose amplitude operand is resident (1152 rows)
#define TC_MAX_ROWS (TC_B_PASSES * TC_PASS_ROWS)
#define TC_IMG_BYTES (2 * TC_PASS_BLOCKS * TC_KR * 2)  // one FP16 amplitude image of a pass: 48 columns (Y, dY of 24 blocks) x KR
#define TC_IMGS_BYTES (TC_B_PASSES * 2 * TC_IMG_BYTES)
#define TC_SMEM (TC_IMGS_BYTES + 2 * TC_MAX_ROWS * 8)   // the images, then two staging buffers of {Y, dY} rows
#define TC_NPC 4                                  // spline pieces staged per unit (an interval spans two or three)
// instruction descriptor of kind::f16: FP16 x FP16 -> FP32, both operands K-major, M 128
#define TC_IDESC(N) ((1u << 4) | ((uint32_t)((N) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24))
// TMEM columns of a CTA (128): the trig operand (A of the MMAs: lane = sample, one column = rows m, m + 1 in FP16)
// and the accumulators
#define TC_COL_CH 0
#define TC_COL_CL 8
#define TC_COL_SH 16
#define TC_COL_SL 24
#define TC_COL_C 32
#define TC_COL_S 80

// FP16, K-major, no swizzle: a core matrix is 8 rows x 16 bytes (8 values of K); K = 16 is two of them, 128 B apart
// (LBO); the next 8 rows are 256 B further (SBO)
__device__ __forceinline__ uint64_t tc_desc16(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)(128 >> 4) << 16;
  d |= (uint64_t)(256 >> 4) << 32;
  d |= (uint64_t)1 << 46;                 // descriptor version of sm_100
  return d;
}
__device__ __forceinline__ int tc_off16(int n, int k) { return (n >> 3) * 256 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2; }
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void tc_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n\t}\n"
               :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0) : "memory");
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t *r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
// x = hi + lo in FP16 (22 significant bits; lo may be subnormal: absolute error <= 2^-25)
__device__ __forceinline__ void tc_split16(float2 x, uint32_t &hi, uint32_t &lo) {
  const __half2 h = __floats2half2_rn(x.x, x.y);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x.x - hf.x, x.y - hf.y);
  hi = *reinterpret_cast<const uint32_t *>(&h);
  lo = *reinterpret_cast<const uint32_t *>(&l);
}
// One accumulator chain of a pass: {hi hi, lo hi, hi lo}, then the commit that arrives on the mbarrier.  Two threads
// issue (one for C, one for S): an MMA costs its issuing thread 60-90 cycles, whatever its size (scripts/micro/mma_rate.cu).
__device__ __forceinline__ void tc_issue_chain(uint32_t tmem_d, uint32_t tmem_a_hi, uint32_t tmem_a_lo, uint64_t descB, int nb,
                                               uint32_t bar_addr) {
  const uint32_t idesc = TC_IDESC(2 * nb);
  tc_mma_ts(tmem_d, tmem_a_hi, descB, idesc, 0u);
  tc_mma_ts(tmem_d, tmem_a_lo, descB, idesc, 1u);
  tc_mma_ts(tmem_d, tmem_a_hi, descB + (uint64_t)(TC_IMG_BYTES >> 4), idesc, 1u);
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar_addr) : "memory");
}
// global -> shared without a register round trip (L1-allocating): 8 B for a {Y, dY} row (a column starts on any
// pair, so wider copies would be misaligned), 16 B for the unit record
__device__ __forceinline__ void tc_cp8(void *s, const void *g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(tc_smem_u32(s)), "l"(g) : "memory");
}
__device__ __forceinline__ void tc_cp16(void *s, const void *g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" :: "r"(tc_smem_u32(s)), "l"(g) : "memory");
}

__global__ void __launch_bounds__(128, 4)
k_synth_tc(const TcUnit *__restrict__ units, int nunits, const double *__restrict__ pc, const float4 *__restrict__ amp,
           float *__restrict__ wave, int *__restrict__ epmax) {
  // per resident pass: hi, lo images of the amplitude operand; then two staging buffers of TC_MAX_ROWS {Y, dY} rows
  extern __shared__ __align__(1024) uint8_t sB[];
  float2 *const stage = reinterpret_cast<float2 *>(sB + TC_IMGS_BYTES);
  __shared__ uint64_t bar;
  __shared__ __align__(16) TcUnit su[2];               // the current and the next unit
  __shared__ double spc[2][TC_NPC * SYNTH_PC];        // their first spline pieces {knot, c0..c4}
  __shared__ float smax[4];
  __shared__ int stop[4];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float2 *__restrict__ amp2 = reinterpret_cast<const float2 *>(amp);

  // ---- operand prefetch, one item (super-pass of a unit) ahead, with cp.async: the item's {Y, dY} rows into a staging
  // buffer (row0 + r at r), and for a new unit its record and spline pieces.  Waited for, and made visible by a
  // barrier, at the end of the item before.  The next unit's column and pieces are loaded when the current unit
  // starts and used after its staging, so that the loads are in flight meanwhile.
  int64_t ncol = 0, npco = 0;
  int nJ = 0, nG = 0, nalo = 0;
  auto locate_unit = [&](int u) {
    const TcUnit *N = units + u;
    ncol = __ldg(&N->col_off); nJ = __ldg(&N->J);
    npco = __ldg(&N->pc_off); nG = __ldg(&N->G); nalo = __ldg(&N->a_lo);
  };
  auto fetch_rows = [&](float2 *dst, const float2 *col, int J, int row0) {    // rows j = 0 (zero) .. J: col[j - 1]
#pragma unroll
    for (int i = 0; i < TC_MAX_ROWS / 128; i++) {
      const int j = row0 + tid + 128 * i;
      if (j >= 1 && j <= J) tc_cp8(dst + tid + 128 * i, col + (j - 1));
    }
  };
  auto fetch_unit = [&](int u, int ub, int buf) {
    if (tid < (int)(sizeof(TcUnit) / 16)) tc_cp16(reinterpret_cast<uint4 *>(&su[ub]) + tid, reinterpret_cast<const uint4 *>(units + u) + tid);
    if (tid < TC_NPC * SYNTH_PC && nG > 0)     // pieces a_lo .. a_lo + 3 (the syllable has G of them)
      tc_cp8(&spc[ub][tid], pc + SYNTH_PC * (npco + min(nalo + tid / SYNTH_PC, nG - 1)) + tid % SYNTH_PC);
    fetch_rows(stage + buf * TC_MAX_ROWS, amp2 + ncol, nJ, 0);
  };
  int ui = blockIdx.x, ub = 0, buf = 0;       // unit, its buffer (su, spc), the current item's staging buffer
  if (ui < nunits) { locate_unit(ui); fetch_unit(ui, 0, 0); }
  asm volatile("cp.async.commit_group;" ::: "memory");

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(tc_smem_u32(&tmem_base_s)), "n"(128));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 2;" :: "r"(tc_smem_u32(&bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const uint32_t tmem_base = tmem_base_s;
  const uint32_t lane_addr = tmem_base + ((uint32_t)(warp * 32) << 16);
  const uint64_t descB = tc_desc16(tc_smem_u32(sB));
  const uint32_t barA = tc_smem_u32(&bar);
  const bool issuer = lane == 0 && warp < 2;         // warp 0: the C chain, warp 1: the S chain
  const uint32_t my_d = tmem_base + (warp == 0 ? TC_COL_C : TC_COL_S);
  const uint32_t my_ahi = tmem_base + (warp == 0 ? TC_COL_CH : TC_COL_SH), my_alo = tmem_base + (warp == 0 ? TC_COL_CL : TC_COL_SL);
  uint32_t phase = 0u;
  bool dead = false;
  TP_DECL

  for (; ui < nunits && !dead; ui += gridDim.x, ub ^= 1) {
    const TcUnit U = su[ub];
    const int un = ui + gridDim.x;
    if (un < nunits) locate_unit(un);
    const bool work = U.kend > U.kbeg;
    const int J = U.J;
    const float2 *__restrict__ col = amp2 + U.col_off;                // {Y, dY} of the interval, row j - 1
    const double *__restrict__ pcs = pc + SYNTH_PC * U.pc_off;
    const double *spcu = spc[ub];
    const int x_first_i = (int)U.x_first;
    const float inv_dx = __frcp_rn((float)(U.xn - U.xg));
    const int nsuper = work ? (J + TC_MAX_ROWS) / TC_MAX_ROWS : 1;    // rows j = 0 (zero) .. J, 1152 per super-pass
    float unit_max = 0.f;

    for (int sp = 0; sp < nsuper && !dead; sp++, buf ^= 1) {
      bool fetched = false;
      auto prefetch = [&]() {
        if (sp + 1 < nsuper) fetch_rows(stage + (buf ^ 1) * TC_MAX_ROWS, col, J, (sp + 1) * TC_MAX_ROWS);
        else if (un < nunits) fetch_unit(un, ub ^ 1, buf ^ 1);
        asm volatile("cp.async.commit_group;" ::: "memory");
        fetched = true;
      };
      if (work) {
        TP(0)
        const int row0 = sp * TC_MAX_ROWS;
        const float2 *stg = stage + buf * TC_MAX_ROWS;
        // ---- amplitude operand: rows row0 .. row0 + 16 blocks - 1, scaled by a power of two so that the largest
        // |Y|, |dY| sits in [2^14, 2^15): hi + lo in FP16 then carry 22 bits of every value down to 2^-39 of the
        // largest.  Rows above the highest one with Y != 0 or dY != 0 (the live top) contribute exactly 0 and are
        // left out in whole block pairs: blocks, passes and the Horner start follow the live top ----
        float mx = 0.f;
        int top = -1;
#pragma unroll
        for (int i = 0; i < TC_MAX_ROWS / 128; i++) {
          const int r = tid + 128 * i, j = row0 + r;
          if (j >= 1 && j <= J) {
            const float2 q = stg[r];
            mx = fmaxf(mx, fmaxf(fabsf(q.x), fabsf(q.y)));
            if (q.x != 0.f || q.y != 0.f) top = r;
          }
        }
#pragma unroll
        for (int of = 16; of > 0; of >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, of));
        top = __reduce_max_sync(0xffffffffu, top);
        if (lane == 0) { smax[warp] = mx; stop[warp] = top; }
        __syncthreads();
        mx = fmaxf(fmaxf(smax[0], smax[1]), fmaxf(smax[2], smax[3]));
        top = max(max(stop[0], stop[1]), max(stop[2], stop[3]));
        const int ex = (mx > 0.f && mx < 3.0e38f) ? ilogbf(mx) : 14;
        const float scale = scalbnf(1.0f, 14 - ex), unscale = scalbnf(1.0f, ex - 14);
        const int lblocks = (top + TC_KR) / TC_KR;                      // blocks up to the live top (0: none)
        const int blocks = (lblocks + 7) & ~7;                          // N = 2 x blocks is a multiple of 16
        const int npass = (blocks + TC_PASS_BLOCKS - 1) / TC_PASS_BLOCKS;
        const int qtop = (((lblocks - 1) % TC_PASS_BLOCKS) >> 1) & 3;  // top block pair of the last pass, in its group
#pragma unroll
        for (int i = 0; i < TC_MAX_ROWS / 128; i++) {
          const int r = tid + 128 * i, j = row0 + r;
          if (r < blocks * TC_KR) {
            const float2 q = (j >= 1 && j <= J) ? stg[r] : make_float2(0.f, 0.f);
            const int p = r / TC_PASS_ROWS, rr = r % TC_PASS_ROWS, b = rr / TC_KR, m = rr % TC_KR;
            const float ys = q.x * scale, ds = q.y * scale;
            const __half yh = __float2half_rn(ys), dh = __float2half_rn(ds);
            const __half yl = __float2half_rn(ys - __half2float(yh)), dl = __float2half_rn(ds - __half2float(dh));
            // accumulator columns of a block pair: {Y_2q, Y_2q+1, dY_2q, dY_2q+1} (register pairs for the packed epilogue)
            uint8_t *hi = sB + p * (2 * TC_IMG_BYTES) + tc_off16(4 * (b >> 1) + (b & 1), m), *lo = hi + TC_IMG_BYTES;
            *reinterpret_cast<__half *>(hi) = yh; *reinterpret_cast<__half *>(hi + 32) = dh;
            *reinterpret_cast<__half *>(lo) = yl; *reinterpret_cast<__half *>(lo + 32) = dl;
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();                               // sB
        TP(1)
        auto pass_blocks = [&](int p) { return min(blocks - p * TC_PASS_BLOCKS, TC_PASS_BLOCKS); };   // 8, 16 or 24

        // phase of sample k of the unit: FP64 closed form of the spline piece; returns integr / (nSubharm + 1) in cycles
        auto sample_phase = [&](int k, float &ww_out) -> double {
          const double v = (k >= U.Ne - 1) ? U.x_last : (U.x_first + (double)k * U.by);
          ww_out = (float)(v - (double)U.xg) * inv_dx;
          const double u = (double)(x_first_i + k);
          int a = 0;                               // piece: largest a with knot <= u; staged ones first
          const int na = min(TC_NPC, U.G - U.a_lo);
          while (a < na - 1 && u >= spcu[SYNTH_PC * (a + 1)]) a++;
          double p0 = spcu[SYNTH_PC * a], p1 = spcu[SYNTH_PC * a + 1], p2 = spcu[SYNTH_PC * a + 2], p3 = spcu[SYNTH_PC * a + 3],
                 p4 = spcu[SYNTH_PC * a + 4], p5 = spcu[SYNTH_PC * a + 5];
          if (a == TC_NPC - 1) {                   // rare: the interval reaches past the staged pieces
            int ag = U.a_lo + a;
            while (ag < U.G - 1 && u >= pcs[SYNTH_PC * (ag + 1)]) ag++;
            const double *pp = pcs + SYNTH_PC * ag;
            p0 = pp[0]; p1 = pp[1]; p2 = pp[2]; p3 = pp[3]; p4 = pp[4]; p5 = pp[5];
          }
          const double M = u - p0;
          const double ph = fma(fma(fma(fma(p5, M, p4), M, p3), M, p2), M, p1);
          const double x = ph * U.inv_sr_np1;
          return x - floor(x);
        };
        // a super-pass after the first with no live row adds exactly 0: its samples keep what the one before wrote.  A
        // first super-pass without one still writes its zeros, and issues no MMA
        if (sp == 0 || npass > 0) {
          float ww_n;
          double x_n = sample_phase(min(U.kbeg + tid, U.kend - 1), ww_n);
          unit_max = 0.f;

          for (int k0 = U.kbeg; k0 < U.kend && !dead; k0 += TC_TILE) {
            // ---- this thread's sample: interval weight and phase (computed one tile ahead, in the shadow of the MMAs) ----
            const bool live = k0 + tid < U.kend;
            const int k = live ? k0 + tid : k0;
            const float ww = ww_n;
            const double x = x_n;
            TP(2)
            // ---- trig operand rows: cos / sin (m theta'), m < KR, hi + lo in FP16, into this thread's TMEM lane; even and
            // odd m are two packed FP32 chains and share a column ----
            if (npass > 0) {
              {
                float s1, c1;
                sincospif(2.0f * (float)x, &s1, &c1);
                const float c2 = fmaf(c1, c1, -(s1 * s1)), s2 = 2.0f * s1 * c1;        // e^{2 i theta'}
                const float2 C2 = make_float2(c2, c2), S2 = make_float2(s2, s2), nS2 = make_float2(-s2, -s2);
                float2 cm = make_float2(1.f, c1), sm = make_float2(0.f, s1);            // rows m, m + 1
                uint32_t ch[8], cl[8], sh[8], sl[8];
#pragma unroll
                for (int h = 0; h < TC_KR / 2; h++) {
                  tc_split16(cm, ch[h], cl[h]); tc_split16(sm, sh[h], sl[h]);
                  const float2 nc = __ffma2_rn(cm, C2, __fmul2_rn(sm, nS2)), ns = __ffma2_rn(cm, S2, __fmul2_rn(sm, C2));
                  cm = nc; sm = ns;
                }
                tc_st8(lane_addr + TC_COL_CH, ch); tc_st8(lane_addr + TC_COL_CL, cl);
                tc_st8(lane_addr + TC_COL_SH, sh); tc_st8(lane_addr + TC_COL_SL, sl);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
              }
              TP(3)
              asm volatile("tcgen05.fence::before_thread_sync;");
              __syncthreads();
              if (issuer) {
                asm volatile("tcgen05.fence::after_thread_sync;");
                tc_issue_chain(my_d, my_ahi, my_alo, descB, pass_blocks(0), barA);
              }
            }
            TP(4)
            // in the shadow of the first MMAs: z = e^{i KR theta'}, z^2, the pass rotation P = e^{i 384 theta'}, E = e^{i row0 theta'}
            float zc, zs;
            { double q = x * (double)TC_KR; q -= floor(q); sincospif(2.0f * (float)q, &zs, &zc); }
            const float zc2 = fmaf(zc, zc, -(zs * zs)), zs2 = 2.0f * zs * zc;
            const float2 z2c = make_float2(zc2, zc2), z2s = make_float2(zs2, zs2), nz2s = make_float2(-zs2, -zs2);
            const float2 ww2 = make_float2(ww, ww);
            float ec = 1.f, es = 0.f, pc_ = 1.f, ps_ = 0.f;
            if (npass > 1) { double q = x * (double)TC_PASS_ROWS; q -= floor(q); sincospif(2.0f * (float)q, &ps_, &pc_); }
            float acc = 0.f, prev = 0.f;
            if (sp > 0) {
              double q = x * (double)row0; q -= floor(q); sincospif(2.0f * (float)q, &es, &ec);
              if (live) prev = wave[U.wave_off + k];
            }
            if (k0 + TC_TILE < U.kend) x_n = sample_phase(min(k0 + TC_TILE + tid, U.kend - 1), ww_n);
            if (k0 == U.kbeg) prefetch();

            for (int p = 0; p < npass; p++) {
              const int nb = pass_blocks(p);
              uint32_t ok = 0, polls = 0;
              while (!ok) {
                asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.b32 %0, 1, 0, p;\n}\n"
                             : "=r"(ok) : "r"(barA), "r"(phase) : "memory");
                if (!ok && ++polls > (1u << 24)) { g_tc_timeout = 1; dead = true; break; }
              }
              phase ^= 1u;
              TP(5)
              asm volatile("tcgen05.fence::after_thread_sync;");
              // ---- R = sum_b z^b (S_b - i C_b): Horner in z^2 from the top live block pair, even and odd blocks as the
              // two halves of packed FP32 pairs; Q = -Im R ----
              float2 Rr = make_float2(0.f, 0.f), Q = make_float2(0.f, 0.f);
              float Cv[2][16], Sv[2][16];                      // 8 blocks = 16 accumulator columns of C and of S, two in flight
              const int g = nb / 8 - 1, qt = p == npass - 1 ? qtop : 3;
              tc_ld16(lane_addr + TC_COL_C + 16 * g, Cv[0]); tc_ld16(lane_addr + TC_COL_S + 16 * g, Sv[0]);
              asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
              for (int it = 0; it < TC_PASS_BLOCKS / 8; it++) {
                const int cur = it & 1;
                if (g - it < 0) break;
                if (g - it - 1 >= 0) {
                  tc_ld16(lane_addr + TC_COL_C + 16 * (g - it - 1), Cv[cur ^ 1]); tc_ld16(lane_addr + TC_COL_S + 16 * (g - it - 1), Sv[cur ^ 1]);
                }
#pragma unroll
                for (int q = 3; q >= 0; q--) {
                  if (it == 0 && q > qt) continue;
                  const float2 Cc = __ffma2_rn(ww2, make_float2(Cv[cur][4 * q + 2], Cv[cur][4 * q + 3]), make_float2(Cv[cur][4 * q], Cv[cur][4 * q + 1]));
                  const float2 Ss = __ffma2_rn(ww2, make_float2(Sv[cur][4 * q + 2], Sv[cur][4 * q + 3]), make_float2(Sv[cur][4 * q], Sv[cur][4 * q + 1]));
                  const float2 nr = __ffma2_rn(Rr, z2c, __ffma2_rn(Q, z2s, Ss)), nq = __ffma2_rn(Rr, nz2s, __ffma2_rn(Q, z2c, Cc));
                  Rr = nr; Q = nq;
                }
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
              }
              asm volatile("tcgen05.fence::before_thread_sync;");
              __syncthreads();                       // the accumulators are free
              if (issuer && p + 1 < npass) {
                asm volatile("tcgen05.fence::after_thread_sync;");
                tc_issue_chain(my_d, my_ahi, my_alo, descB + (uint64_t)(((p + 1) * 2 * TC_IMG_BYTES) >> 4), pass_blocks(p + 1), barA);
              }
              TP(6)
              // R = R_even + z R_odd;  acc += Re (E R)
              const float Rre = fmaf(zc, Rr.y, fmaf(zs, Q.y, Rr.x));            // zc Rr_o - zs Ri_o, Ri_o = -Q_o
              const float Rim = fmaf(zs, Rr.y, fmaf(-zc, Q.y, -Q.x));           // zs Rr_o + zc Ri_o + Ri_e
              acc = fmaf(ec, Rre, fmaf(-es, Rim, acc));
              const float ne = fmaf(ec, pc_, -(es * ps_)), nsn = fmaf(ec, ps_, es * pc_); ec = ne; es = nsn;
              TP(7)
            }
            acc = fmaf(acc, unscale, prev);
            if (live) wave[U.wave_off + k] = acc;
            if (live) unit_max = fmaxf(unit_max, fabsf(acc));
            TP(8)
          }
        }
      }
      if (work && sp == nsuper - 1) {   // max |w| of the epoch over what the last super-pass that ran wrote (tolerance of
#pragma unroll                          // the zero-crossing searches in K6)
        for (int of = 16; of > 0; of >>= 1) unit_max = fmaxf(unit_max, __shfl_xor_sync(0xffffffffu, unit_max, of));
        if (lane == 0 && unit_max > 0.0f) atomicMax(&epmax[U.epmax_idx], float_to_ordered(unit_max));
      }
      if (!fetched) prefetch();
      asm volatile("cp.async.wait_all;" ::: "memory");
      __syncthreads();               // sB, smax, stop and the staging buffer are rewritten next, su / spc one unit later:
                                     // all MMAs completed above, every thread is past its reads; the prefetch landed
    }
  }
  TP_END
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "n"(128));
}

int synth_min_rows();       // kernels_ctrl.cu: the K1 dispatch threshold the work lists were sized with
void launch_build_tiles_tc(const sgb_syllable *syl, const SylCtrl *ctrl, int S, const SylLayout *lay, const Pools &P, TcUnit *units,
                           cudaStream_t st) {
  if (S <= 0) return;
  k_build_units_tc<<<(S + 127) / 128, 128, 0, st>>>(syl, ctrl, S, lay, P, units, synth_min_rows());
}

cudaError_t launch_synth_tc(const TcUnit *units, int n_units, const Pools &P, const float4 *amp, float *wave, int *epmax, cudaStream_t st) {
  if (n_units <= 0) return cudaSuccess;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(k_synth_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = std::min(n_units, 4 * sms);               // persistent: four CTAs (4 x 128 TMEM columns) per SM
  k_synth_tc<<<grid, 128, TC_SMEM, st>>>(units, n_units, P.pc, amp, wave, epmax);
#ifdef TC_PROF
  {
    cudaStreamSynchronize(st);
    unsigned long long h[16], z[16] = {};
    cudaMemcpyFromSymbol(h, g_tc_prof, sizeof h);
    cudaMemcpyToSymbol(g_tc_prof, z, sizeof z);
    double tot = 0;
    for (int i = 0; i < 10; i++) tot += (double)h[i];
    fprintf(stderr, "tcprof grid %d:", grid);
    for (int i = 0; i < 10; i++) fprintf(stderr, " %d:%.1f%%", i, 100.0 * h[i] / tot);
    fprintf(stderr, " cyc/cta %.0f\n", tot / grid);
  }
#endif
  return cudaGetLastError();
}
