// Host engine + C ABI of libsoundgen_b200.so (include/soundgen_b200.h).
//
// The engine owns device memory (grow-only pools), one CUDA stream and the host-side
// layout logic that R's soundgen() performs implicitly with c() / addVectors()
// (R/soundgen.R:632-640, 708-714, 743-748, 813-818, 836-849).  All arithmetic on
// samples happens in the kernels; the host only sizes and places buffers.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "engine.cuh"
#include "hostpar.h"
#include <cstdlib>

// ---- kernel launchers defined in the other translation units ----
void launch_control(const sgb_syllable *, int, bool, const int32_t *, const double *, const double *, const double *, const Pools &,
                    SylCtrl *, SylLayout *, int64_t *, cudaStream_t);
void launch_tiles_amp(const sgb_syllable *, int, const SylCtrl *, const SylLayout *, const Pools &, SynthTile *,
                      int64_t *, double *, float4 *, cudaStream_t);
void launch_rolloff_api(const double *, int, int, const double *, int, const double *, int, const double *, int,
                        double, double, double, double, double, double, double *, int *, double *, int *);
void launch_fp32_peak(float2 *, int, int, int);
void launch_synth(const SynthTile *, int, const sgb_syllable *, const SylCtrl *, const SylLayout *, const Pools &,
                  const float4 *, float *, int *, cudaStream_t);
void launch_build_tiles_tc(const sgb_syllable *, const SylCtrl *, int, const SylLayout *, const Pools &, TcUnit *, cudaStream_t);
void synth_min_rows_set(int);
cudaError_t launch_synth_tc(const TcUnit *, int, const Pools &, const float4 *, float *, int *, cudaStream_t);
int synth_tc_timeout_flag();
void launch_compose(const sgb_syllable *, int, SylCtrl *, const SylLayout *, const Pools &, const double *,
                    const float *, float *, const double *, const double *, const int *, cudaStream_t);
void launch_place_voiced(const sgb_syllable *, int, const SylCtrl *, const SylLayout *, const SylPlace *,
                         const Pools &, const float *, float *, int, cudaStream_t);
void launch_env_tracks(const EnvInst *, int, const sgb_envelope *, const sgb_formant_ref *, const double *,
                       const double *, double *, double *, void *, double *, cudaStream_t);
cudaError_t launch_envelope_f32(const EnvInst *, int, int, int, const sgb_envelope *, const sgb_formant_ref *,
                                const double *, const double *, const double *, const double *, const double *, float *,
                                cudaStream_t);
cudaError_t launch_envelope_f64(const EnvInst *, int, int, int, const sgb_envelope *, const sgb_formant_ref *,
                                const double *, const double *, const double *, const double *, const double *, double *,
                                cudaStream_t);
size_t stft_smem_bytes(int n, double h_in, double h_out, int mode);
size_t stft_smem_bytes_spec(int n, double h_in, double h_out, int mode, int spec);
cudaError_t launch_stft(int mode, int u_is_float, int spec, const FftSeg *, int, const FftJob *, const FftPlan *,
                        const float2 *, const float *, const float *, const void *, const float *, float *, int *,
                        size_t, cudaStream_t);
int stft_spec_of(int n, const int *radix, int npass);
size_t spectrogram_smem_bytes(int n, double h_in, int n_bands, int64_t n_w);
cudaError_t launch_spectrogram(const FftSeg *, int, const SpecRow *, const FftPlan &, const float2 *, const float *,
                               const float *, int, const int32_t *, const float *, int, int, float, float *, size_t,
                               cudaStream_t);
size_t spec_compare_smem_bytes(int method, int64_t max_short);
cudaError_t launch_spec_compare(const float *, const float *, const void *, int, int, int, double, int64_t, double *,
                                cudaStream_t);
size_t cepstra_smem_bytes(int n_in, int n_ceps, int order, int dn);
cudaError_t launch_cepstra(const CepsTile *, int, const CepsRow *, const float *, const float *, float *, int, int, int,
                           int, cudaStream_t);
cudaError_t launch_f0_track(const sgb_syllable *, int, const SylCtrl *, const Pools &, F0Epochs *, const F0Chunk *, int,
                            const int64_t *, const int64_t *, const F0Span *, float *, cudaStream_t);
cudaError_t launch_f0_frames(const F0Seg *, int, const F0Row *, const float *, int, double, float *, cudaStream_t);
void launch_noise_final(const sgb_noise *, int, const NoiseLayout *, const double *, const double *, const int *, int,
                        const float *, float *, void *, double *, const int64_t *, int, cudaStream_t);
size_t contour_tab_bytes();
void launch_sound_mix(const sgb_bout *, int, const BoutLayout *, const sgb_noise *, const NoiseLayout *,
                      const double *, const float *, float *, void *, double *, const int64_t *, bool, int, cudaStream_t);
void launch_finalize(int, const sgb_bout *, int, const BoutLayout *, const sgb_noise *, const NoiseLayout *,
                     const float *, const float *, const float *, const int *, void *, int, cudaStream_t);

int stft_timeout_flag();
int *compose_debug_buffer();
// ------------------------------------------------------------------ errors ---
static thread_local std::string g_err;
static int g_synth_min_rows_override = -1;      // sgb_synth_min_rows_set
static int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  if (code == SGB_ERR_CUDA) {   // a trapped search left its diagnostics in mapped host memory
    int *d = compose_debug_buffer();
    if (d && d[0] > 0) {
      char t[160];
      int n = d[0] < 400 ? d[0] : 400;
      snprintf(t, sizeof t, " | k_compose diagnostics: %d records", d[0]);
      g_err += t;
      for (int i = 0; i < n && i < 24; i++) {
        int *r = d + 8 + i * 10;
        snprintf(t, sizeof t, " [loop %d syl %d ep %d tid %d: %d %d %d %d %d]", r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[8]);
        g_err += t;
      }
    }
  }
  return code;
}
#define CK(call)                                                                               \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      cudaGetLastError();   /* a reported error must not resurface in a later, unrelated call */ \
      return fail(SGB_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
    }                                                                                          \
  } while (0)

// a launch with an invalid configuration only shows in cudaGetLastError(): name the kernel instead of letting
// the next checked call inherit it
#define CKL(what)                                                                                   \
  do {                                                                                              \
    cudaError_t e_ = cudaGetLastError();                                                            \
    if (e_ != cudaSuccess) return fail(SGB_ERR_CUDA, "%s: launch failed: %s", what, cudaGetErrorString(e_)); \
  } while (0)

struct SylSummary { int32_t status, out_len, n_up, nGC, z_used, pad; };
__global__ void k_summary(const SylCtrl *ctrl, int S, SylSummary *out) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  out[s].status = ctrl[s].status; out[s].out_len = ctrl[s].out_len; out[s].n_up = ctrl[s].n_up; out[s].nGC = ctrl[s].nGC;
  out[s].z_used = ctrl[s].z_used; out[s].pad = 0;
}
__global__ void k_fill_int(int *p, int n, int v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
__global__ void k_f32_to_f64(const float *a, double *b, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) b[i] = (double)a[i];
}
__global__ void k_f64_to_f32(const double *a, float *b, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) b[i] = (float)a[i];
}

// ---------------------------------------------------------------- buffers ---
struct DBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

// grow-only page-locked host buffer: small device -> host results land here so that their copies are
// truly asynchronous and the waiting thread can sleep (wait_stream) instead of spinning in a staged copy
struct HBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

// Staging of the device-output exports (sgb_batch_export / sgb_rows_export): the per-row table and the (row, chunk)
// grid travel from pinned host memory to the device.  A slot is reused only once the event recorded after its
// kernel has passed, checked with cudaEventQuery: an export never waits on the host for an earlier one (which may
// itself still wait on the caller's stream); a new slot is added while all are in flight.
struct ExportSlot {
  HBuf h;
  DBuf d;
  cudaEvent_t done = nullptr;
};
struct ExportCtx {
  std::vector<ExportSlot *> slots;
  cudaEvent_t ev_in = nullptr;
  ~ExportCtx() {
    for (auto s : slots) { s->h.release(); s->d.release(); if (s->done) cudaEventDestroy(s->done); delete s; }
    if (ev_in) cudaEventDestroy(ev_in);
  }
};

static int64_t align4(int64_t x) { return (x + 3) & ~(int64_t)3; }

// seq(from, to, by) length: floor((to-from)/by + 1e-10) + 1
static int seq_by_count(double from, double to, double by) {
  if (from == to) return 1;
  return (int)std::floor((to - from) / by + 1e-10) + 1;
}

struct RunState;
struct sgb_batch {
  int device = 0;
  cudaStream_t st = nullptr;
  cudaEvent_t ev[SGB_T_COUNT + 2];
  cudaEvent_t ev_wait = nullptr;   // blocking-sync event: the host thread sleeps instead of spinning (see wait_stream)
  bool have_desc = false, have_run = false;
  // host copies of the small tables
  std::vector<sgb_call> calls;
  std::vector<sgb_bout> bouts;
  std::vector<sgb_syllable> syls;
  std::vector<sgb_noise> noises;
  std::vector<sgb_envelope> envs;
  std::vector<sgb_formant_ref> frefs;
  std::vector<double> h_anchors;   // host copy of the anchor pool (contour_fits)
  int64_t n_pitch = 0, n_anchors = 0, n_formants = 0, n_z = 0, n_u = 0, n_pre = 0;
  int u_is_float = 0;
  // device copies
  DBuf d_bouts, d_syls, d_noises, d_envs, d_frefs, d_pitch, d_anchors, d_formants, d_z, d_u, d_pre;
  DBuf d_gc_off, d_h_off, d_ctrl, d_lay, d_totals, d_summary, d_tiles, d_epmax;
  DBuf p_pitch_w, p_i32[6], p_f64[19], p_pc;
  HBuf h_tot, h_summary, h_lay;   // pinned landing zones of the two mid-run read-backs
  HBuf h_calltab;
  DBuf d_pcm, d_calltab;
  DBuf d_amp, d_amp32, d_wave, d_raw, d_sound, d_voiced, d_filt, d_noise_raw, d_noise_fin, d_env, d_out, d_out64;
  DBuf d_trk, d_mouth, d_formants_late, d_tiles_tc, d_ntabs, d_order, d_mtabs;
  DBuf d_knots, d_koff, d_ctab, d_btabs, d_envk;   // contour knot pool, per-contour offsets, headers (contour.cuh)
  DBuf d_f0ep;                                     // K6's epoch spans replayed for the f0 track (sgb_batch_f0)
  int64_t knot_total = 0;
  bool any_aglobal = false;
  struct RunState *rs = nullptr;     // state carried from run_begin to run_finish
  std::vector<double> late_rows;     // host-drawn formant tracks set between begin and finish
  std::vector<int32_t> h_order;
  bool ctrl_dense = false;
  std::vector<int> late_envs;        // the envelopes they belong to (deferred again at the next run_begin)
  size_t n_frefs_uploaded = 0;
  bool envs_dirty = false;
  DBuf d_bl, d_place, d_nl, d_envinst, d_plans, d_tw, d_win, d_fjobs, d_njobs, d_fsegs, d_nsegs, d_max;
  Pools pools;
  int64_t gc_total = 0, h_total = 0;
  // results
  std::vector<SylSummary> summary;
  std::vector<BoutLayout> bl;
  std::vector<SylPlace> place;
  std::vector<NoiseLayout> nl;
  std::vector<SylLayout> lay_host;
  std::vector<int64_t> call_len, call_off;
  std::vector<int32_t> call_status;
  int64_t total_out = 0;
  int64_t last_amp = 0, last_wave = 0, last_raw = 0, last_tiles = 0, last_sound = 0;
  int last_tc_min_rows = 0;          // K1 dispatch threshold of the last run (the FP32 table's layout per epoch)
  volatile int where = 0;   // progress marker for sgb_batch_debug_state: which wait the host thread is in
  volatile int reached[16] = {0};   // SGB_TRACE=1: stage events the stream has passed (set by host callbacks)
  struct Mark { volatile int *dst; } marks[16];
  bool keep_voiced = false;
  sgb_run_info info;
  ExportCtx *xo = nullptr;           // device-output staging, made on the first export
};

// SGB_TRACE=1: a host callback after every stage records how far the stream got, readable without any
// CUDA call (sgb_batch_debug_state) when a run is stuck.
static const bool g_trace = getenv("SGB_TRACE") != nullptr;
static void CUDART_CB trace_cb(void *p) { *reinterpret_cast<volatile int *>(p) = 1; }
static void trace_mark(sgb_batch *b, int i) {
  if (!g_trace) return;
  cudaLaunchHostFunc(b->st, trace_cb, (void *)&b->reached[i]);
}

// 16-bit PCM of every call's waveform as seewave::savewav writes it (soundgen.R:855-857, seewave.r:5192-5229
// -> tuneR::normalize(unit = "16", level = min(1, max(x))), tuneR normalize.R): centre, scale the largest
// magnitude to `level`, round(x * 32767).  One CTA per row (the whole-row reductions come first); reductions in a
// fixed order (reproducible).  Row r: statistics over its len[r] samples at src + src_off[r]; written: exactly
// cap[r] elements from dst + dst_off[r], the first min(len, cap) samples and then zeros.  The host fetch passes
// dst_off = src_off and cap = len.
__global__ void __launch_bounds__(256)
k_pcm16(const float *__restrict__ src, const int64_t *__restrict__ src_off, const int64_t *__restrict__ len,
        const int64_t *__restrict__ dst_off, const int64_t *__restrict__ cap, int16_t *__restrict__ dst) {
  __shared__ double rs[8], rm[8], ra[8];
  const int64_t n = len[blockIdx.x], c = cap[blockIdx.x], m = n < c ? n : c;
  const float *x = src + src_off[blockIdx.x];
  int16_t *y = dst + dst_off[blockIdx.x];
  double mean = 0.0, am = 0.0, level = 0.0;
  if (n > 0) {                                   // uniform over the CTA
    double sum = 0.0, mx = -INFINITY;
    for (int64_t i = threadIdx.x; i < n; i += 256) { double v = (double)x[i]; sum += v; mx = fmax(mx, v); }
    for (int o = 16; o > 0; o >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, o); mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
    if ((threadIdx.x & 31) == 0) { rs[threadIdx.x >> 5] = sum; rm[threadIdx.x >> 5] = mx; }
    __syncthreads();
    sum = 0.0; mx = -INFINITY;
    for (int w = 0; w < 8; w++) { sum += rs[w]; mx = fmax(mx, rm[w]); }
    mean = sum / (double)n;
    for (int64_t i = threadIdx.x; i < n; i += 256) am = fmax(am, fabs((double)x[i] - mean));
    for (int o = 16; o > 0; o >>= 1) am = fmax(am, __shfl_xor_sync(0xffffffffu, am, o));
    if ((threadIdx.x & 31) == 0) ra[threadIdx.x >> 5] = am;
    __syncthreads();
    am = 0.0;
    for (int w = 0; w < 8; w++) am = fmax(am, ra[w]);
    level = (mx <= 1.0) ? mx : 1.0;
  }
  const bool scale = fabs(am) > 1.5e-8;          // !isTRUE(all.equal(m, 0))
  for (int64_t i = threadIdx.x; i < m; i += 256) {
    double v = (double)x[i] - mean;
    if (scale) v = level * v / am;
    v = rint(v * 32767.0);
    y[i] = (int16_t)fmin(32767.0, fmax(-32768.0, v));
  }
  for (int64_t i = m + threadIdx.x; i < c; i += 256) y[i] = 0;
}

// Float32 rows into caller-owned device memory.  Rows run from 50 ms to many seconds, so the grid is a host-built
// table of (row, chunk) pairs, EXPORT_CHUNK elements each, not one CTA per row.  Chunk k of row r writes elements
// [k * EXPORT_CHUNK, min(cap, (k + 1) * EXPORT_CHUNK)) of the row: the source sample below min(len, cap), else 0.
// Calls are packed back to back with no alignment, so neither side is 16-byte aligned in general: scalar accesses,
// every thread's 32 loads in flight before its stores.
constexpr int EXPORT_THREADS = 256, EXPORT_PER_THREAD = 32, EXPORT_CHUNK = EXPORT_THREADS * EXPORT_PER_THREAD;
__global__ void __launch_bounds__(EXPORT_THREADS)
k_export_f32(const float *__restrict__ src, const int64_t *__restrict__ src_off, const int64_t *__restrict__ len,
             const int64_t *__restrict__ dst_off, const int64_t *__restrict__ cap, const int2 *__restrict__ tab,
             float *__restrict__ dst) {
  const int2 t = tab[blockIdx.x];
  const int64_t c = cap[t.x], n = len[t.x], m = n < c ? n : c;
  const int64_t b0 = (int64_t)t.y * EXPORT_CHUNK + threadIdx.x;
  const float *x = src + src_off[t.x];
  float *y = dst + dst_off[t.x];
  float v[EXPORT_PER_THREAD];
#pragma unroll
  for (int k = 0; k < EXPORT_PER_THREAD; k++) {
    const int64_t i = b0 + (int64_t)k * EXPORT_THREADS;
    v[k] = i < m ? __ldcs(x + i) : 0.0f;         // read once: streaming load
  }
#pragma unroll
  for (int k = 0; k < EXPORT_PER_THREAD; k++) {
    const int64_t i = b0 + (int64_t)k * EXPORT_THREADS;
    if (i < c) y[i] = v[k];
  }
}

// position-weighted checksum of a word array (diagnostics)
__global__ void k_checksum(const uint32_t *p, size_t n, unsigned long long *out) {
  unsigned long long a = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    a += (unsigned long long)p[i] * (unsigned long long)((i % 1000003u) + 1u);
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, a);
}

// Waits for everything queued on the handle's stream WITHOUT spinning: with several handles driven by
// several host threads (and one process per GPU) a spinning cudaStreamSynchronize per thread oversubscribes
// the host cores; a blocking-sync event lets the thread sleep until the stream gets there.
static cudaError_t wait_stream(sgb_batch *b) {
  cudaError_t e = cudaEventRecord(b->ev_wait, b->st);
  if (e != cudaSuccess) return e;
  return cudaEventSynchronize(b->ev_wait);
}

int sgb_fail_msg(int code, const char *msg) { return fail(code, "%s", msg); }

extern "C" {

int sgb_version(void) { return SGB_VERSION; }
const char *sgb_last_error(void) { return g_err.c_str(); }

int sgb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
int sgb_set_device(int device) {
  CK(cudaSetDevice(device));
  return SGB_OK;
}

int sgb_device_pci_bus_id(int device, char *out, int cap) {
  if (!out || cap < 16) return fail(SGB_ERR_INVALID, "bad buffer");
  CK(cudaDeviceGetPCIBusId(out, cap, device));
  return SGB_OK;
}

int sgb_pin(void *ptr, int64_t bytes) {
  if (!ptr || bytes <= 0) return fail(SGB_ERR_INVALID, "bad buffer");
  cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault);
  if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return SGB_OK; }   // pinning is idempotent
  CK(e);
  return SGB_OK;
}
int sgb_unpin(void *ptr) {
  if (!ptr) return fail(SGB_ERR_INVALID, "bad buffer");
  CK(cudaHostUnregister(ptr));
  return SGB_OK;
}
int sgb_measure_fp32_peak(double *out_tflops) {
  if (!out_tflops) return fail(SGB_ERR_INVALID, "null argument");
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  DBuf d;
  CK(d.ensure(sizeof(float2) * 1024));
  CK(cudaMemset(d.p, 0, sizeof(float2) * 1024));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  const int iters = 4096, blocks = sms * 8, threads = 256;
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    CK(cudaEventRecord(e0));
    launch_fp32_peak(d.as<float2>(), iters, blocks, threads);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    // 8 independent FFMA2 chains x 2 lanes x 2 flop per iteration per thread
    double flop = (double)blocks * threads * (double)iters * 8.0 * 2.0 * 2.0;
    best = std::max(best, flop / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  d.release();
  *out_tflops = best;
  return SGB_OK;
}

int sgb_batch_create(sgb_batch **out) {
  compose_debug_buffer();
  if (!out) return fail(SGB_ERR_INVALID, "null out pointer");
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n < 1)
    return fail(SGB_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
  sgb_batch *b = new sgb_batch();
  for (auto &e : b->ev) e = nullptr;
  auto init = [&]() -> int {
    CK(cudaGetDevice(&b->device));
    CK(cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking));
    for (auto &e : b->ev) CK(cudaEventCreate(&e));
    CK(cudaEventCreateWithFlags(&b->ev_wait, cudaEventBlockingSync | cudaEventDisableTiming));
    return SGB_OK;
  };
  int rc = init();
  if (rc != SGB_OK) {            // do not leak a half-built handle
    for (auto &e : b->ev) if (e) cudaEventDestroy(e);
    if (b->ev_wait) cudaEventDestroy(b->ev_wait);
    if (b->st) cudaStreamDestroy(b->st);
    delete b;
    return rc;
  }
  memset(&b->info, 0, sizeof b->info);
  *out = b;
  return SGB_OK;
}

void sgb_batch_destroy(sgb_batch *b) {
  if (!b) return;
  cudaSetDevice(b->device);
  wait_stream(b);
  DBuf *all[] = {&b->d_bouts, &b->d_syls, &b->d_noises, &b->d_envs, &b->d_frefs, &b->d_pitch, &b->d_anchors,
                 &b->d_formants, &b->d_z, &b->d_u, &b->d_pre, &b->d_gc_off, &b->d_h_off, &b->d_ctrl, &b->d_lay,
                 &b->d_totals, &b->d_summary, &b->d_tiles, &b->d_epmax, &b->p_pitch_w, &b->d_amp, &b->d_amp32, &b->d_wave, &b->d_raw,
                 &b->d_sound, &b->d_voiced, &b->d_filt, &b->d_noise_raw, &b->d_noise_fin, &b->d_env, &b->d_out,
                 &b->d_out64, &b->d_bl, &b->d_place, &b->d_nl, &b->d_envinst, &b->d_plans, &b->d_tw, &b->d_win,
                 &b->d_fjobs, &b->d_njobs, &b->d_fsegs, &b->d_nsegs, &b->d_max, &b->d_trk, &b->d_mouth, &b->d_formants_late, &b->d_tiles_tc, &b->d_ntabs, &b->d_order, &b->d_mtabs,
                 &b->d_knots, &b->d_koff, &b->d_ctab, &b->d_btabs, &b->d_envk, &b->d_f0ep};
  for (auto d : all) d->release();
  for (auto &d : b->p_i32) d.release();
  for (auto &d : b->p_f64) d.release();
  b->p_pc.release();
  b->h_tot.release(); b->h_summary.release(); b->h_lay.release(); b->h_calltab.release();
  b->d_pcm.release(); b->d_calltab.release();
  delete b->xo;                    // after wait_stream: no export of this handle is in flight
  delete b->rs;
  for (auto &e : b->ev) cudaEventDestroy(e);
  if (b->ev_wait) cudaEventDestroy(b->ev_wait);
  cudaStreamDestroy(b->st);
  delete b;
}

static int upload_array(sgb_batch *b, DBuf &d, const void *src, size_t bytes) {
  CK(d.ensure(bytes ? bytes : 16));
  if (bytes) CK(cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, b->st));
  return SGB_OK;
}

int sgb_batch_upload(sgb_batch *b, const sgb_batch_desc *D) {
  if (!b || !D) return fail(SGB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(b->device));
  if (D->n_calls < 1 || D->n_bouts < 1 || D->n_syllables < 1)
    return fail(SGB_ERR_INVALID, "empty batch");
  // ---- validate ----
  for (int c = 0; c < D->n_calls; c++) {
    const sgb_call &C = D->calls[c];
    if (C.bout_begin < 0 || C.bout_end > D->n_bouts || C.bout_begin >= C.bout_end)
      return fail(SGB_ERR_INVALID, "call %d: bad bout range", c);
  }
  for (int i = 0; i < D->n_bouts; i++) {
    const sgb_bout &B = D->bouts[i];
    if (B.syl_begin < 0 || B.syl_end > D->n_syllables || B.syl_begin >= B.syl_end)
      return fail(SGB_ERR_INVALID, "bout %d: bad syllable range", i);
    if (B.noise_begin < 0 || B.noise_end > D->n_noises || B.noise_begin > B.noise_end)
      return fail(SGB_ERR_INVALID, "bout %d: bad noise range", i);
    if (B.env_id < 0 || B.env_id >= D->n_envelopes) return fail(SGB_ERR_INVALID, "bout %d: bad env_id", i);
    if (B.wl < 4) return fail(SGB_ERR_INVALID, "bout %d: windowLength_points %d < 4", i, B.wl);
    if (!(B.overlap >= 0.0 && B.overlap < 100.0)) return fail(SGB_ERR_INVALID, "bout %d: overlap out of range", i);
    if (!(B.samplingRate > 0)) return fail(SGB_ERR_INVALID, "bout %d: samplingRate", i);
    if (B.aglobal_n < 0 || (B.aglobal_n > 0 && (B.aglobal_off < 0 || B.aglobal_off + B.aglobal_n > D->n_anchors)))
      return fail(SGB_ERR_INVALID, "bout %d: amplAnchorsGlobal range outside the anchor pool", i);
    if (!(B.throwaway < 0)) return fail(SGB_ERR_INVALID, "bout %d: throwaway must be negative", i);
  }
  for (int s = 0; s < D->n_syllables; s++) {
    const sgb_syllable &Y = D->syllables[s];
    if (Y.kind < 0 || Y.kind > 2) return fail(SGB_ERR_INVALID, "syllable %d: bad kind", s);
    if (Y.kind == 0) { if (Y.silent_len < 0) return fail(SGB_ERR_INVALID, "syllable %d: silent_len", s); continue; }
    const bool dev_pitch = (Y.kind == 1 && Y.pitch_anchor_n > 0);
    if (Y.pitch_len < 1 || Y.pitch_off < 0 || (!dev_pitch && Y.pitch_off + Y.pitch_len > D->n_pitch))
      return fail(SGB_ERR_INVALID, "syllable %d: pitch range outside the pool", s);
    if (Y.kind == 1 && Y.pitch_anchor_n != 0) {
      if (Y.pitch_anchor_n < 0 || Y.pitch_anchor_off < 0 || Y.pitch_anchor_off + Y.pitch_anchor_n > D->n_anchors)
        return fail(SGB_ERR_INVALID, "syllable %d: pitchAnchors range outside the anchor pool", s);
    }
    if (Y.kind == 2) continue;
    if (Y.pitch_len < 3) return fail(SGB_ERR_INVALID, "syllable %d: pitch contour shorter than 3 points", s);
    if (!(Y.samplingRate > 0) || !(Y.pitchSamplingRate > 0) || !(Y.pitchFloor > 0) || !(Y.pitchCeiling >= Y.pitchFloor))
      return fail(SGB_ERR_INVALID, "syllable %d: sampling rates / pitch bounds", s);
    if (Y.z_cap < 0 || Y.z_off < 0 || Y.z_off + Y.z_cap > D->n_z) return fail(SGB_ERR_INVALID, "syllable %d: z range", s);
    if (Y.ampl_n < 0 || (Y.ampl_n > 0 && (Y.ampl_off < 0 || Y.ampl_off + Y.ampl_n > D->n_anchors)))
      return fail(SGB_ERR_INVALID, "syllable %d: amplAnchors range", s);
    if (!(Y.throwaway < 0)) return fail(SGB_ERR_INVALID, "syllable %d: throwaway must be negative", s);
  }
  for (int n = 0; n < D->n_noises; n++) {
    const sgb_noise &N = D->noises[n];
    if (N.len < 1) return fail(SGB_ERR_INVALID, "noise %d: len < 1", n);
    if (N.wl < 4 || (N.wl & 1)) return fail(SGB_ERR_UNSUPPORTED, "noise %d: odd or tiny window", n);
    if (N.env_id >= D->n_envelopes) return fail(SGB_ERR_INVALID, "noise %d: env_id", n);
    if (N.strength_pre_off < 0 && (N.anchor_n < 1 || N.anchor_off < 0 || N.anchor_off + N.anchor_n > D->n_anchors))
      return fail(SGB_ERR_INVALID, "noise %d: anchors", n);
    if (N.strength_pre_off >= 0 && N.strength_pre_off + N.len > D->n_pre) return fail(SGB_ERR_INVALID, "noise %d: pre-evaluated contour range", n);
    double h = N.wl - (N.overlap * N.wl / 100.0);
    if (!(h >= 1.0)) return fail(SGB_ERR_INVALID, "noise %d: hop < 1", n);
    int nc = seq_by_count(1.0, (double)N.len + N.wl, h);
    if (N.u_off < 0 || N.u_off + (int64_t)nc * (N.wl / 2) > D->n_u)
      return fail(SGB_ERR_STREAM, "noise %d: needs %lld uniforms", n, (long long)nc * (N.wl / 2));
  }
  for (int e = 0; e < D->n_envelopes; e++) {
    const sgb_envelope &E = D->envelopes[e];
    if (E.n_formants < 0 || E.n_formants > SGB_MAX_FORMANTS)
      return fail(SGB_ERR_UNSUPPORTED, "envelope %d: %d formants (at most %d)", e, E.n_formants, SGB_MAX_FORMANTS);
    if (E.n_formants > 0 && (E.formant_off < 0 || E.formant_off + E.n_formants > D->n_formant_refs))
      return fail(SGB_ERR_INVALID, "envelope %d: formant refs", e);
    if (E.mouth_n < 0 || (E.mouth_n > 0 && (E.mouth_off < 0 || E.mouth_off + E.mouth_n > D->n_anchors)))
      return fail(SGB_ERR_INVALID, "envelope %d: mouthAnchors range outside the anchor pool", e);
    if (E.tracks_given < 0 || E.tracks_given > 3) return fail(SGB_ERR_INVALID, "envelope %d: tracks_given", e);
    if (E.tracks_given == 2) {
      if (E.nc_fixed < 1 || E.formant_off < 0) return fail(SGB_ERR_INVALID, "envelope %d: literal filter matrix needs nc_fixed >= 1", e);
    } else if (E.n_formants > 0) {
      int np = 0;
      for (int f = 0; f < E.n_formants; f++) {
        const sgb_formant_ref &R = D->formant_index[E.formant_off + f];
        np = std::max(np, (int)R.n);
        if (E.tracks_given == 1 && E.nc_fixed > 0 && R.n < E.nc_fixed)
          return fail(SGB_ERR_INVALID, "envelope %d: formant %d has %d track rows for %d columns", e, f, R.n, E.nc_fixed);
      }
      if (E.tracks_given == 0 && np > 1 && !(E.smoothLinearFactor <= 20.0))    // 2^20 knots per track
        return fail(SGB_ERR_UNSUPPORTED, "envelope %d: smoothLinearFactor above 20", e);
    }
  }
  for (int f = 0; f < D->n_formant_refs; f++) {
    const sgb_formant_ref &R = D->formant_index[f];
    if (R.n < 1 || R.off < 0 || R.off + R.n > D->n_formants) return fail(SGB_ERR_INVALID, "formant ref %d", f);
  }

  b->calls.assign(D->calls, D->calls + D->n_calls);
  b->bouts.assign(D->bouts, D->bouts + D->n_bouts);
  b->syls.assign(D->syllables, D->syllables + D->n_syllables);
  b->noises.assign(D->noises, D->noises + D->n_noises);
  b->envs.assign(D->envelopes, D->envelopes + D->n_envelopes);
  b->frefs.assign(D->formant_index, D->formant_index + D->n_formant_refs);
  b->h_anchors.assign(D->anchors, D->anchors + 2 * D->n_anchors);
  if (b->h_anchors.empty()) b->h_anchors.assign(2, 0.0);
  b->n_pitch = D->n_pitch; b->n_anchors = D->n_anchors; b->n_formants = D->n_formants;
  b->n_z = D->n_z; b->n_u = D->n_u; b->n_pre = D->n_pre; b->u_is_float = D->u_is_float;
  const int S = D->n_syllables;

  CK(cudaEventRecord(b->ev[SGB_T_COUNT], b->st));
  int rc;
  if ((rc = upload_array(b, b->d_bouts, D->bouts, sizeof(sgb_bout) * D->n_bouts))) return rc;
  if ((rc = upload_array(b, b->d_syls, D->syllables, sizeof(sgb_syllable) * S))) return rc;
  {   // K0 runs one warp per syllable and its time grows with the pitch contour: longest first, so that a long
      // syllable scheduled last does not become the kernel's tail (a preset sweep mixes 50 ms and 3 s syllables)
    std::vector<int32_t> &order = b->h_order;     // a member: the copy below is asynchronous
    order.resize((size_t)S);
    for (int s = 0; s < S; s++) order[s] = s;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t c) {
      const int la = b->syls[a].kind == 1 ? b->syls[a].pitch_len : 0, lc = b->syls[c].kind == 1 ? b->syls[c].pitch_len : 0;
      return la > lc;
    });
    if ((rc = upload_array(b, b->d_order, order.data(), sizeof(int32_t) * (size_t)S))) return rc;
    // K0 variant: with no syllable longer than twice the mean, more resident syllables beat fewer registers
    int64_t sum_len = 0; int max_len = 0, nv = 0;
    for (int s = 0; s < S; s++)
      if (b->syls[s].kind == 1) { sum_len += b->syls[s].pitch_len; max_len = std::max(max_len, (int)b->syls[s].pitch_len); nv++; }
    b->ctrl_dense = nv >= 2048 && (int64_t)max_len * nv <= 2 * sum_len;
  }
  if ((rc = upload_array(b, b->d_noises, D->noises, sizeof(sgb_noise) * D->n_noises))) return rc;
  if ((rc = upload_array(b, b->d_envs, D->envelopes, sizeof(sgb_envelope) * D->n_envelopes))) return rc;
  if ((rc = upload_array(b, b->d_frefs, D->formant_index, sizeof(sgb_formant_ref) * D->n_formant_refs))) return rc;
  if ((rc = upload_array(b, b->d_pitch, D->pitch, 8 * (size_t)D->n_pitch))) return rc;
  if ((rc = upload_array(b, b->d_anchors, D->anchors, 16 * (size_t)D->n_anchors))) return rc;
  if ((rc = upload_array(b, b->d_formants, D->formants, 32 * (size_t)D->n_formants))) return rc;
  if ((rc = upload_array(b, b->d_z, D->z, 8 * (size_t)D->n_z))) return rc;
  if ((rc = upload_array(b, b->d_u, D->u, (D->u_is_float ? 4 : 8) * (size_t)D->n_u))) return rc;
  if ((rc = upload_array(b, b->d_pre, D->pre, 8 * (size_t)D->n_pre))) return rc;

  // per-syllable scratch capacities (host-known bounds)
  std::vector<int64_t> gc_off(S + 1), h_off(S + 1);
  int64_t g = 0, h = 0;
  for (int s = 0; s < S; s++) {
    gc_off[s] = g; h_off[s] = h;
    const sgb_syllable &Y = b->syls[s];
    if (Y.kind == 1) {
      g += Y.pitch_len / 2 + 3;
      h += (int64_t)std::ceil((Y.samplingRate / 2.0 - Y.pitchFloor) / Y.pitchFloor) + 2;
    } else {
      g += 1; h += 1;
    }
  }
  gc_off[S] = g; h_off[S] = h;
  b->gc_total = g; b->h_total = h;
  if ((rc = upload_array(b, b->d_gc_off, gc_off.data(), 8 * (size_t)(S + 1)))) return rc;
  if ((rc = upload_array(b, b->d_h_off, h_off.data(), 8 * (size_t)(S + 1)))) return rc;
  // the contour knot pool (contour.cuh): per syllable its pitch and two amplitude contours, then per noise its
  // strength contour, then per bout amplAnchorsGlobal; each contour of n anchors owns 5 n doubles
  const int NN = D->n_noises, NB = D->n_bouts;
  std::vector<int64_t> koff((size_t)3 * S + NN + NB);
  int64_t kt = 0;
  b->any_aglobal = false;
  for (int s = 0; s < S; s++) {
    const sgb_syllable &Y = b->syls[s];
    const int na[3] = {Y.kind == 1 ? Y.pitch_anchor_n : 0, Y.kind == 1 ? Y.ampl_n : 0, Y.kind == 1 ? Y.ampl_n : 0};
    for (int r = 0; r < 3; r++) { koff[3 * (size_t)s + r] = kt; kt += contour_knot_doubles(na[r]); }
  }
  for (int n = 0; n < NN; n++) {
    koff[3 * (size_t)S + n] = kt;
    if (D->noises[n].strength_pre_off < 0) kt += contour_knot_doubles(D->noises[n].anchor_n);
  }
  for (int i = 0; i < NB; i++) {
    koff[3 * (size_t)S + NN + i] = kt;
    kt += contour_knot_doubles(D->bouts[i].aglobal_n);
    if (D->bouts[i].aglobal_n > 0) b->any_aglobal = true;
  }
  b->knot_total = kt;
  if ((rc = upload_array(b, b->d_koff, koff.data(), 8 * koff.size()))) return rc;
  CK(cudaEventRecord(b->ev[SGB_T_COUNT + 1], b->st));
  b->where = 10;
  CK(wait_stream(b));   // gc_off / h_off / koff are stack vectors
  b->where = 0;
  CK(cudaEventElapsedTime(&b->info.ms[SGB_T_H2D], b->ev[SGB_T_COUNT], b->ev[SGB_T_COUNT + 1]));

  int64_t pw = std::max<int64_t>(1, D->n_pitch);   // device-evaluated contours only live in the work pool
  for (int s = 0; s < S; s++)
    if (b->syls[s].kind == 1) pw = std::max<int64_t>(pw, b->syls[s].pitch_off + b->syls[s].pitch_len);
  CK(b->p_pitch_w.ensure(8 * (size_t)pw));
  for (int i = 0; i < 5; i++) CK(b->p_i32[i].ensure(4 * (size_t)g));
  CK(b->p_i32[5].ensure(4 * (size_t)h));
  for (auto &d : b->p_f64) CK(d.ensure(8 * (size_t)g));
  CK(b->p_pc.ensure(8 * (size_t)g * SYNTH_PC));
  Pools &P = b->pools;
  P.pitch_w = b->p_pitch_w.as<double>();
  P.gc = b->p_i32[0].as<int32_t>(); P.nsub = b->p_i32[1].as<int32_t>(); P.rwbin = b->p_i32[2].as<int32_t>();
  P.jidx = b->p_i32[3].as<int32_t>(); P.gcup = b->p_i32[4].as<int32_t>(); P.rowmap = b->p_i32[5].as<int32_t>();
  double **dp[] = {&P.ppg, &P.rw, &P.ro, &P.roct, &P.rk, &P.shimmer, &P.drift, &P.subdep, &P.colmax, &P.kt,
                   &P.sb, &P.sc, &P.sd, &P.phi, &P.t1, &P.t2, &P.t3, &P.t4};
  for (int i = 0; i < 18; i++) *dp[i] = b->p_f64[i].as<double>();
  P.pc = b->p_pc.as<double>();
  P.gc_off = b->d_gc_off.as<int64_t>();
  P.h_off = b->d_h_off.as<int64_t>();
  CK(b->d_knots.ensure(8 * (size_t)std::max<int64_t>(b->knot_total, 1)));
  CK(b->d_ctab.ensure(contour_tab_bytes() * 3 * (size_t)S));
  CK(b->d_btabs.ensure(contour_tab_bytes() * (size_t)D->n_bouts));
  P.ctab = b->d_ctab.as<ContourTab>();
  P.knots = b->d_knots.as<double>();
  P.koff = b->d_koff.as<int64_t>();
  CK(b->d_ctrl.ensure(sizeof(SylCtrl) * (size_t)S));
  CK(b->d_lay.ensure(sizeof(SylLayout) * (size_t)S));
  CK(b->d_totals.ensure(64));
  CK(b->d_summary.ensure(sizeof(SylSummary) * (size_t)S));
  CK(b->d_epmax.ensure(4 * (size_t)S * SGB_MAX_EPOCHS));
  b->late_rows.clear(); b->late_envs.clear(); b->envs_dirty = false;
  b->n_frefs_uploaded = b->frefs.size();
  b->have_desc = true;
  b->have_run = false;
  b->keep_voiced = (D->n_calls <= 64);
  return SGB_OK;
}

// radices for the Stockham passes.  Odd factors go first (largest first): the early passes
// scatter their outputs with stride r, and an odd stride spreads over the shared-memory
// banks where a power of two would collide; by the time the radix-4 / 2 passes run the
// stride s is >= 32 and the accesses are contiguous.
static int plan_radices(int n, int *radix) {
  int np = 0, odd[FFT_MAX_PASS], no = 0;
  int m = n;
  while (m % 2 == 0) m /= 2;
  for (int p = 3; m > 1; p += 2) {
    while (m % p == 0) {
      if (no >= FFT_MAX_PASS) return -1;
      odd[no++] = p; m /= p;
    }
  }
  for (int i = no - 1; i >= 0; i--) radix[np++] = odd[i];
  int pw = n;
  for (int i = 0; i < no; i++) pw /= odd[i];
  while (pw % 4 == 0) { if (np >= FFT_MAX_PASS) return -1; radix[np++] = 4; pw /= 4; }
  while (pw % 2 == 0) { if (np >= FFT_MAX_PASS) return -1; radix[np++] = 2; pw /= 2; }
  if (np >= 2 && radix[np - 2] == 4 && radix[np - 1] == 2) { radix[np - 2] = 8; np--; }   // register radix-8
  return np;
}

struct PlanKey {
  int n; double overlap;
  bool operator<(const PlanKey &o) const { return n < o.n || (n == o.n && overlap < o.overlap); }
};

// A loess contour (3-10 anchors) can fail the way the reference's loess() does ("span is too small"
// after the span-shrinking loop of smoothContours.R:145-152).  The kernels evaluate the contours; the
// host runs the same scalar fit once per contour whose length it knows to learn whether the reference
// call would have stopped.  1, 2 or more than 10 anchors and method 'spline' never fail.
struct FitCheck { int call, na, method, len; double sr, lo, hi; const double *an; };
static bool contour_fits(int na, int method, int len, double samplingRate, bool has_lo, double lo, bool has_hi,
                         double hi, const double *an) {
  if (na < 3 || na > 10 || method != SGB_CONTOUR_LOESS || len < 1) return true;
  ContourTab T;
  double K[5 * 10];
  contour_prepare(&T, K, an, na, len, samplingRate, has_lo, lo, has_hi, hi, false, method);
  return T.status == SGB_OK;
}

// Places an envelope instance's contour knots in the envelope knot pool from doubles `at` on: the mouth-opening
// contour's knots, then per moving formant track (3 per formant) the scratch of k_env_tracks: the nPoints time
// points and values and the 5 arrays of the na = nPoints + 2^smoothLinearFactor knots of approx().  Returns the end.
static int64_t env_knot_layout(EnvInst &I, const sgb_envelope &E, const sgb_formant_ref *refs, int64_t at) {
  I.mouth_koff = -1; I.fit_off = -1;
  if (E.mouth_n > 0) { I.mouth_koff = at; at += contour_knot_doubles(E.mouth_n); }
  if (I.trk_off >= 0 && E.tracks_given == 0) {
    int np = 0;
    for (int f = 0; f < E.n_formants; f++) np = std::max(np, (int)refs[E.formant_off + f].n);
    const int64_t na = (int64_t)std::ceil((double)np + std::exp2(E.smoothLinearFactor)) + 1;  // + 1: exp2 on the device
    I.fit_off = at;
    at += 3 * (int64_t)E.n_formants * (2 * (int64_t)np + 5 * na);
  }
  return at;
}

// FFT plans + twiddle / window tables (seewave hamming.w / hanning.w, seewave.r:7431-7450)
struct PlanTable {
  std::vector<FftPlan> plans;
  std::map<PlanKey, int> idx;
  std::vector<float2> tw;
  std::vector<float> win;
  int get(int n, double overlap) {
    PlanKey key{n, overlap};
    auto it = idx.find(key);
    if (it != idx.end()) return it->second;
    FftPlan pl;
    memset(&pl, 0, sizeof pl);
    pl.n = n;
    pl.npass = plan_radices(n, pl.radix);
    if (pl.npass < 0) return -1;
    pl.h_in = n - (overlap * n / 100.0);
    pl.h_out = n * (100.0 - overlap) / 100.0;
    const size_t t0 = tw.size(), w0 = win.size();
    pl.tw_off = (int64_t)t0; pl.wa_off = (int64_t)w0; pl.ws_off = (int64_t)w0 + n; pl.wh_off = (int64_t)w0 + 2 * n;
    tw.resize(t0 + n);
    win.resize(w0 + 3 * (size_t)n);
    const double two_pi = 2.0 * 3.141592653589793;
    double W0 = 0.0;
    std::vector<double> hann(n);
    for (int i = 0; i < n; i++) {
      double ang = two_pi * (double)i / (double)n;
      tw[t0 + i] = make_float2((float)std::cos(ang), (float)-std::sin(ang));
      double c = std::cos(two_pi * (double)i / (double)(n - 1));
      hann[i] = 0.5 - 0.5 * c;
      W0 += hann[i] * hann[i];
      win[w0 + i] = (float)((0.54 - 0.46 * c) / (double)n);
    }
    for (int i = 0; i < n; i++) win[w0 + n + i] = (float)(hann[i] * pl.h_out / (W0 * (double)n));
    for (int i = 0; i < n; i++) win[w0 + 2 * n + i] = (float)(hann[i] / (double)n);
    plans.push_back(pl);
    idx[key] = (int)plans.size() - 1;
    return (int)plans.size() - 1;
  }
};

// segments: one CTA per sound when there are plenty of sounds, else split runs of frames
// `groups` receives, per compile-time FFT plan (spec), the [begin, end) range of its segments.
struct SegGroup { int spec, begin, end; size_t smem; };
static void make_segs(const std::vector<FftJob> &jobs, const std::vector<FftPlan> &plans, int mode,
                      std::vector<FftSeg> &segs, std::vector<SegGroup> &groups) {
  const int target = 4 * 148;
  int per_job = 1;
  if ((int)jobs.size() < target && !jobs.empty()) per_job = (target + (int)jobs.size() - 1) / (int)jobs.size();
  std::vector<int> spec_of(plans.size());
  for (size_t i = 0; i < plans.size(); i++) spec_of[i] = stft_spec_of(plans[i].n, plans[i].radix, plans[i].npass);
  for (int sp = 0; sp < 7; sp++) {
    SegGroup gr; gr.spec = sp; gr.begin = (int)segs.size(); gr.smem = 0;
    for (int j = 0; j < (int)jobs.size(); j++) {
      if (spec_of[jobs[j].plan] != sp) continue;
      const FftPlan &pl = plans[jobs[j].plan];
      gr.smem = std::max(gr.smem, stft_smem_bytes_spec(pl.n, pl.h_in, pl.h_out, mode, sp));
      int nc = jobs[j].nc;
      int nseg = std::max(1, std::min(per_job, nc / 8));
      int fr = (nc + nseg - 1) / nseg;
      fr += fr & 1;   // keep pairs aligned
      for (int ka = 0; ka < nc; ka += fr) {
        FftSeg sg; sg.job = j; sg.ka = ka; sg.kb = std::min(nc, ka + fr); sg.pad = 0;
        segs.push_back(sg);
      }
    }
    gr.end = (int)segs.size();
    if (gr.end > gr.begin) groups.push_back(gr);
  }
}
// matchLengths(x, len) geometry (R/utilities_math.R:413-444, padDir = 'central')
static void match_lengths(int xlen, int len, int *pad, int *start0) {
  *pad = 0;
  int L = xlen;
  if (xlen == len) { *start0 = 0; return; }
  if (xlen < len) { *pad = len; L = xlen + 2 * len; }
  double halflen = len / 2.0, center = (1 + L) / 2.0;
  *start0 = (int)std::ceil(center - halflen) - 1;
}

struct RunState {
  std::vector<EnvInst> envinst;
  std::vector<FftJob> fjobs, njobs;
  PlanTable PT;
  int64_t sound_total = 0, filt_total = 0, env_total = 0, out_total = 0, noise_total = 0;
  int launches = 0;
  bool begun = false;
};

int sgb_batch_run(sgb_batch *b, sgb_run_info *info_out) {
  int rc = sgb_batch_run_begin(b);
  if (rc != SGB_OK) return rc;
  return sgb_batch_run_finish(b, info_out);
}

int sgb_batch_run_begin(sgb_batch *b) {
  if (!b) return fail(SGB_ERR_INVALID, "null batch");
  if (!b->have_desc) return fail(SGB_ERR_STATE, "sgb_batch_run before sgb_batch_upload");
  if (!b->rs) b->rs = new RunState();
  RunState &R = *b->rs;
  R.begun = false;
  CK(cudaSetDevice(b->device));
  b->have_run = false;           // a failed run must not leave the previous run's results fetchable
  // tracks that arrived during the previous run of this upload: their envelopes wait for new ones again
  for (int e : b->late_envs) b->envs[e].tracks_given = 3;
  b->late_envs.clear(); b->late_rows.clear(); b->frefs.resize(b->n_frefs_uploaded);
  cudaStream_t st = b->st;
  const int S = (int)b->syls.size(), NB = (int)b->bouts.size(), NN = (int)b->noises.size(), NC = (int)b->calls.size();
  sgb_run_info &info = b->info;
  float h2d = info.ms[SGB_T_H2D];
  memset(&info, 0, sizeof info);
  info.ms[SGB_T_H2D] = h2d;
  int launches = 0;
  const Pools &P = b->pools;
  const sgb_syllable *d_syl = b->d_syls.as<sgb_syllable>();
  SylCtrl *d_ctrl = b->d_ctrl.as<SylCtrl>();
  SylLayout *d_lay = b->d_lay.as<SylLayout>();
  int64_t *d_tot = b->d_totals.as<int64_t>();
  cudaEvent_t *ev = b->ev;
  // events: e[0] start, then one after each stage
  if (g_trace) for (int i = 0; i < 16; i++) b->reached[i] = 0;
  CK(cudaEventRecord(ev[0], st)); trace_mark(b, 0);

  // ---- K0 control + size scan ----
  CK(cudaMemsetAsync(d_tot, 0, 64, st));
  static const int tc_min_rows_env = [] {
    const char *e = getenv("SGB_SYNTH");
    if (e && !strcmp(e, "ffma")) return 1 << 30;
    if (e && !strcmp(e, "tc")) return 0;
    const char *m = getenv("SGB_SYNTH_MIN_ROWS");
    return m ? atoi(m) : 224;
  }();
  const int tc_min_rows = g_synth_min_rows_override >= 0 ? g_synth_min_rows_override : tc_min_rows_env;
  synth_min_rows_set(tc_min_rows);
  b->last_tc_min_rows = tc_min_rows;
  launch_control(d_syl, S, b->ctrl_dense, b->d_order.as<int32_t>(), b->d_pitch.as<double>(), b->d_anchors.as<double>(), b->d_z.as<double>(), P, d_ctrl, d_lay,
                 d_tot, st);
  CKL("launch_control");
  launches += 3;
  CK(b->h_tot.ensure(64));
  CK(b->h_summary.ensure(sizeof(SylSummary) * (size_t)S));
  CK(b->h_lay.ensure(sizeof(SylLayout) * (size_t)S));
  int64_t *tot = b->h_tot.as<int64_t>();
  CK(cudaMemcpyAsync(tot, d_tot, 64, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(ev[1], st)); trace_mark(b, 1);
  b->where = 1;
  CK(cudaStreamSynchronize(st));   // short wait on the critical path: spin (the long waits sleep, see wait_stream)
  b->where = 0;
  CK(cudaGetLastError());
  const int64_t amp_total = tot[0], wave_total = tot[1], n_tiles = tot[2], raw_total = tot[3];
  b->last_amp = amp_total; b->last_wave = wave_total; b->last_raw = raw_total; b->last_tiles = n_tiles;
  if (n_tiles > 2000000000LL) return fail(SGB_ERR_UNSUPPORTED, "batch too large: %lld synthesis tiles", (long long)n_tiles);
  CK(b->d_amp.ensure(8 * (size_t)std::max<int64_t>(amp_total, 1)));
  {   // epochs of the tensor-core kernel use the first half of their region ({Y, dY} pairs): a fresh buffer is cleared
      // once so that the unused halves are zeros, not allocator leftovers (sgb_batch_checksums covers the buffer)
    const size_t cap0 = b->d_amp32.cap;
    CK(b->d_amp32.ensure(16 * (size_t)std::max<int64_t>(amp_total, 1)));
    if (b->d_amp32.cap != cap0) CK(cudaMemsetAsync(b->d_amp32.p, 0, b->d_amp32.cap, st));
  }
  CK(b->d_wave.ensure(4 * (size_t)std::max<int64_t>(wave_total, 4)));
  CK(b->d_raw.ensure(4 * (size_t)std::max<int64_t>(raw_total, 4)));
  CK(b->d_tiles.ensure(sizeof(SynthTile) * (size_t)std::max<int64_t>(n_tiles, 1)));

  // ---- K3 amplitude matrices ----
  launch_tiles_amp(d_syl, S, d_ctrl, d_lay, P, b->d_tiles.as<SynthTile>(), d_tot, b->d_amp.as<double>(),
                   b->d_amp32.as<float4>(), st);
  CKL("launch_tiles_amp");
  launches += 2;
  CK(cudaEventRecord(ev[2], st)); trace_mark(b, 2);
  // ---- K1 synthesis ----
  CK(cudaMemsetAsync(b->d_epmax.p, 0, 4 * (size_t)S * SGB_MAX_EPOCHS, st));
  // K1.  Epochs with many rows go to the tensor-core kernel (tcgen05 kind::f16, FP16 hi + lo operands, TMEM
  // accumulators): per 128-sample tile it pays a fixed price (16 trig rows per sample, one MMA round trip per 384
  // rows), which the FP32-pipe kernel of round 1 (blocked Clenshaw on FFMA2, one step per row) undercuts when an
  // epoch has few rows.  SGB_SYNTH=ffma / tc force one kernel; SGB_SYNTH_MIN_ROWS moves the switch.
  const int64_t n_tiles_tc = tot[7];
  if (tc_min_rows < (1 << 30)) {
    if (n_tiles_tc > 2000000000LL) return fail(SGB_ERR_UNSUPPORTED, "batch too large: %lld synthesis units", (long long)n_tiles_tc);
    CK(b->d_tiles_tc.ensure(sizeof(TcUnit) * (size_t)std::max<int64_t>(n_tiles_tc, 1)));
    launch_build_tiles_tc(d_syl, d_ctrl, S, d_lay, P, b->d_tiles_tc.as<TcUnit>(), st);
    CKL("launch_build_tiles_tc");
    CK(launch_synth_tc(b->d_tiles_tc.as<TcUnit>(), (int)n_tiles_tc, P, b->d_amp32.as<float4>(), b->d_wave.as<float>(),
                       b->d_epmax.as<int>(), st));
    if (n_tiles_tc > 0) launches += 2;
  }
  if (tc_min_rows > 0) {
    launch_synth(b->d_tiles.as<SynthTile>(), (int)n_tiles, d_syl, d_ctrl, d_lay, P, b->d_amp32.as<float4>(),
                 b->d_wave.as<float>(), b->d_epmax.as<int>(), st);
    CKL("launch_synth");
    if (n_tiles > 0) launches++;
  }
  CK(cudaEventRecord(ev[3], st)); trace_mark(b, 3);
  // ---- K6 compose ----
  launch_compose(d_syl, S, d_ctrl, d_lay, P, b->d_amp.as<double>(), b->d_wave.as<float>(), b->d_raw.as<float>(),
                 b->d_anchors.as<double>(), b->d_pitch.as<double>(), b->d_epmax.as<int>(), st);
  CKL("launch_compose");
  k_summary<<<(S + 255) / 256, 256, 0, st>>>(d_ctrl, S, b->d_summary.as<SylSummary>());
  launches += 2;
  b->summary.resize(S);
  b->lay_host.resize(S);
  CK(cudaMemcpyAsync(b->h_summary.p, b->d_summary.p, sizeof(SylSummary) * (size_t)S, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(b->h_lay.p, d_lay, sizeof(SylLayout) * (size_t)S, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(tot, d_tot, 64, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(ev[4], st)); trace_mark(b, 4);
  b->where = 2;
  CK(cudaStreamSynchronize(st));
  b->where = 0;
  CK(cudaGetLastError());
  memcpy(b->summary.data(), b->h_summary.p, sizeof(SylSummary) * (size_t)S);
  memcpy(b->lay_host.data(), b->h_lay.p, sizeof(SylLayout) * (size_t)S);
  info.synth_partials = tot[4];
  info.synth_samples = tot[5];

  // ---- host layout (soundgen.R:632-640, 708-714, 743-748, 813-818, 836-849) ----
  b->bl.assign(NB, BoutLayout());
  b->place.assign(S, SylPlace());
  b->nl.assign(NN, NoiseLayout());
  b->call_len.assign(NC, 0); b->call_off.assign(NC, 0); b->call_status.assign(NC, SGB_OK);
  std::vector<EnvInst> &envinst = R.envinst;
  std::vector<FftJob> &fjobs = R.fjobs, &njobs = R.njobs;
  envinst.clear(); fjobs.clear(); njobs.clear();
  R.PT = PlanTable();
  PlanTable &PT = R.PT;
  int64_t sound_total = 0, filt_total = 0, env_total = 0, out_total = 0, noise_total = 0;
  int n_failed = 0;

  auto get_plan = [&](int n, double overlap) -> int { return PT.get(n, overlap); };
  // what an envelope instance of nr x nc reads from the pools must lie inside them (a malformed description
  // must fail its call, not read out of bounds on the device)
  auto env_ok = [&](const sgb_envelope &E, int nr, int nc) -> bool {
    if (E.tracks_given == 2) return E.formant_off >= 0 && E.formant_off + (int64_t)nr * std::max(1, E.nc_fixed) <= b->n_pre;
    if (E.tracks_given == 1)
      for (int f = 0; f < E.n_formants; f++) if (b->frefs[E.formant_off + f].n < nc) return false;
    return true;
  };

  // loess fits that could stop the reference call: collected here, run on the worker threads after the layout
  // (a fit is tens of microseconds of FP64; a preset sweep has three or four per call)
  std::vector<FitCheck> fit_checks;
  auto fit_later = [&](int call, int na, int method, int len, double sr, double lo, double hi, const double *an) {
    if (na < 3 || na > 10 || method != SGB_CONTOUR_LOESS || len < 1) return;
    fit_checks.push_back(FitCheck{call, na, method, len, sr, lo, hi, an});
  };
  std::vector<int64_t> syl_pos, npos, fpos;   // reused across bouts (no allocation per bout)
  for (int c = 0; c < NC; c++) {
    const sgb_call &CL = b->calls[c];
    b->call_off[c] = out_total;
    int64_t clen = 0;
    int wl_running = -1;
    for (int bi = CL.bout_begin; bi < CL.bout_end; bi++) {
      const sgb_bout &B = b->bouts[bi];
      BoutLayout &L = b->bl[bi];
      memset(&L, 0, sizeof L);
      // voiced = c(voiced, syllable, pause)
      syl_pos.assign(B.syl_end - B.syl_begin, 0);
      int64_t vlen = 0;
      bool any_voiced = false;
      for (int s = B.syl_begin; s < B.syl_end; s++) {
        const SylSummary &Y = b->summary[s];
        int len = Y.out_len;
        if (Y.status != SGB_OK) { b->call_status[c] = Y.status; len = 0; }
        else if (b->syls[s].kind != 0 && len > 0) any_voiced = true;
        syl_pos[s - B.syl_begin] = vlen;
        b->place[s].len = len;
        b->place[s].bout = bi;
        vlen += len + b->syls[s].pause_after;
      }
      // pre-filter noise: sound = addVectors(sound, unvoiced[[s]], syllableStartIdx[s])
      int64_t cur = vlen, shift = 0;
      npos.assign(std::max(0, B.noise_end - B.noise_begin), 0);
      bool any_pre = false;
      for (int n = B.noise_begin; n < B.noise_end; n++) {
        const sgb_noise &N = b->noises[n];
        if (N.mix != 0) continue;
        any_pre = true;
        int ip = N.insertion;
        if (ip > 1) { npos[n - B.noise_begin] = ip; cur = std::max<int64_t>(cur, (int64_t)ip + N.len); }
        else if (ip < 1) {
          int64_t pad = 1 - ip;
          shift += pad;
          for (int m = B.noise_begin; m < n; m++) if (b->noises[m].mix == 0) npos[m - B.noise_begin] += pad;
          npos[n - B.noise_begin] = 0;
          cur = std::max<int64_t>(cur + pad, N.len);
        } else { npos[n - B.noise_begin] = 0; cur = std::max<int64_t>(cur, N.len); }
      }
      L.sound_len = (int32_t)cur;
      L.voiced_shift = (int32_t)shift;
      fit_later(c, B.aglobal_n, B.aglobal_method, (int)cur, B.samplingRate, 0.0, -B.throwaway, b->h_anchors.data() + 2 * B.aglobal_off);
      L.sound_off = sound_total;
      for (int s = B.syl_begin; s < B.syl_end; s++) b->place[s].dst_off = L.sound_off + shift + syl_pos[s - B.syl_begin];
      for (int n = B.noise_begin; n < B.noise_end; n++)
        if (b->noises[n].mix == 0) b->nl[n].dst_off = L.sound_off + npos[n - B.noise_begin];
      // filter geometry
      L.bypass = (!any_voiced && !any_pre) ? 1 : 0;   // sum(sound) == 0 (soundgen.R:736)
      if (wl_running < 0) wl_running = B.wl;
      if (!L.bypass) {
        int wl = std::min(wl_running, (int)(cur / 2));     // soundgen.R:743 (persists across bouts)
        wl_running = wl;
        if (wl < 4 || (wl & 1)) {
          b->call_status[c] = SGB_ERR_UNSUPPORTED;
          L.bypass = 1;
        } else {
          L.wl = wl;
          double h_in = wl - (B.overlap * wl / 100.0), h_out = wl * (100.0 - B.overlap) / 100.0;
          L.nc = seq_by_count(1.0, std::max<double>(1.0, (double)(cur - wl)), h_in);
          L.nint = B.moving ? L.nc : 1;
          L.filt_len = (int32_t)std::floor(wl + (L.nc - 1) * h_out);
          L.fft_plan = get_plan(wl, B.overlap);
          if (L.fft_plan < 0) { b->call_status[c] = SGB_ERR_UNSUPPORTED; L.bypass = 1; }
          else if (b->envs[B.env_id].tracks_given != 3 && !env_ok(b->envs[B.env_id], wl / 2, L.nint)) {
            b->call_status[c] = SGB_ERR_INVALID; L.bypass = 1;
          }
        }
      }
      if (L.bypass) { L.filt_len = L.sound_len; L.nc = 0; L.nint = 0; }
      sound_total += align4(cur + 8 + (L.bypass ? 0 : L.wl + 16));
      if (!L.bypass) {
        L.filt_off = filt_total; filt_total += align4(L.filt_len + 4);
        L.env_off = env_total; env_total += align4((int64_t)(L.wl / 2) * L.nint);
        EnvInst I; I.out_off = L.env_off; I.env_id = B.env_id; I.nr = L.wl / 2; I.nc = L.nint; I.col0 = 0; I.trk_off = -1;
        envinst.push_back(I);

        fit_later(c, b->envs[B.env_id].mouth_n, b->envs[B.env_id].mouth_method, L.nint, 16000.0, 0.0, 1.0,
                  b->h_anchors.data() + 2 * b->envs[B.env_id].mouth_off);
        FftJob J; memset(&J, 0, sizeof J);
        J.in_off = L.sound_off; J.out_off = L.filt_off; J.env_off = L.env_off; J.plan = L.fft_plan;
        J.nc = L.nc; J.nint = L.nint; J.xlen = L.filt_len; J.out_len = L.filt_len; J.shift = 0; J.max_slot = bi;
        fjobs.push_back(J);
        info.filter_frames += L.nc;
        info.filter_samples += L.filt_len;
      }
      // post-filter noise: soundFiltered = addVectors(soundFiltered, unvoiced[[s]], syllableStartIdx[s])
      int64_t fcur = L.filt_len, fshift = 0;
      fpos.assign(npos.size(), 0);
      for (int n = B.noise_begin; n < B.noise_end; n++) {
        const sgb_noise &N = b->noises[n];
        if (N.mix != 1) continue;
        int ip = N.insertion;
        if (ip > 1) { fpos[n - B.noise_begin] = ip; fcur = std::max<int64_t>(fcur, (int64_t)ip + N.len); }
        else if (ip < 1) {
          int64_t pad = 1 - ip;
          fshift += pad;
          for (int m = B.noise_begin; m < n; m++) if (b->noises[m].mix == 1) fpos[m - B.noise_begin] += pad;
          fpos[n - B.noise_begin] = 0;
          fcur = std::max<int64_t>(fcur + pad, N.len);
        } else { fpos[n - B.noise_begin] = 0; fcur = std::max<int64_t>(fcur, N.len); }
      }
      L.final_len = (int32_t)fcur;
      L.final_shift = (int32_t)fshift;
      L.out_off = out_total + clen + B.lead_silence;
      for (int n = B.noise_begin; n < B.noise_end; n++)
        if (b->noises[n].mix == 1) b->nl[n].dst_off = L.out_off + fpos[n - B.noise_begin];
      clen += (int64_t)B.lead_silence + fcur + B.tail_silence;
      // noise generation jobs
      for (int n = B.noise_begin; n < B.noise_end; n++) {
        const sgb_noise &N = b->noises[n];
        NoiseLayout &Q = b->nl[n];
        Q.bout = bi;
        Q.raw_off = noise_total; noise_total += align4(N.len + 4);
        double h_in = N.wl - (N.overlap * N.wl / 100.0), h_out = N.wl * (100.0 - N.overlap) / 100.0;
        Q.nc = seq_by_count(1.0, (double)N.len + N.wl, h_in);
        Q.xlen = (int32_t)std::floor(N.wl + (Q.nc - 1) * h_out);
        match_lengths(Q.xlen, N.len, &Q.pad_len, &Q.trim_start);
        if (N.strength_pre_off < 0)
          fit_later(c, N.anchor_n, N.anchor_method, N.len, N.samplingRate, -120.0, 40.0, b->h_anchors.data() + 2 * N.anchor_off);
        Q.fft_plan = get_plan(N.wl, N.overlap);
        Q.env_off = -1; Q.nc_env = 0;
        if (Q.fft_plan < 0) { b->call_status[c] = SGB_ERR_UNSUPPORTED; continue; }
        if (N.env_id >= 0 && !env_ok(b->envs[N.env_id], N.wl / 2, std::max(1, b->envs[N.env_id].nc_fixed))) {
          b->call_status[c] = SGB_ERR_INVALID;        // the noise is generated unfiltered; the call is reported
        } else if (N.env_id >= 0) {
          const sgb_envelope &E = b->envs[N.env_id];
          Q.nc_env = std::max(1, E.nc_fixed);
          Q.env_off = env_total; env_total += align4((int64_t)(N.wl / 2) * Q.nc_env);
          EnvInst I; I.out_off = Q.env_off; I.env_id = N.env_id; I.nr = N.wl / 2; I.nc = Q.nc_env; I.col0 = 0; I.trk_off = -1;
          envinst.push_back(I);
          fit_later(c, E.mouth_n, E.mouth_method, Q.nc_env, 16000.0, 0.0, 1.0, b->h_anchors.data() + 2 * E.mouth_off);
        }
        FftJob J; memset(&J, 0, sizeof J);
        J.in_off = N.u_off; J.out_off = Q.raw_off; J.env_off = Q.env_off; J.plan = Q.fft_plan; J.nc = Q.nc;
        J.nint = Q.nc_env; J.xlen = Q.xlen; J.out_len = N.len; J.shift = Q.trim_start - Q.pad_len;
        J.max_slot = NB + n; J.rolloffNoise = N.rolloffNoise;
        njobs.push_back(J);
        info.noise_samples += N.len;
      }
    }
    b->call_len[c] = clen;
    out_total += clen;          // outputs are packed back to back: one D2H copy fetches them all
  }
  {
    std::vector<char> bad(fit_checks.size(), 0);
    parallel_for((int)fit_checks.size(), [&](int i) {
      const FitCheck &F = fit_checks[i];
      bad[i] = !contour_fits(F.na, F.method, F.len, F.sr, true, F.lo, true, F.hi, F.an);
    });
    for (size_t i = 0; i < bad.size(); i++)
      if (bad[i]) b->call_status[fit_checks[i].call] = SGB_ERR_SYNTH;
  }
  for (int c = 0; c < NC; c++)
    if (b->call_status[c] != SGB_OK) n_failed++;
  b->total_out = out_total;
  info.n_failed = n_failed;
  for (int c = 0; c < NC; c++) info.total_samples += b->call_len[c];
  R.sound_total = sound_total; R.filt_total = filt_total; R.env_total = env_total; R.out_total = out_total;
  R.noise_total = noise_total; R.launches = launches;
  R.begun = true;
  return SGB_OK;
}

int sgb_batch_run_finish(sgb_batch *b, sgb_run_info *info_out) {
  if (!b) return fail(SGB_ERR_INVALID, "null batch");
  if (!b->rs || !b->rs->begun) return fail(SGB_ERR_STATE, "sgb_batch_run_finish before sgb_batch_run_begin");
  RunState &R = *b->rs;
  R.begun = false;
  CK(cudaSetDevice(b->device));
  cudaStream_t st = b->st;
  const int S = (int)b->syls.size(), NB = (int)b->bouts.size(), NN = (int)b->noises.size(), NC = (int)b->calls.size();
  sgb_run_info &info = b->info;
  const Pools &P = b->pools;
  const sgb_syllable *d_syl = b->d_syls.as<sgb_syllable>();
  SylCtrl *d_ctrl = b->d_ctrl.as<SylCtrl>();
  SylLayout *d_lay = b->d_lay.as<SylLayout>();
  cudaEvent_t *ev = b->ev;
  std::vector<EnvInst> &envinst = R.envinst;
  std::vector<FftJob> &fjobs = R.fjobs, &njobs = R.njobs;
  PlanTable &PT = R.PT;
  const int64_t sound_total = R.sound_total, filt_total = R.filt_total, env_total = R.env_total,
                out_total = R.out_total, noise_total = R.noise_total;
  int launches = R.launches;
  for (size_t e = 0; e < b->envs.size(); e++)
    if (b->envs[e].tracks_given == 3) return fail(SGB_ERR_STATE, "envelope %d: deferred formant tracks were never set", (int)e);
  if (b->envs_dirty) {     // host-drawn tracks arrived between begin and finish
    CK(cudaMemcpyAsync(b->d_envs.p, b->envs.data(), sizeof(sgb_envelope) * b->envs.size(), cudaMemcpyHostToDevice, st));
    CK(b->d_frefs.ensure(sizeof(sgb_formant_ref) * b->frefs.size()));
    CK(cudaMemcpyAsync(b->d_frefs.p, b->frefs.data(), sizeof(sgb_formant_ref) * b->frefs.size(), cudaMemcpyHostToDevice, st));
    CK(b->d_formants_late.ensure(8 * std::max<size_t>(b->late_rows.size(), 4)));
    CK(cudaMemcpyAsync(b->d_formants_late.p, b->late_rows.data(), 8 * b->late_rows.size(), cudaMemcpyHostToDevice, st));
    b->envs_dirty = false;
  }

  std::vector<FftSeg> fsegs, nsegs;
  std::vector<SegGroup> fgroups, ngroups;
  make_segs(fjobs, PT.plans, 0, fsegs, fgroups);
  make_segs(njobs, PT.plans, 1, nsegs, ngroups);

  std::vector<FftPlan> &plans = PT.plans;
  std::vector<float2> &tw_host = PT.tw;
  std::vector<float> &win_host = PT.win;
  const int64_t tw_total = (int64_t)tw_host.size(), win_total = (int64_t)win_host.size();
  // ---- upload layout ----
  int max_nc = 0;   // total (instance, column) work items of K4: the kernel runs one warp per item
  int max_f = 0;    // most formants of one of K4's envelopes: sizes its shared memory
  int64_t trk_total = 0, envk_total = 0;
  for (auto &I : envinst) {
    I.col0 = max_nc; max_nc += I.nc;
    const sgb_envelope &E = b->envs[I.env_id];
    max_f = std::max(max_f, E.n_formants);
    bool moving = false;
    if (E.tracks_given == 0)
      for (int f = 0; f < E.n_formants; f++) if (b->frefs[E.formant_off + f].n > 1) moving = true;
    if (moving) { I.trk_off = trk_total; trk_total += (int64_t)I.nc * E.n_formants * 3; }
    envk_total = env_knot_layout(I, E, b->frefs.data(), envk_total);
  }
  CK(b->d_trk.ensure(8 * (size_t)std::max<int64_t>(trk_total, 1)));
  CK(b->d_envk.ensure(8 * (size_t)std::max<int64_t>(envk_total, 1)));
  CK(b->d_mouth.ensure(8 * (size_t)std::max(max_nc, 1)));
  CK(b->d_bl.ensure(sizeof(BoutLayout) * (size_t)NB));
  CK(b->d_place.ensure(sizeof(SylPlace) * (size_t)S));
  CK(b->d_nl.ensure(sizeof(NoiseLayout) * (size_t)std::max(NN, 1)));
  CK(b->d_envinst.ensure(sizeof(EnvInst) * std::max<size_t>(envinst.size(), 1)));
  CK(b->d_plans.ensure(sizeof(FftPlan) * std::max<size_t>(plans.size(), 1)));
  CK(b->d_tw.ensure(8 * (size_t)std::max<int64_t>(tw_total, 1)));
  CK(b->d_win.ensure(4 * (size_t)std::max<int64_t>(win_total, 1)));
  CK(b->d_fjobs.ensure(sizeof(FftJob) * std::max<size_t>(fjobs.size(), 1)));
  CK(b->d_njobs.ensure(sizeof(FftJob) * std::max<size_t>(njobs.size(), 1)));
  CK(b->d_fsegs.ensure(sizeof(FftSeg) * std::max<size_t>(fsegs.size(), 1)));
  CK(b->d_nsegs.ensure(sizeof(FftSeg) * std::max<size_t>(nsegs.size(), 1)));
  CK(b->d_max.ensure(4 * (size_t)(NB + NN + 1)));
  CK(b->d_sound.ensure(4 * (size_t)(sound_total + 64)));
  CK(b->d_filt.ensure(4 * (size_t)(filt_total + 64)));
  CK(b->d_env.ensure(4 * (size_t)(env_total + 64)));
  CK(b->d_noise_raw.ensure(4 * (size_t)(noise_total + 64)));
  CK(b->d_noise_fin.ensure(4 * (size_t)(noise_total + 64)));
  CK(b->d_out.ensure(4 * (size_t)(out_total + 64)));
  auto up = [&](DBuf &d, const void *src, size_t bytes) -> cudaError_t {
    if (!bytes) return cudaSuccess;
    return cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, st);
  };
  CK(up(b->d_bl, b->bl.data(), sizeof(BoutLayout) * (size_t)NB));
  CK(up(b->d_place, b->place.data(), sizeof(SylPlace) * (size_t)S));
  CK(up(b->d_nl, b->nl.data(), sizeof(NoiseLayout) * (size_t)NN));
  CK(up(b->d_envinst, envinst.data(), sizeof(EnvInst) * envinst.size()));
  CK(up(b->d_plans, plans.data(), sizeof(FftPlan) * plans.size()));
  CK(up(b->d_tw, tw_host.data(), 8 * (size_t)tw_total));
  CK(up(b->d_win, win_host.data(), 4 * (size_t)win_total));
  CK(up(b->d_fjobs, fjobs.data(), sizeof(FftJob) * fjobs.size()));
  CK(up(b->d_njobs, njobs.data(), sizeof(FftJob) * njobs.size()));
  CK(up(b->d_fsegs, fsegs.data(), sizeof(FftSeg) * fsegs.size()));
  CK(up(b->d_nsegs, nsegs.data(), sizeof(FftSeg) * nsegs.size()));
  b->last_sound = sound_total;
  CK(cudaMemsetAsync(b->d_sound.p, 0, 4 * (size_t)(sound_total + 64), st));
  CK(cudaMemsetAsync(b->d_out.p, 0, 4 * (size_t)(out_total + 64), st));
  if (noise_total) CK(cudaMemsetAsync(b->d_noise_raw.p, 0, 4 * (size_t)(noise_total + 64), st));
  k_fill_int<<<(NB + NN + 256) / 256, 256, 0, st>>>(b->d_max.as<int>(), NB + NN + 1, ORDERED_NEG_INF);
  launches++;

  const int chunks = (NB >= 1024) ? 4 : ((NB >= 64) ? 16 : 64);
  // ---- voiced syllables -> sound ----
  launch_place_voiced(d_syl, S, d_ctrl, d_lay, b->d_place.as<SylPlace>(), P, b->d_raw.as<float>(),
                      b->d_sound.as<float>(), chunks, st);
  CKL("launch_place_voiced");
  launches++;
  if (b->keep_voiced) {
    CK(b->d_voiced.ensure(4 * (size_t)(sound_total + 64)));
    CK(cudaMemcpyAsync(b->d_voiced.p, b->d_sound.p, 4 * (size_t)(sound_total + 64), cudaMemcpyDeviceToDevice, st));
  }
  CK(cudaEventRecord(ev[5], st)); trace_mark(b, 5);   // assemble (part 1)
  // ---- K4 envelopes (bouts + noises) ----
  CK(b->d_mtabs.ensure(contour_tab_bytes() * std::max<size_t>(envinst.size(), 1)));
  launch_env_tracks(b->d_envinst.as<EnvInst>(), (int)envinst.size(), b->d_envs.as<sgb_envelope>(),
                    b->d_frefs.as<sgb_formant_ref>(), b->d_formants.as<double>(), b->d_anchors.as<double>(),
                    b->d_trk.as<double>(), b->d_mouth.as<double>(), b->d_mtabs.p, b->d_envk.as<double>(), st);
  CKL("launch_env_tracks");
  CK(launch_envelope_f32(b->d_envinst.as<EnvInst>(), (int)envinst.size(), max_nc, max_f, b->d_envs.as<sgb_envelope>(),
                         b->d_frefs.as<sgb_formant_ref>(), b->d_formants.as<double>(), b->d_formants_late.as<double>(),
                         b->d_trk.as<double>(), b->d_mouth.as<double>(), b->d_pre.as<double>(), b->d_env.as<float>(), st));
  if (!envinst.empty()) launches += 2;
  CK(cudaEventRecord(ev[6], st)); trace_mark(b, 6);
  // ---- K5 noise ----
  if (!nsegs.empty()) {
    for (auto &gr : ngroups) {
      if (gr.smem > 226 * 1024) return fail(SGB_ERR_UNSUPPORTED, "noise window too long for shared memory (%zu bytes)", gr.smem);
      cudaError_t le = launch_stft(1, b->u_is_float, gr.spec, b->d_nsegs.as<FftSeg>() + gr.begin, gr.end - gr.begin,
                                   b->d_njobs.as<FftJob>(), b->d_plans.as<FftPlan>(), b->d_tw.as<float2>(), b->d_win.as<float>(),
                                   nullptr, b->d_u.p, b->d_env.as<float>(), b->d_noise_raw.as<float>(), b->d_max.as<int>(),
                                   gr.smem, st);
      if (le != cudaSuccess)
        return fail(SGB_ERR_CUDA, "noise STFT launch failed (plan group %d, %d segments, %zu bytes of shared memory): %s", gr.spec,
                    gr.end - gr.begin, gr.smem, cudaGetErrorString(le));
      launches++;
    }
    CK(b->d_ntabs.ensure(contour_tab_bytes() * (size_t)NN));
    launch_noise_final(b->d_noises.as<sgb_noise>(), NN, b->d_nl.as<NoiseLayout>(), b->d_anchors.as<double>(),
                       b->d_pre.as<double>(), b->d_max.as<int>(), NB, b->d_noise_raw.as<float>(),
                       b->d_noise_fin.as<float>(), b->d_ntabs.p, b->d_knots.as<double>(),
                       b->d_koff.as<int64_t>() + 3 * (size_t)S, 16, st);
    CKL("launch_noise_final");
    launches += 1;
  }
  CK(cudaEventRecord(ev[7], st)); trace_mark(b, 7);
  // ---- sound = voiced + breathing, global envelope ----
  launch_sound_mix(b->d_bouts.as<sgb_bout>(), NB, b->d_bl.as<BoutLayout>(), b->d_noises.as<sgb_noise>(),
                   b->d_nl.as<NoiseLayout>(), b->d_anchors.as<double>(), b->d_noise_fin.as<float>(),
                   b->d_sound.as<float>(), b->d_btabs.p, b->d_knots.as<double>(), b->d_koff.as<int64_t>() + 3 * (size_t)S + NN,
                   b->any_aglobal, chunks, st);
  CKL("launch_sound_mix");
  launches += b->any_aglobal ? 2 : 1;
  CK(cudaEventRecord(ev[8], st)); trace_mark(b, 8);
  // ---- K2 filter ----
  for (auto &gr : fgroups) {
    if (gr.smem > 226 * 1024) return fail(SGB_ERR_UNSUPPORTED, "window too long for shared memory (%zu bytes)", gr.smem);
    CK(launch_stft(0, 0, gr.spec, b->d_fsegs.as<FftSeg>() + gr.begin, gr.end - gr.begin, b->d_fjobs.as<FftJob>(),
                   b->d_plans.as<FftPlan>(), b->d_tw.as<float2>(), b->d_win.as<float>(), b->d_sound.as<float>(),
                   nullptr, b->d_env.as<float>(), b->d_filt.as<float>(), b->d_max.as<int>(), gr.smem, st));
    launches++;
  }
  CK(cudaEventRecord(ev[9], st)); trace_mark(b, 9);
  // ---- normalise, post-filter noise, AM, silences ----
  launch_finalize(0, b->d_bouts.as<sgb_bout>(), NB, b->d_bl.as<BoutLayout>(), b->d_noises.as<sgb_noise>(),
                  b->d_nl.as<NoiseLayout>(), b->d_sound.as<float>(), b->d_filt.as<float>(),
                  b->d_noise_fin.as<float>(), b->d_max.as<int>(), b->d_out.p, chunks, st);
  CKL("launch_finalize");
  launches++;
  CK(cudaEventRecord(ev[10], st)); trace_mark(b, 10);
  b->where = 3;
  CK(wait_stream(b));
  b->where = 0;
  CK(cudaGetLastError());
  if (stft_timeout_flag()) return fail(SGB_ERR_CUDA, "k_stft: a staged (TMA) frame load did not complete");
  if (synth_tc_timeout_flag()) return fail(SGB_ERR_CUDA, "k_synth_tc: a tensor-core completion barrier never flipped");
  info.kernel_launches = launches;
  float ms;
  CK(cudaEventElapsedTime(&ms, ev[0], ev[1])); info.ms[SGB_T_CONTROL] = ms;
  CK(cudaEventElapsedTime(&ms, ev[1], ev[2])); info.ms[SGB_T_AMPL] = ms;
  CK(cudaEventElapsedTime(&ms, ev[2], ev[3])); info.ms[SGB_T_SYNTH] = ms;
  CK(cudaEventElapsedTime(&ms, ev[3], ev[4])); info.ms[SGB_T_COMPOSE] = ms;
  CK(cudaEventElapsedTime(&ms, ev[4], ev[5])); info.ms[SGB_T_ASSEMBLE] = ms;
  CK(cudaEventElapsedTime(&ms, ev[5], ev[6])); info.ms[SGB_T_ENVELOPE] = ms;
  CK(cudaEventElapsedTime(&ms, ev[6], ev[7])); info.ms[SGB_T_NOISE] = ms;
  CK(cudaEventElapsedTime(&ms, ev[7], ev[8])); info.ms[SGB_T_ASSEMBLE] += ms;
  CK(cudaEventElapsedTime(&ms, ev[8], ev[9])); info.ms[SGB_T_FILTER] = ms;
  CK(cudaEventElapsedTime(&ms, ev[9], ev[10])); info.ms[SGB_T_FINALIZE] = ms;
  CK(cudaEventElapsedTime(&ms, ev[0], ev[10])); info.ms[SGB_T_TOTAL] = ms;
  b->have_run = true;
  if (info_out) *info_out = info;
  return SGB_OK;
}

int sgb_batch_bout_geometry(sgb_batch *b, int32_t bout, int32_t *nc, int32_t *nint, int32_t *wl, int32_t *sound_len) {
  if (!b || !b->rs || !(b->rs->begun || b->have_run)) return fail(SGB_ERR_STATE, "no run in progress");
  if (bout < 0 || bout >= (int)b->bl.size()) return fail(SGB_ERR_INVALID, "bout index");
  const BoutLayout &L = b->bl[bout];
  if (nc) *nc = L.nc;
  if (nint) *nint = L.nint;
  if (wl) *wl = L.bypass ? 0 : L.wl;
  if (sound_len) *sound_len = L.sound_len;
  return SGB_OK;
}

int sgb_batch_set_tracks(sgb_batch *b, int32_t env, const double *rows, int32_t n_formants, int32_t nc) {
  if (!b || !b->rs || !b->rs->begun) return fail(SGB_ERR_STATE, "sgb_batch_set_tracks outside run_begin / run_finish");
  if (env < 0 || env >= (int)b->envs.size() || !rows || nc < 1) return fail(SGB_ERR_INVALID, "bad argument");
  if (n_formants < 1 || n_formants > SGB_MAX_FORMANTS)
    return fail(SGB_ERR_UNSUPPORTED, "%d formant tracks (at most %d)", n_formants, SGB_MAX_FORMANTS);
  sgb_envelope &E = b->envs[env];
  E.tracks_given = 1;
  E.n_formants = n_formants;
  E.formant_off = (int64_t)b->frefs.size();
  for (int f = 0; f < n_formants; f++) {
    sgb_formant_ref R;
    R.off = (int64_t)(b->late_rows.size() / 4) + (int64_t)f * nc;
    R.n = nc; R.pad = 1;                 // pad = 1: rows live in the late pool
    b->frefs.push_back(R);
  }
  b->late_rows.insert(b->late_rows.end(), rows, rows + (size_t)4 * n_formants * nc);
  b->late_envs.push_back(env);
  b->envs_dirty = true;
  return SGB_OK;
}

int sgb_batch_z_used(sgb_batch *b, int32_t *out) {
  if (!b || !out) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->rs || !(b->rs->begun || b->have_run)) return fail(SGB_ERR_STATE, "no run");
  for (size_t s = 0; s < b->summary.size(); s++) out[s] = b->summary[s].z_used;
  return SGB_OK;
}

// K1 dispatch threshold for the batches that run after this call (tests; -1 = environment / default 224 rows)
int sgb_synth_min_rows_set(int32_t rows) { g_synth_min_rows_override = rows < 0 ? -1 : rows; return SGB_OK; }

int sgb_abi_sizes(int32_t *out, int32_t cap) {
  const int32_t v[] = {(int32_t)sizeof(sgb_syllable), (int32_t)sizeof(sgb_envelope), (int32_t)sizeof(sgb_noise),
                       (int32_t)sizeof(sgb_bout), (int32_t)sizeof(sgb_call), (int32_t)sizeof(sgb_formant_ref),
                       (int32_t)sizeof(sgb_batch_desc), (int32_t)sizeof(sgb_run_info), (int32_t)sizeof(sgb_soundgen_args),
                       (int32_t)sizeof(sgb_device_out), (int32_t)sizeof(sgb_spec_params),
                       (int32_t)sizeof(sgb_compare_params), (int32_t)sizeof(sgb_ceps_params)};
  if (!out || cap < 9) return fail(SGB_ERR_INVALID, "need room for 9 sizes");
  for (int i = 0; i < 13 && i < cap; i++) out[i] = v[i];
  return SGB_OK;
}

int sgb_batch_lengths(sgb_batch *b, int64_t *out_len) {
  if (!b || !out_len) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  for (size_t c = 0; c < b->call_len.size(); c++) out_len[c] = b->call_len[c];
  return SGB_OK;
}

int sgb_batch_status(sgb_batch *b, int32_t *out_status) {
  if (!b || !out_status) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  for (size_t c = 0; c < b->call_status.size(); c++) out_status[c] = b->call_status[c];
  return SGB_OK;
}

static int fetch_common(sgb_batch *b, void *out, int64_t n, bool f64) {
  if (!b || !out) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  CK(cudaSetDevice(b->device));
  int64_t need = 0;
  for (auto l : b->call_len) need += l;
  if (n < need) return fail(SGB_ERR_INVALID, "output buffer too small: %lld < %lld", (long long)n, (long long)need);
  cudaStream_t st = b->st;
  CK(cudaEventRecord(b->ev[SGB_T_COUNT], st));
  const void *src = b->d_out.p;
  size_t esz = 4;
  if (f64) {
    CK(b->d_out64.ensure(8 * (size_t)(b->total_out + 64)));
    int64_t m = b->total_out;
    if (m > 0) k_f32_to_f64<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(b->d_out.as<float>(), b->d_out64.as<double>(), m);
    src = b->d_out64.p; esz = 8;
  }
  if (need > 0) CK(cudaMemcpyAsync(out, src, (size_t)need * esz, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(b->ev[SGB_T_COUNT + 1], st));
  CK(wait_stream(b));
  CK(cudaEventElapsedTime(&b->info.ms[SGB_T_D2H], b->ev[SGB_T_COUNT], b->ev[SGB_T_COUNT + 1]));
  return SGB_OK;
}
int sgb_batch_fetch_f32(sgb_batch *b, float *out, int64_t n) { return fetch_common(b, out, n, false); }
int sgb_batch_fetch_f64(sgb_batch *b, double *out, int64_t n) { return fetch_common(b, out, n, true); }

// 16-bit PCM (WAV sample format) of every call, normalised as the reference's savePath branch does
// (k_pcm16): halves the device -> host bytes of a data-generation run.
int sgb_batch_fetch_pcm16(sgb_batch *b, int16_t *out, int64_t n) {
  if (!b || !out) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  CK(cudaSetDevice(b->device));
  int64_t need = 0;
  for (auto l : b->call_len) need += l;
  if (n < need) return fail(SGB_ERR_INVALID, "output buffer too small: %lld < %lld", (long long)n, (long long)need);
  const size_t NC = b->call_len.size();
  cudaStream_t st = b->st;
  CK(b->d_pcm.ensure(2 * (size_t)(b->total_out + 64)));
  CK(b->d_calltab.ensure(16 * std::max<size_t>(NC, 1)));
  CK(b->h_calltab.ensure(16 * std::max<size_t>(NC, 1)));
  int64_t *h = b->h_calltab.as<int64_t>();
  for (size_t c = 0; c < NC; c++) { h[c] = b->call_off[c]; h[NC + c] = b->call_len[c]; }
  CK(cudaEventRecord(b->ev[SGB_T_COUNT], st));
  CK(cudaMemcpyAsync(b->d_calltab.p, h, 16 * NC, cudaMemcpyHostToDevice, st));
  const int64_t *d_off = b->d_calltab.as<int64_t>(), *d_len = d_off + NC;
  if (NC > 0) k_pcm16<<<(unsigned)NC, 256, 0, st>>>(b->d_out.as<float>(), d_off, d_len, d_off, d_len, b->d_pcm.as<int16_t>());
  if (need > 0) CK(cudaMemcpyAsync(out, b->d_pcm.p, (size_t)need * 2, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(b->ev[SGB_T_COUNT + 1], st));
  CK(wait_stream(b));
  CK(cudaGetLastError());
  CK(cudaEventElapsedTime(&b->info.ms[SGB_T_D2H], b->ev[SGB_T_COUNT], b->ev[SGB_T_COUNT + 1]));
  return SGB_OK;
}

// ---- device output (sgb_batch_export / sgb_rows_export, sgb_batch_spectrogram / sgb_rows_spectrogram) ----
// `p` must be device (or managed) memory of `device`.
static int on_device(int device, const void *p, const char *what) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(SGB_ERR_INVALID, "%s: not a CUDA allocation (%s)", what, cudaGetErrorString(e)); }
  if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)
    return fail(SGB_ERR_INVALID, "%s is host memory (pinned or pageable), not device memory", what);
  if (a.device != device) return fail(SGB_ERR_INVALID, "%s is memory of device %d, not of device %d", what, a.device, device);
  return SGB_OK;
}

// Checks everything the host can check before anything is queued.  `src` (the rows entries) is checked like dst.
// Row c occupies cap[c] * unit elements of dst (unit: floats per frame of a spectrogram, 1 for the exports).
static int export_check(int device, const float *src, const int64_t *src_off, const int64_t *len, int32_t n,
                        const sgb_device_out *o, int64_t unit, bool pcm16_ok) {
  if (!o) return fail(SGB_ERR_INVALID, "null sgb_device_out");
  if (o->format != SGB_OUT_F32 && !(pcm16_ok && o->format == SGB_OUT_PCM16))
    return fail(SGB_ERR_INVALID, "unsupported output format %d", o->format);
  if (n < 0 || o->dst_elems < 0) return fail(SGB_ERR_INVALID, "negative row count or dst_elems");
  if (n > 0 && (!o->dst_off || !o->cap || !len || (src && !src_off))) return fail(SGB_ERR_INVALID, "null row table");
  std::vector<std::pair<int64_t, int64_t>> rows;
  rows.reserve((size_t)n);
  for (int32_t c = 0; c < n; c++) {
    const int64_t off = o->dst_off[c], cp = o->cap[c];
    if (off < 0 || cp < 0) return fail(SGB_ERR_INVALID, "row %d: negative offset or capacity", c);
    if (off > o->dst_elems || cp > (o->dst_elems - off) / unit)
      return fail(SGB_ERR_INVALID, "row %d: elements [%lld, %lld x %lld more) outside dst (%lld elements)", c,
                  (long long)off, (long long)cp, (long long)unit, (long long)o->dst_elems);
    if (len[c] < 0 || (src && src_off[c] < 0)) return fail(SGB_ERR_INVALID, "row %d: negative source offset or length", c);
    if (cp > 0) rows.push_back({off, cp * unit});
  }
  std::sort(rows.begin(), rows.end());
  for (size_t i = 1; i < rows.size(); i++)
    if (rows[i - 1].first + rows[i - 1].second > rows[i].first)
      return fail(SGB_ERR_INVALID, "rows overlap in dst at element %lld", (long long)rows[i].first);
  if (!rows.empty()) {
    if (!o->dst) return fail(SGB_ERR_INVALID, "null dst");
    const size_t esz = o->format == SGB_OUT_F32 ? 4 : 2;
    if ((uintptr_t)o->dst % esz) return fail(SGB_ERR_INVALID, "dst is not aligned to its element type");
    int rc = on_device(device, o->dst, "dst");
    if (rc != SGB_OK) return rc;
  }
  if (src) {
    if ((uintptr_t)src % 4) return fail(SGB_ERR_INVALID, "src is not aligned to float");
    int rc = on_device(device, src, "src");
    if (rc != SGB_OK) return rc;
  }
  return SGB_OK;
}

// Queues work on `st` (the handle's stream, or the device's export stream) ordered against the caller's stream
// `user` as the header describes.  fill(h) writes `bytes` of host-built tables into a pinned staging slot; launch(d)
// queues the kernels on their device copy.  Arguments were checked before.
static int export_queue(ExportCtx &X, cudaStream_t st, cudaStream_t user, size_t bytes,
                        const std::function<void(char *)> &fill, const std::function<int(const char *)> &launch) {
  if (!X.ev_in) CK(cudaEventCreateWithFlags(&X.ev_in, cudaEventDisableTiming));
  ExportSlot *S = nullptr;
  for (auto s : X.slots) {
    cudaError_t q = cudaEventQuery(s->done);
    if (q == cudaSuccess) { S = s; break; }
    if (q != cudaErrorNotReady) CK(q);
    cudaGetLastError();          // cudaErrorNotReady is not an error to carry forward
  }
  if (!S) {
    S = new ExportSlot();
    cudaError_t e = cudaEventCreateWithFlags(&S->done, cudaEventDisableTiming);
    if (e != cudaSuccess) { delete S; CK(e); }
    X.slots.push_back(S);
  }
  CK(S->h.ensure(std::max<size_t>(bytes, 16)));
  CK(S->d.ensure(std::max<size_t>(bytes, 16)));
  fill(reinterpret_cast<char *>(S->h.p));
  CK(cudaEventRecord(X.ev_in, user));                // the destination is free once the caller's stream gets here
  CK(cudaStreamWaitEvent(st, X.ev_in, 0));
  if (bytes) CK(cudaMemcpyAsync(S->d.p, S->h.p, bytes, cudaMemcpyHostToDevice, st));
  const int rc = launch(reinterpret_cast<const char *>(S->d.p));
  CK(cudaEventRecord(S->done, st));                  // the slot is reused only after its copy has been read
  if (rc != SGB_OK) return rc;
  CK(cudaStreamWaitEvent(user, S->done, 0));        // the caller's later work sees the rows
  return SGB_OK;
}

static int export_rows(ExportCtx &X, cudaStream_t st, const float *src, const int64_t *src_off, const int64_t *len,
                       int32_t n, const sgb_device_out *o) {
  // row table: src_off, len, dst_off, cap (n each), then the (row, chunk) grid of the f32 kernel
  std::vector<int2> grid;
  if (o->format == SGB_OUT_F32) {
    for (int32_t c = 0; c < n; c++)
      for (int64_t k = 0; k * EXPORT_CHUNK < o->cap[c]; k++) grid.push_back(make_int2(c, (int)k));
  }
  const size_t tab_bytes = 32 * (size_t)n, bytes = tab_bytes + sizeof(int2) * grid.size();
  auto fill = [&](char *hp) {
    int64_t *h = reinterpret_cast<int64_t *>(hp);
    for (int32_t c = 0; c < n; c++) {
      h[c] = src_off[c]; h[n + c] = len[c]; h[2 * (size_t)n + c] = o->dst_off[c]; h[3 * (size_t)n + c] = o->cap[c];
    }
    if (!grid.empty()) memcpy(hp + tab_bytes, grid.data(), sizeof(int2) * grid.size());
  };
  auto launch = [&](const char *dp) -> int {
    const int64_t *d = reinterpret_cast<const int64_t *>(dp);
    if (o->format == SGB_OUT_F32) {
      if (!grid.empty())
        k_export_f32<<<(unsigned)grid.size(), EXPORT_THREADS, 0, st>>>(
            src, d, d + n, d + 2 * (size_t)n, d + 3 * (size_t)n, reinterpret_cast<const int2 *>(dp + tab_bytes),
            (float *)o->dst);
      CKL("k_export_f32");
    } else {
      if (n > 0)
        k_pcm16<<<(unsigned)n, 256, 0, st>>>(src, d, d + n, d + 2 * (size_t)n, d + 3 * (size_t)n, (int16_t *)o->dst);
      CKL("k_pcm16");
    }
    return SGB_OK;
  };
  int rc = export_queue(X, st, (cudaStream_t)o->stream, bytes, fill, launch);
  if (rc != SGB_OK) return rc;
  if (o->out_written)
    for (int32_t c = 0; c < n; c++) o->out_written[c] = std::min(len[c], o->cap[c]);
  return SGB_OK;
}

static int no_device() {
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) {
    cudaGetLastError();
    return fail(SGB_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
  }
  return SGB_OK;
}

int sgb_batch_export(sgb_batch *b, const sgb_device_out *o) {
  if (!b) return fail(SGB_ERR_INVALID, "null batch");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  CK(cudaSetDevice(b->device));
  const int32_t n = (int32_t)b->call_len.size();
  int rc = export_check(b->device, nullptr, nullptr, b->call_len.data(), n, o, 1, true);
  if (rc != SGB_OK) return rc;
  if (!b->xo) b->xo = new ExportCtx();
  // queued on the handle's stream: the next run of this handle (same stream) cannot overwrite d_out first
  return export_rows(*b->xo, b->st, b->d_out.as<float>(), b->call_off.data(), b->call_len.data(), n, o);
}

// one export stream + staging per device for rows the caller holds (no handle); exports from several host threads
// to the same device take turns on its lock while they queue (nothing inside waits on the device)
struct DeviceExport {
  std::mutex mu;
  cudaStream_t st = nullptr;
  ExportCtx x;
};
static std::mutex g_dev_export_mu;
static std::map<int, DeviceExport *> g_dev_export;     // kept for the life of the process

static int device_export(int device, DeviceExport **out) {
  std::lock_guard<std::mutex> g(g_dev_export_mu);
  auto it = g_dev_export.find(device);
  if (it == g_dev_export.end()) {
    DeviceExport *D = new DeviceExport();
    cudaError_t e = cudaStreamCreateWithFlags(&D->st, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete D; CK(e); }
    g_dev_export[device] = D;
    *out = D;
  } else {
    *out = it->second;
  }
  return SGB_OK;
}

static int rows_device_check(int32_t device, const float *src, int32_t n) {
  int rc = no_device();
  if (rc != SGB_OK) return rc;
  int nd = 0;
  CK(cudaGetDeviceCount(&nd));
  if (device < 0 || device >= nd) return fail(SGB_ERR_INVALID, "device %d of %d", device, nd);
  if (n > 0 && !src) return fail(SGB_ERR_INVALID, "null src");
  CK(cudaSetDevice(device));
  return SGB_OK;
}

int sgb_rows_export(int32_t device, const float *src, const int64_t *src_off, const int64_t *len, int32_t n,
                    const sgb_device_out *o) {
  int rc = rows_device_check(device, src, n);
  if (rc != SGB_OK) return rc;
  rc = export_check(device, n > 0 ? src : nullptr, src_off, len, n, o, 1, true);
  if (rc != SGB_OK) return rc;
  DeviceExport *D;
  if ((rc = device_export(device, &D)) != SGB_OK) return rc;
  std::lock_guard<std::mutex> g(D->mu);
  return export_rows(D->x, D->st, src, src_off, len, n, o);
}

// ---- spectrograms (K9) ----
// nc = length(seq(1, max(1, len - wl), h)) in 64 bits (seq_by_count), 0 for an empty row
static int64_t spec_nc(int64_t len, int wl, double h) {
  if (len <= 0) return 0;
  const double to = std::max<double>(1.0, (double)(len - wl));
  if (to == 1.0) return 1;
  return (int64_t)std::floor((to - 1.0) / h + 1e-10) + 1;
}

static int spec_geometry(int32_t wl, double overlap, double *h) {
  if (wl < 4 || (wl & 1)) return fail(SGB_ERR_UNSUPPORTED, "window of %d points (odd or < 4) is not supported", wl);
  if (!(overlap >= 0.0 && overlap < 100.0)) return fail(SGB_ERR_INVALID, "overlap %g out of [0, 100)", overlap);
  *h = wl - (overlap * wl / 100.0);
  if (!(*h >= 1.0)) return fail(SGB_ERR_INVALID, "hop %g of a %d-point window is below one sample", *h, wl);
  return SGB_OK;
}

int64_t sgb_spec_frames(int64_t len, int32_t wl, double overlap) {
  double h;
  if (len < 0 || spec_geometry(wl, overlap, &h) != SGB_OK) return -1;
  return spec_nc(len, wl, h);
}

// Everything a spectrogram call queues, built and checked on the host before anything is queued.
struct SpecJob {
  PlanTable PT;
  FftPlan pl;
  int n_feat = 0, n_w = 0;
  size_t smem = 0;
  std::vector<SpecRow> rows;
  std::vector<FftSeg> segs;
  std::vector<int32_t> band_tab;       // lo, len, first weight (n_bands each)
};

// the parameters alone (no device needed)
static int spec_params(const sgb_spec_params *p, SpecJob &J) {
  if (!p) return fail(SGB_ERR_INVALID, "null sgb_spec_params");
  double h;
  int rc = spec_geometry(p->wl, p->overlap, &h);
  if (rc != SGB_OK) return rc;
  if (p->window != SGB_WIN_HAMMING && p->window != SGB_WIN_HANNING) return fail(SGB_ERR_INVALID, "unknown window %d", p->window);
  if (p->db != 0 && p->db != 1) return fail(SGB_ERR_INVALID, "db must be 0 or 1, not %d", p->db);
  if (p->db && !(p->db_floor > 0.0 && std::isfinite(p->db_floor) && (float)p->db_floor > 0.0f))
    return fail(SGB_ERR_INVALID, "db_floor %g: a positive finite float is needed", p->db_floor);
  const int nr = p->wl / 2;
  if (p->n_bands < 0) return fail(SGB_ERR_INVALID, "negative n_bands");
  if (p->n_bands > 0) {
    if (!p->band_lo || !p->band_len || !p->band_w) return fail(SGB_ERR_INVALID, "null band table");
    J.band_tab.resize(3 * (size_t)p->n_bands);
    int64_t nw = 0;
    for (int b = 0; b < p->n_bands; b++) {
      const int32_t lo = p->band_lo[b], ln = p->band_len[b];
      if (lo < 0 || ln < 0 || lo > nr || ln > nr - lo)
        return fail(SGB_ERR_INVALID, "band %d: bins [%d, %d + %d) outside [0, %d)", b, lo, lo, ln, nr);
      for (int j = 0; j < ln; j++)
        if (!std::isfinite(p->band_w[nw + j])) return fail(SGB_ERR_INVALID, "band %d: weight %d is not finite", b, j);
      if (nw + ln > (int64_t)INT32_MAX) return fail(SGB_ERR_UNSUPPORTED, "band weights do not fit in shared memory");
      J.band_tab[b] = lo; J.band_tab[p->n_bands + b] = ln; J.band_tab[2 * (size_t)p->n_bands + b] = (int32_t)nw;
      nw += ln;
    }
    J.n_w = (int)nw;
  }
  J.n_feat = p->n_bands ? p->n_bands : nr;
  J.smem = spectrogram_smem_bytes(p->wl, h, p->n_bands, J.n_w);
  if (J.smem > 226 * 1024) return fail(SGB_ERR_UNSUPPORTED, "window and bands too large for shared memory (%zu bytes)", J.smem);
  const int pi = J.PT.get(p->wl, p->overlap);
  if (pi < 0) return fail(SGB_ERR_UNSUPPORTED, "cannot factor window length %d", p->wl);
  J.pl = J.PT.plans[pi];
  return SGB_OK;
}

// the rows and the destination, after spec_params
static int spec_rows(const sgb_spec_params *p, const float *src, const int64_t *src_off, const int64_t *len, int32_t n,
                     const sgb_device_out *o, int device, SpecJob &J) {
  const double h = J.pl.h_in;
  int rc = export_check(device, src, src_off, len, n, o, J.n_feat, false);
  if (rc != SGB_OK) return rc;
  // rows: the first min(nc, cap) frames are computed, frame pairs completed (a pair is one FFT); the rest are zeros
  std::vector<FftJob> jobs;
  J.rows.resize((size_t)n);
  for (int32_t c = 0; c < n; c++) {
    if (len[c] > INT32_MAX || o->cap[c] > INT32_MAX)
      return fail(SGB_ERR_INVALID, "row %d: %lld samples, %lld frames (at most 2^31 - 1 each)", c, (long long)len[c],
                  (long long)o->cap[c]);
    SpecRow &R = J.rows[c];
    R.src_off = src_off[c]; R.dst_off = o->dst_off[c]; R.len = len[c]; R.cap = o->cap[c];
    R.nc = spec_nc(len[c], p->wl, h);
    FftJob fj;
    memset(&fj, 0, sizeof fj);
    fj.plan = 0;
    fj.nc = (int32_t)std::min(R.nc, R.cap + (R.cap & 1));
    jobs.push_back(fj);
  }
  std::vector<SegGroup> groups;
  make_segs(jobs, J.PT.plans, 0, J.segs, groups);
  const int zf = std::max(1, 8192 / J.n_feat);        // zero-tail segments: about 8192 floats each
  for (int32_t c = 0; c < n; c++)
    for (int64_t k = J.rows[c].nc; k < J.rows[c].cap; k += zf) {
      FftSeg sg; sg.job = c; sg.ka = (int32_t)k; sg.kb = (int32_t)std::min<int64_t>(J.rows[c].cap, k + zf); sg.pad = 0;
      J.segs.push_back(sg);
    }
  if (J.segs.size() > (size_t)INT32_MAX) return fail(SGB_ERR_UNSUPPORTED, "too many segments");
  return SGB_OK;
}

static int spec_queue(ExportCtx &X, cudaStream_t st, const float *src, const SpecJob &J, const sgb_spec_params *p,
                      const sgb_device_out *o) {
  const int N = J.pl.n, nb = p->n_bands;
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t o_rows = 0, o_segs = up16(o_rows + sizeof(SpecRow) * J.rows.size());
  const size_t o_tw = up16(o_segs + sizeof(FftSeg) * J.segs.size()), o_win = up16(o_tw + sizeof(float2) * N);
  const size_t o_band = up16(o_win + sizeof(float) * N), o_w = up16(o_band + sizeof(int32_t) * J.band_tab.size());
  const size_t bytes = o_w + sizeof(float) * J.n_w;
  const int64_t w_off = p->window == SGB_WIN_HANNING ? J.pl.wh_off : J.pl.wa_off;
  auto fill = [&](char *h) {
    if (!J.rows.empty()) memcpy(h + o_rows, J.rows.data(), sizeof(SpecRow) * J.rows.size());
    if (!J.segs.empty()) memcpy(h + o_segs, J.segs.data(), sizeof(FftSeg) * J.segs.size());
    memcpy(h + o_tw, J.PT.tw.data() + J.pl.tw_off, sizeof(float2) * N);
    memcpy(h + o_win, J.PT.win.data() + w_off, sizeof(float) * N);
    if (nb) {
      memcpy(h + o_band, J.band_tab.data(), sizeof(int32_t) * J.band_tab.size());
      memcpy(h + o_w, p->band_w, sizeof(float) * J.n_w);
    }
  };
  auto launch = [&](const char *d) -> int {
    cudaError_t e = launch_spectrogram(reinterpret_cast<const FftSeg *>(d + o_segs), (int)J.segs.size(),
                                       reinterpret_cast<const SpecRow *>(d + o_rows), J.pl,
                                       reinterpret_cast<const float2 *>(d + o_tw), reinterpret_cast<const float *>(d + o_win),
                                       src, nb, reinterpret_cast<const int32_t *>(d + o_band),
                                       reinterpret_cast<const float *>(d + o_w), J.n_w, p->db, (float)p->db_floor,
                                       (float *)o->dst, J.smem, st);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(SGB_ERR_CUDA, "k_spectrogram launch failed (%zu segments, %zu bytes of shared memory): %s",
                  J.segs.size(), J.smem, cudaGetErrorString(e));
    }
    return SGB_OK;
  };
  int rc = export_queue(X, st, (cudaStream_t)o->stream, bytes, fill, launch);
  if (rc != SGB_OK) return rc;
  if (o->out_written)
    for (size_t c = 0; c < J.rows.size(); c++) o->out_written[c] = std::min(J.rows[c].nc, J.rows[c].cap);
  return SGB_OK;
}

int sgb_batch_spectrogram(sgb_batch *b, const sgb_spec_params *p, const sgb_device_out *o) {
  SpecJob J;
  int rc = spec_params(p, J);
  if (rc != SGB_OK) return rc;
  if ((rc = no_device()) != SGB_OK) return rc;
  if (!b) return fail(SGB_ERR_INVALID, "null batch");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  CK(cudaSetDevice(b->device));
  const int32_t n = (int32_t)b->call_len.size();
  rc = spec_rows(p, nullptr, b->call_off.data(), b->call_len.data(), n, o, b->device, J);
  if (rc != SGB_OK) return rc;
  if (!b->xo) b->xo = new ExportCtx();
  // on the handle's stream, like the export: the handle's next run cannot overwrite the rows first
  return spec_queue(*b->xo, b->st, b->d_out.as<float>(), J, p, o);
}

int sgb_rows_spectrogram(int32_t device, const float *src, const int64_t *src_off, const int64_t *len, int32_t n,
                         const sgb_spec_params *p, const sgb_device_out *o) {
  SpecJob J;
  int rc = spec_params(p, J);
  if (rc != SGB_OK) return rc;
  if ((rc = rows_device_check(device, src, n)) != SGB_OK) return rc;
  if (n > 0 && !src_off) return fail(SGB_ERR_INVALID, "null src_off");
  rc = spec_rows(p, n > 0 ? src : nullptr, src_off, len, n, o, device, J);
  if (rc != SGB_OK) return rc;
  DeviceExport *D;
  if ((rc = device_export(device, &D)) != SGB_OK) return rc;
  std::lock_guard<std::mutex> g(D->mu);
  return spec_queue(D->x, D->st, src, J, p, o);
}

// ---- similarity of spectrogram rows (K10) ----
int sgb_rows_compare(int32_t device, const float *a, int64_t a_elems, const float *b, int64_t b_elems,
                     const int64_t *a_off, const int64_t *a_frames, const int64_t *b_off, const int64_t *b_frames,
                     int32_t n, const sgb_compare_params *p, double *dst, int64_t dst_elems, void *stream) {
  // the parameters and the row tables alone (no device needed)
  if (!p) return fail(SGB_ERR_INVALID, "null sgb_compare_params");
  if (p->method != SGB_CMP_COR && p->method != SGB_CMP_COSINE && p->method != SGB_CMP_DTW)
    return fail(SGB_ERR_INVALID, "unknown method %d", p->method);
  if (p->n_feat < 1) return fail(SGB_ERR_INVALID, "n_feat %d < 1", p->n_feat);
  if (!std::isfinite(p->pad)) return fail(SGB_ERR_INVALID, "pad %g is not finite", p->pad);
  if (n < 0 || a_elems < 0 || b_elems < 0 || dst_elems < 0) return fail(SGB_ERR_INVALID, "negative count");
  if (n > 0 && (!a_off || !a_frames || !b_off || !b_frames)) return fail(SGB_ERR_INVALID, "null row table");
  std::vector<int64_t> tab(4 * (size_t)n);       // a_off, a_frames, b_off, b_frames per pair (the kernel's Pair)
  int64_t max_short = 0;
  bool any_cells = false;                         // a pair with frames on both sides reads a and b
  for (int32_t c = 0; c < n; c++) {
    const int64_t ao = a_off[c], af = a_frames[c], bo = b_off[c], bf = b_frames[c];
    if (ao < 0 || af < 0 || bo < 0 || bf < 0) return fail(SGB_ERR_INVALID, "pair %d: negative offset or frames", c);
    if (ao > a_elems || af > (a_elems - ao) / p->n_feat)
      return fail(SGB_ERR_INVALID, "pair %d: row of a [%lld, %lld x %d more) outside a (%lld elements)", c,
                  (long long)ao, (long long)af, p->n_feat, (long long)a_elems);
    if (bo > b_elems || bf > (b_elems - bo) / p->n_feat)
      return fail(SGB_ERR_INVALID, "pair %d: row of b [%lld, %lld x %d more) outside b (%lld elements)", c,
                  (long long)bo, (long long)bf, p->n_feat, (long long)b_elems);
    if (p->method == SGB_CMP_DTW && (af > SGB_CMP_DTW_MAX_FRAMES || bf > SGB_CMP_DTW_MAX_FRAMES))
      return fail(SGB_ERR_UNSUPPORTED, "pair %d: DTW over %lld x %lld frames (at most %d per row)", c, (long long)af,
                  (long long)bf, SGB_CMP_DTW_MAX_FRAMES);
    if (af > 0 && bf > 0) {
      any_cells = true;
      max_short = std::max(max_short, std::min(af, bf));
    }
    tab[4 * (size_t)c] = ao; tab[4 * (size_t)c + 1] = af; tab[4 * (size_t)c + 2] = bo; tab[4 * (size_t)c + 3] = bf;
  }
  if (n > 0 && dst_elems < n) return fail(SGB_ERR_INVALID, "dst has %lld elements for %d scores", (long long)dst_elems, n);
  int rc = rows_device_check(device, nullptr, 0);
  if (rc != SGB_OK) return rc;
  if (n == 0) return SGB_OK;
  if (!dst) return fail(SGB_ERR_INVALID, "null dst");
  if ((uintptr_t)dst % 8) return fail(SGB_ERR_INVALID, "dst is not aligned to double");
  if ((rc = on_device(device, dst, "dst")) != SGB_OK) return rc;
  if (any_cells) {
    if (!a || (uintptr_t)a % 4 || !b || (uintptr_t)b % 4) return fail(SGB_ERR_INVALID, "null or misaligned a / b");
    if ((rc = on_device(device, a, "a")) != SGB_OK || (rc = on_device(device, b, "b")) != SGB_OK) return rc;
  }
  DeviceExport *D;
  if ((rc = device_export(device, &D)) != SGB_OK) return rc;
  std::lock_guard<std::mutex> g(D->mu);
  const size_t bytes = sizeof(int64_t) * tab.size();
  auto fill = [&](char *h) { memcpy(h, tab.data(), bytes); };
  auto launch = [&](const char *d) -> int {
    cudaError_t e = launch_spec_compare(a, b, d, n, p->method, p->n_feat, p->pad, max_short, dst, D->st);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(SGB_ERR_CUDA, "k_spec_compare launch failed (%d pairs, %zu bytes of shared memory): %s", n,
                  spec_compare_smem_bytes(p->method, max_short), cudaGetErrorString(e));
    }
    return SGB_OK;
  };
  return export_queue(D->x, D->st, (cudaStream_t)stream, bytes, fill, launch);
}

// ---- cepstra of spectrogram rows (K11) ----
int sgb_rows_cepstra(int32_t device, const float *src, int64_t src_elems, const int64_t *src_off, const int64_t *frames,
                     int32_t n, const sgb_ceps_params *p, const sgb_device_out *o) {
  // the parameters and the source rows alone (no device needed)
  if (!p) return fail(SGB_ERR_INVALID, "null sgb_ceps_params");
  if (p->n_in < 1 || p->n_ceps < 1) return fail(SGB_ERR_INVALID, "n_in %d, n_ceps %d: at least 1 each", p->n_in, p->n_ceps);
  if (p->delta_order < 0 || p->delta_order > 2) return fail(SGB_ERR_INVALID, "delta_order %d not 0, 1 or 2", p->delta_order);
  if (p->delta_n < 1 || p->delta_n > 8) return fail(SGB_ERR_INVALID, "delta_n %d outside 1..8", p->delta_n);
  if (!p->matrix) return fail(SGB_ERR_INVALID, "null matrix");
  const size_t smem = cepstra_smem_bytes(p->n_in, p->n_ceps, p->delta_order, p->delta_n);
  if (smem > 226 * 1024)
    return fail(SGB_ERR_UNSUPPORTED, "%d inputs, %d cepstra, delta order %d over %d frames: %zu bytes of shared memory",
                p->n_in, p->n_ceps, p->delta_order, p->delta_n, smem);
  const int64_t n_m = (int64_t)p->n_ceps * p->n_in;
  for (int64_t i = 0; i < n_m; i++)
    if (!std::isfinite(p->matrix[i])) return fail(SGB_ERR_INVALID, "matrix element %lld is not finite", (long long)i);
  if (n < 0 || src_elems < 0) return fail(SGB_ERR_INVALID, "negative row count or src_elems");
  if (n > 0 && (!src_off || !frames)) return fail(SGB_ERR_INVALID, "null row table");
  for (int32_t c = 0; c < n; c++) {
    const int64_t so = src_off[c], nc = frames[c];
    if (so < 0 || nc < 0) return fail(SGB_ERR_INVALID, "row %d: negative source offset or frames", c);
    if (nc > INT32_MAX) return fail(SGB_ERR_INVALID, "row %d: %lld frames (at most 2^31 - 1)", c, (long long)nc);
    if (so > src_elems || nc > (src_elems - so) / p->n_in)
      return fail(SGB_ERR_INVALID, "row %d: elements [%lld, %lld x %d more) outside src (%lld elements)", c,
                  (long long)so, (long long)nc, p->n_in, (long long)src_elems);
  }
  int rc = rows_device_check(device, src, n);
  if (rc != SGB_OK) return rc;
  const int n_out = p->n_ceps * (1 + p->delta_order);
  if ((rc = export_check(device, n > 0 ? src : nullptr, src_off, frames, n, o, n_out, false)) != SGB_OK) return rc;
  std::vector<CepsRow> rows((size_t)n);
  std::vector<CepsTile> tiles;
  const int64_t zf = std::max(1, 8192 / n_out);       // zero tails: about 8192 floats per tile
  for (int32_t c = 0; c < n; c++) {
    if (o->cap[c] > INT32_MAX) return fail(SGB_ERR_INVALID, "row %d: %lld frames of capacity (at most 2^31 - 1)", c,
                                           (long long)o->cap[c]);
    const int32_t nc = (int32_t)frames[c], cap = (int32_t)o->cap[c], m = std::min(nc, cap);
    rows[c] = CepsRow{src_off[c], o->dst_off[c], nc, cap};
    for (int64_t t = 0; t < m; t += CEPS_TILE)
      tiles.push_back(CepsTile{c, (int32_t)t, (int32_t)std::min<int64_t>(m, t + CEPS_TILE), 0});
    for (int64_t t = m; t < cap; t += zf) tiles.push_back(CepsTile{c, (int32_t)t, (int32_t)std::min<int64_t>(cap, t + zf), 1});
  }
  if (tiles.size() > (size_t)INT32_MAX) return fail(SGB_ERR_UNSUPPORTED, "too many tiles");
  if (!tiles.empty() && src_elems > 0) {             // the kernel reads src while it writes dst
    const char *s0 = reinterpret_cast<const char *>(src), *s1 = s0 + 4 * src_elems;
    const char *d0 = reinterpret_cast<const char *>(o->dst), *d1 = d0 + 4 * o->dst_elems;
    if (d0 < s1 && s0 < d1) return fail(SGB_ERR_INVALID, "dst overlaps src");
  }
  DeviceExport *D;
  if ((rc = device_export(device, &D)) != SGB_OK) return rc;
  std::lock_guard<std::mutex> g(D->mu);
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t o_tiles = up16(sizeof(CepsRow) * rows.size()), o_m = up16(o_tiles + sizeof(CepsTile) * tiles.size());
  const size_t bytes = o_m + sizeof(float) * (size_t)n_m;
  auto fill = [&](char *h) {
    if (n) memcpy(h, rows.data(), sizeof(CepsRow) * rows.size());
    if (!tiles.empty()) memcpy(h + o_tiles, tiles.data(), sizeof(CepsTile) * tiles.size());
    memcpy(h + o_m, p->matrix, sizeof(float) * (size_t)n_m);
  };
  auto launch = [&](const char *d) -> int {
    cudaError_t e = launch_cepstra(reinterpret_cast<const CepsTile *>(d + o_tiles), (int)tiles.size(),
                                   reinterpret_cast<const CepsRow *>(d), reinterpret_cast<const float *>(d + o_m), src,
                                   (float *)o->dst, p->n_in, p->n_ceps, p->delta_order, p->delta_n, D->st);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(SGB_ERR_CUDA, "k_cepstra launch failed (%zu tiles, %zu bytes of shared memory): %s", tiles.size(),
                  smem, cudaGetErrorString(e));
    }
    return SGB_OK;
  };
  if ((rc = export_queue(D->x, D->st, (cudaStream_t)o->stream, bytes, fill, launch)) != SGB_OK) return rc;
  if (o->out_written)
    for (int32_t c = 0; c < n; c++) o->out_written[c] = std::min(frames[c], o->cap[c]);
  return SGB_OK;
}

// ---- f0 track of the last run (K12a) ----
int sgb_batch_f0(sgb_batch *b, const sgb_device_out *o) {
  if (!b) return fail(SGB_ERR_INVALID, "null batch");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  CK(cudaSetDevice(b->device));
  const int32_t n = (int32_t)b->call_len.size();
  const int S = (int)b->syls.size();
  int rc = export_check(b->device, nullptr, nullptr, b->call_len.data(), n, o, 1, false);
  if (rc != SGB_OK) return rc;
  // voiced spans: syllables of kind 1 that synthesised, in calls that did, where they land in the call's output
  // (bout start + final_shift + the syllable's place in `sound`, cut at filt_len: istft overlap-adds at the stft
  // frame starts, so positions in the filtered bout are positions in `sound`)
  std::vector<F0Span> spans;
  std::vector<F0Chunk> chunks;
  for (int32_t c = 0; c < n; c++) {
    const int32_t s_lo = (int32_t)spans.size();
    if (b->call_status[c] == SGB_OK) {
      const sgb_call &CL = b->calls[c];
      for (int bi = CL.bout_begin; bi < CL.bout_end; bi++) {
        const BoutLayout &L = b->bl[bi];
        const int64_t t_bout = L.out_off - b->call_off[c] + L.final_shift;
        for (int s = b->bouts[bi].syl_begin; s < b->bouts[bi].syl_end; s++) {
          if (b->syls[s].kind != 1 || b->summary[s].status != SGB_OK) continue;
          const int64_t r0 = b->place[s].dst_off - L.sound_off;
          const int64_t m = std::min<int64_t>(b->place[s].len, L.filt_len - r0);
          if (m > 0) spans.push_back(F0Span{t_bout + r0, (int32_t)m, s});
        }
      }
    }
    const int32_t s_hi = (int32_t)spans.size();
    int32_t sp = s_lo;
    for (int64_t k = 0; k * F0_CHUNK < o->cap[c]; k++) {
      while (sp < s_hi && spans[sp].t0 + spans[sp].n <= k * F0_CHUNK) sp++;
      chunks.push_back(F0Chunk{c, (int32_t)k, sp, s_hi});
    }
  }
  if (chunks.size() > (size_t)INT32_MAX) return fail(SGB_ERR_UNSUPPORTED, "too many chunks");
  CK(b->d_f0ep.ensure(sizeof(F0Epochs) * (size_t)std::max(S, 1)));
  if (!b->xo) b->xo = new ExportCtx();
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t o_spans = up16(16 * (size_t)n), o_chunks = up16(o_spans + sizeof(F0Span) * spans.size());
  const size_t bytes = o_chunks + sizeof(F0Chunk) * chunks.size();
  auto fill = [&](char *h) {
    int64_t *t = reinterpret_cast<int64_t *>(h);
    for (int32_t c = 0; c < n; c++) { t[c] = o->dst_off[c]; t[n + c] = o->cap[c]; }
    if (!spans.empty()) memcpy(h + o_spans, spans.data(), sizeof(F0Span) * spans.size());
    if (!chunks.empty()) memcpy(h + o_chunks, chunks.data(), sizeof(F0Chunk) * chunks.size());
  };
  auto launch = [&](const char *d) -> int {
    const int64_t *t = reinterpret_cast<const int64_t *>(d);
    cudaError_t e = launch_f0_track(b->d_syls.as<sgb_syllable>(), S, b->d_ctrl.as<SylCtrl>(), b->pools,
                                    b->d_f0ep.as<F0Epochs>(), reinterpret_cast<const F0Chunk *>(d + o_chunks),
                                    (int)chunks.size(), t, t + n, reinterpret_cast<const F0Span *>(d + o_spans),
                                    (float *)o->dst, b->st);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(SGB_ERR_CUDA, "k_f0_track launch failed (%zu chunks): %s", chunks.size(), cudaGetErrorString(e));
    }
    return SGB_OK;
  };
  // on the handle's stream, like the export: the handle's next run cannot overwrite the spline or SylCtrl first
  if ((rc = export_queue(*b->xo, b->st, (cudaStream_t)o->stream, bytes, fill, launch)) != SGB_OK) return rc;
  if (o->out_written)
    for (int32_t c = 0; c < n; c++) o->out_written[c] = std::min(b->call_len[c], o->cap[c]);
  return SGB_OK;
}

// ---- frame labels of f0 tracks (K12b) ----
int sgb_rows_f0_frames(int32_t device, const float *src, int64_t src_elems, const int64_t *src_off, const int64_t *len,
                       int32_t n, int32_t wl, double overlap, const sgb_device_out *o) {
  // the parameters and the source rows alone (no device needed)
  if (wl < 4 || (wl & 1)) return fail(SGB_ERR_INVALID, "window of %d points: an even wl >= 4 is needed", wl);
  if (!(overlap >= 0.0 && overlap < 100.0)) return fail(SGB_ERR_INVALID, "overlap %g out of [0, 100)", overlap);
  const double h = wl - (overlap * wl / 100.0);
  if (!(h >= 1.0)) return fail(SGB_ERR_INVALID, "hop %g of a %d-point window is below one sample", h, wl);
  if (!o) return fail(SGB_ERR_INVALID, "null sgb_device_out");
  if (o->format != SGB_OUT_F32) return fail(SGB_ERR_INVALID, "unsupported output format %d", o->format);
  if (n < 0 || src_elems < 0) return fail(SGB_ERR_INVALID, "negative row count or src_elems");
  if (n > 0 && (!src_off || !len)) return fail(SGB_ERR_INVALID, "null row table");
  for (int32_t c = 0; c < n; c++) {
    const int64_t so = src_off[c], ln = len[c];
    if (so < 0 || ln < 0) return fail(SGB_ERR_INVALID, "row %d: negative source offset or length", c);
    if (so > src_elems || ln > src_elems - so)
      return fail(SGB_ERR_INVALID, "row %d: samples [%lld, %lld more) outside src (%lld elements)", c, (long long)so,
                  (long long)ln, (long long)src_elems);
  }
  int rc = rows_device_check(device, src, n);
  if (rc != SGB_OK) return rc;
  if ((rc = export_check(device, n > 0 ? src : nullptr, src_off, len, n, o, 2, false)) != SGB_OK) return rc;
  std::vector<F0Row> rows((size_t)n);
  std::vector<F0Seg> segs;
  for (int32_t c = 0; c < n; c++) {
    if (o->cap[c] > INT32_MAX) return fail(SGB_ERR_INVALID, "row %d: %lld frames of capacity (at most 2^31 - 1)", c,
                                           (long long)o->cap[c]);
    const int64_t nc = spec_nc(len[c], wl, h), m = std::min(nc, o->cap[c]);
    rows[c] = F0Row{src_off[c], o->dst_off[c], len[c], nc, o->cap[c]};
    for (int64_t k = 0; k < m; k += F0F_FRAMES)
      segs.push_back(F0Seg{c, (int32_t)k, (int32_t)std::min<int64_t>(m, k + F0F_FRAMES), 0});
    for (int64_t k = m; k < o->cap[c]; k += 4096)    // zero tails: 8192 floats per segment
      segs.push_back(F0Seg{c, (int32_t)k, (int32_t)std::min<int64_t>(o->cap[c], k + 4096), 1});
  }
  if (segs.size() > (size_t)INT32_MAX) return fail(SGB_ERR_UNSUPPORTED, "too many segments");
  if (!segs.empty() && src_elems > 0) {               // the kernel reads src while it writes dst
    const char *s0 = reinterpret_cast<const char *>(src), *s1 = s0 + 4 * src_elems;
    const char *d0 = reinterpret_cast<const char *>(o->dst), *d1 = d0 + 4 * o->dst_elems;
    if (d0 < s1 && s0 < d1) return fail(SGB_ERR_INVALID, "dst overlaps src");
  }
  DeviceExport *D;
  if ((rc = device_export(device, &D)) != SGB_OK) return rc;
  std::lock_guard<std::mutex> g(D->mu);
  const size_t o_segs = (sizeof(F0Row) * rows.size() + 15) & ~(size_t)15;
  const size_t bytes = o_segs + sizeof(F0Seg) * segs.size();
  auto fill = [&](char *hp) {
    if (n) memcpy(hp, rows.data(), sizeof(F0Row) * rows.size());
    if (!segs.empty()) memcpy(hp + o_segs, segs.data(), sizeof(F0Seg) * segs.size());
  };
  auto launch = [&](const char *d) -> int {
    cudaError_t e = launch_f0_frames(reinterpret_cast<const F0Seg *>(d + o_segs), (int)segs.size(),
                                     reinterpret_cast<const F0Row *>(d), src, wl, h, (float *)o->dst, D->st);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(SGB_ERR_CUDA, "k_f0_frames launch failed (%zu segments): %s", segs.size(), cudaGetErrorString(e));
    }
    return SGB_OK;
  };
  if ((rc = export_queue(D->x, D->st, (cudaStream_t)o->stream, bytes, fill, launch)) != SGB_OK) return rc;
  if (o->out_written)
    for (int32_t c = 0; c < n; c++) o->out_written[c] = std::min(rows[c].nc, rows[c].cap);
  return SGB_OK;
}

// Diagnostic for a stuck run (callable from another thread): out[0] = which wait the handle's host thread
// is in (0 none, 10 upload, 1 after control, 2 after compose, 3 end of run), out[1 + i] = 1 if stage event i
// of the current run has been passed by the stream (needs SGB_TRACE=1; events: start, control, ampl, synth, compose, assemble,
// envelope, noise, filter, finalize, end).
int sgb_batch_debug_state(sgb_batch *b, int32_t *out, int32_t cap) {
  if (!b || !out || cap < 12) return fail(SGB_ERR_INVALID, "bad argument");
  out[0] = b->where;
  for (int i = 0; i <= 10; i++) out[1 + i] = b->reached[i];   // no CUDA call here: the driver may be wedged
  return SGB_OK;
}

// Diagnostic: position-weighted 64-bit checksums of the intermediates of the last run
// (0 control pools, 1 spline pieces, 2 tiles, 3 FP32 amplitude table, 4 FP64 amplitude matrices,
//  5 epoch waveforms, 6 composed syllables, 7 bout sounds, 8 output).  Used by the determinism tests.
int sgb_batch_checksums(sgb_batch *b, uint64_t *out, int32_t cap) {
  if (!b || !out || cap < 9) return fail(SGB_ERR_INVALID, "bad argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  CK(cudaSetDevice(b->device));
  DBuf d;
  CK(d.ensure(8 * 16));
  CK(cudaMemsetAsync(d.p, 0, 8 * 16, b->st));
  unsigned long long *acc = d.as<unsigned long long>();
  auto sum = [&](int slot, const void *p, size_t bytes) {
    size_t n = bytes / 4;
    if (!p || n == 0) return;
    k_checksum<<<1024, 256, 0, b->st>>>((const uint32_t *)p, n, acc + slot);
  };
  const size_t g = (size_t)b->gc_total;
  sum(0, b->pools.gcup, 4 * g); sum(0, b->pools.kt, 8 * g); sum(0, b->pools.ppg, 8 * g); sum(0, b->pools.phi, 8 * g);
  sum(1, b->pools.pc, 8 * g * SYNTH_PC);
  sum(2, b->d_tiles.p, sizeof(SynthTile) * (size_t)b->last_tiles);
  sum(2, b->d_epmax.p, 4 * b->syls.size() * SGB_MAX_EPOCHS);
  sum(3, b->d_amp32.p, 16 * (size_t)b->last_amp);
  sum(4, b->d_amp.p, 8 * (size_t)b->last_amp);
  sum(5, b->d_wave.p, 4 * (size_t)b->last_wave);
  sum(6, b->d_raw.p, 4 * (size_t)b->last_raw);
  sum(7, b->d_sound.p, 4 * (size_t)b->last_sound);
  sum(8, b->d_out.p, 4 * (size_t)b->total_out);
  CK(cudaMemcpyAsync(out, d.p, 8 * 9, cudaMemcpyDeviceToHost, b->st));
  CK(wait_stream(b));
  d.release();
  return SGB_OK;
}

int sgb_batch_syllable_len(sgb_batch *b, int32_t syl, int64_t *out_len) {
  if (!b || !out_len) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  if (syl < 0 || syl >= (int)b->syls.size()) return fail(SGB_ERR_INVALID, "syllable index");
  if (b->summary[syl].status != SGB_OK) return fail(b->summary[syl].status, "syllable %d failed (status %d)", syl, b->summary[syl].status);
  *out_len = b->place[syl].len;
  return SGB_OK;
}

int sgb_batch_syllable_fetch(sgb_batch *b, int32_t syl, double *out, int64_t n) {
  int64_t len = 0;
  int rc = sgb_batch_syllable_len(b, syl, &len);
  if (rc) return rc;
  if (!b->keep_voiced) return fail(SGB_ERR_STATE, "intermediates are kept only for batches of <= 64 calls");
  if (n < len) return fail(SGB_ERR_INVALID, "buffer too small");
  CK(cudaSetDevice(b->device));
  std::vector<float> tmp((size_t)len);
  CK(cudaMemcpy(tmp.data(), b->d_voiced.as<float>() + b->place[syl].dst_off, 4 * (size_t)len, cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < len; i++) out[i] = (double)tmp[i];
  return SGB_OK;
}

int sgb_batch_noise_fetch(sgb_batch *b, int32_t noise, double *out, int64_t n) {
  if (!b || !out) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  if (noise < 0 || noise >= (int)b->noises.size()) return fail(SGB_ERR_INVALID, "noise index");
  int64_t len = b->noises[noise].len;
  if (n < len) return fail(SGB_ERR_INVALID, "buffer too small");
  CK(cudaSetDevice(b->device));
  std::vector<float> tmp((size_t)len);
  CK(cudaMemcpy(tmp.data(), b->d_noise_fin.as<float>() + b->nl[noise].raw_off, 4 * (size_t)len, cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < len; i++) out[i] = (double)tmp[i];
  return SGB_OK;
}

static int get_ctrl(sgb_batch *b, int32_t syl, SylCtrl *C) {
  if (!b) return fail(SGB_ERR_INVALID, "null batch");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no completed run");
  if (syl < 0 || syl >= (int)b->syls.size()) return fail(SGB_ERR_INVALID, "syllable index");
  CK(cudaSetDevice(b->device));
  CK(cudaMemcpy(C, b->d_ctrl.as<SylCtrl>() + syl, sizeof(SylCtrl), cudaMemcpyDeviceToHost));
  return SGB_OK;
}

int sgb_batch_artefacts(sgb_batch *b, int32_t syl, sgb_syl_artefacts *out) {
  if (!out) return fail(SGB_ERR_INVALID, "null argument");
  SylCtrl C;
  int rc = get_ctrl(b, syl, &C);
  if (rc) return rc;
  out->nGC = C.nGC; out->nHarmonics = C.nHarmonics; out->rows_kept = C.rows_kept; out->nEpochs = C.nEpochs;
  out->n_upsampled = C.n_up; out->n_jitter_idx = C.n_jidx; out->z_used = C.z_used; out->status = C.status;
  out->raw_max = C.raw_max;
  return SGB_OK;
}

int sgb_batch_artefact_ints(sgb_batch *b, int32_t syl, int which, int32_t *out, int32_t cap) {
  if (!out) return fail(SGB_ERR_INVALID, "null argument");
  SylCtrl C;
  int rc = get_ctrl(b, syl, &C);
  if (rc) return rc;
  std::vector<int64_t> gc_off(2);
  CK(cudaMemcpy(gc_off.data(), b->d_gc_off.as<int64_t>() + syl, 8, cudaMemcpyDeviceToHost));
  const int64_t o = gc_off[0];
  const int32_t *src = nullptr;
  int n = 0;
  switch (which) {
    case 0: src = b->pools.gc + o; n = C.nGC; break;
    case 1: src = b->pools.gcup + o; n = C.nGC + 1; break;
    case 2: src = b->pools.nsub + o; n = C.nGC; break;
    case 3: src = b->pools.rwbin + o; n = C.nGC; break;
    case 4: src = b->pools.jidx + o; n = C.n_jidx; break;
    case 5:
      n = 2 * C.nEpochs;
      if (cap < n) return fail(SGB_ERR_INVALID, "buffer too small");
      for (int e = 0; e < C.nEpochs; e++) { out[2 * e] = C.ep_start[e]; out[2 * e + 1] = C.ep_end[e]; }
      return n;
    case 6:
      n = 2 * C.nEpochs;
      if (cap < n) return fail(SGB_ERR_INVALID, "buffer too small");
      for (int e = 0; e < C.nEpochs; e++) { out[2 * e] = C.ep_zc1[e]; out[2 * e + 1] = C.ep_zc2[e]; }
      return n;
    default: return fail(SGB_ERR_INVALID, "unknown artefact %d", which);
  }
  if (cap < n) return fail(SGB_ERR_INVALID, "buffer too small");
  if (n > 0) CK(cudaMemcpy(out, src, 4 * (size_t)n, cudaMemcpyDeviceToHost));
  return n;
}

// Diagnostic: K3's tables of one epoch of the last run.  shape = {rows, columns, pairs}; f64 gets the rows x columns
// FP64 matrix (column-major), f32 the epoch's 16-byte-per-element FP32 region as K3 left it (pairs: {Y, dY} packed
// at its start, zeros after; otherwise {Y, Y, dY, dY}).  Null f64 and f32 only report the shape.
int sgb_batch_amp_tables(sgb_batch *b, int32_t syl, int32_t epoch, double *f64, float *f32, int64_t cap,
                         int32_t *shape) {
  if (!shape) return fail(SGB_ERR_INVALID, "null argument");
  SylCtrl C;
  int rc = get_ctrl(b, syl, &C);
  if (rc) return rc;
  if (C.status != SGB_OK || C.nGC == 0) return fail(SGB_ERR_STATE, "syllable %d has no amplitude matrices", syl);
  if (epoch < 0 || epoch >= C.nEpochs) return fail(SGB_ERR_INVALID, "epoch index");
  const int64_t rows = C.ep_rows[epoch], cols = C.ep_end[epoch] - C.ep_start[epoch] + 1, n = rows * cols;
  shape[0] = (int32_t)rows; shape[1] = (int32_t)cols; shape[2] = rows >= b->last_tc_min_rows;
  if (!f64 && !f32) return SGB_OK;
  if (!f64 || !f32 || cap < n) return fail(SGB_ERR_INVALID, "buffer too small");
  SylLayout lay;
  CK(cudaMemcpy(&lay, b->d_lay.as<SylLayout>() + syl, sizeof(SylLayout), cudaMemcpyDeviceToHost));
  const int64_t off = lay.amp_off + C.ep_amp_off[epoch];
  CK(cudaMemcpy(f64, b->d_amp.as<double>() + off, 8 * (size_t)n, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(f32, b->d_amp32.as<float4>() + off, 16 * (size_t)n, cudaMemcpyDeviceToHost));
  return SGB_OK;
}

// Diagnostic: the FP32 envelope table K4 wrote for the main filter of bout `index` (kind 0) or for the filter of noise
// `index` (kind 1) in the last run, nr x nint column-major as K2 / K5 read it.  shape = {nr, nint}, {0, 0} for a
// bypassed bout or an unfiltered noise.  A null out only reports the shape.
int sgb_batch_envelope(sgb_batch *b, int32_t kind, int32_t index, float *out, int64_t cap, int32_t *shape) {
  if (!b || !shape) return fail(SGB_ERR_INVALID, "null argument");
  if (!b->have_run) return fail(SGB_ERR_STATE, "no run");
  int64_t off = -1;
  int32_t nr = 0, nint = 0;
  if (kind == 0) {
    if (index < 0 || index >= (int)b->bl.size()) return fail(SGB_ERR_INVALID, "bout index");
    const BoutLayout &L = b->bl[index];
    if (!L.bypass) { off = L.env_off; nr = L.wl / 2; nint = L.nint; }
  } else if (kind == 1) {
    if (index < 0 || index >= (int)b->nl.size()) return fail(SGB_ERR_INVALID, "noise index");
    const NoiseLayout &Q = b->nl[index];
    if (Q.env_off >= 0) { off = Q.env_off; nr = b->noises[index].wl / 2; nint = Q.nc_env; }
  } else {
    return fail(SGB_ERR_INVALID, "kind must be 0 (bout) or 1 (noise)");
  }
  shape[0] = nr; shape[1] = nint;
  const int64_t n = (int64_t)nr * nint;
  if (!out || n == 0) return SGB_OK;
  if (cap < n) return fail(SGB_ERR_INVALID, "buffer too small");
  CK(cudaSetDevice(b->device));
  CK(cudaMemcpyAsync(out, b->d_env.as<float>() + off, 4 * (size_t)n, cudaMemcpyDeviceToHost, b->st));
  CK(cudaStreamSynchronize(b->st));
  return SGB_OK;
}

int sgb_batch_pitch_per_gc(sgb_batch *b, int32_t syl, double *out, int32_t cap) {
  if (!out) return fail(SGB_ERR_INVALID, "null argument");
  SylCtrl C;
  int rc = get_ctrl(b, syl, &C);
  if (rc) return rc;
  if (cap < C.nGC) return fail(SGB_ERR_INVALID, "buffer too small");
  int64_t o;
  CK(cudaMemcpy(&o, b->d_gc_off.as<int64_t>() + syl, 8, cudaMemcpyDeviceToHost));
  if (C.nGC > 0) CK(cudaMemcpy(out, b->pools.ppg + o, 8 * (size_t)C.nGC, cudaMemcpyDeviceToHost));
  return C.nGC;
}

// ------------------------------------------------------------ single calls ---
int sgb_get_rolloff(const double *pitch_per_gc, int32_t nGC, int32_t nHarmonics, const double *rolloff,
                    int32_t n_rolloff, const double *rolloffOct, int32_t n_rolloffOct, const double *rolloffKHz,
                    int32_t n_rolloffKHz, double rolloffParab, double rolloffParabHarm,
                    double rolloffParabCeiling, double baseline, double throwaway, double samplingRate,
                    double *out, int32_t *out_rows) {
  if (!pitch_per_gc || !rolloff || !rolloffOct || !rolloffKHz || !out || !out_rows) return fail(SGB_ERR_INVALID, "null argument");
  if (nGC < 1 || nHarmonics < 2) return fail(SGB_ERR_INVALID, "need nGC >= 1 and nHarmonics >= 2");
  auto okn = [&](int n) { return n == 1 || n == nGC; };
  if (!okn(n_rolloff) || !okn(n_rolloffOct) || !okn(n_rolloffKHz)) return fail(SGB_ERR_INVALID, "vector arguments must have length 1 or nGC");
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) return fail(SGB_ERR_CUDA, "no CUDA device available (no CPU fallback)");
  DBuf dp, dr, dro, drk, dout, drows, dcm, dkept;
  int rc = SGB_OK;
  auto run = [&]() -> int {
    CK(dp.ensure(8 * (size_t)nGC)); CK(dr.ensure(8 * (size_t)n_rolloff)); CK(dro.ensure(8 * (size_t)n_rolloffOct));
    CK(drk.ensure(8 * (size_t)n_rolloffKHz)); CK(dout.ensure(8 * (size_t)nGC * nHarmonics)); CK(drows.ensure(16));
    CK(dcm.ensure(8 * (size_t)nGC)); CK(dkept.ensure(4 * (size_t)nHarmonics));
    CK(cudaMemcpy(dp.p, pitch_per_gc, 8 * (size_t)nGC, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dr.p, rolloff, 8 * (size_t)n_rolloff, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dro.p, rolloffOct, 8 * (size_t)n_rolloffOct, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(drk.p, rolloffKHz, 8 * (size_t)n_rolloffKHz, cudaMemcpyHostToDevice));
    launch_rolloff_api(dp.as<double>(), nGC, nHarmonics, dr.as<double>(), n_rolloff, dro.as<double>(), n_rolloffOct,
                              drk.as<double>(), n_rolloffKHz, rolloffParab, rolloffParabHarm, rolloffParabCeiling,
                              baseline, throwaway, samplingRate, dout.as<double>(), drows.as<int>(), dcm.as<double>(),
                              dkept.as<int>());
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout.p, 8 * (size_t)nGC * nHarmonics, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(out_rows, drows.p, 4, cudaMemcpyDeviceToHost));
    return SGB_OK;
  };
  rc = run();
  dp.release(); dr.release(); dro.release(); drk.release(); dout.release(); drows.release(); dcm.release(); dkept.release();
  return rc;
}

int sgb_get_spectral_envelope(int32_t nr, int32_t nc, const sgb_envelope *env, const double *formants,
                              const int32_t *formant_n, const double *mouth_anchors, double *out) {
  if (!env || !out) return fail(SGB_ERR_INVALID, "null argument");
  if (nr < 1 || nc < 1) return fail(SGB_ERR_INVALID, "nr and nc must be positive");
  if (env->n_formants < 0 || env->n_formants > SGB_MAX_FORMANTS)
    return fail(SGB_ERR_UNSUPPORTED, "%d formants (at most %d)", env->n_formants, SGB_MAX_FORMANTS);
  if (env->n_formants > 0 && (!formants || !formant_n)) return fail(SGB_ERR_INVALID, "formants missing");
  if (env->mouth_n > 0 && !mouth_anchors) return fail(SGB_ERR_INVALID, "mouth anchors missing");
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) return fail(SGB_ERR_CUDA, "no CUDA device available (no CPU fallback)");
  sgb_envelope E = *env;
  std::vector<sgb_formant_ref> refs(std::max(1, E.n_formants));
  int64_t rows = 0;
  for (int f = 0; f < E.n_formants; f++) {
    int n = E.tracks_given ? nc : formant_n[f];
    if (n < 1) return fail(SGB_ERR_INVALID, "formant %d has no rows", f);
    refs[f].off = rows; refs[f].n = n; refs[f].pad = 0; rows += n;
  }
  E.formant_off = 0; E.mouth_off = 0;
  EnvInst I; I.out_off = 0; I.env_id = 0; I.nr = nr; I.nc = nc; I.col0 = 0; I.trk_off = -1;
  int np = 0;
  if (!E.tracks_given) for (int f = 0; f < E.n_formants; f++) np = std::max(np, (int)refs[f].n);
  if (np > 1) {
    if (!(E.smoothLinearFactor <= 20.0)) return fail(SGB_ERR_UNSUPPORTED, "smoothLinearFactor above 20");
    I.trk_off = 0;
  }
  const int64_t env_knots = env_knot_layout(I, E, refs.data(), 0);
  if (E.mouth_n > 0 && !contour_fits(E.mouth_n, E.mouth_method, nc, 16000.0, true, 0.0, true, 1.0, mouth_anchors))
    return fail(SGB_ERR_SYNTH, "loess: span is too small (mouthAnchors)");
  DBuf dE, dR, dF, dA, dI, dO, dT, dM, dTab, dK;
  auto run = [&]() -> int {
    CK(dE.ensure(sizeof E)); CK(dR.ensure(sizeof(sgb_formant_ref) * refs.size())); CK(dF.ensure(32 * (size_t)std::max<int64_t>(rows, 1)));
    CK(dA.ensure(16 * (size_t)std::max(1, E.mouth_n))); CK(dI.ensure(sizeof I)); CK(dO.ensure(8 * (size_t)nr * nc));
    CK(cudaMemcpy(dE.p, &E, sizeof E, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dR.p, refs.data(), sizeof(sgb_formant_ref) * refs.size(), cudaMemcpyHostToDevice));
    if (rows) CK(cudaMemcpy(dF.p, formants, 32 * (size_t)rows, cudaMemcpyHostToDevice));
    if (E.mouth_n) CK(cudaMemcpy(dA.p, mouth_anchors, 16 * (size_t)E.mouth_n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dI.p, &I, sizeof I, cudaMemcpyHostToDevice));
    CK(dT.ensure(8 * (size_t)std::max(1, nc * E.n_formants * 3))); CK(dM.ensure(8 * (size_t)nc));
    CK(dTab.ensure(contour_tab_bytes())); CK(dK.ensure(8 * (size_t)std::max<int64_t>(env_knots, 1)));
    launch_env_tracks(dI.as<EnvInst>(), 1, dE.as<sgb_envelope>(), dR.as<sgb_formant_ref>(), dF.as<double>(),
                      dA.as<double>(), dT.as<double>(), dM.as<double>(), dTab.p, dK.as<double>(), 0);
    CKL("launch_env_tracks");
    CK(launch_envelope_f64(dI.as<EnvInst>(), 1, nc, E.n_formants, dE.as<sgb_envelope>(), dR.as<sgb_formant_ref>(),
                           dF.as<double>(), nullptr, dT.as<double>(), dM.as<double>(), nullptr, dO.as<double>(), 0));
    CK(cudaMemcpy(out, dO.p, 8 * (size_t)nr * nc, cudaMemcpyDeviceToHost));
    return SGB_OK;
  };
  int rc = run();
  dE.release(); dR.release(); dF.release(); dA.release(); dI.release(); dO.release(); dT.release(); dM.release();
  dTab.release(); dK.release();
  return rc;
}

int64_t sgb_filter_len(int64_t len, int32_t wl, double overlap) {
  if (len < 8 || wl < 4) return -1;
  int w = (int)std::min<int64_t>(wl, len / 2);
  double h_in = w - (overlap * w / 100.0), h_out = w * (100.0 - overlap) / 100.0;
  int nc = seq_by_count(1.0, std::max<double>(1.0, (double)(len - w)), h_in);
  return (int64_t)std::floor(w + (nc - 1) * h_out);
}

int sgb_filter(const double *sound, int64_t len, const double *envelope, int32_t nInt, int32_t wl,
               double overlap, double *out, int64_t out_cap) {
  if (!sound || !envelope || !out) return fail(SGB_ERR_INVALID, "null argument");
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) return fail(SGB_ERR_CUDA, "no CUDA device available (no CPU fallback)");
  if (len < 8 || len > 2000000000LL) return fail(SGB_ERR_INVALID, "sound length out of range");
  if (!(overlap >= 0.0 && overlap < 100.0)) return fail(SGB_ERR_INVALID, "overlap out of range");
  int w = (int)std::min<int64_t>(wl, len / 2);     // soundgen.R:743
  if (w < 4 || (w & 1)) return fail(SGB_ERR_UNSUPPORTED, "window of %d points (odd or < 4) is not supported", w);
  PlanTable PT;
  int pi = PT.get(w, overlap);
  if (pi < 0) return fail(SGB_ERR_UNSUPPORTED, "cannot factor window length %d", w);
  const FftPlan &pl = PT.plans[pi];
  const int nr = w / 2;
  const int nc = seq_by_count(1.0, std::max<double>(1.0, (double)(len - w)), pl.h_in);
  if (nInt != 1 && nInt != nc) return fail(SGB_ERR_INVALID, "envelope must have 1 or %d columns, got %d", nc, nInt);
  const int64_t xlen = (int64_t)std::floor(w + (nc - 1) * pl.h_out);
  if (out_cap < xlen) return fail(SGB_ERR_INVALID, "output buffer too small: need %lld", (long long)xlen);
  size_t smem = stft_smem_bytes(w, pl.h_in, pl.h_out, 0);
  if (smem > 226 * 1024) return fail(SGB_ERR_UNSUPPORTED, "window too long for shared memory");
  FftJob J; memset(&J, 0, sizeof J);
  J.in_off = 0; J.out_off = 0; J.env_off = 0; J.plan = 0; J.nc = nc; J.nint = nInt; J.xlen = (int32_t)xlen;
  J.out_len = (int32_t)xlen; J.shift = 0; J.max_slot = 0;
  std::vector<FftJob> jobs(1, J);
  std::vector<FftSeg> segs;
  std::vector<SegGroup> groups;
  make_segs(jobs, PT.plans, 0, segs, groups);
  DBuf d64, dS, dE64, dE, dO, dPl, dTw, dWin, dJ, dSg, dMax, dO64;
  auto run = [&]() -> int {
    const size_t nenv = (size_t)nr * nInt;
    CK(d64.ensure(8 * (size_t)len)); CK(dS.ensure(4 * (size_t)(len + w + 64))); CK(dE64.ensure(8 * nenv));
    CK(dE.ensure(4 * nenv)); CK(dO.ensure(4 * (size_t)(xlen + 64))); CK(dO64.ensure(8 * (size_t)(xlen + 64)));
    CK(dPl.ensure(sizeof(FftPlan))); CK(dTw.ensure(8 * PT.tw.size())); CK(dWin.ensure(4 * PT.win.size()));
    CK(dJ.ensure(sizeof(FftJob))); CK(dSg.ensure(sizeof(FftSeg) * segs.size())); CK(dMax.ensure(16));
    CK(cudaMemcpy(d64.p, sound, 8 * (size_t)len, cudaMemcpyHostToDevice));
    CK(cudaMemset(dS.p, 0, 4 * (size_t)(len + w + 64)));
    k_f64_to_f32<<<(unsigned)((len + 255) / 256), 256>>>(d64.as<double>(), dS.as<float>(), len);
    CK(cudaMemcpy(dE64.p, envelope, 8 * nenv, cudaMemcpyHostToDevice));
    k_f64_to_f32<<<(unsigned)((nenv + 255) / 256), 256>>>(dE64.as<double>(), dE.as<float>(), (int64_t)nenv);
    CK(cudaMemcpy(dPl.p, &pl, sizeof(FftPlan), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dTw.p, PT.tw.data(), 8 * PT.tw.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dWin.p, PT.win.data(), 4 * PT.win.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dJ.p, &J, sizeof J, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dSg.p, segs.data(), sizeof(FftSeg) * segs.size(), cudaMemcpyHostToDevice));
    k_fill_int<<<1, 32>>>(dMax.as<int>(), 4, ORDERED_NEG_INF);
    CK(launch_stft(0, 0, groups[0].spec, dSg.as<FftSeg>(), (int)segs.size(), dJ.as<FftJob>(), dPl.as<FftPlan>(),
                   dTw.as<float2>(), dWin.as<float>(), dS.as<float>(), nullptr, dE.as<float>(), dO.as<float>(),
                   dMax.as<int>(), groups[0].smem, 0));
    CK(cudaDeviceSynchronize());
    int mi;
    CK(cudaMemcpy(&mi, dMax.p, 4, cudaMemcpyDeviceToHost));
    int fi = (mi >= 0) ? mi : (mi ^ 0x7FFFFFFF);
    float mx;
    memcpy(&mx, &fi, 4);
    std::vector<float> tmp((size_t)xlen);
    CK(cudaMemcpy(tmp.data(), dO.p, 4 * (size_t)xlen, cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < xlen; i++) out[i] = (double)tmp[i] / (double)mx;   // soundgen.R:807
    return SGB_OK;
  };
  int rc = run();
  DBuf *all[] = {&d64, &dS, &dE64, &dE, &dO, &dPl, &dTw, &dWin, &dJ, &dSg, &dMax, &dO64};
  for (auto d : all) d->release();
  return rc;
}

}  // extern "C"
