// spart_kernels.cu -- sm_100a kernels and the C ABI of libspart_b200.so.
//
// Data flow for one batch (all buffers in HBM, struct-of-arrays over samples so that every
// warp-wide access is one or two fully used 128-byte lines):
//
//   params [27][n]  --lidf_kernel------>  ws rows F_1..F_12 [12][n]   (block = 128 samples x 12 angles: the
//        reference's truncated leaf-angle iteration, step for step, run as groups of 32 tasks sorted by
//        predicted step count)
//   params + F      --geometry_kernel-> rec [R_COUNT][n]   (one thread per sample: 13-class volume
//        scattering, hot-spot integrals, soil vector weights, SMAC geometry/pressure scalars, ET scale)
//   params + rec    --band_kernel---->  out [n][nb][3]      (one thread per sample, looping over a
//        chunk of <= 16 bands: PROSPECT + BSM + SAILH at the 1-2 wavelengths np.interp touches,
//        SMAC, TOC->TOA; <true> = all samples share the sun / view geometry)
//   params + rec    --spectrum_kernel-> spec [n][9][2162]   (leafopt/soilopt/canopyopt; thread = wavelength)
//   (soillib_* = the band / spectrum kernels with each sample's dry soil read from a soil library,
//    SPART_FLAG_SOIL_LIBRARY)
//
// In band_kernel / spectrum_kernel all lanes of a warp work on the same wavelength, so the
// per-wavelength and per-band constants are warp-uniform shared-memory broadcasts and the
// arithmetic is pure FP64-pipe work; see DESIGN.md for the roofline of each kernel.
#include <cuda_runtime.h>

#include <nvtx3/nvToolsExt.h>

#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/spart_b200.h"
#include "spart_device.cuh"
#include "spart_device_f32.cuh"
#include "lut_kernels.cuh"
#include "sobol_kernels.cuh"
#include "invert_kernels.cuh"

using namespace spart;

// tuning knobs (numeric; build alternatives with tools/build_alt.sh -D... and time them with
// SPART_B200_LIB=<so> python tools/kbench.py): SPART_BAND_CHUNK, SPART_BAND_THREADS, the *_MINBLOCKS values,
// SPART_LIDF_DEG, SPART_LIDF2_R / RA / RB / SUB, and SPART_TAU_SPLIT / SPART_LOG_SPLIT in spart_device.cuh
#ifndef SPART_BAND_CHUNK
#define SPART_BAND_CHUNK 16
#endif
#ifndef SPART_BAND_MINBLOCKS_U
#define SPART_BAND_MINBLOCKS_U 5
#endif
#ifndef SPART_SRF_MINBLOCKS
#define SPART_SRF_MINBLOCKS 5
#endif
#ifndef SPART_BAND_MINBLOCKS
#define SPART_BAND_MINBLOCKS 4
#endif
#ifndef SPART_SAMPLE_MINBLOCKS
#define SPART_SAMPLE_MINBLOCKS 5
#endif

static_assert(LC_COUNT == SPART_NLC, "LC layout");
static_assert(SM_COUNT == SPART_NSMAC, "SMAC layout");
static_assert(SM_USED <= SM_COUNT, "SMAC layout");
static_assert(P_COUNT == SPART_NPAR, "param layout");

// --------------------------------------------------------------------------------------
// error plumbing
// --------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static thread_local int64_t g_launches = 0;

static int fail(int code, const char* fmt, const char* detail = "") {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}
#define CUDA_TRY(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      snprintf(g_err, sizeof(g_err), "%s failed: %s", #expr, cudaGetErrorString(_e));    \
      return (int)_e;                                                                    \
    }                                                                                    \
  } while (0)

// Every kernel launch of the library goes through here, so spart_launch_count() counts each one and a failed
// launch is reported like any other failed CUDA call.
template <typename... KArgs, typename... Args>
static int launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  kernel<<<grid, block, smem, st>>>(std::forward<Args>(args)...);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return SPART_OK;
}

// --------------------------------------------------------------------------------------
// owners of CUDA resources: each releases its resource when it is destroyed or reset, and never writes g_err
// --------------------------------------------------------------------------------------
struct DeviceFree { void operator()(void* p) const { cudaFree(p); } };
struct PinnedFree { void operator()(void* p) const { cudaFreeHost(p); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
template <typename T = void> using DeviceBuf = std::unique_ptr<T, DeviceFree>;
using PinnedBuf = std::unique_ptr<void, PinnedFree>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;

// (Re)allocate a buffer; the old one is released first, so that a grown buffer never coexists with its predecessor.
template <typename T>
static cudaError_t alloc(DeviceBuf<T>& buf, size_t bytes) {
  buf.reset();
  T* p = nullptr;
  const cudaError_t e = cudaMalloc(&p, bytes);
  buf.reset(e == cudaSuccess ? p : nullptr);
  return e;
}
static cudaError_t alloc(PinnedBuf& buf, size_t bytes) {
  buf.reset();
  void* p = nullptr;
  const cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocDefault);
  buf.reset(e == cudaSuccess ? p : nullptr);
  return e;
}
static cudaError_t create(Event& ev, unsigned flags = cudaEventDefault) {
  cudaEvent_t e = nullptr;
  const cudaError_t r = cudaEventCreateWithFlags(&e, flags);
  ev.reset(r == cudaSuccess ? e : nullptr);
  return r;
}
static cudaError_t create(Stream& stream) {
  cudaStream_t s = nullptr;
  const cudaError_t r = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
  stream.reset(r == cudaSuccess ? s : nullptr);
  return r;
}

// --------------------------------------------------------------------------------------
// device-side band table: one row of BT_COUNT doubles per band
// --------------------------------------------------------------------------------------
enum BandTableCol {
  BT_SMAC = 0,                    // SM_COUNT folded SMAC constants
  BT_CONVEA = SM_COUNT,           // SRF-convolved extraterrestrial irradiance
  BT_FRAC,                        // np.interp offset (0 => single knot)
  BT_NPTS,                        // 1 or 2 wavelengths to evaluate
  BT_PAD,
  BT_LC0,                         // LC_COUNT constants at the lower knot
  BT_LC1 = BT_LC0 + LC_COUNT,     // LC_COUNT constants at the upper knot
  BT_COUNT = BT_LC1 + LC_COUNT
};

__constant__ double c_sin_ttli[13];
__constant__ double c_cos_ttli[13];

// Small persistent thread pool for the staging copies of the host-buffer path (pageable caller
// memory <-> pinned staging buffers).  parallel_for(n, f) runs f(0..n-1) on the workers and the
// calling thread and returns when all are done.
class HostPool {
 public:
  explicit HostPool(int workers) {
    for (int i = 0; i < workers; ++i) th_.emplace_back([this] { loop(); });
  }
  ~HostPool() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_work_.notify_all();
    for (auto& t : th_) t.join();
  }
  int size() const { return (int)th_.size() + 1; }
  void parallel_for(int n, const std::function<void(int)>& f) {
    if (n <= 0) return;
    {
      std::lock_guard<std::mutex> lk(mu_);
      job_ = &f;
      njobs_ = n;
      next_ = 0;
      left_ = n;
      ++gen_;
    }
    cv_work_.notify_all();
    drain();
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [this] { return left_ == 0; });
    job_ = nullptr;
  }

 private:
  void drain() {
    for (;;) {
      int i;
      const std::function<void(int)>* f;
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (!job_ || next_ >= njobs_) return;
        i = next_++;
        f = job_;
      }
      (*f)(i);
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (--left_ == 0) cv_done_.notify_all();
      }
    }
  }
  void loop() {
    uint64_t seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_work_.wait(lk, [&] { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
      }
      drain();
    }
  }
  std::vector<std::thread> th_;
  std::mutex mu_;
  std::condition_variable cv_work_, cv_done_;
  const std::function<void(int)>* job_ = nullptr;
  int njobs_ = 0, next_ = 0, left_ = 0;
  uint64_t gen_ = 0;
  bool stop_ = false;
};

struct SpartCtx {
  int device = 0;
  int n_sensors = 0;
  int sm_count = 0;
  DeviceBuf<double> d_lc;               // [LC_COUNT][SPART_NWL]
  std::vector<DeviceBuf<double>> d_band;     // per sensor [nb][BT_COUNT]
  std::vector<DeviceBuf<int32_t>> d_knot;    // per sensor [nb][2]: wl_lo, wl_hi (read by the soil-library kernels)
  std::vector<int> n_bands;
  // optional soil library (spart_create_with_soils): [n_soils + 1][SPART_NWL], the extra last row all NaN
  DeviceBuf<double> d_soils;
  int n_soils = 0;
  // optional SRF tables per sensor (band_mode "srf"): per band the number of non-zero weights and
  // its offset into the concatenated (wavelength index, normalised weight) lists; nullptr when
  // the sensor was created without them
  struct SrfDev {                       // device arrays behind one SrfPlan (all nullptr: no SRF tables)
    int n_wl = 0, n_slots = 0;
    DeviceBuf<int32_t> wl_idx, pair_off, pair_slot, fin_off, fin_band, fin_slot;
    DeviceBuf<double> pair_w;
  };
  std::vector<SrfDev> srf;
  // host-buffer path: lazily created slots (device params / workspace / output, and pinned host
  // staging buffers that are only allocated when the caller's memory is pageable)
  std::mutex mu;
  static const int kSlots = 4;
  Event slot_done[kSlots];                 // the slot's device->host copy has finished
  Event slot_k[kSlots];                    // the slot's kernels have finished
  Stream h2d_stream, d2h_stream;           // one stream per copy direction (see the host path)
  Stream compute_stream, join_stream;
  static const int kInSlots = 3;           // device buffers for the parameter spans of the host path
  DeviceBuf<> in_params[kInSlots];
  Event in_done[kInSlots];                 // the span's host->device copies have finished
  Event in_free[kInSlots];                 // the kernels of all chunks of the span have finished
  int64_t in_cap = 0;                      // samples per span buffer
  PinnedBuf bc_stage;                      // element 0 of the broadcast rows of the current call
  DeviceBuf<> in_ets[kInSlots];            // compact output: the span's etscale values, sent back once per span
  Event ets_done[kInSlots];
  DeviceBuf<double> slot_rec[kSlots];
  DeviceBuf<> slot_out[kSlots];
  PinnedBuf stage_in[kSlots];
  PinnedBuf stage_out[kSlots];
  int64_t slot_cap = 0;        // samples per slot
  size_t slot_out_cap = 0;     // bytes of output per slot
  size_t stage_in_cap = 0, stage_out_cap = 0;   // bytes
  std::unique_ptr<HostPool> pool;
  // optional per-kernel timing of spart_forward_bands (spart_profile_enable / _read)
  mutable std::mutex prof_mu;
  mutable bool profiling = false;
  struct ProfEvents { Event e[4]; };
  mutable std::vector<ProfEvents> prof_pending;
  mutable std::vector<ProfEvents> prof_free;
};

// --------------------------------------------------------------------------------------
// kernels
// --------------------------------------------------------------------------------------
constexpr int kSampleThreads = 128;
// internal launch flag (not part of the ABI): rows 19..21 are broadcast rows, i.e. the batch shares one
// sun / observer geometry by construction
constexpr int kFlagUniform = 1;
// internal launch flag: LIDFa and LIDFb are broadcast rows, the twelve F values were computed once (element 0)
constexpr int kFlagLidfBcast = 1 << 30;
// internal launch flag: the rows hold a caller-supplied leaf inclination distribution lidf_0..lidf_12 themselves
// (SPART_FLAG_USER_LIDF, spart_set_lidf) instead of the cumulative values F_1..F_12 of lidf_kernel
constexpr int kFlagLidfDirect = 1 << 29;
constexpr uint32_t kLidfRows = (1u << P_LIDFA) | (1u << P_LIDFB);
constexpr uint32_t kGeometryRows = (1u << P_SZA) | (1u << P_VZA) | (1u << P_RAA);

__constant__ double c_theta2[12];   // 2 * (pi/180) * theta for theta = 10..80 step 10, 82..88 step 2

#ifndef SPART_LIDF_DEG
#define SPART_LIDF_DEG 6         // degree of the Taylor model of y in stage B of lidf_kernel
#endif
constexpr int kLidfDeg = SPART_LIDF_DEG;

// u <- g(u): Horner evaluation of the degree-kLidfDeg polynomial map of stage B
__device__ __forceinline__ double lidf_poly(const double (&g)[kLidfDeg + 1], double u) {
  double r = g[kLidfDeg];
#pragma unroll
  for (int k = kLidfDeg - 1; k >= 0; --k) r = fma(r, u, g[k]);
  return r;
}

// workspace rows: the per-sample record followed by the 12 cumulative leaf-angle values
constexpr int kRowF = R_COUNT;
constexpr int kWsRows = R_COUNT + 13;     // (the 13th row is used by a caller-supplied distribution only)

// ---- Kernel 1: leaf inclination distribution (CanopyStructure.__init__, sailh.py:340-398) ----------------------
// The reference's dcum is the fixed-point iteration x <- x + (y(x) - x + theta2)/2, y = a sin x + b/2 sin 2x,
// stopped at |dx| <= 1e-8; its result depends on the number of steps taken, so the sequence of iterates has to be
// reproduced, not just its limit.  Exact steps (one sincos each) run until the iterate is close to the fixed point;
// from there on y is replaced by a degree-SPART_LIDF_DEG Taylor model around a point near the fixed point, one
// Horner evaluation per step (see lidf2_hand).  A block takes 128 samples, i.e. 12 x 128 (sample, angle) tasks,
// whose step counts vary widely; so that the 32 lanes of a warp run tasks of about the same length, the work is
// ordered by *predicted* length first:
//   A1  the first exact step of all 12 x 128 tasks of a block, without a sincos (x0 = theta2 is one of twelve
//       constants, whose sine / cosine sit in a table filled by the same sincos_small); from its |dx| and
//       y'(x0) the linear-convergence model predicts the remaining exact steps (or, for a task that hands
//       over at once, the polynomial steps) with two MUFU logarithms;
//   sort the block's 1536 tasks by predicted exact steps, longest first (counting sort, shared-memory atomics);
//   A2  warps fetch groups of 32 consecutive tasks from a block-wide counter and step them until none of the
//       32 runs any more (a vote per step); lanes of a group finish within a step or two of each other;
//   sort by predicted polynomial steps; B: the same with the Taylor-model steps (a vote every
//       SPART_LIDF2_RB steps); results are staged in shared memory and written as 12 coalesced rows.
// The predictions only decide the grouping, never a result: every task runs until its own stop criterion.
// The iteration is one long dependent FP64 chain per lane, so the kernel is kept apart from the others and
// needs the occupancy of SPART_LIDF2_MINBLOCKS blocks per SM to fill the FP64 pipe.
// (The round-1 version, a per-warp task queue, is in git history at 64fd57e.)
#ifndef SPART_LIDF2_RB
#define SPART_LIDF2_RB 4
#endif
#ifndef SPART_LIDF2_RA
#define SPART_LIDF2_RA 1
#endif
#ifndef SPART_LIDF2_R
#define SPART_LIDF2_R 0.15       // hand-over radius of the centred Taylor model
#endif
#ifndef SPART_LIDF2_MINBLOCKS
#define SPART_LIDF2_MINBLOCKS 8
#endif
#ifndef SPART_LIDF2_SUB
#define SPART_LIDF2_SUB 4        // counters per key class in the counting sorts (see lidf2_sort)
#endif
constexpr int kL2Threads = 128;
constexpr int kL2Samples = 128;               // samples per block; task t = angle * kL2Samples + sample
constexpr int kL2Tasks = 12 * kL2Samples;
constexpr int kL2Keys = 64;                   // key classes of the counting sorts
// Runaway guard of the step loops (votes per group).  Inside the model's domain |a| + |b| <= 1 a task needs at most
// ~110 exact and ~460 polynomial steps (on the boundary, where the contraction rate approaches 1); outside it the
// iteration need not converge at all (the reference would loop forever) -- such input ends here with garbage.
constexpr int kL2MaxVotes = 1 << 15;

struct Lidf2Smem {
  double x[kL2Tasks];            // x_1 -> hand-over iterate x_s (or 2 y + theta2 of a task that converged in stage A) -> F
  double a[kL2Samples], b[kL2Samples];
  double theta2[12], sin0[12], cos0[12];
  unsigned short perm[kL2Tasks];
  unsigned short rank[kL2Tasks];
  signed char dq[kL2Tasks];      // (expansion centre - hand-over iterate) * 2^8
  // per task: 0 = converged in stage A ("direct"), 1..63 = predicted polynomial steps of a handed-over task,
  // 128 + k = k more exact steps predicted
  unsigned char key[kL2Tasks];
  int bin[kL2Keys * SPART_LIDF2_SUB];
  int counter, nwork;
};

__device__ __forceinline__ float lidf2_rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float lidf2_lg2(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Hand-over test of an exact step at x with step dx and slope yp = y'(x).  Stage B expands around the Newton
// estimate xc = x + 2 dx / (1 - y') of the fixed point itself.  The truncation error c |x_n - xc|^7 of the
// degree-6 model is then largest for the first polynomial iterates, where it matters least: the iteration
// contracts an error made at distance d from the fixed point by ~1e-8 / d before the stop.  That admits a ten
// times larger hand-over radius than an expansion around the hand-over iterate,
// |2 dx / (1 - y')| <= R (1 - lam)^(1/3) with R = 0.15 (the cube root keeps slowly converging tasks, whose Newton
// estimate is poor and whose errors contract slowly, on exact steps for longer): 2.0 exact steps per task
// instead of 4.3 on the benchmark distribution (the first one is free) for 2.2 more polynomial steps, F within
// 9e-16 of the step-by-step iteration over the whole |a| + |b| <= 1 domain, its boundary included
// (tools/check_lidf_centred.py: NumPy prototype with the kernel's arithmetic; GPU: tools/lidf_parity_scale.py).
// The test is written without a division: 8 |dx|^3 <= R^3 (1 - y')^3 (1 - y') / 2.
__device__ __forceinline__ bool lidf2_hand(double adx, double yp) {
  const double w = 1.0 - yp, w2 = w * w;
  return adx * adx * adx <= (SPART_LIDF2_R * SPART_LIDF2_R * SPART_LIDF2_R / 16.0) * (w2 * w2);
}

// Sort key of a task that leaves an exact step unconverged, from the linear-convergence model in single
// precision (three MUFU.LG2 / RCP pairs; it only decides the grouping): lam = g'(x) = (1 + y') / 2,
//   hand-over:  polynomial steps until |du| = |dx| lam^(n+1) <= 1e-8            -> key 1 .. 63
//   otherwise:  exact steps until the distance |dx| lam^n 2 / (1 - y') <= radius  -> key 128 + (1 .. 31)
// and dq = (centre - next iterate) 2^8 with centre - next iterate =
// (x + 2 dx / (1 - y')) - (x + dx) = dx (1 + y') / (1 - y'): any point within ~1e-2 of the fixed point serves as
// expansion centre (the Newton estimate itself is no better), and xc = x_next + dq 2^-8 is exact in FP64.
__device__ __forceinline__ unsigned char lidf2_leave(double dx, double yp, bool hand, signed char& dq) {
  const float inv_radius = (float)(2.0 / SPART_LIDF2_R);
  const float ypf = (float)yp, dxf = (float)dx;
  const float rw = lidf2_rcp(1.0f - ypf);
  const float lam = fminf(fmaxf(fmaf(0.5f, ypf, 0.5f), 1e-3f), 0.9995f);
  const float r = lidf2_rcp(-lidf2_lg2(lam));
  const float num = fabsf(dxf) * lam * (hand ? 1e8f : inv_radius * rw);
  const int k = __float2int_ru(fminf(fmaxf(lidf2_lg2(num) * r, 0.0f), 100.0f));
  dq = (signed char)__float2int_rn(fminf(fmaxf(dxf * (1.0f + ypf) * rw * 256.0f, -127.0f), 127.0f));
  return hand ? (unsigned char)min(k + 1, 63) : (unsigned char)(128 + min(max(k, 1), 31));
}

// coefficients of the map g(u) = (u + y~(u) + k0) / 2 of stage B, y~ = sum_k y^(k)(xc) u^k / k!, from sin / cos of
// the expansion centre xc: y^(k) = a sin^(k) x + b 2^(k-1) sin^(k) 2x and sin^(k) cycles through (s, c, -s, -c).
// The products a sin, a cos, b sin 2x, b cos 2x are formed once: g_k = C_k (A_k + 2^(k-1) B_k), C_k = +-1 / (2 k!).
__device__ __forceinline__ void lidf2_poly_setup(double a, double b, double s, double c, double k0,
                                                 double (&g)[kLidfDeg + 1]) {
  const double s2 = 2.0 * s * c, c2 = fma(2.0 * c, c, -1.0);
  const double As = a * s, Ac = a * c, Bs = b * s2, Bc = b * c2;
  double fact = 1.0, pow2 = 0.5;        // k!, 2^(k-1)
#pragma unroll
  for (int k = 0; k <= kLidfDeg; ++k) {
    if (k > 0) {
      fact *= (double)k;
      pow2 *= 2.0;
    }
    const double sign = (k & 2) ? -1.0 : 1.0;
    g[k] = (sign * 0.5 / fact) * fma(pow2, (k & 1) ? Bc : Bs, (k & 1) ? Ac : As);
  }
  g[0] = fma(0.5, k0, g[0]);
  g[1] += 0.5;
}

// Counting sort of the block's tasks by binfn(key) in [0, kL2Keys), ascending; leaves the number of tasks in
// front of key class `idle` in S.nwork and resets the group counter.  Every key class owns kL2Sub counters, picked
// by the lane: tasks of one warp instruction mostly share a few key classes, and shared-memory atomics on one
// address serialise (the order inside a key class is irrelevant).
constexpr int kL2Sub = SPART_LIDF2_SUB;
constexpr int kL2Bins = kL2Keys * kL2Sub;
static_assert(kL2Bins % 32 == 0, "bins per lane");
template <typename BinFn>
__device__ __forceinline__ void lidf2_sort(Lidf2Smem& S, BinFn binfn, int idle) {
  const int tid = threadIdx.x, sub = tid & (kL2Sub - 1);
  for (int i = tid; i < kL2Bins; i += kL2Threads) S.bin[i] = 0;
  __syncthreads();
  for (int t = tid; t < kL2Tasks; t += kL2Threads)
    S.rank[t] = (unsigned short)atomicAdd(&S.bin[binfn(S.key[t]) * kL2Sub + sub], 1);
  __syncthreads();
  if (tid < 32) {            // exclusive prefix over the counters: kL2Bins / 32 consecutive ones per lane
    constexpr int kPer = kL2Bins / 32;
    int c[kPer], tot = 0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      c[j] = S.bin[tid * kPer + j];
      tot += c[j];
    }
    int incl = tot;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, d);
      if (tid >= d) incl += v;
    }
    int run = incl - tot;
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      S.bin[tid * kPer + j] = run;
      run += c[j];
    }
  }
  __syncthreads();
  for (int t = tid; t < kL2Tasks; t += kL2Threads)
    S.perm[S.bin[binfn(S.key[t]) * kL2Sub + sub] + S.rank[t]] = (unsigned short)t;
  if (tid == 0) {
    S.nwork = S.bin[idle * kL2Sub];
    S.counter = 0;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kL2Threads, SPART_LIDF2_MINBLOCKS)
lidf_kernel(const double* __restrict__ ab0, const double* __restrict__ ab1, int64_t st0, int64_t st1, int64_t n,
             double* __restrict__ out, int64_t stride_ang, int64_t stride_smp) {
  __shared__ Lidf2Smem S;
  const unsigned full = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t base = (int64_t)blockIdx.x * kL2Samples;
  if (tid < 12) {
    const double th = c_theta2[tid];
    double s, c;
    sincos_small(th, s, c);          // sine / cosine of the first exact step, which starts at x0 = theta2
    S.theta2[tid] = th;
    S.sin0[tid] = s;
    S.cos0[tid] = c;
  }
  const int64_t smp_g = (base + tid < n) ? base + tid : n - 1;     // tail entries shadow the last sample
  const double a = ab0[smp_g * st0], b = ab1[smp_g * st1];         // st = 0: broadcast row
  S.a[tid] = a;
  S.b[tid] = b;
  __syncthreads();

  // ---- A1: first exact step of every task (thread = sample, loop over the angles) ------------------------
#pragma unroll 2
  for (int ang = 0; ang < 12; ++ang) {
    const int t = ang * kL2Samples + tid;
    const double theta2 = S.theta2[ang];
    if (a > 1.0) {                   // sailh.py:371-372: closed form F = 1 - cos(theta), no iteration
      const double y = 0.5 * (SPART_PI * (1.0 - cos(0.5 * theta2)) - theta2);
      S.x[t] = 2.0 * y + theta2;
      S.key[t] = 0;
    } else {
      const double s = S.sin0[ang], c = S.cos0[ang];
      const double y = s * fma(b, c, a);                          // a sin x + b/2 sin 2x at x = theta2
      const double dx = fma(0.5, y, 0.5 * (theta2 - theta2));     // (y - x + theta2) / 2
      const double adx = fabs(dx);
      const double yp = fma(a, c, b * fma(2.0 * c, c, -1.0));     // y'(x) = a cos x + b cos 2x
      const bool conv = !(adx > 1e-8);
      signed char dq;
      const unsigned char key = lidf2_leave(dx, yp, lidf2_hand(adx, yp), dq);
      S.dq[t] = dq;
      S.x[t] = conv ? 2.0 * y + theta2 : theta2 + dx;
      S.key[t] = conv ? (unsigned char)0 : key;
    }
  }
  // (lidf2_sort starts with a barrier)
  lidf2_sort(S, [](unsigned char v) { return v >= 128 ? 159 - (int)v : 32; }, 32);   // 31 .. 1 more steps -> bins 0 .. 30

  // ---- A2: remaining exact steps, groups of 32 tasks of similar predicted length -------------------------
  {
    const int nwork = S.nwork;
    while (true) {
      int g = 0;
      if (lane == 0) g = atomicAdd(&S.counter, 1);
      g = __shfl_sync(full, g, 0);
      if (g * 32 >= nwork) break;
      const int pos = g * 32 + lane;
      const bool has = pos < nwork;
      const int t = S.perm[has ? pos : 0];
      const int ang = t / kL2Samples, smp = t % kL2Samples;
      const double ta = S.a[smp], tb = S.b[smp], theta2 = S.theta2[ang];
      double x = S.x[t], y = 0.0, dx = 1.0, yp = 0.0;
      bool running = has, conv = false;
      int iters = 0;
      do {
#pragma unroll
        for (int rep = 0; rep < SPART_LIDF2_RA; ++rep) {
          if (running) {
            double s, c;
            sincos_small(x, s, c);
            y = s * fma(tb, c, ta);
            dx = fma(0.5, y, 0.5 * (theta2 - x));
            x += dx;
            const double adx = fabs(dx);
            yp = fma(ta, c, tb * fma(2.0 * c, c, -1.0));
            conv = !(adx > 1e-8);                                  // the reference's stop (NaN stops too)
            running = !(conv || lidf2_hand(adx, yp));
          }
        }
      } while (__any_sync(full, running) && ++iters < kL2MaxVotes);   // the cap guards non-convergent garbage input
      if (has) {
        S.x[t] = conv ? 2.0 * y + theta2 : x;
        signed char dq;
        const unsigned char key = lidf2_leave(dx, yp, true, dq);
        S.key[t] = conv ? (unsigned char)0 : key;
        S.dq[t] = dq;
      }
    }
  }
  lidf2_sort(S, [](unsigned char v) { return 63 - (int)(v & 63); }, 63);   // 63 .. 1 polynomial steps -> bins 0 .. 62

  // ---- B: Taylor-model steps, groups of 32 tasks of similar predicted length ----------------------------
  // One group per warp (NG = 1): two neighbouring groups stepped side by side, their Horner chains interleaved,
  // gained nothing (DESIGN.md).  The loops over the one group stay: the same steps written with scalars compile to
  // a different register allocation than the build the measurements under profiles/ were taken on.
  {
    constexpr int NG = 1;
    const int nwork = S.nwork;
    while (true) {
      int g = 0;
      if (lane == 0) g = atomicAdd(&S.counter, NG);
      g = __shfl_sync(full, g, 0);
      if (g * 32 >= nwork) break;
      bool has[NG];
      int t[NG];
      double theta2[NG], k0[NG], u[NG], gk[NG][kLidfDeg + 1];
#pragma unroll
      for (int j = 0; j < NG; ++j) {
        const int pos = (g + j) * 32 + lane;
        has[j] = pos < nwork;
        t[j] = S.perm[has[j] ? pos : 0];
        const int ang = t[j] / kL2Samples, smp = t[j] % kL2Samples;
        theta2[j] = S.theta2[ang];
        const double xs = S.x[t[j]];
        const double xc = xs + (double)S.dq[t[j]] * (1.0 / 256.0);   // expansion centre: near the fixed point
        u[j] = xs - xc;                                               // (exact)
        double s, c;
        sincos_small(xc, s, c);
        k0[j] = theta2[j] - xc;
        lidf2_poly_setup(S.a[smp], S.b[smp], s, c, k0[j], gk[j]);
      }
      bool running = false;
      int iters = 0;
      do {
        // a lane stays on the iterate u from which its first step with |du| <= 1e-8 starts: from then on it
        // repeats that step, so no separate "finished" state is carried through the steps
#pragma unroll
        for (int rep = 0; rep < SPART_LIDF2_RB; ++rep) {
          double un[NG];
#pragma unroll
          for (int j = 0; j < NG; ++j) un[j] = gk[j][kLidfDeg];
#pragma unroll
          for (int k = kLidfDeg - 1; k >= 0; --k)
#pragma unroll
            for (int j = 0; j < NG; ++j) un[j] = fma(un[j], u[j], gk[j][k]);
          running = false;
#pragma unroll
          for (int j = 0; j < NG; ++j) {
            const bool r = fabs(un[j] - u[j]) > 1e-8;     // the reference's stop (NaN stops too)
            u[j] = r ? un[j] : u[j];
            running = running || (r && has[j]);
          }
        }
      } while (__any_sync(full, running) && ++iters < kL2MaxVotes);
#pragma unroll
      for (int j = 0; j < NG; ++j)
        if (has[j]) {
          // y~(u) = 2 g(u) - u - k0, so 2 y + theta2 = 4 g(u) - 2 u - 2 k0 + theta2 at the last iterate
          const double uf = u[j];
          const double unf = lidf_poly(gk[j], uf);
          S.x[t[j]] = (2.0 * (2.0 * unf - uf - k0[j]) + theta2[j]) * (1.0 / SPART_PI);
          S.key[t[j]] = 1;
        }
    }
  }
  __syncthreads();
  if (base + tid < n) {
#pragma unroll
    for (int ang = 0; ang < 12; ++ang) {
      const int t = ang * kL2Samples + tid;
      const double v = S.x[t];
      out[ang * stride_ang + (base + tid) * stride_smp] = (S.key[t] == 0) ? v * (1.0 / SPART_PI) : v;
    }
  }
}

// In-place F -> lidf = diff([0, F_1..F_12, 1]) on a [n][13] buffer whose first 12 entries per
// sample hold the cumulative values (calculate_leafangles, sailh.py:387-396).
__global__ void lidf_diff_kernel(double* __restrict__ out, int64_t n) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  double F[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) F[i] = out[s * 13 + i];
  double prev = 0.0;
#pragma unroll
  for (int i = 0; i < 13; ++i) {
    const double Fi = (i < 12) ? F[i] : 1.0;
    out[s * 13 + i] = Fi - prev;
    prev = Fi;
  }
}

// SMAC scalars that depend on the sun / observer angles only (smac.py:98-102, 125-141), in the order
// m, ln m, cksi, ksiD, Rayleigh phase, 1/(1+us), 1/(1+uv), us uv/(us+uv)
__device__ __forceinline__ void smac_angle_scalars(double us, double uv, double inv_us, double inv_uv, double rel,
                                                   double* o) {
  const double crd = 180.0 / SPART_PI;
  double cksi = -((us * uv) + (sqrt(1.0 - us * us) * sqrt(1.0 - uv * uv) * cos(rel * crd)));
  if (cksi < -1.0) cksi = -1.0;
  const double m = inv_us + inv_uv;
  o[0] = m;
  o[1] = log_fast(m);
  o[2] = cksi;
  o[3] = crd * acos(cksi);
  o[4] = 0.7190443 * (1.0 + (cksi * cksi)) + 0.0412742;
  o[5] = rcp_fast(1.0 + us);
  o[6] = rcp_fast(1.0 + uv);
  o[7] = us * uv * rcp_fast(us + uv);
}

// spart_set_lidf: a caller-supplied leaf inclination distribution [n][13] -> the 13 leaf-angle rows of a workspace
__global__ void lidf_store_kernel(const double* __restrict__ lidf, int64_t n, double* __restrict__ ws) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
#pragma unroll
  for (int i = 0; i < 13; ++i) ws[(size_t)(kRowF + i) * n + s] = lidf[s * 13 + i];
}

// Kernel 2, one thread per sample: everything else that does not depend on wavelength or
// band.  With uniform_geometry != 0 all samples share sun/observer angles (a look-up table
// for one acquisition geometry): the 13-class volume-scattering terms are then evaluated
// once per block by 13 threads instead of once per sample.
__global__ void __launch_bounds__(kSampleThreads, SPART_SAMPLE_MINBLOCKS)
geometry_kernel(const Params P, int64_t n, double* __restrict__ rec, int flags) {
  const int uniform_geometry = flags & kFlagUniform;
  const bool soil_spectrum = (flags & SPART_FLAG_SOIL_SPECTRUM) != 0;
  __shared__ double s_cls[13][4];   // ksli, koli, sobli, sofli per leaf-inclination class
  exp_table_load();               // published by the barrier below
  const int tid = threadIdx.x;
  const int64_t s_raw = (int64_t)blockIdx.x * kSampleThreads + tid;
  const bool valid = s_raw < n;
  const int64_t s = valid ? s_raw : n - 1;

  // sun / observer geometry (sailh.py:59-78)
  const double tts = P.at(P_SZA, s), tto = P.at(P_VZA, s), rel = P.at(P_RAA, s);
  // the parameter rows read after the hot-spot integral: start them towards L1 now
  {
    const int later[] = {P_LAI, P_Q, P_B, P_LAT, P_LON, P_SMP, P_SMC, P_PA, P_UO3, P_UH2O, P_DOY};
#pragma unroll
    for (int i = 0; i < 11; ++i) asm volatile("prefetch.global.L1 [%0];" ::"l"(P.ptr(later[i], s)));
  }
  // uniform geometry: the twelve F loads are issued here, so that their latency overlaps the
  // volume-scattering classes computed by 13 threads of the block
  const int64_t sF = (flags & kFlagLidfBcast) ? 0 : s;      // one leaf-angle distribution for the whole batch
  double F[12];
  if (uniform_geometry) {
#pragma unroll
    for (int i = 0; i < 12; ++i) F[i] = rec[(size_t)(kRowF + i) * n + sF];
  }
  // Scalars that depend on the sun / observer angles only (sailh.py:59-78, smac.py:98-102, 129-141).  With a
  // shared geometry they are the same for every sample: warp 0 computes them (its lanes 0..12 also evaluate the
  // volume-scattering classes) and lane 13 publishes them through shared memory -- the other warps skip three
  // sincos, a cos, an acos, a logarithm and six reciprocals per sample.
  enum { GS_COS_TTS, GS_COS_TTO, GS_INV_CS, GS_INV_CO, GS_DSO, GS_M, GS_LM, GS_CKSI, GS_KSID, GS_RAYPH, GS_INV1PUS,
         GS_INV1PUV, GS_AA3, GS_COUNT };
  __shared__ double s_gs[GS_COUNT];
  double gs[GS_COUNT];     // (only GS_COS_TTS .. GS_DSO stay live in the per-sample path)
  double sin_tts = 0.0, sin_tto = 0.0, psi_rad = 0.0, sin_psi = 0.0, cos_psi = 0.0;   // (per-class path below)
  if (!uniform_geometry || tid < 32) {
    const double psi = fabs(rel - 360.0 * rint(rel / 360.0));
    psi_rad = psi * SPART_DEG2RAD;
    // zenith angles and the folded azimuth are a few radians at most: bounded-range sincos
    double cos_tts, cos_tto;
    sincos_small(tts * SPART_DEG2RAD, sin_tts, cos_tts);
    sincos_small(tto * SPART_DEG2RAD, sin_tto, cos_tto);
    sincos_small(psi_rad, sin_psi, cos_psi);
    const double inv_cs = rcp_fast(cos_tts), inv_co = rcp_fast(cos_tto);
    const double tan_tts = sin_tts * inv_cs, tan_tto = sin_tto * inv_co;
    gs[GS_COS_TTS] = cos_tts;
    gs[GS_COS_TTO] = cos_tto;
    gs[GS_INV_CS] = inv_cs;
    gs[GS_INV_CO] = inv_co;
    // like the reference, a rounding-negative radicand gives NaN (sailh.py:78)
    gs[GS_DSO] = sqrt_fast(tan_tts * tan_tts + tan_tto * tan_tto - 2.0 * tan_tts * tan_tto * cos_psi);
    if (uniform_geometry) {
      smac_angle_scalars(cos_tts, cos_tto, inv_cs, inv_co, rel, &gs[GS_M]);
      if (tid < 13) {
        const double inv_cc = SPART_PI * inv_cs * inv_co;
        double chi_s, chi_o, frho, ftau;
        volscatt_class(sin_tts, cos_tts, sin_tto, cos_tto, psi_rad, sin_psi, cos_psi, c_sin_ttli[tid], c_cos_ttli[tid],
                       chi_s, chi_o, frho, ftau);
        s_cls[tid][0] = chi_s * inv_cs;
        s_cls[tid][1] = chi_o * inv_co;
        s_cls[tid][2] = frho * inv_cc;
        s_cls[tid][3] = ftau * inv_cc;
      }
      if (tid == 13) {
#pragma unroll
        for (int i = 0; i < GS_COUNT; ++i) s_gs[i] = gs[i];
      }
    }
  }
  __syncthreads();
  if (!valid) return;
  if (uniform_geometry) {
#pragma unroll
    for (int i = 0; i <= GS_DSO; ++i) gs[i] = s_gs[i];
  }
  const double cos_tts = gs[GS_COS_TTS], cos_tto = gs[GS_COS_TTO], inv_cs = gs[GS_INV_CS], inv_co = gs[GS_INV_CO];
  const double dso = gs[GS_DSO];
  const double inv_cc = SPART_PI * inv_cs * inv_co;

  // 13 leaf-inclination classes, dotted with lidf (sailh.py:81-97)
  double k = 0.0, K = 0.0, bf = 0.0, sob = 0.0, sof = 0.0;
  if (uniform_geometry) {
    const bool direct = (flags & kFlagLidfDirect) != 0;
    const double F12 = direct ? rec[(size_t)(kRowF + 12) * n + sF] : 1.0;
    double Fprev = 0.0;
#pragma unroll
    for (int i = 0; i < 13; ++i) {
      const double Fi = (i < 12) ? F[i < 12 ? i : 0] : F12;
      const double lidf = direct ? Fi : Fi - Fprev;       // sailh.py:395: lidf = diff(F)
      Fprev = Fi;
      k += s_cls[i][0] * lidf;
      K += s_cls[i][1] * lidf;
      bf += (c_cos_ttli[i] * c_cos_ttli[i]) * lidf;
      sob += s_cls[i][2] * lidf;
      sof += s_cls[i][3] * lidf;
    }
  } else {
    const bool direct = (flags & kFlagLidfDirect) != 0;
    const int last = direct ? 12 : 11;          // rows to fetch
    double Fprev = 0.0;
    double Fnext = rec[(size_t)kRowF * n + sF];
#pragma unroll 1
    for (int i = 0; i < 13; ++i) {
      const double Fi = (i <= last) ? Fnext : 1.0;
      if (i < last) Fnext = rec[(size_t)(kRowF + i + 1) * n + sF];   // in flight during volscatt_class
      const double lidf = direct ? Fi : Fi - Fprev;                  // sailh.py:395: lidf = diff(F)
      Fprev = Fi;
      double chi_s, chi_o, frho, ftau;
      volscatt_class(sin_tts, cos_tts, sin_tto, cos_tto, psi_rad, sin_psi, cos_psi, c_sin_ttli[i], c_cos_ttli[i], chi_s,
                     chi_o, frho, ftau);
      k += (chi_s * inv_cs) * lidf;
      K += (chi_o * inv_co) * lidf;
      bf += (c_cos_ttli[i] * c_cos_ttli[i]) * lidf;
      sob += (frho * inv_cc) * lidf;
      sof += (ftau * inv_cc) * lidf;
    }
  }

  const double LAI = P.at(P_LAI, s), q = P.at(P_Q, s);
  double sumpso, pso2w;
  hotspot_integrals(K, k, LAI, q, dso, sumpso, pso2w);

  const double tau_ss = exp_fast(-k * LAI), tau_oo = exp_fast(-K * LAI);
  rec[R_K_SUN * n + s] = k;
  rec[R_K_OBS * n + s] = K;
  rec[R_BF * n + s] = bf;
  rec[R_SOB * n + s] = sob;
  rec[R_SOF * n + s] = sof;
  rec[R_TAUSS * n + s] = tau_ss;
  rec[R_TAUOO * n + s] = tau_oo;
  rec[R_SUMPSO * n + s] = sumpso;
  rec[R_PSO2W * n + s] = pso2w;
  rec[R_Z * n + s] = (1.0 - tau_ss * tau_oo) * rcp_fast(K + k);

  // BSM soil-vector weights and Poisson mean (bsm.py:49-51, 101)
  {
    const double B = P.at(P_B, s);
    double slat, clat, slon, clon;
    sincos_small(P.at(P_LAT, s) * SPART_PI / 180.0, slat, clat);
    sincos_small(P.at(P_LON, s) * SPART_PI / 180.0, slon, clon);
    // with a user-supplied dry-soil spectrum (bsm.py:42-43) the context's first soil vector IS that
    // spectrum and the weights are (1, 0, 0): rdry = 1 * spectrum + 0 + 0 exactly
    rec[R_F1 * n + s] = soil_spectrum ? 1.0 : B * slat;
    rec[R_F2 * n + s] = soil_spectrum ? 0.0 : B * clat * slon;
    rec[R_F3 * n + s] = soil_spectrum ? 0.0 : B * clat * clon;
    const double mu = (P.at(P_SMP, s) - 5.0) * rcp_fast(P.at(P_SMC, s));
    rec[R_MU * n + s] = mu;
    rec[R_EMU * n + s] = exp_fast(-mu);
  }

  // SMAC per-sample scalars (smac.py:98-102, 129-141); the angle-only ones were formed above
  {
    const double us = cos_tts, uv = cos_tto;    // cos(tts*cdr), cos(tto*cdr)
    const double Peq = P.at(P_PA, s) * (1.0 / 1013.25);
    if (uniform_geometry) {
#pragma unroll
      for (int i = GS_M; i < GS_COUNT; ++i) gs[i] = s_gs[i];
    } else {
      smac_angle_scalars(cos_tts, cos_tto, inv_cs, inv_co, rel, &gs[GS_M]);
    }
    const double m = gs[GS_M];
    rec[R_US * n + s] = us;
    rec[R_UV * n + s] = uv;
    rec[R_M * n + s] = m;
    rec[R_PEQ * n + s] = Peq;
    rec[R_LO3 * n + s] = log_fast(P.at(P_UO3, s) * m);
    rec[R_LH2O * n + s] = log_fast(P.at(P_UH2O, s) * m);
    rec[R_LM * n + s] = gs[GS_LM];
    rec[R_LPEQ * n + s] = log_fast(Peq);
    rec[R_CKSI * n + s] = gs[GS_CKSI];
    rec[R_KSID * n + s] = gs[GS_KSID];
    rec[R_RAYPH * n + s] = gs[GS_RAYPH];
    rec[R_INVUS * n + s] = inv_cs;
    rec[R_INVUV * n + s] = inv_co;
    rec[R_INV1PUS * n + s] = gs[GS_INV1PUS];
    rec[R_INV1PUV * n + s] = gs[GS_INV1PUV];
    rec[R_AA3 * n + s] = gs[GS_AA3];
    // extraterrestrial radiance scale (SPART.py:345-353)
    const double b = 2.0 * SPART_PI * P.at(P_DOY, s) * (1.0 / 365.0);
    double sb, cb, s2b, c2b;
    sincos_small(b, sb, cb);
    sincos_small(2.0 * b, s2b, c2b);
    const double cf = 1.00011 + 0.034221 * cb + 0.00128 * sb + 0.000719 * c2b + 0.000077 * s2b;
    rec[R_ETSCALE * n + s] = cf * us * (1.0 / SPART_PI);
  }
}

__device__ __forceinline__ CanopyGeo load_geo(const Params& P,
                                              const double* __restrict__ rec, int64_t n, int64_t s) {
  CanopyGeo G;
  G.LAI = P.at(P_LAI, s);
  G.k = rec[R_K_SUN * n + s];
  G.K = rec[R_K_OBS * n + s];
  G.bf = rec[R_BF * n + s];
  G.sob = rec[R_SOB * n + s];
  G.sof = rec[R_SOF * n + s];
  G.tau_ss = rec[R_TAUSS * n + s];
  G.tau_oo = rec[R_TAUOO * n + s];
  G.sumpso = rec[R_SUMPSO * n + s];
  G.pso2w = rec[R_PSO2W * n + s];
  G.Z = rec[R_Z * n + s];
  return G;
}

__device__ __forceinline__ SoilPar load_soil(const Params& P,
                                             const double* __restrict__ rec, int64_t n, int64_t s) {
  SoilPar S;
  S.f1 = rec[R_F1 * n + s];
  S.f2 = rec[R_F2 * n + s];
  S.f3 = rec[R_F3 * n + s];
  S.mu = rec[R_MU * n + s];
  S.emu = rec[R_EMU * n + s];
  S.film = P.at(P_FILM, s);
  return S;
}

#ifndef SPART_BAND_THREADS
#define SPART_BAND_THREADS 128
#endif
constexpr int kBandThreads = SPART_BAND_THREADS;
constexpr int kBandChunk = SPART_BAND_CHUNK;   // bands handled by one block (per-sample state is loaded once per chunk)

__device__ __forceinline__ AtmSample load_atm(const Params& P, const double* __restrict__ rec, int64_t n, int64_t s) {
  AtmSample A;
  A.us = rec[R_US * n + s];
  A.uv = rec[R_UV * n + s];
  A.m = rec[R_M * n + s];
  A.Peq = rec[R_PEQ * n + s];
  A.lo3 = rec[R_LO3 * n + s];
  A.lh2o = rec[R_LH2O * n + s];
  A.lm = rec[R_LM * n + s];
  A.lpeq = rec[R_LPEQ * n + s];
  A.cksi = rec[R_CKSI * n + s];
  A.ksiD = rec[R_KSID * n + s];
  A.ray_phase = rec[R_RAYPH * n + s];
  A.taup550 = P.at(P_AOT, s);
  A.inv_us = rec[R_INVUS * n + s];
  A.inv_uv = rec[R_INVUV * n + s];
  A.inv_1pus = rec[R_INV1PUS * n + s];
  A.inv_1puv = rec[R_INV1PUV * n + s];
  A.aa3 = rec[R_AA3 * n + s];
  return A;
}

// The band kernels park the soil and canopy state in shared memory (one column per thread, no synchronisation
// needed) and re-read it per wavelength right before use: soil before bsm_point, canopy before sailh_point.  That
// keeps 34 registers less live across the leaf model; the re-reads are volatile so that the compiler keeps them
// where they are instead of hoisting them back into registers.
constexpr int kStateRows = 17;
__device__ __forceinline__ void park_state(double (*st)[kBandThreads], const SoilPar& S, const CanopyGeo& G) {
  const double v[kStateRows] = {S.f1, S.f2, S.f3, S.mu, S.emu, S.film, G.LAI, G.k, G.K, G.bf, G.sob, G.sof,
                                G.tau_ss, G.tau_oo, G.sumpso, G.pso2w, G.Z};
#pragma unroll
  for (int i = 0; i < kStateRows; ++i) st[i][threadIdx.x] = v[i];
}

__device__ __forceinline__ SoilPar reload_soil(volatile double (*st)[kBandThreads]) {
  const int t = threadIdx.x;
  SoilPar S;
  S.f1 = st[0][t]; S.f2 = st[1][t]; S.f3 = st[2][t]; S.mu = st[3][t]; S.emu = st[4][t]; S.film = st[5][t];
  return S;
}

__device__ __forceinline__ CanopyGeo reload_geo(volatile double (*st)[kBandThreads]) {
  const int t = threadIdx.x;
  CanopyGeo G;
  G.LAI = st[6][t]; G.k = st[7][t]; G.K = st[8][t]; G.bf = st[9][t]; G.sob = st[10][t]; G.sof = st[11][t];
  G.tau_ss = st[12][t]; G.tau_oo = st[13][t]; G.sumpso = st[14][t]; G.pso2w = st[15][t]; G.Z = st[16][t];
  return G;
}

// Dry-soil source of the band-path kernels (the `Soil` parameter of their bodies below).
//   GsvSoil:     the record's soil-vector weights times the context's three GSV vectors -- the B / lat / lon
//                model, or a user spectrum in GSV0 with weights (1, 0, 0) (SPART_FLAG_SOIL_SPECTRUM).
//   LibrarySoil: row `index` of the context's soil library, index = params row 9 (SPART_FLAG_SOIL_LIBRARY).  The
//                geometry kernels then run with SPART_FLAG_SOIL_SPECTRUM, so the record is that of a user spectrum
//                and, since 1 * x + 0 * y + 0 * z == x, every sample equals bit for bit a run with
//                soil_spectrum = its library row.  The index is read from params, not from the record, so
//                SPART_FLAG_REUSE_RECORD works unchanged.
// `wl` is the index into 400..2400 nm of the wavelength whose constants `lc` holds; GsvSoil does not need it.
struct SoilLib {                // device view of a context's soil library
  const double* rows;           // [k + 1][SPART_NWL]; row k is all NaN
  int k;
};

struct GsvSoil {
  static constexpr bool kLibrary = false;
  template <typename T>
  __device__ __forceinline__ static GsvSoil select(const ParamsT<T>&, int64_t, const SoilLib&) { return {}; }
  __device__ __forceinline__ void point(const SoilPar& S, const double* lc, int, double& rwet, double& rdry) const {
    bsm_point(S, lc, rwet, rdry);
  }
  __device__ __forceinline__ float point_f(const spart::f32::SoilParF& S, const float* lc, int) const {
    return spart::f32::bsm_point_f(S, lc);
  }
};

struct LibrarySoil {
  static constexpr bool kLibrary = true;
  const double* row;
  // An index that is not a whole number in [0, k) (NaN included) selects the NaN row: the address stays inside the
  // library and every soil-dependent output of the sample is NaN.  float -> double is exact, so F32_IO indices
  // are judged the same way.
  template <typename T>
  __device__ __forceinline__ static LibrarySoil select(const ParamsT<T>& P, int64_t s, const SoilLib& lib) {
    const double v = (double)P.at(P_B, s);
    const bool ok = v >= 0.0 && v < (double)lib.k && v == trunc(v);
    return {lib.rows + (size_t)(ok ? (int)v : lib.k) * SPART_NWL};
  }
  __device__ __forceinline__ void point(const SoilPar& S, const double* lc, int wl, double& rwet, double& rdry) const {
    rdry = __ldg(row + wl);
    bsm_wet(S, lc, rdry, rwet);
  }
  __device__ __forceinline__ float point_f(const spart::f32::SoilParF& S, const float* lc, int wl) const {
    return spart::f32::bsm_wet_f(S, lc, (float)__ldg(row + wl));
  }
};

// One thread per sample, looping over a chunk of up to kBandChunk bands; blockIdx.x = band
// chunk, blockIdx.y = sample tile.  The per-sample state (leaf, soil, canopy geometry, SMAC
// scalars: 44 doubles) is read from HBM once per chunk and kept in registers; the per-band
// constants are warp-uniform shared-memory broadcasts.  knots: [nb][2] wavelength indices of the
// band's np.interp knots, read by LibrarySoil only.
template <bool kUniform, class Soil>
__device__ __forceinline__ void band_body(const Params& P, int64_t n, const double* __restrict__ rec,
                                          const double* __restrict__ band_table, int nb, double* __restrict__ out,
                                          int compact, const SoilLib& lib, const int32_t* __restrict__ knots) {
  __shared__ TauTable s_tau;
  __shared__ double s_bt[kBandChunk][BT_COUNT];
  __shared__ double s_ug[kUniform ? kBandChunk : 1][UG_COUNT];
  __shared__ int s_knot[Soil::kLibrary ? kBandChunk : 1][2];
  const int b0 = blockIdx.x * kBandChunk;
  const int nbc = min(kBandChunk, nb - b0);
  load_tau_table(&s_tau);
  exp_table_load();
  for (int i = threadIdx.x; i < nbc * BT_COUNT; i += blockDim.x)
    (&s_bt[0][0])[i] = band_table[(size_t)b0 * BT_COUNT + i];
  if (Soil::kLibrary)
    for (int i = threadIdx.x; i < nbc * 2; i += blockDim.x) (&s_knot[0][0])[i] = knots[(size_t)b0 * 2 + i];
  __syncthreads();
  if (kUniform) {
    // all samples share the geometry: fold it into per-band constants, one thread per band,
    // from the record of the tile's first sample
    if (threadIdx.x < nbc) {
      const int64_t s0 = (int64_t)blockIdx.y * kBandThreads;
      AtmGeometry g;
      g.us = rec[R_US * n + s0];
      g.uv = rec[R_UV * n + s0];
      g.m = rec[R_M * n + s0];
      g.lm = rec[R_LM * n + s0];
      g.cksi = rec[R_CKSI * n + s0];
      g.ksiD = rec[R_KSID * n + s0];
      g.ray_phase = rec[R_RAYPH * n + s0];
      g.inv_us = rec[R_INVUS * n + s0];
      g.inv_uv = rec[R_INVUV * n + s0];
      g.inv_1pus = rec[R_INV1PUS * n + s0];
      g.inv_1puv = rec[R_INV1PUV * n + s0];
      g.aa3 = rec[R_AA3 * n + s0];
      smac_fold_geometry(g, &s_bt[threadIdx.x][BT_SMAC], s_ug[threadIdx.x]);
    }
    __syncthreads();
  }
  const int64_t s = (int64_t)blockIdx.y * kBandThreads + threadIdx.x;
  if (s >= n) return;

  const LeafPar L = load_leaf(P, s);
  const Soil soil = Soil::select(P, s, lib);
  __shared__ double s_st[kStateRows][kBandThreads];
  park_state(s_st, load_soil(P, rec, n, s), load_geo(P, rec, n, s));
  AtmSample A;
  AtmColumn C;
  if (kUniform) {
    C.Peq = rec[R_PEQ * n + s];
    C.lo3 = rec[R_LO3 * n + s];
    C.lh2o = rec[R_LH2O * n + s];
    C.lpeq = rec[R_LPEQ * n + s];
    C.taup550 = P.at(P_AOT, s);
  } else {
    A = load_atm(P, rec, n, s);
  }
  const double etscale = rec[R_ETSCALE * n + s];
  // full output: [n][nb][3]; compact output (SPART_FLAG_COMPACT_OUT): [n][nb][2] followed by etscale[n]
  const int nout = compact ? 2 : SPART_NOUT;
  double* o = out + ((size_t)s * nb + b0) * nout;
  if (compact && blockIdx.x == 0) out[(size_t)n * nb * 2 + s] = etscale;

#pragma unroll 1
  for (int bi = 0; bi < nbc; ++bi) {
    const double* bt = s_bt[bi];
    // PROSPECT + BSM + SAILH at the one or two wavelengths np.interp touches (SPART.py:220-223)
    double rso = 0.0, rdo = 0.0, rsd = 0.0, rdd = 0.0;
    const int npts = (__double2hiint(bt[BT_NPTS]) >= 0x40000000) ? 2 : 1;   // 2.0 or 1.0, integer-pipe test
#pragma unroll 1
    for (int pt = 0; pt < npts; ++pt) {
      const double* lc = &bt[BT_LC0 + pt * LC_COUNT];
      double refl, tran, kchl, rwet, rdry, a0, a1, a2, a3;
      prospect_point<false>(L, lc, &s_tau, refl, tran, kchl);
      soil.point(reload_soil(s_st), lc, Soil::kLibrary ? s_knot[bi][pt] : 0, rwet, rdry);
      sailh_point(reload_geo(s_st), refl, tran, rwet, a0, a1, a2, a3);
      if (pt == 0) {
        rso = a0; rdo = a1; rsd = a2; rdd = a3;
      } else {
        const double fr = bt[BT_FRAC];
        rso = (a0 - rso) * fr + rso;
        rdo = (a1 - rdo) * fr + rdo;
        rsd = (a2 - rsd) * fr + rsd;
        rdd = (a3 - rdd) * fr + rdd;
      }
    }
    double R_TOC, R_TOA, L_TOA;
    if (kUniform)
      smac_toa_band_uniform(C, &bt[BT_SMAC], s_ug[bi], bt[BT_CONVEA], etscale, rso, rdo, rdd, rsd, R_TOC, R_TOA,
                            L_TOA);
    else
      smac_toa_band(A, &bt[BT_SMAC], bt[BT_CONVEA], etscale, rso, rdo, rdd, rsd, R_TOC, R_TOA, L_TOA);
    o[bi * nout + 0] = R_TOC;
    o[bi * nout + 1] = R_TOA;
    if (!compact) o[bi * nout + 2] = L_TOA;
  }
}

template <bool kUniform>
__global__ void __launch_bounds__(kBandThreads, kUniform ? SPART_BAND_MINBLOCKS_U : SPART_BAND_MINBLOCKS)
band_kernel(const Params P, int64_t n, const double* __restrict__ rec,
            const double* __restrict__ band_table, int nb, double* __restrict__ out, int compact) {
  band_body<kUniform, GsvSoil>(P, n, rec, band_table, nb, out, compact, SoilLib{nullptr, 0}, nullptr);
}

// band_kernel with the dry soil of each sample taken from the soil library (SPART_FLAG_SOIL_LIBRARY)
template <bool kUniform>
__global__ void __launch_bounds__(kBandThreads, kUniform ? SPART_BAND_MINBLOCKS_U : SPART_BAND_MINBLOCKS)
soillib_bands(const Params P, int64_t n, const double* __restrict__ rec, const double* __restrict__ band_table,
              int nb, double* __restrict__ out, int compact, const SoilLib lib, const int32_t* __restrict__ knots) {
  band_body<kUniform, LibrarySoil>(P, n, rec, band_table, nb, out, compact, lib, knots);
}

// Band kernel of the SRF mode (SPART_FLAG_SRF_BANDS): the four canopy reflectances of a band are
// the spectral-response-weighted means over the band's support (calculate_spectral_convolution,
// SPART.py:358-396, applied to canopyopt) instead of np.interp samples at the band centre.
//
// Bands overlap (TerraAqua-MODIS lists 2006 (wavelength, weight) pairs on 694 distinct wavelengths),
// so the leaf / soil / canopy model is evaluated ONCE per distinct wavelength, in ascending order, and
// its four reflectances are added into every band that contains the wavelength.  A band's accumulators
// live in a shared-memory slot (one column per thread); spart_create assigns slots by interval colouring
// (bands whose supports overlap get different slots: a handful suffices) and lists, per wavelength, the
// (slot, weight) pairs to add and the bands that are complete after it: for those SMAC + TOC->TOA run
// right away and the slot is cleared.  Each band still sums its samples in ascending wavelength order.
// thread = sample, block = sample tile; everything about wavelengths / bands is warp-uniform.
constexpr int kSrfChunk = 32;

struct SrfPlan {               // device pointers, built by spart_create
  int n_wl;                    // steps: distinct wavelengths, ascending, then one per band without SRF weight
  int n_slots;                 // accumulator slots (max. number of simultaneously open bands + 1 spare)
  const int32_t* wl_idx;       // [n_wl] index into 400..2400 nm
  const int32_t* pair_off;     // [n_wl + 1] offsets into pair_slot / pair_w
  const int32_t* pair_slot;
  const double* pair_w;        // normalised SRF weights
  const int32_t* fin_off;      // [n_wl + 1] offsets into fin_band / fin_slot: bands complete after wavelength i
  const int32_t* fin_band;
  const int32_t* fin_slot;
};

template <class Soil>
__device__ __forceinline__ void srf_body(const Params& P, int64_t n, const double* __restrict__ rec,
                                         const double* __restrict__ band_table, const double* __restrict__ lc_table,
                                         const SrfPlan& plan, int nb, double* __restrict__ out, int compact,
                                         const SoilLib& lib) {
  extern __shared__ double s_acc[];            // [n_slots][4][kBandThreads]
  __shared__ TauTable s_tau;
  __shared__ double s_lc[kSrfChunk][LC_COUNT];
  __shared__ int s_poff[kSrfChunk + 1], s_foff[kSrfChunk + 1];
  const int t = threadIdx.x;
  load_tau_table(&s_tau);
  exp_table_load();
  for (int i = 0; i < plan.n_slots * 4; ++i) s_acc[i * kBandThreads + t] = 0.0;
  const int64_t s_raw = (int64_t)blockIdx.x * kBandThreads + t;
  const bool valid = s_raw < n;
  const int64_t s = valid ? s_raw : n - 1;
  const LeafPar L = load_leaf(P, s);
  const Soil soil = Soil::select(P, s, lib);
  __shared__ double s_st[kStateRows][kBandThreads];
  park_state(s_st, load_soil(P, rec, n, s), load_geo(P, rec, n, s));
  const double etscale = rec[R_ETSCALE * n + s];
  const int nout = compact ? 2 : SPART_NOUT;
  if (compact && valid) out[(size_t)n * nb * 2 + s] = etscale;

  for (int c0 = 0; c0 < plan.n_wl; c0 += kSrfChunk) {
    const int m = min(kSrfChunk, plan.n_wl - c0);
    __syncthreads();
    for (int i = t; i < m * LC_COUNT; i += blockDim.x)
      s_lc[i / LC_COUNT][i % LC_COUNT] = lc_table[(size_t)(i % LC_COUNT) * SPART_NWL + plan.wl_idx[c0 + i / LC_COUNT]];
    for (int i = t; i <= m; i += blockDim.x) {
      s_poff[i] = plan.pair_off[c0 + i];
      s_foff[i] = plan.fin_off[c0 + i];
    }
    __syncthreads();
#pragma unroll 1
    for (int j = 0; j < m; ++j) {
      double refl, tran, kchl, rwet, rdry, a0, a1, a2, a3;
      prospect_point<false>(L, s_lc[j], &s_tau, refl, tran, kchl);
      soil.point(reload_soil(s_st), s_lc[j], Soil::kLibrary ? __ldg(plan.wl_idx + c0 + j) : 0, rwet, rdry);
      sailh_point(reload_geo(s_st), refl, tran, rwet, a0, a1, a2, a3);
      // add into every band that contains this wavelength (own column of the slot: no synchronisation)
#pragma unroll 1
      for (int p = s_poff[j]; p < s_poff[j + 1]; ++p) {
        const double w = __ldg(plan.pair_w + p);
        double* acc = s_acc + (size_t)__ldg(plan.pair_slot + p) * 4 * kBandThreads + t;
        acc[0 * kBandThreads] = fma(w, a0, acc[0 * kBandThreads]);     // rso
        acc[1 * kBandThreads] = fma(w, a1, acc[1 * kBandThreads]);     // rdo
        acc[2 * kBandThreads] = fma(w, a2, acc[2 * kBandThreads]);     // rsd
        acc[3 * kBandThreads] = fma(w, a3, acc[3 * kBandThreads]);     // rdd
      }
      // bands whose last wavelength this was: atmosphere + TOC -> TOA, then the slot is free again
#pragma unroll 1
      for (int f = s_foff[j]; f < s_foff[j + 1]; ++f) {
        const int b = __ldg(plan.fin_band + f);
        double* acc = s_acc + (size_t)__ldg(plan.fin_slot + f) * 4 * kBandThreads + t;
        const double rso = acc[0 * kBandThreads], rdo = acc[1 * kBandThreads], rsd = acc[2 * kBandThreads],
                     rdd = acc[3 * kBandThreads];
        acc[0 * kBandThreads] = acc[1 * kBandThreads] = acc[2 * kBandThreads] = acc[3 * kBandThreads] = 0.0;
        const AtmSample A = load_atm(P, rec, n, s);
        const double* bt = band_table + (size_t)b * BT_COUNT;
        double R_TOC, R_TOA, L_TOA;
        smac_toa_band(A, bt + BT_SMAC, __ldg(bt + BT_CONVEA), etscale, rso, rdo, rdd, rsd, R_TOC, R_TOA, L_TOA);
        if (valid) {
          double* o = out + ((size_t)s * nb + b) * nout;
          o[0] = R_TOC;
          o[1] = R_TOA;
          if (!compact) o[2] = L_TOA;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(kBandThreads, SPART_SRF_MINBLOCKS)
band_kernel_srf(const Params P, int64_t n, const double* __restrict__ rec,
                const double* __restrict__ band_table, const double* __restrict__ lc_table, const SrfPlan plan,
                int nb, double* __restrict__ out, int compact) {
  srf_body<GsvSoil>(P, n, rec, band_table, lc_table, plan, nb, out, compact, SoilLib{nullptr, 0});
}

// band_kernel_srf with the dry soil of each sample taken from the soil library (SPART_FLAG_SOIL_LIBRARY)
__global__ void __launch_bounds__(kBandThreads, SPART_SRF_MINBLOCKS)
soillib_srf(const Params P, int64_t n, const double* __restrict__ rec, const double* __restrict__ band_table,
            const double* __restrict__ lc_table, const SrfPlan plan, int nb, double* __restrict__ out, int compact,
            const SoilLib lib) {
  srf_body<LibrarySoil>(P, n, rec, band_table, lc_table, plan, nb, out, compact, lib);
}

// SMAC alone (the reference's SMAC(angles, atm, coefs), smac.py:14-213): the nine
// AtmosphericOptics arrays per (sample, band); thread = sample, blockIdx.x = band.
__global__ void __launch_bounds__(kBandThreads)
smac_kernel(const Params P, int64_t n, const double* __restrict__ rec,
            const double* __restrict__ band_table, int nb, double* __restrict__ out) {
  __shared__ double s_c[SM_COUNT];
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < SM_COUNT; i += blockDim.x) s_c[i] = band_table[(size_t)b * BT_COUNT + BT_SMAC + i];
  exp_table_load();
  __syncthreads();
  const int64_t s = (int64_t)blockIdx.y * kBandThreads + threadIdx.x;
  if (s >= n) return;
  const AtmOptics O = smac_band(load_atm(P, rec, n, s), s_c);
  double* o = out + (size_t)s * 9 * nb + b;
  o[0 * nb] = O.Ta_s;
  o[1 * nb] = O.Ta_o;
  o[2 * nb] = O.Tg;
  o[3 * nb] = O.Ra_dd;
  o[4 * nb] = O.Ra_so;
  o[5 * nb] = O.Ta_ss;
  o[6 * nb] = O.Ta_sd;
  o[7 * nb] = O.Ta_oo;
  o[8 * nb] = O.Ta_do;
}

// SAILH on caller-supplied spectra (the reference's SAILH(soil, leafopt, canopy, angles),
// sailh.py:14-237): thread = wavelength (coalesced reads of the three input spectra and writes
// of the four outputs), blockIdx.y = sample; the sample's canopy record is a broadcast load.
__global__ void __launch_bounds__(256)
sailh_spectra_kernel(const Params P, int64_t n, const double* __restrict__ rec,
                     const double* __restrict__ rs, const double* __restrict__ rho, const double* __restrict__ tau,
                     int64_t stride, int64_t s0, double* __restrict__ out) {
  exp_table_load();
  __syncthreads();
  const int w = blockIdx.x * 256 + threadIdx.x;
  const int64_t s = s0 + blockIdx.y;
  if (w >= SPART_NWL_S || s >= n) return;
  const CanopyGeo G = load_geo(P, rec, n, s);
  double rso, rdo, rsd, rdd;
  sailh_point(G, rho[s * stride + w], tau[s * stride + w], rs[s * stride + w], rso, rdo, rsd, rdd);
  double* o = out + (size_t)s * 4 * SPART_NWL_S;
  o[0 * SPART_NWL_S + w] = rso;
  o[1 * SPART_NWL_S + w] = rdo;
  o[2 * SPART_NWL_S + w] = rsd;
  o[3 * SPART_NWL_S + w] = rdd;
}

// ---- FP32 mode (SPART_FP32) -----------------------------------------------------------------
// Two kernels: per-sample geometry (leaf angles by safeguarded Newton, volume scattering,
// hot-spot integrals, soil / atmosphere scalars) and the band kernel.  The per-sample record
// is kept as float [R_COUNT][n] in the same workspace; parameters are read and results are
// written as TIO: double, or float with SPART_FLAG_F32_IO.
__constant__ float c_sin_ttli_f[13];
__constant__ float c_cos_ttli_f[13];
__constant__ float c_theta2_f[12];

template <typename TIO>
__global__ void __launch_bounds__(kSampleThreads)
geometry_kernel_f32(const ParamsT<TIO> P, int64_t n, float* __restrict__ rec, int flags) {
  using namespace spart::f32;
  const int uniform_geometry = flags & kFlagUniform;
  const bool soil_spectrum = (flags & SPART_FLAG_SOIL_SPECTRUM) != 0;
  __shared__ float s_cls[13][4];
  const int tid = threadIdx.x;
  const int64_t s_raw = (int64_t)blockIdx.x * kSampleThreads + tid;
  const bool valid = s_raw < n;
  const int64_t s = valid ? s_raw : n - 1;

  const double tts_d = P.at(P_SZA, s), tto_d = P.at(P_VZA, s), rel_d = P.at(P_RAA, s);
  const float tts = (float)tts_d, tto = (float)tto_d, rel = (float)rel_d;
  const float psi = fabsf(rel - 360.0f * rintf(rel / 360.0f));
  const float psi_rad = psi * (SPART_PI_F / 180.0f);
  float sin_tts, cos_tts, sin_tto, cos_tto;
  sincosf(tts * (SPART_PI_F / 180.0f), &sin_tts, &cos_tts);
  sincosf(tto * (SPART_PI_F / 180.0f), &sin_tto, &cos_tto);
  const float inv_cs = rcp(cos_tts), inv_co = rcp(cos_tto);
  float sin_psi, cos_psi;
  sincosf(psi_rad, &sin_psi, &cos_psi);
  // dso (sailh.py:78) is a difference of O(1) terms that vanishes in the hot spot: a degree away from it single
  // precision has no digits left, so this one per-sample scalar is formed in FP64 from the angles as given
  float dso;
  double us_d, uv_d, ss_d, so_d;       // cos / sin of the two zenith angles in FP64, reused by the SMAC scalars below
  {
    double sp, cp;
    sincos_small(tts_d * SPART_DEG2RAD, ss_d, us_d);
    sincos_small(tto_d * SPART_DEG2RAD, so_d, uv_d);
    const double psi_d = fabs(rel_d - 360.0 * rint(rel_d / 360.0));
    sincos_small(psi_d * SPART_DEG2RAD, sp, cp);
    (void)sp;
    const double ts = ss_d * rcp_fast(us_d), to = so_d * rcp_fast(uv_d);
    const double d2 = ts * ts + to * to - 2.0 * ts * to * cp;
    dso = (float)sqrt_fast(fmax(d2, 0.0));
  }
  const float inv_cc = SPART_PI_F * inv_cs * inv_co;

  if (uniform_geometry) {
    if (tid < 13) {
      float chi_s, chi_o, frho, ftau;
      volscatt_class_f(sin_tts, cos_tts, sin_tto, cos_tto, psi_rad, sin_psi, cos_psi, c_sin_ttli_f[tid], c_cos_ttli_f[tid],
                       chi_s, chi_o, frho, ftau);
      s_cls[tid][0] = chi_s * inv_cs;
      s_cls[tid][1] = chi_o * inv_co;
      s_cls[tid][2] = frho * inv_cc;
      s_cls[tid][3] = ftau * inv_cc;
    }
    __syncthreads();
  }
  if (!valid) return;

  const float a = (float)P.at(P_LIDFA, s), b = (float)P.at(P_LIDFB, s);
  float k = 0.0f, K = 0.0f, bf = 0.0f, sob = 0.0f, sof = 0.0f;
  float Fprev = 0.0f;
#pragma unroll 1
  for (int i = 0; i < 13; ++i) {
    const float Fi = (i < 12) ? dcum_newton_f(a, b, c_theta2_f[i]) : 1.0f;
    const float lidf = Fi - Fprev;
    Fprev = Fi;
    float ksli, koli, sobli, sofli;
    if (uniform_geometry) {
      ksli = s_cls[i][0]; koli = s_cls[i][1]; sobli = s_cls[i][2]; sofli = s_cls[i][3];
    } else {
      float chi_s, chi_o, frho, ftau;
      volscatt_class_f(sin_tts, cos_tts, sin_tto, cos_tto, psi_rad, sin_psi, cos_psi, c_sin_ttli_f[i], c_cos_ttli_f[i], chi_s,
                       chi_o, frho, ftau);
      ksli = chi_s * inv_cs; koli = chi_o * inv_co; sobli = frho * inv_cc; sofli = ftau * inv_cc;
    }
    k += ksli * lidf;
    K += koli * lidf;
    bf += (c_cos_ttli_f[i] * c_cos_ttli_f[i]) * lidf;
    sob += sobli * lidf;
    sof += sofli * lidf;
  }

  const float LAI = (float)P.at(P_LAI, s), q = (float)P.at(P_Q, s);
  float sumpso, pso2w;
  hotspot_integrals_f(K, k, LAI, q, dso, sumpso, pso2w);
  const float tau_ss = __expf(-k * LAI), tau_oo = __expf(-K * LAI);
  rec[R_K_SUN * n + s] = k;
  rec[R_K_OBS * n + s] = K;
  rec[R_BF * n + s] = bf;
  rec[R_SOB * n + s] = sob;
  rec[R_SOF * n + s] = sof;
  rec[R_TAUSS * n + s] = tau_ss;
  rec[R_TAUOO * n + s] = tau_oo;
  rec[R_SUMPSO * n + s] = sumpso;
  rec[R_PSO2W * n + s] = pso2w;
  rec[R_Z * n + s] = one_minus_exp(-(k + K) * LAI) * rcp(K + k);

  {
    const float B = (float)P.at(P_B, s);
    float slat, clat, slon, clon;
    sincosf((float)P.at(P_LAT, s) * (SPART_PI_F / 180.0f), &slat, &clat);
    sincosf((float)P.at(P_LON, s) * (SPART_PI_F / 180.0f), &slon, &clon);
    // with a user-supplied dry-soil spectrum (bsm.py:42-43) the context's first soil vector IS that
    // spectrum and the weights are (1, 0, 0): rdry = 1 * spectrum + 0 + 0 exactly
    rec[R_F1 * n + s] = soil_spectrum ? 1.0f : B * slat;
    rec[R_F2 * n + s] = soil_spectrum ? 0.0f : B * clat * slon;
    rec[R_F3 * n + s] = soil_spectrum ? 0.0f : B * clat * clon;
    const float mu = ((float)P.at(P_SMP, s) - 5.0f) / (float)P.at(P_SMC, s);
    rec[R_MU * n + s] = mu;
    rec[R_EMU * n + s] = __expf(-mu);
  }

  {
    // the scattering-angle terms keep FP64: cos(rel * 180/pi) has an argument of ~1e4 rad (smac.py:130)
    const double crd = 180.0 / SPART_PI;
    double cksi = -((us_d * uv_d) + (sqrt_fast(1.0 - us_d * us_d) * sqrt_fast(1.0 - uv_d * uv_d) * cos(rel_d * crd)));
    if (cksi < -1.0) cksi = -1.0;
    const float us = (float)us_d, uv = (float)uv_d;
    const float Peq = (float)(P.at(P_PA, s) / 1013.25);
    const float inv_us = rcp(us), inv_uv = rcp(uv);
    const float m = inv_us + inv_uv;
    rec[R_US * n + s] = us;
    rec[R_UV * n + s] = uv;
    rec[R_M * n + s] = m;
    rec[R_PEQ * n + s] = Peq;
    rec[R_LO3 * n + s] = logf((float)P.at(P_UO3, s) * m);
    rec[R_LH2O * n + s] = logf((float)P.at(P_UH2O, s) * m);
    rec[R_LM * n + s] = logf(m);
    rec[R_LPEQ * n + s] = (float)log(P.at(P_PA, s) / 1013.25);   // ln of a number close to 1
    rec[R_CKSI * n + s] = (float)cksi;
    rec[R_KSID * n + s] = (float)(crd * acos(cksi));
    rec[R_RAYPH * n + s] = (float)(0.7190443 * (1.0 + (cksi * cksi)) + 0.0412742);
    rec[R_INVUS * n + s] = inv_us;
    rec[R_INVUV * n + s] = inv_uv;
    rec[R_INV1PUS * n + s] = rcp(1.0f + us);
    rec[R_INV1PUV * n + s] = rcp(1.0f + uv);
    rec[R_AA3 * n + s] = us * uv * rcp(us + uv);
    const float bb = 2.0f * SPART_PI_F * (float)P.at(P_DOY, s) / 365.0f;
    float sb, cb, s2b, c2b;
    sincosf(bb, &sb, &cb);
    sincosf(2.0f * bb, &s2b, &c2b);
    const float cf = 1.00011f + 0.034221f * cb + 0.00128f * sb + 0.000719f * c2b + 0.000077f * s2b;
    rec[R_ETSCALE * n + s] = cf * us / SPART_PI_F;
  }
}

template <typename TIO, class Soil>
__device__ __forceinline__ void band_body_f32(const ParamsT<TIO>& P, int64_t n, const float* __restrict__ rec,
                                              const double* __restrict__ band_table, int nb, TIO* __restrict__ out,
                                              int compact, const SoilLib& lib, const int32_t* __restrict__ knots) {
  using namespace spart::f32;
  __shared__ TauTableF s_tau;
  __shared__ float s_bt[kBandChunk][BT_COUNT];
  __shared__ int s_knot[Soil::kLibrary ? kBandChunk : 1][2];
  const int b0 = blockIdx.x * kBandChunk;
  const int nbc = min(kBandChunk, nb - b0);
  load_tau_table_f(&s_tau);
  exp_table_load();       // the FP64 Stokes solve of near-conservative leaves uses the table-driven exp
  for (int i = threadIdx.x; i < nbc * BT_COUNT; i += blockDim.x)
    (&s_bt[0][0])[i] = (float)band_table[(size_t)b0 * BT_COUNT + i];
  if (Soil::kLibrary)
    for (int i = threadIdx.x; i < nbc * 2; i += blockDim.x) (&s_knot[0][0])[i] = knots[(size_t)b0 * 2 + i];
  __syncthreads();
  const int64_t s = (int64_t)blockIdx.y * kBandThreads + threadIdx.x;
  if (s >= n) return;

  const LeafParF L = load_leaf_f(P, s);
  const Soil soil = Soil::select(P, s, lib);
  SoilParF S;
  S.f1 = rec[R_F1 * n + s]; S.f2 = rec[R_F2 * n + s]; S.f3 = rec[R_F3 * n + s];
  S.mu = rec[R_MU * n + s]; S.emu = rec[R_EMU * n + s]; S.film = (float)P.at(P_FILM, s);
  CanopyGeoF G;
  G.LAI = (float)P.at(P_LAI, s);
  G.k = rec[R_K_SUN * n + s]; G.K = rec[R_K_OBS * n + s]; G.bf = rec[R_BF * n + s];
  G.sob = rec[R_SOB * n + s]; G.sof = rec[R_SOF * n + s];
  G.tau_ss = rec[R_TAUSS * n + s]; G.tau_oo = rec[R_TAUOO * n + s];
  G.sumpso = rec[R_SUMPSO * n + s]; G.pso2w = rec[R_PSO2W * n + s]; G.Z = rec[R_Z * n + s];
  AtmSampleF A;
  A.us = rec[R_US * n + s]; A.uv = rec[R_UV * n + s]; A.m = rec[R_M * n + s]; A.Peq = rec[R_PEQ * n + s];
  A.lo3 = rec[R_LO3 * n + s]; A.lh2o = rec[R_LH2O * n + s]; A.lm = rec[R_LM * n + s]; A.lpeq = rec[R_LPEQ * n + s];
  A.cksi = rec[R_CKSI * n + s]; A.ksiD = rec[R_KSID * n + s]; A.ray_phase = rec[R_RAYPH * n + s];
  A.taup550 = (float)P.at(P_AOT, s);
  A.inv_us = rec[R_INVUS * n + s]; A.inv_uv = rec[R_INVUV * n + s];
  A.inv_1pus = rec[R_INV1PUS * n + s]; A.inv_1puv = rec[R_INV1PUV * n + s]; A.aa3 = rec[R_AA3 * n + s];
  const float etscale = rec[R_ETSCALE * n + s];
  const int nout = compact ? 2 : SPART_NOUT;
  TIO* o = out + ((size_t)s * nb + b0) * nout;
  if (compact && blockIdx.x == 0) out[(size_t)n * nb * 2 + s] = (TIO)etscale;

#pragma unroll 1
  for (int bi = 0; bi < nbc; ++bi) {
    const float* bt = s_bt[bi];
    float rso = 0.0f, rdo = 0.0f, rsd = 0.0f, rdd = 0.0f;
    const int npts = (bt[BT_NPTS] > 1.5f) ? 2 : 1;
#pragma unroll 1
    for (int pt = 0; pt < npts; ++pt) {
      const float* lc = &bt[BT_LC0 + pt * LC_COUNT];
      float refl, tran, absorb, a0, a1, a2, a3;
      prospect_point_f(L, lc, &s_tau, refl, tran, absorb);
      const float rwet = soil.point_f(S, lc, Soil::kLibrary ? s_knot[bi][pt] : 0);
      sailh_point_f(G, refl, tran, absorb, rwet, a0, a1, a2, a3);
      if (pt == 0) {
        rso = a0; rdo = a1; rsd = a2; rdd = a3;
      } else {
        const float fr = bt[BT_FRAC];
        rso = (a0 - rso) * fr + rso;
        rdo = (a1 - rdo) * fr + rdo;
        rsd = (a2 - rsd) * fr + rsd;
        rdd = (a3 - rdd) * fr + rdd;
      }
    }
    float R_TOC, R_TOA, L_TOA;
    smac_toa_band_f(A, &bt[BT_SMAC], bt[BT_CONVEA], etscale, rso, rdo, rdd, rsd, R_TOC, R_TOA, L_TOA);
    o[bi * nout + 0] = (TIO)R_TOC;
    o[bi * nout + 1] = (TIO)R_TOA;
    if (!compact) o[bi * nout + 2] = (TIO)L_TOA;
  }
}

template <typename TIO>
__global__ void __launch_bounds__(kBandThreads)
band_kernel_f32(const ParamsT<TIO> P, int64_t n, const float* __restrict__ rec,
                const double* __restrict__ band_table, int nb, TIO* __restrict__ out, int compact) {
  band_body_f32<TIO, GsvSoil>(P, n, rec, band_table, nb, out, compact, SoilLib{nullptr, 0}, nullptr);
}

// band_kernel_f32 with the dry soil of each sample taken from the soil library (SPART_FLAG_SOIL_LIBRARY)
template <typename TIO>
__global__ void __launch_bounds__(kBandThreads)
soillib_bands_f32(const ParamsT<TIO> P, int64_t n, const float* __restrict__ rec, const double* __restrict__ band_table,
                  int nb, TIO* __restrict__ out, int compact, const SoilLib lib, const int32_t* __restrict__ knots) {
  band_body_f32<TIO, LibrarySoil>(P, n, rec, band_table, nb, out, compact, lib, knots);
}

// Full-spectrum planes (leafopt / soilopt / canopyopt): thread = wavelength, blockIdx.y = sample.
// Every load of the per-wavelength constants and every store of the nine output planes is then
// coalesced along the wavelength axis (the output is 155 KB per sample, so this kernel lives on
// its store pattern); the sample's parameters and record are warp-uniform broadcast loads.
constexpr int kSpecThreads = 256;

template <class Soil>
__device__ __forceinline__ void spectrum_body(const Params& P, int64_t n, const double* __restrict__ rec,
                                              const double* __restrict__ lc_table, int64_t s0, double rho_thermal,
                                              double tau_thermal, double* __restrict__ out, const SoilLib& lib) {
  __shared__ TauTable s_tau;
  load_tau_table(&s_tau);
  exp_table_load();
  __syncthreads();
  const int w = blockIdx.x * kSpecThreads + threadIdx.x;
  const int64_t s = s0 + blockIdx.y;
  if (w >= SPART_NWL_S || s >= n) return;
  const LeafPar L = load_leaf(P, s);
  const SoilPar S = load_soil(P, rec, n, s);
  const CanopyGeo G = load_geo(P, rec, n, s);
  double lc[LC_COUNT];
  const int wc = min(w, SPART_NWL - 1);     // thermal wavelengths re-use the 2400 nm soil constants (SPART.py:440)
#pragma unroll
  for (int r = 0; r < LC_COUNT; ++r) lc[r] = lc_table[(size_t)r * SPART_NWL + wc];
  double refl, tran, kchl, rwet, rdry, rso, rdo, rsd, rdd;
  Soil::select(P, s, lib).point(S, lc, wc, rwet, rdry);
  if (w < SPART_NWL) {
    prospect_point<true>(L, lc, &s_tau, refl, tran, kchl);
  } else {  // thermal assumptions (SPART.py:461-466): LeafBiology.rho_thermal / tau_thermal
    refl = rho_thermal;
    tran = tau_thermal;
    kchl = 0.0;
  }
  sailh_point(G, refl, tran, rwet, rso, rdo, rsd, rdd);
  double* o = out + (size_t)s * SPART_NSPEC * SPART_NWL_S + w;
  o[0 * SPART_NWL_S] = refl;
  o[1 * SPART_NWL_S] = tran;
  o[2 * SPART_NWL_S] = kchl;
  o[3 * SPART_NWL_S] = rwet;
  o[4 * SPART_NWL_S] = rdry;
  o[5 * SPART_NWL_S] = rso;
  o[6 * SPART_NWL_S] = rdo;
  o[7 * SPART_NWL_S] = rsd;
  o[8 * SPART_NWL_S] = rdd;
}

__global__ void __launch_bounds__(kSpecThreads)
spectrum_kernel(const Params P, int64_t n, const double* __restrict__ rec,
                const double* __restrict__ lc_table, int64_t s0, double rho_thermal, double tau_thermal,
                double* __restrict__ out) {
  spectrum_body<GsvSoil>(P, n, rec, lc_table, s0, rho_thermal, tau_thermal, out, SoilLib{nullptr, 0});
}

// spectrum_kernel with the dry soil of each sample taken from the soil library (SPART_FLAG_SOIL_LIBRARY)
__global__ void __launch_bounds__(kSpecThreads)
soillib_spectrum(const Params P, int64_t n, const double* __restrict__ rec, const double* __restrict__ lc_table,
                 int64_t s0, double rho_thermal, double tau_thermal, double* __restrict__ out, const SoilLib lib) {
  spectrum_body<LibrarySoil>(P, n, rec, lc_table, s0, rho_thermal, tau_thermal, out, lib);
}

// ---- peak micro-benchmarks ---------------------------------------------------------------
template <typename T>
__global__ void fma_chain_kernel(T* out, int iters, T a, T b) {
  T x0 = (T)threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6,
    x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
    x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
  }
  T r = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (r == (T)-12345.678) out[0] = r;   // never true; keeps the chain alive
}

// Dependent DFMA chains on register operands, one chain per warp: a degree-6 Horner step u <- g(u) with seven
// per-thread coefficients (the inner loop of lidf_kernel's stage B without its compare).  Eight warps per
// scheduler; what this sustains is the FP64 issue ceiling of code like the leaf-angle / band kernels.
__global__ void __launch_bounds__(1024, 1) fp64_register_chain_kernel(double* out, int iters) {
  double g[7];
  const double base[7] = {0.01, 0.45, 0.1, -0.05, 0.01, 0.002, -0.0003};    // a contraction towards ~0.018
#pragma unroll
  for (int k = 0; k < 7; ++k) g[k] = base[k] * (1.0 + 1e-9 * threadIdx.x);
  double u = 1e-6 * threadIdx.x;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int rep = 0; rep < 4; ++rep) {
      double r = g[6];
#pragma unroll
      for (int k = 5; k >= 0; --k) r = fma(r, u, g[k]);
      u = r;
    }
  }
  if (u == -12345.678) out[0] = u;   // never true; keeps the chain alive
}

// Best rate of four timed runs of `run(d)` on the default stream, the first run not counted (warm-up); `d` is a
// device scratch double the kernels may write, `flops` the work of one run.
template <typename Run>
static int time_peak(double flops, double* tflops, Run run) {
  DeviceBuf<double> d;
  Event e0, e1;
  CUDA_TRY(alloc(d, sizeof(double)));
  CUDA_TRY(create(e0));
  CUDA_TRY(create(e1));
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    CUDA_TRY(cudaEventRecord(e0.get()));
    const int rc = run(d.get());
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(e1.get()));
    CUDA_TRY(cudaEventSynchronize(e1.get()));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0.get(), e1.get()));
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  *tflops = best;
  return SPART_OK;
}

template <typename T>
static int time_fma(int sm_count, double* tflops) {
  const int iters = 1 << 14, threads = 512, blocks = sm_count * 8;
  return time_peak(2.0 * 8.0 * (double)iters * threads * (double)blocks, tflops, [&](double* d) {
    return launch(fma_chain_kernel<T>, blocks, threads, 0, nullptr, (T*)d, iters, (T)1.0000001, (T)1e-7);
  });
}

// --------------------------------------------------------------------------------------
// C ABI
// --------------------------------------------------------------------------------------
namespace {

// Makes `device` current for the duration of an entry point and restores the caller's device on
// exit, so that the library never changes the calling thread's (PyTorch's) current device.
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
    else if (err == cudaSuccess) prev = -1;      // nothing to restore
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define GUARD_DEVICE(dev)                                                                  \
  DeviceGuard _guard(dev);                                                                 \
  if (_guard.err != cudaSuccess) {                                                         \
    snprintf(g_err, sizeof(g_err), "cudaSetDevice(%d) failed: %s", (int)(dev), cudaGetErrorString(_guard.err)); \
    return (int)_guard.err;                                                                \
  }

// NVTX range around a group of launches (the reference annotates its stages with nvtx,
// SPART.py:191-227); a no-op unless a profiler is attached.
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

}  // namespace

constexpr int kSrfMaxSlots = 24;      // 24 x 4 x 128 doubles = 96 KB of accumulators at most

// __constant__ tables are per device: upload them once for every device that is used.  The dynamic shared-memory
// cap of the SRF kernels is set here too, once, to the largest plan spart_create accepts: the attribute belongs to
// the kernel and device, not to a context, so setting it per call to that call's plan size would let a concurrent
// call with a smaller plan lower it between another thread's set and launch.
static int init_device_constants(int device) {
  static std::mutex mu;
  static bool done[64] = {false};
  std::lock_guard<std::mutex> lock(mu);
  if (device < 0 || device >= 64) return fail(SPART_EINVAL, "device index out of range%s");
  if (done[device]) return SPART_OK;
  GUARD_DEVICE(device);
  CUDA_TRY(cudaMemcpyToSymbol(c_tau_coef, SPART_TAU_COEF_H, sizeof(SPART_TAU_COEF_H)));
  CUDA_TRY(cudaMemcpyToSymbol(c_tau_mid, SPART_TAU_MID_H, sizeof(SPART_TAU_MID_H)));
  CUDA_TRY(cudaMemcpyToSymbol(c_tau_invhalf, SPART_TAU_INVHALF_H, sizeof(SPART_TAU_INVHALF_H)));
  CUDA_TRY(cudaMemcpyToSymbol(f32::c_tauf_coef, SPART_TAUF_COEF_H, sizeof(SPART_TAUF_COEF_H)));
  double sl[13], cl[13];
  for (int i = 0; i < 13; ++i) {  // litab (sailh.py:49): 5,15,...,75, 81,83,...,89 degrees
    const double li = (i < 8) ? 5.0 + 10.0 * i : 81.0 + 2.0 * (i - 8);
    sl[i] = sin(li * (M_PI / 180.0));
    cl[i] = cos(li * (M_PI / 180.0));
  }
  double th2[12];
  for (int i = 0; i < 12; ++i) {  // dcum angles (sailh.py:388-393) and x0 = 2*rd*theta (sailh.py:376)
    const double theta = (i < 8) ? 10.0 * (i + 1) : 80.0 + 2.0 * (i - 7);
    th2[i] = 2.0 * (M_PI / 180.0) * theta;
  }
  CUDA_TRY(cudaMemcpyToSymbol(c_theta2, th2, sizeof(th2)));
  {
    float th2f[12], slf[13], clf[13];
    for (int i = 0; i < 12; ++i) th2f[i] = (float)th2[i];
    for (int i = 0; i < 13; ++i) {
      slf[i] = (float)sl[i];
      clf[i] = (float)cl[i];
    }
    CUDA_TRY(cudaMemcpyToSymbol(c_theta2_f, th2f, sizeof(th2f)));
    CUDA_TRY(cudaMemcpyToSymbol(c_sin_ttli_f, slf, sizeof(slf)));
    CUDA_TRY(cudaMemcpyToSymbol(c_cos_ttli_f, clf, sizeof(clf)));
  }
  CUDA_TRY(cudaMemcpyToSymbol(c_sin_ttli, sl, sizeof(sl)));
  CUDA_TRY(cudaMemcpyToSymbol(c_cos_ttli, cl, sizeof(cl)));
  const int srf_max_bytes = (int)(sizeof(double) * kSrfMaxSlots * 4 * kBandThreads);
  CUDA_TRY(cudaFuncSetAttribute(band_kernel_srf, cudaFuncAttributeMaxDynamicSharedMemorySize, srf_max_bytes));
  CUDA_TRY(cudaFuncSetAttribute(soillib_srf, cudaFuncAttributeMaxDynamicSharedMemorySize, srf_max_bytes));

  done[device] = true;
  return SPART_OK;
}

extern "C" {

int spart_abi_version(void) { return SPART_ABI_VERSION; }
const char* spart_last_error(void) { return g_err; }
int64_t spart_launch_count(void) { return g_launches; }

int spart_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int spart_destroy(SpartCtx* ctx) {
  if (!ctx) return SPART_OK;
  DeviceGuard guard(ctx->device);
  // work of device-path calls may still be queued on callers' streams and read the context's tables: wait for
  // everything on the device, not only for the host path's own streams, before anything is freed
  cudaDeviceSynchronize();
  delete ctx;
  return SPART_OK;
}

}  // extern "C"

template <typename T>
static int upload(const std::vector<T>& v, DeviceBuf<T>& d) {
  CUDA_TRY(alloc(d, sizeof(T) * (v.empty() ? 1 : v.size())));
  if (!v.empty()) CUDA_TRY(cudaMemcpy(d.get(), v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
  return SPART_OK;
}

// SRF band mode: turn the per-band (wavelength, weight) lists into the schedule band_kernel_srf walks --
// distinct wavelengths in ascending order, per wavelength the (accumulator slot, weight) pairs to add and
// the bands that are complete after it.  Slots are an interval colouring of the bands' supports.
static int build_srf_plan(const SpartSensor& S, SpartCtx::SrfDev& dev) {
  const int nb = S.n_bands;
  std::vector<int64_t> off(nb + 1, 0);
  for (int b = 0; b < nb; ++b) {
    if (S.srf_len[b] < 0) return fail(SPART_EINVAL, "spart_create: negative SRF length%s");
    off[b + 1] = off[b] + S.srf_len[b];
  }
  const int64_t total = off[nb];
  std::vector<char> used(SPART_NWL, 0);
  for (int64_t k = 0; k < total; ++k) {
    if (S.srf_idx[k] < 0 || S.srf_idx[k] >= SPART_NWL)
      return fail(SPART_EINVAL, "spart_create: SRF wavelength index outside 400..2400 nm%s");
    used[S.srf_idx[k]] = 1;
  }
  std::vector<int32_t> wl_idx, pos(SPART_NWL, -1);
  for (int w = 0; w < SPART_NWL; ++w)
    if (used[w]) {
      pos[w] = (int32_t)wl_idx.size();
      wl_idx.push_back(w);
    }
  const int U = (int)wl_idx.size();
  // first / last position of every band on the distinct-wavelength axis
  std::vector<int> first(nb, U), last(nb, -1);
  for (int b = 0; b < nb; ++b)
    for (int64_t k = off[b]; k < off[b + 1]; ++k) {
      const int q = pos[S.srf_idx[k]];
      if (q < first[b]) first[b] = q;
      if (q > last[b]) last[b] = q;
    }
  // interval colouring: walk the wavelengths, release the slots of finished bands, hand the lowest free
  // slot to every band that starts
  std::vector<int> slot(nb, -1), free_slots;
  int n_slots = 0;
  std::vector<std::vector<int>> starts(U + 1), ends(U + 1);
  for (int b = 0; b < nb; ++b)
    if (last[b] >= 0) {
      starts[first[b]].push_back(b);
      ends[last[b]].push_back(b);
    }
  for (int q = 0; q < U; ++q) {
    for (int b : starts[q]) {
      if (free_slots.empty()) free_slots.push_back(n_slots++);
      slot[b] = free_slots.back();
      free_slots.pop_back();
    }
    for (int b : ends[q]) free_slots.push_back(slot[b]);
  }
  const int spare = n_slots++;          // only for bands without any SRF weight, see the end of the plan
  if (n_slots > kSrfMaxSlots) return fail(SPART_EINVAL, "spart_create: too many overlapping bands for the SRF band mode%s");
  if (U == 0) return fail(SPART_EINVAL, "spart_create: SRF tables without a single sample%s");
  // per wavelength: pairs in ascending band order (each band's own sum keeps its ascending wavelength order)
  std::vector<std::vector<std::pair<int, double>>> pairs(U);
  for (int b = 0; b < nb; ++b)
    for (int64_t k = off[b]; k < off[b + 1]; ++k) pairs[pos[S.srf_idx[k]]].push_back({slot[b], S.srf_w[k]});
  std::vector<int32_t> pair_off(U + 1, 0), pair_slot, fin_off(U + 1, 0), fin_band, fin_slot;
  std::vector<double> pair_w;
  for (int q = 0; q < U; ++q) {
    for (auto& pr : pairs[q]) {
      pair_slot.push_back(pr.first);
      pair_w.push_back(pr.second);
    }
    pair_off[q + 1] = (int32_t)pair_slot.size();
    for (int b : ends[q]) {
      fin_band.push_back(b);
      fin_slot.push_back(slot[b]);
    }
    fin_off[q + 1] = (int32_t)fin_band.size();
  }
  // A band without any SRF weight is 0 / 0 in calculate_spectral_convolution (SPART.py:389-396): its band
  // reflectances, and with them R_TOC, R_TOA and L_TOA, are NaN.  Each such band gets one more step (a repeat
  // of the last wavelength) that adds a NaN weight into the spare slot and finishes the band from there; the
  // kernel needs no test of its own for it.
  for (int b = 0; b < nb; ++b)
    if (last[b] < 0) {
      wl_idx.push_back(wl_idx[U - 1]);
      pair_slot.push_back(spare);
      pair_w.push_back(__builtin_nan(""));
      pair_off.push_back((int32_t)pair_slot.size());
      fin_band.push_back(b);
      fin_slot.push_back(spare);
      fin_off.push_back((int32_t)fin_band.size());
    }
  dev.n_wl = (int)wl_idx.size();
  dev.n_slots = n_slots;
  int rc;
  if ((rc = upload(wl_idx, dev.wl_idx)) || (rc = upload(pair_off, dev.pair_off)) ||
      (rc = upload(pair_slot, dev.pair_slot)) || (rc = upload(pair_w, dev.pair_w)) ||
      (rc = upload(fin_off, dev.fin_off)) || (rc = upload(fin_band, dev.fin_band)) ||
      (rc = upload(fin_slot, dev.fin_slot)))
    return rc;
  return SPART_OK;
}

// body of spart_create; on any failure the caller deletes the partially built context, which releases it
static int create_into(SpartCtx* ctx, const SpartTables* tables, const SpartSensor* sensors, int32_t n_sensors,
                       const double* soils, int32_t n_soils, int32_t device) {
  CUDA_TRY(cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device));
  int rc = init_device_constants(device);
  if (rc) return rc;
  const size_t lc_bytes = sizeof(double) * LC_COUNT * SPART_NWL;
  CUDA_TRY(alloc(ctx->d_lc, lc_bytes));
  CUDA_TRY(cudaMemcpy(ctx->d_lc.get(), tables->lc, lc_bytes, cudaMemcpyHostToDevice));
  if (soils) {
    // the library plus one row of NaN that invalid sample indices are pointed at
    const size_t lib_bytes = sizeof(double) * (size_t)n_soils * SPART_NWL;
    const std::vector<double> nan_row(SPART_NWL, __builtin_nan(""));
    CUDA_TRY(alloc(ctx->d_soils, lib_bytes + sizeof(double) * SPART_NWL));
    CUDA_TRY(cudaMemcpy(ctx->d_soils.get(), soils, lib_bytes, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(ctx->d_soils.get() + (size_t)n_soils * SPART_NWL, nan_row.data(), sizeof(double) * SPART_NWL,
                        cudaMemcpyHostToDevice));
    ctx->n_soils = n_soils;
  }

  ctx->n_bands.resize(n_sensors);
  ctx->d_band.resize(n_sensors);
  ctx->d_knot.resize(n_sensors);
  ctx->srf.resize(n_sensors);
  for (int i = 0; i < n_sensors; ++i) {
    const SpartSensor& S = sensors[i];
    std::vector<double> bt((size_t)S.n_bands * BT_COUNT, 0.0);
    for (int b = 0; b < S.n_bands; ++b) {
      double* row = &bt[(size_t)b * BT_COUNT];
      for (int r = 0; r < SM_COUNT; ++r) row[BT_SMAC + r] = S.smac[(size_t)r * S.n_bands + b];
      row[BT_CONVEA] = S.conv_ea[b];
      row[BT_FRAC] = S.wl_frac[b];
      row[BT_NPTS] = (S.wl_hi[b] != S.wl_lo[b]) ? 2.0 : 1.0;
      for (int r = 0; r < LC_COUNT; ++r) {
        row[BT_LC0 + r] = tables->lc[(size_t)r * SPART_NWL + S.wl_lo[b]];
        row[BT_LC1 + r] = tables->lc[(size_t)r * SPART_NWL + S.wl_hi[b]];
      }
    }
    std::vector<int32_t> knots((size_t)S.n_bands * 2);
    for (int b = 0; b < S.n_bands; ++b) {
      knots[(size_t)b * 2] = S.wl_lo[b];
      knots[(size_t)b * 2 + 1] = S.wl_hi[b];
    }
    ctx->n_bands[i] = S.n_bands;
    if ((rc = upload(bt, ctx->d_band[i])) || (rc = upload(knots, ctx->d_knot[i]))) return rc;
    if (S.srf_idx && S.srf_len && S.srf_w) {
      rc = build_srf_plan(S, ctx->srf[i]);
      if (rc) return rc;
    }
  }
  return SPART_OK;
}

static int create_ctx(const SpartTables* tables, const SpartSensor* sensors, int32_t n_sensors, const double* soils,
                      int32_t n_soils, int32_t device, SpartCtx** out) {
  if (!tables || !tables->lc || !out || n_sensors < 0 || (n_sensors > 0 && !sensors))
    return fail(SPART_EINVAL, "spart_create: null argument%s");
  if (tables->n_wl != SPART_NWL) return fail(SPART_EINVAL, "spart_create: tables->n_wl must be 2001%s");
  int ndev = spart_device_count();
  if (ndev <= 0) return fail(SPART_ENODEV, "spart_create: no CUDA device (this library has no CPU fallback)%s");
  if (device < 0 || device >= ndev) return fail(SPART_EINVAL, "spart_create: device index out of range%s");
  for (int i = 0; i < n_sensors; ++i) {
    const SpartSensor& S = sensors[i];
    if (S.n_bands <= 0 || !S.wl_lo || !S.wl_hi || !S.wl_frac || !S.smac || !S.conv_ea)
      return fail(SPART_EINVAL, "spart_create: incomplete sensor%s");
    for (int b = 0; b < S.n_bands; ++b)
      if (S.wl_lo[b] < 0 || S.wl_lo[b] >= SPART_NWL || S.wl_hi[b] < S.wl_lo[b] || S.wl_hi[b] >= SPART_NWL)
        return fail(SPART_EINVAL, "spart_create: band knot outside 400..2400 nm%s");
  }
  GUARD_DEVICE(device);
  std::unique_ptr<SpartCtx> ctx(new (std::nothrow) SpartCtx());
  if (!ctx) return fail(SPART_ENOMEM, "spart_create: out of host memory%s");
  ctx->device = device;
  ctx->n_sensors = n_sensors;
  const int rc = create_into(ctx.get(), tables, sensors, n_sensors, soils, n_soils, device);
  if (rc) return rc;
  *out = ctx.release();
  return SPART_OK;
}

extern "C" {

int spart_create(const SpartTables* tables, const SpartSensor* sensors, int32_t n_sensors, int32_t device,
                 SpartCtx** out) {
  return create_ctx(tables, sensors, n_sensors, nullptr, 0, device, out);
}

int spart_create_with_soils(const SpartTables* tables, const SpartSensor* sensors, int32_t n_sensors,
                            const double* soils, int32_t n_soils, int32_t device, SpartCtx** out) {
  if (!soils) return fail(SPART_EINVAL, "spart_create_with_soils: null soil library%s");
  // F32_IO carries the index as a float, which holds every whole number only up to 2^24
  if (n_soils < 1 || n_soils > (1 << 24)) return fail(SPART_EINVAL, "spart_create_with_soils: need 1 <= n_soils <= 2^24%s");
  return create_ctx(tables, sensors, n_sensors, soils, n_soils, device, out);
}

size_t spart_workspace_bytes(const SpartCtx* ctx, int64_t n) {
  (void)ctx;
  if (n < 0) return 0;
  return sizeof(double) * (size_t)kWsRows * (size_t)n;
}

}  // extern "C"

static int launch_lidf(const Params& P, int64_t n_batch, double* ws, cudaStream_t st) {
  // LIDFa and LIDFb both broadcast rows (a look-up table with one leaf-angle distribution): the twelve
  // iterations run once, geometry_kernel reads element 0 of the F rows (kFlagLidfBcast)
  const int64_t n = ((P.bc & kLidfRows) == kLidfRows) ? 1 : n_batch;
  return launch(lidf_kernel, (unsigned)((n + kL2Samples - 1) / kL2Samples), kL2Threads, 0, st, P.ptr(P_LIDFA, 0),
                P.ptr(P_LIDFB, 0), ((P.bc >> P_LIDFA) & 1u) ? 0 : 1, ((P.bc >> P_LIDFB) & 1u) ? 0 : 1, n,
                ws + (size_t)kRowF * n_batch, n_batch, 1);
}

static int launch_geometry(const Params& P, int64_t n, double* ws, int kflags, cudaStream_t st) {
  if ((P.bc & kLidfRows) == kLidfRows && !(kflags & kFlagLidfDirect)) kflags |= kFlagLidfBcast;
  return launch(geometry_kernel, (unsigned)((n + kSampleThreads - 1) / kSampleThreads), kSampleThreads, 0, st, P, n,
                ws, kflags);
}

static int check_batch(const SpartCtx* ctx, const void* params, int64_t n, int64_t ld, uint32_t bc, const void* ws,
                       const void* out, const char* who) {
  if (!ctx || !params || !out || (!ws && n > 0)) return fail(SPART_EINVAL, "%s: null argument", who);
  if (n < 0 || ld < n) return fail(SPART_EINVAL, "%s: need 0 <= n <= ld", who);
  if (bc >> SPART_NPAR) return fail(SPART_EINVAL, "%s: broadcast_rows has bits beyond row 26", who);
  if (n > (int64_t)65535 * kBandThreads)
    return fail(SPART_EINVAL, "%s: n exceeds 65535*128 samples per call; split the batch", who);
  return SPART_OK;
}

static const int kKnownFlags = SPART_FLAG_SOIL_SPECTRUM | SPART_FLAG_SRF_BANDS | SPART_FLAG_REUSE_RECORD |
                               SPART_FLAG_F32_IO | SPART_FLAG_COMPACT_OUT | SPART_FLAG_USER_LIDF |
                               SPART_FLAG_SOIL_LIBRARY;

// SPART_FLAG_SOIL_LIBRARY needs a context with a library and excludes SPART_FLAG_SOIL_SPECTRUM
static int check_soil_library(const SpartCtx* ctx, int32_t flags, const char* who) {
  if (!(flags & SPART_FLAG_SOIL_LIBRARY)) return SPART_OK;
  if (flags & SPART_FLAG_SOIL_SPECTRUM)
    return fail(SPART_EINVAL, "%s: SPART_FLAG_SOIL_LIBRARY and SPART_FLAG_SOIL_SPECTRUM exclude each other", who);
  if (!ctx->d_soils) return fail(SPART_EINVAL, "%s: SPART_FLAG_SOIL_LIBRARY needs a context created with a soil library", who);
  return SPART_OK;
}

// the geometry kernels see a library run as a user-spectrum run: soil weights (1, 0, 0)
static int soil_kflags(int32_t flags) {
  return (flags & (SPART_FLAG_SOIL_SPECTRUM | SPART_FLAG_SOIL_LIBRARY)) ? SPART_FLAG_SOIL_SPECTRUM : 0;
}

// flag / precision combinations shared by the device and the host entry point
static int check_mode(const SpartCtx* ctx, int32_t sensor, int32_t precision, int32_t flags, const char* who) {
  if (sensor < 0 || sensor >= ctx->n_sensors) return fail(SPART_EINVAL, "%s: unknown sensor", who);
  if (precision != SPART_FP64 && precision != SPART_FP32)
    return fail(SPART_EINVAL, "%s: precision must be SPART_FP64 or SPART_FP32", who);
  if (flags & ~kKnownFlags) return fail(SPART_EINVAL, "%s: unknown flag bit", who);
  if ((flags & SPART_FLAG_F32_IO) && precision != SPART_FP32)
    return fail(SPART_EINVAL, "%s: SPART_FLAG_F32_IO needs SPART_FP32", who);
  if ((flags & SPART_FLAG_USER_LIDF) && precision != SPART_FP64)
    return fail(SPART_EINVAL, "%s: SPART_FLAG_USER_LIDF needs SPART_FP64", who);
  if ((flags & SPART_FLAG_USER_LIDF) && (flags & SPART_FLAG_REUSE_RECORD))
    return fail(SPART_EINVAL, "%s: SPART_FLAG_USER_LIDF and SPART_FLAG_REUSE_RECORD exclude each other", who);
  if (flags & SPART_FLAG_SRF_BANDS) {
    if (precision != SPART_FP64) return fail(SPART_EINVAL, "%s: SRF band mode needs SPART_FP64", who);
    if (!ctx->srf[sensor].pair_w) return fail(SPART_EINVAL, "%s: this sensor was created without SRF tables", who);
  }
  return check_soil_library(ctx, flags, who);
}

template <typename TIO>
static int launch_fp32(const SpartCtx* ctx, int sensor, const void* params_dev, const void* params_bc_dev, int64_t n,
                       int64_t ld, uint32_t bc, int kflags, bool reuse, bool compact, bool library, float* rec,
                       void* out_dev,
                       dim3 grid, cudaStream_t st, bool prof, const SpartCtx::ProfEvents& pe) {
  const ParamsT<TIO> P{(const TIO*)params_dev, ld, bc, (const TIO*)params_bc_dev};
  const double* band = ctx->d_band[sensor].get();
  const int nb = ctx->n_bands[sensor];
  if (prof) CUDA_TRY(cudaEventRecord(pe.e[1].get(), st));
  if (!reuse) {
    NvtxRange r("spart::geometry_f32");
    const int rc = launch(geometry_kernel_f32<TIO>, (unsigned)((n + kSampleThreads - 1) / kSampleThreads),
                          kSampleThreads, 0, st, P, n, rec, kflags);
    if (rc) return rc;
  }
  if (prof) CUDA_TRY(cudaEventRecord(pe.e[2].get(), st));
  NvtxRange r("spart::bands_f32");
  if (library)
    return launch(soillib_bands_f32<TIO>, grid, kBandThreads, 0, st, P, n, rec, band, nb, (TIO*)out_dev,
                  compact ? 1 : 0, SoilLib{ctx->d_soils.get(), ctx->n_soils}, ctx->d_knot[sensor].get());
  return launch(band_kernel_f32<TIO>, grid, kBandThreads, 0, st, P, n, rec, band, nb, (TIO*)out_dev, compact ? 1 : 0);
}

// spart_forward_bands with a separate base for the broadcast rows (see ParamsT); the host-buffer path calls it on
// chunks of a device-resident span
static int forward_bands_impl(const SpartCtx* ctx, int32_t sensor, const void* params_dev, const void* params_bc_dev,
                              int64_t n, int64_t ld, uint32_t broadcast_rows, int32_t precision, int32_t flags,
                              void* workspace_dev, void* out_dev, void* stream) {
  int rc = check_batch(ctx, params_dev, n, ld, broadcast_rows, workspace_dev, out_dev, "spart_forward_bands");
  if (rc) return rc;
  rc = check_mode(ctx, sensor, precision, flags, "spart_forward_bands");
  if (rc) return rc;
  if (n == 0) return SPART_OK;
  GUARD_DEVICE(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  double* rec = (double*)workspace_dev;
  // the call's profiling events: released on any return before they are handed to prof_pending
  SpartCtx::ProfEvents pe;
  bool prof = false;
  {
    std::lock_guard<std::mutex> lock(ctx->prof_mu);
    if (ctx->profiling) {
      prof = true;
      if (!ctx->prof_free.empty()) {
        pe = std::move(ctx->prof_free.back());
        ctx->prof_free.pop_back();
      } else {
        for (Event& e : pe.e) CUDA_TRY(create(e));
      }
    }
  }
  const int nb = ctx->n_bands[sensor];
  const double* band = ctx->d_band[sensor].get();
  dim3 grid((unsigned)((nb + kBandChunk - 1) / kBandChunk), (unsigned)((n + kBandThreads - 1) / kBandThreads));
  const bool reuse = (flags & SPART_FLAG_REUSE_RECORD) != 0;   // workspace already holds this batch's record
  const int compact = (flags & SPART_FLAG_COMPACT_OUT) ? 1 : 0;
  // one sun / observer geometry for the whole batch by construction: rows 19..21 are broadcast rows
  const bool uniform = (broadcast_rows & kGeometryRows) == kGeometryRows;
  const bool user_lidf = (flags & SPART_FLAG_USER_LIDF) != 0;   // the workspace holds the caller's distribution
  const bool library = (flags & SPART_FLAG_SOIL_LIBRARY) != 0;    // per-sample dry soil from the context's library
  const SoilLib lib{ctx->d_soils.get(), ctx->n_soils};
  const int kflags = soil_kflags(flags) | (uniform ? kFlagUniform : 0) | (user_lidf ? kFlagLidfDirect : 0);
  if (prof) CUDA_TRY(cudaEventRecord(pe.e[0].get(), st));
  if (precision == SPART_FP64) {
    const Params P{(const double*)params_dev, ld, broadcast_rows, (const double*)params_bc_dev};
    double* out = (double*)out_dev;
    if (!reuse && !user_lidf) {
      NvtxRange r("spart::leaf_angles");
      rc = launch_lidf(P, n, rec, st);
      if (rc) return rc;
    }
    if (prof) CUDA_TRY(cudaEventRecord(pe.e[1].get(), st));
    if (!reuse) {
      NvtxRange r("spart::geometry");
      rc = launch_geometry(P, n, rec, kflags, st);
      if (rc) return rc;
    }
    if (prof) CUDA_TRY(cudaEventRecord(pe.e[2].get(), st));
    NvtxRange r("spart::bands");
    if (flags & SPART_FLAG_SRF_BANDS) {
      const SpartCtx::SrfDev& v = ctx->srf[sensor];
      const SrfPlan plan{v.n_wl, v.n_slots, v.wl_idx.get(), v.pair_off.get(), v.pair_slot.get(), v.pair_w.get(),
                         v.fin_off.get(), v.fin_band.get(), v.fin_slot.get()};
      const size_t acc_bytes = sizeof(double) * v.n_slots * 4 * kBandThreads;
      const unsigned blocks = (unsigned)((n + kBandThreads - 1) / kBandThreads);
      // the kernels' dynamic shared-memory cap was set to the kSrfMaxSlots bound once per device
      if (library)
        rc = launch(soillib_srf, blocks, kBandThreads, acc_bytes, st, P, n, rec, band, ctx->d_lc.get(), plan, nb, out,
                    compact, lib);
      else
        rc = launch(band_kernel_srf, blocks, kBandThreads, acc_bytes, st, P, n, rec, band, ctx->d_lc.get(), plan, nb,
                    out, compact);
    } else if (library) {
      rc = launch(uniform ? soillib_bands<true> : soillib_bands<false>, grid, kBandThreads, 0, st, P, n, rec, band, nb,
                  out, compact, lib, ctx->d_knot[sensor].get());
    } else {
      rc = launch(uniform ? band_kernel<true> : band_kernel<false>, grid, kBandThreads, 0, st, P, n, rec, band, nb,
                  out, compact);
    }
  } else if (flags & SPART_FLAG_F32_IO) {   // SPART_FP32: the leaf angles are solved inside the geometry kernel
    rc = launch_fp32<float>(ctx, sensor, params_dev, params_bc_dev, n, ld, broadcast_rows, kflags, reuse, compact,
                            library, (float*)rec, out_dev, grid, st, prof, pe);
  } else {
    rc = launch_fp32<double>(ctx, sensor, params_dev, params_bc_dev, n, ld, broadcast_rows, kflags, reuse, compact,
                             library, (float*)rec, out_dev, grid, st, prof, pe);
  }
  if (rc) return rc;
  if (prof) {
    CUDA_TRY(cudaEventRecord(pe.e[3].get(), st));
    std::lock_guard<std::mutex> lock(ctx->prof_mu);
    ctx->prof_pending.push_back(std::move(pe));
  }
  return SPART_OK;
}

extern "C" {

int spart_forward_bands(const SpartCtx* ctx, int32_t sensor, const void* params_dev, int64_t n, int64_t ld,
                        uint32_t broadcast_rows, int32_t precision, int32_t flags, void* workspace_dev, void* out_dev,
                        void* stream) {
  return forward_bands_impl(ctx, sensor, params_dev, params_dev, n, ld, broadcast_rows, precision, flags,
                            workspace_dev, out_dev, stream);
}

int spart_forward_bands_bc(const SpartCtx* ctx, int32_t sensor, const void* params_dev, const void* params_bc_dev,
                           int64_t n, int64_t ld, uint32_t broadcast_rows, int32_t precision, int32_t flags,
                           void* workspace_dev, void* out_dev, void* stream) {
  if (!params_bc_dev) return fail(SPART_EINVAL, "spart_forward_bands_bc: null broadcast base%s");
  return forward_bands_impl(ctx, sensor, params_dev, params_bc_dev, n, ld, broadcast_rows, precision, flags,
                            workspace_dev, out_dev, stream);
}

int spart_profile_enable(SpartCtx* ctx, int32_t on) {
  if (!ctx) return fail(SPART_EINVAL, "spart_profile_enable: null context%s");
  std::lock_guard<std::mutex> lock(ctx->prof_mu);
  ctx->profiling = on != 0;
  for (auto& pe : ctx->prof_pending) ctx->prof_free.push_back(std::move(pe));
  ctx->prof_pending.clear();
  return SPART_OK;
}

int spart_profile_read(SpartCtx* ctx, double* kernel_ms, int64_t* calls) {
  if (!ctx || !kernel_ms || !calls) return fail(SPART_EINVAL, "spart_profile_read: null argument%s");
  GUARD_DEVICE(ctx->device);
  std::lock_guard<std::mutex> lock(ctx->prof_mu);
  double acc[SPART_NKERNELS] = {0.0, 0.0, 0.0};
  for (auto& pe : ctx->prof_pending) {
    CUDA_TRY(cudaEventSynchronize(pe.e[3].get()));
    for (int k = 0; k < SPART_NKERNELS; ++k) {
      float ms = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&ms, pe.e[k].get(), pe.e[k + 1].get()));
      acc[k] += ms;
    }
  }
  for (int k = 0; k < SPART_NKERNELS; ++k) kernel_ms[k] = acc[k];
  *calls = (int64_t)ctx->prof_pending.size();
  for (auto& pe : ctx->prof_pending) ctx->prof_free.push_back(std::move(pe));
  ctx->prof_pending.clear();
  return SPART_OK;
}

int spart_forward_spectrum(const SpartCtx* ctx, const double* params_dev, int64_t n, int64_t ld, int32_t flags,
                           double rho_thermal, double tau_thermal, void* workspace_dev, double* out_dev,
                           void* stream) {
  int rc = check_batch(ctx, params_dev, n, ld, 0, workspace_dev, out_dev, "spart_forward_spectrum");
  if (rc) return rc;
  if (flags & ~(SPART_FLAG_SOIL_SPECTRUM | SPART_FLAG_USER_LIDF | SPART_FLAG_SOIL_LIBRARY))
    return fail(SPART_EINVAL, "spart_forward_spectrum: unknown flag bit%s");
  rc = check_soil_library(ctx, flags, "spart_forward_spectrum");
  if (rc) return rc;
  if (n == 0) return SPART_OK;
  GUARD_DEVICE(ctx->device);
  NvtxRange r("spart::spectrum");
  cudaStream_t st = (cudaStream_t)stream;
  double* rec = (double*)workspace_dev;
  const Params P{params_dev, ld, 0u};
  const bool user_lidf = (flags & SPART_FLAG_USER_LIDF) != 0;     // spart_set_lidf filled the workspace
  if (!user_lidf) {
    rc = launch_lidf(P, n, rec, st);
    if (rc) return rc;
  }
  rc = launch_geometry(P, n, rec, soil_kflags(flags) | (user_lidf ? kFlagLidfDirect : 0), st);
  if (rc) return rc;
  for (int64_t s0 = 0; s0 < n; s0 += 65535) {
    const unsigned ny = (unsigned)((n - s0 < 65535) ? (n - s0) : 65535);
    dim3 grid((SPART_NWL_S + kSpecThreads - 1) / kSpecThreads, ny);
    if (flags & SPART_FLAG_SOIL_LIBRARY)
      rc = launch(soillib_spectrum, grid, kSpecThreads, 0, st, P, n, rec, ctx->d_lc.get(), s0, rho_thermal,
                  tau_thermal, out_dev, SoilLib{ctx->d_soils.get(), ctx->n_soils});
    else
      rc = launch(spectrum_kernel, grid, kSpecThreads, 0, st, P, n, rec, ctx->d_lc.get(), s0, rho_thermal,
                  tau_thermal, out_dev);
    if (rc) return rc;
  }
  return SPART_OK;
}

int spart_smac(const SpartCtx* ctx, int32_t sensor, const double* params_dev, int64_t n, int64_t ld,
               void* workspace_dev, double* out_dev, void* stream) {
  int rc = check_batch(ctx, params_dev, n, ld, 0, workspace_dev, out_dev, "spart_smac");
  if (rc) return rc;
  if (sensor < 0 || sensor >= ctx->n_sensors) return fail(SPART_EINVAL, "spart_smac: unknown sensor%s");
  if (n == 0) return SPART_OK;
  GUARD_DEVICE(ctx->device);
  NvtxRange r("spart::smac");
  cudaStream_t st = (cudaStream_t)stream;
  double* rec = (double*)workspace_dev;
  const Params P{params_dev, ld, 0u};
  rc = launch_lidf(P, n, rec, st);
  if (rc) return rc;
  rc = launch_geometry(P, n, rec, 0, st);
  if (rc) return rc;
  const int nb = ctx->n_bands[sensor];
  dim3 grid((unsigned)nb, (unsigned)((n + kBandThreads - 1) / kBandThreads));
  return launch(smac_kernel, grid, kBandThreads, 0, st, P, n, rec, ctx->d_band[sensor].get(), nb, out_dev);
}

int spart_sailh(const SpartCtx* ctx, const double* params_dev, int64_t n, int64_t ld, const double* soil_refl_dev,
                const double* leaf_refl_dev, const double* leaf_tran_dev, int64_t spectra_stride,
                void* workspace_dev, double* out_dev, void* stream) {
  int rc = check_batch(ctx, params_dev, n, ld, 0, workspace_dev, out_dev, "spart_sailh");
  if (rc) return rc;
  if (!soil_refl_dev || !leaf_refl_dev || !leaf_tran_dev) return fail(SPART_EINVAL, "spart_sailh: null spectrum%s");
  if (spectra_stride != 0 && spectra_stride < SPART_NWL_S)
    return fail(SPART_EINVAL, "spart_sailh: spectra_stride must be 0 (shared spectra) or >= 2162%s");
  if (n == 0) return SPART_OK;
  GUARD_DEVICE(ctx->device);
  NvtxRange r("spart::sailh");
  cudaStream_t st = (cudaStream_t)stream;
  double* rec = (double*)workspace_dev;
  const Params P{params_dev, ld, 0u};
  rc = launch_lidf(P, n, rec, st);
  if (rc) return rc;
  rc = launch_geometry(P, n, rec, 0, st);
  if (rc) return rc;
  for (int64_t s0 = 0; s0 < n; s0 += 65535) {
    const unsigned ny = (unsigned)((n - s0 < 65535) ? (n - s0) : 65535);
    dim3 grid((SPART_NWL_S + 255) / 256, ny);
    rc = launch(sailh_spectra_kernel, grid, 256, 0, st, P, n, rec, soil_refl_dev, leaf_refl_dev, leaf_tran_dev,
                spectra_stride, s0, out_dev);
    if (rc) return rc;
  }
  return SPART_OK;
}

size_t spart_lut_workspace_bytes(int64_t m) { return m > 0 ? sizeof(unsigned long long) * (size_t)m : 0; }

}  // extern "C"

// argument check of spart_lut_nearest (`who`, max_bands 32, k 1), spart_lut_nearest_tc (max_bands 30) and
// spart_lut_topk (max_bands 32, 1 <= k <= kLutTopkMax)
static int check_lut(const char* who, int max_bands, int32_t k, const float* lut_dev, int64_t n, int32_t n_bands,
                     const float* obs_dev, int64_t m, int64_t index_offset, const void* workspace_dev,
                     const int64_t* best_index_dev, const float* best_cost_dev, const unsigned long long* packed_dev) {
  if (k < 1 || k > kLutTopkMax) {
    snprintf(g_err, sizeof(g_err), "%s: need 1 <= k <= %d", who, kLutTopkMax);
    return SPART_EINVAL;
  }
  if (!lut_dev || !obs_dev || (!workspace_dev && m > 0)) return fail(SPART_EINVAL, "%s: null argument", who);
  if (!packed_dev && (!best_index_dev || !best_cost_dev))
    return fail(SPART_EINVAL, "%s: need best_index_dev + best_cost_dev or packed_dev", who);
  if (n <= 0 || n > 0x7fffffffLL || m < 0 || n_bands < 1 || n_bands > max_bands || index_offset < 0 ||
      index_offset + n > 0xffffffffLL) {
    snprintf(g_err, sizeof(g_err),
             "%s: need 1 <= n < 2^31, m >= 0, 1 <= n_bands <= %d, index_offset + n < 2^32", who, max_bands);
    return SPART_EINVAL;
  }
  return SPART_OK;
}

// The grid of a LUT search: `obs_per_block` observations by LUT slices of whole `tile`-entry tiles, enough slices
// that the grid fills the GPU a few times over, but at most `max_slices`.
struct LutPlan {
  dim3 grid;
  int64_t per_slice;
};
static int plan_lut(int64_t n, int64_t m, int64_t tile, int obs_per_block, int64_t max_slices, LutPlan& p) {
  int dev = 0, sms = 148;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int64_t obs_blocks = (m + obs_per_block - 1) / obs_per_block;
  int64_t slices = (8LL * sms + obs_blocks - 1) / obs_blocks;
  const int64_t tiles = (n + tile - 1) / tile;
  if (slices > tiles) slices = tiles;
  if (slices > max_slices) slices = max_slices;
  if (slices > 65535) slices = 65535;
  if (slices < 1) slices = 1;
  const int64_t per_slice = (n + slices - 1) / slices;
  p.per_slice = ((per_slice + tile - 1) / tile) * tile;
  p.grid = dim3((unsigned)obs_blocks, (unsigned)((n + p.per_slice - 1) / p.per_slice));
  return SPART_OK;
}

// The (cost, index) words of a single-best search, reset to "no entry": with packed_dev they are the result (a
// sharded search min-reduces them across GPUs before unpacking); otherwise they live in the workspace.
static int reset_words(void* workspace_dev, unsigned long long* packed_dev, int64_t m, cudaStream_t st,
                       unsigned long long*& best) {
  best = packed_dev ? packed_dev : (unsigned long long*)workspace_dev;
  CUDA_TRY(cudaMemsetAsync(best, 0xff, sizeof(unsigned long long) * m, st));
  return SPART_OK;
}

// spart_lut_topk: observations per block by k; the heaps take [k][block] words of shared memory, at most
// kLutTopkHeapBytes (k = 32 with 256 observations, k = 128 with 64).  At k = 32, 256 observations per block measured
// 0.80x the pairs/s of spart_lut_nearest against 0.59x with 128 (2 entries per unrolled step).  The slice count is
// capped at what plan_lut gives on a 148-SM GPU, which makes the workspace ([slices][m][k] words) a function of
// (n, m, k) alone.
constexpr int kLutTopkHeapBytes = 65536;
static int topk_obs_per_block(int32_t k) { return k <= 32 ? 256 : 64; }
static int64_t topk_slices(int64_t n, int64_t m, int32_t k) {
  const int64_t obs_blocks = (m + topk_obs_per_block(k) - 1) / topk_obs_per_block(k);
  int64_t slices = (8LL * 148 + obs_blocks - 1) / obs_blocks;
  const int64_t tiles = (n + kLutTile - 1) / kLutTile;
  if (slices > tiles) slices = tiles;
  return slices < 1 ? 1 : slices;
}

// spart_lut_topk_merge: warps per block so that the heads and cursors ([warps][L] words + bytes) fit 48 KB
constexpr int kLutMergeMaxLists = 4096;
static int merge_warps(int64_t L) {
  const int64_t w = 49152 / (9 * L);
  return w > 8 ? 8 : (w < 1 ? 1 : (int)w);
}
static int launch_topk_merge(const unsigned long long* lists, int64_t L, int64_t m, int32_t k, int64_t* idx,
                             float* cost, unsigned long long* packed, cudaStream_t st) {
  const int warps = merge_warps(L);
  return launch(lut_topk_merge_kernel, (unsigned)((m + warps - 1) / warps), 32 * warps, (size_t)(9 * L * warps), st,
                lists, (int)L, m, (int)k, idx, cost, packed);
}

extern "C" {

int spart_lut_nearest(const float* lut_dev, int64_t n, int32_t n_bands, const float* obs_dev, int64_t m,
                      const float* weights_dev, int64_t index_offset, void* workspace_dev, int64_t* best_index_dev,
                      float* best_cost_dev, unsigned long long* packed_dev, void* stream) {
  int rc = check_lut("spart_lut_nearest", 32, 1, lut_dev, n, n_bands, obs_dev, m, index_offset, workspace_dev,
                     best_index_dev, best_cost_dev, packed_dev);
  if (rc || m == 0) return rc;
  NvtxRange r("spart::lut_nearest");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* best = nullptr;
  LutPlan p;
  rc = reset_words(workspace_dev, packed_dev, m, st, best);
  if (!rc) rc = plan_lut(n, m, kLutTile, kLutObs, 65535, p);
  if (rc) return rc;
  // one instance per group of four bands
  decltype(&lut_nearest_kernel<1>) const kernels[] = {lut_nearest_kernel<1>, lut_nearest_kernel<2>,
                                                      lut_nearest_kernel<3>, lut_nearest_kernel<4>,
                                                      lut_nearest_kernel<5>, lut_nearest_kernel<6>,
                                                      lut_nearest_kernel<7>, lut_nearest_kernel<8>};
  rc = launch(kernels[(n_bands + 3) / 4 - 1], p.grid, kLutObs, 0, st, lut_dev, n, n_bands, obs_dev, m, weights_dev,
              p.per_slice, (unsigned)index_offset, best);
  if (rc || packed_dev) return rc;
  return launch(lut_unpack_kernel, (unsigned)((m + 255) / 256), 256, 0, st, best, m, best_index_dev, best_cost_dev);
}

int spart_lut_nearest_tc(const float* lut_dev, int64_t n, int32_t n_bands, const float* obs_dev, int64_t m,
                         const float* weights_dev, int64_t index_offset, void* workspace_dev, int64_t* best_index_dev,
                         float* best_cost_dev, unsigned long long* packed_dev, void* stream) {
  int rc = check_lut("spart_lut_nearest_tc", 30, 1, lut_dev, n, n_bands, obs_dev, m, index_offset, workspace_dev,
                     best_index_dev, best_cost_dev, packed_dev);
  if (rc || m == 0) return rc;
  NvtxRange r("spart::lut_nearest_tc");
  cudaStream_t st = (cudaStream_t)stream;
  const int ks = (n_bands + 2 + 7) / 8;                 // bands + the two |l|^2 slots, in k-steps of 8
  unsigned long long* best = nullptr;
  LutPlan p;
  rc = reset_words(workspace_dev, packed_dev, m, st, best);
  if (!rc) rc = plan_lut(n, m, kTcTile, kTcWarps * 16 * (ks <= 2 ? 4 : 2), 65535, p);
  if (rc) return rc;
  const unsigned off = (unsigned)index_offset;
  const auto kernel = ks <= 2 ? lut_nearest_tc_kernel<2, 4> : ks == 3 ? lut_nearest_tc_kernel<3, 2>
                                                                   : lut_nearest_tc_kernel<4, 2>;
  rc = launch(kernel, p.grid, kTcWarps * 32, 0, st, lut_dev, n, n_bands, obs_dev, m, weights_dev, p.per_slice, off,
              best);
  if (rc) return rc;
  rc = launch(lut_refine_kernel, (unsigned)((m + 255) / 256), 256, 0, st, lut_dev, n_bands, obs_dev, m, weights_dev,
              off, best);
  if (rc || packed_dev) return rc;
  return launch(lut_unpack_kernel, (unsigned)((m + 255) / 256), 256, 0, st, best, m, best_index_dev, best_cost_dev);
}

int spart_lut_unpack(const unsigned long long* packed_dev, int64_t m, int64_t* best_index_dev, float* best_cost_dev,
                     void* stream) {
  if (!packed_dev || !best_index_dev || !best_cost_dev || m < 0)
    return fail(SPART_EINVAL, "spart_lut_unpack: bad argument%s");
  if (m == 0) return SPART_OK;
  return launch(lut_unpack_kernel, (unsigned)((m + 255) / 256), 256, 0, (cudaStream_t)stream, packed_dev, m,
                best_index_dev, best_cost_dev);
}

size_t spart_lut_topk_workspace_bytes(int64_t n, int64_t m, int32_t k) {
  if (n <= 0 || m <= 0 || k < 1 || k > kLutTopkMax) return 0;
  return sizeof(unsigned long long) * (size_t)topk_slices(n, m, k) * (size_t)m * (size_t)k;
}

int spart_lut_topk(const float* lut_dev, int64_t n, int32_t n_bands, const float* obs_dev, int64_t m, int32_t k,
                   const float* weights_dev, int64_t index_offset, void* workspace_dev, int64_t* best_index_dev,
                   float* best_cost_dev, unsigned long long* packed_dev, void* stream) {
  int rc = check_lut("spart_lut_topk", 32, k, lut_dev, n, n_bands, obs_dev, m, index_offset, workspace_dev,
                     best_index_dev, best_cost_dev, packed_dev);
  if (rc || m == 0) return rc;
  NvtxRange r("spart::lut_topk");
  cudaStream_t st = (cudaStream_t)stream;
  const int obs_per_block = topk_obs_per_block(k);
  LutPlan p;
  rc = plan_lut(n, m, kLutTile, obs_per_block, topk_slices(n, m, k), p);
  if (rc) return rc;
  decltype(&lut_topk_kernel<1>) const kernels[] = {lut_topk_kernel<1>, lut_topk_kernel<2>, lut_topk_kernel<3>,
                                                   lut_topk_kernel<4>, lut_topk_kernel<5>, lut_topk_kernel<6>,
                                                   lut_topk_kernel<7>, lut_topk_kernel<8>};
  const auto kernel = kernels[(n_bands + 3) / 4 - 1];
  const size_t heap_bytes = sizeof(unsigned long long) * (size_t)k * obs_per_block;
  // the cap is per kernel and device: every call sets the same bound, so calls with different k on other host
  // threads never lower it under each other
  CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLutTopkHeapBytes));
  unsigned long long* lists = (unsigned long long*)workspace_dev;
  rc = launch(kernel, p.grid, obs_per_block, heap_bytes, st, lut_dev, n, n_bands, obs_dev, m, weights_dev,
              p.per_slice, (unsigned)index_offset, (int)k, lists);
  if (rc) return rc;
  return launch_topk_merge(lists, p.grid.y, m, k, packed_dev ? nullptr : best_index_dev,
                           packed_dev ? nullptr : best_cost_dev, packed_dev, st);
}

int spart_lut_topk_merge(const unsigned long long* lists_dev, int64_t n_lists, int64_t m, int32_t k,
                         int64_t* best_index_dev, float* best_cost_dev, unsigned long long* packed_dev, void* stream) {
  if ((!lists_dev && m > 0) || (!packed_dev && (!best_index_dev || !best_cost_dev)))
    return fail(SPART_EINVAL, "spart_lut_topk_merge: need lists_dev and best_index_dev + best_cost_dev or packed_dev%s");
  if (n_lists < 1 || n_lists > kLutMergeMaxLists || m < 0 || k < 1 || k > kLutTopkMax) {
    snprintf(g_err, sizeof(g_err), "spart_lut_topk_merge: need 1 <= n_lists <= %d, m >= 0, 1 <= k <= %d",
             kLutMergeMaxLists, kLutTopkMax);
    return SPART_EINVAL;
  }
  if (m == 0) return SPART_OK;
  return launch_topk_merge(lists_dev, n_lists, m, k, packed_dev ? nullptr : best_index_dev,
                           packed_dev ? nullptr : best_cost_dev, packed_dev, (cudaStream_t)stream);
}

int spart_lut_moments_accumulate(const void* params_dev, int32_t n_params, int64_t stride_param, int64_t stride_entry,
                                 int32_t flags, int64_t index_offset, int64_t n_local, const int64_t* index_dev,
                                 int64_t m, int32_t k, const double* centre_dev, double* acc_dev, void* stream) {
  if ((!params_dev && n_local > 0) || ((!index_dev || !acc_dev) && m > 0))
    return fail(SPART_EINVAL, "spart_lut_moments_accumulate: null argument%s");
  if (n_params < 1 || stride_param < 0 || stride_entry < 0 || (flags & ~SPART_FLAG_F32_IO) || index_offset < 0 ||
      n_local < 0 || index_offset + n_local > 0xffffffffLL || m < 0 || k < 1) {
    return fail(SPART_EINVAL, "spart_lut_moments_accumulate: need n_params >= 1, strides >= 0, flags 0 or "
                              "SPART_FLAG_F32_IO, index_offset, n_local >= 0, index_offset + n_local < 2^32, m >= 0, "
                              "k >= 1%s");
  }
  if (m == 0) return SPART_OK;
  const unsigned blocks = (unsigned)((m * (n_params + 1) + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & SPART_FLAG_F32_IO)
    return launch(lut_moments_kernel<float>, blocks, 256, 0, st, (const float*)params_dev, (int)n_params,
                  stride_param, stride_entry, index_offset, n_local, index_dev, m, (int)k, centre_dev, acc_dev);
  return launch(lut_moments_kernel<double>, blocks, 256, 0, st, (const double*)params_dev, (int)n_params,
                stride_param, stride_entry, index_offset, n_local, index_dev, m, (int)k, centre_dev, acc_dev);
}

int spart_lut_moments_finish(const double* sum_dev, const double* sq_dev, int64_t m, int32_t n_params,
                             double* mean_dev, double* std_dev, int64_t* count_dev, void* stream) {
  if ((!sum_dev || !mean_dev || !count_dev || (sq_dev && !std_dev)) && m > 0)
    return fail(SPART_EINVAL, "spart_lut_moments_finish: null argument%s");
  if (m < 0 || n_params < 1) return fail(SPART_EINVAL, "spart_lut_moments_finish: need m >= 0, n_params >= 1%s");
  if (m == 0) return SPART_OK;
  return launch(lut_moments_finish_kernel, (unsigned)((m * (n_params + 1) + 255) / 256), 256, 0, (cudaStream_t)stream,
                sum_dev, sq_dev, m, (int)n_params, mean_dev, std_dev, count_dev);
}

int spart_set_lidf(const double* lidf_dev, int64_t n, void* workspace_dev, void* stream) {
  if (!lidf_dev || (!workspace_dev && n > 0)) return fail(SPART_EINVAL, "spart_set_lidf: null argument%s");
  if (n < 0) return fail(SPART_EINVAL, "spart_set_lidf: n < 0%s");
  if (n == 0) return SPART_OK;
  return launch(lidf_store_kernel, (unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream, lidf_dev, n,
                (double*)workspace_dev);
}

int spart_leafangles(const double* ab_dev, int64_t n, int64_t ld, double* out_dev, void* stream) {
  if (!ab_dev || !out_dev) return fail(SPART_EINVAL, "spart_leafangles: null argument%s");
  if (n < 0 || ld < n) return fail(SPART_EINVAL, "spart_leafangles: need 0 <= n <= ld%s");
  if (n == 0) return SPART_OK;
  {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    int rc = init_device_constants(dev);
    if (rc) return rc;
  }
  NvtxRange r("spart::leaf_angles");
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = launch(lidf_kernel, (unsigned)((n + kL2Samples - 1) / kL2Samples), kL2Threads, 0, st, ab_dev,
                        ab_dev + ld, 1, 1, n, out_dev, 1, 13);
  if (rc) return rc;
  return launch(lidf_diff_kernel, (unsigned)((n + 255) / 256), 256, 0, st, out_dev, n);
}

}  // extern "C"

// ---- sensitivity analysis -----------------------------------------------------------------
static uint64_t splitmix64(uint64_t& state) {
  uint64_t z = (state += 0x9e3779b97f4a7c15ull);
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

// Dimension `dim` draws words 32 dim .. 32 dim + 31 of the SplitMix64 stream of `seed`: 31 for the strictly-lower
// rows of L, one for the shift, so its scramble does not depend on how many dimensions a call uses.
static void sobol_scramble(uint64_t seed, int dim, unsigned (&v)[32], unsigned& shift) {
  uint64_t state = seed + 32ull * (uint64_t)dim * 0x9e3779b97f4a7c15ull;
  unsigned row[32];                   // row r of L (r = 0: most significant bit) as a mask over the input bits
  row[0] = 1u << 31;
  for (int r = 1; r < 32; ++r)
    row[r] = ((unsigned)(splitmix64(state) & ((1ull << r) - 1)) << (32 - r)) | (1u << (31 - r));
  shift = (unsigned)splitmix64(state);
  for (int j = 0; j < 32; ++j) {
    unsigned out = 0;
    for (int r = 0; r < 32; ++r) out |= (unsigned)(__builtin_popcount(row[r] & v[j]) & 1) << (31 - r);
    v[j] = out;
  }
}

extern "C" {

int spart_sobol_design(const int32_t* rows, const double* lo, const double* hi, int32_t n_vary, uint64_t seed,
                       int32_t scramble, int64_t first, int64_t count, int32_t saltelli, double* params_dev,
                       int64_t ld, void* stream) {
  if (!rows || !lo || !hi || (!params_dev && count > 0))
    return fail(SPART_EINVAL, "spart_sobol_design: null argument%s");
  if (n_vary < 1 || n_vary > kSobolMaxVary || (scramble != 0 && scramble != 1) || (saltelli != 0 && saltelli != 1))
    return fail(SPART_EINVAL, "spart_sobol_design: need 1 <= n_vary <= 27, scramble and saltelli 0 or 1%s");
  if (first < 0 || count < 0 || first > (1ll << 32) || count > (1ll << 32) - first)
    return fail(SPART_EINVAL, "spart_sobol_design: need first, count >= 0 and first + count <= 2^32%s");
  if (ld < (saltelli ? (int64_t)(n_vary + 2) * count : count))
    return fail(SPART_EINVAL, "spart_sobol_design: ld is below the number of samples written%s");
  SobolDesignArgs a;
  unsigned used = 0;
  for (int p = 0; p < n_vary; ++p) {
    if (rows[p] < 0 || rows[p] >= SPART_NPAR || (used >> rows[p] & 1u))
      return fail(SPART_EINVAL, "spart_sobol_design: rows must be distinct values in 0..26%s");
    used |= 1u << rows[p];
    if (!(std::isfinite(lo[p]) && std::isfinite(hi[p]) && lo[p] < hi[p]))
      return fail(SPART_EINVAL, "spart_sobol_design: need finite lo < hi%s");
    a.row[p] = rows[p];
    a.lo[p] = lo[p];
    a.hi[p] = hi[p];
  }
  if (count == 0) return SPART_OK;
  for (int d = 0; d < (saltelli ? 2 : 1) * n_vary; ++d) {
    memcpy(a.v[d], SPART_SOBOL_V[d], sizeof(a.v[d]));
    a.shift[d] = 0;
    if (scramble) sobol_scramble(seed, d, a.v[d], a.shift[d]);
  }
  NvtxRange r("spart::sobol_design");
  const dim3 grid((unsigned)((count + kSobolThreads - 1) / kSobolThreads), (unsigned)n_vary);
  return launch(sobol_design_kernel, grid, kSobolThreads, 0, (cudaStream_t)stream, a, (int)n_vary, first, count,
                (int)saltelli, params_dev, ld);
}

size_t spart_sobol_acc_elems(int32_t n_out, int32_t n_vary) {
  if (n_out < 1 || n_vary < 1 || n_vary > kSobolMaxVary) return 0;
  return (size_t)kSobolSlices * (size_t)(n_vary + 1) * (size_t)n_out * kSobolSums;
}

int spart_sobol_accumulate(const double* f_dev, int64_t n, int32_t n_out, int32_t n_vary, const double* ref_dev,
                           double* acc_dev, void* stream) {
  if ((!f_dev && n > 0) || !ref_dev || !acc_dev) return fail(SPART_EINVAL, "spart_sobol_accumulate: null argument%s");
  if (n < 0 || n_out < 1 || n_vary < 1 || n_vary > kSobolMaxVary)
    return fail(SPART_EINVAL, "spart_sobol_accumulate: need n >= 0, n_out >= 1, 1 <= n_vary <= 27%s");
  if (n == 0) return SPART_OK;
  NvtxRange r("spart::sobol_accumulate");
  return launch(sobol_accumulate_kernel, dim3((unsigned)(n_vary + 1), kSobolSlices), kSobolThreads, 0,
                (cudaStream_t)stream, f_dev, n, (int)n_out, (int)n_vary, ref_dev, acc_dev);
}

int spart_sobol_finish(const double* acc_dev, const double* ref_dev, int64_t n_total, int32_t n_out, int32_t n_vary,
                       double* mean_dev, double* var_dev, double* first_dev, double* total_dev, double* first_se_dev,
                       double* total_se_dev, void* stream) {
  if (!acc_dev || !ref_dev || !mean_dev || !var_dev || !first_dev || !total_dev || !first_se_dev || !total_se_dev)
    return fail(SPART_EINVAL, "spart_sobol_finish: null argument%s");
  if (n_total < 1 || n_out < 1 || n_vary < 1 || n_vary > kSobolMaxVary)
    return fail(SPART_EINVAL, "spart_sobol_finish: need n_total >= 1, n_out >= 1, 1 <= n_vary <= 27%s");
  const int64_t threads = (int64_t)n_out * n_vary;
  return launch(sobol_finish_kernel, (unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream, acc_dev, ref_dev,
                n_total, (int)n_out, (int)n_vary, mean_dev, var_dev, first_dev, total_dev, first_se_dev, total_se_dev);
}

}  // extern "C"

// ---- retrieval by bounded Levenberg-Marquardt ------------------------------------------------
// Checks the box of the varied parameters (lo, hi may be NULL: then only n_vary is checked) and fills `a`.
static int invert_args(const char* who, const int32_t* rows, const double* lo, const double* hi, int32_t n_vary,
                       int32_t n_starts, InvertArgs& a) {
  if (n_vary < 1 || n_vary > kInvMaxVary) return fail(SPART_EINVAL, "%s: need 1 <= n_vary <= 16", who);
  if (n_starts < 1) return fail(SPART_EINVAL, "%s: need n_starts >= 1", who);
  if (!lo || !hi) return fail(SPART_EINVAL, "%s: null argument", who);
  a = InvertArgs{};
  a.n_vary = n_vary;
  a.n_starts = n_starts;
  unsigned used = 0;
  for (int p = 0; p < n_vary; ++p) {
    if (rows) {
      if (rows[p] < 0 || rows[p] >= SPART_NPAR || (used >> rows[p] & 1u))
        return fail(SPART_EINVAL, "%s: rows must be distinct values in 0..26", who);
      used |= 1u << rows[p];
      a.row[p] = rows[p];
    }
    if (!(std::isfinite(lo[p]) && std::isfinite(hi[p]) && lo[p] < hi[p]))
      return fail(SPART_EINVAL, "%s: need finite lo < hi", who);
    a.lo[p] = lo[p];
    a.hi[p] = hi[p];
  }
  return SPART_OK;
}

extern "C" {

size_t spart_invert_state_rows(int32_t n_vary) {
  return (n_vary < 1 || n_vary > kInvMaxVary) ? 0 : (size_t)inv_rows(n_vary);
}

int spart_invert_design(const int32_t* rows, const double* lo, const double* hi, int32_t n_vary,
                        const int32_t* obs_rows, int32_t n_obs_rows, const double* obs_values_dev,
                        int64_t ld_values, const double* base, int32_t n_starts, const double* state_dev,
                        int64_t n_tracks, const int32_t* active_dev, int64_t n_active, double* params_dev,
                        int64_t ld, void* stream) {
  static const char* who = "spart_invert_design";
  if (!rows || !base || (n_obs_rows > 0 && (!obs_rows || !obs_values_dev)) ||
      (n_active > 0 && (!state_dev || !active_dev || !params_dev)))
    return fail(SPART_EINVAL, "spart_invert_design: null argument%s");
  InvertArgs a;
  if (const int rc = invert_args(who, rows, lo, hi, n_vary, n_starts, a)) return rc;
  if (n_tracks < 0 || n_active < 0 || n_active > n_tracks || n_tracks * (n_vary + 1) > INT32_MAX)
    return fail(SPART_EINVAL, "spart_invert_design: need 0 <= n_active <= n_tracks and n_tracks (n_vary + 1) < 2^31%s");
  if (ld < n_active * (n_vary + 1) || (n_active > 0 && ld < 1))
    return fail(SPART_EINVAL, "spart_invert_design: ld is below the number of samples written%s");
  if (n_obs_rows < 0 || n_obs_rows > SPART_NPAR - n_vary || (n_obs_rows > 0 && ld_values < n_tracks / n_starts))
    return fail(SPART_EINVAL, "spart_invert_design: need 0 <= n_obs_rows <= 27 - n_vary and ld_values >= "
                              "n_tracks / n_starts%s");
  unsigned used = 0;
  for (int p = 0; p < n_vary; ++p) used |= 1u << rows[p];
  for (int k = 0; k < n_obs_rows; ++k) {
    if (obs_rows[k] < 0 || obs_rows[k] >= SPART_NPAR || (used >> obs_rows[k] & 1u))
      return fail(SPART_EINVAL, "spart_invert_design: obs_rows must be distinct rows in 0..26 that are not varied%s");
    used |= 1u << obs_rows[k];
    a.obs_row[k] = obs_rows[k];
  }
  a.n_obs_rows = n_obs_rows;
  for (int r = 0; r < SPART_NPAR; ++r) {
    a.base[r] = base[r];
    if (!(used >> r & 1u)) a.bcast_row[a.n_bcast++] = r;
  }
  if (n_active == 0) return SPART_OK;
  NvtxRange r("spart::invert_design");
  const int64_t n = n_active * (n_vary + 1);
  return launch(invert_design_kernel, (unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream, a, obs_values_dev,
                ld_values, state_dev, n_tracks, active_dev, n_active, params_dev, ld);
}

int spart_invert_step(const double* lo, const double* hi, int32_t n_vary, int32_t n_starts, const double* f_dev,
                      int32_t n_bands, int32_t column, const double* obs_dev, const double* weights_dev, double ftol,
                      double xtol, int32_t max_iter, double* state_dev, int64_t n_tracks, const int32_t* active_dev,
                      int64_t n_active, void* stream) {
  static const char* who = "spart_invert_step";
  if (n_active > 0 && (!f_dev || !obs_dev || !state_dev || !active_dev))
    return fail(SPART_EINVAL, "spart_invert_step: null argument%s");
  InvertArgs a;
  if (const int rc = invert_args(who, nullptr, lo, hi, n_vary, n_starts, a)) return rc;
  if (n_tracks < 0 || n_active < 0 || n_active > n_tracks || n_tracks > INT32_MAX)
    return fail(SPART_EINVAL, "spart_invert_step: need 0 <= n_active <= n_tracks < 2^31%s");
  if (n_bands < 1 || column < 0 || column >= SPART_NOUT || max_iter < 1)
    return fail(SPART_EINVAL, "spart_invert_step: need n_bands >= 1, column 0..2 and max_iter >= 1%s");
  if (!(ftol >= 0.0 && xtol >= 0.0 && std::isfinite(ftol) && std::isfinite(xtol)))
    return fail(SPART_EINVAL, "spart_invert_step: need finite ftol, xtol >= 0%s");
  if (n_active == 0) return SPART_OK;
  NvtxRange r("spart::invert_step");
  return launch(invert_step_kernel, (unsigned)((n_active + kInvThreads - 1) / kInvThreads), kInvThreads,
                sizeof(double) * kInvThreads * inv_shared(n_vary), (cudaStream_t)stream, a, f_dev, (int)n_bands,
                (int)column, obs_dev, weights_dev, ftol, xtol, (int)max_iter, state_dev, n_tracks, active_dev,
                n_active);
}

int spart_invert_finish(const double* lo, const double* hi, int32_t n_vary, int32_t n_starts, int32_t n_bands,
                        int32_t absolute_sigma, const double* state_dev, int64_t n_obs, double* x_dev,
                        double* cost_dev, double* std_dev, int32_t* status_dev, int32_t* start_dev,
                        int32_t* iterations_dev, int64_t* n_forward_dev, void* stream) {
  static const char* who = "spart_invert_finish";
  if (n_obs > 0 && (!state_dev || !x_dev || !cost_dev || !std_dev || !status_dev || !start_dev || !iterations_dev ||
                    !n_forward_dev))
    return fail(SPART_EINVAL, "spart_invert_finish: null argument%s");
  InvertArgs a;
  if (const int rc = invert_args(who, nullptr, lo, hi, n_vary, n_starts, a)) return rc;
  if (n_obs < 0 || n_obs * n_starts > INT32_MAX || n_bands < 1 || (absolute_sigma != 0 && absolute_sigma != 1))
    return fail(SPART_EINVAL, "spart_invert_finish: need 0 <= n_obs n_starts < 2^31, n_bands >= 1 and "
                              "absolute_sigma 0 or 1%s");
  if (n_obs == 0) return SPART_OK;
  NvtxRange r("spart::invert_finish");
  return launch(invert_finish_kernel, (unsigned)((n_obs + kInvThreads - 1) / kInvThreads), kInvThreads,
                sizeof(double) * kInvThreads * inv_shared(n_vary), (cudaStream_t)stream, a, (int)n_bands,
                (int)absolute_sigma, state_dev, n_obs, x_dev, cost_dev, std_dev, status_dev, start_dev,
                iterations_dev, n_forward_dev);
}

}  // extern "C"

// ---- host-buffer path ---------------------------------------------------------------------
static bool is_pinned_host(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// buffers, streams and events of the host path: kInSlots parameter spans of `span` samples, kSlots record /
// output slots of `chunk` samples, pinned staging buffers for pageable caller memory
static int ensure_slots(SpartCtx* ctx, int64_t span, int64_t chunk, size_t out_bytes, bool stage_in, bool stage_out) {
  const size_t in_bytes = sizeof(double) * P_COUNT * (size_t)span;
  for (Stream* s : {&ctx->h2d_stream, &ctx->d2h_stream, &ctx->compute_stream, &ctx->join_stream}) {
    if (!*s) CUDA_TRY(create(*s));
    CUDA_TRY(cudaStreamSynchronize(s->get()));
  }
  // a buffer below its capacity field is (re)allocated; the fields are raised once every buffer has grown
  for (int i = 0; i < SpartCtx::kSlots; ++i) {
    if (!ctx->slot_done[i]) CUDA_TRY(create(ctx->slot_done[i], cudaEventDisableTiming));
    if (!ctx->slot_k[i]) CUDA_TRY(create(ctx->slot_k[i], cudaEventDisableTiming));
    if (ctx->slot_cap < chunk) CUDA_TRY(alloc(ctx->slot_rec[i], sizeof(double) * kWsRows * chunk));
    if (ctx->slot_out_cap < out_bytes) CUDA_TRY(alloc(ctx->slot_out[i], out_bytes));
    if (stage_out && ctx->stage_out_cap < out_bytes) CUDA_TRY(alloc(ctx->stage_out[i], out_bytes));
  }
  if (!ctx->bc_stage) CUDA_TRY(alloc(ctx->bc_stage, sizeof(double) * P_COUNT));
  for (int i = 0; i < SpartCtx::kInSlots; ++i) {
    if (!ctx->in_done[i]) CUDA_TRY(create(ctx->in_done[i], cudaEventDisableTiming));
    if (!ctx->in_free[i]) CUDA_TRY(create(ctx->in_free[i], cudaEventDisableTiming));
    if (!ctx->ets_done[i]) CUDA_TRY(create(ctx->ets_done[i], cudaEventDisableTiming));
    if (ctx->in_cap < span) {
      CUDA_TRY(alloc(ctx->in_params[i], in_bytes));
      CUDA_TRY(alloc(ctx->in_ets[i], sizeof(double) * (size_t)span));
    }
    if (stage_in && ctx->stage_in_cap < in_bytes) CUDA_TRY(alloc(ctx->stage_in[i], in_bytes));
  }
  if (ctx->slot_cap < chunk) ctx->slot_cap = chunk;
  if (ctx->in_cap < span) ctx->in_cap = span;
  if (ctx->slot_out_cap < out_bytes) ctx->slot_out_cap = out_bytes;
  if (stage_in && ctx->stage_in_cap < in_bytes) ctx->stage_in_cap = in_bytes;
  if (stage_out && ctx->stage_out_cap < out_bytes) ctx->stage_out_cap = out_bytes;
  if ((stage_in || stage_out) && !ctx->pool) {
    int want = 12;      // copy threads: 4 / 8 / 12 / 16 -> 60 / 85 / 98 / 94 M simulations/s from pageable arrays
    if (const char* e = getenv("SPART_HOST_THREADS")) want = atoi(e);
    const int hw = (int)std::thread::hardware_concurrency();
    if (hw > 0 && want > hw) want = hw;
    if (want < 1) want = 1;
    ctx->pool.reset(new (std::nothrow) HostPool(want - 1));
    if (!ctx->pool) return fail(SPART_ENOMEM, "spart_forward_bands_host: out of host memory%s");
  }
  return SPART_OK;
}

// memcpy of `bytes` split into ~1 MiB pieces over the pool
static void pool_memcpy(HostPool* pool, void* dst, const void* src, size_t bytes) {
  const size_t piece = (size_t)1 << 20;
  const int n = (int)((bytes + piece - 1) / piece);
  pool->parallel_for(n, [&](int i) {
    const size_t o = (size_t)i * piece;
    memcpy((char*)dst + o, (const char*)src + o, (bytes - o < piece) ? bytes - o : piece);
  });
}

extern "C" {

int spart_forward_bands_host(SpartCtx* ctx, int32_t sensor, const void* params_host, int64_t n, int64_t ld,
                             uint32_t broadcast_rows, int32_t precision, int32_t flags, void* out_host) {
  const char* who = "spart_forward_bands_host";
  if (!ctx || !params_host || !out_host) return fail(SPART_EINVAL, "%s: null argument", who);
  if (n < 0 || ld < n) return fail(SPART_EINVAL, "%s: need 0 <= n <= ld", who);
  if (broadcast_rows >> SPART_NPAR) return fail(SPART_EINVAL, "%s: broadcast_rows has bits beyond row 26", who);
  if (flags & SPART_FLAG_REUSE_RECORD) return fail(SPART_EINVAL, "%s: SPART_FLAG_REUSE_RECORD is a device-path flag", who);
  if (flags & SPART_FLAG_USER_LIDF) return fail(SPART_EINVAL, "%s: SPART_FLAG_USER_LIDF is a device-path flag", who);
  int rc = check_mode(ctx, sensor, precision, flags, who);
  if (rc) return rc;
  if (n == 0) return SPART_OK;
  std::lock_guard<std::mutex> lock(ctx->mu);
  GUARD_DEVICE(ctx->device);
  NvtxRange range("spart::forward_bands_host");
  const int nb = ctx->n_bands[sensor];
  const size_t elt = (flags & SPART_FLAG_F32_IO) ? sizeof(float) : sizeof(double);
  const bool compact = (flags & SPART_FLAG_COMPACT_OUT) != 0;
  const int nout = compact ? 2 : SPART_NOUT;
  // The pipeline has two granularities.
  //   Spans (up to 128 Ki samples) are the unit of the host->device copy: one 2-D copy per run of rows into one of
  //   kInSlots device buffers.  A host->device copy issued next to a saturated device->host stream pays ~40 us
  //   of latency per copy operation on this box, so few, large operations matter (SPART_HOST_TRACE timeline).
  //   Chunks (up to 64 Ki samples) are the unit of the kernels and of the device->host copy: a span's chunks are
  //   evaluated in place (params = span + offset, broadcast rows from the span's first elements, see ParamsT),
  //   so results start to flow back after the first chunk, not after the first span.
  // Streams: ONE per copy direction (each slot's own stream first carried its copies too: the host->device copy of
  // a later chunk then queued behind the device->host copy of an earlier one), ONE compute stream (with a stream per
  // output slot the chunks of a span share the SMs and finish together, a span's worth of kernel time after its
  // copy; on one stream they finish one after the other and results flow back sooner) and a join stream, tied
  // together by events:
  //   H2D(span j)  waits until the kernels of every chunk of span j - kInSlots have finished (join stream)
  //   kernels(i)   wait for H2D(span of i) and for D2H(i - kSlots)   (the slot's output buffer is free)
  //   D2H(i)       waits for kernels(i)
  // The first spans are small (32 Ki, 96 Ki samples) and the last chunk is split down to 16 Ki, because the first
  // H2D + kernels and the last D2H overlap with nothing.  SPART_HOST_SPAN / SPART_HOST_CHUNK override the sizes.
  int64_t span_max = 1 << 17, chunk = 1 << 16;      // best of {96, 128, 192, 256} Ki x {32, 48, 64, 128} Ki on 1M samples
  if (const char* e = getenv("SPART_HOST_SPAN")) {
    const long long v = atoll(e);
    if (v >= 1024) span_max = v;
  }
  if (const char* e = getenv("SPART_HOST_CHUNK")) {
    const long long v = atoll(e);
    if (v >= 1024) chunk = v;
  }
  const int64_t cap_by_out = ((int64_t)256 << 20) / ((int64_t)nb * SPART_NOUT * 8);   // <= ~256 MB of output per slot
  if (chunk > cap_by_out) chunk = cap_by_out > 1024 ? cap_by_out : 1024;
  chunk = (chunk / 128) * 128;
  if (span_max < chunk) span_max = chunk;
  span_max = (span_max / chunk) * chunk;
  if (chunk > n) chunk = n;
  if (span_max > n) span_max = n;
  struct Span { int64_t s0, m; };
  std::vector<Span> spans;
  {
    int64_t s0 = 0;
    for (int64_t c = (1 << 15); c < span_max && n - s0 >= 4 * c; c *= 3) {     // 32 Ki, 96 Ki
      const int64_t m = (c / 128) * 128;
      spans.push_back({s0, m});
      s0 += m;
    }
    while (s0 < n) {
      const int64_t m = (n - s0 < span_max) ? n - s0 : span_max;
      spans.push_back({s0, m});
      s0 += m;
    }
  }
  // pageable caller memory is staged through pinned buffers by the copy threads (a cudaMemcpyAsync on
  // pageable memory is a synchronous single-threaded driver copy); pinned or registered memory is
  // DMA'd directly
  const bool stage_in = !is_pinned_host(params_host), stage_out = !is_pinned_host(out_host);
  const size_t out_chunk_bytes = ((size_t)chunk * nb * nout + (compact ? (size_t)chunk : 0)) * elt;
  rc = ensure_slots(ctx, span_max, chunk, out_chunk_bytes, stage_in, stage_out);
  if (rc) return rc;
  const char* pin = (const char*)params_host;
  char* pout = (char*)out_host;
  char* pets = pout + (size_t)n * nb * 2 * elt;      // compact output: etscale[n] follows [n][nb][2]

  struct Pending { int64_t s0 = 0, m = 0; bool live = false; } pend[SpartCtx::kSlots];
  // SPART_HOST_TRACE=1 (tuning aid): CUDA events per span and per chunk, printed as a timeline when the call ends
  const bool trace = getenv("SPART_HOST_TRACE") != nullptr;
  struct TraceEv { Event e[2]; int64_t m; int slot; bool span; };
  std::vector<TraceEv> tev;
  Event trace_t0;
  if (trace) {
    create(trace_t0);
    cudaEventRecord(trace_t0.get(), ctx->h2d_stream.get());
  }
  auto trace_new = [&](int64_t m, int slot, bool span) {
    if (!trace) return;
    TraceEv t;
    for (auto& e : t.e) create(e);
    t.m = m;
    t.slot = slot;
    t.span = span;
    tev.push_back(std::move(t));
  };
  auto mark = [&](int which, cudaStream_t st) {
    if (trace) cudaEventRecord(tev.back().e[which].get(), st);
  };
  // wait for a slot's chunk and, with a pageable output, copy it from the pinned staging buffer into the
  // caller's array (the staging buffer may then be reused)
  auto unstage = [&](int slot) -> int {
    Pending& q = pend[slot];
    if (!q.live) return SPART_OK;
    q.live = false;
    CUDA_TRY(cudaEventSynchronize(ctx->slot_done[slot].get()));
    const size_t main_bytes = (size_t)q.m * nb * nout * elt;
    pool_memcpy(ctx->pool.get(), pout + (size_t)q.s0 * nb * nout * elt, ctx->stage_out[slot].get(), main_bytes);
    if (compact) memcpy(pets + (size_t)q.s0 * elt, (char*)ctx->stage_out[slot].get() + main_bytes, (size_t)q.m * elt);
    return SPART_OK;
  };
  auto run = [&]() -> int {
    cudaStream_t sin = ctx->h2d_stream.get(), sout = ctx->d2h_stream.get();
    cudaStream_t st = ctx->compute_stream.get(), sjoin = ctx->join_stream.get();
    bool in_used[SpartCtx::kInSlots] = {}, used[SpartCtx::kSlots] = {};
    int slot = 0;
    std::vector<int> fifo;       // pageable output: slots whose chunks are still to be copied out, oldest first
    // The rows of a span buffer are ctx->in_cap elements apart whatever the span's length, so the broadcast
    // elements have fixed places: they go in once per call and buffer, while the link is still idle (a tiny copy
    // issued later, next to a saturated device->host stream, costs as much as 2 MB of payload).
    const int64_t dld = ctx->in_cap;
    if (broadcast_rows) {
      for (int r = 0; r < P_COUNT; ++r)
        if ((broadcast_rows >> r) & 1u)
          memcpy((char*)ctx->bc_stage.get() + (size_t)r * elt, pin + (size_t)r * ld * elt, elt);
      for (int i = 0; i < SpartCtx::kInSlots && i < (int)spans.size(); ++i)
        for (int r0 = 0; r0 < P_COUNT;) {
          if (!((broadcast_rows >> r0) & 1u)) {
            ++r0;
            continue;
          }
          int r1 = r0 + 1;
          while (r1 < P_COUNT && ((broadcast_rows >> r1) & 1u)) ++r1;
          CUDA_TRY(cudaMemcpy2DAsync((char*)ctx->in_params[i].get() + (size_t)r0 * dld * elt, (size_t)dld * elt,
                                     (char*)ctx->bc_stage.get() + (size_t)r0 * elt, elt, elt, r1 - r0,
                                     cudaMemcpyHostToDevice, sin));
          r0 = r1;
        }
    }
    // compact result in pinned memory: the etscale values travel once per span instead of once per chunk
    const bool ets_per_span = compact && !stage_out;
    for (size_t j = 0; j < spans.size(); ++j) {
      const int islot = (int)(j % SpartCtx::kInSlots);
      const int64_t sp0 = spans[j].s0, sm = spans[j].m;
      // ---- host -> device: the span's parameter rows (ld apart on the host, sm apart on the device; a
      // broadcast row moves one element)
      const char* src = pin;
      size_t src_pitch = (size_t)ld * elt;
      size_t src_off = (size_t)sp0 * elt;
      if (stage_in) {
        // the staging buffer has been read
        if (in_used[islot]) CUDA_TRY(cudaEventSynchronize(ctx->in_done[islot].get()));
        char* stg = (char*)ctx->stage_in[islot].get();
        ctx->pool->parallel_for(P_COUNT, [&](int r) {
          if (!((broadcast_rows >> r) & 1u))
            memcpy(stg + (size_t)r * sm * elt, pin + (size_t)r * ld * elt + (size_t)sp0 * elt, (size_t)sm * elt);
        });
        src = stg;
        src_pitch = (size_t)sm * elt;
        src_off = 0;
      }
      if (in_used[islot]) CUDA_TRY(cudaStreamWaitEvent(sin, ctx->in_free[islot].get(), 0));
      trace_new(sm, islot, true);
      mark(0, sin);
      for (int r0 = 0; r0 < P_COUNT;) {     // runs of per-sample rows become one 2-D copy each
        if ((broadcast_rows >> r0) & 1u) {
          ++r0;
          continue;
        }
        int r1 = r0 + 1;
        while (r1 < P_COUNT && !((broadcast_rows >> r1) & 1u)) ++r1;
        CUDA_TRY(cudaMemcpy2DAsync((char*)ctx->in_params[islot].get() + (size_t)r0 * dld * elt, (size_t)dld * elt,
                                   src + (size_t)r0 * src_pitch + src_off, src_pitch, (size_t)sm * elt, r1 - r0,
                                   cudaMemcpyHostToDevice, sin));
        r0 = r1;
      }
      CUDA_TRY(cudaEventRecord(ctx->in_done[islot].get(), sin));
      mark(1, sin);
      in_used[islot] = true;
      // ---- the span's chunks: kernels in place, device -> host
      std::vector<int64_t> sizes;
      for (int64_t left = sm; left > 0;) {
        int64_t m = left < chunk ? left : chunk;
        if (j + 1 == spans.size() && left <= chunk && m >= (1 << 15)) m = ((m / 2 + 127) / 128) * 128;   // tail: halve
        sizes.push_back(m);
        left -= m;
      }
      int64_t off = 0;
      for (size_t ci = 0; ci < sizes.size(); off += sizes[ci], ++ci, slot = (slot + 1) % SpartCtx::kSlots) {
        const int64_t m = sizes[ci], s0 = sp0 + off;
        int rc2 = unstage(slot);      // pageable output: the slot's previous chunk leaves its staging buffer
        if (rc2) return rc2;
        trace_new(m, slot, false);
        CUDA_TRY(cudaStreamWaitEvent(st, ctx->in_done[islot].get(), 0));
        if (used[slot]) CUDA_TRY(cudaStreamWaitEvent(st, ctx->slot_done[slot].get(), 0));
        if (ets_per_span && ci == 0 && j >= (size_t)SpartCtx::kInSlots)
          CUDA_TRY(cudaStreamWaitEvent(st, ctx->ets_done[islot].get(), 0));   // the span buffer's etscale array is free
        rc2 = forward_bands_impl(ctx, sensor, (const char*)ctx->in_params[islot].get() + (size_t)off * elt,
                                 ctx->in_params[islot].get(), m, dld, broadcast_rows, precision, flags,
                                 ctx->slot_rec[slot].get(), ctx->slot_out[slot].get(), st);
        if (rc2) return rc2;
        const size_t main_bytes = (size_t)m * nb * nout * elt;
        if (ets_per_span)
          CUDA_TRY(cudaMemcpyAsync((char*)ctx->in_ets[islot].get() + (size_t)off * elt,
                                   (char*)ctx->slot_out[slot].get() + main_bytes, (size_t)m * elt,
                                   cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(cudaEventRecord(ctx->slot_k[slot].get(), st));
        mark(0, st);
        CUDA_TRY(cudaStreamWaitEvent(sjoin, ctx->slot_k[slot].get(), 0));
        CUDA_TRY(cudaStreamWaitEvent(sout, ctx->slot_k[slot].get(), 0));
        if (stage_out) {
          CUDA_TRY(cudaMemcpyAsync(ctx->stage_out[slot].get(), ctx->slot_out[slot].get(),
                                   main_bytes + (compact ? m * elt : 0), cudaMemcpyDeviceToHost, sout));
        } else {
          CUDA_TRY(cudaMemcpyAsync(pout + (size_t)s0 * nb * nout * elt, ctx->slot_out[slot].get(), main_bytes,
                                   cudaMemcpyDeviceToHost, sout));
        }
        CUDA_TRY(cudaEventRecord(ctx->slot_done[slot].get(), sout));
        mark(1, sout);
        used[slot] = true;
        if (stage_out) {
          pend[slot].s0 = s0;
          pend[slot].m = m;
          pend[slot].live = true;
          // copy finished chunks out of their staging buffers while the newer ones are on the GPU: two chunks stay
          // in flight behind the one just enqueued (waiting for the newest would drain the pipeline)
          fifo.push_back(slot);
          while (fifo.size() > 2) {
            rc2 = unstage(fifo.front());
            fifo.erase(fifo.begin());
            if (rc2) return rc2;
          }
        }
      }
      CUDA_TRY(cudaEventRecord(ctx->in_free[islot].get(), sjoin));    // every chunk of this span has been evaluated
      if (ets_per_span) {          // (the d2h stream has already waited for the kernels of all chunks of the span)
        CUDA_TRY(cudaMemcpyAsync(pets + (size_t)sp0 * elt, ctx->in_ets[islot].get(), (size_t)sm * elt,
                                 cudaMemcpyDeviceToHost, sout));
        CUDA_TRY(cudaEventRecord(ctx->ets_done[islot].get(), sout));
      }
    }
    for (int i = 0; i < SpartCtx::kSlots; ++i) {
      const int rc2 = unstage(i);
      if (rc2) return rc2;
    }
    return SPART_OK;
  };
  rc = run();
  // on success and on failure alike: nothing of this call may still be in flight (the copy streams read and
  // write the caller's memory) when it returns
  for (const Stream* sy : {&ctx->compute_stream, &ctx->h2d_stream, &ctx->d2h_stream, &ctx->join_stream}) {
    const cudaError_t e = cudaStreamSynchronize(sy->get());
    if (e != cudaSuccess && rc == SPART_OK) {
      snprintf(g_err, sizeof(g_err), "cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
      rc = (int)e;
    }
  }
  if (trace) {
    fprintf(stderr, "spart_forward_bands_host trace [ms from the first enqueue]\n"
                    "  span  <samples> <buffer> | H2D start .. end\n  chunk <samples> <slot>   | kernels end | D2H end\n");
    for (size_t i = 0; i < tev.size(); ++i) {
      float t[2] = {0, 0};
      for (int k = 0; k < 2; ++k) cudaEventElapsedTime(&t[k], trace_t0.get(), tev[i].e[k].get());
      if (tev[i].span)
        fprintf(stderr, "  span  %7lld %d | %7.3f .. %7.3f\n", (long long)tev[i].m, tev[i].slot, t[0], t[1]);
      else
        fprintf(stderr, "  chunk %7lld %d |            %7.3f | %7.3f\n", (long long)tev[i].m, tev[i].slot, t[0], t[1]);
    }
  }
  return rc;
}

int spart_measure_peaks(int32_t device, double* fp64_tflops, double* fp32_tflops) {
  if (!fp64_tflops || !fp32_tflops) return fail(SPART_EINVAL, "spart_measure_peaks: null argument%s");
  const int ndev = spart_device_count();
  if (ndev <= 0) return fail(SPART_ENODEV, "spart_measure_peaks: no CUDA device%s");
  if (device < 0 || device >= ndev) return fail(SPART_EINVAL, "spart_measure_peaks: device index out of range%s");
  GUARD_DEVICE(device);
  int sm = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device));
  int rc = time_fma<double>(sm, fp64_tflops);
  if (rc) return rc;
  return time_fma<float>(sm, fp32_tflops);
}

int spart_measure_fp64_chain(int32_t device, double* tflops) {
  if (!tflops) return fail(SPART_EINVAL, "spart_measure_fp64_chain: null argument%s");
  const int ndev = spart_device_count();
  if (ndev <= 0) return fail(SPART_ENODEV, "spart_measure_fp64_chain: no CUDA device%s");
  if (device < 0 || device >= ndev) return fail(SPART_EINVAL, "spart_measure_fp64_chain: device index out of range%s");
  GUARD_DEVICE(device);
  int sm = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device));
  const int iters = 1 << 12, threads = 1024, blocks = sm;     // 8 warps per scheduler
  return time_peak(2.0 * 6.0 * 4.0 * (double)iters * threads * (double)blocks, tflops, [&](double* d) {
    return launch(fp64_register_chain_kernel, blocks, threads, 0, nullptr, d, iters);
  });
}

}  // extern "C"
