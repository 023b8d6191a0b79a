// batotp_cuda.cu — extern "C" boundary (include/batotp_cuda.h) and the chunk pipeline that
// strings the kernels of k_input.cuh / k_sweep.cuh / k_output.cuh together.
//
// Build (product):  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -lineinfo
//                   -shared -Xcompiler -fPIC  -> batotp_b200/lib/libbatotp_cuda.so
// There is no CPU fallback in that library.  The same file compiles with g++ and
// -DBATOTP_HOST_EMU into a TEST-ONLY emulation library (see emu.h) used by the CPU CI.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/batotp_cuda.h"
#include "k_output.cuh"
#include "k_sweep.cuh"
#include "k_sweep_group.cuh"
#include "k_mvc.cuh"

#ifndef BATOTP_HOST_EMU
#include <cuda_runtime.h>
#else
thread_local emu_dim3 threadIdx, blockIdx, blockDim, gridDim;
thread_local EmuCta *emu_cta = nullptr;
#endif

// ----------------------------------------------------------------------------- runtime shims
namespace {

struct Err {
  std::string msg;
  bool oom = false;  // a device allocation failed (or would fail): the batch call retries with smaller chunks
  int fitB = 0;      // with oom: how many trajectories per chunk the free memory would hold (0 = unknown)
  bool planned = false;  // with oom: refused by the planner before anything was freed or allocated (workspaces intact)
};

#ifndef BATOTP_HOST_EMU
#define CU_CHECK(call)                                                                      \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess) {                                                                \
      char buf_[512];                                                                       \
      snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
               __FILE__, __LINE__);                                                         \
      throw Err{buf_};                                                                      \
    }                                                                                       \
  } while (0)
// tuning aid: BATOTP_TRACE=1 prints the chunk decisions of a batch call, the planner's refusals and the time spent in
// cudaMalloc / cudaFree to stderr
inline bool g_trace() {
  static const bool on = getenv("BATOTP_TRACE") != nullptr;
  return on;
}
inline double g_now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static double g_allocMs = 0, g_freeMs = 0;
inline void *g_alloc(size_t bytes) {
  void *p = nullptr;
  const double t0 = g_trace() ? g_now_ms() : 0;
  const cudaError_t e = cudaMalloc(&p, bytes ? bytes : 8);
  if (g_trace()) g_allocMs += g_now_ms() - t0;
  if (e != cudaSuccess) {
    cudaGetLastError();  // not sticky: clear it
    char buf[256];
    snprintf(buf, sizeof buf, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    Err er{buf};
    er.oom = (e == cudaErrorMemoryAllocation);
    throw er;
  }
  return p;
}
inline void g_free(void *p) {
  const double t0 = g_trace() ? g_now_ms() : 0;
  if (p) cudaFree(p);
  if (g_trace()) g_freeMs += g_now_ms() - t0;
}
inline void g_zero(void *p, size_t bytes, cudaStream_t s) { CU_CHECK(cudaMemsetAsync(p, 0, bytes, s)); }
inline void g_h2d(void *d, const void *h, size_t bytes, cudaStream_t s) {
  CU_CHECK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyDefault, s));
}
inline void g_d2h(void *h, const void *d, size_t bytes, cudaStream_t s) {
  CU_CHECK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDefault, s));
}
inline void g_d2d(void *d, const void *s0, size_t bytes, cudaStream_t s) {
  CU_CHECK(cudaMemcpyAsync(d, s0, bytes, cudaMemcpyDeviceToDevice, s));
}
inline void g_d2h_2d(void *h, size_t hp, const void *d, size_t dp, size_t width, size_t rows, cudaStream_t s) {
  CU_CHECK(cudaMemcpy2DAsync(h, hp, d, dp, width, rows, cudaMemcpyDefault, s));
}
inline void g_h2d_2d(void *d, size_t dp, const void *h, size_t hp, size_t width, size_t rows, cudaStream_t s) {
  CU_CHECK(cudaMemcpy2DAsync(d, dp, h, hp, width, rows, cudaMemcpyHostToDevice, s));
}
inline void g_d2d_2d(void *d, size_t dp, const void *s0, size_t sp, size_t width, size_t rows, cudaStream_t s) {
  CU_CHECK(cudaMemcpy2DAsync(d, dp, s0, sp, width, rows, cudaMemcpyDeviceToDevice, s));
}
inline void g_sync(cudaStream_t s) { CU_CHECK(cudaStreamSynchronize(s)); }
inline void g_event_record(cudaEvent_t e, cudaStream_t s) { CU_CHECK(cudaEventRecord(e, s)); }
inline void g_stream_wait(cudaStream_t s, cudaEvent_t e) { CU_CHECK(cudaStreamWaitEvent(s, e, 0)); }
inline void g_check_launch() { CU_CHECK(cudaGetLastError()); }
#else
inline bool g_trace() {
  static const bool on = getenv("BATOTP_TRACE") != nullptr;
  return on;
}
inline double g_now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static double g_allocMs = 0, g_freeMs = 0;
inline void *g_alloc(size_t bytes) { return calloc(1, bytes ? bytes : 8); }
inline void g_free(void *p) { free(p); }
inline void g_zero(void *p, size_t bytes, cudaStream_t) { memset(p, 0, bytes); }
inline void g_h2d(void *d, const void *h, size_t bytes, cudaStream_t) { memcpy(d, h, bytes); }
inline void g_d2h(void *h, const void *d, size_t bytes, cudaStream_t) { memcpy(h, d, bytes); }
inline void g_d2d(void *d, const void *s0, size_t bytes, cudaStream_t) { memmove(d, s0, bytes); }
inline void copy2d(void *d, size_t dp, const void *s0, size_t sp, size_t width, size_t rows) {
  for (size_t r = 0; r < rows; ++r) memcpy((char *)d + r * dp, (const char *)s0 + r * sp, width);
}
inline void g_d2h_2d(void *h, size_t hp, const void *d, size_t dp, size_t width, size_t rows, cudaStream_t) {
  copy2d(h, hp, d, dp, width, rows);
}
inline void g_h2d_2d(void *d, size_t dp, const void *h, size_t hp, size_t width, size_t rows, cudaStream_t) {
  copy2d(d, dp, h, hp, width, rows);
}
inline void g_d2d_2d(void *d, size_t dp, const void *s0, size_t sp, size_t width, size_t rows, cudaStream_t) {
  copy2d(d, dp, s0, sp, width, rows);
}
inline void g_sync(cudaStream_t) {}
typedef int cudaEvent_t;
inline void g_event_record(cudaEvent_t, cudaStream_t) {}
inline void g_stream_wait(cudaStream_t, cudaEvent_t) {}
inline void g_check_launch() {}
#endif

inline int cdiv(int a, int b) { return (a + b - 1) / b; }
#ifndef SWEEP_GROUP_MAX_B
#define SWEEP_GROUP_MAX_B 16384  // chunks up to this size take the group-per-trajectory sweep kernel (automatic mode) ...
#endif
#ifndef SWEEP_GROUP_MAX_B_EXACT
#define SWEEP_GROUP_MAX_B_EXACT 32768  // ... or this size when the limits need the exact verification (Cartesian / torque
                                       // rows: no float filters, so the lane kernel pays 14+ IEEE divisions per
                                       // verification and the group kernel stays ahead for longer: CSPR x19072 351 vs ~270 ms)
#endif
// bytes the device can still hand out (host emulation: "plenty")
inline size_t g_free_bytes() {
#ifndef BATOTP_HOST_EMU
  size_t fr = 0, tot = 0;
  if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) return (size_t)1 << 62;
  return fr;
#else
  // TEST-ONLY (host emulation): BATOTP_EMU_FREE_MB pretends the device has that much memory left, so that the
  // CPU suite can walk the "chunk does not fit" paths
  if (const char *e = getenv("BATOTP_EMU_FREE_MB")) return (size_t)atoll(e) << 20;
  return (size_t)1 << 62;
#endif
}

// robot.cpp:291-322 — cable attachment points of the CSPR (host, once)
Pmat make_pmat() {
  Pmat pm;
  const double cible1[3] = {1.0941, -4.9074, 2.5542};
  const double delta1[3] = {-0.765, 0.112, 3.74};
  const double cible3[3] = {0.2098, 5.3409, 2.6236};
  const double delta2[3] = {0.43, 0.125, 3.615};
  double p1[3], p2[3];
  const double p3[3] = {-5.9751, 0.1399, 6.1543};
  for (int i = 0; i < 3; ++i) {
    p1[i] = cible1[i] + delta1[i];
    p2[i] = cible3[i] + delta2[i];
  }
  const int ind[3] = {1, 0, 2};
  for (int i = 0; i < 3; ++i) {
    const int it = ind[i];
    pm.p[i][0] = -p1[it];
    pm.p[i][1] = -p2[it];
    pm.p[i][2] = -p3[it];
  }
  double cen[3];
  for (int i = 0; i < 3; ++i) cen[i] = 1 / 3.0 * (pm.p[i][0] + pm.p[i][1] + pm.p[i][2]);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) pm.p[i][j] -= cen[i];
  return pm;
}

}  // namespace

// ----------------------------------------------------------------------------- context
#define NSETS 4
// The shapes the two device workspaces are allocated for.  A shape holds every input of its array list (chunk_arrays,
// out_arrays), so a held workspace serves a request when its shape covers the request's (ws_covers, out_covers).
// B = 0 / Bo = 0: nothing held.
struct WsShape {  // chunk-resident arrays; J..trq: the configuration's rows, which also size the output arrays
  int B = 0, Nc = 0, Sc = 0, J = 0, Cin = 0, C = 0, R = 0, RT = 0;
  bool trq = false;
};
struct OutShape {  // output sub-chunk arrays (rows as in the chunk's shape: ensure_ws drops these arrays with its own)
  int Bo = 0, Sc = 0, Oc = 0, Os = 0, OutC = 0, rowP = 0, histP = 0;
  bool keepF64 = false, fused = false;
};
struct batotp_ctx {
  int device = 0;
  cudaStream_t stream = 0;
  std::string err;
  int chunk = 0;  // trajectories per resident chunk; 0 = automatic (auto_chunk)
  long launches = 0;
  DevCfg cfg;
  bool haveCfg = false;
  Ws w;
  WsShape wsHeld;
  OutShape outHeld;
  std::vector<void *> wsAllocs;   // chunk-resident arrays
  size_t wsBytes = 0, outBytes = 0;  // bytes held by wsAllocs / outAllocs
  int learnedChunk = 0;              // automatic chunking: the chunk size the last batch call of this configuration ended with
  std::vector<void *> outAllocs;  // output sub-chunk arrays
  int outChunk = 8192;            // trajectories per output pass
  // row pitch (points) of the packed float32 rows / histories: the caller's out_cap / hist_cap inside
  // batotp_cuda_optimize_batch (a sub-chunk then leaves in one contiguous copy), 0 = the device capacities
  int rowPitch = 0, histPitch = 0;
  // ragged result layout (batotp_batch_out.row_offset): the blocks of a sub-chunk are packed back to back in the
  // staging set and leave in one copy; where they go in the caller's buffer comes from a counter shared by the
  // contexts that work on one batch
  bool ragged = false;
  std::atomic<long long> *ragNext = nullptr;
  std::vector<long long> ragOffHost;  // [B + 1] prefix sums of the resident chunk's output lengths (w.ragOff on the device)
  long long ragChunkBase = 0;         // where the chunk's blocks start in the caller's buffers
  long long ragBase[NSETS] = {}, ragTotal[NSETS] = {};
  int curSet = 0;
  int maxSteps = 65536;           // largest RK-step capacity the automatic retries grow to (per sweep)
  // cfg.dyn_source = 1: the caller's point function for a1..a4 (Robot::call_dynSerial's contract)
  batotp_dyn_fn dynFn = nullptr;
  void *dynUser = nullptr;
  int sweepKernel = 0;            // 0 automatic (by chunk size), 1 one trajectory per lane (k_sweep), 2 a group of lanes per trajectory (k_sweep_group)
  int stepHint = 0;               // RK-step capacity a chunk starts with (0 = automatic: max(1024, 2 x grid points))
  // Thomas factor tables
  double *d_cN = nullptr;  // Thomas tables (ensure_tabs)
  int tabN = 0;
  Pmat pm;
  // staged inputs
  // two input staging sets: while chunk k is computed from one, the host rows of chunk k+1 travel into the other
  // on the copy stream (issue_inputs); d_tres / d_n0 point into the set bound to the resident chunk
  struct InSet {
    void *theta = nullptr, *cart = nullptr;
    double *ts = nullptr, *tres = nullptr;
    int *n0 = nullptr;
    size_t capTheta = 0, capCart = 0, capInB = 0, capInTs = 0;  // bytes (theta, cart), trajectories, timestamps
    std::vector<double> tresHost;
    const batotp_batch_in *src = nullptr;  // what the set holds: chunk [first, first+B) of this batch
    int first = -1, B = 0;
    bool onCopyStream = false;
#ifndef BATOTP_HOST_EMU
    cudaEvent_t ev = nullptr;
#else
    cudaEvent_t ev = 0;
#endif
  } inSet[2];
  int curIn = 0;
  double *d_tres = nullptr;
  int *d_n0 = nullptr;
  bool copiesPending = false;  // row copies of the previous chunk may still be in flight on the copy stream
  const void *in_theta = nullptr, *in_cart = nullptr;  // device views used by k_in_load
  const double *in_ts = nullptr;
  bool inF64 = false, hasTheta = false, hasCart = false;
  int B = 0, n0max = 0;
  // staged outputs
  float *d_thetaOut = nullptr, *d_cartOut = nullptr, *d_trqOut = nullptr, *d_histOut = nullptr;  // current set
  // NSETS sets of packed-output staging buffers: the rows of sub-chunk k travel to the host on the copy stream
  // while the kernels of the following sub-chunks fill the other sets - and, since nothing but the output phase
  // touches a set, while the NEXT chunk's input phase and sweeps run: when the host link is the bottleneck (several
  // GPUs sharing it) the copy engine then never idles
  float *o_thetaOut[NSETS] = {}, *o_cartOut[NSETS] = {}, *o_trqOut[NSETS] = {}, *o_histOut[NSETS] = {};
  bool setBusy[NSETS] = {};  // a copy out of the set has been enqueued since its rows were last awaited (evCopied)
  int setNext = 0;           // the staging sets rotate across sub-chunks AND chunks
  cudaStream_t copyStream = 0;
  double *d_cartOutD = nullptr;
  double *d_outD = nullptr;  // [Bo][J+C+J][OutC] FP64 final rows (keepF64)
  bool keepF64 = false;
  int mxSteps = 0;  // largest nFwd/nRev of the resident chunk (launch extents of the output phase)
  int allocPhase = 0;  // which workspace was being (re)allocated last: 0 chunk arrays, 1 output sub-chunk arrays
  // which buffers hold the final rows after interp_output
  // high-water marks so that steady-state chunks need no planning sync
  int hwNc = 0, hwSc = 0;
  std::vector<TrajState> hst;
  int phase = 0;  // 0 none, 1 loaded, 2 input done, 3 sweeps done, 4 output done
  bool lastHaveN0 = false;
  // measurement (bench.py): device time of the sweep kernel and whole-context event timer
  double sweepMs = 0;
  long sweepLaunches = 0;
  // one record per sweep launch since the last reset: device ms, trajectories of the chunk, kernel (1 lane, 2 group)
  struct SweepRec {
    double ms;
    int B, kernel;
  };
  std::vector<SweepRec> sweepLog;
  int lastSweepKernel = 1;
  // trajectories one launch of the sweep kernels keeps resident (SMs x CTAs per SM x lanes / lanes per trajectory),
  // learnt from the launches of the current configuration ([0] lane kernel, [1] group kernel; key = its dispatch key)
  int sweepCap[2] = {0, 0}, sweepCapKey = -1;
  long long cntVerify = 0, cntSteps = 0, cntTraj = 0;
  // optional per-kernel device timing (batotp_cuda_set_profile): serialises every launch
  bool profile = false;
  std::map<std::string, std::pair<double, long>> prof;
  // tail overlap (batotp_cuda_optimize_batch): a last chunk that fills at most one sweep CTA per SM runs on a second
  // context (own streams and workspaces, one host thread) next to the output / input phases of the full chunks
  batotp_ctx *helper = nullptr;
  bool tailOverlap = true;
  int walkerKernel = 0;  // sequential walkers of the input phase (cumulative norms, interpSpecial march): 0 by chunk size, 1 one thread per trajectory, 2 point-parallel increments + a group of lanes per trajectory
  // stragglers: the few trajectories of a chunk that outgrow the step capacity keep BATOTP_ST_STEP_CAP for the
  // moment and are re-run together, with a larger capacity, after the chunks of the batch (optimize_batch)
  std::vector<int> stragglers;  // indices in the caller's batch
  int stragglerSc = 0;          // the step capacity they outgrew
  int chunkFirst = 0;           // index of the resident chunk's first trajectory in the caller's batch
  bool collectStragglers = false;
  std::function<void()> onSweepsDone;  // called once the sweeps of a chunk have completed on the device
  std::function<void()> beforeSweeps;  // called after interpInputData of a chunk has been enqueued (may block)
#ifndef BATOTP_HOST_EMU
  cudaEvent_t evS0 = nullptr, evS1 = nullptr, evT[2] = {nullptr, nullptr}, evP[2] = {nullptr, nullptr};
  cudaEvent_t evOut[NSETS] = {}, evCopied[NSETS] = {};
  bool sweepPending = false;
#else
  cudaEvent_t evOut[NSETS] = {}, evCopied[NSETS] = {};
#endif
};

namespace {

// brackets one launch with events when profiling is on (and waits for it: measurement mode only)
struct ProfScope {
  batotp_ctx *h;
  const char *name;
  ProfScope(batotp_ctx *h_, const char *n) : h(h_), name(n) {
#ifndef BATOTP_HOST_EMU
    if (h->profile) {
      if (!h->evP[0]) {
        cudaEventCreate(&h->evP[0]);
        cudaEventCreate(&h->evP[1]);
      }
      cudaEventRecord(h->evP[0], h->stream);
    }
#endif
  }
  ~ProfScope() {
#ifndef BATOTP_HOST_EMU
    if (h->profile) {
      cudaEventRecord(h->evP[1], h->stream);
      cudaEventSynchronize(h->evP[1]);
      float ms = 0;
      cudaEventElapsedTime(&ms, h->evP[0], h->evP[1]);
      auto &e = h->prof[name];
      e.first += ms;
      e.second++;
    }
#endif
  }
};

#define LAUNCH_T(h, kern, nthreads, ...)                                                    \
  do {                                                                                      \
    const int nth_ = (nthreads);                                                            \
    if (nth_ > 0) {                                                                         \
      ProfScope ps_((h), #kern);                                                            \
      BATOTP_LAUNCH(kern, dim3(cdiv(nth_, 128)), dim3(128), (h)->stream, __VA_ARGS__);      \
      g_check_launch();                                                                     \
      (h)->launches++;                                                                      \
    }                                                                                       \
  } while (0)
// (trajectory, point) kernels: a 3-D grid, x over the nb trajectories (fastest), y/z over the points; the
// kernel receives (..., npts, nb) last and decomposes with TP_DECOMP
inline void tp_dims(long long fast, long long slow, dim3 &grid, dim3 &block) {
  int bdx = 128;
  if (fast < 128) {
    bdx = 32;
    while (bdx < fast) bdx <<= 1;
  }
  const int bdy = 128 / bdx;
  const long long rows = (slow + bdy - 1) / bdy;
  const long long gy = std::min<long long>(rows, 32768);
  const long long gz = (rows + gy - 1) / gy;
  grid = dim3((unsigned)((fast + bdx - 1) / bdx), (unsigned)gy, (unsigned)gz);
  block = dim3(bdx, bdy, 1);
}
#define LAUNCH_TP(h, kern, npts, nb, ...)                                                   \
  do {                                                                                      \
    const long long np_ = (long long)(npts), nb_ = (long long)(nb);                         \
    if (np_ > 0 && nb_ > 0) {                                                               \
      dim3 g_, b_;                                                                          \
      tp_dims(nb_, np_, g_, b_);                                                            \
      ProfScope ps_((h), #kern);                                                            \
      BATOTP_LAUNCH(kern, g_, b_, (h)->stream, __VA_ARGS__, (int)np_, (int)nb_);            \
      g_check_launch();                                                                     \
      (h)->launches++;                                                                      \
    }                                                                                       \
  } while (0)
// (point, trajectory) kernels with points fastest (PT_DECOMP)
#define LAUNCH_PT(h, kern, npts, nb, ...)                                                   \
  do {                                                                                      \
    const long long np_ = (long long)(npts), nb_ = (long long)(nb);                         \
    if (np_ > 0 && nb_ > 0) {                                                               \
      dim3 g_, b_;                                                                          \
      tp_dims(np_, nb_, g_, b_);                                                            \
      ProfScope ps_((h), #kern);                                                            \
      BATOTP_LAUNCH(kern, g_, b_, (h)->stream, __VA_ARGS__, (int)np_, (int)nb_);            \
      g_check_launch();                                                                     \
      (h)->launches++;                                                                      \
    }                                                                                       \
  } while (0)

void free_ws(batotp_ctx *h) {
  for (void *p : h->wsAllocs) g_free(p);
  h->wsAllocs.clear();
  h->wsBytes = 0;
  h->wsHeld = WsShape();
}
void free_out(batotp_ctx *h) {
  for (void *p : h->outAllocs) g_free(p);
  h->outAllocs.clear();
  h->outBytes = 0;
  h->outHeld = OutShape();
}

// allocating visitor of chunk_arrays / out_arrays (a count of 0 leaves the member null)
struct Allocate {
  std::vector<void *> &allocs;
  size_t &bytes;
  template <class T>
  void operator()(T *&p, size_t count) {
    p = nullptr;
    if (count == 0) return;
    p = (T *)g_alloc(count * sizeof(T));
    allocs.push_back(p);
    bytes += count * sizeof(T);
  }
};

void ensure_tabs(batotp_ctx *h, int n) {
  if (n <= h->tabN) return;
  g_free(h->d_cN);
  n = std::max(n + 64, 4096);
  // [cN | dN | rN | cC | dC | rC], n doubles each
  std::vector<double> t((size_t)6 * n, 1.0);
  double *cN = t.data(), *dN = cN + n, *rN = dN + n, *cC = rN + n, *dC = cC + n, *rC = dC + n;
  // spline.cpp:259-268 (natural) and 229-237 (clamped): the same divisions, tabulated
  cN[0] = 1.0;
  if (n > 1) cN[1] = 1.0 / 4.0;
  for (int i = 2; i < n; ++i) cN[i] = 1.0 / (4.0 - 1.0 * cN[i - 1]);
  cC[0] = 1.0 / 2.0;
  for (int i = 1; i < n; ++i) cC[i] = 1.0 / (4.0 - 1.0 * cC[i - 1]);
  // denominators of row i and their correctly rounded reciprocals (for sdiv::div)
  for (int i = 1; i < n; ++i) {
    dN[i] = 4.0 - 1.0 * cN[i - 1];
    rN[i] = 1.0 / dN[i];
    dC[i] = 4.0 - 1.0 * cC[i - 1];
    rC[i] = 1.0 / dC[i];
  }
  h->d_cN = (double *)g_alloc((size_t)6 * n * sizeof(double));
  g_h2d(h->d_cN, t.data(), (size_t)6 * n * sizeof(double), h->stream);
  g_sync(h->stream);
  h->tabN = n;
}
inline ThomasTabs thomas_tabs(const batotp_ctx *h) {
  const double *p = h->d_cN;
  const size_t n = (size_t)h->tabN;
  return ThomasTabs{p, p + n, p + 2 * n, p + 3 * n, p + 4 * n, p + 5 * n};
}

// glibc's x86-64 sin/cos come in two arithmetics, selected at load time: with fused multiply-adds on a CPU that
// has FMA and AVX2, without otherwise (sysdeps/x86_64/fpu/multiarch/ifunc-avx-fma4.h; the FMA4 variant of old AMD
// parts contracts the same expressions)
bool host_libm_uses_fma() {
#if defined(__x86_64__) && (defined(__GNUC__) || defined(__clang__))
  static const bool v = [] {
    // BATOTP_TRIG_VARIANT=1|3 overrides the detection (a process started with GLIBC_TUNABLES=glibc.cpu.hwcaps=-FMA
    // runs the plain variant on an FMA machine: that is how the test suite checks both)
    if (const char *e = getenv("BATOTP_TRIG_VARIANT")) {
      if (e[0] == '1') return false;
      if (e[0] == '3') return true;
    }
    return (__builtin_cpu_supports("fma") && __builtin_cpu_supports("avx2")) || __builtin_cpu_supports("fma4");
  }();
  return v;
#else
  return false;
#endif
}

int oversample_cap(const batotp_ctx *h, int Sc) {
  // nPtsMVCout bound for nFwd <= Sc (ba.cpp:1667-1685)
  const batotp_cfg &c = h->cfg.c;
  double outRes = c.out_res, sm = c.out_smooth_fact;
  const double integRes = c.is_auto_integ_res ? 0.004 : c.integ_res;  // auto: >= minIntegRes (ba.cpp:512)
  if (outRes < integRes) {
    sm *= std::max(c.out_res / integRes, 1.0);
    outRes = integRes;
  }
  const double integMax = c.is_auto_integ_res ? 0.2 : c.integ_res;
  const double n = sm * (std::ceil(integMax * (double)(Sc - 1) / outRes + 1.0) + 1.0);
  return std::max((int)n + 8, 16);
}

// smoothing decided on the host when it is uniform over the batch (ba.cpp:1667-1672, 1838)
bool smooth_uniform_on(const batotp_ctx *h) {
  const batotp_cfg &c = h->cfg.c;
  if (c.is_auto_integ_res) return false;
  double sm = c.out_smooth_fact;
  if (c.out_res < c.integ_res) sm *= std::max(c.out_res / c.integ_res, 1.0);
  return sm > 1.5;
}

int kin_mode(const batotp_ctx *h, int where);
// the oversampled output rows feed nothing but the smoothing stage (do_interp_output's fused path)
bool fused_out(const batotp_ctx *h) {
  return !h->cfg.trqOn && smooth_uniform_on(h) && kin_mode(h, 2) == 0 && (int)h->cfg.c.out_smooth_fact <= 11;
}

int final_cap(const batotp_ctx *h, int Sc, int Os) {
  const batotp_cfg &c = h->cfg.c;
  const double integMax = c.is_auto_integ_res ? 0.2 : c.integ_res;
  const double tLast = integMax * (double)(Sc - 1);
  const int n = (int)std::ceil(tLast / c.out_res) + 8;
  return std::max(std::max(n, 16), Os);
}

// capacities of the output arrays for a step capacity Sc: oversampled, smoothed and final points
struct OutCaps { int Oc, Os, OutC; };
OutCaps out_caps(const batotp_ctx *h, int Sc) {
  const int Oc = oversample_cap(h, Sc);
  const int Os = (!h->cfg.trqOn && smooth_uniform_on(h)) ? (int)(Oc / h->cfg.c.out_smooth_fact) + 16 : Oc;
  return {Oc, Os, final_cap(h, Sc, Os)};
}

// The chunk-resident arrays (input phase + sweeps) of a workspace shaped s, as f(Ws member, element count).
template <class F>
void chunk_arrays(Ws &w, const WsShape &s, F &&f) {
  const size_t b = (size_t)s.B, n = (size_t)s.Nc, sc = (size_t)s.Sc, R = (size_t)s.R;
  f(w.P, b * R * n);
  f(w.Q, b * R * n);
  f(w.M, b * R * n);
  f(w.sC, b * n);
  f(w.nrm, b * 2 * n);
  f(w.tab, b * n * s.RT * 4);
  f(w.hist, b * 4 * sc);
  f(w.flags, b * 2 * sc);
  f(w.st, b);
  f(w.mS, b * sc);
  const size_t t = s.trq ? b : 0;  // torque only
  f(w.A, t * 4 * s.J * n);
  f(w.AM, t * 4 * s.J * n);
  f(w.GD, t * R * n);
  f(w.GD2, t * R * n);
  f(w.queue, 4);
  f(w.ragOff, b + 1);
}

// The output sub-chunk arrays of a workspace shaped s, as f(member, element count); a count of 0: not used.
template <class F>
void out_arrays(batotp_ctx *h, const OutShape &s, F &&f) {
  const DevCfg &c = h->cfg;
  Ws &w = h->w;
  const size_t b = (size_t)s.Bo, R = (size_t)c.R, Oc = (size_t)s.Oc, Os = (size_t)s.Os, OutC = (size_t)s.OutC;
  const size_t t = c.trqOn ? b : 0;  // torque only
  f(w.sOut, b * Oc);
  f(w.segO, b * Oc);
  f(w.tauO, b * Oc);
  f(w.O5, s.fused ? 8 : b * R * Oc);  // untouched on the fused path
  f(w.OA, b * R * Os);
  f(w.OM, b * R * Os);
  f(w.OD, t * R * Oc);
  f(w.OD2, t * R * Oc);
  f(w.Trq, t * MAXD * Oc);
  f(w.Trq2, t * MAXD * Oc);
  f(w.TrqM, t * MAXD * Oc);
  for (int q = 0; q < NSETS; ++q) {
    f(h->o_thetaOut[q], b * c.J * s.rowP);
    f(h->o_cartOut[q], b * std::max(c.Cin, 1) * s.rowP);
    f(h->o_trqOut[q], t * c.J * s.rowP);
    f(h->o_histOut[q], b * 4 * s.histP);
  }
  f(h->d_cartOutD, c.C == 7 ? b * 7 * OutC : 0);
  f(h->d_outD, s.keepF64 ? b * (c.J + c.C + c.J) * OutC : 0);  // k_out_pack's layout
}

// (with a step hint the step capacity asked for is taken literally, not "at least")
bool ws_covers(const WsShape &held, const WsShape &n, bool exactSc) {
  return n.B <= held.B && n.Nc <= held.Nc && (exactSc ? n.Sc == held.Sc : n.Sc <= held.Sc) && n.J == held.J &&
         n.Cin == held.Cin && n.C == held.C && n.R == held.R && n.RT == held.RT && n.trq == held.trq;
}
// the output arrays of a sub-chunk of Bo trajectories of a chunk with step capacity Sc, at the pitches in use
OutShape out_shape(const batotp_ctx *h, int Bo, int Sc, int minOutC = 0) {
  const OutCaps k = out_caps(h, Sc);
  const int OutC = std::max(k.OutC, minOutC);
  return {Bo, Sc, k.Oc, k.Os, OutC, h->rowPitch > 0 ? h->rowPitch : OutC, h->histPitch > 0 ? h->histPitch : Sc,
          h->keepF64, fused_out(h)};
}
// (the output arrays belong to one step capacity of the chunk)
bool out_covers(const OutShape &held, const OutShape &n) {
  return n.Bo <= held.Bo && n.Sc == held.Sc && n.Oc <= held.Oc && n.Os <= held.Os && n.OutC <= held.OutC &&
         n.rowP <= held.rowP && n.histP <= held.histP && n.keepF64 == held.keepF64 && n.fused == held.fused;
}

// The planner's footprints of a chunk shaped s: its arrays, the part of them that grows with each trajectory, and the
// output arrays of its first sub-chunk.  They are the lists of arrays themselves, summed.
struct Footprints { size_t chunk, perTraj, out; };
Footprints footprints(batotp_ctx *h, const WsShape &s) {
  size_t n = 0;
  auto add = [&n](auto *&p, size_t count) { n += count * sizeof(*p); };
  auto chunk_bytes = [&](int B) {
    WsShape sb = s;
    sb.B = B;
    n = 0;
    chunk_arrays(h->w, sb, add);
    return n;
  };
  const size_t chunk = chunk_bytes(s.B), perTraj = chunk_bytes(1) - chunk_bytes(0);
  n = 0;
  out_arrays(h, out_shape(h, std::min(s.B, h->outChunk), s.Sc), add);
  return {chunk, perTraj, n};
}

// A chunk whose arrays would not fit is refused before anything is freed or allocated, with the size that would fit
// (the batch call continues with smaller chunks - and finds the workspace of its previous call intact: releasing and
// re-allocating ~130 GB costs 170 ms).  Beside the chunk arrays the context will ask for the output arrays of one
// sub-chunk and some slack for the input staging sets / the tail helper.
void plan_chunk(batotp_ctx *h, const WsShape &want) {
#ifndef BATOTP_HOST_EMU
  const size_t held = h->wsBytes + h->outBytes;  // released if the new workspace goes ahead
#else
  const size_t held = 0;  // (BATOTP_EMU_FREE_MB is what this context may use in total)
#endif
  const Footprints fp = footprints(h, want);
  const size_t fr = g_free_bytes() + held;
  const size_t reserve = ((size_t)2 << 30) + fp.out;
  const double room = (double)(fr > reserve ? fr - reserve : 0);
  if ((double)fp.chunk > 0.94 * room) {
    char buf[200];
    snprintf(buf, sizeof buf, "chunk of %d trajectories needs %.1f GB of workspace (%zu bytes each), %.1f GB free",
             want.B, (double)fp.chunk * 1e-9, fp.perTraj, (double)fr * 1e-9);
    Err er{buf};
    er.oom = true;
    er.fitB = (int)std::min<double>(2.0e9, 0.9 * room / (double)fp.perTraj);
    er.planned = true;
    throw er;
  }
}

// chunk-resident arrays (input phase + sweeps)
void ensure_ws(batotp_ctx *h, int B, int Nc, int Sc) {
  const DevCfg &c = h->cfg;
  const WsShape want{B, Nc, Sc, c.J, c.Cin, c.C, c.R, c.RT, c.trqOn != 0};
  if (ws_covers(h->wsHeld, want, h->stepHint > 0)) {
    h->w.B = B;
    return;
  }
  h->allocPhase = 0;
  plan_chunk(h, want);
  free_ws(h);
  free_out(h);
  Ws &w = h->w;
  memset(&w, 0, sizeof(w));
  w.cfg = h->cfg;
  w.B = B;
  w.Nc = Nc;
  w.Sc = Sc;
  w.R = want.R;
  w.RT = want.RT;
  w.AD = want.J;
  chunk_arrays(w, want, Allocate{h->wsAllocs, h->wsBytes});
  if (want.trq) g_zero(w.A, (size_t)B * 4 * w.AD * Nc * sizeof(double), h->stream);
  h->wsHeld = want;
  ensure_tabs(h, std::max(Nc, Sc) + 8);
}

inline int row_pitch(const batotp_ctx *h) { return h->rowPitch > 0 ? h->rowPitch : h->w.OutC; }
inline int hist_pitch(const batotp_ctx *h) { return h->histPitch > 0 ? h->histPitch : h->w.Sc; }

void select_out_set(batotp_ctx *h, int q) {
  h->curSet = q;
  h->d_thetaOut = h->o_thetaOut[q];
  h->d_cartOut = h->o_cartOut[q];
  h->d_trqOut = h->o_trqOut[q];
  h->d_histOut = h->o_histOut[q];
}

// output sub-chunk arrays, sized from the step capacity of the resident chunk
void ensure_out(batotp_ctx *h, int Bo, int minOutC = 0) {
  Ws &w = h->w;
  const OutShape want = out_shape(h, Bo, w.Sc, minOutC);
  if (out_covers(h->outHeld, want)) return;
  free_out(h);
  h->allocPhase = 1;
  out_arrays(h, want, Allocate{h->outAllocs, h->outBytes});
  h->outHeld = want;
  for (bool &busy : h->setBusy) busy = false;  // (free_out has waited for the device)
  select_out_set(h, 0);
  w.Oc = want.Oc;
  w.Os = want.Os;
  w.OutC = want.OutC;
  ensure_tabs(h, std::max(std::max(w.Nc, w.Sc), want.Oc) + 8);
}

void set_cfg(batotp_ctx *h, const batotp_cfg *cfg) {
  DevCfg d;
  memset(&d, 0, sizeof(d));
  d.c = *cfg;
  d.J = cfg->n_joints;
  d.Cin = cfg->n_cart;
  const bool quat = (cfg->path_type == BATOTP_CART || cfg->path_type == BATOTP_BOTH) && cfg->n_cart == 6;
  d.C = quat ? 7 : cfg->n_cart;
  d.cartOn = (cfg->is_cart_vel_on || cfg->is_cart_acc_on) ? 1 : 0;
  d.trqOn = cfg->is_trq_on ? 1 : 0;
  if (d.C < 3) d.C = 3;  // adjust_s / interpSpecial always read cart rows 0..2 (ba.cpp:463, 697)
  // A joint-only generic robot (no kinematic model, joint path, no Cartesian or torque limits) has Cartesian rows
  // that are zero throughout (ba.cpp:245-280 with no fwdKin): only its joint rows are stored, and the kernels read
  // the Cartesian rows as a literal 0.0.  (isInterpOnly re-samples and returns whatever rows the input had.)
  const bool jointOnly = cfg->robot_type == BATOTP_GENJNT && cfg->path_type == BATOTP_JOINT && !d.cartOn && !d.trqOn &&
                         !cfg->is_interp_only;
  d.R = jointOnly ? d.J : d.J + d.C;
  d.RT = d.J + (d.cartOn ? 3 : 0) + (d.trqOn ? 4 * d.J : 0);
  d.quadThresh = cfg->cart_thresh * cfg->cart_thresh;
  d.pm = h->pm;
  // strict trig on the device: the arithmetic variant of the host libm this process runs against (k_trig.cuh)
  d.trigDev = (cfg->trig_mode == 1) ? (host_libm_uses_fma() ? 3 : 1) : 0;
  const double Bt[6][6] = {{1. / 5, 3. / 40, 44. / 45, 19372. / 6561, 9017. / 3168, 35. / 384},
                           {0, 9. / 40, -56. / 15, -25360. / 2187, -355. / 33, 0},
                           {0, 0, 32. / 9, 64448. / 6561, 46732. / 5247, 500. / 1113},
                           {0, 0, 0, -212. / 729, 49. / 176, 125. / 192},
                           {0, 0, 0, 0, -5103. / 18656, -2187. / 6784},
                           {0, 0, 0, 0, 0, 11. / 84}};  // ba.cpp:58-63, literals as written there
  memcpy(d.B, Bt, sizeof(Bt));
  for (int i = 0; i < MAXD; ++i) {
    d.accMaxF[i] = (float)cfg->jnt_acc_max[i];
    d.velMaxF[i] = (float)std::fabs(cfg->jnt_vel_max[i]);
  }
  if (!h->haveCfg || memcmp(&h->cfg.c, cfg, sizeof(batotp_cfg)) != 0) {
    h->hwNc = 0;  // capacity high-water marks belong to one configuration
    h->hwSc = 0;
  }
  h->cfg = d;
  h->w.cfg = d;  // the options travel with every launch (Ws is a kernel parameter)
  h->haveCfg = true;
}

int check_cfg(batotp_ctx *h) {
  const batotp_cfg &c = h->cfg.c;
  if (c.n_joints < 1 || c.n_joints > MAXD || c.n_cart < 0 || c.n_cart > MAXD) {
    h->err = "nJoints/nCart outside 1..7";
    return -1;
  }
  if (c.is_svd) {
    h->err = "isSVD=1 is outside the accelerated scope (SURVEY §8f rank 3)";
    return -1;
  }
  if (c.is_trq_on && c.is_parallel && !c.is_par2ser && !(c.is_cart_vel_on || c.is_cart_acc_on)) {
    h->err = "parallel-mechanism torque limits without isPar2Ser need a Cartesian limit switched on: setA reads the "
             "Cartesian point, which the reference only refreshes then (ba.cpp:1363-1380, 1408-1411)";
    return -1;
  }
  if (c.is_trq_on && c.dyn_source == 1) {
    if (c.is_parallel) {
      h->err = "dyn_source = 1 (a caller-supplied dynamic model) serves serial mechanisms only";
      return -1;
    }
    if (!h->dynFn) {
      h->err = "dyn_source = 1 needs a point function: call batotp_cuda_set_dyn_callback first";
      return -1;
    }
  } else if (c.is_trq_on && !((c.robot_type == BATOTP_RR && !c.is_parallel) || (c.robot_type == BATOTP_CSPR3DOF && c.is_parallel))) {
    h->err = "torque limits need a dynamic model: batotp has one for RR (serial) and CSPR3DOF (parallel) only (robot.cpp:349-360, 463-474); supply yours with dyn_source = 1 + batotp_cuda_set_dyn_callback";
    return -1;
  }
  if (c.is_interp_only && c.path_type == BATOTP_CART) {
    h->err = "isInterpOnly needs joint data: the reference sizes the result by theta[0] (ba.cpp:141)";
    return -1;
  }
  return 0;
}

// ---- strict-parity trig: the host evaluates the trig-bearing point functions with its libm,
//      exactly as the reference does (DESIGN.md §trig).  Rows travel D2H/H2D around the call.
//      `base` is a point-major array [npts][nb][R]; b0 = chunk index of its first trajectory.
void host_rows_apply(batotp_ctx *h, double *base, int npts, int nb, int b0, bool over, int kind) {
  // kind 1: fwdKin (theta rows -> cart rows); kind 2: aa2qVect on cart rows 3..6
  const DevCfg &c = h->cfg;
  const int R = c.R, J = c.J;
  h->hst.resize(h->B);
  g_d2h(h->hst.data(), h->w.st, (size_t)h->B * sizeof(TrajState), h->stream);
  g_sync(h->stream);
  int nmax = 0;
  for (int bl = 0; bl < nb; ++bl) {
    const TrajState &s = h->hst[b0 + bl];
    if (s.status & ST_FATAL_MASK) continue;
    nmax = std::max(nmax, over ? s.nOver : s.nPts);
  }
  nmax = std::min(nmax, npts);
  if (nmax <= 0) return;
  std::vector<double> buf((size_t)nmax * nb * R);
  g_d2h(buf.data(), base, buf.size() * sizeof(double), h->stream);
  g_sync(h->stream);
  const int nth = std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
  const size_t pst = (size_t)nb * R;
  auto work = [&](int tid) {
    for (int bl = tid; bl < nb; bl += nth) {
      const TrajState &s = h->hst[b0 + bl];
      if (s.status & ST_FATAL_MASK) continue;
      const int n = std::min(over ? s.nOver : s.nPts, nmax);
      double *r0 = buf.data() + (size_t)bl * R;
      if (kind == 1) {
        for (int i = 0; i < n; ++i) {
          double *p = r0 + (size_t)i * pst;
          double xyz[3];
          if (c.c.robot_type == BATOTP_KUKA) {
            fk_kuka_point(Trig{0}, p, xyz);
            for (int q = 0; q < 3; ++q) p[J + q] = xyz[q];
          } else if (c.c.robot_type == BATOTP_RR) {
            fk_rr_point(Trig{0}, p, xyz);
            p[J] = xyz[0];
            p[J + 1] = xyz[1];
          }
        }
      } else if (kind == 2) {
        double aa[3] = {r0[J + 3], r0[J + 4], r0[J + 5]}, q[4], qprev[4];
        aa2q_dev(Trig{0}, aa, qprev);
        for (int i = 0; i < n; ++i) {
          double *p = r0 + (size_t)i * pst;
          aa[0] = p[J + 3];
          aa[1] = p[J + 4];
          aa[2] = p[J + 5];
          aa2q_dev(Trig{0}, aa, q);
          double qdir = 0;
          for (int j = 0; j < 4; ++j) qdir += q[j] * qprev[j];
          if (qdir < 0.0)
            for (int j = 0; j < 4; ++j) q[j] = -q[j];
          for (int j = 0; j < 4; ++j) qprev[j] = q[j];
          p[J + 3] = q[0];
          p[J + 4] = q[1];
          p[J + 5] = q[2];
          p[J + 6] = q[3];
        }
      }
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nth; ++t) th.emplace_back(work, t);
  work(0);
  for (auto &x : th) x.join();
  g_h2d(base, buf.data(), buf.size() * sizeof(double), h->stream);
  g_sync(h->stream);
}

// kinematics after a resampling stage (ba.cpp:245-280 mode 0; ba.cpp:616-632 mode 1; ba.cpp:1723-1741 mode 2)
int kin_mode(const batotp_ctx *h, int where) {
  const DevCfg &c = h->cfg;
  const int pt = c.c.path_type;
  int mode = 0;
  if (pt == BATOTP_JOINT) {
    if (where == 0)
      mode = c.cartOn ? 1 : 3;
    else
      mode = (c.c.robot_type == BATOTP_GENJNT) ? (where == 1 ? 3 : 0) : 1;
    if (mode == 1 && !(c.c.robot_type == BATOTP_KUKA || c.c.robot_type == BATOTP_RR)) mode = 0;  // no model
  } else if (pt == BATOTP_CART) {
    if (where == 0)
      mode = (c.c.is_jnt_vel_on || c.c.is_jnt_acc_on || c.c.is_trq_on) ? 2 : 4;
    else
      mode = 2;
    if (mode == 2 && c.c.robot_type != BATOTP_CSPR3DOF) mode = 0;
  }
  return mode;
}

void apply_kinematics(batotp_ctx *h, int where) {
  const DevCfg &c = h->cfg;
  const bool over = (where == 2);
  double *base = over ? h->w.O5 : h->w.P;
  const int npts = over ? h->w.Oc : h->w.Nc;
  const int nb = over ? h->w.Bo : h->w.B;
  const int b0 = over ? h->w.b0 : 0;
  const int mode = kin_mode(h, where);
  if (mode == 0) return;
  if (mode == 3 && c.R == c.J) return;  // the zeroed Cartesian rows are not stored
  if (mode == 1 && c.c.trig_mode == 2) {
    host_rows_apply(h, base, npts, nb, b0, over, 1);
    return;
  }
  LAUNCH_TP(h, k_pointfn, npts, nb, h->w, base, b0, mode, over ? 1 : 0, h->pm);
}

void thomas_rows(batotp_ctx *h, double *src, double *dst, int nb, int b0, int rows, int rowsPerTraj, int nsel,
                 int clamped) {
  const ThomasTabs t = thomas_tabs(h);
  LAUNCH_T(h, k_thomas_rows, nb * rows, h->w, src, dst, nb, b0, rows, rowsPerTraj, nsel, clamped, t);
}

// One launch of a sweep kernel over the resident chunk: nt threads per CTA, `lanes` lanes per trajectory.  kind 1 is
// the lane kernel, 2 the group kernel: it names the launch in sweepLog and selects the sweepCap slot the launch fills.
template <typename Kernel>
void launch_sweep_kernel(batotp_ctx *h, Kernel kern, int kind, int nt, size_t smem, int lanes, const char *name) {
  g_zero(h->w.queue, sizeof(int) * 4, h->stream);
  h->lastSweepKernel = kind;
#ifndef BATOTP_HOST_EMU
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (smem) CU_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int perSm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, kern, nt, smem);
  if (perSm < 1) perSm = 1;
  int blocks = (int)std::min<long long>((long long)sms * perSm, ((long long)h->B * lanes + nt - 1) / nt);
  if (blocks < 1) blocks = 1;
  h->sweepCap[kind - 1] = sms * perSm * nt / lanes;
  if (!h->evS0) {
    CU_CHECK(cudaEventCreate(&h->evS0));
    CU_CHECK(cudaEventCreate(&h->evS1));
  }
  CU_CHECK(cudaEventRecord(h->evS0, h->stream));
#else
  int blocks = 1;
  if (const char *e = getenv("BATOTP_EMU_SWEEP_CAP")) h->sweepCap[kind - 1] = atoi(e);  // TEST-ONLY: pretend this occupancy
#endif
  {
    ProfScope ps_(h, name);
    BATOTP_LAUNCH_WARP(kern, dim3(blocks), dim3(nt), smem, h->stream, h->w);
    g_check_launch();
  }
#ifndef BATOTP_HOST_EMU
  CU_CHECK(cudaEventRecord(h->evS1, h->stream));
  h->sweepPending = true;
#endif
  h->launches++;
  h->sweepLaunches++;
}

template <int J, bool CART, bool TRQ, bool PAR = false>
void launch_sweep(batotp_ctx *h, bool group) {
  if (group)
    launch_sweep_kernel(h, k_sweep_group<J, CART, TRQ>, 2, SWG_NT, 0, GroupShape<J, CART>::G, "k_sweep_group");
  else
    launch_sweep_kernel(h, k_sweep<J, CART, TRQ, PAR>, 1, SW_NT, SweepLayout<J, CART, TRQ, PAR>::bytes, 1, "k_sweep");
}

// Which sweep kernel serves a chunk of B trajectories: one trajectory per lane (k_sweep.cuh: the fewest issue slots
// per trajectory, the choice when the chunk fills the machine) or a group of lanes per trajectory (k_sweep_group.cuh:
// a quarter of the latency per point, the choice when the latency of one trajectory bounds the launch).  Torque limits
// of a parallel mechanism without Par2Ser (ba.cpp:1463-1491) have the lane kernel only, whatever sweepKernel asks.
bool group_sweep(const DevCfg &c, int sweepKernel, int B) {
  if (c.trqOn && c.c.is_parallel && !c.c.is_par2ser) return false;
  if (sweepKernel == 1) return false;
  if (sweepKernel == 2) return true;
  const bool exact = c.cartOn || c.trqOn;
  return B <= (exact ? SWEEP_GROUP_MAX_B_EXACT : SWEEP_GROUP_MAX_B);
}

int dispatch_sweep(batotp_ctx *h) {
  const DevCfg &c = h->cfg;
  const int key = c.J * 4 + (c.cartOn ? 2 : 0) + (c.trqOn ? 1 : 0);
  const bool par = c.trqOn && c.c.is_parallel && !c.c.is_par2ser;
  const int capKey = key * 2 + (par ? 1 : 0);
  if (capKey != h->sweepCapKey) {  // another kernel instance: its occupancy is not known yet
    h->sweepCap[0] = h->sweepCap[1] = 0;
    h->sweepCapKey = capKey;
  }
  if (par) {  // one trajectory per lane only (group_sweep)
    if (key == 3 * 4 + 3) {
      launch_sweep<3, true, true, true>(h, false);
      return 0;
    }
    h->err = "parallel-mechanism torque limits without isPar2Ser are instantiated for 3 joints + Cartesian limits (CSPR3DOF)";
    return -1;
  }
  const bool group = group_sweep(c, h->sweepKernel, h->B);
  switch (key) {
    case 7 * 4 + 0: launch_sweep<7, false, false>(h, group); return 0;  // GEN7DOF
    case 7 * 4 + 2: launch_sweep<7, true, false>(h, group); return 0;   // KUKA-LWR-IV
    case 7 * 4 + 3: launch_sweep<7, true, true>(h, group); return 0;    // KUKA-LWR-IV with a caller-supplied torque model
    case 7 * 4 + 1: launch_sweep<7, false, true>(h, group); return 0;   // 7 joints, torque model, no Cartesian limits
    case 6 * 4 + 3: launch_sweep<6, true, true>(h, group); return 0;
    case 6 * 4 + 2: launch_sweep<6, true, false>(h, group); return 0;   // UR5
    case 6 * 4 + 0: launch_sweep<6, false, false>(h, group); return 0;
    case 2 * 4 + 3: launch_sweep<2, true, true>(h, group); return 0;    // RR
    case 3 * 4 + 3: launch_sweep<3, true, true>(h, group); return 0;    // CSPR3DOF (Par2Ser)
    case 3 * 4 + 2: launch_sweep<3, true, false>(h, group); return 0;
    case 2 * 4 + 2: launch_sweep<2, true, false>(h, group); return 0;
    default:
      h->err = "no sweep kernel instantiated for this (nJoints, Cartesian, torque) combination; add a line to dispatch_sweep()";
      return -1;
  }
}

}  // namespace
#include "host_strict.inl"
namespace {
// ---- phases ---------------------------------------------------------------------------
void free_inset(batotp_ctx::InSet &q) {
  g_free(q.theta);
  g_free(q.cart);
  g_free(q.ts);
  g_free(q.tres);
  g_free(q.n0);
  q.theta = q.cart = nullptr;
  q.ts = q.tres = nullptr;
  q.n0 = nullptr;
  q.capTheta = q.capCart = q.capInB = q.capInTs = 0;
  q.src = nullptr;
  q.first = -1;
}

// host rows of chunk [first, first+B) -> staging set `qi`, enqueued on stream `st`
void issue_inputs(batotp_ctx *h, const batotp_batch_in *in, int first, int B, int qi, cudaStream_t st, bool onCopy) {
  const DevCfg &c = h->cfg;
  batotp_ctx::InSet &q = h->inSet[qi];
  const int n0 = in->n0_max;
  const bool f64 = (in->theta_f64 || in->cart_f64);
  const size_t es = f64 ? 8 : 4;
  const size_t thBytes = (size_t)B * c.J * n0 * es, caBytes = (size_t)B * c.Cin * n0 * es;
  const void *th = f64 ? (const void *)in->theta_f64 : (const void *)in->theta_f32;
  const void *ca = f64 ? (const void *)in->cart_f64 : (const void *)in->cart_f32;
#ifndef BATOTP_HOST_EMU
  if (!q.ev) CU_CHECK(cudaEventCreateWithFlags(&q.ev, cudaEventDisableTiming));
  CU_CHECK(cudaEventSynchronize(q.ev));  // the set's previous transfer has left tresHost
#endif
  q.src = nullptr;
  // resident rows are used where they are; host rows need room for what this call copies (the staging set may
  // have been sized for another robot / path length: each block keeps its own capacity)
  const size_t needTh = (in->on_device || !th) ? 0 : thBytes, needCa = (in->on_device || !ca) ? 0 : caBytes;
  const size_t needTs = (in->on_device || !in->timestamp) ? 0 : (size_t)B * n0;
  if (needTh > q.capTheta || needCa > q.capCart || (size_t)B > q.capInB || needTs > q.capInTs || !q.tres) {
    const size_t capB = std::max((size_t)B, q.capInB);
    const size_t cTh = std::max(needTh, q.capTheta), cCa = std::max(needCa, q.capCart), cTs = std::max(needTs, q.capInTs);
    free_inset(q);
    if (cTh) q.theta = g_alloc(cTh);
    if (cCa) q.cart = g_alloc(cCa);
    if (cTs) q.ts = (double *)g_alloc(cTs * 8);
    q.tres = (double *)g_alloc(capB * 8);
    q.n0 = (int *)g_alloc(capB * 4);
    q.capTheta = cTh;
    q.capCart = cCa;
    q.capInB = capB;
    q.capInTs = cTs;
  }
  q.tresHost.resize(B);
  for (int b = 0; b < B; ++b) q.tresHost[b] = in->tres ? in->tres[first + b] : in->tres_all;  // per-trajectory tres (small)
  g_h2d(q.tres, q.tresHost.data(), (size_t)B * 8, st);
  if (!in->on_device) {
    if (th) g_h2d(q.theta, (const char *)th + (size_t)first * c.J * n0 * es, thBytes, st);
    if (ca) g_h2d(q.cart, (const char *)ca + (size_t)first * c.Cin * n0 * es, caBytes, st);
    if (in->timestamp) g_h2d(q.ts, in->timestamp + (size_t)first * n0, (size_t)B * n0 * 8, st);
  }
  if (in->n0) g_h2d(q.n0, in->n0 + first, (size_t)B * 4, st);
  g_event_record(q.ev, st);
  q.src = in;
  q.first = first;
  q.B = B;
  q.onCopyStream = onCopy;
}

// binds the staging set that holds chunk [first, first+B) (transferring it now if no prefetch did)
void stage_inputs(batotp_ctx *h, const batotp_batch_in *in, int first, int B) {
  const DevCfg &c = h->cfg;
  const int n0 = in->n0_max;
  ProfScope ps_(h, "copy_h2d(stage)");
  int qi = -1;
  for (int k = 0; k < 2; ++k)
    if (h->inSet[k].src == in && h->inSet[k].first == first && h->inSet[k].B == B) qi = k;
  if (qi < 0) {
    qi = h->curIn ^ 1;
    issue_inputs(h, in, first, B, qi, h->stream, false);
  } else if (h->inSet[qi].onCopyStream) {
    g_stream_wait(h->stream, h->inSet[qi].ev);
  }
  h->curIn = qi;
  const batotp_ctx::InSet &q = h->inSet[qi];
  h->inSet[qi].src = nullptr;  // consumed: a later call with the same arguments must transfer again
  h->inF64 = (in->theta_f64 || in->cart_f64);
  h->hasTheta = (in->theta_f32 || in->theta_f64);
  h->hasCart = (in->cart_f32 || in->cart_f64);
  const size_t es = h->inF64 ? 8 : 4;
  const void *th = h->inF64 ? (const void *)in->theta_f64 : (const void *)in->theta_f32;
  const void *ca = h->inF64 ? (const void *)in->cart_f64 : (const void *)in->cart_f32;
  if (in->on_device) {
    h->in_theta = th ? (const char *)th + (size_t)first * c.J * n0 * es : nullptr;
    h->in_cart = ca ? (const char *)ca + (size_t)first * c.Cin * n0 * es : nullptr;
    h->in_ts = in->timestamp ? in->timestamp + (size_t)first * n0 : nullptr;
  } else {
    h->in_theta = th ? q.theta : nullptr;
    h->in_cart = ca ? q.cart : nullptr;
    h->in_ts = in->timestamp ? q.ts : nullptr;
  }
  h->d_tres = q.tres;
  h->d_n0 = q.n0;
  h->B = B;
  h->n0max = n0;
}

void run_load_prepare(batotp_ctx *h, bool haveN0) {
  Ws &w = h->w;
  w.B = h->B;
  const int *n0 = haveN0 ? h->d_n0 : nullptr;
  if (h->inF64)
    LAUNCH_TP(h, (k_in_load<double>), h->n0max, h->B, w, (const double *)h->in_theta, (const double *)h->in_cart, n0,
              h->d_tres);
  else
    LAUNCH_TP(h, (k_in_load<float>), h->n0max, h->B, w, (const float *)h->in_theta, (const float *)h->in_cart, n0,
              h->d_tres);
  LAUNCH_T(h, k_in_prepare, h->B, w, h->in_ts, h->n0max, h->hasTheta ? 1 : 0, h->hasCart ? 1 : 0);
}

// returns max over trajectories of (nNew, nPts) for capacity planning
int read_plan_max(batotp_ctx *h, int *anyGridCap) {
  h->hst.resize(h->B);
  g_d2h(h->hst.data(), h->w.st, (size_t)h->B * sizeof(TrajState), h->stream);
  g_sync(h->stream);
  int mx = 0, cap = 0;
  for (int b = 0; b < h->B; ++b) {
    const TrajState &s = h->hst[b];
    if (s.status & ST_GRID_CAP) cap = 1;
    if (s.status & ST_FATAL_MASK) continue;
    mx = std::max(mx, std::max(s.nNew, s.nPts));
  }
  if (anyGridCap) *anyGridCap = cap;
  return mx;
}

#define WALKER_GROUP_MAX_B 32768
int do_interp_input(batotp_ctx *h, bool haveN0, bool planSync) {
  const DevCfg &c = h->cfg;
  Ws &w = h->w;
  const int B = h->B;
  const bool adjust = !(c.c.s_weights[1] + c.c.s_weights[2] < 1e-8);  // ba.cpp:416
  run_load_prepare(h, haveN0);
  const int pt = c.c.path_type;
  if ((pt == BATOTP_CART || pt == BATOTP_BOTH) && c.Cin == 6) {  // ba.cpp:185-192
    if (c.c.trig_mode == 2)
      host_rows_apply(h, w.P, w.Nc, B, 0, false, 2);
    else
      LAUNCH_T(h, k_aa2q, B, w);
  }
  if (c.c.input_decim_fact > 1 || c.c.smooth_window > 1) {
    LAUNCH_T(h, k_in_smooth_decimate, B * c.R, w);
    LAUNCH_T(h, k_in_decim_fix, B, w);
  }
  apply_kinematics(h, 0);
  if (adjust) {
    // chunks that do not fill the machine are bound by the latency of one trajectory in the one-thread-per-trajectory
    // walkers: their per-point work goes to point-parallel / group kernels (measured on the B200: KUKA x4096 march
    // 107 -> 24.5 ms, cumulative norms 23.5 -> 12.4 ms; GEN7DOF x56832 19.5 -> 22.6 and 2.2 -> 3.1 ms, hence the switch)
    const bool smallChunk = h->walkerKernel == 2 || (h->walkerKernel == 0 && B <= WALKER_GROUP_MAX_B);
    if (smallChunk) LAUNCH_TP(h, k_adjust_inc, w.Nc, B, w);
    LAUNCH_T(h, k_adjust_s, B, w, 1, smallChunk ? 1 : 0);
    if (planSync) {
      const int mx = read_plan_max(h, nullptr);
      const int need = (int)(mx * 1.125) + 64;
      if (need > w.Nc) return need;  // caller grows the workspace and restarts the chunk
    }
    thomas_rows(h, w.P, w.M, B, 0, c.R, c.R, 0, 0);
    if (smallChunk && c.J + MAXD <= MG && c.R <= MG) {  // a group of lanes per trajectory (k_input.cuh)
      ProfScope ps_(h, "k_march_group");
      BATOTP_LAUNCH_WARP(k_march_group, dim3((unsigned)(((long long)B * MG + 127) / 128)), dim3(128), 0, h->stream, w);
      g_check_launch();
      h->launches++;
    } else if (c.J == 7 && c.R == 7)
      LAUNCH_T(h, (k_march<7, 0>), B, w);
    else if (c.J == 7 && c.R == 10)
      LAUNCH_T(h, (k_march<7, 3>), B, w);
    else if (c.J == 6 && c.R == 13)
      LAUNCH_T(h, (k_march<6, 7>), B, w);
    else if (c.J == 3 && c.R == 6)
      LAUNCH_T(h, (k_march<3, 3>), B, w);
    else if (c.J == 2 && c.R == 5)
      LAUNCH_T(h, (k_march<2, 3>), B, w);
    else
      LAUNCH_T(h, (k_march<0, 0>), B, w);
    std::swap(w.P, w.Q);
    apply_kinematics(h, 1);
    if (smallChunk) LAUNCH_TP(h, k_adjust_inc, w.Nc, B, w);
    LAUNCH_T(h, k_adjust_s, B, w, 0, smallChunk ? 1 : 0);
    thomas_rows(h, w.P, w.M, B, 0, c.R, c.R, 0, 0);
    LAUNCH_TP(h, k_resample, w.Nc, B, w);
    LAUNCH_TP(h, k_resample_check, w.Nc, B, w);
    LAUNCH_T(h, k_resample_commit, B, w);
    std::swap(w.P, w.Q);
    apply_kinematics(h, 1);
  }
  // ba.cpp:297-305: final splines on the uniform grid, then the dynamic model
  thomas_rows(h, w.P, w.M, B, 0, c.R, c.R, 0, 0);
  LAUNCH_T(h, k_final_plan, B, w);
  if (c.trqOn) {
    LAUNCH_TP(h, k_eval_grid, w.Nc, B, w);
    if (!c.c.is_parallel && (c.c.trig_mode == 2 || c.c.dyn_source == 1))
      host_dyn_rr_grid(h);
    else
      LAUNCH_TP(h, k_dyn_grid, w.Nc, B, w, h->pm);
    thomas_rows(h, w.A, w.AM, B, 0, 4 * w.AD, 4 * w.AD, 0, 0);
  }
  {  // the segment table, tiled through shared memory
    const long long rows = cdiv(w.Nc, BT_SEGS);
    const long long gy = std::min<long long>(rows, 32768), gz = (rows + gy - 1) / gy;
    ProfScope ps_(h, "k_build_table_tile");
    if (!c.trqOn && w.RT <= BT_ROWS) {  // kinematic rows only
      BATOTP_LAUNCH_WARP((k_build_table_tile<BT_TRAJ, BT_ROWS>), dim3((unsigned)cdiv(B, BT_TRAJ), (unsigned)gy, (unsigned)gz),
                         dim3(BT_TRAJ, BT_SEGS, 1), 0, h->stream, w, w.Nc, B);
    } else if (w.RT <= BT_ROWS_DYN) {  // with the dynamics rows
      BATOTP_LAUNCH_WARP((k_build_table_tile<BT_TRAJ_DYN, BT_ROWS_DYN>),
                         dim3((unsigned)cdiv(B, BT_TRAJ_DYN), (unsigned)gy, (unsigned)gz), dim3(BT_TRAJ_DYN, BT_SEGS, 1), 0,
                         h->stream, w, w.Nc, B);
    } else {
      LAUNCH_TP(h, k_build_table, w.Nc, B, w);
    }
    g_check_launch();
    h->launches++;
  }
  h->phase = 2;
  return 0;
}

// BA::interpInputData with _isInterpOnly (ba.cpp:139-159) for the resident chunk: re-sample every row with
// natural splines at outRes; the result is packed like an optimised trajectory (one output "sub-chunk" =
// the whole chunk, whose point-major layout the packing kernel reads directly).
int do_interp_only(batotp_ctx *h, bool haveN0) {
  const DevCfg &c = h->cfg;
  for (int attempt = 0; attempt < 4; ++attempt) {
    int Nc = std::max(std::max(h->hwNc, h->n0max + 8), h->w.Nc);
    ensure_ws(h, h->B, Nc, std::max(h->hwSc, 1024));
    Ws &w = h->w;
    w.B = h->B;
    run_load_prepare(h, haveN0);
    int gridCap = 0;
    read_plan_max(h, &gridCap);
    int mx = 0;  // largest re-sampled length, the trajectories that only ran out of room included
    for (int b = 0; b < h->B; ++b) {
      const TrajState &t = h->hst[b];
      if (t.status & (ST_FATAL_MASK & ~ST_GRID_CAP)) continue;
      mx = std::max(mx, std::max(t.nNew, t.nPts));
    }
    if (gridCap || mx + 8 > w.Nc) {  // the re-sampled rows need more room
      h->hwNc = std::max(h->hwNc, mx + 64);
      free_ws(h);
      continue;
    }
    const int pt = c.c.path_type;
    if ((pt == BATOTP_CART || pt == BATOTP_BOTH) && c.Cin == 6) {  // ba.cpp:145-148
      if (c.c.trig_mode == 2)
        host_rows_apply(h, w.P, w.Nc, h->B, 0, false, 2);
      else
        LAUNCH_T(h, k_aa2q, h->B, w);
    }
    thomas_rows(h, w.P, w.M, h->B, 0, c.R, c.R, 0, 0);
    LAUNCH_TP(h, k_resample, w.Nc, h->B, w);
    LAUNCH_TP(h, k_resample_check, w.Nc, h->B, w);
    LAUNCH_T(h, k_resample_commit, h->B, w);
    std::swap(w.P, w.Q);
    ensure_out(h, h->B, mx + 8);
    w.b0 = 0;
    w.Bo = h->B;
    LAUNCH_T(h, k_interp_only_finish, h->B, w);
    select_out_set(h, 0);
    const bool strictQuat = (c.C == 7 && c.c.trig_mode != 0);
    const int rp = row_pitch(h), hp = hist_pitch(h);
    if (h->d_trqOut) g_zero(h->d_trqOut, (size_t)h->B * c.J * rp * sizeof(float), h->stream);  // no torque rows here
    LAUNCH_PT(h, k_out_pack, std::max(w.OutC, rp), h->B, w, w.P, w.M, (double *)nullptr, (double *)nullptr, h->d_thetaOut,
              h->d_cartOut, (float *)nullptr, strictQuat ? h->d_cartOutD : (double *)nullptr, h->d_outD, rp,
              (const long long *)nullptr, 0ll);
    LAUNCH_PT(h, k_pack_hist, std::max(w.Sc, hp), h->B, w, h->d_histOut, hp);
    h->phase = 4;
    return 0;
  }
  h->err = "grid capacity retry limit reached";
  return -1;
}

int do_sweeps(batotp_ctx *h) {
  if (dispatch_sweep(h) != 0) return -1;
  h->phase = 3;
  return 0;
}

// interpOutputData for the sub-chunk [b0, b0+Bo) of the resident chunk
void do_interp_output(batotp_ctx *h, int b0, int Bo) {
  const DevCfg &c = h->cfg;
  ensure_out(h, Bo);
  Ws &w = h->w;
  w.b0 = b0;
  w.Bo = Bo;
  const ThomasTabs t = thomas_tabs(h);
  // launch extents from the longest trajectory of the chunk rather than from the capacities (held Os == Oc: no
  // smoothing, or capacities too small for it to shrink them - the smoothed rows then span the oversampled extent)
  const OutCaps l = out_caps(h, std::max(h->mxSteps, 4));
  const int lOc = std::min(w.Oc, l.Oc), lOs = (w.Os == w.Oc) ? lOc : std::min(w.Os, l.Os);
  // s(t) of the whole resident chunk is planned with its first sub-chunk: one launch of the sequential solve over
  // the chunk's trajectories instead of one per sub-chunk (mS is chunk-resident, [B][Sc])
  if (b0 == 0) LAUNCH_T(h, k_out_plan, h->B, w, t);
  {  // s(t) at the oversampled sites and their segments, 32x32 tiles
    const long long rows = cdiv(lOc, 32);
    const long long gy = std::min<long long>(rows, 32768), gz = (rows + gy - 1) / gy;
    ProfScope ps_(h, "k_out_s_segs");
    BATOTP_LAUNCH_WARP(k_out_s_segs, dim3((unsigned)cdiv(Bo, 32), (unsigned)gy, (unsigned)gz), dim3(32, 8, 1), 0, h->stream,
                       w, lOc, Bo);
    g_check_launch();
    h->launches++;
  }
  LAUNCH_T(h, k_out_segs, Bo, w);
  double *cur = w.O5;
  int curCap = w.Oc;
  double *trqCur = w.Trq;
  if (fused_out(h)) {
    // the oversampled rows have no other consumer: evaluate, smooth and decimate in one pass (O5 is not touched)
    LAUNCH_T(h, k_out_smooth_plan, Bo, w);
    {
      const int wv = (int)c.c.out_smooth_fact;  // smooth()'s window half-width (util.cpp:261-263) when the row is long enough
      const int wMid = wv / 2 + wv % 2 - 1;
      const bool jointRows = c.c.path_type == BATOTP_JOINT;  // rows 0..J-1 driven, the others zero
      if (jointRows && wMid == 2 && c.J == 7)
        LAUNCH_TP(h, (k_out_eval_smooth_rows<2, 7>), lOs, Bo, w, w.OA);
      else if (jointRows && wMid == 2 && c.J == 6)
        LAUNCH_TP(h, (k_out_eval_smooth_rows<2, 6>), lOs, Bo, w, w.OA);
      else
      switch (wMid) {
        case 1: LAUNCH_TP(h, k_out_eval_smooth<1>, lOs, (long long)Bo * c.R, w, w.OA); break;
        case 2: LAUNCH_TP(h, k_out_eval_smooth<2>, lOs, (long long)Bo * c.R, w, w.OA); break;
        case 3: LAUNCH_TP(h, k_out_eval_smooth<3>, lOs, (long long)Bo * c.R, w, w.OA); break;
        case 4: LAUNCH_TP(h, k_out_eval_smooth<4>, lOs, (long long)Bo * c.R, w, w.OA); break;
        default: LAUNCH_TP(h, k_out_eval_smooth<5>, lOs, (long long)Bo * c.R, w, w.OA); break;  // others: generic path
      }
    }
    cur = w.OA;
    curCap = w.Os;
  } else {
    LAUNCH_TP(h, k_out_eval, lOc, (long long)Bo * c.R, w);
    apply_kinematics(h, 2);
    if (c.trqOn) {
      // re-spline theta(t) (and cart(t) for the parallel robot) to get time derivatives
      thomas_rows(h, w.O5, w.OM, Bo, b0, c.c.is_parallel ? c.R : c.J, c.R, 1, c.c.is_parallel ? 0 : 1);
      LAUNCH_TP(h, k_out_knot_eval, lOc, Bo, w);
      if (!c.c.is_parallel && (c.c.trig_mode == 2 || c.c.dyn_source == 1))
        host_dyn_rr_out(h);
      else
        LAUNCH_TP(h, k_out_trq, lOc, Bo, w, h->pm);
      cur = w.OA;
    }
    LAUNCH_T(h, k_out_smooth_plan, Bo, w);
    if (smooth_uniform_on(h) || c.c.is_auto_integ_res) {
      double *dst = (cur == w.O5) ? w.OA : w.O5;
      const int dstCap = (cur == w.O5) ? w.Os : w.Oc;
      LAUNCH_TP(h, k_out_smooth, std::min(curCap, dstCap), Bo, w, cur, dst);
      cur = dst;
      curCap = dstCap;
      trqCur = w.Trq2;
    }
  }
  LAUNCH_T(h, k_out_final_plan, Bo, w);
  // natural splines of the rows for the final resample (ba.cpp:1889-1915; used where isReinterp).
  // OM has at least the capacity of `cur` by construction (Os == Oc whenever cur can be O5 here).
  const bool needRe = (c.c.out_res < c.c.integ_res) || c.c.is_auto_integ_res;
  if (needRe) {
    thomas_rows(h, cur, w.OM, Bo, b0, c.R, c.R, 2, 0);
    if (c.trqOn) thomas_rows(h, trqCur, w.TrqM, Bo, b0, c.J, MAXD, 2, 0);
  }
  const bool strictQuat = (c.C == 7 && c.c.trig_mode != 0);
  const int rp = row_pitch(h), hp = hist_pitch(h);
  const long long *rag = nullptr;
  long long rag0 = 0;
  if (h->ragged) {
    // ragged layout: the chunk's block offsets were computed on the host from the sweep results (plan_ragged: the
    // output length is a function of the step count) and uploaded once; the sub-chunk's blocks are packed back to
    // back in the staging set, i.e. relative to the first of them
    rag = h->w.ragOff + b0;
    rag0 = h->ragOffHost[b0];
    h->ragBase[h->curSet] = h->ragChunkBase + rag0;
    h->ragTotal[h->curSet] = h->ragOffHost[b0 + Bo] - rag0;
  }
  float *cartDst = h->ragged ? (float *)nullptr : h->d_cartOut;
  if (c.c.robot_type == BATOTP_GENJNT && c.C != 7 && c.Cin <= MAXD && !c.trqOn && !h->d_outD && rp > 0 && Bo > 0) {
    // generic robot, float rows only: warp-per-tile staging through shared memory (k_out_pack_rows)
    const long long rows = cdiv(Bo, OP_WARPS);
    const long long gy = std::min<long long>(rows, 32768), gz = (rows + gy - 1) / gy;
    ProfScope ps_(h, "k_out_pack_rows");
    BATOTP_LAUNCH_WARP(k_out_pack_rows, dim3((unsigned)cdiv(rp, 32), (unsigned)gy, (unsigned)gz),
                       dim3(32, OP_WARPS, 1), 0, h->stream, w, cur, w.OM, h->d_thetaOut, cartDst, rp, rag, rag0, rp, Bo);
    g_check_launch();
    h->launches++;
  } else {
    LAUNCH_PT(h, k_out_pack, std::max(w.OutC, rp), Bo, w, cur, w.OM, trqCur, w.TrqM, h->d_thetaOut, cartDst,
              h->d_trqOut, strictQuat ? h->d_cartOutD : (double *)nullptr, h->d_outD, rp, rag, rag0);
  }
  LAUNCH_PT(h, k_pack_hist, std::max(w.Sc, hp), Bo, w, h->d_histOut, hp);
  h->phase = 4;
}

}  // namespace

// FP64 pipe peak of this device, measured (MEASURED_PEAKS.json has no FP64 entry): 16 independent
// accumulator chains per thread, either fused multiply-adds (2 flop each) or alternating
// multiply / add (1 flop each: the ceiling of a -fmad=false kernel).  Returns TFLOP/s.
#ifndef BATOTP_HOST_EMU
template <bool FMA>
__global__ void __launch_bounds__(256) k_fp64_peak(double *out, int iters, double a, double b) {
  double x[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) x[q] = 1.0 + 1e-9 * (threadIdx.x + q);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      if (FMA)
        x[q] = __fma_rn(x[q], a, b);
      else {
        x[q] = __dmul_rn(x[q], a);
        x[q] = __dadd_rn(x[q], b);
      }
    }
  }
  double sacc = 0;
#pragma unroll
  for (int q = 0; q < 16; ++q) sacc += x[q];
  out[blockIdx.x * blockDim.x + threadIdx.x] = sacc;
}
#endif

// Self-test of the shared-reciprocal division (k_sweep.cuh sdiv::) against the compiler's '/':
// pseudo-random operand pairs (full-range mantissas; exponents concentrated in the working range,
// a share of them near and beyond the fast-path window so that the fallback is exercised too).
#ifndef BATOTP_HOST_EMU
__device__ __forceinline__ unsigned long long st_mix(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double st_operand(unsigned long long bits, unsigned long long sel) {
  const unsigned long long mant = bits & 0x000FFFFFFFFFFFFFull, sign = bits & 0x8000000000000000ull;
  long long e;
  const unsigned k = (unsigned)(sel & 15u);
  if (k < 12)
    e = 1023 + (long long)((sel >> 8) % 81) - 40;  // 2^-40 .. 2^40
  else if (k < 14)
    e = 1023 + (long long)((sel >> 8) % 2001) - 1000;  // anywhere
  else
    e = ((sel >> 8) & 1) ? (long long)((sel >> 16) % 80) : 2046 - (long long)((sel >> 16) % 80);  // extremes
  if (e < 0) e = 0;
  if (e > 2046) e = 2046;
  return __longlong_as_double((long long)(sign | ((unsigned long long)e << 52) | mant));
}
__global__ void k_selftest_div(unsigned long long seed, int perThread, unsigned long long *mismatch,
                               unsigned long long *fastTaken) {
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long bad = 0, fast = 0;
  unsigned long long z = st_mix(seed ^ (t * 0xD1342543DE82EF95ull));
  for (int it = 0; it < perThread; ++it) {
    const unsigned long long ba = st_mix(z), bb = st_mix(ba), sel = st_mix(bb);
    z = sel;
    const double b = st_operand(bb, sel >> 20);
    const sdiv::Rcp rc = sdiv::prep(b);
    // several numerators per denominator, like the kernels use it
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double a = st_operand(st_mix(ba + k), sel + k * 977);
      const double q1 = sdiv::div(a, b, rc);
      const double q2 = a / b;
      if (__double_as_longlong(q1) != __double_as_longlong(q2) && !(q1 != q1 && q2 != q2)) bad++;
      const double q0 = __dmul_rn(a, rc.r);
      const double q = __fma_rn(rc.r, __fma_rn(-b, q0, a), q0);
      if (rc.ok && sdiv::exp_ok(a) && sdiv::exp_ok(q)) fast++;
      // the tabulated-reciprocal form of the Thomas recurrences: r = RN(1/b) formed by an IEEE division
      const sdiv::Rcp rt = {1.0 / b, rc.ok};
      const double q3 = sdiv::div(a, b, rt);
      if (__double_as_longlong(q3) != __double_as_longlong(q2) && !(q3 != q3 && q2 != q2)) bad++;
      // the constant-divisor form used by the spline coefficients
      const double s1 = sdiv::div6(a), s2 = a / 6.0;
      if (__double_as_longlong(s1) != __double_as_longlong(s2) && !(s1 != s1 && s2 != s2)) bad++;
    }
  }
  atomicAdd(mismatch, bad);
  atomicAdd(fastTaken, fast);
}
#endif

// Self-test of the strict trigonometry (k_trig.cuh) against the libm of the host this process runs on: the device
// evaluates sin / cos at pseudo-random arguments (several magnitudes: the working range of joint angles in radians,
// the Taylor and table branches, the pi/2 reductions, tiny arguments), the host repeats them with its own sin / cos.
__host__ __device__ inline unsigned long long tt_mix(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__host__ __device__ inline double tt_arg(unsigned long long seed, long long i) {
  const unsigned long long a = tt_mix(seed ^ ((unsigned long long)i * 0xD1342543DE82EF95ull)), b = tt_mix(a);
  const double u = (double)(a >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;  // [-1, 1)
  switch ((unsigned)(b & 15u)) {
    case 0: return u * 0.13;        // TAYLOR_SIN
    case 1: case 2: case 3: return u * 0.86;   // table branch
    case 4: case 5: case 6: return u * 2.43;   // pi/2 - |x|
    case 7: case 8: case 9: case 10: return u * 3.4;  // +-195 degrees: every joint range of the shipped robots
    case 11: case 12: return u * 13.0;         // reduce_sincos, a few turns
    case 13: return u * 1.0e4;
    case 14: return u * 1.0e8;                 // up to the end of the ported range
    default: {                                 // tiny and subnormal-adjacent magnitudes
      const int e = (int)((b >> 8) % 60);
      return ldexp(u, -e);
    }
  }
}
__global__ void k_selftest_trig(unsigned long long seed, long long first, int n, int mode, double *xs, double *ss,
                                double *cs) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const double x = tt_arg(seed, first + t);
  const Trig tg{mode};
  xs[t] = x;
  ss[t] = tg.s(x);
  cs[t] = tg.c(x);
}

// Self-test of the branch-free bracket update of the sweep kernel (Bisect::step_any) against the reference-shaped
// one (Bisect::step, ba.cpp:1270-1321) on random problems "feasible iff sdot^2 <= T": same result code and same next
// candidate after every verification, same settled value and iteration count.  kinds: thresholds all over the
// range, at / next to a candidate, zero, negative start.  One problem per call; runs as a device kernel in the
// product build and sequentially in the host emulation.
__host__ __device__ inline bool bisect_problem_differs(unsigned long long seed, long long k) {
  unsigned long long z = tt_mix(seed ^ ((unsigned long long)k * 0xD1342543DE82EF95ull));
  auto rnd = [&]() {
    z = tt_mix(z);
    return (double)(z >> 11) * (1.0 / 9007199254740992.0);
  };
  const int kind = (int)(rnd() * 8);
  double start = exp((rnd() - 0.5) * 40.0);
  if (kind == 5) start = -start;
  if (kind == 6) start = 0.0;
  double T = start * start * exp(-rnd() * (kind == 1 ? 60.0 : 6.0));
  if (kind == 2) T = 0.0;                          // nothing but sdot = 0 is feasible
  if (kind == 3) T = -1.0;                         // nothing is feasible: the bracket collapses or 100 passes
  if (kind == 4) T = start * start * (1.0 + 1e-3);  // feasible at once
  if (kind == 7) {                                 // threshold exactly at a candidate of the sequence
    Bisect p;
    p.begin(start);
    const int stop = 1 + (int)(rnd() * 12);
    for (int it = 0; it < stop; ++it)
      if (p.step(true) != 0) break;
    T = p.sdotCur * p.sdotCur;
  }
  Bisect a, b;
  a.begin(start);
  b.begin(start);
  int ra = 0, rb = 0, guard = 0;
  while (ra == 0 && rb == 0 && guard++ < 300) {
    const bool va = !(a.sdotCur * a.sdotCur <= T), vb = !(b.sdotCur * b.sdotCur <= T);
    ra = a.step(va);
    rb = b.step_any(vb);
    if (ra != rb) return true;
    if (ra == 0 && a.sdotCur != b.sdotCur && !(a.sdotCur != a.sdotCur && b.sdotCur != b.sdotCur)) return true;
  }
  const double inB = (rb == 2) ? start : b.sdotCur;  // what the sweep kernel forms after the loop
  if (ra != rb || a.nIter != b.nIter) return true;
  return a.sdotIn != inB && !(a.sdotIn != a.sdotIn && inB != inB);
}
__global__ void k_selftest_bisect(unsigned long long seed, long long first, int n, unsigned long long *bad) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  if (bisect_problem_differs(seed, first + t)) {
#ifdef BATOTP_HOST_EMU
    (*bad)++;
#else
    atomicAdd(bad, 1ull);
#endif
  }
}

// ----------------------------------------------------------------------------- C ABI
extern "C" {

int batotp_cuda_device_count(void) {
#ifndef BATOTP_HOST_EMU
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
#else
  return 1;
#endif
}

int batotp_cuda_create(int device, batotp_handle *out) {
  if (!out) return -1;
  *out = nullptr;
#ifndef BATOTP_HOST_EMU
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    fprintf(stderr, "batotp_cuda: no CUDA device available (this library has no CPU fallback)\n");
    return -1;
  }
  if (device < 0 || device >= n) return -1;
  if (cudaSetDevice(device) != cudaSuccess) return -1;
#endif
  batotp_ctx *h = new batotp_ctx();
  h->device = device;
  memset(&h->w, 0, sizeof(h->w));
#ifndef BATOTP_HOST_EMU
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->copyStream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return -1;
  }
  for (int q = 0; q < NSETS; ++q)
    if (cudaEventCreateWithFlags(&h->evOut[q], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->evCopied[q], cudaEventDisableTiming) != cudaSuccess) {
      delete h;
      return -1;
    }
#endif
  h->pm = make_pmat();
  *out = h;
  return 0;
}

int batotp_cuda_destroy(batotp_handle h) {
  if (!h) return -1;
  if (h->helper) batotp_cuda_destroy(h->helper);
  h->helper = nullptr;
  free_ws(h);
  free_out(h);
  g_free(h->d_cN);
  for (int k = 0; k < 2; ++k) {
    free_inset(h->inSet[k]);
#ifndef BATOTP_HOST_EMU
    if (h->inSet[k].ev) cudaEventDestroy(h->inSet[k].ev);
#endif
  }
#ifndef BATOTP_HOST_EMU
  cudaStreamDestroy(h->stream);
  cudaStreamDestroy(h->copyStream);
  for (int q = 0; q < NSETS; ++q) {
    if (h->evOut[q]) cudaEventDestroy(h->evOut[q]);
    if (h->evCopied[q]) cudaEventDestroy(h->evCopied[q]);
  }
#endif
  delete h;
  return 0;
}

const char *batotp_cuda_last_error(batotp_handle h) { return h ? h->err.c_str() : "null handle"; }

int batotp_cuda_set_chunk(batotp_handle h, int chunk) {
  if (!h || chunk < 0) return -1;
  h->chunk = chunk;
  h->learnedChunk = 0;
  return 0;
}

long batotp_cuda_launch_count(batotp_handle h) { return h ? h->launches : 0; }

int batotp_cuda_fp64_peak(batotp_handle h, double *tflops_fma, double *tflops_nofma) {
#ifndef BATOTP_HOST_EMU
  if (!h) return -1;
  try {
    CU_CHECK(cudaSetDevice(h->device));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    const int blocks = sms * 8, threads = 256, iters = 4096;
    double *d = (double *)g_alloc((size_t)blocks * threads * 8);
    cudaEvent_t e0, e1;
    CU_CHECK(cudaEventCreate(&e0));
    CU_CHECK(cudaEventCreate(&e1));
    double best[2] = {0, 0};
    for (int mode = 0; mode < 2; ++mode)
      for (int rep = 0; rep < 6; ++rep) {
        CU_CHECK(cudaEventRecord(e0, h->stream));
        if (mode == 0)
          k_fp64_peak<true><<<blocks, threads, 0, h->stream>>>(d, iters, 1.0000001, 1e-9);
        else
          k_fp64_peak<false><<<blocks, threads, 0, h->stream>>>(d, iters, 1.0000001, 1e-9);
        CU_CHECK(cudaEventRecord(e1, h->stream));
        CU_CHECK(cudaEventSynchronize(e1));
        float ms = 0;
        CU_CHECK(cudaEventElapsedTime(&ms, e0, e1));
        const double flop = (double)blocks * threads * iters * 16 * 2;  // both variants: 2 flop per chain step
        const double tf = flop / (ms * 1e-3) * 1e-12;
        if (rep > 0 && tf > best[mode]) best[mode] = tf;
      }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    g_free(d);
    if (tflops_fma) *tflops_fma = best[0];
    if (tflops_nofma) *tflops_nofma = best[1];
    return 0;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
#else
  if (tflops_fma) *tflops_fma = 0;
  if (tflops_nofma) *tflops_nofma = 0;
  return h ? 0 : -1;
#endif
}

int batotp_cuda_selftest_div(batotp_handle h, unsigned long long seed, long long n, long long *mismatches,
                             long long *fast_path_taken) {
#ifndef BATOTP_HOST_EMU
  if (!h) return -1;
  try {
    CU_CHECK(cudaSetDevice(h->device));
    unsigned long long *d = (unsigned long long *)g_alloc(16);
    g_zero(d, 16, h->stream);
    const int threads = 256, perThread = 256;
    long long blocks = (n / 3 + (long long)threads * perThread - 1) / ((long long)threads * perThread);
    if (blocks < 1) blocks = 1;
    k_selftest_div<<<(unsigned)blocks, threads, 0, h->stream>>>(seed, perThread, d, d + 1);
    CU_CHECK(cudaGetLastError());
    unsigned long long out[2] = {0, 0};
    g_d2h(out, d, 16, h->stream);
    g_sync(h->stream);
    g_free(d);
    if (mismatches) *mismatches = (long long)out[0];
    if (fast_path_taken) *fast_path_taken = (long long)out[1];
    return 0;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
#else
  (void)seed;
  (void)n;
  if (mismatches) *mismatches = 0;
  if (fast_path_taken) *fast_path_taken = 0;
  return h ? 0 : -1;
#endif
}

int batotp_cuda_selftest_trig(batotp_handle h, unsigned long long seed, long long n, long long *mismatches,
                              int *variant) {
  if (!h || n < 0) return -1;
  try {
#ifndef BATOTP_HOST_EMU
    CU_CHECK(cudaSetDevice(h->device));
#endif
    const int mode = host_libm_uses_fma() ? 3 : 1;
    if (variant) *variant = mode;
    const int M = 1 << 22;
    double *d = (double *)g_alloc((size_t)3 * M * 8);
    std::vector<double> hb((size_t)3 * M);
    long long bad = 0;
    const unsigned nth = std::max(1u, std::min(std::thread::hardware_concurrency(), 64u));
    for (long long at = 0; at < n; at += M) {
      const int m = (int)std::min<long long>(M, n - at);
      LAUNCH_T(h, k_selftest_trig, m, seed, at, m, mode, d, d + M, d + 2 * (size_t)M);
      g_d2h(hb.data(), d, (size_t)3 * M * 8, h->stream);
      g_sync(h->stream);
      std::vector<long long> part(nth, 0);
      auto work = [&](unsigned tid) {
        long long b = 0;
        for (int i = (int)tid; i < m; i += (int)nth) {
          const double x = hb[i];
          const double sr = sin(x), cr = cos(x);  // the host libm: what the reference calls
          if (memcmp(&sr, &hb[(size_t)M + i], 8) != 0) b++;
          if (memcmp(&cr, &hb[2 * (size_t)M + i], 8) != 0) b++;
        }
        part[tid] = b;
      };
      std::vector<std::thread> th;
      for (unsigned t = 1; t < nth; ++t) th.emplace_back(work, t);
      work(0);
      for (auto &x : th) x.join();
      for (long long v : part) bad += v;
    }
    g_free(d);
    if (mismatches) *mismatches = bad;
    return 0;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}

int batotp_cuda_set_keep_f64(batotp_handle h, int on) {
  if (!h) return -1;
  h->keepF64 = on != 0;
  return 0;
}

int batotp_cuda_stats(batotp_handle h, double *out, int n) {
  if (!h || !out) return -1;
  const double v[6] = {h->sweepMs, (double)h->sweepLaunches, (double)h->cntVerify, (double)h->cntSteps,
                       (double)h->cntTraj, (double)h->launches};
  for (int i = 0; i < n && i < 6; ++i) out[i] = v[i];
  return 0;
}
int batotp_cuda_sweep_log(batotp_handle h, double *ms, int *n_traj, int *kernel, int cap) {
  if (!h) return -1;
  const int n = (int)h->sweepLog.size();
  for (int i = 0; i < n && i < cap; ++i) {
    if (ms) ms[i] = h->sweepLog[i].ms;
    if (n_traj) n_traj[i] = h->sweepLog[i].B;
    if (kernel) kernel[i] = h->sweepLog[i].kernel;
  }
  return n;
}
int batotp_cuda_stats_reset(batotp_handle h) {
  if (!h) return -1;
  h->sweepMs = 0;
  h->sweepLaunches = 0;
  h->sweepLog.clear();
  h->cntVerify = h->cntSteps = h->cntTraj = 0;
  h->launches = 0;
  return 0;
}
int batotp_cuda_set_profile(batotp_handle h, int on) {
  if (!h) return -1;
  h->profile = on != 0;
  h->prof.clear();
  return 0;
}
int batotp_cuda_profile_dump(batotp_handle h, char *buf, int cap) {
  if (!h || !buf || cap < 1) return -1;
  std::string o;
  char line[256];
  for (const auto &kv : h->prof) {
    snprintf(line, sizeof line, "%s,%.4f,%ld\n", kv.first.c_str(), kv.second.first, kv.second.second);
    o += line;
  }
  const int n = (int)std::min(o.size(), (size_t)cap - 1);
  memcpy(buf, o.data(), n);
  buf[n] = 0;
  return n;
}
#ifdef BATOTP_HOST_EMU
// TEST-ONLY (host emulation build): counters of the sweep kernel's float filters, see k_sweep.cuh
int batotp_emu_filter_stats(long long *out, int n, int reset) {
  for (int i = 0; i < n && i < 16; ++i) out[i] = g_emu_filter[i];
  if (reset) memset(g_emu_filter, 0, sizeof(g_emu_filter));
  return 0;
}
// TEST-ONLY: perturb the float reciprocal of the sweep kernel's models by k ulps (see f_rcp)
int batotp_emu_set_rcp_ulps(int k) {
  g_emu_rcp_ulps = k;
  return 0;
}
// TEST-ONLY: the planner's footprints of the chunk workspace the context holds - its chunk arrays, the output arrays
// of its first sub-chunk, the bytes per trajectory - beside the bytes actually held and the trajectories the chunk
// arrays were allocated for: {chunk, out, perTraj, wsBytes, outBytes, B}
int batotp_emu_workspace_plan(batotp_handle h, size_t *out) {
  if (!h || !out) return -1;
  const Footprints fp = footprints(h, h->wsHeld);
  const size_t v[6] = {fp.chunk, fp.out, fp.perTraj, h->wsBytes, h->outBytes, (size_t)h->wsHeld.B};
  memcpy(out, v, sizeof v);
  return 0;
}
#endif
int batotp_cuda_selftest_bisect(batotp_handle h, unsigned long long seed, long long n, long long *mismatches) {
  if (!h || n < 0) return -1;
  try {
#ifndef BATOTP_HOST_EMU
    CU_CHECK(cudaSetDevice(h->device));
#endif
    unsigned long long *d = (unsigned long long *)g_alloc(8);
    g_zero(d, 8, h->stream);
    const int M = 1 << 24;
    for (long long at = 0; at < n; at += M) {
      const int m = (int)std::min<long long>(M, n - at);
      LAUNCH_T(h, k_selftest_bisect, m, seed, at, m, d);
    }
    unsigned long long bad = 0;
    g_d2h(&bad, d, 8, h->stream);
    g_sync(h->stream);
    g_free(d);
    if (mismatches) *mismatches = (long long)bad;
    return 0;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}

int batotp_cuda_timer(batotp_handle h, int which, double *elapsed_ms) {
#ifndef BATOTP_HOST_EMU
  if (!h || which < 0 || which > 1) return -1;
  try {
    CU_CHECK(cudaSetDevice(h->device));
    if (!h->evT[0]) {
      CU_CHECK(cudaEventCreate(&h->evT[0]));
      CU_CHECK(cudaEventCreate(&h->evT[1]));
    }
    CU_CHECK(cudaEventRecord(h->evT[which], h->stream));
    if (which == 1) {
      CU_CHECK(cudaEventSynchronize(h->evT[1]));
      float ms = 0;
      CU_CHECK(cudaEventElapsedTime(&ms, h->evT[0], h->evT[1]));
      if (elapsed_ms) *elapsed_ms = ms;
    }
    return 0;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
#else
  (void)which;
  if (elapsed_ms) *elapsed_ms = 0;
  return h ? 0 : -1;
#endif
}

// The sweep kernel keeps one trajectory per lane resident for a whole sweep (SMs x SW_MIN_BLOCKS CTAs of
// SW_NT lanes) and its duration hardly depends on how many lanes are filled (it is bound by the latency of
// one trajectory), so a chunk larger than the resident lanes leaves a thin second wave running on its own and
// a smaller one wastes lanes: automatic chunking takes full waves and leaves the remainder to the last chunk
// (measured on the 131072-path step: 817 ms against 828 ms for three equal chunks).
static int auto_chunk(batotp_handle h, int B) {
  int sms = 148;
#ifndef BATOTP_HOST_EMU
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
#else
  (void)h;
#endif
  const int lanes = sms * SW_MIN_BLOCKS * SW_NT;
  return std::max(SW_NT, std::min(lanes, cdiv(B, SW_NT) * SW_NT));
}

static int load_chunk(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in, int first, int B) {
#ifndef BATOTP_HOST_EMU
  CU_CHECK(cudaSetDevice(h->device));
#endif
  if (cfg) {
    set_cfg(h, cfg);
    if (check_cfg(h) != 0) return -1;
  }
  if (!h->haveCfg) {
    h->err = "no configuration loaded";
    return -1;
  }
  if (!(in->theta_f32 || in->theta_f64 || in->cart_f32 || in->cart_f64)) {
    h->err = "batch input holds neither joint nor Cartesian data";
    return -1;
  }
  if ((in->theta_f32 || in->cart_f32) && (in->theta_f64 || in->cart_f64)) {
    h->err = "mixing float32 and float64 payloads is not supported";
    return -1;
  }
  if (in->n0_max < 1) {
    h->err = "batch input: n0_max must be at least 1";
    return -1;
  }
  if (in->n0)  // caller-supplied lengths index the payload rows: never trust them past the row pitch
    for (int b = 0; b < B; ++b)
      if (in->n0[first + b] < 1 || in->n0[first + b] > in->n0_max) {
        char buf[160];
        snprintf(buf, sizeof buf, "batch input: n0[%d] = %d is outside 1..n0_max (%d)", first + b, in->n0[first + b],
                 in->n0_max);
        h->err = buf;
        return -1;
      }
  stage_inputs(h, in, first, B);
  h->phase = 1;
  return 0;
}

// one chunk through interpInputData with capacity planning / retry
static int chunk_interp_input(batotp_handle h, bool haveN0) {
  int Nc = std::max(h->hwNc, h->n0max + 8);
  bool plan = (h->hwNc == 0);
  for (int attempt = 0; attempt < 8; ++attempt) {
    // the step capacity follows the grid the planning pass finds (a sweep takes about as many steps as the
    // grid has points; twice that leaves room), or what earlier chunks needed
    const int Sc = std::min(h->maxSteps, std::max(h->hwSc, h->stepHint > 0 ? h->stepHint : std::max(1024, 2 * Nc)));
    ensure_ws(h, h->B, Nc, Sc);
    h->w.B = h->B;
    const int need = do_interp_input(h, haveN0, plan);
    if (need > 0) {  // planning pass asked for more room
      Nc = need;
      plan = false;
      continue;
    }
    int gridCap = 0;
    const int mx = read_plan_max(h, &gridCap);
    if (gridCap) {
      Nc = std::max((int)(Nc * 1.5), (int)(mx * 1.125) + 64);
      plan = false;
      continue;
    }
    h->hwNc = std::max(h->hwNc, Nc);
    return 0;
  }
  h->err = "grid capacity retry limit reached";
  return -1;
}

// Ragged result layout: the output length of a trajectory follows from its forward sweep (ba.cpp:1664-1685 output
// resolution, 1838-1871 smoothing / decimation, 1873-1921 final sizes - the arithmetic of k_out_plan,
// k_out_smooth_plan and k_out_final_plan), so the host lays the chunk's blocks out as soon as the sweeps are back:
// prefix sums -> w.ragOff, and the chunk's place in the caller's buffers from the shared counter.  (A trajectory
// the output phase rejects later keeps its reserved block and reports n_out = 0.)
static void plan_ragged(batotp_handle h) {
  const batotp_cfg &c = h->cfg.c;
  const int B = h->B;
  h->ragOffHost.resize((size_t)B + 1);
  long long acc = 0;
  for (int b = 0; b < B; ++b) {
    h->ragOffHost[b] = acc;
    const TrajState &s = h->hst[b];
    if (s.status & ST_FATAL_MASK) continue;
    const double outResT = c.out_res;
    double outRes = outResT, outSmooth = c.out_smooth_fact;
    bool re = false;
    if (outRes < s.integRes) {
      re = true;
      outRes = s.integRes;
      outSmooth *= std::max(outResT / outRes, 1.);
    }
    const double tLast = s.tStep * (double)(s.nFwd - 1);
    int nOver = (int)(outSmooth * std::ceil(tLast / outRes + 1.));
    nOver = std::max(nOver, 4);
    const int nSm = outSmooth > 1.5 ? std::max((int)((nOver - 1) / outSmooth) + 1, 4) : nOver;
    const int nOut = re ? std::max((int)(std::ceil(tLast / outResT)), 4) : nSm;
    acc += nOut;
  }
  h->ragOffHost[B] = acc;
  h->ragChunkBase = h->ragNext->fetch_add(acc);
  g_h2d(h->w.ragOff, h->ragOffHost.data(), ((size_t)B + 1) * sizeof(long long), h->stream);
}

static int chunk_sweeps_output(batotp_handle h, bool haveN0) {
  for (int attempt = 0; attempt < 10; ++attempt) {
    if (do_sweeps(h) != 0) return -1;
    h->hst.resize(h->B);
    g_d2h(h->hst.data(), h->w.st, (size_t)h->B * sizeof(TrajState), h->stream);
    g_sync(h->stream);
#ifndef BATOTP_HOST_EMU
    if (h->sweepPending) {
      float ms = 0;
      CU_CHECK(cudaEventElapsedTime(&ms, h->evS0, h->evS1));
      h->sweepMs += ms;
      if (h->sweepLog.size() < 4096) h->sweepLog.push_back({(double)ms, h->B, h->lastSweepKernel});
      h->sweepPending = false;
    }
#endif
    bool stepCap = false;
    int mxF = 0, nCap = 0;
    for (int b = 0; b < h->B; ++b) {
      if (h->hst[b].status & ST_STEP_CAP) {
        stepCap = true;
        nCap++;
      }
      mxF = std::max(mxF, std::max(h->hst[b].nFwd, h->hst[b].nRev));
    }
    h->mxSteps = mxF;
    if (stepCap && h->collectStragglers && nCap <= std::max(8, h->B / 64) && h->w.Sc < h->maxSteps) {
      // a few trajectories outgrew a capacity that serves the rest of the chunk: they keep BATOTP_ST_STEP_CAP for
      // now (the output phase skips them) and are re-run together after the chunks of the batch, instead of the
      // whole chunk being redone with twice the capacity for their sake
      for (int b = 0; b < h->B; ++b)
        if ((h->hst[b].status & ST_STEP_CAP) && !(h->hst[b].status & (ST_FATAL_MASK & ~ST_STEP_CAP)))
          h->stragglers.push_back(h->chunkFirst + b);
      h->stragglerSc = std::max(h->stragglerSc, h->w.Sc);
      stepCap = false;
    }
    if (!stepCap) {
      for (int b = 0; b < h->B; ++b) {
        const TrajState &t = h->hst[b];
        if (t.status & ST_FATAL_MASK) continue;
        h->cntVerify += t.nVerify;
        h->cntSteps += (t.nRev - 1) + (t.nFwd - 1);
        h->cntTraj++;
      }
      h->hwSc = std::max(h->hwSc, std::min(h->w.Sc, (int)(mxF * 1.25) + 64));
      if (h->ragged) plan_ragged(h);
      return 0;
    }
    // A trajectory that crawls (e.g. an infeasible path whose bisection keeps failing, ba.cpp:1307-1319) runs
    // until maxIntegTime in the reference.  The step capacity follows it up to maxSteps; beyond that the
    // trajectory keeps BATOTP_ST_STEP_CAP (reported as not optimised) instead of holding the batch hostage.
    if ((long long)h->w.Sc * 2 > (long long)h->maxSteps) {
      for (int b = 0; b < h->B; ++b) {
        const TrajState &t = h->hst[b];
        if (t.status & ST_FATAL_MASK) continue;
        h->cntVerify += t.nVerify;
        h->cntSteps += (t.nRev - 1) + (t.nFwd - 1);
        h->cntTraj++;
      }
      h->hwSc = std::max(h->hwSc, h->w.Sc);  // the next chunks start with this capacity: one pass each
      if (h->ragged) plan_ragged(h);
      return 0;
    }
    // grow the step capacity and redo the chunk from the start (the status word is sticky)
    const int Sc = h->w.Sc * 2;
    const int Nc = h->w.Nc;
    ensure_ws(h, h->B, Nc, Sc);
    h->w.B = h->B;
    const int need = do_interp_input(h, haveN0, false);
    (void)need;
  }
  h->err = "step capacity retry limit reached";
  return -1;
}

int batotp_cuda_load(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in) {
  if (!h || !in) return -1;
  try {
    h->lastHaveN0 = in->n0 != nullptr;
    h->inSet[0].src = h->inSet[1].src = nullptr;
    h->rowPitch = h->histPitch = 0;  // phase-wise calls pack at the device capacities
    h->ragged = false;
    h->chunkFirst = 0;
    h->collectStragglers = false;
    const int rc = load_chunk(h, cfg, in, 0, in->B);
    if (rc == 0) g_sync(h->stream);  // the caller's arrays are free again when this call returns
    return rc;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}
int batotp_cuda_interp_input(batotp_handle h) {
  if (!h || h->phase < 1) return -1;
  try {
    if (h->cfg.c.is_interp_only) return do_interp_only(h, h->lastHaveN0);  // result ready for batotp_cuda_fetch
    return chunk_interp_input(h, h->lastHaveN0);
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}
int batotp_cuda_sweeps(batotp_handle h) {
  if (!h || h->phase < 2) return -1;
  try {
    return chunk_sweeps_output(h, h->lastHaveN0);
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}
int batotp_cuda_interp_output(batotp_handle h) {
  if (!h || h->phase < 3) return -1;
  try {
    if (h->B > h->outChunk) h->outChunk = h->B;  // the phase-wise API keeps one sub-chunk resident
    do_interp_output(h, 0, h->B);
    g_sync(h->stream);
    return 0;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}

// per-trajectory scalars of the chunk trajectories [b0, b0+Bo) -> the caller's arrays (host arrays: synchronous,
// small; device arrays: one kernel on the context's stream)
static void fetch_scalars(batotp_handle h, batotp_batch_out *out, int first, int b0, int Bo) {
  const Ws &w = h->w;
  if (out->on_device) {
    const ScalarOut so{out->status, out->n_rev, out->n_fwd, out->n_out, out->n_cart_out, out->n_grid,
                       out->t_total, out->t_rev, out->s_last_sec, out->out_sres};
    LAUNCH_T(h, k_fetch_scalars, Bo, w, so, first, b0, Bo);
    return;
  }
  h->hst.resize(h->B);
  g_d2h(h->hst.data() + b0, w.st + b0, (size_t)Bo * sizeof(TrajState), h->stream);
  g_sync(h->stream);
  for (int bl = 0; bl < Bo; ++bl) {
    const TrajState &s = h->hst[b0 + bl];
    const int g = first + b0 + bl;
    if (out->status) out->status[g] = s.status;
    if (out->n_rev) out->n_rev[g] = s.nRev;
    if (out->n_fwd) out->n_fwd[g] = s.nFwd;
    if (out->n_out) out->n_out[g] = (s.status & ST_FATAL_MASK) ? 0 : s.nOut;
    if (out->n_cart_out) out->n_cart_out[g] = (s.status & ST_FATAL_MASK) ? 0 : s.nCartOut;
    if (out->n_grid) out->n_grid[g] = s.nPtsC;
    if (out->t_total) out->t_total[g] = s.tFwd;
    if (out->t_rev) out->t_rev[g] = s.tRev;
    if (out->s_last_sec) out->s_last_sec[g] = s.sLastSec;
    if (out->out_sres) out->out_sres[g] = s.sresOut;
  }
}

// one block of packed rows (rows x `have` points at device pitch dp) -> the caller's block at pitch `want`:
// a single contiguous copy when the staging set was packed at the caller's pitch
static void copy_rows(void *dst, size_t want, const void *src, size_t dp, size_t rows, size_t es, cudaStream_t cs) {
  if (want == dp)
    g_d2h(dst, src, rows * dp * es, cs);
  else
    g_d2h_2d(dst, want * es, src, dp * es, std::min(want, dp) * es, rows, cs);
}

// packed float32 rows / histories / flags of the current output sub-chunk -> the caller's buffers (host or
// device memory), enqueued on stream `cs` (the staging set is the one selected when the sub-chunk was packed)
static void fetch_rows(batotp_handle h, batotp_batch_out *out, int first, cudaStream_t cs) {
  const DevCfg &c = h->cfg;
  const Ws &w = h->w;
  const int Bo = w.Bo, g0 = first + w.b0;
  const size_t oc = (size_t)out->out_cap, rp = (size_t)row_pitch(h);
  if (h->ragged) {
    // the sub-chunk's blocks, back to back in the staging set -> their place in the caller's buffer, in one copy;
    // the offsets were computed when the sub-chunk was packed (do_interp_output)
    const long long base = h->ragBase[h->curSet], total = h->ragTotal[h->curSet];
    if (base + total > out->ragged_cap) {
      char buf[160];
      snprintf(buf, sizeof buf, "ragged_cap (%lld points) is too small: %lld points needed so far", out->ragged_cap,
               base + total);
      throw Err{buf};
    }
    for (int bl = 0; bl < Bo; ++bl) out->row_offset[g0 + bl] = h->ragChunkBase + h->ragOffHost[w.b0 + bl];
    if (out->theta_out && total > 0)
      g_d2h(out->theta_out + (size_t)base * c.J, h->d_thetaOut, (size_t)total * c.J * 4, cs);
    if (out->trq_out && c.trqOn && total > 0)
      g_d2h(out->trq_out + (size_t)base * c.J, h->d_trqOut, (size_t)total * c.J * 4, cs);
  } else {
    if (out->theta_out && oc > 0)
      copy_rows(out->theta_out + (size_t)g0 * c.J * oc, oc, h->d_thetaOut, rp, (size_t)Bo * c.J, 4, cs);
    if (out->trq_out && oc > 0 && c.trqOn)
      copy_rows(out->trq_out + (size_t)g0 * c.J * oc, oc, h->d_trqOut, rp, (size_t)Bo * c.J, 4, cs);
  }
  if (out->cart_out && oc > 0 && c.Cin > 0 && !(c.C == 7 && c.c.trig_mode != 0))
    copy_rows(out->cart_out + (size_t)g0 * c.Cin * oc, oc, h->d_cartOut, rp, (size_t)Bo * c.Cin, 4, cs);
  const size_t hc = (size_t)out->hist_cap, hp = (size_t)hist_pitch(h);
  if (out->hist && hc > 0) copy_rows(out->hist + (size_t)g0 * 4 * hc, hc, h->d_histOut, hp, (size_t)Bo * 4, 4, cs);
  if (out->flags && hc > 0)
    copy_rows(out->flags + (size_t)g0 * 2 * hc, hc, w.flags + (size_t)w.b0 * 2 * w.Sc, (size_t)w.Sc, (size_t)Bo * 2, 1, cs);
}

// copy the results of the current output sub-chunk [w.b0, w.b0+w.Bo) to the caller's buffers;
// `first` = index of the resident chunk's first trajectory in the caller's batch
static void fetch_sub(batotp_handle h, batotp_batch_out *out, int first) {
  const DevCfg &c = h->cfg;
  const Ws &w = h->w;
  ProfScope ps_(h, "copy_d2h(fetch)");
  const bool strictQuatOut = out->cart_out && out->out_cap > 0 && c.Cin > 0 && c.C == 7 && c.c.trig_mode != 0;
  if (out->on_device && strictQuatOut)
    throw Err{"batotp_batch_out.on_device: axis-angle rows in strict-trig mode are finished on the host; use trig_mode 0"};
  fetch_scalars(h, out, first, w.b0, w.Bo);
  fetch_rows(h, out, first, h->stream);
  if (strictQuatOut) host_q2aa_out(h, out, first + w.b0);
  g_sync(h->stream);
}

int batotp_cuda_fetch(batotp_handle h, batotp_batch_out *out) {
  if (!h || !out || h->phase < 4) return -1;
  try {
    fetch_sub(h, out, 0);
    return 0;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}

// one resident chunk [at, at+B) of the caller's batch through the whole path
static void process_chunk(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in, batotp_batch_out *out,
                          int at, int B, int nextB) {
  if (load_chunk(h, cfg, in, at, B) != 0) throw Err{h->err};
  h->lastHaveN0 = in->n0 != nullptr;
  h->chunkFirst = at;
  // the staging sets are packed at the caller's pitches: a sub-chunk then leaves in one contiguous copy
  h->ragged = out->row_offset != nullptr && h->ragNext != nullptr;
  h->rowPitch = (!h->ragged && (out->theta_out || out->cart_out || out->trq_out) && out->out_cap > 0) ? out->out_cap : 0;
  h->histPitch = (out->hist && out->hist_cap > 0) ? out->hist_cap : 0;
  if (nextB > 0 && !in->on_device && !h->profile) {
    // the host rows of the next chunk travel while this one is computed
    try {
      issue_inputs(h, in, at + B, nextB, h->curIn ^ 1, h->copyStream, true);
    } catch (const Err &) {
      h->inSet[h->curIn ^ 1].src = nullptr;  // no room for the second set: that chunk is staged when its turn comes
    }
  }
  if (h->cfg.c.is_interp_only) {  // ba.cpp:139-159: re-sample only
    if (do_interp_only(h, h->lastHaveN0) != 0) throw Err{h->err};
    fetch_sub(h, out, at);
    return;
  }
  if (chunk_interp_input(h, h->lastHaveN0) != 0) throw Err{h->err};
  if (h->beforeSweeps) h->beforeSweeps();
  if (h->copiesPending && out->flags && out->hist_cap > 0) {
    // the switching flags travel straight out of the chunk workspace, which the sweeps overwrite: when they were
    // asked for, the sweeps queue up behind the previous chunk's copies.  (Rows and histories leave from the
    // staging sets, which only the output phase touches: their copies go on beside the next chunk's sweeps.)
    for (int q = 0; q < NSETS; ++q)
      if (h->setBusy[q]) {
        g_stream_wait(h->stream, h->evCopied[q]);
        h->setBusy[q] = false;
      }
    h->copiesPending = false;
  }
  if (chunk_sweeps_output(h, h->lastHaveN0) != 0) throw Err{h->err};
  if (h->onSweepsDone) h->onSweepsDone();
  {
      const DevCfg &c = h->cfg;
      const bool strictQuatOut = out->cart_out && out->out_cap > 0 && c.Cin > 0 && c.C == 7 && c.c.trig_mode != 0;
      if (strictQuatOut || h->profile) {  // host post-processing per sub-chunk / serialised measurement
        for (int b0 = 0; b0 < B; b0 += h->outChunk) {
          do_interp_output(h, b0, std::min(h->outChunk, B - b0));
          fetch_sub(h, out, at);
        }
      } else {
        // rows of sub-chunk k go to the host on the copy stream while sub-chunk k+1 is computed into the
        // other staging set
        for (int b0 = 0; b0 < B; b0 += h->outChunk) {
          ensure_out(h, std::min(h->outChunk, B - b0));
          const int q = h->setNext;
          h->setNext = (q + 1) % NSETS;
          if (h->setBusy[q]) g_stream_wait(h->stream, h->evCopied[q]);  // the set's last rows have reached the host
          select_out_set(h, q);
          do_interp_output(h, b0, std::min(h->outChunk, B - b0));
          g_event_record(h->evOut[q], h->stream);
          g_stream_wait(h->copyStream, h->evOut[q]);
          fetch_rows(h, out, at, h->copyStream);
          g_event_record(h->evCopied[q], h->copyStream);
          h->setBusy[q] = true;
        }
        fetch_scalars(h, out, at, 0, B);
        h->copiesPending = true;  // waited for before the next chunk's sweeps, or before the call returns
      }
  }
}

int batotp_cuda_set_tail_overlap(batotp_handle h, int on) {
  if (!h) return -1;
  h->tailOverlap = on != 0;
  return 0;
}

// drain both streams of a context without raising (error paths)
static void sync_quiet(batotp_handle h) {
#ifndef BATOTP_HOST_EMU
  cudaStreamSynchronize(h->stream);
  cudaStreamSynchronize(h->copyStream);
#endif
  h->copiesPending = false;
}

// trajectories per round of the sweep kernel a chunk of B trajectories of this configuration would take (0: not known)
static int sweep_round_capacity(batotp_handle h, const batotp_cfg *cfg, int B) {
  if (!h->haveCfg || memcmp(&h->cfg.c, cfg, sizeof(batotp_cfg)) != 0) return 0;  // learnt for another configuration
  return h->sweepCap[group_sweep(h->cfg, h->sweepKernel, B) ? 1 : 0];
}

// The chunks [0, mainB) of a batch on context h, one after the other (out-of-memory: smaller chunks)
static void run_chunks(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in, batotp_batch_out *out,
                       int from, int mainB, int &chunk, bool &first) {
  for (int at = from; at < mainB;) {
    // A sweep launch lasts whole rounds of the trajectories it keeps resident (it is bound by the latency of one
    // trajectory), so a chunk of 1.5 rounds pays for 2 (CSPR3DOF on the B200: 9472 paths per round; memory allows
    // 14464..19072 per chunk).  Once the occupancy of the configuration's kernel is known, a chunk that is not the
    // last one of its batch is cut to whole rounds - what it leaves moves on to the next chunk - and the last one when
    // its final round would be less than a quarter full (a fuller round is cheaper than another chunk).
    auto whole_rounds = [&](int n, int left) {
      const int cap = h->chunk == 0 ? sweep_round_capacity(h, cfg, n) : 0;  // (an explicit chunk setting is taken literally)
      if (cap <= 0 || n <= cap) return n;
      return (left > n || n % cap < cap / 4) ? n / cap * cap : n;
    };
    const int B = whole_rounds(std::min(chunk, mainB - at), mainB - at);
    const int nextB = whole_rounds(std::min(chunk, mainB - at - B), mainB - at - B);
    const double tC0 = g_trace() ? g_now_ms() : 0;
    if (g_trace())
      fprintf(stderr, "[batotp] chunk at %d: %d paths (chunk setting %d, round capacity %d; capB %d capNc %d capSc %d; alloc %.1f ms free %.1f ms so far)\n",
              at, B, chunk, sweep_round_capacity(h, cfg, B), h->wsHeld.B, h->wsHeld.Nc, h->wsHeld.Sc, g_allocMs, g_freeMs);
    try {
      process_chunk(h, first ? cfg : nullptr, in, out, at, B, nextB);
    } catch (const Err &e) {
      // a workspace did not fit (long paths, many rows): release everything and go on with smaller chunks
      if (!e.oom) throw;
      if (g_trace()) fprintf(stderr, "[batotp]   refused after %.1f ms: %s (fits: %d, alloc phase %d)\n", g_now_ms() - tC0, e.msg.c_str(), e.fitB, h->allocPhase);
      g_sync(h->stream);
      g_sync(h->copyStream);
      h->copiesPending = false;
      h->inSet[0].src = h->inSet[1].src = nullptr;
      if (!e.planned) {  // (a refusal by the planner has left the workspaces of the previous chunks / calls as they were)
        free_ws(h);
        free_out(h);
      }
      const int chunk0 = chunk, out0 = h->outChunk;
      if (e.fitB > 0 && e.fitB < B)  // the workspace planner knows what fits
        chunk = std::max(1, e.fitB >= SW_NT ? e.fitB / SW_NT * SW_NT : e.fitB);
      else if (h->allocPhase == 1 && std::min(h->outChunk, B) > 1)
        h->outChunk = std::max(1, std::min(h->outChunk, B) / 2);
      else
        chunk = std::max(1, B > 2 * SW_NT ? (B / 2 + SW_NT - 1) / SW_NT * SW_NT : B / 2);
      if ((chunk >= chunk0 || chunk >= B) && h->outChunk >= std::min(out0, B)) throw;  // nothing left to shrink
      continue;
    }
    if (g_trace()) fprintf(stderr, "[batotp]   done in %.1f ms (Nc %d Sc %d, stragglers so far %zu)\n", g_now_ms() - tC0, h->w.Nc, h->w.Sc, h->stragglers.size());
    first = false;
    at += B;
  }
}

// Stragglers.  The trajectories that outgrew the step capacity of their chunk (chunk_sweeps_output) are gathered
// into one small batch and run again with four times that capacity (growing further, up to maxSteps, by the
// ordinary capacity retries of a chunk); their results replace the BATOTP_ST_STEP_CAP placeholders in the caller's
// arrays.  Trajectories are independent, so the results are the ones a single large-capacity pass would give.
static void run_stragglers(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in, batotp_batch_out *out) {
  std::vector<int> idx = h->stragglers;
  h->stragglers.clear();
  std::sort(idx.begin(), idx.end());
  idx.erase(std::unique(idx.begin(), idx.end()), idx.end());
  const int n = (int)idx.size();
  if (n == 0) return;
  const DevCfg &c = h->cfg;
  const int n0 = in->n0_max, J = c.J, Cin = c.Cin;
  const bool f64 = (in->theta_f64 || in->cart_f64);
  const size_t es = f64 ? 8 : 4;
  const void *th = f64 ? (const void *)in->theta_f64 : (const void *)in->theta_f32;
  const void *ca = f64 ? (const void *)in->cart_f64 : (const void *)in->cart_f32;
  const size_t thRow = (size_t)J * n0 * es, caRow = (size_t)Cin * n0 * es;
  // ---- gather the inputs (host rows into host vectors, resident rows into a device block)
  std::vector<char> hTh, hCa;
  std::vector<double> hTs, hTres(n);
  std::vector<int> hN0(n);
  void *dTh = nullptr, *dCa = nullptr;
  double *dTs = nullptr;
  struct Guard {
    void *&a, *&b;
    double *&c;
    ~Guard() {
      g_free(a);
      g_free(b);
      g_free(c);
    }
  } guard{dTh, dCa, dTs};
  if (in->on_device) {
    if (th) dTh = g_alloc((size_t)n * thRow);
    if (ca) dCa = g_alloc((size_t)n * caRow);
    if (in->timestamp) dTs = (double *)g_alloc((size_t)n * n0 * 8);
  } else {
    if (th) hTh.resize((size_t)n * thRow);
    if (ca) hCa.resize((size_t)n * caRow);
    if (in->timestamp) hTs.resize((size_t)n * n0);
  }
  for (int k = 0; k < n; ++k) {
    const size_t g = (size_t)idx[k];
    hTres[k] = in->tres ? in->tres[g] : in->tres_all;
    hN0[k] = in->n0 ? in->n0[g] : n0;
    if (in->on_device) {
      if (th) g_d2d((char *)dTh + k * thRow, (const char *)th + g * thRow, thRow, h->stream);
      if (ca) g_d2d((char *)dCa + k * caRow, (const char *)ca + g * caRow, caRow, h->stream);
      if (in->timestamp) g_d2d(dTs + (size_t)k * n0, in->timestamp + g * n0, (size_t)n0 * 8, h->stream);
    } else {
      if (th) memcpy(hTh.data() + k * thRow, (const char *)th + g * thRow, thRow);
      if (ca) memcpy(hCa.data() + k * caRow, (const char *)ca + g * caRow, caRow);
      if (in->timestamp) memcpy(hTs.data() + (size_t)k * n0, in->timestamp + g * n0, (size_t)n0 * 8);
    }
  }
  batotp_batch_in in2 = *in;
  in2.B = n;
  in2.n0 = in->n0 ? hN0.data() : nullptr;
  in2.tres = hTres.data();
  const void *pTh = in->on_device ? dTh : (th ? (void *)hTh.data() : nullptr);
  const void *pCa = in->on_device ? dCa : (ca ? (void *)hCa.data() : nullptr);
  in2.theta_f32 = f64 ? nullptr : (const float *)pTh;
  in2.cart_f32 = f64 ? nullptr : (const float *)pCa;
  in2.theta_f64 = f64 ? (const double *)pTh : nullptr;
  in2.cart_f64 = f64 ? (const double *)pCa : nullptr;
  in2.timestamp = in->timestamp ? (in->on_device ? dTs : hTs.data()) : nullptr;
  // ---- results into host vectors with the caller's pitches
  // (ragged layout: the stragglers are computed into a pitched temporary wide enough for the step ceiling and
  // appended to the caller's buffer block by block)
  const bool ragOut = out->row_offset != nullptr;
  const size_t oc = ragOut ? (size_t)final_cap(h, h->maxSteps, 0) : (size_t)out->out_cap, hc = (size_t)out->hist_cap;
  std::vector<int> oI[6];
  std::vector<double> oD[4];
  for (auto &v : oI) v.assign(n, 0);
  for (auto &v : oD) v.assign(n, 0.0);
  std::vector<float> oTh, oCa, oTq, oHist;
  std::vector<unsigned char> oFl;
  batotp_batch_out o2;
  memset(&o2, 0, sizeof(o2));
  o2.out_cap = (int)oc;
  o2.hist_cap = out->hist_cap;
  o2.status = oI[0].data();
  o2.n_rev = oI[1].data();
  o2.n_fwd = oI[2].data();
  o2.n_out = oI[3].data();
  o2.n_cart_out = oI[4].data();
  o2.n_grid = oI[5].data();
  o2.t_total = oD[0].data();
  o2.t_rev = oD[1].data();
  o2.s_last_sec = oD[2].data();
  o2.out_sres = oD[3].data();
  if (out->theta_out && oc) { oTh.assign((size_t)n * J * oc, 0.f); o2.theta_out = oTh.data(); }
  if (out->cart_out && oc && Cin > 0) { oCa.assign((size_t)n * Cin * oc, 0.f); o2.cart_out = oCa.data(); }
  if (out->trq_out && oc && c.trqOn) { oTq.assign((size_t)n * J * oc, 0.f); o2.trq_out = oTq.data(); }
  if (out->hist && hc) { oHist.assign((size_t)n * 4 * hc, 0.f); o2.hist = oHist.data(); }
  if (out->flags && hc) { oFl.assign((size_t)n * 2 * hc, 0); o2.flags = oFl.data(); }
  // ---- run them as one chunk with a larger step capacity; the capacity marks of the batch are put back after
  std::atomic<long long> *const keepRag = h->ragNext;
  h->ragNext = nullptr;  // the temporary is pitched
  const int keepHwSc = h->hwSc;
  const bool keepCollect = h->collectStragglers;
  h->collectStragglers = false;
  h->hwSc = (int)std::min<long long>(h->maxSteps, (long long)std::max(h->stragglerSc, 1024) * 4);
  h->stragglerSc = 0;
  g_sync(h->stream);
  g_sync(h->copyStream);
  h->copiesPending = false;
  h->inSet[0].src = h->inSet[1].src = nullptr;
  try {
    int chunk2 = n;
    bool first2 = true;
    run_chunks(h, cfg, &in2, &o2, 0, n, chunk2, first2);  // (with its out-of-memory retries)
    g_sync(h->copyStream);
    g_sync(h->stream);
    h->copiesPending = false;
  } catch (...) {
    h->hwSc = keepHwSc;
    h->collectStragglers = keepCollect;
    h->ragNext = keepRag;
    throw;
  }
  h->hwSc = keepHwSc;
  h->collectStragglers = keepCollect;
  h->ragNext = keepRag;
  free_ws(h);  // the large-capacity workspace is not what the next batch needs
  free_out(h);
  // ---- scatter
  auto put = [&](void *dst, const void *src, size_t bytes) {
    if (!bytes) return;
    if (out->on_device)
      g_h2d(dst, src, bytes, h->stream);
    else
      memcpy(dst, src, bytes);
  };
  for (int k = 0; k < n; ++k) {
    const size_t g = (size_t)idx[k];
    int *const dI[6] = {out->status, out->n_rev, out->n_fwd, out->n_out, out->n_cart_out, out->n_grid};
    double *const dD[4] = {out->t_total, out->t_rev, out->s_last_sec, out->out_sres};
    for (int q = 0; q < 6; ++q)
      if (dI[q]) put(dI[q] + g, &oI[q][k], sizeof(int));
    for (int q = 0; q < 4; ++q)
      if (dD[q]) put(dD[q] + g, &oD[q][k], sizeof(double));
    if (ragOut) {
      const long long nn = oI[3][k];  // n_out
      const long long base = keepRag->fetch_add(nn);
      if (base + nn > out->ragged_cap) throw Err{"ragged_cap is too small for the re-run stragglers"};
      out->row_offset[g] = base;
      for (int r = 0; r < J; ++r) {
        if (o2.theta_out) memcpy(out->theta_out + (size_t)base * J + (size_t)r * nn, oTh.data() + ((size_t)k * J + r) * oc, (size_t)nn * 4);
        if (o2.trq_out) memcpy(out->trq_out + (size_t)base * J + (size_t)r * nn, oTq.data() + ((size_t)k * J + r) * oc, (size_t)nn * 4);
      }
    } else {
      if (o2.theta_out) put(out->theta_out + g * J * oc, oTh.data() + (size_t)k * J * oc, (size_t)J * oc * 4);
      if (o2.cart_out) put(out->cart_out + g * Cin * oc, oCa.data() + (size_t)k * Cin * oc, (size_t)Cin * oc * 4);
      if (o2.trq_out) put(out->trq_out + g * J * oc, oTq.data() + (size_t)k * J * oc, (size_t)J * oc * 4);
    }
    if (o2.hist) put(out->hist + g * 4 * hc, oHist.data() + (size_t)k * 4 * hc, 4 * hc * 4);
    if (o2.flags) put(out->flags + g * 2 * hc, oFl.data() + (size_t)k * 2 * hc, 2 * hc);
  }
  g_sync(h->stream);
}

// Tail overlap.  The sweep kernel is bound by the latency of one trajectory, so a last chunk that fills only a
// fraction of the resident lanes costs a whole sweep on its own (131072 paths = 2 full waves + 17408 paths).  When
// that tail fits into ONE sweep CTA per SM it leaves two thirds of every SM free: it is handed to a second context
// (own streams and workspaces, driven by one host thread): its input interpolation runs at once, its sweeps
// start when the sweeps of the first full chunk have completed, so that they run beside the bandwidth-bound
// output / input phases of the full chunks instead of after them.  Results are the same bytes either way (trajectories are independent).
int batotp_cuda_optimize_batch(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in,
                               batotp_batch_out *out) {
  if (!h || !cfg || !in || !out) return -1;
  std::atomic<long long> ragCounter{0};  // ragged layout: the next free point of the caller's row buffers
  h->ragNext = nullptr;
  if (out->row_offset) {
    if (out->on_device || out->cart_out || !out->theta_out || out->ragged_cap <= 0 || cfg->is_interp_only) {
      h->err = "ragged rows (row_offset): host buffers, theta_out (+ trq_out) only, cart_out = NULL, ragged_cap > 0, "
               "not with isInterpOnly";
      return -1;
    }
    h->ragNext = &ragCounter;
  }
  struct RagReset {
    batotp_ctx *h;
    ~RagReset() {
      h->ragNext = nullptr;
      h->ragged = false;
      if (h->helper) {
        h->helper->ragNext = nullptr;
        h->helper->ragged = false;
      }
    }
  } ragReset{h};
  bool first = true;
  int chunk = h->chunk > 0 ? h->chunk : auto_chunk(h, in->B);
  const int chunkAuto = chunk;
  // what the workspace planner allowed in the previous call of this configuration: start there (a refused first
  // attempt costs the staging of its inputs)
  const bool sameCfg = h->haveCfg && memcmp(&h->cfg.c, cfg, sizeof(batotp_cfg)) == 0;
  if (h->chunk == 0 && sameCfg && h->learnedChunk > 0) chunk = std::min(chunk, h->learnedChunk);
  if (!sameCfg) h->learnedChunk = 0;
  {
    // whole rounds of the sweep kernel (run_chunks): applied to the chunk setting itself when the occupancy is already
    // known, so that the tail below is what whole-round chunks leave over
    const int cap = h->chunk == 0 ? sweep_round_capacity(h, cfg, chunk) : 0;
    if (cap > 0 && chunk > cap && in->B > chunk) chunk = chunk / cap * cap;
  }
  int mainB = in->B, tail = 0;
  std::thread tailThread;
  std::mutex mu;
  std::condition_variable cv;
  int go = 0;  // 0 wait, 1 run the tail, 2 skip it
  struct { bool failed = false, oom = false; std::string msg; } tailRes;
  auto signal = [&](int v) {
    std::lock_guard<std::mutex> lk(mu);
    if (go == 0) go = v;
    cv.notify_all();
  };
  auto finish_tail = [&](int v) {  // every exit path: let the tail thread go (or skip) and wait for it
    h->onSweepsDone = nullptr;
    if (tailThread.joinable()) {
      signal(v);
      tailThread.join();
    }
  };
  try {
    h->inSet[0].src = h->inSet[1].src = nullptr;
    h->stragglers.clear();
    h->stragglerSc = 0;
    h->collectStragglers = !cfg->is_interp_only;
    if (h->tailOverlap && !h->profile && !out->on_device && !cfg->is_interp_only && in->B > chunk) {
      int sms = 148;
#ifndef BATOTP_HOST_EMU
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
#endif
      const int t = in->B % chunk;
      if (t > 0 && t <= sms * SW_NT) {
        if (!h->helper && batotp_cuda_create(h->device, &h->helper) != 0) h->helper = nullptr;
        if (h->helper) {
          tail = t;
          mainB = in->B - tail;
          batotp_ctx *hp = h->helper;
          hp->tailOverlap = false;
          hp->chunk = 0;
          hp->outChunk = h->outChunk;
          hp->maxSteps = h->maxSteps;
          if (hp->stepHint != h->stepHint) hp->hwSc = 0;
          hp->stepHint = h->stepHint;
          hp->keepF64 = h->keepF64;
          hp->sweepKernel = h->sweepKernel;
          hp->walkerKernel = h->walkerKernel;
          hp->dynFn = h->dynFn;
          hp->dynUser = h->dynUser;
          hp->ragNext = h->ragNext;
          hp->stragglers.clear();
          hp->stragglerSc = 0;
          hp->collectStragglers = true;
          h->onSweepsDone = [&]() { signal(1); };
          // the tail's input interpolation runs at once (beside that of the first full chunk); its sweeps wait
          // until the sweeps of the first full chunk have completed, so that they run beside output / input phases
          hp->beforeSweeps = [&]() {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return go != 0; });
            if (go != 1) throw Err{"tail chunk skipped"};
          };
          tailThread = std::thread([&, hp]() {
            try {
              hp->inSet[0].src = hp->inSet[1].src = nullptr;
              const bool same = hp->haveCfg && memcmp(&hp->cfg.c, cfg, sizeof(batotp_cfg)) == 0;
              process_chunk(hp, same ? nullptr : cfg, in, out, mainB, tail, 0);
              g_sync(hp->copyStream);
              hp->copiesPending = false;
              hp->beforeSweeps = nullptr;
            } catch (const Err &e) {
              hp->beforeSweeps = nullptr;
              tailRes.failed = true;
              tailRes.oom = e.oom;
              tailRes.msg = e.msg;
              sync_quiet(hp);
            } catch (...) {
              hp->beforeSweeps = nullptr;
              tailRes.failed = true;
              tailRes.msg = "unexpected exception in the tail chunk";
              sync_quiet(hp);
            }
          });
        }
      }
    }
    run_chunks(h, cfg, in, out, 0, mainB, chunk, first);
    if (h->chunk == 0 && chunk < chunkAuto) h->learnedChunk = chunk;  // the out-of-memory handling shrank it
    finish_tail(1);
    if (tail > 0) {
      batotp_ctx *hp = h->helper;
      h->sweepMs += hp->sweepMs;
      h->sweepLaunches += hp->sweepLaunches;
      h->sweepLog.insert(h->sweepLog.end(), hp->sweepLog.begin(), hp->sweepLog.end());
      h->cntVerify += hp->cntVerify;
      h->cntSteps += hp->cntSteps;
      h->cntTraj += hp->cntTraj;
      h->launches += hp->launches;
      batotp_cuda_stats_reset(hp);
      h->stragglers.insert(h->stragglers.end(), hp->stragglers.begin(), hp->stragglers.end());
      h->stragglerSc = std::max(h->stragglerSc, hp->stragglerSc);
      hp->stragglers.clear();
      if (tailRes.failed) {
        if (!tailRes.oom) throw Err{tailRes.msg};
        // no room for the second context's workspaces: release them and run the tail here
        free_ws(hp);
        free_out(hp);
        run_chunks(h, cfg, in, out, mainB, in->B, chunk, first);
      }
    }
    g_sync(h->copyStream);  // every row has reached the caller's buffers
    h->copiesPending = false;
    if (!h->stragglers.empty()) run_stragglers(h, cfg, in, out);
    h->collectStragglers = false;
    return 0;
  } catch (const Err &e) {
    finish_tail(2);
    h->collectStragglers = false;
    h->err = e.msg;
#ifndef BATOTP_HOST_EMU
    cudaStreamSynchronize(h->copyStream);
#endif
    h->copiesPending = false;
    return -1;
  } catch (...) {
    finish_tail(2);
    h->err = "unexpected exception in batotp_cuda_optimize_batch";
    return -1;
  }
}

int batotp_cuda_mvc_per_sample(batotp_handle h, double sdot_start, double *sdot_out, int cap) {
  if (!h || h->phase < 2 || !sdot_out) return -1;
  try {
    return run_mvc_per_sample(h, sdot_start, sdot_out, cap);
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}

int batotp_cuda_get_f64(batotp_handle h, const char *name, int traj, int row, double *buf, int cap) {
  if (!h || !name || h->phase < 2 || traj < 0 || traj >= h->B || row < 0 || cap < 0) return -1;
  try {
    const DevCfg &c = h->cfg;
    const Ws &w = h->w;
    {  // row must exist in the family the name selects
      const std::string nn(name);
      const bool thetaFam = nn.compare(0, 5, "theta") == 0 || nn == "trq_out" || nn[0] == 'a';
      const bool cartFam = nn.compare(0, 4, "cart") == 0;
      if ((thetaFam && row >= c.J) || (cartFam && row >= c.C)) return -1;
    }
    TrajState s;
    g_d2h(&s, w.st + traj, sizeof(TrajState), h->stream);
    g_sync(h->stream);
    const std::string n(name);
    const double *src = nullptr;
    size_t stride = 1;  // in doubles
    int len = 0;
    const size_t pst = (size_t)w.B * c.R, ast = (size_t)w.B * 4 * w.AD;
    auto prow = [&](const double *base, int r) { return base + (size_t)traj * c.R + r; };
    auto arow = [&](const double *base, int k, int r) { return base + (size_t)traj * 4 * w.AD + (size_t)k * w.AD + r; };
    if (n == "integ_res" || n == "t_step" || n == "t_total" || n == "t_rev") {
      // per-trajectory scalars of the sweeps (integRes may be the automatically chosen step, ba.cpp:493-556)
      const double v = n == "integ_res" ? s.integRes : (n == "t_step" ? s.tStep : (n == "t_total" ? s.tFwd : s.tRev));
      if (buf && cap > 0) buf[0] = v;
      return 1;
    }
    if ((n == "cartC_y" || n == "cartC_m") && c.R == c.J) {  // Cartesian rows that are not stored: zeros
      if (s.status & ST_FATAL_MASK) return 0;
      for (int i = 0; buf && i < std::min(s.nPtsC, cap); ++i) buf[i] = 0.0;
      return s.nPtsC;
    }
    if (n == "thetaC_y") { src = prow(w.P, row); stride = pst; len = s.nPtsC; }
    else if (n == "thetaC_m") { src = prow(w.M, row); stride = pst; len = s.nPtsC; }
    else if (n == "cartC_y") { src = prow(w.P, c.J + row); stride = pst; len = s.nPtsC; }
    else if (n == "cartC_m") { src = prow(w.M, c.J + row); stride = pst; len = s.nPtsC; }
    else if (n == "theta" && c.trqOn) { src = prow(w.Q, row); stride = pst; len = s.nPts; }
    else if (n == "cart" && c.trqOn) { src = prow(w.Q, c.J + row); stride = pst; len = s.nPts; }
    else if (n.size() == 2 && n[0] == 'a' && n[1] >= '1' && n[1] <= '4' && c.trqOn) { src = arow(w.A, n[1] - '1', row); stride = ast; len = s.nPts; }
    else if (n.size() == 5 && n[0] == 'a' && n.substr(2) == "C_m" && c.trqOn) { src = arow(w.AM, n[1] - '1', row); stride = ast; len = s.nPts; }
    else if (h->phase >= 3 && n == "s_rev") { src = w.hist + (size_t)traj * 4 * w.Sc + (w.Sc - s.nRev); len = s.nRev; }
    else if (h->phase >= 3 && n == "sdot_rev") { src = w.hist + (size_t)traj * 4 * w.Sc + w.Sc + (w.Sc - s.nRev); len = s.nRev; }
    else if (h->phase >= 3 && n == "s_fwd") { src = w.hist + (size_t)traj * 4 * w.Sc + 2 * (size_t)w.Sc; len = s.nFwd; }
    else if (h->phase >= 3 && n == "sdot_fwd") { src = w.hist + (size_t)traj * 4 * w.Sc + 3 * (size_t)w.Sc; len = s.nFwd; }
    else if (h->phase >= 4 && h->d_outD && traj >= w.b0 && traj < w.b0 + w.Bo &&
             (n == "theta_out" || n == "cart_out" || n == "trq_out")) {
      const int rows = c.J + c.C + c.J, bl = traj - w.b0;  // k_out_pack's layout of outD
      auto orow_ = [&](int r) { return h->d_outD + ((size_t)bl * rows + r) * w.OutC; };
      if (n == "theta_out") { src = orow_(row); len = s.nOut; }
      else if (n == "trq_out") { src = orow_(c.J + c.C + row); len = s.nOut; }
      else {
        len = s.nCartOut;
        if (c.C == 7 && row >= 3) {  // q2aaVect (ba.cpp:382-403) with the host libm
          if (s.status & ST_FATAL_MASK) return 0;
          std::vector<double> q((size_t)4 * std::max(len, 1));
          for (int k = 0; k < 4; ++k) g_d2h(q.data() + (size_t)k * len, orow_(c.J + 3 + k), (size_t)len * 8, h->stream);
          g_sync(h->stream);
          for (int i = 0; i < len && i < cap; ++i) {
            const double qq[4] = {q[i], q[(size_t)len + i], q[(size_t)2 * len + i], q[(size_t)3 * len + i]};
            double aa[3];
            q2aa_dev(qq, aa);
            if (buf) buf[i] = aa[row - 3];
          }
          return len;
        }
        src = orow_(c.J + row);
      }
    }
    else return -1;
    if (s.status & ST_FATAL_MASK) return 0;
    const int m = std::min(len, cap);
    if (buf && m > 0) {
      if (stride == 1)
        g_d2h(buf, src, (size_t)m * sizeof(double), h->stream);
      else
        g_d2h_2d(buf, sizeof(double), src, stride * sizeof(double), sizeof(double), (size_t)m, h->stream);
      g_sync(h->stream);
    }
    return len;
  } catch (const Err &e) {
    h->err = e.msg;
    return -1;
  }
}

int batotp_cuda_set_max_steps(batotp_handle h, int n) {
  if (!h || n < 1024) return -1;
  h->maxSteps = n;
  return 0;
}

int batotp_cuda_set_dyn_callback(batotp_handle h, batotp_dyn_fn fn, void *user) {
  if (!h) return -1;
  h->dynFn = fn;
  h->dynUser = user;
  return 0;
}

int batotp_cuda_set_sweep_kernel(batotp_handle h, int mode) {
  if (!h || mode < 0 || mode > 2) return -1;
  h->sweepKernel = mode;
  return 0;
}

int batotp_cuda_set_walker_kernel(batotp_handle h, int mode) {
  if (!h || mode < 0 || mode > 2) return -1;
  h->walkerKernel = mode;
  return 0;
}

int batotp_cuda_set_step_hint(batotp_handle h, int n) {
  if (!h || n < 0) return -1;
  h->stepHint = n;
  h->hwSc = 0;  // the hint replaces what earlier chunks have learnt
  return 0;
}

int batotp_cuda_set_out_chunk(batotp_handle h, int n) {
  if (!h || n < 1) return -1;
  h->outChunk = n;
  return 0;
}

}  // extern "C"
