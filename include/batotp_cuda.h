/* batotp_cuda.h — the extern "C" boundary of the B200-native Bisection Algorithm path.
 *
 * This layer does not exist in the reference (SURVEY §8b); it is what a host-language
 * binding of batotp's time-optimisation step binds to.  Every entry point replaces a
 * BATOTP::BA member (reference file:line cited on each); buffers are plain pointers
 * and sizes, caller-owned (pin them for full copy bandwidth), the return convention is
 * the reference's: 0 = ok, -1 = error (+ message via batotp_cuda_last_error).
 *
 * There is no CPU fallback: every call fails with -1 when no CUDA device is usable.
 */
#ifndef BATOTP_CUDA_H
#define BATOTP_CUDA_H

#include "batotp_cfg.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct batotp_ctx *batotp_handle;

/* per-trajectory status word (bit set); 0 = optimised.  Mirrors BA's -1 returns and
 * BA::ErrorOptimization (ba.h:176) without aborting the batch. */
#define BATOTP_ST_TOO_SHORT 1        /* ba.cpp:129-133,175-179 */
#define BATOTP_ST_IDENTICAL 2        /* ba.cpp:484-488 */
#define BATOTP_ST_SRES_SMALL 4       /* ba.cpp:607-611 */
#define BATOTP_ST_GRID_CAP 8         /* internal capacity; retried automatically */
#define BATOTP_ST_MAX_INTEG_TIME 16  /* ba.cpp:1117-1122 = BA::MAX_INTEGRATION_TIME */
#define BATOTP_ST_STEP_CAP 32        /* internal capacity; retried automatically up to batotp_cuda_set_max_steps */
#define BATOTP_ST_NUMERIC 64         /* NaN in a segment search (the reference would not return) */
#define BATOTP_ST_BISECT_FAIL 128    /* informational: ba.cpp:1307-1319 returned -1 somewhere (sweep ignores it) */
#define BATOTP_ST_DIV0 256           /* spline.cpp:82-86 */
#define BATOTP_ST_UNSUPPORTED 512    /* option outside the accelerated scope */
#define BATOTP_ST_FATAL_MASK (1 | 2 | 4 | 8 | 16 | 32 | 64 | 256 | 512)

/* ---- device enumeration / lifetime ---------------------------------------------------- */
int batotp_cuda_device_count(void);
/* one context per device and host thread; owns the chunk workspace in HBM */
int batotp_cuda_create(int device, batotp_handle *out);
int batotp_cuda_destroy(batotp_handle h);
const char *batotp_cuda_last_error(batotp_handle h);
/* trajectories resident per device pass (input interpolation + both sweeps run over the whole chunk; the
 * tables and histories of one chunk live in HBM).  0 (default) = automatic: chunks of the sweep kernel's
 * resident lanes (SMs x 3 CTAs x 128 = 56832 on a B200), the remainder in the last chunk */
int batotp_cuda_set_chunk(batotp_handle h, int chunk);
/* trajectories per interpOutputData pass inside a chunk (bounds the oversampled-output buffers); default 8192 */
int batotp_cuda_set_out_chunk(batotp_handle h, int n);
/* largest Runge-Kutta step capacity (per sweep) the automatic capacity retries grow to; default 65536.  A
 * trajectory that needs more steps (the reference would run it until maxIntegTime, ba.cpp:1117-1122) keeps
 * BATOTP_ST_STEP_CAP and is reported as not optimised; n >= 1024 */
int batotp_cuda_set_max_steps(batotp_handle h, int n);
/* which sweep kernel serves a chunk.  0 (default) = by chunk size; 1 = one trajectory per lane (k_sweep.cuh: fewest
 * issue slots per trajectory, for chunks that fill the device); 2 = a group of 8 (or 4) lanes per trajectory
 * (k_sweep_group.cuh: a fraction of the latency per Runge-Kutta stage, for small batches and single paths).  Both
 * produce the same bits. */
int batotp_cuda_set_sweep_kernel(batotp_handle h, int mode);
/* the strictly sequential walkers of interpInputData (cumulative norms of adjust_s, ba.cpp:423-446; the constant-ds
 * march of interpSpecial, ba.cpp:651-781).  0 (default) = by chunk size; 1 = one thread per trajectory (chunks that fill
 * the device); 2 = point-parallel norm increments + a group of 16 lanes per trajectory for the march (small chunks:
 * the walk is bound by the latency of one trajectory).  Both produce the same bits. */
int batotp_cuda_set_walker_kernel(batotp_handle h, int mode);
/* Runge-Kutta step capacity (per sweep) a chunk starts with; 0 (default) = automatic: max(1024, 2 x grid points),
 * then what earlier chunks of the same configuration needed.  Inside batotp_cuda_optimize_batch the few trajectories
 * of a chunk that outgrow the capacity ("stragglers", at most max(8, chunk/64)) are re-run together with a
 * larger one after the chunks of the batch; when more do, the chunk is redone with twice the capacity. */
int batotp_cuda_set_step_hint(batotp_handle h, int n);
/* tail overlap of batotp_cuda_optimize_batch (default on): when the last chunk of a batch fills at most one sweep
 * CTA per SM (<= SMs x 128 trajectories) it runs on a second context inside the library (own streams and
 * workspaces, one host thread), beside the output / input phases of the full chunks instead of after them.
 * Results are identical either way; 0 switches it off (one context, chunks strictly one after the other) */
int batotp_cuda_set_tail_overlap(batotp_handle h, int on);
/* number of kernels launched by this context since creation (for the benchmark's gpu_launches) */
long batotp_cuda_launch_count(batotp_handle h);
/* measurement hooks for bench.py.
 * _stats: out[0] device ms spent in the sweep kernel (CUDA events on the launching stream),
 *         out[1] sweep launches, out[2] constraint verifications (ba.cpp:1449 calls),
 *         out[3] RK steps, out[4] trajectories, out[5] all kernel launches — since the last reset.
 * _timer(which=0) records an event on the context's stream, _timer(which=1) records a second one,
 *         waits for it and returns the elapsed device milliseconds between the two. */
int batotp_cuda_stats(batotp_handle h, double *out, int n);
/* one record per sweep launch since the last reset (at most 4096 kept): device milliseconds, trajectories of the
 * chunk, kernel (1 = one trajectory per lane, 2 = a group of lanes per trajectory).  Returns the number of records. */
int batotp_cuda_sweep_log(batotp_handle h, double *ms, int *n_traj, int *kernel, int cap);
int batotp_cuda_stats_reset(batotp_handle h);
int batotp_cuda_timer(batotp_handle h, int which, double *elapsed_ms);
/* per-kernel device timing for tuning runs: when on, every launch is bracketed by CUDA events and waited
 * for (so the pipeline is serialised: never combine with a throughput measurement).
 * _profile_dump writes "kernel,total_ms,launches" lines into buf and returns the length. */
int batotp_cuda_set_profile(batotp_handle h, int on);
int batotp_cuda_profile_dump(batotp_handle h, char *buf, int cap);
/* measured FP64-pipe peak of the device in TFLOP/s: fused multiply-add chains, and separate
 * multiply + add chains (the ceiling of this library's -fmad=false kernels) */
int batotp_cuda_fp64_peak(batotp_handle h, double *tflops_fma, double *tflops_nofma);
/* device self-test: the kernels' shared-reciprocal division against the compiler's IEEE '/' on about n
 * pseudo-random operand pairs; reports bitwise mismatches (must be 0) and how many took the fast path */
int batotp_cuda_selftest_div(batotp_handle h, unsigned long long seed, long long n, long long *mismatches,
                             long long *fast_path_taken);

/* device self-test of the sweep kernel's branch-free bisection step (Bisect::step_any, k_sweep.cuh) against the
 * reference-shaped control flow of ba.cpp:1270-1321 on n random feasibility thresholds; mismatches must be 0 */
int batotp_cuda_selftest_bisect(batotp_handle h, unsigned long long seed, long long n, long long *mismatches);
/* device self-test of the strict trigonometry (cfg.trig_mode 1): the device port of the host libm's sin / cos
 * (robot.cpp:130-136, 196-199, 408-419 and util.cpp:544-549 call them) against the libm of the host this process
 * runs on, at n pseudo-random arguments over the working range and beyond; reports bitwise mismatches (must be 0
 * for trig_mode 1 to reproduce the reference on this host; otherwise use trig_mode 2) and the arithmetic variant
 * in use (1: products and sums rounded separately, 3: fused multiply-adds, as glibc selects on an FMA+AVX2 CPU) */
int batotp_cuda_selftest_trig(batotp_handle h, unsigned long long seed, long long n, long long *mismatches,
                              int *variant);

/* ---- dynamic models batotp does not have (SURVEY 8f rank 4) ----------------------------------
 * The reference evaluates tau = a1*sddot + a2*sdot^2 + a3*sdot + a4 through Robot::call_dynSerial (robot.cpp:349-360),
 * which knows the RR robot only; its README asks a user to add other models to robot.cpp.  Here the model is a point
 * function of the caller: with cfg.dyn_source = 1 and cfg.is_trq_on = 1 the library calls fn for every grid point of
 * every trajectory (findDynModel, ba.cpp:905-914: joint values and their s-derivatives in, a1..a4 out, n_joints
 * entries each) and again at the output sites (ba.cpp:1815-1825: time derivatives in; trq = a2 + a3 + a4), on the
 * host's cores between device stages; splines, sweeps and limits run on the device as for RR.  fn must be
 * thread-safe.  Serial mechanisms only. */
typedef void (*batotp_dyn_fn)(void *user, int n_joints, const double *theta, const double *thetaD,
                              const double *thetaD2, double *a1, double *a2, double *a3, double *a4);
int batotp_cuda_set_dyn_callback(batotp_handle h, batotp_dyn_fn fn, void *user);

/* ---- batch input: what BA::loadTrajectoryData leaves in Traj (ba.cpp:2206-2461) -------- */
typedef struct batotp_batch_in {
  int B;                  /* trajectories */
  int n0_max;             /* row pitch (points) of the payload arrays */
  const int *n0;          /* [B] points per path, or NULL: all n0_max   (always a HOST pointer) */
  const double *tres;     /* [B] tresInput per path, or NULL: tres_all  (always a HOST pointer) */
  double tres_all;
  /* BIN-file payload layout (ba.cpp:2283-2299): [B][coordinate][n0_max]; NULL = block absent.
   * float32 as in the files, or float64 for CSV-sourced paths (exactly one family non-NULL) */
  const float *theta_f32;
  const float *cart_f32;
  const double *theta_f64;
  const double *cart_f64;
  const double *timestamp; /* [B][n0_max] CSV timestamps or NULL (ba.cpp:98-127) */
  int on_device;           /* 1: the payload pointers are device pointers already resident in HBM */
} batotp_batch_in;

/* ---- batch output: what BA::writeOutputData would serialise (ba.cpp:2510-2759) --------- */
typedef struct batotp_batch_out {
  int out_cap;   /* in: row pitch (points) of theta_out/cart_out/trq_out */
  int hist_cap;  /* in: row pitch (points) of hist/flags */
  /* per trajectory [B]; any pointer may be NULL */
  int *status;
  int *n_rev, *n_fwd;    /* points of the reverse / forward s-sdot curves (switching counts) */
  int *n_out;            /* Traj::nPts after interpOutputData */
  int *n_cart_out;       /* length of the Cartesian rows (trajWriteBIN's is_cartFull test) */
  int *n_grid;           /* knots of the s-grid after interpInputData */
  double *t_total;       /* Traj::tTotalTraj (forward sweep) */
  double *t_rev;         /* reverse-sweep time */
  double *s_last_sec;    /* Traj::sLastSec */
  double *out_sres;      /* Traj::sres after interpOutputData */
  /* float32 rows in trajWriteBIN order */
  float *theta_out;      /* [B][nJoints][out_cap] */
  float *cart_out;       /* [B][nCart][out_cap] */
  float *trq_out;        /* [B][nJoints][out_cap] */
  float *hist;           /* [B][4][hist_cap]: s_rev, sdot_rev (ascending s), s_fwd, sdot_fwd  (sdotWrite) */
  unsigned char *flags;  /* [B][2][hist_cap]: per RK step, integration order:
                            bits0-2 sub-steps limited by a velocity limit/MVC (ba.cpp:1093),
                            bits3-5 sub-steps with an active bisection, bit6 isOn_sdot (ba.cpp:1211) */
  int on_device;         /* 1: the pointers above are device pointers */
  /* Ragged rows (optional; batotp_cuda_optimize_batch only).  With row_offset != NULL the float32 joint rows are
   * packed at their own length instead of the pitch out_cap: trajectory g's block is
   *     theta_out[row_offset[g] * nJoints ...] = [nJoints][n_out[g]]
   * - exactly the joint payload trajWriteBIN writes (ba.cpp:2617-2647) - and trq_out likewise; blocks are laid out in
   * completion order (row_offset says where), ragged_cap is the capacity of theta_out / trq_out in POINTS
   * (sum of n_out over the batch; the call fails when it does not suffice).  No padding crosses the host link.
   * cart_out must be NULL in this mode; host buffers only. */
  long long *row_offset; /* [B] out: first point of trajectory g's block */
  long long ragged_cap;  /* in: capacity in points */
} batotp_batch_out;

/* BA::optimize (ba.cpp:2538-2573) over a batch: interpInputData -> sweep(-1) -> sweep(+1) ->
 * interpOutputData for every path, chunked through the device. */
int batotp_cuda_optimize_batch(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in,
                               batotp_batch_out *out);

/* ---- phase-wise calls, mirroring batest's sequence (test/main.cpp:55-86) ---------------- */
/* They operate on one resident chunk (B <= chunk size) so that a BATOTP::BA facade can fill
 * Traj between calls.  batotp_cuda_load replaces loadTrajectoryData's hand-over,
 * _interp_input = BA::interpInputData (ba.cpp:95), _sweeps = BA::sweep x2 (ba.cpp:979; the
 * reverse pass must precede the forward pass, so both run in one launch),
 * _interp_output = BA::interpOutputData (ba.cpp:1661), _fetch = copy results out. */
int batotp_cuda_load(batotp_handle h, const batotp_cfg *cfg, const batotp_batch_in *in);
int batotp_cuda_interp_input(batotp_handle h);
int batotp_cuda_sweeps(batotp_handle h);
int batotp_cuda_interp_output(batotp_handle h);
int batotp_cuda_fetch(batotp_handle h, batotp_batch_out *out);

/* Derived product (SURVEY §8a A10): per-sample maximum-velocity curve on the s-grid, one
 * thread per (path, sample): the sweep's own per-point functions evaluated at every knot.
 * Call after batotp_cuda_interp_input.  sdot_out: [B][cap] host doubles. */
int batotp_cuda_mvc_per_sample(batotp_handle h, double sdot_start, double *sdot_out, int cap);

/* FP64 inspection of the resident chunk (tests, and Traj filling by the facade).
 * name: "theta","cart" (grid/out rows), "thetaC_y","thetaC_m","cartC_y","cartC_m" (spline knots /
 * second-derivative solution), "a1".."a4","a1C_m".."a4C_m", "s_rev","sdot_rev","s_fwd","sdot_fwd",
 * "theta_out","cart_out","trq_out" (FP64 before the float cast); scalars (length 1): "integ_res" (the step the
 * sweeps used: _integRes or the automatic one, ba.cpp:493-556), "t_step", "t_total", "t_rev".
 * Returns the length, or -1 for an unknown name / a row the configuration does not have. */
int batotp_cuda_get_f64(batotp_handle h, const char *name, int traj, int row, double *buf, int cap);

/* keep FP64 copies of the final rows on the device so that batotp_cuda_get_f64 can return
 * "theta_out"/"cart_out"/"trq_out" before the float cast (the facade fills Traj with them). */
int batotp_cuda_set_keep_f64(batotp_handle h, int on);

/* ---- host-side file formats, byte-compatible with the reference (no CUDA involved) ------ */
int batotp_read_config(const char *path, batotp_cfg *cfg, char *traj_file_name, int name_cap); /* BA::readConfigData ba.cpp:1942-2087 */
/* BA::trajReadBIN ba.cpp:2257-2312: rows are malloc'ed [coord][n0] float32 (NULL if the block is absent); free with batotp_free */
int batotp_read_traj_bin(const char *path, int n_joints, int n_cart, double *tres, int *n0, float **theta, float **cart);
/* BA::trajReadCSV ba.cpp:2322-2461: FP64 rows + timestamps; header names ';'-joined */
int batotp_read_traj_csv(const char *path, int n_joints, int n_cart, int is_generic, double *tres, int *n0,
                         double **theta, double **cart, double **timestamp, char *header, int header_cap);
void batotp_free(void *p);
/* BA::trajWriteBIN ba.cpp:2582-2651 (cart / trq NULL = block absent; pitch = row stride in points) */
int batotp_write_traj_bin(const char *path, double sres, unsigned n_pts, int n_joints, const float *theta, int n_cart,
                          const float *cart, const float *trq, int pitch);
/* BA::sdotWrite ba.cpp:2726-2759 */
int batotp_write_s_sdot(const char *path, double sres, int n_rev, const float *s_rev, const float *sdot_rev,
                        int n_fwd, const float *s_fwd, const float *sdot_fwd);
/* BA::trajWriteCSV ba.cpp:2660-2717 */
int batotp_write_traj_csv(const char *path, const char *header, double sres, int n_pts, int n_joints,
                          const float *theta, int n_cart, const float *cart, int pitch);

/* ---- batch writer: BA::writeOutputData (ba.cpp:2510-2528) for the trajectories of a batch result --------
 * `threads` writer threads serialise <dir>/traj_out_<index>.dat (trajWriteBIN, ba.cpp:2582-2651) and, when the
 * result carries the histories and is_sdotOut is set, <dir>/s-sdot_<index>.dat (sdotWrite, ba.cpp:2726-2759),
 * index = base_index + b printed as %07lld, for b in [first, first+count).  _submit returns at once; the arrays
 * of `out` must stay untouched until _wait returns, so a caller that alternates two result buffers overlaps
 * the file output of chunk k with batotp_cuda_optimize_batch on chunk k+1.  Trajectories that were not
 * optimised (fatal status) get no file, like the reference's early returns.  _wait returns -1 if a file failed. */
typedef struct batotp_writer *batotp_writer_handle;
int batotp_writer_create(const char *dir, int threads, batotp_writer_handle *out);
int batotp_writer_submit(batotp_writer_handle w, const batotp_cfg *cfg, const batotp_batch_out *out,
                         long long base_index, int first, int count);
int batotp_writer_wait(batotp_writer_handle w, long long *files_written, long long *files_failed);
int batotp_writer_destroy(batotp_writer_handle w);

#ifdef __cplusplus
}
#endif
#endif /* BATOTP_CUDA_H */
