/* cngp.h - C ABI of the B200-native GP slip-prediction hot path (corenav-GP).
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI for this path - it crosses two
 * ROS topics and one service - so each entry point below names the reference interface it replaces:
 *
 *   cngp_predict_batch          replaces GPy's GPRegression build + m.predict() loop as called from
 *                               core_navigation/script/gp_slip_node.py:35,47-50 (rows a3, a6), for B windows at once
 *   cngp_lml_grad_batch         replaces the objective/gradient evaluation inside m.optimize(),
 *                               gp_slip_node.py:36 (rows a3, a4), for C hyper-parameter candidates x B windows
 *   cngp_lml_grad_windows       the same objective with one hyper-parameter vector per window (the evaluation each
 *                               L-BFGS-B iteration of B concurrent m.optimize() calls makes)
 *   cngp_optimize_batch         replaces m.optimize() itself (gp_slip_node.py:36; paramz L-BFGS-B on softplus hypers)
 *   cngp_gp_slip_batch          replaces the whole callback gp_slip_node.py:16-63 (rows a1-a7): train split,
 *                               prediction grid, predict, mean[n:], sigma = 2 sqrt(var[n:])
 *   cngp_zupt_lookahead_batch   replaces the loop of GpPredictor::GPCallBack, gp_predictor/src/gp_predictor.cpp:58-130
 *                               (rows a9-a12), with the SetStopping response (core_navigation/srv/SetStopping.srv:1-7,
 *                               CoreNav.cpp:652-676) passed as plain arrays
 *   cngp_llh_to_enu             replaces GpPredictor::llh_to_enu, gp_predictor.cpp:144-178
 *   cngp_slip_record_batch      replaces the slip extraction + GP_Input recorder of CoreNav::Update, CoreNav.cpp:244-329
 *   cngp_ekf_context_batch      replaces insErrorStateModel_LNF / calc_Q (CoreNav.cpp:411-527) behind SetStopping
 *   cngp_chol_large*            the N = 32768 single-window factorisation of BASELINE.json configs[4] (same math as a3)
 *   cngp_*_ragged               the same entry points for windows of different sizes in one call (recorder output)
 *
 * Conventions: plain C, int status returns (0 = ok, negative = error; text via cngp_last_error), no exceptions
 * cross the ABI, caller-owned buffers, row-major, FP64.  Every array argument is either a HOST pointer or a DEVICE
 * pointer according to the `mem` argument of the call (CNGP_MEM_HOST / CNGP_MEM_DEVICE); host calls copy in and
 * out through the context's pinned staging area and return after the results are in the caller's buffers; device
 * calls are stream-ordered on the context's stream and return immediately (use cngp_sync).  One context per GPU;
 * a context is not thread-safe.  There is NO CPU fallback: without a CUDA device cngp_create fails.
 */
#ifndef CNGP_H_
#define CNGP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CNGP_VERSION 100

/* ---- status codes ---- */
#define CNGP_OK 0
#define CNGP_ERR_INVALID (-1)     /* bad argument */
#define CNGP_ERR_CUDA (-2)        /* CUDA runtime error, see cngp_last_error */
#define CNGP_ERR_UNSUPPORTED (-3) /* shape outside what the kernels cover */
#define CNGP_ERR_NOMEM (-4)

/* ---- memory space of the array arguments of a call ---- */
#define CNGP_MEM_HOST 0
#define CNGP_MEM_DEVICE 1

/* ---- kernel families (GPy names; gp_slip_node.py:31-34, "Kernel Selection/README.md":18-20) ---- */
#define CNGP_K_RBF 1         /* variance, lengthscale            sigma^2 exp(-r^2/2) */
#define CNGP_K_MAT32 2       /* variance, lengthscale */
#define CNGP_K_MAT52 3       /* variance, lengthscale */
#define CNGP_K_RATQUAD 4     /* variance, lengthscale, power     sigma^2 (1 + r^2/2)^-power */
#define CNGP_K_STDPERIODIC 5 /* variance, period, lengthscale    sigma^2 exp(-0.5 (sin(pi d/p)/l)^2) */
#define CNGP_K_BROWNIAN 6    /* variance */
#define CNGP_K_LINEAR 7      /* variance */
#define CNGP_K_BIAS 8        /* variance */
#define CNGP_K_WHITE 9       /* variance */
#define CNGP_OP_ADD 16
#define CNGP_OP_MUL 17
#define CNGP_MAX_OPS 32      /* postfix program length */
#define CNGP_MAX_PARAMS 24   /* kernel hyper-parameters (noise excluded) */
#define CNGP_MAX_N 256       /* batched windows: training points per window */

/* A composite covariance as a postfix program over the families above, e.g. "rbf*brownian" ->
 * {RBF, BROWNIAN, MUL}.  theta of a window = the leaf hyper-parameters in program order followed by the Gaussian
 * noise variance, so theta has n_params + 1 entries. */
typedef struct cngp_kernel {
  int32_t n_ops;
  int32_t ops[CNGP_MAX_OPS];
  int32_t n_params; /* filled by cngp_kernel_parse / cngp_kernel_finalize */
} cngp_kernel;

/* Parse "rbf*brownian", "se+periodic", "(rbf+linear)*brownian+white" ... (names as in the oracle / GPy). */
int cngp_kernel_parse(const char* text, cngp_kernel* out);
/* Validate a hand-filled program and compute n_params. */
int cngp_kernel_finalize(cngp_kernel* k);

typedef struct cngp_ctx cngp_ctx;

typedef struct cngp_config {
  int32_t device;            /* CUDA device ordinal */
  int32_t jitter_retry;      /* 0: a non-PD window gets status < 0 and NaN outputs; 1: GPy jitchol ladder
                                (mean(diag)*1e-6, x10, 5 tries) - status = tries used */
  int64_t scratch_bytes;     /* device scratch for factors (0 = default 2 GiB); windows are processed in chunks */
  int32_t precision;         /* CNGP_PRECISION_F64 (default; 1e-9 parity) or CNGP_PRECISION_F32 (1e-4): the predictive
                                mean / variance phase of cngp_predict_batch / cngp_gp_slip_batch runs on the TF32 tensor
                                cores with the 3xTF32 split (FP32-level accuracy); factorisation, LML and every other
                                entry point stay FP64.  Arrays at the ABI are double in both modes. */
  int32_t reserved[7];
} cngp_config;

#define CNGP_PRECISION_F64 0
#define CNGP_PRECISION_F32 1

void cngp_default_config(cngp_config* cfg);
int cngp_create(const cngp_config* cfg, cngp_ctx** out);
void cngp_destroy(cngp_ctx* ctx);
const char* cngp_last_error(cngp_ctx* ctx); /* ctx may be NULL: last create error */
int cngp_sync(cngp_ctx* ctx);
/* Make the context launch on an existing cudaStream_t (e.g. torch's current stream; 0 is the legacy default
 * stream), or back on the context's own non-blocking stream when use_own != 0. */
int cngp_set_stream(cngp_ctx* ctx, void* cuda_stream, int32_t use_own);
/* Switch the precision mode of an existing context (see cngp_config.precision). */
int cngp_set_precision(cngp_ctx* ctx, int32_t precision);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
int64_t cngp_launch_count(cngp_ctx* ctx);
int cngp_version(void);

/* Per-kernel device timing with CUDA events recorded on the launching stream around every kernel this context
 * launches (bench.py's roofline numbers).  cngp_profile_read synchronises the recorded events, returns the accumulated
 * milliseconds and launch count of one kernel class, and optionally resets them. */
#define CNGP_PROF_FIT 0        /* gp_fit_kernel: assembly + Cholesky + z + LML */
#define CNGP_PROF_VAR 1        /* gp_var_kernel: predictive mean / variance */
#define CNGP_PROF_GRAD 2       /* gp_grad_kernel: L^-1, K^-1, gradient contraction */
#define CNGP_PROF_LOOKAHEAD 3  /* zupt_lookahead_kernel */
#define CNGP_PROF_LARGE 4      /* large-N blocked Cholesky kernels */
#define CNGP_PROF_MISC 5
#define CNGP_PROF_KERNELS 6
int cngp_set_profiling(cngp_ctx* ctx, int32_t on);
int cngp_profile_read(cngp_ctx* ctx, int32_t kernel_id, double* total_ms, int64_t* launches, int32_t reset);

/* Exact-GP prediction for B independent windows (rows a3 + a6).
 *   theta   [B][P] (theta_stride = P) or one shared vector (theta_stride = 0); P = kernel->n_params + 1, noise last
 *   x, y    [B][N] training inputs / targets
 *   xstar   [B][M] (xstar_stride = M) or shared [M] (xstar_stride = 0)
 *   mean    [B][M]  K*' alpha
 *   var     [B][M]  max(k** - sum V^2, 1e-15) + noise   (GPy predict, include_likelihood=True)
 *   lml     [B]     log marginal likelihood (may be NULL)
 *   status  [B]     0 ok; k > 0: jitter tries that were needed (jitter_retry=1); -k: factorisation failed at pivot k
 *                   (1-based) - mean/var/lml of that window are NaN; (may be NULL)
 */
int cngp_predict_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                       const double* x, const double* y, const double* xstar, int64_t xstar_stride,
                       int64_t B, int32_t N, int32_t M,
                       double* mean, double* var, double* lml, int32_t* status, int32_t mem);

/* Log marginal likelihood and its gradient for C candidates x B windows (rows a3 + a4).
 *   theta [C][P]; x, y [B][N]; lml [C][B]; grad [C][B][P] (d LML / d theta, noise last; may be NULL); status [C][B] */
int cngp_lml_grad_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t C,
                        const double* x, const double* y, int64_t B, int32_t N,
                        double* lml, double* grad, int32_t* status, int32_t mem);

/* The same objective for n_problems independent (hyper-parameter vector, window) pairs: problem p evaluates theta
 * row p [n_problems][P] on window window_of_problem[p] of the B windows.  This is what every iteration of a batch of
 * independent m.optimize() runs needs (gp_slip_node.py:36): each window is at its own theta, and windows that have
 * converged drop out of the list.  lml [n_problems]; grad [n_problems][P] (may be NULL); status [n_problems]. */
int cngp_lml_grad_windows(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t n_problems,
                          const int32_t* window_of_problem, const double* x, const double* y, int64_t B, int32_t N,
                          double* lml, double* grad, int32_t* status, int32_t mem);

/* Batched hyper-parameter fit (row a4): L-BFGS (history 10) on softplus-transformed [theta, noise] from theta0,
 * one independent optimiser per window, objective/gradient on the GPU.  theta0 [B][P] or shared (stride 0);
 * theta_out [B][P]; lml_out [B]; iters_out [B] (may be NULL).  HOST memory only. */
int cngp_optimize_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta0, int64_t theta0_stride,
                        const double* x, const double* y, int64_t B, int32_t N, int32_t max_iters,
                        double* theta_out, double* lml_out, int32_t* iters_out);
/* The same with the array arguments in device memory when mem = CNGP_MEM_DEVICE (stream-ordered, returns after the
 * optimisers have finished; results are left in the device buffers). */
int cngp_optimize_batch_mem(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta0, int64_t theta0_stride,
                        const double* x, const double* y, int64_t B, int32_t N, int32_t max_iters,
                        double* theta_out, double* lml_out, int32_t* iters_out, int32_t mem);

/* The node callback for B windows of n samples each (rows a1-a7): train on the first int(0.9 n) samples, predict on
 * arange(min(time), max(time) + horizon, 1), keep entries [n:], sigma = 2 sqrt(var).  m_out = number of kept points
 * per window (must be equal across the batch: same n and same ceil(span)); mean/sigma [B][m_cap].  theta [B][P] or
 * shared; pass theta = NULL to fit the hypers first (cngp_optimize_batch from all-ones, as GPy does). HOST memory. */
int cngp_gp_slip_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                       const double* time_array, const double* slip_array, int64_t B, int32_t n,
                       int32_t horizon, int32_t m_cap, double* mean, double* sigma, int32_t* m_out, int32_t* status);

/* ---- ragged window batches ----
 * The windows GP_Input carries differ in size (CoreNav.cpp:264-300: n_samples from min_samples up to the window length,
 * stamps with gaps), so these entry points take per-window counts.  Window b has n[b] valid samples in a row of ld
 * doubles of x / y (time_array / slip_array) and m[b] valid test points in a row of ldm doubles of xstar / mean / var /
 * sigma.  Entries beyond n[b] and m[b] are never read and never written (NaN there does not matter).  A window with
 * n[b] = 0 is skipped: nothing is written for it and its status is 0.  The windows are grouped on the device by
 * ceil(n[b] / 8) and every group runs the launch shape of the fixed-size entry points, so results equal theirs; each
 * call makes one small device-to-host read (the group sizes).  All arrays follow `mem`. */

/* cngp_predict_batch (gp_slip_node.py:35,47-50, rows a3 + a6) for ragged windows: theta [B][P] or shared (stride 0);
 * x, y [B][ld]; xstar, mean, var [B][ldm]; lml [B] (lml uses each window's own n: -n/2 log 2 pi); status [B]. */
int cngp_predict_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                        const double* x, const double* y, const int32_t* n, int32_t ld, const double* xstar,
                        const int32_t* m, int32_t ldm, int64_t B, double* mean, double* var, double* lml,
                        int32_t* status, int32_t mem);

/* cngp_lml_grad_batch (gp_slip_node.py:36, rows a3 + a4) for C candidates x B ragged windows: theta [C][P];
 * x, y [B][ld]; lml [C][B]; grad [C][B][P] (may be NULL); status [C][B]. */
int cngp_lml_grad_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t C, const double* x,
                         const double* y, const int32_t* n, int32_t ld, int64_t B, double* lml, double* grad,
                         int32_t* status, int32_t mem);

/* cngp_optimize_batch_mem (m.optimize(), gp_slip_node.py:36, row a4) for ragged windows: theta0 [B][P] or shared
 * (stride 0) or NULL (all ones, as GPy); theta_out [B][P]; lml_out, iters_out [B] (may be NULL). */
int cngp_optimize_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta0, int64_t theta0_stride,
                         const double* x, const double* y, const int32_t* n, int32_t ld, int64_t B, int32_t max_iters,
                         double* theta_out, double* lml_out, int32_t* iters_out, int32_t mem);

/* The node callback gp_slip_node.py:16-63 (rows a1-a7) for ragged windows, e.g. cngp_slip_record_batch output in place
 * (rows [B * max_windows] of cap doubles, n = n_samples of the published windows, 0 elsewhere).  Per window:
 * ntr = int(0.9 n) training samples, grid arange(min, max + horizon, 1), m_out[b] = len(grid) - n published points
 * in mean / sigma [B][ldm] (sigma = 2 sqrt(var)).  n[b] < 2: m_out[b] = 0, status 0, nothing written.  n[b] > ld or
 * m_out[b] > ldm: CNGP_ERR_INVALID before any work; ntr > CNGP_MAX_N: CNGP_ERR_UNSUPPORTED.  theta [B][P] or shared;
 * NULL fits the hypers first (cngp_optimize_ragged from all ones). */
int cngp_gp_slip_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                        const double* time_array, const double* slip_array, const int32_t* n, int32_t ld, int64_t B,
                        int32_t horizon, int32_t ldm, double* mean, double* sigma, int32_t* m_out, int32_t* status,
                        int32_t mem);

/* ---- stop predictor ---- */
typedef struct cngp_stop_config {
  double v_nom;      /* 0.8    gp_predictor.cpp:73-75 */
  double floor_a;    /* 0.03   :80-81 */
  double floor_b;    /* 0.05   :82-83 */
  double track;      /* 0.685  :85 */
  double scale;      /* 25     :88 */
  double thresh;     /* 3.00   :102 */
  int32_t ratio;     /* 5      :64,67 */
  int32_t fix_h_packing; /* 0 = reference behaviour: H(r,c) = Hvec[r*4+c] (gp_predictor.cpp:38-42) */
  double init_llh[3];    /* core_navigation/config/init_params.yaml:13-16 */
  double init_ecef[3];   /* core_navigation/config/init_params.yaml:9-12 */
} cngp_stop_config;

void cngp_default_stop_config(cngp_stop_config* c);

/* which context arrays carry one entry per window (else shared by the batch) */
#define CNGP_PERWIN_P 1
#define CNGP_PERWIN_Q 2
#define CNGP_PERWIN_STM 4
#define CNGP_PERWIN_H 8
#define CNGP_PERWIN_POS 16

/* Covariance look-ahead + 3-sigma error observer for B windows (rows a9-a12).
 *   mean, sigma [B][M] (GP_Output); P, Q, STM [.][225] row-major 15x15; Hvec [.][60]; pos [.][3] (lat, lon, h)
 *   triggered [B] 0/1; i_stop [B] = odometry updates performed when the loop ended (the reference's `i`);
 *   step_stop [B] = slip_i at the trigger or ratio*M; xy_err [B] = last horizontal error computed.
 * The 15 x 15 algebra runs on the FP64 tensor cores (one mma.sync.m8n8k4.f64 is bit for bit an ascending fma chain, the
 * order the oracle uses); one warp per window, windows claimed dynamically.  Test hook: the environment variable
 * CNGP_LOOKAHEAD_KERNEL ("tc" default / "warp" / "cta") selects the tensor-core kernel or one of the two scalar kernels of
 * round 1; all three produce the same bits. */
int cngp_zupt_lookahead_batch(cngp_ctx* ctx, const double* mean, const double* sigma, int64_t B, int32_t M,
                              const double* P, const double* Q, const double* STM, const double* Hvec,
                              const double* pos, int32_t per_window, const cngp_stop_config* cfg,
                              int32_t* triggered, int32_t* i_stop, int32_t* step_stop, double* xy_err, int32_t mem);

/* The same, also returning what the reference leaves in GpPredictor's public members after the callback
 * (gp_predictor.h:36-43): P_final [B][225] = P_pred after the last step executed, K_final [B][60] = K_pred (15 x 4) and
 * R_final [B][16] = R_IP of the last update; each may be NULL (K_final / R_final need P_final). */
int cngp_zupt_lookahead_batch_ex(cngp_ctx* ctx, const double* mean, const double* sigma, int64_t B, int32_t M,
                                 const double* P, const double* Q, const double* STM, const double* Hvec,
                                 const double* pos, int32_t per_window, const cngp_stop_config* cfg,
                                 int32_t* triggered, int32_t* i_stop, int32_t* step_stop, double* xy_err,
                                 double* P_final, double* K_final, double* R_final, int32_t mem);

/* cngp_zupt_lookahead_batch_ex (gp_predictor.cpp:58-130, rows a9-a12) for GP_Output of ragged length: mean, sigma
 * [B][ldm] with m[b] <= ldm points in row b.  The loop of window b runs ratio * m[b] steps (the reference's
 * slip_i < ratio * mean.size()), so a window that does not trigger reports step_stop = ratio * m[b]; m[b] = 0 gives
 * triggered = 0.  P_final / K_final / R_final may be NULL as in _batch_ex. */
int cngp_zupt_lookahead_ragged(cngp_ctx* ctx, const double* mean, const double* sigma, int64_t B, const int32_t* m,
                               int32_t ldm, const double* P, const double* Q, const double* STM, const double* Hvec,
                               const double* pos, int32_t per_window, const cngp_stop_config* cfg, int32_t* triggered,
                               int32_t* i_stop, int32_t* step_stop, double* xy_err, double* P_final, double* K_final,
                               double* R_final, int32_t mem);

/* The filter's own covariance recursion for B operating points (SURVEY.md 8f row N4): n_steps IMU steps of
 * P <- STM P STM' + Q (CoreNav.cpp:101) with the odometry update's Joseph form every ratio-th step (CoreNav.cpp:226-230)
 * - the covariance CoreNav::Update hands to the SetStopping service as P_pred (CoreNav.cpp:291-292).
 *   P0, Q, STM [.][225] row-major; H [.][60] the TRUE 4 x 15 measurement matrix, row-major (not the service's packing);
 *   R [.][16] the filter's odometry noise; per_window: CNGP_PERWIN_P | _Q | _STM | _H as above, CNGP_PERWIN_POS for R;
 *   n_steps must be a multiple of ratio; P_out [B][225]. */
int cngp_ekf_covariance_batch(cngp_ctx* ctx, const double* P0, const double* Q, const double* STM, const double* H,
                              const double* R, int64_t B, int32_t n_steps, int32_t ratio, int32_t per_window,
                              double* P_out, int32_t mem);

/* GpPredictor::llh_to_enu for n points on the device (lat, lon, h -> E, N, U); llh, enu [n][3]. */
int cngp_llh_to_enu(cngp_ctx* ctx, const double* llh, int64_t n, const cngp_stop_config* cfg, double* enu, int32_t mem);

/* EKF context generation for B operating points (SURVEY.md 8f row N4): the matrices CoreNav serves through
 * SetStopping (row a9), computed on the device for Monte-Carlo look-ahead runs.  Replaces the pure functions
 * CoreNav::insErrorStateModel_LNF (core_navigation/src/CoreNav.cpp:411-470) and CoreNav::calc_Q (:471-527) evaluated
 * as CoreNav::Propagate does (:58-72), and the odometry H of :191-220 in its instantaneous form.
 *   llh [B][3] lat, lon (rad), height (m); vel [B][3] nav-frame velocity; att [B][3] roll, pitch, yaw;
 *   f_ib_b [B][3] specific force (body); dt IMU step (s); dt_odo odometry step (s, H24 divides by it)
 *   STM, Q [B][225] row-major 15x15; Hvec [B][60] packed as HvecData[r*4+c] (CoreNav.cpp:669-673); Hvec may be NULL */
int cngp_ekf_context_batch(cngp_ctx* ctx, const double* llh, const double* vel, const double* att, const double* f_ib_b,
                           int64_t B, double dt, double dt_odo, double* STM, double* Q, double* Hvec, int32_t mem);

/* Slip extraction + GP window recorder for B independent drives of T odometry updates each - the producer of
 * core_nav/GP_Input (SURVEY.md 8f row N1).  Replaces CoreNav::Update, core_navigation/src/CoreNav.cpp:176-183, :190,
 * :244-258 (slip = max over the four wheels of (v_wheel - vlin) / v_wheel, dead-band, clamp) and :264-329 (recorder).
 *   joint     [B][T][4]  wheel joint rates (rad/s: front-left, front-right, back-left, back-right; CoreNav.cpp:178-181)
 *   att       [B][T][3]  roll, pitch, yaw before the update (Cn2bUnc, CoreNav.cpp:190)
 *   vel       [B][T][3]  INS velocity (nav frame) after the update (CoreNav.cpp:232,244)
 *   cmd       [B][T]     cmd[0] of the drive command (CoreNav.cpp:264)
 *   stop_cmd  [B][T]     seconds-to-stop received since the previous update (CoreNav.cpp:755-758), NaN = none; may be NULL
 *   slip      [B][T]     per-update slip (may be NULL)
 *   time_array, slip_array [B][max_windows][cap]   recorded windows (counts are 1-based update numbers, CoreNav.cpp:286)
 *   n_samples, published, stop_update [B][max_windows]   samples recorded (may exceed cap: only cap are stored),
 *                        published = n_samples >= 15 (CoreNav.cpp:300), index of the update that closed the window
 *   n_windows [B]        windows closed (may exceed max_windows: only max_windows are stored) */
typedef struct cngp_slip_config {
  double wheel_radius;   /* InsConst.h:17   0.11 m */
  double cmd_min;        /* CoreNav.cpp:264 0.2 */
  double rear_min;       /* CoreNav.cpp:247 0.001 */
  int32_t arm_delay;     /* CoreNav.cpp:270 10 updates */
  int32_t window;        /* CoreNav.cpp:271 150 updates */
  int32_t min_samples;   /* CoreNav.cpp:300 15 */
  int32_t reserved;
} cngp_slip_config;
void cngp_default_slip_config(cngp_slip_config* cfg);
int cngp_slip_record_batch(cngp_ctx* ctx, const double* joint, const double* att, const double* vel, const double* cmd,
                           const double* stop_cmd, int64_t B, int32_t T, const cngp_slip_config* cfg,
                           int32_t max_windows, int32_t cap, double* slip, double* time_array, double* slip_array,
                           int32_t* n_samples, int32_t* published, int32_t* stop_update, int32_t* n_windows, int32_t mem);

/* ---- large single window (BASELINE.json configs[4]: N = 32768) ----
 * Blocked right-looking FP64 Cholesky of Ky = K(x,x) + (noise + 1e-8) I - the same inference as cngp_predict_batch
 * (row a3: GPy ExactGaussianInference as reached from gp_slip_node.py:35) for a window too large for shared memory.
 * The matrix lives in HBM as 8x8 tiles, column-tile-major, in block columns of CNGP_LARGE_NB columns dealt
 * cyclically to `world` GPUs (block column c belongs to rank c % world).  Per block column k: the owner factors the
 * diagonal block, inverts it and forms the panel (rows below) - cngp_large_factor_panel; the panel buffer is then
 * broadcast (NCCL, by the caller: corenav_gp_b200/large.py) and every rank subtracts panel x panel^T from its own
 * block columns - cngp_large_update, the only dense contraction (FP64 tensor cores fed by bulk-TMA copies).  y rides
 * along as one extra matrix row, so z = L^-1 y, y' Ky^-1 y and the LML come out of the factorisation itself.
 * All pointers of the cngp_large_* primitives are DEVICE pointers except `theta` and the plan. */
#define CNGP_LARGE_NB 256
typedef struct cngp_large_plan {
  int64_t N;                 /* training points */
  int64_t n_pad;             /* N rounded up to a multiple of CNGP_LARGE_NB (identity padding) */
  int32_t world, rank;
  int64_t row_tiles;         /* allocated 8-row tiles per column tile: n_pad/8 + 16; tile n_pad/8 carries y / z */
  int64_t n_blockcols;       /* n_pad / CNGP_LARGE_NB */
  int64_t n_local_blockcols; /* block columns of this rank */
  int64_t local_doubles;     /* size of this rank's matrix storage A */
  int64_t panel_doubles;     /* size of one panel buffer */
  int64_t winv_doubles;      /* inverted diagonal blocks of the local block columns (kept for the back substitution) */
  int64_t chunk_blocks;      /* 0 (cngp_large_make_plan): panels in one piece.  Otherwise the rows of every panel are cut at
                              * multiples of chunk_blocks x 128 rows (even, >= row_tiles/16/CNGP_LARGE_MAX_CHUNKS) and each
                              * piece is stored contiguously - the unit the multi-GPU driver pipelines (panel GEMM of a
                              * chunk -> its broadcast -> the update of the next block column with it).  The caller sets it
                              * after cngp_large_make_plan, the same on every rank. */
} cngp_large_plan;
#define CNGP_LARGE_MAX_CHUNKS 16
int cngp_large_make_plan(int64_t N, int32_t world, int32_t rank, cngp_large_plan* plan);
/* Fill this rank's block columns: Ky tiles on and below the diagonal blocks, the y row, identity padding. */
int cngp_large_assemble(cngp_ctx* ctx, const cngp_large_plan* plan, const cngp_kernel* kernel, const double* theta,
                        const double* x, const double* y, double* A);
/* Owner of block column k: factor + invert the diagonal block, panel = rows below x inv(L_kk)^T, written to `panel`
 * and back into A.  The panel buffer is compact: with r0 = (k+1) NB/8 and R = row_tiles - r0, tile (k-tile kt, row tile
 * rt >= r0) is at panel[(kt R + rt - r0) 64], so the first (NB/8) R 64 doubles are what the other ranks need.  logdet[k] = log det of the diagonal block; status[k] = 0 or -(failing pivot, 1-based in block). */
int cngp_large_factor_panel(cngp_ctx* ctx, const cngp_large_plan* plan, double* A, int64_t k, double* panel,
                            double* winv, double* logdet, int32_t* status);
/* The same in pieces, for the two-stream driver (flags, OR-ed):
 *   CNGP_LARGE_DEFER_COPY  step 4 (copying the panel back under the diagonal block of A) is left to cngp_large_copy_back,
 *                          issued off the panel chain (nothing before the backward sweep reads the copy);
 *   CNGP_LARGE_DIAG_ONLY   factor and invert the diagonal block only;   CNGP_LARGE_PANEL_ONLY   form the panel only - so
 *                          that the rows below the diagonal block can still be updated (cngp_large_update_part) on another
 *                          stream while the block is factored. */
#define CNGP_LARGE_DEFER_COPY 1
#define CNGP_LARGE_DIAG_ONLY 2
#define CNGP_LARGE_PANEL_ONLY 4
#define CNGP_LARGE_ROWS_ALL 0
#define CNGP_LARGE_ROWS_DIAG 1
#define CNGP_LARGE_ROWS_BELOW 2
/* chunk >= 0 (absolute chunk id, see chunk_blocks): the panel rows of that chunk only; -1: all rows. */
int cngp_large_factor_panel_ex(cngp_ctx* ctx, const cngp_large_plan* plan, double* A, int64_t k, double* panel,
                            double* winv, double* logdet, int32_t* status, int32_t flags, int32_t chunk);
int cngp_large_copy_back(cngp_ctx* ctx, const cngp_large_plan* p, double* A, int64_t k, const double* panel);
/* The chunks of panel k that hold rows: id of the first, how many, and offsets[0 .. count] (doubles) delimiting them in
 * the panel buffer - chunk first + i is panel[offsets[i] .. offsets[i+1]), one contiguous broadcast payload. */
int cngp_large_panel_chunks(const cngp_large_plan* plan, int64_t k, int32_t* first, int32_t* count, int64_t* offsets);
/* cngp_large_update restricted, for ONE block column, to its diagonal block or to the rows below it, and / or
 * (chunk >= 0) to the rows of one chunk of the panel. */
int cngp_large_update_part(cngp_ctx* ctx, const cngp_large_plan* plan, double* A, int64_t k, const double* panel,
                           int64_t c_lo, int64_t c_hi, int32_t rows, int32_t chunk);
/* Every rank: A(:, c) -= panel panel(c)^T for its block columns c in [max(c_lo, k+1), c_hi). */
int cngp_large_update(cngp_ctx* ctx, const cngp_large_plan* plan, double* A, int64_t k, const double* panel,
                      int64_t c_lo, int64_t c_hi);
/* After the last panel: z [n_pad] (this rank's columns, 0 elsewhere), sums[0] = sum of this rank's logdet[k],
 * sums[1] = sum of this rank's z^2, sums[2] = first failing pivot (1-based, global) of this rank's blocks or 0. */
int cngp_large_reduce(cngp_ctx* ctx, const cngp_large_plan* plan, const double* A, const double* logdet,
                      const int32_t* status, double* z, double* sums);
/* One step of alpha = L^-T z, last block column first: the owner of block column j computes alpha[j NB .. (j+1) NB)
 * from z and alpha of the later blocks (which must already be in `alpha` on this rank). */
int cngp_large_backsolve_step(cngp_ctx* ctx, const cngp_large_plan* plan, const double* A, const double* winv,
                              int64_t j, const double* z, double* alpha);
/* The same sweep with the work taken off its serial path: the owner of j finishes alpha_j = inv(L_jj)^T (z_j - s_j)
 * (cngp_large_backsolve_finish), alpha_j is broadcast, and EVERY rank adds L(block row j, c)^T alpha_j to s_c for its block
 * columns c < j (cngp_large_backsolve_apply).  s [n_pad] starts as zeros.  Same bits on every world size. */
int cngp_large_backsolve_finish(cngp_ctx* ctx, const cngp_large_plan* plan, const double* winv, int64_t j, const double* z,
                                const double* s, double* alpha);
int cngp_large_backsolve_apply(cngp_ctx* ctx, const cngp_large_plan* plan, const double* A, int64_t j, const double* alpha,
                               double* s);
/* r = Ky v for the same covariance, evaluated on the fly (no matrix stored): the residual check of the solve. */
int cngp_large_matvec(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x, const double* v,
                      int64_t N, double* r);

/* The whole single-GPU sequence: assemble, factor, logdet, quad = y' Ky^-1 y, lml, alpha = Ky^-1 y [N] (may be NULL).
 * x, y, alpha follow `mem`; logdet/quad/lml are HOST scalars (may be NULL).  Returns CNGP_OK, or a positive value
 * = the (1-based) pivot at which the factorisation broke down. */
int cngp_chol_large(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x, const double* y,
                    int64_t N, double* logdet, double* quad, double* lml, double* alpha, int32_t mem);

/* ---- predict on the large window from its stored factor ----
 * After the factorisation and the backward sweep, A (block columns of L below their diagonal blocks), winv and alpha
 * are all a predict pass reads, so any number of passes, at any test points x* [M], can follow one factorisation:
 *   mean = K(x*, x) alpha,   var = max(k(x*, x*) - sum_i W_i^2, 1e-15) + noise,   W = L^-1 K(x, x*)
 * (cngp_predict_batch's definition).  W is a forward sweep over R = K(x*, x), stored like A with the test points as rows
 * (M rounded up to a multiple of 128, zero beyond M) and dealt out block-cyclically as A is.  Per block column k:
 *   owner of k:  cngp_large_predict_panel    W_k = R(:, k) inv(L_kk)^T and L(rows below the diagonal block, k) into one
 *                                            payload; s[k][m] = sum over the block's columns of W_k(m, .)^2
 *   all ranks:   broadcast of the payload (by the caller; nothing with one rank)
 *   all ranks:   cngp_large_predict_update   R(:, c) -= W_k L(c, k)^T for its block columns c in [max(c_lo, k+1), c_hi)
 * then s is summed over the ranks (zero outside the owners' rows, so the sum is exact) and cngp_large_predict_finish
 * gives mean and var from alpha (all of it on every rank) and s, adding the s[k] in increasing k.  Every R(:, c) is written
 * by one rank in increasing k, so the results have the same bits on every world size.  Device pointers except theta. */
/* Buffer sizes in doubles for M test points: R of this rank, the payload of block column k (k = 0 is the largest), s. */
int cngp_large_predict_sizes(const cngp_large_plan* plan, int64_t M, int64_t k, int64_t* r_doubles,
                             int64_t* payload_doubles, int64_t* s_doubles);
/* R = K(x*, x) for this rank's block columns. */
int cngp_large_predict_assemble(cngp_ctx* ctx, const cngp_large_plan* plan, const cngp_kernel* kernel, const double* theta,
                                const double* x, const double* xstar, int64_t M, double* R);
/* Owner of block column k: payload = [W_k ; L(rows > k, k)] ([k-tile][row tile] each), s[k][0 .. M). */
int cngp_large_predict_panel(cngp_ctx* ctx, const cngp_large_plan* plan, const double* A, const double* winv,
                             const double* R, int64_t M, int64_t k, double* payload, double* s);
int cngp_large_predict_update(cngp_ctx* ctx, const cngp_large_plan* plan, double* R, int64_t M, int64_t k,
                              const double* payload, int64_t c_lo, int64_t c_hi);
/* mean, var [M] from alpha [n_pad] and the rank-summed s [n_blockcols][M]. */
int cngp_large_predict_finish(cngp_ctx* ctx, const cngp_large_plan* plan, const cngp_kernel* kernel, const double* theta,
                              const double* x, const double* alpha, const double* xstar, int64_t M, const double* s,
                              double* mean, double* var);
/* The whole single-GPU sequence: cngp_chol_large's factorisation, then the predict pass at xstar [M].  x, y, xstar,
 * mean, var follow `mem`; logdet/quad/lml are HOST scalars (may be NULL).  Returns CNGP_OK, or the failing pivot as in
 * cngp_chol_large - then mean, var, logdet, quad and lml are NaN. */
int cngp_chol_large_predict(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x,
                            const double* y, int64_t N, const double* xstar, int64_t M, double* mean, double* var,
                            double* logdet, double* quad, double* lml, int32_t mem);

/* ---- LML gradient on the large window from its stored factor ----
 * The same definitions as cngp_lml_grad_batch (GPy ExactGaussianInference dL_dK + kern.update_gradients_full):
 *   Ky = K + (noise + 1e-8) I,   dLML/dtheta_p = 1/2 sum_{i,j < N} (alpha_i alpha_j - (Ky^-1)_ij) dK_ij/dtheta_p,
 *   noise (last entry): 1/2 (alpha' alpha - tr Ky^-1);  natural (not log) parameters, leaf parameters in program order.
 * Like the predict pass it reads only A, winv and alpha, so any number of predict and gradient passes, in any order, can
 * follow one factorisation.  With V = L^-T (upper triangular), Ky^-1 = V V^T = sum_k V_k V_k^T, and V is the predict
 * sweep with R = I: W_k = V_k, non-zero in rows < NB (k+1) only.  RG stores R like A (n_pad/8 row tiles per column tile,
 * block-cyclic); once block column k of R has given W_k it holds G(:, k) = -(Ky^-1)(:, k) (lower part) instead.
 * Per block column k:
 *   owner of k:  cngp_large_grad_panel    payload = [W_k (rows < NB (k+1)) ; L(rows > k, k)], n_pad x NB doubles for any k
 *   all ranks:   broadcast of the payload (by the caller; nothing with one rank)
 *   all ranks:   cngp_large_grad_update   its block columns c in [c_lo, c_hi): c > k  R(rows < NB (k+1), c) -= W_k L(c, k)^T
 *                                                                           c <= k G(I, c) -= W_k(I) W_k(c)^T, c <= I <= k
 * then cngp_large_grad_contract writes part[c][p] for this rank's block columns (zero elsewhere), the parts are summed
 * over the ranks (each row comes from one rank, so the sum is exact) and cngp_large_grad_finish adds them in increasing c.
 * Every R(:, c) and G(:, c) is written by one rank in increasing k: the same bits on every world size.  Device pointers
 * except theta and the plan. */
/* Buffer sizes in doubles: RG of this rank, one payload, part [n_blockcols][CNGP_MAX_PARAMS + 1]. */
int cngp_large_grad_sizes(const cngp_large_plan* plan, int64_t* rg_doubles, int64_t* payload_doubles, int64_t* part_doubles);
/* RG = I on this rank's block columns. */
int cngp_large_grad_begin(cngp_ctx* ctx, const cngp_large_plan* plan, double* RG);
int cngp_large_grad_panel(cngp_ctx* ctx, const cngp_large_plan* plan, const double* A, const double* winv, double* RG,
                          int64_t k, double* payload);
int cngp_large_grad_update(cngp_ctx* ctx, const cngp_large_plan* plan, double* RG, int64_t k, const double* payload,
                           int64_t c_lo, int64_t c_hi);
/* part[c][0 .. P) = sum over the entries i >= j of block column c of (alpha_i alpha_j - (Ky^-1)_ij) dK_ij/dtheta, the
 * entries off the diagonal counted twice; alpha [n_pad] whole on every rank. */
int cngp_large_grad_contract(cngp_ctx* ctx, const cngp_large_plan* plan, const cngp_kernel* kernel, const double* theta,
                             const double* x, const double* alpha, const double* RG, double* part);
/* grad [P] = 1/2 sum_c part[c] from the rank-summed part. */
int cngp_large_grad_finish(cngp_ctx* ctx, const cngp_large_plan* plan, const cngp_kernel* kernel, const double* part,
                           double* grad);
/* The whole single-GPU sequence: cngp_chol_large's factorisation, then the gradient pass.  x, y, grad [P] follow `mem`;
 * logdet/quad/lml are HOST scalars (may be NULL).  Returns CNGP_OK, or the failing pivot as in cngp_chol_large - then
 * grad, logdet, quad and lml are NaN. */
int cngp_chol_large_grad(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x, const double* y,
                         int64_t N, double* logdet, double* quad, double* lml, double* grad, int32_t mem);

#ifdef __cplusplus
}
#endif
#endif /* CNGP_H_ */
