// Host orchestration of the two entry points that sit directly behind the node callback
// core_navigation/script/gp_slip_node.py:16-63:
//
//   cngp_optimize_batch   m.optimize() (gp_slip_node.py:36) for B windows at once, entirely on the device.  GPy hands the objective to paramz'
//                         "lbfgsb" optimiser = scipy.optimize.fmin_l_bfgs_b (L-BFGS-B 3.0, m = 10, factr = 1e7,
//                         pgtol = 1e-5, maxfun = maxiter = 1000) on Logexp (softplus) transformed positives.  With no
//                         bounds L-BFGS-B is L-BFGS with the More-Thuente line search (MINPACK-2 dcsrch/dcstep,
//                         ftol 1e-3, gtol 0.9, xtol 0.1, first step 1/||g||, at most 20 trial points per search).  That
//                         published algorithm is restated below as an explicit per-window state machine so that all B
//                         optimisers advance in lock step: every round evaluates ONE trial point per still-active
//                         window in a single batched GPU launch.  Objective, gradient AND the O(m P) two-loop recursions,
//                         line searches and convergence tests run on the GPU (opt_feed_kernel); the host only
//                         enqueues launches and reads one progress integer every few iterations.
//   cngp_gp_slip_batch    the whole callback (rows a1-a7): 90 % train split, [optional fit], prediction grid
//                         arange(min, max + horizon, 1), predict, keep [n:], sigma = 2 sqrt(var) (fused into the
//                         variance kernel's epilogue).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "cngp_internal.h"
#include "lbfgsb_host.h"

using namespace cngp_host;

namespace {

// grow-only device buffers of the context (slots 30..41 belong to the optimiser): no cudaMalloc / cudaFree per call
enum { SLOT_OPT_X = 30, SLOT_OPT_Y, SLOT_OPT_TH, SLOT_OPT_MAP, SLOT_OPT_LML, SLOT_OPT_GRAD, SLOT_OPT_ST, SLOT_OPT_STATE,
       SLOT_OPT_DONE, SLOT_OPT_NACT, SLOT_OPT_OUT, SLOT_OPT_TH0 };

}  // namespace

// ---- device side of the optimiser: one L-BFGS-B state machine per window, advanced by a kernel ----
namespace {

__global__ void opt_init_kernel(Optimizer* st, const double* theta0, long long theta0_stride, int P, int max_iters,
                                long long B, double* theta, int* win_map, int* done) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double ones[kMaxP];
  for (int i = 0; i < P; ++i) ones[i] = 1.0;      // GPy initialises every hyper-parameter and the noise at 1.0
  Optimizer& o = st[b];
  o.init(theta0 ? theta0 + (theta0_stride ? b * theta0_stride : 0) : ones, P, max_iters);
  for (int i = 0; i < P; ++i) theta[b * P + i] = softplus(o.zt[i]);
  win_map[b] = (int)b;
  done[b] = 0;
}

// Consume the objective / gradient evaluated at every still-active window's trial point and publish the next one.
// One WARP per window: the 5 KB state machine is copied into shared memory by the 32 lanes (coalesced), lane 0 runs the
// L-BFGS-B step on the shared copy, and the lanes copy it back.  (One THREAD per window walking its state in global memory
// - a few thousand dependent, uncoalesced accesses - took longer per iteration at B = 4096 than the factorisations:
// tools/bench_configs.py callback, 105 ms per call of which 51 ms in gp_fit_kernel + gp_grad_kernel.)
constexpr int FEED_WPB = 8;
static_assert(sizeof(Optimizer) % 8 == 0, "Optimizer is copied as 64-bit words");
__global__ void __launch_bounds__(FEED_WPB * 32) opt_feed_kernel(Optimizer* st, const double* lml, const double* grad,
                                                                 const int* status, int P, long long B, double* theta,
                                                                 int* done, int* n_active) {
  extern __shared__ __align__(16) unsigned char feed_sm[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * FEED_WPB + w;
  if (b >= B || done[b]) return;
  Optimizer* so = reinterpret_cast<Optimizer*>(feed_sm) + w;
  constexpr int NW64 = (int)(sizeof(Optimizer) / 8);
  unsigned long long* gw = reinterpret_cast<unsigned long long*>(st + b);
  unsigned long long* sw = reinterpret_cast<unsigned long long*>(so);
  for (int i = lane; i < NW64; i += 32) sw[i] = gw[i];
  __syncwarp();
  if (lane == 0) {
    Optimizer& o = *so;
    double gz[kMaxP];
    double fv;
    if (status[b] < 0 || !isfinite(lml[b])) {   // not positive definite: a wall, as in the CPU path
      fv = 1e300;
      for (int i = 0; i < P; ++i) gz[i] = 0.0;
    } else {
      fv = -lml[b];
      for (int i = 0; i < P; ++i) gz[i] = -grad[b * P + i] * softplus_gradfactor(theta[b * P + i]);
    }
    o.feed(fv, gz);
    if (o.done) {
      done[b] = 1;
    } else {
      for (int i = 0; i < P; ++i) theta[b * P + i] = softplus(o.zt[i]);
      atomicAdd(n_active, 1);
    }
  }
  __syncwarp();
  for (int i = lane; i < NW64; i += 32) gw[i] = sw[i];
}

__global__ void opt_result_kernel(const Optimizer* st, int P, long long B, double* theta_out, double* lml_out, int* iters_out) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const Optimizer& o = st[b];
  for (int i = 0; i < P; ++i) theta_out[b * P + i] = softplus(o.z[i]);
  if (lml_out) lml_out[b] = -o.f;
  if (iters_out) iters_out[b] = o.nfev;
}

}  // namespace

// m.optimize() for B windows.  Every L-BFGS-B state machine lives in device memory and is advanced by opt_feed_kernel;
// one iteration is  gp_fit_kernel -> gp_grad_kernel -> opt_feed_kernel  on the context's stream with NO host round trip:
// the host enqueues OPT_BLIND iterations at a time and only then reads one integer (windows still active).  Finished
// windows are skipped by the kernels themselves (FitArgs::skip), so the tail of a batch costs empty launches, not work.
int cngp_optimize_impl(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta0, int64_t theta0_stride,
                       const double* x, const double* y, int64_t B, int32_t N, int32_t max_iters, double* theta_out,
                       double* lml_out, int32_t* iters_out, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !x || !y || !theta_out || B < 0 || N <= 0) return cngp_set_error(ctx, CNGP_ERR_INVALID, "optimize: bad argument");
  if (B == 0) return CNGP_OK;
  cngp_kernel kk = *kernel;
  if (cngp_kernel_finalize(&kk) != CNGP_OK) return cngp_set_error(ctx, CNGP_ERR_INVALID, "optimize: invalid kernel expression");
  const int P = kk.n_params + 1;
  if (P > kMaxP) return cngp_set_error(ctx, CNGP_ERR_UNSUPPORTED, "optimize: too many hyper-parameters");
  if (max_iters <= 0) max_iters = 1000;
  const bool host = mem == CNGP_MEM_HOST;

  // Everything below is ordered on the context's stream on the context's device.
  if (cudaSetDevice(cngp_ctx_device(ctx)) != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize: cudaSetDevice failed");
  cudaStream_t s = cngp_ctx_stream(ctx);
  const size_t xy = sizeof(double) * (size_t)B * N;
  const double *d_x = x, *d_y = y, *d_th0 = theta0;
  double* d_out = theta_out; double* d_lout = lml_out; int* d_iout = iters_out;
  if (host) {
    double* bx = (double*)cngp_ctx_buf(ctx, SLOT_OPT_X, xy);
    double* by = (double*)cngp_ctx_buf(ctx, SLOT_OPT_Y, xy);
    double* bo = (double*)cngp_ctx_buf(ctx, SLOT_OPT_OUT, sizeof(double) * B * (P + 1) + sizeof(int) * B);
    double* b0 = theta0 ? (double*)cngp_ctx_buf(ctx, SLOT_OPT_TH0, sizeof(double) * (theta0_stride ? B * theta0_stride : P)) : nullptr;
    if (!bx || !by || !bo || (theta0 && !b0)) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "optimize: device allocation failed");
    if (cudaMemcpyAsync(bx, x, xy, cudaMemcpyHostToDevice, s) != cudaSuccess ||
        cudaMemcpyAsync(by, y, xy, cudaMemcpyHostToDevice, s) != cudaSuccess ||
        (theta0 && cudaMemcpyAsync(b0, theta0, sizeof(double) * (theta0_stride ? B * theta0_stride : P),
                                   cudaMemcpyHostToDevice, s) != cudaSuccess))
      return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize: upload failed");
    d_x = bx; d_y = by; d_th0 = b0;
    d_out = bo; d_lout = bo + (size_t)B * P; d_iout = (int*)(bo + (size_t)B * (P + 1));
  }
  const OptBucket all{0, B, N, d_x, d_y, nullptr};
  const int rc = cngp_optimize_run(ctx, &kk, d_th0, theta0_stride, B, max_iters, &all, 1, d_out, d_lout, d_iout);
  if (rc) return rc;
  if (host) {
    if (cudaMemcpyAsync(theta_out, d_out, sizeof(double) * B * P, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        (lml_out && cudaMemcpyAsync(lml_out, d_lout, sizeof(double) * B, cudaMemcpyDeviceToHost, s) != cudaSuccess) ||
        (iters_out && cudaMemcpyAsync(iters_out, d_iout, sizeof(int) * B, cudaMemcpyDeviceToHost, s) != cudaSuccess) ||
        cudaStreamSynchronize(s) != cudaSuccess)
      return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize: download failed");
  }
  return CNGP_OK;
}

// The optimiser loop over B windows held in buckets (see OptBucket): one fit + gradient per bucket and one
// opt_feed_kernel over all B windows per iteration.  Every pointer is a device pointer.
int cngp_optimize_run(cngp_ctx* ctx, const cngp_kernel* kernel, const double* d_th0, int64_t theta0_stride, int64_t B,
                      int32_t max_iters, const OptBucket* buckets, int n_buckets, double* d_out, double* d_lout,
                      int32_t* d_iout) {
  cngp_kernel kk = *kernel;
  if (cngp_kernel_finalize(&kk) != CNGP_OK) return cngp_set_error(ctx, CNGP_ERR_INVALID, "optimize: invalid kernel expression");
  const int P = kk.n_params + 1;
  if (P > kMaxP) return cngp_set_error(ctx, CNGP_ERR_UNSUPPORTED, "optimize: too many hyper-parameters");
  if (max_iters <= 0) max_iters = 1000;
  cudaStream_t s = cngp_ctx_stream(ctx);
  Optimizer* d_st = (Optimizer*)cngp_ctx_buf(ctx, SLOT_OPT_STATE, sizeof(Optimizer) * (size_t)B);
  double* d_th = (double*)cngp_ctx_buf(ctx, SLOT_OPT_TH, sizeof(double) * B * P);
  int* d_map = (int*)cngp_ctx_buf(ctx, SLOT_OPT_MAP, sizeof(int) * B);
  double* d_lml = (double*)cngp_ctx_buf(ctx, SLOT_OPT_LML, sizeof(double) * B);
  double* d_grad = (double*)cngp_ctx_buf(ctx, SLOT_OPT_GRAD, sizeof(double) * B * P);
  int* d_st_fit = (int*)cngp_ctx_buf(ctx, SLOT_OPT_ST, sizeof(int) * B);
  int* d_done = (int*)cngp_ctx_buf(ctx, SLOT_OPT_DONE, sizeof(int) * B);
  int* d_nact = (int*)cngp_ctx_buf(ctx, SLOT_OPT_NACT, 64);
  if (!d_st || !d_th || !d_map || !d_lml || !d_grad || !d_st_fit || !d_done || !d_nact)
    return cngp_set_error(ctx, CNGP_ERR_NOMEM, "optimize: device allocation failed");
  const unsigned blocks = (unsigned)((B + 63) / 64);
  // d_map[b] = b: problem p of a bucket is the bucket's window p (theta row p of the bucket's slice)
  opt_init_kernel<<<blocks, 64, 0, s>>>(d_st, d_th0, theta0_stride, P, max_iters, B, d_th, d_map, d_done);
  constexpr int OPT_BLIND = 6;
  const unsigned feed_blocks = (unsigned)((B + FEED_WPB - 1) / FEED_WPB);
  const size_t feed_smem = sizeof(Optimizer) * FEED_WPB;
  if (cudaFuncSetAttribute(opt_feed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)feed_smem) != cudaSuccess)
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize: shared memory attribute");
  int n_active = 1;
  for (int round = 0; n_active > 0 && round * OPT_BLIND <= max_iters + OPT_BLIND; ++round) {
    for (int k = 0; k < OPT_BLIND; ++k) {
      if (cudaMemsetAsync(d_nact, 0, sizeof(int), s) != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize: memset failed");
      for (int k = 0; k < n_buckets; ++k) {
        const OptBucket& bk = buckets[k];
        const int rc = cngp_lml_grad_impl(ctx, &kk, d_th + bk.off * P, bk.nb, bk.x, bk.y, bk.nb, bk.ld, d_lml + bk.off,
                                          d_grad + bk.off * P, d_st_fit + bk.off, CNGP_MEM_DEVICE, d_map, d_done + bk.off,
                                          bk.n_win);
        if (rc) return rc;
      }
      cngp_ctx_begin(ctx, CNGP_PROF_MISC);
      opt_feed_kernel<<<feed_blocks, FEED_WPB * 32, feed_smem, s>>>(d_st, d_lml, d_grad, d_st_fit, P, B, d_th, d_done, d_nact);
      cngp_ctx_end(ctx);
    }
    if (cudaMemcpyAsync(&n_active, d_nact, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess)
      return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize: progress read failed");
  }
  opt_result_kernel<<<blocks, 64, 0, s>>>(d_st, P, B, d_out, d_lout, d_iout);
  if (cudaGetLastError() != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize: kernel launch failed");
  return CNGP_OK;
}

extern "C" int cngp_optimize_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta0, int64_t theta0_stride,
                                   const double* x, const double* y, int64_t B, int32_t N, int32_t max_iters,
                                   double* theta_out, double* lml_out, int32_t* iters_out) {
  return cngp_optimize_impl(ctx, kernel, theta0, theta0_stride, x, y, B, N, max_iters, theta_out, lml_out, iters_out,
                            CNGP_MEM_HOST);
}

extern "C" int cngp_optimize_batch_mem(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta0,
                                       int64_t theta0_stride, const double* x, const double* y, int64_t B, int32_t N,
                                       int32_t max_iters, double* theta_out, double* lml_out, int32_t* iters_out,
                                       int32_t mem) {
  return cngp_optimize_impl(ctx, kernel, theta0, theta0_stride, x, y, B, N, max_iters, theta_out, lml_out, iters_out, mem);
}

namespace {
// gp_slip_node.py:45,59-61: X_ = arange(X.min(), X.max() + horizon, 1); the published part is X_[len(X):]
__global__ void grid_fill_kernel(const double* t0, int n, long long M, long long B, double* grid) {
  for (long long b = blockIdx.x; b < B; b += gridDim.x)
    for (long long k = threadIdx.x; k < M; k += blockDim.x) grid[b * M + k] = t0[b] + (double)(n + k);
}
}  // namespace

extern "C" int cngp_gp_slip_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                                  const double* time_array, const double* slip_array, int64_t B, int32_t n,
                                  int32_t horizon, int32_t m_cap, double* mean, double* sigma, int32_t* m_out,
                                  int32_t* status) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !time_array || !slip_array || !mean || !sigma || !m_out || B < 0 || n <= 0 || horizon < 0)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "gp_slip: bad argument");
  *m_out = 0;
  if (B == 0) return CNGP_OK;
  if (cudaSetDevice(cngp_ctx_device(ctx)) != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "gp_slip: cudaSetDevice failed");
  cngp_kernel kk = *kernel;
  if (cngp_kernel_finalize(&kk) != CNGP_OK) return cngp_set_error(ctx, CNGP_ERR_INVALID, "gp_slip: invalid kernel expression");
  const int P = kk.n_params + 1;
  // gp_slip_node.py:27-30: per = 0.9; train = first int(per * len(X)) samples (double product, then truncation)
  const int ntr = (int)(0.9 * (double)n);
  if (ntr < 1) return cngp_set_error(ctx, CNGP_ERR_INVALID, "gp_slip: fewer than 2 samples");
  if (ntr > CNGP_MAX_N) return cngp_set_error(ctx, CNGP_ERR_UNSUPPORTED, "gp_slip: int(0.9 n) exceeds CNGP_MAX_N");
  // gp_slip_node.py:45: X_ = arange(X.min(), X.max() + horizon, 1) -> start + k, ceil(stop - start) points
  std::vector<double> t0((size_t)B);
  int64_t len = -1;
  for (int64_t b = 0; b < B; ++b) {
    const double* t = time_array + b * n;
    double lo = t[0], hi = t[0];
    for (int i = 1; i < n; ++i) { lo = std::min(lo, t[i]); hi = std::max(hi, t[i]); }
    const int64_t l = (int64_t)std::ceil((hi + (double)horizon) - lo);
    if (len >= 0 && l != len)
      return cngp_set_error(ctx, CNGP_ERR_UNSUPPORTED, "gp_slip: windows of one batch must span the same number of grid points");
    len = l;
    t0[b] = lo;
  }
  const int64_t M = len - n;                      // gp_slip_node.py:59-61: entries [len(X):] are published
  if (M <= 0) return CNGP_OK;
  if (M > m_cap) return cngp_set_error(ctx, CNGP_ERR_INVALID, "gp_slip: m_cap too small");

  // Everything between the caller's arrays and the kernels stays on the device: the training split is a strided upload
  // (no host repacking), the prediction grid is generated in place, the fitted hyper-parameters never leave the GPU, and
  // the outputs come back with one strided copy each.  (Round 1 staged x, y, the B x M grid, mean and sigma through
  // pageable std::vectors and uploaded x, y twice - at B = 4096 half of the call.)
  cudaStream_t s = cngp_ctx_stream(ctx);
  enum { SLOT_CB_XTR = 44, SLOT_CB_YTR, SLOT_CB_GRID, SLOT_CB_MU, SLOT_CB_SG, SLOT_CB_TH, SLOT_CB_T0, SLOT_CB_STATUS };
  double* d_xtr = (double*)cngp_ctx_buf(ctx, SLOT_CB_XTR, sizeof(double) * (size_t)B * ntr);
  double* d_ytr = (double*)cngp_ctx_buf(ctx, SLOT_CB_YTR, sizeof(double) * (size_t)B * ntr);
  double* d_grid = (double*)cngp_ctx_buf(ctx, SLOT_CB_GRID, sizeof(double) * (size_t)B * M);
  double* d_mu = (double*)cngp_ctx_buf(ctx, SLOT_CB_MU, sizeof(double) * (size_t)B * M);
  double* d_sg = (double*)cngp_ctx_buf(ctx, SLOT_CB_SG, sizeof(double) * (size_t)B * M);
  const size_t th_doubles = theta ? (theta_stride ? (size_t)B * theta_stride : (size_t)P) : (size_t)B * P;
  double* d_th = (double*)cngp_ctx_buf(ctx, SLOT_CB_TH, sizeof(double) * th_doubles);
  double* d_t0 = (double*)cngp_ctx_buf(ctx, SLOT_CB_T0, sizeof(double) * (size_t)B);
  int* d_status = (int*)cngp_ctx_buf(ctx, SLOT_CB_STATUS, sizeof(int) * (size_t)B);
  if (!d_xtr || !d_ytr || !d_grid || !d_mu || !d_sg || !d_th || !d_t0 || !d_status)
    return cngp_set_error(ctx, CNGP_ERR_NOMEM, "gp_slip: device allocation failed");
  if (cudaMemcpy2DAsync(d_xtr, sizeof(double) * ntr, time_array, sizeof(double) * n, sizeof(double) * ntr, (size_t)B,
                        cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaMemcpy2DAsync(d_ytr, sizeof(double) * ntr, slip_array, sizeof(double) * n, sizeof(double) * ntr, (size_t)B,
                        cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaMemcpyAsync(d_t0, t0.data(), sizeof(double) * (size_t)B, cudaMemcpyHostToDevice, s) != cudaSuccess ||
      (theta && cudaMemcpyAsync(d_th, theta, sizeof(double) * th_doubles, cudaMemcpyHostToDevice, s) != cudaSuccess))
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "gp_slip: upload failed");
  grid_fill_kernel<<<(unsigned)std::min<int64_t>(B, 65535), 128, 0, s>>>(d_t0, n, M, B, d_grid);
  int64_t th_stride = theta_stride;
  if (!theta) {                                   // gp_slip_node.py:35-36: all-ones start, then m.optimize()
    const int rc = cngp_optimize_impl(ctx, &kk, nullptr, 0, d_xtr, d_ytr, B, ntr, 1000, d_th, nullptr, nullptr, CNGP_MEM_DEVICE);
    if (rc) return rc;
    th_stride = P;
  }
  const int rc = cngp_predict_impl(ctx, &kk, d_th, th_stride, d_xtr, d_ytr, d_grid, M, B, ntr, (int32_t)M, d_mu, d_sg, nullptr,
                                   d_status, CNGP_MEM_DEVICE, /*sigma_mode=*/1);
  if (rc) return rc;
  if (cudaMemcpy2DAsync(mean, sizeof(double) * m_cap, d_mu, sizeof(double) * M, sizeof(double) * M, (size_t)B,
                        cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaMemcpy2DAsync(sigma, sizeof(double) * m_cap, d_sg, sizeof(double) * M, sizeof(double) * M, (size_t)B,
                        cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      (status && cudaMemcpyAsync(status, d_status, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, s) != cudaSuccess) ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "gp_slip: download failed");
  *m_out = (int32_t)M;
  return CNGP_OK;
}
