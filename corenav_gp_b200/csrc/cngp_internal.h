// Internal (non-ABI) entry points shared between the translation units of libcngp.
#pragma once
#include "../../include/cngp.h"

// cngp_predict_batch with the output transform of the node callback: sigma_mode = 1 writes 2 sqrt(var) into `var`.
int cngp_predict_impl(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                      const double* x, const double* y, const double* xstar, int64_t xstar_stride, int64_t B, int32_t N,
                      int32_t M, double* mean, double* var, double* lml, int32_t* status, int32_t mem, int sigma_mode,
                      const int32_t* n_win = nullptr, const int32_t* m_win = nullptr);
// Ragged batches (device memory only): n_win [B] valid training points per window, all with ceil(n_win / 8) ==
// ceil(N / 8) - N is then the row stride of x / y; m_win [B] <= M valid test points per window - M is the row stride of
// xstar / mean / var and nothing at or beyond m_win[b] is written.  Either may be null (every window full).

// cngp_lml_grad_batch (win_map == nullptr) / cngp_lml_grad_windows (win_map given).
int cngp_lml_grad_impl(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t C, const double* x,
                       const double* y, int64_t B, int32_t N, double* lml, double* grad, int32_t* status, int32_t mem,
                       const int32_t* win_map, const int32_t* skip = nullptr,   // skip[p] != 0: problem p is left untouched
                       const int32_t* n_win = nullptr);                          // per-window valid counts, as above

// The batched optimiser over windows held in buckets (gp_slip.cu): bucket k is windows [off, off + nb) of the optimiser
// state, with x / y rows of stride ld and per-window counts n_win (null: all ld points valid).  Device pointers only.
struct OptBucket {
  int64_t off, nb;
  int32_t ld;
  const double* x;
  const double* y;
  const int32_t* n_win;
};
int cngp_optimize_run(cngp_ctx* ctx, const cngp_kernel* kernel, const double* d_th0, int64_t theta0_stride, int64_t B,
                      int32_t max_iters, const OptBucket* buckets, int n_buckets, double* d_out, double* d_lout,
                      int32_t* d_iout);

// error text of a context (cngp_api.cu)
int cngp_set_error(cngp_ctx* ctx, int code, const char* text);

// ---- context internals for the other translation units (chol_large.cu) ----
#ifdef __CUDACC__
#include <cuda_runtime.h>
namespace cngp { struct KProg; }
cudaStream_t cngp_ctx_stream(cngp_ctx* ctx);
int cngp_ctx_device(cngp_ctx* ctx);
void cngp_ctx_begin(cngp_ctx* ctx, int prof_id);   // counts one kernel launch (+ opens a timing span when profiling)
void cngp_ctx_end(cngp_ctx* ctx);
void* cngp_ctx_buf(cngp_ctx* ctx, size_t slot, size_t bytes);   // grow-only device buffer `slot`
int cngp_build_kprog(const cngp_kernel* k, cngp::KProg* kp);
int cngp_sm_count(void);
#endif
