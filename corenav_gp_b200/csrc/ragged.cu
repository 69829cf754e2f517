// Ragged window batches: every window carries its own number of training points n[b] (row stride ld) and of test
// points m[b] (row stride ldm) - what the recorder (cngp_slip_record_batch) produces, since n_samples and the stamp span
// differ from window to window.
//
// The windows are grouped on the device by tile count nt_b = ceil(n_b / 8) (32 buckets at CNGP_MAX_N = 256): one CTA
// counts every bucket, takes the exclusive prefix and scatters the window indices into a permutation, stably (a window
// keeps its place within its bucket).  The host then reads back ONE small record - the bucket sizes, the largest and
// smallest m and the smallest n of each bucket, and the validation flags - and runs, per non-empty bucket, the launch
// shape today's code picks for that nt (cngp_predict_impl / cngp_lml_grad_impl on the bucket's windows gathered into
// contiguous rows of 8 nt doubles).  A window is padded by at most 7 identity rows; the kernels take the per-window
// counts (FitArgs / GradArgs / VarArgs::n_win, VarArgs::m_win) for the padding, the masks and the LML constant.
// Results are scattered back to the caller's rows; entries beyond n[b] / m[b] are never read and never written.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "cngp_internal.h"

namespace {

constexpr int RB = CNGP_MAX_N / 8;   // buckets: nt = 1 .. 32

struct RaggedStats {
  int count[RB];   // windows per bucket
  int max_m[RB];   // largest m of the bucket
  int min_m[RB];   // smallest m of the bucket
  int min_n[RB];   // smallest n of the bucket (== 8 nt: every window of the bucket is full)
  int flags;       // 1: some n or m outside [0, ld] / [0, ldm];  2: some n > CNGP_MAX_N
  int prep_flags;  // the same bits, from ragged_slip_prep_kernel
};

// grow-only context buffers of the ragged entry points
enum { SLOT_RG_STATS = 60, SLOT_RG_PERM, SLOT_RG_X, SLOT_RG_Y, SLOT_RG_XS, SLOT_RG_TH, SLOT_RG_N, SLOT_RG_M, SLOT_RG_MEAN,
       SLOT_RG_VAR, SLOT_RG_LML, SLOT_RG_ST, SLOT_RG_GRAD, SLOT_RG_T0, SLOT_RG_NTR, SLOT_RG_ITERS,
       SLOT_RG_IN0 = 80 };

__device__ __forceinline__ int warp_min(int v) {
  for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_max(int v) {
  for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// One CTA of RB warps; warp k owns bucket nt = k + 1.  Pass 1 counts (ballot over 32 windows at a time), thread 0 takes
// the exclusive prefix, pass 2 writes perm in window order.  Windows with n = 0 (or invalid) belong to no bucket.
__global__ void __launch_bounds__(RB * 32) ragged_bucket_kernel(const int* n, const int* m, long long B, int ld, int ldm,
                                                                int* perm, RaggedStats* st) {
  __shared__ int s_base[RB];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nt = w + 1;
  int cnt = 0, mx = 0, mnm = INT_MAX, mnn = INT_MAX, flags = 0;
  auto member = [&](long long b, int& nb, int& mb) -> bool {
    nb = 0; mb = 0;
    if (b >= B) return false;
    nb = n[b];
    mb = m ? m[b] : 0;
    return nb > 0 && nb <= ld && nb <= CNGP_MAX_N && mb >= 0 && mb <= ldm && (nb + 7) / 8 == nt;
  };
  for (long long b0 = 0; b0 < B; b0 += 32) {
    int nb, mb;
    const bool mine = member(b0 + lane, nb, mb);
    if (w == 0 && b0 + lane < B) {
      if (nb < 0 || nb > ld || mb < 0 || mb > ldm) flags |= 1;
      else if (nb > CNGP_MAX_N) flags |= 2;
    }
    cnt += __popc(__ballot_sync(0xffffffffu, mine));
    if (mine) { mx = max(mx, mb); mnm = min(mnm, mb); mnn = min(mnn, nb); }
  }
  mx = warp_max(mx); mnm = warp_min(mnm); mnn = warp_min(mnn);
  for (int o = 16; o; o >>= 1) flags |= __shfl_xor_sync(0xffffffffu, flags, o);
  if (lane == 0) {
    s_base[w] = cnt;
    st->count[w] = cnt; st->max_m[w] = mx; st->min_m[w] = cnt ? mnm : 0; st->min_n[w] = cnt ? mnn : 0;
    if (w == 0) st->flags = flags;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int k = 0; k < RB; ++k) { const int c = s_base[k]; s_base[k] = acc; acc += c; }
  }
  __syncthreads();
  int pos = s_base[w];
  for (long long b0 = 0; b0 < B; b0 += 32) {
    int nb, mb;
    const bool mine = member(b0 + lane, nb, mb);
    const unsigned bal = __ballot_sync(0xffffffffu, mine);
    if (mine) perm[pos + __popc(bal & ((1u << lane) - 1u))] = (int)(b0 + lane);
    pos += __popc(bal);
  }
}

// Node callback per window (gp_slip_node.py:27-30,45,59-61): ntr = int(0.9 n), t0 = min(time), m = ceil(max + horizon -
// min) - n published points.  n < 2: nothing to do (ntr = m = 0).  One warp per window.
__global__ void ragged_slip_prep_kernel(const double* time_array, const int* n, long long B, int ld, int horizon, int ldm,
                                        int* ntr, int* m, double* t0, RaggedStats* st) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const int nb = n[b];
  int flag = 0, tr = 0, mb = 0;
  double lo = 0.0;
  if (nb < 0 || nb > ld) {
    flag = 1;
  } else if (nb >= 2) {
    const double* t = time_array + b * (long long)ld;
    double l = t[0], h = t[0];
    for (int i = lane; i < nb; i += 32) { l = fmin(l, t[i]); h = fmax(h, t[i]); }
    for (int o = 16; o; o >>= 1) {
      l = fmin(l, __shfl_xor_sync(0xffffffffu, l, o));
      h = fmax(h, __shfl_xor_sync(0xffffffffu, h, o));
    }
    lo = l;
    const double len = ceil((h + (double)horizon) - l);
    mb = (int)fmax(len - (double)nb, 0.0);
    tr = (int)(0.9 * (double)nb);
    if (len - (double)nb > (double)ldm) flag = 1;
    else if (tr > CNGP_MAX_N) flag = 2;
  }
  if (lane == 0) {
    if (flag) { atomicOr(&st->prep_flags, flag); tr = 0; mb = 0; }
    ntr[b] = tr; m[b] = mb; t0[b] = lo;
  }
}

struct GatherArgs {
  const int* perm;                 // this bucket's slice of the permutation
  long long nb;
  const int* n; const int* m;      // caller counts (n: the training points used)
  const double* x; const double* y; long long ld_in;
  const double* xs; long long ldm_in;    // caller test points, or null: grid t0[b] + n_grid[b] + k
  const double* t0; const int* n_grid;
  const double* theta; long long theta_stride; int P;   // per-window theta rows to gather, or null
  int ldg, ldmg;                   // gathered strides: 8 nt, the bucket's largest m
  double* xg; double* yg; double* xsg; double* thg; int* ng; int* mg;
};

// Window j of the bucket <- caller row perm[j].  Padding: x, y = 0 (never read, the kernels mask by n); test points beyond
// m repeat a valid stamp of the window, so that they stay inside its lag table (their outputs are not stored).
__global__ void ragged_gather_kernel(const GatherArgs a) {
  for (long long j = blockIdx.x; j < a.nb; j += gridDim.x) {
    const long long b = a.perm[j];
    const int nb = a.n[b], mb = a.m ? a.m[b] : 0;
    const double* xr = a.x + b * a.ld_in;
    for (int i = threadIdx.x; i < a.ldg; i += blockDim.x) {
      a.xg[j * a.ldg + i] = i < nb ? xr[i] : 0.0;
      a.yg[j * a.ldg + i] = i < nb ? a.y[b * a.ld_in + i] : 0.0;
    }
    if (a.xsg) {
      auto test_point = [&](int k) -> double {
        return a.xs ? a.xs[b * a.ldm_in + k] : a.t0[b] + (double)(a.n_grid[b] + k);
      };
      for (int k = threadIdx.x; k < a.ldmg; k += blockDim.x)
        a.xsg[j * a.ldmg + k] = k < mb ? test_point(k) : (mb > 0 ? test_point(mb - 1) : xr[0]);
    }
    if (a.thg)
      for (int i = threadIdx.x; i < a.P; i += blockDim.x) a.thg[j * a.P + i] = a.theta[b * a.theta_stride + i];
    if (threadIdx.x == 0) {
      a.ng[j] = nb;
      if (a.mg) a.mg[j] = mb;
    }
  }
}

// predict outputs of one bucket -> caller rows (m[b] entries of mean / var, lml, status)
__global__ void ragged_scatter_predict_kernel(const int* perm, long long nb, const int* mg, int ldmg, const double* mean_s,
                                              const double* var_s, const double* lml_s, const int* st_s, long long ldm,
                                              double* mean, double* var, double* lml, int* status) {
  for (long long j = blockIdx.x; j < nb; j += gridDim.x) {
    const long long b = perm[j];
    const int mb = mg[j];
    for (int k = threadIdx.x; k < mb; k += blockDim.x) {
      mean[b * ldm + k] = mean_s[j * ldmg + k];
      var[b * ldm + k] = var_s[j * ldmg + k];
    }
    if (threadIdx.x == 0) {
      if (lml) lml[b] = lml_s[j];
      if (status) status[b] = st_s[j];
    }
  }
}

// C x nb problems of one bucket -> [C][B] caller layout (rows of P for grad); also optimiser outputs (C = 1)
__global__ void ragged_scatter_problems_kernel(const int* perm, long long nb, long long C, long long B, int P,
                                               const double* lml_s, const double* grad_s, const int* st_s,
                                               double* lml, double* grad, int* status) {
  const long long total = C * nb;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long c = t / nb, j = t - c * nb;
    const long long dst = c * B + perm[j];
    if (lml) lml[dst] = lml_s[t];
    if (status) status[dst] = st_s[t];
    if (grad)
      for (int i = 0; i < P; ++i) grad[dst * P + i] = grad_s[t * P + i];
  }
}

unsigned grid_of(long long n) { return (unsigned)std::max<long long>(1, std::min<long long>(n, 65535)); }

// The buckets of one call, from the single read-back of RaggedStats.
struct Plan {
  RaggedStats h;
  int* d_perm = nullptr;
  long long Bv = 0;                // windows in some bucket
  std::vector<int> ks;             // non-empty buckets
  std::vector<long long> off;      // first window of bucket k in the permutation
  std::vector<long long> xoff;     // first double of bucket k in the gathered x / y
  std::vector<long long> soff;     // first double of bucket k in the gathered test points / outputs
  long long xtot = 0, stot = 0;
};

int make_plan(cngp_ctx* ctx, const int* d_n, const int* d_m, long long B, int ld, int ldm, RaggedStats* d_st, Plan& pl,
              const char* what) {
  cudaStream_t s = cngp_ctx_stream(ctx);
  pl.d_perm = (int*)cngp_ctx_buf(ctx, SLOT_RG_PERM, sizeof(int) * (size_t)B);
  if (!pl.d_perm) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "ragged: permutation buffer");
  cngp_ctx_begin(ctx, CNGP_PROF_MISC);
  ragged_bucket_kernel<<<1, RB * 32, 0, s>>>(d_n, d_m, B, ld, ldm, pl.d_perm, d_st);
  cngp_ctx_end(ctx);
  // the one device-to-host read of the call
  if (cudaMemcpyAsync(&pl.h, d_st, sizeof(RaggedStats), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "ragged: bucket read-back failed");
  const int flags = pl.h.flags | pl.h.prep_flags;
  if (flags & 1) {
    char msg[160];
    snprintf(msg, sizeof msg, "%s: some window has n > ld (%d), m > ldm (%d) or a negative count", what, ld, ldm);
    return cngp_set_error(ctx, CNGP_ERR_INVALID, msg);
  }
  if (flags & 2) {
    char msg[160];
    snprintf(msg, sizeof msg, "%s: some window has more than CNGP_MAX_N = %d training points", what, CNGP_MAX_N);
    return cngp_set_error(ctx, CNGP_ERR_UNSUPPORTED, msg);
  }
  long long o = 0;
  for (int k = 0; k < RB; ++k) {
    if (!pl.h.count[k]) continue;
    pl.ks.push_back(k);
    pl.off.push_back(o);
    pl.xoff.push_back(pl.xtot);
    pl.soff.push_back(pl.stot);
    o += pl.h.count[k];
    pl.xtot += (long long)pl.h.count[k] * 8 * (k + 1);
    pl.stot += (long long)pl.h.count[k] * pl.h.max_m[k];
  }
  pl.Bv = o;
  return CNGP_OK;
}

// Gathered copies of every bucket, laid out one bucket after the other.
struct Gathered {
  double *x = nullptr, *y = nullptr, *xs = nullptr, *th = nullptr;
  int *n = nullptr, *m = nullptr;
};

int gather_all(cngp_ctx* ctx, const Plan& pl, GatherArgs ga, bool want_xs, bool want_theta, int P, Gathered& g) {
  g.x = (double*)cngp_ctx_buf(ctx, SLOT_RG_X, sizeof(double) * (size_t)std::max<long long>(pl.xtot, 1));
  g.y = (double*)cngp_ctx_buf(ctx, SLOT_RG_Y, sizeof(double) * (size_t)std::max<long long>(pl.xtot, 1));
  g.n = (int*)cngp_ctx_buf(ctx, SLOT_RG_N, sizeof(int) * (size_t)std::max<long long>(pl.Bv, 1));
  g.m = (int*)cngp_ctx_buf(ctx, SLOT_RG_M, sizeof(int) * (size_t)std::max<long long>(pl.Bv, 1));
  g.xs = want_xs ? (double*)cngp_ctx_buf(ctx, SLOT_RG_XS, sizeof(double) * (size_t)std::max<long long>(pl.stot, 1)) : nullptr;
  g.th = want_theta ? (double*)cngp_ctx_buf(ctx, SLOT_RG_TH, sizeof(double) * (size_t)std::max<long long>(pl.Bv * P, 1)) : nullptr;
  if (!g.x || !g.y || !g.n || !g.m || (want_xs && !g.xs) || (want_theta && !g.th))
    return cngp_set_error(ctx, CNGP_ERR_NOMEM, "ragged: gather buffers");
  cudaStream_t s = cngp_ctx_stream(ctx);
  for (size_t i = 0; i < pl.ks.size(); ++i) {
    const int k = pl.ks[i];
    GatherArgs a = ga;
    a.perm = pl.d_perm + pl.off[i];
    a.nb = pl.h.count[k];
    a.ldg = 8 * (k + 1);
    a.ldmg = pl.h.max_m[k];
    a.xg = g.x + pl.xoff[i]; a.yg = g.y + pl.xoff[i];
    a.xsg = want_xs && a.ldmg > 0 ? g.xs + pl.soff[i] : nullptr;
    a.thg = want_theta ? g.th + pl.off[i] * P : nullptr;
    a.P = P;
    a.ng = g.n + pl.off[i]; a.mg = g.m + pl.off[i];
    cngp_ctx_begin(ctx, CNGP_PROF_MISC);
    ragged_gather_kernel<<<grid_of(a.nb), 128, 0, s>>>(a);
    cngp_ctx_end(ctx);
  }
  if (cudaGetLastError() != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "ragged: gather launch failed");
  return CNGP_OK;
}

// Host-memory calls: the caller's arrays go to grow-only device buffers first (outputs too, so that the entries this call
// does not write come back unchanged), the device path runs, and the outputs are copied home.
struct HostStage {
  cngp_ctx* ctx;
  bool host;
  int slot = SLOT_RG_IN0;
  bool err = false;
  struct Out { void* h; void* d; size_t bytes; };
  std::vector<Out> outs;
  template <class T> T* put(T* p, size_t count, bool output) {
    if (!host || !p || count == 0) return p;
    void* d = cngp_ctx_buf(ctx, slot++, sizeof(T) * count);
    if (!d || cudaMemcpyAsync(d, p, sizeof(T) * count, cudaMemcpyHostToDevice, cngp_ctx_stream(ctx)) != cudaSuccess) {
      err = true;
      return nullptr;
    }
    if (output) outs.push_back({(void*)p, d, sizeof(T) * count});
    return (T*)d;
  }
  int finish(const char* what) {
    cudaStream_t s = cngp_ctx_stream(ctx);
    if (host) {
      for (auto& o : outs)
        if (cudaMemcpyAsync(o.h, o.d, o.bytes, cudaMemcpyDeviceToHost, s) != cudaSuccess) err = true;
      if (cudaStreamSynchronize(s) != cudaSuccess) err = true;
    }
    if (err) return cngp_set_error(ctx, CNGP_ERR_CUDA, what);
    return CNGP_OK;
  }
};

// Predict every bucket of a gathered plan and scatter the results.  th: shared theta (stride 0) or gathered rows (stride P).
int predict_buckets(cngp_ctx* ctx, const cngp_kernel* kk, const Plan& pl, const Gathered& g, const double* th,
                    int64_t th_stride, int sigma_mode, long long ldm, double* mean, double* var, double* lml,
                    int* status) {
  cudaStream_t s = cngp_ctx_stream(ctx);
  const size_t so = (size_t)std::max<long long>(pl.stot, 1), bv = (size_t)std::max<long long>(pl.Bv, 1);
  double* mean_s = (double*)cngp_ctx_buf(ctx, SLOT_RG_MEAN, sizeof(double) * so);
  double* var_s = (double*)cngp_ctx_buf(ctx, SLOT_RG_VAR, sizeof(double) * so);
  double* lml_s = (double*)cngp_ctx_buf(ctx, SLOT_RG_LML, sizeof(double) * bv);
  int* st_s = (int*)cngp_ctx_buf(ctx, SLOT_RG_ST, sizeof(int) * bv);
  if (!mean_s || !var_s || !lml_s || !st_s) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "ragged predict: output buffers");
  for (size_t i = 0; i < pl.ks.size(); ++i) {
    const int k = pl.ks[i], nt = k + 1, nb = pl.h.count[k], M = pl.h.max_m[k];
    const bool full_n = pl.h.min_n[k] == 8 * nt, equal_m = pl.h.min_m[k] == M;
    const double* thk = th_stride ? th + pl.off[i] * th_stride : th;
    const int rc = cngp_predict_impl(ctx, kk, thk, th_stride, g.x + pl.xoff[i], g.y + pl.xoff[i],
                                     M ? g.xs + pl.soff[i] : nullptr, M, nb, 8 * nt, M, mean_s + pl.soff[i],
                                     var_s + pl.soff[i], lml_s + pl.off[i], st_s + pl.off[i], CNGP_MEM_DEVICE, sigma_mode,
                                     full_n ? nullptr : g.n + pl.off[i], equal_m ? nullptr : g.m + pl.off[i]);
    if (rc) return rc;
    cngp_ctx_begin(ctx, CNGP_PROF_MISC);
    ragged_scatter_predict_kernel<<<grid_of(nb), 128, 0, s>>>(pl.d_perm + pl.off[i], nb, g.m + pl.off[i], M,
                                                              mean_s + pl.soff[i], var_s + pl.soff[i], lml_s + pl.off[i],
                                                              st_s + pl.off[i], ldm, mean, var, lml, status);
    cngp_ctx_end(ctx);
  }
  if (cudaGetLastError() != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "ragged predict: scatter launch failed");
  return CNGP_OK;
}

int finalize_kernel(cngp_ctx* ctx, const cngp_kernel* kernel, cngp_kernel& kk, const char* what) {
  if (!kernel) return cngp_set_error(ctx, CNGP_ERR_INVALID, what);
  kk = *kernel;
  if (cngp_kernel_finalize(&kk) != CNGP_OK) return cngp_set_error(ctx, CNGP_ERR_INVALID, what);
  return CNGP_OK;
}

RaggedStats* stats_buf(cngp_ctx* ctx) {
  RaggedStats* d = (RaggedStats*)cngp_ctx_buf(ctx, SLOT_RG_STATS, sizeof(RaggedStats));
  if (d && cudaMemsetAsync(d, 0, sizeof(RaggedStats), cngp_ctx_stream(ctx)) != cudaSuccess) return nullptr;
  return d;
}

}  // namespace

extern "C" int cngp_predict_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                                   const double* x, const double* y, const int32_t* n, int32_t ld, const double* xstar,
                                   const int32_t* m, int32_t ldm, int64_t B, double* mean, double* var, double* lml,
                                   int32_t* status, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  cngp_kernel kk;
  if (finalize_kernel(ctx, kernel, kk, "predict_ragged: invalid kernel expression")) return CNGP_ERR_INVALID;
  const int P = kk.n_params + 1;
  if (!theta || !x || !y || !n || !m || B < 0 || ld <= 0 || ldm < 0 || (theta_stride != 0 && theta_stride < P) ||
      (ldm > 0 && (!xstar || !mean || !var)))
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "predict_ragged: bad argument");
  if (B == 0) return CNGP_OK;
  if (cudaSetDevice(cngp_ctx_device(ctx)) != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "predict_ragged: cudaSetDevice failed");
  HostStage hs{ctx, mem == CNGP_MEM_HOST};
  const size_t bb = (size_t)B;
  const double* d_th = hs.put(theta, theta_stride ? bb * theta_stride : (size_t)P, false);
  const double* d_x = hs.put(x, bb * ld, false);
  const double* d_y = hs.put(y, bb * ld, false);
  const int* d_n = hs.put(n, bb, false);
  const int* d_m = hs.put(m, bb, false);
  const double* d_xs = hs.put(xstar, bb * ldm, false);
  double* d_mean = hs.put(mean, bb * ldm, true);
  double* d_var = hs.put(var, bb * ldm, true);
  double* d_lml = hs.put(lml, bb, true);
  int* d_status = hs.put(status, bb, true);
  RaggedStats* d_st = stats_buf(ctx);
  if (hs.err || !d_st) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "predict_ragged: staging failed");
  cudaStream_t s = cngp_ctx_stream(ctx);
  if (d_status && cudaMemsetAsync(d_status, 0, sizeof(int) * bb, s) != cudaSuccess)
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "predict_ragged: memset failed");
  Plan pl;
  int rc = make_plan(ctx, d_n, d_m, B, ld, ldm, d_st, pl, "predict_ragged");
  if (rc) return rc;
  GatherArgs ga;
  memset(&ga, 0, sizeof ga);
  ga.n = d_n; ga.m = d_m; ga.x = d_x; ga.y = d_y; ga.ld_in = ld; ga.xs = d_xs; ga.ldm_in = ldm;
  ga.theta = d_th; ga.theta_stride = theta_stride;
  Gathered g;
  if ((rc = gather_all(ctx, pl, ga, true, theta_stride != 0, P, g))) return rc;
  rc = predict_buckets(ctx, &kk, pl, g, theta_stride ? g.th : d_th, theta_stride ? P : 0, 0, ldm, d_mean, d_var, d_lml,
                       d_status);
  if (rc) return rc;
  return hs.finish("predict_ragged: copy-out failed");
}

extern "C" int cngp_lml_grad_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t C,
                                    const double* x, const double* y, const int32_t* n, int32_t ld, int64_t B,
                                    double* lml, double* grad, int32_t* status, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  cngp_kernel kk;
  if (finalize_kernel(ctx, kernel, kk, "lml_grad_ragged: invalid kernel expression")) return CNGP_ERR_INVALID;
  const int P = kk.n_params + 1;
  if (!theta || !x || !y || !n || !lml || C < 0 || B < 0 || ld <= 0)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "lml_grad_ragged: bad argument");
  if (B == 0 || C == 0) return CNGP_OK;
  if (cudaSetDevice(cngp_ctx_device(ctx)) != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "lml_grad_ragged: cudaSetDevice failed");
  HostStage hs{ctx, mem == CNGP_MEM_HOST};
  const size_t bb = (size_t)B, cb = (size_t)C * B;
  const double* d_th = hs.put(theta, (size_t)C * P, false);
  const double* d_x = hs.put(x, bb * ld, false);
  const double* d_y = hs.put(y, bb * ld, false);
  const int* d_n = hs.put(n, bb, false);
  double* d_lml = hs.put(lml, cb, true);
  double* d_grad = hs.put(grad, cb * P, true);
  int* d_status = hs.put(status, cb, true);
  RaggedStats* d_st = stats_buf(ctx);
  if (hs.err || !d_st) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "lml_grad_ragged: staging failed");
  cudaStream_t s = cngp_ctx_stream(ctx);
  if (d_status && cudaMemsetAsync(d_status, 0, sizeof(int) * cb, s) != cudaSuccess)
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "lml_grad_ragged: memset failed");
  Plan pl;
  int rc = make_plan(ctx, d_n, nullptr, B, ld, 0, d_st, pl, "lml_grad_ragged");
  if (rc) return rc;
  GatherArgs ga;
  memset(&ga, 0, sizeof ga);
  ga.n = d_n; ga.x = d_x; ga.y = d_y; ga.ld_in = ld;
  Gathered g;
  if ((rc = gather_all(ctx, pl, ga, false, false, P, g))) return rc;
  const size_t pv = (size_t)std::max<long long>(pl.Bv, 1) * C;
  double* lml_s = (double*)cngp_ctx_buf(ctx, SLOT_RG_LML, sizeof(double) * pv);
  int* st_s = (int*)cngp_ctx_buf(ctx, SLOT_RG_ST, sizeof(int) * pv);
  double* grad_s = d_grad ? (double*)cngp_ctx_buf(ctx, SLOT_RG_GRAD, sizeof(double) * pv * P) : nullptr;
  if (!lml_s || !st_s || (d_grad && !grad_s)) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "lml_grad_ragged: output buffers");
  for (size_t i = 0; i < pl.ks.size(); ++i) {
    const int k = pl.ks[i], nt = k + 1, nb = pl.h.count[k];
    const long long po = pl.off[i] * C;   // bucket i's problems: [C][nb] from po
    rc = cngp_lml_grad_impl(ctx, &kk, d_th, C, g.x + pl.xoff[i], g.y + pl.xoff[i], nb, 8 * nt, lml_s + po,
                            grad_s ? grad_s + po * P : nullptr, st_s + po, CNGP_MEM_DEVICE, nullptr, nullptr,
                            pl.h.min_n[k] == 8 * nt ? nullptr : g.n + pl.off[i]);
    if (rc) return rc;
    cngp_ctx_begin(ctx, CNGP_PROF_MISC);
    ragged_scatter_problems_kernel<<<grid_of((C * nb + 127) / 128), 128, 0, s>>>(
        pl.d_perm + pl.off[i], nb, C, B, P, lml_s + po, grad_s ? grad_s + po * P : nullptr, st_s + po, d_lml, d_grad,
        d_status);
    cngp_ctx_end(ctx);
  }
  if (cudaGetLastError() != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "lml_grad_ragged: launch failed");
  return hs.finish("lml_grad_ragged: copy-out failed");
}

namespace {
// the optimiser over the gathered buckets of a plan; results in gathered (bucket) order
int optimize_buckets(cngp_ctx* ctx, const cngp_kernel* kk, const Plan& pl, const Gathered& g, const double* th0,
                     int64_t th0_stride, int max_iters, double* th_s, double* lml_s, int* it_s) {
  std::vector<OptBucket> bk;
  for (size_t i = 0; i < pl.ks.size(); ++i) {
    const int k = pl.ks[i], nt = k + 1;
    bk.push_back(OptBucket{pl.off[i], pl.h.count[k], 8 * nt, g.x + pl.xoff[i], g.y + pl.xoff[i],
                           pl.h.min_n[k] == 8 * nt ? nullptr : g.n + pl.off[i]});
  }
  return cngp_optimize_run(ctx, kk, th0, th0_stride, pl.Bv, max_iters, bk.data(), (int)bk.size(), th_s, lml_s, it_s);
}
}  // namespace

extern "C" int cngp_optimize_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta0,
                                    int64_t theta0_stride, const double* x, const double* y, const int32_t* n,
                                    int32_t ld, int64_t B, int32_t max_iters, double* theta_out, double* lml_out,
                                    int32_t* iters_out, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  cngp_kernel kk;
  if (finalize_kernel(ctx, kernel, kk, "optimize_ragged: invalid kernel expression")) return CNGP_ERR_INVALID;
  const int P = kk.n_params + 1;
  if (!x || !y || !n || !theta_out || B < 0 || ld <= 0 || (theta0 && theta0_stride != 0 && theta0_stride < P))
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "optimize_ragged: bad argument");
  if (B == 0) return CNGP_OK;
  if (cudaSetDevice(cngp_ctx_device(ctx)) != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize_ragged: cudaSetDevice failed");
  HostStage hs{ctx, mem == CNGP_MEM_HOST};
  const size_t bb = (size_t)B;
  const double* d_th0 = hs.put(theta0, theta0_stride ? bb * theta0_stride : (size_t)P, false);
  const double* d_x = hs.put(x, bb * ld, false);
  const double* d_y = hs.put(y, bb * ld, false);
  const int* d_n = hs.put(n, bb, false);
  double* d_th = hs.put(theta_out, bb * P, true);
  double* d_lml = hs.put(lml_out, bb, true);
  int* d_it = hs.put(iters_out, bb, true);
  RaggedStats* d_st = stats_buf(ctx);
  if (hs.err || !d_st) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "optimize_ragged: staging failed");
  Plan pl;
  int rc = make_plan(ctx, d_n, nullptr, B, ld, 0, d_st, pl, "optimize_ragged");
  if (rc) return rc;
  const bool per_win = d_th0 && theta0_stride;
  GatherArgs ga;
  memset(&ga, 0, sizeof ga);
  ga.n = d_n; ga.x = d_x; ga.y = d_y; ga.ld_in = ld; ga.theta = d_th0; ga.theta_stride = theta0_stride;
  Gathered g;
  if ((rc = gather_all(ctx, pl, ga, false, per_win, P, g))) return rc;
  const size_t bv = (size_t)std::max<long long>(pl.Bv, 1);
  double* th_s = (double*)cngp_ctx_buf(ctx, SLOT_RG_GRAD, sizeof(double) * bv * P);
  double* lml_s = (double*)cngp_ctx_buf(ctx, SLOT_RG_LML, sizeof(double) * bv);
  int* it_s = (int*)cngp_ctx_buf(ctx, SLOT_RG_ITERS, sizeof(int) * bv);
  if (!th_s || !lml_s || !it_s) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "optimize_ragged: output buffers");
  if (pl.Bv > 0) {
    rc = optimize_buckets(ctx, &kk, pl, g, per_win ? g.th : d_th0, per_win ? P : 0, max_iters, th_s, lml_s, it_s);
    if (rc) return rc;
    cngp_ctx_begin(ctx, CNGP_PROF_MISC);
    ragged_scatter_problems_kernel<<<grid_of((pl.Bv + 127) / 128), 128, 0, cngp_ctx_stream(ctx)>>>(
        pl.d_perm, pl.Bv, 1, B, P, lml_s, th_s, it_s, d_lml, d_th, d_it);
    cngp_ctx_end(ctx);
    if (cudaGetLastError() != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "optimize_ragged: launch failed");
  }
  return hs.finish("optimize_ragged: copy-out failed");
}

extern "C" int cngp_gp_slip_ragged(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                                   const double* time_array, const double* slip_array, const int32_t* n, int32_t ld,
                                   int64_t B, int32_t horizon, int32_t ldm, double* mean, double* sigma, int32_t* m_out,
                                   int32_t* status, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  cngp_kernel kk;
  if (finalize_kernel(ctx, kernel, kk, "gp_slip_ragged: invalid kernel expression")) return CNGP_ERR_INVALID;
  const int P = kk.n_params + 1;
  if (!time_array || !slip_array || !n || !mean || !sigma || !m_out || B < 0 || ld <= 0 || ldm < 0 || horizon < 0 ||
      (theta && theta_stride != 0 && theta_stride < P))
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "gp_slip_ragged: bad argument");
  if (B == 0) return CNGP_OK;
  if (cudaSetDevice(cngp_ctx_device(ctx)) != cudaSuccess) return cngp_set_error(ctx, CNGP_ERR_CUDA, "gp_slip_ragged: cudaSetDevice failed");
  HostStage hs{ctx, mem == CNGP_MEM_HOST};
  const size_t bb = (size_t)B;
  const double* d_th = hs.put(theta, theta_stride ? bb * theta_stride : (size_t)P, false);
  const double* d_t = hs.put(time_array, bb * ld, false);
  const double* d_s = hs.put(slip_array, bb * ld, false);
  const int* d_n = hs.put(n, bb, false);
  double* d_mean = hs.put(mean, bb * ldm, true);
  double* d_sigma = hs.put(sigma, bb * ldm, true);
  int* d_mout = hs.put(m_out, bb, true);
  int* d_status = hs.put(status, bb, true);
  RaggedStats* d_st = stats_buf(ctx);
  int* d_ntr = (int*)cngp_ctx_buf(ctx, SLOT_RG_NTR, sizeof(int) * bb);
  int* d_m = (int*)cngp_ctx_buf(ctx, SLOT_RG_ITERS + 1, sizeof(int) * bb);
  double* d_t0 = (double*)cngp_ctx_buf(ctx, SLOT_RG_T0, sizeof(double) * bb);
  if (hs.err || !d_st || !d_ntr || !d_m || !d_t0) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "gp_slip_ragged: staging failed");
  cudaStream_t s = cngp_ctx_stream(ctx);
  if (d_status && cudaMemsetAsync(d_status, 0, sizeof(int) * bb, s) != cudaSuccess)
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "gp_slip_ragged: memset failed");
  cngp_ctx_begin(ctx, CNGP_PROF_MISC);
  ragged_slip_prep_kernel<<<(unsigned)((B + 7) / 8), 256, 0, s>>>(d_t, d_n, B, ld, horizon, ldm, d_ntr, d_m, d_t0, d_st);
  cngp_ctx_end(ctx);
  Plan pl;
  int rc = make_plan(ctx, d_ntr, d_m, B, INT_MAX, INT_MAX, d_st, pl, "gp_slip_ragged");
  if (rc) return rc;
  if (cudaMemcpyAsync(d_mout, d_m, sizeof(int) * bb, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
    return cngp_set_error(ctx, CNGP_ERR_CUDA, "gp_slip_ragged: m_out copy failed");
  GatherArgs ga;
  memset(&ga, 0, sizeof ga);
  ga.n = d_ntr; ga.m = d_m; ga.x = d_t; ga.y = d_s; ga.ld_in = ld; ga.t0 = d_t0; ga.n_grid = d_n;
  ga.theta = d_th; ga.theta_stride = theta_stride;
  const bool per_win = theta && theta_stride;
  Gathered g;
  if ((rc = gather_all(ctx, pl, ga, true, per_win, P, g))) return rc;
  const double* th = per_win ? g.th : d_th;
  int64_t th_stride = per_win ? P : 0;
  if (!theta && pl.Bv > 0) {   // gp_slip_node.py:35-36: all-ones start, then m.optimize()
    const size_t bv = (size_t)pl.Bv;
    double* th_s = (double*)cngp_ctx_buf(ctx, SLOT_RG_GRAD, sizeof(double) * bv * P);
    if (!th_s) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "gp_slip_ragged: theta buffer");
    if ((rc = optimize_buckets(ctx, &kk, pl, g, nullptr, 0, 1000, th_s, nullptr, nullptr))) return rc;
    th = th_s;
    th_stride = P;
  }
  if ((rc = predict_buckets(ctx, &kk, pl, g, th, th_stride, 1, ldm, d_mean, d_sigma, nullptr, d_status))) return rc;
  return hs.finish("gp_slip_ragged: copy-out failed");
}
