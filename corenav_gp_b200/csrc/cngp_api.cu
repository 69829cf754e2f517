// C-ABI entry points of libcngp (include/cngp.h): context, kernel-expression parsing, batched predict,
// LML/gradient, look-ahead.  Host-side orchestration only; all arithmetic is in the kernels.
#include <cuda_runtime.h>

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "cngp_internal.h"
#include "gp_fit.cuh"
#include "gp_fit_toeplitz.cuh"
#include "gp_grad.cuh"
#include "gp_toep_group.cuh"
#include "gp_var.cuh"
#include "gp_var32.cuh"
#include "gp_var_toeplitz.cuh"

extern "C" int cngp_launch_lookahead(const double*, const double*, long long, int, const double*, const double*,
                                     const double*, const double*, const double*, int, const cngp_stop_config*, int*,
                                     int*, int*, double*, unsigned long long*, double*, double*, double*, const double*, int,
                                     cudaStream_t, const int* m_win = nullptr);
extern "C" int cngp_launch_llh_to_enu(const double*, long long, const cngp_stop_config*, double*, cudaStream_t);
extern "C" int cngp_launch_ekf_context(const double*, const double*, const double*, const double*, long long, double, double,
                                       double*, double*, double*, cudaStream_t);
extern "C" int cngp_launch_slip_record(const double*, const double*, const double*, const double*, const double*, long long,
                                       int, const cngp_slip_config*, int, int, double*, double*, double*, int*, int*, int*,
                                       int*, cudaStream_t);

using namespace cngp;

namespace {
std::string g_create_error;
int g_sm_count = 148;
}

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

struct cngp_ctx {
  cngp_config cfg;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;   // host-memory calls: results of one slab go home while the next slab computes
  std::string err;
  long long launches = 0;
  double* scratch = nullptr;  // factors (L / W tiles) + z
  size_t scratch_bytes = 0;
  std::vector<DevBuf> bufs;   // grow-only staging for host-memory calls
  // optional per-kernel timing with CUDA events on the launching stream (cngp_set_profiling)
  bool profiling = false;
  struct Span { int id; cudaEvent_t e0, e1; };
  std::vector<Span> spans;
  std::vector<cudaEvent_t> event_pool;
  double prof_ms[CNGP_PROF_KERNELS] = {0};
  long long prof_n[CNGP_PROF_KERNELS] = {0};

  cudaEvent_t get_event() {
    if (!event_pool.empty()) { cudaEvent_t e = event_pool.back(); event_pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
  void begin(int id) {
    launches++;
    if (!profiling) return;
    Span sp{id, get_event(), get_event()};
    cudaEventRecord(sp.e0, stream);
    spans.push_back(sp);
  }
  void end() {
    if (!profiling) return;
    cudaEventRecord(spans.back().e1, stream);
  }
  void collect() {
    for (auto& sp : spans) {
      float ms = 0.f;
      if (cudaEventSynchronize(sp.e1) == cudaSuccess && cudaEventElapsedTime(&ms, sp.e0, sp.e1) == cudaSuccess) {
        prof_ms[sp.id] += ms;
        prof_n[sp.id]++;
      }
      event_pool.push_back(sp.e0);
      event_pool.push_back(sp.e1);
    }
    spans.clear();
  }

  void* buf(size_t slot, size_t bytes) {
    if (bufs.size() <= slot) bufs.resize(slot + 1);
    DevBuf& b = bufs[slot];
    if (b.cap < bytes) {
      if (b.p) cudaFree(b.p);
      b.p = nullptr;
      b.cap = 0;
      if (cudaMalloc(&b.p, bytes) != cudaSuccess) return nullptr;
      b.cap = bytes;
    }
    return b.p;
  }
};

static int fail(cngp_ctx* c, int code, const char* fmt, ...) {
  char tmp[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tmp, sizeof tmp, fmt, ap);
  va_end(ap);
  if (c) c->err = tmp; else g_create_error = tmp;
  return code;
}

int cngp_set_error(cngp_ctx* ctx, int code, const char* text) { return fail(ctx, code, "%s", text); }
cudaStream_t cngp_ctx_stream(cngp_ctx* ctx) { return ctx->stream; }
int cngp_ctx_device(cngp_ctx* ctx) { return ctx->cfg.device; }
void cngp_ctx_begin(cngp_ctx* ctx, int prof_id) { ctx->begin(prof_id); }
void cngp_ctx_end(cngp_ctx* ctx) { ctx->end(); }
void* cngp_ctx_buf(cngp_ctx* ctx, size_t slot, size_t bytes) { return ctx->buf(slot, bytes); }
int cngp_sm_count(void) { return g_sm_count; }

#define CU(c, call)                                                                                  \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) return fail(c, CNGP_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));   \
  } while (0)

// ------------------------------------------------------------------------------------------------------------
// kernel expressions
// ------------------------------------------------------------------------------------------------------------
static int leaf_from_name(const std::string& s) {
  static const struct { const char* n; int t; } tab[] = {
      {"rbf", CNGP_K_RBF}, {"se", CNGP_K_RBF}, {"mat32", CNGP_K_MAT32}, {"matern32", CNGP_K_MAT32},
      {"mat52", CNGP_K_MAT52}, {"matern52", CNGP_K_MAT52}, {"ratquad", CNGP_K_RATQUAD}, {"rq", CNGP_K_RATQUAD},
      {"stdperiodic", CNGP_K_STDPERIODIC}, {"periodic", CNGP_K_STDPERIODIC}, {"per", CNGP_K_STDPERIODIC},
      {"brownian", CNGP_K_BROWNIAN}, {"linear", CNGP_K_LINEAR}, {"bias", CNGP_K_BIAS}, {"const", CNGP_K_BIAS},
      {"white", CNGP_K_WHITE}};
  for (auto& e : tab)
    if (s == e.n) return e.t;
  return 0;
}

extern "C" int cngp_kernel_finalize(cngp_kernel* k) {
  if (!k || k->n_ops <= 0 || k->n_ops > CNGP_MAX_OPS) return CNGP_ERR_INVALID;
  int depth = 0, np = 0;
  for (int i = 0; i < k->n_ops; ++i) {
    const int op = k->ops[i];
    if (op >= CNGP_K_RBF && op <= CNGP_K_WHITE) {
      ++depth;
      np += leaf_nparams(op);
    } else if (op == CNGP_OP_ADD || op == CNGP_OP_MUL) {
      if (depth < 2) return CNGP_ERR_INVALID;
      --depth;
    } else {
      return CNGP_ERR_INVALID;
    }
  }
  if (depth != 1 || np > CNGP_MAX_PARAMS) return CNGP_ERR_INVALID;
  k->n_params = np;
  return CNGP_OK;
}

extern "C" int cngp_kernel_parse(const char* text, cngp_kernel* out) {
  if (!text || !out) return CNGP_ERR_INVALID;
  std::vector<int> outq;
  std::vector<char> st;
  std::string cur;
  auto flush = [&]() -> bool {
    if (cur.empty()) return true;
    const int t = leaf_from_name(cur);
    cur.clear();
    if (!t) return false;
    outq.push_back(t);
    return true;
  };
  auto prec = [](char c) { return c == '+' ? 1 : 2; };
  for (const char* p = text; *p; ++p) {
    const char ch = (char)tolower((unsigned char)*p);
    if (ch == ' ') continue;
    if (ch == '+' || ch == '*') {
      if (!flush()) return CNGP_ERR_INVALID;
      while (!st.empty() && st.back() != '(' && prec(st.back()) >= prec(ch)) {
        outq.push_back(st.back() == '+' ? CNGP_OP_ADD : CNGP_OP_MUL);
        st.pop_back();
      }
      st.push_back(ch);
    } else if (ch == '(') {
      st.push_back(ch);
    } else if (ch == ')') {
      if (!flush()) return CNGP_ERR_INVALID;
      while (!st.empty() && st.back() != '(') {
        outq.push_back(st.back() == '+' ? CNGP_OP_ADD : CNGP_OP_MUL);
        st.pop_back();
      }
      if (st.empty()) return CNGP_ERR_INVALID;
      st.pop_back();
    } else {
      cur.push_back(ch);
    }
  }
  if (!flush()) return CNGP_ERR_INVALID;
  while (!st.empty()) {
    if (st.back() == '(') return CNGP_ERR_INVALID;
    outq.push_back(st.back() == '+' ? CNGP_OP_ADD : CNGP_OP_MUL);
    st.pop_back();
  }
  if (outq.empty() || (int)outq.size() > CNGP_MAX_OPS) return CNGP_ERR_INVALID;
  memset(out, 0, sizeof *out);
  out->n_ops = (int)outq.size();
  for (size_t i = 0; i < outq.size(); ++i) out->ops[i] = outq[i];
  return cngp_kernel_finalize(out);
}

// postfix program -> sum of products of leaves
static int build_kprog(const cngp_kernel* k, KProg* kp) {
  cngp_kernel kk = *k;
  if (cngp_kernel_finalize(&kk) != CNGP_OK) return CNGP_ERR_INVALID;
  typedef std::vector<std::pair<int, int>> Term;  // (leaf type, param offset)
  std::vector<std::vector<Term>> st;
  int poff = 0;
  for (int i = 0; i < kk.n_ops; ++i) {
    const int op = kk.ops[i];
    if (op < CNGP_OP_ADD) {
      st.push_back({Term{{op, poff}}});
      poff += leaf_nparams(op);
    } else {
      std::vector<Term> b = st.back(); st.pop_back();
      std::vector<Term> a = st.back(); st.pop_back();
      std::vector<Term> r;
      if (op == CNGP_OP_ADD) {
        r = a;
        r.insert(r.end(), b.begin(), b.end());
      } else {
        for (auto& ta : a)
          for (auto& tb : b) {
            Term t = ta;
            t.insert(t.end(), tb.begin(), tb.end());
            r.push_back(t);
          }
      }
      st.push_back(r);
    }
  }
  memset(kp, 0, sizeof *kp);
  int nl = 0;
  kp->n_terms = (int)st.back().size();
  if (kp->n_terms > CNGP_MAX_LEAVES) return CNGP_ERR_UNSUPPORTED;
  for (int t = 0; t < kp->n_terms; ++t) {
    kp->term_start[t] = nl;
    for (auto& lf : st.back()[t]) {
      if (nl >= CNGP_MAX_LEAVES) return CNGP_ERR_UNSUPPORTED;
      kp->leaf_type[nl] = lf.first;
      kp->leaf_param[nl] = lf.second;
      ++nl;
    }
  }
  kp->term_start[kp->n_terms] = nl;
  kp->n_leaves = nl;
  kp->n_params = kk.n_params;
  kp->fast_id = 0;
  return CNGP_OK;
}
int cngp_build_kprog(const cngp_kernel* k, cngp::KProg* kp) { return build_kprog(k, kp); }

// ------------------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------------------
extern "C" int cngp_version(void) { return CNGP_VERSION; }

extern "C" void cngp_default_config(cngp_config* cfg) {
  memset(cfg, 0, sizeof *cfg);
  cfg->device = 0;
  cfg->jitter_retry = 0;
  cfg->scratch_bytes = 0;
}

extern "C" int cngp_create(const cngp_config* cfg, cngp_ctx** out) {
  if (!out) return fail(nullptr, CNGP_ERR_INVALID, "cngp_create: out is null");
  *out = nullptr;
  cngp_config c;
  if (cfg) c = *cfg; else cngp_default_config(&c);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, CNGP_ERR_CUDA, "cngp_create: no CUDA device (%s) - libcngp has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (c.device < 0 || c.device >= ndev) return fail(nullptr, CNGP_ERR_INVALID, "cngp_create: bad device %d", c.device);
  if (c.precision != CNGP_PRECISION_F64 && c.precision != CNGP_PRECISION_F32)
    return fail(nullptr, CNGP_ERR_INVALID, "cngp_create: unknown precision mode %d", c.precision);
  CU(nullptr, cudaSetDevice(c.device));
  cudaDeviceProp prop;
  CU(nullptr, cudaGetDeviceProperties(&prop, c.device));
  if (prop.major != 10)
    return fail(nullptr, CNGP_ERR_UNSUPPORTED, "cngp_create: device %s is sm_%d%d; this library is built for sm_100a only",
                prop.name, prop.major, prop.minor);
  g_sm_count = prop.multiProcessorCount;
  cngp_ctx* ctx = new cngp_ctx();
  ctx->cfg = c;
  if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return fail(nullptr, CNGP_ERR_CUDA, "cngp_create: cudaStreamCreate failed");
  }
  ctx->stream = ctx->own_stream;
  ctx->scratch_bytes = c.scratch_bytes > 0 ? (size_t)c.scratch_bytes : ((size_t)2 << 30);
  *out = ctx;
  return CNGP_OK;
}

extern "C" void cngp_destroy(cngp_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->cfg.device);
  cudaStreamSynchronize(ctx->stream);
  ctx->collect();
  for (auto e : ctx->event_pool) cudaEventDestroy(e);
  for (auto& b : ctx->bufs)
    if (b.p) cudaFree(b.p);
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
}

extern "C" const char* cngp_last_error(cngp_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int cngp_sync(cngp_ctx* ctx) {
  if (!ctx) return CNGP_ERR_INVALID;
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return CNGP_OK;
}

extern "C" int cngp_set_stream(cngp_ctx* ctx, void* s, int32_t use_own) {
  if (!ctx) return CNGP_ERR_INVALID;
  ctx->collect();
  ctx->stream = use_own ? ctx->own_stream : (cudaStream_t)s;  // s == 0 is the legacy default stream
  return CNGP_OK;
}

extern "C" int cngp_set_precision(cngp_ctx* ctx, int32_t precision) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (precision != CNGP_PRECISION_F64 && precision != CNGP_PRECISION_F32) return fail(ctx, CNGP_ERR_INVALID, "set_precision: unknown mode %d", precision);
  ctx->cfg.precision = precision;
  return CNGP_OK;
}

extern "C" int64_t cngp_launch_count(cngp_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int cngp_set_profiling(cngp_ctx* ctx, int32_t on) {
  if (!ctx) return CNGP_ERR_INVALID;
  ctx->collect();
  ctx->profiling = on != 0;
  return CNGP_OK;
}

extern "C" int cngp_profile_read(cngp_ctx* ctx, int32_t kernel_id, double* total_ms, int64_t* launches, int32_t reset) {
  if (!ctx || kernel_id < 0 || kernel_id >= CNGP_PROF_KERNELS) return CNGP_ERR_INVALID;
  ctx->collect();
  if (total_ms) *total_ms = ctx->prof_ms[kernel_id];
  if (launches) *launches = ctx->prof_n[kernel_id];
  if (reset) { ctx->prof_ms[kernel_id] = 0.0; ctx->prof_n[kernel_id] = 0; }
  return CNGP_OK;
}

static int ensure_scratch(cngp_ctx* ctx) {
  if (ctx->scratch) return CNGP_OK;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  cudaError_t e = cudaMalloc((void**)&ctx->scratch, ctx->scratch_bytes);
  if (e != cudaSuccess) {
    ctx->scratch = nullptr;
    return fail(ctx, CNGP_ERR_NOMEM, "scratch allocation of %zu bytes failed: %s", ctx->scratch_bytes,
                cudaGetErrorString(e));
  }
  return CNGP_OK;
}

// staging helpers for host-memory calls
struct Stage {
  cngp_ctx* ctx;
  int mem;
  size_t slot = 0;
  int err = CNGP_OK;
  struct Out { void* host; void* dev; size_t bytes; };
  std::vector<Out> outs;
  const void* in(const void* host, size_t bytes) {
    if (!host || bytes == 0) return host;
    if (mem == CNGP_MEM_DEVICE) return host;
    void* d = ctx->buf(slot++, bytes);
    if (!d) { err = CNGP_ERR_NOMEM; return nullptr; }
    if (cudaMemcpyAsync(d, host, bytes, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) err = CNGP_ERR_CUDA;
    return d;
  }
  void* out(void* host, size_t bytes) {
    if (!host || bytes == 0) return host;
    if (mem == CNGP_MEM_DEVICE) return host;
    void* d = ctx->buf(slot++, bytes);
    if (!d) { err = CNGP_ERR_NOMEM; return nullptr; }
    outs.push_back({host, d, bytes});
    return d;
  }
  const void* in_alloc(const void* host, size_t bytes) {   // device room only: the caller issues the copies
    if (!host || bytes == 0 || mem == CNGP_MEM_DEVICE) return host;
    void* d = ctx->buf(slot++, bytes);
    if (!d) err = CNGP_ERR_NOMEM;
    return d;
  }
  void forget(void* host) {   // this output is copied home by the caller
    for (auto& o : outs)
      if (o.host == host) o.bytes = 0;
  }
  int finish() {
    if (mem == CNGP_MEM_DEVICE) return err;
    for (auto& o : outs)
      if (o.bytes && cudaMemcpyAsync(o.host, o.dev, o.bytes, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) err = CNGP_ERR_CUDA;
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) err = CNGP_ERR_CUDA;
    return err;
  }
};

// ------------------------------------------------------------------------------------------------------------
// batched predict
// ------------------------------------------------------------------------------------------------------------
template <int NT_MAX, int G, int WG, int NSLOT, int CT, int KID, bool TAB = false>
static int launch_var_k(cngp_ctx* ctx, VarArgs& va, long long nwin, cudaStream_t s) {
  const long long nrounds = (va.mt - va.mt0 + WG - 1) / WG;
  const long long units = nwin * nrounds;
  const long long grid = std::min<long long>((units + G - 1) / G, g_sm_count);   // persistent: one CTA per SM
  const size_t smem = var_smem_bytes(G, WG, NSLOT, CT);
  if (KID == KID_GENERIC && !TAB) {
    va.kstage = (double*)ctx->buf(12, (size_t)grid * G * WG * NT_MAX * 64 * sizeof(double));
    if (!va.kstage) return CNGP_ERR_NOMEM;
  }
  const bool full = va.nt == NT_MAX && va.N == NT_MAX * 8 && !va.n_win;
  auto kfn = full ? gp_var_kernel<NT_MAX, G, WG, NSLOT, CT, KID, true, TAB> : gp_var_kernel<NT_MAX, G, WG, NSLOT, CT, KID, false, TAB>;
  cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kfn<<<(unsigned)grid, G * WG * 32, smem, s>>>(va);
  return CNGP_OK;
}
template <int NT_MAX, int G, int WG, int NSLOT, int CT>
static int launch_var(cngp_ctx* ctx, int kid, VarArgs& va, long long nwin, cudaStream_t s) {
  if (va.n_lazy) {
    // Stationary expression: the lag-table kernel and the lazy kernel are both launched; phase A counted the windows
    // without a valid table (non-integer stamps) and exactly one of the two runs, the other returns at once.
    const int rc = launch_var_k<NT_MAX, G, WG, NSLOT, CT, KID_RBF, true>(ctx, va, nwin, s);
    if (rc) return rc;
    ctx->launches++;
  }
  switch (kid) {
    case KID_RBF: return launch_var_k<NT_MAX, G, WG, NSLOT, CT, KID_RBF>(ctx, va, nwin, s);
    case KID_RBF_PER: return launch_var_k<NT_MAX, G, WG, NSLOT, CT, KID_RBF_PER>(ctx, va, nwin, s);
    case KID_RBF_BROWN: return launch_var_k<NT_MAX, G, WG, NSLOT, CT, KID_RBF_BROWN>(ctx, va, nwin, s);
    default: return launch_var_k<NT_MAX, G, WG, NSLOT, CT, KID_GENERIC>(ctx, va, nwin, s);
  }
}
// FP32 mode: ten warps x 16 test points per round (M = 600 -> 38 sixteen-point tiles -> 4 rounds, 95 % of the slots used)
template <int NT_MAX>
static int launch_var32(cngp_ctx* ctx, VarArgs& va, long long nwin, cudaStream_t s) {
  constexpr int WG = 10, NSLOT = 3, CT = 64;
  va.mt = (va.M + 15) / 16;
  va.mt0 = 0;
  const long long nrounds = (va.mt + WG - 1) / WG;
  const long long units = nwin * nrounds;
  const long long grid = std::min<long long>(units, g_sm_count);
  const size_t smem = var32_smem_bytes(NSLOT, CT);
  va.kstage = (double*)ctx->buf(12, (size_t)grid * WG * NT_MAX * 32 * 16);
  if (!va.kstage) return CNGP_ERR_NOMEM;
  const bool full = va.nt == NT_MAX && va.N == NT_MAX * 8 && !va.n_win;
  auto kfn = full ? gp_var32_kernel<NT_MAX, WG, NSLOT, CT, true> : gp_var32_kernel<NT_MAX, WG, NSLOT, CT, false>;
  cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kfn<<<(unsigned)grid, WG * 32, smem, s>>>(va);
  return CNGP_OK;
}

template <int KID, int NW, int T>
static void launch_fit_k(const FitArgs& fa, long long nprob, cudaStream_t s) {
  const size_t smem = fit_smem_bytes(fa.nt, NW * T);
  cudaFuncSetAttribute(gp_fit_kernel<KID, NW, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  gp_fit_kernel<KID, NW, T><<<(unsigned)nprob, (NW + 1) * 32, smem, s>>>(fa);   // NW workers + the diagonal warp
}
template <int KID>
static void launch_fit_w(const FitArgs& fa, long long nprob, cudaStream_t s) {
  // row tiles (nt) must fit NW workers x T slots
  if (fa.nt <= 8) launch_fit_k<KID, 4, 2>(fa, nprob, s);
  else if (fa.nt <= 16) launch_fit_k<KID, 8, 2>(fa, nprob, s);
  else if (fa.nt <= 18) launch_fit_k<KID, 9, 2>(fa, nprob, s);   // the reference's own window (134 of 149 samples): two CTAs per SM
  else launch_fit_k<KID, FIT_NW_FULL, FIT_T_FULL>(fa, nprob, s);
}
template <int KID>
static void launch_fit_toeplitz(const FitArgs& fa, long long nprob, cudaStream_t s) {
  const size_t smem = toep_smem_bytes(fa.nt);
  cudaFuncSetAttribute(gp_fit_toeplitz_kernel<KID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  gp_fit_toeplitz_kernel<KID><<<(unsigned)((nprob + TOEP_WARPS - 1) / TOEP_WARPS), TOEP_WARPS * 32, smem, s>>>(fa, nprob);
}
// Phase A of a chunk.  With lag tables on and more problems than SMs, gp_fit_toeplitz_kernel first takes the windows
// whose Ky is Toeplitz (uniform integer stamps) and well conditioned, and marks them in done (slot SLOT_FIT_DONE,
// [n_problems], merged with fa.skip); gp_fit_kernel then factors the others.  Up to one problem per SM gp_fit_kernel
// finishes the whole chunk in its single-window time, which is shorter than one warp's Schur recursion (one N = 100
// window on a B200: 36 us against 89 us); beyond that its waves run one after the other and the Schur path wins
// (4096 windows of N = 256: 0.57 ms against 2.37 ms).
enum { SLOT_FIT_DONE = 26 };
static int launch_fit(cngp_ctx* ctx, int kid, const FitArgs& fa_in, long long n_problems, long long nprob, cudaStream_t s) {
  FitArgs fa = fa_in;
  if (fa.lag_ok && kid != KID_RBF_BROWN && nprob > g_sm_count) {
    fa.done = (int*)ctx->buf(SLOT_FIT_DONE, sizeof(int) * (size_t)n_problems);
    if (!fa.done) return CNGP_ERR_NOMEM;
    // the features of KID_RBF are those of the interpreter: only the periodic phases need their own instance
    if (kid == KID_RBF_PER) launch_fit_toeplitz<KID_RBF_PER>(fa, nprob, s);
    else launch_fit_toeplitz<KID_GENERIC>(fa, nprob, s);
    ctx->launches++;
    fa.skip = fa.done;
  }
  switch (kid) {
    case KID_RBF: launch_fit_w<KID_RBF>(fa, nprob, s); break;
    case KID_RBF_PER: launch_fit_w<KID_RBF_PER>(fa, nprob, s); break;
    case KID_RBF_BROWN: launch_fit_w<KID_RBF_BROWN>(fa, nprob, s); break;
    default: launch_fit_w<KID_GENERIC>(fa, nprob, s); break;
  }
  return CNGP_OK;
}

// Phase B of a chunk, first step.  With lag tables on, FP64 and more windows than SMs (the gate of the Schur fit),
// gp_var_toeplitz_kernel takes the windows whose Ky is Toeplitz and whose test points lie on the training lattice, and
// marks them in taken (slot SLOT_VAR_TAKEN, [nw]); var_compact_kernel lists the others (slot SLOT_VAR_LIST: count, then
// the list) for gp_var_kernel.  On one window the warp's recurrence is latency-bound, and gp_var_kernel's single window
// is spread over a whole SM, so below the gate every window stays on gp_var_kernel.
enum { SLOT_VAR_TAKEN = 27, SLOT_VAR_LIST = 28 };
static int launch_var_toeplitz(cngp_ctx* ctx, VarArgs& va, long long nw, cudaStream_t s) {
  int* taken = (int*)ctx->buf(SLOT_VAR_TAKEN, sizeof(int) * (size_t)nw);
  int* lst = (int*)ctx->buf(SLOT_VAR_LIST, sizeof(int) * ((size_t)nw + 32));
  if (!taken || !lst) return CNGP_ERR_NOMEM;
  const size_t smem = tvt_smem_bytes(va.nt, va.M);
  cudaFuncSetAttribute(gp_var_toeplitz_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  gp_var_toeplitz_kernel<<<(unsigned)((nw + TVT_WARPS - 1) / TVT_WARPS), TVT_WARPS * 32, smem, s>>>(va, taken);
  var_compact_kernel<<<1, 1024, 0, s>>>(taken, nw, lst + 32, lst);
  ctx->launches += 2;
  va.list = lst + 32;
  va.list_count = lst;
  return CNGP_OK;
}

// Shared covariance (gp_toep_group.cuh, DESIGN.md section 4.2d).  Under the gate of the Toeplitz kernels and with one
// theta for the whole call, the chunk's largest group of windows with the same key is factored once: the key and group
// kernels, the group's Schur fit into a slot of its own (slot SLOT_TG_DATA: factor | z | L_jj | table | meta |
// integer stamps | variance row | mean row | log det) and the member kernel, which clears flag (slot SLOT_TG_FLAG,
// [n_windows]) for whatever goes back to the per-window kernels.  Those then run with flag as their skip list.
enum { SLOT_TG_KEY = 29, SLOT_TG_FLAG = 30, SLOT_TG_LIST = 31, SLOT_TG_REC = 32, SLOT_TG_DATA = 33 };
struct TGroup {
  int* flag = nullptr;
  int* list = nullptr;
  int* rec = nullptr;
  double* gvar = nullptr;
};
static int launch_toep_group(cngp_ctx* ctx, const FitArgs& fa, const VarArgs& va, const int* m_win, long long B,
                             long long nw, TGroup& tg, cudaStream_t s) {
  const int nt = fa.nt, R = 8 * nt, M = fa.M;
  int4* key = (int4*)ctx->buf(SLOT_TG_KEY, sizeof(int4) * (size_t)nw);
  tg.flag = (int*)ctx->buf(SLOT_TG_FLAG, sizeof(int) * (size_t)B);
  tg.list = (int*)ctx->buf(SLOT_TG_LIST, sizeof(int) * (size_t)nw);
  tg.rec = (int*)ctx->buf(SLOT_TG_REC, sizeof(int) * TG_INTS);
  const size_t nd = (size_t)tiles_in_lower(nt) * 64 + R + (size_t)nt * 64 + VAR_TAB_MAX + VAR_META + R / 2 + 2 * (size_t)M + 1;
  double* gd = (double*)ctx->buf(SLOT_TG_DATA, sizeof(double) * nd);
  if (!key || !tg.flag || !tg.list || !tg.rec || !gd) return CNGP_ERR_NOMEM;
  double* gL = gd;
  double* gz = gL + (size_t)tiles_in_lower(nt) * 64;
  double* gdiag = gz + R;
  double* gtab = gdiag + (size_t)nt * 64;
  double* gmeta = gtab + VAR_TAB_MAX;
  int* gxi = (int*)(gmeta + VAR_META);
  tg.gvar = gmeta + VAR_META + R / 2;
  double* gmean = tg.gvar + M;
  double* glogdet = gmean + M;

  toep_key_kernel<<<(unsigned)((nw + TG_KEY_WARPS - 1) / TG_KEY_WARPS), TG_KEY_WARPS * 32, 0, s>>>(fa, m_win, nw, key);
  toep_group_kernel<<<1, 1024, 0, s>>>(key, nw, fa.problem0, tg.flag, tg.list, tg.rec);
  // the one-window fit: the first member's stamps, y = 0
  FitArgs g = fa;
  g.problem0 = 0; g.win_map = tg.rec + TG_REP; g.skip = tg.rec + TG_NONE; g.theta_mode = 0;
  g.y = nullptr; g.L = gL; g.z = gz; g.feat = nullptr; g.lml = nullptr; g.logdet = glogdet; g.quad = nullptr;
  g.status = nullptr; g.ktab = gtab; g.kmeta = gmeta; g.kxi = gxi; g.n_lazy = nullptr; g.done = tg.rec + TG_FIT;
  g.ldiag = gdiag; g.f32_factor = 0;
#ifdef CNGP_TG_TIMING
  {
    unsigned long long z[16] = {};
    z[10] = ~0ull;
    cudaMemcpyToSymbolAsync(tg_stamp, z, sizeof z, 0, cudaMemcpyHostToDevice, s);
  }
#endif
  const size_t fsmem = tgf_smem_bytes(nt);
  cudaFuncSetAttribute(gp_toep_group_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem);
  gp_toep_group_fit_kernel<<<1, TGF_THREADS, fsmem, s>>>(g);
  ctx->launches += 2;   // + the begin() below that re-opens the fit span
  ctx->end();
  ctx->begin(CNGP_PROF_VAR);
  TGArgs t;
  memset(&t, 0, sizeof t);
  t.g = va;
  t.g.L = gL; t.g.z = gz; t.g.ktab = gtab; t.g.kmeta = gmeta; t.g.kxi = gxi; t.g.status = nullptr;
  t.ldiag = gdiag; t.logdet = glogdet; t.gvar = tg.gvar; t.gmean = gmean;
  t.y = fa.y; t.lml = fa.lml; t.status = fa.status; t.mean = va.mean; t.flag = tg.flag; t.list = tg.list; t.rec = tg.rec;
  t.w0 = fa.problem0;
  const size_t smem = tg_smem_bytes(nt, M);
  cudaFuncSetAttribute(gp_toep_member_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  gp_toep_member_kernel<<<(unsigned)(1 + (nw + TG_WARPS - 1) / TG_WARPS), TG_WARPS * 32, smem, s>>>(t);
#ifdef CNGP_TG_TIMING
  {
    unsigned long long h[16];
    cudaStreamSynchronize(s);
    cudaMemcpyFromSymbol(h, tg_stamp, sizeof h);
    auto us = [&](int i, int from) { return h[i] ? 1e-3 * (double)(long long)(h[i] - h[from]) : -1.0; };
    fprintf(stderr, "tg_timing fit_us prologue %.1f generators %.1f recursion %.1f outputs %.1f end %.1f"
            " | member_us var_row %.1f members_start %.1f z %.1f alpha %.1f members_end %.1f\n",
            us(1, 0), us(2, 0), us(3, 0), us(4, 0), us(5, 0), us(9, 8), us(10, 8), us(12, 8), us(13, 8), us(11, 8));
  }
#endif
  ctx->end();
  ctx->begin(CNGP_PROF_FIT);
  return CNGP_OK;
}

// every leaf a function of |x - x'| only (White: zero off the diagonal) - what the lag tables of gp_fit.cuh need
static bool kprog_stationary(const KProg& kp) {
  for (int u = 0; u < kp.n_leaves; ++u)
    if (kp.leaf_type[u] == CNGP_K_BROWNIAN || kp.leaf_type[u] == CNGP_K_LINEAR) return false;
  return true;
}
static bool lag_tables_enabled() {
  const char* e = getenv("CNGP_NO_LAG_TABLES");   // tests force the lazy path with it
  return !(e && atoi(e));
}

int cngp_predict_impl(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                      const double* x, const double* y, const double* xstar, int64_t xstar_stride, int64_t B, int32_t N,
                      int32_t M, double* mean, double* var, double* lml, int32_t* status, int32_t mem, int sigma_mode,
                      const int32_t* n_win, const int32_t* m_win) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !theta || !x || !y || B < 0 || N <= 0 || M < 0) return fail(ctx, CNGP_ERR_INVALID, "predict: bad argument");
  if (M > 0 && (!xstar || !mean || !var)) return fail(ctx, CNGP_ERR_INVALID, "predict: xstar/mean/var null");
  if (N > CNGP_MAX_N) return fail(ctx, CNGP_ERR_UNSUPPORTED, "predict: N=%d > %d (use cngp_chol_large)", N, CNGP_MAX_N);
  if (B == 0) return CNGP_OK;
  KProg kp;
  int rc = build_kprog(kernel, &kp);
  if (rc) return fail(ctx, rc, "predict: invalid kernel expression");
  const int P = kp.n_params + 1;
  if (theta_stride != 0 && theta_stride < P) return fail(ctx, CNGP_ERR_INVALID, "predict: theta_stride < n_params+1");
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if ((rc = ensure_scratch(ctx))) return rc;

  Stage st{ctx, mem};
  // Host-memory calls work in slabs: x / y of slab k+1 arrive and mean / var of slab k-1 leave on a second stream while
  // slab k computes (16 x (N + M) bytes per window cross PCIe).
  const bool pipelined = mem == CNGP_MEM_HOST && M > 0 && B >= 1024;
  const double* d_theta = (const double*)st.in(theta, sizeof(double) * (theta_stride ? (size_t)B * theta_stride : P));
  const double* d_x = (const double*)(pipelined ? st.in_alloc(x, sizeof(double) * (size_t)B * N) : st.in(x, sizeof(double) * (size_t)B * N));
  const double* d_y = (const double*)(pipelined ? st.in_alloc(y, sizeof(double) * (size_t)B * N) : st.in(y, sizeof(double) * (size_t)B * N));
  const double* d_xs = M ? (const double*)st.in(xstar, sizeof(double) * (xstar_stride ? (size_t)B * xstar_stride : M)) : nullptr;
  double* d_mean = M ? (double*)st.out(mean, sizeof(double) * (size_t)B * M) : nullptr;
  double* d_var = M ? (double*)st.out(var, sizeof(double) * (size_t)B * M) : nullptr;
  double* d_lml = (double*)st.out(lml, sizeof(double) * (size_t)B);
  int* d_status = (int*)st.out(status, sizeof(int) * (size_t)B);
  if (st.err) return fail(ctx, st.err, "predict: staging failed");
  if (!d_status) {  // phase B needs the status to poison failed windows
    d_status = (int*)ctx->buf(15, sizeof(int) * (size_t)B);
    if (!d_status) return fail(ctx, CNGP_ERR_NOMEM, "predict: status buffer");
  }

  const int nt = (N + 7) / 8, mt = (M + 7) / 8;
  const int kid = match_fast_kernel(kp);
  const bool lag_ok = kprog_stationary(kp) && lag_tables_enabled();
  const size_t per_problem = ((size_t)tiles_in_lower(nt) * 64 + (size_t)nt * 8 * 5 +
                              (lag_ok ? (size_t)VAR_TAB_MAX + VAR_META + (size_t)nt * 4 : 0)) * sizeof(double);
  int* d_nlazy = nullptr;
  if (lag_ok && !(d_nlazy = (int*)ctx->buf(16, 256))) return fail(ctx, CNGP_ERR_NOMEM, "predict: flag buffer");
  const size_t slack = 64 * 64;   // >= the largest chunk (tiles x 64 doubles)   // gp_var_kernel's first (partial) chunk may start before the first tile
  if (ctx->scratch_bytes < slack * 8 + per_problem)
    return fail(ctx, CNGP_ERR_NOMEM, "predict: scratch_bytes = %zu cannot hold one window (%zu bytes needed)",
                ctx->scratch_bytes, slack * 8 + per_problem);
  long long chunk = (long long)((ctx->scratch_bytes - slack * 8) / per_problem);
  cudaEvent_t pending_inputs = nullptr;
  auto send_inputs = [&](long long w0, long long nw, cudaStream_t s) -> int {   // x, y of the slab [w0, w0 + nw)
    if (w0 >= B || nw <= 0) return 0;
    const size_t off = (size_t)w0 * N, bytes = sizeof(double) * (size_t)nw * N;
    if (cudaMemcpyAsync((double*)d_x + off, x + off, bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) return 1;
    if (cudaMemcpyAsync((double*)d_y + off, y + off, bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) return 1;
    return 0;
  };
  if (pipelined) {
    if (!ctx->copy_stream && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess)
      return fail(ctx, CNGP_ERR_CUDA, "predict: cudaStreamCreate failed");
    st.forget(mean);
    st.forget(var);
  }
  // Slab schedule.  Device calls: as many windows as the scratch holds.  Pipelined host calls: what cannot overlap is the
  // upload of the FIRST slab and the download of the LAST one, so those two are short (about two waves of the
  // one-CTA-per-window factorisation) and the slabs in between long, all but the last a multiple of the SM count.
  std::vector<std::pair<long long, long long>> slabs;
  {
    const long long sm = g_sm_count;
    const long long head = 2 * sm, mid = ((B - head) / 3 / sm) * sm;
    if (pipelined && mid >= 2 * sm && mid <= chunk) {
      slabs.push_back({0, head});
      for (int k = 0; k < 3; ++k) slabs.push_back({head + k * mid, mid});
      if (head + 3 * mid < B) slabs.push_back({head + 3 * mid, B - head - 3 * mid});
    } else {
      if (pipelined) chunk = std::min<long long>(chunk, (B + 3) / 4);
      for (long long w0 = 0; w0 < B; w0 += chunk) slabs.push_back({w0, std::min<long long>(chunk, B - w0)});
    }
  }
  if (pipelined && send_inputs(slabs[0].first, slabs[0].second, ctx->stream))
    return fail(ctx, CNGP_ERR_CUDA, "predict: input copy failed");
  for (size_t si = 0; si < slabs.size(); ++si) {
    const long long w0 = slabs[si].first, nw = slabs[si].second;
    if (pipelined && si + 1 < slabs.size()) {   // next slab's inputs travel while this slab computes
      if (send_inputs(slabs[si + 1].first, slabs[si + 1].second, ctx->copy_stream)) return fail(ctx, CNGP_ERR_CUDA, "predict: input copy failed");
      cudaEvent_t arrived = ctx->get_event();
      CU(ctx, cudaEventRecord(arrived, ctx->copy_stream));
      pending_inputs = arrived;
    }
    double* Lbuf = ctx->scratch + slack;
    double* zbuf = Lbuf + (size_t)nw * tiles_in_lower(nt) * 64;
    double* fbuf = zbuf + (size_t)nw * nt * 8;
    double* tbuf = fbuf + (size_t)nw * nt * 8 * 4;                 // lag tables | meta | integer stamps
    double* mbuf = tbuf + (size_t)nw * VAR_TAB_MAX;
    int* xibuf = (int*)(mbuf + (size_t)nw * VAR_META);
    FitArgs fa;
    memset(&fa, 0, sizeof fa);
    fa.kp = kp;
    fa.theta = d_theta; fa.theta_stride = theta_stride; fa.theta_mode = theta_stride ? 1 : 0;
    fa.win_map = nullptr;
    if (lag_ok) {
      fa.lag_ok = 1;
      fa.xstar = d_xs; fa.xstar_stride = xstar_stride; fa.M = M;
      fa.ktab = M > 0 ? tbuf : nullptr; fa.kmeta = M > 0 ? mbuf : nullptr; fa.kxi = xibuf; fa.n_lazy = d_nlazy;
      CU(ctx, cudaMemsetAsync(d_nlazy, 0, sizeof(int), ctx->stream));
    }
    const bool f32 = ctx->cfg.precision == CNGP_PRECISION_F32;
    fa.f32_factor = (f32 && M > 0) ? 1 : 0;
    fa.x = d_x; fa.y = d_y; fa.N = N; fa.nt = nt; fa.n_windows = (int)B; fa.problem0 = w0;
    fa.L = Lbuf; fa.z = zbuf; fa.feat = fbuf; fa.lml = d_lml; fa.logdet = nullptr; fa.quad = nullptr;
    fa.status = d_status;
    fa.jitter_retry = ctx->cfg.jitter_retry;
    fa.Asrc = nullptr; fa.a_col_stride = 0;
    fa.n_win = n_win;
    VarArgs va;
    memset(&va, 0, sizeof va);
    // the gate of the Toeplitz kernels (launch_fit, launch_var_toeplitz), one theta for the call
    const bool toep = !f32 && lag_ok && nw > g_sm_count && M > 0;
    const bool grouped = toep && theta_stride == 0;
    TGroup tg;
    ctx->begin(CNGP_PROF_FIT);
    if (M > 0) {
      va.kp = kp;
      va.ktab = tbuf; va.kmeta = mbuf; va.kxi = xibuf; va.n_lazy = lag_ok ? d_nlazy : nullptr;
      va.theta = d_theta; va.theta_stride = theta_stride; va.theta_mode = theta_stride ? 1 : 0;
      va.xstar = d_xs; va.xstar_stride = xstar_stride;
      va.N = N; va.nt = nt; va.M = M; va.mt = mt; va.mt0 = 0; va.window0 = w0; va.n_windows_launch = nw;
      va.L = Lbuf; va.z = zbuf; va.feat = fbuf; va.status = d_status; va.mean = d_mean; va.var = d_var;
      va.sigma_mode = sigma_mode;
      va.kstage = nullptr;
      va.n_win = n_win; va.m_win = m_win;
    }
    if (grouped) {
      rc = launch_toep_group(ctx, fa, va, m_win, B, nw, tg, ctx->stream);
      if (rc) {
        ctx->end();
        return fail(ctx, rc, "predict: shared-covariance buffers");
      }
      fa.skip = tg.flag;
      va.skip = tg.flag;
    }
    rc = launch_fit(ctx, kid, fa, B, nw, ctx->stream);
    ctx->end();
    if (rc) return fail(ctx, rc, "predict: flag buffer");
    if (M > 0) {
      ctx->begin(CNGP_PROF_VAR);
      int vrc = CNGP_OK;
      if (toep) vrc = launch_var_toeplitz(ctx, va, nw, ctx->stream);
      if (vrc) {
        ctx->end();
        return fail(ctx, vrc, "predict: flag buffer");
      }
      if (f32) {
        va.n_lazy = nullptr;
        va.kmeta = lag_ok ? mbuf : nullptr;      // the FP32 kernel picks table or interpreter per window
        if (nt <= 8) vrc = launch_var32<8>(ctx, va, nw, ctx->stream);
        else if (nt <= 16) vrc = launch_var32<16>(ctx, va, nw, ctx->stream);
        else vrc = launch_var32<32>(ctx, va, nw, ctx->stream);
      }
      else if (nt <= 8) vrc = launch_var<8, 1, 16, 6, 16>(ctx, kid, va, nw, ctx->stream);
      else if (nt <= 16) vrc = launch_var<16, 1, 16, 6, 16>(ctx, kid, va, nw, ctx->stream);
#ifdef CNGP_VAR_TUNE   // tuning builds only: alternative shapes selected by the environment
      else if (getenv("CNGP_VAR_VARIANT") && atoi(getenv("CNGP_VAR_VARIANT")) == 1) vrc = launch_var<32, 1, 12, 4, 32>(ctx, kid, va, nw, ctx->stream);
      else if (getenv("CNGP_VAR_VARIANT") && atoi(getenv("CNGP_VAR_VARIANT")) == 2) vrc = launch_var<32, 1, 12, 6, 32>(ctx, kid, va, nw, ctx->stream);
      else if (getenv("CNGP_VAR_VARIANT") && atoi(getenv("CNGP_VAR_VARIANT")) == 3) vrc = launch_var<32, 1, 12, 8, 16>(ctx, kid, va, nw, ctx->stream);
#endif
      else if (mt > 12 && mt % 12 >= 1 && mt % 12 <= 3) {
        // A round of 12 test tiles streams the factor once; a last round of 1..3 tiles would stream it for a quarter of
        // the warps.  Those tiles go to a second launch in which every CTA runs four groups of three warps, each
        // streaming the factor of a different window, so all twelve warps stay busy.
        va.mt = mt - mt % 12;
        vrc = launch_var<32, 1, 12, 3, 64>(ctx, kid, va, nw, ctx->stream);
        ctx->end();
        ctx->begin(CNGP_PROF_VAR);
        va.mt0 = va.mt; va.mt = mt;
        if (!vrc) vrc = launch_var<32, 4, 3, 3, 16>(ctx, kid, va, nw, ctx->stream);
      }
      else vrc = launch_var<32, 1, 12, 3, 64>(ctx, kid, va, nw, ctx->stream);
      if (grouped && !vrc) {
        toep_var_broadcast_kernel<<<(unsigned)((nw + 3) / 4), 128, 0, ctx->stream>>>(tg.list, tg.rec, tg.flag, tg.gvar, d_var,
                                                                                     w0, M);
        ctx->launches++;
      }
      ctx->end();
      if (vrc) return fail(ctx, vrc, "predict: staging buffer for the generic kernel path");
    }
    CU(ctx, cudaGetLastError());
    if (pipelined) {
      cudaEvent_t done = ctx->get_event();
      CU(ctx, cudaEventRecord(done, ctx->stream));
      CU(ctx, cudaStreamWaitEvent(ctx->copy_stream, done, 0));
      const size_t off = (size_t)w0 * M, bytes = sizeof(double) * (size_t)nw * M;
      CU(ctx, cudaMemcpyAsync(mean + off, d_mean + off, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
      CU(ctx, cudaMemcpyAsync(var + off, d_var + off, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
      ctx->event_pool.push_back(done);   // its wait is enqueued: free for re-use
      if (pending_inputs) {               // the next slab may start once its inputs have landed
        CU(ctx, cudaStreamWaitEvent(ctx->stream, pending_inputs, 0));
        ctx->event_pool.push_back(pending_inputs);
        pending_inputs = nullptr;
      }
    }
  }
  rc = st.finish();
  if (pipelined && cudaStreamSynchronize(ctx->copy_stream) != cudaSuccess) rc = rc ? rc : CNGP_ERR_CUDA;
  if (rc) return fail(ctx, rc, "predict: copy-out failed: %s", cudaGetErrorString(cudaGetLastError()));
  return CNGP_OK;
}

extern "C" int cngp_predict_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t theta_stride,
                                  const double* x, const double* y, const double* xstar, int64_t xstar_stride,
                                  int64_t B, int32_t N, int32_t M, double* mean, double* var, double* lml,
                                  int32_t* status, int32_t mem) {
  return cngp_predict_impl(ctx, kernel, theta, theta_stride, x, y, xstar, xstar_stride, B, N, M, mean, var, lml, status,
                           mem, 0, nullptr, nullptr);
}

// ------------------------------------------------------------------------------------------------------------
// LML + gradient for C candidates x B windows (win_map == null), or for n_prob independent (theta row, window)
// problems: problem p uses theta row p and window win_map[p] of the B windows (C = n_prob then).
// ------------------------------------------------------------------------------------------------------------
int cngp_lml_grad_impl(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t C, const double* x,
                       const double* y, int64_t B, int32_t N, double* lml, double* grad, int32_t* status, int32_t mem,
                       const int32_t* win_map, const int32_t* skip, const int32_t* n_win) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !theta || !x || !y || C < 0 || B < 0 || N <= 0) return fail(ctx, CNGP_ERR_INVALID, "lml_grad: bad argument");
  if (N > CNGP_MAX_N) return fail(ctx, CNGP_ERR_UNSUPPORTED, "lml_grad: N=%d > %d", N, CNGP_MAX_N);
  if (C == 0 || B == 0) return CNGP_OK;
  KProg kp;
  int rc = build_kprog(kernel, &kp);
  if (rc) return fail(ctx, rc, "lml_grad: invalid kernel expression");
  const int P = kp.n_params + 1;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if ((rc = ensure_scratch(ctx))) return rc;
  const long long n_prob = win_map ? (long long)C : (long long)C * B;

  Stage st{ctx, mem};
  const double* d_theta = (const double*)st.in(theta, sizeof(double) * (size_t)C * P);
  const double* d_x = (const double*)st.in(x, sizeof(double) * (size_t)B * N);
  const double* d_y = (const double*)st.in(y, sizeof(double) * (size_t)B * N);
  const int* d_map = (const int*)st.in(win_map, sizeof(int) * (size_t)n_prob);
  double* d_lml = (double*)st.out(lml, sizeof(double) * (size_t)n_prob);
  double* d_grad = (double*)st.out(grad, sizeof(double) * (size_t)n_prob * P);
  int* d_status = (int*)st.out(status, sizeof(int) * (size_t)n_prob);
  if (st.err) return fail(ctx, st.err, "lml_grad: staging failed");
  if (!d_status) {
    d_status = (int*)ctx->buf(15, sizeof(int) * (size_t)n_prob);
    if (!d_status) return fail(ctx, CNGP_ERR_NOMEM, "lml_grad: status buffer");
  }

  const int nt = (N + 7) / 8;
  const size_t ltiles = (size_t)tiles_in_lower(nt) * 64;
  const size_t per_problem = (ltiles * ((grad && nt > GRAD_SMEM_NT) ? 2 : 1) + (size_t)nt * 8 * 2) * sizeof(double);   // W only for the global variant
  if (ctx->scratch_bytes < per_problem)
    return fail(ctx, CNGP_ERR_NOMEM, "lml_grad: scratch_bytes = %zu cannot hold one problem (%zu bytes needed)",
                ctx->scratch_bytes, per_problem);
  const long long chunk = (long long)(ctx->scratch_bytes / per_problem);
  for (long long p0 = 0; p0 < n_prob; p0 += chunk) {
    const long long np = std::min<long long>(chunk, n_prob - p0);
    double* Lbuf = ctx->scratch;
    double* Wbuf = Lbuf + (size_t)np * ltiles;
    double* zbuf = (grad && nt > GRAD_SMEM_NT) ? Wbuf + (size_t)np * ltiles : Wbuf;
    double* abuf = zbuf + (size_t)np * nt * 8;
    FitArgs fa;
    memset(&fa, 0, sizeof fa);
    fa.kp = kp;
    fa.lag_ok = (kprog_stationary(kp) && lag_tables_enabled()) ? 1 : 0;   // K(X,X) by integer lag when the stamps allow
    fa.skip = skip;
    fa.theta = d_theta; fa.theta_stride = P; fa.theta_mode = d_map ? 3 : 2;
    fa.win_map = d_map;
    fa.x = d_x; fa.y = d_y; fa.N = N; fa.nt = nt; fa.n_windows = (int)B; fa.problem0 = p0;
    fa.L = Lbuf; fa.z = zbuf; fa.feat = nullptr; fa.lml = d_lml; fa.logdet = nullptr; fa.quad = nullptr;
    fa.status = d_status;
    fa.jitter_retry = ctx->cfg.jitter_retry;
    fa.Asrc = nullptr; fa.a_col_stride = 0;
    fa.n_win = n_win;
    ctx->begin(CNGP_PROF_FIT);
    rc = launch_fit(ctx, match_fast_kernel(kp), fa, n_prob, np, ctx->stream);
    ctx->end();
    if (rc) return fail(ctx, rc, "lml_grad: flag buffer");
    if (grad) {
      GradArgs ga;
      ga.kp = kp;
      ga.theta = d_theta; ga.theta_stride = P; ga.win_map = d_map;
      ga.x = d_x; ga.N = N; ga.nt = nt; ga.n_windows = (int)B; ga.problem0 = p0;
      ga.L = Lbuf; ga.W = Wbuf; ga.z = zbuf; ga.alpha = abuf; ga.status = d_status; ga.grad = d_grad;
      ga.skip = skip;
      ga.n_win = n_win;
      // uniform-stamp contraction of gp_grad_kernel: stationary expressions, or few product terms with Brownian / Linear factors
      ga.lag_ok = fa.lag_ok ? 1 : ((lag_tables_enabled() && kp.n_terms <= GRAD_UNI_TERMS) ? 2 : 0);
      ctx->begin(CNGP_PROF_GRAD);
      if (nt <= GRAD_SMEM_NT) {
        const size_t gsm = grad_smem_bytes(nt);
        cudaFuncSetAttribute(gp_grad_kernel<GRAD_WARPS_SMEM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm);
        gp_grad_kernel<GRAD_WARPS_SMEM, true><<<(unsigned)np, GRAD_WARPS_SMEM * 32, gsm, ctx->stream>>>(ga);
      } else {
        gp_grad_kernel<GRAD_WARPS_GLOBAL, false><<<(unsigned)np, GRAD_WARPS_GLOBAL * 32, 0, ctx->stream>>>(ga);
      }
      ctx->end();
    }
    CU(ctx, cudaGetLastError());
  }
  rc = st.finish();
  if (rc) return fail(ctx, rc, "lml_grad: copy-out failed: %s", cudaGetErrorString(cudaGetLastError()));
  return CNGP_OK;
}

extern "C" int cngp_lml_grad_batch(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t C,
                                   const double* x, const double* y, int64_t B, int32_t N, double* lml, double* grad,
                                   int32_t* status, int32_t mem) {
  return cngp_lml_grad_impl(ctx, kernel, theta, C, x, y, B, N, lml, grad, status, mem, nullptr);
}

extern "C" int cngp_lml_grad_windows(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, int64_t n_problems,
                                     const int32_t* window_of_problem, const double* x, const double* y, int64_t B,
                                     int32_t N, double* lml, double* grad, int32_t* status, int32_t mem) {
  if (!window_of_problem) return ctx ? fail(ctx, CNGP_ERR_INVALID, "lml_grad_windows: window_of_problem is null") : CNGP_ERR_INVALID;
  return cngp_lml_grad_impl(ctx, kernel, theta, n_problems, x, y, B, N, lml, grad, status, mem, window_of_problem);
}

// ------------------------------------------------------------------------------------------------------------
// stop predictor
// ------------------------------------------------------------------------------------------------------------
extern "C" void cngp_default_stop_config(cngp_stop_config* c) {
  c->v_nom = 0.8; c->floor_a = 0.03; c->floor_b = 0.05; c->track = 0.685; c->scale = 25.0; c->thresh = 3.0;
  c->ratio = 5; c->fix_h_packing = 0;
  c->init_llh[0] = 0.693457963620326; c->init_llh[1] = -1.39498384275845; c->init_llh[2] = 334.993517334743;
  c->init_ecef[0] = 859153.015300000; c->init_ecef[1] = -4836303.72660000; c->init_ecef[2] = 4055378.50100000;
}

extern "C" int cngp_zupt_lookahead_batch(cngp_ctx* ctx, const double* mean, const double* sigma, int64_t B, int32_t M,
                                         const double* P, const double* Q, const double* STM, const double* Hvec,
                                         const double* pos, int32_t per_window, const cngp_stop_config* cfg,
                                         int32_t* triggered, int32_t* i_stop, int32_t* step_stop, double* xy_err,
                                         int32_t mem) {
  return cngp_zupt_lookahead_batch_ex(ctx, mean, sigma, B, M, P, Q, STM, Hvec, pos, per_window, cfg, triggered, i_stop,
                                      step_stop, xy_err, nullptr, nullptr, nullptr, mem);
}

namespace {
// any m[b] outside [0, ldm] sets *bad
__global__ void ragged_m_check_kernel(const int* m, long long B, int ldm, int* bad) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B && (m[b] < 0 || m[b] > ldm)) atomicOr(bad, 1);
}
}  // namespace

// M: points per window, or (m != null) the row stride of mean / sigma with m[b] <= M points in row b
static int lookahead_impl(cngp_ctx* ctx, const double* mean, const double* sigma, int64_t B, int32_t M, const int32_t* m,
                          const double* P, const double* Q, const double* STM, const double* Hvec, const double* pos,
                          int32_t per_window, const cngp_stop_config* cfg, int32_t* triggered, int32_t* i_stop,
                          int32_t* step_stop, double* xy_err, double* P_final, double* K_final, double* R_final,
                          int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if ((K_final || R_final) && !P_final) return fail(ctx, CNGP_ERR_INVALID, "lookahead: K_final / R_final need P_final");
  if (!mean || !sigma || !P || !Q || !STM || !Hvec || !pos || !triggered || !i_stop || B < 0 || M <= 0)
    return fail(ctx, CNGP_ERR_INVALID, "lookahead: bad argument");
  if (B == 0) return CNGP_OK;
  cngp_stop_config c;
  if (cfg) c = *cfg; else cngp_default_stop_config(&c);
  if (c.ratio <= 0) return fail(ctx, CNGP_ERR_INVALID, "lookahead: ratio must be positive");
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  Stage st{ctx, mem};
  const int* d_m = (const int*)st.in(m, sizeof(int) * (size_t)B);
  if (m) {   // every count within its row: one flag read back (device memory) or a host loop
    if (mem == CNGP_MEM_HOST) {
      for (int64_t b = 0; b < B; ++b)
        if (m[b] < 0 || m[b] > M) return fail(ctx, CNGP_ERR_INVALID, "lookahead_ragged: m[%lld] = %d outside [0, ldm = %d]", (long long)b, m[b], M);
    } else {
      int* d_bad = (int*)ctx->buf(20, 64);
      int bad = 0;
      if (!d_bad) return fail(ctx, CNGP_ERR_NOMEM, "lookahead_ragged: flag buffer");
      CU(ctx, cudaMemsetAsync(d_bad, 0, sizeof(int), ctx->stream));
      ragged_m_check_kernel<<<(unsigned)((B + 255) / 256), 256, 0, ctx->stream>>>(d_m, B, M, d_bad);
      CU(ctx, cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
      CU(ctx, cudaStreamSynchronize(ctx->stream));
      if (bad) return fail(ctx, CNGP_ERR_INVALID, "lookahead_ragged: some m[b] outside [0, ldm = %d]", M);
    }
  }
  auto cnt = [&](int bit, size_t sz) { return sizeof(double) * sz * ((per_window & bit) ? (size_t)B : 1); };
  const double* d_mean = (const double*)st.in(mean, sizeof(double) * (size_t)B * M);
  const double* d_sigma = (const double*)st.in(sigma, sizeof(double) * (size_t)B * M);
  const double* d_P = (const double*)st.in(P, cnt(CNGP_PERWIN_P, 225));
  const double* d_Q = (const double*)st.in(Q, cnt(CNGP_PERWIN_Q, 225));
  const double* d_F = (const double*)st.in(STM, cnt(CNGP_PERWIN_STM, 225));
  const double* d_H = (const double*)st.in(Hvec, cnt(CNGP_PERWIN_H, 60));
  const double* d_pos = (const double*)st.in(pos, cnt(CNGP_PERWIN_POS, 3));
  int* d_trig = (int*)st.out(triggered, sizeof(int) * (size_t)B);
  int* d_i = (int*)st.out(i_stop, sizeof(int) * (size_t)B);
  int* d_step = (int*)st.out(step_stop, sizeof(int) * (size_t)B);
  double* d_xy = (double*)st.out(xy_err, sizeof(double) * (size_t)B);
  if (st.err) return fail(ctx, st.err, "lookahead: staging failed");
  if (!d_step) d_step = (int*)ctx->buf(14, sizeof(int) * (size_t)B);
  if (!d_xy) d_xy = (double*)ctx->buf(13, sizeof(double) * (size_t)B);
  if (!d_step || !d_xy) return fail(ctx, CNGP_ERR_NOMEM, "lookahead: buffers");
  ctx->begin(CNGP_PROF_LOOKAHEAD);
  unsigned long long* d_counter = (unsigned long long*)ctx->buf(17, 64);
  if (!d_counter) return fail(ctx, CNGP_ERR_NOMEM, "lookahead: work counter");
  double* d_Pf = (double*)st.out(P_final, sizeof(double) * 225 * (size_t)B);
  double* d_Kf = (double*)st.out(K_final, sizeof(double) * 60 * (size_t)B);
  double* d_Rf = (double*)st.out(R_final, sizeof(double) * 16 * (size_t)B);
  if (st.err) return fail(ctx, st.err, "lookahead: staging failed");
  if (d_Kf) CU(ctx, cudaMemsetAsync(d_Kf, 0, sizeof(double) * 60 * (size_t)B, ctx->stream));   // windows without an update
  if (d_Rf) CU(ctx, cudaMemsetAsync(d_Rf, 0, sizeof(double) * 16 * (size_t)B, ctx->stream));
  const int e = cngp_launch_lookahead(d_mean, d_sigma, B, M, d_P, d_Q, d_F, d_H, d_pos, per_window, &c, d_trig, d_i,
                                      d_step, d_xy, d_counter, d_Pf, d_Kf, d_Rf, nullptr, 0, ctx->stream, d_m);
  ctx->end();
  if (e) return fail(ctx, CNGP_ERR_CUDA, "lookahead launch: %s", cudaGetErrorString((cudaError_t)e));
  const int rc = st.finish();
  if (rc) return fail(ctx, rc, "lookahead: copy-out failed: %s", cudaGetErrorString(cudaGetLastError()));
  return CNGP_OK;
}

extern "C" int cngp_zupt_lookahead_batch_ex(cngp_ctx* ctx, const double* mean, const double* sigma, int64_t B, int32_t M,
                                            const double* P, const double* Q, const double* STM, const double* Hvec,
                                            const double* pos, int32_t per_window, const cngp_stop_config* cfg,
                                            int32_t* triggered, int32_t* i_stop, int32_t* step_stop, double* xy_err,
                                            double* P_final, double* K_final, double* R_final, int32_t mem) {
  return lookahead_impl(ctx, mean, sigma, B, M, nullptr, P, Q, STM, Hvec, pos, per_window, cfg, triggered, i_stop,
                        step_stop, xy_err, P_final, K_final, R_final, mem);
}

extern "C" int cngp_zupt_lookahead_ragged(cngp_ctx* ctx, const double* mean, const double* sigma, int64_t B,
                                          const int32_t* m, int32_t ldm, const double* P, const double* Q,
                                          const double* STM, const double* Hvec, const double* pos, int32_t per_window,
                                          const cngp_stop_config* cfg, int32_t* triggered, int32_t* i_stop,
                                          int32_t* step_stop, double* xy_err, double* P_final, double* K_final,
                                          double* R_final, int32_t mem) {
  if (!m) return ctx ? fail(ctx, CNGP_ERR_INVALID, "lookahead_ragged: m is null") : CNGP_ERR_INVALID;
  return lookahead_impl(ctx, mean, sigma, B, ldm, m, P, Q, STM, Hvec, pos, per_window, cfg, triggered, i_stop, step_stop,
                        xy_err, P_final, K_final, R_final, mem);
}

// The filter's own covariance recursion for B operating points (SURVEY.md 8f row N4, the P half): n_steps IMU steps of
// P <- STM P STM' + Q (CoreNav.cpp:101) with the odometry update's Joseph form every `ratio`-th step
// (K = P H'(H P H' + R)^-1, P <- (I-KH) P (I-KH)' + K R K', CoreNav.cpp:226-230) - what stands in P_ when
// CoreNav::Update copies it to P_pred for the SetStopping service (CoreNav.cpp:291-292).  Runs on the tensor-core
// look-ahead kernel with the true 4 x 15 H (row-major), the filter's constant R and no error observer.
extern "C" int cngp_ekf_covariance_batch(cngp_ctx* ctx, const double* P0, const double* Q, const double* STM,
                                         const double* H, const double* R, int64_t B, int32_t n_steps, int32_t ratio,
                                         int32_t per_window, double* P_out, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!P0 || !Q || !STM || !H || !R || !P_out || B < 0 || n_steps <= 0 || ratio <= 0 || n_steps % ratio != 0)
    return fail(ctx, CNGP_ERR_INVALID, "ekf_covariance: bad argument (n_steps must be a positive multiple of ratio)");
  if (B == 0) return CNGP_OK;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  cngp_stop_config c;
  cngp_default_stop_config(&c);
  c.ratio = ratio;
  c.fix_h_packing = 1;                       // H is given as the true row-major 4 x 15 matrix
  c.thresh = 1e300;                          // no trigger: all n_steps are executed
  const int M = n_steps / ratio;
  Stage st{ctx, mem};
  auto cnt = [&](int bit, size_t sz) { return sizeof(double) * sz * ((per_window & bit) ? (size_t)B : 1); };
  const double* d_P = (const double*)st.in(P0, cnt(CNGP_PERWIN_P, 225));
  const double* d_Q = (const double*)st.in(Q, cnt(CNGP_PERWIN_Q, 225));
  const double* d_F = (const double*)st.in(STM, cnt(CNGP_PERWIN_STM, 225));
  const double* d_H = (const double*)st.in(H, cnt(CNGP_PERWIN_H, 60));
  const double* d_R = (const double*)st.in(R, cnt(CNGP_PERWIN_POS, 16));     // the R bit re-uses the position slot
  double* d_out = (double*)st.out(P_out, sizeof(double) * 225 * (size_t)B);
  if (st.err) return fail(ctx, st.err, "ekf_covariance: staging failed");
  // the slip arrays are not used on this path (fixed R) and the observer cannot trigger: they get harmless storage
  double* d_ms = (double*)ctx->buf(18, sizeof(double) * (size_t)M);
  int* d_i4 = (int*)ctx->buf(19, sizeof(int) * 3 * (size_t)B);
  double* d_xy = (double*)ctx->buf(13, sizeof(double) * (size_t)B);
  double* d_pos = (double*)ctx->buf(14, sizeof(double) * 3);
  unsigned long long* d_counter = (unsigned long long*)ctx->buf(17, 64);
  if (!d_ms || !d_i4 || !d_xy || !d_pos || !d_counter) return fail(ctx, CNGP_ERR_NOMEM, "ekf_covariance: buffers");
  CU(ctx, cudaMemsetAsync(d_ms, 0, sizeof(double) * (size_t)M, ctx->stream));
  CU(ctx, cudaMemcpyAsync(d_pos, c.init_llh, sizeof(double) * 3, cudaMemcpyHostToDevice, ctx->stream));
  ctx->begin(CNGP_PROF_LOOKAHEAD);
  const int pw = per_window & (CNGP_PERWIN_P | CNGP_PERWIN_Q | CNGP_PERWIN_STM | CNGP_PERWIN_H);
  // mean / sigma: one zero row shared by every window (M < 0 = row stride 0)
  const int e = cngp_launch_lookahead(d_ms, d_ms, B, -M, d_P, d_Q, d_F, d_H, d_pos, pw, &c, d_i4, d_i4 + B, d_i4 + 2 * B,
                                      d_xy, d_counter, d_out, nullptr, nullptr, d_R, (per_window & CNGP_PERWIN_POS) ? 1 : 0,
                                      ctx->stream);
  ctx->end();
  if (e) return fail(ctx, CNGP_ERR_CUDA, "ekf_covariance launch: %s", cudaGetErrorString((cudaError_t)e));
  const int rc = st.finish();
  if (rc) return fail(ctx, rc, "ekf_covariance: copy-out failed: %s", cudaGetErrorString(cudaGetLastError()));
  return CNGP_OK;
}

extern "C" int cngp_llh_to_enu(cngp_ctx* ctx, const double* llh, int64_t n, const cngp_stop_config* cfg, double* enu,
                               int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!llh || !enu || n < 0) return fail(ctx, CNGP_ERR_INVALID, "llh_to_enu: bad argument");
  if (n == 0) return CNGP_OK;
  cngp_stop_config c;
  if (cfg) c = *cfg; else cngp_default_stop_config(&c);
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  Stage st{ctx, mem};
  const double* d_in = (const double*)st.in(llh, sizeof(double) * 3 * (size_t)n);
  double* d_out = (double*)st.out(enu, sizeof(double) * 3 * (size_t)n);
  if (st.err) return fail(ctx, st.err, "llh_to_enu: staging failed");
  ctx->begin(CNGP_PROF_MISC);
  const int e = cngp_launch_llh_to_enu(d_in, n, &c, d_out, ctx->stream);
  ctx->end();
  if (e) return fail(ctx, CNGP_ERR_CUDA, "llh_to_enu launch: %s", cudaGetErrorString((cudaError_t)e));
  const int rc = st.finish();
  if (rc) return fail(ctx, rc, "llh_to_enu: copy-out failed");
  return CNGP_OK;
}

// ------------------------------------------------------------------------------------------------------------
// slip extraction + window recorder (the producer of GP_Input)
// ------------------------------------------------------------------------------------------------------------
extern "C" void cngp_default_slip_config(cngp_slip_config* c) {
  c->wheel_radius = 0.11; c->cmd_min = 0.2; c->rear_min = 0.001; c->arm_delay = 10; c->window = 150; c->min_samples = 15;
  c->reserved = 0;
}

extern "C" int cngp_slip_record_batch(cngp_ctx* ctx, const double* joint, const double* att, const double* vel,
                                      const double* cmd, const double* stop_cmd, int64_t B, int32_t T,
                                      const cngp_slip_config* cfg, int32_t max_windows, int32_t cap, double* slip,
                                      double* time_array, double* slip_array, int32_t* n_samples, int32_t* published,
                                      int32_t* stop_update, int32_t* n_windows, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!joint || !att || !vel || !cmd || !time_array || !slip_array || !n_samples || !published || !stop_update ||
      !n_windows || B < 0 || T <= 0 || max_windows <= 0 || cap <= 0)
    return fail(ctx, CNGP_ERR_INVALID, "slip_record: bad argument");
  if (B == 0) return CNGP_OK;
  cngp_slip_config c;
  if (cfg) c = *cfg; else cngp_default_slip_config(&c);
  if (c.window <= 0 || c.arm_delay < 0) return fail(ctx, CNGP_ERR_INVALID, "slip_record: bad recorder configuration");
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  Stage st{ctx, mem};
  const size_t bt = (size_t)B * T, bw = (size_t)B * max_windows;
  const double* d_joint = (const double*)st.in(joint, sizeof(double) * bt * 4);
  const double* d_att = (const double*)st.in(att, sizeof(double) * bt * 3);
  const double* d_vel = (const double*)st.in(vel, sizeof(double) * bt * 3);
  const double* d_cmd = (const double*)st.in(cmd, sizeof(double) * bt);
  const double* d_scmd = (const double*)st.in(stop_cmd, sizeof(double) * bt);
  double* d_slip = (double*)st.out(slip, sizeof(double) * bt);
  double* d_ta = (double*)st.out(time_array, sizeof(double) * bw * cap);
  double* d_sa = (double*)st.out(slip_array, sizeof(double) * bw * cap);
  int* d_ns = (int*)st.out(n_samples, sizeof(int) * bw);
  int* d_pu = (int*)st.out(published, sizeof(int) * bw);
  int* d_su = (int*)st.out(stop_update, sizeof(int) * bw);
  int* d_nw = (int*)st.out(n_windows, sizeof(int) * (size_t)B);
  if (st.err) return fail(ctx, st.err, "slip_record: staging failed");
  // windows that never close and samples never recorded read as zero
  CU(ctx, cudaMemsetAsync(d_ta, 0, sizeof(double) * bw * cap, ctx->stream));
  CU(ctx, cudaMemsetAsync(d_sa, 0, sizeof(double) * bw * cap, ctx->stream));
  CU(ctx, cudaMemsetAsync(d_ns, 0, sizeof(int) * bw, ctx->stream));
  CU(ctx, cudaMemsetAsync(d_pu, 0, sizeof(int) * bw, ctx->stream));
  CU(ctx, cudaMemsetAsync(d_su, 0xff, sizeof(int) * bw, ctx->stream));
  ctx->begin(CNGP_PROF_MISC);
  const int e = cngp_launch_slip_record(d_joint, d_att, d_vel, d_cmd, d_scmd, B, T, &c, max_windows, cap, d_slip, d_ta,
                                        d_sa, d_ns, d_pu, d_su, d_nw, ctx->stream);
  ctx->end();
  if (e) return fail(ctx, CNGP_ERR_CUDA, "slip_record launch: %s", cudaGetErrorString((cudaError_t)e));
  const int rc = st.finish();
  if (rc) return fail(ctx, rc, "slip_record: copy-out failed");
  return CNGP_OK;
}

// ------------------------------------------------------------------------------------------------------------
// EKF context generation (STM, Q, H of the SetStopping service)
// ------------------------------------------------------------------------------------------------------------
extern "C" int cngp_ekf_context_batch(cngp_ctx* ctx, const double* llh, const double* vel, const double* att,
                                      const double* f_ib_b, int64_t B, double dt, double dt_odo, double* STM, double* Q,
                                      double* Hvec, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!llh || !vel || !att || !f_ib_b || !STM || !Q || B < 0 || !(dt > 0.0) || !(dt_odo > 0.0))
    return fail(ctx, CNGP_ERR_INVALID, "ekf_context: bad argument");
  if (B == 0) return CNGP_OK;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  Stage st{ctx, mem};
  const size_t b3 = sizeof(double) * 3 * (size_t)B;
  const double* d_llh = (const double*)st.in(llh, b3);
  const double* d_vel = (const double*)st.in(vel, b3);
  const double* d_att = (const double*)st.in(att, b3);
  const double* d_fib = (const double*)st.in(f_ib_b, b3);
  double* d_S = (double*)st.out(STM, sizeof(double) * 225 * (size_t)B);
  double* d_Q = (double*)st.out(Q, sizeof(double) * 225 * (size_t)B);
  double* d_H = (double*)st.out(Hvec, sizeof(double) * 60 * (size_t)B);
  if (st.err) return fail(ctx, st.err, "ekf_context: staging failed");
  ctx->begin(CNGP_PROF_MISC);
  const int e = cngp_launch_ekf_context(d_llh, d_vel, d_att, d_fib, B, dt, dt_odo, d_S, d_Q, d_H, ctx->stream);
  ctx->end();
  if (e) return fail(ctx, CNGP_ERR_CUDA, "ekf_context launch: %s", cudaGetErrorString((cudaError_t)e));
  const int rc = st.finish();
  if (rc) return fail(ctx, rc, "ekf_context: copy-out failed");
  return CNGP_OK;
}
