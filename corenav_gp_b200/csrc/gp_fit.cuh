// Phase A of the batched exact GP: assemble Ky = K(X,X) + (noise + 1e-8) I, factor it, solve z = L^-1 y, LML.
//
// Replaces GPy ExactGaussianInference.inference as reached from GPRegression(...) at
// core_navigation/script/gp_slip_node.py:35 (row a3): kern.K, pdinv -> jitchol -> dpotrf, dpotrs, logdet.
//
// One CTA per (candidate, window) problem: NW worker warps + one DIAGONAL warp.  Left-looking tile Cholesky over
// 8-wide tile columns with a one-column look-ahead, so that the only serial chain of the algorithm - the in-warp
// factorisation + inversion of the 8x8 diagonal tile (chol8_inv8, ~1.3k cycles of dependent shuffles / rsqrt / fma
// per column) - runs on the diagonal warp WHILE the workers accumulate the bulk of the next column.
//
// Row tiles are OWNED: row i belongs to worker i % NW for the whole factorisation (slot t = i / NW of that warp), so a
// worker's tiles of the current column, of the next column and the factor tiles it has just produced all stay in
// registers under compile-time indices, and the k = j term of the look-ahead needs one operand from shared memory only.
// (Measured alternatives, tools/fit_bench.cu: dedicated evaluator warps staging Ky ahead of the factorisation lose -
// their scalar FP64 work crawls behind the workers' DMMA on the shared FP64 pipe - and so does moving the diagonal warp
// to a sub-partition of its own; evaluating in a phase of its own, all workers at once, is what the pipe likes.)
//
//   workers, step j:  (b) S(i, j+1) = sum_{k<j} L(i,k) L(j+1,k)^T for their rows i >= j+1 (one pass over the tile pool:
//                         1 + A 16-byte loads and 2A DMMA per k for A live rows), evaluate Ky(i, j+1) (the kernel
//                         matrix is never materialised); the owner of row j+1 parks the diagonal tile's partial sum and
//                         carries the forward solve for z along as two scalar FMA per k on the tiles it loads anyway
//                     --- barrier 1: inv(L_jj) published by the diagonal warp ---
//                     (d) L(i,j) = C(i,j) inv(L_jj)^T -> registers, tile pool, global (for phase B); z_j
//                     --- barrier 2 ---
//                     (a) C(i, j+1) = Ky(i, j+1) - S(i, j+1) - L(i,j) L(j+1,j)^T
//   diagonal warp:    chol8_inv8(C(j,j)) -> inv(L_jj); arrive on barrier 1; wait on barrier 2;
//                     C(j+1,j+1) = parked partial - L(j+1,j) L(j+1,j)^T.
//
// Every update and the triangular solve below the diagonal (through the explicitly inverted 8x8 diagonal tile) are
// tile_mma = FP64 DMMA.
// Output factor layout (consumed by gp_var.cuh / gp_grad.cuh): column-block-major tiles, tile (j,j) holds
// inv(L_jj) (lower triangular), tiles (i>j, j) hold L_ij.
#pragma once
#include "kernel_eval.cuh"

namespace cngp {

constexpr int NPAD = CNGP_MAX_N + 8;
constexpr int FIT_NW_FULL = 11, FIT_T_FULL = 3;   // workers x row-tile slots for nt > 16 (CNGP_MAX_N = 256: nt <= 32)
// Shared-memory tile pool.  With h = ceil(nt/2): columns k < h are packed one after the other, column k holding its
// rows k..nt-1 (tile (i,k) at cb(k) + i - k, cb(k) = k nt - k(k-1)/2).  Rows < h are dead once column h starts, so
// column k = h + m re-uses the dead head of column m (h - m >= nt - k tiles): tile (i,k) at cb(m) + i - k.  Walking k
// for a fixed row therefore advances by nt-1, nt-2, ... tiles in BOTH ranges, with one pointer for all rows of a
// column.  392 tiles (196 KB) at nt = 32 instead of 528.
__host__ __device__ __forceinline__ int fit_pool_tiles(int nt) {
  const int h = (nt + 1) / 2;
  return h * nt - h * (h - 1) / 2;
}
// + slack: rows beyond nt-1 of a partially filled last slot are read (never used) by the unpredicated pool loop
constexpr size_t fit_smem_bytes(int nt, int slots_total) {
  return (size_t)(((nt + 1) / 2) * nt - ((nt + 1) / 2) * (((nt + 1) / 2) - 1) / 2 + (slots_total > nt ? slots_total - nt : 0)) * 512;
}

struct FitArgs {
  KProg kp;
  const double* theta;   // hyper-parameters, noise last
  long long theta_stride;
  int theta_mode;        // 0 shared, 1 per window (problem % n_windows), 2 per candidate (problem / n_windows),
                         // 3 per problem (theta row = problem; the window comes from win_map)
  const int* win_map;    // [n_problems] window of each problem (theta_mode 3), or null
  const double* x;       // [n_windows][N]
  const double* y;       // [n_windows][N]
  int N, nt;             // nt = ceil(N / 8)
  int n_windows;
  long long problem0;    // first problem of this launch (chunking)
  double* L;             // [chunk][tiles_in_lower(nt)][64]
  double* z;             // [chunk][nt*8]   z = L^-1 y
  double* feat;          // [chunk][4][nt*8] per-point features (x, x^2, cos, sin) for phase B, or null
  double* lml;           // [n_problems] or null
  double* logdet;        // [n_problems] or null
  double* quad;          // [n_problems] or null   y' Ky^-1 y
  int* status;           // [n_problems] or null
  int jitter_retry;
  // lag tables (see above).  lag_ok: the expression is stationary (host check); the rest may be null (fit-only callers)
  int lag_ok;
  const double* xstar;   // [n_windows][M] or [M]: test stamps, so that the table covers the cross-covariance lags
  long long xstar_stride;
  int M;
  double* ktab;          // [chunk][VAR_TAB_MAX]
  double* kmeta;         // [chunk][VAR_META]
  int* kxi;              // [chunk][nt*8]  training stamps as integer offsets from the base stamp
  const int* skip;       // [n_problems] or null: problems with skip[p] != 0 are left untouched (finished optimiser windows)
  int f32_factor;        // FP32 mode: write the factor tiles split hi/lo TF32 (tile_store_split) for gp_var32_kernel
  int* n_lazy;           // += 1 for every window of the launch whose table is NOT valid (gp_var_kernel picks its path on it)
  // KID_TILES only (large-N blocked Cholesky, chol_large.cu): the SPD block is read from tile storage instead of being
  // evaluated - tile (i, j) of the block at Asrc + j * a_col_stride + i * 64 (lower tiles only are read).
  const double* Asrc;
  long long a_col_stride;
  // ragged batches: valid training points of each window (n_win[window] <= N, ceil(n_win / 8) == nt); N is then the row
  // stride of x / y only, and the window is identity-padded beyond its own count.  null: every window has N points.
  const int* n_win;
  int* done;             // [n_problems] gp_fit_toeplitz_kernel only: 1 for the problems it factored (or skipped), else 0
  double* ldiag;         // gp_fit_toeplitz_kernel only, or null: [nt][64] the diagonal tiles L_jj themselves (row-major) of
                         // problem 0 of the launch - the one-window fit of a shared covariance (gp_toep_group.cuh)
#ifdef CNGP_FIT_TIMING
  long long* dbg;        // tools/fit_bench.cu: per-warp phase cycle counters of block 0, [warp][8]
#endif
};

// Which lag tables a window gets (both false: the lazy evaluators).
struct LagTab {
  bool fit_tab;          // K(X,X) by integer lag: every stamp an integer, the span of the training stamps < FIT_TAB_MAX
  bool var_tab;          // the whole table (training and test lags) for gp_var_kernel
};

// Stamp extent of one window, the part of the lag-table decision that writes nothing: every training stamp and every
// one of the M test stamps an integer with |x| < 2^26 (x^2 and x x' stay exact integers, r^2 of the expanded form is
// exact), the base stamp, the span of the training stamps and the largest lag of K(X,X) and K(X,X*).  fit_lag_tables
// and the shared-covariance qualification (gp_toep_group.cuh) both decide from it.
struct LagExtent {
  bool ok;
  double base, span, dmax;
  __device__ __forceinline__ bool fit_tab() const { return ok && span < (double)FIT_TAB_MAX; }
  __device__ __forceinline__ bool var_tab() const { return ok && dmax < (double)VAR_TAB_MAX; }
};
template <int NTH>
__device__ __forceinline__ LagExtent lag_extent(const FitArgs& a, int win, int N, int tid, const double* fx, double* s_mm,
                                                int* s_okv) {
  constexpr int NWARPS = NTH / 32;
  const int lane = tid & 31, w = tid >> 5;
  const double big = 67108864.0;   // 2^26
  double xlo = 1e300, xhi = -1e300, slo = 1e300, shi = -1e300;
  int ok = 1;
  for (int i = tid; i < N; i += NTH) {
    const double v = fx[i];
    ok &= (v == rint(v)) && (fabs(v) < big);
    xlo = fmin(xlo, v); xhi = fmax(xhi, v);
  }
  if (a.xstar) {
    const double* xs = a.xstar + (a.xstar_stride ? (long long)win * a.xstar_stride : 0);
    for (int i = tid; i < a.M; i += NTH) {
      const double v = xs[i];
      ok &= (v == rint(v)) && (fabs(v) < big);
      slo = fmin(slo, v); shi = fmax(shi, v);
    }
  }
  for (int o = 16; o; o >>= 1) {
    xlo = fmin(xlo, __shfl_xor_sync(0xffffffffu, xlo, o)); xhi = fmax(xhi, __shfl_xor_sync(0xffffffffu, xhi, o));
    slo = fmin(slo, __shfl_xor_sync(0xffffffffu, slo, o)); shi = fmax(shi, __shfl_xor_sync(0xffffffffu, shi, o));
    ok &= __shfl_xor_sync(0xffffffffu, ok, o);
  }
  if (NWARPS > 1) {
    if (lane == 0) { s_mm[w] = xlo; s_mm[NWARPS + w] = xhi; s_mm[2 * NWARPS + w] = slo; s_mm[3 * NWARPS + w] = shi; s_okv[w] = ok; }
    __syncthreads();
    for (int i = 0; i < NWARPS; ++i) {
      xlo = fmin(xlo, s_mm[i]); xhi = fmax(xhi, s_mm[NWARPS + i]); slo = fmin(slo, s_mm[2 * NWARPS + i]); shi = fmax(shi, s_mm[3 * NWARPS + i]);
      ok &= s_okv[i];
    }
  }
  const double base = fmin(xlo, slo);
  return LagExtent{ok != 0, base, xhi - xlo, fmax(xhi, shi) - base};   // span: largest lag inside K(X,X)
}

// Lag-table prologue of one window, shared by gp_fit_kernel (NTH = the whole CTA) and gp_fit_toeplitz_kernel (NTH = one
// warp), so that both write the same table bits and take the same table / lazy decision.  fx: the window's stamps.
// s_tab: k by lag for the caller's own assembly, or null.  s_xi: training stamps minus the base stamp.  tid 0 writes
// *s_kdiag (K(x,x), White included) and the window's meta row; the caller syncs before reading them.  For NTH > 32,
// s_mm [4][NTH / 32] and s_okv [NTH / 32] carry the cross-warp reduction.  The caller counts the window in n_lazy.
template <int NTH>
__device__ __forceinline__ LagTab fit_lag_tables(const FitArgs& a, long long lp, int win, int N, int nt, int tid,
                                                 const double* fx, const KProg* kps, const LeafConst* hc, double noise,
                                                 double* s_tab, int* s_xi, double* s_kdiag, double* s_mm, int* s_okv) {
  const LagExtent ex = lag_extent<NTH>(a, win, N, tid, fx, s_mm, s_okv);
  const double base = ex.base, span = ex.span, dmax = ex.dmax;
  const bool fit_tab = ex.fit_tab();
  const bool var_tab = a.ktab && ex.var_tab();
  if (fit_tab || var_tab) {
    const int nl = (int)(var_tab ? dmax : span) + 1;
    double* gt = var_tab ? a.ktab + lp * (long long)VAR_TAB_MAX : nullptr;
    for (int d = tid; d < nl; d += NTH) {
      const double v = keval_generic_cross(kps, hc, (double)d, 0.0);
      if (s_tab && fit_tab && d < FIT_TAB_MAX && (double)d <= span) s_tab[d] = v;
      if (gt) gt[d] = v;
    }
    for (int i = tid; i < nt * 8; i += NTH) {
      const int xi = i < N ? (int)(fx[i] - base) : 0;
      s_xi[i] = xi;
      if (var_tab) a.kxi[lp * (long long)(nt * 8) + i] = xi;
    }
    if (tid == 0) *s_kdiag = keval_generic_sym(kps, hc, 0.0, 0.0, true);
  }
  if (tid == 0 && a.kmeta) {
    double* km = a.kmeta + lp * (long long)VAR_META;
    km[0] = kdiag_eval(*kps, hc, 0.0);
    km[1] = base;
    km[2] = noise;
    km[3] = var_tab ? 1.0 : 0.0;
  }
  return LagTab{fit_tab, var_tab};
}

#ifdef CNGP_FIT_TIMING
#define FIT_STAMP(ph) do { const long long now_ = clock64(); t_acc[ph] += now_ - t_last; t_last = now_; } while (0)
#else
#define FIT_STAMP(ph) do { } while (0)
#endif

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// In-warp Cholesky of an 8x8 SPD tile held in the lane layout, fused with the inverse of the factor.  This is the
// critical path of every tile column, so it is built for latency: the tile stays in registers, column k is exchanged
// with independent shuffles, the pivot uses rsqrt (sqrt + div cost 165 dependent cycles, rsqrt 80), and the inverse
// rides along for free: the row operations of the elimination are applied to an identity tile in the same step
// (forward substitution L X = I by columns: X[k] = x[k] / L[k][k], x[r] -= L[r][k] X[k]), so there is no second pass.
// The logarithms of the pivots are NOT taken here - the pivots are parked in dpiv and logged in parallel at the end.
// On return linv holds inv(L) row-major (zeros above the diagonal) and dpiv[0..7] the diagonal of L.
// Returns the failing pivot (1-based) or 0.
__device__ __forceinline__ int chol8_inv8(tile2 c, int lane, double* linv, double* dpiv) {
  const int r = lane >> 2, q = lane & 3;
  int fail = 0;
  tile2 x{r == 2 * q ? 1.0 : 0.0, r == 2 * q + 1 ? 1.0 : 0.0};
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const double v = (k & 1) ? c.b : c.a;                              // my entry of column pair k>>1
    const double pk = __shfl_sync(0xffffffffu, v, 4 * k + (k >> 1));     // T[k][k]
    const double trk = __shfl_sync(0xffffffffu, v, 4 * r + (k >> 1));    // T[r][k]
    const double tc0 = __shfl_sync(0xffffffffu, v, 8 * q + (k >> 1));    // T[2q][k]
    const double tc1 = __shfl_sync(0xffffffffu, v, 8 * q + 4 + (k >> 1));// T[2q+1][k]
    const double xka = __shfl_sync(0xffffffffu, x.a, 4 * k + q);         // x[k][2q]
    const double xkb = __shfl_sync(0xffffffffu, x.b, 4 * k + q);         // x[k][2q+1]
    if (!(pk > 0.0) && fail == 0) fail = k + 1;
    const double rs = rsqrt(pk);
    const double lrk = trk * rs;
    if (2 * q > k && r >= 2 * q) c.a = fma(-lrk, tc0 * rs, c.a);
    if (2 * q + 1 > k && r >= 2 * q + 1) c.b = fma(-lrk, tc1 * rs, c.b);
    const double xsa = xka * rs, xsb = xkb * rs;
    if (r == k) { x.a = xsa; x.b = xsb; }
    if (r > k) { x.a = fma(-lrk, xsa, x.a); x.b = fma(-lrk, xsb, x.b); }
    if (lane == 0) dpiv[k] = pk * rs;
  }
  tile_store(linv, lane, x);
  __syncwarp();
  return fail;
}


template <int N> struct FitIC { static constexpr int value = N; };

// Row residue of worker warp w (its rows are residue + NW t).  Identity.  Rows with a higher index live longer, so
// residue r carries pass work ~ sum_t (r + NW t)^2 and the sub-partitions (warp id % 4) are unevenly loaded; dealing the
// residues so that the four sub-partitions carry equal work was measured (tools/fit_bench.cu, round 2): {8,4,0} {7,5,1}
// {6,3,2} {9,10}+diag 2.23 ms, {9,0,10} {8,1,2} {7,3,4} {5,6}+diag 2.29 ms, identity 2.19 ms - the per-column critical
// path is the diagonal warp's chol8 + the panel phase, not the heaviest worker, so balancing the passes buys nothing.
template <int NW>
__device__ __forceinline__ int fit_residue(int w) {
  return w;
}

// NW workers, T row-tile slots per worker: nt <= NW * T.
template <int KID, int NW, int T>
__global__ void __launch_bounds__((NW + 1) * 32, NW * T > 18 ? 1 : 2) gp_fit_kernel(const FitArgs a) {
  constexpr int FIT_THREADS = (NW + 1) * 32;
  extern __shared__ __align__(128) double pool[];               // tile pool, see fit_pool_tiles
  __shared__ __align__(16) double fx[NPAD], fxx[NPAD], fc[NPAD], fs[NPAD];   // per-point features
  __shared__ double ys[NPAD];
  __shared__ __align__(16) double zs[NPAD];
  __shared__ LeafConst hc[CNGP_MAX_LEAVES];
  __shared__ KProg kps;
  __shared__ __align__(16) double linv[64];      // inv(L_jj) of the current column (diagonal warp -> workers)
  __shared__ __align__(16) double dpart[2][64];  // Ky(c,c) - sum_{k<c-1} ... of column c, buffer c & 1 (owner -> diagonal warp)
  __shared__ __align__(16) double etab[128];     // exp_tab tables scaled by the leaf variances
  __shared__ double dpiv[NPAD];          // diagonal of L (pivots), logged in parallel at the end
  __shared__ double s_red[NW + 1], s_red2[NW + 1];
  __shared__ int s_fail;
  __shared__ double s_tab[KID == KID_TILES ? 1 : FIT_TAB_MAX];   // k by integer lag, lags 0 .. span
  __shared__ int s_xi[KID == KID_TILES ? 2 : NPAD];              // training stamps minus the base stamp
  __shared__ double s_mm[4 * (NW + 1)];
  __shared__ int s_okv[NW + 1];
  __shared__ double s_kdiag;

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int wr = fit_residue<NW>(w);               // row residue of a worker warp
  const int r = lane >> 2, q = lane & 3;
  const long long lp = blockIdx.x;                 // problem within this launch
  const long long p = a.problem0 + lp;             // global problem
  if (a.skip && a.skip[p]) return;
  const int win = a.win_map ? a.win_map[p] : (int)(p % a.n_windows);
  const long long ti = a.theta_mode == 0 ? 0 : (a.theta_mode == 1 ? (long long)win : (a.theta_mode == 3 ? p : p / a.n_windows));
  const double* th = a.theta + ti * a.theta_stride;
  const int ld = a.N, N = a.n_win ? a.n_win[win] : a.N, nt = a.nt;
  const int h = (nt + 1) / 2;                       // columns >= h re-use the dead heads of columns < h
  const double noise = (KID == KID_TILES) ? 0.0 : th[a.kp.n_params];
  FastK<KID> fk;
  if (KID != KID_GENERIC && KID != KID_TILES) {
    fk.init(th);
    fk.base = a.x[(long long)win * ld];        // phase origin: the window's first stamp (gp_var_kernel uses the same)
    if (tid < 64) {
      const double t = EXP2_TAB64[tid];
      etab[tid] = fk.scale1() * t;
      etab[64 + tid] = fk.scale2() * t;
    }
  }

  for (int i = tid; i < nt * 8; i += FIT_THREADS) {
    const double xv = (KID != KID_TILES && i < N) ? a.x[(long long)win * ld + i] : 0.0;
    ys[i] = (KID != KID_TILES && i < N) ? a.y[(long long)win * ld + i] : 0.0;
    PointFeat f{xv, __dmul_rn(xv, xv), 0.0, 0.0};
    if (KID != KID_GENERIC && KID != KID_TILES) f = fk.point(xv);
    fx[i] = f.x; fxx[i] = f.xx; fc[i] = f.c; fs[i] = f.s;
    if (a.feat) {
      double* fp = a.feat + lp * (long long)(4 * nt * 8);
      fp[i] = f.x; fp[nt * 8 + i] = f.xx; fp[2 * nt * 8 + i] = f.c; fp[3 * nt * 8 + i] = f.s;
    }
  }
  if (KID == KID_GENERIC || (KID != KID_TILES && a.lag_ok)) {
    if (tid < a.kp.n_leaves) hc[tid] = leaf_prepare(a.kp.leaf_type[tid], th + a.kp.leaf_param[tid]);
    if (tid == 0) kps = a.kp;
  }
  __syncthreads();

  // ---- lag table (stationary expression, integer stamps) ----
  bool tabmode = false;
  if (KID != KID_TILES && a.lag_ok) {
    const LagTab lt = fit_lag_tables<FIT_THREADS>(a, lp, win, N, nt, tid, fx, &kps, hc, noise, s_tab, s_xi, &s_kdiag,
                                                  s_mm, s_okv);
    tabmode = lt.fit_tab;
    if (tid == 0 && a.kmeta && !lt.var_tab && a.n_lazy) atomicAdd(a.n_lazy, 1);
    __syncthreads();
  } else if (KID != KID_TILES && tid == 0 && a.n_lazy) {
    atomicAdd(a.n_lazy, 1);
  }

  const bool full_window = N == 8 * nt;
  auto feat_at = [&](int i) -> PointFeat {
    if (KID == KID_GENERIC) return PointFeat{fx[i], 0.0, 0.0, 0.0};
    if (KID == KID_RBF_PER) return PointFeat{fx[i], fxx[i], fc[i], fs[i]};
    return PointFeat{fx[i], fxx[i], 0.0, 0.0};
  };
  // Ky(row, col) without the diagonal term; identity padding beyond N
  auto ky_entry = [&](int row, int col, const PointFeat& fa, const PointFeat& fb) -> double {
    if (KID == KID_TILES) return 0.0;   // never used: the tiles are loaded
    if (row < N && col < N) {
      if (KID == KID_GENERIC) return keval_generic_sym(&kps, hc, fa.x, fb.x, row == col);
      return fk.eval_tab(fa, fb, row == col, etab);
    }
    return (row == col) ? 1.0 : 0.0;
  };
  // lag-table form of a Ky tile: xr = integer stamp of my row, xc = stamps of my two columns
  auto ky_tab = [&](int xr, int2 xc, int i, int c, double dadd) -> tile2 {
    const int c0 = 8 * c + 2 * q, c1 = c0 + 1, row = 8 * i + r;
    double v0 = s_tab[abs(xr - xc.x)], v1 = s_tab[abs(xr - xc.y)];     // two shared-memory lookups by integer lag
    if (i == c) {    // true diagonal entries: K(x,x) of the expression (White included) + noise + jitter
      if (row == c0) v0 = s_kdiag + dadd;
      if (row == c1) v1 = s_kdiag + dadd;
    }
    if (!full_window) {   // identity padding beyond N
      if (row >= N || c0 >= N) v0 = (row == c0) ? 1.0 : 0.0;
      if (row >= N || c1 >= N) v1 = (row == c1) ? 1.0 : 0.0;
    }
    return tile2{v0, v1};
  };
  // tile (i, c) of Ky in the lane layout (dadd on the diagonal entries), evaluated or - KID_TILES - loaded
  auto ky_tile = [&](int i, int c, double dadd) -> tile2 {
    if (KID == KID_TILES) {
      const double2 av = *reinterpret_cast<const double2*>(a.Asrc + c * a.a_col_stride + (long long)i * 64 + 2 * lane);
      return tile2{av.x, av.y};
    }
    const int c0 = 8 * c + 2 * q, c1 = c0 + 1, row = 8 * i + r;
    if (tabmode) return ky_tab(s_xi[row], *reinterpret_cast<const int2*>(s_xi + c0), i, c, dadd);
    if (KID != KID_GENERIC && full_window && i != c) {   // interior tile of an unpadded window: no diagonal, no padding
      const PointFeat fr = feat_at(row);
      const double2 x2 = *reinterpret_cast<const double2*>(fx + c0), xx2 = *reinterpret_cast<const double2*>(fxx + c0);
      double2 c2 = make_double2(0.0, 0.0), s2 = make_double2(0.0, 0.0);
      if (KID == KID_RBF_PER) { c2 = *reinterpret_cast<const double2*>(fc + c0); s2 = *reinterpret_cast<const double2*>(fs + c0); }
      return tile2{fk.eval_tab(fr, PointFeat{x2.x, xx2.x, c2.x, s2.x}, false, etab),
                   fk.eval_tab(fr, PointFeat{x2.y, xx2.y, c2.y, s2.y}, false, etab)};
    }
    const PointFeat fr = feat_at(row), f0 = feat_at(c0), f1 = feat_at(c1);
    double v0 = ky_entry(row, c0, fr, f0), v1 = ky_entry(row, c1, fr, f1);
    if (row == c0 && row < N) v0 += dadd;
    if (row == c1 && row < N) v1 += dadd;
    return tile2{v0, v1};
  };
  // pool slot of factor tile (i, k)
  auto pool_idx = [&](int i, int k) -> int {
    const int m = k < h ? k : k - h;
    return m * nt - m * (m - 1) / 2 + i - k;
  };

  double* Lp = a.L + lp * (long long)tiles_in_lower(nt) * 64;
  double* poolL = pool + 2 * lane;                       // lane-offset view of the pool
  const int max_attempts = (a.jitter_retry && KID != KID_TILES) ? 6 : 1;
  double extra = 0.0;
  int fail_pivot = 0, attempts_used = 0;

  for (int attempt = 0; attempt < max_attempts; ++attempt) {
    if (attempt == 1) {
      // GPy jitchol: jitter = mean(diag(Ky)) * 1e-6, then x10 per retry
      double s = 0.0;
      for (int i = tid; i < N; i += FIT_THREADS) {
        const PointFeat f = feat_at(i);
        s += (tabmode ? s_kdiag : ky_entry(i, i, f, f)) + noise + CNGP_JITTER;
      }
      for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) s_red[w] = s;
      __syncthreads();
      s = 0.0;
      for (int i = 0; i <= NW; ++i) s += s_red[i];
      extra = s / N * 1e-6;
    } else if (attempt > 1) {
      extra *= 10.0;
    }
    if (tid == 0) s_fail = 0;
    __syncthreads();
    const double dadd = noise + CNGP_JITTER + extra;
#ifdef CNGP_FIT_TIMING
    long long t_acc[6] = {0, 0, 0, 0, 0, 0};
    long long t_last = clock64();
#endif

    if (w == NW) {
      // ================= diagonal warp =================
      tile2 Cd = ky_tile(0, 0, dadd);
      for (int j = 0; j < nt; ++j) {
        const int f = chol8_inv8(Cd, lane, linv, dpiv + 8 * j);
        if (lane == 0 && f && s_fail == 0) s_fail = 8 * j + f;
        FIT_STAMP(0);
        named_bar_arrive(1, FIT_THREADS);                           // inv(L_jj) is in linv
        if (a.f32_factor) tile_store_split(Lp + (long long)tile_index(j, j, nt) * 64, lane, tile_load(linv, lane));
        else tile_store(Lp + (long long)tile_index(j, j, nt) * 64, lane, tile_load(linv, lane));
        named_bar_sync(2, FIT_THREADS);                             // column j stored, dpart of column j+1 parked
        FIT_STAMP(1);
        if (j + 1 < nt) {
          const tile2 Y = tile_load(pool + pool_idx(j + 1, j) * 64, lane);
          tile2 S = tile_load(dpart[(j + 1) & 1], lane);
          tile_mma(S, tile2{-Y.a, -Y.b}, Y);
          Cd = S;
        }
        FIT_STAMP(2);
      }
    } else {
      // ================= worker warps =================
      // slot t of this warp is row tile i = wr + NW t, for every column (wr: the warp's row residue, see fit_residue)
      tile2 Ccur[T], Lt[T];
      int xrow[T];                  // lag-table mode: integer stamp of my row in slot t
#pragma unroll
      for (int t = 0; t < T; ++t) xrow[t] = (tabmode && wr + NW * t < nt) ? s_xi[8 * (wr + NW * t) + r] : 0;
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int i = wr + NW * t;
        Ccur[t] = (i >= 1 && i < nt) ? ky_tile(i, 0, dadd) : tile2{0.0, 0.0};   // (0,0) is the diagonal warp's
        Lt[t] = tile2{0.0, 0.0};
      }
      double za = 0.0, zb = 0.0;    // sum_k L(c,k) z_k in the lane layout, for the next diagonal row c this warp owns

      for (int j = 0; j < nt; ++j) {
        const int c = j + 1;
        // ---- (b) look-ahead: partial sums of column c over k < j, Ky tiles of column c ----
        const int t0 = c > wr ? (c - wr + NW - 1) / NW : 0;     // first slot with a row >= c
        const bool own_diag = t0 < T && wr + NW * t0 == c && c < nt;
        tile2 S0[T], S1[T], Kn[T];
#pragma unroll
        for (int t = 0; t < T; ++t) {
          S0[t] = tile2{0.0, 0.0};
          S1[t] = tile2{0.0, 0.0};
          Kn[t] = tile2{0.0, 0.0};
        }
        if (c < nt && wr + NW * t0 < nt && t0 < T) {
          // pool pass over slots T0..T-1 (compile-time T0): Y = (c,k) and X_t = (i_t,k) sit in the same pool column.
          // Slots whose row is beyond nt-1 read (and never use) whatever follows the column - see fit_smem_bytes.
          auto pass = [&](auto t0c, int k0, int k1, const double* pY) {
            constexpr int T0 = decltype(t0c)::value;
            if (k0 >= k1) return;
            const double* pX = pY + (wr - c) * 64;
            int pitch = (nt - 1) * 64;
            const double* zp = zs + 8 * k0 + 2 * q;
            tile2 Y = tile_load(pY, 0), X[T], Yn{0.0, 0.0}, Xn[T];
#pragma unroll
            for (int t = T0; t < T; ++t) X[t] = tile_load(pX + t * NW * 64, 0);
            for (int k = k0; k < k1; k += 2) {
              pY += pitch; pX += pitch; pitch -= 64;
              if (k + 1 < k1) {
                Yn = tile_load(pY, 0);
#pragma unroll
                for (int t = T0; t < T; ++t) Xn[t] = tile_load(pX + t * NW * 64, 0);
              }
#pragma unroll
              for (int t = T0; t < T; ++t) dmma884(S0[t].a, S0[t].b, X[t].a, Y.a);
#pragma unroll
              for (int t = T0; t < T; ++t) dmma884(S0[t].a, S0[t].b, X[t].b, Y.b);
              if (own_diag) {
                const double2 zk = *reinterpret_cast<const double2*>(zp);
                za = fma(Y.a, zk.x, za); zb = fma(Y.b, zk.y, zb);
              }
              if (k + 1 >= k1) break;
              pY += pitch; pX += pitch; pitch -= 64;
              if (k + 2 < k1) {
                Y = tile_load(pY, 0);
#pragma unroll
                for (int t = T0; t < T; ++t) X[t] = tile_load(pX + t * NW * 64, 0);
              }
#pragma unroll
              for (int t = T0; t < T; ++t) dmma884(S1[t].a, S1[t].b, Xn[t].a, Yn.a);
#pragma unroll
              for (int t = T0; t < T; ++t) dmma884(S1[t].a, S1[t].b, Xn[t].b, Yn.b);
              if (own_diag) {
                const double2 zk = *reinterpret_cast<const double2*>(zp + 8);
                za = fma(Yn.a, zk.x, za); zb = fma(Yn.b, zk.y, zb);
              }
              zp += 16;
            }
          };
          auto both = [&](auto t0c) {
            pass(t0c, 0, j < h ? j : h, poolL + c * 64);          // columns k < min(j, h)
            if (j > h) pass(t0c, h, j, poolL + (c - h) * 64);     // columns h <= k < j
          };
          if (T == 1 || t0 == 0) both(FitIC<0>{});
          else if (T == 2 || t0 == 1) both(FitIC<(T > 1 ? 1 : 0)>{});
          else if (T == 3 || t0 == 2) both(FitIC<(T > 2 ? 2 : 0)>{});
          else both(FitIC<(T > 3 ? 3 : 0)>{});
          FIT_STAMP(0);
          // Ky tiles of column c (never stored); the diagonal row's partial result goes to the diagonal warp
          int2 xc2 = make_int2(0, 0);
          if (tabmode) xc2 = *reinterpret_cast<const int2*>(s_xi + 8 * c + 2 * q);
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int i = wr + NW * t;
            if (t >= t0 && i < nt) {
              S0[t].a += S1[t].a; S0[t].b += S1[t].b;
              Kn[t] = tabmode ? ky_tab(xrow[t], xc2, i, c, dadd) : ky_tile(i, c, dadd);
              if (i == c) tile_store(dpart[c & 1], lane, tile2{Kn[t].a - S0[t].a, Kn[t].b - S0[t].b});
            }
          }
        }
        FIT_STAMP(1);
        named_bar_sync(1, FIT_THREADS);                             // inv(L_jj) published
        FIT_STAMP(2);
        // ---- (d) rows below the diagonal: L(i,j) = C(i,j) inv(L_jj)^T -> registers, pool, global; z_j ----
        {
          const tile2 Yinv = tile_load(linv, lane);
          double* colj = Lp + (long long)tile_index(j, j, nt) * 64;
          double* pcol = pool + pool_idx(j, j) * 64;
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int i = wr + NW * t;
            if (i > j && i < nt) {
              tile2 L{0.0, 0.0};
              tile_mma(L, Ccur[t], Yinv);
              Lt[t] = L;
              tile_store(pcol + (i - j) * 64, lane, L);
              if (a.f32_factor) tile_store_split(colj + (i - j) * 64, lane, L);
              else tile_store(colj + (i - j) * 64, lane, L);
            }
          }
          if (wr == j % NW) {
            // z_j = inv(L_jj) (y_j - sum_k L(j,k) z_k): reduce the lane partials over q, then an 8x8 mat-vec in-warp
            double s = za + zb;
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            const double tr = ys[8 * j + r] - s;                                   // t[r], same on the 4 lanes of row r
            const double t0v = __shfl_sync(0xffffffffu, tr, 8 * q), t1v = __shfl_sync(0xffffffffu, tr, 8 * q + 4);
            double zv = fma(Yinv.a, t0v, Yinv.b * t1v);
            zv += __shfl_xor_sync(0xffffffffu, zv, 1);
            zv += __shfl_xor_sync(0xffffffffu, zv, 2);
            if (q == 0) zs[8 * j + r] = zv;
            za = 0.0; zb = 0.0;
          }
        }
        FIT_STAMP(3);
        named_bar_sync(2, FIT_THREADS);
        FIT_STAMP(4);
        // ---- (a) finish column c with the k = j term (X operand: the factor tile this warp has just produced) ----
        if (c < nt) {
          const tile2 Y = tile_load(pool + pool_idx(c, j) * 64, lane);
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int i = wr + NW * t;
            if (i > c && i < nt) {
              tile_mma(S0[t], Lt[t], Y);
              Ccur[t] = tile2{Kn[t].a - S0[t].a, Kn[t].b - S0[t].b};
            }
          }
          if (own_diag) {
            const double2 zk = *reinterpret_cast<const double2*>(zs + 8 * j + 2 * q);
            za = fma(Y.a, zk.x, za); zb = fma(Y.b, zk.y, zb);
          }
        }
        FIT_STAMP(5);
      }
    }
#ifdef CNGP_FIT_TIMING
    if (lane == 0 && blockIdx.x == 0)
      for (int k = 0; k < 6; ++k) a.dbg[w * 8 + k] += t_acc[k];
#endif
    __syncthreads();
    fail_pivot = s_fail;
    attempts_used = attempt;
    if (fail_pivot == 0) break;
    __syncthreads();
  }

  // ---- outputs: z, quad = z'z, logdet = 2 sum log L_kk, lml ----
  double* zp = a.z + lp * (long long)(nt * 8);
  double qs = 0.0, hl = 0.0;
  for (int i = tid; i < nt * 8; i += FIT_THREADS) {
    const double v = zs[i];
    zp[i] = v;
    qs += v * v;
    hl += log(dpiv[i]);      // padded rows have pivot 1
  }
  for (int o = 16; o; o >>= 1) {
    qs += __shfl_xor_sync(0xffffffffu, qs, o);
    hl += __shfl_xor_sync(0xffffffffu, hl, o);
  }
  if (lane == 0) { s_red[w] = qs; s_red2[w] = hl; }
  __syncthreads();
  if (tid == 0) {
    double quad = 0.0, hls = 0.0;
    for (int i = 0; i <= NW; ++i) { quad += s_red[i]; hls += s_red2[i]; }
    const double logdet = 2.0 * hls;
    const double nanv = __longlong_as_double(0x7ff8000000000000LL);
    const bool bad = fail_pivot != 0;
    if (a.quad) a.quad[p] = bad ? nanv : quad;
    if (a.logdet) a.logdet[p] = bad ? nanv : logdet;
    if (a.lml) a.lml[p] = bad ? nanv : 0.5 * (-(double)N * CNGP_LOG_2PI - logdet - quad);
    if (a.status) a.status[p] = bad ? -fail_pivot : attempts_used;
  }
}

}  // namespace cngp
