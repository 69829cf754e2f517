// Predict for windows that share one covariance (DESIGN.md section 4.2d).
//
// On the Toeplitz path everything but y is a function of theta, the stamp step d and the counts: with one theta for the
// whole call, windows with the same key (n, mc, d, m_s) - n training points, mc test points x_0 + (m_s + j) d - have
// bit-identical factors, lag tables, log det, t = Ky^-1 e_{n-1} and variance rows, whatever their x_0 and y.  A chunk
// then factors its largest such group once:
//   1. toep_key_kernel: every window's key, or -1 if the Schur fit or the Toeplitz variance would not take it on its
//      stamps alone (the predicates are the ones those kernels use: lag_extent, toep_uniform, tvt_lattice, TvtShape).
//   2. toep_group_kernel: the group = the windows with the key of the first qualifying window, in window order.
//   3. gp_toep_group_fit_kernel: gp_fit_toeplitz_kernel's factorisation of ONE problem on a whole CTA: the first
//      member's stamps with y = 0 (so that its acceptance depends on theta and the key only), into a slot of its own;
//      it also writes the diagonal tiles L_jj themselves.
//   4. gp_toep_member_kernel: CTA 0 runs gp_var_toeplitz_kernel's window code on that slot (the variance row); every
//      other warp takes one member: z = L^-1 y in the Schur recursion's own order, alpha by the same back substitution,
//      the mean by the same chain without the variance terms, and the LML from the group's log det.  The members of a
//      CTA read the factor from shared copies of its tile columns.
//   5. The per-window kernels run as before with the members marked (FitArgs::skip, VarArgs::skip), and
//      toep_var_broadcast_kernel copies the variance row to the members.
// A member gets exactly the bits the per-window Toeplitz path gives it.  Whatever that path would not take goes back to
// it before it runs: the whole group if the one-window fit or variance is not accepted (both depend on theta and the key
// only), one member if its own z, alpha or mean is not finite.
#pragma once
#include "gp_var_toeplitz.cuh"

namespace cngp {

#ifdef CNGP_TG_TIMING
// timing builds only (tools/toep_group_phases.py --timing): %globaltimer stamps, ns, of the group's fit and member
// kernels; cngp_api.cu resets them before the fit and prints them after the member kernel
__device__ unsigned long long tg_stamp[16];
__device__ __forceinline__ unsigned long long tg_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TG_STAMP(i) (tg_stamp[i] = tg_now())
#define TG_STAMP_MIN(i) atomicMin(&tg_stamp[i], tg_now())
#define TG_STAMP_MAX(i) atomicMax(&tg_stamp[i], tg_now())
#else
#define TG_STAMP(i) do { } while (0)
#define TG_STAMP_MIN(i) do { } while (0)
#define TG_STAMP_MAX(i) do { } while (0)
#endif

// group record (ints)
enum { TG_COUNT, TG_REP, TG_NONE, TG_FIT, TG_VAR, TG_N, TG_MC, TG_D, TG_MS, TG_INTS };
constexpr int TG_KEY_WARPS = 8;   // windows per CTA of toep_key_kernel
constexpr int TG_WARPS = 8;       // members per CTA of gp_toep_member_kernel

// 1. one warp per window of the chunk: key[lw] = (n, mc, d, m_s), or x = -1
__global__ void __launch_bounds__(TG_KEY_WARPS * 32) toep_key_kernel(const FitArgs a, const int* m_win, long long nw,
                                                                      int4* key) {
  __shared__ int s_xi_all[TG_KEY_WARPS][CNGP_MAX_N];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long lw = (long long)blockIdx.x * TG_KEY_WARPS + w;
  if (lw >= nw) return;
  const int win = (int)((a.problem0 + lw) % a.n_windows);
  const int n = a.n_win ? a.n_win[win] : a.N;
  const int mc = m_win ? m_win[win] : a.M;
  const double* x = a.x + (long long)win * a.N;
  int* xi = s_xi_all[w];
  const LagExtent ex = lag_extent<32>(a, win, n, lane, x, nullptr, nullptr);
  bool ok = ex.fit_tab() && ex.var_tab() && n >= 2 && mc >= 1;
  int d = 1, ms = 0;
  if (ok) {
    for (int i = lane; i < n; i += 32) xi[i] = (int)(x[i] - ex.base);   // fit_lag_tables' integer stamps
    __syncwarp();
    ok = toep_uniform(xi, n, lane, d);
    const double* xs = a.xstar + (a.xstar_stride ? (long long)win * a.xstar_stride : 0);
    ok = ok && tvt_lattice(xs, ex.base, xi[0], d, mc, lane, ms);
    ok = ok && TvtShape(n, ms, mc).need <= tvt_tab_cap(a.nt, a.M);
  }
  ok = __all_sync(0xffffffffu, ok);
  if (lane == 0) key[lw] = ok ? make_int4(n, mc, d, ms) : make_int4(-1, 0, 0, 0);
}

// 2. one CTA of 1024 threads: the members list[0 .. count) in window order (ballot + block scan, a fixed order),
// flag[w0 + lw] = 1 for the members and 0 for the other windows of the chunk, and the record
__global__ void __launch_bounds__(1024) toep_group_kernel(const int4* key, long long nw, long long w0, int* flag,
                                                          int* list, int* rec) {
  __shared__ int wsum[32];
  __shared__ int wpre[32];
  __shared__ int first;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (threadIdx.x == 0) first = INT_MAX;
  __syncthreads();
  for (long long i = threadIdx.x; i < nw; i += 1024)
    if (key[i].x >= 0) {
      atomicMin(&first, (int)i);
      break;
    }
  __syncthreads();
  const int f0 = first;
  const int4 k0 = f0 < nw ? key[f0] : make_int4(-1, 0, 0, 0);
  int base = 0;
  for (long long b0 = 0; b0 < nw; b0 += 1024) {
    const long long i = b0 + threadIdx.x;
    bool f = false;
    if (i < nw) {
      const int4 k = key[i];
      f = k0.x >= 0 && k.x == k0.x && k.y == k0.y && k.z == k0.z && k.w == k0.w;
      flag[w0 + i] = f ? 1 : 0;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) wsum[w] = __popc(bal);
    __syncthreads();
    if (w == 0) {
      const int v = wsum[lane];
      int incl = v;
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
      }
      wpre[lane] = incl - v;
    }
    __syncthreads();
    if (f) list[base + wpre[w] + __popc(bal & ((1u << lane) - 1u))] = (int)i;
    base += wpre[31] + wsum[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    rec[TG_COUNT] = base;
    rec[TG_REP] = (int)(w0 + (f0 < nw ? f0 : 0));
    rec[TG_NONE] = base == 0 ? 1 : 0;
    rec[TG_FIT] = 0;
    rec[TG_VAR] = 0;
    rec[TG_N] = k0.x; rec[TG_MC] = k0.y; rec[TG_D] = k0.z; rec[TG_MS] = k0.w;
  }
}

// 3. The group's factor on one CTA: gp_fit_toeplitz_kernel's arithmetic for its one problem (the first member's stamps,
// y = 0), with one row per thread instead of eight rows per lane, so a Schur step is a few instructions per thread and
// one barrier.  Every value is the per-window kernel's:
//  - the lag table and the generators are per entry / per row, whichever thread evaluates them;
//  - rho, s2, is, piv, ipiv and minp2 are recomputed identically by every thread;
//  - a row takes exactly the operations it takes there: the shift and the rotation only touch the rows of the "slots"
//    (32-row blocks) at or below the one of row k, and row 32 s reads 0 where slot s is the first live one;
//  - with y = 0 the residual stays +0 (fma(-u, +0, +0) = +0), so z and the quad are exact zeros.  The per-window
//    kernel refuses a problem whose residual is not finite: here that is a u value that is not finite in a live row, or
//    an ipiv that is not finite at some step.
// The tile columns leave through a ring of TGF_NS column copies: TGF_OUT_WARPS warps store the tiles below the diagonal,
// invert L_JJ in-warp and write ldiag, off the recursion's chain.  The log det is reduced in the per-window kernel's
// order (per lane over the slots, then the xor tree).
constexpr int TGF_ROWS = CNGP_MAX_N;   // recursion threads: one per row
constexpr int TGF_OUT_WARPS = 2;
constexpr int TGF_THREADS = TGF_ROWS + 32 * TGF_OUT_WARPS;
constexpr int TGF_NS = 4;              // tile-column copies in the ring
enum { TGF_BAR_STEP = 1, TGF_BAR_FULL = 2, TGF_BAR_EMPTY = 2 + TGF_NS };
static_assert(TGF_BAR_EMPTY + TGF_NS <= 16, "named barriers");
__host__ __device__ __forceinline__ size_t tgf_smem_bytes(int nt) { return (size_t)TGF_NS * 64 * nt * sizeof(double); }

__global__ void __launch_bounds__(TGF_THREADS, 1) gp_toep_group_fit_kernel(const FitArgs a) {
  extern __shared__ __align__(16) double tgf_ring[];   // [TGF_NS][8][R]: columns 8J .. 8J+7 of tile column J
  __shared__ KProg kps;
  __shared__ LeafConst hc[CNGP_MAX_LEAVES];
  __shared__ double s_ub[2][TGF_ROWS / 32];   // u of lane 31 of every warp, before the shift of the next step
  __shared__ double s_vb[2];                  // v_{k+1} for step k
  __shared__ double s_piv[TGF_ROWS];          // pivots (1 on the padding rows)
  __shared__ double s_ipiv[TGF_NS][8];        // 1 / L_kk of the tile columns in the ring
  __shared__ double s_dtile[64];              // L_JJ, row-major (first output warp)
  __shared__ double s_mm[4 * (TGF_THREADS / 32)];
  __shared__ int s_okv[TGF_THREADS / 32];
  __shared__ double s_kdiag;
  const unsigned FULL = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) { kps = a.kp; TG_STAMP(0); }
  if (a.skip && a.skip[0]) {
    if (tid == 0) a.done[0] = 1;
    return;
  }
  const int win = a.win_map ? a.win_map[0] : 0;
  const double* th = a.theta;
  const int ld = a.N, N = a.n_win ? a.n_win[win] : a.N, nt = a.nt, R = 8 * nt;
  const double noise = th[a.kp.n_params];
  if (N < 1) {
    if (tid == 0) a.done[0] = 0;
    return;
  }

  // ---- prologue on the whole CTA: stamps, lag tables, uniform stamps ----
  double* fx = tgf_ring;                                   // prologue only
  int* s_xi = reinterpret_cast<int*>(tgf_ring + R);
  for (int i = tid; i < R; i += TGF_THREADS) fx[i] = i < N ? a.x[(long long)win * ld + i] : 0.0;
  if (tid < a.kp.n_leaves) hc[tid] = leaf_prepare(a.kp.leaf_type[tid], th + a.kp.leaf_param[tid]);
  __syncthreads();
  const LagTab lt = fit_lag_tables<TGF_THREADS>(a, 0, win, N, nt, tid, fx, &kps, hc, noise, nullptr, s_xi, &s_kdiag, s_mm,
                                                s_okv);
  __syncthreads();
  int d = 1;
  const bool uni = lt.fit_tab && toep_uniform(s_xi, N, tid, d);   // thread tid checks rows tid, tid + 32, ...
  if (!__syncthreads_and(uni)) {
    if (tid == 0) a.done[0] = 0;
    return;
  }
  if (tid == 0) TG_STAMP(1);

  // ---- generators (every thread keeps the scalars of the recursion) ----
  const double t0 = s_kdiag + (noise + CNGP_JITTER);
  double piv = sqrt(t0), ipiv = 1.0 / piv, minp2 = t0;
  bool good = true, fin = true;
  double* Lp = a.L;
  if (tid < TGF_ROWS) {
    const int i = tid, sl = i >> 5;
    double u = 0.0;
    if (i == 0) u = piv;
    else if (i < N) u = keval_generic_cross(&kps, hc, (double)(i * d), 0.0) * ipiv;
    double v = i == 0 ? 0.0 : u;
    s_piv[i] = 1.0;
    if (lane == 31) s_ub[0][w] = u;
    if (i == 1) s_vb[0] = v;
    named_bar_sync(TGF_BAR_STEP, TGF_ROWS);   // s_ub, s_vb of step 0
    if (tid == 0) TG_STAMP(2);
    for (int k = 0; k < R; ++k) {
      const int SB = k >> 5, J = k >> 3, slot = J % TGF_NS, par = k & 1;
      const bool live = sl >= SB;
      if ((k & 7) == 0 && J >= TGF_NS) named_bar_sync(TGF_BAR_EMPTY + slot, TGF_THREADS);   // the copy is free
      if (k >= N) {   // identity padding: L(:, k) = e_k
        if (live) u = i == k ? 1.0 : 0.0;
        piv = 1.0; ipiv = 1.0;
      }
      if (i < R) tgf_ring[(slot * 8 + (k & 7)) * R + i] = u;
      if (i == 0) s_ipiv[slot][k & 7] = ipiv;
      if (i == k) s_piv[k] = piv;
      if (live) fin &= isfinite(u);
      fin &= isfinite(ipiv);
      if (k + 1 < N) {
        const double sh = __shfl_up_sync(FULL, u, 1);
        if (live && 32 * sl < R) {
          const double prev = sl == SB ? 0.0 : s_ub[par][w - 1];
          u = i >= N ? 0.0 : (lane == 0 ? prev : sh);
        }
        const double rho = s_vb[par] * ipiv;
        good &= fabs(rho) < 1.0;
        const double s2 = (1.0 - rho) * (1.0 + rho);
        const double is = rsqrt(s2);
        if (live) {
          const double un = fma(-rho, v, u) * is;
          v = fma(-rho, u, v) * is;
          u = un;
        }
        piv *= s2 * is;
        ipiv *= is;
        minp2 = fmin(minp2, piv * piv);
        if (i == k + 1) { u = piv; v = 0.0; }
      }
      if (lane == 31) s_ub[par ^ 1][w] = u;
      if (i == k + 2) s_vb[par ^ 1] = v;
      if ((k & 7) == 7) named_bar_arrive(TGF_BAR_FULL + slot, TGF_THREADS);   // tile column J is in the ring
      named_bar_sync(TGF_BAR_STEP, TGF_ROWS);
    }
    if (tid == 0) TG_STAMP(3);
  } else {
    // ---- output warps: tile column J from the ring to the packed factor, inv(L_JJ), ldiag ----
    const int ot = tid - TGF_ROWS;
    for (int J = 0; J < nt; ++J) {
      const int slot = J % TGF_NS;
      const double* st = tgf_ring + (size_t)slot * 8 * R;
      named_bar_sync(TGF_BAR_FULL + slot, TGF_THREADS);
      double* colJ = Lp + (long long)tile_index(J, J, nt) * 64;   // row i of tile column J at colJ + (i - 8J) 8
      const int npairs = 4 * (R - 8 * J - 8);
      for (int e = ot; e < npairs; e += 32 * TGF_OUT_WARPS) {
        const int i = 8 * J + 8 + (e >> 2), c = 2 * (e & 3);
        *reinterpret_cast<double2*>(colJ + (i - 8 * J) * 8 + c) = make_double2(st[c * R + i], st[(c + 1) * R + i]);
      }
      if (ot < 32) {
        s_dtile[lane] = st[(lane & 7) * R + 8 * J + (lane >> 3)];
        s_dtile[32 + lane] = st[(lane & 7) * R + 8 * J + 4 + (lane >> 3)];
        const double* ipiv8 = s_ipiv[slot];
        __syncwarp();
        // inv(L_JJ) by forward substitution on the identity, as gp_fit_toeplitz_kernel does it
        const int r = lane >> 2, q = lane & 3;
        tile2 x{r == 2 * q ? 1.0 : 0.0, r == 2 * q + 1 ? 1.0 : 0.0};
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const double xka = __shfl_sync(FULL, x.a, 4 * m + q), xkb = __shfl_sync(FULL, x.b, 4 * m + q);
          const double xsa = xka * ipiv8[m], xsb = xkb * ipiv8[m];
          const double lrm = s_dtile[8 * r + m];
          if (r == m) { x.a = xsa; x.b = xsb; }
          if (r > m) { x.a = fma(-lrm, xsa, x.a); x.b = fma(-lrm, xsb, x.b); }
        }
        tile_store(colJ, lane, x);
        if (a.ldiag) {
          a.ldiag[J * 64 + lane] = s_dtile[lane];
          a.ldiag[J * 64 + 32 + lane] = s_dtile[32 + lane];
        }
        __syncwarp();
      }
      if (J + TGF_NS < nt) named_bar_arrive(TGF_BAR_EMPTY + slot, TGF_THREADS);
    }
    if (ot == 0) TG_STAMP(4);
  }

  // ---- accept or hand the group back to the per-window path ----
  fin = fin && isfinite(piv) && isfinite(ipiv);
  good = good && minp2 >= TOEP_MIN_PIVOT2 * t0;
  const bool ok = __syncthreads_and(tid >= TGF_ROWS || (good && fin));
  if (w == 0) {
    double hl = 0.0;
    bool pf = true;
#pragma unroll
    for (int s = 0; s < TGF_ROWS / 32; ++s) {
      const double pv = s_piv[lane + 32 * s];
      pf &= isfinite(pv);
      hl += log(pv);
    }
    for (int o = 16; o; o >>= 1) hl += __shfl_xor_sync(FULL, hl, o);
    const bool acc = ok && __all_sync(FULL, pf);
    if (acc)
      for (int i = lane; i < R; i += 32) a.z[i] = 0.0;
    if (lane == 0) {
      if (acc && a.logdet) a.logdet[0] = 2.0 * hl;
      a.done[0] = acc ? 1 : 0;
      TG_STAMP(5);
    }
  }
}

struct TGArgs {
  VarArgs g;              // the group's slot: L, z (zeros), ktab, kmeta, kxi of the one-window fit; counts and test
                          // stamps of the call (read at window rec[TG_REP]); status null
  const double* ldiag;    // [nt][64] the diagonal tiles L_jj (row-major) of the group's factor
  const double* logdet;   // the group's log det
  double* gvar;           // [M] the group's variance row
  double* gmean;          // [M] the one-window fit's mean (y = 0; not used)
  const double* y;        // [n_windows][N]
  double* lml;            // [n_windows] or null
  int* status;            // [n_windows]
  double* mean;           // [n_windows][M]
  int* flag;              // [n_windows] members (cleared for what goes back to the per-window path)
  const int* list;        // members, local to the chunk
  int* rec;
  long long w0;           // first window of the chunk
};

// shared room of a member CTA: the chain table, then per warp z | alpha, then two copies of a factor tile column.
// The table and the per-warp room are rounded up to an even count of doubles: the back substitution reads z in 16-byte
// pairs, and the column copies are filled by 16-byte asynchronous copies.  A column copy holds the tiles I = J .. nt-1
// of tile column J and then L_JJ from ldiag, row by row with TG_RS doubles per row of 8: with 80-byte rows, the eight
// lanes of a 16-byte load phase that read consecutive rows hit distinct banks.
constexpr int TG_RS = 10;
__host__ __device__ __forceinline__ int tg_tab_doubles(int nt, int M) { return (tvt_tab_cap(nt, M) + 1) & ~1; }
__host__ __device__ __forceinline__ int tg_member_doubles(int nt) { return 2 * 8 * nt + TVT_P + 1; }
__host__ __device__ __forceinline__ int tg_col_doubles(int nt) { return 8 * (nt + 1) * TG_RS; }
__host__ __device__ __forceinline__ size_t tg_smem_bytes(int nt, int M) {
  const int members = tg_tab_doubles(nt, M) + TG_WARPS * tg_member_doubles(nt) + 2 * tg_col_doubles(nt);
  const int grp = tvt_warp_doubles(nt, M);
  return (size_t)(members > grp ? members : grp) * sizeof(double);
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// tile column J of the group's factor (and, with diag, L_JJ) -> buf, by the whole CTA; the caller waits and syncs
__device__ __forceinline__ void tg_stage_col(double* buf, const double* Lp, const double* ldiag, int J, int nt,
                                             bool diag) {
  const int rc = 8 * (nt - J), rows = rc + (diag ? 8 : 0);
  const double* col = Lp + (long long)tile_index(J, J, nt) * 64;
  for (int g = threadIdx.x; g < 4 * rows; g += TG_WARPS * 32) {
    const int r = g >> 2, c = 2 * (g & 3);
    cp_async16(buf + r * TG_RS + c, r < rc ? col + r * 8 + c : ldiag + J * 64 + (r - rc) * 8 + c);
  }
  cp_async_commit();
}

// 4. CTA 0: the group's variance row (warp 0); CTAs 1..: one member per warp.  The warps of a CTA walk the factor's
// tile columns together - up for z, down for alpha - and read each column from one shared copy, which the CTA fills
// with the next column while it works on the current one.  So every warp takes part in every column, also one without
// a member or whose member has failed; such a warp writes nothing.
__global__ void __launch_bounds__(TG_WARPS * 32, 2) gp_toep_member_kernel(const TGArgs t) {
  extern __shared__ __align__(16) double tg_smem[];
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int* rec = t.rec;
  if (rec[TG_NONE]) return;
  const int count = rec[TG_COUNT];
  const bool fit_ok = rec[TG_FIT] != 0;
  if (blockIdx.x == 0) {
    if (w != 0) return;
    if (lane == 0) TG_STAMP(8);
    const bool ok = fit_ok && tvt_window(t.g, 0, rec[TG_REP], tg_smem, t.gmean, t.gvar, lane);
    if (lane == 0) { rec[TG_VAR] = ok ? 1 : 0; TG_STAMP(9); }
    if (!ok)   // the whole group goes back to the per-window path
      for (int i = lane; i < count; i += 32) t.flag[t.w0 + t.list[i]] = 0;
    return;
  }
  if (threadIdx.x == 0) TG_STAMP_MIN(10);
  const long long idx = (long long)(blockIdx.x - 1) * TG_WARPS + w;
  const bool have = idx < count;
  const long long win = have ? t.w0 + t.list[idx] : 0;
  if (!fit_ok) {
    if (have && lane == 0) t.flag[win] = 0;
    return;
  }
  const int nt = t.g.nt, R = 8 * nt, M = t.g.M;
  const int n = rec[TG_N], mc = rec[TG_MC], d = rec[TG_D], ms = rec[TG_MS];
  const TvtShape sh(n, ms, mc);
  double* s_tab = tg_smem;   // the group's chain table, shared by the CTA's members
  double* s_z = tg_smem + tg_tab_doubles(nt, M) + (size_t)w * tg_member_doubles(nt);
  double* s_al = s_z + R;
  double* const s_col = tg_smem + tg_tab_doubles(nt, M) + (size_t)TG_WARPS * tg_member_doubles(nt);
  const int CD = tg_col_doubles(nt);
  const double* Lp = t.g.L;
  tg_stage_col(s_col, Lp, t.ldiag, 0, nt, true);
  tvt_table(s_tab, t.g.ktab, sh, n, d, threadIdx.x, TG_WARPS * 32);
  int cur = 0;   // the column copy being read: s_col + cur CD

  // ---- z = L^-1 y: gp_fit_toeplitz_kernel's recursion with the stored columns (rows dealt the same way) ----
  double rr[TOEP_SLOTS];
#pragma unroll
  for (int s = 0; s < TOEP_SLOTS; ++s) {
    const int i = lane + 32 * s;
    rr[s] = have && i < n ? t.y[win * (long long)t.g.N + i] : 0.0;
  }
  auto block = [&](auto sbc) {
    constexpr int SB = decltype(sbc)::value;
    const int J1 = min(4 * SB + 4, nt);
    for (int J = 4 * SB; J < J1; ++J) {
      cp_async_wait_all();
      __syncthreads();   // column J is in the copy cur; every warp is done with the other copy
      // the next column: J + 1 for z, or the last one, where the back substitution starts
      tg_stage_col(s_col + (cur ^ 1) * CD, Lp, t.ldiag, J + 1 < nt ? J + 1 : nt - 1, nt, J + 1 < nt);
      const double* colJ = s_col + cur * CD;
      for (int h = 0; h < 2; ++h) {
        // column k = 8J + 4h + c of L at the rows of this lane: the tiles below the diagonal, L_JJ from ldiag, zero above
        double lk[TOEP_SLOTS][4];
#pragma unroll
        for (int s = SB; s < TOEP_SLOTS; ++s) {
          const int i = lane + 32 * s, I = i >> 3;
          double2 l0 = make_double2(0.0, 0.0), l1 = make_double2(0.0, 0.0);
          const double* src = colJ + (I == J ? 8 * (nt - J) + (i & 7) : i - 8 * J) * TG_RS + 4 * h;
          if (I >= J && I < nt) {
            l0 = *reinterpret_cast<const double2*>(src);
            l1 = *reinterpret_cast<const double2*>(src + 2);
          }
          lk[s][0] = l0.x; lk[s][1] = l0.y; lk[s][2] = l1.x; lk[s][3] = l1.y;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int k = 8 * J + 4 * h + c, kk = k & 31;
          const double ipiv = colJ[(4 * h + c) * (TG_RS + 1)];   // diagonal of the stored inv(L_JJ): 1 / L_kk, bit for bit
          const double zk = __shfl_sync(FULL, rr[SB], kk) * ipiv;
#pragma unroll
          for (int s = SB; s < TOEP_SLOTS; ++s) rr[s] = fma(-lk[s][c], zk, rr[s]);
          if (lane == kk) rr[SB] = zk;
        }
      }
      cur ^= 1;
    }
  };
  static_assert(TOEP_SLOTS == 8 && (TVT_P & 1), "unrolled slot blocks below; tg_member_doubles rounds 2R + TVT_P up");
  block(FitIC<0>{});
  if (R > 32) block(FitIC<1>{});
  if (R > 64) block(FitIC<2>{});
  if (R > 96) block(FitIC<3>{});
  if (R > 128) block(FitIC<4>{});
  if (R > 160) block(FitIC<5>{});
  if (R > 192) block(FitIC<6>{});
  if (R > 224) block(FitIC<7>{});
  bool fin = true;
#pragma unroll
  for (int s = 0; s < TOEP_SLOTS; ++s) {
    fin &= isfinite(rr[s]);
    if (lane + 32 * s < R) s_z[lane + 32 * s] = rr[s];
  }
  bool live = have && __all_sync(FULL, fin);
  if (lane == 0) TG_STAMP_MAX(12);
  if (have && !live && lane == 0) t.flag[win] = 0;
  const double qs = toep_quad(rr);
  __syncwarp();

  // ---- alpha = Ky^-1 y (tvt_backsub<false>'s steps on the shared column copies) and the mean ----
  {
    double inv_last = 0.0, maxinv2 = 0.0;
    for (int J = nt - 1; J >= 0; --J) {
      cp_async_wait_all();
      __syncthreads();
      if (J > 0) tg_stage_col(s_col + (cur ^ 1) * CD, Lp, t.ldiag, J - 1, nt, false);
      tvt_backsub_col<false, TG_RS>(s_col + cur * CD, J, s_z, n, nt, lane, s_al, nullptr, inv_last, maxinv2);
      cur ^= 1;
    }
  }
  if (lane == 0) TG_STAMP_MAX(13);
  if (!live) return;   // no barrier below
  const int npad = (n + TVT_P - 1) / TVT_P * TVT_P;
  for (int i = lane; i < npad; i += 32) {
    if (i < n) fin &= isfinite(s_al[i]);
    else s_al[i] = 0.0;
  }
  if (!__all_sync(FULL, fin)) {
    if (lane == 0) t.flag[win] = 0;
    return;
  }
  __syncwarp();
  fin = tvt_chain<false>(s_tab, s_al, nullptr, nullptr, n, sh, ms, mc, 0.0, 0.0, 0.0, 0.0, 0, t.mean + win * (long long)M,
                         nullptr, lane);
  fin = __all_sync(FULL, fin);
  if (lane == 0) {
    if (fin) {
      if (t.lml) t.lml[win] = toep_lml(n, *t.logdet, qs);
      t.status[win] = 0;
    } else {
      t.flag[win] = 0;   // the per-window path rewrites the mean row
    }
    TG_STAMP_MAX(11);
  }
}

// 5. the group's variance row to every member still flagged; one warp per member
__global__ void __launch_bounds__(128) toep_var_broadcast_kernel(const int* list, const int* rec, const int* flag,
                                                                 const double* gvar, double* var, long long w0, int M) {
  const int lane = threadIdx.x & 31;
  const long long idx = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (rec[TG_NONE] || idx >= rec[TG_COUNT]) return;
  const long long win = w0 + list[idx];
  if (!flag[win]) return;
  const int mc = rec[TG_MC];
  double* dst = var + win * (long long)M;
  for (int j = lane; j < mc; j += 32) dst[j] = gvar[j];
}

}  // namespace cngp
