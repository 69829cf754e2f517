// Predict for windows that share one covariance (DESIGN.md section 4.2d).
//
// On the Toeplitz path everything but y is a function of theta, the stamp step d and the counts: with one theta for the
// whole call, windows with the same key (n, mc, d, m_s) - n training points, mc test points x_0 + (m_s + j) d - have
// bit-identical factors, lag tables, log det, t = Ky^-1 e_{n-1} and variance rows, whatever their x_0 and y.  A chunk
// then factors its largest such group once:
//   1. toep_key_kernel: every window's key, or -1 if the Schur fit or the Toeplitz variance would not take it on its
//      stamps alone (the predicates are the ones those kernels use: lag_extent, toep_uniform, tvt_lattice, TvtShape).
//   2. toep_group_kernel: the group = the windows with the key of the first qualifying window, in window order.
//   3. gp_fit_toeplitz_kernel on ONE problem: the first member's stamps with y = 0 (so that its acceptance depends on
//      theta and the key only), into a slot of its own; it also writes the diagonal tiles L_jj themselves.
//   4. gp_toep_member_kernel: CTA 0 runs gp_var_toeplitz_kernel's window code on that slot (the variance row); every
//      other warp takes one member: z = L^-1 y in the Schur recursion's own order, alpha by the same back substitution,
//      the mean by the same chain without the variance terms, and the LML from the group's log det.
//   5. The per-window kernels run as before with the members marked (FitArgs::skip, VarArgs::skip), and
//      toep_var_broadcast_kernel copies the variance row to the members.
// A member gets exactly the bits the per-window Toeplitz path gives it.  Whatever that path would not take goes back to
// it before it runs: the whole group if the one-window fit or variance is not accepted (both depend on theta and the key
// only), one member if its own z, alpha or mean is not finite.
#pragma once
#include "gp_var_toeplitz.cuh"

namespace cngp {

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

// shared room of a member CTA: the chain table, then per warp z | alpha.  Both rounded up to an even count of doubles:
// the back substitution reads z in 16-byte pairs.
__host__ __device__ __forceinline__ int tg_tab_doubles(int nt, int M) { return (tvt_tab_cap(nt, M) + 1) & ~1; }
__host__ __device__ __forceinline__ int tg_member_doubles(int nt) { return 2 * 8 * nt + TVT_P + 1; }
__host__ __device__ __forceinline__ size_t tg_smem_bytes(int nt, int M) {
  const int members = tg_tab_doubles(nt, M) + TG_WARPS * tg_member_doubles(nt);
  const int grp = tvt_warp_doubles(nt, M);
  return (size_t)(members > grp ? members : grp) * sizeof(double);
}

// 4. CTA 0: the group's variance row (warp 0); CTAs 1..: one member per warp
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
    const bool ok = fit_ok && tvt_window(t.g, 0, rec[TG_REP], tg_smem, t.gmean, t.gvar, lane);
    if (lane == 0) rec[TG_VAR] = ok ? 1 : 0;
    if (!ok)   // the whole group goes back to the per-window path
      for (int i = lane; i < count; i += 32) t.flag[t.w0 + t.list[i]] = 0;
    return;
  }
  const int nt = t.g.nt, R = 8 * nt, M = t.g.M;
  const int n = rec[TG_N], mc = rec[TG_MC], d = rec[TG_D], ms = rec[TG_MS];
  const TvtShape sh(n, ms, mc);
  double* s_tab = tg_smem;   // the group's chain table, shared by the CTA's members
  if (fit_ok) tvt_table(s_tab, t.g.ktab, sh, n, d, threadIdx.x, TG_WARPS * 32);
  __syncthreads();
  const long long idx = (long long)(blockIdx.x - 1) * TG_WARPS + w;
  if (idx >= count) return;
  const long long win = t.w0 + t.list[idx];
  if (!fit_ok) {
    if (lane == 0) t.flag[win] = 0;
    return;
  }
  double* s_z = tg_smem + tg_tab_doubles(nt, M) + (size_t)w * tg_member_doubles(nt);
  double* s_al = s_z + R;

  // ---- z = L^-1 y: gp_fit_toeplitz_kernel's recursion with the stored columns (rows dealt the same way) ----
  const double* Lp = t.g.L;
  double rr[TOEP_SLOTS];
#pragma unroll
  for (int s = 0; s < TOEP_SLOTS; ++s) {
    const int i = lane + 32 * s;
    rr[s] = i < n ? t.y[win * (long long)t.g.N + i] : 0.0;
  }
  auto block = [&](auto sbc) {
    constexpr int SB = decltype(sbc)::value;
    const int J1 = min(4 * SB + 4, nt);
    for (int J = 4 * SB; J < J1; ++J) {
      const double* colJ = Lp + (long long)tile_index(J, J, nt) * 64;
      for (int h = 0; h < 2; ++h) {
        // column k = 8J + 4h + c of L at the rows of this lane: the tiles below the diagonal, L_JJ from ldiag, zero above
        double lk[TOEP_SLOTS][4];
#pragma unroll
        for (int s = SB; s < TOEP_SLOTS; ++s) {
          const int i = lane + 32 * s, I = i >> 3;
          double2 l0 = make_double2(0.0, 0.0), l1 = make_double2(0.0, 0.0);
          const double* src = I == J ? t.ldiag + J * 64 + (i & 7) * 8 + 4 * h
                                     : colJ + (I - J) * 64 + (i & 7) * 8 + 4 * h;
          if (I >= J && I < nt) {
            l0 = *reinterpret_cast<const double2*>(src);
            l1 = *reinterpret_cast<const double2*>(src + 2);
          }
          lk[s][0] = l0.x; lk[s][1] = l0.y; lk[s][2] = l1.x; lk[s][3] = l1.y;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int k = 8 * J + 4 * h + c, kk = k & 31;
          const double ipiv = colJ[9 * (4 * h + c)];   // diagonal of the stored inv(L_JJ): 1 / L_kk, bit for bit
          const double zk = __shfl_sync(FULL, rr[SB], kk) * ipiv;
#pragma unroll
          for (int s = SB; s < TOEP_SLOTS; ++s) rr[s] = fma(-lk[s][c], zk, rr[s]);
          if (lane == kk) rr[SB] = zk;
        }
      }
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
  if (!__all_sync(FULL, fin)) {
    if (lane == 0) t.flag[win] = 0;
    return;
  }
  const double qs = toep_quad(rr);
  __syncwarp();

  // ---- alpha = Ky^-1 y and the mean ----
  tvt_backsub<false>(Lp, s_z, n, nt, lane, s_al, nullptr);
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
