// Phase B for windows whose Ky is Toeplitz and whose test points lie on the lattice of the training stamps
// (DESIGN.md section 4.2c).
//
// With stamps x_i = x_0 + i d and a stationary expression, Ky = K + s I is symmetric Toeplitz (s = t0 - k*(0): noise,
// jitter and any White variance, which K* does not have).  The column of the test point p_m = x_0 + m d is
// k_m[i] = k*((i - m) d), so k_{m+1} = Z k_m + k*(-(m+1) d) e_0 (Z the down-shift), and A = Ky^-1 has displacement
// rank 2: with a = A e_0, gamma = a_0 and t = J a (A is persymmetric),  A - Z^T A Z = (t t^T - (Z^T a)(Z^T a)^T) / gamma.
// Hence q_m = k_m^T A k_m obeys the scalar recurrence
//     q_{m+1} = q_m + ((a^T k_{m+1})^2 - (t^T k_m)^2) / gamma,
// anchored in closed form at m = 0 and m = n-1, where k_m = (Ky - s I) e_m:  q = t0 - 2 s + s^2 gamma.  The variance
// phase then costs three dot products of length n per chain point (a^T k, t^T k and the mean alpha^T k) instead of the
// N^2 M forward substitution of gp_var_kernel.
//
// One warp per window, TVT_WARPS windows per CTA.
//   1. alpha = A y and w = A e_{n-1} = t by ONE back substitution with two right-hand sides over the stored factor:
//      L^T [alpha, w] = [z, e_{n-1} / L_{n-1,n-1}]  (z from phase A; the diagonal tiles hold inv(L_jj)).  The factor is
//      read once, tile column by tile column, each tile as one 16-byte load per lane.
//   2. The chain m0 .. m_end (m0 = n-1 if the first test point is at or beyond x_{n-1}, else 0) is dealt over the lanes
//      in blocks of TVT_P consecutive points.  A lane slides its TVT_P table values along i in a register ring, so one
//      table load (conflict-free: TVT_P is odd) feeds 3 TVT_P FMA; alpha_i, a_i, t_i are warp-wide broadcasts.
//   3. The increments are summed in a fixed order (sequential inside a lane, then a warp scan of the lane totals, then
//      the carry of the previous pass), so the results do not depend on scheduling.
//
// A window is taken only if its own data allow it: phase A status 0, a valid lag table, uniform integer stamps with
// d >= 1, consecutive lattice test points x_0 + (m_s + j) d (m_s >= 0), the chain's table within the warp's shared
// room, the conditioning guard of the Schur fit (min_k L_kk^2 >= TOEP_MIN_PIVOT2 t0, read from the inverted diagonal
// tiles) and every value finite.  taken[lw] says which; gp_var_kernel handles the others through the compacted list.
#pragma once
#include "gp_fit_toeplitz.cuh"
#include "gp_var.cuh"

namespace cngp {

constexpr int TVT_WARPS = 4;   // windows per CTA
constexpr int TVT_P = 9;       // chain points per lane and pass: odd, so lanes TVT_P doubles apart hit distinct banks

// shared table room (doubles) of one warp: the chain of a test grid of M consecutive points covers at most n + M lags
__host__ __device__ __forceinline__ int tvt_tab_cap(int nt, int M) {
  const int R = 8 * nt, span = (M < VAR_TAB_MAX ? M : VAR_TAB_MAX) + R;
  return TVT_P + R + (span + 32 * TVT_P - 1) / (32 * TVT_P) * (32 * TVT_P);
}
// per warp: alpha, a, t (8 nt + TVT_P each, zero beyond n) | the chain's lag table
__host__ __device__ __forceinline__ int tvt_warp_doubles(int nt, int M) { return 3 * (8 * nt + TVT_P) + tvt_tab_cap(nt, M); }
__host__ __device__ __forceinline__ size_t tvt_smem_bytes(int nt, int M) { return (size_t)TVT_WARPS * tvt_warp_doubles(nt, M) * sizeof(double); }

// Test points x_0 + (m_s + j) d, j < mc, consecutive on the lattice of the stamps (m_s >= 0): this lane's share of the
// check (the caller takes the warp vote).  base: the window's base stamp, xi0 = x_0 - base.
__device__ __forceinline__ bool tvt_lattice(const double* xs, double base, int xi0, int d, int mc, int lane, int& ms) {
  const int mi0 = (int)(xs[0] - base) - xi0;   // offset of the first test point from x_0, in stamp units
  bool ok = mi0 >= 0 && mi0 % d == 0;
  ms = ok ? mi0 / d : 0;
  for (int j = lane; ok && j < mc; j += 32) ok = (int)(xs[j] - base) - xi0 == mi0 + j * d;
  return ok;
}
// The chain of a window with n training points and the test grid m_s .. m_s + mc - 1: chain points m0 .. mend, the
// passes over them and the table entries the passes read
struct TvtShape {
  int m0, mend, passes, need;
  __device__ __forceinline__ TvtShape(int n, int ms, int mc) {
    m0 = ms >= n - 1 ? n - 1 : 0;
    mend = ms + mc - 1;
    passes = (mend - m0 + 1 + 32 * TVT_P - 1) / (32 * TVT_P);
    need = TVT_P + n - 1 + passes * 32 * TVT_P;
  }
};

// [alpha, w] = L^-T [z, e_{n-1} / L_{n-1,n-1}] by one back substitution over the stored factor, tile column
// J = nt-1 .. 0, into s_al (and, with W, s_t).  W also returns max_k inv(L)_kk^2 over k < n (the conditioning guard).
// Without W the alpha half is the same arithmetic, so alpha has the same bits either way.
// tvt_backsub_col is the step of tile column J: col holds its tiles I = J .. nt-1 (inv(L_JJ) first) as rows
// 8 (I - J) + r of RS doubles each - RS = 8 in the packed factor, more where a shared-memory copy pads its rows.
template <bool W, int RS>
__device__ __forceinline__ void tvt_backsub_col(const double* col, int J, const double* zp, int n, int nt, int lane,
                                                double* s_al, double* s_t, double& inv_last, double& maxinv2) {
  const unsigned FULL = 0xffffffffu;
  const int r = lane >> 2, q = lane & 3;
  col += r * RS + 2 * q;
  const double2 dg = *reinterpret_cast<const double2*>(col);   // inv(L_JJ), row r, columns 2q, 2q+1
  double c0a = 0.0, c0b = 0.0, c1a = 0.0, c1b = 0.0;             // (L_IJ^T x_I) for columns 2q, 2q+1: alpha | w
#pragma unroll 8
  for (int I = J + 1; I < nt; ++I) {
    const double2 l = *reinterpret_cast<const double2*>(col + (I - J) * 8 * RS);
    const double xa = s_al[8 * I + r];
    c0a = fma(l.x, xa, c0a); c0b = fma(l.y, xa, c0b);
    if (W) {
      const double xw = s_t[8 * I + r];
      c1a = fma(l.x, xw, c1a); c1b = fma(l.y, xw, c1b);
    }
  }
  // rows of the diagonal tile: pivots of the guard, 1 / L_{n-1,n-1}
  const int row = 8 * J + r;
  const double dv = (r == 2 * q) ? dg.x : (r == 2 * q + 1 ? dg.y : 0.0);
  if (W) {
    if ((r >> 1) == q && row < n) maxinv2 = fmax(maxinv2, dv * dv);
    if (J == nt - 1) {
      const int kl = (n - 1) & 7;   // n-1 lies in the last tile column
      inv_last = __shfl_sync(FULL, dv, 4 * kl + (kl >> 1));
    }
  }
  for (int o = 4; o < 32; o <<= 1) {
    c0a += __shfl_xor_sync(FULL, c0a, o); c0b += __shfl_xor_sync(FULL, c0b, o);
    if (W) { c1a += __shfl_xor_sync(FULL, c1a, o); c1b += __shfl_xor_sync(FULL, c1b, o); }
  }
  // right-hand sides of rows 8J + 2q (+1), then gathered to row r = lane >> 2
  const int ca = 8 * J + 2 * q;
  const double2 zz = *reinterpret_cast<const double2*>(zp + ca);
  const double b0a = zz.x - c0a, b0b = zz.y - c0b;
  const double g0a = __shfl_sync(FULL, b0a, r >> 1), g0b = __shfl_sync(FULL, b0b, r >> 1);
  const double h0 = (r & 1) ? g0b : g0a;
  double h1 = 0.0;
  if (W) {
    const double b1a = (ca == n - 1 ? inv_last : 0.0) - c1a, b1b = (ca + 1 == n - 1 ? inv_last : 0.0) - c1b;
    const double g1a = __shfl_sync(FULL, b1a, r >> 1), g1b = __shfl_sync(FULL, b1b, r >> 1);
    h1 = (r & 1) ? g1b : g1a;
  }
  // x_J[c] = sum_r inv(L_JJ)[r][c] rhs[r]  (lower triangle only)
  const double la = r >= 2 * q ? dg.x : 0.0, lb = r >= 2 * q + 1 ? dg.y : 0.0;
  double x0a = la * h0, x0b = lb * h0, x1a = 0.0, x1b = 0.0;
  if (W) { x1a = la * h1; x1b = lb * h1; }
  for (int o = 4; o < 32; o <<= 1) {
    x0a += __shfl_xor_sync(FULL, x0a, o); x0b += __shfl_xor_sync(FULL, x0b, o);
    if (W) { x1a += __shfl_xor_sync(FULL, x1a, o); x1b += __shfl_xor_sync(FULL, x1b, o); }
  }
  if (r == 0) {
    s_al[ca] = x0a; s_al[ca + 1] = x0b;
    if (W) { s_t[ca] = x1a; s_t[ca + 1] = x1b; }
  }
  __syncwarp();
}
template <bool W>
__device__ __forceinline__ double tvt_backsub(const double* Lp, const double* zp, int n, int nt, int lane, double* s_al,
                                              double* s_t) {
  const unsigned FULL = 0xffffffffu;
  double inv_last = 0.0, maxinv2 = 0.0;
  for (int J = nt - 1; J >= 0; --J)
    tvt_backsub_col<W, 8>(Lp + (long long)tile_index(J, J, nt) * 64, J, zp, n, nt, lane, s_al, s_t, inv_last, maxinv2);
  if (W)
    for (int o = 16; o; o >>= 1) maxinv2 = fmax(maxinv2, __shfl_xor_sync(FULL, maxinv2, o));
  return maxinv2;
}

// s_tab[j] = k*(|L| d), L = j - TVT_P - (n-1) + m0 the lag (in lattice steps) of chain offset c and row i at
// j = TVT_P + n-1 + c - i; entries outside the real (c, i) range are 0.  Threads tid, tid + nth, ...
__device__ __forceinline__ void tvt_table(double* s_tab, const double* ktab, const TvtShape& sh, int n, int d, int tid,
                                          int nth) {
  const int lmin = sh.m0 - (n - 1);
  for (int j = tid; j < sh.need; j += nth) {
    const int L = j - TVT_P - (n - 1) + sh.m0;
    s_tab[j] = (L >= lmin && L <= sh.mend) ? ktab[(L < 0 ? -L : L) * d] : 0.0;
  }
}

// The chain.  Every lane runs TVT_P consecutive chain points per pass; the mean alpha^T k always, and with UV the
// recurrence terms a^T k, t^T k and the variance.  Returns this lane's "every result finite".
template <bool UV>
__device__ __forceinline__ bool tvt_chain(const double* s_tab, const double* s_al, const double* s_a, const double* s_t,
                                          int n, const TvtShape& sh, int ms, int mc, double q0, double igam, double kss,
                                          double noise, int sigma_mode, double* mean, double* var, int lane) {
  const unsigned FULL = 0xffffffffu;
  const int npad = (n + TVT_P - 1) / TVT_P * TVT_P;
  const int cout0 = ms - sh.m0;   // chain offset of test point 0
  double carry = 0.0, vcarry = 0.0;   // sum of the increments of the earlier passes; t^T k of the last point before
  bool fin = true;
  for (int pass = 0; pass < sh.passes; ++pass) {
    const int c0 = pass * 32 * TVT_P + lane * TVT_P;   // this lane's first chain offset
    const double* tb = s_tab + TVT_P + (n - 1) + c0;    // K(i, p) = tb[p - i]
    double kw[TVT_P], mu[TVT_P], u[TVT_P], v[TVT_P];
#pragma unroll
    for (int p = 0; p < TVT_P; ++p) {
      kw[p] = p ? tb[p] : 0.0;   // slot (p - i) mod P holds K(i, p); slot 0 is loaded at i = 0
      mu[p] = 0.0; u[p] = 0.0; v[p] = 0.0;
    }
    for (int i0 = 0; i0 < npad; i0 += TVT_P) {
#pragma unroll
      for (int st = 0; st < TVT_P; ++st) {
        const int i = i0 + st;
        kw[(TVT_P - st) % TVT_P] = tb[-i];
        const double al = s_al[i];
#pragma unroll
        for (int p = 0; p < TVT_P; ++p) {
          const double k = kw[(p - st + TVT_P) % TVT_P];
          mu[p] = fma(al, k, mu[p]);
        }
        if (UV) {
          const double aa = s_a[i], tt = s_t[i];
#pragma unroll
          for (int p = 0; p < TVT_P; ++p) {
            const double k = kw[(p - st + TVT_P) % TVT_P];
            u[p] = fma(aa, k, u[p]);
            v[p] = fma(tt, k, v[p]);
          }
        }
      }
    }
    if (!UV) {
#pragma unroll
      for (int p = 0; p < TVT_P; ++p) {
        const int j = c0 + p - cout0;
        if (j >= 0 && j < mc) {
          fin &= isfinite(mu[p]);
          mean[j] = mu[p];
        }
      }
      continue;
    }
    // increments delta_c = u_c^2 - v_{c-1}^2 (delta_0 = 0: the anchor), summed in chain order
    double vprev = __shfl_up_sync(FULL, v[TVT_P - 1], 1);
    if (lane == 0) vprev = vcarry;
    double ps[TVT_P];
    double acc = 0.0;
#pragma unroll
    for (int p = 0; p < TVT_P; ++p) {
      const double vp = p ? v[p - 1] : vprev;
      const double dl = (c0 + p == 0) ? 0.0 : fma(u[p], u[p], -vp * vp);
      acc += dl;
      ps[p] = acc;
    }
    double incl = acc;
    for (int o = 1; o < 32; o <<= 1) {
      const double y = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += y;
    }
    double excl = __shfl_up_sync(FULL, incl, 1);
    if (lane == 0) excl = 0.0;
    const double base = carry + excl;
#pragma unroll
    for (int p = 0; p < TVT_P; ++p) {
      const int j = c0 + p - cout0;   // test point of chain offset c0 + p
      if (j >= 0 && j < mc) {
        const double qm = fma(base + ps[p], igam, q0);
        const double vv = fmax(kss - qm, CNGP_VAR_FLOOR) + noise;
        const double out = sigma_mode ? 2.0 * sqrt(vv) : vv;
        fin &= isfinite(mu[p]) && isfinite(out);
        mean[j] = mu[p];
        var[j] = out;
      }
    }
    carry += __shfl_sync(FULL, incl, 31);
    vcarry = __shfl_sync(FULL, v[TVT_P - 1], 31);
  }
  return fin;
}

// One window on one warp: slot lw of the phase-A buffers (factor, z, table, meta, integer stamps), window win of the
// call (counts, test stamps, status), results to mean_row / var_row.  s_w: the warp's shared room (tvt_warp_doubles).
// Returns (warp-uniform) whether the window was taken; a window not taken has had nothing written.
__device__ __forceinline__ bool tvt_window(const VarArgs& a, long long lw, long long win, double* s_w, double* mean_row,
                                           double* var_row, int lane) {
  const unsigned FULL = 0xffffffffu;
  const int nt = a.nt, R = 8 * nt, M = a.M;
  const int cap = tvt_tab_cap(nt, M);
  double* s_al = s_w;
  double* s_a = s_al + R + TVT_P;
  double* s_t = s_a + R + TVT_P;
  double* s_tab = s_t + R + TVT_P;

  // ---- the window's own qualification (no factor read yet) ----
  const double* km = a.kmeta + lw * (long long)VAR_META;
  const int* xi = a.kxi + lw * (long long)R;
  const int n = a.n_win ? a.n_win[win] : a.N;
  const int mc = a.m_win ? a.m_win[win] : M;
  bool ok = km[3] != 0.0 && n >= 2 && mc >= 1 && !(a.status && a.status[win] != 0);
  int d = 1, ms = 0;
  if (ok) {
    ok = toep_uniform(xi, n, lane, d);
    const double* xs = a.xstar + (a.xstar_stride ? win * a.xstar_stride : 0);
    ok = ok && tvt_lattice(xs, km[1], xi[0], d, mc, lane, ms);
  }
  const TvtShape sh(n, ms, mc);
  ok = ok && sh.need <= cap;
  if (!__all_sync(FULL, ok)) return false;

  // ---- [alpha, w] = L^-T [z, e_{n-1} / L_{n-1,n-1}] ----
  const double maxinv2 = tvt_backsub<true>(a.L + lw * (long long)tiles_in_lower(nt) * 64, a.z + lw * (long long)R, n, nt,
                                           lane, s_al, s_t);

  // ---- anchor, guard, a = J t, zero padding, the chain's lag table ----
  const double kss = km[0], noise = km[2];
  const double* ktab = a.ktab + lw * (long long)VAR_TAB_MAX;
  const double t0 = kss + (noise + CNGP_JITTER);
  const double s = t0 - ktab[0];
  const double gam = s_t[n - 1];
  const double q0 = t0 - 2.0 * s + s * s * gam;
  // min_k L_kk^2 >= g t0  <=>  max_k inv(L)_kk^2 <= 1 / (g t0)
  bool good = maxinv2 * (TOEP_MIN_PIVOT2 * t0) <= 1.0 && isfinite(q0) && gam > 0.0;
  const int npad = (n + TVT_P - 1) / TVT_P * TVT_P;
  for (int i = lane; i < npad; i += 32) {
    if (i < n) {
      good &= isfinite(s_al[i]) && isfinite(s_t[i]);
      s_a[i] = s_t[n - 1 - i];
    } else {
      s_al[i] = 0.0; s_a[i] = 0.0; s_t[i] = 0.0;
    }
  }
  tvt_table(s_tab, ktab, sh, n, d, lane, 32);
  if (!__all_sync(FULL, good)) return false;
  __syncwarp();

  // ---- the chain; a window with a non-finite result is left to gp_var_kernel, which rewrites every entry ----
  const bool fin = tvt_chain<true>(s_tab, s_al, s_a, s_t, n, sh, ms, mc, q0, 1.0 / gam, kss, noise, a.sigma_mode,
                                   mean_row, var_row, lane);
  return __all_sync(FULL, fin);
}

__global__ void __launch_bounds__(TVT_WARPS * 32, 3) gp_var_toeplitz_kernel(const VarArgs a, int* taken) {
  extern __shared__ __align__(16) double tvt_smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long lw = (long long)blockIdx.x * TVT_WARPS + w;   // window within this launch
  if (lw >= a.n_windows_launch) return;
  const long long win = a.window0 + lw;
  if (a.skip && a.skip[win]) {   // a member of a shared covariance: gp_toep_member_kernel has its results
    if (lane == 0) taken[lw] = 1;
    return;
  }
  const bool ok = tvt_window(a, lw, win, tvt_smem + (size_t)w * tvt_warp_doubles(a.nt, a.M), a.mean + win * (long long)a.M,
                             a.var + win * (long long)a.M, lane);
  if (lane == 0) taken[lw] = ok ? 1 : 0;
}

// The windows of a launch that gp_var_toeplitz_kernel did not take, in increasing order (ballot + block scan, a fixed
// order): list[0 .. *count).  One CTA of 1024 threads.
__global__ void __launch_bounds__(1024) var_compact_kernel(const int* taken, long long nw, int* list, int* count) {
  __shared__ int wsum[32];
  __shared__ int wpre[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int base = 0;
  for (long long b0 = 0; b0 < nw; b0 += 1024) {
    const long long i = b0 + threadIdx.x;
    const bool f = i < nw && !taken[i];
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
  if (threadIdx.x == 0) *count = base;
}

}  // namespace cngp
