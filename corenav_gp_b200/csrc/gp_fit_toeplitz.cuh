// Phase A for windows whose Ky is a symmetric positive-definite Toeplitz matrix (DESIGN.md section 4.1).
//
// With a stationary expression and stamps base + i d (d >= 1 an integer: every recorder window without a pause), Ky(i, j)
// depends on |i - j| only.  The generalised Schur algorithm then produces the Cholesky factor column by column from the
// first column t of Ky in ~2 N^2 flop instead of N^3 / 3: with the generators u = t / sqrt(t0), v = u (v_0 = 0),
//     for k = 0 .. n-1:   L(k:, k) = u(k:);  u <- u shifted down one row;
//                         rho = v_{k+1} / u_{k+1};  (u, v) <- ((u - rho v), (v - rho u)) / sqrt(1 - rho^2)   (rows > k)
// and u_{k+1} after the rotation is the next pivot, u_k sqrt(1 - rho^2).  z = L^-1 y rides along as a forward
// substitution on the column just produced.
//
// One warp per window, rows dealt cyclically over the lanes (row lane + 32 s in slot s), so a step is a few shuffles and
// FMA per live slot and its only serial dependence is the broadcast of v_{k+1}; TOEP_WARPS windows share a CTA and a SM
// runs many of them at once.  The output is exactly what gp_fit_kernel writes, in the same layouts (packed factor tiles
// with inv(L_jj) on the diagonal, TF32 hi/lo halves in FP32 mode, z, features, lag tables, LML / log det / quad, status 0),
// so phase B and the gradient do not know which kernel factored a window.  Half a tile column (four steps) is staged in
// shared memory and leaves as full 32-byte sectors; the 8x8 diagonal tile is inverted in-warp once its column is done.
//
// A window is taken only if it qualifies, decided here from its own data: lag tables on (stationary expression), the
// fit table valid, uniform integer stamps, every |rho| < 1, every value finite and min_k L_kk^2 >= TOEP_MIN_PIVOT2 t0.
// Any other window is left to gp_fit_kernel (done[p] = 0), which keeps the jitter ladder and the status codes.
#pragma once
#include "gp_fit.cuh"

namespace cngp {

constexpr int TOEP_WARPS = 4;                 // windows per CTA
constexpr int TOEP_SLOTS = CNGP_MAX_N / 32;   // row slots per lane
static_assert(CNGP_MAX_N % 32 == 0, "rows are dealt over the 32 lanes");
// Conditioning guard.  min_k L_kk^2 / t0 tracks 1 / cond(Ky): 0.11 to 0.14 for rbf, rbf+stdperiodic, mat32+bias and
// ratquad+stdperiodic*rbf at noise 1e-3 (the benchmark window: cond 750), 6.5e-3 for mat52+white at noise 1e-3
// (cond 1.6e4), 1e-3 for stdperiodic at noise 1e-3.  Just above the guard (ratio 1.5e-2; lengthscales x1 to x100,
// N = 100 and 256) the Schur fit, the variance recurrence and the shared-covariance group are within 1.4e-13 of a float80
// exact GP in mean, 1.4e-14 in variance and 1.9e-13 in LML (max(1, |ref|) relative; the tile Cholesky: 1.1e-13, 1.4e-15,
// 1.1e-12), and the gradients they feed are as close as the tile path's - measured on a B200 by
// tests/test_gpu_toeplitz_conditioning.py.  (The 1e-10 gaps between the Schur and the tile mean seen with a metric
// floored at 1e-3 max|mean| are both paths' rounding on a tail that decays to zero, not an error.)  Below the guard the
// windows take the tile Cholesky; the guard keeps the ill-conditioned ones (cond 1e6 and beyond) on the path whose
// jitter ladder and status codes handle them.
constexpr double TOEP_MIN_PIVOT2 = 1e-2;

// stage stride: one column of the staged half tile column, rows rounded up to the 32 lanes
__host__ __device__ __forceinline__ int toep_col_stride(int nt) { return (8 * nt + 31) & ~31; }
__host__ __device__ __forceinline__ size_t toep_smem_bytes(int nt) { return (size_t)TOEP_WARPS * 4 * toep_col_stride(nt) * sizeof(double); }

// Uniform stamps x_i = x_0 + i d with d >= 1, from the integer stamps xi[0 .. n) (this lane's share of the check; the
// caller takes the warp vote).  n < 2 passes with d = 1.
__device__ __forceinline__ bool toep_uniform(const int* xi, int n, int lane, int& d) {
  d = 1;
  if (n < 2) return true;
  d = xi[1] - xi[0];
  bool ok = d >= 1;
  for (int i = lane; i < n; i += 32) ok &= (xi[i] - xi[0] == i * d);
  return ok;
}
// z'z of the warp's rows (sequential over the slots, then the xor tree) and the LML: the Schur fit and the members of a
// shared covariance (gp_toep_group.cuh) compute them here, so both give the same bits
__device__ __forceinline__ double toep_quad(const double (&rr)[TOEP_SLOTS]) {
  double qs = 0.0;
#pragma unroll
  for (int s = 0; s < TOEP_SLOTS; ++s) qs += rr[s] * rr[s];
  for (int o = 16; o; o >>= 1) qs += __shfl_xor_sync(0xffffffffu, qs, o);
  return qs;
}
__device__ __forceinline__ double toep_lml(int N, double logdet, double qs) {
  return 0.5 * (-(double)N * CNGP_LOG_2PI - logdet - qs);
}

// KID only selects the per-point features written for phase B (the periodic phases for KID_RBF_PER); the factorisation
// itself reads the lag table, built by the interpreter for every expression.
template <int KID>
__global__ void __launch_bounds__(TOEP_WARPS * 32, 4) gp_fit_toeplitz_kernel(const FitArgs a, long long nprob) {
  extern __shared__ __align__(16) double toep_smem[];
  __shared__ KProg kps;
  __shared__ LeafConst hc_all[TOEP_WARPS][CNGP_MAX_LEAVES];
  __shared__ double dtile_all[TOEP_WARPS][64];   // L_jj of the current tile column, row-major
  __shared__ double ipiv_all[TOEP_WARPS][8];     // 1 / L_kk of the current tile column
  __shared__ double kdiag_all[TOEP_WARPS];

  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (threadIdx.x == 0) kps = a.kp;
  __syncthreads();
  const long long lp = (long long)blockIdx.x * TOEP_WARPS + w;   // problem within this launch
  if (lp >= nprob) return;
  const long long p = a.problem0 + lp;
  if (a.skip && a.skip[p]) {
    if (lane == 0) a.done[p] = 1;
    return;
  }
  const int win = a.win_map ? a.win_map[p] : (int)(p % a.n_windows);
  const long long ti = a.theta_mode == 0 ? 0 : (a.theta_mode == 1 ? (long long)win : (a.theta_mode == 3 ? p : p / a.n_windows));
  const double* th = a.theta + ti * a.theta_stride;
  const int ld = a.N, N = a.n_win ? a.n_win[win] : a.N, nt = a.nt, R = 8 * nt, CS = toep_col_stride(nt);
  const double noise = th[a.kp.n_params];
  LeafConst* hc = hc_all[w];
  double* stage = toep_smem + (size_t)w * 4 * CS;   // [4][CS]: columns 4h .. 4h+3 of the current tile column
  double* dtile = dtile_all[w];
  double* ipiv8 = ipiv_all[w];
  double* fx = stage;                               // prologue only: stamps, then integer stamps
  int* s_xi = reinterpret_cast<int*>(stage + CS);
  if (N < 1) {
    if (lane == 0) a.done[p] = 0;
    return;
  }

  // ---- prologue: features, lag tables (the same code as gp_fit_kernel's) ----
  FastK<KID> fk;
  if (KID != KID_GENERIC) {
    fk.init(th);
    fk.base = a.x[(long long)win * ld];
  }
  for (int i = lane; i < R; i += 32) {
    const double xv = i < N ? a.x[(long long)win * ld + i] : 0.0;
    PointFeat f{xv, __dmul_rn(xv, xv), 0.0, 0.0};
    if (KID != KID_GENERIC) f = fk.point(xv);
    fx[i] = f.x;
    if (a.feat) {
      double* fp = a.feat + lp * (long long)(4 * R);
      fp[i] = f.x; fp[R + i] = f.xx; fp[2 * R + i] = f.c; fp[3 * R + i] = f.s;
    }
  }
  if (lane < a.kp.n_leaves) hc[lane] = leaf_prepare(a.kp.leaf_type[lane], th + a.kp.leaf_param[lane]);
  __syncwarp();
  const LagTab lt = fit_lag_tables<32>(a, lp, win, N, nt, lane, fx, &kps, hc, noise, nullptr, s_xi, &kdiag_all[w],
                                       nullptr, nullptr);
  __syncwarp();

  // ---- uniform stamps: x_i = x_0 + i d ----
  int d = 1;
  const bool ok = lt.fit_tab && toep_uniform(s_xi, N, lane, d);
  if (!__all_sync(0xffffffffu, ok)) {
    if (lane == 0) a.done[p] = 0;
    return;
  }
  __syncwarp();   // the stage takes over the prologue's room

  // ---- generators from the first column of Ky (same values as the tile path's lag table) ----
  const double t0 = kdiag_all[w] + (noise + CNGP_JITTER);
  double piv = sqrt(t0), ipiv = 1.0 / piv, minp2 = t0;
  double u[TOEP_SLOTS], v[TOEP_SLOTS], rr[TOEP_SLOTS], pv[TOEP_SLOTS];
#pragma unroll
  for (int s = 0; s < TOEP_SLOTS; ++s) {
    const int i = lane + 32 * s;
    double ui = 0.0;
    if (i == 0) ui = piv;
    else if (i < N) ui = keval_generic_cross(&kps, hc, (double)(i * d), 0.0) * ipiv;
    u[s] = ui;
    v[s] = i == 0 ? 0.0 : ui;
    rr[s] = (i < N && a.y) ? a.y[(long long)win * ld + i] : 0.0;   // residual y - L z (y = 0 without y), row k becomes z_k at step k
    pv[s] = 1.0;                                          // pivots (1 on the padding rows)
  }
  bool good = true;
  double* Lp = a.L + lp * (long long)tiles_in_lower(nt) * 64;
  const bool f32 = a.f32_factor != 0;

  // one Schur step; SB = slot of row k (slots below it are dead: rows < k are zero in u and v)
  auto step = [&](auto sbc, int k) {
    constexpr int SB = decltype(sbc)::value;
    const int kk = k & 31;
    if (k >= N) {   // identity padding: L(:, k) = e_k, z_k = 0
#pragma unroll
      for (int t = SB; t < TOEP_SLOTS; ++t) u[t] = (32 * t + lane == k) ? 1.0 : 0.0;
      piv = 1.0; ipiv = 1.0;
    }
    // column k of L -> stage
#pragma unroll
    for (int t = SB; t < TOEP_SLOTS; ++t)
      if (32 * t < R) stage[(k & 3) * CS + 32 * t + lane] = u[t];
    if (lane == 0) ipiv8[k & 7] = ipiv;
    // z_k = r_k / L_kk, r -= L(:, k) z_k
    const double zk = __shfl_sync(0xffffffffu, rr[SB], kk) * ipiv;
#pragma unroll
    for (int t = SB; t < TOEP_SLOTS; ++t) rr[t] = fma(-u[t], zk, rr[t]);
    if (lane == kk) { rr[SB] = zk; pv[SB] = piv; }
    if (k + 1 < N) {
      // shift u down one row (lane 0 takes lane 31's row of the slot before).  Row N - 1 falls off the end: the rows
      // at and beyond N are identity padding and must stay zero in every column k < N.
      double prev = 0.0;
#pragma unroll
      for (int t = SB; t < TOEP_SLOTS; ++t) {
        if (32 * t < R) {
          const double sh = __shfl_sync(0xffffffffu, u[t], (lane + 31) & 31);
          u[t] = (32 * t + lane >= N) ? 0.0 : (lane == 0 ? prev : sh);
          prev = sh;
        }
      }
      constexpr int SN = SB + 1 < TOEP_SLOTS ? SB + 1 : SB;
      const double vb = __shfl_sync(0xffffffffu, kk == 31 ? v[SN] : v[SB], (kk + 1) & 31);
      const double rho = vb * ipiv;                  // u_{k+1} after the shift is L_kk
      good &= fabs(rho) < 1.0;
      const double s2 = (1.0 - rho) * (1.0 + rho);
      const double is = rsqrt(s2);
#pragma unroll
      for (int t = SB; t < TOEP_SLOTS; ++t) {
        const double un = fma(-rho, v[t], u[t]) * is;
        v[t] = fma(-rho, u[t], v[t]) * is;
        u[t] = un;
      }
      piv *= s2 * is;
      ipiv *= is;
      minp2 = fmin(minp2, piv * piv);
      if (kk == 31) {
        if (lane == 0) { u[SN] = piv; v[SN] = 0.0; }
      } else if (lane == kk + 1) {
        u[SB] = piv; v[SB] = 0.0;
      }
    }
    if ((k & 3) == 3) {
      // half tile column h of tile column J is complete: rows below the diagonal tile leave, the diagonal tile's part
      // goes to dtile
      __syncwarp();
      const int J = k >> 3, h = (k >> 2) & 1;
      dtile[(lane >> 2) * 8 + 4 * h + (lane & 3)] = stage[(lane & 3) * CS + 8 * J + (lane >> 2)];
      double* colJ = Lp + (long long)tile_index(J, J, nt) * 64 + 4 * h;   // row i of tile column J at colJ + (i - 8J) 8
      const int npairs = 2 * (R - 8 * J - 8);
      for (int e = lane; e < npairs; e += 32) {
        const int i = 8 * J + 8 + (e >> 1), c = 2 * (e & 1);
        const double x0 = stage[c * CS + i], x1 = stage[(c + 1) * CS + i];
        double* dst = colJ + (i - 8 * J) * 8 + c;
        if (f32) pair_store_split(dst, x0, x1);
        else *reinterpret_cast<double2*>(dst) = make_double2(x0, x1);
      }
      __syncwarp();
      if (h == 1) {
        // inv(L_JJ) by forward substitution on the identity (as in chol8_inv8), in the lane layout
        const int r = lane >> 2, q = lane & 3;
        tile2 x{r == 2 * q ? 1.0 : 0.0, r == 2 * q + 1 ? 1.0 : 0.0};
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const double xka = __shfl_sync(0xffffffffu, x.a, 4 * m + q), xkb = __shfl_sync(0xffffffffu, x.b, 4 * m + q);
          const double xsa = xka * ipiv8[m], xsb = xkb * ipiv8[m];
          const double lrm = dtile[8 * r + m];
          if (r == m) { x.a = xsa; x.b = xsb; }
          if (r > m) { x.a = fma(-lrm, xsa, x.a); x.b = fma(-lrm, xsb, x.b); }
        }
        double* dst = Lp + (long long)tile_index(J, J, nt) * 64;
        if (f32) tile_store_split(dst, lane, x);
        else tile_store(dst, lane, x);
        if (a.ldiag) {
          a.ldiag[J * 64 + lane] = dtile[lane];
          a.ldiag[J * 64 + 32 + lane] = dtile[32 + lane];
        }
        __syncwarp();
      }
    }
  };
  // slot-block loop: SB is a compile-time index so that every register array stays in registers
  auto block = [&](auto sbc) {
    constexpr int SB = decltype(sbc)::value;
    const int k1 = min(32 * SB + 32, R);
    for (int k = 32 * SB; k < k1; ++k) step(sbc, k);
  };
  static_assert(TOEP_SLOTS == 8, "unrolled slot blocks below");
  block(FitIC<0>{});
  if (R > 32) block(FitIC<1>{});
  if (R > 64) block(FitIC<2>{});
  if (R > 96) block(FitIC<3>{});
  if (R > 128) block(FitIC<4>{});
  if (R > 160) block(FitIC<5>{});
  if (R > 192) block(FitIC<6>{});
  if (R > 224) block(FitIC<7>{});

  // ---- accept or hand the window to gp_fit_kernel ----
  double hl = 0.0;
  bool fin = isfinite(piv) && isfinite(ipiv);
#pragma unroll
  for (int s = 0; s < TOEP_SLOTS; ++s) {
    fin &= isfinite(rr[s]) && isfinite(pv[s]);
    hl += log(pv[s]);   // padded rows have pivot 1
  }
  good = good && fin && minp2 >= TOEP_MIN_PIVOT2 * t0;
  if (!__all_sync(0xffffffffu, good)) {
    if (lane == 0) a.done[p] = 0;
    return;
  }
  double* zp = a.z + lp * (long long)R;
#pragma unroll
  for (int s = 0; s < TOEP_SLOTS; ++s)
    if (lane + 32 * s < R) zp[lane + 32 * s] = rr[s];
  const double qs = toep_quad(rr);
  for (int o = 16; o; o >>= 1) hl += __shfl_xor_sync(0xffffffffu, hl, o);
  if (lane == 0) {
    const double logdet = 2.0 * hl;
    if (a.quad) a.quad[p] = qs;
    if (a.logdet) a.logdet[p] = logdet;
    if (a.lml) a.lml[p] = toep_lml(N, logdet, qs);
    if (a.status) a.status[p] = 0;
    if (a.kmeta && !lt.var_tab && a.n_lazy) atomicAdd(a.n_lazy, 1);
    a.done[p] = 1;
  }
}

}  // namespace cngp
