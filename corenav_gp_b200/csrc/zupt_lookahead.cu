// Batched stop predictor: unscented transform of predicted slip -> odometry noise R_IP, 15-state covariance
// look-ahead with a Joseph-form update every `ratio`-th step, and the 3-sigma horizontal error observer.
//
// Replaces the loop body of GpPredictor::GPCallBack, /root/reference/gp_predictor/src/gp_predictor.cpp:64-124
// (rows a10-a12 of SURVEY.md section 8) and GpPredictor::llh_to_enu (:144-178), for B independent windows.
// Reference quirks kept (SURVEY.md App. B): H(r,c) = Hvec[r*4+c]; sigma is used as the sigma-point offset and the UT
// covariance is squared again; update happens before the error check; only the +3 sigma point triggers.
//
// One warp per window; P and the temporaries live in shared memory, each lane owns up to 8 of the 225 outputs of a
// 15x15 product and evaluates its dot products as ascending-index fma chains starting from 0 - the same operation
// order as the C oracle, so (triggered, i) is reproducible bit for bit.  This translation unit is compiled with
// -fmad=false: every fused operation below is an explicit fma().
#include <cuda_runtime.h>
#include <stdlib.h>
#include "../../include/cngp.h"

namespace cngp {

constexpr int LA_WARPS = 4;

struct LookaheadArgs {
  const double* mean;   // [B][M]
  const double* sigma;  // [B][M]
  long long B;
  int M;
  const double* P; const double* Q; const double* STM; const double* Hvec; const double* pos;
  int per_window;
  cngp_stop_config cfg;
  int* triggered; int* i_stop; int* step_stop; double* xy_err;
  unsigned long long* next_window;   // tensor-core kernel: work counter (windows are claimed one at a time), or null
  // optional final state per window (the reference leaves it in public members, gp_predictor.h:36-43): P_pred after the
  // last step executed, K_pred and R_IP of the last update - row-major [225], [60] (15 x 4), [16]
  double* P_final; double* K_final; double* R_final;
  // EKF covariance recursion (cngp_ekf_covariance_batch): a fixed odometry noise R [16] or [B][16] replaces the UT of the
  // predicted slip (CoreNav.cpp:228 uses the filter's constant R_), tensor-core kernel only
  const double* R_fixed; int R_per_window;
  long long ms_stride;   // row stride of mean / sigma: M, or 0 when every window shares one row
  const int* m_win;      // ragged batches: GP_Output points of each window (<= M; the loop runs ratio * m_win[b] steps), or null
};

struct LlhConst {
  double e2, one_m_e2;          // e*e, 1 - e*e with e = sqrt(1 - (b/a)^2)
  double Rm[3][3];              // ECEF -> ENU rotation at init_llh
};

// Deterministic sin / cos: Cody-Waite reduction by pi/2 in three fma steps, then the classic degree-13 / 14 minimax
// polynomials on [-pi/4, pi/4] as fma Horner chains.  Only IEEE-exact operations in a fixed order (this TU is built with
// -fmad=false), so the C oracle (its trig_mode = 1, built with -ffp-contract=off) returns the same bits
// and the stop decision is reproducible at a 0-ulp margin; within 1 ulp of libm / libdevice.  tan = sin / cos.
__device__ __forceinline__ void det_sincos(double x, double& sn, double& cs) {
  const double k = rint(x * 6.36619772367581382433e-01);
  double r = fma(-k, 1.57079632679489655800e+00, x);
  r = fma(-k, 6.12323399573676603587e-17, r);
  r = fma(-k, -1.49738490485916983000e-33, r);
  const double z = r * r;
  double ps = 1.58969099521155010221e-10;
  ps = fma(ps, z, -2.50507602534068634195e-08);
  ps = fma(ps, z, 2.75573137070700676789e-06);
  ps = fma(ps, z, -1.98412698298579493134e-04);
  ps = fma(ps, z, 8.33333333332248946124e-03);
  ps = fma(ps, z, -1.66666666666666324348e-01);
  const double s = fma(r * z, ps, r);
  double pc = -1.13596475577881948265e-11;
  pc = fma(pc, z, 2.08757232129817482790e-09);
  pc = fma(pc, z, -2.75573143513906633035e-07);
  pc = fma(pc, z, 2.48015872894767294178e-05);
  pc = fma(pc, z, -1.38888888888741095749e-03);
  pc = fma(pc, z, 4.16666666666666019037e-02);
  const double hz = 0.5 * z;
  const double w = 1.0 - hz;
  const double c = w + (((1.0 - w) - hz) + (z * z) * pc);
  const long long q = (long long)k & 3;
  sn = (q == 0) ? s : (q == 1) ? c : (q == 2) ? -s : -c;
  cs = (q == 0) ? c : (q == 1) ? -s : (q == 2) ? -c : s;
}

__device__ __forceinline__ LlhConst llh_prepare(const cngp_stop_config& c) {
  LlhConst k;
  const double a = 6378137.0000, b = 6356752.3142;
  const double boa = b / a;
  const double e = sqrt(1 - boa * boa);
  k.e2 = e * e;
  k.one_m_e2 = 1 - e * e;
  double sinPhi, cosPhi, sinLam, cosLam;
  det_sincos(c.init_llh[0], sinPhi, cosPhi);
  det_sincos(c.init_llh[1], sinLam, cosLam);
  k.Rm[0][0] = -1 * sinLam; k.Rm[0][1] = cosLam; k.Rm[0][2] = 0;
  k.Rm[1][0] = (-1 * sinPhi) * cosLam; k.Rm[1][1] = (-1 * sinPhi) * sinLam; k.Rm[1][2] = cosPhi;
  k.Rm[2][0] = cosPhi * cosLam; k.Rm[2][1] = cosPhi * sinLam; k.Rm[2][2] = sinPhi;
  return k;
}

// gp_predictor.cpp:144-178 given the five trigonometric values of (lat, lon)
__device__ __forceinline__ void llh_to_enu_trig(double sinphi, double cosphi, double tanphi, double sinlam, double coslam,
                                                double h, const LlhConst& k, const cngp_stop_config& c, double enu[3]) {
  const double a = 6378137.0000;
  const double tan2phi = tanphi * tanphi;
  const double tmpden = sqrt(1 + k.one_m_e2 * tan2phi);
  const double x1 = (a * coslam) / tmpden + h * coslam * cosphi;
  const double y1 = (a * sinlam) / tmpden + h * sinlam * cosphi;
  const double tmp3 = sqrt(1 - k.e2 * sinphi * sinphi);
  const double z1 = (a * k.one_m_e2 * sinphi) / tmp3 + h * sinphi;
  const double d0 = x1 - c.init_ecef[0], d1 = y1 - c.init_ecef[1], d2 = z1 - c.init_ecef[2];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    double acc = 0.0;
    acc = fma(k.Rm[r][0], d0, acc);
    acc = fma(k.Rm[r][1], d1, acc);
    acc = fma(k.Rm[r][2], d2, acc);
    enu[r] = acc;
  }
}

__device__ __forceinline__ void llh_to_enu_dev(double lat, double lon, double h, const LlhConst& k,
                                               const cngp_stop_config& c, double enu[3]) {
  double sp, cp, sl, cl;
  det_sincos(lat, sp, cp);
  det_sincos(lon, sl, cl);
  llh_to_enu_trig(sp, cp, sp / cp, sl, cl, h, k, c, enu);
}

// closed-form 4x4 inverse through 2x2 minors (Eigen's fixed-size inverse at gp_predictor.cpp:90 is the same math)
__device__ __forceinline__ void inv4(const double* m /*[16] row-major*/, double* o) {
#define M_(r, c) m[(r) * 4 + (c)]
  const double s0 = M_(0, 0) * M_(1, 1) - M_(1, 0) * M_(0, 1);
  const double s1 = M_(0, 0) * M_(1, 2) - M_(1, 0) * M_(0, 2);
  const double s2 = M_(0, 0) * M_(1, 3) - M_(1, 0) * M_(0, 3);
  const double s3 = M_(0, 1) * M_(1, 2) - M_(1, 1) * M_(0, 2);
  const double s4 = M_(0, 1) * M_(1, 3) - M_(1, 1) * M_(0, 3);
  const double s5 = M_(0, 2) * M_(1, 3) - M_(1, 2) * M_(0, 3);
  const double c5 = M_(2, 2) * M_(3, 3) - M_(3, 2) * M_(2, 3);
  const double c4 = M_(2, 1) * M_(3, 3) - M_(3, 1) * M_(2, 3);
  const double c3 = M_(2, 1) * M_(3, 2) - M_(3, 1) * M_(2, 2);
  const double c2 = M_(2, 0) * M_(3, 3) - M_(3, 0) * M_(2, 3);
  const double c1 = M_(2, 0) * M_(3, 2) - M_(3, 0) * M_(2, 2);
  const double c0 = M_(2, 0) * M_(3, 1) - M_(3, 0) * M_(2, 1);
  const double det = s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0;
  const double id = 1.0 / det;
  o[0] = (M_(1, 1) * c5 - M_(1, 2) * c4 + M_(1, 3) * c3) * id;
  o[1] = (-M_(0, 1) * c5 + M_(0, 2) * c4 - M_(0, 3) * c3) * id;
  o[2] = (M_(3, 1) * s5 - M_(3, 2) * s4 + M_(3, 3) * s3) * id;
  o[3] = (-M_(2, 1) * s5 + M_(2, 2) * s4 - M_(2, 3) * s3) * id;
  o[4] = (-M_(1, 0) * c5 + M_(1, 2) * c2 - M_(1, 3) * c1) * id;
  o[5] = (M_(0, 0) * c5 - M_(0, 2) * c2 + M_(0, 3) * c1) * id;
  o[6] = (-M_(3, 0) * s5 + M_(3, 2) * s2 - M_(3, 3) * s1) * id;
  o[7] = (M_(2, 0) * s5 - M_(2, 2) * s2 + M_(2, 3) * s1) * id;
  o[8] = (M_(1, 0) * c4 - M_(1, 1) * c2 + M_(1, 3) * c0) * id;
  o[9] = (-M_(0, 0) * c4 + M_(0, 1) * c2 - M_(0, 3) * c0) * id;
  o[10] = (M_(3, 0) * s4 - M_(3, 1) * s2 + M_(3, 3) * s0) * id;
  o[11] = (-M_(2, 0) * s4 + M_(2, 1) * s2 - M_(2, 3) * s0) * id;
  o[12] = (-M_(1, 0) * c3 + M_(1, 1) * c1 - M_(1, 2) * c0) * id;
  o[13] = (M_(0, 0) * c3 - M_(0, 1) * c1 + M_(0, 2) * c0) * id;
  o[14] = (-M_(3, 0) * s3 + M_(3, 1) * s1 - M_(3, 2) * s0) * id;
  o[15] = (M_(2, 0) * s3 - M_(2, 1) * s1 + M_(2, 2) * s0) * id;
#undef M_
}

// gp_predictor.cpp:69-88
__device__ __forceinline__ void ut_R(double mean, double sigma, const cngp_stop_config& c, double* R /*[16]*/) {
  const double chi0 = c.v_nom / (1.0 - mean);
  const double chi1 = c.v_nom / (1.0 - (mean + sigma));
  const double chi2 = c.v_nom / (1.0 - (mean - sigma));
  const double est = (chi0 + chi1 + chi2) / 3.0;
  const double cov = ((chi0 - est) * (chi0 - est) + (chi1 - est) * (chi1 - est) + (chi2 - est) * (chi2 - est)) / 3.0;
  const double c2 = cov * cov;
  const double fa = c.floor_a * c.floor_a, fb = c.floor_b * c.floor_b;
  const double R2[4] = {fmax(fa, c2), fmax(fa, c2), fmax(fb, c2), fb};
  const double it = 1 / c.track;
  const double R1[4][4] = {{0.5, 0.5, 0.0, 0.0}, {it, -it, 0.0, 0.0}, {0.0, 0.0, 1.0, 0.0}, {0.0, 0.0, 0.0, 1.0}};
  double Bm[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int k = 0; k < 4; ++k) Bm[a][k] = (c.scale * R1[a][k]) * R2[k];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      double acc = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) acc = fma(Bm[a][k], R1[b][k], acc);
      R[a * 4 + b] = acc;
    }
}

// Cheap rigorous upper bound of the horizontal ENU displacement between (lat, lon, h) and (lat + dl, lon + dm, h + dh):
// walk the three coordinates one at a time.  The meridian and parallel chords are at most Rb dl and Rb cmax dm long
// (Rb >= any radius of curvature + height, cmax >= |cos| along the way) and perpendicular up to dm / 2, the height step
// only shows in the horizontal plane of init_llh through the tilt (<= tilt0 + dl + dm) between the two verticals.
// While the bound stays below the threshold the exact observer (five trigonometric calls) cannot trigger and is skipped.
struct ObsBound {
  double habs, coslat0, tilt0;
  bool usable;
  double c1, c2, c3, t2;   // square-root-free form of the same bound (obs_cannot_trigger_sq)
};
__device__ __forceinline__ ObsBound obs_prepare(double lat, double lon, double h, const cngp_stop_config& c) {
  ObsBound o;
  o.habs = fabs(h);
  o.coslat0 = fabs(cos(lat));
  o.tilt0 = fabs(lat - c.init_llh[0]) + fabs(lon - c.init_llh[1]);
  o.usable = fabs(lat) < 1.4;       // the closed form of gp_predictor.cpp:150-160 is the ellipsoid map away from the poles
  // The same bound without square roots, from u = |P66|, v = |P77|, hh = |P88| (dl = 3 sqrt u ...), valid while
  // dl, dm < 1e-3 rad and dh < 1e3 m:  bound <= 1.0011 sqrt(X) + y,  X = Rb1^2 9 (u + (coslat0 + 1e-3)^2 v),
  // y = dh tilt1, and (s + y)^2 <= (1 + 1e-3) s^2 + 1001 y^2.  It is ~0.2 % more conservative than the form above (a few
  // more exact evaluations close to the threshold) and takes three square roots off every step of the look-ahead.
  const double Rb1 = 6.4e6 + o.habs + 1.0e3, tilt1 = fmin(1.0, o.tilt0 + 2.0e-3);
  o.c1 = 1.001 * 1.0011 * 1.0011 * 9.0 * Rb1 * Rb1;
  o.c2 = (o.coslat0 + 1.0e-3) * (o.coslat0 + 1.0e-3);
  o.c3 = 1001.0 * 9.0 * tilt1 * tilt1;
  o.t2 = c.thresh > 1.0e-3 ? (c.thresh - 1.0e-6) * (c.thresh - 1.0e-6) : -1.0;
  return o;
}
__device__ __forceinline__ bool obs_cannot_trigger_sq(const ObsBound& o, double u, double v, double hh) {
  return o.usable && (9.0 * u < 1.0e-6) && (9.0 * v < 1.0e-6) && (9.0 * hh < 1.0e6) &&
         (o.c1 * (u + o.c2 * v) + o.c3 * hh < o.t2);                                   // NaN compares false: exact path
}
__device__ __forceinline__ bool obs_cannot_trigger(const ObsBound& o, double dl, double dm, double dh, double thresh) {
  const double Rb = 6.4e6 + o.habs + dh;
  const double A = Rb * dl, Bq = Rb * (o.coslat0 + dl) * dm;
  const double tilt = fmin(1.0, o.tilt0 + dl + dm);
  const double bound = sqrt(A * A + Bq * Bq) * (1.0 + dm) + dh * tilt;
  return o.usable && dl < 0.1 && (bound * (1.0 + 1e-9) + 1e-6 < thresh);     // NaN compares false: exact path
}


// ---------------------------------------------------------------------------------------------------------------------
// Tensor-core look-ahead.  One FP64 tensor-core instruction  mma.sync.m8n8k4.f64  returns, bit for bit, the ascending-k
// chain of fma  d = fma(a3,b3, fma(a2,b2, fma(a1,b1, fma(a0,b0,c))))  (tools/dmma_semantics.cu: 1 280 000 of 1 280 000
// outputs identical on B200; descending / pairwise / mul+add orders do not match).  An ascending-index fma chain starting
// from 0 is exactly how the C oracle forms every dot product of the look-ahead, so the 15 x 15 algebra can run on the
// FP64 tensor pipe - matrices zero-padded to 16 x 16 = 2 x 2 tiles, a 15-term chain = four k4 instructions whose 16th
// term is fma(0, 0, acc) = acc - and still reproduce (triggered, i, step, xy_err) bit for bit.
//
// One warp per window.  Matrices live in shared memory row-major with a leading dimension of 20 doubles (12 for the
// 16 x 4 ones): with that stride the A-fragment loads M[8 ri + g][4 ks + t], the B-fragment loads M[4 ks + t][8 ci + g]
// and the 16-byte D-fragment stores M[8 ri + g][8 ci + 2t .. +1] all hit every bank pair exactly twice per warp - the
// minimum for 8-byte accesses.  The fragments of the constant operands (STM as A and, transposed, as B; Q as accumulator
// fragments; H) stay in registers for the whole window.  A propagation step is 32 instructions (F P, then (F P) F' + Q),
// an update 64 (P H', H P, S, K, I - K H, K R, (I-KH) P, (..)(I-KH)' + (K R) K'), against ~6000 scalar fma with two
// shared-memory loads each in the scalar kernels below.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int TC_LD = 20, TC_LD4 = 12;
// Working set per warp (doubles).  Buffers with disjoint lifetimes share storage: I - K H lives where H P and P H' were
// (both dead once K is formed), K R in the head of T (dead between the propagation and the Joseph products; it is pulled
// into registers before T is written again).  11 KB per warp: two CTAs of eight warps per SM.
constexpr int TC_P = 0, TC_T = 320, TC_KR = 320, TC_HP = 640, TC_PHT = 800, TC_A = 640, TC_K = 992, TC_H = 1184,
              TC_S = 1344, TC_R = 1360, TC_WS = 1376;
constexpr int TC_WARPS = 8;

__device__ __forceinline__ void dmma(double2& d, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d.x), "+d"(d.y) : "d"(a), "d"(b));
}
__device__ __forceinline__ double pick16(const double* v, int idx) {   // v is a register array: unrolled selects
  double r = v[0];
#pragma unroll
  for (int e = 1; e < 16; ++e) r = (idx == e) ? v[e] : r;
  return r;
}

__global__ void __launch_bounds__(TC_WARPS * 32, 2) zupt_lookahead_tc_kernel(const LookaheadArgs a) {
  extern __shared__ __align__(16) double smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  double* ws = smem + (long long)w * TC_WS;
  // Windows run anywhere between 1 and ratio * M steps (early exit at the trigger), so they are not dealt statically:
  // every warp claims the next unclaimed window from a global counter until none is left.  (Without a counter - small
  // batches, one warp per CTA - warp k of the grid takes window k.)
  for (long long b = (long long)blockIdx.x * (blockDim.x >> 5) + w;; ) {
  if (a.next_window) {
    unsigned long long nb = 0;
    if (lane == 0) nb = atomicAdd(a.next_window, 1ULL);
    b = (long long)__shfl_sync(0xffffffffu, nb, 0);
  }
  if (b >= a.B) return;
  __syncwarp();
  double *Ps = ws + TC_P, *Ts = ws + TC_T, *As = ws + TC_A, *Hs = ws + TC_H, *HPs = ws + TC_HP, *PHts = ws + TC_PHT,
         *Ks = ws + TC_K, *KRs = ws + TC_KR, *Ss = ws + TC_S, *Rs = ws + TC_R;
  const cngp_stop_config& cfg = a.cfg;
  const int pw = a.per_window;
  const double* gP = a.P + ((pw & CNGP_PERWIN_P) ? b * 225 : 0);
  const double* gQ = a.Q + ((pw & CNGP_PERWIN_Q) ? b * 225 : 0);
  const double* gF = a.STM + ((pw & CNGP_PERWIN_STM) ? b * 225 : 0);
  const double* gH = a.Hvec + ((pw & CNGP_PERWIN_H) ? b * 60 : 0);
  const double* gpos = a.pos + ((pw & CNGP_PERWIN_POS) ? b * 3 : 0);

  for (int i = lane; i < TC_WS; i += 32) ws[i] = 0.0;           // zero padding everywhere
  __syncwarp();
  for (int i = lane; i < 225; i += 32) {
    const int rr = i / 15, cc = i % 15;
    Ps[rr * TC_LD + cc] = gP[i];
    Ts[rr * TC_LD + cc] = gF[i];                                // the STM passes through T's storage on its way to registers
  }
  for (int i = lane; i < 60; i += 32) {
    const int rr = i / 15, cc = i % 15;
    Hs[rr * TC_LD + cc] = gH[cfg.fix_h_packing ? rr * 15 + cc : rr * 4 + cc];   // gp_predictor.cpp:38-42 aliasing index
  }
  __syncwarp();
  // constant fragments.  Ff[ri][ks] = F[8ri+g][4ks+t]: A fragment of F, and B fragment of F' for column tile ri.
  double Ff[2][4], Hf[4], Hb[2];
  double2 Qd[2][2];
#pragma unroll
  for (int ri = 0; ri < 2; ++ri)
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) Ff[ri][ks] = Ts[(8 * ri + g) * TC_LD + 4 * ks + t];
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) Hf[ks] = Hs[g * TC_LD + 4 * ks + t];       // A fragment of H (rows 4..7 are padding)
#pragma unroll
  for (int ci = 0; ci < 2; ++ci) Hb[ci] = Hs[t * TC_LD + 8 * ci + g];       // B fragment of H as the 4 x 16 right factor
#pragma unroll
  for (int ri = 0; ri < 2; ++ri)
#pragma unroll
    for (int ci = 0; ci < 2; ++ci) {
      const int rr = 8 * ri + g, c0 = 8 * ci + 2 * t;
      Qd[ri][ci].x = (rr < 15 && c0 < 15) ? gQ[rr * 15 + c0] : 0.0;
      Qd[ri][ci].y = (rr < 15 && c0 + 1 < 15) ? gQ[rr * 15 + c0 + 1] : 0.0;
    }
  const double lat = gpos[0], lon = gpos[1], hgt = gpos[2];
  const LlhConst lk = llh_prepare(cfg);
  double enu0[3];
  llh_to_enu_dev(lat, lon, hgt, lk, cfg, enu0);
  const ObsBound ob = obs_prepare(lat, lon, hgt, cfg);
  __syncwarp();

  const double* mean = a.mean + b * a.ms_stride;
  const double* sigma = a.sigma + b * a.ms_stride;
  const int nsteps = cfg.ratio * (a.m_win ? a.m_win[b] : a.M);
  int i_upd = 0, trig = 0, step = nsteps;
  double xy = 0.0;
  // R1 of gp_predictor.cpp:84-87 seen from this lane: row g (as the left factor), rows 2t, 2t+1 (as the right factor)
  const double it = 1 / cfg.track;
  auto r1 = [&](int row, int k) -> double {
    return row == 0 ? (k < 2 ? 0.5 : 0.0) : row == 1 ? (k == 0 ? it : k == 1 ? -it : 0.0) : (row == k && row < 4 ? 1.0 : 0.0);
  };

  for (int slip_i = 0; slip_i < nsteps; ++slip_i) {
    // ---- P = F P F' + Q ----
    {
      double2 Td[2][2];
#pragma unroll
      for (int ri = 0; ri < 2; ++ri)
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) Td[ri][ci] = make_double2(0.0, 0.0);
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const double b0 = Ps[(4 * ks + t) * TC_LD + g], b1 = Ps[(4 * ks + t) * TC_LD + 8 + g];
        dmma(Td[0][0], Ff[0][ks], b0); dmma(Td[0][1], Ff[0][ks], b1);
        dmma(Td[1][0], Ff[1][ks], b0); dmma(Td[1][1], Ff[1][ks], b1);
      }
#pragma unroll
      for (int ri = 0; ri < 2; ++ri)
#pragma unroll
        for (int ci = 0; ci < 2; ++ci)
          *reinterpret_cast<double2*>(Ts + (8 * ri + g) * TC_LD + 8 * ci + 2 * t) = Td[ri][ci];
      __syncwarp();
      double2 Pd[2][2];
#pragma unroll
      for (int ri = 0; ri < 2; ++ri)
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) Pd[ri][ci] = make_double2(0.0, 0.0);
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const double a0 = Ts[g * TC_LD + 4 * ks + t], a1 = Ts[(8 + g) * TC_LD + 4 * ks + t];
        dmma(Pd[0][0], a0, Ff[0][ks]); dmma(Pd[0][1], a0, Ff[1][ks]);
        dmma(Pd[1][0], a1, Ff[0][ks]); dmma(Pd[1][1], a1, Ff[1][ks]);
      }
#pragma unroll
      for (int ri = 0; ri < 2; ++ri)
#pragma unroll
        for (int ci = 0; ci < 2; ++ci)
          *reinterpret_cast<double2*>(Ps + (8 * ri + g) * TC_LD + 8 * ci + 2 * t) =
              make_double2(Pd[ri][ci].x + Qd[ri][ci].x, Pd[ri][ci].y + Qd[ri][ci].y);
      __syncwarp();
    }
    if (slip_i % cfg.ratio == 0) {
      // ---- UT -> R_IP (this lane's two entries R[g][2t], R[g][2t+1]; only g < 4, t < 2 are real) ----
      {
        const double mu = mean[i_upd], sg = sigma[i_upd];
        const double chi0 = cfg.v_nom / (1.0 - mu);
        const double chi1 = cfg.v_nom / (1.0 - (mu + sg));
        const double chi2 = cfg.v_nom / (1.0 - (mu - sg));
        const double est = (chi0 + chi1 + chi2) / 3.0;
        const double cov = ((chi0 - est) * (chi0 - est) + (chi1 - est) * (chi1 - est) + (chi2 - est) * (chi2 - est)) / 3.0;
        const double c2 = cov * cov;
        const double fa = cfg.floor_a * cfg.floor_a, fb = cfg.floor_b * cfg.floor_b;
        const double R2[4] = {fmax(fa, c2), fmax(fa, c2), fmax(fb, c2), fb};
        double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const double bm = (cfg.scale * r1(g, k)) * R2[k];
          acc0 = fma(bm, r1(2 * t, k), acc0);
          acc1 = fma(bm, r1(2 * t + 1, k), acc1);
        }
        if (a.R_fixed && g < 4 && t < 2) {
          const double* rf = a.R_fixed + (a.R_per_window ? b * 16 : 0);
          acc0 = rf[g * 4 + 2 * t]; acc1 = rf[g * 4 + 2 * t + 1];
        }
        if (g < 4 && t < 2) { Rs[g * 4 + 2 * t] = acc0; Rs[g * 4 + 2 * t + 1] = acc1; }
      }
      // ---- P H' (16 x 8) and H P (8 x 16) ----
      {
        double2 D0 = make_double2(0.0, 0.0), D1 = D0, E0 = D0, E1 = D0;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const double a0 = Ps[g * TC_LD + 4 * ks + t], a1 = Ps[(8 + g) * TC_LD + 4 * ks + t];
          dmma(D0, a0, Hf[ks]); dmma(D1, a1, Hf[ks]);                       // P H': B fragment of H' = A fragment of H
          const double b0 = Ps[(4 * ks + t) * TC_LD + g], b1 = Ps[(4 * ks + t) * TC_LD + 8 + g];
          dmma(E0, Hf[ks], b0); dmma(E1, Hf[ks], b1);                       // H P
        }
        *reinterpret_cast<double2*>(PHts + g * TC_LD4 + 2 * t) = D0;
        *reinterpret_cast<double2*>(PHts + (8 + g) * TC_LD4 + 2 * t) = D1;
        *reinterpret_cast<double2*>(HPs + g * TC_LD + 2 * t) = E0;
        *reinterpret_cast<double2*>(HPs + g * TC_LD + 8 + 2 * t) = E1;
      }
      __syncwarp();
      // ---- S = (H P) H' + R ----
      {
        double2 Sd = make_double2(0.0, 0.0);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) dmma(Sd, HPs[g * TC_LD + 4 * ks + t], Hf[ks]);
        if (g < 4 && t < 2) {
          Ss[g * 4 + 2 * t] = Sd.x + Rs[g * 4 + 2 * t];
          Ss[g * 4 + 2 * t + 1] = Sd.y + Rs[g * 4 + 2 * t + 1];
        }
      }
      __syncwarp();
      // ---- K = (P H') S^-1,  I - K H,  K R ----
      {
        double Sl[16], Sil[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) Sl[e] = Ss[e];
        inv4(Sl, Sil);
        const double sib = g < 4 ? pick16(Sil, t * 4 + g) : 0.0;            // B fragment of S^-1: Si[t][g]
        double2 K0 = make_double2(0.0, 0.0), K1 = K0;
        dmma(K0, PHts[g * TC_LD4 + t], sib);
        dmma(K1, PHts[(8 + g) * TC_LD4 + t], sib);
        *reinterpret_cast<double2*>(Ks + g * TC_LD4 + 2 * t) = K0;
        *reinterpret_cast<double2*>(Ks + (8 + g) * TC_LD4 + 2 * t) = K1;
      }
      __syncwarp();
      double Af[2][4];     // A fragments of I - K H, kept for both products below
      double Kf[2];        // A fragments of K (= B fragments of K')
      {
        Kf[0] = Ks[g * TC_LD4 + t]; Kf[1] = Ks[(8 + g) * TC_LD4 + t];
        double2 Ad[2][2];
#pragma unroll
        for (int ri = 0; ri < 2; ++ri)
#pragma unroll
          for (int ci = 0; ci < 2; ++ci) {
            Ad[ri][ci] = make_double2(0.0, 0.0);
            dmma(Ad[ri][ci], Kf[ri], Hb[ci]);
            const int rr = 8 * ri + g, c0 = 8 * ci + 2 * t;
            Ad[ri][ci].x = ((rr == c0 && rr < 15) ? 1.0 : 0.0) - Ad[ri][ci].x;
            Ad[ri][ci].y = ((rr == c0 + 1 && rr < 15) ? 1.0 : 0.0) - Ad[ri][ci].y;
            *reinterpret_cast<double2*>(As + rr * TC_LD + c0) = Ad[ri][ci];
          }
        const double rb = g < 4 ? Rs[t * 4 + g] : 0.0;                      // B fragment of R: R[t][g]
        double2 KR0 = make_double2(0.0, 0.0), KR1 = KR0;
        dmma(KR0, Kf[0], rb);
        dmma(KR1, Kf[1], rb);
        *reinterpret_cast<double2*>(KRs + g * TC_LD4 + 2 * t) = KR0;
        *reinterpret_cast<double2*>(KRs + (8 + g) * TC_LD4 + 2 * t) = KR1;
      }
      __syncwarp();
      // ---- Joseph form: P = ((I-KH) P) (I-KH)' + (K R) K' ----
      {
#pragma unroll
        for (int ri = 0; ri < 2; ++ri)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) Af[ri][ks] = As[(8 * ri + g) * TC_LD + 4 * ks + t];
        const double kr0 = KRs[g * TC_LD4 + t], kr1 = KRs[(8 + g) * TC_LD4 + t];
        __syncwarp();        // K R shares storage with T: every lane has its fragment before T is written
        double2 Td[2][2];
#pragma unroll
        for (int ri = 0; ri < 2; ++ri)
#pragma unroll
          for (int ci = 0; ci < 2; ++ci) Td[ri][ci] = make_double2(0.0, 0.0);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const double b0 = Ps[(4 * ks + t) * TC_LD + g], b1 = Ps[(4 * ks + t) * TC_LD + 8 + g];
          dmma(Td[0][0], Af[0][ks], b0); dmma(Td[0][1], Af[0][ks], b1);
          dmma(Td[1][0], Af[1][ks], b0); dmma(Td[1][1], Af[1][ks], b1);
        }
#pragma unroll
        for (int ri = 0; ri < 2; ++ri)
#pragma unroll
          for (int ci = 0; ci < 2; ++ci)
            *reinterpret_cast<double2*>(Ts + (8 * ri + g) * TC_LD + 8 * ci + 2 * t) = Td[ri][ci];
        __syncwarp();
        double2 Pd[2][2], Gd[2][2];
#pragma unroll
        for (int ri = 0; ri < 2; ++ri)
#pragma unroll
          for (int ci = 0; ci < 2; ++ci) {
            Pd[ri][ci] = make_double2(0.0, 0.0);
            Gd[ri][ci] = make_double2(0.0, 0.0);
            dmma(Gd[ri][ci], ri ? kr1 : kr0, Kf[ci]);
          }
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const double a0 = Ts[g * TC_LD + 4 * ks + t], a1 = Ts[(8 + g) * TC_LD + 4 * ks + t];
          dmma(Pd[0][0], a0, Af[0][ks]); dmma(Pd[0][1], a0, Af[1][ks]);
          dmma(Pd[1][0], a1, Af[0][ks]); dmma(Pd[1][1], a1, Af[1][ks]);
        }
#pragma unroll
        for (int ri = 0; ri < 2; ++ri)
#pragma unroll
          for (int ci = 0; ci < 2; ++ci)
            *reinterpret_cast<double2*>(Ps + (8 * ri + g) * TC_LD + 8 * ci + 2 * t) =
                make_double2(Pd[ri][ci].x + Gd[ri][ci].x, Pd[ri][ci].y + Gd[ri][ci].y);
        __syncwarp();
      }
      ++i_upd;
    }
    // ---- error observer ----
    const double p66 = fabs(Ps[6 * TC_LD + 6]), p77 = fabs(Ps[7 * TC_LD + 7]), p88 = fabs(Ps[8 * TC_LD + 8]);
    if (slip_i + 1 < nsteps && obs_cannot_trigger_sq(ob, p66, p77, p88)) continue;      // no square roots on this path
    const double dl3 = 3.0 * sqrt(p66), dm3 = 3.0 * sqrt(p77), dh3 = 3.0 * sqrt(p88);
    if (slip_i + 1 < nsteps && obs_cannot_trigger(ob, dl3, dm3, dh3, cfg.thresh)) continue;
    const double lat3 = lat + dl3;
    const double lon3 = lon + dm3;
    const double h3 = hgt + dh3;
    double tsn, tcs;                               // lane 0: latitude, lane 1: longitude
    det_sincos(lane == 0 ? lat3 : lon3, tsn, tcs);
    const double sp = __shfl_sync(0xffffffffu, tsn, 0), cp = __shfl_sync(0xffffffffu, tcs, 0),
                 sl = __shfl_sync(0xffffffffu, tsn, 1), cl = __shfl_sync(0xffffffffu, tcs, 1);
    const double tp = sp / cp;
    double enu3[3];
    llh_to_enu_trig(sp, cp, tp, sl, cl, h3, lk, cfg, enu3);
    const double dx = enu3[0] - enu0[0], dy = enu3[1] - enu0[1];
    xy = sqrt(dx * dx + dy * dy);
    if (xy > cfg.thresh) { trig = 1; step = slip_i; break; }
  }
  if (lane == 0) {
    a.triggered[b] = trig;
    a.i_stop[b] = i_upd;
    a.step_stop[b] = step;
    a.xy_err[b] = xy;
  }
  if (a.P_final) {
    __syncwarp();
    for (int i = lane; i < 225; i += 32) a.P_final[b * 225 + i] = Ps[(i / 15) * TC_LD + i % 15];
    if (a.K_final) for (int i = lane; i < 60; i += 32) a.K_final[b * 60 + i] = Ks[(i / 4) * TC_LD4 + i % 4];
    if (a.R_final && lane < 16) a.R_final[b * 16 + lane] = Rs[lane];
  }
  if (!a.next_window) return;
  }   // next claimed window
}

// ---------------------------------------------------------------------------------------------------------------------
// Scalar kernels (round 1): the same algebra as explicit fma chains.  Kept as an independent implementation of the same
// bits - tests/test_gpu_lookahead.py runs all three on one batch and demands identical xy_err - and selectable with
// CNGP_LOOKAHEAD_KERNEL = warp | cta.
// ---------------------------------------------------------------------------------------------------------------------
// per-warp shared-memory working set (doubles)
constexpr int LA_P = 0, LA_T = 225, LA_A = 450, LA_PHT = 675, LA_K = 735, LA_KR = 795, LA_S = 855, LA_SI = 871,
              LA_R = 887, LA_F = 903, LA_Q = 1128, LA_H = 1353, LA_HP = 1413, LA_WS = 1473 + 3;  // padded to an even count

__global__ void __launch_bounds__(LA_WARPS * 32) zupt_lookahead_kernel(const LookaheadArgs a) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long b = (long long)blockIdx.x * LA_WARPS + w;
  if (b >= a.B) return;
  double* ws = smem + (long long)w * LA_WS;
  double *P = ws + LA_P, *T = ws + LA_T, *A = ws + LA_A, *PHt = ws + LA_PHT, *K = ws + LA_K, *KR = ws + LA_KR,
         *S = ws + LA_S, *Si = ws + LA_SI, *R = ws + LA_R, *F = ws + LA_F, *Q = ws + LA_Q, *H = ws + LA_H, *HP = ws + LA_HP;
  const cngp_stop_config& cfg = a.cfg;
  const int pw = a.per_window;
  const double* gP = a.P + ((pw & CNGP_PERWIN_P) ? b * 225 : 0);
  const double* gQ = a.Q + ((pw & CNGP_PERWIN_Q) ? b * 225 : 0);
  const double* gF = a.STM + ((pw & CNGP_PERWIN_STM) ? b * 225 : 0);
  const double* gH = a.Hvec + ((pw & CNGP_PERWIN_H) ? b * 60 : 0);
  const double* gpos = a.pos + ((pw & CNGP_PERWIN_POS) ? b * 3 : 0);
  for (int i = lane; i < 225; i += 32) { P[i] = gP[i]; Q[i] = gQ[i]; F[i] = gF[i]; }
  for (int i = lane; i < 60; i += 32) {
    const int rr = i / 15, cc = i % 15;
    H[i] = gH[cfg.fix_h_packing ? rr * 15 + cc : rr * 4 + cc];  // gp_predictor.cpp:38-42 aliasing index
  }
  const double lat = gpos[0], lon = gpos[1], hgt = gpos[2];
  const LlhConst lk = llh_prepare(cfg);
  double enu0[3];
  llh_to_enu_dev(lat, lon, hgt, lk, cfg, enu0);
  const ObsBound ob = obs_prepare(lat, lon, hgt, cfg);
  __syncwarp();

  // unit rows 9..14 in the STM (true for every CoreNav::insErrorStateModel_LNF output): see the propagation below
  bool unit_ok = true;
  for (int i = lane; i < 90; i += 32) {
    const int rr = 9 + i / 15, cc = i % 15;
    unit_ok = unit_ok && F[rr * 15 + cc] == (rr == cc ? 1.0 : 0.0);
  }
  const bool bias_rows_identity = __all_sync(0xffffffffu, unit_ok);

  const double* mean = a.mean + b * a.ms_stride;
  const double* sigma = a.sigma + b * a.ms_stride;
  const int nsteps = cfg.ratio * (a.m_win ? a.m_win[b] : a.M);
  int i_upd = 0, trig = 0, step = nsteps;
  double xy = 0.0;

  for (int slip_i = 0; slip_i < nsteps; ++slip_i) {
    // ---- P = F P F' + Q ----
    if (bias_rows_identity) {
      // Rows 9..14 of the STM are unit rows (the bias states are constants, CoreNav.cpp:462-468), so rows 9..14 of F P are
      // rows of P and columns 9..14 of (F P) F' are columns of F P: 90 of the 225 entries of each product are copies.
      // The copied value is what the full dot product returns (every other term is an exact zero), so the result is
      // unchanged up to the sign of zeros.
#pragma unroll
      for (int t = 0; t < 5; ++t) {
        const int idx = lane + 32 * t;         // rows 0..8 are the first 135 entries
        if (idx < 135) {
          const int rr = idx / 15, kk = idx % 15;
          double acc = 0.0;
#pragma unroll
          for (int j = 0; j < 15; ++j) acc = fma(F[rr * 15 + j], P[j * 15 + kk], acc);
          T[idx] = acc;
        }
      }
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        const int idx = 135 + lane + 32 * t;
        if (idx < 225) T[idx] = P[idx];
      }
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 5; ++t) {
        const int e = lane + 32 * t;
        if (e < 135) {
          const int rr = e / 9, cc = e % 9, idx = rr * 15 + cc;
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < 15; ++k) acc = fma(T[rr * 15 + k], F[cc * 15 + k], acc);
          P[idx] = acc + Q[idx];
        }
      }
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        const int e = lane + 32 * t;
        if (e < 90) {
          const int idx = (e / 6) * 15 + 9 + e % 6;
          P[idx] = T[idx] + Q[idx];
        }
      }
      __syncwarp();
    } else {
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int idx = lane + 32 * t;
        if (idx < 225) {
          const int rr = idx / 15, kk = idx % 15;
          double acc = 0.0;
#pragma unroll
          for (int j = 0; j < 15; ++j) acc = fma(F[rr * 15 + j], P[j * 15 + kk], acc);
          T[idx] = acc;
        }
      }
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int idx = lane + 32 * t;
        if (idx < 225) {
          const int rr = idx / 15, cc = idx % 15;
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < 15; ++k) acc = fma(T[rr * 15 + k], F[cc * 15 + k], acc);
          P[idx] = acc + Q[idx];
        }
      }
      __syncwarp();
    }
    if (slip_i % cfg.ratio == 0) {
      // ---- UT -> R_IP, K = P H' (H P H' + R)^-1, Joseph update ----
      double Rl[16];
      ut_R(mean[i_upd], sigma[i_upd], cfg, Rl);
      if (lane < 16) R[lane] = Rl[lane];
      for (int idx = lane; idx < 60; idx += 32) {
        const int rr = idx / 4, mm = idx % 4;
        double acc = 0.0;
#pragma unroll
        for (int c = 0; c < 15; ++c) acc = fma(P[rr * 15 + c], H[mm * 15 + c], acc);
        PHt[idx] = acc;
      }
      // S = (H P) H' + R: H_*P_pred*H_.transpose() is parsed left to right (gp_predictor.cpp:90)
      for (int idx = lane; idx < 60; idx += 32) {
        const int mm = idx / 15, c = idx % 15;
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 15; ++j) acc = fma(H[mm * 15 + j], P[j * 15 + c], acc);
        HP[idx] = acc;
      }
      __syncwarp();
      if (lane < 16) {
        const int mm = lane / 4, nn = lane % 4;
        double acc = 0.0;
#pragma unroll
        for (int c = 0; c < 15; ++c) acc = fma(HP[mm * 15 + c], H[nn * 15 + c], acc);
        S[lane] = acc + R[lane];
      }
      __syncwarp();
      {
        double Sl[16], Sil[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) Sl[e] = S[e];
        inv4(Sl, Sil);
        if (lane < 16) Si[lane] = Sil[lane];
      }
      __syncwarp();
      for (int idx = lane; idx < 60; idx += 32) {
        const int rr = idx / 4, mm = idx % 4;
        double acc = 0.0;
#pragma unroll
        for (int n = 0; n < 4; ++n) acc = fma(PHt[rr * 4 + n], Si[n * 4 + mm], acc);
        K[idx] = acc;
      }
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int idx = lane + 32 * t;
        if (idx < 225) {
          const int rr = idx / 15, cc = idx % 15;
          double acc = 0.0;
#pragma unroll
          for (int m = 0; m < 4; ++m) acc = fma(K[rr * 4 + m], H[m * 15 + cc], acc);
          A[idx] = (rr == cc ? 1.0 : 0.0) - acc;
        }
      }
      for (int idx = lane; idx < 60; idx += 32) {
        const int rr = idx / 4, nn = idx % 4;
        double acc = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) acc = fma(K[rr * 4 + m], R[m * 4 + nn], acc);
        KR[idx] = acc;
      }
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int idx = lane + 32 * t;
        if (idx < 225) {
          const int rr = idx / 15, kk = idx % 15;
          double acc = 0.0;
#pragma unroll
          for (int j = 0; j < 15; ++j) acc = fma(A[rr * 15 + j], P[j * 15 + kk], acc);
          T[idx] = acc;
        }
      }
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int idx = lane + 32 * t;
        if (idx < 225) {
          const int rr = idx / 15, cc = idx % 15;
          double a1 = 0.0, a2 = 0.0;
#pragma unroll
          for (int k = 0; k < 15; ++k) a1 = fma(T[rr * 15 + k], A[cc * 15 + k], a1);
#pragma unroll
          for (int n = 0; n < 4; ++n) a2 = fma(KR[rr * 4 + n], K[cc * 4 + n], a2);
          P[idx] = a1 + a2;
        }
      }
      __syncwarp();
      ++i_upd;
    }
    // ---- error observer ----
    const double dl3 = 3.0 * sqrt(fabs(P[6 * 15 + 6])), dm3 = 3.0 * sqrt(fabs(P[7 * 15 + 7])),
                 dh3 = 3.0 * sqrt(fabs(P[8 * 15 + 8]));
    if (slip_i + 1 < nsteps && obs_cannot_trigger(ob, dl3, dm3, dh3, cfg.thresh)) continue;
    const double lat3 = lat + dl3;
    const double lon3 = lon + dm3;
    const double h3 = hgt + dh3;
    double tsn, tcs;                               // lane 0: latitude, lane 1: longitude
    det_sincos(lane == 0 ? lat3 : lon3, tsn, tcs);
    const double sp = __shfl_sync(0xffffffffu, tsn, 0), cp = __shfl_sync(0xffffffffu, tcs, 0),
                 sl = __shfl_sync(0xffffffffu, tsn, 1), cl = __shfl_sync(0xffffffffu, tcs, 1);
    const double tp = sp / cp;
    double enu3[3];
    llh_to_enu_trig(sp, cp, tp, sl, cl, h3, lk, cfg, enu3);
    const double dx = enu3[0] - enu0[0], dy = enu3[1] - enu0[1];
    xy = sqrt(dx * dx + dy * dy);
    if (xy > cfg.thresh) { trig = 1; step = slip_i; break; }
  }
  if (lane == 0) {
    a.triggered[b] = trig;
    a.i_stop[b] = i_upd;
    a.step_stop[b] = step;
    a.xy_err[b] = xy;
  }
  if (a.P_final) {
    __syncwarp();
    for (int i = lane; i < 225; i += 32) a.P_final[b * 225 + i] = P[i];
    if (a.K_final) for (int i = lane; i < 60; i += 32) a.K_final[b * 60 + i] = K[i];
    if (a.R_final && lane < 16) a.R_final[b * 16 + lane] = R[lane];
  }
}

// Small batches (the reference's own use: ONE window per callback, gp_predictor.cpp:16): the look-ahead is a chain of up
// to 2995 dependent 15x15 steps, and one warp per window spends ~7 k cycles on each.  Here a CTA of 256 threads takes the
// window - one thread per matrix entry, every dot product in the same ascending-index fma order as the warp kernel (so
// the results are the same bits), the five trigonometric values of the observer on five different warps - which cuts
// the step to about a seventh.  Used when the batch cannot fill the GPU with warps anyway (LA_CTA_MAX_B).
constexpr int LA_CTA_THREADS = 256;
constexpr long long LA_CTA_MAX_B = 592;   // 4 windows per SM

__global__ void __launch_bounds__(LA_CTA_THREADS) zupt_lookahead_cta_kernel(const LookaheadArgs a) {
  extern __shared__ double ws[];
  const int tid = threadIdx.x;
  const long long b = blockIdx.x;
  double *P = ws + LA_P, *T = ws + LA_T, *A = ws + LA_A, *PHt = ws + LA_PHT, *K = ws + LA_K, *KR = ws + LA_KR,
         *S = ws + LA_S, *Si = ws + LA_SI, *R = ws + LA_R, *F = ws + LA_F, *Q = ws + LA_Q, *H = ws + LA_H, *HP = ws + LA_HP;
  const cngp_stop_config& cfg = a.cfg;
  const int pw = a.per_window;
  const double* gP = a.P + ((pw & CNGP_PERWIN_P) ? b * 225 : 0);
  const double* gQ = a.Q + ((pw & CNGP_PERWIN_Q) ? b * 225 : 0);
  const double* gF = a.STM + ((pw & CNGP_PERWIN_STM) ? b * 225 : 0);
  const double* gH = a.Hvec + ((pw & CNGP_PERWIN_H) ? b * 60 : 0);
  const double* gpos = a.pos + ((pw & CNGP_PERWIN_POS) ? b * 3 : 0);
  if (tid < 225) { P[tid] = gP[tid]; Q[tid] = gQ[tid]; F[tid] = gF[tid]; }
  if (tid < 60) {
    const int rr = tid / 15, cc = tid % 15;
    H[tid] = gH[cfg.fix_h_packing ? rr * 15 + cc : rr * 4 + cc];
  }
  const double lat = gpos[0], lon = gpos[1], hgt = gpos[2];
  const LlhConst lk = llh_prepare(cfg);
  double enu0[3];
  llh_to_enu_dev(lat, lon, hgt, lk, cfg, enu0);
  const ObsBound ob = obs_prepare(lat, lon, hgt, cfg);
  __syncthreads();
  bool unit_ok = true;
  if (tid < 90) {
    const int rr = 9 + tid / 15, cc = tid % 15;
    unit_ok = F[rr * 15 + cc] == (rr == cc ? 1.0 : 0.0);
  }
  const bool bias_rows_identity = __syncthreads_and(unit_ok);

  const double* mean = a.mean + b * a.ms_stride;
  const double* sigma = a.sigma + b * a.ms_stride;
  const int nsteps = cfg.ratio * (a.m_win ? a.m_win[b] : a.M);
  const bool ent = tid < 225;
  const int rr = tid / 15, cc = tid % 15;      // entry (rr, cc) of a 15x15 matrix
  const int r4 = tid / 4, m4 = tid % 4;        // entry (r4, m4) of a 15x4 matrix (tid < 60), (m4', n4) of 4x4 (tid < 16)
  int i_upd = 0, trig = 0, step = nsteps;
  double xy = 0.0;

  for (int slip_i = 0; slip_i < nsteps; ++slip_i) {
    // ---- P = F P F' + Q ----
    if (ent) {
      double acc;
      if (bias_rows_identity && rr >= 9) {
        acc = P[tid];
      } else {
        acc = 0.0;
#pragma unroll
        for (int j = 0; j < 15; ++j) acc = fma(F[rr * 15 + j], P[j * 15 + cc], acc);
      }
      T[tid] = acc;
    }
    __syncthreads();
    if (ent) {
      double acc;
      if (bias_rows_identity && cc >= 9) {
        acc = T[tid];
      } else {
        acc = 0.0;
#pragma unroll
        for (int k = 0; k < 15; ++k) acc = fma(T[rr * 15 + k], F[cc * 15 + k], acc);
      }
      P[tid] = acc + Q[tid];
    }
    __syncthreads();
    if (slip_i % cfg.ratio == 0) {
      // ---- UT -> R_IP, K = P H' (H P H' + R)^-1, Joseph update ----
      double Rl[16];
      ut_R(mean[i_upd], sigma[i_upd], cfg, Rl);
      if (tid < 16) R[tid] = Rl[tid];
      if (tid < 60) {
        double acc = 0.0;
#pragma unroll
        for (int c = 0; c < 15; ++c) acc = fma(P[r4 * 15 + c], H[m4 * 15 + c], acc);
        PHt[tid] = acc;
      } else if (tid >= 64 && tid < 124) {      // S = (H P) H' + R, left to right as gp_predictor.cpp:90 parses
        const int e = tid - 64, mm = e / 15, c = e % 15;
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 15; ++j) acc = fma(H[mm * 15 + j], P[j * 15 + c], acc);
        HP[e] = acc;
      }
      __syncthreads();
      if (tid < 16) {
        double acc = 0.0;
#pragma unroll
        for (int c = 0; c < 15; ++c) acc = fma(HP[r4 * 15 + c], H[m4 * 15 + c], acc);
        S[tid] = acc + R[tid];
      }
      __syncthreads();
      {
        double Sl[16], Sil[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) Sl[e] = S[e];
        inv4(Sl, Sil);
        if (tid < 16) Si[tid] = Sil[tid];
      }
      __syncthreads();
      if (tid < 60) {
        double acc = 0.0;
#pragma unroll
        for (int n = 0; n < 4; ++n) acc = fma(PHt[r4 * 4 + n], Si[n * 4 + m4], acc);
        K[tid] = acc;
      }
      __syncthreads();
      if (ent) {
        double acc = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) acc = fma(K[rr * 4 + m], H[m * 15 + cc], acc);
        A[tid] = (rr == cc ? 1.0 : 0.0) - acc;
      }
      if (tid < 60) {
        double acc = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) acc = fma(K[r4 * 4 + m], R[m * 4 + m4], acc);
        KR[tid] = acc;
      }
      __syncthreads();
      if (ent) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 15; ++j) acc = fma(A[rr * 15 + j], P[j * 15 + cc], acc);
        T[tid] = acc;
      }
      __syncthreads();
      if (ent) {
        double a1 = 0.0, a2 = 0.0;
#pragma unroll
        for (int k = 0; k < 15; ++k) a1 = fma(T[rr * 15 + k], A[cc * 15 + k], a1);
#pragma unroll
        for (int n = 0; n < 4; ++n) a2 = fma(KR[rr * 4 + n], K[cc * 4 + n], a2);
        P[tid] = a1 + a2;
      }
      __syncthreads();
      ++i_upd;
    }
    // ---- error observer ----
    const double dl3 = 3.0 * sqrt(fabs(P[6 * 15 + 6])), dm3 = 3.0 * sqrt(fabs(P[7 * 15 + 7])),
                 dh3 = 3.0 * sqrt(fabs(P[8 * 15 + 8]));
    if (slip_i + 1 < nsteps && obs_cannot_trigger(ob, dl3, dm3, dh3, cfg.thresh)) continue;   // same P in every thread
    const double lat3 = lat + dl3;
    const double lon3 = lon + dm3;
    const double h3 = hgt + dh3;
    double sp, cp, sl, cl;                         // cheap enough (about 40 fma) to repeat in every thread
    det_sincos(lat3, sp, cp);
    det_sincos(lon3, sl, cl);
    double enu3[3];
    llh_to_enu_trig(sp, cp, sp / cp, sl, cl, h3, lk, cfg, enu3);
    const double dx = enu3[0] - enu0[0], dy = enu3[1] - enu0[1];
    xy = sqrt(dx * dx + dy * dy);
    if (xy > cfg.thresh) { trig = 1; step = slip_i; break; }
  }
  if (tid == 0) {
    a.triggered[b] = trig;
    a.i_stop[b] = i_upd;
    a.step_stop[b] = step;
    a.xy_err[b] = xy;
  }
  if (a.P_final) {
    __syncthreads();
    if (tid < 225) a.P_final[b * 225 + tid] = P[tid];
    if (a.K_final && tid < 60) a.K_final[b * 60 + tid] = K[tid];
    if (a.R_final && tid < 16) a.R_final[b * 16 + tid] = R[tid];
  }
}

__global__ void llh_to_enu_kernel(const double* llh, long long n, cngp_stop_config cfg, double* enu) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const LlhConst lk = llh_prepare(cfg);
  double e[3];
  llh_to_enu_dev(llh[3 * i], llh[3 * i + 1], llh[3 * i + 2], lk, cfg, e);
  enu[3 * i] = e[0]; enu[3 * i + 1] = e[1]; enu[3 * i + 2] = e[2];
}

}  // namespace cngp

extern "C" int cngp_launch_lookahead(const double* mean, const double* sigma, long long B, int M, const double* P,
                                     const double* Q, const double* STM, const double* Hvec, const double* pos,
                                     int per_window, const cngp_stop_config* cfg, int* triggered, int* i_stop,
                                     int* step_stop, double* xy_err, unsigned long long* work_counter,
                                     double* P_final, double* K_final, double* R_final, const double* R_fixed,
                                     int R_per_window, cudaStream_t stream, const int* m_win) {
  using namespace cngp;
  // M < 0: |M| entries of mean / sigma shared by every window (cngp_ekf_covariance_batch)
  LookaheadArgs a{mean, sigma, B, M < 0 ? -M : M, P, Q, STM, Hvec, pos, per_window, *cfg, triggered, i_stop, step_stop,
                  xy_err, nullptr, P_final, K_final, R_final, R_fixed, R_per_window, M < 0 ? 0LL : (long long)M, m_win};
  const size_t smem = (size_t)LA_WARPS * LA_WS * sizeof(double);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(zupt_lookahead_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    attr_set = true;
  }
  const char* force = getenv("CNGP_LOOKAHEAD_KERNEL");     // "tc" (default) / "warp" / "cta": tests run all on one batch
  if (!force || force[0] == 't' || R_fixed) {
    // few windows: one warp per CTA so that they spread over the SMs; many: eight warps per CTA
    const int wpc = B <= 4 * 148 ? 1 : TC_WARPS;
    const size_t tsm = (size_t)TC_WARPS * TC_WS * sizeof(double);
    static bool tc_attr = false;
    if (!tc_attr) {
      cudaFuncSetAttribute(zupt_lookahead_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm);
      cudaFuncSetAttribute(zupt_lookahead_tc_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);   // two CTAs per SM
      tc_attr = true;
    }
    long long grid = (B + wpc - 1) / wpc;
    if (wpc == TC_WARPS && work_counter && grid > 2 * 148) {     // persistent: two CTAs per SM claim windows dynamically
      if (cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), stream) != cudaSuccess) return (int)cudaGetLastError();
      a.next_window = work_counter;
      grid = 2 * 148;
    }
    zupt_lookahead_tc_kernel<<<(unsigned)grid, wpc * 32, (size_t)wpc * TC_WS * sizeof(double), stream>>>(a);
    return (int)cudaGetLastError();
  }
  const bool cta = force[0] == 'c';
  if (cta) {
    zupt_lookahead_cta_kernel<<<(unsigned)B, LA_CTA_THREADS, LA_WS * sizeof(double), stream>>>(a);
    return (int)cudaGetLastError();
  }
  const long long grid = (B + LA_WARPS - 1) / LA_WARPS;
  zupt_lookahead_kernel<<<(unsigned)grid, LA_WARPS * 32, smem, stream>>>(a);
  return (int)cudaGetLastError();
}

extern "C" int cngp_launch_llh_to_enu(const double* llh, long long n, const cngp_stop_config* cfg, double* enu,
                                      cudaStream_t stream) {
  cngp::llh_to_enu_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(llh, n, *cfg, enu);
  return (int)cudaGetLastError();
}
