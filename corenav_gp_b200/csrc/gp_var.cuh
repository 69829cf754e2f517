// Phase B of the batched exact GP: predictive mean and variance at M test points per window.
//
// Replaces GPy PosteriorExact._raw_predict + Gaussian.predictive_values as reached from the per-point loop
// m.predict([[x]]) at core_navigation/script/gp_slip_node.py:47-50 (row a6):
//     mu = Kx' alpha,  tmp = dtrtrs(L, Kx),  var = max(Kxx - sum(tmp^2), 1e-15) + sigma_n^2.
//
// Work decomposition.  One WARP owns 8 test points and runs a right-looking forward substitution V^T = K*^T L^-T over
// the tile columns of L:  V_j = (K*_j + A_j) inv(L_jj)^T,  then  A_j' -= V_j L(j',j)^T  for every j' > j - all
// tile_mma (FP64 DMMA).  The 8 x N block A of accumulated updates lives in registers (64 doubles per lane at N = 256);
// the rows of V never leave registers; mean = V' z with z = L^-1 y from phase A (no back-substitution),
// var = k** - sum V^2.  K*^T is evaluated LAZILY, one 8x8 tile per column step, right behind the two dependent DMMA of
// the diagonal step, so the scalar FP64 work of the covariance function (exp_tab, kernel_eval.cuh) interleaves with the
// tensor work instead of forming a phase of its own; it never touches memory.  (Arbitrary kernel expressions go
// through the out-of-line interpreter, which cannot be called with 64 live accumulators: for them the tiles are
// evaluated up front by a rolled loop into a per-warp global staging line that stays in L1/L2.)
//
// Data movement.  The substitution consumes the packed tiles of L in exactly their storage order.  A persistent CTA
// (one per SM) is split into G independent GROUPS of WG warps; a group takes one UNIT = (window, round of WG test
// tiles) at a time - units are dealt round-robin over all groups of the grid, so neighbouring groups work on the same
// window and the factor is read from HBM once and from L2 afterwards - and streams that window's factor (270 KB at
// N = 256) through its own shared-memory ring filled by 1-D bulk asynchronous copies (cp.async.bulk -> UBLKCP,
// completion counted on mbarriers).  There is no producer warp: the last warp of the group to release a ring slot
// issues the copy that refills it, VAR_NSLOT chunks ahead, across unit boundaries.  Small groups keep the round
// quantisation loss low (M = 600: 75 test tiles = 18.75 rounds of 4) and let the groups drift apart, so the pipe sees
// a mix of phases.  Every tile costs each warp one 16-byte LDS per lane and two DMMA.
#pragma once
#include "kernel_eval.cuh"

namespace cngp {

constexpr int VAR_MAX_CT = 64;                  // largest chunk (tiles) any instantiation uses: sizes the slack
constexpr int VAR_MAX_SLOTS = 8;
// dynamic shared memory: G rings (NSLOT chunks of CT tiles) | per-warp exp tables (2 x 64) | padding
constexpr size_t var_smem_bytes(int groups, int wg, int nslot, int ct) {
  return (size_t)groups * nslot * ct * 512 + (size_t)groups * wg * 128 * 8 + 128;
}

struct VarArgs {
  KProg kp;
  const double* theta;
  long long theta_stride;
  int theta_mode;          // 0 shared, 1 per window
  const double* xstar;     // [n_windows][M] or [M]
  long long xstar_stride;  // M or 0
  int N, nt, M, mt;        // mt = ceil(M / 8): test tiles [mt0, mt) are handled by this launch
  int mt0;
  long long window0;       // first window of this launch
  long long n_windows_launch;
  const double* L;         // [chunk][tiles][64]  (phase A output; one chunk of slack before the first window)
  const double* z;         // [chunk][nt*8]
  const double* feat;      // [chunk][4][nt*8]  per-point features of the training inputs (phase A output)
  const int* status;       // [n_windows] (phase A), may be null
  double* mean;            // [n_windows][M]
  double* var;             // [n_windows][M]
  int sigma_mode;          // 0: var;  1: write sigma = 2 sqrt(var) instead (gp_slip_node.py:61)
  double* kstage;          // generic kernels only: [grid][warps][nt_max*64] staging of K*^T tiles
  // lag-table path (gp_fit.cuh "Lag tables"): K*(i,k) = ktab[|x*_k - x_i|], phase A output
  const double* ktab;      // [chunk][VAR_TAB_MAX]
  const double* kmeta;     // [chunk][VAR_META]
  const int* kxi;          // [chunk][nt*8]
  const int* n_lazy;       // windows of this launch without a valid table: the TAB kernel runs iff it is 0, the lazy one
                           // iff it is not (both are launched; one of them returns at once).  null: lazy only.
  // ragged batches (null: every window has N training / M test points).  n_win[win]: valid training points, ceil(/8) == nt;
  // m_win[win] <= M: valid test points - mean / var entries at or beyond it are not written (M stays the row stride).
  const int* n_win;
  const int* m_win;
  // windows left by gp_var_toeplitz_kernel (null: every window of the launch): local windows list[0 .. *list_count) in
  // increasing order, in place of 0 .. n_windows_launch-1
  const int* list;
  const int* list_count;
  // gp_var_toeplitz_kernel only, or null: [n_windows] windows whose results come from gp_toep_member_kernel (members of a
  // shared covariance, gp_toep_group.cuh) - marked taken and left untouched
  const int* skip;
};

struct VarGroupShared {
  unsigned long long full[VAR_MAX_SLOTS];   // mbarriers: chunk landed (transaction bytes)
  unsigned long long empty[VAR_MAX_SLOTS];  // mbarriers: every warp of the group has released the chunk
  int ce_max, nchunks, nrounds, n_tiles, ct;
  long long unit0, n_units, unit_stride;
  const double* Lbase;
  const int* list;
  uint32_t ring_u32, full_u32;
};

// Issue the bulk copy of chunk `gc` of the group's stream (units x chunks, in consumption order) into `slot`.
// Stateless - the position is decoded from gc - so refill duties may be carried out by different warps in any order.
// Called by one lane; kept out of line: it is the rare path.
static __device__ __noinline__ void var_issue_chunk(const VarGroupShared* sh, int gc, int slot) {
  const int k = gc / sh->nchunks;
  const int ce = sh->ce_max - (gc - k * sh->nchunks);
  const long long u = sh->unit0 + (long long)k * sh->unit_stride;
  if (u >= sh->n_units) return;
  const long long lw = sh->list ? sh->list[u / sh->nrounds] : u / sh->nrounds;
  const int ct = sh->ct;
  const double* src = sh->Lbase + (lw + 1) * (long long)sh->n_tiles * 64 - (long long)(ct * ce + ct) * 64;
  mbar_expect_tx(sh->full_u32 + 8 * slot, ct * 512);
  bulk_g2s(sh->ring_u32 + slot * ct * 512, src, ct * 512, sh->full_u32 + 8 * slot);
}

// FULL: nt == NT_MAX and N == 8 nt (no padding) - drops every per-column guard from the unrolled code.
// TAB: K* comes from the window's lag table (two cached global loads per tile and lane) instead of being evaluated -
// nothing but the DMMA stream and the mean / variance reductions is left on the FP64 pipe.  KID is ignored then.
template <int NT_MAX, int G, int WG, int NSLOT, int VAR_CT, int KID, bool FULL, bool TAB = false>
__global__ void __launch_bounds__(G * WG * 32, 1) gp_var_kernel(const VarArgs a) {
  if (a.n_lazy && ((*a.n_lazy == 0) != TAB)) return;
  const long long n_windows = a.list ? (long long)*a.list_count : a.n_windows_launch;
  if (n_windows == 0) return;
  static_assert(NSLOT <= VAR_MAX_SLOTS && VAR_CT <= VAR_MAX_CT, "ring too deep / chunk too large");
  constexpr int WARPS = G * WG;
  constexpr int VAR_CHUNK_DOUBLES = VAR_CT * 64;
  extern __shared__ __align__(128) unsigned char dsm[];
  __shared__ LeafConst hc_all[KID == KID_GENERIC ? WARPS : 1][CNGP_MAX_LEAVES];
  __shared__ KProg kps;
  __shared__ VarGroupShared shg[G];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int grp = w / WG, wg = w % WG;
  const int r = lane >> 2, q = lane & 3;
  const int nt = FULL ? NT_MAX : a.nt, M = a.M, mt = a.mt;
  const int n8 = nt * 8;
  const int n_tiles = tiles_in_lower(nt);
  const int ce_max = (n_tiles - 1) / VAR_CT;      // chunk ids count from the END of a window's factor
  const int nchunks = ce_max + 1;
  const int nrounds = (mt - a.mt0 + WG - 1) / WG;
  const long long n_units = n_windows * nrounds;
  const long long unit_stride = (long long)gridDim.x * G;
  const long long unit0 = (long long)blockIdx.x * G + grp;

  VarGroupShared& sh = shg[grp];
  double* ring = reinterpret_cast<double*>(dsm) + (size_t)grp * NSLOT * VAR_CHUNK_DOUBLES;
  double* tab = reinterpret_cast<double*>(dsm) + (size_t)G * NSLOT * VAR_CHUNK_DOUBLES + (size_t)w * 128;
  const uint32_t ring_u32 = smem_u32(ring);
  const uint32_t full_u32 = smem_u32(&sh.full[0]);

  if (threadIdx.x == 0 && KID == KID_GENERIC && !TAB) kps = a.kp;
  const uint32_t empty_u32 = smem_u32(&sh.empty[0]);
  if (wg == 0 && lane == 0) {
    for (int s = 0; s < NSLOT; ++s) { mbar_init(full_u32 + 8 * s, 1); mbar_init(empty_u32 + 8 * s, WG); }
    sh.ce_max = ce_max; sh.nchunks = nchunks; sh.nrounds = nrounds; sh.n_tiles = n_tiles; sh.ct = VAR_CT;
    sh.unit0 = unit0; sh.n_units = n_units; sh.unit_stride = unit_stride;
    sh.Lbase = a.L; sh.list = a.list; sh.ring_u32 = ring_u32; sh.full_u32 = full_u32;
    mbar_fence_init();
    for (int s = 0; s < NSLOT; ++s) var_issue_chunk(&sh, s, s);   // chunk g of the group goes to slot g % NSLOT
  }
  __syncthreads();

  LeafConst* hc = hc_all[KID == KID_GENERIC ? w : 0];
  double* kst = (KID == KID_GENERIC && !TAB) ? a.kstage + ((size_t)blockIdx.x * WARPS + w) * (size_t)(NT_MAX * 64) + 2 * lane : nullptr;
  int g = 0;   // chunk counter of this warp within its group's stream (over units x chunks)

  for (long long u = unit0; u < n_units; u += unit_stride) {
    const long long ui = u / nrounds;
    const long long lw = a.list ? a.list[ui] : ui;    // window within this launch
    const int round = (int)(u - ui * nrounds);
    const long long win = a.window0 + lw;
    const double* th = a.theta + (a.theta_mode == 0 ? 0 : win) * a.theta_stride;
    const int m8 = a.mt0 + round * WG + wg;
    int slot = g % NSLOT;
    uint32_t parity = (uint32_t)(g / NSLOT) & 1u;
    int gc = g, duty = g % WG;     // running chunk index of this warp; warp (gc mod WG) has refill duty at chunk gc
    g += nchunks;
    // Ring protocol.  Every warp of the group waits for and releases every chunk (mbarrier arrive on empty[slot] - fire
    // and forget), so no warp runs more than NSLOT chunks ahead of another, which is what makes waiting on a phase
    // PARITY safe.  The refill of a slot is a rotating duty: when warp (gc mod WG) releases chunk gc it makes sure
    // chunk gc-1 has been released by everybody (normally long true) and issues chunk gc-1+NSLOT into that slot.
    auto release_chunk = [&]() {
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(empty_u32 + 8 * slot);
        if (duty == wg && gc > 0) {
          const int ps = slot == 0 ? NSLOT - 1 : slot - 1;
          mbar_wait(empty_u32 + 8 * ps, slot == 0 ? parity ^ 1u : parity);
          var_issue_chunk(&sh, gc - 1 + NSLOT, ps);
        }
      }
      ++gc;
      if (++duty == WG) duty = 0;
      if (++slot == NSLOT) { slot = 0; parity ^= 1u; }
    };
    if (m8 >= mt) {   // no test tile for this warp in the window's last round: just keep the ring protocol going
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(full_u32 + 8 * slot, parity);
        release_chunk();
      }
      continue;
    }

    FastK<KID> fk;
    if (TAB) {
    } else if (KID == KID_GENERIC) {
      __syncwarp();
      if (lane < a.kp.n_leaves) hc[lane] = leaf_prepare(a.kp.leaf_type[lane], th + a.kp.leaf_param[lane]);
      __syncwarp();
    } else {
      fk.init(th);
      __syncwarp();
      const double s1 = fk.scale1(), s2 = fk.scale2();
      const double t0 = EXP2_TAB64[lane], t1 = EXP2_TAB64[lane + 32];
      tab[lane] = s1 * t0; tab[lane + 32] = s1 * t1;
      tab[64 + lane] = s2 * t0; tab[96 + lane] = s2 * t1;
      __syncwarp();
    }
    const double* fp = a.feat + lw * (long long)(4 * n8) + 2 * q;
    const double* zp = a.z + lw * (long long)n8 + 2 * q;
    const double* km = TAB ? a.kmeta + lw * (long long)VAR_META : nullptr;
    const double noise = TAB ? km[2] : th[a.kp.n_params];
    const bool bad = a.status && a.status[win] < 0;
    const int N = FULL ? NT_MAX * 8 : (a.n_win ? a.n_win[win] : a.N);

    const int m = min(8 * m8 + r, M - 1);
    const double xm = a.xstar[(a.xstar_stride ? win * a.xstar_stride : 0) + m];
    PointFeat fm{xm, 0.0, 0.0, 0.0};
    if (!TAB && KID != KID_GENERIC) {
      fk.base = a.feat[lw * (long long)(4 * n8)];      // the window's first training stamp, as in phase A
      fm = fk.point(xm);
    }
    const double* ktab = TAB ? a.ktab + lw * (long long)VAR_TAB_MAX : nullptr;
    const int* xip = TAB ? a.kxi + lw * (long long)n8 + 2 * q : nullptr;
    const int mi = TAB ? (int)(xm - km[1]) : 0;        // my test stamp as an offset from the window's base stamp

    // K*^T tile of training tile column j = nt-1-J (rows: my 8 test points), in the lane layout
    auto kstar_tile = [&](const int J) -> double2 {
      if (TAB) {
        const int c0 = 8 * (nt - 1 - J);
        const int2 xi2 = __ldg(reinterpret_cast<const int2*>(xip + c0));
        double2 v;
        v.x = __ldg(ktab + abs(mi - xi2.x));
        v.y = __ldg(ktab + abs(mi - xi2.y));
        if (!FULL) {
          if (c0 + 2 * q >= N) v.x = 0.0;
          if (c0 + 2 * q + 1 >= N) v.y = 0.0;
        }
        return v;
      }
      if (KID == KID_GENERIC) return *reinterpret_cast<const double2*>(kst + J * 64);
      const int c0 = 8 * (nt - 1 - J);     // + 2q is folded into fp
      const double2 x2 = *reinterpret_cast<const double2*>(fp + c0);
      const double2 xx2 = *reinterpret_cast<const double2*>(fp + n8 + c0);
      double2 cc2 = make_double2(0.0, 0.0), ss2 = make_double2(0.0, 0.0);
      if (KID == KID_RBF_PER) {
        cc2 = *reinterpret_cast<const double2*>(fp + 2 * n8 + c0);
        ss2 = *reinterpret_cast<const double2*>(fp + 3 * n8 + c0);
      }
      double2 v;
      v.x = fk.eval_tab(PointFeat{x2.x, xx2.x, cc2.x, ss2.x}, fm, false, tab);
      v.y = fk.eval_tab(PointFeat{x2.y, xx2.y, cc2.y, ss2.y}, fm, false, tab);
      if (!FULL) {   // padded training columns
        if (c0 + 2 * q >= N) v.x = 0.0;
        if (c0 + 2 * q + 1 >= N) v.y = 0.0;
      }
      return v;
    };
    if (!TAB && KID == KID_GENERIC) {   // rolled up-front evaluation through the interpreter (no accumulators live yet)
#pragma unroll 1
      for (int J = nt - 1; J >= 0; --J) {
        const int c0 = 8 * (nt - 1 - J) + 2 * q;
        const double2 x2 = *reinterpret_cast<const double2*>(fp + 8 * (nt - 1 - J));
        double2 v = make_double2(0.0, 0.0);
        if (c0 < N) v.x = keval_generic_cross(&kps, hc, x2.x, xm);
        if (c0 + 1 < N) v.y = keval_generic_cross(&kps, hc, x2.y, xm);
        *reinterpret_cast<double2*>(kst + J * 64) = v;
      }
    }

    // ---- forward substitution over the streamed tiles ----
    tile2 A[NT_MAX];
#pragma unroll
    for (int J = 0; J < NT_MAX; ++J) A[J] = tile2{0.0, 0.0};
    double vs = 0.0, ms = 0.0;
    const double* cptr = ring + slot * VAR_CHUNK_DOUBLES + 2 * lane;
    // tile at distance e (1-based) from the end of the factor: chunk id and offset inside the chunk are
    // compile-time after unrolling; the ring slot advances by one per chunk.
    auto next_tile = [&](const int e, const bool first) -> tile2 {
      const int ce = (e - 1) / VAR_CT;
      if (first || (e - 1) % VAR_CT == VAR_CT - 1) mbar_wait(full_u32 + 8 * slot, parity);
      const double2 v = *reinterpret_cast<const double2*>(cptr + (VAR_CT * ce + VAR_CT - e) * 64);
      if ((e - 1) % VAR_CT == 0) {     // chunk drained by this warp
        release_chunk();
        cptr = ring + slot * VAR_CHUNK_DOUBLES + 2 * lane;
      }
      return tile2{v.x, v.y};
    };

    double2 kv = kstar_tile(nt - 1);
#pragma unroll
    for (int J = NT_MAX - 1; J >= 0; --J) {
      if (FULL || J < nt) {
        const int e0 = (J + 1) * (J + 2) / 2;   // distance from the end of tile (J, d = 0)
        const tile2 Yd = next_tile(e0, J == nt - 1);
        const tile2 X{kv.x + A[J].a, kv.y + A[J].b};
        tile2 V{0.0, 0.0};
        tile_mma(V, X, Yd);
        if (J > 0) kv = kstar_tile(J - 1);      // independent scalar FP64 work behind the two dependent DMMA
        const double2 zz = *reinterpret_cast<const double2*>(zp + 8 * (nt - 1 - J));
        vs = fma(V.a, V.a, vs);
        vs = fma(V.b, V.b, vs);
        ms = fma(V.a, zz.x, ms);
        ms = fma(V.b, zz.y, ms);
        const tile2 nV{-V.a, -V.b};
        // two tiles per step with their DMMA pairs interleaved (a dependent DMMA costs 26 cycles, issue 16)
#pragma unroll
        for (int J2 = J - 1; J2 >= 1; J2 -= 2) {
          const tile2 Ya = next_tile(e0 - (J - J2), false);
          const tile2 Yb = next_tile(e0 - (J - J2) - 1, false);
          dmma884(A[J2].a, A[J2].b, nV.a, Ya.a);
          dmma884(A[J2 - 1].a, A[J2 - 1].b, nV.a, Yb.a);
          dmma884(A[J2].a, A[J2].b, nV.b, Ya.b);
          dmma884(A[J2 - 1].a, A[J2 - 1].b, nV.b, Yb.b);
        }
        if (J & 1) {   // J tiles below the diagonal: one left over when J is odd
          const tile2 Yl = next_tile(e0 - J, false);
          tile_mma(A[0], nV, Yl);
        }
      }
    }
    vs += __shfl_xor_sync(0xffffffffu, vs, 1);
    vs += __shfl_xor_sync(0xffffffffu, vs, 2);
    ms += __shfl_xor_sync(0xffffffffu, ms, 1);
    ms += __shfl_xor_sync(0xffffffffu, ms, 2);
    if (q == 0 && 8 * m8 + r < (a.m_win ? a.m_win[win] : M)) {
      const double kss = TAB ? km[0] : (KID == KID_GENERIC) ? kdiag_eval(kps, hc, xm) : fk.kdiag(xm);
      const double nanv = __longlong_as_double(0x7ff8000000000000LL);
      a.mean[win * M + m] = bad ? nanv : ms;
      const double vv = fmax(kss - vs, CNGP_VAR_FLOOR) + noise;
      a.var[win * M + m] = bad ? nanv : (a.sigma_mode ? 2.0 * sqrt(vv) : vv);
    }
  }
}

}  // namespace cngp
