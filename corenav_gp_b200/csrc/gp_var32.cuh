// FP32 mode (cngp_config.precision = CNGP_PRECISION_F32, north_star tolerance 1e-4) of phase B: predictive mean and
// variance on the TF32 tensor cores with the 3xTF32 split, i.e. FP32-level accuracy at tensor-core rate.
//
// Same algorithm and data movement as gp_var.cuh (row a6: mu = Kx' alpha, dtrtrs, var = Kxx - sum(tmp^2) + noise,
// gp_slip_node.py:47-50 -> GPy PosteriorExact._raw_predict): a persistent CTA streams each window's factor once per
// round through a bulk-TMA / mbarrier ring and every warp runs the right-looking forward substitution
// V^T = K*^T L^-T over the 8x8 tiles in storage order.  What changes is the tile product:
//
//   * a warp owns SIXTEEN test points and uses  mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 :  the 16 x 8
//     accumulator fragment (lane (g,t): rows g, g+8; columns 2t, 2t+1) is, with the k index permuted (slot t <-> column
//     2t, slot t+4 <-> column 2t+1), also a valid A fragment, and the B fragment of  D += X Y^T  for lane (g,t) is
//     Y[g][2t], Y[g][2t+1] - exactly the row-major 8x8 tile layout of the FP64 path - so, as there, no shuffle and
//     no layout conversion is needed between the steps of the substitution;
//   * phase A (gp_fit_kernel, FP64 - it is latency-bound, a narrower type would not make it faster) writes every
//     factor tile already SPLIT: lane (g,t) stores float4 {hi(Y[g][2t]), hi(Y[g][2t+1]), lo(..), lo(..)} with
//     hi = tf32(x), lo = tf32(x - hi): 512 B per tile as before, one 16-byte shared-memory load per lane and tile;
//   * a product is three MMAs,  D += Xlo Yhi + Xhi Ylo + Xhi Yhi  (the lo-lo term is below FP32 rounding), accumulated
//     in FP32.  Per test point and tile that is 3/16 MMA instead of 2/8 DMMA.
//
// K*^T is staged up front per unit (from the window's lag table when phase A built one, else through the interpreter)
// as FP32 accumulator fragments in a per-warp global line that stays in L1/L2.  Outputs are written as FP64 so the ABI
// does not change; only their accuracy does (tests/test_gpu_fp32_mode.py: 1e-4 against the FP64 oracle).
#pragma once
#include "gp_var.cuh"

namespace cngp {

// D(16x8, f32) += A(16x8, tf32) * B(8x8, tf32)
__device__ __forceinline__ void mma_tf32(float4& d, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d.x), "+f"(d.y), "+f"(d.z), "+f"(d.w)
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// hi / lo TF32 split of an accumulator fragment, laid out as an A fragment (see the header comment)
struct SplitA {
  uint32_t h0, h1, h2, h3, l0, l1, l2, l3;
};
__device__ __forceinline__ SplitA split_a(const float4& x) {
  SplitA s;
  // A fragment order: (row g, slot t) = x.x, (row g+8, slot t) = x.z, (row g, slot t+4) = x.y, (row g+8, slot t+4) = x.w
  s.h0 = to_tf32(x.x); s.h1 = to_tf32(x.z); s.h2 = to_tf32(x.y); s.h3 = to_tf32(x.w);
  s.l0 = to_tf32(x.x - __uint_as_float(s.h0)); s.l1 = to_tf32(x.z - __uint_as_float(s.h1));
  s.l2 = to_tf32(x.y - __uint_as_float(s.h2)); s.l3 = to_tf32(x.w - __uint_as_float(s.h3));
  return s;
}
// D += X Y^T with X split, Y = {hi(2t), hi(2t+1), lo(2t), lo(2t+1)} as stored by phase A
__device__ __forceinline__ void tile_mma32(float4& d, const SplitA& x, const float4& y) {
  const uint32_t yh0 = __float_as_uint(y.x), yh1 = __float_as_uint(y.y), yl0 = __float_as_uint(y.z), yl1 = __float_as_uint(y.w);
  mma_tf32(d, x.l0, x.l1, x.l2, x.l3, yh0, yh1);
  mma_tf32(d, x.h0, x.h1, x.h2, x.h3, yl0, yl1);
  mma_tf32(d, x.h0, x.h1, x.h2, x.h3, yh0, yh1);
}

constexpr size_t var32_smem_bytes(int nslot, int ct) { return (size_t)nslot * ct * 512 + 128; }

template <int NT_MAX, int WG, int NSLOT, int VAR_CT, bool FULL>
__global__ void __launch_bounds__(WG * 32, 1) gp_var32_kernel(const VarArgs a) {
  static_assert(NSLOT <= VAR_MAX_SLOTS && VAR_CT <= VAR_MAX_CT, "ring too deep / chunk too large");
  constexpr int VAR_CHUNK_FLOATS = VAR_CT * 128;
  extern __shared__ __align__(128) unsigned char dsm[];
  __shared__ LeafConst hc_all[WG][CNGP_MAX_LEAVES];
  __shared__ KProg kps;
  __shared__ VarGroupShared shg[1];
  const int lane = threadIdx.x & 31, wg = threadIdx.x >> 5;
  const int g8 = lane >> 2, t = lane & 3;
  const int nt = FULL ? NT_MAX : a.nt, M = a.M, mt = a.mt;   // mt = ceil(M / 16) here
  const int n8 = nt * 8;
  const int n_tiles = tiles_in_lower(nt);
  const int ce_max = (n_tiles - 1) / VAR_CT;
  const int nchunks = ce_max + 1;
  const int nrounds = (mt + WG - 1) / WG;
  const long long n_units = a.n_windows_launch * nrounds;
  const long long unit_stride = gridDim.x;
  const long long unit0 = blockIdx.x;

  VarGroupShared& sh = shg[0];
  float* ring = reinterpret_cast<float*>(dsm);
  const uint32_t ring_u32 = smem_u32(ring);
  const uint32_t full_u32 = smem_u32(&sh.full[0]);
  const uint32_t empty_u32 = smem_u32(&sh.empty[0]);
  if (threadIdx.x == 0) kps = a.kp;
  if (wg == 0 && lane == 0) {
    for (int s = 0; s < NSLOT; ++s) { mbar_init(full_u32 + 8 * s, 1); mbar_init(empty_u32 + 8 * s, WG); }
    sh.ce_max = ce_max; sh.nchunks = nchunks; sh.nrounds = nrounds; sh.n_tiles = n_tiles; sh.ct = VAR_CT;
    sh.unit0 = unit0; sh.n_units = n_units; sh.unit_stride = unit_stride;
    sh.Lbase = a.L; sh.list = nullptr; sh.ring_u32 = ring_u32; sh.full_u32 = full_u32;   // every window of the launch
    mbar_fence_init();
    for (int s = 0; s < NSLOT; ++s) var_issue_chunk(&sh, s, s);
  }
  __syncthreads();

  LeafConst* hc = hc_all[wg];
  float4* kst = reinterpret_cast<float4*>(a.kstage) + ((size_t)blockIdx.x * WG + wg) * (size_t)(NT_MAX * 32) + lane;
  int g = 0;

  for (long long u = unit0; u < n_units; u += unit_stride) {
    const long long lw = u / nrounds;
    const int round = (int)(u - lw * nrounds);
    const long long win = a.window0 + lw;
    const double* th = a.theta + (a.theta_mode == 0 ? 0 : win) * a.theta_stride;
    const int m16 = round * WG + wg;
    int slot = g % NSLOT;
    uint32_t parity = (uint32_t)(g / NSLOT) & 1u;
    int gc = g, duty = g % WG;
    g += nchunks;
    auto release_chunk = [&]() {    // ring protocol of gp_var.cuh
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
    if (m16 >= mt) {
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(full_u32 + 8 * slot, parity);
        release_chunk();
      }
      continue;
    }

    const double* km = a.kmeta ? a.kmeta + lw * (long long)VAR_META : nullptr;
    const bool tab = km && km[3] != 0.0;
    const double noise = th[a.kp.n_params];
    const bool bad = a.status && a.status[win] < 0;
    const int N = FULL ? NT_MAX * 8 : (a.n_win ? a.n_win[win] : a.N);
    const int m_lo = min(16 * m16 + g8, M - 1), m_hi = min(16 * m16 + 8 + g8, M - 1);
    const double* xsp = a.xstar + (a.xstar_stride ? win * a.xstar_stride : 0);
    const double x_lo = xsp[m_lo], x_hi = xsp[m_hi];
    const double* zp = a.z + lw * (long long)n8 + 2 * t;

    // ---- stage K*^T for my 16 test points as accumulator fragments (rolled; nothing else is live yet) ----
    if (tab) {
      const double* ktab = a.ktab + lw * (long long)VAR_TAB_MAX;
      const int* xip = a.kxi + lw * (long long)n8 + 2 * t;
      const int mi_lo = (int)(x_lo - km[1]), mi_hi = (int)(x_hi - km[1]);
#pragma unroll 4
      for (int J = nt - 1; J >= 0; --J) {
        const int c0 = 8 * (nt - 1 - J);
        const int2 xi2 = __ldg(reinterpret_cast<const int2*>(xip + c0));
        float4 v;
        v.x = (float)__ldg(ktab + abs(mi_lo - xi2.x)); v.y = (float)__ldg(ktab + abs(mi_lo - xi2.y));
        v.z = (float)__ldg(ktab + abs(mi_hi - xi2.x)); v.w = (float)__ldg(ktab + abs(mi_hi - xi2.y));
        if (!FULL) {
          if (c0 + 2 * t >= N) { v.x = 0.f; v.z = 0.f; }
          if (c0 + 2 * t + 1 >= N) { v.y = 0.f; v.w = 0.f; }
        }
        kst[J * 32] = v;
      }
    } else {
      __syncwarp();
      if (lane < a.kp.n_leaves) hc[lane] = leaf_prepare(a.kp.leaf_type[lane], th + a.kp.leaf_param[lane]);
      __syncwarp();
      const double* fp = a.feat + lw * (long long)(4 * n8) + 2 * t;      // row 0 of the features: the training stamps
#pragma unroll 1
      for (int J = nt - 1; J >= 0; --J) {
        const int c0 = 8 * (nt - 1 - J);
        const double2 x2 = *reinterpret_cast<const double2*>(fp + c0);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c0 + 2 * t < N) {
          v.x = (float)keval_generic_cross(&kps, hc, x2.x, x_lo);
          v.z = (float)keval_generic_cross(&kps, hc, x2.x, x_hi);
        }
        if (c0 + 2 * t + 1 < N) {
          v.y = (float)keval_generic_cross(&kps, hc, x2.y, x_lo);
          v.w = (float)keval_generic_cross(&kps, hc, x2.y, x_hi);
        }
        kst[J * 32] = v;
      }
    }
    __syncwarp();

    // ---- forward substitution over the streamed tiles ----
    float4 A[NT_MAX];
#pragma unroll
    for (int J = 0; J < NT_MAX; ++J) A[J] = make_float4(0.f, 0.f, 0.f, 0.f);
    float vs_lo = 0.f, vs_hi = 0.f, ms_lo = 0.f, ms_hi = 0.f;
    const float* cptr = ring + slot * VAR_CHUNK_FLOATS + 4 * lane;
    auto next_tile = [&](const int e, const bool first) -> float4 {
      const int ce = (e - 1) / VAR_CT;
      if (first || (e - 1) % VAR_CT == VAR_CT - 1) mbar_wait(full_u32 + 8 * slot, parity);
      const float4 v = *reinterpret_cast<const float4*>(cptr + (VAR_CT * ce + VAR_CT - e) * 128);
      if ((e - 1) % VAR_CT == 0) {
        release_chunk();
        cptr = ring + slot * VAR_CHUNK_FLOATS + 4 * lane;
      }
      return v;
    };

    float4 kv = kst[(nt - 1) * 32];
#pragma unroll
    for (int J = NT_MAX - 1; J >= 0; --J) {
      if (FULL || J < nt) {
        const int e0 = (J + 1) * (J + 2) / 2;
        const float4 Yd = next_tile(e0, J == nt - 1);
        const float4 X = make_float4(kv.x + A[J].x, kv.y + A[J].y, kv.z + A[J].z, kv.w + A[J].w);
        float4 V = make_float4(0.f, 0.f, 0.f, 0.f);
        tile_mma32(V, split_a(X), Yd);
        if (J > 0) kv = kst[(J - 1) * 32];
        const double2 zz = *reinterpret_cast<const double2*>(zp + 8 * (nt - 1 - J));
        const float z0 = (float)zz.x, z1 = (float)zz.y;
        vs_lo = fmaf(V.x, V.x, vs_lo); vs_lo = fmaf(V.y, V.y, vs_lo);
        vs_hi = fmaf(V.z, V.z, vs_hi); vs_hi = fmaf(V.w, V.w, vs_hi);
        ms_lo = fmaf(V.x, z0, ms_lo); ms_lo = fmaf(V.y, z1, ms_lo);
        ms_hi = fmaf(V.z, z0, ms_hi); ms_hi = fmaf(V.w, z1, ms_hi);
        const SplitA nV = split_a(make_float4(-V.x, -V.y, -V.z, -V.w));
#pragma unroll
        for (int J2 = J - 1; J2 >= 0; --J2) {
          const float4 Ya = next_tile(e0 - (J - J2), false);
          tile_mma32(A[J2], nV, Ya);
        }
      }
    }
    vs_lo += __shfl_xor_sync(0xffffffffu, vs_lo, 1); vs_lo += __shfl_xor_sync(0xffffffffu, vs_lo, 2);
    vs_hi += __shfl_xor_sync(0xffffffffu, vs_hi, 1); vs_hi += __shfl_xor_sync(0xffffffffu, vs_hi, 2);
    ms_lo += __shfl_xor_sync(0xffffffffu, ms_lo, 1); ms_lo += __shfl_xor_sync(0xffffffffu, ms_lo, 2);
    ms_hi += __shfl_xor_sync(0xffffffffu, ms_hi, 1); ms_hi += __shfl_xor_sync(0xffffffffu, ms_hi, 2);
    if (t < 2) {     // lane t = 0 writes the point of row g, t = 1 the point of row g + 8
      const int mrow = 16 * m16 + g8 + 8 * t;
      if (mrow < (a.m_win ? a.m_win[win] : M)) {
        const double xm = t ? x_hi : x_lo;
        const double kss = tab ? km[0] : kdiag_eval(kps, hc, xm);
        const double vsum = t ? (double)vs_hi : (double)vs_lo, msum = t ? (double)ms_hi : (double)ms_lo;
        const double nanv = __longlong_as_double(0x7ff8000000000000LL);
        a.mean[win * M + mrow] = bad ? nanv : msum;
        const double vv = fmax(kss - vsum, CNGP_VAR_FLOOR) + noise;
        a.var[win * M + mrow] = bad ? nanv : (a.sigma_mode ? 2.0 * sqrt(vv) : vv);
      }
    }
    __syncwarp();
  }
}

}  // namespace cngp
