// Shared device/host definitions for the cngp kernels (sm_100a).
//
// Tile algebra used by every linear-algebra kernel here
// -----------------------------------------------------
// All matrices are cut into 8x8 FP64 tiles stored row-major (64 doubles = 512 B).  A warp holds a tile as two
// doubles per lane: lane = 4*r + q  (r = lane>>2 row, q = lane&3)  holds  T[r][2q] and T[r][2q+1]  - which is both
// the accumulator (C/D) fragment layout of  mma.sync.aligned.m8n8k4.f64  and exactly one 16-byte load per lane.
// With the k index of the two k4-steps permuted (step s uses k = 2q+s), the same registers are also valid A and B
// fragments, so   tile_mma(D, X, Y):  D += X * Y^T   needs no shuffle and no layout conversion:
//     step s:  A[r][q] = X[r][2q+s],  B[q][n] = Y[n][2q+s]   =>   D[r][n] += sum_q X[r][2q+s] * Y[n][2q+s].
// Cholesky, triangular solves (with explicitly inverted 8x8 diagonal tiles), L^-1, K^-1 = W^T W and the
// predictive-variance substitution are all written as sequences of tile_mma, i.e. FP64 tensor-core DMMA.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/cngp.h"

#define CNGP_JITTER 1e-8          // GPy exact_gaussian_inference.py: Ky = K + (sigma_n^2 + 1e-8) I
#define CNGP_VAR_FLOOR 1e-15      // GPy posterior.py: np.clip(var, 1e-15, inf)
#define CNGP_LOG_2PI 1.8378770664093454836

namespace cngp {

struct tile2 {
  double a, b;  // T[r][2q], T[r][2q+1]
};

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(d0), "+d"(d1)
      : "d"(a), "d"(b));
}

// D += X * Y^T  (all three in the lane layout above)
__device__ __forceinline__ void tile_mma(tile2& d, const tile2& x, const tile2& y) {
  dmma884(d.a, d.b, x.a, y.a);
  dmma884(d.a, d.b, x.b, y.b);
}

__device__ __forceinline__ tile2 tile_load(const double* tile, int lane) {
  const double2 v = *reinterpret_cast<const double2*>(tile + 2 * lane);
  return tile2{v.x, v.y};
}
__device__ __forceinline__ void tile_store(double* tile, int lane, const tile2& t) {
  *reinterpret_cast<double2*>(tile + 2 * lane) = make_double2(t.a, t.b);
}

// FP32 mode (gp_var32.cuh): a factor tile is stored SPLIT for the 3xTF32 tensor-core product - lane 4r+q writes
// float4 {hi(T[r][2q]), hi(T[r][2q+1]), lo(T[r][2q]), lo(T[r][2q+1])}, hi = tf32(x), lo = tf32(x - hi): 512 B as before.
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// the 16 bytes of one entry pair (T[r][2q], T[r][2q+1]), at the place the two doubles would take
__device__ __forceinline__ void pair_store_split(double* dst, double x0, double x1) {
  const float a = (float)x0, b = (float)x1;
  const uint32_t ha = to_tf32(a), hb = to_tf32(b);
  const uint32_t la = to_tf32(a - __uint_as_float(ha)), lb = to_tf32(b - __uint_as_float(hb));
  *reinterpret_cast<uint4*>(dst) = make_uint4(ha, hb, la, lb);
}
__device__ __forceinline__ void tile_store_split(double* tile, int lane, const tile2& t) {
  pair_store_split(tile + 2 * lane, t.a, t.b);
}

// Packed lower-triangular tile storage, column-major: column j holds tiles i = j..nt-1 and starts after the
// nt + (nt-1) + ... tiles of columns 0..j-1.  Seen from the END of the buffer, column j (J = nt-1-j) starts
// (J+1)(J+2)/2 tiles before the end - independent of nt - and the forward substitution of gp_var.cuh consumes the
// tiles in exactly this linear order, which is what lets it stream them with bulk asynchronous copies.
__host__ __device__ __forceinline__ int tile_index(int i, int j, int nt) {
  return j * nt - j * (j - 1) / 2 + (i - j);
}
__host__ __device__ __forceinline__ int tiles_in_lower(int nt) { return nt * (nt + 1) / 2; }

// Lag tables.  The reference's stamps are integer update counts (CoreNav.cpp:286) and its prediction grid has step 1
// (gp_slip_node.py:45), so for a stationary expression k(x, x') is a function of the INTEGER lag |x - x'| only: at most
// span + horizon + 1 distinct values per window instead of N(N+1)/2 + N M evaluations.  gp_fit_kernel detects this per
// window (every stamp and every test point an integer below 2^26, which also makes GPy's expanded-form r^2 exact), builds
// the table once - with the same interpreter as the lazy path - keeps the lags of K(X,X) in shared memory for its own
// assembly and writes the whole table out for gp_var_kernel.  Non-integer stamps or other kernels take the lazy
// evaluators as before.
constexpr int FIT_TAB_MAX = 1024;     // lags of K(X,X) kept in shared memory (span of the training stamps)
constexpr int VAR_TAB_MAX = 2048;     // lags of the whole table (training + test stamps), doubles per window in scratch
constexpr int VAR_META = 8;           // doubles per window: [0] Kdiag(x*) (constant for stationary kernels), [1] base stamp,
                                      // [2] noise variance, [3] 1.0 if the table is valid

// ---- mbarrier + bulk asynchronous copy (TMA, 1-D) helpers ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_inval(uint32_t bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
// polling wait (test_wait returns at once): no suspend / wake-up latency, for waits that sit on a critical path
__device__ __forceinline__ void mbar_spin(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// global -> shared bulk copy, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src_gmem), "r"(bytes), "r"(bar)
               : "memory");
}

// ------------------------------------------------------------------------------------------------------------
// covariance functions.  A kernel expression (postfix program, cngp.h) is expanded on the host into a sum of
// products of leaves; the device evaluates   k = sum_t prod_u leaf_{t,u}.
// ------------------------------------------------------------------------------------------------------------
#define CNGP_MAX_LEAVES 24
struct KProg {
  int n_terms;
  int n_leaves;                      // total leaves over all terms
  int n_params;                      // kernel hyper-parameters (noise excluded)
  int term_start[CNGP_MAX_LEAVES + 1];
  int leaf_type[CNGP_MAX_LEAVES];    // CNGP_K_*
  int leaf_param[CNGP_MAX_LEAVES];   // offset of the leaf's first hyper-parameter in theta
  int fast_id;                       // 0 generic, else a specialised evaluator (see kernel_eval.cuh)
};

}  // namespace cngp
