// Large single-window exact GP (BASELINE.json configs[4], N = 32768): blocked right-looking FP64 Cholesky in HBM.
//
// Same inference as gp_fit.cuh (row a3: GPy ExactGaussianInference reached from GPRegression(...) at
// core_navigation/script/gp_slip_node.py:35 - Ky = K + (sigma_n^2 + 1e-8) I, dpotrf, dpotrs, logdet, LML) for a window
// that does not fit one SM.  Nothing in the reference runs at this size; the algorithm is the textbook blocked
// factorisation, organised for B200:
//
//  * storage: 8x8 FP64 tiles (the lane layout of cngp_common.cuh), column-tile-major: tile (rt, ct) at
//    A[(ct * row_tiles + rt) * 64].  For a fixed column tile the row tiles are contiguous, so a 16-tile operand slab
//    is ONE 8 KB bulk-TMA copy, and a warp reads/writes a C tile as one 512 B coalesced access.
//  * block columns of NB = 256 columns, dealt cyclically over `world` GPUs (1-D block-cyclic); y is carried as one
//    extra row tile under the matrix so z = L^-1 y falls out of the factorisation (as in gp_fit_kernel).
//  * per block column k (owner only): the 256x256 diagonal block is factored by gp_fit_kernel<KID_TILES> (the same
//    in-shared-memory tile Cholesky as the batched windows), inverted tile-wise (large_trinv_kernel), and the panel
//    below is formed as a product with the inverse - a GEMM, not a substitution.
//  * trailing update C -= P P^T (large_gemm_kernel, mode 1): the only dense contraction, N^3/3 flop.  128x128 C tiles
//    per CTA, 8 consumer warps x 32 accumulator tiles in registers (mma.sync m8n8k4 f64 - FP64 has no tcgen05 kind),
//    operands streamed through a 4-stage shared-memory ring by a producer warp issuing cp.async.bulk (UBLKCP) with
//    mbarrier completion; C is loaded straight into the accumulators before the main loop and stored once.
//  * predict pass (after the factorisation, reading only A, winv and alpha): W = L^-1 K(x, x*) as a forward sweep over
//    R = K(x*, x) in the same block-cyclic shape - the owner forms W_k with the panel product, every rank updates its
//    block columns of R with the same CTA body as the trailing update (cngp.h, cngp_large_predict_*).
//  * gradient pass (after the factorisation, reading the same A, winv and alpha): the predict sweep with R = I gives V = L^-T block column by block column,
//    and every rank accumulates its block columns of Ky^-1 = sum_k V_k V_k^T with the trailing update's kernel, then
//    contracts them against dK/dtheta evaluated in registers (cngp.h, cngp_large_grad_*).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <type_traits>
#include <vector>

#include "cngp_internal.h"
#include "gp_fit.cuh"
#include "gp_grad.cuh"

using namespace cngp;

namespace {

constexpr int LG_NB = CNGP_LARGE_NB;     // columns per block column
constexpr int LG_BT = LG_NB / 8;         // 32 tiles
constexpr int LG_BLK = 16;               // CTA tile edge in tiles (128 rows / columns)
constexpr int LG_KC = 2;                 // k-tiles per pipeline stage
constexpr int LG_STAGES = 4;
constexpr int LG_CONSUMERS = 8;
constexpr int LG_THREADS = LG_CONSUMERS * 32;
constexpr int LG_SLAB = LG_BLK * 64;     // doubles in a 16-tile slab (8 KB)
constexpr int LG_STAGE_DOUBLES = 2 * LG_KC * LG_SLAB;
constexpr size_t LG_SMEM = (size_t)LG_STAGES * LG_STAGE_DOUBLES * 8;

// ------------------------------------------------------------------------------------------------------------
// assembly
// ------------------------------------------------------------------------------------------------------------
struct AsmArgs {
  KProg kp;
  const double* theta;   // device [P]
  const double* x;       // device [N]
  const double* y;       // device [N]
  long long N, n_pad;
  long long row_tiles;
  int world, rank;
  double* A;
};

constexpr int ASM_WARPS = 8;
constexpr int ASM_TILES_PER_WARP = 8;

// grid (ceil(row_tiles / 64), local column tiles); each warp writes 8 consecutive row tiles of one column tile
template <int KID>
__global__ void __launch_bounds__(ASM_WARPS * 32) large_assemble_kernel(const AsmArgs a) {
  __shared__ LeafConst hc[CNGP_MAX_LEAVES];
  __shared__ KProg kps;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, r = lane >> 2, q = lane & 3;
  const long long lct = blockIdx.y;
  const long long c = (lct / LG_BT) * a.world + a.rank;          // global block column
  const long long gct = c * LG_BT + lct % LG_BT;                 // global column tile
  const long long NT = a.n_pad / 8;
  FastK<KID> fk;
  if (KID == KID_GENERIC) {
    if (threadIdx.x < a.kp.n_leaves)
      hc[threadIdx.x] = leaf_prepare(a.kp.leaf_type[threadIdx.x], a.theta + a.kp.leaf_param[threadIdx.x]);
    if (threadIdx.x == 0) kps = a.kp;
    __syncthreads();
  } else {
    fk.init(a.theta);
  }
  const double dadd = a.theta[a.kp.n_params] + CNGP_JITTER;
  const long long c0 = 8 * gct + 2 * q, c1 = c0 + 1;
  const double xc0 = c0 < a.N ? a.x[c0] : 0.0, xc1 = c1 < a.N ? a.x[c1] : 0.0;
  PointFeat f0{xc0, 0.0, 0.0, 0.0}, f1{xc1, 0.0, 0.0, 0.0};
  if (KID != KID_GENERIC) { f0 = fk.point(xc0); f1 = fk.point(xc1); }
  const long long first_rt = (gct / LG_BLK) * LG_BLK;            // whole diagonal 16x16 tile blocks are filled
  double* col = a.A + lct * a.row_tiles * 64;
  for (int t = 0; t < ASM_TILES_PER_WARP; ++t) {
    const long long rt = ((long long)blockIdx.x * ASM_WARPS + w) * ASM_TILES_PER_WARP + t;
    if (rt >= a.row_tiles || rt < first_rt) continue;            // storage is zero-filled beforehand
    tile2 v{0.0, 0.0};
    if (rt < NT) {
      const long long row = 8 * rt + r;
      if (row < a.N) {
        const double xr = a.x[row];
        if (KID == KID_GENERIC) {
          if (c0 < a.N) v.a = keval_generic_sym(&kps, hc, xr, xc0, row == c0);
          if (c1 < a.N) v.b = keval_generic_sym(&kps, hc, xr, xc1, row == c1);
        } else {
          const PointFeat fr = fk.point(xr);
          if (c0 < a.N) v.a = fk.eval(fr, f0, row == c0);
          if (c1 < a.N) v.b = fk.eval(fr, f1, row == c1);
        }
        if (row == c0) v.a += dadd;
        if (row == c1) v.b += dadd;
      } else {
        if (row == c0) v.a = 1.0;                                // identity padding
        if (row == c1) v.b = 1.0;
      }
    } else if (rt == NT) {
      if (r == 0) { v.a = c0 < a.N ? a.y[c0] : 0.0; v.b = c1 < a.N ? a.y[c1] : 0.0; }
    }
    tile_store(col + rt * 64, lane, v);
  }
}

// ------------------------------------------------------------------------------------------------------------
// inverse of the factored diagonal block: W = L^-1 as 32 x 32 tiles in [k-tile][row-tile] order (the Y operand
// layout of large_gemm_kernel), from the packed factor gp_fit_kernel writes (diagonal tiles already inverted).
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ tile2 tile_load_transposed(const double* tile, int lane) {
  const int r = lane >> 2, q = lane & 3;
  return tile2{tile[(2 * q) * 8 + r], tile[(2 * q + 1) * 8 + r]};
}

// One CTA per tile column j of X = L^-1, one warp per row tile i.  With WT(i,j) = X(i,j)^T:
//   WT(j,j) = inv(L_jj)^T,   WT(i,j) = -(sum_{k=j}^{i-1} WT(k,j) L(i,k)^T) inv(L_ii)^T.
// Right-looking inside the column: as soon as WT(k,j) is published (shared memory, double-buffered) every warp i > k
// adds its term WT(k,j) L(i,k)^T to the sum it keeps in registers, and warp k+1 - whose sum is then complete - finishes
// and publishes WT(k+1,j).  The dependent chain per step is two tile products and one CTA barrier; the L tiles are
// prefetched one step ahead.  (Round 1 ran all 32 columns on ONE CTA, two per warp, each step re-reading its column
// from global memory: 76 us on the serial panel chain of every block column; this is 32 CTAs and a few microseconds.)
constexpr int TRI_WARPS = LG_BT;
__global__ void __launch_bounds__(TRI_WARPS * 32) large_trinv_kernel(const double* __restrict__ Lp, double* __restrict__ W) {
  __shared__ __align__(16) double cur[2][64];
  constexpr int nt = LG_BT;
  const int lane = threadIdx.x & 31, i = threadIdx.x >> 5, j = blockIdx.x;
  const int r = lane >> 2, q = lane & 3;
  tile2 acc{0.0, 0.0}, mine{0.0, 0.0};
  if (i == j) {
    mine = tile_load_transposed(Lp + (long long)tile_index(j, j, nt) * 64, lane);
    tile_store(cur[0], lane, mine);
  }
  tile2 lnext{0.0, 0.0}, linv{0.0, 0.0};
  if (i > j) {
    lnext = tile_load(Lp + (long long)tile_index(i, j, nt) * 64, lane);
    linv = tile_load(Lp + (long long)tile_index(i, i, nt) * 64, lane);
  }
  __syncthreads();
  for (int k = j; k + 1 < nt; ++k) {
    if (i > k) {
      const tile2 lik = lnext;
      if (k + 1 < i) lnext = tile_load(Lp + (long long)tile_index(i, k + 1, nt) * 64, lane);
      tile_mma(acc, tile_load(cur[(k - j) & 1], lane), lik);
      if (i == k + 1) {
        const tile2 nT{-acc.a, -acc.b};
        tile_mma(mine, nT, linv);
        tile_store(cur[(k + 1 - j) & 1], lane, mine);
      }
    }
    __syncthreads();
  }
  // W tile (row tile i, k-tile j) = X(i,j) = WT(i,j)^T at W[(j * 32 + i) * 64]; zero above the diagonal
  double* out = W + ((long long)j * nt + i) * 64;
  out[(2 * q) * 8 + r] = mine.a;          // mine is zero for i < j
  out[(2 * q + 1) * 8 + r] = mine.b;
}

// ------------------------------------------------------------------------------------------------------------
// tile GEMM:  C(rt, ct) (-)= sum_k X(k, rt) Y(k, n)^T
// ------------------------------------------------------------------------------------------------------------
// Panel buffer layout.  A panel holds the rows below its diagonal block: row tiles r0 .. row_tiles, 32 k-tiles wide.
// It is cut into CHUNKS of rows at fixed absolute positions (every `cs` 16-tile row blocks, cs even; cs = 0: one chunk),
// each chunk stored compactly on its own - [k-tile][row tile of the chunk] - one after the other, so that a chunk is ONE
// contiguous range: the unit of the broadcast, of the panel GEMM and of the update of the next block column, which the
// driver pipelines chunk by chunk (large.py).  The chunk of row tile rt and where its tiles are:
struct PanelGeom {
  long long r0, row_tiles;
  int cs;                      // chunk size in 16-tile row blocks, 0 = single chunk
};
struct ChunkLoc { long long base, kstride; };   // tile (kt, rt) of the chunk at P + base + kt * kstride + rt * 64
__host__ __device__ inline int chunk_count_abs(long long row_tiles, int cs) {
  if (cs <= 0) return 1;
  const long long rb = row_tiles / LG_BLK;
  return rb / cs > 1 ? (int)(rb / cs) : 1;             // the last chunk takes the remainder
}
__host__ __device__ inline void chunk_rows(const PanelGeom& g, int chunk, long long& lo, long long& hi) {
  const int n = chunk_count_abs(g.row_tiles, g.cs);
  if (g.cs <= 0) { lo = g.r0; hi = g.row_tiles; return; }
  lo = (long long)chunk * g.cs * LG_BLK;
  hi = chunk == n - 1 ? g.row_tiles : (long long)(chunk + 1) * g.cs * LG_BLK;
  if (lo < g.r0) lo = g.r0;
  if (hi < lo) hi = lo;
}
__host__ __device__ inline int chunk_of(const PanelGeom& g, long long rt) {
  if (g.cs <= 0) return 0;
  const int n = chunk_count_abs(g.row_tiles, g.cs);
  const long long c = rt / ((long long)g.cs * LG_BLK);
  return (int)(c < n - 1 ? c : n - 1);
}
__host__ __device__ inline ChunkLoc chunk_loc(const PanelGeom& g, long long rt) {
  long long lo, hi;
  chunk_rows(g, chunk_of(g, rt), lo, hi);
  ChunkLoc c;
  c.kstride = (hi - lo) * 64;
  c.base = (long long)LG_BT * 64 * (lo - g.r0) - lo * 64;   // every chunk before this one holds 32 k-tiles of its rows
  return c;
}

struct GemmArgs {
  const double* X; long long x_kstride;   // X tile (k, rt) at X + k * x_kstride + rt * 64
  const double* Y; long long y_kstride;   // Y tile (k, n)  at Y + k * y_kstride + n * 64
  double* C;       long long c_cstride;   // C tile (rt, ct) at C + ct * c_cstride + rt * 64
  int mode;       // 0: C = X Y^T, Y lower-triangular inverse block (k-tiles up to the column block's last tile); C is
                  //    the panel buffer `panel` in the chunked layout `pg`
                  // 1: C -= X Y^T over all 32 k-tiles; column blocks are local block-cyclic, lower blocks only; X and Y
                  //    are both the panel buffer `panel` (layout `pg`)
  int rb0;        // first row block of the launch (units of 16 tiles); blockIdx.x counts from it
  int lcb0;       // mode 1: first local column block (units of 16 tiles); blockIdx.y counts from it
  int world, rank;
  double* panel;
  PanelGeom pg;
};

// One 16 x 16-tile block of C, rows rt0.. and columns ct0..:  C = sum_{k < KT} X(k, rt0..) Y(k, n0..)^T, or with `sub`
// C -= the same (C loaded into the accumulators first).  The CTA body of large_gemm_kernel and large_pred_update_kernel.
__device__ __forceinline__ void gemm_block(const double* Xb, long long xks, const double* Yb, long long yks, double* Cb,
                                           long long ccs, long long rt0, long long n0, long long ct0, int KT, bool sub,
                                           double* ring, unsigned long long* bars);

__global__ void __launch_bounds__(LG_THREADS, 1) large_gemm_kernel(const GemmArgs a) {
  extern __shared__ __align__(128) double ring[];
  __shared__ unsigned long long bars[2 * LG_STAGES];
  const long long rt0 = (long long)(a.rb0 + blockIdx.x) * LG_BLK;
  long long n0, ct0;
  int KT;
  if (a.mode == 0) {
    n0 = ct0 = (long long)blockIdx.y * LG_BLK;
    KT = ((int)blockIdx.y + 1) * LG_BLK;
  } else {
    const long long lct0 = (long long)(a.lcb0 + blockIdx.y) * LG_BLK;
    const long long c = (lct0 / LG_BT) * a.world + a.rank;
    n0 = c * LG_BT + lct0 % LG_BT;       // panel rows that face this column block
    ct0 = lct0;
    KT = LG_BT;
    if (rt0 < n0) return;                // block strictly above the diagonal
  }
  // operands: a 16-tile block never straddles two chunks of the panel (chunk boundaries are multiples of 16 tiles)
  const double *Xb, *Yb;
  long long xks, yks, ccs;
  double* Cb;
  if (a.mode == 0) {
    const ChunkLoc c = chunk_loc(a.pg, rt0);
    Xb = a.X; xks = a.x_kstride; Yb = a.Y; yks = a.y_kstride;
    Cb = a.panel + c.base; ccs = c.kstride;
  } else {
    const ChunkLoc cx = chunk_loc(a.pg, rt0), cy = chunk_loc(a.pg, n0);
    Xb = a.panel + cx.base; xks = cx.kstride;
    Yb = a.panel + cy.base; yks = cy.kstride;
    Cb = a.C; ccs = a.c_cstride;
  }
  gemm_block(Xb, xks, Yb, yks, Cb, ccs, rt0, n0, ct0, KT, a.mode == 1, ring, bars);
}

__device__ __forceinline__ void gemm_block(const double* Xb, long long xks, const double* Yb, long long yks, double* Cb,
                                           long long ccs, long long rt0, long long n0, long long ct0, int KT, bool sub,
                                           double* ring, unsigned long long* bars) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const uint32_t full_u32 = smem_u32(&bars[0]), empty_u32 = smem_u32(&bars[LG_STAGES]);
  if (tid == 0) {
    for (int s = 0; s < LG_STAGES; ++s) { mbar_init(full_u32 + 8 * s, 1); mbar_init(empty_u32 + 8 * s, LG_CONSUMERS); }
    mbar_fence_init();
  }
  __syncthreads();
  const int n_it = KT / LG_KC;
  const uint32_t ring_u32 = smem_u32(ring);
  // one lane streams the operand slabs of iteration `it`: LG_KC k-tiles of X and of Y into slot it % LG_STAGES
  auto issue = [&](int it) {
    const int s = it % LG_STAGES;
    mbar_expect_tx(full_u32 + 8 * s, LG_STAGE_DOUBLES * 8);
    const uint32_t dst = ring_u32 + s * LG_STAGE_DOUBLES * 8;
#pragma unroll
    for (int kk = 0; kk < LG_KC; ++kk) {
      const long long k = (long long)it * LG_KC + kk;
      bulk_g2s(dst + kk * LG_SLAB * 8, Xb + k * xks + rt0 * 64, LG_SLAB * 8, full_u32 + 8 * s);
      bulk_g2s(dst + (LG_KC + kk) * LG_SLAB * 8, Yb + k * yks + n0 * 64, LG_SLAB * 8, full_u32 + 8 * s);
    }
  };
  if (tid == 0)
    for (int it = 0; it < LG_STAGES - 1 && it < n_it; ++it) issue(it);

  // ---- consumers: warp (wr, wc) owns row tiles wr*8 .. +8 and column tiles wc*4 .. +4 of the block ----
  const int wr = w >> 2, wc = w & 3;
  tile2 acc[8][4];
  double* cbase = Cb + (ct0 + wc * 4) * ccs + (rt0 + wr * 8) * 64 + 2 * lane;
  if (sub) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const double2 v = *reinterpret_cast<const double2*>(cbase + j * ccs + i * 64);
        acc[i][j] = tile2{v.x, v.y};
      }
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i][j] = tile2{0.0, 0.0};
  }
  const bool neg = sub;
  for (int it = 0; it < n_it; ++it) {
    const int s = it % LG_STAGES;
    // refill duty rotates over the warps: the slot consumed at iteration it-1 gets iteration it + LG_STAGES - 1
    if (w == (it % LG_CONSUMERS) && lane == 0 && it + LG_STAGES - 1 < n_it) {
      if (it >= 1) mbar_wait(empty_u32 + 8 * ((it - 1) % LG_STAGES), (uint32_t)((it - 1) / LG_STAGES) & 1u);
      issue(it + LG_STAGES - 1);
    }
    __syncwarp();
    mbar_wait(full_u32 + 8 * s, (uint32_t)(it / LG_STAGES) & 1u);
    const double* xs = ring + s * LG_STAGE_DOUBLES + wr * 8 * 64 + 2 * lane;
    const double* ys = ring + s * LG_STAGE_DOUBLES + LG_KC * LG_SLAB + wc * 4 * 64 + 2 * lane;
#pragma unroll
    for (int kk = 0; kk < LG_KC; ++kk) {
      tile2 Yf[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double2 v = *reinterpret_cast<const double2*>(ys + kk * LG_SLAB + j * 64);
        Yf[j] = tile2{v.x, v.y};
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const double2 v = *reinterpret_cast<const double2*>(xs + kk * LG_SLAB + i * 64);
        const tile2 Xf = neg ? tile2{-v.x, -v.y} : tile2{v.x, v.y};
#pragma unroll
        for (int j = 0; j < 4; ++j) tile_mma(acc[i][j], Xf, Yf[j]);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_u32 + 8 * s);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 8; ++i)
      *reinterpret_cast<double2*>(cbase + j * ccs + i * 64) = make_double2(acc[i][j].a, acc[i][j].b);
}

// ------------------------------------------------------------------------------------------------------------
// z gather / reductions / back substitution / matvec
// ------------------------------------------------------------------------------------------------------------
// z[8 gct + c] = row 0 of tile (n_pad/8, lct); sums[0] = sum logdet of local blocks, sums[1] = sum z^2,
// sums[2] = first failing pivot (global, 1-based) or 0.  One CTA.
__global__ void __launch_bounds__(1024) large_reduce_kernel(const double* A, long long row_tiles, long long NT,
                                                            long long n_local_ct, int world, int rank,
                                                            const double* logdet, const int* status,
                                                            long long n_blockcols, double* z, double* sums) {
  __shared__ double red[32];
  double qs = 0.0;
  for (long long i = threadIdx.x; i < n_local_ct * 8; i += blockDim.x) {
    const long long lct = i / 8, cc = i % 8;
    const long long c = (lct / LG_BT) * world + rank;
    const long long gct = c * LG_BT + lct % LG_BT;
    const double v = A[(lct * row_tiles + NT) * 64 + cc];
    z[8 * gct + cc] = v;
    qs += v * v;
  }
  for (int o = 16; o; o >>= 1) qs += __shfl_xor_sync(0xffffffffu, qs, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = qs;
  __syncthreads();
  if (threadIdx.x == 0) {
    double ld = 0.0, fp = 0.0;
    for (long long k = rank; k < n_blockcols; k += world) {
      ld += logdet[k];
      if (status[k] < 0 && fp == 0.0) fp = (double)(k * LG_NB - status[k]);
    }
    double q2 = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) q2 += red[i];
    sums[0] = ld; sums[1] = q2; sums[2] = fp;
  }
}

// partial[chunk][c] = sum over this chunk's row tiles (below the diagonal block) of L(row, c) alpha(row)
constexpr int BACK_CHUNKS = 32;
__global__ void __launch_bounds__(256) large_back_partial_kernel(const double* Acol /* block column base */,
                                                                 long long row_tiles, long long rt_first, long long NT,
                                                                 const double* alpha, double* partial) {
  __shared__ double red[8][8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, r = lane >> 2, q = lane & 3;
  const int kt = blockIdx.x, chunk = blockIdx.y;
  const long long n_rt = NT - rt_first;
  const long long per = (n_rt + BACK_CHUNKS - 1) / BACK_CHUNKS;
  const long long lo = rt_first + chunk * per, hi = min(NT, lo + per);
  double s0 = 0.0, s1 = 0.0;
  for (long long rt = lo + w; rt < hi; rt += 8) {
    const double2 v = *reinterpret_cast<const double2*>(Acol + ((long long)kt * row_tiles + rt) * 64 + 2 * lane);
    const double al = alpha[8 * rt + r];
    s0 = fma(v.x, al, s0);
    s1 = fma(v.y, al, s1);
  }
  for (int o = 4; o < 32; o <<= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if (r == 0) { red[w][2 * q] = s0; red[w][2 * q + 1] = s1; }
  __syncthreads();
  if (threadIdx.x < 8) {
    double s = 0.0;
    for (int i = 0; i < 8; ++i) s += red[i][threadIdx.x];
    partial[chunk * LG_NB + kt * 8 + threadIdx.x] = s;
  }
}

// alpha_j = inv(L_jj)^T (z_j - sum_chunks partial).  1024 threads: column c of the 256 x 256 inverse is summed in four
// row segments of 64 (a single thread walking a whole column made this 39 us of pure load latency per block column -
// 5 ms of the 128-step backward sweep).
__device__ __forceinline__ void back_finish_block(const double* W, const double* zj, const double* partial, int nparts,
                                                  double* alpha_j, double* t, double (*seg_sum)[LG_NB]) {
  const int c = threadIdx.x % LG_NB, seg = threadIdx.x / LG_NB;
  if (seg == 0) {
    double s = zj[c];
    for (int ch = 0; ch < nparts; ++ch) s -= partial[ch * LG_NB + c];
    t[c] = s;
  }
  __syncthreads();
  // alpha[c] = sum_row W[row][c] t[row];  W element (row, c) is in tile (k-tile c/8, row tile row/8)
  const double* wt = W + (long long)(c / 8) * LG_BT * 64 + (c % 8);
  const int lo = max(c - (c % 8), seg * (LG_NB / 4)), hi = (seg + 1) * (LG_NB / 4);
  double acc = 0.0;
  for (int row = lo; row < hi; ++row) acc = fma(wt[(row / 8) * 64 + (row % 8) * 8], t[row], acc);
  seg_sum[seg][c] = acc;
  __syncthreads();
  if (seg == 0) alpha_j[c] = ((seg_sum[0][c] + seg_sum[1][c]) + seg_sum[2][c]) + seg_sum[3][c];
}

__global__ void __launch_bounds__(4 * LG_NB) large_back_finish_kernel(const double* W, const double* zj, const double* partial,
                                                                      int nparts, double* alpha_j) {
  __shared__ double t[LG_NB];
  __shared__ double seg_sum[4][LG_NB];
  back_finish_block(W, zj, partial, nparts, alpha_j, t, seg_sum);
}

// one warp: out[0..7] += sum over the 32 row tiles at `col` (consecutive tiles of one column tile) of tile^T alpha
__device__ __forceinline__ void back_apply_column_tile(const double* col, const double* al, double* out, int lane) {
  const int r = lane >> 2, q = lane & 3;
  col += 2 * lane;
  double s0 = 0.0, s1 = 0.0;
#pragma unroll 8
  for (int t = 0; t < LG_BT; ++t) {
    const double2 v = *reinterpret_cast<const double2*>(col + t * 64);
    const double a = al[8 * t + r];
    s0 = fma(v.x, a, s0);
    s1 = fma(v.y, a, s1);
  }
  for (int o = 4; o < 32; o <<= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if (r == 0) {
    out[2 * q] += s0;
    out[2 * q + 1] += s1;
  }
}

__global__ void __launch_bounds__(256) large_back_apply_kernel(const double* A, long long row_tiles, long long j,
                                                               long long n_lct, int world, int rank,
                                                               const double* alpha_j, double* s) {
  __shared__ double al[LG_NB];
  for (int i = threadIdx.x; i < LG_NB; i += blockDim.x) al[i] = alpha_j[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long lct = (long long)blockIdx.x * 8 + w;
  if (lct >= n_lct) return;
  const long long c = (lct / LG_BT) * world + rank;
  back_apply_column_tile(A + (lct * row_tiles + j * LG_BT) * 64, al, s + 8 * (c * LG_BT + lct % LG_BT), lane);
}

// r = Ky v with Ky evaluated on the fly; one warp per row
template <int KID>
__global__ void __launch_bounds__(256) large_matvec_kernel(KProg kp, const double* theta, const double* x,
                                                           const double* v, long long N, double* out) {
  __shared__ LeafConst hc[CNGP_MAX_LEAVES];
  __shared__ KProg kps;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  FastK<KID> fk;
  if (KID == KID_GENERIC) {
    if (threadIdx.x < kp.n_leaves) hc[threadIdx.x] = leaf_prepare(kp.leaf_type[threadIdx.x], theta + kp.leaf_param[threadIdx.x]);
    if (threadIdx.x == 0) kps = kp;
    __syncthreads();
  } else {
    fk.init(theta);
  }
  const long long row = (long long)blockIdx.x * 8 + w;
  if (row >= N) return;
  const double xr = x[row];
  PointFeat fr{xr, 0.0, 0.0, 0.0};
  if (KID != KID_GENERIC) fr = fk.point(xr);
  double s = 0.0;
  for (long long c = lane; c < N; c += 32) {
    const double xc = x[c];
    double k;
    if (KID == KID_GENERIC) k = keval_generic_sym(&kps, hc, xr, xc, row == c);
    else k = fk.eval(fr, fk.point(xc), row == c);
    if (row == c) k += theta[kp.n_params] + CNGP_JITTER;
    s = fma(k, v[c], s);
  }
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[row] = s;
}

// ------------------------------------------------------------------------------------------------------------
// predict pass over the stored factor: W = L^-1 K(x, x*) as a forward sweep on R = K(x*, x), block column by block column
// ------------------------------------------------------------------------------------------------------------
// R is stored like A but with m_tiles row tiles (test points, 8 per tile, padded to a multiple of 128 so that every GEMM
// block is whole): tile (mt, local column tile lct) at R[(lct * m_tiles + mt) * 64].  Rows m >= M and columns >= N are 0.
struct PredAsmArgs {
  KProg kp;
  const double* theta;   // device [P]
  const double* x;       // device [N]
  const double* xstar;   // device [M]
  long long N, M, m_tiles;
  long long lct0;        // first local column tile of the launch (blockIdx.y counts from it)
  int world, rank;
  double* R;
};

// grid (ceil(m_tiles / 8), local column tiles); one warp per tile
template <int KID>
__global__ void __launch_bounds__(256) large_pred_assemble_kernel(const PredAsmArgs a) {
  __shared__ LeafConst hc[CNGP_MAX_LEAVES];
  __shared__ KProg kps;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, r = lane >> 2, q = lane & 3;
  FastK<KID> fk;
  if (KID == KID_GENERIC) {
    if (threadIdx.x < a.kp.n_leaves)
      hc[threadIdx.x] = leaf_prepare(a.kp.leaf_type[threadIdx.x], a.theta + a.kp.leaf_param[threadIdx.x]);
    if (threadIdx.x == 0) kps = a.kp;
    __syncthreads();
  } else {
    fk.init(a.theta);                                             // phase origin 0, as large_assemble_kernel
  }
  const long long mt = (long long)blockIdx.x * 8 + w;
  if (mt >= a.m_tiles) return;
  const long long lct = a.lct0 + blockIdx.y;
  const long long gct = ((lct / LG_BT) * a.world + a.rank) * LG_BT + lct % LG_BT;
  const long long m = 8 * mt + r, c0 = 8 * gct + 2 * q, c1 = c0 + 1;
  tile2 v{0.0, 0.0};
  if (m < a.M) {
    const double xm = a.xstar[m];
    if (KID == KID_GENERIC) {
      if (c0 < a.N) v.a = keval_generic_cross(&kps, hc, a.x[c0], xm);
      if (c1 < a.N) v.b = keval_generic_cross(&kps, hc, a.x[c1], xm);
    } else {
      const PointFeat fm = fk.point(xm);
      if (c0 < a.N) v.a = fk.eval(fk.point(a.x[c0]), fm, false);
      if (c1 < a.N) v.b = fk.eval(fk.point(a.x[c1]), fm, false);
    }
  }
  tile_store(a.R + (lct * a.m_tiles + mt) * 64, lane, v);
}

// R(:, c) -= W_k L(c, k)^T for this rank's block columns c: grid (m_tiles / 16, local 16-tile column blocks).
// W tile (k-tile kt, test tile mt) at W + kt * w_kstride + mt * 64; L tile (kt, global row tile n) at Lp + kt * l_kstride
// + n * 64 (Lp is offset so that n counts from 0).
struct PredUpdArgs {
  const double* W; long long w_kstride;
  const double* Lp; long long l_kstride;
  double* R; long long r_cstride;
  int lcb0, world, rank;
};
__global__ void __launch_bounds__(LG_THREADS, 1) large_pred_update_kernel(const PredUpdArgs a) {
  extern __shared__ __align__(128) double ring[];
  __shared__ unsigned long long bars[2 * LG_STAGES];
  const long long lct0 = (long long)(a.lcb0 + blockIdx.y) * LG_BLK;
  const long long n0 = ((lct0 / LG_BT) * a.world + a.rank) * LG_BT + lct0 % LG_BT;
  gemm_block(a.W, a.w_kstride, a.Lp, a.l_kstride, a.R, a.r_cstride, (long long)blockIdx.x * LG_BLK, n0, lct0, LG_BT, true,
             ring, bars);
}

// s[m] = sum over the 256 columns of W_k of W(m, i)^2, in a fixed order; one warp per test tile
__global__ void __launch_bounds__(256) large_pred_sumsq_kernel(const double* W, long long m_tiles, long long M, double* s) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, r = lane >> 2, q = lane & 3;
  const long long mt = (long long)blockIdx.x * 8 + w;
  if (mt >= m_tiles) return;
  double acc = 0.0;
  for (int kt = 0; kt < LG_BT; ++kt) {
    const tile2 v = tile_load(W + (kt * m_tiles + mt) * 64, lane);
    acc = fma(v.a, v.a, acc);
    acc = fma(v.b, v.b, acc);
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  if (q == 0 && 8 * mt + r < M) s[8 * mt + r] = acc;
}

// mean[m] = K(x*_m, x) alpha (one warp per test point, large_matvec_kernel's order); var[m] = max(k(x*_m, x*_m) -
// sum_k s[k][m], 1e-15) + noise with the block sums added in increasing k
template <int KID>
__global__ void __launch_bounds__(256) large_pred_finish_kernel(KProg kp, const double* theta, const double* x,
                                                                const double* alpha, long long N, const double* xstar,
                                                                long long M, const double* s, long long n_blockcols,
                                                                double* mean, double* var) {
  __shared__ LeafConst hc[CNGP_MAX_LEAVES];
  __shared__ KProg kps;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  FastK<KID> fk;
  if (KID == KID_GENERIC) {
    if (threadIdx.x < kp.n_leaves) hc[threadIdx.x] = leaf_prepare(kp.leaf_type[threadIdx.x], theta + kp.leaf_param[threadIdx.x]);
    if (threadIdx.x == 0) kps = kp;
    __syncthreads();
  } else {
    fk.init(theta);
  }
  const long long m = (long long)blockIdx.x * 8 + w;
  if (m >= M) return;
  const double xm = xstar[m];
  PointFeat fm{xm, 0.0, 0.0, 0.0};
  if (KID != KID_GENERIC) fm = fk.point(xm);
  double acc = 0.0;
  for (long long c = lane; c < N; c += 32) {
    const double k = KID == KID_GENERIC ? keval_generic_cross(&kps, hc, x[c], xm) : fk.eval(fk.point(x[c]), fm, false);
    acc = fma(k, alpha[c], acc);
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    double vs = 0.0;
    for (long long k = 0; k < n_blockcols; ++k) vs += s[k * M + m];
    const double kss = KID == KID_GENERIC ? kdiag_eval(kps, hc, xm) : fk.kdiag(xm);
    mean[m] = acc;
    var[m] = fmax(kss - vs, CNGP_VAR_FLOOR) + theta[kp.n_params];
  }
}

// ------------------------------------------------------------------------------------------------------------
// LML gradient pass over the stored factor: V = L^-T as the forward sweep of the predict pass with R = I
// ------------------------------------------------------------------------------------------------------------
// RG is stored like A but with NT = n_pad/8 row tiles per column tile: tile (rt, lct) at RG[(lct * NT + rt) * 64].  Block
// column c holds R(:, c) until W_c = V_c is formed from it, and G(:, c) = -(sum_{k >= c} V_k V_k^T)(:, c) after that (kept
// negated so that the accumulation is the subtracting CTA body of the trailing update): the two never live at once.
constexpr int GRAD_STRIDE = CNGP_MAX_PARAMS + 1;    // one gradient row: kernel parameters, noise in the slot P - 1

// R = I on this rank's block columns (the storage is zero-filled beforehand); one thread per local column tile
__global__ void __launch_bounds__(256) large_grad_identity_kernel(double* RG, long long NT, long long n_lct, int world, int rank) {
  const long long lct = (long long)blockIdx.x * 256 + threadIdx.x;
  if (lct >= n_lct) return;
  const long long gct = ((lct / LG_BT) * world + rank) * LG_BT + lct % LG_BT;
  double* t = RG + (lct * NT + gct) * 64;
  for (int i = 0; i < 8; ++i) t[i * 9] = 1.0;
}

// One entry of dL/dK (weight wgt, mirrored entry included) against dK/dtheta at (xa, xb), gp_grad_kernel's sum and product
// rules: each leaf's derivatives times the values of the other leaves of its product term.  Expressions of up to
// GRAD_FAST_LEAVES leaves accumulate per leaf (gl), larger ones straight into the parameter slots (g).
__device__ __forceinline__ void large_grad_entry(const KProg& kp, const double* thv, const GradConst* gcs, const int* lt0,
                                                 const int* lt1, double wgt, double xa, double xb, double r2, bool same,
                                                 double (&gl)[GRAD_FAST_LEAVES][3], double (&g)[GRAD_STRIDE]) {
  if (kp.n_leaves <= GRAD_FAST_LEAVES) {
#pragma unroll
    for (int ul = 0; ul < GRAD_FAST_LEAVES; ++ul) {
      if (ul < kp.n_leaves) {
        double others = 1.0, dv[3];
        for (int u2 = lt0[ul]; u2 < lt1[ul]; ++u2)
          if (u2 != ul) others *= leaf_value_grad_c<true>(kp.leaf_type[u2], thv + kp.leaf_param[u2], gcs[u2], xa, xb, r2, same, dv);
        leaf_value_grad_c<true>(kp.leaf_type[ul], thv + kp.leaf_param[ul], gcs[ul], xa, xb, r2, same, dv);
        const double ww = wgt * others;
        gl[ul][0] += ww * dv[0]; gl[ul][1] += ww * dv[1]; gl[ul][2] += ww * dv[2];
      }
    }
  } else {
    for (int u = 0; u < kp.n_leaves; ++u) {
      double others = 1.0, dv[3];
      for (int u2 = lt0[u]; u2 < lt1[u]; ++u2)
        if (u2 != u) others *= leaf_value_grad_c<true>(kp.leaf_type[u2], thv + kp.leaf_param[u2], gcs[u2], xa, xb, r2, same, dv);
      leaf_value_grad_c<true>(kp.leaf_type[u], thv + kp.leaf_param[u], gcs[u], xa, xb, r2, same, dv);
      const int np = leaf_nparams(kp.leaf_type[u]), po = kp.leaf_param[u];
      const double ww = wgt * others;
#pragma unroll
      for (int i = 0; i < CNGP_MAX_PARAMS; ++i) {
        const int jj = i - po;
        if (jj >= 0 && jj < np) g[i] += ww * (jj == 0 ? dv[0] : (jj == 1 ? dv[1] : dv[2]));
      }
    }
  }
}

// partial[lct][p] = sum over the entries i >= j (i, j < N) of local column tile lct of  w_ij dK_ij/dtheta_p,
// w_ij = alpha_i alpha_j + G_ij (G = -Ky^-1), doubled off the diagonal; the noise slot gets the diagonal weights.
// One CTA per column tile, warp w takes row tiles gct + w, gct + w + 8, ...; the sums are reduced in a fixed order.
constexpr int GC_WARPS = 8;
__global__ void __launch_bounds__(GC_WARPS * 32) large_grad_contract_kernel(const KProg kp, const double* theta, const double* x,
                                                                            const double* alpha, const double* RG, long long N,
                                                                            long long NT, int world, int rank, double* partial) {
  __shared__ double thv[GRAD_STRIDE];
  __shared__ GradConst gcs[CNGP_MAX_LEAVES];
  __shared__ int lt0[CNGP_MAX_LEAVES], lt1[CNGP_MAX_LEAVES];
  __shared__ double gred[GC_WARPS][GRAD_STRIDE];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, r = lane >> 2, q = lane & 3;
  const int P = kp.n_params + 1;
  if (tid < P) thv[tid] = theta[tid];
  if (tid < kp.n_leaves) gcs[tid] = grad_prepare(kp.leaf_type[tid], theta + kp.leaf_param[tid]);
  if (tid < kp.n_terms)
    for (int u = kp.term_start[tid]; u < kp.term_start[tid + 1]; ++u) { lt0[u] = kp.term_start[tid]; lt1[u] = kp.term_start[tid + 1]; }
  __syncthreads();
  const long long lct = blockIdx.x;
  const long long gct = ((lct / LG_BT) * world + rank) * LG_BT + lct % LG_BT;
  double g[GRAD_STRIDE];
#pragma unroll
  for (int i = 0; i < GRAD_STRIDE; ++i) g[i] = 0.0;
  double gl[GRAD_FAST_LEAVES][3];
#pragma unroll
  for (int i = 0; i < GRAD_FAST_LEAVES; ++i) gl[i][0] = gl[i][1] = gl[i][2] = 0.0;
  const long long j0 = 8 * gct + 2 * q;
  const double xb0 = j0 < N ? x[j0] : 0.0, xb1 = j0 + 1 < N ? x[j0 + 1] : 0.0;
  const double ab0 = j0 < N ? alpha[j0] : 0.0, ab1 = j0 + 1 < N ? alpha[j0 + 1] : 0.0;
  const long long rt_end = min(NT, (N + 7) / 8);
  for (long long rt = gct + w; rt < rt_end; rt += GC_WARPS) {
    const double2 v = *reinterpret_cast<const double2*>(RG + (lct * NT + rt) * 64 + 2 * lane);
    const long long i = 8 * rt + r;
    if (i >= N) continue;
    const double xa = x[i], ai = alpha[i];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const long long j = j0 + e;
      if (j > i || j >= N) continue;
      const bool same = i == j;
      double wgt = ai * (e ? ab1 : ab0) + (e ? v.y : v.x);
      if (!same) wgt += wgt;
      const double xb = e ? xb1 : xb0;
      const double r2 = same ? 0.0 : r2_expanded(xa, xb);
      if (same) g[CNGP_MAX_PARAMS] += wgt;                 // noise: trace(dL_dK)
      large_grad_entry(kp, thv, gcs, lt0, lt1, wgt, xa, xb, r2, same, gl, g);
    }
  }
  if (kp.n_leaves <= GRAD_FAST_LEAVES) {
#pragma unroll
    for (int ul = 0; ul < GRAD_FAST_LEAVES; ++ul) {
      if (ul < kp.n_leaves) {
        const int np = leaf_nparams(kp.leaf_type[ul]), po = kp.leaf_param[ul];
#pragma unroll
        for (int i = 0; i < CNGP_MAX_PARAMS; ++i) {
          const int jj = i - po;
          if (jj >= 0 && jj < np) g[i] += (jj == 0 ? gl[ul][0] : (jj == 1 ? gl[ul][1] : gl[ul][2]));
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < GRAD_STRIDE; ++i) {
    double v = g[i];
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) gred[w][i] = v;
  }
  __syncthreads();
  if (tid < GRAD_STRIDE) {
    double v = 0.0;
    if (tid < P) {
      const int src = tid == P - 1 ? CNGP_MAX_PARAMS : tid;
      for (int ww = 0; ww < GC_WARPS; ++ww) v += gred[ww][src];
    }
    partial[lct * GRAD_STRIDE + tid] = v;
  }
}

// part[c][p] = sum over the 32 column tiles of this rank's block column c of partial, in increasing column tile
__global__ void __launch_bounds__(32) large_grad_part_kernel(const double* partial, int world, int rank, double* part) {
  const long long l = blockIdx.x, c = l * world + rank;
  const int p = threadIdx.x;
  if (p >= GRAD_STRIDE) return;
  double s = 0.0;
  for (int t = 0; t < LG_BT; ++t) s += partial[(l * LG_BT + t) * GRAD_STRIDE + p];
  part[c * GRAD_STRIDE + p] = s;
}

// grad[p] = 1/2 sum_c part[c][p], c increasing
__global__ void __launch_bounds__(32) large_grad_finish_kernel(const double* part, long long n_blockcols, int P, double* grad) {
  const int p = threadIdx.x;
  if (p >= P) return;
  double s = 0.0;
  for (long long c = 0; c < n_blockcols; ++c) s += part[c * GRAD_STRIDE + p];
  grad[p] = 0.5 * s;
}

template <typename F>
void dispatch_kid(int kid, F&& f) {
  switch (kid) {
    case KID_RBF: f(std::integral_constant<int, KID_RBF>()); break;
    case KID_RBF_PER: f(std::integral_constant<int, KID_RBF_PER>()); break;
    case KID_RBF_BROWN: f(std::integral_constant<int, KID_RBF_BROWN>()); break;
    default: f(std::integral_constant<int, KID_GENERIC>()); break;
  }
}

int cuda_fail(cngp_ctx* ctx, const char* what, cudaError_t e) {
  char tmp[256];
  snprintf(tmp, sizeof tmp, "%s: %s", what, cudaGetErrorString(e));
  return cngp_set_error(ctx, CNGP_ERR_CUDA, tmp);
}
#define LCU(ctx, call)                                        \
  do {                                                        \
    cudaError_t e_ = (call);                                  \
    if (e_ != cudaSuccess) return cuda_fail(ctx, #call, e_);  \
  } while (0)

// scratch slots of the context used here
enum { SLOT_THETA = 20, SLOT_LPACK = 21, SLOT_WT = 22, SLOT_Z33 = 23, SLOT_PARTIAL = 24, SLOT_GPART = 25 };

inline PanelGeom panel_geom(const cngp_large_plan* p, long long k) {
  PanelGeom g;
  g.r0 = (k + 1) * LG_BT;
  g.row_tiles = p->row_tiles;
  g.cs = (int)p->chunk_blocks;
  return g;
}

inline long long local_index_of(long long c_lo, int world, int rank) {   // smallest l with l*world + rank >= c_lo
  if (c_lo <= rank) return 0;
  return (c_lo - rank + world - 1) / world;
}

}  // namespace

extern "C" int cngp_large_make_plan(int64_t N, int32_t world, int32_t rank, cngp_large_plan* p) {
  if (!p || N <= 0 || world <= 0 || rank < 0 || rank >= world) return CNGP_ERR_INVALID;
  memset(p, 0, sizeof *p);     // chunk_blocks = 0: panels in one piece (the caller may set it, see cngp.h)
  p->N = N;
  p->n_pad = (N + LG_NB - 1) / LG_NB * LG_NB;
  p->world = world;
  p->rank = rank;
  p->row_tiles = p->n_pad / 8 + LG_BLK;
  p->n_blockcols = p->n_pad / LG_NB;
  p->n_local_blockcols = p->n_blockcols > rank ? (p->n_blockcols - rank + world - 1) / world : 0;
  p->local_doubles = p->n_local_blockcols * LG_BT * p->row_tiles * 64;
  p->panel_doubles = (int64_t)LG_BT * p->row_tiles * 64;
  p->winv_doubles = p->n_local_blockcols * LG_BT * LG_BT * 64;
  return CNGP_OK;
}

extern "C" int cngp_large_assemble(cngp_ctx* ctx, const cngp_large_plan* p, const cngp_kernel* kernel, const double* theta,
                                   const double* x, const double* y, double* A) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !kernel || !theta || !x || !y || !A) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_assemble: bad argument");
  KProg kp;
  int rc = cngp_build_kprog(kernel, &kp);
  if (rc) return cngp_set_error(ctx, rc, "large_assemble: invalid kernel expression");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  const int P = kp.n_params + 1;
  double* d_theta = (double*)cngp_ctx_buf(ctx, SLOT_THETA, sizeof(double) * (CNGP_MAX_PARAMS + 1));
  if (!d_theta) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "large_assemble: theta buffer");
  LCU(ctx, cudaMemcpyAsync(d_theta, theta, sizeof(double) * P, cudaMemcpyHostToDevice, s));
  LCU(ctx, cudaStreamSynchronize(s));   // theta is a host stack/array of the caller
  if (p->n_local_blockcols == 0) return CNGP_OK;
  LCU(ctx, cudaMemsetAsync(A, 0, sizeof(double) * (size_t)p->local_doubles, s));
  AsmArgs a;
  a.kp = kp; a.theta = d_theta; a.x = x; a.y = y; a.N = p->N; a.n_pad = p->n_pad; a.row_tiles = p->row_tiles;
  a.world = p->world; a.rank = p->rank; a.A = A;
  const long long n_local_ct = p->n_local_blockcols * LG_BT;
  const int per_cta = ASM_WARPS * ASM_TILES_PER_WARP;
  // grid.y is limited to 65535: launch in slices of column tiles
  for (long long y0 = 0; y0 < n_local_ct; y0 += 32768) {
    const long long ny = std::min<long long>(32768, n_local_ct - y0);
    AsmArgs as = a;
    as.A = A + y0 * p->row_tiles * 64;
    // the kernel derives the global column from blockIdx.y, so slices must start on a block-column boundary
    // (32768 is a multiple of 32) and carry their offset through `rank`-relative arithmetic:
    const long long l0 = y0 / LG_BT;
    as.rank = (int)(p->rank + l0 * p->world);   // (lct / 32) * world + rank  ==  ((lct + y0) / 32) * world + p->rank
    dim3 grid((unsigned)((p->row_tiles + per_cta - 1) / per_cta), (unsigned)ny);
    cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
    dispatch_kid(match_fast_kernel(kp), [&](auto kid) {
      large_assemble_kernel<decltype(kid)::value><<<grid, ASM_WARPS * 32, 0, s>>>(as);
    });
    cngp_ctx_end(ctx);
  }
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_factor_panel(cngp_ctx* ctx, const cngp_large_plan* p, double* A, int64_t k, double* panel,
                                       double* winv, double* logdet, int32_t* status) {
  return cngp_large_factor_panel_ex(ctx, p, A, k, panel, winv, logdet, status, 0, -1);
}

// 4. of cngp_large_factor_panel on its own: the panel is this block column of L - copy it back under the diagonal block.
// Nothing before the backward sweep reads it there, so the two-stream driver takes it off the panel chain.
extern "C" int cngp_large_copy_back(cngp_ctx* ctx, const cngp_large_plan* p, double* A, int64_t k, const double* panel) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !A || !panel || k < 0 || k >= p->n_blockcols) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_copy_back: bad argument");
  if (k % p->world != p->rank) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_copy_back: not the owner of this block column");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  const long long l = k / p->world, cstride = p->row_tiles * 64;
  double* Acol = A + l * LG_BT * cstride;
  const PanelGeom pg = panel_geom(p, k);
  for (int c = chunk_of(pg, pg.r0); c < chunk_count_abs(pg.row_tiles, pg.cs); ++c) {
    long long lo, hi;
    chunk_rows(pg, c, lo, hi);
    if (hi <= lo) continue;
    const ChunkLoc loc = chunk_loc(pg, lo);
    LCU(ctx, cudaMemcpy2DAsync(Acol + lo * 64, cstride * 8, panel + loc.base + lo * 64, loc.kstride * 8, (size_t)(hi - lo) * 512,
                               LG_BT, cudaMemcpyDeviceToDevice, cngp_ctx_stream(ctx)));
  }
  return CNGP_OK;
}

// Live chunks of panel k: *first = absolute id of the first one, *count = how many, offsets[0 .. count] = where each starts
// in the panel buffer (doubles; offsets[count] = end of the payload).  offsets must hold CNGP_LARGE_MAX_CHUNKS + 1 entries.
extern "C" int cngp_large_panel_chunks(const cngp_large_plan* p, int64_t k, int32_t* first, int32_t* count, int64_t* offsets) {
  if (!p || !first || !count || !offsets || k < 0 || k >= p->n_blockcols) return CNGP_ERR_INVALID;
  const PanelGeom pg = panel_geom(p, k);
  const int n = chunk_count_abs(pg.row_tiles, pg.cs);
  if (n > CNGP_LARGE_MAX_CHUNKS) return CNGP_ERR_INVALID;
  const int c0 = chunk_of(pg, pg.r0);
  *first = c0;
  int m = 0;
  for (int c = c0; c < n; ++c) {
    long long lo, hi;
    chunk_rows(pg, c, lo, hi);
    offsets[m++] = (long long)LG_BT * 64 * (lo - pg.r0);
    if (c == n - 1) offsets[m] = (long long)LG_BT * 64 * (hi - pg.r0);
  }
  *count = m;
  return CNGP_OK;
}

extern "C" int cngp_large_factor_panel_ex(cngp_ctx* ctx, const cngp_large_plan* p, double* A, int64_t k, double* panel,
                                          double* winv, double* logdet, int32_t* status, int32_t flags, int32_t chunk) {
  if (!ctx) return CNGP_ERR_INVALID;
  const bool defer_copy_back = flags & CNGP_LARGE_DEFER_COPY, do_diag = !(flags & CNGP_LARGE_PANEL_ONLY), do_panel = !(flags & CNGP_LARGE_DIAG_ONLY);
  if (!p || !A || !panel || !winv || !logdet || !status || k < 0 || k >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_factor_panel: bad argument");
  if (k % p->world != p->rank) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_factor_panel: not the owner of this block column");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  const long long l = k / p->world;
  const long long cstride = p->row_tiles * 64;
  double* Acol = A + l * LG_BT * cstride;                 // block column k
  const long long rdiag = k * LG_BT;                      // first row tile of the diagonal block
  double* Lpack = (double*)cngp_ctx_buf(ctx, SLOT_LPACK, sizeof(double) * tiles_in_lower(LG_BT) * 64);
  double* z33 = (double*)cngp_ctx_buf(ctx, SLOT_Z33, sizeof(double) * (LG_NB + 8));
  if (!Lpack || !z33) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "large_factor_panel: scratch");
  double* Wk = winv + l * LG_BT * LG_BT * 64;

  if (do_diag) {
  // 1. diagonal block: tile Cholesky in shared memory (diagonal tiles come out inverted)
  FitArgs fa;
  memset(&fa, 0, sizeof fa);
  fa.theta = nullptr; fa.theta_stride = 0; fa.theta_mode = 0; fa.win_map = nullptr;
  fa.x = nullptr; fa.y = nullptr; fa.N = LG_NB; fa.nt = LG_BT; fa.n_windows = 1; fa.problem0 = 0;
  fa.L = Lpack; fa.z = z33; fa.feat = nullptr; fa.lml = nullptr; fa.logdet = logdet + k; fa.quad = nullptr;
  fa.status = status + k; fa.jitter_retry = 0;
  fa.Asrc = Acol + rdiag * 64; fa.a_col_stride = cstride;
  // logdet / status are indexed by the kernel with the problem id p = problem0 + blockIdx.x = 0
  const size_t smem = fit_smem_bytes(LG_BT, FIT_NW_FULL * FIT_T_FULL);
  LCU(ctx, cudaFuncSetAttribute(gp_fit_kernel<KID_TILES, FIT_NW_FULL, FIT_T_FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  gp_fit_kernel<KID_TILES, FIT_NW_FULL, FIT_T_FULL><<<1, (FIT_NW_FULL + 1) * 32, smem, s>>>(fa);   // workers + the diagonal warp
  cngp_ctx_end(ctx);
  // 2. inverse of the block factor
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_trinv_kernel<<<LG_BT, TRI_WARPS * 32, 0, s>>>(Lpack, Wk);
  cngp_ctx_end(ctx);
  }
  if (!do_panel) { LCU(ctx, cudaGetLastError()); return CNGP_OK; }
  // 3. panel = (rows below the diagonal block) inv(L_kk)^T, all of it or the rows of one chunk (chunk >= 0: absolute id)
  const PanelGeom pg = panel_geom(p, k);
  long long lo = pg.r0, hi = p->row_tiles;
  if (chunk >= 0) {
    if (chunk >= chunk_count_abs(pg.row_tiles, pg.cs)) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_factor_panel: no such chunk");
    chunk_rows(pg, chunk, lo, hi);
  }
  if (hi > lo) {
    GemmArgs g;
    memset(&g, 0, sizeof g);
    g.X = Acol; g.x_kstride = cstride;
    g.Y = Wk; g.y_kstride = (long long)LG_BT * 64;
    g.panel = panel; g.pg = pg;
    g.mode = 0; g.rb0 = (int)(lo / LG_BLK); g.lcb0 = 0; g.world = p->world; g.rank = p->rank;
    LCU(ctx, cudaFuncSetAttribute(large_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_SMEM));
    cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
    large_gemm_kernel<<<dim3((unsigned)((hi - lo) / LG_BLK), LG_BT / LG_BLK), LG_THREADS, LG_SMEM, s>>>(g);
    cngp_ctx_end(ctx);
  }
  LCU(ctx, cudaGetLastError());
  // 4. the panel is this block column of L: copy it back under the diagonal block (or leave that to cngp_large_copy_back)
  if (!defer_copy_back) return cngp_large_copy_back(ctx, p, A, k, panel);
  return CNGP_OK;
}

extern "C" int cngp_large_update(cngp_ctx* ctx, const cngp_large_plan* p, double* A, int64_t k, const double* panel,
                                 int64_t c_lo, int64_t c_hi) {
  return cngp_large_update_part(ctx, p, A, k, panel, c_lo, c_hi, CNGP_LARGE_ROWS_ALL, -1);
}

// rows: CNGP_LARGE_ROWS_ALL, or - for ONE block column - only its diagonal block (so that the block can be factored while
// the rows below are still being updated on another stream) / only the rows below it.
extern "C" int cngp_large_update_part(cngp_ctx* ctx, const cngp_large_plan* p, double* A, int64_t k, const double* panel,
                                      int64_t c_lo, int64_t c_hi, int32_t rows, int32_t chunk) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !A || !panel || k < 0 || k >= p->n_blockcols) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_update: bad argument");
  c_lo = std::max<int64_t>(c_lo, k + 1);
  c_hi = std::min<int64_t>(c_hi, p->n_blockcols);
  if (c_lo >= c_hi) return CNGP_OK;
  const long long l_lo = local_index_of(c_lo, p->world, p->rank), l_hi = local_index_of(c_hi, p->world, p->rank);
  if (l_lo >= l_hi) return CNGP_OK;
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  const long long cstride = p->row_tiles * 64;
  const int RB = (int)(p->row_tiles / LG_BLK);
  const long long c_first = l_lo * p->world + p->rank;
  const int rb0 = (int)(c_first * LG_BT / LG_BLK);
  const PanelGeom pg = panel_geom(p, k);
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.panel = const_cast<double*>(panel); g.pg = pg;
  g.C = A; g.c_cstride = cstride;
  g.mode = 1; g.rb0 = rb0; g.world = p->world; g.rank = p->rank;
  LCU(ctx, cudaFuncSetAttribute(large_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_SMEM));
  const long long ncb = (l_hi - l_lo) * (LG_BT / LG_BLK);
  int rb_first = rb0, rb_count = RB - rb0;
  if (rows != CNGP_LARGE_ROWS_ALL || chunk >= 0) {
    if (l_hi - l_lo != 1) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_update_part: a row part needs exactly one block column");
    const int diag_blocks = LG_BT / LG_BLK;
    if (rows == CNGP_LARGE_ROWS_DIAG) rb_count = diag_blocks;
    else if (rows == CNGP_LARGE_ROWS_BELOW) { rb_first = rb0 + diag_blocks; rb_count = RB - rb_first; }
    if (chunk >= 0) {        // ... intersected with the rows of one chunk of the panel
      if (chunk >= chunk_count_abs(pg.row_tiles, pg.cs)) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_update_part: no such chunk");
      long long lo, hi;
      chunk_rows(pg, chunk, lo, hi);
      const int b_lo = std::max<int>(rb_first, (int)(lo / LG_BLK)), b_hi = std::min<int>(rb_first + rb_count, (int)(hi / LG_BLK));
      rb_first = b_lo; rb_count = b_hi - b_lo;
    }
    if (rb_count <= 0) return CNGP_OK;
    g.rb0 = rb_first;
  }
  for (long long y0 = 0; y0 < ncb; y0 += 65535) {
    g.lcb0 = (int)(l_lo * (LG_BT / LG_BLK) + y0);
    const unsigned ny = (unsigned)std::min<long long>(65535, ncb - y0);
    cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
    large_gemm_kernel<<<dim3((unsigned)rb_count, ny), LG_THREADS, LG_SMEM, s>>>(g);
    cngp_ctx_end(ctx);
  }
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_reduce(cngp_ctx* ctx, const cngp_large_plan* p, const double* A, const double* logdet,
                                 const int32_t* status, double* z, double* sums) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !A || !logdet || !status || !z || !sums) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_reduce: bad argument");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  LCU(ctx, cudaMemsetAsync(z, 0, sizeof(double) * (size_t)p->n_pad, s));
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_reduce_kernel<<<1, 1024, 0, s>>>(A, p->row_tiles, p->n_pad / 8, p->n_local_blockcols * LG_BT, p->world, p->rank,
                                         logdet, status, p->n_blockcols, z, sums);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_backsolve_step(cngp_ctx* ctx, const cngp_large_plan* p, const double* A, const double* winv,
                                         int64_t j, const double* z, double* alpha) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !A || !winv || !z || !alpha || j < 0 || j >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_backsolve_step: bad argument");
  if (j % p->world != p->rank) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_backsolve_step: not the owner");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  double* partial = (double*)cngp_ctx_buf(ctx, SLOT_PARTIAL, sizeof(double) * BACK_CHUNKS * LG_NB);
  if (!partial) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "large_backsolve_step: scratch");
  const long long l = j / p->world;
  const long long cstride = p->row_tiles * 64;
  const double* Acol = A + l * LG_BT * cstride;
  const long long NT = p->n_pad / 8;
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_back_partial_kernel<<<dim3(LG_BT, BACK_CHUNKS), 256, 0, s>>>(Acol, p->row_tiles, (j + 1) * LG_BT, NT, alpha, partial);
  cngp_ctx_end(ctx);
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_back_finish_kernel<<<1, 4 * LG_NB, 0, s>>>(winv + l * LG_BT * LG_BT * 64, z + j * LG_NB, partial, BACK_CHUNKS, alpha + j * LG_NB);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

// The lazy backward sweep (see large_back_apply_kernel), last block column first:
//   owner of j:  cngp_large_backsolve_finish  alpha_j = inv(L_jj)^T (z_j - s_j)      -> broadcast alpha_j
//   every rank:  cngp_large_backsolve_apply   s_c += L(block row j, c)^T alpha_j for its block columns c < j
// s [n_pad] starts as zeros.
extern "C" int cngp_large_backsolve_finish(cngp_ctx* ctx, const cngp_large_plan* p, const double* winv, int64_t j,
                                           const double* z, const double* s_acc, double* alpha) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !winv || !z || !s_acc || !alpha || j < 0 || j >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_backsolve_finish: bad argument");
  if (j % p->world != p->rank) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_backsolve_finish: not the owner");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  const long long l = j / p->world;
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_back_finish_kernel<<<1, 4 * LG_NB, 0, cngp_ctx_stream(ctx)>>>(winv + l * LG_BT * LG_BT * 64, z + j * LG_NB,
                                                                      s_acc + j * LG_NB, 1, alpha + j * LG_NB);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_backsolve_apply(cngp_ctx* ctx, const cngp_large_plan* p, const double* A, int64_t j,
                                          const double* alpha, double* s_acc) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !A || !alpha || !s_acc || j < 0 || j >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_backsolve_apply: bad argument");
  const long long n_lct = local_index_of(j, p->world, p->rank) * LG_BT;     // local column tiles of block columns < j
  if (n_lct <= 0) return CNGP_OK;
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_back_apply_kernel<<<(unsigned)((n_lct + 7) / 8), 256, 0, cngp_ctx_stream(ctx)>>>(A, p->row_tiles, j, n_lct, p->world,
                                                                                      p->rank, alpha + j * LG_NB, s_acc);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_matvec(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x,
                                 const double* v, int64_t N, double* r) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !theta || !x || !v || !r || N <= 0) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_matvec: bad argument");
  KProg kp;
  int rc = cngp_build_kprog(kernel, &kp);
  if (rc) return cngp_set_error(ctx, rc, "large_matvec: invalid kernel expression");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  double* d_theta = (double*)cngp_ctx_buf(ctx, SLOT_THETA, sizeof(double) * (CNGP_MAX_PARAMS + 1));
  if (!d_theta) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "large_matvec: theta buffer");
  LCU(ctx, cudaMemcpyAsync(d_theta, theta, sizeof(double) * (kp.n_params + 1), cudaMemcpyHostToDevice, s));
  LCU(ctx, cudaStreamSynchronize(s));
  cngp_ctx_begin(ctx, CNGP_PROF_MISC);
  dispatch_kid(match_fast_kernel(kp), [&](auto kid) {
    large_matvec_kernel<decltype(kid)::value><<<(unsigned)((N + 7) / 8), 256, 0, s>>>(kp, d_theta, x, v, N, r);
  });
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

// ------------------------------------------------------------------------------------------------------------
// predict pass (see cngp.h): R = K(x*, x) swept forward through the stored factor
// ------------------------------------------------------------------------------------------------------------
namespace {
inline long long pred_m_tiles(int64_t M) { return (M + 8 * LG_BLK - 1) / (8 * LG_BLK) * LG_BLK; }
inline long long pred_payload_doubles(const cngp_large_plan* p, long long m_tiles, int64_t k) {
  return (long long)LG_BT * 64 * (m_tiles + p->n_pad / 8 - (k + 1) * LG_BT);
}
int upload_theta(cngp_ctx* ctx, const KProg& kp, const double* theta, double** d_theta, const char* what) {
  *d_theta = (double*)cngp_ctx_buf(ctx, SLOT_THETA, sizeof(double) * (CNGP_MAX_PARAMS + 1));
  if (!*d_theta) return cngp_set_error(ctx, CNGP_ERR_NOMEM, what);
  cudaStream_t s = cngp_ctx_stream(ctx);
  LCU(ctx, cudaMemcpyAsync(*d_theta, theta, sizeof(double) * (kp.n_params + 1), cudaMemcpyHostToDevice, s));
  LCU(ctx, cudaStreamSynchronize(s));   // theta is a host stack/array of the caller
  return CNGP_OK;
}
}  // namespace

extern "C" int cngp_large_predict_sizes(const cngp_large_plan* p, int64_t M, int64_t k, int64_t* r_doubles,
                                        int64_t* payload_doubles, int64_t* s_doubles) {
  if (!p || M <= 0 || k < 0 || k >= p->n_blockcols) return CNGP_ERR_INVALID;
  const long long mt = pred_m_tiles(M);
  if (r_doubles) *r_doubles = p->n_local_blockcols * LG_BT * mt * 64;
  if (payload_doubles) *payload_doubles = pred_payload_doubles(p, mt, k);
  if (s_doubles) *s_doubles = p->n_blockcols * M;
  return CNGP_OK;
}

extern "C" int cngp_large_predict_assemble(cngp_ctx* ctx, const cngp_large_plan* p, const cngp_kernel* kernel,
                                           const double* theta, const double* x, const double* xstar, int64_t M, double* R) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !kernel || !theta || !x || !xstar || !R || M <= 0)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_predict_assemble: bad argument");
  KProg kp;
  int rc = cngp_build_kprog(kernel, &kp);
  if (rc) return cngp_set_error(ctx, rc, "large_predict_assemble: invalid kernel expression");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  double* d_theta;
  if ((rc = upload_theta(ctx, kp, theta, &d_theta, "large_predict_assemble: theta buffer"))) return rc;
  PredAsmArgs a;
  a.kp = kp; a.theta = d_theta; a.x = x; a.xstar = xstar; a.N = p->N; a.M = M; a.m_tiles = pred_m_tiles(M);
  a.world = p->world; a.rank = p->rank; a.R = R;
  const long long n_local_ct = p->n_local_blockcols * LG_BT;
  for (long long y0 = 0; y0 < n_local_ct; y0 += 65535) {      // grid.y is limited to 65535
    a.lct0 = y0;
    const dim3 grid((unsigned)((a.m_tiles + 7) / 8), (unsigned)std::min<long long>(65535, n_local_ct - y0));
    cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
    dispatch_kid(match_fast_kernel(kp), [&](auto kid) {
      large_pred_assemble_kernel<decltype(kid)::value><<<grid, 256, 0, cngp_ctx_stream(ctx)>>>(a);
    });
    cngp_ctx_end(ctx);
  }
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_predict_panel(cngp_ctx* ctx, const cngp_large_plan* p, const double* A, const double* winv,
                                        const double* R, int64_t M, int64_t k, double* payload, double* s) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !A || !winv || !R || !payload || !s || M <= 0 || k < 0 || k >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_predict_panel: bad argument");
  if (k % p->world != p->rank) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_predict_panel: not the owner of this block column");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t st = cngp_ctx_stream(ctx);
  const long long l = k / p->world, mt = pred_m_tiles(M), NT = p->n_pad / 8, r0 = (k + 1) * LG_BT;
  // W_k = R(:, k) inv(L_kk)^T: the panel product of large_gemm_kernel (mode 0) with the test rows as the panel rows
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.X = R + l * LG_BT * mt * 64; g.x_kstride = mt * 64;
  g.Y = winv + l * LG_BT * LG_BT * 64; g.y_kstride = (long long)LG_BT * 64;
  g.panel = payload; g.pg.r0 = 0; g.pg.row_tiles = mt; g.pg.cs = 0;
  g.mode = 0; g.world = p->world; g.rank = p->rank;
  LCU(ctx, cudaFuncSetAttribute(large_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_SMEM));
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_gemm_kernel<<<dim3((unsigned)(mt / LG_BLK), LG_BT / LG_BLK), LG_THREADS, LG_SMEM, st>>>(g);
  cngp_ctx_end(ctx);
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_pred_sumsq_kernel<<<(unsigned)((mt + 7) / 8), 256, 0, st>>>(payload, mt, M, s + k * M);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  // L(rows below the diagonal block, k) from A behind W_k, without the y / z row tile: [k-tile][row tile - r0]
  if (NT > r0) {
    const long long cstride = p->row_tiles * 64;
    LCU(ctx, cudaMemcpy2DAsync(payload + (long long)LG_BT * mt * 64, (size_t)(NT - r0) * 512, A + l * LG_BT * cstride + r0 * 64,
                               (size_t)cstride * 8, (size_t)(NT - r0) * 512, LG_BT, cudaMemcpyDeviceToDevice, st));
  }
  return CNGP_OK;
}

extern "C" int cngp_large_predict_update(cngp_ctx* ctx, const cngp_large_plan* p, double* R, int64_t M, int64_t k,
                                         const double* payload, int64_t c_lo, int64_t c_hi) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !R || !payload || M <= 0 || k < 0 || k >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_predict_update: bad argument");
  c_lo = std::max<int64_t>(c_lo, k + 1);
  c_hi = std::min<int64_t>(c_hi, p->n_blockcols);
  if (c_lo >= c_hi) return CNGP_OK;
  const long long l_lo = local_index_of(c_lo, p->world, p->rank), l_hi = local_index_of(c_hi, p->world, p->rank);
  if (l_lo >= l_hi) return CNGP_OK;
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  const long long mt = pred_m_tiles(M), NT = p->n_pad / 8, r0 = (k + 1) * LG_BT;
  PredUpdArgs a;
  a.W = payload; a.w_kstride = mt * 64;
  a.Lp = payload + (long long)LG_BT * mt * 64 - r0 * 64; a.l_kstride = (NT - r0) * 64;
  a.R = R; a.r_cstride = mt * 64;
  a.world = p->world; a.rank = p->rank;
  LCU(ctx, cudaFuncSetAttribute(large_pred_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_SMEM));
  const long long ncb = (l_hi - l_lo) * (LG_BT / LG_BLK);
  for (long long y0 = 0; y0 < ncb; y0 += 65535) {
    a.lcb0 = (int)(l_lo * (LG_BT / LG_BLK) + y0);
    const unsigned ny = (unsigned)std::min<long long>(65535, ncb - y0);
    cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
    large_pred_update_kernel<<<dim3((unsigned)(mt / LG_BLK), ny), LG_THREADS, LG_SMEM, cngp_ctx_stream(ctx)>>>(a);
    cngp_ctx_end(ctx);
  }
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_predict_finish(cngp_ctx* ctx, const cngp_large_plan* p, const cngp_kernel* kernel,
                                         const double* theta, const double* x, const double* alpha, const double* xstar,
                                         int64_t M, const double* s, double* mean, double* var) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !kernel || !theta || !x || !alpha || !xstar || !s || !mean || !var || M <= 0)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_predict_finish: bad argument");
  KProg kp;
  int rc = cngp_build_kprog(kernel, &kp);
  if (rc) return cngp_set_error(ctx, rc, "large_predict_finish: invalid kernel expression");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  double* d_theta;
  if ((rc = upload_theta(ctx, kp, theta, &d_theta, "large_predict_finish: theta buffer"))) return rc;
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  dispatch_kid(match_fast_kernel(kp), [&](auto kid) {
    large_pred_finish_kernel<decltype(kid)::value><<<(unsigned)((M + 7) / 8), 256, 0, cngp_ctx_stream(ctx)>>>(
        kp, d_theta, x, alpha, p->N, xstar, M, s, p->n_blockcols, mean, var);
  });
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

// ------------------------------------------------------------------------------------------------------------
// LML gradient pass (see cngp.h): the predict sweep with R = I, Ky^-1 accumulated block column by block column
// ------------------------------------------------------------------------------------------------------------
extern "C" int cngp_large_grad_sizes(const cngp_large_plan* p, int64_t* rg_doubles, int64_t* payload_doubles,
                                     int64_t* part_doubles) {
  if (!p || p->n_blockcols <= 0) return CNGP_ERR_INVALID;
  if (rg_doubles) *rg_doubles = p->n_local_blockcols * LG_BT * (p->n_pad / 8) * 64;
  if (payload_doubles) *payload_doubles = (long long)LG_BT * 64 * (p->n_pad / 8);     // [W_k ; L(rows > k, k)], any k
  if (part_doubles) *part_doubles = p->n_blockcols * GRAD_STRIDE;
  return CNGP_OK;
}

extern "C" int cngp_large_grad_begin(cngp_ctx* ctx, const cngp_large_plan* p, double* RG) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !RG) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_grad_begin: bad argument");
  if (p->n_local_blockcols == 0) return CNGP_OK;
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t st = cngp_ctx_stream(ctx);
  const long long NT = p->n_pad / 8, n_lct = p->n_local_blockcols * LG_BT;
  LCU(ctx, cudaMemsetAsync(RG, 0, sizeof(double) * (size_t)(n_lct * NT * 64), st));
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_grad_identity_kernel<<<(unsigned)((n_lct + 255) / 256), 256, 0, st>>>(RG, NT, n_lct, p->world, p->rank);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_grad_panel(cngp_ctx* ctx, const cngp_large_plan* p, const double* A, const double* winv, double* RG,
                                     int64_t k, double* payload) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !A || !winv || !RG || !payload || k < 0 || k >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_grad_panel: bad argument");
  if (k % p->world != p->rank) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_grad_panel: not the owner of this block column");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t st = cngp_ctx_stream(ctx);
  const long long l = k / p->world, NT = p->n_pad / 8, r0 = (k + 1) * LG_BT;
  double* Rk = RG + l * LG_BT * NT * 64;
  // W_k = R(rows < 256 (k+1), k) inv(L_kk)^T: the panel product (large_gemm_kernel mode 0), as in cngp_large_predict_panel
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.X = Rk; g.x_kstride = NT * 64;
  g.Y = winv + l * LG_BT * LG_BT * 64; g.y_kstride = (long long)LG_BT * 64;
  g.panel = payload; g.pg.r0 = 0; g.pg.row_tiles = r0; g.pg.cs = 0;
  g.mode = 0; g.world = p->world; g.rank = p->rank;
  LCU(ctx, cudaFuncSetAttribute(large_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_SMEM));
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_gemm_kernel<<<dim3((unsigned)(r0 / LG_BLK), LG_BT / LG_BLK), LG_THREADS, LG_SMEM, st>>>(g);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  // L(rows below the diagonal block, k) behind W_k: [k-tile][row tile - r0]
  if (NT > r0) {
    const long long cstride = p->row_tiles * 64;
    LCU(ctx, cudaMemcpy2DAsync(payload + (long long)LG_BT * r0 * 64, (size_t)(NT - r0) * 512, A + l * LG_BT * cstride + r0 * 64,
                               (size_t)cstride * 8, (size_t)(NT - r0) * 512, LG_BT, cudaMemcpyDeviceToDevice, st));
  }
  // R(:, k) is consumed: block column k becomes G(:, k).  Rows below its diagonal block are zero already (R(:, k) has
  // none), the diagonal block held R(k, k)
  LCU(ctx, cudaMemset2DAsync(Rk + k * LG_BT * 64, (size_t)NT * 512, 0, (size_t)LG_BT * 512, LG_BT, st));
  return CNGP_OK;
}

extern "C" int cngp_large_grad_update(cngp_ctx* ctx, const cngp_large_plan* p, double* RG, int64_t k, const double* payload,
                                      int64_t c_lo, int64_t c_hi) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !RG || !payload || k < 0 || k >= p->n_blockcols)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_grad_update: bad argument");
  c_lo = std::max<int64_t>(c_lo, 0);
  c_hi = std::min<int64_t>(c_hi, p->n_blockcols);
  if (c_lo >= c_hi) return CNGP_OK;
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t st = cngp_ctx_stream(ctx);
  const long long NT = p->n_pad / 8, r0 = (k + 1) * LG_BT;
  const int rbk = (int)(r0 / LG_BLK);                     // 16-tile row blocks of W_k
  // sweep: R(rows < 256 (k+1), c) -= W_k L(c, k)^T for c > k - large_pred_update_kernel over W_k's rows only
  {
    const long long l_lo = local_index_of(std::max<int64_t>(c_lo, k + 1), p->world, p->rank);
    const long long l_hi = local_index_of(c_hi, p->world, p->rank);
    if (l_lo < l_hi) {
      PredUpdArgs a;
      a.W = payload; a.w_kstride = r0 * 64;
      a.Lp = payload + (long long)LG_BT * r0 * 64 - r0 * 64; a.l_kstride = (NT - r0) * 64;
      a.R = RG; a.r_cstride = NT * 64;
      a.world = p->world; a.rank = p->rank;
      LCU(ctx, cudaFuncSetAttribute(large_pred_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_SMEM));
      const long long ncb = (l_hi - l_lo) * (LG_BT / LG_BLK);
      for (long long y0 = 0; y0 < ncb; y0 += 65535) {
        a.lcb0 = (int)(l_lo * (LG_BT / LG_BLK) + y0);
        const unsigned ny = (unsigned)std::min<long long>(65535, ncb - y0);
        cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
        large_pred_update_kernel<<<dim3((unsigned)rbk, ny), LG_THREADS, LG_SMEM, st>>>(a);
        cngp_ctx_end(ctx);
      }
    }
  }
  // accumulation: G(I, J) -= W_k(I) W_k(J)^T for J <= k, J <= I <= k - the trailing update (large_gemm_kernel mode 1) with
  // W_k as the panel; blocks above the diagonal return at once
  {
    const long long l_lo = local_index_of(c_lo, p->world, p->rank);
    const long long l_hi = local_index_of(std::min<int64_t>(c_hi, k + 1), p->world, p->rank);
    if (l_lo < l_hi) {
      const long long c_first = l_lo * p->world + p->rank;
      GemmArgs g;
      memset(&g, 0, sizeof g);
      g.panel = const_cast<double*>(payload); g.pg.r0 = 0; g.pg.row_tiles = r0; g.pg.cs = 0;
      g.C = RG; g.c_cstride = NT * 64;
      g.mode = 1; g.rb0 = (int)(c_first * LG_BT / LG_BLK); g.world = p->world; g.rank = p->rank;
      LCU(ctx, cudaFuncSetAttribute(large_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_SMEM));
      const long long ncb = (l_hi - l_lo) * (LG_BT / LG_BLK);
      for (long long y0 = 0; y0 < ncb; y0 += 65535) {
        g.lcb0 = (int)(l_lo * (LG_BT / LG_BLK) + y0);
        const unsigned ny = (unsigned)std::min<long long>(65535, ncb - y0);
        cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
        large_gemm_kernel<<<dim3((unsigned)(rbk - g.rb0), ny), LG_THREADS, LG_SMEM, st>>>(g);
        cngp_ctx_end(ctx);
      }
    }
  }
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_grad_contract(cngp_ctx* ctx, const cngp_large_plan* p, const cngp_kernel* kernel, const double* theta,
                                        const double* x, const double* alpha, const double* RG, double* part) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !kernel || !theta || !x || !alpha || !RG || !part)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_grad_contract: bad argument");
  KProg kp;
  int rc = cngp_build_kprog(kernel, &kp);
  if (rc) return cngp_set_error(ctx, rc, "large_grad_contract: invalid kernel expression");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  double* d_theta;
  if ((rc = upload_theta(ctx, kp, theta, &d_theta, "large_grad_contract: theta buffer"))) return rc;
  cudaStream_t st = cngp_ctx_stream(ctx);
  LCU(ctx, cudaMemsetAsync(part, 0, sizeof(double) * (size_t)(p->n_blockcols * GRAD_STRIDE), st));
  const long long n_lct = p->n_local_blockcols * LG_BT;
  if (n_lct == 0) return CNGP_OK;
  double* partial = (double*)cngp_ctx_buf(ctx, SLOT_GPART, sizeof(double) * (size_t)(n_lct * GRAD_STRIDE));
  if (!partial) return cngp_set_error(ctx, CNGP_ERR_NOMEM, "large_grad_contract: scratch");
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_grad_contract_kernel<<<(unsigned)n_lct, GC_WARPS * 32, 0, st>>>(kp, d_theta, x, alpha, RG, p->N, p->n_pad / 8,
                                                                          p->world, p->rank, partial);
  cngp_ctx_end(ctx);
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_grad_part_kernel<<<(unsigned)p->n_local_blockcols, 32, 0, st>>>(partial, p->world, p->rank, part);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

extern "C" int cngp_large_grad_finish(cngp_ctx* ctx, const cngp_large_plan* p, const cngp_kernel* kernel, const double* part,
                                      double* grad) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!p || !kernel || !part || !grad) return cngp_set_error(ctx, CNGP_ERR_INVALID, "large_grad_finish: bad argument");
  KProg kp;
  int rc = cngp_build_kprog(kernel, &kp);
  if (rc) return cngp_set_error(ctx, rc, "large_grad_finish: invalid kernel expression");
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cngp_ctx_begin(ctx, CNGP_PROF_LARGE);
  large_grad_finish_kernel<<<1, 32, 0, cngp_ctx_stream(ctx)>>>(part, p->n_blockcols, kp.n_params + 1, grad);
  cngp_ctx_end(ctx);
  LCU(ctx, cudaGetLastError());
  return CNGP_OK;
}

namespace {
struct DevMem {
  void* p = nullptr;
  ~DevMem() { if (p) cudaFree(p); }
  bool alloc(size_t bytes) { return cudaMalloc(&p, std::max<size_t>(bytes, 16)) == cudaSuccess; }
};
}  // namespace

extern "C" int cngp_chol_large(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x,
                               const double* y, int64_t N, double* logdet, double* quad, double* lml, double* alpha,
                               int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !theta || !x || !y || N <= 0) return cngp_set_error(ctx, CNGP_ERR_INVALID, "chol_large: bad argument");
  cngp_large_plan p;
  cngp_large_make_plan(N, 1, 0, &p);
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  DevMem dA, dP, dW, dld, dst, dz, dal, dsum, dx, dy, dsa;
  if (!dA.alloc(sizeof(double) * p.local_doubles) || !dP.alloc(sizeof(double) * p.panel_doubles) ||
      !dW.alloc(sizeof(double) * p.winv_doubles) || !dld.alloc(sizeof(double) * p.n_blockcols) ||
      !dst.alloc(sizeof(int) * p.n_blockcols) || !dz.alloc(sizeof(double) * p.n_pad) ||
      !dal.alloc(sizeof(double) * p.n_pad) || !dsum.alloc(sizeof(double) * 4) || !dsa.alloc(sizeof(double) * p.n_pad))
    return cngp_set_error(ctx, CNGP_ERR_NOMEM, "chol_large: device allocation failed");
  const double *d_x = x, *d_y = y;
  if (mem == CNGP_MEM_HOST) {
    if (!dx.alloc(sizeof(double) * N) || !dy.alloc(sizeof(double) * N))
      return cngp_set_error(ctx, CNGP_ERR_NOMEM, "chol_large: device allocation failed");
    LCU(ctx, cudaMemcpyAsync(dx.p, x, sizeof(double) * N, cudaMemcpyHostToDevice, s));
    LCU(ctx, cudaMemcpyAsync(dy.p, y, sizeof(double) * N, cudaMemcpyHostToDevice, s));
    d_x = (const double*)dx.p; d_y = (const double*)dy.p;
  }
  int rc = cngp_large_assemble(ctx, &p, kernel, theta, d_x, d_y, (double*)dA.p);
  if (rc) return rc;
  LCU(ctx, cudaMemsetAsync(dP.p, 0, sizeof(double) * p.panel_doubles, s));
  for (int64_t k = 0; k < p.n_blockcols; ++k) {
    if ((rc = cngp_large_factor_panel(ctx, &p, (double*)dA.p, k, (double*)dP.p, (double*)dW.p, (double*)dld.p, (int*)dst.p))) return rc;
    if ((rc = cngp_large_update(ctx, &p, (double*)dA.p, k, (const double*)dP.p, k + 1, p.n_blockcols))) return rc;
  }
  if ((rc = cngp_large_reduce(ctx, &p, (const double*)dA.p, (const double*)dld.p, (const int*)dst.p, (double*)dz.p, (double*)dsum.p))) return rc;
  if (alpha) {
    LCU(ctx, cudaMemsetAsync(dal.p, 0, sizeof(double) * p.n_pad, s));
    LCU(ctx, cudaMemsetAsync(dsa.p, 0, sizeof(double) * p.n_pad, s));
    for (int64_t j = p.n_blockcols - 1; j >= 0; --j) {
      if ((rc = cngp_large_backsolve_finish(ctx, &p, (const double*)dW.p, j, (const double*)dz.p, (const double*)dsa.p, (double*)dal.p))) return rc;
      if ((rc = cngp_large_backsolve_apply(ctx, &p, (const double*)dA.p, j, (const double*)dal.p, (double*)dsa.p))) return rc;
    }
    LCU(ctx, cudaMemcpyAsync(alpha, dal.p, sizeof(double) * N, mem == CNGP_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s));
  }
  double sums[3];
  LCU(ctx, cudaMemcpyAsync(sums, dsum.p, sizeof sums, cudaMemcpyDeviceToHost, s));
  LCU(ctx, cudaStreamSynchronize(s));
  const bool bad = sums[2] != 0.0;
  const double nanv = std::nan("");
  if (logdet) *logdet = bad ? nanv : sums[0];
  if (quad) *quad = bad ? nanv : sums[1];
  if (lml) *lml = bad ? nanv : 0.5 * (-(double)N * CNGP_LOG_2PI - sums[0] - sums[1]);
  return bad ? (int)sums[2] : CNGP_OK;
}

extern "C" int cngp_chol_large_predict(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x,
                                       const double* y, int64_t N, const double* xstar, int64_t M, double* mean,
                                       double* var, double* logdet, double* quad, double* lml, int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !theta || !x || !y || !xstar || !mean || !var || N <= 0 || M <= 0)
    return cngp_set_error(ctx, CNGP_ERR_INVALID, "chol_large_predict: bad argument");
  cngp_large_plan p;
  cngp_large_make_plan(N, 1, 0, &p);
  int64_t r_doubles, payload_doubles, s_doubles;
  cngp_large_predict_sizes(&p, M, 0, &r_doubles, &payload_doubles, &s_doubles);
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  DevMem dA, dP, dW, dld, dst, dz, dal, dsum, dx, dy, dsa, dxs, dR, dpay, ds, dmean, dvar;
  if (!dA.alloc(sizeof(double) * p.local_doubles) || !dP.alloc(sizeof(double) * p.panel_doubles) ||
      !dW.alloc(sizeof(double) * p.winv_doubles) || !dld.alloc(sizeof(double) * p.n_blockcols) ||
      !dst.alloc(sizeof(int) * p.n_blockcols) || !dz.alloc(sizeof(double) * p.n_pad) ||
      !dal.alloc(sizeof(double) * p.n_pad) || !dsum.alloc(sizeof(double) * 4) || !dsa.alloc(sizeof(double) * p.n_pad) ||
      !dR.alloc(sizeof(double) * r_doubles) || !dpay.alloc(sizeof(double) * payload_doubles) ||
      !ds.alloc(sizeof(double) * s_doubles))
    return cngp_set_error(ctx, CNGP_ERR_NOMEM, "chol_large_predict: device allocation failed");
  const double *d_x = x, *d_y = y, *d_xs = xstar;
  double *d_mean = mean, *d_var = var;
  if (mem == CNGP_MEM_HOST) {
    if (!dx.alloc(sizeof(double) * N) || !dy.alloc(sizeof(double) * N) || !dxs.alloc(sizeof(double) * M) ||
        !dmean.alloc(sizeof(double) * M) || !dvar.alloc(sizeof(double) * M))
      return cngp_set_error(ctx, CNGP_ERR_NOMEM, "chol_large_predict: device allocation failed");
    LCU(ctx, cudaMemcpyAsync(dx.p, x, sizeof(double) * N, cudaMemcpyHostToDevice, s));
    LCU(ctx, cudaMemcpyAsync(dy.p, y, sizeof(double) * N, cudaMemcpyHostToDevice, s));
    LCU(ctx, cudaMemcpyAsync(dxs.p, xstar, sizeof(double) * M, cudaMemcpyHostToDevice, s));
    d_x = (const double*)dx.p; d_y = (const double*)dy.p; d_xs = (const double*)dxs.p;
    d_mean = (double*)dmean.p; d_var = (double*)dvar.p;
  }
  // the factorisation and the backward sweep of cngp_chol_large
  int rc = cngp_large_assemble(ctx, &p, kernel, theta, d_x, d_y, (double*)dA.p);
  if (rc) return rc;
  LCU(ctx, cudaMemsetAsync(dP.p, 0, sizeof(double) * p.panel_doubles, s));
  for (int64_t k = 0; k < p.n_blockcols; ++k) {
    if ((rc = cngp_large_factor_panel(ctx, &p, (double*)dA.p, k, (double*)dP.p, (double*)dW.p, (double*)dld.p, (int*)dst.p))) return rc;
    if ((rc = cngp_large_update(ctx, &p, (double*)dA.p, k, (const double*)dP.p, k + 1, p.n_blockcols))) return rc;
  }
  if ((rc = cngp_large_reduce(ctx, &p, (const double*)dA.p, (const double*)dld.p, (const int*)dst.p, (double*)dz.p, (double*)dsum.p))) return rc;
  double sums[3];
  LCU(ctx, cudaMemcpyAsync(sums, dsum.p, sizeof sums, cudaMemcpyDeviceToHost, s));
  LCU(ctx, cudaStreamSynchronize(s));
  const double nanv = std::nan("");
  if (sums[2] != 0.0) {                      // not positive definite: nothing below reads the broken factor
    if (logdet) *logdet = nanv;
    if (quad) *quad = nanv;
    if (lml) *lml = nanv;
    if (mem == CNGP_MEM_HOST) {
      std::fill(mean, mean + M, nanv);
      std::fill(var, var + M, nanv);
    } else {
      std::vector<double> nans((size_t)M, nanv);
      LCU(ctx, cudaMemcpyAsync(mean, nans.data(), sizeof(double) * M, cudaMemcpyHostToDevice, s));
      LCU(ctx, cudaMemcpyAsync(var, nans.data(), sizeof(double) * M, cudaMemcpyHostToDevice, s));
      LCU(ctx, cudaStreamSynchronize(s));
    }
    return (int)sums[2];
  }
  LCU(ctx, cudaMemsetAsync(dal.p, 0, sizeof(double) * p.n_pad, s));
  LCU(ctx, cudaMemsetAsync(dsa.p, 0, sizeof(double) * p.n_pad, s));
  for (int64_t j = p.n_blockcols - 1; j >= 0; --j) {
    if ((rc = cngp_large_backsolve_finish(ctx, &p, (const double*)dW.p, j, (const double*)dz.p, (const double*)dsa.p, (double*)dal.p))) return rc;
    if ((rc = cngp_large_backsolve_apply(ctx, &p, (const double*)dA.p, j, (const double*)dal.p, (double*)dsa.p))) return rc;
  }
  // the predict pass, block column by block column (one rank: no look-ahead needed)
  if ((rc = cngp_large_predict_assemble(ctx, &p, kernel, theta, d_x, d_xs, M, (double*)dR.p))) return rc;
  for (int64_t k = 0; k < p.n_blockcols; ++k) {
    if ((rc = cngp_large_predict_panel(ctx, &p, (const double*)dA.p, (const double*)dW.p, (const double*)dR.p, M, k,
                                       (double*)dpay.p, (double*)ds.p))) return rc;
    if ((rc = cngp_large_predict_update(ctx, &p, (double*)dR.p, M, k, (const double*)dpay.p, k + 1, p.n_blockcols))) return rc;
  }
  if ((rc = cngp_large_predict_finish(ctx, &p, kernel, theta, d_x, (const double*)dal.p, d_xs, M, (const double*)ds.p,
                                      d_mean, d_var))) return rc;
  if (mem == CNGP_MEM_HOST) {
    LCU(ctx, cudaMemcpyAsync(mean, d_mean, sizeof(double) * M, cudaMemcpyDeviceToHost, s));
    LCU(ctx, cudaMemcpyAsync(var, d_var, sizeof(double) * M, cudaMemcpyDeviceToHost, s));
  }
  LCU(ctx, cudaStreamSynchronize(s));
  if (logdet) *logdet = sums[0];
  if (quad) *quad = sums[1];
  if (lml) *lml = 0.5 * (-(double)N * CNGP_LOG_2PI - sums[0] - sums[1]);
  return CNGP_OK;
}

extern "C" int cngp_chol_large_grad(cngp_ctx* ctx, const cngp_kernel* kernel, const double* theta, const double* x,
                                    const double* y, int64_t N, double* logdet, double* quad, double* lml, double* grad,
                                    int32_t mem) {
  if (!ctx) return CNGP_ERR_INVALID;
  if (!kernel || !theta || !x || !y || !grad || N <= 0) return cngp_set_error(ctx, CNGP_ERR_INVALID, "chol_large_grad: bad argument");
  KProg kp;
  int rc = cngp_build_kprog(kernel, &kp);
  if (rc) return cngp_set_error(ctx, rc, "chol_large_grad: invalid kernel expression");
  const int P = kp.n_params + 1;
  cngp_large_plan p;
  cngp_large_make_plan(N, 1, 0, &p);
  int64_t rg_doubles, payload_doubles, part_doubles;
  cngp_large_grad_sizes(&p, &rg_doubles, &payload_doubles, &part_doubles);
  LCU(ctx, cudaSetDevice(cngp_ctx_device(ctx)));
  cudaStream_t s = cngp_ctx_stream(ctx);
  DevMem dA, dP, dW, dld, dst, dz, dal, dsum, dx, dy, dsa, dRG, dpay, dpart, dgrad;
  if (!dA.alloc(sizeof(double) * p.local_doubles) || !dP.alloc(sizeof(double) * p.panel_doubles) ||
      !dW.alloc(sizeof(double) * p.winv_doubles) || !dld.alloc(sizeof(double) * p.n_blockcols) ||
      !dst.alloc(sizeof(int) * p.n_blockcols) || !dz.alloc(sizeof(double) * p.n_pad) ||
      !dal.alloc(sizeof(double) * p.n_pad) || !dsum.alloc(sizeof(double) * 4) || !dsa.alloc(sizeof(double) * p.n_pad) ||
      !dRG.alloc(sizeof(double) * rg_doubles) || !dpay.alloc(sizeof(double) * payload_doubles) ||
      !dpart.alloc(sizeof(double) * part_doubles) || !dgrad.alloc(sizeof(double) * P))
    return cngp_set_error(ctx, CNGP_ERR_NOMEM, "chol_large_grad: device allocation failed");
  const double *d_x = x, *d_y = y;
  if (mem == CNGP_MEM_HOST) {
    if (!dx.alloc(sizeof(double) * N) || !dy.alloc(sizeof(double) * N))
      return cngp_set_error(ctx, CNGP_ERR_NOMEM, "chol_large_grad: device allocation failed");
    LCU(ctx, cudaMemcpyAsync(dx.p, x, sizeof(double) * N, cudaMemcpyHostToDevice, s));
    LCU(ctx, cudaMemcpyAsync(dy.p, y, sizeof(double) * N, cudaMemcpyHostToDevice, s));
    d_x = (const double*)dx.p; d_y = (const double*)dy.p;
  }
  // the factorisation and the backward sweep of cngp_chol_large
  if ((rc = cngp_large_assemble(ctx, &p, kernel, theta, d_x, d_y, (double*)dA.p))) return rc;
  LCU(ctx, cudaMemsetAsync(dP.p, 0, sizeof(double) * p.panel_doubles, s));
  for (int64_t k = 0; k < p.n_blockcols; ++k) {
    if ((rc = cngp_large_factor_panel(ctx, &p, (double*)dA.p, k, (double*)dP.p, (double*)dW.p, (double*)dld.p, (int*)dst.p))) return rc;
    if ((rc = cngp_large_update(ctx, &p, (double*)dA.p, k, (const double*)dP.p, k + 1, p.n_blockcols))) return rc;
  }
  if ((rc = cngp_large_reduce(ctx, &p, (const double*)dA.p, (const double*)dld.p, (const int*)dst.p, (double*)dz.p, (double*)dsum.p))) return rc;
  double sums[3];
  LCU(ctx, cudaMemcpyAsync(sums, dsum.p, sizeof sums, cudaMemcpyDeviceToHost, s));
  LCU(ctx, cudaStreamSynchronize(s));
  const double nanv = std::nan("");
  if (sums[2] != 0.0) {                      // not positive definite: nothing below reads the broken factor
    if (logdet) *logdet = nanv;
    if (quad) *quad = nanv;
    if (lml) *lml = nanv;
    std::vector<double> nans((size_t)P, nanv);
    if (mem == CNGP_MEM_HOST) {
      std::copy(nans.begin(), nans.end(), grad);
    } else {
      LCU(ctx, cudaMemcpyAsync(grad, nans.data(), sizeof(double) * P, cudaMemcpyHostToDevice, s));
      LCU(ctx, cudaStreamSynchronize(s));
    }
    return (int)sums[2];
  }
  LCU(ctx, cudaMemsetAsync(dal.p, 0, sizeof(double) * p.n_pad, s));
  LCU(ctx, cudaMemsetAsync(dsa.p, 0, sizeof(double) * p.n_pad, s));
  for (int64_t j = p.n_blockcols - 1; j >= 0; --j) {
    if ((rc = cngp_large_backsolve_finish(ctx, &p, (const double*)dW.p, j, (const double*)dz.p, (const double*)dsa.p, (double*)dal.p))) return rc;
    if ((rc = cngp_large_backsolve_apply(ctx, &p, (const double*)dA.p, j, (const double*)dal.p, (double*)dsa.p))) return rc;
  }
  // the gradient pass, block column by block column (one rank: no look-ahead needed)
  if ((rc = cngp_large_grad_begin(ctx, &p, (double*)dRG.p))) return rc;
  for (int64_t k = 0; k < p.n_blockcols; ++k) {
    if ((rc = cngp_large_grad_panel(ctx, &p, (const double*)dA.p, (const double*)dW.p, (double*)dRG.p, k, (double*)dpay.p))) return rc;
    if ((rc = cngp_large_grad_update(ctx, &p, (double*)dRG.p, k, (const double*)dpay.p, 0, p.n_blockcols))) return rc;
  }
  if ((rc = cngp_large_grad_contract(ctx, &p, kernel, theta, d_x, (const double*)dal.p, (const double*)dRG.p, (double*)dpart.p))) return rc;
  double* d_grad = mem == CNGP_MEM_HOST ? (double*)dgrad.p : grad;
  if ((rc = cngp_large_grad_finish(ctx, &p, kernel, (const double*)dpart.p, d_grad))) return rc;
  if (mem == CNGP_MEM_HOST) LCU(ctx, cudaMemcpyAsync(grad, d_grad, sizeof(double) * P, cudaMemcpyDeviceToHost, s));
  LCU(ctx, cudaStreamSynchronize(s));
  if (logdet) *logdet = sums[0];
  if (quad) *quad = sums[1];
  if (lml) *lml = 0.5 * (-(double)N * CNGP_LOG_2PI - sums[0] - sums[1]);
  return CNGP_OK;
}
