// estep.cu -- K1: fused CPD / BCPD E-step for sm_100a.
//
// Replaces CpdRegistrationState.P (registration/config/CPD.scala:54-75) together with the reductions
// the reference takes from it: P1 = sum(P, Axis._1) (CPD.scala:36, :122, :139), Pt1 = sum(P, Axis._0)
// (:140), P*X (:145), and BCPD.computeP + reductions (other/algorithms/cpd/BCPD.scala:167-184, :200-209).
// The M x N matrix is never materialised.  Two sweeps over the pairs are inherent (the column
// denominators need every row before any P_ij is final):
//
//   sweep A  (estep_colsum_kernel)  colsum_j = sum_i f_i K_ij            thread owns CA columns in registers,
//                                                                        rows stream through shared memory
//   estep_den_kernel                den_j = a*colsum_j + c ; w_j = 1/den_j ; Pt1_j = colsum_j * w_j ;
//                                   packs {x_j, w_j, w_j x_j} for sweep B
//   sweep B  (estep_rowsum_kernel)  P1_i = f_i sum_j K_ij w_j ; PX_i = f_i sum_j K_ij (w_j x_j)
//                                   thread owns RB rows + 4 accumulators in registers, columns stream
//                                   through shared memory
//   estep_rowreduce_kernel          fixed-order sum of the per-CTA partials (deterministic, no atomics)
//
// K_ij = exp(-|x_j - y_i|^2 / (2 sigma2)) in FP64 (FP32 cannot represent the 1e-159 column sums of
// DemoCPD's sigma2 = 1, SURVEY.md 7.1).  The kernel is bound by the FP64 FMA pipe, not by HBM:
// bytes are 24(M+N) in, 8(4M+N) out against 2 x 20..24 FP64 instructions per pair.
// CPD:  f_i = 1, a = 1, c = w/(1-w) (2 pi sigma2)^{3/2} M/N           (CPD.scala:69-72)
// BCPD: f_i = (1-w) (2 pi sigma2)^{-3/2} exp(-s/(2 sigma2) 3 Sigma_mm) alpha_m, a = (1-w), c = w/N
//                                                                     (BCPD.scala:170-181)
#include "batch.cuh"
#include "estep.cuh"
#include "exp2_poly.cuh"

#include <algorithm>
#include <utility>
#include <vector>

namespace gingr {

// tuning knobs (overridable with -D for experiments; the defaults are the measured best on B200)
#ifndef ESTEP_CA
#define ESTEP_CA 6
#endif
#ifndef ESTEP_RB
#define ESTEP_RB 4
#endif
#ifndef ESTEP_MINB_A
#define ESTEP_MINB_A 2
#endif
#ifndef ESTEP_UNROLL_A
#define ESTEP_UNROLL_A 1
#endif
#ifndef ESTEP_UNROLL_B
#define ESTEP_UNROLL_B 1
#endif
#define ESTEP_PRAGMA(x) _Pragma(#x)
#define ESTEP_UNROLL(n) ESTEP_PRAGMA(unroll n)
#ifndef ESTEP_MINB_B
#define ESTEP_MINB_B 4
#endif
constexpr int TPB = 256;       // threads per CTA in sweep A and the small kernels
constexpr int TPB_B = 128;     // threads per CTA in sweep B: 512-row blocks, small enough for the sweep-B bound to bite
constexpr int CA = ESTEP_CA;   // columns per thread, sweep A
constexpr int RB = ESTEP_RB;   // rows per thread, sweep B
constexpr int TILE_ROWS = 512; // rows staged per shared-memory tile in sweep A
constexpr int TILE_COLS = 256; // columns staged per shared-memory tile in sweep B
// Culling units.  fit_soa is in the k-d order of estep_row_order and the target shard in that of estep_target_order, so
// each aligned unit below is a subtree with a tight bounding box.
constexpr int COLS_A = TPB * CA;     // sweep-A column block (target points)
constexpr int SUB_A = 32;            // sweep-A model sub-tile (rows)
constexpr int ROWS_B = TPB_B * RB;   // sweep-B row block (model points)
constexpr int TILE_B = 64;           // sweep-B target tile (columns)
static_assert(TILE_ROWS % SUB_A == 0 && TILE_COLS % TILE_B == 0 && COLS_A % TILE_B == 0 && ROWS_B % SUB_A == 0, "tiles");
// Below this many pairs the three extra launches of the cull cost more than they can save (and C3-size problems stay as
// they were); at the C4 size they cost < 0.1 % of a dense E-step.
constexpr double CULL_MIN_PAIRS = 1.0 * (1 << 27);

// True when every pair of this launch satisfies 0 <= d2 * |negk64| < 2^31 - 2^18 (gauss_exp2_tab<SAFE>):
// scal[7] = upper bound of d2 from the coordinate ranges of both clouds (<= 0 / non-finite: unknown).
__device__ __forceinline__ bool estep_safe_range(const double* __restrict__ scal) {
  const double sigma2 = scal[0], d2max = scal[7];
  return sigma2 > 0.0 && d2max > 0.0 && d2max * (GAUSS_SCALE * 1.4426950408889634074 / (2.0 * sigma2)) < 2146435072.0;
}

// Expanded-distance fast path: -k |x - y|^2 = (-k |x|^2) + (-k |y|^2) + (2 k x) . y  needs 1 add + 3 FMA per pair
// instead of 3 subtractions + 1 multiply + 2 FMA + the scaling FMA of the exponential (14 / 17 FP64 instructions per
// pair in sweep A / B instead of 16 / 19).  The cancellation costs an absolute error of about
// 4 eps |k64| (|x|^2 + |y|^2) in the scaled exponent, so the path is only taken while |k64| d2max < 2^22
// (relative error of every K_ij below 4e-11, typically 1e-13); smaller sigma2 / larger extents use the difference form.
__device__ __forceinline__ bool estep_expand_ok(const double* __restrict__ scal) {
  const double sigma2 = scal[0], d2max = scal[7];
  return sigma2 > 0.0 && d2max > 0.0 && d2max * (64.0 * 1.4426950408889634074 / (2.0 * sigma2)) < 4194304.0;
}

// ytile[t] = {y, -k64 |y|^2};  per column px = 2 k64 x (3 values), cx = -k64 |x|^2
__device__ __forceinline__ void colsum_tile_expanded(int cnt, const double4* __restrict__ ytile, const double (&px)[CA],
                                                     const double (&py)[CA], const double (&pz)[CA], const double (&cx)[CA],
                                                     double (&acc)[CA], const unsigned int* s_tab, int lane_off) {
ESTEP_UNROLL(ESTEP_UNROLL_A)
  for (int t = 0; t < cnt; ++t) {
    const double4 y = ytile[t];
#pragma unroll
    for (int c = 0; c < CA; ++c) {
      double u = cx[c] + y.w;
      u = fma(pz[c], y.z, u);
      u = fma(py[c], y.y, u);
      u = fma(px[c], y.x, u);
      acc[c] += gauss_exp2_tab_u(u, s_tab, lane_off);
    }
  }
}

// xtile[2 t] = {2 k64 x, -k64 |x|^2}, xtile[2 t + 1] = {w, w x};  per row y and cy = -k64 |y|^2
__device__ __forceinline__ void rowsum_tile_expanded(int cnt, const double4* __restrict__ xtile, const double (&yx)[RB],
                                                     const double (&yy)[RB], const double (&yz)[RB], const double (&cy)[RB],
                                                     double (&a0)[RB], double (&a1)[RB], double (&a2)[RB], double (&a3)[RB],
                                                     const unsigned int* s_tab, int lane_off) {
ESTEP_UNROLL(ESTEP_UNROLL_B)
  for (int t = 0; t < cnt; ++t) {
    const double4 xa = xtile[2 * t];
    const double4 xb = xtile[2 * t + 1];
#pragma unroll
    for (int q = 0; q < RB; ++q) {
      double u = xa.w + cy[q];
      u = fma(xa.z, yz[q], u);
      u = fma(xa.y, yy[q], u);
      u = fma(xa.x, yx[q], u);
      const double k = gauss_exp2_tab_u(u, s_tab, lane_off);
      a0[q] = fma(k, xb.x, a0[q]);
      a1[q] = fma(k, xb.y, a1[q]);
      a2[q] = fma(k, xb.z, a2[q]);
      a3[q] = fma(k, xb.w, a3[q]);
    }
  }
}

template <bool SAFE>
__device__ __forceinline__ void colsum_tile(int cnt, const double4* __restrict__ ytile, const double (&xj)[CA],
                                            const double (&yj)[CA], const double (&zj)[CA], double (&acc)[CA],
                                            double negk, const unsigned int* s_tab, int lane_off) {
#pragma unroll 2
  for (int t = 0; t < cnt; ++t) {
    const double4 y = ytile[t];
#pragma unroll
    for (int c = 0; c < CA; ++c) {
      const double dx = xj[c] - y.x, dy = yj[c] - y.y, dz = zj[c] - y.z;
      double d2 = dx * dx;
      d2 = fma(dy, dy, d2);
      d2 = fma(dz, dz, d2);
      acc[c] = fma(gauss_exp2_tab<SAFE>(d2, negk, s_tab, lane_off), y.w, acc[c]);
    }
  }
}

template <bool SAFE>
__device__ __forceinline__ void rowsum_tile(int cnt, const double4* __restrict__ xtile, const double (&yx)[RB],
                                            const double (&yy)[RB], const double (&yz)[RB], double (&a0)[RB],
                                            double (&a1)[RB], double (&a2)[RB], double (&a3)[RB], double negk,
                                            const unsigned int* s_tab, int lane_off) {
#pragma unroll 2
  for (int t = 0; t < cnt; ++t) {
    const double4 xa = xtile[2 * t];
    const double4 xb = xtile[2 * t + 1];
#pragma unroll
    for (int q = 0; q < RB; ++q) {
      const double dx = xa.x - yx[q], dy = xa.y - yy[q], dz = xa.z - yz[q];
      double d2 = dx * dx;
      d2 = fma(dy, dy, d2);
      d2 = fma(dz, dz, d2);
      const double k = gauss_exp2_tab<SAFE>(d2, negk, s_tab, lane_off);
      a0[q] = fma(k, xa.w, a0[q]);
      a1[q] = fma(k, xb.x, a1[q]);
      a2[q] = fma(k, xb.y, a2[q]);
      a3[q] = fma(k, xb.z, a3[q]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// sweep A: column sums.   grid = (col blocks, row splits)
// fit  : moving points SoA [3][M] (+ row factor f[M]), target: SoA [3][N]
// part : [gridDim.y][N] partial column sums
// ---------------------------------------------------------------------------------------------
GINGR_KERNEL((TPB, ESTEP_MINB_A), estep_colsum_kernel, int M, int N, const double* __restrict__ fit,
                                                           const double* __restrict__ rowf,
                                                           const double* __restrict__ target,
                                                           const double* __restrict__ scal,
                                                           const int* __restrict__ list, const int* __restrict__ nlive,
                                                           double* __restrict__ part) {
  __shared__ double4 ytile[TILE_ROWS];
  __shared__ __align__(16) unsigned int s_tab[GAUSS_TAB_BYTES / 4];
  gauss_tab_fill(s_tab, threadIdx.x, TPB);
  const int lane_off = (threadIdx.x & 15) * 8;
  const double sigma2 = scal[0];
  const double negk = -GAUSS_SCALE * 1.4426950408889634074 / (2.0 * sigma2);
  // this CTA's contiguous share of the column block's live sub-tiles (all sub-tiles, in order, without a list)
  const int nsub = (M + SUB_A - 1) / SUB_A;
  const int* lst = list ? list + (size_t)blockIdx.x * nsub : nullptr;
  const int nl = list ? nlive[blockIdx.x] : nsub;
  const int per = (nl + gridDim.y - 1) / gridDim.y;
  const int e_begin = min(nl, (int)blockIdx.y * per);
  const int e_end = min(nl, e_begin + per);
  constexpr int SUBS = TILE_ROWS / SUB_A;   // sub-tiles gathered per shared-memory tile
  // model row of staged row t of the tile starting at live entry e0; only the last sub-tile of the model is partial, and
  // lists are ascending, so a tile's rows are the first cnt
  auto row_of = [&](int e0, int t) { return (lst ? lst[e0 + t / SUB_A] : e0 + t / SUB_A) * SUB_A + t % SUB_A; };
  auto tile_rows = [&](int e0, int ne) {
    const int last = lst ? lst[e0 + ne - 1] : e0 + ne - 1;
    return (ne - 1) * SUB_A + min(SUB_A, M - last * SUB_A);
  };

  double xj[CA], yj[CA], zj[CA], acc[CA];
  int col[CA];
#pragma unroll
  for (int c = 0; c < CA; ++c) {
    col[c] = (blockIdx.x * CA + c) * TPB + threadIdx.x;
    const int j = min(col[c], N - 1);
    xj[c] = target[j];
    yj[c] = target[N + j];
    zj[c] = target[2 * N + j];
    acc[c] = 0.0;
  }
  const bool safe = estep_safe_range(scal);
  const bool expand = rowf == nullptr && estep_expand_ok(scal);
  if (expand) {
    double cx[CA];
#pragma unroll
    for (int c = 0; c < CA; ++c) {
      cx[c] = negk * (xj[c] * xj[c] + yj[c] * yj[c] + zj[c] * zj[c]);
      xj[c] *= -2.0 * negk; yj[c] *= -2.0 * negk; zj[c] *= -2.0 * negk;
    }
    for (int e0 = e_begin; e0 < e_end; e0 += SUBS) {
      const int cnt = tile_rows(e0, min(SUBS, e_end - e0));
      __syncthreads();
      for (int t = threadIdx.x; t < cnt; t += TPB) {
        const int i = row_of(e0, t);
        const double a = fit[i], b = fit[M + i], c = fit[2 * M + i];
        ytile[t] = make_double4(a, b, c, negk * (a * a + b * b + c * c));
      }
      __syncthreads();
      colsum_tile_expanded(cnt, ytile, xj, yj, zj, cx, acc, s_tab, lane_off);
    }
  } else {
    for (int e0 = e_begin; e0 < e_end; e0 += SUBS) {
      const int cnt = tile_rows(e0, min(SUBS, e_end - e0));
      __syncthreads();
      for (int t = threadIdx.x; t < cnt; t += TPB) {
        const int i = row_of(e0, t);
        ytile[t] = make_double4(fit[i], fit[M + i], fit[2 * M + i], rowf ? rowf[i] : 1.0);
      }
      __syncthreads();
      if (safe) colsum_tile<true>(cnt, ytile, xj, yj, zj, acc, negk, s_tab, lane_off);
      else colsum_tile<false>(cnt, ytile, xj, yj, zj, acc, negk, s_tab, lane_off);
    }
  }
#pragma unroll
  for (int c = 0; c < CA; ++c)
    if (col[c] < N) part[(size_t)blockIdx.y * N + col[c]] = acc[c];
}

// ---------------------------------------------------------------------------------------------
// denominators.  scal[1] = a, scal[2] = c.  pack[j] = {x, y, z, w_j, w_j x, w_j y, w_j z, 0} * {1,1,1,2^-64,...}
// xpx_part[blockIdx.x] = sum over the block's columns of Pt1_j |x_j|^2  (CPD.scala:142)
// Columns are in the order of target_soa; pt1 is written at the shard index tperm[j].
// tw (may be null): per sweep-B target tile {min w_j, max w_j}, max = +inf when some w_j is not finite.
// ---------------------------------------------------------------------------------------------
GINGR_KERNEL((TPB), estep_den_kernel, int N, int splits, const double* __restrict__ part,
                                                        const double* __restrict__ target,
                                                        const int* __restrict__ tperm,
                                                        const double* __restrict__ scal, double* __restrict__ pack,
                                                        double* __restrict__ pt1, double* __restrict__ xpx_part,
                                                        double* __restrict__ tw) {
  static_assert(TPB % TILE_B == 0 && TILE_B % 32 == 0, "den tiles");
  __shared__ double red[TPB / 32];
  __shared__ double wlo[TPB / 32], whi[TPB / 32];
  const int j = blockIdx.x * TPB + threadIdx.x;
  double xpx = 0.0;
  double lo = INFINITY, hi = -INFINITY;
  if (j < N) {
    double s = 0.0;
    for (int k = 0; k < splits; ++k) s += part[(size_t)k * N + j];
    s *= GAUSS_BIAS_UNSCALE;  // the sweeps accumulate 2^64 K (exp2_poly.cuh); exact power-of-two rescale
    const double den = scal[1] * s + scal[2];
    const double w = 1.0 / den;
    const double p = s / den;
    const double x = target[j], y = target[N + j], z = target[2 * N + j];
    double4* o = reinterpret_cast<double4*>(pack + (size_t)j * 8);
    const double wb = w * GAUSS_BIAS_UNSCALE;  // sweep B multiplies 2^64 K by these
    if (estep_expand_ok(scal)) {   // layout of rowsum_tile_expanded
      const double negk = -GAUSS_SCALE * 1.4426950408889634074 / (2.0 * scal[0]);
      o[0] = make_double4(-2.0 * negk * x, -2.0 * negk * y, -2.0 * negk * z, negk * (x * x + y * y + z * z));
      o[1] = make_double4(wb, wb * x, wb * y, wb * z);
    } else {
      o[0] = make_double4(x, y, z, wb);
      o[1] = make_double4(wb * x, wb * y, wb * z, 0.0);
    }
    pt1[tperm[j]] = p;
    xpx = p * (x * x + y * y + z * z);
    lo = w;
    hi = fabs(w) < INFINITY ? w : INFINITY;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    xpx += __shfl_down_sync(0xffffffffu, xpx, o);
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) {
    red[threadIdx.x >> 5] = xpx;
    wlo[threadIdx.x >> 5] = lo;
    whi[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  constexpr int WPT = TILE_B / 32;   // warps per tile
  if (tw && threadIdx.x < TPB / TILE_B && (blockIdx.x * TPB + threadIdx.x * TILE_B) < N) {
    double l = INFINITY, h = -INFINITY;
    for (int k = 0; k < WPT; ++k) {
      l = fmin(l, wlo[threadIdx.x * WPT + k]);
      h = fmax(h, whi[threadIdx.x * WPT + k]);
    }
    const size_t t = (size_t)blockIdx.x * (TPB / TILE_B) + threadIdx.x;
    tw[2 * t] = l;
    tw[2 * t + 1] = h;
  }
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int k = 0; k < TPB / 32; ++k) s += red[k];
    xpx_part[blockIdx.x] = s;
  }
}

// ---------------------------------------------------------------------------------------------
// sweep B: row sums.   grid = (row blocks, column splits)
// part : [gridDim.y][4][M]  (P1, PX.x, PX.y, PX.z) partials, without the row factor
// ---------------------------------------------------------------------------------------------
GINGR_KERNEL((TPB_B, ESTEP_MINB_B), estep_rowsum_kernel, int M, int N, const double* __restrict__ fit,
                                                           const double* __restrict__ pack,
                                                           const double* __restrict__ scal,
                                                           const int* __restrict__ list, const int* __restrict__ nlive,
                                                           double* __restrict__ part) {
  __shared__ double4 xtile[TILE_COLS * 2];
  __shared__ __align__(16) unsigned int s_tab[GAUSS_TAB_BYTES / 4];
  gauss_tab_fill(s_tab, threadIdx.x, TPB_B);
  const int lane_off = (threadIdx.x & 15) * 8;
  const double sigma2 = scal[0];
  const double negk = -GAUSS_SCALE * 1.4426950408889634074 / (2.0 * sigma2);
  // this CTA's contiguous share of the row block's live target tiles (all tiles, in order, without a list)
  const int ntt = (N + TILE_B - 1) / TILE_B;
  const int* lst = list ? list + (size_t)blockIdx.x * ntt : nullptr;
  const int nl = list ? nlive[blockIdx.x] : ntt;
  const int per = (nl + gridDim.y - 1) / gridDim.y;
  const int e_begin = min(nl, (int)blockIdx.y * per);
  const int e_end = min(nl, e_begin + per);
  constexpr int TILES = TILE_COLS / TILE_B;   // target tiles gathered per shared-memory tile

  double yx[RB], yy[RB], yz[RB], a0[RB], a1[RB], a2[RB], a3[RB];
  int row[RB];
#pragma unroll
  for (int q = 0; q < RB; ++q) {
    row[q] = (blockIdx.x * RB + q) * TPB_B + threadIdx.x;
    const int i = min(row[q], M - 1);
    yx[q] = fit[i];
    yy[q] = fit[M + i];
    yz[q] = fit[2 * M + i];
    a0[q] = a1[q] = a2[q] = a3[q] = 0.0;
  }
  const double4* pack4 = reinterpret_cast<const double4*>(pack);
  const bool safe = estep_safe_range(scal);
  const bool expand = estep_expand_ok(scal);   // the same predicate chose the pack layout in estep_den_kernel
  double cy[RB];
#pragma unroll
  for (int q = 0; q < RB; ++q) cy[q] = negk * (yx[q] * yx[q] + yy[q] * yy[q] + yz[q] * yz[q]);
  for (int e0 = e_begin; e0 < e_end; e0 += TILES) {
    // only the last tile of the target is partial and lists are ascending: the staged columns are the first cnt
    const int ne = min(TILES, e_end - e0);
    const int last = lst ? lst[e0 + ne - 1] : e0 + ne - 1;
    const int cnt = (ne - 1) * TILE_B + min(TILE_B, N - last * TILE_B);
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * cnt; t += TPB_B) {
      const int c = t >> 1;
      const int j = (lst ? lst[e0 + c / TILE_B] : e0 + c / TILE_B) * TILE_B + c % TILE_B;
      xtile[t] = pack4[(size_t)j * 2 + (t & 1)];
    }
    __syncthreads();
    if (expand) rowsum_tile_expanded(cnt, xtile, yx, yy, yz, cy, a0, a1, a2, a3, s_tab, lane_off);
    else if (safe) rowsum_tile<true>(cnt, xtile, yx, yy, yz, a0, a1, a2, a3, negk, s_tab, lane_off);
    else rowsum_tile<false>(cnt, xtile, yx, yy, yz, a0, a1, a2, a3, negk, s_tab, lane_off);
  }
#pragma unroll
  for (int q = 0; q < RB; ++q)
    if (row[q] < M) {
      double* o = part + (size_t)blockIdx.y * 4 * M;
      o[row[q]] = a0[q];
      o[M + row[q]] = a1[q];
      o[2 * M + row[q]] = a2[q];
      o[3 * M + row[q]] = a3[q];
    }
}

// fixed-order reduction of the row partials; applies the row factor (in fit_soa order).  out: [4][M], row perm[i] of the
// caller's order
GINGR_KERNEL((TPB), estep_rowreduce_kernel, int M, int splits, const double* __restrict__ part,
                                                              const double* __restrict__ rowf,
                                                              const int* __restrict__ perm,
                                                              double* __restrict__ out) {
  // one thread per (quantity q, row i): 4 M threads instead of M (the M-thread form ran at 7 % occupancy: 51 us at
  // M = 20 000); two interleaved partial sums over the splits, fixed order
  const int idx = blockIdx.x * TPB + threadIdx.x;
  if (idx >= 4 * M) return;
  const int q = idx / M, i = idx - q * M;
  const double f = rowf ? rowf[i] : 1.0;
  double s0 = 0.0, s1 = 0.0;
  int k = 0;
  for (; k + 1 < splits; k += 2) {
    s0 += part[((size_t)k * 4 + q) * M + i];
    s1 += part[((size_t)(k + 1) * 4 + q) * M + i];
  }
  if (k < splits) s0 += part[((size_t)k * 4 + q) * M + i];
  out[(size_t)q * M + perm[i]] = f * (s0 + s1);
}

// ---------------------------------------------------------------------------------------------
// Culling.  A tile pair is dropped only when the bounds below prove that all the pairs it holds together change every
// affected sum by at most 2^-60 of itself.  Boxes are {lo x, lo y, lo z, hi x, hi y, hi z}; k = 1 / (2 sigma2).
// ---------------------------------------------------------------------------------------------
constexpr double LN2_60 = 41.588830833596715;   // 60 ln 2
constexpr double CULL_SLACK = 1.0;              // e^-1 more, for the rounding of the bounds below
constexpr double CULL_REL = 1e-12;              // relative slack on box distances

// squared distance bounds between any point of box a and any point of box b
__device__ __forceinline__ void box_d2(const double* a, const double* __restrict__ b, double& dmin2, double& dmax2) {
  dmin2 = 0.0;
  dmax2 = 0.0;
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double gap = fmax(0.0, fmax(a[d] - b[3 + d], b[d] - a[3 + d]));
    const double far = fmax(fabs(a[3 + d] - b[d]), fabs(b[3 + d] - a[d]));
    dmin2 = fma(gap, gap, dmin2);
    dmax2 = fma(far, far, dmax2);
  }
}

// union of boxes [b, e) of `boxes`
__device__ __forceinline__ void box_union(const double* __restrict__ boxes, int b, int e, double (&u)[6]) {
#pragma unroll
  for (int d = 0; d < 3; ++d) { u[d] = INFINITY; u[3 + d] = -INFINITY; }
  for (int t = b; t < e; ++t)
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      u[d] = fmin(u[d], boxes[6 * t + d]);
      u[3 + d] = fmax(u[3 + d], boxes[6 * t + 3 + d]);
    }
}

__device__ __forceinline__ double block_reduce_min(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  v = red[0];
  for (int k = 1; k < TPB / 32; ++k) v = fmin(v, red[k]);
  return v;
}

// Appends the units with keep set, in index order, to lst[base...]: a block-wide exclusive scan (no atomics, so the list
// is the same in every run).  Returns the new length.
__device__ __forceinline__ int block_append(bool keep, int unit, int* lst, int base, int* wsum) {
  const unsigned b = __ballot_sync(0xffffffffu, keep);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) wsum[wid] = __popc(b);
  __syncthreads();
  int off = base, total = base;
  for (int k = 0; k < TPB / 32; ++k) {
    if (k < wid) off += wsum[k];
    total += wsum[k];
  }
  if (keep) lst[off + __popc(b & ((1u << lane) - 1u))] = unit;
  return total;
}

// Boxes of the sweep-A model sub-tiles (SUB_A rows of fit_soa) and of the sweep-B target tiles (TILE_B columns of
// target_soa); one warp per box.
GINGR_KERNEL((TPB), estep_boxes_kernel, int M, int N, const double* __restrict__ fit, const double* __restrict__ target,
                                                      double* __restrict__ rbox, double* __restrict__ tbox) {
  const int w = (blockIdx.x * TPB + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nsub = (M + SUB_A - 1) / SUB_A, ntt = (N + TILE_B - 1) / TILE_B;
  if (w >= nsub + ntt) return;
  const bool model = w < nsub;
  const double* src = model ? fit : target;
  const int n = model ? M : N, size = model ? SUB_A : TILE_B, t = model ? w : w - nsub;
  const int b = t * size, e = min(n, b + size);
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = b + lane; i < e; i += 32)
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const double v = src[(size_t)d * n + i];
      lo[d] = fmin(lo[d], v);
      hi[d] = fmax(hi[d], v);
    }
#pragma unroll
  for (int d = 0; d < 3; ++d)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[d] = fmin(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
      hi[d] = fmax(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
    }
  if (lane < 6) (model ? rbox : tbox)[6 * t + lane] = lane < 3 ? lo[lane] : hi[lane - 3];
}

// Sweep-A live lists, one CTA per column block C.  With U_C = min_T dmax2(C, T), every column of C has a model point
// within sqrt(U_C): colsum_j >= exp(-k U_C).  A sub-tile T with k (dmin2(C, T) - U_C) >= ln M + 60 ln 2 holds pairs of
// K <= exp(-k U_C) 2^-60 / M, so all culled pairs of a column add at most 2^-60 colsum_j, whatever the row factors of
// CPD.  live[0] counts the live (C, T) pairs.
GINGR_KERNEL((TPB), estep_cull_a_kernel, int M, int N, const double* __restrict__ rbox, const double* __restrict__ tbox,
                                                       const double* __restrict__ scal, int* __restrict__ list,
                                                       int* __restrict__ nlive, unsigned long long* __restrict__ live) {
  __shared__ double red[TPB / 32];
  __shared__ int wsum[TPB / 32];
  const int nsub = (M + SUB_A - 1) / SUB_A, ntt = (N + TILE_B - 1) / TILE_B;
  constexpr int TPC = COLS_A / TILE_B;
  double cb[6];
  box_union(tbox, blockIdx.x * TPC, min(ntt, ((int)blockIdx.x + 1) * TPC), cb);
  const double sigma2 = scal[0];
  const bool ok = sigma2 > 0.0 && sigma2 < INFINITY;
  double u = INFINITY, dmin2, dmax2;
  for (int s = threadIdx.x; s < nsub; s += TPB) {
    box_d2(cb, rbox + 6 * s, dmin2, dmax2);
    u = fmin(u, dmax2);
  }
  u = block_reduce_min(u, red);
  const double bar = u * (1.0 + CULL_REL) + 2.0 * sigma2 * (log((double)M) + LN2_60 + CULL_SLACK);
  int* lst = list + (size_t)blockIdx.x * nsub;
  int n = 0;
  for (int s0 = 0; s0 < nsub; s0 += TPB) {
    const int s = s0 + threadIdx.x;
    bool keep = false;
    if (s < nsub) {
      box_d2(cb, rbox + 6 * s, dmin2, dmax2);
      keep = !(ok && dmin2 * (1.0 - CULL_REL) >= bar);
    }
    n = block_append(keep, s, lst, n, wsum);
  }
  if (threadIdx.x == 0) {
    nlive[blockIdx.x] = n;
    atomicAdd(live, (unsigned long long)n);
  }
}

// Sweep-B live lists, one CTA per row block B.  With V_B = max_T (-k dmax2(B, T) + ln min_T w), every row of B has
// P1_i >= exp(V_B) (CPD: row factor 1).  A target tile T with -k dmin2(B, T) + ln max_T w <= V_B - (ln N + 60 ln 2) holds
// terms K_ij w_j <= exp(V_B) 2^-60 / N, so all culled terms of a row add at most 2^-60 P1_i to P1_i (and 2^-60 P1_i
// max|x| to PX_i).  Nothing is culled when some w_j is not finite: the dense sums carry that NaN / Inf into P1 and PX.
// live[1] counts the live (B, T) pairs.
GINGR_KERNEL((TPB), estep_cull_b_kernel, int M, int N, const double* __restrict__ rbox, const double* __restrict__ tbox,
                                                       const double* __restrict__ tw, const double* __restrict__ scal,
                                                       int* __restrict__ list, int* __restrict__ nlive,
                                                       unsigned long long* __restrict__ live) {
  __shared__ double red[TPB / 32];
  __shared__ int wsum[TPB / 32];
  const int nsub = (M + SUB_A - 1) / SUB_A, ntt = (N + TILE_B - 1) / TILE_B;
  constexpr int SPB = ROWS_B / SUB_A;
  double rb[6];
  box_union(rbox, blockIdx.x * SPB, min(nsub, ((int)blockIdx.x + 1) * SPB), rb);
  const double sigma2 = scal[0];
  const double k = 1.0 / (2.0 * sigma2);
  double v = -INFINITY, dmin2, dmax2;
  int bad = !(sigma2 > 0.0 && sigma2 < INFINITY);
  for (int t = threadIdx.x; t < ntt; t += TPB) {
    box_d2(rb, tbox + 6 * t, dmin2, dmax2);
    if (!(tw[2 * t + 1] < INFINITY)) bad = 1;
    v = fmax(v, -k * dmax2 * (1.0 + CULL_REL) + log(tw[2 * t]));
  }
  bad = __syncthreads_or(bad);
  v = -block_reduce_min(-v, red);
  const double bar = v - (log((double)N) + LN2_60 + CULL_SLACK);
  int* lst = list + (size_t)blockIdx.x * ntt;
  int n = 0;
  for (int t0 = 0; t0 < ntt; t0 += TPB) {
    const int t = t0 + threadIdx.x;
    bool keep = false;
    if (t < ntt) {
      box_d2(rb, tbox + 6 * t, dmin2, dmax2);
      keep = bad || -k * dmin2 * (1.0 - CULL_REL) + log(tw[2 * t + 1]) > bar;
    }
    n = block_append(keep, t, lst, n, wsum);
  }
  if (threadIdx.x == 0) {
    nlive[blockIdx.x] = n;
    atomicAdd(live + 1, (unsigned long long)n);
  }
}

// sets *flag when any of the n doubles is NaN / Inf (the E-step kernels assume finite input, exp2_poly.cuh)
__global__ void validate_finite_kernel(int n, const double* __restrict__ v, int* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !(fabs(v[i]) < INFINITY)) *flag = 1;
}

// AoS [n][3] -> SoA [3][n]
__global__ void aos_to_soa_kernel(int n, const double* __restrict__ aos, double* __restrict__ soa) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    soa[i] = aos[3 * i];
    soa[n + i] = aos[3 * i + 1];
    soa[2 * n + i] = aos[3 * i + 2];
  }
}

// CPD scalars: scal[0] = sigma2 (input), scal[3] = w, scal[4] = M/N_total -> scal[1] = a = 1, scal[2] = c
__global__ void estep_cpd_scalars_kernel(double* scal) {
  const double sigma2 = scal[0], w = scal[3], ratio = scal[4];
  const double t = 2.0 * 3.14159265358979323846 * sigma2;
  scal[1] = 1.0;
  scal[2] = w / (1.0 - w) * (t * sqrt(t)) * ratio;  // pow(2 pi sigma2, 3/2)  CPD.scala:69-70
}

// BCPD row factors and scalars.  scal[0] = sigma2, scal[3] = w, scal[5] = s, scal[6] = 1/N_total
__global__ void estep_bcpd_rowf_kernel(int M, const double* __restrict__ sigma_mm, const double* __restrict__ alpha,
                                       double* __restrict__ scal, double* __restrict__ rowf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const double sigma2 = scal[0], w = scal[3], s = scal[5];
  if (i < M) {
    const double t = 2.0 * 3.14159265358979323846 * sigma2;
    const double norm = 1.0 / (t * sqrt(t));
    rowf[i] = (1.0 - w) * norm * exp(-s / (2.0 * sigma2) * (3.0 * sigma_mm[i])) * alpha[i];
  }
  if (i == 0) {
    scal[1] = 1.0 - w;
    scal[2] = w * scal[6];
  }
}

// ---------------------------------------------------------------------------------------------
// computeInitialSigma2 (CPD.scala:81-90): sum_ij |x_j - m_i|^2 / (3 N M), evaluated in O(M + N) about the
// common centroid c:  sum_ij |x_j - m_i|^2 = N sum|m_i - c|^2 + M sum|x_j - c|^2 - 2 (sum(m_i - c)).(sum(x_j - c))
// (centring keeps the three terms free of cancellation).  One CTA, fixed-order tree reductions.
// m: AoS [M][3], x: SoA [3][N].
// ---------------------------------------------------------------------------------------------
__device__ double block_sum_1024(double v, double* red) {
  __syncthreads();
  red[threadIdx.x] = v;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  return red[0];
}

__global__ void __launch_bounds__(1024) initial_sigma2_kernel(int M, const double* __restrict__ m, int N,
                                                              const double* __restrict__ x,
                                                              double* __restrict__ out) {
  __shared__ double red[1024];
  double c[3];
  for (int d = 0; d < 3; ++d) {
    double s = 0.0;
    for (int i = threadIdx.x; i < M; i += 1024) s += m[3 * i + d];
    for (int j = threadIdx.x; j < N; j += 1024) s += x[(size_t)d * N + j];
    c[d] = block_sum_1024(s, red) / (double)(M + N);
  }
  double a = 0.0, sm[3] = {0, 0, 0};
  for (int i = threadIdx.x; i < M; i += 1024)
    for (int d = 0; d < 3; ++d) {
      const double v = m[3 * i + d] - c[d];
      a = fma(v, v, a);
      sm[d] += v;
    }
  double b = 0.0, sx[3] = {0, 0, 0};
  for (int j = threadIdx.x; j < N; j += 1024)
    for (int d = 0; d < 3; ++d) {
      const double v = x[(size_t)d * N + j] - c[d];
      b = fma(v, v, b);
      sx[d] += v;
    }
  const double A = block_sum_1024(a, red), B = block_sum_1024(b, red);
  double dot = 0.0;
  for (int d = 0; d < 3; ++d) {
    const double p = block_sum_1024(sm[d], red);
    const double q = block_sum_1024(sx[d], red);
    dot += p * q;
  }
  if (threadIdx.x == 0) out[0] = ((double)N * A + (double)M * B - 2.0 * dot) / (3.0 * (double)N * (double)M);
}

int32_t initial_sigma2_enqueue(gingr_ctx* ctx, int M, const double* d_pts_aos, int N, const double* d_target_soa,
                               double* d_out) {
  initial_sigma2_kernel<<<1, 1024, 0, ctx->stream>>>(M, d_pts_aos, N, d_target_soa, d_out);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// Number of splits s (1 <= s <= max_splits) of the streamed dimension such that the grid of blocks * s CTAs fills
// whole waves of `capacity` resident CTAs: the kernels are throughput bound, so a last wave that is 10 % full
// costs a whole wave (ncu: 4.05 waves/SM on sweep B before this planner).  Prefers 2..6 waves.
static int pick_splits_for_waves(int blocks, int max_splits, int capacity) {
  if (blocks >= 8 * capacity || max_splits <= 1) return 1;
  int best = 1;
  double best_score = -1.0;
  for (int s = 1; s <= max_splits; ++s) {
    const double ctas = (double)blocks * s;
    const double waves = ctas / capacity;
    if (waves > 6.0 && best_score >= 0.0) break;
    const double fill = waves / ceil(waves);
    // below one wave: plain parallelism counts; above: fill of the last wave, slight preference for more waves
    const double score = waves < 1.0 ? waves : 1.0 + fill + 0.002 * waves;
    if (score > best_score) {
      best_score = score;
      best = s;
    }
  }
  return best;
}

void estep_plan(const gingr_ctx* ctx, int M, int N, EstepPlan* p) {
  int occ_a = 4, occ_b = 4;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_a, estep_colsum_kernel, TPB, 0);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_b, estep_rowsum_kernel, TPB_B, 0);
  p->nsub = ceil_div(M, SUB_A);
  p->ntt = ceil_div(N, TILE_B);
  p->col_blocks = ceil_div(N, COLS_A);
  p->row_splits = pick_splits_for_waves(p->col_blocks, ceil_div(M, 128), max(occ_a, 1) * ctx->num_sms);
  p->row_blocks = ceil_div(M, ROWS_B);
  p->col_splits = pick_splits_for_waves(p->row_blocks, ceil_div(N, 128), max(occ_b, 1) * ctx->num_sms);
  p->den_blocks = ceil_div(N, TPB);
  p->cull = (double)M * (double)N >= CULL_MIN_PAIRS;
  // tuning / test overrides (tools/time_estep_phases.py, tools/time_estep_cull.py, tests/test_estep_cull_gpu.py)
  if (const char* e = getenv("GINGR_ESTEP_SPLITS_A")) if (atoi(e) > 0) p->row_splits = std::min(atoi(e), ceil_div(M, 128));
  if (const char* e = getenv("GINGR_ESTEP_SPLITS_B")) if (atoi(e) > 0) p->col_splits = std::min(atoi(e), ceil_div(N, 128));
  if (const char* e = getenv("GINGR_ESTEP_CULL")) if (*e) p->cull = atoi(e) != 0;
  if (getenv("GINGR_ESTEP_VERBOSE"))
    fprintf(stderr, "estep plan M=%d N=%d: sweep A %d x %d CTAs (occupancy %d), sweep B %d x %d CTAs (occupancy %d), cull %d\n", M,
            N, p->col_blocks, p->row_splits, occ_a, p->row_blocks, p->col_splits, occ_b, (int)p->cull);
}

// k-d order of n points (AoS): perm[k] = index of the point at position k.  Each range is split along the longest edge of
// its bounding box at the median, rounded to a multiple of `big` while the range is longer than `big` and of `small`
// below, so every aligned run of `big` and of `small` points is a subtree.  Non-finite input keeps the identity order.
static void kd_order(const double* aos, int n, int big, int small, std::vector<int32_t>& perm) {
  perm.resize(n);
  for (int k = 0; k < n; ++k) perm[k] = k;
  for (size_t k = 0; k < (size_t)3 * n; ++k)
    if (!(fabs(aos[k]) < INFINITY)) return;
  std::vector<std::pair<int, int>> todo{{0, n}};
  while (!todo.empty()) {
    const auto [lo, hi] = todo.back();
    todo.pop_back();
    const int g = hi - lo > big ? big : small;
    if (hi - lo <= g) continue;
    double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int k = lo; k < hi; ++k)
      for (int d = 0; d < 3; ++d) {
        mn[d] = std::min(mn[d], aos[3 * (size_t)perm[k] + d]);
        mx[d] = std::max(mx[d], aos[3 * (size_t)perm[k] + d]);
      }
    int ax = 0;
    for (int d = 1; d < 3; ++d)
      if (mx[d] - mn[d] > mx[ax] - mn[ax]) ax = d;
    const int mid = lo + ceil_div(hi - lo, g) / 2 * g;
    std::nth_element(perm.begin() + lo, perm.begin() + mid, perm.begin() + hi, [&](int a, int b) {
      const double u = aos[3 * (size_t)a + ax], v = aos[3 * (size_t)b + ax];
      return u < v || (u == v && a < b);
    });
    todo.push_back({lo, mid});
    todo.push_back({mid, hi});
  }
}

void estep_row_order(const double* aos, int M, std::vector<int32_t>& perm) { kd_order(aos, M, ROWS_B, SUB_A, perm); }
void estep_target_order(const double* aos, int N, std::vector<int32_t>& perm) { kd_order(aos, N, COLS_A, TILE_B, perm); }

int32_t EstepWorkspace::ensure(gingr_ctx* ctx, int M, int N) {
  estep_plan(ctx, M, N, &plan);
  GINGR_CUDA_TRY(ctx, colpart.alloc((size_t)plan.row_splits * N));
  GINGR_CUDA_TRY(ctx, pack.alloc((size_t)N * 8));
  GINGR_CUDA_TRY(ctx, pt1.alloc((size_t)N));
  GINGR_CUDA_TRY(ctx, xpx_part.alloc((size_t)plan.den_blocks));
  GINGR_CUDA_TRY(ctx, rowpart.alloc((size_t)plan.col_splits * 4 * M));
  GINGR_CUDA_TRY(ctx, rows.alloc((size_t)4 * M));
  GINGR_CUDA_TRY(ctx, fit_soa.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, rowf.alloc((size_t)M));
  GINGR_CUDA_TRY(ctx, scal.alloc(16));
  GINGR_CUDA_TRY(ctx, row_perm.alloc((size_t)M));
  GINGR_CUDA_TRY(ctx, rbox.alloc((size_t)6 * plan.nsub));
  GINGR_CUDA_TRY(ctx, tbox.alloc((size_t)6 * plan.ntt));
  GINGR_CUDA_TRY(ctx, tw.alloc((size_t)2 * plan.den_blocks * (TPB / TILE_B)));
  GINGR_CUDA_TRY(ctx, list_a.alloc((size_t)plan.col_blocks * plan.nsub));
  GINGR_CUDA_TRY(ctx, list_b.alloc((size_t)plan.row_blocks * plan.ntt));
  GINGR_CUDA_TRY(ctx, nlive.alloc((size_t)plan.col_blocks + plan.row_blocks));
  if (!live.p) {
    GINGR_CUDA_TRY(ctx, live.alloc(2));
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(live.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
  }
  return GINGR_OK;
}

int32_t EstepWorkspace::set_row_order(gingr_ctx* ctx, int M, const int32_t* perm) {
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(row_perm.p, perm, sizeof(int32_t) * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GINGR_OK;
}

// Enqueue the E-step on ctx->stream.  fit_soa (in the order of ws.row_perm) / rowf (may be null; same order) / scal must be
// set up by the caller: scal[0] = sigma2, scal[1] = a, scal[2] = c.  target_soa is in the order of target_perm.
// Results in the callers' orders: ws.pt1 [N], ws.rows [4][M], ws.xpx_part.
int32_t estep_enqueue(gingr_ctx* ctx, EstepWorkspace& ws, int M, int N, const double* target_soa, const int32_t* target_perm,
                      bool use_rowf, const EstepEvents* ev) {
  const EstepPlan& p = ws.plan;
  const double* rowf = use_rowf ? ws.rowf.p : nullptr;
  // the bounds assume a row factor of 1 (CPD)
  const bool cull = p.cull && !use_rowf;
  cudaStream_t st = ctx->stream;
  if (ev) cudaEventRecord(ev->a0, st);
  if (cull) {
    GINGR_LAUNCH(ctx, estep_boxes_kernel, ceil_div(32 * (p.nsub + p.ntt), TPB), TPB, 0, st, M, N, ws.fit_soa.p, target_soa,
                 ws.rbox.p, ws.tbox.p);
    GINGR_LAUNCHED(ctx);
    GINGR_LAUNCH(ctx, estep_cull_a_kernel, p.col_blocks, TPB, 0, st, M, N, ws.rbox.p, ws.tbox.p, ws.scal.p, ws.list_a.p, ws.nlive.p,
                 ws.live.p);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_LAUNCH(ctx, estep_colsum_kernel, dim3(p.col_blocks, p.row_splits), TPB, 0, st, M, N, ws.fit_soa.p, rowf, target_soa,
               ws.scal.p, cull ? ws.list_a.p : nullptr, ws.nlive.p, ws.colpart.p);
  if (ev) cudaEventRecord(ev->a1, st);
  GINGR_LAUNCHED(ctx);
  GINGR_LAUNCH(ctx, estep_den_kernel, p.den_blocks, TPB, 0, st, N, p.row_splits, ws.colpart.p, target_soa, target_perm, ws.scal.p,
               ws.pack.p, ws.pt1.p, ws.xpx_part.p, cull ? ws.tw.p : nullptr);
  GINGR_LAUNCHED(ctx);
  if (ev) cudaEventRecord(ev->b0, st);
  int* nlive_b = ws.nlive.p + p.col_blocks;
  if (cull) {
    GINGR_LAUNCH(ctx, estep_cull_b_kernel, p.row_blocks, TPB, 0, st, M, N, ws.rbox.p, ws.tbox.p, ws.tw.p, ws.scal.p, ws.list_b.p,
                 nlive_b, ws.live.p);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_LAUNCH(ctx, estep_rowsum_kernel, dim3(p.row_blocks, p.col_splits), TPB_B, 0, st, M, N, ws.fit_soa.p, ws.pack.p, ws.scal.p,
               cull ? ws.list_b.p : nullptr, nlive_b, ws.rowpart.p);
  if (ev) cudaEventRecord(ev->b1, st);
  GINGR_LAUNCHED(ctx);
  GINGR_LAUNCH(ctx, estep_rowreduce_kernel, ceil_div(4 * M, TPB), TPB, 0, st, M, p.col_splits, ws.rowpart.p, rowf, ws.row_perm.p,
               ws.rows.p);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t aos_to_soa_enqueue(gingr_ctx* ctx, int n, const double* d_aos, double* d_soa) {
  aos_to_soa_kernel<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, d_aos, d_soa);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t validate_finite_enqueue(gingr_ctx* ctx, int n, const double* d_v, int* d_flag) {
  validate_finite_kernel<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, d_v, d_flag);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

int32_t estep_cpd_scalars_enqueue(gingr_ctx* ctx, double* d_scal) {
  estep_cpd_scalars_kernel<<<1, 1, 0, ctx->stream>>>(d_scal);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

int32_t estep_bcpd_rowf_enqueue(gingr_ctx* ctx, int M, const double* d_sigma_mm, const double* d_alpha,
                                double* d_scal, double* d_rowf) {
  estep_bcpd_rowf_kernel<<<ceil_div(M, 256), 256, 0, ctx->stream>>>(M, d_sigma_mm, d_alpha, d_scal, d_rowf);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

}  // namespace gingr
