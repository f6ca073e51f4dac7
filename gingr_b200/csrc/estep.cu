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
#define ESTEP_MINB_B 2
#endif
constexpr int TPB = 256;       // threads per CTA in both sweeps
constexpr int CA = ESTEP_CA;   // columns per thread, sweep A
constexpr int RB = ESTEP_RB;   // rows per thread, sweep B
constexpr int TILE_ROWS = 512; // rows staged per shared-memory tile in sweep A
constexpr int TILE_COLS = 256; // columns staged per shared-memory tile in sweep B

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
                                                           double* __restrict__ part) {
  __shared__ double4 ytile[TILE_ROWS];
  __shared__ __align__(16) unsigned int s_tab[GAUSS_TAB_BYTES / 4];
  gauss_tab_fill(s_tab, threadIdx.x, TPB);
  const int lane_off = (threadIdx.x & 15) * 8;
  const double sigma2 = scal[0];
  const double negk = -GAUSS_SCALE * 1.4426950408889634074 / (2.0 * sigma2);
  const int rows_per_split = (M + gridDim.y - 1) / gridDim.y;
  const int i_begin = blockIdx.y * rows_per_split;
  const int i_end = min(M, i_begin + rows_per_split);

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
    for (int i0 = i_begin; i0 < i_end; i0 += TILE_ROWS) {
      const int cnt = min(TILE_ROWS, i_end - i0);
      __syncthreads();
      for (int t = threadIdx.x; t < cnt; t += TPB) {
        const int i = i0 + t;
        const double a = fit[i], b = fit[M + i], c = fit[2 * M + i];
        ytile[t] = make_double4(a, b, c, negk * (a * a + b * b + c * c));
      }
      __syncthreads();
      colsum_tile_expanded(cnt, ytile, xj, yj, zj, cx, acc, s_tab, lane_off);
    }
  } else {
    for (int i0 = i_begin; i0 < i_end; i0 += TILE_ROWS) {
      const int cnt = min(TILE_ROWS, i_end - i0);
      __syncthreads();
      for (int t = threadIdx.x; t < cnt; t += TPB) {
        const int i = i0 + t;
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
// ---------------------------------------------------------------------------------------------
GINGR_KERNEL((TPB), estep_den_kernel, int N, int splits, const double* __restrict__ part,
                                                        const double* __restrict__ target,
                                                        const double* __restrict__ scal, double* __restrict__ pack,
                                                        double* __restrict__ pt1, double* __restrict__ xpx_part) {
  __shared__ double red[TPB / 32];
  const int j = blockIdx.x * TPB + threadIdx.x;
  double xpx = 0.0;
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
    pt1[j] = p;
    xpx = p * (x * x + y * y + z * z);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) xpx += __shfl_down_sync(0xffffffffu, xpx, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = xpx;
  __syncthreads();
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
GINGR_KERNEL((TPB, ESTEP_MINB_B), estep_rowsum_kernel, int M, int N, const double* __restrict__ fit,
                                                           const double* __restrict__ pack,
                                                           const double* __restrict__ scal,
                                                           double* __restrict__ part) {
  __shared__ double4 xtile[TILE_COLS * 2];
  __shared__ __align__(16) unsigned int s_tab[GAUSS_TAB_BYTES / 4];
  gauss_tab_fill(s_tab, threadIdx.x, TPB);
  const int lane_off = (threadIdx.x & 15) * 8;
  const double sigma2 = scal[0];
  const double negk = -GAUSS_SCALE * 1.4426950408889634074 / (2.0 * sigma2);
  const int cols_per_split = (N + gridDim.y - 1) / gridDim.y;
  const int j_begin = blockIdx.y * cols_per_split;
  const int j_end = min(N, j_begin + cols_per_split);

  double yx[RB], yy[RB], yz[RB], a0[RB], a1[RB], a2[RB], a3[RB];
  int row[RB];
#pragma unroll
  for (int q = 0; q < RB; ++q) {
    row[q] = (blockIdx.x * RB + q) * TPB + threadIdx.x;
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
  for (int j0 = j_begin; j0 < j_end; j0 += TILE_COLS) {
    const int cnt = min(TILE_COLS, j_end - j0);
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * cnt; t += TPB) xtile[t] = pack4[(size_t)j0 * 2 + t];
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

// fixed-order reduction of the row partials; applies the row factor.  out: [4][M]
GINGR_KERNEL((TPB), estep_rowreduce_kernel, int M, int splits, const double* __restrict__ part,
                                                              const double* __restrict__ rowf,
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
  out[(size_t)q * M + i] = f * (s0 + s1);
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
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_b, estep_rowsum_kernel, TPB, 0);
  p->col_blocks = ceil_div(N, TPB * CA);
  p->row_splits = pick_splits_for_waves(p->col_blocks, ceil_div(M, 128), max(occ_a, 1) * ctx->num_sms);
  p->row_blocks = ceil_div(M, TPB * RB);
  p->col_splits = pick_splits_for_waves(p->row_blocks, ceil_div(N, 128), max(occ_b, 1) * ctx->num_sms);
  p->den_blocks = ceil_div(N, TPB);
  // tuning overrides (tools/time_estep_phases.py)
  if (const char* e = getenv("GINGR_ESTEP_SPLITS_A")) if (atoi(e) > 0) p->row_splits = std::min(atoi(e), ceil_div(M, 128));
  if (const char* e = getenv("GINGR_ESTEP_SPLITS_B")) if (atoi(e) > 0) p->col_splits = std::min(atoi(e), ceil_div(N, 128));
  if (getenv("GINGR_ESTEP_VERBOSE"))
    fprintf(stderr, "estep plan M=%d N=%d: sweep A %d x %d CTAs (occupancy %d), sweep B %d x %d CTAs (occupancy %d)\n", M, N,
            p->col_blocks, p->row_splits, occ_a, p->row_blocks, p->col_splits, occ_b);
}

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
  return GINGR_OK;
}

// Enqueue the E-step on ctx->stream.  fit_soa / rowf (may be null) / scal must be set up by the caller:
// scal[0] = sigma2, scal[1] = a, scal[2] = c.  Results: ws.pt1 [N], ws.rows [4][M], ws.xpx_part.
int32_t estep_enqueue(gingr_ctx* ctx, EstepWorkspace& ws, int M, int N, const double* target_soa, bool use_rowf,
                      const EstepEvents* ev) {
  const EstepPlan& p = ws.plan;
  const double* rowf = use_rowf ? ws.rowf.p : nullptr;
  cudaStream_t st = ctx->stream;
  if (ev) cudaEventRecord(ev->a0, st);
  GINGR_LAUNCH(ctx, estep_colsum_kernel, dim3(p.col_blocks, p.row_splits), TPB, 0, st, M, N, ws.fit_soa.p, rowf, target_soa,
                                                                        ws.scal.p, ws.colpart.p);
  if (ev) cudaEventRecord(ev->a1, st);
  GINGR_LAUNCHED(ctx);
  GINGR_LAUNCH(ctx, estep_den_kernel, p.den_blocks, TPB, 0, st, N, p.row_splits, ws.colpart.p, target_soa, ws.scal.p, ws.pack.p,
                                                 ws.pt1.p, ws.xpx_part.p);
  GINGR_LAUNCHED(ctx);
  if (ev) cudaEventRecord(ev->b0, st);
  GINGR_LAUNCH(ctx, estep_rowsum_kernel, dim3(p.row_blocks, p.col_splits), TPB, 0, st, M, N, ws.fit_soa.p, ws.pack.p, ws.scal.p,
                                                                        ws.rowpart.p);
  if (ev) cudaEventRecord(ev->b1, st);
  GINGR_LAUNCHED(ctx);
  GINGR_LAUNCH(ctx, estep_rowreduce_kernel, ceil_div(4 * M, TPB), TPB, 0, st, M, p.col_splits, ws.rowpart.p, rowf, ws.rows.p);
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
