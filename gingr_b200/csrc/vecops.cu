// vecops.cu -- K3c: HBM-bound passes over the GPMM basis and small dense helpers (sm_100a).
//
//   gemv_rows   out[k] = sum_a Phi[k][a] v[a]      instance / posterior mean evaluation at the mesh points:
//               scalismo `instance(alpha) = ref + mean + basis (sqrt(lambda) * alpha)` (SURVEY.md A1), call sites
//               GingrAlgorithm.scala:211, :222, :224 and ModelFittingParameters.scala:134.  One warp per row,
//               two right-hand sides per pass (instance(alpha_old) and instance(alpha_new) share the read) while both
//               fit shared memory (r <= 12 800), one per pass up to r = 25 600.
//   gemvT       out[a] = s_a sum_k Phi[k][a] u[k]   right-hand side Q^T L^-1 (y - m) of the regression
//               (SURVEY.md A3).  Thread per column, rows split over CTAs, fixed-order reduction.
// Both read Phi (8 * 3M * r bytes) exactly once; Phi is row-major [3M][rp] so both are fully coalesced.
#include <stdint.h>

#include <algorithm>

#include "batch.cuh"
#include "posterior.cuh"

namespace gingr {

GINGR_KERNEL_T((int NVEC), (NVEC), (256), gemv_rows_kernel, int rows, int r, int rp, const double* __restrict__ phi,
               const double* __restrict__ v0, const double* __restrict__ v1, const double* __restrict__ scale /*may be null*/,
               double* __restrict__ out0, double* __restrict__ out1) {
  extern __shared__ double sv[];  // [NVEC][r]
  for (int a = threadIdx.x; a < r; a += 256) {
    const double sc = scale ? scale[a] : 1.0;   // instance(alpha): v = sqrt(lambda) * alpha, folded into the staging
    sv[a] = scale ? sc * v0[a] : v0[a];
    if (NVEC > 1) sv[r + a] = scale ? sc * v1[a] : v1[a];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * 256 + threadIdx.x) >> 5, nwarps = (gridDim.x * 256) >> 5;
  for (int k = warp; k < rows; k += nwarps) {
    const double* row = phi + (size_t)k * rp;
    double s0 = 0.0, s1 = 0.0;
    // rp is a multiple of 8: 16-byte vector loads
    for (int a = lane * 2; a < r; a += 64) {
      const double2 p = *reinterpret_cast<const double2*>(row + a);
      s0 = fma(p.x, sv[a], s0);
      if (a + 1 < r) s0 = fma(p.y, sv[a + 1], s0);
      if (NVEC > 1) {
        s1 = fma(p.x, sv[r + a], s1);
        if (a + 1 < r) s1 = fma(p.y, sv[r + a + 1], s1);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      if (NVEC > 1) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    if (lane == 0) {
      out0[k] = s0;
      if (NVEC > 1) out1[k] = s1;
    }
  }
}

constexpr int GT_ROWS = 512;  // max rows per CTA of gemvT

// rows per CTA: ~2 CTAs of rows per SM so that small problems (C1-C3: a few hundred rows) still spread over the
// machine instead of one CTA walking every row with dependent loads; large problems keep long streaming CTAs
static int gemvT_rows_per_cta(const gingr_ctx* ctx, int rows) {
  const int want = ceil_div(std::max(rows, 1), 2 * ctx->num_sms);
  return std::max(16, std::min(GT_ROWS, (want + 3) / 4 * 4));
}

GINGR_KERNEL((256), gemvT_kernel, int rows, int rp, int rows_per_cta, const double* __restrict__ phi,
                                                    const double* __restrict__ u, double* __restrict__ part) {
  __shared__ double su[GT_ROWS];
  const int k0 = blockIdx.y * rows_per_cta;
  const int cnt = min(rows_per_cta, rows - k0);
  for (int t = threadIdx.x; t < cnt; t += 256) su[t] = u[k0 + t];
  __syncthreads();
  const int a = blockIdx.x * 256 + threadIdx.x;
  if (a >= rp) return;
  const double* p = phi + (size_t)k0 * rp + a;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int t = 0;
  for (; t + 4 <= cnt; t += 4) {
    s0 = fma(p[(size_t)t * rp], su[t], s0);
    s1 = fma(p[(size_t)(t + 1) * rp], su[t + 1], s1);
    s2 = fma(p[(size_t)(t + 2) * rp], su[t + 2], s2);
    s3 = fma(p[(size_t)(t + 3) * rp], su[t + 3], s3);
  }
  for (; t < cnt; ++t) s0 = fma(p[(size_t)t * rp], su[t], s0);
  part[(size_t)blockIdx.y * rp + a] = (s0 + s1) + (s2 + s3);
}

// Sum of the `splits` partial vectors, fixed order (deterministic).  A CTA owns 32 columns; 8 groups of threads walk the
// splits interleaved and are combined through shared memory: the one-thread-per-column form walked ~300 strided loads in a
// dependent add chain from 8 CTAs (35 us at rank 2000, more than the streaming pass it follows on 8 GPUs).
GINGR_KERNEL((256), gemvT_reduce_kernel, int r, int rp, int splits, const double* __restrict__ part,
                                                           const double* __restrict__ scale, double* __restrict__ out) {
  __shared__ double sp[8][33];
  const int c = threadIdx.x & 31, q = threadIdx.x >> 5;
  const int a = blockIdx.x * 32 + c;
  double s0 = 0.0, s1 = 0.0;
  if (a < r) {
    int k = q;
    for (; k + 8 < splits; k += 16) {
      s0 += part[(size_t)k * rp + a];
      s1 += part[(size_t)(k + 8) * rp + a];
    }
    if (k < splits) s0 += part[(size_t)k * rp + a];
  }
  sp[q][c] = s0 + s1;
  __syncthreads();
  if (q == 0 && a < r) {
    const double s = ((sp[0][c] + sp[1][c]) + (sp[2][c] + sp[3][c])) + ((sp[4][c] + sp[5][c]) + (sp[6][c] + sp[7][c]));
    out[a] = scale ? scale[a] * s : s;
  }
}

// y = A x for a dense r x r row-major matrix: one warp per row, four independent accumulators per lane (the
// one-accumulator form ran at 1.7 TB/s on a matrix that mostly sits in L2)
GINGR_KERNEL((256), dense_matvec_kernel, int r, const double* __restrict__ A, int ld,
                                                           const double* __restrict__ x, double* __restrict__ y,
                                                           int* __restrict__ flag_in, int* __restrict__ flag_out) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * 256 + threadIdx.x) >> 5;
  if (row >= r) return;
  const double* p = A + (size_t)row * ld;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  bool bad_in = false;
  int b = lane;
  for (; b + 96 < r; b += 128) {
    const double x0 = x[b], x1 = x[b + 32], x2 = x[b + 64], x3 = x[b + 96];
    bad_in = bad_in || !(fabs(x0) < INFINITY) || !(fabs(x1) < INFINITY) || !(fabs(x2) < INFINITY) || !(fabs(x3) < INFINITY);
    s0 = fma(p[b], x0, s0);
    s1 = fma(p[b + 32], x1, s1);
    s2 = fma(p[b + 64], x2, s2);
    s3 = fma(p[b + 96], x3, s3);
  }
  for (; b < r; b += 32) {
    const double xb = x[b];
    bad_in = bad_in || !(fabs(xb) < INFINITY);
    s0 = fma(p[b], xb, s0);
  }
  double s = (s0 + s1) + (s2 + s3);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  // optional finiteness flags of the operand / the result (what separate check_finite launches did)
  if (flag_in && row == 0 && __any_sync(0xffffffffu, bad_in) && lane == 0) *flag_in = 1;
  if (lane == 0) {
    y[row] = s;
    if (flag_out && !(fabs(s) < INFINITY)) *flag_out = 1;
  }
}

// The same product with TWO warps per row and 16-byte loads, four per lane in flight: a 32 MB matrix that the Gram has pushed
// out of L2 ran at 2.2 TB/s with one warp per row and 8-byte loads (2000 warps x 1 KB in flight).  Needs 16-byte aligned A and
// x and an even pitch.  Block = 4 rows x 2 halves; the halves meet in shared memory (fixed order).
GINGR_KERNEL((256), dense_matvec2_kernel, int r, const double* __restrict__ A, int ld, const double* __restrict__ x,
             double* __restrict__ y, int* __restrict__ flag_in, int* __restrict__ flag_out) {
  __shared__ double sp[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = blockIdx.x * 4 + (warp >> 1), half = warp & 1;
  double s = 0.0;
  bool bad_in = false;
  if (row < r) {
    const int n2 = r >> 1, h2 = (n2 + 1) >> 1;                 // pairs of columns; the first half takes h2 of them
    const int b1 = half ? n2 : h2;
    const double2* p2 = reinterpret_cast<const double2*>(A + (size_t)row * ld);
    const double2* x2 = reinterpret_cast<const double2*>(x);
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, a4 = 0.0, a5 = 0.0, a6 = 0.0, a7 = 0.0;
    int b = (half ? h2 : 0) + lane;
    for (; b + 96 < b1; b += 128) {
      const double2 m0 = p2[b], m1 = p2[b + 32], m2 = p2[b + 64], m3 = p2[b + 96];
      const double2 v0 = x2[b], v1 = x2[b + 32], v2 = x2[b + 64], v3 = x2[b + 96];
      bad_in = bad_in || !(fabs(v0.x) < INFINITY) || !(fabs(v0.y) < INFINITY) || !(fabs(v1.x) < INFINITY) || !(fabs(v1.y) < INFINITY) ||
               !(fabs(v2.x) < INFINITY) || !(fabs(v2.y) < INFINITY) || !(fabs(v3.x) < INFINITY) || !(fabs(v3.y) < INFINITY);
      a0 = fma(m0.x, v0.x, a0); a1 = fma(m0.y, v0.y, a1);
      a2 = fma(m1.x, v1.x, a2); a3 = fma(m1.y, v1.y, a3);
      a4 = fma(m2.x, v2.x, a4); a5 = fma(m2.y, v2.y, a5);
      a6 = fma(m3.x, v3.x, a6); a7 = fma(m3.y, v3.y, a7);
    }
    for (; b < b1; b += 32) {
      const double2 m0 = p2[b], v0 = x2[b];
      bad_in = bad_in || !(fabs(v0.x) < INFINITY) || !(fabs(v0.y) < INFINITY);
      a0 = fma(m0.x, v0.x, a0); a1 = fma(m0.y, v0.y, a1);
    }
    if (half == 1 && (r & 1) && lane == 0) {                   // odd r: the last column
      const double xv = x[r - 1];
      bad_in = bad_in || !(fabs(xv) < INFINITY);
      a0 = fma(A[(size_t)row * ld + r - 1], xv, a0);
    }
    s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (flag_in && row == 0 && __any_sync(0xffffffffu, bad_in) && lane == 0) *flag_in = 1;
  }
  if (lane == 0) sp[warp] = s;
  __syncthreads();
  if (half == 0 && lane == 0 && row < r) {
    const double t = sp[warp] + sp[warp + 1];
    y[row] = t;
    if (flag_out && !(fabs(t) < INFINITY)) *flag_out = 1;
  }
}

__global__ void transpose_kernel(int n, const double* __restrict__ A, int lda, double* __restrict__ B, int ldb) {
  __shared__ double tile[32][33];
  const int x = blockIdx.x * 32 + threadIdx.x, y0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (x < n && y0 + j < n) tile[j][threadIdx.x] = A[(size_t)(y0 + j) * lda + x];
  __syncthreads();
  const int xo = blockIdx.y * 32 + threadIdx.x, yo0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (xo < n && yo0 + j < n) B[(size_t)(yo0 + j) * ldb + xo] = tile[threadIdx.x][j];
}

__global__ void slab_transpose_kernel(int rows, int nc, const double* __restrict__ tmp, double* __restrict__ dst,
                                      int ld_dst) {
  __shared__ double tile[32][33];
  const int k = blockIdx.x * 32 + threadIdx.x;  // row of Phi (contiguous in tmp)
  const int j0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (k < rows && j0 + j < nc) tile[j][threadIdx.x] = tmp[(size_t)(j0 + j) * rows + k];
  __syncthreads();
  const int jo = j0 + threadIdx.x, k0 = blockIdx.x * 32;
  for (int q = threadIdx.y; q < 32; q += 8)
    if (jo < nc && k0 + q < rows) dst[(size_t)(k0 + q) * ld_dst + jo] = tile[threadIdx.x][q];
}

GINGR_KERNEL_NB(build_regression_system_kernel, int r, int rp, const double* __restrict__ S, double eps,
                                               double* __restrict__ B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int a = blockIdx.y;
  if (b >= rp) return;
  B[(size_t)a * rp + b] = (b < r ? S[(size_t)a * rp + b] : 0.0) + (a == b ? eps : 0.0);
  B[(size_t)(r + a) * rp + b] = a == b ? 1.0 : 0.0;
}

GINGR_KERNEL_NB(add_vectors_kernel, int n, const double* __restrict__ a, const double* __restrict__ b,
                                   double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}

int32_t slab_transpose_enqueue(gingr_ctx* ctx, int rows, int nc, const double* d_tmp, double* d_dst, int ld_dst) {
  slab_transpose_kernel<<<dim3(ceil_div(rows, 32), ceil_div(nc, 32)), dim3(32, 8), 0, ctx->stream>>>(rows, nc, d_tmp,
                                                                                                     d_dst, ld_dst);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t build_regression_system_enqueue(gingr_ctx* ctx, int r, int rp, const double* d_S, double eps, double* d_B) {
  GINGR_LAUNCH(ctx, build_regression_system_kernel, dim3(ceil_div(rp, 256), r), 256, 0, ctx->stream, r, rp, d_S, eps, d_B);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t add_vectors_enqueue(gingr_ctx* ctx, int n, const double* d_a, const double* d_b, double* d_out) {
  GINGR_LAUNCH(ctx, add_vectors_kernel, ceil_div(n, 256), 256, 0, ctx->stream, n, d_a, d_b, d_out);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// ---------------------------------------------------------------------------------------------
int32_t gemv_rows_enqueue(gingr_ctx* ctx, int rows, int r, int rp, const double* d_phi, int nvec, const double* d_v0,
                          const double* d_v1, double* d_out0, double* d_out1, const double* d_scale) {
  if (rows <= 0) return GINGR_OK;
  // one row per warp; four when many chains share the launch (batch.cuh) -- a row's dot product does not depend on it
  const int blocks = std::max(1, std::min(ctx->num_sms * 4, ceil_div(rows, ctx->rec ? 32 : 8)));
  // two vectors that do not fit shared memory together (r > 12 800) are two one-vector passes: the same per-row sums
  if (nvec == 2 && (size_t)2 * r * sizeof(double) > 200 * 1024) {
    GINGR_TRY(gemv_rows_enqueue(ctx, rows, r, rp, d_phi, 1, d_v0, nullptr, d_out0, nullptr, d_scale));
    return gemv_rows_enqueue(ctx, rows, r, rp, d_phi, 1, d_v1, nullptr, d_out1, nullptr, d_scale);
  }
  const size_t smem = (size_t)nvec * r * sizeof(double);
  if (smem > 48 * 1024) {
    static bool set1 = false, set2 = false;
    if (nvec == 1 && !set1) {
      GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(gemv_rows_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      set1 = true;
    }
    if (nvec == 2 && !set2) {
      GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(gemv_rows_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      set2 = true;
    }
    if (smem > 200 * 1024) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "rank too large for gemv_rows shared memory");
  }
  if (nvec == 1)
    GINGR_LAUNCH_T(ctx, gemv_rows_kernel, (1), blocks, 256, smem, ctx->stream, rows, r, rp, d_phi, d_v0, d_v0, d_scale, d_out0, d_out0);
  else
    GINGR_LAUNCH_T(ctx, gemv_rows_kernel, (2), blocks, 256, smem, ctx->stream, rows, r, rp, d_phi, d_v0, d_v1, d_scale, d_out0, d_out1);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int gemvT_splits(const gingr_ctx* ctx, int rows) {
  return std::max(1, ceil_div(rows, gemvT_rows_per_cta(ctx, rows)));
}

int32_t gemvT_enqueue(gingr_ctx* ctx, int rows, int r, int rp, const double* d_phi, const double* d_u,
                      const double* d_scale, double* d_part, double* d_out) {
  const int splits = gemvT_splits(ctx, rows);
  if (rows > 0) {
    GINGR_LAUNCH(ctx, gemvT_kernel, dim3(ceil_div(rp, 256), splits), 256, 0, ctx->stream, rows, rp, gemvT_rows_per_cta(ctx, rows), d_phi,
                                                                           d_u, d_part);
    GINGR_LAUNCHED(ctx);
  } else {
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(d_part, 0, sizeof(double) * rp, ctx->stream));
  }
  GINGR_LAUNCH(ctx, gemvT_reduce_kernel, ceil_div(r, 32), 256, 0, ctx->stream, r, rp, splits, d_part, d_scale, d_out);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t dense_matvec_enqueue(gingr_ctx* ctx, int r, const double* d_A, int ld, const double* d_x, double* d_y,
                             int* d_flag_in, int* d_flag_out) {
  // (short rows -- the rank-50 chains of C5 -- are better off with one warp per row: 856 k against 762 k MH steps/s)
  if (r >= 512 && (ld & 1) == 0 && ((((uintptr_t)d_A) | ((uintptr_t)d_x)) & 15) == 0)
    GINGR_LAUNCH(ctx, dense_matvec2_kernel, ceil_div(r, 4), 256, 0, ctx->stream, r, d_A, ld, d_x, d_y, d_flag_in, d_flag_out);
  else
    GINGR_LAUNCH(ctx, dense_matvec_kernel, ceil_div(r * 32, 256), 256, 0, ctx->stream, r, d_A, ld, d_x, d_y, d_flag_in, d_flag_out);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t transpose_enqueue(gingr_ctx* ctx, int n, const double* d_A, int lda, double* d_B, int ldb) {
  transpose_kernel<<<dim3(ceil_div(n, 32), ceil_div(n, 32)), dim3(32, 8), 0, ctx->stream>>>(n, d_A, lda, d_B, ldb);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

}  // namespace gingr
