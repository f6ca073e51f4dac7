// basis_rotate.cu -- basis of the posterior model on the FP64 tensor pipe (sm_100a):
//     Phi'[3i + d][j] = scale[j] * sum_e R[d][e] (Phi U)[3i + e][j]        i.e.  Phi' = (I (x) R) Phi U diag(scale)
// Phi [rows][rp] and the output row-major, U [rp][rp] row-major and zero padded (update.cu: gingr_model_posterior).
//
// Plain tiled GEMM: one CTA per 96 x 128 output tile (96 rows = 32 whole vertices, so the per-vertex rotation fits in the
// epilogue), 8 warps of 48 x 32 (6 x 4 DMMA.8x8x4 accumulator fragments), k in chunks of 16 through a 4-stage cp.async
// pipeline.  Every output element is one fixed-order sum over k (no split-K): two calls give the same bits.
// The CTA index runs along the columns first, so the CTAs that share a row slab of Phi run together and U (r^2 doubles,
// 32 MB at r = 2000) stays in L2.
#include "dmma.cuh"
#include "posterior.cuh"

namespace gingr {

namespace {
constexpr int BR_BM = 96;                  // tile rows (multiple of 3 and of 8)
constexpr int BR_BN = 128;                 // tile columns
constexpr int BR_BK = 16;                  // k per pipeline stage
constexpr int BR_STAGES = 4;
constexpr int BR_PA = BR_BK + 4;           // sA[m][k] pitch (== 4 mod 16: conflict-free A fragment loads)
constexpr int BR_PB = BR_BN + 4;           // sB[k][n] pitch (== 4 mod 16: conflict-free B fragment loads)
constexpr int BR_PC = BR_BN + 4;           // epilogue tile pitch
constexpr int BR_THREADS = 256;
constexpr int BR_WM = 48, BR_WN = 32;      // warp tile: 2 x 4 warps
constexpr int BR_MI = BR_WM / 8, BR_NJ = BR_WN / 8;
constexpr int BR_STAGE_DOUBLES = BR_BM * BR_PA + BR_BK * BR_PB;
constexpr size_t BR_SMEM = (size_t)BR_STAGES * BR_STAGE_DOUBLES * sizeof(double);
static_assert(BR_BM % 3 == 0 && BR_BM % 8 == 0, "a tile owns whole vertices");
static_assert((size_t)BR_BM * BR_PC * sizeof(double) <= BR_SMEM, "the epilogue tile reuses the pipeline stages");
}  // namespace

__global__ void __launch_bounds__(BR_THREADS, 1) basis_rotate_kernel(int rows, int rp, int ntn, const double* __restrict__ phi,
                                                                     const double* __restrict__ U,
                                                                     const double* __restrict__ scale,
                                                                     const double* __restrict__ Rm, double* __restrict__ out) {
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 2, wn = warp & 3;
  const int g = lane >> 2, t = lane & 3;
  const int m0 = (blockIdx.x / ntn) * BR_BM, n0 = (blockIdx.x % ntn) * BR_BN;
  const int nchunks = (rp + BR_BK - 1) / BR_BK;

  auto issue = [&](int chunk) {
    double* sA = smem + (size_t)(chunk % BR_STAGES) * BR_STAGE_DOUBLES;
    double* sB = sA + BR_BM * BR_PA;
    const int k0 = chunk * BR_BK;
    // A: 96 rows x 8 pieces of 16 bytes; B: 16 rows x 64 pieces
#pragma unroll
    for (int q = 0; q < BR_BM * (BR_BK / 2) / BR_THREADS; ++q) {
      const int e = tid + q * BR_THREADS;
      const int mr = e / (BR_BK / 2), kc = (e % (BR_BK / 2)) * 2;
      const bool ok = m0 + mr < rows && k0 + kc < rp;
      cp_async16(sA + mr * BR_PA + kc, ok ? (const void*)(phi + (size_t)(m0 + mr) * rp + k0 + kc) : (const void*)phi, ok ? 16 : 0);
    }
#pragma unroll
    for (int q = 0; q < BR_BK * (BR_BN / 2) / BR_THREADS; ++q) {
      const int e = tid + q * BR_THREADS;
      const int kr = e / (BR_BN / 2), nc = (e % (BR_BN / 2)) * 2;
      const bool ok = k0 + kr < rp && n0 + nc < rp;
      cp_async16(sB + kr * BR_PB + nc, ok ? (const void*)(U + (size_t)(k0 + kr) * rp + n0 + nc) : (const void*)U, ok ? 16 : 0);
    }
  };

  double acc[BR_MI][BR_NJ][2];
#pragma unroll
  for (int i = 0; i < BR_MI; ++i)
#pragma unroll
    for (int j = 0; j < BR_NJ; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int p = 0; p < BR_STAGES - 1; ++p) {
    if (p < nchunks) issue(p);
    cp_async_commit();
  }
  for (int ch = 0; ch < nchunks; ++ch) {
    cp_async_wait<BR_STAGES - 2>();
    __syncthreads();   // chunk ch has landed for every thread, and the stage refilled below is no longer read
    if (ch + BR_STAGES - 1 < nchunks) issue(ch + BR_STAGES - 1);
    cp_async_commit();
    const double* sA = smem + (size_t)(ch % BR_STAGES) * BR_STAGE_DOUBLES;
    const double* tA = sA + (wm * BR_WM + g) * BR_PA + t;
    const double* tB = sA + BR_BM * BR_PA + t * BR_PB + wn * BR_WN + g;
#pragma unroll
    for (int k4 = 0; k4 < BR_BK / 4; ++k4) {
      double af[BR_MI], bf[BR_NJ];
#pragma unroll
      for (int i = 0; i < BR_MI; ++i) af[i] = tA[i * 8 * BR_PA + k4 * 4];
#pragma unroll
      for (int j = 0; j < BR_NJ; ++j) bf[j] = tB[k4 * 4 * BR_PB + j * 8];
#pragma unroll
      for (int i = 0; i < BR_MI; ++i)
#pragma unroll
        for (int j = 0; j < BR_NJ; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
  }
  cp_async_wait<0>();
  __syncthreads();   // every warp is done with the stages: the tile goes through shared memory

  // epilogue: column scale into the staged tile, then the rotation of each vertex's three rows.  Explicitly rounded
  // products and sums (no contraction into FMA).
  double* sC = smem;
#pragma unroll
  for (int j = 0; j < BR_NJ; ++j) {
    const int col = wn * BR_WN + j * 8 + 2 * t;
    const double s0 = n0 + col < rp ? scale[n0 + col] : 0.0, s1 = n0 + col + 1 < rp ? scale[n0 + col + 1] : 0.0;
#pragma unroll
    for (int i = 0; i < BR_MI; ++i) {
      const int row = wm * BR_WM + i * 8 + g;
      *reinterpret_cast<double2*>(sC + row * BR_PC + col) = make_double2(__dmul_rn(acc[i][j][0], s0), __dmul_rn(acc[i][j][1], s1));
    }
  }
  __syncthreads();
  double R[9];
#pragma unroll
  for (int q = 0; q < 9; ++q) R[q] = Rm[q];
  const int ncols = min(BR_BN, rp - n0);
  for (int e = tid; e < (BR_BM / 3) * BR_BN; e += BR_THREADS) {
    const int v = e / BR_BN, c = e % BR_BN;
    const int row = m0 + 3 * v;
    if (row >= rows || c >= ncols) continue;
    const double x = sC[(3 * v) * BR_PC + c], y = sC[(3 * v + 1) * BR_PC + c], z = sC[(3 * v + 2) * BR_PC + c];
#pragma unroll
    for (int d = 0; d < 3; ++d)
      out[(size_t)(row + d) * rp + n0 + c] =
          __dadd_rn(__dadd_rn(__dmul_rn(R[3 * d], x), __dmul_rn(R[3 * d + 1], y)), __dmul_rn(R[3 * d + 2], z));
  }
}

int32_t basis_rotate_enqueue(gingr_ctx* ctx, int rows, int rp, const double* d_phi, const double* d_U, const double* d_scale,
                             const double* d_R, double* d_out) {
  if (rows <= 0 || rp <= 0) return GINGR_OK;
  if (rows % 3 != 0 || rp % 8 != 0) return gingr_fail(ctx, GINGR_ERR_ARG, "basis_rotate_enqueue: rows must hold whole vertices, rp a multiple of 8");
  GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(basis_rotate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BR_SMEM));
  const int ntm = ceil_div(rows, BR_BM), ntn = ceil_div(rp, BR_BN);
  basis_rotate_kernel<<<ntm * ntn, BR_THREADS, BR_SMEM, ctx->stream>>>(rows, rp, ntn, d_phi, d_U, d_scale, d_R, d_out);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

}  // namespace gingr
