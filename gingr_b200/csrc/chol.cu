// chol.cu -- K3b: backward substitutions  c = L^-T z  against a Cholesky factor on the device (sm_100a).
//
// The factorisation is chol_df.cu's (one persistent data-flow kernel; chol_small_kernel for n <= 64); it performs the
// forward substitution L^-1 b on right-hand sides stored as extra rows, and its own back substitution reads the inverses
// of the diagonal blocks it published in the workspace (chol_backsolve_z_kernel).  The kernels here need the factor
// alone: they solve against every one-block factor (n <= 64) and against factors whose workspace inverses belong to
// another factorisation (the kept factors of a Metropolis-Hastings chain).
//   chol_backsolve_kernel        sync-free multi-CTA kernel: one CTA per 64-block, taken by ticket, consuming solved blocks
//                                as their ready flags appear
//   chol_backsolve_small_kernel  n <= 64: one warp substitutes, right-looking
#include "batch.cuh"
#include "posterior.cuh"

namespace gingr {

constexpr int NB = 64;
constexpr int SP = NB + 1;  // shared pitch for the scalar kernels

// ---------------------------------------------------------------------------------------------
// backward substitution  L^T c = z,  one CTA per 64-block, blocks become ready from the last one up.
// A CTA takes its block from an atomic ticket: ticket t solves block k = nb - 1 - t and waits only for the blocks
// i > k, which tickets smaller than its own hold.  A ticket is drawn only by a running CTA, so every block waited for
// belongs to a resident CTA that itself waits only for smaller tickets: the spin waits cannot deadlock whatever the grid
// size (nb may exceed the SM count) or whatever else occupies the GPU.  The arithmetic depends on the block alone, not
// on the CTA that solves it.
// Each CTA first inverts its own diagonal block (off the critical path: it would otherwise spin on the
// ready flags), accumulates  z_k - sum_{i>k} L_ik^T c_i  as the c_i appear, and finishes with the
// 64 x 64 product  c_k = D^-T acc.
// flags: nb + 2 ints (block flags, finished CTAs, ticket), zero on entry; the last CTA out zeroes them again, so a
// captured graph replays without a memset node.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) chol_backsolve_kernel(int n, const double* __restrict__ L, int ld,
                                                             const double* __restrict__ z, double* __restrict__ c,
                                                             volatile int* __restrict__ flags) {
  __shared__ double sD[NB * SP];  // lower: D ; strict upper: (D^-1)^T ; diagonal of D^-1 in sZd
  __shared__ double sZd[NB];
  __shared__ double sc[NB];
  __shared__ double sacc[4][NB];
  __shared__ double acc[NB];
  __shared__ int s_ticket;
  const int nb = (n + NB - 1) / NB;
  const int tid = threadIdx.x;
  if (tid == 0) s_ticket = atomicAdd((int*)&flags[nb + 1], 1);
  __syncthreads();
  const int k = nb - 1 - s_ticket;  // the first tickets own the last blocks (solved first)
  const int k0 = k * NB, kcnt = min(NB, n - k0);
  for (int e = tid; e < NB * NB; e += 256) {
    const int i = e >> 6, j = e & 63;
    sD[i * SP + j] = (i < kcnt && j <= i) ? L[(size_t)(k0 + i) * ld + k0 + j] : (i == j ? 1.0 : 0.0);
  }
  if (tid < NB) acc[tid] = tid < kcnt ? z[k0 + tid] : 0.0;
  __syncthreads();
  // Z = D^-1 by columns: thread (col = tid & 63, part = tid >> 6) -- the 4 parts split the inner sums
  {
    const int col = tid & 63, part = tid >> 6;
    // one warp-pair per ... keep it simple: part 0 does the column, sequentially
    if (part == 0) {
      // Z[i][col] lives at sD[col][i] (i > col); thread `col` only touches row `col` of the upper triangle
      const double zcc = 1.0 / sD[col * SP + col];
      sZd[col] = zcc;
      for (int i = col + 1; i < NB; ++i) {
        double s0 = sD[i * SP + col] * zcc, s1 = 0.0;
        int kk = col + 1;
        for (; kk + 1 < i; kk += 2) {
          s0 = fma(sD[i * SP + kk], sD[col * SP + kk], s0);
          s1 = fma(sD[i * SP + kk + 1], sD[col * SP + kk + 1], s1);
        }
        if (kk < i) s0 = fma(sD[i * SP + kk], sD[col * SP + kk], s0);
        sD[col * SP + i] = -(s0 + s1) / sD[i * SP + i];
      }
    }
  }
  const int col = tid & 63, part = tid >> 6;
  double s = 0.0;
  for (int i = nb - 1; i > k; --i) {
    if (tid == 0) {
      while (flags[i] == 0) {
      }
    }
    __syncthreads();
    __threadfence();
    const int i0 = i * NB, icnt = min(NB, n - i0);
    if (tid < NB) sc[tid] = tid < icnt ? __ldcg(c + i0 + tid) : 0.0;
    __syncthreads();
    if (col < kcnt) {
      const int r_begin = part * 16, r_end = min(icnt, r_begin + 16);
      for (int rr = r_begin; rr < r_end; ++rr) s = fma(L[(size_t)(i0 + rr) * ld + k0 + col], sc[rr], s);
    }
  }
  sacc[part][col] = s;
  __syncthreads();
  if (tid < NB) acc[tid] -= (sacc[0][tid] + sacc[1][tid]) + (sacc[2][tid] + sacc[3][tid]);
  __syncthreads();
  // c_k = D^-T acc :  c[j] = sum_{i >= j} Z[i][j] acc[i]   (4 partial sums per output)
  {
    double t = part == 0 ? sZd[col] * acc[col] : 0.0;
    for (int i = col + 1 + part; i < NB; i += 4) t = fma(sD[col * SP + i], acc[i], t);
    sacc[part][col] = t;
  }
  __syncthreads();
  if (tid < kcnt) c[k0 + tid] = (sacc[0][tid] + sacc[1][tid]) + (sacc[2][tid] + sacc[3][tid]);
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    flags[k] = 1;
    if (atomicAdd((int*)&flags[nb], 1) == nb - 1) {   // last CTA out: every flag has been read and every ticket drawn
      for (int e = 0; e <= nb + 1; ++e) flags[e] = 0;
    }
  }
}

// n <= 64 (one block): plain right-looking back substitution by 64 threads -- the general kernel would spend 50 us
// inverting the diagonal block with one thread per column, which only pays when it hides behind the flag waits.
GINGR_KERNEL((128), chol_backsolve_small_kernel, int n, const double* __restrict__ L, int ld,
                                                                   const double* __restrict__ z, double* __restrict__ c) {
  __shared__ double sLs[NB * SP];
  __shared__ double sinv[NB];
  // four warps bring the block in (coalesced rows; one warp alone spent 10 us of its 20 here), warp 0 substitutes
  for (int e = threadIdx.x; e < NB * NB; e += 128) {
    const int i = e >> 6, j = e & 63;
    sLs[i * SP + j] = (i < n && j <= i) ? L[(size_t)i * ld + j] : (i == j ? 1.0 : 0.0);
  }
  __syncthreads();
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  sinv[lane] = 1.0 / sLs[lane * SP + lane];
  sinv[lane + 32] = 1.0 / sLs[(lane + 32) * SP + lane + 32];
  __syncwarp();
  // lane holds the running right-hand sides of unknowns lane and lane + 32; unknown j = L^T row j needs L[j][k], k < j
  double a0 = lane < n ? z[lane] : 0.0, a1 = lane + 32 < n ? z[lane + 32] : 0.0;
#pragma unroll 8
  for (int j = 63; j >= 32; --j) {
    const double cj = __shfl_sync(0xffffffffu, a1 * sinv[j], j - 32);
    if (lane + 32 == j) a1 = cj;
    else if (lane + 32 < j) a1 = fma(-sLs[j * SP + lane + 32], cj, a1);
    a0 = fma(-sLs[j * SP + lane], cj, a0);
  }
#pragma unroll 8
  for (int j = 31; j >= 0; --j) {
    const double cj = __shfl_sync(0xffffffffu, a0 * sinv[j], j);
    if (lane == j) a0 = cj;
    else if (lane < j) a0 = fma(-sLs[j * SP + lane], cj, a0);
  }
  if (lane < n) c[lane] = a0;
  if (lane + 32 < n) c[lane + 32] = a1;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
int32_t chol_backsolve_enqueue(gingr_ctx* ctx, int n, const double* d_L, int ld, const double* d_z, double* d_c,
                               int* d_flags, CholWs* ws) {
  const int nb = ceil_div(n, NB);
  if (ws != nullptr && nb > 1) return chol_backsolve_z_enqueue(ctx, n, d_L, ld, d_z, d_c, *ws);
  if (nb == 1) {
    GINGR_LAUNCH(ctx, chol_backsolve_small_kernel, 1, 128, 0, ctx->stream, n, d_L, ld, d_z, d_c);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    return GINGR_OK;
  }
  chol_backsolve_kernel<<<nb, 256, 0, ctx->stream>>>(n, d_L, ld, d_z, d_c, d_flags);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

}  // namespace gingr
