// chol.cu -- K3b: on-device r x r Cholesky factorisation and triangular solves (sm_100a).
//
// Replaces `Minv = breeze.linalg.pinv(M)` of scalismo's regression (SURVEY.md A3; call sites
// GingrAlgorithm.scala:300, :215, :236).  M = Q^T L^-1 Q + I is symmetric positive definite, so
// M^-1 b is obtained from M = L L^T; a failed pivot (M not SPD / non-finite input) is reported through
// d_info and becomes FittingStatuses.ModelFlexibilityError where the reference's Try fails.
//
// Blocked right-looking factorisation, block 64:
//   chol_panel_kernel   every CTA factorises the 64 x 64 diagonal block redundantly (no extra launch / grid
//                       sync; warp-level in-register 32 x 32 factorisations) and solves its own 128 panel rows
//   chol_syrk_kernel    trailing update C -= X X^T on DMMA.8x8x4 (64 x 64 tiles, K = 64)
// Rows below the square part (right-hand sides stored as extra rows) ride along, which performs the
// forward substitution L^-1 b inside the factorisation.  The backward substitution L^-T z is a sync-free
// multi-CTA kernel: one CTA per 64-block, taken by ticket, consuming solved blocks as their ready flags appear.
#include <stdlib.h>

#include <algorithm>

#include "batch.cuh"
#include "posterior.cuh"

namespace gingr {

constexpr int NB = 64;
constexpr int SP = NB + 1;  // shared pitch for the scalar kernels

// ---------------------------------------------------------------------------------------------
// panel kernel.  Every CTA factorises the 64 x 64 diagonal block redundantly (no extra launch, no grid sync)
// and then solves its own PR rows of the panel.  The diagonal block is done recursively on 32 x 32 halves:
//   L11 = chol32(A11)            one warp, lane i owns row i in REGISTERS, pivots/columns move by shuffles:
//                                no block barrier inside the 32 sequential column steps
//   L21 = A21 L11^-T             one warp, lane = row, right-looking substitution against L11 in shared memory
//   A22 -= L21 L21^T             all threads
//   L22 = chol32(A22)
// The panel rows are solved one row per thread, the row held in registers (x[64]), right-looking so the 63
// updates of a step are independent FMAs; L is read from shared memory as a broadcast.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sa), "l"(gmem) : "memory");
}

#ifdef CHOL_TIMING
// tuning build only (tools/build_variant.sh timing chol.cu -DCHOL_TIMING): clock64 per phase of the panel kernel, block 0
__device__ unsigned long long chol_timing[8];
#define CT_MARK(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) { const long long now = clock64(); atomicAdd(&chol_timing[k], (unsigned long long)(now - ct_last)); ct_last = now; } } while (0)
#else
#define CT_MARK(k) ((void)0)
#endif

constexpr int PR = 128;  // panel rows (threads) per CTA
constexpr size_t PANEL_SMEM = ((size_t)NB * SP + NB + (size_t)PR * SP) * sizeof(double);

// In-register Cholesky of a 32 x 32 block: lane i holds row i (a[k], k <= i).  On return a[k] = L[i][k] for
// k <= i and *invd = 1 / L[i][i].  Returns true if a pivot was not positive and finite.
__device__ __forceinline__ bool warp_chol32(double (&a)[32], int lane, double* invd) {
  bool bad = false;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const double d = __shfl_sync(0xffffffffu, a[j], j);
    if (!(d > 0.0) || !(d < INFINITY)) bad = true;
    const double rs = rsqrt(d);
    const double l = a[j] * rs;  // lane j: sqrt(d); lanes > j: L[i][j]
    a[j] = l;
    if (lane == j) *invd = rs;
#pragma unroll
    for (int k = j + 1; k < 32; ++k) {
      const double lk = __shfl_sync(0xffffffffu, l, k);  // L[k][j]
      a[k] = fma(-l, lk, a[k]);
    }
  }
  return bad;
}

// x <- x L^-T for one row held in registers: L (NC x NC lower, pitch SP) and 1/diag in shared memory.
template <int NC>
__device__ __forceinline__ void row_trsm(double (&x)[NC], const double* __restrict__ sLm,
                                         const double* __restrict__ sInv) {
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    x[j] *= sInv[j];
    const double xj = x[j];
#pragma unroll
    for (int m = j + 1; m < NC; ++m) x[m] = fma(-xj, sLm[m * SP + j], x[m]);
  }
}

// x <- x L^-T for ONE row by a whole warp (lane holds x[lane] and x[lane + 32]): the pivot element is scaled by its owner
// and broadcast by a shuffle, every lane updates its two later elements.  64 short steps instead of the 2016 dependent
// FMA + shared-memory loads of the thread-per-row form: used when a CTA has only a few rows (the right-hand-side row
// of a small system).
__device__ __forceinline__ void warp_row_trsm64(double* __restrict__ xrow /*shared, 64 values*/, const double* __restrict__ sLm,
                                                const double* __restrict__ sInv, int lane) {
  double x0 = xrow[lane], x1 = xrow[lane + 32];
#pragma unroll 8
  for (int j = 0; j < 32; ++j) {
    const double xj = __shfl_sync(0xffffffffu, x0 * sInv[j], j);
    if (lane == j) x0 = xj;
    else if (lane > j) x0 = fma(-xj, sLm[lane * SP + j], x0);
    x1 = fma(-xj, sLm[(lane + 32) * SP + j], x1);
  }
#pragma unroll 8
  for (int j = 32; j < 64; ++j) {
    const double xj = __shfl_sync(0xffffffffu, x1 * sInv[j], j - 32);
    if (lane + 32 == j) x1 = xj;
    else if (lane + 32 > j) x1 = fma(-xj, sLm[(lane + 32) * SP + j], x1);
  }
  xrow[lane] = x0;
  xrow[lane + 32] = x1;
}

__global__ void __launch_bounds__(PR) chol_panel_kernel(int nrows, int j0, int jb, double* __restrict__ A, int ld,
                                                        int* __restrict__ info) {
  extern __shared__ __align__(16) double psm[];
  double* sL = psm;                    // [64][65] diagonal block -> L (lower)
  double* sInvD = psm + NB * SP;       // [64] 1 / L[j][j]
  double* sX = psm + NB * SP + NB;     // [PR][65] panel rows
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = j0 + jb + blockIdx.x * PR;
  const int cnt = max(0, min(PR, nrows - i0));
#ifdef CHOL_TIMING
  long long ct_last = clock64();
#endif
  // All 96 loads of a thread are issued as asynchronous 8-byte copies before anything waits: the load phase was a
  // quarter of the kernel (ncu: long-scoreboard stalls) when every global load stalled the scheduler's only warp in turn.
  for (int e = tid; e < NB * NB; e += PR) {
    const int i = e >> 6, k = e & 63;
    if (i < jb && k <= i) cp_async8(&sL[i * SP + k], &A[(size_t)(j0 + i) * ld + j0 + k]);
    else sL[i * SP + k] = (i == k ? 1.0 : 0.0);
  }
  for (int e = tid; e < PR * NB; e += PR) {
    const int i = e >> 6, k = e & 63;
    if (i < cnt && k < jb) cp_async8(&sX[i * SP + k], &A[(size_t)(i0 + i) * ld + j0 + k]);
    else sX[i * SP + k] = 0.0;
  }
  asm volatile("cp.async.wait_all;\n" ::: "memory");
  __syncthreads();
  CT_MARK(0);   // loads
  // All four warps run the warp-level pieces redundantly and convergently (no divergent region around the
  // shuffles); only warp 0 stores.  h = 0: (L11, L21, A22 update), h = 1: L22 -- one copy of the unrolled code.
  bool bad = false;
#pragma unroll 1
  for (int h = 0; h < 2; ++h) {
    double* blk = sL + (h * 32) * SP + h * 32;  // A11 or A22
    double a[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) a[k] = blk[lane * SP + k];
    double invd = 0.0;
    bad = warp_chol32(a, lane, &invd) || bad;
    __syncthreads();  // every warp has read the block
    CT_MARK(1);   // chol32
    if (warp == 0) {
#pragma unroll
      for (int k = 0; k < 32; ++k)
        if (k <= lane) blk[lane * SP + k] = a[k];
      sInvD[h * 32 + lane] = invd;
    }
    __syncthreads();
    if (h == 0) {
      // L21 = A21 L11^-T  (lane = row of A21)
      double x[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) x[k] = sL[(32 + lane) * SP + k];
      row_trsm<32>(x, sL, sInvD);
      __syncthreads();
      CT_MARK(2);   // trsm32
      if (warp == 0) {
#pragma unroll
        for (int k = 0; k < 32; ++k) sL[(32 + lane) * SP + k] = x[k];
      }
      __syncthreads();
      // A22 -= L21 L21^T : thread -> row i = tid / 4, 8 columns
      const int i = tid >> 2, k0 = (tid & 3) * 8;
      const double* li = sL + (32 + i) * SP;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int k = k0 + q;
        if (k <= i) {
          const double* lk = sL + (32 + k) * SP;
          double s0 = 0.0, s1 = 0.0;
#pragma unroll
          for (int c = 0; c < 32; c += 2) {
            s0 = fma(li[c], lk[c], s0);
            s1 = fma(li[c + 1], lk[c + 1], s1);
          }
          sL[(32 + i) * SP + 32 + k] -= s0 + s1;
        }
      }
      __syncthreads();
      CT_MARK(3);   // A22 update
    }
  }
  if (blockIdx.x == 0) {
    if (bad && tid == 0) info[0] = 1;
    for (int e = tid; e < NB * NB; e += PR) {
      const int i = e >> 6, k = e & 63;
      if (i < jb && k <= i) A[(size_t)(j0 + i) * ld + j0 + k] = sL[i * SP + k];
    }
  }
  CT_MARK(4);   // store of L
  if (cnt > 0 && cnt <= 4) {
    if (warp < cnt) warp_row_trsm64(sX + warp * SP, sL, sInvD, lane);   // a few rows: one warp per row
  } else if (cnt > 0) {
    double x[NB];
#pragma unroll
    for (int k = 0; k < NB; ++k) x[k] = sX[tid * SP + k];
    row_trsm<NB>(x, sL, sInvD);
#pragma unroll
    for (int k = 0; k < NB; ++k) sX[tid * SP + k] = x[k];
  }
  __syncthreads();
  CT_MARK(5);   // panel rows
  for (int e = tid; e < PR * NB; e += PR) {
    const int i = e >> 6, k = e & 63;
    if (i < cnt && k < jb) A[(size_t)(i0 + i) * ld + j0 + k] = sX[i * SP + k];
  }
  CT_MARK(6);   // store of the panel
}

// ---------------------------------------------------------------------------------------------
// trailing update on DMMA:  C[i][k] -= sum_c X[i][c] X[k][c],  c in [j0, j0 + 64)
// grid (col tiles, row tiles) over the region rows >= r0, cols in [r0, n); tiles above the diagonal exit.
// ---------------------------------------------------------------------------------------------
constexpr int UP = NB + 4;  // pitch == 4 mod 16: conflict-free DMMA fragment loads
constexpr size_t SYRK_SMEM = 2 * NB * UP * sizeof(double);

__device__ __forceinline__ void dmma884s(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(128) chol_syrk_kernel(int nrows, int n, int j0, int jb, int r0, int tk_begin,
                                                        double* __restrict__ A, int ld) {
  extern __shared__ __align__(16) double sm[];
  double* sI = sm;            // [64][UP] rows of the row tile
  double* sK = sm + NB * UP;  // [64][UP] rows of the column tile
  const int ti = blockIdx.y, tk = blockIdx.x + tk_begin;
  const int i0 = r0 + ti * NB, k0 = r0 + tk * NB;
  if (k0 > i0 || k0 >= n || i0 >= nrows) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 1, wn = warp & 1, g = lane >> 2, t = lane & 3;
  const int icnt = min(NB, nrows - i0), kcnt = min(NB, n - k0);
  for (int e = tid; e < NB * NB; e += 128) {
    const int i = e / NB, c = e % NB;
    sI[i * UP + c] = (i < icnt && c < jb) ? A[(size_t)(i0 + i) * ld + j0 + c] : 0.0;
    sK[i * UP + c] = (i < kcnt && c < jb) ? A[(size_t)(k0 + i) * ld + j0 + c] : 0.0;
  }
  __syncthreads();
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
#pragma unroll 4
  for (int c4 = 0; c4 < NB / 4; ++c4) {
    double af[4], bf[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) af[i] = sI[(wm * 32 + i * 8 + g) * UP + c4 * 4 + t];
#pragma unroll
    for (int j = 0; j < 4; ++j) bf[j] = sK[(wn * 32 + j * 8 + g) * UP + c4 * 4 + t];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma884s(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int row = wm * 32 + i * 8 + g, col = wn * 32 + j * 8 + 2 * t;
      if (row < icnt) {
        double* p = A + (size_t)(i0 + row) * ld + k0 + col;
        if (col + 1 < kcnt) {
          double2 v = *reinterpret_cast<double2*>(p);
          v.x -= acc[i][j][0];
          v.y -= acc[i][j][1];
          *reinterpret_cast<double2*>(p) = v;
        } else if (col < kcnt) {
          p[0] -= acc[i][j][0];
        }
      }
    }
}

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
int32_t cholesky_enqueue(gingr_ctx* ctx, int n, int nrows, double* d_A, int ld, int* d_info, CholWs* ws) {
  static const int env_df = [] { const char* e = getenv("GINGR_CHOL_DF"); return e ? atoi(e) : 1; }();
  if (ws != nullptr && env_df != 0) return cholesky_df_enqueue(ctx, n, nrows, d_A, ld, d_info, *ws);
  static thread_local int attr_device = -1;  // once per device (and host thread): not a stream operation
  if (attr_device != ctx->device) {
    GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(chol_syrk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)SYRK_SMEM));
    GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)PANEL_SMEM));
    attr_device = ctx->device;
  }
  cudaStream_t st = ctx->stream;
  // Lookahead: the trailing update of step j is split into A(j) = the next block column (what the next panel
  // needs) on the main stream and B(j) = everything to the right of it on the low-priority side stream, which then
  // overlaps panel(j + 1).  Dependencies: B(j) after panel(j); A(j) after B(j - 1) (both update block column j + 1).
  // Inside a stream capture these event edges become graph dependencies.
  static const int env_la = [] { const char* e = getenv("GINGR_CHOL_LOOKAHEAD"); return e ? atoi(e) : 1; }();
  const int nb = ceil_div(n, NB);
  const bool lookahead = env_la != 0 && ctx->side_stream != nullptr && nb >= 4;
  if (lookahead && (int)ctx->chol_events.size() < 2 * nb) {
    const size_t old = ctx->chol_events.size();
    ctx->chol_events.resize((size_t)2 * nb);
    for (size_t k = old; k < ctx->chol_events.size(); ++k)
      GINGR_CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->chol_events[k], cudaEventDisableTiming));
  }
  int last_b = -1;
  for (int j0 = 0, j = 0; j0 < n; j0 += NB, ++j) {
    const int jb = std::min(NB, n - j0);
    const int below = nrows - (j0 + jb);
    const int pblocks = std::max(1, ceil_div(below, PR));
    chol_panel_kernel<<<pblocks, PR, PANEL_SMEM, st>>>(nrows, j0, jb, d_A, ld, d_info);
    GINGR_LAUNCHED(ctx);
    if (below > 0 && j0 + jb < n) {
      const int r0 = j0 + jb;
      const int nti = ceil_div(nrows - r0, NB), ntk = ceil_div(n - r0, NB);
      if (!lookahead || ntk < 2) {
        if (last_b >= 0) { GINGR_CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->chol_events[2 * last_b + 1], 0)); last_b = -1; }
        chol_syrk_kernel<<<dim3(ntk, nti), 128, SYRK_SMEM, st>>>(nrows, n, j0, jb, r0, 0, d_A, ld);
        GINGR_LAUNCHED(ctx);
      } else {
        cudaEvent_t ev_p = ctx->chol_events[2 * j], ev_b = ctx->chol_events[2 * j + 1];
        GINGR_CUDA_TRY(ctx, cudaEventRecord(ev_p, st));
        GINGR_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->side_stream, ev_p, 0));
        chol_syrk_kernel<<<dim3(ntk - 1, nti), 128, SYRK_SMEM, ctx->side_stream>>>(nrows, n, j0, jb, r0, 1, d_A, ld);  // B(j)
        GINGR_LAUNCHED(ctx);
        GINGR_CUDA_TRY(ctx, cudaEventRecord(ev_b, ctx->side_stream));
        if (last_b >= 0) GINGR_CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->chol_events[2 * last_b + 1], 0));
        chol_syrk_kernel<<<dim3(1, nti), 128, SYRK_SMEM, st>>>(nrows, n, j0, jb, r0, 0, d_A, ld);                       // A(j)
        GINGR_LAUNCHED(ctx);
        last_b = j;
      }
    }
  }
  if (last_b >= 0) GINGR_CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->chol_events[2 * last_b + 1], 0));
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t chol_backsolve_enqueue(gingr_ctx* ctx, int n, const double* d_L, int ld, const double* d_z, double* d_c,
                               int* d_flags, CholWs* ws) {
  const int nb = ceil_div(n, NB);
  static const int env_df = [] { const char* e = getenv("GINGR_CHOL_DF"); return e ? atoi(e) : 1; }();
  if (ws != nullptr && env_df != 0 && nb > 1) return chol_backsolve_z_enqueue(ctx, n, d_L, ld, d_z, d_c, *ws);
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

#ifdef CHOL_TIMING
extern "C" GINGR_API int32_t gingr_debug_chol_timing(unsigned long long* out, int32_t reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, gingr::chol_timing, sizeof(unsigned long long) * 8);
  if (reset) {
    unsigned long long z[8] = {0};
    cudaMemcpyToSymbol(gingr::chol_timing, z, sizeof(z));
  }
  return 0;
}
#endif
