// chol_df.cu -- K3b: the r x r Cholesky factorisation as ONE persistent data-flow kernel (sm_100a).
//
// Replaces `Minv = breeze.linalg.pinv(M)` of scalismo's regression (SURVEY.md A3; call sites
// GingrAlgorithm.scala:300, :215, :236) together with chol.cu's back substitution.  The factorisation is the one
// replicated, latency-bound step of a multi-GPU iteration, so what counts is its CRITICAL PATH, not its flops
// (r^3/3 = 2.7 GFLOP at r = 2000 is 0.1 ms of DMMA): the previous form (one panel kernel + one or two trailing-update
// kernels per 64-column step, 32 dependent steps of ~47 us) is replaced by a tile data-flow:
//
//   * the lower triangle is cut into 64 x 64 tiles; TASKS are handed out in a topological order by an atomic ticket
//     counter to a persistent grid (one CTA of 8 warps per SM).  A task keeps its accumulators in registers and
//     subtracts X_ik X_jk^T (DMMA.8x8x4) for every k as soon as the two operand tiles are flagged final (left-looking,
//     operands double-buffered through cp.async);
//   * task T(i, j) (off-diagonal tile): waits for Z_j = L_jj^-1 and finishes with X_ij = A_ij Z_j^T as a (triangular)
//     DMMA product -- no substitution anywhere outside the diagonal blocks;
//   * task D(j) owns the diagonal tile (j, j) AND the tile (j, j-1) left of it: when Z_{j-1} appears it forms X_{j,j-1},
//     keeps it in shared memory, applies the last update to the diagonal tile, factorises the 64 x 64 block inside
//     the CTA (see potrf64), publishes Z_j and raises the flag.  Between two diagonal factorisations the critical
//     path is therefore  flag -> one triangular tile product -> one tile product -- with no trip through global memory;
//   * a CTA only ever waits for tasks with a smaller ticket, and every ticket that was drawn belongs to a running
//     CTA, so the spin waits cannot deadlock whatever else occupies the GPU.  No launch boundary, no grid-wide barrier.
//
// Rows below the square part (right-hand sides stored as extra rows) ride along, which performs the forward
// substitution L^-1 b inside the factorisation (as chol.cu's kernels did).
#include <stdlib.h>

#include <algorithm>

#include "batch.cuh"
#include "posterior.cuh"

namespace gingr {

namespace {

constexpr int TB = 64;                 // tile edge
constexpr int TP = TB + 4;             // shared pitch, == 4 (mod 16): conflict-free DMMA fragment loads
constexpr int DF_THREADS = 256;
constexpr int TILE_DOUBLES = TB * TP;  // 4352
// shared memory: 6 tile buffers (2 stages x 2 operands + the two input tiles of a diagonal task), diag(L), the
// sub-diagonal entries L[2s+1][2s] and the step flags of the in-CTA factorisation
constexpr size_t DF_SMEM = (size_t)(6 * TILE_DOUBLES + TB + 32 + 32) * sizeof(double) + 64;

__device__ __forceinline__ int ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Release at gpu scope AFTER a CTA barrier: cumulative, so the plain global stores of every thread of the CTA that
// happened before the barrier are visible to whoever acquires the flag -- no separate __threadfence() (it cost a second
// fence per flag on the critical path; the same pattern as CUTLASS's Semaphore::release).
__device__ __forceinline__ void st_release(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
// barrier of the two warps (64 threads) that own the pivot columns of a factorisation step
__device__ __forceinline__ void bar_pair(int id) { asm volatile("bar.sync %0, 64;\n" ::"r"(id) : "memory"); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

#ifdef DF_TIMING
// tuning build only (tools/build_variant.sh dft chol_df.cu -DDF_TIMING): per tile 8 globaltimer stamps (ns) and, for
// diagonal tiles, clock64 phase stamps of the in-CTA factorisation; read with gingr_debug_chol_df_timing
__device__ unsigned long long df_stamps[64 * 64 * 16];
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define DF_STAMP(tile, k) do { if (threadIdx.x == 0 && (tile) < 64 * 64) df_stamps[(tile) * 16 + (k)] = gtime(); } while (0)
#define DF_CLOCK(tile, k) do { if (threadIdx.x == 0 && (tile) < 64 * 64) df_stamps[(tile) * 16 + 8 + (k)] = (unsigned long long)clock64(); } while (0)
// per-step profile of the in-CTA factorisation of tile 0 (lane 0 of the warp that executes the marked code)
__device__ long long potrf_prof[32 * 8];
#define PF_MARK(s, k) do { if ((threadIdx.x & 31) == 0 && tile_id == 0) potrf_prof[(s) * 8 + (k)] = clock64(); } while (0)
#else
#define PF_MARK(s, k) ((void)0)
#define DF_STAMP(tile, k) ((void)0)
#define DF_CLOCK(tile, k) ((void)0)
#endif

struct DfParams {
  double* A;
  int ld, n, nrows, nb, nbr, ntasks;
  int* sync;      // [0] ticket counter, [1] finished CTAs, [2 ...] flags[nbr][nb]
  double* linv;   // [nb][64][64] inverses of the diagonal blocks
  int* info;
};

// 64 rows x 64 columns of A starting at (row0, col0) -> s (pitch TP); rows >= rows_valid and columns >= ld are zero-filled
__device__ __forceinline__ void load_tile_async(double* s, const double* __restrict__ A, int ld, int row0, int col0,
                                                int rows_valid, int tid) {
#pragma unroll 4
  for (int e = tid; e < TB * (TB / 2); e += DF_THREADS) {
    const int i = e >> 5, c = (e & 31) * 2;
    double* dst = s + i * TP + c;
    if (i < rows_valid && col0 + c < ld) cp_async16(dst, A + (size_t)(row0 + i) * ld + col0 + c);   // never past the row pitch
    else *reinterpret_cast<double2*>(dst) = make_double2(0.0, 0.0);
  }
}

// Warp tile of the 8 warps: 16 rows x 32 columns; acc[i][j] = rows wm*16 + i*8 + g, columns wn*32 + j*8 + 2t (+1).
// acc += I K^T over the 64 columns of the two shared tiles
__device__ __forceinline__ void mma_tile(double (&acc)[2][4][2], const double* __restrict__ sI,
                                         const double* __restrict__ sK, int wm, int wn, int g, int t) {
#pragma unroll 4
  for (int c4 = 0; c4 < TB / 4; ++c4) {
    double af[2], bf[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) af[i] = sI[(wm * 16 + i * 8 + g) * TP + c4 * 4 + t];
#pragma unroll
    for (int j = 0; j < 4; ++j) bf[j] = sK[(wn * 32 + j * 8 + g) * TP + c4 * 4 + t];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
  }
}

// diagonal task: accV += I K^T and (unless this warp sits in the unused upper-right quarter) accS += I I^T
__device__ __forceinline__ void mma_tile2(double (&accV)[2][4][2], double (&accS)[2][4][2], const double* __restrict__ sI,
                                          const double* __restrict__ sK, bool doS, int wm, int wn, int g, int t) {
#pragma unroll 2
  for (int c4 = 0; c4 < TB / 4; ++c4) {
    double af[2], bk[4], bi[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) af[i] = sI[(wm * 16 + i * 8 + g) * TP + c4 * 4 + t];
#pragma unroll
    for (int j = 0; j < 4; ++j) bk[j] = sK[(wn * 32 + j * 8 + g) * TP + c4 * 4 + t];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma884(accV[i][j][0], accV[i][j][1], af[i], bk[j]);
    if (doS) {
#pragma unroll
      for (int j = 0; j < 4; ++j) bi[j] = sI[(wn * 32 + j * 8 + g) * TP + c4 * 4 + t];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(accS[i][j][0], accS[i][j][1], af[i], bi[j]);
    }
  }
}

// X = V Z^T with Z lower triangular (Z = L^-1): column c of X only needs k <= c, so a fragment column block jj stops at
// k4 < wn*8 + jj*2 + 2
__device__ __forceinline__ void mma_tile_lower(double (&acc)[2][4][2], const double* __restrict__ sI,
                                               const double* __restrict__ sK, int wm, int wn, int g, int t) {
#pragma unroll 2
  for (int c4 = 0; c4 < TB / 4; ++c4) {
    if (c4 >= wn * 8 + 8) break;
    double af[2], bf[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) af[i] = sI[(wm * 16 + i * 8 + g) * TP + c4 * 4 + t];
#pragma unroll
    for (int j = 0; j < 4; ++j) bf[j] = sK[(wn * 32 + j * 8 + g) * TP + c4 * 4 + t];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (c4 < wn * 8 + j * 2 + 2) {
#pragma unroll
        for (int i = 0; i < 2; ++i) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
      }
    }
  }
}

#include "chol_potrf.cuh"

GINGR_KERNEL((DF_THREADS, 1), chol_df_kernel, const DfParams& P) {
  extern __shared__ __align__(16) double dsm[];
  double* bufI0 = dsm;                       // stage 0, row operand    | X_{j,j-1} of a diagonal task
  double* bufK0 = dsm + TILE_DOUBLES;        // stage 0, column operand | Z of the finishing product
  double* bufI1 = dsm + 2 * TILE_DOUBLES;    // stage 1, row operand    | potrf: factor exchange G2
  double* bufK1 = dsm + 3 * TILE_DOUBLES;    // stage 1, column operand | potrf: rows below the square part
  double* sV0 = dsm + 4 * TILE_DOUBLES;      // input / updated value of the off-diagonal tile
  double* sA0 = dsm + 5 * TILE_DOUBLES;      // input / updated value of the diagonal tile (diagonal tasks)
  double* sDiag = dsm + 6 * TILE_DOUBLES;    // [64]
  double* sSub = sDiag + TB;                 // [32]
  unsigned long long* sBar = reinterpret_cast<unsigned long long*>(sSub + 32);   // [32] step barriers of potrf64
  __shared__ int s_task, s_pre[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // warp tile: 16 rows x 32 columns.  wm = warp & 3 puts one left-half and one right-half warp on every SM sub-partition
  // (warp % 4): the triangular products give the right half 2.6x the work of the left one
  const int wm = warp & 3, wn = warp >> 2, g = lane >> 2, t = lane & 3;
  int* flags = P.sync + 2;
  const double* __restrict__ A = P.A;
  const int ld = P.ld, nb = P.nb;
  if (tid < 32) mbar_init(&sBar[tid], 1);
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  unsigned potrf_calls = 0;   // the loop-top barrier orders the initialisation before the first use

  for (;;) {
    __syncthreads();   // s_task / shared buffers of the previous task are free
    if (tid == 0) s_task = atomicAdd(&P.sync[0], 1);
    __syncthreads();
    int tt = s_task;
    if (tt >= P.ntasks) break;
    // ---- ticket -> task.  Column j: D(j) first, then T(i, j) for the rows i that no diagonal task owns -------------
    int j = 0;
    for (;;) {
      const int cnt = (P.nbr - j - 1) + (j + 1 >= nb ? 1 : 0);
      if (tt < cnt) break;
      tt -= cnt;
      ++j;
    }
    const bool isD = (tt == 0);
    const int rb = isD ? j : ((j + 1 >= nb) ? j + tt : j + 1 + tt);   // row block of the task
    const int cb = isD ? j - 1 : j;                                    // column block of its off-diagonal tile (-1: none)
    const bool hasV = cb >= 0;
    const int r0 = rb * TB;
    const int rcnt = min(TB, P.nrows - r0);                            // valid rows
    const int vb = hasV ? min(TB, P.n - cb * TB) : 0;                  // valid columns of the off-diagonal tile
    const int tile_id = rb * nb + (isD ? j : cb);
    (void)tile_id;
    DF_STAMP(tile_id, 0);

    // the task's own input tiles (their group completes long before it is needed)
    if (hasV) load_tile_async(sV0, A, ld, r0, cb * TB, rcnt, tid);
    if (isD) load_tile_async(sA0, A, ld, r0, r0, rcnt, tid);
    cp_async_commit();

    double accV[2][4][2], accS[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) accV[a][b][0] = accV[a][b][1] = accS[a][b][0] = accS[a][b][1] = 0.0;
    const bool doS = isD && !(wm < 2 && wn == 1);   // the upper-right quarter of a diagonal tile is never used

    // ---- left-looking updates over k < cb: V += X_{rb,k} X_{cb,k}^T, diagonal task also S += X_{rb,k} X_{rb,k}^T ----
    if (cb > 0) {
      const int* fI = flags + rb * nb;
      const int* fK = flags + cb * nb;
      if (tid == 0) {
        while (ld_acquire(fI) == 0) {}
        while (ld_acquire(fK) == 0) {}
      }
      __syncthreads();
      load_tile_async(bufI0, A, ld, r0, 0, rcnt, tid);
      load_tile_async(bufK0, A, ld, cb * TB, 0, TB, tid);
      cp_async_commit();
      for (int k = 0; k < cb; ++k) {
        const int st = k & 1;
        const double* sI = st ? bufI1 : bufI0;
        const double* sK = st ? bufK1 : bufK0;
        const bool more = (k + 1 < cb);
        if (tid == 0) {
          int pre = 0;
          if (more) pre = (ld_acquire(fI + k + 1) != 0) && (ld_acquire(fK + k + 1) != 0);
          s_pre[st] = pre;        // two slots: a slow reader of step k cannot see the value of step k + 1
        }
        cp_async_wait_all();
        __syncthreads();          // stage k landed; every thread is past the product of step k - 1; s_pre visible
        const bool pre = s_pre[st] != 0;
        if (more && pre) {
          load_tile_async(st ? bufI0 : bufI1, A, ld, r0, (k + 1) * TB, rcnt, tid);
          load_tile_async(st ? bufK0 : bufK1, A, ld, cb * TB, (k + 1) * TB, TB, tid);
          cp_async_commit();
        }
        if (isD) mma_tile2(accV, accS, sI, sK, doS, wm, wn, g, t);
        else mma_tile(accV, sI, sK, wm, wn, g, t);
        if (more && !pre) {
          if (tid == 0) {
            while (ld_acquire(fI + k + 1) == 0) {}
            while (ld_acquire(fK + k + 1) == 0) {}
          }
          __syncthreads();
          load_tile_async(st ? bufI0 : bufI1, A, ld, r0, (k + 1) * TB, rcnt, tid);
          load_tile_async(st ? bufK0 : bufK1, A, ld, cb * TB, (k + 1) * TB, TB, tid);
          cp_async_commit();
        }
      }
    }
    cp_async_wait_all();
    __syncthreads();   // the input tiles landed; the stage buffers are free
    DF_STAMP(tile_id, 1);

    if (hasV) {
      // ---- sV0 <- A - V (masked to the valid part);  X = sV0 Z^T with Z = L_cb^-1 ------------------------------------
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int row = wm * 16 + a * 8 + g, col = wn * 32 + b * 8 + 2 * t;
          double2* p = reinterpret_cast<double2*>(sV0 + row * TP + col);
          double2 v = *p;
          v.x = (row < rcnt && col < vb) ? v.x - accV[a][b][0] : 0.0;
          v.y = (row < rcnt && col + 1 < vb) ? v.y - accV[a][b][1] : 0.0;
          *p = v;
          accV[a][b][0] = accV[a][b][1] = 0.0;
        }
      if (tid == 0) while (ld_acquire(&flags[cb * nb + cb]) == 0) {}
      __syncthreads();
      DF_STAMP(tile_id, 2);
      {
        const double* Z = P.linv + (size_t)cb * TB * TB;
#pragma unroll 4
        for (int e = tid; e < TB * (TB / 2); e += DF_THREADS) {
          const int r = e >> 5, c = (e & 31) * 2;
          cp_async16(bufK0 + r * TP + c, Z + r * TB + c);
        }
        cp_async_commit();
      }
      cp_async_wait_all();
      __syncthreads();
      mma_tile_lower(accV, sV0, bufK0, wm, wn, g, t);
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int row = wm * 16 + a * 8 + g, col = wn * 32 + b * 8 + 2 * t;
          if (isD) *reinterpret_cast<double2*>(bufI0 + row * TP + col) = make_double2(accV[a][b][0], accV[a][b][1]);
          if (row < rcnt) {
            double* p = P.A + (size_t)(r0 + row) * ld + cb * TB + col;
            if (col + 1 < vb) *reinterpret_cast<double2*>(p) = make_double2(accV[a][b][0], accV[a][b][1]);
            else if (col < vb) p[0] = accV[a][b][0];
          }
        }
      __syncthreads();   // every thread's stores are issued; X is complete in shared memory (diagonal task)
      if (tid == DF_THREADS - 1) {   // the last warp pays for the fence, not the warp that leads the diagonal factorisation
        st_release(&flags[rb * nb + cb], 1);
      }
      DF_STAMP(tile_id, 3);
      if (!isD) continue;
      // the last update of the diagonal tile, with X_{j,j-1} straight from shared memory
      if (doS) mma_tile(accS, bufI0, bufI0, wm, wn, g, t);
    }

    // ---- diagonal task: sA0 <- A_jj - S, factorise, publish --------------------------------------------------------
    const int jb = min(TB, P.n - r0);      // valid columns of this block column
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int row = wm * 16 + a * 8 + g, col = wn * 32 + b * 8 + 2 * t;
        double2* p = reinterpret_cast<double2*>(sA0 + row * TP + col);
        double2 v = *p;
        v.x = (row < rcnt && col < jb) ? v.x - accS[a][b][0] : 0.0;
        v.y = (row < rcnt && col + 1 < jb) ? v.y - accS[a][b][1] : 0.0;
        *p = v;
      }
    __syncthreads();
    // rows >= jb of a diagonal tile lie below the square part (right-hand sides): set them aside, pad with identity
    const int ecnt = rcnt - jb;     // > 0 only in the last block column
    if (jb < TB) {
      for (int e = tid; e < TB * TB; e += DF_THREADS) {
        const int r = e >> 6, c = e & 63;
        if (r >= jb) {
          bufK1[r * TP + c] = sA0[r * TP + c];
          sA0[r * TP + c] = (r == c) ? 1.0 : 0.0;
        }
      }
      __syncthreads();
    }
    DF_STAMP(tile_id, 4);
    const double2* G2 = reinterpret_cast<const double2*>(bufI1);
    // Z = L^-1 is all the waiting tasks of this block column need: its rows go out WHILE the factorisation runs (the warps
    // whose columns are eliminated copy them, potrf64), only the first 8 rows are left for afterwards
    double* Z = P.linv + (size_t)j * TB * TB;
    const bool bad = potrf64(sA0, reinterpret_cast<double2*>(bufI1), sDiag, sSub, sBar, potrf_calls & 1u, tid, tile_id, Z);
    ++potrf_calls;
    DF_STAMP(tile_id, 5);
    if (bad && tid == 0) P.info[0] = 1;
    {
      const int c = tid >> 5, k = (tid & 31) * 2;     // 8 rows x 32 column pairs = 256 threads
      *reinterpret_cast<double2*>(Z + c * TB + k) = make_double2(potrf_Z(G2, c, k), potrf_Z(G2, c, k + 1));
    }
    __syncthreads();
    if (tid == 0) {
      st_release(&flags[j * nb + j], 1);
    }
    DF_STAMP(tile_id, 6);
    // ... then L and the solved extra rows, which nothing inside this kernel reads (a diagonal tile is never an operand)
    for (int e = tid; e < TB * TB; e += DF_THREADS) {
      const int r = e >> 6, c = e & 63;
      if (r < jb && c <= r) P.A[(size_t)(r0 + r) * ld + r0 + c] = potrf_L(G2, sDiag, sSub, r, c);
    }
    if (ecnt > 0) {
      for (int e = tid; e < ecnt * TB; e += DF_THREADS) {
        const int r = jb + (e >> 6), c = e & 63;
        if (c < jb) {
          const double* er = bufK1 + r * TP;
          double s0 = 0.0;
          for (int k = 0; k <= c; ++k) s0 = fma(er[k], potrf_Z(G2, c, k), s0);
          P.A[(size_t)(r0 + r) * ld + r0 + c] = s0;
        }
      }
    }
  }
  // ---- the last CTA out resets the tickets and flags for the next launch (no memset node in the captured graph) ----
  __shared__ int s_last;
  if (tid == 0) s_last = (atomicAdd(&P.sync[1], 1) == (int)gridDim.x - 1);
  __syncthreads();
  if (s_last) {
    for (int e = tid; e < P.nbr * nb; e += DF_THREADS) flags[e] = 0;
    if (tid == 0) { P.sync[0] = 0; P.sync[1] = 0; }
  }
}

// ---------------------------------------------------------------------------------------------
// n <= 64: the whole matrix is ONE diagonal block.  The data-flow kernel above would run its single task with 216 registers
// and 209 KB of shared memory -- one CTA per SM, which is what bounds a batch of 1024 chains of rank 50 (batch.cuh: 7 waves of
// 17 us).  Here: load, potrf64, write L, forward-substitute the rows below the square (x = b Z^T with Z = L^-1 from the same
// pass), 70 KB and <= 128 registers: two CTAs per SM, and nothing but the factorisation between load and store.
// ---------------------------------------------------------------------------------------------
constexpr size_t SMALL_SMEM = (size_t)(TILE_DOUBLES + TB * G2P * 2 + TB + 32 + 32) * sizeof(double) + 64;

GINGR_KERNEL((DF_THREADS, 2), chol_small_kernel, int n, int nrows, double* __restrict__ A, int ld, int* __restrict__ info) {
  extern __shared__ __align__(16) unsigned char small_smem[];
  double* sT = reinterpret_cast<double*>(small_smem);                  // [64][TP] the block, later a batch of extra rows
  double2* G2 = reinterpret_cast<double2*>(sT + TILE_DOUBLES);           // [64][G2P]
  double* sDiag = reinterpret_cast<double*>(G2 + TB * G2P);             // [64]
  double* sSub = sDiag + TB;                                            // [32]
  unsigned long long* sBar = reinterpret_cast<unsigned long long*>(sSub + 32);   // [32]
  const int tid = threadIdx.x;
  if (tid < 32) mbar_init(&sBar[tid], 1);
  for (int e = tid; e < TB * TB; e += DF_THREADS) {
    const int r = e >> 6, c = e & 63;
    sT[r * TP + c] = (r < n && c <= r) ? A[(size_t)r * ld + c] : (r == c ? 1.0 : 0.0);   // identity-padded beyond the valid part
  }
  __syncthreads();
  const bool bad = potrf64(sT, G2, sDiag, sSub, sBar, 0u, tid, 0);
  if (bad && tid == 0) info[0] = 1;
  for (int e = tid; e < TB * TB; e += DF_THREADS) {
    const int r = e >> 6, c = e & 63;
    if (r < n && c <= r) A[(size_t)r * ld + c] = potrf_L(G2, sDiag, sSub, r, c);
  }
  // rows below the square part (right-hand sides): x[c] = sum_{k <= c} b[k] Z[c][k], 64 rows at a time through sT
  for (int e0 = n; e0 < nrows; e0 += TB) {
    const int cnt = min(TB, nrows - e0);
    __syncthreads();
    for (int e = tid; e < cnt * TB; e += DF_THREADS) {
      const int r = e >> 6, c = e & 63;
      sT[r * TP + c] = c < n ? A[(size_t)(e0 + r) * ld + c] : 0.0;
    }
    __syncthreads();
    for (int e = tid; e < cnt * TB; e += DF_THREADS) {
      const int r = e >> 6, c = e & 63;
      if (c < n) {
        const double* er = sT + r * TP;
        double s0 = 0.0;
        for (int k = 0; k <= c; ++k) s0 = fma(er[k], potrf_Z(G2, c, k), s0);
        A[(size_t)(e0 + r) * ld + c] = s0;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// backward substitution  L^T c = z  with the published inverses Z_k = L_kk^-1 of the factorisation above: one CTA per
// 64-block, blocks become ready from the last one up.  CTA k accumulates  z_k - sum_{i>k} L_ik^T c_i  as the c_i appear
// and finishes with c_k = Z_k^T acc.  Everything the critical step needs is in shared memory BEFORE its flag arrives:
// Z_k, and the L_ik blocks stream through a two-deep cp.async ring one block ahead of the flags, so between two flags
// there is one 64 x 64 mat-vec from shared memory, one more with Z_k^T, a fence and the flag (chol.cu's kernel inverted
// its diagonal block itself and read every L_ik from global memory after the flag: 5.6 us per block, now ~2).
// flags: nb + 1 ints, zero on entry; the last CTA out zeroes them again.
// ---------------------------------------------------------------------------------------------
constexpr int BS_THREADS = 256;
constexpr size_t BS_SMEM = (size_t)(3 * TB * TB + TB + 4 * TB + TB) * sizeof(double);

__global__ void __launch_bounds__(BS_THREADS) chol_backsolve_z_kernel(int n, const double* __restrict__ L, int ld,
                                                                      const double* __restrict__ z, double* __restrict__ c,
                                                                      const double* __restrict__ linv, int* flags) {
  extern __shared__ __align__(16) double bsm[];
  double* sZ = bsm;                    // [64][64] Z_k
  double* sLb = bsm + TB * TB;         // [2][64][64] L_ik ring
  double* sc = bsm + 3 * TB * TB;      // [64] c_i
  double* sacc = sc + TB;              // [4][64] partial sums
  double* acc = sacc + 4 * TB;         // [64]
  const int nb = (n + TB - 1) / TB;
  const int k = nb - 1 - (int)blockIdx.x;   // first CTAs own the last blocks (solved first)
  const int tid = threadIdx.x, col = tid & 63, part = tid >> 6;
  const int k0 = k * TB, kcnt = min(TB, n - k0);
  auto load_block = [&](double* dst, int i) {   // rows of block i, columns of block k (k < i: all 64 columns exist)
    const int i0 = i * TB, icnt = min(TB, n - i0);
#pragma unroll 4
    for (int e = tid; e < TB * (TB / 2); e += BS_THREADS) {
      const int r = e >> 5, cc = (e & 31) * 2;
      if (r < icnt) cp_async16(dst + r * TB + cc, L + (size_t)(i0 + r) * ld + k0 + cc);
      else *reinterpret_cast<double2*>(dst + r * TB + cc) = make_double2(0.0, 0.0);
    }
  };
  {
    const double* Z = linv + (size_t)k * TB * TB;
#pragma unroll 4
    for (int e = tid; e < TB * (TB / 2); e += BS_THREADS) cp_async16(sZ + 2 * e, Z + 2 * e);
  }
  if (k + 1 < nb) load_block(sLb, nb - 1);
  cp_async_commit();
  if (tid < TB) acc[tid] = tid < kcnt ? z[k0 + tid] : 0.0;
  double s = 0.0;
  for (int i = nb - 1; i > k; --i) {
    const int st = (nb - 1 - i) & 1;
    __syncthreads();   // the other ring slot was read by the products of the previous step: every thread is past them
    if (i - 1 > k) load_block(sLb + (st ^ 1) * TB * TB, i - 1);
    cp_async_commit();
    if (tid == 0) while (ld_acquire(&flags[i]) == 0) {}
    asm volatile("cp.async.wait_group 1;\n" ::: "memory");
    __syncthreads();
    const int i0 = i * TB;
    if (tid < TB) sc[tid] = (i0 + tid < n) ? __ldcg(c + i0 + tid) : 0.0;
    __syncthreads();
    const double* Lb = sLb + st * TB * TB;
#pragma unroll
    for (int rr = 0; rr < 16; ++rr) s = fma(Lb[(part * 16 + rr) * TB + col], sc[part * 16 + rr], s);
  }
  cp_async_wait_all();
  sacc[part * TB + col] = s;
  __syncthreads();
  if (tid < TB) acc[tid] -= (sacc[tid] + sacc[TB + tid]) + (sacc[2 * TB + tid] + sacc[3 * TB + tid]);
  __syncthreads();
  // c_k = Z_k^T acc :  c[j] = sum_{i >= j} Z[i][j] acc[i]   (4 partial sums per output)
  {
    double t = 0.0;
#pragma unroll
    for (int rr = 0; rr < 16; ++rr) {
      const int i = part * 16 + rr;
      t = fma(sZ[i * TB + col], acc[i], t);     // Z is lower triangular with zeros above the diagonal
    }
    sacc[part * TB + col] = t;
  }
  __syncthreads();
  if (tid < kcnt) c[k0 + tid] = (sacc[tid] + sacc[TB + tid]) + (sacc[2 * TB + tid] + sacc[3 * TB + tid]);
  __syncthreads();
  if (tid == 0) {
    st_release(&flags[k], 1);
    if (atomicAdd(&flags[nb], 1) == nb - 1) {   // last CTA out: every flag has been read for the last time
      for (int e = 0; e <= nb; ++e) flags[e] = 0;
    }
  }
}

}  // namespace

int32_t CholWs::alloc(gingr_ctx* ctx, int n, int nrows) {
  const int nb = ceil_div(n, TB), nbr = ceil_div(nrows, TB);
  const size_t ns = 2 + (size_t)nb * nbr;
  if (sync.n < ns) {
    GINGR_CUDA_TRY(ctx, sync.alloc(ns));
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(sync.p, 0, sizeof(int) * ns, ctx->stream));
  }
  GINGR_CUDA_TRY(ctx, linv.alloc((size_t)nb * TB * TB));
  if (bsync.n < (size_t)nb + 1) {
    GINGR_CUDA_TRY(ctx, bsync.alloc((size_t)nb + 1));
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(bsync.p, 0, sizeof(int) * ((size_t)nb + 1), ctx->stream));
  }
  cap_n = std::max(cap_n, n);
  cap_nrows = std::max(cap_nrows, nrows);
  return GINGR_OK;
}

int32_t cholesky_df_enqueue(gingr_ctx* ctx, int n, int nrows, double* d_A, int ld, int* d_info, CholWs& ws) {
  static thread_local int attr_device = -1;
  if (attr_device != ctx->device) {
    GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(chol_df_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DF_SMEM));
    attr_device = ctx->device;
  }
  DfParams P;
  P.A = d_A;
  P.ld = ld;
  P.n = n;
  P.nrows = nrows;
  P.nb = ceil_div(n, TB);
  P.nbr = ceil_div(nrows, TB);
  P.ntasks = 0;   // per block column: the diagonal task + the rows no diagonal task owns
  for (int j = 0; j < P.nb; ++j) P.ntasks += (P.nbr - j - 1) + (j + 1 >= P.nb ? 1 : 0);
  if ((size_t)(2 + (size_t)P.nb * P.nbr) > ws.sync.n || (size_t)P.nb * TB * TB > ws.linv.n)
    return gingr_fail(ctx, GINGR_ERR_ARG, "cholesky: workspace too small");
  if ((ld & 1) != 0 || (((uintptr_t)d_A) & 15) != 0) return gingr_fail(ctx, GINGR_ERR_ARG, "cholesky: matrix must be 16-byte aligned with an even pitch");
  static const int env_small = [] { const char* e = getenv("GINGR_CHOL_SMALL"); return e ? atoi(e) : 1; }();
  if (P.nb == 1 && env_small) {
    static thread_local int attr_small = -1;
    if (attr_small != ctx->device) {
      GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(chol_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM));
      attr_small = ctx->device;
    }
    GINGR_LAUNCH(ctx, chol_small_kernel, 1, DF_THREADS, SMALL_SMEM, ctx->stream, n, nrows, d_A, ld, d_info);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    return GINGR_OK;
  }
  P.sync = ws.sync.p;
  P.linv = ws.linv.p;
  P.info = d_info;
  const int grid = std::min(P.ntasks, ctx->num_sms);
  GINGR_LAUNCH(ctx, chol_df_kernel, grid, DF_THREADS, DF_SMEM, ctx->stream, P);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t chol_backsolve_z_enqueue(gingr_ctx* ctx, int n, const double* d_L, int ld, const double* d_z, double* d_c, CholWs& ws) {
  static thread_local int attr_device = -1;
  if (attr_device != ctx->device) {
    GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(chol_backsolve_z_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BS_SMEM));
    attr_device = ctx->device;
  }
  const int nb = ceil_div(n, TB);
  if ((size_t)nb + 1 > ws.bsync.n || (size_t)nb * TB * TB > ws.linv.n) return gingr_fail(ctx, GINGR_ERR_ARG, "back solve: workspace too small");
  if (nb > ctx->num_sms) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "rank too large for the sync-free back solve");
  chol_backsolve_z_kernel<<<nb, BS_THREADS, BS_SMEM, ctx->stream>>>(n, d_L, ld, d_z, d_c, ws.linv.p, ws.bsync.p);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

}  // namespace gingr

#ifdef DF_TIMING
extern "C" GINGR_API int32_t gingr_debug_potrf_profile(long long* out) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, gingr::potrf_prof, sizeof(long long) * 32 * 8);
  return 0;
}
extern "C" GINGR_API int32_t gingr_debug_chol_df_timing(unsigned long long* out, int32_t count) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, gingr::df_stamps, sizeof(unsigned long long) * (size_t)count);
  return 0;
}
#endif
