// gram.cu -- K3a: weighted Gram matrix of the GPMM basis on the FP64 tensor pipe (sm_100a).
//
// Replaces the dense products of scalismo's regression at the call site GingrAlgorithm.scala:300
// (`model.transform(rigid).posterior(obs)`; SURVEY.md A3):  Mx = Q^T L^-1 Q + I_r  with
// Q = Phi' diag(sqrt(lambda)), L^-1 = blockdiag(inv(cov_i)).  For the isotropic noise GiNGR's CPD/ICP
// configs hand over (CPD.scala:120-128, ICP.scala:90-92) cov_i = v_i I3 and the rotation of the posed model
// cancels ((I (x) R)^T (W (x) I3) (I (x) R) = W (x) I3), so
//     Mx = I + D G D,   G = Phi^T diag(w_row) Phi,   w_row[3i+d] = 1 / v_i,   D = diag(sqrt(lambda)).
// G is a real dense FP64 contraction (3n x r by r) and runs on DMMA: tcgen05 has no FP64 kind, the sm_100a
// FP64 tensor instruction is mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4; the m16n8k{4,8,16} PTX shapes lower to it).
//
// Kernel: only the lower-triangular 128x128 tiles are computed (symmetric minimum 3n r (r+1) flop).
// One persistent CTA per SM works through a static list of (tile, k-chunk range) segments (split-K schedule
// built on the host, GramPlan::build): with T tiles on n SMs, T "main" CTAs each own one tile and walk the
// rows of Phi in lockstep from the top (every row slab is fetched from HBM once and served to the other
// tiles from L2), while the remaining n - T CTAs take the bottom slab of every tile, so all SMs finish
// together for any r.  Each segment accumulates in registers (warp tile 64x32 = 32 DMMA accumulator
// fragments), operands stream global -> shared with a 3-stage cp.async pipeline ([k][col] tiles of 32 rows,
// pitch 132 doubles: conflict-free LDS.64 fragment loads), the row weights are multiplied into the B
// fragments.  Partial tiles go to a workspace and are summed in fixed
// order by gram_finish_kernel (deterministic; no atomics), which also applies D, adds I and the landmark
// blocks (full 3x3 covariances, GeneralRegistrationState.scala:43-62).
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "batch.cuh"
#include "dmma.cuh"
#include "posterior.cuh"

namespace gingr {

constexpr int BT = 128;          // output tile edge
constexpr int BK = 32;           // rows of Phi per pipeline stage
constexpr int STAGES = 3;
constexpr int PITCH = BT + 4;    // smem row pitch in doubles (== 4 mod 16 -> conflict-free fragment loads)
#ifndef GRAM_WARPS_M
#define GRAM_WARPS_M 2           // warps along the tile rows: 2 -> 8 warps of 64x32, 4 -> 16 warps of 32x32
#endif
constexpr int GRAM_THREADS = GRAM_WARPS_M * 4 * 32;
constexpr int WTM = BT / GRAM_WARPS_M;   // warp tile rows
constexpr int MI = WTM / 8;              // 8-row DMMA fragments per warp tile
constexpr size_t GRAM_SMEM = (size_t)STAGES * (2 * BK * PITCH + BK) * sizeof(double);

// segment of work of one CTA: tile (ta >= tb), chunk range [c0, c1), output slot
struct GramSegment {
  int ta, tb, c0, c1, slot, pad0, pad1, pad2;
};

// phi: [rows][rp] row-major, wrow: [rows] (may be null = unit weights)
__global__ void __launch_bounds__(GRAM_THREADS, 1) gram_streamk_kernel(int rows, int rp,
                                                                       const double* __restrict__ phi,
                                                                       const double* __restrict__ wrow,
                                                                       const GramSegment* __restrict__ segs,
                                                                       const int* __restrict__ seg_begin,
                                                                       double* __restrict__ partial) {
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;                                   // [STAGES][BK][PITCH]
  double* sB = sA + (size_t)STAGES * BK * PITCH;       // [STAGES][BK][PITCH]
  double* sW = sB + (size_t)STAGES * BK * PITCH;       // [STAGES][BK]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 2, wn = warp & 3;             // GRAM_WARPS_M x 4 warps, warp tile WTM x 32
  const int g = lane >> 2, t = lane & 3;

  for (int si = seg_begin[blockIdx.x]; si < seg_begin[blockIdx.x + 1]; ++si) {
    const GramSegment sg = segs[si];
    const int a0 = sg.ta * BT, b0 = sg.tb * BT;
    const bool diag = sg.ta == sg.tb;
    const int nchunks = sg.c1 - sg.c0;

    double acc[MI][4][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    auto issue = [&](int chunk) {
      const int stage = chunk % STAGES;
      const int krow0 = (sg.c0 + chunk) * BK;
      double* dA = sA + (size_t)stage * BK * PITCH;
      double* dB = sB + (size_t)stage * BK * PITCH;
      // BK rows x 64 16-byte pieces per operand tile, BK * 64 / 256 per thread
#pragma unroll
      for (int q = 0; q < BK * 64 / GRAM_THREADS; ++q) {
        const int e = tid + q * GRAM_THREADS;
        const int kr = e >> 6, c2 = (e & 63) * 2;
        const int krow = krow0 + kr;
        const bool rok = krow < rows;
        {
          const int col = a0 + c2;
          const bool ok = rok && col < rp;
          cp_async16(dA + kr * PITCH + c2, ok ? (const void*)(phi + (size_t)krow * rp + col) : (const void*)phi,
                     ok ? 16 : 0);
        }
        if (!diag) {
          const int col = b0 + c2;
          const bool ok = rok && col < rp;
          cp_async16(dB + kr * PITCH + c2, ok ? (const void*)(phi + (size_t)krow * rp + col) : (const void*)phi,
                     ok ? 16 : 0);
        }
      }
      if (tid < BK) {
        const int krow = krow0 + tid;
        const bool ok = krow < rows && wrow != nullptr;
        cp_async8(sW + stage * BK + tid, ok ? (const void*)(wrow + krow) : (const void*)phi, ok ? 8 : 0);
      }
    };

    __syncthreads();  // previous segment's readers are done with the stages
#pragma unroll
    for (int p = 0; p < STAGES - 1; ++p) {
      if (p < nchunks) issue(p);
      cp_async_commit();
    }
    for (int ch = 0; ch < nchunks; ++ch) {
      cp_async_wait<STAGES - 2>();
      __syncthreads();
      if (ch + STAGES - 1 < nchunks) issue(ch + STAGES - 1);
      cp_async_commit();
      const int stage = ch % STAGES;
      const double* tA = sA + (size_t)stage * BK * PITCH + wm * WTM + g;
      const double* tB = (diag ? sA : sB) + (size_t)stage * BK * PITCH + wn * 32 + g;
      const double* tW = sW + stage * BK;
#pragma unroll
      for (int k4 = 0; k4 < BK / 4; ++k4) {
        const int kk = k4 * 4 + t;
        const double wk = wrow ? tW[kk] : 1.0;
        double af[MI], bf[4];
#pragma unroll
        for (int i = 0; i < MI; ++i) af[i] = tA[kk * PITCH + i * 8];
#pragma unroll
        for (int j = 0; j < 4; ++j) bf[j] = tB[kk * PITCH + j * 8] * wk;
#pragma unroll
        for (int i = 0; i < MI; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
      }
    }
    cp_async_wait<0>();
    // store the partial tile: slot-major [slot][128][128]
    double* out = partial + (size_t)sg.slot * BT * BT;
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int row = wm * WTM + i * 8 + g, col = wn * 32 + j * 8 + 2 * t;
        *reinterpret_cast<double2*>(out + (size_t)row * BT + col) = make_double2(acc[i][j][0], acc[i][j][1]);
      }
  }
}

// ---------------------------------------------------------------------------------------------
// Warp-specialised variant (default): 8 consumer warps + 1 producer warp, stages handed over through mbarriers
// instead of a CTA-wide barrier per chunk.  ncu on the barrier version: 6 % of the warp samples sit in `barrier`
// and 7 % in `short scoreboard` right after it (the whole CTA drains the DMMA pipe every 32 rows); here a consumer
// warp only waits for "its" stage to be full and the producer refills a stage as soon as the 8 warps released it,
// also across segment boundaries (the partial-tile store of one segment overlaps the loads of the next).
//   full[s]   count 32 + transaction bytes: every producer lane arrives (lane 0 with expect_tx) and issues one
//             cp.async.bulk (global -> shared, 1 KB, completes on the mbarrier) per operand row
//   empty[s]  count 8 : one arrive per consumer warp after its last fragment load of the stage
// ---------------------------------------------------------------------------------------------
// Measured and NOT kept (round 2): skipping the fragments a tile does not need -- above the diagonal of the 16 diagonal
// tiles, past rank r in the last tile row (2000 -> 2048 padding), together 10 % of the DMMA slots -- with cyclic column
// fragments per warp (so that the four sub-partitions stay balanced on a diagonal tile) and a cost-weighted schedule.
// The masked loop itself is free (7.74 ms with every mask full, 7.72 ms for the cyclic mapping alone, against 7.75 ms),
// but as soon as fragments are really skipped the kernel takes 8.99 ms with the equal-chunk schedule and 14.1 ms with the
// weighted one: the CTAs of the cheaper tiles run ahead of the lockstep in which all CTAs walk the chunk index together,
// and the 512 KB strip of Phi that every tile shares per chunk no longer meets its readers in L2.
constexpr int GRAM_WS_THREADS = 256 + 32;
constexpr size_t GRAM_WS_SMEM = GRAM_SMEM + 2 * STAGES * sizeof(unsigned long long);

__device__ __forceinline__ void mbar_init(unsigned addr, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(addr), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(unsigned addr) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_cp_async_arrive(unsigned addr) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned addr, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(addr),
      "r"(parity)
      : "memory");
}

GINGR_KERNEL((GRAM_WS_THREADS, 1), gram_ws_kernel, int rows, int rp, const double* __restrict__ phi,
                                                                     const double* __restrict__ wrow,
                                                                     const double* __restrict__ resid, int r,
                                                                     const GramSegment* __restrict__ segs,
                                                                     const int* __restrict__ seg_begin,
                                                                     double* __restrict__ partial) {
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;                                   // [STAGES][BK][PITCH]
  double* sB = sA + (size_t)STAGES * BK * PITCH;       // [STAGES][BK][PITCH]
  double* sW = sB + (size_t)STAGES * BK * PITCH;       // [STAGES][BK]
  const unsigned bar0 = (unsigned)__cvta_generic_to_shared(sW + STAGES * BK);  // full[STAGES], empty[STAGES]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar0 + 8 * s, 32);
      mbar_init(bar0 + 8 * (STAGES + s), 8);
    }
  }
  __syncthreads();
  const int s_first = seg_begin[blockIdx.x], s_last = seg_begin[blockIdx.x + 1];

  if (warp == 8) {
    // ---------------- producer: one bulk copy (TMA engine, SASS UBLKCP) per operand row and lane ----------------
    unsigned it = 0;
    for (int si = s_first; si < s_last; ++si) {
      const GramSegment sg = segs[si];
      const int a0 = sg.ta * BT, b0 = sg.tb * BT;
      const bool diag = sg.ta == sg.tb;
      const unsigned bytes_a = (unsigned)(min(BT, rp - a0) * 8), bytes_b = diag ? 0u : (unsigned)(min(BT, rp - b0) * 8);
      // rhs for free: in the last tile row the first column of the A panel past the bulk copy (global index rp: the
      // copy also brings the zero padding [r, rp) of Phi) carries the residual of the row, so that output row rp of those
      // tiles is  sum_k resid_k w_k Phi[k][.]  = Phi^T W resid
      const int rcol = (resid != nullptr && rp - a0 > 0 && rp - a0 < BT) ? rp - a0 : -1;
      for (int ch = sg.c0; ch < sg.c1; ++ch, ++it) {
        const int stage = it % STAGES;
        const int krow = ch * BK + lane;                 // this lane's row of the chunk
        const bool rok = krow < rows;
        const double wv = (rok && wrow) ? wrow[krow] : 0.0;   // issued before the wait: latency off the critical path
        mbar_wait(bar0 + 8 * (STAGES + stage), ((it / STAGES) & 1) ^ 1);  // stage released by all consumer warps
        double* dA = sA + (size_t)stage * BK * PITCH + lane * PITCH;
        double* dB = sB + (size_t)stage * BK * PITCH + lane * PITCH;
        sW[stage * BK + lane] = wv;
        if (!rok) {  // rows past the end of Phi contribute zero (the tail chunk only)
          for (int c = 0; c < BT; ++c) { dA[c] = 0.0; if (!diag) dB[c] = 0.0; }
        } else if (rcol >= 0) {
          dA[rcol] = resid[krow];
        }
        const int valid = min(BK, rows - ch * BK);
        const unsigned full_bar = bar0 + 8 * stage;
        if (lane == 0) {
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(full_bar),
                       "r"((unsigned)valid * (bytes_a + bytes_b))
                       : "memory");
        } else {
          mbar_arrive(full_bar);  // releases this lane's plain stores (weights, zero rows)
        }
        if (rok) {
          const double* src = phi + (size_t)krow * rp;
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                           (unsigned)__cvta_generic_to_shared(dA)),
                       "l"(src + a0), "r"(bytes_a), "r"(full_bar)
                       : "memory");
          if (!diag)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                             (unsigned)__cvta_generic_to_shared(dB)),
                         "l"(src + b0), "r"(bytes_b), "r"(full_bar)
                         : "memory");
        }
      }
    }
    return;
  }

  // ---------------- consumers ----------------
  const int g = lane >> 2, t = lane & 3;
  if (rp < 64) {
    // rank < 64 (one tile, its upper-left quarter incl. the rhs in row rp: the small problems of batched chains, C1): the 64 x 64 corner is cut
    // into 16 x 32 pieces, one per warp -- with the 64 x 32 pieces below two warps would do all the MMAs and six none
    const int r0w = (warp & 3) * 16, c0w = (warp >> 2) * 32;
    unsigned it = 0;
    for (int si = s_first; si < s_last; ++si) {
      const GramSegment sg = segs[si];
      double acc[2][4][2];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
      for (int ch = sg.c0; ch < sg.c1; ++ch, ++it) {
        const int stage = it % STAGES;
        mbar_wait(bar0 + 8 * stage, (it / STAGES) & 1);
        const double* tA = sA + (size_t)stage * BK * PITCH + r0w + g;
        const double* tB = sA + (size_t)stage * BK * PITCH + c0w + g;    // one tile: always diagonal
        const double* tW = sW + stage * BK;
#pragma unroll
        for (int k4 = 0; k4 < BK / 4; ++k4) {
          const int kk = k4 * 4 + t;
          const double wk = wrow ? tW[kk] : 1.0;
          double af[2], bf[4];
#pragma unroll
          for (int i = 0; i < 2; ++i) af[i] = tA[kk * PITCH + i * 8];
#pragma unroll
          for (int j = 0; j < 4; ++j) bf[j] = tB[kk * PITCH + j * 8] * wk;
          if (k4 == BK / 4 - 1) {
            __syncwarp();
            if (lane == 0) mbar_arrive(bar0 + 8 * (STAGES + stage));
          }
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
      }
      double* out = partial + (size_t)sg.slot * BT * BT;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int row = r0w + i * 8 + g, col = c0w + j * 8 + 2 * t;
          *reinterpret_cast<double2*>(out + (size_t)row * BT + col) = make_double2(acc[i][j][0], acc[i][j][1]);
        }
    }
    return;
  }
  const int wm = warp >> 2, wn = warp & 3;             // 2 x 4 warps, warp tile 64 x 32
  unsigned it = 0;
  for (int si = s_first; si < s_last; ++si) {
    const GramSegment sg = segs[si];
    const bool diag = sg.ta == sg.tb;
    // a warp whose 64 x 32 piece lies past the matrix (rank far below the tile edge: the small problems of batched chains;
    // row rp may carry the rhs) only keeps the pipeline's barriers moving; the finish never reads its part of the tile
    const bool idle = sg.ta * BT + wm * 64 > rp || sg.tb * BT + wn * 32 >= rp;
    double acc[8][4][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    for (int ch = sg.c0; ch < sg.c1; ++ch, ++it) {
      const int stage = it % STAGES;
      mbar_wait(bar0 + 8 * stage, (it / STAGES) & 1);
      if (idle) {
        __syncwarp();
        if (lane == 0) mbar_arrive(bar0 + 8 * (STAGES + stage));
        continue;
      }
      const double* tA = sA + (size_t)stage * BK * PITCH + wm * 64 + g;
      const double* tB = (diag ? sA : sB) + (size_t)stage * BK * PITCH + wn * 32 + g;
      const double* tW = sW + stage * BK;
#pragma unroll
      for (int k4 = 0; k4 < BK / 4; ++k4) {
        const int kk = k4 * 4 + t;
        const double wk = wrow ? tW[kk] : 1.0;
        double af[8], bf[4];
#pragma unroll
        for (int i = 0; i < 8; ++i) af[i] = tA[kk * PITCH + i * 8];
#pragma unroll
        for (int j = 0; j < 4; ++j) bf[j] = tB[kk * PITCH + j * 8] * wk;
        if (k4 == BK / 4 - 1) {  // last fragment loads of the stage are in registers: hand the stage back
          __syncwarp();
          if (lane == 0) mbar_arrive(bar0 + 8 * (STAGES + stage));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
      }
    }
    if (idle) continue;
    double* out = partial + (size_t)sg.slot * BT * BT;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int row = wm * 64 + i * 8 + g, col = wn * 32 + j * 8 + 2 * t;
        *reinterpret_cast<double2*>(out + (size_t)row * BT + col) = make_double2(acc[i][j][0], acc[i][j][1]);
      }
  }
}

// Sum the partial tiles in slot order and emit  out = add_identity * I + D (G + LM) D  (both triangles).
// tile_first[t] .. tile_first[t+1] are the slots of lower-triangular tile t (t = ta (ta+1)/2 + tb).
// Landmark term: LM[a][b] = sum_l sum_{d,e} phi_l[d][a] A_l[d][e] phi_l[e][b]  with lm_rows [L][3][rp], lm_A [L][9].
GINGR_KERNEL((256), gram_finish_kernel, int r, int rp, int ld_out, const double* __restrict__ partial,
                                                          const int* __restrict__ tile_first,
                                                          const double* __restrict__ sqrt_lambda,
                                                          double add_identity, int L,
                                                          const double* __restrict__ lm_rows,
                                                          const double* __restrict__ lm_A, double* __restrict__ out,
                                                          int packed /*1: packed lower tiles, 2: matrix without the mirror*/,
                                                          int rhs_row /*1: row rp of the last tile row holds Phi^T W resid*/,
             int nt, int slices /*grid (nt, nt * slices): blockIdx.z is left to the batched form (batch.cuh)*/) {
  const int ta = blockIdx.y % nt, tb = blockIdx.x, slice = blockIdx.y / nt;
  if (tb > ta) return;
  const int tile = ta * (ta + 1) / 2 + tb;
  const int s0 = tile_first[tile], s1 = tile_first[tile + 1];
  if (rhs_row && ta == nt - 1) {
    // the rhs that rode along (gram_ws_kernel): out[r][b] = sqrt_lambda[b] * sum of the partials, no identity, no mirror
    const int row = rp - ta * BT;
    for (int col = slice * 256 + threadIdx.x; col < BT; col += 256 * slices) {
      const int b = tb * BT + col, e = row * BT + col;
      if (b >= r) continue;
      double s = 0.0;
      for (int k = s0; k < s1; ++k) s += partial[(size_t)k * BT * BT + e];
      const double v = (sqrt_lambda ? sqrt_lambda[b] : 1.0) * s;
      if (packed == 1) out[(size_t)tile * BT * BT + e] = v;
      else out[(size_t)r * ld_out + b] = v;
    }
  }
  // blockIdx.z slices the elements of the tile: a small matrix has few tiles and would otherwise be finished by a
  // handful of latency-bound CTAs
  const int e_end = min(BT, r - ta * BT) * BT;   // rows of the tile inside the matrix (a small rank uses a corner of its one tile)
  for (int e = slice * 256 + threadIdx.x; e < e_end; e += 256 * slices) {
    const int row = e / BT, col = e % BT;
    const int a = ta * BT + row, b = tb * BT + col;
    if (a >= r || b >= r || b > a) continue;
    double s = 0.0;
    for (int k = s0; k < s1; ++k) s += partial[(size_t)k * BT * BT + e];
    for (int l = 0; l < L; ++l) {
      const double* pr = lm_rows + (size_t)l * 3 * rp;
      const double* A = lm_A + l * 9;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const double pa = pr[d * rp + a];
        s += pa * (A[d * 3] * pr[b] + A[d * 3 + 1] * pr[rp + b] + A[d * 3 + 2] * pr[2 * rp + b]);
      }
    }
    const double da = sqrt_lambda ? sqrt_lambda[a] : 1.0, db = sqrt_lambda ? sqrt_lambda[b] : 1.0;
    const double v = da * s * db;
    if (packed == 1) {   // lower tiles back to back (what a multi-rank iteration all-reduces: half of the full rectangle)
      out[(size_t)tile * BT * BT + e] = v + (a == b ? add_identity : 0.0);
      continue;
    }
    out[(size_t)a * ld_out + b] = v + (a == b ? add_identity : 0.0);
    if (a != b && packed != 2) out[(size_t)b * ld_out + a] = v;   // the mirror is a column-wise (uncoalesced) write
  }
}

// ---------------------------------------------------------------------------------------------
// host side: static stream-K schedule
// ---------------------------------------------------------------------------------------------
int32_t GramPlan::build(gingr_ctx* ctx, int rows_, int r_, int rp_, int max_cta) {
  rows = rows_;
  r = r_;
  rp = rp_;
  nt = ceil_div(r, BT);
  ntiles = nt * (nt + 1) / 2;
  nchunks = std::max(1, ceil_div(rows, BK));
  ncta = max_cta > 0 ? std::min(ctx->num_sms, max_cta) : ctx->num_sms;
  const int n = ncta, K = nchunks;
  std::vector<std::pair<int, int>> tile_ab(ntiles);
  for (int a = 0, k = 0; a < nt; ++a)
    for (int b = 0; b <= a; ++b) tile_ab[k++] = {a, b};
  struct Seg { int cta, tile, c0, c1; };
  std::vector<Seg> list;
  // full rounds: n tiles at a time, every CTA walks all K chunks of its tile (lockstep -> L2 reuse)
  const int full_rounds = ntiles / n, rem = ntiles % n;
  for (int round = 0; round < full_rounds; ++round)
    for (int c = 0; c < n; ++c) list.push_back({c, round * n + c, 0, K});
  if (rem > 0) {
    // last round: rem main CTAs take chunks [0, K1) of their tile, the other n - rem CTAs share the bottom
    // slabs [K1, K) of all rem tiles; every CTA ends up with ~ rem K / n chunks
    // equal chunk counts would leave the n - rem tail CTAs late: each of their ~rem / (n - rem) + 1 pieces costs a
    // pipeline refill and a 128 KB partial tile on top of its chunks (about 0.75 chunk times, from the phase times of the
    // 8-GPU iteration: 235 chunks per tile, 12 tail CTAs with 11-12 pieces each).  K1 minimises the later of the two.
    int K1 = (int)((int64_t)K * rem / n);
    {
      const double ov = 0.75, pieces = (double)rem / (n - rem) + 1.0;
      double best_t = 1e300;
      int best_k = K1;
      for (int k = std::max(0, K1 - 2); k <= std::min(K, K1 + 8); ++k) {
        const double t_main = k > 0 ? k + ov : 0.0, t_tail = (double)rem * (K - k) / (n - rem) + (K - k > 0 ? ov * pieces : 0.0);
        const double t = std::max(t_main, t_tail);
        if (t < best_t) { best_t = t; best_k = k; }
      }
      K1 = best_k;
    }
    const int base_tile = full_rounds * n;
    for (int c = 0; c < rem; ++c)
      if (K1 > 0) list.push_back({c, base_tile + c, 0, K1});
    const int tail = K - K1, ntail = n - rem;
    const int64_t total = (int64_t)rem * tail;
    for (int j = 0; j < ntail; ++j) {
      int64_t u = total * j / ntail;
      const int64_t u1 = total * (j + 1) / ntail;
      while (u < u1) {
        const int tile = (int)(u / tail), c0 = (int)(u % tail);
        const int c1 = (int)std::min<int64_t>(tail, c0 + (u1 - u));
        list.push_back({rem + j, base_tile + tile, K1 + c0, K1 + c1});
        u += c1 - c0;
      }
    }
  }
  // slots: segments of a tile are numbered consecutively (ascending chunk) -> fixed summation order
  std::vector<int> order(list.size());
  for (size_t i = 0; i < list.size(); ++i) order[i] = (int)i;
  std::sort(order.begin(), order.end(), [&](int x, int y) {
    return list[x].tile != list[y].tile ? list[x].tile < list[y].tile : list[x].c0 < list[y].c0;
  });
  std::vector<int> slot_of(list.size());
  std::vector<int> tile_first(ntiles + 1, 0);
  for (size_t s = 0; s < order.size(); ++s) {
    slot_of[order[s]] = (int)s;
    tile_first[list[order[s]].tile + 1] = (int)s + 1;
  }
  for (int tix = 1; tix <= ntiles; ++tix) tile_first[tix] = std::max(tile_first[tix], tile_first[tix - 1]);
  // per-CTA lists in launch order (a CTA's main segment first, then its tail pieces)
  std::vector<GramSegment> segs;
  std::vector<int> seg_begin(n + 1, 0);
  for (int c = 0; c < n; ++c) {
    seg_begin[c] = (int)segs.size();
    for (size_t i = 0; i < list.size(); ++i)
      if (list[i].cta == c) {
        GramSegment g;
        g.ta = tile_ab[list[i].tile].first;
        g.tb = tile_ab[list[i].tile].second;
        g.c0 = list[i].c0;
        g.c1 = list[i].c1;
        g.slot = slot_of[i];
        g.pad0 = g.pad1 = g.pad2 = 0;
        segs.push_back(g);
      }
  }
  seg_begin[n] = (int)segs.size();
  nsegs = (int)segs.size();
  GINGR_CUDA_TRY(ctx, d_segs.alloc(std::max<size_t>(segs.size(), 1) * sizeof(GramSegment) / sizeof(int)));
  GINGR_CUDA_TRY(ctx, d_seg_begin.alloc(seg_begin.size()));
  GINGR_CUDA_TRY(ctx, d_tile_first.alloc(tile_first.size()));
  GINGR_CUDA_TRY(ctx, d_partial.alloc((size_t)std::max(nsegs, 1) * BT * BT));
  if (nsegs > 0)
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_segs.p, segs.data(), segs.size() * sizeof(GramSegment), cudaMemcpyHostToDevice,
                                        ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_seg_begin.p, seg_begin.data(), seg_begin.size() * sizeof(int),
                                      cudaMemcpyHostToDevice, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_tile_first.p, tile_first.data(), tile_first.size() * sizeof(int),
                                      cudaMemcpyHostToDevice, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // host vectors go out of scope
  GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(gram_streamk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)GRAM_SMEM));
  GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(gram_ws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)GRAM_WS_SMEM));
  return GINGR_OK;
}

// partial tiles of G = Phi^T diag(wrow) Phi  (wrow may be null)
bool gram_rhs_fusable(const GramPlan& plan) {
  static const int use_ws = [] { const char* e = getenv("GINGR_GRAM_WS"); return e ? atoi(e) : 1; }();
  static const int fuse = [] { const char* e = getenv("GINGR_GRAM_RHS"); return e ? atoi(e) : 1; }();
  // the same answer on every rank (a rank without rows just contributes zero partials)
  return fuse && use_ws && GRAM_WARPS_M == 2 && (plan.rp % BT) != 0;
}

int32_t gram_partials_enqueue(gingr_ctx* ctx, GramPlan& plan, const double* d_phi, const double* d_wrow,
                              cudaEvent_t ev0, cudaEvent_t ev1, const double* d_resid) {
  if (d_resid && !gram_rhs_fusable(plan)) return gingr_fail(ctx, GINGR_ERR_ARG, "gram: the rhs cannot ride along for this rank");
  if (ev0) cudaEventRecord(ev0, ctx->stream);
  if (plan.rows > 0 && plan.nsegs > 0) {
    static const int use_ws = [] { const char* e = getenv("GINGR_GRAM_WS"); return e ? atoi(e) : 1; }();
    if (use_ws && GRAM_WARPS_M == 2)
      GINGR_LAUNCH(ctx, gram_ws_kernel, plan.ncta, GRAM_WS_THREADS, GRAM_WS_SMEM, ctx->stream, 
          plan.rows, plan.rp, d_phi, d_wrow, d_resid, plan.r, reinterpret_cast<const GramSegment*>(plan.d_segs.p), plan.d_seg_begin.p,
          plan.d_partial.p);
    else
      gram_streamk_kernel<<<plan.ncta, GRAM_THREADS, GRAM_SMEM, ctx->stream>>>(
          plan.rows, plan.rp, d_phi, d_wrow, reinterpret_cast<const GramSegment*>(plan.d_segs.p), plan.d_seg_begin.p,
          plan.d_partial.p);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
  } else {
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(plan.d_partial.p, 0, plan.d_partial.n * sizeof(double), ctx->stream));
  }
  if (ev1) cudaEventRecord(ev1, ctx->stream);
  return GINGR_OK;
}

// out[r x r] (pitch ld_out) = add_identity I + D (sum of partial tiles + landmark blocks) D
// out (LOWER triangle, pitch ld_out) <- the lower tiles of a packed buffer [tile][128][128] (tile = ta (ta + 1) / 2 + tb)
__global__ void __launch_bounds__(256) gram_unpack_kernel(int r, int rp, int ld_out, const double* __restrict__ packed,
                                                          double* __restrict__ out, int rhs_row) {
  const int ta = blockIdx.y, tb = blockIdx.x;
  if (tb > ta) return;
  const int tile = ta * (ta + 1) / 2 + tb;
  for (int e = blockIdx.z * 256 + threadIdx.x; e < BT * BT; e += 256 * gridDim.z) {
    const int row = e / BT, col = e % BT;
    const int a = ta * BT + row, b = tb * BT + col;
    if (a >= r || b >= r || b > a) continue;
    out[(size_t)a * ld_out + b] = packed[(size_t)tile * BT * BT + e];   // lower triangle: all the factorisation reads
  }
  if (rhs_row && ta == (int)gridDim.y - 1) {
    const int row = rp - ta * BT;
    for (int col = blockIdx.z * 256 + threadIdx.x; col < BT; col += 256 * gridDim.z) {
      const int b = tb * BT + col;
      if (b < r) out[(size_t)r * ld_out + b] = packed[(size_t)tile * BT * BT + row * BT + col];
    }
  }
}

size_t gram_packed_doubles(const GramPlan& plan) { return (size_t)(plan.nt * (plan.nt + 1) / 2) * BT * BT; }

int32_t gram_unpack_enqueue(gingr_ctx* ctx, GramPlan& plan, const double* d_packed, int ld_out, double* d_out, bool rhs_row) {
  const int tiles = plan.nt * (plan.nt + 1) / 2;
  const int slices = std::max(1, std::min(64, (8 * ctx->num_sms) / std::max(tiles, 1)));
  gram_unpack_kernel<<<dim3(plan.nt, plan.nt, slices), 256, 0, ctx->stream>>>(plan.r, plan.rp, ld_out, d_packed, d_out, rhs_row ? 1 : 0);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t gram_finish_enqueue(gingr_ctx* ctx, GramPlan& plan, const double* d_partial, const double* d_sqrt_lambda,
                            double add_identity, int L, const double* d_lm_rows, const double* d_lm_A, int ld_out,
                            double* d_out, bool packed, bool lower_only, bool rhs_row) {
  const int tiles = plan.nt * (plan.nt + 1) / 2;
  // (chains batched in one launch fill the machine by themselves: batch.cuh)
  // ~8 CTAs per SM: the kernel is a latency-bound stream of a few dependent loads per element
  const int slices = ctx->rec ? 1 : std::max(1, std::min(64, (8 * ctx->num_sms) / std::max(tiles, 1)));
  GINGR_LAUNCH(ctx, gram_finish_kernel, dim3(plan.nt, plan.nt * slices), 256, 0, ctx->stream, plan.r, plan.rp, ld_out, d_partial,
                                                                      plan.d_tile_first.p, d_sqrt_lambda, add_identity,
                                                                      L, d_lm_rows, d_lm_A, d_out, packed ? 1 : (lower_only ? 2 : 0),
                                                                      rhs_row ? 1 : 0, plan.nt, slices);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

}  // namespace gingr
