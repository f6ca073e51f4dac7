// posterior.cuh -- host-side interface of the K3 posterior kernels (gram.cu, chol.cu, vecops.cu).
#pragma once
#include "common.cuh"

namespace gingr {

// ---- gram.cu -------------------------------------------------------------------------------------
struct GramPlan {
  int rows = 0, r = 0, rp = 0;
  int nt = 0, ntiles = 0, nchunks = 0, ncta = 0, nsegs = 0;
  DevBuf<int> d_segs;        // GramSegment[nsegs]
  DevBuf<int> d_seg_begin;   // [ncta + 1]
  DevBuf<int> d_tile_first;  // [ntiles + 1]
  DevBuf<double> d_partial;  // [nsegs][128][128]
  // max_cta > 0 caps the CTAs of the schedule (many chains batched in one launch: a chain's Gram on few CTAs, batch.cuh)
  int32_t build(gingr_ctx* ctx, int rows, int r, int rp, int max_cta = 0);
};
// d_resid (optional, needs gram_rhs_fusable): per-row residuals c_k; row r of the last tile row then comes out as
// sum_k c_k w_k Phi[k][.] = Phi^T W c -- the right-hand side of the regression without a pass of its own over Phi
// (finish / unpack with rhs_row = true emit it as row r of the matrix)
bool gram_rhs_fusable(const GramPlan& plan);
int32_t gram_partials_enqueue(gingr_ctx* ctx, GramPlan& plan, const double* d_phi, const double* d_wrow,
                              cudaEvent_t ev0 = nullptr, cudaEvent_t ev1 = nullptr, const double* d_resid = nullptr);
// packed: d_out receives the lower tiles back to back ([tile][128][128], gram_packed_doubles) instead of the r x r matrix --
// what a multi-rank iteration all-reduces (half the bytes); gram_unpack_enqueue then writes the lower triangle of the matrix.
int32_t gram_finish_enqueue(gingr_ctx* ctx, GramPlan& plan, const double* d_partial, const double* d_sqrt_lambda,
                            double add_identity, int L, const double* d_lm_rows, const double* d_lm_A, int ld_out,
                            double* d_out, bool packed = false, bool lower_only = false, bool rhs_row = false);
// lower_only: the strict upper triangle is not written (the Cholesky factorisation reads the lower one only; the mirror
// is a column-wise write that costs as much as the rest of the kernel)
size_t gram_packed_doubles(const GramPlan& plan);
int32_t gram_unpack_enqueue(gingr_ctx* ctx, GramPlan& plan, const double* d_packed, int ld_out, double* d_out,
                            bool rhs_row = false);

// ---- chol.cu -------------------------------------------------------------------------------------
// In-place blocked Cholesky A = L L^T of the leading n x n block (lower triangle, row-major, pitch ld) of a
// matrix with nrows >= n rows.  The extra rows i >= n are carried through the panel solves, so on return
// row n + q holds  L^-1 b_q  for the right-hand side b_q that was stored there (forward substitution for free).
// d_info[0] is set to 1 if a non-positive / non-finite pivot appears (matrix not SPD).
// Workspace of the data-flow factorisation (chol_df.cu): tile tickets / flags and the inverses of the diagonal blocks.
// One per concurrent factorisation (a registration owns one); alloc() outside stream capture.
struct CholWs {
  DevBuf<int> sync, bsync;   // factorisation tickets / flags; flags of the back substitution
  DevBuf<double> linv;
  int cap_n = 0, cap_nrows = 0;
  int32_t alloc(gingr_ctx* ctx, int n, int nrows);
};
// ws == nullptr (or GINGR_CHOL_DF=0): the kernel-per-step form of chol.cu; else one persistent data-flow kernel.
int32_t cholesky_enqueue(gingr_ctx* ctx, int n, int nrows, double* d_A, int ld, int* d_info, CholWs* ws = nullptr);
int32_t cholesky_df_enqueue(gingr_ctx* ctx, int n, int nrows, double* d_A, int ld, int* d_info, CholWs& ws);
// c = L^-T z  (sync-free multi-CTA backward substitution).  d_flags: >= ceil(n/64) ints of scratch.
// ws (optional): the workspace the factor was computed with by the data-flow kernel -- the back substitution then uses
// the published inverses of the diagonal blocks (chol_df.cu); GINGR_CHOL_DF=0 or ws == nullptr: chol.cu's kernel.
int32_t chol_backsolve_enqueue(gingr_ctx* ctx, int n, const double* d_L, int ld, const double* d_z, double* d_c,
                               int* d_flags, CholWs* ws = nullptr);
int32_t chol_backsolve_z_enqueue(gingr_ctx* ctx, int n, const double* d_L, int ld, const double* d_z, double* d_c, CholWs& ws);

// ---- basis_rotate.cu -----------------------------------------------------------------------------
// out[3i + d][j] = scale[j] * sum_e R[d][e] (Phi U)[3i + e][j]  on DMMA: Phi, out [rows][rp], U [rp][rp] (all row-major,
// zero padded), scale [rp], d_R: 9 doubles (row-major rotation) on the device.  rows a multiple of 3, rp of 8.
int32_t basis_rotate_enqueue(gingr_ctx* ctx, int rows, int rp, const double* d_phi, const double* d_U, const double* d_scale,
                             const double* d_R, double* d_out);

// ---- vecops.cu -----------------------------------------------------------------------------------
// out_q[k] = sum_a phi[k][a] v_q[a],  q < nvec (1 or 2), k < rows
// d_scale (optional): the vectors are multiplied elementwise by it while they are staged (instance(alpha) = Phi (sqrt(lambda) alpha))
int32_t gemv_rows_enqueue(gingr_ctx* ctx, int rows, int r, int rp, const double* d_phi, int nvec, const double* d_v0,
                          const double* d_v1, double* d_out0, double* d_out1, const double* d_scale = nullptr);
// out[a] = scale[a] * sum_k phi[k][a] u[k]   (scale may be null).  d_part: >= gemvT_splits(ctx, rows) * rp doubles
int gemvT_splits(const gingr_ctx* ctx, int rows);
int32_t gemvT_enqueue(gingr_ctx* ctx, int rows, int r, int rp, const double* d_phi, const double* d_u,
                      const double* d_scale, double* d_part, double* d_out);
// y[a] = sum_b A[a][b] x[b]  for a dense r x r row-major matrix (pitch ld)
// d_flag_in / d_flag_out (optional): set to 1 when x / y holds a non-finite value
int32_t dense_matvec_enqueue(gingr_ctx* ctx, int r, const double* d_A, int ld, const double* d_x, double* d_y,
                             int* d_flag_in = nullptr, int* d_flag_out = nullptr);
// B[c][r] = A[r][c]  (n x n, pitches lda / ldb)
int32_t transpose_enqueue(gingr_ctx* ctx, int n, const double* d_A, int lda, double* d_B, int ldb);

// dst[k * ld_dst + j] = tmp[j * rows + k]  (column slab [nc][rows] -> row-major rows of Phi)
int32_t slab_transpose_enqueue(gingr_ctx* ctx, int rows, int nc, const double* d_tmp, double* d_dst, int ld_dst);
// B = [eps I + S ; I]  ((2r) x r, pitch rp)
int32_t build_regression_system_enqueue(gingr_ctx* ctx, int r, int rp, const double* d_S, double eps, double* d_B);
int32_t add_vectors_enqueue(gingr_ctx* ctx, int n, const double* d_a, const double* d_b, double* d_out);

}  // namespace gingr
