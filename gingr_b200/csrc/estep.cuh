// estep.cuh -- host-side interface of the K1 E-step kernels (estep.cu).
#pragma once
#include "common.cuh"

namespace gingr {

struct EstepPlan {
  int col_blocks = 0, row_splits = 0;  // sweep A grid
  int row_blocks = 0, col_splits = 0;  // sweep B grid
  int den_blocks = 0;
};

struct EstepWorkspace {
  EstepPlan plan;
  DevBuf<double> colpart;   // [row_splits][N]
  DevBuf<double> pack;      // [N][8]
  DevBuf<double> pt1;       // [N]      Pt1 (CPD) / nu' (BCPD)
  DevBuf<double> xpx_part;  // [den_blocks] partial sums of Pt1_j |x_j|^2
  DevBuf<double> rowpart;   // [col_splits][4][M]
  DevBuf<double> rows;      // [4][M]   P1, PX.x, PX.y, PX.z
  DevBuf<double> fit_soa;   // [3][M]
  DevBuf<double> rowf;      // [M]      BCPD row factors
  DevBuf<double> scal;      // [16]     0 sigma2, 1 a, 2 c, 3 w, 4 M/N, 5 s, 6 1/N
  int32_t ensure(gingr_ctx* ctx, int M, int N);
};

void estep_plan(const gingr_ctx* ctx, int M, int N, EstepPlan* p);
struct EstepEvents {
  cudaEvent_t a0, a1, b0, b1;  // around the sweep A and sweep B kernels
};
int32_t estep_enqueue(gingr_ctx* ctx, EstepWorkspace& ws, int M, int N, const double* target_soa, bool use_rowf,
                      const EstepEvents* ev = nullptr);
int32_t validate_finite_enqueue(gingr_ctx* ctx, int n, const double* d_v, int* d_flag);
int32_t aos_to_soa_enqueue(gingr_ctx* ctx, int n, const double* d_aos, double* d_soa);
int32_t estep_cpd_scalars_enqueue(gingr_ctx* ctx, double* d_scal);
int32_t estep_bcpd_rowf_enqueue(gingr_ctx* ctx, int M, const double* d_sigma_mm, const double* d_alpha,
                                double* d_scal, double* d_rowf);

int32_t initial_sigma2_enqueue(gingr_ctx* ctx, int M, const double* d_pts_aos, int N, const double* d_target_soa,
                               double* d_out);

}  // namespace gingr
