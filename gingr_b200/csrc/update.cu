// update.cu -- the full GiNGR iteration on the device: GingrAlgorithm.update (api/GingrAlgorithm.scala:192-254)
// with computePosterior (:281-302), the CPD / ICP plugin functions (registration/config/CPD.scala:32-49,
// :120-147; ICP.scala:37-51, :90-99), the rigid / similarity extraction (:260-279) and the fit refresh of
// GingrGeneratorWrapper.propose (sampling/generators/GingrGeneratorWrapper.scala:28-39).
//
// One call enqueues a fixed sequence of kernels on the ctx stream; every scalar the kernels need (pose,
// sigma2, status flags) lives in a small device-resident state block, so iterations can be chained without
// host round trips (gingr_update_chain).  Data flow of one iteration (SURVEY.md 3.2 / 3.3):
//
//   pose_kernel            R = Rz(phi) Ry(theta) Rx(psi) from the Euler angles of the state
//   [CPD] E-step (estep.cu) on this rank's target shard  -> P1, PX, Pt1 ; all-reduce over ranks
//   [ICP] closest point (closest.cu)                     -> cp, 0/1 weights
//   obs_kernel             correspondence point, observation weight 1/var, residual u = w R^T (y - m'),
//                          per-row weights; sums for the sigma2 update (pre-update fit, CPD.scala:133-147)
//   gemvT                  rhs = D Phi^T u                         (Q^T L^-1 (y - m))
//   gram (DMMA) + finish   Mx = I + D Phi^T W Phi D (+ landmark blocks) ; all-reduce over ranks
//   cholesky (+ rhs row)   z = L^-1 rhs ; backsolve c = L^-T z     (posterior mean coefficients)
//   shrink                 alpha* = W0 (S c)   == transformedModelInit.coefficients(posterior.mean) (:214-216)
//   combine                alpha_c = alpha + (alpha* - alpha) stepLength                          (:218-220)
//   gemv_rows x2           instance(alpha) and instance(alpha_c) at the mesh points               (:222-224)
//   procrustes             Umeyama about the origin, Euler round trips                             (:227-231)
//   gemvT + W0             alpha_new = transformedModel.coefficients(newshape)                    (:234-237)
//   finalize               new state or ModelFlexibilityError, sigma2 hook                        (:239-251)
//   gemv_rows + pose       fit = s (R instance(alpha_new) + t)            (ModelFittingParameters.scala:130-143)
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "closest.cuh"
#include "batch.cuh"
#include "estep.cuh"
#include "grid.cuh"
#include "nccl_dl.cuh"
#include "posterior.cuh"

namespace gingr {

// ---- device state block layout (doubles) ---------------------------------------------------------
enum {
  DS_SCALE = 0, DS_T = 1, DS_EULER = 4, DS_CENTER = 7, DS_SIGMA2 = 10, DS_STEP = 11, DS_R = 12,
  DS_NEW_SCALE = 24, DS_NEW_T = 25, DS_NEW_EULER = 28, DS_R1 = 31, DS_R2 = 40,
  DS_NEW_SIGMA2 = 50, DS_NP = 51, DS_XPX = 52, DS_YPY = 53, DS_TRPXY = 54,
  DS_MUX = 56, DS_MUY = 59, DS_S2X = 62, DS_SXY = 63, DS_COUNT = 80
};
enum { IS_GT = 0, IS_ITER = 1, IS_STATUS = 2, IS_INFO = 3, IS_FAIL_POST = 4, IS_FAIL_COEF = 5, IS_RETRY = 6, IS_COUNT = 16 };
constexpr int RETRY_COUNTER_INIT = 10;  // GingrAlgorithm.scala:69-70

__device__ __forceinline__ void euler_to_matrix_dev(double phi, double theta, double psi, double* R) {
  const double cph = cos(phi), sph = sin(phi), cth = cos(theta), sth = sin(theta), cps = cos(psi), sps = sin(psi);
  R[0] = cth * cph; R[1] = sps * sth * cph - cps * sph; R[2] = sps * sph + cps * sth * cph;
  R[3] = cth * sph; R[4] = cps * cph + sps * sth * sph; R[5] = cps * sth * sph - sps * cph;
  R[6] = -sth;      R[7] = sps * cth;                   R[8] = cps * cth;
}

// RotationSpace3D.rotMatrixToEulerAngles (Slabaugh), SURVEY.md A4
__device__ __forceinline__ void matrix_to_euler_dev(const double* R, double* e) {
  if (fabs(fabs(R[6]) - 1.0) > 0.0001) {
    const double theta = asin(-R[6]);
    const double ct = cos(theta);
    e[0] = atan2(R[3] / ct, R[0] / ct);
    e[1] = theta;
    e[2] = atan2(R[7] / ct, R[8] / ct);
  } else if (fabs(R[6] + 1.0) < 0.0001) {
    e[0] = 0.0; e[1] = 3.14159265358979323846 / 2.0; e[2] = atan2(R[1], R[2]);
  } else {
    e[0] = 0.0; e[1] = -3.14159265358979323846 / 2.0; e[2] = atan2(-R[1], -R[2]);
  }
}

GINGR_KERNEL_NB(pose_kernel, double* ds, int* is) {
  euler_to_matrix_dev(ds[DS_EULER], ds[DS_EULER + 1], ds[DS_EULER + 2], ds + DS_R);
  is[IS_INFO] = 0;
  is[IS_FAIL_POST] = 0;
  is[IS_FAIL_COEF] = 0;
}

// fit_i = s (R (ref_i + mean_i + a_i) + t)  for the local point range [m0, m0 + Ml); a: [3 Ml] local.
// pose offsets select which (scale, t, R) of the state block to use.
GINGR_KERNEL_NB(fit_from_instance_kernel, int m0, int Ml, const double* __restrict__ ref, const double* __restrict__ mean,
                                         const double* __restrict__ a, const double* __restrict__ ds, int off_s,
                                         int off_t, int off_R, double* __restrict__ out /*[3 Ml] local*/) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Ml) return;
  const int gi = m0 + i;
  const double* R = ds + off_R;
  const double s = ds[off_s];
  const double x = ref[3 * gi] + mean[3 * gi] + a[3 * i];
  const double y = ref[3 * gi + 1] + mean[3 * gi + 1] + a[3 * i + 1];
  const double z = ref[3 * gi + 2] + mean[3 * gi + 2] + a[3 * i + 2];
  out[3 * i] = (R[0] * x + R[1] * y + R[2] * z + ds[off_t]) * s;
  out[3 * i + 1] = (R[3] * x + R[4] * y + R[5] * z + ds[off_t + 1]) * s;
  out[3 * i + 2] = (R[6] * x + R[7] * y + R[8] * z + ds[off_t + 2]) * s;
}

// v[a] = sqrt_lambda[a] * alpha[a]
GINGR_KERNEL_NB(scale_vec_kernel, int r, const double* __restrict__ sl, const double* __restrict__ alpha,
                                 double* __restrict__ out) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a < r) out[a] = sl[a] * alpha[a];
}

// gather padded all-gather blocks [nranks][3 Mmax] into fit [3 M]
__global__ void compact_gather_kernel(int M, int nranks, int Mmax, const double* __restrict__ gathered,
                                      double* __restrict__ fit) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= 3 * M) return;
  const int i = e / 3, d = e % 3;
  const int base = M / nranks, rem = M % nranks;
  // rank owning point i
  int rk, start;
  if (i < rem * (base + 1)) { rk = i / (base + 1); start = rk * (base + 1); }
  else { rk = rem + (i - rem * (base + 1)) / max(base, 1); start = rem * (base + 1) + (rk - rem) * base; }
  fit[e] = gathered[(size_t)rk * 3 * Mmax + 3 * (i - start) + d];
}

// ---- CPD: fit and scalars for the E-step from the state block ----------------------------------
// What the CPD E-step needs from the fit, in one pass and one launch (were four: two finite checks, the AoS -> SoA copy and a
// one-block reduction): fit_soa (row i of it is point perm[i], the E-step's k-d order), the failure flag for a non-finite fit / sigma2, and -- by the last block to finish, which
// also resets the two words of `sync` for the next launch -- the scalars: scal[0] = sigma2, scal[1] = a = 1, scal[2] = c
// (CPD.scala:69-70), scal[7] = bound of the pair distances from max |coordinate| of fit and target (gauss_exp2_tab<SAFE>).
// The maximum is exact in any order, so the result does not depend on which block comes last.
GINGR_KERNEL((256), cpd_prepare_kernel, int M, const double* __restrict__ fit /*AoS*/, const int* __restrict__ perm,
                                                          double* __restrict__ fit_soa,
                                                          const double* __restrict__ ds, double w, double ratio,
                                                          double target_maxabs, int* __restrict__ fail_flag,
                                                          unsigned long long* __restrict__ sync /*[2]: max bits, ticket*/,
                                                          double* __restrict__ scal) {
  __shared__ double red[8];
  const int i = blockIdx.x * 256 + threadIdx.x;
  double m = 0.0;
  int bad = 0;
  if (i < M) {
    const size_t p = 3 * (size_t)perm[i];
    const double x = fit[p], y = fit[p + 1], z = fit[p + 2];
    fit_soa[i] = x; fit_soa[M + i] = y; fit_soa[2 * (size_t)M + i] = z;
    bad = !(fabs(x) < INFINITY) || !(fabs(y) < INFINITY) || !(fabs(z) < INFINITY);
    m = fmax(fmax(fabs(x), fabs(y)), fabs(z));
  }
  bad = __syncthreads_or(bad);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (int k = 1; k < 8; ++k) m = fmax(m, red[k]);
  if (bad) *fail_flag = 1;
  atomicMax(sync, (unsigned long long)__double_as_longlong(m));   // non-negative doubles order like their bit patterns
  __threadfence();
  if (atomicAdd(sync + 1, 1ULL) != (unsigned long long)gridDim.x - 1) return;
  __threadfence();
  const double fmaxabs = __longlong_as_double((long long)atomicExch(sync, 0ULL));
  sync[1] = 0ULL;
  const double sigma2 = ds[DS_SIGMA2];
  if (!(fabs(sigma2) < INFINITY)) *fail_flag = 1;
  const double t = 2.0 * 3.14159265358979323846 * sigma2;
  scal[0] = sigma2;
  scal[1] = 1.0;
  scal[2] = w / (1.0 - w) * (t * sqrt(t)) * ratio;  // CPD.scala:69-70
  const double s2 = fmaxabs + target_maxabs;
  scal[7] = 3.0 * s2 * s2;
}

// xpx total (fixed order) appended behind the row block for the all-reduce.  One CTA of 256 threads.
GINGR_KERNEL_NB(xpx_total_kernel, int nparts, const double* __restrict__ parts, double* __restrict__ out) {
  __shared__ double red[256];
  double s = 0.0;
  for (int k = threadIdx.x; k < nparts; k += 256) s += parts[k];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}

// ---- observations ---------------------------------------------------------------------------------
// CPD (CPD.scala:32-49, :120-128): point PX_i / P1_i, variance sigma2 * lambda / P1_i.
// ICP (ICP.scala:37-51, :90-92):  point cp_i (kept only if w_i == 1), variance sigma2.
// Output for local points [m0, m0 + Ml): wrow[3 Ml], u[3 Ml] = w R^T (y - (R (ref + mean) + t)).
// Sums for CPD's sigma2 update over ALL points (every rank computes the same): per-block partials of
// P1, P1 |fit|^2, fit . PX.
struct ObsArgs {
  int algo, M, m0, Ml, use_lm, L;
  double lambda;
};

GINGR_KERNEL((256), obs_kernel, const ObsArgs& a, const double* __restrict__ rows /*[4][M] CPD*/,
                                                  const double* __restrict__ cp /*[M][3] ICP*/,
                                                  const uint8_t* __restrict__ w01,
                                                  const double* __restrict__ wcnt /*reversed ICP, else null*/,
                                                  const double* __restrict__ fit,
                                                  const double* __restrict__ ref, const double* __restrict__ mean,
                                                  const int32_t* __restrict__ lm_pid, const double* __restrict__ ds,
                                                  int* __restrict__ is, double* __restrict__ wrow,
                                                  double* __restrict__ u, double* __restrict__ sums_part /*[blocks][3]*/,
                                                  double* __restrict__ resid /*[3 Ml] unweighted R^T residual, may be null*/) {
  __shared__ double red[3][8];
  const int i = blockIdx.x * 256 + threadIdx.x;
  double sP1 = 0.0, sY = 0.0, sT = 0.0;
  if (i < a.M) {
    const double sigma2 = ds[DS_SIGMA2];
    double px, py, pz, wt;
    if (a.algo == GINGR_ALGO_CPD) {
      const double p1 = rows[i];
      const double X = rows[(size_t)a.M + i], Y = rows[(size_t)2 * a.M + i], Z = rows[(size_t)3 * a.M + i];
      const double inv = 1.0 / p1;
      px = X * inv; py = Y * inv; pz = Z * inv;
      const double var = sigma2 * a.lambda * inv;  // eye(3) * sigma2 * lambda * P1inv(id)  CPD.scala:125
      wt = 1.0 / var;
      if (!(var < INFINITY) || !(var > 0.0) || !(wt < INFINITY)) is[IS_FAIL_POST] = 1;  // breeze inv(cov) not finite
      const double fx = fit[3 * i], fy = fit[3 * i + 1], fz = fit[3 * i + 2];
      sP1 = p1;
      sY = p1 * (fx * fx + fy * fy + fz * fz);
      sT = fx * X + fy * Y + fz * Z;
    } else {
      px = cp[3 * i]; py = cp[3 * i + 1]; pz = cp[3 * i + 2];
      // pairs with w != 1 are dropped (ICP.scala:50); reversed direction: cnt observations of this vertex, cp = their mean
      const double cnt = wcnt ? wcnt[i] : (w01[i] ? 1.0 : 0.0);
      wt = cnt > 0.0 ? cnt / sigma2 : 0.0;
      if (cnt > 0.0 && (!(wt < INFINITY) || !(wt > 0.0))) is[IS_FAIL_POST] = 1;
    }
    if (a.use_lm)
      for (int l = 0; l < a.L; ++l)
        if (lm_pid[l] == i) wt = 0.0;  // correspondences at landmark ids are replaced (GingrAlgorithm.scala:288-296)
    const int li = i - a.m0;
    if (li >= 0 && li < a.Ml) {
      const double* R = ds + DS_R;
      const double bx = ref[3 * i] + mean[3 * i], by = ref[3 * i + 1] + mean[3 * i + 1], bz = ref[3 * i + 2] + mean[3 * i + 2];
      double rx = px - (R[0] * bx + R[1] * by + R[2] * bz + ds[DS_T]);
      double ry = py - (R[3] * bx + R[4] * by + R[5] * bz + ds[DS_T + 1]);
      double rz = pz - (R[6] * bx + R[7] * by + R[8] * bz + ds[DS_T + 2]);
      if (wt == 0.0) { rx = ry = rz = 0.0; }  // dropped observation: contributes nothing (and no 0 * NaN)
      wrow[3 * li] = wrow[3 * li + 1] = wrow[3 * li + 2] = wt;
      const double q0 = R[0] * rx + R[3] * ry + R[6] * rz, q1 = R[1] * rx + R[4] * ry + R[7] * rz,
                   q2 = R[2] * rx + R[5] * ry + R[8] * rz;
      u[3 * li] = wt * q0;
      u[3 * li + 1] = wt * q1;
      u[3 * li + 2] = wt * q2;
      if (resid) { resid[3 * li] = q0; resid[3 * li + 1] = q1; resid[3 * li + 2] = q2; }   // the Gram applies the weight itself
    }
  }
  // block sums (fixed order)
  double v[3] = {sP1, sY, sT};
#pragma unroll
  for (int q = 0; q < 3; ++q) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_down_sync(0xffffffffu, v[q], o);
    if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = v[q];
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    for (int k = 0; k < 8; ++k) s += red[threadIdx.x][k];
    sums_part[blockIdx.x * 3 + threadIdx.x] = s;
  }
}

// sigma2 hook: CPD (xPx - 2 trPXY + yPy) / (3 Np) (CPD.scala:133-147); ICP linear anneal (ICP.scala:96-99)
GINGR_KERNEL_NB(sigma2_kernel, int algo, int nblocks, const double* __restrict__ sums_part, const double* __restrict__ xpx,
                              double sigma_step, double end_sigma, double* __restrict__ ds) {
  // one warp: lane l adds the block partials l, l + 32, ... in order, then a fixed shuffle tree (deterministic)
  const int lane = threadIdx.x;
  if (algo == GINGR_ALGO_CPD) {
    double np = 0.0, ypy = 0.0, tr = 0.0;
    for (int k = lane; k < nblocks; k += 32) {
      np += sums_part[3 * k];
      ypy += sums_part[3 * k + 1];
      tr += sums_part[3 * k + 2];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      np += __shfl_xor_sync(0xffffffffu, np, o);
      ypy += __shfl_xor_sync(0xffffffffu, ypy, o);
      tr += __shfl_xor_sync(0xffffffffu, tr, o);
    }
    if (lane == 0) {
      ds[DS_NP] = np; ds[DS_XPX] = xpx[0]; ds[DS_YPY] = ypy; ds[DS_TRPXY] = tr;
      ds[DS_NEW_SIGMA2] = (xpx[0] - 2.0 * tr + ypy) / (np * 3.0);
    }
  } else if (lane == 0) {
    ds[DS_NEW_SIGMA2] = fmax(ds[DS_SIGMA2] - sigma_step, end_sigma);
  }
}

// ---- landmarks ------------------------------------------------------------------------------------
// A_l = R^T C_l^-1 R ; rhs += D Phi_l^T A_l R^T (y_l - (R (ref + mean)_pid + t))   for local landmarks
GINGR_KERNEL_NB(landmark_prepare_kernel, int L, const double* __restrict__ cinv, const double* __restrict__ ds,
                                        double* __restrict__ A) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L) return;
  const double* R = ds + DS_R;
  const double* C = cinv + 9 * l;
  double T[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) T[3 * i + j] = C[3 * i] * R[j] + C[3 * i + 1] * R[3 + j] + C[3 * i + 2] * R[6 + j];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) A[9 * l + 3 * i + j] = R[i] * T[j] + R[3 + i] * T[3 + j] + R[6 + i] * T[6 + j];
}

GINGR_KERNEL_NB(landmark_rhs_kernel, int r, int rp, int L, const int32_t* __restrict__ pid,
                                    const double* __restrict__ pts, const double* __restrict__ A,
                                    const double* __restrict__ lm_rows, const double* __restrict__ ref,
                                    const double* __restrict__ mean, const double* __restrict__ sl,
                                    const double* __restrict__ ds, double* __restrict__ rhs) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= r) return;
  const double* R = ds + DS_R;
  double s = 0.0;
  for (int l = 0; l < L; ++l) {
    const int p = pid[l];
    const double bx = ref[3 * p] + mean[3 * p], by = ref[3 * p + 1] + mean[3 * p + 1], bz = ref[3 * p + 2] + mean[3 * p + 2];
    const double rx = pts[3 * l] - (R[0] * bx + R[1] * by + R[2] * bz + ds[DS_T]);
    const double ry = pts[3 * l + 1] - (R[3] * bx + R[4] * by + R[5] * bz + ds[DS_T + 1]);
    const double rz = pts[3 * l + 2] - (R[6] * bx + R[7] * by + R[8] * bz + ds[DS_T + 2]);
    const double qx = R[0] * rx + R[3] * ry + R[6] * rz, qy = R[1] * rx + R[4] * ry + R[7] * rz,
                 qz = R[2] * rx + R[5] * ry + R[8] * rz;
    const double* Al = A + 9 * l;
    const double vx = Al[0] * qx + Al[1] * qy + Al[2] * qz, vy = Al[3] * qx + Al[4] * qy + Al[5] * qz,
                 vz = Al[6] * qx + Al[7] * qy + Al[8] * qz;
    const double* pr = lm_rows + (size_t)l * 3 * rp;
    s += pr[a] * vx + pr[rp + a] * vy + pr[2 * rp + a] * vz;
  }
  rhs[a] += sl[a] * s;
}

// gather the 3 basis rows of each landmark vertex: lm_rows [L][3][rp]
GINGR_KERNEL_NB(gather_rows_kernel, int L, int rp, int m0, const int32_t* __restrict__ pid, const double* __restrict__ phi,
                                   double* __restrict__ out) {
  const int l = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= 3 * rp) return;
  const int d = e / rp, a = e % rp;
  out[(size_t)l * 3 * rp + e] = phi[((size_t)3 * (pid[l] - m0) + d) * rp + a];
}

// ---- posterior sampling -----------------------------------------------------------------------------
// posterior.sample() (GingrAlgorithm.scala:211; scalismo: mean + Phi' U_s (sqrt(s) z), SURVEY.md A3) draws the
// coefficients from N(c, Minv).  With Mx = L L^T the same distribution is  c + L^-T z = L^-T (L^-1 rhs + z):
// z is added to the forward-substituted right-hand side before the back solve.  (scalismo rotates the basis with
// an SVD and uses its own RNG stream, so the individual draws differ; the distribution is identical.)
// z comes from Philox4x32-10 keyed by the caller's seed, counter = (pair index, iteration, 0, 0), and Box-Muller in
// FP64 -- a counter-based stream that any host (the oracle, the JVM) can reproduce.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t* out) {
#pragma unroll
  for (int round = 0; round < 10; ++round) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

GINGR_KERNEL_NB(add_normal_kernel, int r, uint64_t seed, const int* __restrict__ counter, double* __restrict__ y) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;  // pair index: entries 2p, 2p + 1
  if (2 * p >= r) return;
  uint32_t x[4];
  philox4x32_10((uint32_t)p, (uint32_t)counter[0], 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), x);
  const double u1 = ((double)(x[0] >> 5) * 67108864.0 + (double)(x[1] >> 6) + 0.5) * (1.0 / 9007199254740992.0);
  const double u2 = ((double)(x[2] >> 5) * 67108864.0 + (double)(x[3] >> 6) + 0.5) * (1.0 / 9007199254740992.0);
  const double rad = sqrt(-2.0 * log(u1));
  const double ang = 6.283185307179586476925 * u2;
  y[2 * p] += rad * cos(ang);
  if (2 * p + 1 < r) y[2 * p + 1] += rad * sin(ang);
}

// ---- small vector kernels -------------------------------------------------------------------------
GINGR_KERNEL_NB(check_finite_kernel, int n, const double* __restrict__ v, int* __restrict__ flag) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a < n && !(fabs(v[a]) < INFINITY)) *flag = 1;
}

// alpha_c = alpha + (alpha* - alpha) * stepLength   (GingrAlgorithm.scala:218-220)
GINGR_KERNEL_NB(combine_kernel, int r, const double* __restrict__ alpha, const double* __restrict__ astar,
                               const double* __restrict__ ds, double* __restrict__ out) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a < r) out[a] = alpha[a] + (astar[a] - alpha[a]) * ds[DS_STEP];
}

// X_i = ref + mean + a (currentFitNoTransform, :224), Y_i = R (ref + mean + b) + t (newshape, :222), local points.
// pass 0: partial sums of X and Y ; pass 1: centred sums |X - mux|^2 and (Y - muy)(X - mux)^T.
GINGR_KERNEL((256), procrustes_sums_kernel, int pass, int m0, int Ml, const double* __restrict__ ref,
                                                              const double* __restrict__ mean,
                                                              const double* __restrict__ a, const double* __restrict__ b,
                                                              const double* __restrict__ ds,
                                                              double* __restrict__ newshape /*[3 Ml]*/,
                                                              double* __restrict__ part /*[blocks][16]*/) {
  __shared__ double red[16][8];
  const int i = blockIdx.x * 256 + threadIdx.x;
  double v[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) v[q] = 0.0;
  if (i < Ml) {
    const int gi = m0 + i;
    const double* R = ds + DS_R;
    const double cx = ref[3 * gi] + mean[3 * gi], cy = ref[3 * gi + 1] + mean[3 * gi + 1], cz = ref[3 * gi + 2] + mean[3 * gi + 2];
    const double X0 = cx + a[3 * i], X1 = cy + a[3 * i + 1], X2 = cz + a[3 * i + 2];
    const double bx = cx + b[3 * i], by = cy + b[3 * i + 1], bz = cz + b[3 * i + 2];
    const double Y0 = R[0] * bx + R[1] * by + R[2] * bz + ds[DS_T];
    const double Y1 = R[3] * bx + R[4] * by + R[5] * bz + ds[DS_T + 1];
    const double Y2 = R[6] * bx + R[7] * by + R[8] * bz + ds[DS_T + 2];
    if (pass == 0) {
      newshape[3 * i] = Y0; newshape[3 * i + 1] = Y1; newshape[3 * i + 2] = Y2;
      v[0] = X0; v[1] = X1; v[2] = X2; v[3] = Y0; v[4] = Y1; v[5] = Y2;
    } else if (pass == 2) {
      // several ranks: ONE pass and one all-reduce.  Moments about fixed points every rank knows -- p0 = (ref + mean) of
      // vertex 0 for x, its posed image q0 = R p0 + t for y -- so that centring them afterwards cancels nothing that
      // matters (the shifted coordinates are of the size of the shape, wherever it sits).
      newshape[3 * i] = Y0; newshape[3 * i + 1] = Y1; newshape[3 * i + 2] = Y2;
      const double p0x = ref[0] + mean[0], p0y = ref[1] + mean[1], p0z = ref[2] + mean[2];
      const double x0 = X0 - p0x, x1 = X1 - p0y, x2 = X2 - p0z;
      const double y0 = Y0 - (R[0] * p0x + R[1] * p0y + R[2] * p0z + ds[DS_T]);
      const double y1 = Y1 - (R[3] * p0x + R[4] * p0y + R[5] * p0z + ds[DS_T + 1]);
      const double y2 = Y2 - (R[6] * p0x + R[7] * p0y + R[8] * p0z + ds[DS_T + 2]);
      v[0] = x0 * x0 + x1 * x1 + x2 * x2;
      v[1] = y0 * x0; v[2] = y0 * x1; v[3] = y0 * x2;
      v[4] = y1 * x0; v[5] = y1 * x1; v[6] = y1 * x2;
      v[7] = y2 * x0; v[8] = y2 * x1; v[9] = y2 * x2;
      v[10] = x0; v[11] = x1; v[12] = x2; v[13] = y0; v[14] = y1; v[15] = y2;
    } else {
      const double x0 = X0 - ds[DS_MUX], x1 = X1 - ds[DS_MUX + 1], x2 = X2 - ds[DS_MUX + 2];
      const double y0 = Y0 - ds[DS_MUY], y1 = Y1 - ds[DS_MUY + 1], y2 = Y2 - ds[DS_MUY + 2];
      v[0] = x0 * x0 + x1 * x1 + x2 * x2;
      v[1] = y0 * x0; v[2] = y0 * x1; v[3] = y0 * x2;
      v[4] = y1 * x0; v[5] = y1 * x1; v[6] = y1 * x2;
      v[7] = y2 * x0; v[8] = y2 * x1; v[9] = y2 * x2;
    }
  }
#pragma unroll
  for (int q = 0; q < 16; ++q) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_down_sync(0xffffffffu, v[q], o);
    if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = v[q];
  }
  __syncthreads();
  if (threadIdx.x < 16) {
    double s = 0.0;
    for (int k = 0; k < 8; ++k) s += red[threadIdx.x][k];
    part[blockIdx.x * 16 + threadIdx.x] = s;
  }
}

GINGR_KERNEL_NB(procrustes_reduce_kernel, int nblocks, int count, const double* __restrict__ part,
                                         double* __restrict__ out /*[16]*/) {
  const int q = threadIdx.x;
  if (q >= count) return;
  double s = 0.0;
  for (int k = 0; k < nblocks; ++k) s += part[k * 16 + q];
  out[q] = s;
}

GINGR_KERNEL_NB(procrustes_means_kernel, int M, const double* __restrict__ sums, double* __restrict__ ds) {
  for (int d = 0; d < 3; ++d) {
    ds[DS_MUX + d] = sums[d] / M;
    ds[DS_MUY + d] = sums[3 + d] / M;
  }
}

// 3x3 SVD by one-sided Jacobi (Hestenes): A V = U diag(s), s sorted descending.
__device__ void svd3(const double* Ain, double* U, double* S, double* V) {
  double A[9], Vm[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  for (int i = 0; i < 9; ++i) A[i] = Ain[i];
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = 0.0;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        double alpha = 0, beta = 0, gamma = 0;
        for (int k = 0; k < 3; ++k) {
          alpha += A[3 * k + p] * A[3 * k + p];
          beta += A[3 * k + q] * A[3 * k + q];
          gamma += A[3 * k + p] * A[3 * k + q];
        }
        if (gamma == 0.0) continue;
        off = fmax(off, fabs(gamma) / sqrt(alpha * beta));
        const double zeta = (beta - alpha) / (2.0 * gamma);
        const double tt = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + tt * tt), s = c * tt;
        for (int k = 0; k < 3; ++k) {
          const double ap = A[3 * k + p], aq = A[3 * k + q];
          A[3 * k + p] = c * ap - s * aq;
          A[3 * k + q] = s * ap + c * aq;
          const double vp = Vm[3 * k + p], vq = Vm[3 * k + q];
          Vm[3 * k + p] = c * vp - s * vq;
          Vm[3 * k + q] = s * vp + c * vq;
        }
      }
    if (off < 2.3e-16) break;  // columns orthogonal to machine precision
  }
  double sv[3];
  for (int j = 0; j < 3; ++j) sv[j] = sqrt(A[j] * A[j] + A[3 + j] * A[3 + j] + A[6 + j] * A[6 + j]);
  int idx[3] = {0, 1, 2};
  for (int i = 0; i < 2; ++i)
    for (int j = i + 1; j < 3; ++j)
      if (sv[idx[j]] > sv[idx[i]]) { const int tmp = idx[i]; idx[i] = idx[j]; idx[j] = tmp; }
  for (int j = 0; j < 3; ++j) {
    const int c = idx[j];
    S[j] = sv[c];
    for (int k = 0; k < 3; ++k) {
      U[3 * k + j] = sv[c] > 0.0 ? A[3 * k + c] / sv[c] : 0.0;
      V[3 * k + j] = Vm[3 * k + c];
    }
  }
  // a zero singular value leaves a zero column in U: complete it to a right-handed orthonormal frame
  if (S[2] <= 0.0) {
    U[2] = U[3] * U[7] - U[6] * U[4];
    U[5] = U[6] * U[1] - U[0] * U[7];
    U[8] = U[0] * U[4] - U[3] * U[1];
  }
}

__device__ double det3(const double* A) {
  return A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) + A[2] * (A[3] * A[7] - A[4] * A[6]);
}

// Umeyama about the origin (LandmarkRegistration.{rigid,similarity}3DLandmarkRegistration, SURVEY.md A4;
// GingrAlgorithm.scala:227-231, :260-279) and the Euler round trips of the state update (:239-243,
// GeneralRegistrationState.scala:83-87).  sums: [0] sum |x - mux|^2, [1..9] sum (y - muy)(x - mux)^T
__device__ void procrustes_solve_dev(int M, const double* __restrict__ sums, double* __restrict__ ds,
                                     const int* __restrict__ is) {
  const int gt = is[IS_GT];
  double R1[9], t[3], c = 1.0;
  if (gt == GINGR_NO_TRANSFORMS) {
    for (int i = 0; i < 9; ++i) R1[i] = (i % 4 == 0) ? 1.0 : 0.0;
    t[0] = t[1] = t[2] = 0.0;
  } else {
    double Sxy[9], U[9], S[3], V[9], Rm[9];
    const double s2x = sums[0] / M;
    for (int i = 0; i < 9; ++i) Sxy[i] = sums[1 + i] / M;
    svd3(Sxy, U, S, V);
    const double sign = det3(Sxy) < 0.0 ? -1.0 : 1.0;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        Rm[3 * i + j] = U[3 * i] * V[3 * j] + U[3 * i + 1] * V[3 * j + 1] + sign * U[3 * i + 2] * V[3 * j + 2];
    if (gt == GINGR_SIMILARITY_TRANSFORMS) c = (S[0] + S[1] + sign * S[2]) / s2x;
    for (int i = 0; i < 3; ++i)
      t[i] = ds[DS_MUY + i] - c * (Rm[3 * i] * ds[DS_MUX] + Rm[3 * i + 1] * ds[DS_MUX + 1] + Rm[3 * i + 2] * ds[DS_MUX + 2]);
    double e[3];
    matrix_to_euler_dev(Rm, e);  // the registration result carries the rotation as Euler angles
    euler_to_matrix_dev(e[0], e[1], e[2], R1);
  }
  double e2[3];
  matrix_to_euler_dev(R1, e2);  // updateRotation(Rotation) -> Euler angles stored in the state
  ds[DS_NEW_SCALE] = c;
  for (int i = 0; i < 3; ++i) { ds[DS_NEW_T + i] = t[i]; ds[DS_NEW_EULER + i] = e2[i]; }
  for (int i = 0; i < 9; ++i) ds[DS_R1 + i] = R1[i];
  euler_to_matrix_dev(e2[0], e2[1], e2[2], ds + DS_R2);
}

GINGR_KERNEL_NB(procrustes_solve_kernel, int M, const double* __restrict__ sums, double* __restrict__ ds,
                                        const int* __restrict__ is) {
  procrustes_solve_dev(M, sums, ds, is);
}

// several ranks: the all-reduced shifted moments of the single pass (pass 2 of procrustes_sums_kernel) -> means and
// centred sums, then the same solve
GINGR_KERNEL_NB(procrustes_moments_solve_kernel, int M, double* __restrict__ sums /*[16]*/, const double* __restrict__ ref,
                                                const double* __restrict__ mean, double* __restrict__ ds,
                                                const int* __restrict__ is) {
  const double* R = ds + DS_R;
  const double p0[3] = {ref[0] + mean[0], ref[1] + mean[1], ref[2] + mean[2]};
  double mx[3], my[3];
  for (int d = 0; d < 3; ++d) {
    mx[d] = sums[10 + d] / M;
    my[d] = sums[13 + d] / M;
    ds[DS_MUX + d] = mx[d] + p0[d];
    ds[DS_MUY + d] = my[d] + (R[3 * d] * p0[0] + R[3 * d + 1] * p0[1] + R[3 * d + 2] * p0[2] + ds[DS_T + d]);
  }
  sums[0] -= M * (mx[0] * mx[0] + mx[1] * mx[1] + mx[2] * mx[2]);
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) sums[1 + 3 * a + b] -= M * my[a] * mx[b];
  procrustes_solve_dev(M, sums, ds, is);
}

// single rank: sum of the block partials (block order, as procrustes_reduce_kernel) followed by what consumes them:
// the means after pass 0, the rotation / translation / scale after pass 1
GINGR_KERNEL_NB(procrustes_reduce_then_kernel, int pass, int nblocks, int M, const double* __restrict__ part,
                                              double* __restrict__ sums /*[16]*/, double* __restrict__ ds,
                                              const int* __restrict__ is) {
  const int q = threadIdx.x;
  // lane l adds the blocks l, l + 32, ... of every quantity in order, then a fixed shuffle tree (deterministic)
  for (int c = 0; c < 10; ++c) {
    double s = 0.0;
    for (int k = q; k < nblocks; k += 32) s += part[k * 16 + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (q == 0) sums[c] = s;
  }
  __syncwarp();
  if (q != 0) return;
  if (pass == 0) {
    for (int d = 0; d < 3; ++d) {
      ds[DS_MUX + d] = sums[d] / M;
      ds[DS_MUY + d] = sums[3 + d] / M;
    }
  } else {
    procrustes_solve_dev(M, sums, ds, is);
  }
}

// u_i = R1^T (newshape_i - (R1 (ref + mean)_i + t_new))  for the second `coefficients` call (:234-237)
GINGR_KERNEL_NB(coeff_residual_kernel, int m0, int Ml, const double* __restrict__ newshape, const double* __restrict__ ref,
                                      const double* __restrict__ mean, const double* __restrict__ ds,
                                      double* __restrict__ u) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Ml) return;
  const int gi = m0 + i;
  const double* R = ds + DS_R1;
  const double bx = ref[3 * gi] + mean[3 * gi], by = ref[3 * gi + 1] + mean[3 * gi + 1], bz = ref[3 * gi + 2] + mean[3 * gi + 2];
  const double rx = newshape[3 * i] - (R[0] * bx + R[1] * by + R[2] * bz + ds[DS_NEW_T]);
  const double ry = newshape[3 * i + 1] - (R[3] * bx + R[4] * by + R[5] * bz + ds[DS_NEW_T + 1]);
  const double rz = newshape[3 * i + 2] - (R[6] * bx + R[7] * by + R[8] * bz + ds[DS_NEW_T + 2]);
  u[3 * i] = R[0] * rx + R[3] * ry + R[6] * rz;
  u[3 * i + 1] = R[1] * rx + R[4] * ry + R[7] * rz;
  u[3 * i + 2] = R[2] * rx + R[5] * ry + R[8] * rz;
}

// Commit the iteration (GingrAlgorithm.scala:193-208, :239-251): on success pose/scale/alpha/sigma2 are
// replaced; a failed posterior leaves the state unchanged (status ModelFlexibilityError if iteration > 0; in the
// probabilistic branch only once the retry counter of :69-70 has run out), a
// failed `coefficients` sets ModelFlexibilityError.  DS_R2 is left holding the rotation of the committed state.
GINGR_KERNEL_NB(finalize_kernel, int r, int probabilistic, const double* __restrict__ alpha_new, double* __restrict__ alpha,
                                double* __restrict__ ds, int* __restrict__ is) {
  __shared__ int mode;  // 0 commit, 1 keep
  if (threadIdx.x == 0) {
    const bool fail_post = is[IS_INFO] != 0 || is[IS_FAIL_POST] != 0;
    const bool fail_coef = is[IS_FAIL_COEF] != 0;
    if (fail_post) {
      if (is[IS_ITER] > 0) {
        if (probabilistic && is[IS_RETRY] != 0) is[IS_RETRY] -= 1;  // :197-202 retry: state returned unchanged
        else is[IS_STATUS] = GINGR_STATUS_MODEL_FLEXIBILITY_ERROR;
      }
      mode = 1;
    } else {
      is[IS_RETRY] = min(RETRY_COUNTER_INIT, is[IS_RETRY] + 1);  // :210
      if (fail_coef) {
        is[IS_STATUS] = GINGR_STATUS_MODEL_FLEXIBILITY_ERROR;
        mode = 1;
      } else {
        mode = 0;
        ds[DS_SCALE] = ds[DS_NEW_SCALE];
        for (int i = 0; i < 3; ++i) { ds[DS_T + i] = ds[DS_NEW_T + i]; ds[DS_EULER + i] = ds[DS_NEW_EULER + i]; }
        ds[DS_SIGMA2] = ds[DS_NEW_SIGMA2];
      }
    }
    if (mode == 1) euler_to_matrix_dev(ds[DS_EULER], ds[DS_EULER + 1], ds[DS_EULER + 2], ds + DS_R2);
  }
  __syncthreads();
  if (mode == 0)
    for (int a = threadIdx.x; a < r; a += blockDim.x) alpha[a] = alpha_new[a];
}

GINGR_KERNEL_NB(bump_iteration_kernel, int* is) { is[IS_ITER] += 1; }

GINGR_KERNEL_NB(set_iteration_kernel, int* is, int iteration, int status) {
  is[IS_ITER] = iteration;
  is[IS_STATUS] = status;
}

}  // namespace gingr

// =================================================================================================
// handles
// =================================================================================================
using namespace gingr;

struct gingr_registration {
  gingr_ctx* ctx = nullptr;
  const gingr_model* model = nullptr;
  const gingr_target* target = nullptr;
  gingr_config cfg;
  // landmarks (all, replicated) and the subset whose vertex lives in this rank's shard
  int L = 0, Ll = 0;
  DevBuf<int32_t> lm_pid;      // [L] all landmark vertex ids (for the correspondence filter)
  DevBuf<int32_t> lml_pid;     // [Ll] local
  DevBuf<double> lml_pts, lml_cinv, lml_A, lml_rows;
  // workspaces
  EstepWorkspace estep;
  ClosestWorkspace closest;
  GramPlan gram;
  DevBuf<double> fit_normals;  // [M][3] vertex normals of the current fit (ICP mesh flavours)
  DevBuf<double> fit_soa;      // [3][M] (reversed ICP: the fit is the mesh that is searched)
  SpatialGrid fit_pgrid, fit_tgrid;  // uniform grids over the moving fit, rebuilt every iteration (K2 at scale)
  bool use_fit_pgrid = false, use_fit_tgrid = false;
  DevBuf<int32_t> rev_tid;     // [N] reversed ICP: template vertex each target vertex maps back to
  DevBuf<double> rev_cp, rev_wcnt;  // [M][3], [M] folded observations of the reversed direction
  DevBuf<int32_t> rev_scratch;      // [3 M + N + 1] lists of the O(N + M) fold (large problems)
  DevBuf<double> rows_ext;     // [4 M + 8]  E-step rows + xPx (all-reduced together)
  DevBuf<double> Mx;           // [(r + 8)][rp]  posterior matrix + rhs row
  DevBuf<double> Mx_packed;    // several ranks: lower tiles of the partial posterior matrix + rhs, all-reduced as one buffer
  DevBuf<double> Mx_raw;       // [(r + 1)][rp]  copy of Mx and rhs before the factorisation (MCMC only, mcmc.cuh)
  bool keep_raw = false;
  bool skip_fit_refresh = false;        // MH step: the proposal's fit is evaluated after the random override
  const int* sample_counter = nullptr;  // device counter keyed into the posterior-sample stream (null: the iteration)
  std::unique_ptr<struct McmcState> mcmc;  // Metropolis-Hastings chain state (mcmc.cuh), created by gingr_mcmc_configure
  DevBuf<unsigned long long> prep_sync;   // [2] cpd_prepare_kernel: running maximum and block ticket (self-resetting)
  DevBuf<double> wrow, u, resid, inst_a, inst_b, newshape, fit_local, gathered, fit;
  DevBuf<double> vec;          // 8 * rp scratch vectors
  DevBuf<double> gt_part, sums_part, pro_part, pro_sums;
  DevBuf<double> ds;
  DevBuf<int> is, flags;
  CholWs cholws;               // tickets / flags / diagonal-block inverses of the data-flow Cholesky (chol_df.cu)
  DevBuf<double> alpha;
  int retry_counter = RETRY_COUNTER_INIT;  // mirror of the device counter, refreshed by download_state
  // One iteration captured as a CUDA graph: the ~100-launch sequence of a small registration (C1-C3 sizes) is
  // launch-latency bound, the graph replays it with one driver call.  Key = (probabilistic, seed).
  GraphExec graph_exec;
  int graph_prob = -1;
  uint64_t graph_seed = 0;
  int64_t graph_launches = 0;
  bool state_valid = false;        // the device holds a consistent state (pose, alpha, fit)
  bool host_mirror_current = false;  // ... and last_out / last_alpha are that state (false after device-resident chains)
  gingr_state last_out;
  std::vector<double> last_alpha;
  // profiling: per recorded iteration 14 events
  bool profiling = false;
  std::vector<cudaEvent_t> events;
  int prof_iters = 0;
  static constexpr int EV_PER_ITER = 14, EV_MAX_ITERS = 256;
  cudaEvent_t* ev(int k) { return profiling && prof_iters < EV_MAX_ITERS ? &events[(size_t)prof_iters * EV_PER_ITER + k] : nullptr; }
  void rec(int k) { if (cudaEvent_t* e = ev(k)) cudaEventRecord(*e, ctx->stream); }
  ~gingr_registration();   // defined behind mcmc.cuh, where McmcState is complete
};

static int32_t model_build_constants(gingr_ctx* ctx, gingr_model* m);
static int32_t model_upload_topology(gingr_ctx* ctx, gingr_model* m, const int32_t* tri, int T);
static void drop_graph(gingr_registration* g);
static uint64_t g_batch_epoch = 1;   // bumped whenever a chain's captured sequence goes stale (drop_graph, mcmc_release): so are batched plans
static void mcmc_invalidate(gingr_registration* g);  // mcmc.cuh: the device state changed outside the MH chain
static void mcmc_drop_chain_graph(gingr_registration* g);   // mcmc.cuh: the captured MH step of the chain is stale

// reference triangles, vertex -> triangle adjacency and boundary flags of a model (ICP mesh flavours)
static int32_t model_upload_topology(gingr_ctx* ctx, gingr_model* m, const int32_t* tri, int T) {
  const int M = m->M;
  cudaStream_t st = ctx->stream;
  m->T = T;
  if (T <= 0) return GINGR_OK;
  for (int k = 0; k < 3 * T; ++k)
    if (tri[k] < 0 || tri[k] >= M) return gingr_fail(ctx, GINGR_ERR_ARG, "model triangle index out of range");
  std::vector<int32_t> off, adj;
  std::vector<uint8_t> bflags;
  build_vertex_adjacency(M, T, tri, &off, &adj);
  compute_boundary_flags(M, T, tri, &bflags);
  GINGR_CUDA_TRY(ctx, m->boundary.alloc((size_t)M));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->boundary.p, bflags.data(), (size_t)M, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, m->tri.alloc((size_t)3 * T));
  GINGR_CUDA_TRY(ctx, m->adj_off.alloc(off.size()));
  GINGR_CUDA_TRY(ctx, m->adj.alloc(adj.size()));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->tri.p, tri, sizeof(int32_t) * 3 * (size_t)T, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->adj_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->adj.p, adj.data(), adj.size() * 4, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));   // off / adj / bflags are stack vectors
  return GINGR_OK;
}

// new basis rows / mean of point i = those of old point idx[i]  (NearestNeighborInterpolator)
__global__ void rereference_rows_kernel(int M2, int rp, const int32_t* __restrict__ idx, const double* __restrict__ phi,
                                        const double* __restrict__ mean, double* __restrict__ phi2, double* __restrict__ mean2) {
  const int row = blockIdx.x;          // 3 * i + d of the new model
  const int i = row / 3, d = row % 3;
  const size_t src = (size_t)3 * idx[i] + d;
  for (int a = threadIdx.x; a < rp; a += blockDim.x) phi2[(size_t)row * rp + a] = phi[src * rp + a];
  if (threadIdx.x == 0) mean2[row] = mean[src];
}

extern "C" {

int32_t gingr_model_upload(gingr_ctx* ctx, int32_t M, int32_t r, const double* ref_pts, const double* mean,
                           const double* basis, int64_t ld_basis, const double* variance, const int32_t* tri,
                           int32_t T, gingr_model** out) {
  if (!ctx || !out || !ref_pts || !mean || !basis || !variance || M <= 0 || r <= 0 || ld_basis < 3 * (int64_t)M ||
      T < 0 || (T > 0 && !tri))
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_upload: bad argument");
  for (int k = 0; k < r; ++k)
    if (!(variance[k] >= 0.0)) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_upload: negative or NaN variance");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  std::unique_ptr<gingr_model> m(new gingr_model());
  m->ctx = ctx;
  m->M = M;
  m->r = r;
  m->rp = (r + 7) / 8 * 8;
  shard_range(M, ctx->nranks, ctx->rank, &m->m0, &m->Ml);
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, m->ref.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, m->mean.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, m->sqrt_lambda.alloc((size_t)m->rp));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->ref.p, ref_pts, sizeof(double) * 3 * (size_t)M, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->mean.p, mean, sizeof(double) * 3 * (size_t)M, cudaMemcpyHostToDevice, st));
  std::vector<double> sl((size_t)m->rp, 0.0);
  for (int k = 0; k < r; ++k) sl[k] = sqrt(variance[k]);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->sqrt_lambda.p, sl.data(), sizeof(double) * m->rp, cudaMemcpyHostToDevice, st));
  // basis: column-major host -> row-major [3 Ml][rp] device, in column slabs through a transpose kernel
  const size_t rows = (size_t)3 * m->Ml;
  GINGR_CUDA_TRY(ctx, m->phi.alloc(std::max<size_t>(rows, 1) * m->rp));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(m->phi.p, 0, sizeof(double) * std::max<size_t>(rows, 1) * m->rp, st));
  if (rows > 0) {
    const int slab = 128;
    DevBuf<double> tmp;
    GINGR_CUDA_TRY(ctx, tmp.alloc((size_t)slab * rows));
    for (int a0 = 0; a0 < r; a0 += slab) {
      const int nc = std::min(slab, r - a0);
      GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(tmp.p, rows * sizeof(double), basis + (size_t)a0 * ld_basis + (size_t)3 * m->m0,
                                            (size_t)ld_basis * sizeof(double), rows * sizeof(double), nc,
                                            cudaMemcpyHostToDevice, st));
      GINGR_TRY(slab_transpose_enqueue(ctx, (int)rows, nc, tmp.p, m->phi.p + a0, m->rp));
    }
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  }
  GINGR_TRY(model_upload_topology(ctx, m.get(), tri, T));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  GINGR_TRY(model_build_constants(ctx, m.get()));
  *out = m.release();
  return GINGR_OK;
}

int32_t gingr_model_destroy(gingr_model* m) {
  if (!m) return GINGR_OK;
  cudaSetDevice(m->ctx->device);
  delete m;
  return GINGR_OK;
}

// model.newReference(newRef, NearestNeighborInterpolator()) (api/registration/SimpleRegistrator.scala:90-92; scalismo
// semantics SURVEY.md A7): every new reference point takes the mean deformation and the three basis rows of its
// NEAREST old reference point (exact argmin, lowest index on ties: the K2 vertex search); the variances are kept.  The
// basis is no longer orthonormal afterwards, so the constants of the `coefficients` regression are rebuilt.
int32_t gingr_model_new_reference(gingr_ctx* ctx, const gingr_model* model, int32_t M2, const double* new_ref,
                                  const int32_t* tri, int32_t T, gingr_model** out) {
  if (!ctx || !model || !out || !new_ref || M2 <= 0 || T < 0 || (T > 0 && !tri))
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_new_reference: bad argument");
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_model_new_reference: single-GPU entry point (re-reference before sharding)");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int M = model->M, r = model->r, rp = model->rp;
  std::unique_ptr<gingr_model> m(new gingr_model());
  m->ctx = ctx;
  m->M = M2; m->r = r; m->rp = rp; m->m0 = 0; m->Ml = M2;
  GINGR_CUDA_TRY(ctx, m->ref.alloc((size_t)3 * M2));
  GINGR_CUDA_TRY(ctx, m->mean.alloc((size_t)3 * M2));
  GINGR_CUDA_TRY(ctx, m->sqrt_lambda.alloc((size_t)rp));
  GINGR_CUDA_TRY(ctx, m->phi.alloc((size_t)3 * M2 * rp));
  {   // the search scratch is freed before the regression constants are built
    DevBuf<double> old_soa, d2;
    DevBuf<int32_t> idx;
    ClosestWorkspace ws;
    SpatialGrid pgrid;
    GINGR_CUDA_TRY(ctx, old_soa.alloc((size_t)3 * M));
    GINGR_CUDA_TRY(ctx, d2.alloc((size_t)M2));
    GINGR_CUDA_TRY(ctx, idx.alloc((size_t)M2));
    GINGR_TRY(ws.ensure(ctx, M2, M, 0, 0));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->ref.p, new_ref, sizeof(double) * 3 * (size_t)M2, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->sqrt_lambda.p, model->sqrt_lambda.p, sizeof(double) * rp, cudaMemcpyDeviceToDevice, st));
    GINGR_TRY(aos_to_soa_enqueue(ctx, M, model->ref.p, old_soa.p));
    if (grid_wanted(M)) {
      VertexArray va;
      va.p = model->ref.p;
      GINGR_TRY(pgrid.ensure(ctx, M, M, false));
      GINGR_TRY(grid_build_points_enqueue(ctx, pgrid, M, va));
    }
    GINGR_TRY(nn_vertex_enqueue(ctx, ws, M2, m->ref.p, M, old_soa.p, d2.p, idx.p, pgrid.built ? &pgrid : nullptr));
    rereference_rows_kernel<<<3 * M2, 128, 0, st>>>(M2, rp, idx.p, model->phi.p, model->mean.p, m->phi.p, m->mean.p);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  }
  GINGR_TRY(model_upload_topology(ctx, m.get(), tri, T));
  GINGR_TRY(model_build_constants(ctx, m.get()));
  *out = m.release();
  return GINGR_OK;
}

}  // extern "C"

// S = D Phi^T Phi D and W0 = (1e-5 I + S)^-1: the constants of scalismo's `coefficients` regression (all M
// points, noise 1e-5 I3; SURVEY.md A3).  Phi'^T Phi' = Phi^T Phi for any rigid pose, so they are per model.
static int32_t model_build_constants(gingr_ctx* ctx, gingr_model* m) {
  const int r = m->r, rp = m->rp;
  GramPlan plan;
  GINGR_TRY(plan.build(ctx, 3 * m->Ml, r, rp));
  GINGR_CUDA_TRY(ctx, m->S.alloc((size_t)rp * rp));
  GINGR_CUDA_TRY(ctx, m->W0.alloc((size_t)rp * rp));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(m->S.p, 0, sizeof(double) * rp * rp, ctx->stream));
  GINGR_TRY(gram_partials_enqueue(ctx, plan, m->phi.p, nullptr));
  GINGR_TRY(gram_finish_enqueue(ctx, plan, plan.d_partial.p, m->sqrt_lambda.p, 0.0, 0, nullptr, nullptr, rp, m->S.p));
  GINGR_TRY(comm_allreduce_sum(ctx, m->S.p, (size_t)rp * rp));
  // B = [1e-5 I + S ; I]  (2r x r), factorise; rows r..2r-1 then hold L^-T... i.e. Rm with Rm L^T = I
  DevBuf<double> B, Rt;
  DevBuf<int> info;
  GINGR_CUDA_TRY(ctx, B.alloc((size_t)2 * r * rp));
  GINGR_CUDA_TRY(ctx, Rt.alloc((size_t)r * rp));
  GINGR_CUDA_TRY(ctx, info.alloc(4));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(info.p, 0, sizeof(int) * 4, ctx->stream));
  GINGR_TRY(build_regression_system_enqueue(ctx, r, rp, m->S.p, 1e-5, B.p));
  CholWs cws;
  GINGR_TRY(cws.alloc(ctx, r, 2 * r));
  GINGR_TRY(cholesky_enqueue(ctx, r, 2 * r, B.p, rp, info.p, &cws));
  // W0 = Rm Rm^T = Gram of Rm^T
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(Rt.p, 0, sizeof(double) * r * rp, ctx->stream));
  GINGR_TRY(transpose_enqueue(ctx, r, B.p + (size_t)r * rp, rp, Rt.p, rp));
  GramPlan plan2;
  GINGR_TRY(plan2.build(ctx, r, r, rp));
  GINGR_TRY(gram_partials_enqueue(ctx, plan2, Rt.p, nullptr));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(m->W0.p, 0, sizeof(double) * rp * rp, ctx->stream));
  GINGR_TRY(gram_finish_enqueue(ctx, plan2, plan2.d_partial.p, nullptr, 0.0, 0, nullptr, nullptr, rp, m->W0.p));
  int h_info = 0;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(&h_info, info.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (h_info != 0) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_upload: basis/variance not finite (1e-5 I + S not SPD)");
  m->has_regression_constants = true;
  return GINGR_OK;
}

// -------------------------------------------------------------------------------------------------
// building blocks shared by the kernel-level K3 entry points and gingr_update
// -------------------------------------------------------------------------------------------------
namespace gingr {

// instance coefficients -> local mesh rows: out[3 Ml] = Phi_local (sqrt_lambda * alpha) for 1 or 2 alphas
static int32_t instance_rows(gingr_ctx* ctx, const gingr_model* m, double* d_vec_scratch, int nvec, const double* d_alpha0,
                             const double* d_alpha1, double* d_out0, double* d_out1) {
  (void)d_vec_scratch;   // sqrt(lambda) * alpha is formed while the vectors are staged in the row pass
  return gemv_rows_enqueue(ctx, 3 * m->Ml, m->r, m->rp, m->phi.p, nvec, d_alpha0, d_alpha1, d_out0, d_out1, m->sqrt_lambda.p);
}

// local fit rows -> full fit on every rank
static int32_t gather_fit(gingr_ctx* ctx, const gingr_model* m, const double* d_fit_local, double* d_gathered,
                          double* d_fit) {
  if (ctx->nranks == 1) {
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_fit, d_fit_local, sizeof(double) * 3 * (size_t)m->M, cudaMemcpyDeviceToDevice,
                                        ctx->stream));
    return GINGR_OK;
  }
  const int Mmax = ceil_div(m->M, ctx->nranks);
  GINGR_TRY(comm_allgather(ctx, d_fit_local, d_gathered, (size_t)3 * Mmax));
  compact_gather_kernel<<<ceil_div(3 * m->M, 256), 256, 0, ctx->stream>>>(m->M, ctx->nranks, Mmax, d_gathered, d_fit);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

}  // namespace gingr

struct PosteriorScratch {
  GramPlan gram;
  DevBuf<double> Mx, wrow, u, vec, gt_part, inst, fit_local, gathered, fit, ds;
  DevBuf<int> is, flags;
  gingr::CholWs cholws;
};

namespace gingr {
// rows r + 1 + k of the system <- row k of Q = Phi diag(sqrt(lambda)): riding through the factorisation as extra rows they
// come out as Q_k L^-T, whose 3 x 3 Gram blocks are the posterior covariances at the mesh points
__global__ void posterior_cov_rows_kernel(int rows, int r, int rp, const double* __restrict__ phi,
                                          const double* __restrict__ sqrt_lambda, double* __restrict__ out) {
  const int k = blockIdx.y;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < rp; c += gridDim.x * blockDim.x)
    out[(size_t)k * rp + c] = c < r ? phi[(size_t)k * rp + c] * sqrt_lambda[c] : 0.0;
}
// rows r + 1 + k of the system <- sqrt(lambda_k) e_k: they come out as the rows of B = D L^-T, B B^T = D Mx^-1 D
__global__ void posterior_model_rows_kernel(int r, int rp, const double* __restrict__ sqrt_lambda, double* __restrict__ out) {
  const int k = blockIdx.y;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < rp; c += gridDim.x * blockDim.x)
    out[(size_t)k * rp + c] = c == k ? sqrt_lambda[k] : 0.0;
}
// cov_i = R (X_i X_i^T) R^T with X_i the three solved rows of vertex i; one warp per vertex
__global__ void __launch_bounds__(256) posterior_cov_kernel(int M, int r, int rp, const double* __restrict__ X,
                                                            const double* __restrict__ ds, double* __restrict__ cov) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= M) return;
  const double* x0 = X + (size_t)(3 * i) * rp;
  const double* x1 = x0 + rp;
  const double* x2 = x1 + rp;
  double s[6] = {0, 0, 0, 0, 0, 0};
  for (int c = lane; c < r; c += 32) {
    const double a = x0[c], b = x1[c], d = x2[c];
    s[0] = fma(a, a, s[0]); s[1] = fma(a, b, s[1]); s[2] = fma(a, d, s[2]);
    s[3] = fma(b, b, s[3]); s[4] = fma(b, d, s[4]); s[5] = fma(d, d, s[5]);
  }
#pragma unroll
  for (int q = 0; q < 6; ++q)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[q] += __shfl_xor_sync(0xffffffffu, s[q], o);
  if (lane == 0) {
    const double C[9] = {s[0], s[1], s[2], s[1], s[3], s[4], s[2], s[4], s[5]};
    const double* R = ds + DS_R;
    double T[9];
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) T[3 * a + b] = R[3 * a] * C[b] + R[3 * a + 1] * C[3 + b] + R[3 * a + 2] * C[6 + b];
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b)
        cov[(size_t)9 * i + 3 * a + b] = T[3 * a] * R[3 * b] + T[3 * a + 1] * R[3 * b + 1] + T[3 * a + 2] * R[3 * b + 2];
  }
}

// CUDA events at the phase boundaries of a posterior-model build (gingr_posterior_model_profile); destroyed on every exit
struct PosteriorModelEvents {
  cudaEvent_t e[5] = {};
  ~PosteriorModelEvents() {
    for (cudaEvent_t x : e)
      if (x) cudaEventDestroy(x);
  }
  int32_t create(gingr_ctx* ctx) {
    for (cudaEvent_t& x : e) GINGR_CUDA_TRY(ctx, cudaEventCreate(&x));
    return GINGR_OK;
  }
  int32_t record(gingr_ctx* ctx, int k) {
    GINGR_CUDA_TRY(ctx, cudaEventRecord(e[k], ctx->stream));
    return GINGR_OK;
  }
};
}  // namespace gingr
// posterior_model.cuh: the model from the factorised system (rows B = D L^-T behind the rhs row), c and the pose in d_ds
static int32_t posterior_model_finish(gingr_ctx* ctx, const gingr_model* m, const double* d_B, const double* d_c,
                                      const double* d_ds, gingr::PosteriorModelEvents& ev, gingr_model** out);

// the regression of model.transform(R, t).posterior(obs): coefficients, mean mesh and (optionally) the covariance blocks
// or the posterior model itself
static int32_t posterior_core(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t, int32_t n,
                              const int32_t* pid, const double* points, int32_t noise_kind, const double* noise,
                              double* coeffs, double* mean_pts, double* cov_pts, gingr_model** model_out = nullptr) {
  if (!ctx || !model || !R || !t || n < 0 || (n > 0 && (!pid || !points || !noise)) || noise_kind < 0 || noise_kind > 1)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_posterior_mean: bad argument");
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_posterior_mean: single-GPU entry point");
  const gingr_model* m = model;
  const int M = m->M, r = m->r, rp = m->rp;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  gingr::PosteriorModelEvents ev;
  if (model_out) {
    GINGR_TRY(ev.create(ctx));
    GINGR_TRY(ev.record(ctx, 0));
  }
  // Host-side marshalling of the observation list into per-vertex weights / residuals.  Isotropic
  // observations of the same vertex add up (W = sum 1/var, W y = sum y/var); full-covariance ones become
  // "landmark" blocks.
  std::vector<double> wrow((size_t)3 * M, 0.0), u((size_t)3 * M, 0.0);
  std::vector<int32_t> lpid;
  std::vector<double> lpts, lcinv;
  std::vector<double> href((size_t)3 * M), hmean((size_t)3 * M);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(href.data(), m->ref.p, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(hmean.data(), m->mean.p, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  bool bad = false;
  for (int k = 0; k < n; ++k) {
    const int p = pid[k];
    if (p < 0 || p >= M) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_posterior_mean: point id out of range");
    if (noise_kind == 0) {
      const double var = noise[k];
      if (!(var > 0.0) || !(var < INFINITY)) { bad = true; continue; }
      const double w = 1.0 / var;
      double b[3], res[3];
      for (int d = 0; d < 3; ++d) b[d] = href[3 * p + d] + hmean[3 * p + d];
      for (int d = 0; d < 3; ++d)
        res[d] = points[3 * k + d] - (R[3 * d] * b[0] + R[3 * d + 1] * b[1] + R[3 * d + 2] * b[2] + t[d]);
      for (int d = 0; d < 3; ++d) {
        wrow[3 * p + d] += w;
        u[3 * p + d] += w * (R[d] * res[0] + R[3 + d] * res[1] + R[6 + d] * res[2]);
      }
    } else {
      const double* C = noise + 9 * (size_t)k;
      double inv[9];
      const double det = C[0] * (C[4] * C[8] - C[5] * C[7]) - C[1] * (C[3] * C[8] - C[5] * C[6]) +
                         C[2] * (C[3] * C[7] - C[4] * C[6]);
      if (!(fabs(det) > 0.0) || !(fabs(det) < INFINITY)) { bad = true; continue; }
      inv[0] = (C[4] * C[8] - C[5] * C[7]) / det; inv[1] = (C[2] * C[7] - C[1] * C[8]) / det; inv[2] = (C[1] * C[5] - C[2] * C[4]) / det;
      inv[3] = (C[5] * C[6] - C[3] * C[8]) / det; inv[4] = (C[0] * C[8] - C[2] * C[6]) / det; inv[5] = (C[2] * C[3] - C[0] * C[5]) / det;
      inv[6] = (C[3] * C[7] - C[4] * C[6]) / det; inv[7] = (C[1] * C[6] - C[0] * C[7]) / det; inv[8] = (C[0] * C[4] - C[1] * C[3]) / det;
      lpid.push_back(p);
      for (int d = 0; d < 3; ++d) lpts.push_back(points[3 * k + d]);
      for (int d = 0; d < 9; ++d) lcinv.push_back(inv[d]);
    }
  }
  if (bad) return GINGR_MODEL_FLEXIBILITY;
  const int L = (int)lpid.size();
  PosteriorScratch s;
  GINGR_TRY(s.gram.build(ctx, 3 * M, r, rp));
  cudaStream_t st = ctx->stream;
  DevBuf<int32_t> d_lpid;
  DevBuf<double> d_lpts, d_lcinv, d_lA, d_lrows;
  // rows carried through the factorisation: Q for the covariance, D for the posterior model
  const int xrows = cov_pts ? 3 * M : (model_out ? r : 0);
  GINGR_CUDA_TRY(ctx, s.Mx.alloc((size_t)(r + 8 + xrows) * rp));
  GINGR_CUDA_TRY(ctx, s.wrow.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, s.u.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, s.vec.alloc((size_t)8 * rp));
  GINGR_CUDA_TRY(ctx, s.gt_part.alloc((size_t)gemvT_splits(ctx, 3 * M) * rp));
  GINGR_CUDA_TRY(ctx, s.inst.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, s.fit_local.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, s.ds.alloc(DS_COUNT));
  GINGR_CUDA_TRY(ctx, s.is.alloc(IS_COUNT));
  GINGR_CUDA_TRY(ctx, s.flags.alloc(256));
  GINGR_TRY(s.cholws.alloc(ctx, r, r + 1 + xrows));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(s.Mx.p, 0, sizeof(double) * (size_t)(r + 8) * rp, st));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(s.is.p, 0, sizeof(int) * IS_COUNT, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(s.wrow.p, wrow.data(), sizeof(double) * 3 * M, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(s.u.p, u.data(), sizeof(double) * 3 * M, cudaMemcpyHostToDevice, st));
  double hds[DS_COUNT];
  memset(hds, 0, sizeof(hds));
  hds[DS_SCALE] = 1.0;
  for (int d = 0; d < 3; ++d) hds[DS_T + d] = t[d];
  for (int d = 0; d < 9; ++d) hds[DS_R + d] = R[d];
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(s.ds.p, hds, sizeof(hds), cudaMemcpyHostToDevice, st));
  double* rhs = s.Mx.p + (size_t)r * rp;
  GINGR_TRY(gemvT_enqueue(ctx, 3 * M, r, rp, m->phi.p, s.u.p, m->sqrt_lambda.p, s.gt_part.p, rhs));
  if (L > 0) {
    GINGR_CUDA_TRY(ctx, d_lpid.alloc(L));
    GINGR_CUDA_TRY(ctx, d_lpts.alloc(3 * L));
    GINGR_CUDA_TRY(ctx, d_lcinv.alloc(9 * L));
    GINGR_CUDA_TRY(ctx, d_lA.alloc(9 * L));
    GINGR_CUDA_TRY(ctx, d_lrows.alloc((size_t)L * 3 * rp));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_lpid.p, lpid.data(), sizeof(int32_t) * L, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_lpts.p, lpts.data(), sizeof(double) * 3 * L, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_lcinv.p, lcinv.data(), sizeof(double) * 9 * L, cudaMemcpyHostToDevice, st));
    GINGR_LAUNCH(ctx, gather_rows_kernel, dim3(ceil_div(3 * rp, 256), L), 256, 0, st, L, rp, 0, d_lpid.p, m->phi.p, d_lrows.p);
    GINGR_LAUNCH(ctx, landmark_prepare_kernel, ceil_div(L, 64), 64, 0, st, L, d_lcinv.p, s.ds.p, d_lA.p);
    GINGR_LAUNCH(ctx, landmark_rhs_kernel, ceil_div(r, 256), 256, 0, st, r, rp, L, d_lpid.p, d_lpts.p, d_lA.p, d_lrows.p, m->ref.p,
                                                          m->mean.p, m->sqrt_lambda.p, s.ds.p, rhs);
    ctx->launches += 3;
  }
  GINGR_TRY(gram_partials_enqueue(ctx, s.gram, m->phi.p, s.wrow.p));
  GINGR_TRY(gram_finish_enqueue(ctx, s.gram, s.gram.d_partial.p, m->sqrt_lambda.p, 1.0, L, d_lrows.p, d_lA.p, rp, s.Mx.p, false, true));
  if (cov_pts) {
    gingr::posterior_cov_rows_kernel<<<dim3(ceil_div(rp, 256), xrows), 256, 0, st>>>(xrows, r, rp, m->phi.p, m->sqrt_lambda.p,
                                                                                 s.Mx.p + (size_t)(r + 1) * rp);
    GINGR_LAUNCHED(ctx);
  } else if (model_out) {
    gingr::posterior_model_rows_kernel<<<dim3(ceil_div(rp, 256), r), 256, 0, st>>>(r, rp, m->sqrt_lambda.p, s.Mx.p + (size_t)(r + 1) * rp);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_TRY(cholesky_enqueue(ctx, r, r + 1 + xrows, s.Mx.p, rp, s.is.p + IS_INFO, &s.cholws));
  double* c = s.vec.p;
  GINGR_TRY(chol_backsolve_enqueue(ctx, r, s.Mx.p, rp, rhs, c, s.flags.p, &s.cholws));
  GINGR_LAUNCH(ctx, check_finite_kernel, ceil_div(r, 256), 256, 0, st, r, c, s.is.p + IS_FAIL_POST);
  GINGR_LAUNCHED(ctx);
  if (model_out) GINGR_TRY(ev.record(ctx, 1));
  if (mean_pts) {
    GINGR_TRY(instance_rows(ctx, m, s.vec.p + 2 * rp, 1, c, nullptr, s.inst.p, nullptr));
    GINGR_LAUNCH(ctx, fit_from_instance_kernel, ceil_div(M, 256), 256, 0, st, 0, M, m->ref.p, m->mean.p, s.inst.p, s.ds.p, DS_SCALE, DS_T,
                                                               DS_R, s.fit_local.p);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mean_pts, s.fit_local.p, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, st));
  }
  DevBuf<double> d_cov;
  if (cov_pts) {
    GINGR_CUDA_TRY(ctx, d_cov.alloc((size_t)9 * M));
    gingr::posterior_cov_kernel<<<ceil_div(M, 8), 256, 0, st>>>(M, r, rp, s.Mx.p + (size_t)(r + 1) * rp, s.ds.p, d_cov.p);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(cov_pts, d_cov.p, sizeof(double) * 9 * M, cudaMemcpyDeviceToHost, st));
  }
  int his[IS_COUNT];
  if (coeffs) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(coeffs, c, sizeof(double) * r, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(his, s.is.p, sizeof(int) * IS_COUNT, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (his[IS_INFO] || his[IS_FAIL_POST]) return GINGR_MODEL_FLEXIBILITY;
  if (model_out) return posterior_model_finish(ctx, m, s.Mx.p + (size_t)(r + 1) * rp, c, s.ds.p, ev, model_out);
  return GINGR_OK;
}

extern "C" {

// ---- K3 kernel-level entry points -----------------------------------------------------------------
int32_t gingr_posterior_mean(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t, int32_t n,
                             const int32_t* pid, const double* points, int32_t noise_kind, const double* noise,
                             double* coeffs, double* mean_pts) {
  return posterior_core(ctx, model, R, t, n, pid, points, noise_kind, noise, coeffs, mean_pts, nullptr);
}

int32_t gingr_model_posterior(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t, int32_t n,
                              const int32_t* pid, const double* points, int32_t noise_kind, const double* noise,
                              gingr_model** out) {
  if (!out) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_posterior: bad argument");
  *out = nullptr;
  return posterior_core(ctx, model, R, t, n, pid, points, noise_kind, noise, nullptr, nullptr, nullptr, out);
}

int32_t gingr_posterior_covariance(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t, int32_t n,
                                   const int32_t* pid, const double* points, int32_t noise_kind, const double* noise,
                                   double* cov_pts) {
  if (!cov_pts) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_posterior_covariance: bad argument");
  return posterior_core(ctx, model, R, t, n, pid, points, noise_kind, noise, nullptr, nullptr, cov_pts);
}

int32_t gingr_coefficients(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t,
                           const double* mesh_pts, double* coeffs) {
  if (!ctx || !model || !R || !t || !mesh_pts || !coeffs)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_coefficients: bad argument");
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_coefficients: single-GPU entry point");
  const gingr_model* m = model;
  const int M = m->M, r = m->r, rp = m->rp;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> mesh, u, part, vec, ds;
  DevBuf<int> flag;
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, mesh.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, u.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, vec.alloc((size_t)4 * rp));
  GINGR_CUDA_TRY(ctx, part.alloc((size_t)gemvT_splits(ctx, 3 * M) * rp));
  GINGR_CUDA_TRY(ctx, ds.alloc(DS_COUNT));
  GINGR_CUDA_TRY(ctx, flag.alloc(4));
  double hds[DS_COUNT];
  memset(hds, 0, sizeof(hds));
  for (int d = 0; d < 3; ++d) hds[DS_NEW_T + d] = t[d];
  for (int d = 0; d < 9; ++d) hds[DS_R1 + d] = R[d];
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(ds.p, hds, sizeof(hds), cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mesh.p, mesh_pts, sizeof(double) * 3 * M, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(flag.p, 0, sizeof(int) * 4, st));
  GINGR_LAUNCH(ctx, coeff_residual_kernel, ceil_div(M, 256), 256, 0, st, 0, M, mesh.p, m->ref.p, m->mean.p, ds.p, u.p);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(gemvT_enqueue(ctx, 3 * M, r, rp, m->phi.p, u.p, m->sqrt_lambda.p, part.p, vec.p));
  GINGR_TRY(dense_matvec_enqueue(ctx, r, m->W0.p, rp, vec.p, vec.p + rp));
  GINGR_LAUNCH(ctx, check_finite_kernel, ceil_div(r, 256), 256, 0, st, r, vec.p + rp, flag.p);
  GINGR_LAUNCHED(ctx);
  int hflag = 0;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(coeffs, vec.p + rp, sizeof(double) * r, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(&hflag, flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return hflag ? GINGR_MODEL_FLEXIBILITY : GINGR_OK;
}

int32_t gingr_spd_solve(gingr_ctx* ctx, int32_t n, const double* A, int32_t nrhs, const double* B, double* L_out,
                        double* Y_out, double* x_out, int32_t reps, double* ms_out) {
  if (!ctx || !A || n < 1 || nrhs < 0 || (nrhs > 0 && !B) || (x_out && nrhs < 1) || reps < 1)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_spd_solve: bad argument");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int np = (n + 7) / 8 * 8, nrows = n + nrhs;
  DevBuf<double> in, work, x;
  DevBuf<int> info, flags;
  CholWs ws;
  struct TimingEvents {   // destroyed on every exit
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    ~TimingEvents() {
      if (e0) cudaEventDestroy(e0);
      if (e1) cudaEventDestroy(e1);
    }
  } ev;
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, in.alloc((size_t)nrows * np));
  GINGR_CUDA_TRY(ctx, work.alloc((size_t)(nrows + 8) * np));
  GINGR_CUDA_TRY(ctx, x.alloc(np));
  GINGR_CUDA_TRY(ctx, info.alloc(4));
  GINGR_CUDA_TRY(ctx, flags.alloc((size_t)ceil_div(n, 64) + 8));
  GINGR_TRY(ws.alloc(ctx, n, nrows));
  GINGR_CUDA_TRY(ctx, cudaEventCreate(&ev.e0));
  GINGR_CUDA_TRY(ctx, cudaEventCreate(&ev.e1));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(in.p, 0, sizeof(double) * (size_t)nrows * np, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(in.p, sizeof(double) * np, A, sizeof(double) * n, sizeof(double) * n, n, cudaMemcpyHostToDevice, st));
  if (nrhs > 0)
    GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(in.p + (size_t)n * np, sizeof(double) * np, B, sizeof(double) * n, sizeof(double) * n, nrhs,
                                          cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(info.p, 0, sizeof(int) * 4, st));
  float ms_total = 0.f;
  for (int it = 0; it < reps; ++it) {
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(work.p, in.p, sizeof(double) * (size_t)nrows * np, cudaMemcpyDeviceToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaEventRecord(ev.e0, st));
    GINGR_TRY(cholesky_enqueue(ctx, n, nrows, work.p, np, info.p, &ws));
    if (nrhs > 0) GINGR_TRY(chol_backsolve_enqueue(ctx, n, work.p, np, work.p + (size_t)n * np, x.p, flags.p, &ws));
    GINGR_CUDA_TRY(ctx, cudaEventRecord(ev.e1, st));
    GINGR_CUDA_TRY(ctx, cudaEventSynchronize(ev.e1));
    float ms = 0.f;
    GINGR_CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ev.e0, ev.e1));
    ms_total += ms;
  }
  if (ms_out) *ms_out = (double)ms_total / reps;
  int h_info = 0;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(&h_info, info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  if (L_out) {
    GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(L_out, sizeof(double) * n, work.p, sizeof(double) * np, sizeof(double) * n, n,
                                          cudaMemcpyDeviceToHost, st));
  }
  if (Y_out && nrhs > 0)
    GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(Y_out, sizeof(double) * n, work.p + (size_t)n * np, sizeof(double) * np, sizeof(double) * n, nrhs,
                                          cudaMemcpyDeviceToHost, st));
  if (x_out) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(x_out, x.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (L_out)
    for (int i = 0; i < n; ++i)
      for (int k = i + 1; k < n; ++k) L_out[(size_t)i * n + k] = 0.0;
  return h_info ? GINGR_MODEL_FLEXIBILITY : GINGR_OK;
}

int32_t gingr_model_instance(gingr_ctx* ctx, const gingr_model* model, const gingr_state* stt, const double* alpha,
                             double* fit) {
  if (!ctx || !model || !stt || !alpha || !fit) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_instance: bad argument");
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_model_instance: single-GPU entry point");
  if (stt->rank != model->r) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_instance: state rank does not match the model rank");
  if (stt->center[0] != 0.0 || stt->center[1] != 0.0 || stt->center[2] != 0.0)
    return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "rotation centre must be the origin (GeneralRegistrationState.scala:147)");
  const gingr_model* m = model;
  const int M = m->M, r = m->r, rp = m->rp;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> vec, inst, out, ds;
  DevBuf<int> is;
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, vec.alloc((size_t)4 * rp));
  GINGR_CUDA_TRY(ctx, inst.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, out.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, ds.alloc(DS_COUNT));
  GINGR_CUDA_TRY(ctx, is.alloc(IS_COUNT));
  double hds[DS_COUNT];
  memset(hds, 0, sizeof(hds));
  hds[DS_SCALE] = stt->scale;
  for (int d = 0; d < 3; ++d) { hds[DS_T + d] = stt->translation[d]; hds[DS_EULER + d] = stt->euler[d]; }
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(ds.p, hds, sizeof(hds), cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(vec.p, alpha, sizeof(double) * r, cudaMemcpyHostToDevice, st));
  GINGR_LAUNCH(ctx, pose_kernel, 1, 1, 0, st, ds.p, is.p);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(instance_rows(ctx, m, vec.p + rp, 1, vec.p, nullptr, inst.p, nullptr));
  GINGR_LAUNCH(ctx, fit_from_instance_kernel, ceil_div(M, 256), 256, 0, st, 0, M, m->ref.p, m->mean.p, inst.p, ds.p, DS_SCALE, DS_T, DS_R,
                                                             out.p);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(fit, out.p, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return GINGR_OK;
}

// ---- registration handle ---------------------------------------------------------------------------
int32_t gingr_registration_create(gingr_ctx* ctx, const gingr_model* model, const gingr_target* target,
                                  const gingr_config* cfg, gingr_registration** out) {
  if (!ctx || !model || !target || !cfg || !out) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_registration_create: bad argument");
  if (cfg->algorithm != GINGR_ALGO_CPD && cfg->algorithm != GINGR_ALGO_ICP)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_registration_create: unknown algorithm");
  if (cfg->algorithm == GINGR_ALGO_CPD && !(cfg->w >= 0.0 && cfg->w < 1.0))
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_registration_create: CPD w must be in [0, 1)");
  if (cfg->algorithm == GINGR_ALGO_ICP) {
    if (cfg->correspondence_method < GINGR_TRIANGULAR_CLOSEST_POINT || cfg->correspondence_method > GINGR_POINTCLOUD_CLOSEST_POINT)
      return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_registration_create: unknown correspondence method");
    if (cfg->correspondence_method != GINGR_POINTCLOUD_CLOSEST_POINT && (model->T <= 0 || target->T <= 0))
      return gingr_fail(ctx, GINGR_ERR_ARG, "the mesh flavours of the ICP correspondence need model and target triangles");
  }
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  std::unique_ptr<gingr_registration> g(new gingr_registration());
  g->ctx = ctx;
  g->model = model;
  g->target = target;
  g->cfg = *cfg;
  const int M = model->M, r = model->r, rp = model->rp, Ml = model->Ml;
  const int Mmax = ceil_div(M, ctx->nranks);
  if (cfg->algorithm == GINGR_ALGO_CPD) {
    GINGR_TRY(g->estep.ensure(ctx, M, std::max(target->N, 1)));
    // the fit moves about the reference points, so their k-d order keeps the E-step's model tiles compact
    std::vector<double> ref((size_t)3 * M);
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(ref.data(), model->ref.p, sizeof(double) * ref.size(), cudaMemcpyDeviceToHost, ctx->stream));
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<int32_t> perm;
    estep_row_order(ref.data(), M, perm);
    GINGR_TRY(g->estep.set_row_order(ctx, M, perm.data()));
  } else {
    const bool rev = cfg->reverse_correspondence_direction != 0;
    GINGR_TRY(rev ? g->closest.ensure(ctx, target->N_total, M, model->T, target->T)
                  : g->closest.ensure(ctx, M, target->N_total, target->T, model->T));
    GINGR_CUDA_TRY(ctx, g->fit_normals.alloc((size_t)3 * M));
    const bool mesh_flavour = cfg->correspondence_method != GINGR_POINTCLOUD_CLOSEST_POINT;
    if (grid_wanted(M)) {
      // the fit is scanned by the self-intersection test of the mesh flavours (both directions) and, in the
      // reversed direction, by the vertex / surface searches themselves
      if (mesh_flavour && model->T > 0) {
        GINGR_TRY(g->fit_tgrid.ensure(ctx, M, model->T, true));
        g->use_fit_tgrid = true;
      }
      if (rev) {
        GINGR_TRY(g->fit_pgrid.ensure(ctx, M, M, false));
        g->use_fit_pgrid = true;
      }
    }
    if (rev) {
      GINGR_CUDA_TRY(ctx, g->fit_soa.alloc((size_t)3 * M));
      GINGR_CUDA_TRY(ctx, g->rev_tid.alloc((size_t)target->N_total));
      GINGR_CUDA_TRY(ctx, g->rev_cp.alloc((size_t)3 * M));
      GINGR_CUDA_TRY(ctx, g->rev_wcnt.alloc((size_t)M));
      GINGR_CUDA_TRY(ctx, g->rev_scratch.alloc((size_t)3 * M + target->N_total + 1));
    }
  }
  GINGR_TRY(g->gram.build(ctx, 3 * Ml, r, rp));
  GINGR_CUDA_TRY(ctx, g->rows_ext.alloc((size_t)4 * M + 8));
  GINGR_CUDA_TRY(ctx, g->Mx.alloc((size_t)(r + 8) * rp));
  if (ctx->nranks > 1) GINGR_CUDA_TRY(ctx, g->Mx_packed.alloc(gram_packed_doubles(g->gram) + rp));
  GINGR_CUDA_TRY(ctx, g->prep_sync.alloc(2));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->prep_sync.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
  GINGR_CUDA_TRY(ctx, g->wrow.alloc((size_t)3 * Mmax));
  GINGR_CUDA_TRY(ctx, g->u.alloc((size_t)3 * Mmax));
  GINGR_CUDA_TRY(ctx, g->resid.alloc((size_t)3 * Mmax));
  GINGR_CUDA_TRY(ctx, g->inst_a.alloc((size_t)3 * Mmax));
  GINGR_CUDA_TRY(ctx, g->inst_b.alloc((size_t)3 * Mmax));
  GINGR_CUDA_TRY(ctx, g->newshape.alloc((size_t)3 * Mmax));
  GINGR_CUDA_TRY(ctx, g->fit_local.alloc((size_t)3 * Mmax));
  GINGR_CUDA_TRY(ctx, g->gathered.alloc((size_t)3 * Mmax * ctx->nranks));
  GINGR_CUDA_TRY(ctx, g->fit.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, g->vec.alloc((size_t)8 * rp));
  GINGR_CUDA_TRY(ctx, g->gt_part.alloc((size_t)gemvT_splits(ctx, 3 * Ml) * rp));
  GINGR_CUDA_TRY(ctx, g->sums_part.alloc((size_t)3 * ceil_div(M, 256)));
  GINGR_CUDA_TRY(ctx, g->pro_part.alloc((size_t)16 * ceil_div(std::max(Ml, 1), 256)));
  GINGR_CUDA_TRY(ctx, g->pro_sums.alloc(32));
  GINGR_CUDA_TRY(ctx, g->ds.alloc(DS_COUNT));
  GINGR_CUDA_TRY(ctx, g->is.alloc(IS_COUNT));
  GINGR_CUDA_TRY(ctx, g->flags.alloc(256));
  GINGR_TRY(g->cholws.alloc(ctx, r, r + 1));
  GINGR_CUDA_TRY(ctx, g->alpha.alloc((size_t)rp));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->Mx.p, 0, sizeof(double) * (size_t)(r + 8) * rp, ctx->stream));
  if (g->Mx_packed.p) GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->Mx_packed.p, 0, sizeof(double) * g->Mx_packed.n, ctx->stream));   // unused slots stay 0
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->fit_local.p, 0, sizeof(double) * 3 * Mmax, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->ds.p, 0, sizeof(double) * DS_COUNT, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->is.p, 0, sizeof(int) * IS_COUNT, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->is.p + IS_RETRY, &g->retry_counter, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->alpha.p, 0, sizeof(double) * rp, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->rows_ext.p, 0, sizeof(double) * ((size_t)4 * M + 8), ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  *out = g.release();
  return GINGR_OK;
}

int32_t gingr_registration_destroy(gingr_registration* g) {
  if (!g) return GINGR_OK;
  cudaSetDevice(g->ctx->device);
  cudaStreamSynchronize(g->ctx->stream);
  ++g_batch_epoch;   // a later registration can get this address: batched plans that name this one are stale
  for (auto& e : g->events) cudaEventDestroy(e);
  delete g;
  return GINGR_OK;
}

int32_t gingr_registration_set_landmarks(gingr_registration* g, int32_t L, const int32_t* pid, const double* points,
                                         const double* cov) {
  if (!g || L < 0 || (L > 0 && (!pid || !points || !cov))) return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "set_landmarks: bad argument");
  gingr_ctx* ctx = g->ctx;
  const gingr_model* m = g->model;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  std::vector<int32_t> lpid;
  std::vector<double> lpts, lcinv;
  for (int l = 0; l < L; ++l) {
    if (pid[l] < 0 || pid[l] >= m->M) return gingr_fail(ctx, GINGR_ERR_ARG, "set_landmarks: vertex id out of range");
    const double* C = cov + 9 * (size_t)l;
    const double det = C[0] * (C[4] * C[8] - C[5] * C[7]) - C[1] * (C[3] * C[8] - C[5] * C[6]) + C[2] * (C[3] * C[7] - C[4] * C[6]);
    if (!(fabs(det) > 0.0) || !(fabs(det) < INFINITY)) return gingr_fail(ctx, GINGR_ERR_ARG, "set_landmarks: singular covariance");
    if (pid[l] >= m->m0 && pid[l] < m->m0 + m->Ml) {
      lpid.push_back(pid[l]);
      for (int d = 0; d < 3; ++d) lpts.push_back(points[3 * l + d]);
      const double inv[9] = {(C[4] * C[8] - C[5] * C[7]) / det, (C[2] * C[7] - C[1] * C[8]) / det, (C[1] * C[5] - C[2] * C[4]) / det,
                             (C[5] * C[6] - C[3] * C[8]) / det, (C[0] * C[8] - C[2] * C[6]) / det, (C[2] * C[3] - C[0] * C[5]) / det,
                             (C[3] * C[7] - C[4] * C[6]) / det, (C[1] * C[6] - C[0] * C[7]) / det, (C[0] * C[4] - C[1] * C[3]) / det};
      for (int d = 0; d < 9; ++d) lcinv.push_back(inv[d]);
    }
  }
  g->L = L;
  g->Ll = (int)lpid.size();
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, g->lm_pid.alloc(std::max(L, 1)));
  if (L > 0) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->lm_pid.p, pid, sizeof(int32_t) * L, cudaMemcpyHostToDevice, st));
  const int Ll = g->Ll;
  GINGR_CUDA_TRY(ctx, g->lml_pid.alloc(std::max(Ll, 1)));
  GINGR_CUDA_TRY(ctx, g->lml_pts.alloc(std::max(3 * Ll, 1)));
  GINGR_CUDA_TRY(ctx, g->lml_cinv.alloc(std::max(9 * Ll, 1)));
  GINGR_CUDA_TRY(ctx, g->lml_A.alloc(std::max(9 * Ll, 1)));
  GINGR_CUDA_TRY(ctx, g->lml_rows.alloc(std::max<size_t>((size_t)Ll * 3 * m->rp, 1)));
  if (Ll > 0) {
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->lml_pid.p, lpid.data(), sizeof(int32_t) * Ll, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->lml_pts.p, lpts.data(), sizeof(double) * 3 * Ll, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->lml_cinv.p, lcinv.data(), sizeof(double) * 9 * Ll, cudaMemcpyHostToDevice, st));
    GINGR_LAUNCH(ctx, gather_rows_kernel, dim3(ceil_div(3 * m->rp, 256), Ll), 256, 0, st, Ll, m->rp, m->m0, g->lml_pid.p, m->phi.p,
                                                                          g->lml_rows.p);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  g->state_valid = false;
  drop_graph(g);  // the landmark buffers (and their count) are baked into the captured launches
  return GINGR_OK;
}

}  // extern "C"

// -------------------------------------------------------------------------------------------------
// state upload / fit evaluation / one iteration
// -------------------------------------------------------------------------------------------------
static int32_t upload_state(gingr_registration* g, const gingr_state* s, const double* alpha) {
  gingr_ctx* ctx = g->ctx;
  if (s->rank != g->model->r) return gingr_fail(ctx, GINGR_ERR_ARG, "state rank does not match the model rank");
  if (s->center[0] != 0.0 || s->center[1] != 0.0 || s->center[2] != 0.0)
    return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "rotation centre must be the origin (GeneralRegistrationState.scala:147)");
  double* h = ctx->h_pinned;
  memset(h, 0, sizeof(double) * DS_COUNT);
  h[DS_SCALE] = s->scale;
  for (int d = 0; d < 3; ++d) { h[DS_T + d] = s->translation[d]; h[DS_EULER + d] = s->euler[d]; h[DS_CENTER + d] = s->center[d]; }
  h[DS_SIGMA2] = s->sigma2;
  h[DS_STEP] = s->step_length;
  int* hi = reinterpret_cast<int*>(h + DS_COUNT);
  memset(hi, 0, sizeof(int) * IS_COUNT);
  hi[IS_GT] = s->global_transformation;
  hi[IS_ITER] = s->iteration;
  hi[IS_STATUS] = s->status;
  hi[IS_RETRY] = g->retry_counter;  // the counter belongs to the algorithm instance, not to the state (:70)
  double* ha = h + DS_COUNT + IS_COUNT;
  if ((size_t)(DS_COUNT + IS_COUNT + g->model->r) > ctx->h_pinned_count) {
    // large ranks: alpha goes straight from the caller's buffer
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->alpha.p, alpha, sizeof(double) * g->model->r, cudaMemcpyHostToDevice, ctx->stream));
  } else {
    memcpy(ha, alpha, sizeof(double) * g->model->r);
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->alpha.p, ha, sizeof(double) * g->model->r, cudaMemcpyHostToDevice, ctx->stream));
  }
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->ds.p, h, sizeof(double) * DS_COUNT, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->is.p, hi, sizeof(int) * IS_COUNT, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_LAUNCH(ctx, pose_kernel, 1, 1, 0, ctx->stream, g->ds.p, g->is.p);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

// fit = s (R instance(alpha) + t) with the pose at the given state-block offsets; result in g->fit (all ranks)
static int32_t evaluate_fit(gingr_registration* g, int off_s, int off_t, int off_R) {
  gingr_ctx* ctx = g->ctx;
  const gingr_model* m = g->model;
  GINGR_TRY(instance_rows(ctx, m, g->vec.p + 6 * m->rp, 1, g->alpha.p, nullptr, g->inst_a.p, nullptr));
  if (m->Ml > 0) {
    GINGR_LAUNCH(ctx, fit_from_instance_kernel, ceil_div(m->Ml, 256), 256, 0, ctx->stream, m->m0, m->Ml, m->ref.p, m->mean.p, g->inst_a.p,
                                                                            g->ds.p, off_s, off_t, off_R,
                                                                            ctx->nranks == 1 ? g->fit.p : g->fit_local.p);
    GINGR_LAUNCHED(ctx);
  }
  if (ctx->nranks == 1) return GINGR_OK;   // one rank owns every row: the fit was written in place
  return gather_fit(ctx, m, g->fit_local.p, g->gathered.p, g->fit.p);
}

// The iteration in two phases, so that the Metropolis-Hastings chain (mcmc.cuh) can keep the posterior of a state and
// reuse it (scalismo's Memoize of cashedPosterior, GingrAlgorithm.scala:68):
//   posterior phase  correspondence -> observations -> rhs, Gram -> Cholesky with the forward substitution; leaves
//                    L and z = L^-1 rhs in g->Mx (and, if g->keep_raw, the unfactorised Mx in g->Mx_raw)
//   update phase     (sample |) back solve -> alpha* -> Procrustes -> alpha_new -> commit -> fit
static int32_t enqueue_posterior_phase(gingr_registration* g) {
  gingr_ctx* ctx = g->ctx;
  const gingr_model* m = g->model;
  const gingr_target* tg = g->target;
  const gingr_config& cfg = g->cfg;
  const int M = m->M, r = m->r, rp = m->rp, Ml = m->Ml, m0 = m->m0;
  cudaStream_t st = ctx->stream;
  double* vec = g->vec.p;  // [0] c_post  [1] S c  [2] alpha*  [3] alpha_c  [4] q  [5] alpha_new  [6,7] scaled scratch
  // events: 0/1 iteration, 2..5 E-step sweeps, 6/7 Gram, 8/9 Cholesky + back solve, 10/11 closest point, 12/13 unused
  g->rec(0);
  GINGR_LAUNCH(ctx, pose_kernel, 1, 1, 0, st, g->ds.p, g->is.p);
  GINGR_LAUNCHED(ctx);
  // ---- correspondence -------------------------------------------------------------------------------
  const double* icp_cp = nullptr;
  const double* icp_wcnt = nullptr;
  if (cfg.algorithm == GINGR_ALGO_CPD) {
    // non-finite fit / sigma2 / target: the reference's P is all NaN and the posterior fails
    if (tg->nonfinite) GINGR_TRY(validate_finite_enqueue(ctx, 3 * tg->N_total, tg->verts.p, g->is.p + IS_FAIL_POST));
    GINGR_LAUNCH(ctx, cpd_prepare_kernel, ceil_div(M, 256), 256, 0, st, M, g->fit.p, g->estep.row_perm.p, g->estep.fit_soa.p, g->ds.p, cfg.w,
                                                         (double)M / (double)tg->N_total, tg->maxabs, g->is.p + IS_FAIL_POST,
                                                         g->prep_sync.p, g->estep.scal.p);
    GINGR_LAUNCHED(ctx);
    if (tg->N > 0) {
      EstepEvents ee;
      const bool pe = g->ev(2) != nullptr;
      if (pe) { ee.a0 = *g->ev(2); ee.a1 = *g->ev(3); ee.b0 = *g->ev(4); ee.b1 = *g->ev(5); }
      GINGR_TRY(estep_enqueue(ctx, g->estep, M, tg->N, tg->soa.p, tg->soa_perm.p, false, pe ? &ee : nullptr));
      GINGR_CUDA_TRY(ctx, gingr_copy_d2d(ctx, g->rows_ext.p, g->estep.rows.p, sizeof(double) * 4 * (size_t)M, st));
      GINGR_LAUNCH(ctx, xpx_total_kernel, 1, 256, 0, st, g->estep.plan.den_blocks, g->estep.xpx_part.p, g->rows_ext.p + (size_t)4 * M);
      GINGR_LAUNCHED(ctx);
    } else {
      GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->rows_ext.p, 0, sizeof(double) * ((size_t)4 * M + 8), st));
    }
    GINGR_TRY(comm_allreduce_sum(ctx, g->rows_ext.p, (size_t)4 * M + 8));
  } else {
    g->rec(10);
    const bool mesh_flavour = cfg.correspondence_method != GINGR_POINTCLOUD_CLOSEST_POINT;
    MeshView fv, tv;
    fv.n = M; fv.aos = g->fit.p; fv.T = m->T; fv.tri = m->tri.p; fv.boundary = m->boundary.p;
    if (mesh_flavour) {
      GINGR_TRY(vertex_normals_enqueue(ctx, M, g->fit.p, m->tri.p, m->adj_off.p, m->adj.p, g->fit_normals.p));
      fv.normals = g->fit_normals.p;
    }
    tv.n = tg->N_total; tv.aos = tg->aos.p; tv.soa = tg->verts.p; tv.T = tg->T; tv.tri = tg->tri.p;
    tv.normals = tg->normals.p; tv.boundary = tg->boundary.p;
    tv.pgrid = tg->pgrid.get(); tv.tgrid = tg->tgrid.get();
    VertexArray fva;
    fva.p = g->fit.p;
    if (g->use_fit_tgrid) {
      GINGR_TRY(grid_build_triangles_enqueue(ctx, g->fit_tgrid, M, fva, m->T, m->tri.p));
      fv.tgrid = &g->fit_tgrid;
    }
    if (g->use_fit_pgrid) {
      GINGR_TRY(grid_build_points_enqueue(ctx, g->fit_pgrid, M, fva));
      fv.pgrid = &g->fit_pgrid;
    }
    if (!cfg.reverse_correspondence_direction) {
      // several ranks: every rank searches only the vertices of its own basis shard [m0, m0 + Ml) -- the queries are
      // split across the GPUs (SURVEY 8e, ClosestPointRegistrator.scala:74-131), and since a rank's observation rows ARE
      // those vertices nothing has to be gathered.  (The reversed direction folds target queries onto template vertices
      // and stays replicated.)
      if (ctx->nranks > 1) GINGR_TRY(icp_correspondence_enqueue(ctx, g->closest, fv, tv, cfg.correspondence_method, m0, Ml));
      else GINGR_TRY(icp_correspondence_enqueue(ctx, g->closest, fv, tv, cfg.correspondence_method));
      icp_cp = g->closest.cp.p;
    } else {
      // closestPointCorrespondenceReversal (ClosestPointRegistrator.scala:34-45): search from the target to the fit,
      // map every corresponding point back to its nearest fit vertex, observe the TARGET point there
      GINGR_TRY(aos_to_soa_enqueue(ctx, M, g->fit.p, g->fit_soa.p));
      fv.soa = g->fit_soa.p;
      GINGR_TRY(icp_correspondence_enqueue(ctx, g->closest, tv, fv, cfg.correspondence_method));
      GINGR_TRY(nn_vertex_enqueue(ctx, g->closest, tg->N_total, g->closest.cp.p, M, g->fit_soa.p, g->closest.d2.p,
                                  g->rev_tid.p, fv.pgrid, g->closest.qorder.get()));
      GINGR_TRY(reverse_fold_enqueue(ctx, M, tg->N_total, g->rev_tid.p, g->closest.w.p, tg->aos.p, g->rev_cp.p,
                                     g->rev_wcnt.p, g->rev_scratch.p));
      icp_cp = g->rev_cp.p;
      icp_wcnt = g->rev_wcnt.p;
    }
    g->rec(11);
  }
  // ---- observations, sigma2 hook ----------------------------------------------------------------------
  ObsArgs oa;
  oa.algo = cfg.algorithm; oa.M = M; oa.m0 = m0; oa.Ml = Ml; oa.use_lm = cfg.use_landmark_correspondence && g->L > 0;
  oa.L = g->L; oa.lambda = cfg.lambda;
  const int oblocks = ceil_div(M, 256);
  // the right-hand side D Phi^T W resid rides along in the Gram (no pass of its own over Phi) unless landmarks add their
  // own terms to it or the rank is a multiple of the tile edge (no spare column in the last tile row)
  const bool use_lm = cfg.use_landmark_correspondence && g->Ll > 0;
  const bool any_lm = cfg.use_landmark_correspondence && g->L > 0;
  const bool rhs_fused = !any_lm && gram_rhs_fusable(g->gram);
  GINGR_LAUNCH(ctx, obs_kernel, oblocks, 256, 0, st, oa, g->rows_ext.p, icp_cp, g->closest.w.p, icp_wcnt, g->fit.p, m->ref.p, m->mean.p,
                                      g->lm_pid.p, g->ds.p, g->is.p, g->wrow.p, g->u.p, g->sums_part.p,
                                      rhs_fused ? g->resid.p : nullptr);
  GINGR_LAUNCHED(ctx);
  const double sigma_step = cfg.algorithm == GINGR_ALGO_ICP ? (cfg.initial_sigma - cfg.end_sigma) / (double)cfg.max_iterations : 0.0;
  GINGR_LAUNCH(ctx, sigma2_kernel, 1, 32, 0, st, cfg.algorithm, oblocks, g->sums_part.p, g->rows_ext.p + (size_t)4 * M, sigma_step,
                                 cfg.end_sigma, g->ds.p);
  GINGR_LAUNCHED(ctx);
  // ---- posterior: rhs, Gram, Cholesky --------------------------------------------------------------------
  // several ranks: the partial matrix is written as packed lower tiles with the rhs behind them, so that ONE all-reduce of
  // half the bytes of the (r + 1) x rp rectangle combines both; it is unpacked into g->Mx afterwards
  const bool packed = ctx->nranks > 1;
  const size_t packed_n = packed ? gram_packed_doubles(g->gram) : 0;
  double* rhs = packed ? g->Mx_packed.p + packed_n : g->Mx.p + (size_t)r * rp;
  if (!rhs_fused) GINGR_TRY(gemvT_enqueue(ctx, 3 * Ml, r, rp, m->phi.p, g->u.p, m->sqrt_lambda.p, g->gt_part.p, rhs));
  if (use_lm) {
    GINGR_LAUNCH(ctx, landmark_prepare_kernel, ceil_div(g->Ll, 64), 64, 0, st, g->Ll, g->lml_cinv.p, g->ds.p, g->lml_A.p);
    GINGR_LAUNCH(ctx, landmark_rhs_kernel, ceil_div(r, 256), 256, 0, st, r, rp, g->Ll, g->lml_pid.p, g->lml_pts.p, g->lml_A.p, g->lml_rows.p,
                                                          m->ref.p, m->mean.p, m->sqrt_lambda.p, g->ds.p, rhs);
    ctx->launches += 2;
  }
  GINGR_TRY(gram_partials_enqueue(ctx, g->gram, m->phi.p, g->wrow.p, g->ev(6) ? *g->ev(6) : nullptr,
                                  g->ev(7) ? *g->ev(7) : nullptr, rhs_fused ? g->resid.p : nullptr));
  if (packed) {
    GINGR_TRY(gram_finish_enqueue(ctx, g->gram, g->gram.d_partial.p, m->sqrt_lambda.p, ctx->rank == 0 ? 1.0 : 0.0,
                                  use_lm ? g->Ll : 0, g->lml_rows.p, g->lml_A.p, rp, g->Mx_packed.p, true, false, rhs_fused));
    GINGR_TRY(comm_allreduce_sum(ctx, g->Mx_packed.p, packed_n + (rhs_fused ? 0 : (size_t)r)));
    GINGR_TRY(gram_unpack_enqueue(ctx, g->gram, g->Mx_packed.p, rp, g->Mx.p, rhs_fused));
    if (!rhs_fused)
      GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(g->Mx.p + (size_t)r * rp, rhs, sizeof(double) * r, cudaMemcpyDeviceToDevice, st));
  } else {
    // the upper triangle is only read from the kept copy of the MH chain (mcmc.cuh: dense products with the raw matrix)
    GINGR_TRY(gram_finish_enqueue(ctx, g->gram, g->gram.d_partial.p, m->sqrt_lambda.p, 1.0, use_lm ? g->Ll : 0, g->lml_rows.p,
                                  g->lml_A.p, rp, g->Mx.p, false, !g->keep_raw, rhs_fused));
  }
  if (g->keep_raw)
    GINGR_CUDA_TRY(ctx, gingr_copy_d2d(ctx, g->Mx_raw.p, g->Mx.p, sizeof(double) * (size_t)(r + 1) * rp, st));
  g->rec(8);
  GINGR_TRY(cholesky_enqueue(ctx, r, r + 1, g->Mx.p, rp, g->is.p + IS_INFO, &g->cholws));
  return GINGR_OK;
}

// fresh_factor: g->Mx was factorised by the posterior phase right before (its block inverses still sit in g->cholws); the
// MH chain calls this on a KEPT factor that was copied around since, and then takes chol.cu's back substitution
static int32_t enqueue_update_phase(gingr_registration* g, int probabilistic, uint64_t seed, bool fresh_factor = false) {
  gingr_ctx* ctx = g->ctx;
  const gingr_model* m = g->model;
  const gingr_config& cfg = g->cfg;
  const int M = m->M, r = m->r, rp = m->rp, Ml = m->Ml, m0 = m->m0;
  cudaStream_t st = ctx->stream;
  double* vec = g->vec.p;
  double* rhs = g->Mx.p + (size_t)r * rp;
  (void)cfg;
  if (probabilistic) {  // posterior.sample() instead of posterior.mean (:211)
    // counter of the Philox stream: the state's iteration (gingr_update) or the chain's MH step (mcmc.cuh)
    GINGR_LAUNCH(ctx, add_normal_kernel, ceil_div(ceil_div(r, 2), 128), 128, 0, st, r, seed, g->sample_counter ? g->sample_counter : g->is.p + IS_ITER,
                                                                     rhs);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_TRY(chol_backsolve_enqueue(ctx, r, g->Mx.p, rp, rhs, vec, g->flags.p, fresh_factor ? &g->cholws : nullptr));
  g->rec(9);
  // ---- alpha* = coefficients(posterior mean) = W0 S c ; combine ---------------------------------------------
  // (a non-finite c is flagged by the first product, a non-finite alpha_new by the last: no separate launches)
  GINGR_TRY(dense_matvec_enqueue(ctx, r, m->S.p, rp, vec, vec + rp, g->is.p + IS_FAIL_POST, nullptr));
  GINGR_TRY(dense_matvec_enqueue(ctx, r, m->W0.p, rp, vec + rp, vec + 2 * rp));
  GINGR_LAUNCH(ctx, combine_kernel, ceil_div(r, 256), 256, 0, st, r, g->alpha.p, vec + 2 * rp, g->ds.p, vec + 3 * rp);
  GINGR_LAUNCHED(ctx);
  // ---- instances, Procrustes -----------------------------------------------------------------------------------
  GINGR_TRY(instance_rows(ctx, m, vec + 6 * rp, 2, g->alpha.p, vec + 3 * rp, g->inst_a.p, g->inst_b.p));
  const int pblocks = ceil_div(std::max(Ml, 1), 256);
  if (ctx->nranks == 1) {
    for (int pass = 0; pass < 2; ++pass) {
      GINGR_LAUNCH(ctx, procrustes_sums_kernel, pblocks, 256, 0, st, pass, m0, Ml, m->ref.p, m->mean.p, g->inst_a.p, g->inst_b.p, g->ds.p,
                                                      g->newshape.p, g->pro_part.p);
      GINGR_LAUNCHED(ctx);
      // one rank: the block partials are summed (same fixed order) by the kernel that consumes the sums
      GINGR_LAUNCH(ctx, procrustes_reduce_then_kernel, 1, 32, 0, st, pass, pblocks, M, g->pro_part.p, g->pro_sums.p, g->ds.p, g->is.p);
      GINGR_LAUNCHED(ctx);
    }
  } else {
    // several ranks: one pass of shifted moments and ONE all-reduce of 16 doubles (two latency-bound all-reduces and the
    // second pass over the shard before)
    GINGR_LAUNCH(ctx, procrustes_sums_kernel, pblocks, 256, 0, st, 2, m0, Ml, m->ref.p, m->mean.p, g->inst_a.p, g->inst_b.p, g->ds.p,
                                                    g->newshape.p, g->pro_part.p);
    GINGR_LAUNCHED(ctx);
    GINGR_LAUNCH(ctx, procrustes_reduce_kernel, 1, 32, 0, st, Ml > 0 ? pblocks : 0, 16, g->pro_part.p, g->pro_sums.p);
    GINGR_LAUNCHED(ctx);
    GINGR_TRY(comm_allreduce_sum(ctx, g->pro_sums.p, 16));
    GINGR_LAUNCH(ctx, procrustes_moments_solve_kernel, 1, 1, 0, st, M, g->pro_sums.p, m->ref.p, m->mean.p, g->ds.p, g->is.p);
    GINGR_LAUNCHED(ctx);
  }
  // ---- alpha_new = transformedModel.coefficients(newshape) ---------------------------------------------------------
  if (Ml > 0) {
    GINGR_LAUNCH(ctx, coeff_residual_kernel, ceil_div(Ml, 256), 256, 0, st, m0, Ml, g->newshape.p, m->ref.p, m->mean.p, g->ds.p, g->u.p);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_TRY(gemvT_enqueue(ctx, 3 * Ml, r, rp, m->phi.p, g->u.p, m->sqrt_lambda.p, g->gt_part.p, vec + 4 * rp));
  GINGR_TRY(comm_allreduce_sum(ctx, vec + 4 * rp, (size_t)r));
  GINGR_TRY(dense_matvec_enqueue(ctx, r, m->W0.p, rp, vec + 4 * rp, vec + 5 * rp, nullptr, g->is.p + IS_FAIL_COEF));
  // ---- commit, refresh the fit ------------------------------------------------------------------------------------------
  GINGR_LAUNCH(ctx, finalize_kernel, 1, 256, 0, st, r, probabilistic, vec + 5 * rp, g->alpha.p, g->ds.p, g->is.p);
  GINGR_LAUNCHED(ctx);
  if (!g->skip_fit_refresh) GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R2));
  g->rec(1);
  if (g->profiling && g->prof_iters < gingr_registration::EV_MAX_ITERS) g->prof_iters++;
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

static int32_t enqueue_iteration(gingr_registration* g, int probabilistic = 0, uint64_t seed = 0) {
  GINGR_TRY(enqueue_posterior_phase(g));
  return enqueue_update_phase(g, probabilistic, seed, true);
}

static bool graphs_enabled(const gingr_ctx* ctx) {
  static const int env = [] { const char* e = getenv("GINGR_CUDA_GRAPH"); return e ? atoi(e) : 2; }();
  // GINGR_CUDA_GRAPH: 0 = off, 1 = single-GPU contexts only, 2 (default) = also capture the NCCL collectives of a
  // multi-rank iteration (NCCL >= 2.9 supports stream capture; the ranks run the same deterministic sequence)
  return env != 0 && (ctx->nranks == 1 || env >= 2);
}

static void drop_graph(gingr_registration* g) {
  ++g_batch_epoch;
  g->graph_exec.reset();
  g->graph_prob = -1;
}

// Captures into `exec` what enqueue() puts on the ctx stream.  *launches receives the launches enqueue() counted; nothing
// ran yet, so they are taken off ctx->launches again, and every replay adds them.
template <typename F>
static int32_t capture_graph(gingr_ctx* ctx, GraphExec& exec, int64_t* launches, F&& enqueue) {
  exec.reset();
  const int64_t l0 = ctx->launches;
  GINGR_CUDA_TRY(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
  const int32_t rc = enqueue();
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
  *launches = ctx->launches - l0;
  ctx->launches = l0;
  if (rc < 0) {
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  GINGR_CUDA_TRY(ctx, e);
  const cudaError_t e2 = cudaGraphInstantiate(&exec.h, graph, 0);
  cudaGraphDestroy(graph);
  GINGR_CUDA_TRY(ctx, e2);
  return GINGR_OK;
}

// The captured iteration of g for (probabilistic, seed); captured again when the key changed.
static int32_t iteration_graph(gingr_registration* g, int probabilistic, uint64_t seed) {
  if (g->graph_exec.h && g->graph_prob == probabilistic && (!probabilistic || g->graph_seed == seed)) return GINGR_OK;
  drop_graph(g);
  GINGR_TRY(capture_graph(g->ctx, g->graph_exec, &g->graph_launches, [&] { return enqueue_iteration(g, probabilistic, seed); }));
  g->graph_prob = probabilistic;
  g->graph_seed = seed;
  return GINGR_OK;
}

// One iteration, through the captured graph when possible (not while profiling: the events live outside graphs).
static int32_t run_iteration(gingr_registration* g, int probabilistic, uint64_t seed) {
  gingr_ctx* ctx = g->ctx;
  if (g->profiling || !graphs_enabled(ctx)) return enqueue_iteration(g, probabilistic, seed);
  GINGR_TRY(iteration_graph(g, probabilistic, seed));
  GINGR_CUDA_TRY(ctx, cudaGraphLaunch(g->graph_exec.h, ctx->stream));
  ctx->launches += g->graph_launches;
  return GINGR_OK;
}

static int32_t download_state(gingr_registration* g, gingr_state* out, double* alpha_out, double* fit_out) {
  gingr_ctx* ctx = g->ctx;
  const gingr_model* m = g->model;
  double* h = ctx->h_pinned;
  int* hi = reinterpret_cast<int*>(h + DS_COUNT);
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(h, g->ds.p, sizeof(double) * DS_COUNT, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(hi, g->is.p, sizeof(int) * IS_COUNT, cudaMemcpyDeviceToHost, st));
  if (alpha_out) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(alpha_out, g->alpha.p, sizeof(double) * m->r, cudaMemcpyDeviceToHost, st));
  if (fit_out) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(fit_out, g->fit.p, sizeof(double) * 3 * (size_t)m->M, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  out->scale = h[DS_SCALE];
  for (int d = 0; d < 3; ++d) { out->translation[d] = h[DS_T + d]; out->euler[d] = h[DS_EULER + d]; out->center[d] = h[DS_CENTER + d]; }
  out->sigma2 = h[DS_SIGMA2];
  out->step_length = h[DS_STEP];
  out->global_transformation = hi[IS_GT];
  out->iteration = hi[IS_ITER];
  out->status = hi[IS_STATUS];
  out->rank = m->r;
  g->retry_counter = hi[IS_RETRY];
  return GINGR_OK;
}

// equal up to the bookkeeping fields the host-side `propose` touches (iteration, status)
static bool same_state(gingr_state a, const gingr_state& b) {
  a.iteration = b.iteration;
  a.status = b.status;
  return memcmp(&a, &b, sizeof(gingr_state)) == 0;
}

// Pool of streams the batched entry points (gingr_update_batch, gingr_mcmc_batch) replay the chains' graphs on: one pool
// per host thread and device, created on first use.
struct ChainStreamPool {
  static constexpr int NS = 64;   // allocated; GINGR_BATCH_STREAMS (default 16) of them are used
  cudaStream_t streams[NS] = {nullptr};
  cudaEvent_t fork_ev = nullptr, join_ev[NS] = {nullptr};
  int device = -1;
  int used = 16;
};

static int32_t chain_stream_pool(gingr_ctx* ctx, ChainStreamPool** out) {
  static thread_local ChainStreamPool pool;
  if (pool.device != ctx->device) {
    for (int q = 0; q < ChainStreamPool::NS; ++q) {
      GINGR_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&pool.streams[q], cudaStreamNonBlocking));
      GINGR_CUDA_TRY(ctx, cudaEventCreateWithFlags(&pool.join_ev[q], cudaEventDisableTiming));
    }
    GINGR_CUDA_TRY(ctx, cudaEventCreateWithFlags(&pool.fork_ev, cudaEventDisableTiming));
    pool.device = ctx->device;
    const char* e = getenv("GINGR_BATCH_STREAMS");
    if (e && atoi(e) > 0) pool.used = std::min(atoi(e), (int)ChainStreamPool::NS);
  }
  *out = &pool;
  return GINGR_OK;
}

// Replay `iters` times the graphs of n chains on the pool's streams (chain k always on stream k % ns, so its steps stay
// ordered).  post(k, stream) enqueues what follows a chain's graph (may be empty).  Measured: the replay rate is bound by
// the device-side launch processing of the graph nodes (about 0.5 us per kernel node), not by the host -- more streams
// than 16 or several launching host threads do not raise it (profiles/r02_small_problems.md).
template <typename G, typename P>
static int32_t replay_chain_graphs(gingr_ctx* ctx, ChainStreamPool* sp, int n, int iters, G&& graph_of, P&& post) {
  const int ns = std::min(sp->used, n);
  GINGR_CUDA_TRY(ctx, cudaEventRecord(sp->fork_ev, ctx->stream));
  for (int q = 0; q < ns; ++q) GINGR_CUDA_TRY(ctx, cudaStreamWaitEvent(sp->streams[q], sp->fork_ev, 0));
  for (int it = 0; it < iters; ++it)
    for (int k = 0; k < n; ++k) {
      GINGR_CUDA_TRY(ctx, cudaGraphLaunch(graph_of(k), sp->streams[k % ns]));
      post(k, sp->streams[k % ns]);
    }
  for (int q = 0; q < ns; ++q) {
    GINGR_CUDA_TRY(ctx, cudaEventRecord(sp->join_ev[q], sp->streams[q]));
    GINGR_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, sp->join_ev[q], 0));
  }
  return GINGR_OK;
}

// ---- many chains, ONE kernel sequence (batch.cuh) ---------------------------------------------------------------------
// Every chain's step is recorded (arguments only, nothing is launched), the sequences are checked to be the same launch
// for launch, the argument tuples go to the device as [launch][chain] arrays and the batched forms of the kernels are
// captured as one graph: blockIdx.z = chain.  A plan is kept until the set of chains, the seed, the kind of step or a
// chain's configuration changes.  Users: gingr_mcmc_batch (mcmc.cuh) and gingr_update_batch.  Each keeps one plan per host
// thread on the heap and never deletes it: a plan is never freed at thread or process exit, where the CUDA runtime may
// already be shut down.
struct BatchPlan {
  std::vector<gingr_registration*> regs;
  std::vector<double> step_lengths;
  uint64_t seed = 0, epoch = 0;
  int device = -1, kind = 0;    // kind: 1 update (deterministic), 3 update (sampled), 2 Metropolis-Hastings step
  bool unsupported = false;     // a launch / copy on the path is not batch-aware, or the chains differ: per-chain graphs
  int nlaunch = 0;
  DevBuf<unsigned char> d_args;
  GraphExec exec;
  void drop() {
    exec.reset();
    regs.clear();
    step_lengths.clear();
    unsupported = false;
    nlaunch = 0;
  }
};

static bool batch_plan_current(const BatchPlan& bp, gingr_ctx* ctx, gingr_registration** regs, int n, uint64_t seed, int kind) {
  if (bp.epoch != g_batch_epoch || bp.device != ctx->device || bp.seed != seed || bp.kind != kind || (int)bp.regs.size() != n)
    return false;
  for (int k = 0; k < n; ++k)
    if (bp.regs[k] != regs[k] || bp.step_lengths[k] != regs[k]->last_out.step_length) return false;
  return true;
}

// a chain's Gram on few CTAs: with n chains in one launch the machine is filled by the chains, and the empty CTAs of the
// 148-wide schedule would each still cost a slot with 200 KB of shared memory
static int32_t batch_cap_gram(gingr_ctx* ctx, gingr_registration** regs, int n) {
  const int cap = std::max(1, (2 * ctx->num_sms) / n);
  for (int k = 0; k < n; ++k) {
    gingr_registration* g = regs[k];
    if (g->gram.ncta > cap) {
      GINGR_TRY(g->gram.build(ctx, g->gram.rows, g->gram.r, g->gram.rp, cap));
      drop_graph(g);
      mcmc_invalidate(g);   // a kept posterior was formed in the other summation order
      mcmc_drop_chain_graph(g);
    }
  }
  return GINGR_OK;
}

template <typename F>
static int32_t batch_plan_build(gingr_ctx* ctx, gingr_registration** regs, int n, uint64_t seed, int kind, BatchPlan& bp,
                                F&& enqueue_chain) {
  bp.drop();
  bp.epoch = g_batch_epoch;
  bp.device = ctx->device;
  bp.seed = seed;
  bp.kind = kind;
  bp.regs.assign(regs, regs + n);
  for (int k = 0; k < n; ++k) bp.step_lengths.push_back(regs[k]->last_out.step_length);
  cudaStream_t st = ctx->stream;
  // 1. record: inside a capture, so that whatever is not batch-aware is caught in the discarded graph instead of running
  std::vector<LaunchRecorder> rec((size_t)n);
  const int64_t l0 = ctx->launches;
  GINGR_CUDA_TRY(ctx, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  int32_t rc = GINGR_OK;
  for (int k = 0; k < n && rc >= 0; ++k) {
    ctx->rec = &rec[k];
    rc = enqueue_chain(k);
  }
  ctx->rec = nullptr;
  ctx->launches = l0;
  cudaGraph_t stray = nullptr;
  const cudaError_t ec = cudaStreamEndCapture(st, &stray);
  size_t stray_nodes = 0;
  if (stray) {
    cudaGraphGetNodes(stray, nullptr, &stray_nodes);
    cudaGraphDestroy(stray);
  }
  if (rc < 0) return rc;
  GINGR_CUDA_TRY(ctx, ec);
  // 2. the same sequence for every chain?
  bool same = stray_nodes == 0 && !rec[0].recs.empty();
  const std::vector<LaunchRecord>& r0 = rec[0].recs;
  for (int k = 1; k < n && same; ++k) {
    const std::vector<LaunchRecord>& rk = rec[k].recs;
    same = rk.size() == r0.size();
    for (size_t i = 0; i < r0.size() && same; ++i)
      same = rk[i].fn == r0[i].fn && rk[i].arg_bytes == r0[i].arg_bytes && rk[i].smem == r0[i].smem &&
             rk[i].grid.x == r0[i].grid.x && rk[i].grid.y == r0[i].grid.y && rk[i].grid.z == r0[i].grid.z &&
             rk[i].block.x == r0[i].block.x && rk[i].block.y == r0[i].block.y && rk[i].block.z == r0[i].block.z;
  }
  for (size_t i = 0; i < r0.size() && same; ++i) same = r0[i].grid.z == 1;
  if (!same) {
    if (getenv("GINGR_BATCH_VERBOSE"))
      fprintf(stderr, "gingr batch: not batchable (%zu stray stream operations, %zu recorded launches): per-chain graphs\n",
              stray_nodes, r0.size());
    bp.unsupported = true;
    return GINGR_OK;
  }
  // 3. argument arrays [launch][chain]
  std::vector<size_t> off(r0.size());
  size_t total = 0;
  for (size_t i = 0; i < r0.size(); ++i) {
    off[i] = total;
    total += ((size_t)r0[i].arg_bytes * n + 255) / 256 * 256;
  }
  std::vector<unsigned char> h(total, 0);
  for (size_t i = 0; i < r0.size(); ++i)
    for (int k = 0; k < n; ++k)
      memcpy(h.data() + off[i] + (size_t)k * r0[i].arg_bytes, rec[k].args.data() + rec[k].recs[i].arg_off, r0[i].arg_bytes);
  GINGR_CUDA_TRY(ctx, bp.d_args.alloc(total));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(bp.d_args.p, h.data(), total, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  // 4. the batched sequence as one graph
  for (size_t i = 0; i < r0.size(); ++i)
    if (r0[i].smem > 48 * 1024)
      GINGR_CUDA_TRY(ctx, cudaFuncSetAttribute(r0[i].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)r0[i].smem));
  GINGR_CUDA_TRY(ctx, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  cudaError_t el = cudaSuccess;
  for (size_t i = 0; i < r0.size() && el == cudaSuccess; ++i) {
    const void* p = bp.d_args.p + off[i];
    void* params[1] = {(void*)&p};
    el = cudaLaunchKernel(r0[i].fn, dim3(r0[i].grid.x, r0[i].grid.y, (unsigned)n), r0[i].block, params, r0[i].smem, st);
  }
  cudaGraph_t graph = nullptr;
  const cudaError_t e2 = cudaStreamEndCapture(st, &graph);
  if (el != cudaSuccess || e2 != cudaSuccess) {
    if (graph) cudaGraphDestroy(graph);
    GINGR_CUDA_TRY(ctx, el);
    GINGR_CUDA_TRY(ctx, e2);
  }
  const cudaError_t e3 = cudaGraphInstantiate(&bp.exec.h, graph, 0);
  cudaGraphDestroy(graph);
  GINGR_CUDA_TRY(ctx, e3);
  bp.nlaunch = (int)r0.size();
  return GINGR_OK;
}

extern "C" {

int32_t gingr_initialize_state(gingr_registration* g, gingr_state* s, const double* alpha, double* fit_out) {
  if (!g || !s || !alpha) return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_initialize_state: bad argument");
  mcmc_invalidate(g);
  gingr_ctx* ctx = g->ctx;
  const gingr_model* m = g->model;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  s->rank = m->r;
  if (g->cfg.algorithm == GINGR_ALGO_ICP || g->cfg.has_initial_sigma) {
    s->sigma2 = g->cfg.initial_sigma;  // ICP.scala:74-78 ; CPD.scala:94 (initialSigma given)
  } else {
    // computeInitialSigma2 over model.mean = ref + meanVector (CPD.scala:95)
    DevBuf<double> mp, outv;
    GINGR_CUDA_TRY(ctx, mp.alloc((size_t)3 * m->M));
    GINGR_CUDA_TRY(ctx, outv.alloc(4));
    add_vectors_enqueue(ctx, 3 * m->M, m->ref.p, m->mean.p, mp.p);
    GINGR_TRY(initial_sigma2_enqueue(ctx, m->M, mp.p, g->target->N_total, g->target->verts.p, outv.p));
    double v = 0.0;
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(&v, outv.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    s->sigma2 = v;
  }
  GINGR_TRY(upload_state(g, s, alpha));
  GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R));
  gingr_state tmp;
  GINGR_TRY(download_state(g, &tmp, nullptr, fit_out));
  g->last_out = *s;
  g->host_mirror_current = true;
  g->last_alpha.assign(alpha, alpha + m->r);
  g->state_valid = true;
  return GINGR_OK;
}

int32_t gingr_update(gingr_registration* g, const gingr_state* state_in, const double* alpha_in, int32_t probabilistic,
                     uint64_t seed, gingr_state* state_out, double* alpha_out, double* fit_out) {
  if (!g || !state_in || !alpha_in || !state_out || !alpha_out)
    return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_update: bad argument");
  mcmc_invalidate(g);
  gingr_ctx* ctx = g->ctx;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const gingr_model* m = g->model;
  // Re-seed the device state unless the caller hands back exactly what the previous call returned
  // (then the device-resident fit is already the fit of this state).
  const bool resume = g->state_valid && g->host_mirror_current && same_state(*state_in, g->last_out) &&
                      memcmp(alpha_in, g->last_alpha.data(), sizeof(double) * m->r) == 0;
  if (!resume) {
    GINGR_TRY(upload_state(g, state_in, alpha_in));
    GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R));
  } else {
    GINGR_LAUNCH(ctx, set_iteration_kernel, 1, 1, 0, ctx->stream, g->is.p, state_in->iteration, state_in->status);
    GINGR_LAUNCHED(ctx);
  }
  g->state_valid = false;
  GINGR_TRY(run_iteration(g, probabilistic != 0, seed));
  GINGR_TRY(download_state(g, state_out, alpha_out, fit_out));
  g->last_out = *state_out;
  g->host_mirror_current = true;
  g->last_alpha.assign(alpha_out, alpha_out + m->r);
  g->state_valid = true;
  return GINGR_OK;
}

int32_t gingr_update_chain(gingr_registration* g, int32_t iters) {
  if (!g || iters < 0) return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_update_chain: bad argument");
  gingr_ctx* ctx = g->ctx;
  if (!g->state_valid) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_update_chain: no device-resident state (call gingr_initialize_state / gingr_update first)");
  mcmc_invalidate(g);
  g->host_mirror_current = false;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  for (int k = 0; k < iters; ++k) {
    GINGR_TRY(run_iteration(g, 0, 0));
    GINGR_LAUNCH(ctx, bump_iteration_kernel, 1, 1, 0, ctx->stream, g->is.p);  // GingrGeneratorWrapper.propose: updateIteration()
    GINGR_LAUNCHED(ctx);
  }
  return GINGR_OK;
}

int32_t gingr_update_chain_sampled(gingr_registration* g, int32_t iters, uint64_t seed) {
  if (!g || iters < 0) return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_update_chain_sampled: bad argument");
  gingr_ctx* ctx = g->ctx;
  if (!g->state_valid) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_update_chain_sampled: no device-resident state");
  mcmc_invalidate(g);
  g->host_mirror_current = false;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  for (int k = 0; k < iters; ++k) {
    GINGR_TRY(run_iteration(g, 1, seed));  // the Philox counter carries the device iteration number
    GINGR_LAUNCH(ctx, bump_iteration_kernel, 1, 1, 0, ctx->stream, g->is.p);
    GINGR_LAUNCHED(ctx);
  }
  return GINGR_OK;
}

// Independent registrations / MCMC chains (SURVEY.md 8e "replicas only"; BASELINE config 5): every chain is its own
// gingr_registration (own state and workspaces; model and target handles are shared), its iteration is one captured
// CUDA graph, and the graphs of different chains are replayed round-robin on a small pool of streams so that the
// launch-latency-bound kernels of ~16 chains are in flight at once.  No collective, no cross-chain data.
int32_t gingr_update_batch(gingr_registration** regs, int32_t n, int32_t iters, int32_t probabilistic, uint64_t seed) {
  if (!regs || n <= 0 || iters < 0) return gingr_fail(nullptr, GINGR_ERR_ARG, "gingr_update_batch: bad argument");
  gingr_ctx* ctx = regs[0]->ctx;
  for (int k = 0; k < n; ++k) {
    if (!regs[k] || regs[k]->ctx != ctx) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_update_batch: chains must share one ctx");
    if (!regs[k]->state_valid) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_update_batch: chain without device-resident state");
    if (regs[k]->profiling) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_update_batch: profiling is per registration");
    mcmc_invalidate(regs[k]);
    regs[k]->host_mirror_current = false;
  }
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_update_batch: chains are replicas, one ctx per GPU without a communicator");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  // one batched kernel sequence per iteration for all chains (batch.cuh) when every launch of the iteration is batch-aware
  // (the ICP flavours on the scans; the CPD E-step is not: per-chain graphs), GINGR_UPDATE_BATCHED=0: always per-chain graphs
  static const int batched = [] { const char* e = getenv("GINGR_UPDATE_BATCHED"); return e ? atoi(e) : 1; }();
  if (batched && n >= 2 && n <= 65535 && graphs_enabled(ctx)) {
    static thread_local BatchPlan& bp = *new BatchPlan();   // never deleted (BatchPlan)
    const int kind = probabilistic ? 3 : 1;
    if (!batch_plan_current(bp, ctx, regs, n, seed, kind)) {
      int32_t rc = batch_cap_gram(ctx, regs, n);
      if (rc >= 0)
        rc = batch_plan_build(ctx, regs, n, seed, kind, bp, [&](int k) -> int32_t {
          GINGR_TRY(enqueue_iteration(regs[k], probabilistic != 0, seed + (uint64_t)k));
          GINGR_LAUNCH(ctx, bump_iteration_kernel, 1, 1, 0, ctx->stream, regs[k]->is.p);
          GINGR_LAUNCHED(ctx);
          return GINGR_OK;
        });
      if (rc < 0) { bp.drop(); return rc; }
    }
    if (!bp.unsupported) {
      for (int it = 0; it < iters; ++it) GINGR_CUDA_TRY(ctx, cudaGraphLaunch(bp.exec.h, ctx->stream));
      ctx->launches += (int64_t)iters * bp.nlaunch;
      return GINGR_OK;
    }
  }
  ChainStreamPool* sp = nullptr;
  GINGR_TRY(chain_stream_pool(ctx, &sp));
  // capture (or re-key) every chain's graph on the ctx stream first: capture is not concurrent
  for (int k = 0; k < n; ++k) GINGR_TRY(iteration_graph(regs[k], probabilistic != 0, seed + (uint64_t)k));
  GINGR_TRY(replay_chain_graphs(ctx, sp, n, iters, [&](int k) { return regs[k]->graph_exec.h; },
                                [&](int k, cudaStream_t st) { GINGR_LAUNCH(ctx, bump_iteration_kernel, 1, 1, 0, st, regs[k]->is.p); }));
  for (int k = 0; k < n; ++k) ctx->launches += (int64_t)iters * (regs[k]->graph_launches + 1);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

int32_t gingr_registration_set_profiling(gingr_registration* g, int32_t enable) {
  if (!g) return GINGR_ERR_ARG;
  gingr_ctx* ctx = g->ctx;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (enable && g->events.empty()) {
    g->events.resize((size_t)gingr_registration::EV_PER_ITER * gingr_registration::EV_MAX_ITERS);
    for (auto& e : g->events) GINGR_CUDA_TRY(ctx, cudaEventCreate(&e));
  }
  g->profiling = enable != 0;
  g->prof_iters = 0;
  if (g->estep.live.p) GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->estep.live.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
  return GINGR_OK;
}

int32_t gingr_registration_get_profile(gingr_registration* g, double* ms, int32_t* iterations) {
  if (!g || !ms || !iterations) return GINGR_ERR_ARG;
  gingr_ctx* ctx = g->ctx;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 8; ++k) ms[k] = 0.0;
  const bool cpd = g->cfg.algorithm == GINGR_ALGO_CPD && g->target->N > 0;
  for (int it = 0; it < g->prof_iters; ++it) {
    cudaEvent_t* e = &g->events[(size_t)it * gingr_registration::EV_PER_ITER];
    float t = 0.f;
    auto el = [&](int a, int b) { t = 0.f; cudaEventElapsedTime(&t, e[a], e[b]); return (double)t; };
    if (cpd) { ms[0] += el(2, 3); ms[1] += el(4, 5); } else if (g->cfg.algorithm == GINGR_ALGO_ICP) { ms[5] += el(10, 11); }
    ms[2] += el(6, 7);
    ms[3] += el(8, 9);
    ms[4] += el(0, 1);
  }
  if (cpd) {
    const EstepPlan& p = g->estep.plan;
    unsigned long long live[2] = {0, 0};
    if (p.cull) {
      GINGR_CUDA_TRY(ctx, cudaMemcpy(live, g->estep.live.p, sizeof(live), cudaMemcpyDeviceToHost));
      GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g->estep.live.p, 0, sizeof(live), ctx->stream));
    }
    ms[6] = p.cull ? (double)live[0] / ((double)p.col_blocks * p.nsub) : g->prof_iters;
    ms[7] = p.cull ? (double)live[1] / ((double)p.row_blocks * p.ntt) : g->prof_iters;
  }
  *iterations = g->prof_iters;
  g->prof_iters = 0;
  cudaGetLastError();
  return GINGR_OK;
}

int32_t gingr_state_download(gingr_registration* g, gingr_state* state_out, double* alpha_out, double* fit_out) {
  if (!g || !state_out) return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_state_download: bad argument");
  GINGR_CUDA_TRY(g->ctx, cudaSetDevice(g->ctx->device));
  GINGR_TRY(download_state(g, state_out, alpha_out, fit_out));
  g->last_out = *state_out;
  g->host_mirror_current = true;
  if (alpha_out) g->last_alpha.assign(alpha_out, alpha_out + g->model->r);
  else g->state_valid = false;
  return GINGR_OK;
}

}  // extern "C"

#include "mcmc.cuh"
#include "gpmm.cuh"
#include "posterior_model.cuh"

gingr_registration::~gingr_registration() = default;
