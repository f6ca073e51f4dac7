/*
 * gingr_cuda.h -- C ABI of libgingr_cuda.so, the B200 (sm_100a) implementation of GiNGR's
 * per-iteration hot path `GingrAlgorithm.update`.
 *
 * The reference (unibas-gravis/GiNGR, Scala 3) has NO native / FFI boundary today; the
 * extension surface is the Scala trait `GingrAlgorithm[State, config]`
 * (src/main/scala/gingr/api/GingrAlgorithm.scala:65).  A Scala shim (scala/ in this repo,
 * binding shown in INTEGRATION.md) subclasses that trait, overrides `update` (:192) and
 * `generatorCombined` (:177) and calls the entry points below through Panama FFM / JNI.
 * Each entry point cites the reference statement it replaces (paths relative to
 * /root/reference/src/main/scala/gingr/).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - All floating point is IEEE double (the reference is Breeze/scalismo Double end to end);
 *     indices are int32 (scalismo PointId(id: Int)).
 *   - Host arrays are caller-owned: inputs are read-only, outputs are caller-allocated.
 *     Points are row-major [n][3].  The GPMM basis is COLUMN-major [3M x r] with leading
 *     dimension `ld_basis` (Breeze DenseMatrix layout of scalismo's basisMatrix), row 3*pid+d.
 *   - Device memory is library-owned behind opaque handles and freed only by *_destroy.
 *   - A gingr_ctx is bound to one CUDA device and is single-threaded (the reference calls
 *     `update` from one thread per algorithm instance, GingrAlgorithm.scala:70).  Distinct
 *     contexts may be used concurrently.  Multi-GPU = one process (or thread) per GPU, each
 *     with its own ctx, joined by gingr_comm_init (NCCL).
 *   - Every function returns an int32 status: 0 = OK, 1 = MODEL_FLEXIBILITY (the numerical
 *     failure the reference maps to FittingStatuses.ModelFlexibilityError,
 *     GingrAlgorithm.scala:194-208, :214-217, :235-251), negative = error; text via
 *     gingr_last_error.  No exceptions cross the ABI.  There is no CPU fallback: without a
 *     CUDA device gingr_ctx_create fails with GINGR_ERR_CUDA.
 */
#ifndef GINGR_CUDA_H
#define GINGR_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GINGR_API __attribute__((visibility("default")))

/* ---- status codes -------------------------------------------------------------------------- */
#define GINGR_OK 0
#define GINGR_MODEL_FLEXIBILITY 1 /* non-finite result or matrix not SPD */
#define GINGR_ERR_ARG (-1)
#define GINGR_ERR_CUDA (-2)
#define GINGR_ERR_NCCL (-3)
#define GINGR_ERR_UNSUPPORTED (-4)

/* ---- enums mirroring the reference --------------------------------------------------------- */
/* api/FittingStatuses.scala:20-23 (Enumeration order) */
#define GINGR_STATUS_NONE 0
#define GINGR_STATUS_MAX_ITERATION 1
#define GINGR_STATUS_CONVERGED 2
#define GINGR_STATUS_MODEL_FLEXIBILITY_ERROR 3
/* api/GlobalTranformationType.scala:20-24 */
#define GINGR_SIMILARITY_TRANSFORMS 0
#define GINGR_RIGID_TRANSFORMS 1
#define GINGR_NO_TRANSFORMS 2
/* registration/config/ICP.scala:29-33 ICPCorrespondenceMethod */
#define GINGR_TRIANGULAR_CLOSEST_POINT 0
#define GINGR_ALONG_NORMAL_CLOSEST_POINT 1
#define GINGR_POINTCLOUD_CLOSEST_POINT 2
/* which GingrAlgorithm subclass */
#define GINGR_ALGO_CPD 0 /* registration/config/CPD.scala:117 CpdRegistration */
#define GINGR_ALGO_ICP 1 /* registration/config/ICP.scala:84 IcpRegistration */

typedef struct gingr_ctx gingr_ctx;
typedef struct gingr_model gingr_model;               /* scalismo PointDistributionModel on device */
typedef struct gingr_target gingr_target;             /* target TriangleMesh on device */
typedef struct gingr_registration gingr_registration; /* model + target + config + workspaces */

/*
 * POD mirror of the numeric part of GeneralRegistrationState (api/GeneralRegistrationState.scala:28-41)
 * and ModelFittingParameters (api/ModelFittingParameters.scala:31-74).  The shape coefficient
 * vector alpha[rank] travels beside it as a plain double array.  `model`, `target`, landmarks live
 * in the handles; `fit` is an explicit array argument.
 */
typedef struct gingr_state {
  double scale;          /* ScaleParameter.s */
  double translation[3]; /* PoseParameters.translation */
  double euler[3];       /* EulerAngles phi, theta, psi  (R = Rz(phi) Ry(theta) Rx(psi)) */
  double center[3];      /* EulerRotation.center -- GiNGR always uses the origin */
  double sigma2;         /* GeneralRegistrationState.sigma2 */
  double step_length;    /* GeneralRegistrationState.stepLength */
  int32_t global_transformation; /* GINGR_*_TRANSFORMS */
  int32_t iteration;
  int32_t status; /* GINGR_STATUS_* */
  int32_t rank;   /* length of alpha */
} gingr_state;

/*
 * POD mirror of CpdConfiguration (registration/config/CPD.scala:105-115) and IcpConfiguration
 * (registration/config/ICP.scala:54-66).  The `converged` closure stays on the host side.
 */
typedef struct gingr_config {
  int32_t algorithm; /* GINGR_ALGO_* */
  int32_t max_iterations;
  double threshold;
  int32_t use_landmark_correspondence;
  int32_t has_initial_sigma; /* CPD: initialSigma: Option[Double] */
  double initial_sigma;      /* CPD (if has_initial_sigma) / ICP initialSigma (used as sigma2, ICP.scala:74-78) */
  double w;                  /* CPD outlier weight */
  double lambda;             /* CPD noise scaling (CPD.scala:114, :125) */
  double end_sigma;          /* ICP */
  int32_t reverse_correspondence_direction; /* ICP */
  int32_t correspondence_method;            /* ICP, GINGR_*_CLOSEST_POINT */
} gingr_config;

/* ---- context --------------------------------------------------------------------------------- */
GINGR_API int32_t gingr_version(void);
GINGR_API int32_t gingr_ctx_create(int32_t device, gingr_ctx** out);
GINGR_API int32_t gingr_ctx_destroy(gingr_ctx* ctx);
/* Text of the last error on this ctx (or of the last ctx-less error when ctx == NULL). */
GINGR_API const char* gingr_last_error(const gingr_ctx* ctx);
/* cudaStream_t all work of this ctx is enqueued on (for CUDA-event timing by the caller). */
GINGR_API void* gingr_ctx_stream(gingr_ctx* ctx);
GINGR_API int32_t gingr_ctx_synchronize(gingr_ctx* ctx);
/* Number of kernels this ctx has launched so far (bench.py's gpu_launches). */
GINGR_API int64_t gingr_ctx_launch_count(const gingr_ctx* ctx);

/* ---- multi-GPU (new: the reference has no distributed code; SURVEY.md 8e) ------------------- */
/* Rank 0 creates an id and ships it to the other ranks by any host channel. */
GINGR_API int32_t gingr_comm_unique_id(char id[128]);
/* Join an NCCL communicator of `nranks` contexts.  After this call, target points (E-step) and
 * GPMM basis rows (Gram, fit evaluation) uploaded through this ctx are sharded by rank and the
 * partial sums are combined with ncclAllReduce inside gingr_update. */
GINGR_API int32_t gingr_comm_init(gingr_ctx* ctx, int32_t nranks, int32_t rank, const char id[128]);

/* ---- uploads ----------------------------------------------------------------------------------- */
/* scalismo PointDistributionModel: reference points, meanVector, basisMatrix, variance
 * (SURVEY.md A1).  tri may be NULL (T = 0) for CPD-only use; ICP needs the reference triangles. */
GINGR_API int32_t gingr_model_upload(gingr_ctx* ctx, int32_t M, int32_t r, const double* ref_pts /*[3M]*/,
                                     const double* mean /*[3M]*/, const double* basis /*col-major*/,
                                     int64_t ld_basis, const double* variance /*[r]*/,
                                     const int32_t* tri /*[3T]*/, int32_t T, gingr_model** out);
GINGR_API int32_t gingr_model_destroy(gingr_model* m);
/* model.newReference(newRef, NearestNeighborInterpolator()) of SimpleRegistrator.decimateState
 * (api/registration/SimpleRegistrator.scala:84-106; scalismo semantics SURVEY.md A7): every new reference point takes
 * the mean deformation and basis rows of its nearest old reference point (exact argmin, ties -> lowest index), on the
 * device, from the resident basis.  The decimated reference mesh itself (scalismo's quadric `decimate`) is the caller's.
 * Used with gingr_target_upload of the decimated target to run the multi-resolution schedule of
 * examples/DemoMultiResolution.scala:39-47 without re-uploading a basis. */
GINGR_API int32_t gingr_model_new_reference(gingr_ctx* ctx, const gingr_model* model, int32_t M2,
                                            const double* new_ref_pts /*[3 M2]*/, const int32_t* tri /*[3T]*/,
                                            int32_t T, gingr_model** out);
/* GPMM construction (SURVEY.md 8f item 4): GPMMTriangleMesh3D(reference, relativeTolerance).Gaussian(sigma, scaling) /
 * .GaussianMixture(pars) (api/gpmm/GPMMHelper.scala:99-129) = GPMM.construct (:39-54) = scalismo
 * LowRankGaussianProcess.approximateGPCholesky (SURVEY.md A7) for DiagonalKernel(sum_q scaling_q GaussianKernel(sigma_q), 3):
 * pivoted Cholesky until trace(residual) <= rel_tol * trace(K) (at most max_rank columns, 0 = no cap), then the KL basis
 * (orthonormal columns, variances) -- all on the device; the mean is zero.  The basis is unique only up to rotations inside
 * the (triple) eigenspaces: rank, variances and the covariance basis diag(variance) basis^T are what is defined. */
GINGR_API int32_t gingr_gpmm_gaussian_mixture(gingr_ctx* ctx, int32_t M, const double* ref_pts /*[3M]*/,
                                              const int32_t* tri /*[3T]*/, int32_t T, int32_t n_kernels,
                                              const double* sigma /*[n]*/, const double* scaling /*[n]*/, double rel_tol,
                                              int32_t max_rank, gingr_model** out, int32_t* rank_out);
/* The mirror-symmetric Gaussian (mixture) model: scalismo's symmetrised kernel about the plane x = 0 (the tutorial's
 * "XmirroredKernel"), with S = diag(-1, 1, 1), k the scalar mixture above and k_m(x, y) = k(S x, y):
 *   K(x, y) = DiagonalKernel(k, 3) + DiagonalKernel(-k_m, k_m, k_m)
 *           = diag(k(x, y) - k(S x, y),  k(x, y) + k(S x, y),  k(x, y) + k(S x, y)).
 * Left and right halves of the template deform as mirror images, and points on the plane do not move off it (their
 * x rows of the basis are exactly zero).  The plane is fixed at x = 0: the caller centres the template on it.
 * Arguments, validation, stopping rule and outputs are those of gingr_gpmm_gaussian_mixture. */
GINGR_API int32_t gingr_gpmm_gaussian_symmetric(gingr_ctx* ctx, int32_t M, const double* ref_pts /*[3M]*/,
                                                const int32_t* tri /*[3T]*/, int32_t T, int32_t n_kernels,
                                                const double* sigma /*[n]*/, const double* scaling /*[n]*/, double rel_tol,
                                                int32_t max_rank, gingr_model** out, int32_t* rank_out);
/* The inverse-Laplacian model: the look-up kernel of the model chooser (api/gpmm LaplacianHelper.scala:26-55 with
 * MatrixHelper.pinv :23-26), the GP form of a mesh-graph stiffness term -- vertices close on the triangle graph move
 * together, vertices merely close in space do not.  This project's reading of that kernel (unit weights, the role of
 * gamma and the parameter names are not verified against the reference):
 *   L = D - A, the combinatorial graph Laplacian of the triangle edges (unit weights, each undirected edge once however
 *       many triangles share it, self-edges of degenerate triangles ignored);
 *   Ks = scaling (L + gamma I)^-1 for gamma > 0, and for gamma = 0 the pseudo-inverse scaling L^+ = scaling ((L + P)^-1 - P),
 *       P = sum_c 1_c 1_c^T / |c| over the connected components c of the edge graph (a vertex in no triangle is a component
 *       of its own);
 *   K = DiagonalKernel(Ks, 3) = Ks (x) I3, then approximateGPCholesky with the stopping rule and outputs of
 *       gingr_gpmm_gaussian_mixture; the mean is zero.
 * Ks is formed densely on the device, so M <= 6000 (GINGR_ERR_UNSUPPORTED above).  Its spectrum decays like 1/k: at
 * rel_tol 0.01 the rank is about 0.97-0.99 of 3M, and the registrations take rank <= 9472 (about M <= 3200 at rel_tol 0.01):
 * larger templates want max_rank.  With gamma = 0 the kernel has rank 3 (M - #components): at rel_tol = 0 the
 * factorisation goes on past that rank and takes up to 3 * #components more columns from the rounding-level residual of
 * the null space, so a full-rank gamma = 0 model wants a small positive rel_tol (1e-12 suffices).  Requires T > 0,
 * indices in [0, M), scaling > 0 and gamma >= 0 finite, rel_tol >= 0, max_rank >= 0 and a single-GPU context.  Returns GINGR_MODEL_FLEXIBILITY with *out = NULL when L + gamma I is not
 * numerically positive definite (a gamma far below the rounding of L) or Ks is not finite. */
GINGR_API int32_t gingr_gpmm_inverse_laplacian(gingr_ctx* ctx, int32_t M, const double* ref_pts /*[3M]*/,
                                               const int32_t* tri /*[3T]*/, int32_t T, double scaling, double gamma,
                                               double rel_tol, int32_t max_rank, gingr_model** out, int32_t* rank_out);
/* The model as scalismo stores it (SURVEY.md A1): meanVector, basisMatrix column-major with leading dimension ld_basis,
 * variance.  Any output may be NULL (M_out / r_out give the sizes to allocate). */
GINGR_API int32_t gingr_model_download(gingr_ctx* ctx, const gingr_model* model, int32_t* M_out, int32_t* r_out,
                                       double* ref_pts /*[3M]*/, double* mean /*[3M]*/, double* basis, int64_t ld_basis,
                                       double* variance /*[r]*/);
GINGR_API int32_t gingr_target_upload(gingr_ctx* ctx, int32_t N, const double* pts /*[3N]*/,
                                      const int32_t* tri /*[3T]*/, int32_t T, gingr_target** out);
GINGR_API int32_t gingr_target_destroy(gingr_target* t);

/* ---- K1: CPD / BCPD E-step ------------------------------------------------------------------- */
/* Replaces CpdRegistrationState.P (CPD.scala:54-75) + its reductions: P1 = sum(P,Axis._1)
 * (CPD.scala:36, :122, :139), Pt1 = sum(P,Axis._0) (:140), PX = P*X (:145).  P is never
 * materialised.  Any output pointer may be NULL. */
GINGR_API int32_t gingr_cpd_estep(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* fit /*[3M]*/,
                                  double sigma2, double w, double* P1 /*[M]*/, double* Pt1 /*[N]*/,
                                  double* PX /*[3M]*/);
/* Replaces BCPD.computeP + the P reductions of BCPD.Iteration
 * (other/algorithms/cpd/BCPD.scala:167-184, :200-209); quirks of the reference kept. */
GINGR_API int32_t gingr_bcpd_estep(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* y /*[3M]*/,
                                   const double* sigma_mm /*[M]*/, const double* alpha /*[M]*/, double sigma2,
                                   double s, double w, double* nu /*[M]*/, double* nu_prime /*[N]*/,
                                   double* n_hat /*[1]*/, double* x_hat /*[3M]*/);
/* computeInitialSigma2 (CPD.scala:81-90): sum_ij |x_j - m_i|^2 / (3 N M). */
GINGR_API int32_t gingr_cpd_initial_sigma2(gingr_ctx* ctx, const gingr_target* target, int32_t M,
                                           const double* pts /*[3M]*/, double* sigma2_out);

/* ---- K2: ICP closest-point correspondence ---------------------------------------------------- */
/* Replaces closestPointCorrespondence of registration/utils/ClosestPointRegistrator.scala
 * (:74-96 triangular, :98-131 along normal, :133-160 point cloud).  `tpl` / `tpl_tri` are the template
 * (current fit) vertices and triangles.  Outputs per template vertex: idx = nearest target vertex id
 * (exact argmin, ties -> lowest index), cp = corresponding point, w = 0/1 robustness weight,
 * mean_distance = the second component of the reference's result. */
GINGR_API int32_t gingr_icp_closest(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* tpl /*[3M]*/,
                                    const int32_t* tpl_tri /*[3T]*/, int32_t T, int32_t method, int32_t* idx /*[M]*/,
                                    double* cp /*[3M]*/, uint8_t* w /*[M]*/, double* mean_distance /*[1]*/);
/* closestPointCorrespondenceReversal (ClosestPointRegistrator.scala:34-45): the search runs from every TARGET
 * vertex j to the template; outputs per target vertex: tpl_id = template.findClosestPoint(corresponding point).id,
 * w = the weight of that search.  The observation the reference forms is (tpl_id[j], target point j, w[j]). */
GINGR_API int32_t gingr_icp_closest_reversal(gingr_ctx* ctx, const gingr_target* target, int32_t M,
                                             const double* tpl /*[3M]*/, const int32_t* tpl_tri /*[3T]*/, int32_t T,
                                             int32_t method, int32_t* tpl_id /*[N]*/, uint8_t* w /*[N]*/,
                                             double* mean_distance /*[1]*/);

/* ---- K3: low-rank GPMM posterior ------------------------------------------------------------- */
/* Replaces model.transform(rigid).posterior(obs).mean (GingrAlgorithm.scala:297-301, :211;
 * scalismo regression, SURVEY.md A3): weighted Gram Q^T L^-1 Q + I on the FP64 tensor pipe,
 * Cholesky solve, mean evaluation at all M points.
 * R[9] row-major rotation about the origin, t[3]; n observations (pid, point); noise_kind 0:
 * noise[n] isotropic variances (cov_i = noise_i * I3), 1: noise[9n] full row-major covariances. */
GINGR_API int32_t gingr_posterior_mean(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t,
                                       int32_t n, const int32_t* pid, const double* points /*[3n]*/,
                                       int32_t noise_kind, const double* noise, double* coeffs /*[r]*/,
                                       double* mean_pts /*[3M]*/);
/* The COVARIANCE of the same posterior at the mesh points: scalismo's `posterior` (GingrAlgorithm.scala:300) returns a
 * model whose covariance helper/PosteriorHelper.scala:26-80 turns into per-vertex variance maps; here
 *   cov_i = R Phi_i D Mx^-1 D Phi_i^T R^T   (3 x 3, row-major, cov[9 i ..]),  Mx = Q^T L^-1 Q + I  as above,
 * evaluated exactly: the rows of Q = Phi D ride through the Cholesky factorisation as extra rows (Q_i L^-T), their
 * 3 x 3 Gram blocks are the covariances.  Same observation arguments as gingr_posterior_mean. */
GINGR_API int32_t gingr_posterior_covariance(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t,
                                             int32_t n, const int32_t* pid, const double* points /*[3n]*/,
                                             int32_t noise_kind, const double* noise, double* cov_pts /*[9M]*/);
/* scalismo model.transform(R, t).posterior(trainingData) (SURVEY.md A3; call site GingrAlgorithm.scala:299-300) as a
 * new model handle.  Observation arguments exactly as gingr_posterior_mean.  The new model: reference R ref_i + t with the
 * source model's triangles, mean R (mean_i + Phi_i D c) (c: the coefficients of gingr_posterior_mean, D = diag(sqrt(lambda))),
 * basis (I (x) R) Phi U, variance s in descending order (stable) with U diag(s) U^T = D Mx^-1 D.  Indices with variance 0 in
 * the source model keep the unit vector e_k and variance 0.  The basis is unique up to rotations inside degenerate
 * eigenspaces.  Returns GINGR_MODEL_FLEXIBILITY with *out = NULL for non-finite noise or a failed factorisation.
 * Single-GPU contexts only. */
GINGR_API int32_t gingr_model_posterior(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t,
                                        int32_t n, const int32_t* pid, const double* points /*[3n]*/, int32_t noise_kind,
                                        const double* noise, gingr_model** out);
/* Device times of the last posterior model built on the ctx (gingr_model_posterior, gingr_registration_posterior_model),
 * CUDA events in ms: [0] observations, system assembly and factorisation, [1] eigenpairs (Jacobi), [2] basis product,
 * [3] mean, reference and regression constants, [4] the whole call.  sweeps (may be NULL): Jacobi sweeps. */
GINGR_API int32_t gingr_posterior_model_profile(const gingr_ctx* ctx, double* ms /*[5]*/, int32_t* sweeps);
/* Replaces model.transform(rigid).coefficients(mesh) (GingrAlgorithm.scala:215, :236): regression on
 * all M points with noise 1e-5 * I3. */
GINGR_API int32_t gingr_coefficients(gingr_ctx* ctx, const gingr_model* model, const double* R, const double* t,
                                     const double* mesh_pts /*[3M]*/, double* coeffs /*[r]*/);
/* Kernel-level entry of the r x r solve inside the regression -- scalismo's `Minv = pinv(Mx); c = Minv * rhs`
 * (SURVEY.md A3; call sites GingrAlgorithm.scala:300, :215, :236) -- as the on-device Cholesky the iteration uses.
 * A[n*n] row-major symmetric positive definite (only the lower triangle is read); B[nrhs*n]: right-hand sides as rows.
 * Outputs (each may be NULL): L_out[n*n] the factor (lower, row-major, strict upper part zero); Y_out[nrhs*n] the rows
 * L^-1 b_q (forward substitution, carried through the factorisation); x_out[n] = A^-1 b_0 (needs nrhs >= 1).
 * reps >= 1 factorisations are run back to back on the same input; ms_out (may be NULL) receives the device time of
 * ONE factorisation + back substitution (CUDA events on the library's stream).
 * Returns GINGR_MODEL_FLEXIBILITY when A is not positive definite / not finite. */
GINGR_API int32_t gingr_spd_solve(gingr_ctx* ctx, int32_t n, const double* A, int32_t nrhs, const double* B,
                                  double* L_out, double* Y_out, double* x_out, int32_t reps, double* ms_out);
/* Replaces ModelFittingParameters.modelInstanceShapePoseScale (ModelFittingParameters.scala:130-143):
 * fit = s * (R * instance(alpha) + t). */
GINGR_API int32_t gingr_model_instance(gingr_ctx* ctx, const gingr_model* model, const gingr_state* st,
                                       const double* alpha /*[r]*/, double* fit /*[3M]*/);

/* ---- the full iteration ------------------------------------------------------------------------ */
GINGR_API int32_t gingr_registration_create(gingr_ctx* ctx, const gingr_model* model, const gingr_target* target,
                                            const gingr_config* cfg, gingr_registration** out);
GINGR_API int32_t gingr_registration_destroy(gingr_registration* reg);
/* GeneralRegistrationState.landmarkCorrespondences (GeneralRegistrationState.scala:43-62), already
 * resolved by the host: nearest reference vertex id, target landmark point, 3x3 row-major covariance. */
GINGR_API int32_t gingr_registration_set_landmarks(gingr_registration* reg, int32_t L, const int32_t* pid,
                                                   const double* points /*[3L]*/, const double* cov /*[9L]*/);
/* initializeState (CPD.scala:92-103 / ICP.scala:74-86): sets st->sigma2 (computeInitialSigma2 over
 * model.mean for CPD without initialSigma) and evaluates the initial fit. */
GINGR_API int32_t gingr_initialize_state(gingr_registration* reg, gingr_state* st /*in/out*/,
                                         const double* alpha /*[r]*/, double* fit_out /*[3M], may be NULL*/);
/* GingrAlgorithm.update (GingrAlgorithm.scala:192-254), followed by the
 * fit refresh of GingrGeneratorWrapper.propose (sampling/generators/GingrGeneratorWrapper.scala:28-39)
 * delivered in fit_out (state_out->iteration is NOT incremented here: that stays with `propose`).
 * state_out->status is GINGR_STATUS_MODEL_FLEXIBILITY_ERROR exactly where the reference's Try fails;
 * the function's own return value is then GINGR_OK (the state carries the failure, as in the reference).
 * probabilistic != 0: posterior.sample() replaces posterior.mean (:211).  The coefficients are drawn from
 * N(c, Minv) as c + L^-T z with z ~ N(0, I_r) from Philox4x32-10 (key = seed, counter = (pair, iteration, 0, 0)) +
 * Box-Muller: the same distribution as scalismo's SVD-rotated basis, not the same draws.  The retry counter of
 * GingrAlgorithm.scala:69-70, :197-202 lives in the registration handle. */
GINGR_API int32_t gingr_update(gingr_registration* reg, const gingr_state* state_in, const double* alpha_in /*[r]*/,
                               int32_t probabilistic, uint64_t seed, gingr_state* state_out,
                               double* alpha_out /*[r]*/, double* fit_out /*[3M], may be NULL*/);
/* Device-resident chaining for throughput runs: enqueue `iters` consecutive update+propose steps
 * starting from the state of the last gingr_update / gingr_initialize_state without host round trips. */
GINGR_API int32_t gingr_update_chain(gingr_registration* reg, int32_t iters);
/* The same with probabilistic = true in every step (a chain of informed posterior-sample proposals that are all
 * accepted, i.e. GeneratorWrapperStochastic.gingrPropose without the MH accept/reject of the caller). */
GINGR_API int32_t gingr_update_chain_sampled(gingr_registration* reg, int32_t iters, uint64_t seed);
/* Independent registrations / MCMC chains batched on one GPU (BASELINE config 5; SURVEY.md 8e "replicas only"):
 * `iters` update+propose steps of each of the n registrations (all created on the same ctx, typically sharing one
 * model and one target handle, each with its own device-resident state).  Chain k uses seed + k when
 * probabilistic != 0.  All chains advance through ONE batched kernel sequence per iteration (every kernel launched once
 * with blockIdx.z = chain; csrc/batch.cuh) when every launch of the iteration has a batched form -- CPD and the ICP flavours
 * on the scans do --, otherwise (uniform-grid searches of large meshes, the reversed correspondence direction) the chains'
 * captured iteration graphs are replayed on a pool of streams.  The call returns
 * after enqueueing, results are read with gingr_state_download per chain.  Per chain the arithmetic is that of the chain
 * alone, up to the summation order of its Gram partials when many chains share the GPU. */
GINGR_API int32_t gingr_update_batch(gingr_registration** regs, int32_t n, int32_t iters, int32_t probabilistic,
                                     uint64_t seed);
/* Read back the device-resident state after gingr_update_chain / gingr_update_batch. */
GINGR_API int32_t gingr_state_download(gingr_registration* reg, gingr_state* state_out, double* alpha_out,
                                       double* fit_out);

/* GingrAlgorithm.computePosterior(current) (GingrAlgorithm.scala:281-302): the correspondences and uncertainties of the
 * registration's configuration (CPD E-step / ICP flavours, landmarks) at `state`, then the posterior model as
 * gingr_model_posterior builds it.  The device-resident state is replaced (the next gingr_update uploads its own). */
GINGR_API int32_t gingr_registration_posterior_model(gingr_registration* reg, const gingr_state* state,
                                                     const double* alpha /*[r]*/, gingr_model** out);

/* ---- probabilistic registration: Metropolis-Hastings with the informed GiNGR proposal (SURVEY.md 8f item 1) ---- */
/* sampling/evaluators/IndependentPointDistanceEvaluator.scala:26-32 EvaluationMode */
#define GINGR_EVAL_MODEL_TO_TARGET 0
#define GINGR_EVAL_TARGET_TO_MODEL 1
#define GINGR_EVAL_SYMMETRIC 2
/* POD mirror of ProbabilisticSettings(IndependentPoints(state, uncertainty, mode, evaluatedPoints), randomMixture)
 * (GingrAlgorithm.scala:40-50, sampling/Evaluator.scala:43-60) and of the defaults of Generator.DefaultRandom
 * (sampling/Generator.scala:27-83). */
typedef struct gingr_mcmc_settings {
  double random_mixture;   /* weight of the random generators in MixtureProposal(rm *: random + (1 - rm) *: informed) */
  double uncertainty;      /* sdev of the Gaussian point-distance likelihood */
  int32_t evaluation_mode; /* GINGR_EVAL_* */
  int32_t reserved;
  double rot_sdev[3];      /* yaw (psi), pitch (theta), roll (phi); Generator.defaultRotation = 0.01 */
  double trans_sdev[3];    /* x, y, z; Generator.defaultTranslation = 0.1 */
  double shape_sdev[3];    /* RandomShape steps; default 1.0, 0.1, 0.01 */
} gingr_mcmc_settings;
/* Attach the probabilistic settings to a registration.  model_ids / target_ids: the comparison points of the distance
 * evaluator (numberOfPointsForComparison; the reference decimates, the host passes the ids it wants), n = 0: all. */
GINGR_API int32_t gingr_mcmc_configure(gingr_registration* reg, const gingr_mcmc_settings* settings,
                                       const int32_t* model_ids, int32_t n_model_ids, const int32_t* target_ids,
                                       int32_t n_target_ids);
/* EvaluatorWrapper.logValue of a state (sampling/evaluators/EvaluatorWrapper.scala:23-33): out[0] = ModelEvaluator
 * (ModelEvaluator.scala:25-32), out[1] = IndependentPointDistanceEvaluator (:54-78); the product evaluator is their sum. */
GINGR_API int32_t gingr_evaluate_log_value(gingr_registration* reg, const gingr_state* state, const double* alpha,
                                           double* out /*[2]*/);
/* GeneratorWrapperStochastic.logTransitionProbability(from, to) (GeneratorWrapperStochastic.scala:42-63): log density of
 * the informed proposal; -inf where the reference returns Double.NegativeInfinity. */
GINGR_API int32_t gingr_log_transition_probability(gingr_registration* reg, const gingr_state* from,
                                                   const double* from_alpha, const gingr_state* to,
                                                   const double* to_alpha, double* out /*[1]*/);
/* `iters` steps of scalismo's MetropolisHastings (SURVEY.md A5) with generatorCombined (GingrAlgorithm.scala:177-190) and
 * the evaluators above, starting at the device-resident state, entirely on the device: choice of the generator, informed
 * or random proposal, posterior of the proposal (kept when accepted), both transition densities of the mixture, accept /
 * reject, best-sample tracking.  Random numbers: Philox4x32-10, key = seed, counter = (index, MH step, purpose, 0). */
GINGR_API int32_t gingr_mcmc_chain(gingr_registration* reg, int32_t iters, uint64_t seed);
/* Independent chains batched on one GPU (BASELINE config 5); chain k uses seed + k.  One batched kernel sequence per MH
 * step serves all chains (see gingr_update_batch); a step with a launch that has no batched form falls back to per-chain
 * step graphs. */
GINGR_API int32_t gingr_mcmc_batch(gingr_registration** regs, int32_t n, int32_t iters, uint64_t seed);
/* values[16] / counts[32]: see mcmc.cuh (log values of current / proposal / best, transition densities, accept counts per
 * generator). */
GINGR_API int32_t gingr_mcmc_stats(gingr_registration* reg, double* values /*[16]*/, int32_t* counts /*[32]*/);
/* BestAndCurrentSampleLogger.currentBestSample (GingrAlgorithm.scala:160-163). */
GINGR_API int32_t gingr_mcmc_best(gingr_registration* reg, gingr_state* state_out, double* alpha_out, double* fit_out);

/* ---- measurement hooks (new; used by bench.py for the roofline numbers) ------------------------ */
/* Per-phase device timing with CUDA events recorded on the ctx stream around the kernels of gingr_update /
 * gingr_update_chain.  ms[8]: 0 = E-step sweep A kernels, 1 = E-step sweep B kernels (each with its cull kernels), 2 = Gram (DMMA) kernel,
 * 3 = Cholesky + back substitution, 4 = whole iteration, 5 = closest-point search (ICP), 6 and 7 = CPD: live fraction
 * of the tile pairs of sweep A / B (1 when nothing was culled; not a time).  Values are sums over `iterations` iterations since the last
 * call (the call synchronises the stream and resets the counters). */
GINGR_API int32_t gingr_registration_set_profiling(gingr_registration* reg, int32_t enable);
GINGR_API int32_t gingr_registration_get_profile(gingr_registration* reg, double* ms /*[8]*/, int32_t* iterations);

#ifdef __cplusplus
}
#endif
#endif /* GINGR_CUDA_H */
