// mcmc.cuh -- the probabilistic registration step on the device (included by update.cu; SURVEY.md 8f item 1).
//
// Replaces, for one chain, what the reference runs on the JVM around `update(current, probabilistic = true)`:
//   GeneratorWrapperStochastic.logTransitionProbability   sampling/generators/GeneratorWrapperStochastic.scala:42-63
//   the random pose / shape proposals                     RandomPoseUpdateProposal.scala:30-111,
//                                                         RandomShapeUpdateProposal.scala:23-51,
//                                                         GaussianDenseVectorProposal.scala:25-42
//   the mixture of generators                             Generator.scala:31-83, GingrAlgorithm.scala:177-190
//   the evaluators                                        ModelEvaluator.scala:25-32,
//                                                         IndependentPointDistanceEvaluator.scala:54-78, Evaluator.scala:43-60
//   the accept / reject of scalismo's MetropolisHastings  (SURVEY.md A5) and BestAndCurrentSampleLogger
//
// logTransitionProbability without the SVD.  The reference projects `toMesh` on the POSTERIOR model of `from`
// (mean' + Phi' D c, basis Phi' U_s, variance s with U_s diag(s) U_s^T = A = D Mx^-1 D) by a regression with noise
// eps = 1e-5 and takes the N(0, I) log density of the coefficients c'.  With K = U_s sqrt(s) (K K^T = A):
//     c' = (K^T G K + eps I)^-1 K^T Phi'^T resid = K^T (G A + eps I)^-1 b ,   G = Phi^T Phi,  b = Phi'^T resid
//     |c'|^2 = b^T (A G + eps I)^-1 A (G A + eps I)^-1 b
// and with the substitution w = D u:   (S + eps Mx) u = D b ,   |c'|^2 = u^T Mx u ,   S = D G D  (the model constant
// of the `coefficients` regression).  One r x r Cholesky of S + eps Mx and a quadratic form: no SVD, no division by
// lambda, and every piece is an existing kernel.  (tests/test_mcmc_gpu.py compares with the literal SVD form.)
//
// Random numbers: Philox4x32-10 keyed by the chain's seed, counter = (index, MH step, purpose, 0):
//   purpose 0  posterior.sample() normals (pairs, as in gingr_update)      purpose 1  index 0: (u_choice, u_accept)
//   purpose 2  perturbation normals of the random proposals (pairs)
// The same distributions as the reference's scalismo / Breeze generators, not the same draws; the oracle consumes the
// identical stream, so device and oracle chains can be compared step by step.
//
// One MH step is a fixed kernel sequence (captured as a CUDA graph): the informed proposal is always computed and the
// chosen random leaf overrides it, both directions of the informed transition density are evaluated, and the
// accept / reject is a set of flag-conditioned copies -- no host round trip inside a chain.
#pragma once

namespace gingr {

enum { LEAF_INFORMED = 0, LEAF_ROT_YAW = 1, LEAF_ROT_PITCH = 2, LEAF_ROT_ROLL = 3, LEAF_TRANS_X = 4, LEAF_TRANS_Y = 5,
       LEAF_TRANS_Z = 6, LEAF_SHAPE_0 = 7, LEAF_SHAPE_1 = 8, LEAF_SHAPE_2 = 9, LEAF_COUNT = 10 };
// doubles of the chain
enum { MD_LP_CUR = 0 /*prior, distance*/, MD_LP_PROP = 2, MD_TINF_FW = 4, MD_TINF_BW = 5, MD_U_ACCEPT = 6, MD_A = 7,
       MD_LP_BEST = 8, MD_FW = 9, MD_BW = 10, MD_TINF_CUR = 11 /*informed density of the current state (stepLength = 1)*/,
       MD_COUNT = 16 };
// ints of the chain
enum { MI_STEP = 0, MI_LEAF = 1, MI_ACCEPT = 2, MI_ACCEPTED = 3, MI_BEST_UPDATED = 4, MI_NAN = 5, MI_INFO2 = 6,
       MI_PROPOSED = 8 /*[LEAF_COUNT]*/, MI_ACCEPTED_LEAF = 18 /*[LEAF_COUNT]*/, MI_COUNT = 32 };

constexpr double LOG_2PI = 1.8378770664093454835606594728112;

__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6) + 0.5) * (1.0 / 9007199254740992.0);
}

// normal number `idx` of the (step, purpose) stream (Box-Muller pairs)
__device__ __forceinline__ double philox_normal(uint64_t seed, uint32_t step, uint32_t purpose, int idx) {
  uint32_t x[4];
  philox4x32_10((uint32_t)(idx >> 1), step, purpose, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), x);
  const double rad = sqrt(-2.0 * log(u53(x[0], x[1])));
  const double ang = 6.283185307179586476925 * u53(x[2], x[3]);
  return (idx & 1) ? rad * sin(ang) : rad * cos(ang);
}

struct McmcDev {
  double rho;            // randomMixture
  double sd[9];          // yaw, pitch, roll, x, y, z, shape steps
};

__host__ __device__ inline void leaf_weights(double rho, double* w) {
  // MixtureProposal(rho *: DefaultRandom + (1 - rho) *: informed), DefaultRandom = 0.5 pose + 0.5 shape, pose = 0.5
  // rotation (3 axes, equal) + 0.5 translation (3 axes, equal), shape = 3 steps, equal.  Generator.scala:31-83
  w[LEAF_INFORMED] = 1.0 - rho;
  for (int k = 0; k < 3; ++k) {
    w[LEAF_ROT_YAW + k] = rho * 0.5 * 0.5 / 3.0;
    w[LEAF_TRANS_X + k] = rho * 0.5 * 0.5 / 3.0;
    w[LEAF_SHAPE_0 + k] = rho * 0.5 / 3.0;
  }
}

// the Euler angle a rotation leaf perturbs: YawAxis -> psi, PitchAxis -> theta, RollAxis -> phi
// (RandomPoseUpdateProposal.scala:40-44); DS_EULER holds (phi, theta, psi)
__host__ __device__ inline int leaf_euler_slot(int leaf) { return leaf == LEAF_ROT_YAW ? 2 : leaf == LEAF_ROT_PITCH ? 1 : 0; }

// which generator of the mixture proposes (flattened leaves, Generator.scala:31-83) and the uniform of the accept test
__device__ void mcmc_choose(const McmcDev& p, uint64_t seed, int* __restrict__ mi, double* __restrict__ md) {
  uint32_t x[4];
  philox4x32_10(0u, (uint32_t)mi[MI_STEP], 1u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), x);
  const double uc = u53(x[0], x[1]);
  md[MD_U_ACCEPT] = u53(x[2], x[3]);
  double w[LEAF_COUNT];
  leaf_weights(p.rho, w);
  int leaf = LEAF_COUNT - 1;
  double acc = 0.0;
  for (int k = 0; k < LEAF_COUNT; ++k) {
    acc += w[k];
    if (uc < acc) { leaf = k; break; }
  }
  if (w[leaf] <= 0.0) leaf = LEAF_INFORMED;   // rounding at the upper end with rho = 0
  mi[MI_LEAF] = leaf;
  mi[MI_PROPOSED + leaf] += 1;
}

// the chosen random leaf replaces the informed proposal: all parameters of the current state (snapshot) with one
// Gaussian perturbation; sigma2 and status are those of the current state (the random generators do not touch them)
GINGR_KERNEL((256), mcmc_random_override_kernel, const McmcDev& p, uint64_t seed, int r, const int* __restrict__ mi,
                                                                   const double* __restrict__ s_ds, const int* __restrict__ s_is,
                                                                   const double* __restrict__ s_alpha, double* __restrict__ ds,
                                                                   int* __restrict__ is, double* __restrict__ alpha,
                                                                   int* mi_rw, double* __restrict__ md) {
  if (threadIdx.x == 0) mcmc_choose(p, seed, mi_rw, md);   // the informed update before this kernel does not depend on it
  __syncthreads();
  const int leaf = mi_rw[MI_LEAF];
  const uint32_t step = (uint32_t)mi_rw[MI_STEP];
  if (leaf != LEAF_INFORMED) {
    if (threadIdx.x == 0) {
      ds[DS_SCALE] = s_ds[DS_SCALE];
      for (int d = 0; d < 3; ++d) { ds[DS_T + d] = s_ds[DS_T + d]; ds[DS_EULER + d] = s_ds[DS_EULER + d]; }
      ds[DS_SIGMA2] = s_ds[DS_SIGMA2];
      is[IS_STATUS] = s_is[IS_STATUS];
      is[IS_RETRY] = s_is[IS_RETRY];   // update() is not called for a random proposal: its retry bookkeeping is undone
      if (leaf >= LEAF_ROT_YAW && leaf <= LEAF_ROT_ROLL)
        ds[DS_EULER + leaf_euler_slot(leaf)] += p.sd[leaf - LEAF_ROT_YAW] * philox_normal(seed, step, 2u, 0);
      else if (leaf >= LEAF_TRANS_X && leaf <= LEAF_TRANS_Z)
        ds[DS_T + (leaf - LEAF_TRANS_X)] += p.sd[3 + leaf - LEAF_TRANS_X] * philox_normal(seed, step, 2u, 0);
    }
    const double sdev = leaf >= LEAF_SHAPE_0 ? p.sd[6 + leaf - LEAF_SHAPE_0] : 0.0;
    for (int a = threadIdx.x; a < r; a += blockDim.x)
      alpha[a] = s_alpha[a] + (leaf >= LEAF_SHAPE_0 ? sdev * philox_normal(seed, step, 2u, a) : 0.0);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    euler_to_matrix_dev(ds[DS_EULER], ds[DS_EULER + 1], ds[DS_EULER + 2], ds + DS_R2);
    is[IS_ITER] = s_is[IS_ITER] + 1;   // GingrGeneratorWrapper.propose: updateIteration()
  }
}

// ---- evaluators ---------------------------------------------------------------------------------------------
GINGR_KERNEL_NB(gather_aos_kernel, int n, const int32_t* __restrict__ ids, const double* __restrict__ src, double* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int j = ids ? ids[i] : i;
  dst[3 * i] = src[3 * j]; dst[3 * i + 1] = src[3 * j + 1]; dst[3 * i + 2] = src[3 * j + 2];
}

// sum_i logPdf_{N(0, sd)}(sqrt(d2_i)) = sum_i (-d2_i / (2 sd^2) - log(sd sqrt(2 pi)))   (Breeze Gaussian.logPdf);
// one block, fixed-order tree; out[0] (accumulate ? += : =) weight * sum
GINGR_KERNEL((256), mcmc_distance_logpdf_kernel, int n, const double* __restrict__ d2, double sd, double weight,
                                                                   int accumulate, double* __restrict__ out, int r,
                                                                   const double* __restrict__ alpha /*null: no prior*/) {
  __shared__ double red[256];
  if (alpha) {   // ModelEvaluator of the same state in the same launch: out[-1] = log N(alpha; 0, I_r)
    double sa = 0.0;
    for (int a = threadIdx.x; a < r; a += 256) sa += alpha[a] * alpha[a];
    red[threadIdx.x] = sa;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) out[-1] = -0.5 * red[0] - 0.5 * (double)r * LOG_2PI;
    __syncthreads();
  }
  const double lognorm = log(sd * 2.5066282746310005024157652848110);
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) {
    const double dist = sqrt(d2[i]);   // (closestPointOnSurface(pt).point - pt).norm
    s += -(dist * dist) / (2.0 * sd * sd) - lognorm;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (accumulate ? out[0] : 0.0) + weight * red[0];
}

// ---- informed transition density ---------------------------------------------------------------------------------
// u_i = R^T (mesh_i - t) - ref_i - mean_i     (residual of `mesh` against the posed model mean, rotated back)
GINGR_KERNEL_NB(mcmc_residual_kernel, int M, const double* __restrict__ mesh, const double* __restrict__ ref,
                                     const double* __restrict__ mean, const double* __restrict__ R, const double* __restrict__ t,
                                     double* __restrict__ u) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const double x = mesh[3 * i] - t[0], y = mesh[3 * i + 1] - t[1], z = mesh[3 * i + 2] - t[2];
  u[3 * i] = R[0] * x + R[3] * y + R[6] * z - ref[3 * i] - mean[3 * i];
  u[3 * i + 1] = R[1] * x + R[4] * y + R[7] * z - ref[3 * i + 1] - mean[3 * i + 1];
  u[3 * i + 2] = R[2] * x + R[5] * y + R[8] * z - ref[3 * i + 2] - mean[3 * i + 2];
}

// B[a][b] = S[a][b] + eps * Mx[a][b] (a, b < r);  row r: rhs = b_proj - S c
GINGR_KERNEL_NB(mcmc_build_system_kernel, int r, int rp, const double* __restrict__ S, const double* __restrict__ Mx, double eps,
                                         const double* __restrict__ bproj, const double* __restrict__ Sc, double* __restrict__ B,
                                         int* __restrict__ info2) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e == 0) info2[0] = 0;   // the factorisation that follows reports a failed pivot here
  if (e >= (r + 1) * rp) return;
  const int a = e / rp, b = e % rp;
  if (a < r) B[e] = b < r ? S[(size_t)a * rp + b] + eps * Mx[(size_t)a * rp + b] : 0.0;
  else B[e] = b < r ? bproj[b] - Sc[b] : 0.0;
}

// out = -0.5 u^T (Mx u) - r/2 log(2 pi), or -inf when the posterior of `from` failed / the solve failed / not finite
// (GeneratorWrapperStochastic.scala:44-45, :58-60)
GINGR_KERNEL((256), mcmc_quadform_kernel, int r, const double* __restrict__ u, const double* __restrict__ Mxu,
                                                            const int* __restrict__ from_is, const int* __restrict__ info2,
                                                            double* __restrict__ out) {
  __shared__ double red[256];
  double s = 0.0;
  for (int a = threadIdx.x; a < r; a += 256) s += u[a] * Mxu[a];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double v = -0.5 * red[0] - 0.5 * (double)r * LOG_2PI;
    if (from_is[IS_INFO] != 0 || from_is[IS_FAIL_POST] != 0 || info2[0] != 0 || !(fabs(v) < INFINITY)) v = -INFINITY;
    out[0] = v;
  }
}

// alpha_comp = from + (to - from) / stepLength   (GeneratorWrapperStochastic.scala:48-50)
GINGR_KERNEL_NB(mcmc_compensate_kernel, int r, const double* __restrict__ from, const double* __restrict__ to, double step,
                                       double* __restrict__ out) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a < r) out[a] = from[a] + (to[a] - from[a]) / step;
}

// ---- decision -------------------------------------------------------------------------------------------------
__device__ __forceinline__ double gauss_logpdf(double x, double sd) {   // Breeze Gaussian(0, sd).logPdf / GaussianEvaluator.logDensity
  return -(x * x) / (2.0 * sd * sd) - log(sd * 2.5066282746310005024157652848110);
}

// log sum_k w_k exp(t_k) of the flattened mixture for the move a -> b (scalismo MixtureProposal.logTransitionProbability)
__device__ double mixture_log_transition(const McmcDev& p, int r, const double* a_ds, const double* a_alpha, const double* b_ds,
                                         const double* b_alpha, double t_informed, double shape_ss /*sum (b-a)^2*/,
                                         bool shape_equal) {
  double w[LEAF_COUNT];
  leaf_weights(p.rho, w);
  const bool scale_eq = a_ds[DS_SCALE] == b_ds[DS_SCALE];
  const bool trans_eq = a_ds[DS_T] == b_ds[DS_T] && a_ds[DS_T + 1] == b_ds[DS_T + 1] && a_ds[DS_T + 2] == b_ds[DS_T + 2];
  const bool rot_eq = a_ds[DS_EULER] == b_ds[DS_EULER] && a_ds[DS_EULER + 1] == b_ds[DS_EULER + 1] && a_ds[DS_EULER + 2] == b_ds[DS_EULER + 2];
  double s = w[LEAF_INFORMED] * exp(t_informed);
  for (int k = 0; k < 3; ++k) {
    if (scale_eq && trans_eq && shape_equal) {   // only the rotation may differ (RandomPoseUpdateProposal.scala:50-56)
      const int slot = leaf_euler_slot(LEAF_ROT_YAW + k);
      s += w[LEAF_ROT_YAW + k] * exp(gauss_logpdf(b_ds[DS_EULER + slot] - a_ds[DS_EULER + slot], p.sd[k]));
    }
    if (scale_eq && rot_eq && shape_equal)       // only the translation may differ (:96-102)
      s += w[LEAF_TRANS_X + k] * exp(gauss_logpdf(b_ds[DS_T + k] - a_ds[DS_T + k], p.sd[3 + k]));
    if (scale_eq && rot_eq && trans_eq) {        // only the shape may differ (RandomShapeUpdateProposal.scala:42-50)
      const double sd = p.sd[6 + k];
      s += w[LEAF_SHAPE_0 + k] * exp(-shape_ss / (2.0 * sd * sd) - (double)r * log(sd * 2.5066282746310005024157652848110));
    }
  }
  return log(s);
}

GINGR_KERNEL((256), mcmc_decide_kernel, const McmcDev& p, int r, int fw_cached, const double* __restrict__ s_ds, const int* __restrict__ s_is,
                                                          const double* __restrict__ s_alpha, const double* __restrict__ ds,
                                                          const double* __restrict__ alpha, double* __restrict__ md,
                                                          int* __restrict__ mi) {
  __shared__ double red[256];
  __shared__ int neq[256];
  double ss = 0.0;
  int ne = 0;
  for (int a = threadIdx.x; a < r; a += 256) {
    const double d = alpha[a] - s_alpha[a];
    ss += d * d;
    ne += (alpha[a] != s_alpha[a]);
  }
  red[threadIdx.x] = ss;
  neq[threadIdx.x] = ne;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) { red[threadIdx.x] += red[threadIdx.x + o]; neq[threadIdx.x] += neq[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  const bool shape_equal = neq[0] == 0;
  // stepLength = 1: logTransitionProbability(from, to) only looks at `from` (its fit projected on its own posterior), so
  // the density of the current state is the one computed when it was proposed (scalismo memoises the posterior alike)
  if (fw_cached) md[MD_TINF_FW] = md[MD_TINF_CUR];
  const double fw = mixture_log_transition(p, r, s_ds, s_alpha, ds, alpha, md[MD_TINF_FW], red[0], shape_equal);
  const double bw = mixture_log_transition(p, r, ds, alpha, s_ds, s_alpha, md[MD_TINF_BW], red[0], shape_equal);
  md[MD_FW] = fw;
  md[MD_BW] = bw;
  const double lp_cur = md[MD_LP_CUR] + md[MD_LP_CUR + 1], lp_prop = md[MD_LP_PROP] + md[MD_LP_PROP + 1];
  int accept = 0;
  if (s_is[IS_STATUS] == GINGR_STATUS_MODEL_FLEXIBILITY_ERROR) {
    accept = 0;   // the reference stops the chain at a ModelFlexibilityError state (GingrAlgorithm.scala:150-153)
  } else if (fw != fw || bw != bw) {
    mi[MI_NAN] += 1;   // scalismo throws "NaN transition Probability!": counted, proposal dropped
  } else {
    const double ratio = (fw == -INFINITY || bw == -INFINITY) ? -INFINITY : fw - bw;   // SURVEY.md A5
    const double a = lp_prop - lp_cur - ratio;
    md[MD_A] = a;
    accept = (a > 0.0 || md[MD_U_ACCEPT] < exp(a)) ? 1 : 0;
  }
  mi[MI_ACCEPT] = accept;
  if (accept) {
    mi[MI_ACCEPTED] += 1;
    mi[MI_ACCEPTED_LEAF + mi[MI_LEAF]] += 1;
    md[MD_LP_CUR] = md[MD_LP_PROP];
    md[MD_LP_CUR + 1] = md[MD_LP_PROP + 1];
    md[MD_TINF_CUR] = md[MD_TINF_BW];
  }
  // BestAndCurrentSampleLogger: the chain state of this iteration (proposal if accepted, else current) vs the best
  const double lp_now = accept ? lp_prop : lp_cur;
  const int better = lp_now > md[MD_LP_BEST] ? 1 : 0;
  mi[MI_BEST_UPDATED] = better && accept;   // a rejected step leaves the (already logged) current state
  if (better) md[MD_LP_BEST] = lp_now;
  mi[MI_STEP] += 1;
}

// Several (conditional) copies in one launch: the replay rate of a chain's step graph is bound by its node count
// (profiles/r02_small_problems.md), so the snapshot and the accept / reject / best-sample copies are one node each.
// Segment q copies n 8-byte words when (flag == nullptr) or ((*flag != 0) == when).
struct CopySegments {
  static constexpr int MAXSEG = 12;
  int count = 0;
  const int* flag[MAXSEG];
  int when[MAXSEG];
  double* dst[MAXSEG];
  const double* src[MAXSEG];
  unsigned long long n[MAXSEG];
  void add(const int* f, int w, void* d, const void* s_, size_t words) {
    flag[count] = f; when[count] = w; dst[count] = (double*)d; src[count] = (const double*)s_; n[count] = words; ++count;
  }
};

GINGR_KERNEL((256), multi_copy_kernel, const CopySegments& seg) {
  for (int q = 0; q < seg.count; ++q) {
    if (seg.flag[q] && ((*seg.flag[q] != 0) != (seg.when[q] != 0))) continue;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < seg.n[q]; i += (size_t)gridDim.x * 256) seg.dst[q][i] = seg.src[q][i];
  }
}

template <typename T>
__global__ void cond_copy_kernel(const int* __restrict__ flag, int when, T* __restrict__ dst, const T* __restrict__ src, size_t n) {
  if ((*flag != 0) != (when != 0)) return;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

// on reject the working state returns to the snapshot, except the retry counter, which belongs to the algorithm
// instance and not to the state (GingrAlgorithm.scala:70)
// ... and the best sample's int block when the accepted proposal is the new best (one launch for both int blocks)
GINGR_KERNEL_NB(mcmc_restore_ints_kernel, const int* __restrict__ flag, int* __restrict__ is, const int* __restrict__ s_is,
                                         const int* __restrict__ best_flag, int* __restrict__ best_is) {
  if (*flag == 0) {
    for (int k = 0; k < IS_COUNT; ++k)
      if (k != IS_RETRY) is[k] = s_is[k];
  }
  if (*best_flag != 0)
    for (int k = 0; k < IS_COUNT; ++k) best_is[k] = is[k];
}

// ---- sample collection: LogHelper.samplesFromLog (LogHelper.scala:29-43) and the moments behind
// PosteriorHelper.computeDistanceMapFromMeshes* (PosteriorHelper.scala:31-79), accumulated on the device ---------------
// Per vertex ACC_WORDS doubles: [0, 3) mean fit position, [3, 9) scatter sum (x - mean)(x - mean)^T as xx xy xz yy yz zz,
// [9, 12) sum of the unit vertex normals of the collected fits; the sample count per vertex beside them.  The products
// feeding sums are rounded one by one (no FMA contraction), so that tests/test_mcmc_samples_host.py restates them in numpy.
constexpr int ACC_WORDS = 12;
__device__ __constant__ const int SCATTER_ROW[6] = {0, 0, 0, 1, 1, 2}, SCATTER_COL[6] = {0, 1, 2, 1, 2, 2};

// vertex_normals_kernel (closest.cu) for one vertex: the normalised mean of the unit normals of the adjacent triangles
__device__ __forceinline__ void vertex_normal_rn(int i, const double* __restrict__ v, const int32_t* __restrict__ tri,
                                                 const int32_t* __restrict__ adj_off, const int32_t* __restrict__ adj, double* nrm) {
  double ax = 0, ay = 0, az = 0;
  const int b = adj_off[i], e = adj_off[i + 1];
  for (int k = b; k < e; ++k) {
    const int t = adj[k];
    const double* a = v + 3 * tri[3 * t];
    const double* bb = v + 3 * tri[3 * t + 1];
    const double* c = v + 3 * tri[3 * t + 2];
    const double ux = bb[0] - a[0], uy = bb[1] - a[1], uz = bb[2] - a[2];
    const double wx = c[0] - a[0], wy = c[1] - a[1], wz = c[2] - a[2];
    double nx = __dsub_rn(__dmul_rn(uy, wz), __dmul_rn(uz, wy));
    double ny = __dsub_rn(__dmul_rn(uz, wx), __dmul_rn(ux, wz));
    double nz = __dsub_rn(__dmul_rn(ux, wy), __dmul_rn(uy, wx));
    const double len = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny)), __dmul_rn(nz, nz)));
    nx /= len; ny /= len; nz /= len;
    ax += nx; ay += ny; az += nz;
  }
  const int cnt = e - b;
  if (cnt > 0) { ax /= cnt; ay /= cnt; az /= cnt; }
  const double len = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az)));
  nrm[0] = ax / len; nrm[1] = ay / len; nrm[2] = az / len;
}

// Chain state i = mi[MI_STEP] (0: the primed start state, i >= 1: the state after the i-th MH step, in the working
// buffers) is collected when i >= burn_in, (i - burn_in) % every == 0, i < total and the state before it (prev_is, null
// for i = 0) is not a ModelFlexibilityError state.  Every thread decides from values no thread of the launch writes, so a
// step that collects nothing is one early-exiting launch.  Welford update in FP64; tri = null: no normals (no triangles).
GINGR_KERNEL((256), mcmc_collect_kernel, int M, const int* __restrict__ mi, const int* __restrict__ prev_is, int burn_in,
                                         int every, int total, const double* __restrict__ fit, const int32_t* __restrict__ tri,
                                         const int32_t* __restrict__ adj_off, const int32_t* __restrict__ adj,
                                         double* __restrict__ acc, long long* __restrict__ cnt) {
  const int i = mi[MI_STEP];
  if (i < burn_in || i >= total || (i - burn_in) % every != 0) return;
  if (prev_is && prev_is[IS_STATUS] == GINGR_STATUS_MODEL_FLEXIBILITY_ERROR) return;
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const long long n = cnt[m] + 1;
  cnt[m] = n;
  double* a = acc + (size_t)ACC_WORDS * m;
  double d[3], e[3];
  for (int k = 0; k < 3; ++k) {
    const double x = fit[3 * (size_t)m + k];
    d[k] = x - a[k];
    a[k] = a[k] + d[k] / (double)n;
    e[k] = x - a[k];
  }
  for (int q = 0; q < 6; ++q) a[3 + q] = __dadd_rn(a[3 + q], __dmul_rn(d[SCATTER_ROW[q]], e[SCATTER_COL[q]]));
  if (tri) {
    double nrm[3];
    vertex_normal_rn(m, fit, tri, adj_off, adj, nrm);
    for (int k = 0; k < 3; ++k) a[9 + k] += nrm[k];
  }
}

// gingr_mcmc_samples: the statistics of n chains pooled with Chan et al.'s pairwise formula in the order of the chains,
// one thread per vertex.  Outputs: mean [3M], covariance S / (n - 1) [9M] row-major, mean of the normals [3M], count.
__global__ void __launch_bounds__(256) mcmc_samples_pool_kernel(int M, int n, const double* const* __restrict__ accs,
                                                                const long long* const* __restrict__ cnts,
                                                                double* __restrict__ mean, double* __restrict__ cov,
                                                                double* __restrict__ normal, long long* __restrict__ count) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  long long na = 0;
  double mu[3] = {0, 0, 0}, S[6] = {0, 0, 0, 0, 0, 0}, ns[3] = {0, 0, 0};
  for (int c = 0; c < n; ++c) {
    const long long nb = cnts[c][m];
    if (nb == 0) continue;
    const double* b = accs[c] + (size_t)ACC_WORDS * m;
    if (na == 0) {
      for (int k = 0; k < 3; ++k) { mu[k] = b[k]; ns[k] = b[9 + k]; }
      for (int q = 0; q < 6; ++q) S[q] = b[3 + q];
      na = nb;
      continue;
    }
    const long long nn = na + nb;
    const double f = (double)nb / (double)nn, w = __dmul_rn((double)na, (double)nb) / (double)nn;
    double d[3];
    for (int k = 0; k < 3; ++k) {
      d[k] = b[k] - mu[k];
      mu[k] = __dadd_rn(mu[k], __dmul_rn(d[k], f));
      ns[k] += b[9 + k];
    }
    for (int q = 0; q < 6; ++q) S[q] = __dadd_rn(S[q] + b[3 + q], __dmul_rn(__dmul_rn(d[SCATTER_ROW[q]], d[SCATTER_COL[q]]), w));
    na = nn;
  }
  if (m == 0) count[0] = na;
  const double dn = (double)na;
  for (int k = 0; k < 3; ++k) { mean[3 * (size_t)m + k] = na > 0 ? mu[k] : NAN; normal[3 * (size_t)m + k] = ns[k] / dn; }
  for (int q = 0; q < 6; ++q) {
    const double c = S[q] / (dn - 1.0);
    cov[9 * (size_t)m + 3 * SCATTER_ROW[q] + SCATTER_COL[q]] = c;
    cov[9 * (size_t)m + 3 * SCATTER_COL[q] + SCATTER_ROW[q]] = c;
  }
}

}  // namespace gingr

// =================================================================================================
struct McmcState {
  gingr_mcmc_settings cfg;
  gingr::McmcDev dev;
  int n_model_ids = 0, n_target_ids = 0;      // 0 = all points
  DevBuf<int32_t> model_ids, target_ids;
  // snapshot of the current state while a proposal occupies the working buffers
  DevBuf<double> s_ds, s_alpha, s_fit, s_fac;
  DevBuf<int> s_is;
  // posterior of the current state (raw Mx + rhs row, posterior-mean coefficients); the proposal's live in the
  // working buffers g->Mx_raw / cm_prop
  DevBuf<double> raw_cur, cm_cur, cm_prop;
  DevBuf<double> best_ds, best_alpha, best_fit;
  DevBuf<int> best_is;
  DevBuf<double> md;
  DevBuf<int> mi;
  // scratch of the transition density and the evaluators
  DevBuf<double> sys, vecs, u3m, inst, q_pts, target_sub;
  gingr::ClosestWorkspace ws_m2t, ws_t2m;
  gingr::SpatialGrid fit_tgrid;
  bool use_fit_tgrid = false;
  // sample collection (gingr_mcmc_collect; every = 0: off): per-vertex moments [M][ACC_WORDS] and counts [M]
  int col_burn_in = 0, col_every = 0, col_total = 0;
  DevBuf<double> col_acc;
  DevBuf<long long> col_cnt;
  bool primed = false;
  GraphExec graph_exec;
  uint64_t graph_seed = 0;
  int64_t graph_launches = 0;
};

using namespace gingr;

static void mcmc_release(gingr_registration* g) {
  if (!g->mcmc) return;
  ++g_batch_epoch;   // a batched plan that names this chain is stale
  g->mcmc.reset();
}

// gingr_initialize_state / gingr_update / gingr_update_chain* / gingr_update_batch moved the device-resident state: the kept
// posterior, log values and best sample of the chain no longer describe it, the next gingr_mcmc_chain starts afresh
static void mcmc_invalidate(gingr_registration* g) {
  if (g && g->mcmc) g->mcmc->primed = false;
}

static void mcmc_drop_chain_graph(gingr_registration* g) {
  if (g && g->mcmc) g->mcmc->graph_exec.reset();
}

// EvaluatorWrapper.logValue pieces of the state in the working buffers (fit, alpha): out[0] = ModelEvaluator,
// out[1] = IndependentPointDistanceEvaluator
// d_surface_d2 (optional): squared distances of ALL points of d_fit to the target surface when a correspondence search on
// the same points has just produced them (ClosestWorkspace::surf_d2) -- the same scan is then not run a second time
static int32_t enqueue_log_value(gingr_registration* g, const double* d_fit, const double* d_alpha, double* d_out,
                                 const double* d_surface_d2 = nullptr) {
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  const gingr_model* m = g->model;
  const gingr_target* tg = g->target;
  cudaStream_t st = ctx->stream;
  const int M = m->M, N = tg->N_total;
  const int mode = mc->cfg.evaluation_mode;
  const double sd = mc->cfg.uncertainty;
  int acc = 0;
  if (mode == GINGR_EVAL_MODEL_TO_TARGET || mode == GINGR_EVAL_SYMMETRIC) {
    // points of the sample at the comparison ids against the target surface (:54-60)
    const int nq = mc->n_model_ids > 0 ? mc->n_model_ids : M;
    const double* q = d_fit;
    if (mc->n_model_ids > 0) {
      GINGR_LAUNCH(ctx, gather_aos_kernel, ceil_div(nq, 256), 256, 0, st, nq, mc->model_ids.p, d_fit, mc->q_pts.p);
      GINGR_LAUNCHED(ctx);
      q = mc->q_pts.p;
    }
    const double* d2 = mc->ws_m2t.d2.p;
    if (d_surface_d2 && mc->n_model_ids == 0) {
      d2 = d_surface_d2;
    } else {
      MeshView tv;
      tv.n = N; tv.aos = tg->aos.p; tv.soa = tg->verts.p; tv.T = tg->T; tv.tri = tg->tri.p; tv.tgrid = tg->tgrid.get();
      GINGR_TRY(surface_distance_enqueue(ctx, mc->ws_m2t, nq, q, tv));
    }
    GINGR_LAUNCH(ctx, mcmc_distance_logpdf_kernel, 1, 256, 0, st, nq, d2, sd, mode == GINGR_EVAL_SYMMETRIC ? 0.5 : 1.0, acc,
                                                   d_out + 1, m->r, d_alpha);
    GINGR_LAUNCHED(ctx);
    acc = 1;
  }
  if (mode == GINGR_EVAL_TARGET_TO_MODEL || mode == GINGR_EVAL_SYMMETRIC) {
    // the comparison points of the target against the surface of the sample (:62-67)
    const int nq = mc->n_target_ids > 0 ? mc->n_target_ids : N;
    const double* q = mc->n_target_ids > 0 ? mc->target_sub.p : tg->aos.p;
    GINGR_TRY(aos_to_soa_enqueue(ctx, M, d_fit, mc->inst.p));
    MeshView fv;
    fv.n = M; fv.aos = d_fit; fv.soa = mc->inst.p; fv.T = m->T; fv.tri = m->tri.p;
    if (mc->use_fit_tgrid) {
      VertexArray va;
      va.p = d_fit;
      GINGR_TRY(grid_build_triangles_enqueue(ctx, mc->fit_tgrid, M, va, m->T, m->tri.p));
      fv.tgrid = &mc->fit_tgrid;
    }
    GINGR_TRY(surface_distance_enqueue(ctx, mc->ws_t2m, nq, q, fv));
    GINGR_LAUNCH(ctx, mcmc_distance_logpdf_kernel, 1, 256, 0, st, nq, mc->ws_t2m.d2.p, sd, mode == GINGR_EVAL_SYMMETRIC ? 0.5 : 1.0, acc,
                                                   d_out + 1, m->r, acc ? nullptr : d_alpha);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// log density of the informed proposal for the move `from` -> toMesh, from the kept posterior of `from`:
// raw = [Mx ; rhs] before the factorisation, cmean = posterior-mean coefficients, from_ds / from_is = the state blocks
// of `from` after its posterior phase (DS_R = its rotation, DS_T its translation, fail flags).
static int32_t enqueue_log_transition(gingr_registration* g, const double* d_raw, const double* d_cmean, const double* d_from_ds,
                                      const int* d_from_is, const double* d_to_mesh, double* d_out) {
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  const gingr_model* m = g->model;
  const int M = m->M, r = m->r, rp = m->rp;
  cudaStream_t st = ctx->stream;
  double* v = mc->vecs.p;   // [0] b_proj  [1] S c  [2] u  [3] Mx u
  GINGR_LAUNCH(ctx, mcmc_residual_kernel, ceil_div(M, 256), 256, 0, st, M, d_to_mesh, m->ref.p, m->mean.p, d_from_ds + DS_R, d_from_ds + DS_T,
                                                         mc->u3m.p);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(gemvT_enqueue(ctx, 3 * M, r, rp, m->phi.p, mc->u3m.p, m->sqrt_lambda.p, g->gt_part.p, v));
  GINGR_TRY(dense_matvec_enqueue(ctx, r, m->S.p, rp, d_cmean, v + rp));
  GINGR_LAUNCH(ctx, mcmc_build_system_kernel, ceil_div((r + 1) * rp, 256), 256, 0, st, r, rp, m->S.p, d_raw, 1e-5, v, v + rp, mc->sys.p,
                                                                        mc->mi.p + MI_INFO2);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(cholesky_df_enqueue(ctx, r, r + 1, mc->sys.p, rp, mc->mi.p + MI_INFO2, g->cholws));
  GINGR_TRY(chol_backsolve_enqueue(ctx, r, mc->sys.p, rp, mc->sys.p + (size_t)r * rp, v + 2 * rp, g->flags.p));
  GINGR_TRY(dense_matvec_enqueue(ctx, r, d_raw, rp, v + 2 * rp, v + 3 * rp));
  GINGR_LAUNCH(ctx, mcmc_quadform_kernel, 1, 256, 0, st, r, v + 2 * rp, v + 3 * rp, d_from_is, mc->mi.p + MI_INFO2, d_out);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// toMesh of logTransitionProbability(from, to) (GeneratorWrapperStochastic.scala:46-51): from.fit when stepLength == 1,
// else the UNPOSED instance of the compensated coefficients.  Returns the device pointer holding it.
static int32_t enqueue_to_mesh(gingr_registration* g, double step_length, const double* d_from_fit, const double* d_from_alpha,
                               const double* d_to_alpha, const double** out) {
  if (step_length == 1.0) { *out = d_from_fit; return GINGR_OK; }
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  const gingr_model* m = g->model;
  const int M = m->M, r = m->r, rp = m->rp;
  double* v = mc->vecs.p;
  GINGR_LAUNCH(ctx, mcmc_compensate_kernel, ceil_div(r, 256), 256, 0, ctx->stream, r, d_from_alpha, d_to_alpha, step_length, v + 4 * rp);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(instance_rows(ctx, m, v + 5 * rp, 1, v + 4 * rp, nullptr, mc->inst.p, nullptr));
  add_vectors_enqueue(ctx, 3 * M, m->ref.p, m->mean.p, mc->u3m.p);
  add_vectors_enqueue(ctx, 3 * M, mc->u3m.p, mc->inst.p, mc->inst.p);
  *out = mc->inst.p;
  return GINGR_OK;
}

// collection of the chain state in the working buffers (mcmc_collect_kernel); prev_is = null for the start state
static int32_t enqueue_collect(gingr_registration* g, const int* prev_is) {
  McmcState* mc = g->mcmc.get();
  if (mc->col_every <= 0) return GINGR_OK;
  gingr_ctx* ctx = g->ctx;
  const gingr_model* m = g->model;
  const bool normals = m->T > 0;
  GINGR_LAUNCH(ctx, mcmc_collect_kernel, ceil_div(m->M, 256), 256, 0, ctx->stream, m->M, mc->mi.p, prev_is, mc->col_burn_in,
               mc->col_every, mc->col_total, g->fit.p, normals ? m->tri.p : nullptr, normals ? m->adj_off.p : nullptr,
               normals ? m->adj.p : nullptr, mc->col_acc.p, mc->col_cnt.p);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

static int32_t collect_reset(gingr_registration* g) {
  McmcState* mc = g->mcmc.get();
  if (mc->col_every <= 0) return GINGR_OK;
  const size_t M = (size_t)g->model->M;
  GINGR_CUDA_TRY(g->ctx, cudaMemsetAsync(mc->col_acc.p, 0, sizeof(double) * ACC_WORDS * M, g->ctx->stream));
  GINGR_CUDA_TRY(g->ctx, cudaMemsetAsync(mc->col_cnt.p, 0, sizeof(long long) * M, g->ctx->stream));
  return GINGR_OK;
}

// posterior-mean coefficients of the state whose factor + z sit in g->Mx
static int32_t enqueue_posterior_mean_coeffs(gingr_registration* g, double* d_out) {
  const gingr_model* m = g->model;
  return chol_backsolve_enqueue(g->ctx, m->r, g->Mx.p, m->rp, g->Mx.p + (size_t)m->r * m->rp, d_out, g->flags.p);
}

// the surface distances the posterior phase of g->fit left behind, when its correspondence search was the triangular
// closest point of the fit's vertices on the target (the evaluator's own query)
static const double* posterior_surface_d2(const gingr_registration* g) {
  const gingr_config& cfg = g->cfg;
  return (cfg.algorithm == GINGR_ALGO_ICP && cfg.correspondence_method == GINGR_TRIANGULAR_CLOSEST_POINT &&
          !cfg.reverse_correspondence_direction && g->ctx->nranks == 1)
             ? g->closest.surf_d2.p
             : nullptr;
}

// Posterior + evaluators of the device-resident state: the chain starts from it.
static int32_t mcmc_prime(gingr_registration* g) {
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  const gingr_model* m = g->model;
  const int M = m->M, r = m->r, rp = m->rp;
  cudaStream_t st = ctx->stream;
  g->keep_raw = true;
  mc->graph_exec.reset();   // the captured step bakes in the state's stepLength (toMesh of the transition density)
  // a new chain: step counter (the Philox stream position) and statistics start at zero
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(mc->md.p, 0, sizeof(double) * MD_COUNT, st));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(mc->mi.p, 0, sizeof(int) * MI_COUNT, st));
  GINGR_TRY(collect_reset(g));
  GINGR_TRY(enqueue_posterior_phase(g));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->raw_cur.p, g->Mx_raw.p, sizeof(double) * (size_t)(r + 1) * rp, cudaMemcpyDeviceToDevice, st));
  GINGR_TRY(enqueue_posterior_mean_coeffs(g, mc->cm_cur.p));
  GINGR_TRY(enqueue_log_value(g, g->fit.p, g->alpha.p, mc->md.p + MD_LP_CUR, posterior_surface_d2(g)));
  if (g->last_out.step_length == 1.0)   // the informed density of the start state (fit on its own posterior)
    GINGR_TRY(enqueue_log_transition(g, g->Mx_raw.p, mc->cm_cur.p, g->ds.p, g->is.p, g->fit.p, mc->md.p + MD_TINF_CUR));
  // best = current
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->best_ds.p, g->ds.p, sizeof(double) * DS_COUNT, cudaMemcpyDeviceToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->best_is.p, g->is.p, sizeof(int) * IS_COUNT, cudaMemcpyDeviceToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->best_alpha.p, g->alpha.p, sizeof(double) * r, cudaMemcpyDeviceToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->best_fit.p, g->fit.p, sizeof(double) * 3 * (size_t)M, cudaMemcpyDeviceToDevice, st));
  GINGR_TRY(enqueue_collect(g, nullptr));   // chain state 0
  // MD_LP_BEST = lp_cur
  double h[2];
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(h, mc->md.p + MD_LP_CUR, sizeof(double) * 2, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  const double best = h[0] + h[1];
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->md.p + MD_LP_BEST, &best, sizeof(double), cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  mc->primed = true;
  return GINGR_OK;
}

// One Metropolis-Hastings step on the working state (which holds the current state after its posterior phase).
static int32_t enqueue_mcmc_step(gingr_registration* g, uint64_t seed) {
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  const gingr_model* m = g->model;
  const int M = m->M, r = m->r, rp = m->rp;
  cudaStream_t st = ctx->stream;
  const size_t fac_n = (size_t)(r + 1) * rp;
  // 1. snapshot of the current state (one node; the int block travels as 8 doubles)
  static_assert(IS_COUNT % 2 == 0, "the int state block is copied as doubles");
  {
    CopySegments sg;
    sg.add(nullptr, 0, mc->s_ds.p, g->ds.p, DS_COUNT);
    sg.add(nullptr, 0, mc->s_is.p, g->is.p, IS_COUNT / 2);
    sg.add(nullptr, 0, mc->s_alpha.p, g->alpha.p, r);
    sg.add(nullptr, 0, mc->s_fit.p, g->fit.p, (size_t)3 * M);
    sg.add(nullptr, 0, mc->s_fac.p, g->Mx.p, fac_n);
    GINGR_LAUNCH(ctx, multi_copy_kernel, 16, 256, 0, st, sg);
    GINGR_LAUNCHED(ctx);
  }
  // 3. the informed proposal update(current, probabilistic = true) from the kept posterior ...
  g->sample_counter = mc->mi.p + MI_STEP;
  g->skip_fit_refresh = true;   // the fit is evaluated once, after the random override
  const int32_t rc = enqueue_update_phase(g, 1, seed);
  g->skip_fit_refresh = false;
  g->sample_counter = nullptr;
  GINGR_TRY(rc);
  // 4. ... replaced by the chosen random leaf; iteration + 1; fit of the proposal
  GINGR_LAUNCH(ctx, mcmc_random_override_kernel, 1, 256, 0, st, mc->dev, seed, r, mc->mi.p, mc->s_ds.p, mc->s_is.p, mc->s_alpha.p, g->ds.p,
                                                 g->is.p, g->alpha.p, mc->mi.p, mc->md.p);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R2));
  // 5. posterior of the proposal (kept if accepted: the reference memoises it for the next update)
  GINGR_TRY(enqueue_posterior_phase(g));
  GINGR_TRY(enqueue_posterior_mean_coeffs(g, mc->cm_prop.p));
  // 6. informed transition densities, both directions
  const double step_length = g->last_out.step_length;
  const bool fw_cached = step_length == 1.0;   // MD_TINF_CUR holds it (mcmc_prime / the accepting step)
  const double* to_mesh = nullptr;
  if (!fw_cached) {
    GINGR_TRY(enqueue_to_mesh(g, step_length, mc->s_fit.p, mc->s_alpha.p, g->alpha.p, &to_mesh));
    GINGR_TRY(enqueue_log_transition(g, mc->raw_cur.p, mc->cm_cur.p, mc->s_ds.p, mc->s_is.p, to_mesh, mc->md.p + MD_TINF_FW));
  }
  GINGR_TRY(enqueue_to_mesh(g, step_length, g->fit.p, g->alpha.p, mc->s_alpha.p, &to_mesh));
  GINGR_TRY(enqueue_log_transition(g, g->Mx_raw.p, mc->cm_prop.p, g->ds.p, g->is.p, to_mesh, mc->md.p + MD_TINF_BW));
  // 7. evaluators of the proposal (its posterior phase, step 5, searched the same points)
  GINGR_TRY(enqueue_log_value(g, g->fit.p, g->alpha.p, mc->md.p + MD_LP_PROP, posterior_surface_d2(g)));
  // 8. accept / reject
  GINGR_LAUNCH(ctx, mcmc_decide_kernel, 1, 256, 0, st, mc->dev, r, fw_cached ? 1 : 0, mc->s_ds.p, mc->s_is.p, mc->s_alpha.p, g->ds.p, g->alpha.p, mc->md.p, mc->mi.p);
  GINGR_LAUNCHED(ctx);
  const int* acc = mc->mi.p + MI_ACCEPT;
  const int* bu = mc->mi.p + MI_BEST_UPDATED;
  // reject: the working state returns to the snapshot (ints by their own kernel: the retry counter stays);
  // accept: the proposal's posterior becomes the current one; best sample (only ever an accepted proposal)
  GINGR_LAUNCH(ctx, mcmc_restore_ints_kernel, 1, 1, 0, st, acc, g->is.p, mc->s_is.p, bu, mc->best_is.p);
  GINGR_LAUNCHED(ctx);
  {
    CopySegments sg;
    sg.add(acc, 0, g->ds.p, mc->s_ds.p, DS_COUNT);
    sg.add(acc, 0, g->alpha.p, mc->s_alpha.p, r);
    sg.add(acc, 0, g->fit.p, mc->s_fit.p, (size_t)3 * M);
    sg.add(acc, 0, g->Mx.p, mc->s_fac.p, fac_n);
    sg.add(acc, 1, mc->raw_cur.p, g->Mx_raw.p, fac_n);
    sg.add(acc, 1, mc->cm_cur.p, mc->cm_prop.p, r);
    sg.add(bu, 1, mc->best_ds.p, g->ds.p, DS_COUNT);
    sg.add(bu, 1, mc->best_alpha.p, g->alpha.p, r);
    sg.add(bu, 1, mc->best_fit.p, g->fit.p, (size_t)3 * M);
    GINGR_LAUNCH(ctx, multi_copy_kernel, 16, 256, 0, st, sg);
    GINGR_LAUNCHED(ctx);
  }
  // 9. sample collection of the state the step leaves (only when switched on: the step is otherwise unchanged)
  GINGR_TRY(enqueue_collect(g, mc->s_is.p));
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

static int32_t mcmc_capture(gingr_registration* g, uint64_t seed) {
  McmcState* mc = g->mcmc.get();
  if (mc->graph_exec.h && mc->graph_seed == seed) return GINGR_OK;
  GINGR_TRY(capture_graph(g->ctx, mc->graph_exec, &mc->graph_launches, [&] { return enqueue_mcmc_step(g, seed); }));
  mc->graph_seed = seed;
  return GINGR_OK;
}

static int32_t mcmc_check(gingr_registration* g, const char* who) {
  if (!g) return gingr_fail(nullptr, GINGR_ERR_ARG, who);
  if (!g->mcmc) return gingr_fail(g->ctx, GINGR_ERR_ARG, "call gingr_mcmc_configure first");
  if (g->ctx->nranks != 1) return gingr_fail(g->ctx, GINGR_ERR_UNSUPPORTED, "MCMC chains are replicas: one ctx per GPU without a communicator");
  return GINGR_OK;
}

extern "C" {

int32_t gingr_mcmc_configure(gingr_registration* g, const gingr_mcmc_settings* s, const int32_t* model_ids, int32_t n_model_ids,
                             const int32_t* target_ids, int32_t n_target_ids) {
  if (!g || !s || n_model_ids < 0 || n_target_ids < 0 || (n_model_ids > 0 && !model_ids) || (n_target_ids > 0 && !target_ids))
    return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_mcmc_configure: bad argument");
  gingr_ctx* ctx = g->ctx;
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_mcmc_configure: single-GPU chains only");
  if (g->cfg.algorithm == GINGR_ALGO_BCPD) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_mcmc_configure: BCPD registrations are deterministic");
  if (!(s->random_mixture >= 0.0 && s->random_mixture <= 1.0) || !(s->uncertainty > 0.0) || s->evaluation_mode < 0 ||
      s->evaluation_mode > 2)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_configure: randomMixture in [0, 1], uncertainty > 0, mode 0..2");
  for (int k = 0; k < 3; ++k)
    if (!(s->rot_sdev[k] > 0.0) || !(s->trans_sdev[k] > 0.0) || !(s->shape_sdev[k] > 0.0))
      return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_configure: proposal standard deviations must be positive");
  const gingr_model* m = g->model;
  const gingr_target* tg = g->target;
  const int M = m->M, r = m->r, rp = m->rp, N = tg->N_total;
  const int mode = s->evaluation_mode;
  const bool m2t = mode != GINGR_EVAL_TARGET_TO_MODEL, t2m = mode != GINGR_EVAL_MODEL_TO_TARGET;
  if (m2t && tg->T <= 0) return gingr_fail(ctx, GINGR_ERR_ARG, "the distance evaluator needs the target triangles");
  if (t2m && m->T <= 0) return gingr_fail(ctx, GINGR_ERR_ARG, "the target-to-model evaluator needs the model triangles");
  for (int k = 0; k < n_model_ids; ++k)
    if (model_ids[k] < 0 || model_ids[k] >= M) return gingr_fail(ctx, GINGR_ERR_ARG, "model comparison id out of range");
  for (int k = 0; k < n_target_ids; ++k)
    if (target_ids[k] < 0 || target_ids[k] >= N) return gingr_fail(ctx, GINGR_ERR_ARG, "target comparison id out of range");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  mcmc_release(g);
  g->mcmc = std::make_unique<McmcState>();
  McmcState* mc = g->mcmc.get();
  mc->cfg = *s;
  mc->dev.rho = s->random_mixture;
  for (int k = 0; k < 3; ++k) { mc->dev.sd[k] = s->rot_sdev[k]; mc->dev.sd[3 + k] = s->trans_sdev[k]; mc->dev.sd[6 + k] = s->shape_sdev[k]; }
  mc->n_model_ids = n_model_ids;
  mc->n_target_ids = n_target_ids;
  cudaStream_t st = ctx->stream;
  const size_t fac_n = (size_t)(r + 1) * rp;
  GINGR_CUDA_TRY(ctx, mc->s_ds.alloc(DS_COUNT)); GINGR_CUDA_TRY(ctx, mc->s_is.alloc(IS_COUNT));
  GINGR_CUDA_TRY(ctx, mc->s_alpha.alloc(rp)); GINGR_CUDA_TRY(ctx, mc->s_fit.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, mc->s_fac.alloc(fac_n)); GINGR_CUDA_TRY(ctx, mc->raw_cur.alloc(fac_n));
  GINGR_CUDA_TRY(ctx, g->Mx_raw.alloc(fac_n));
  GINGR_CUDA_TRY(ctx, mc->cm_cur.alloc(rp)); GINGR_CUDA_TRY(ctx, mc->cm_prop.alloc(rp));
  GINGR_CUDA_TRY(ctx, mc->best_ds.alloc(DS_COUNT)); GINGR_CUDA_TRY(ctx, mc->best_is.alloc(IS_COUNT));
  GINGR_CUDA_TRY(ctx, mc->best_alpha.alloc(rp)); GINGR_CUDA_TRY(ctx, mc->best_fit.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, mc->md.alloc(MD_COUNT)); GINGR_CUDA_TRY(ctx, mc->mi.alloc(MI_COUNT));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(mc->md.p, 0, sizeof(double) * MD_COUNT, st));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(mc->mi.p, 0, sizeof(int) * MI_COUNT, st));
  GINGR_CUDA_TRY(ctx, mc->sys.alloc((size_t)(r + 8) * rp)); GINGR_CUDA_TRY(ctx, mc->vecs.alloc((size_t)8 * rp));
  GINGR_CUDA_TRY(ctx, mc->u3m.alloc((size_t)3 * M)); GINGR_CUDA_TRY(ctx, mc->inst.alloc((size_t)3 * M));
  if (m2t) {
    const int nq = n_model_ids > 0 ? n_model_ids : M;
    GINGR_TRY(mc->ws_m2t.ensure(ctx, nq, N, tg->T, 0));
    GINGR_CUDA_TRY(ctx, mc->q_pts.alloc((size_t)3 * nq));
    if (n_model_ids > 0) {
      GINGR_CUDA_TRY(ctx, mc->model_ids.alloc(n_model_ids));
      GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->model_ids.p, model_ids, sizeof(int32_t) * n_model_ids, cudaMemcpyHostToDevice, st));
    }
  }
  if (t2m) {
    const int nq = n_target_ids > 0 ? n_target_ids : N;
    GINGR_TRY(mc->ws_t2m.ensure(ctx, nq, M, m->T, 0));
    if (n_target_ids > 0) {
      GINGR_CUDA_TRY(ctx, mc->target_ids.alloc(n_target_ids));
      GINGR_CUDA_TRY(ctx, mc->target_sub.alloc((size_t)3 * n_target_ids));
      GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->target_ids.p, target_ids, sizeof(int32_t) * n_target_ids, cudaMemcpyHostToDevice, st));
      GINGR_LAUNCH(ctx, gather_aos_kernel, ceil_div(n_target_ids, 256), 256, 0, st, n_target_ids, mc->target_ids.p, tg->aos.p, mc->target_sub.p);
      GINGR_LAUNCHED(ctx);
    }
    if (grid_wanted(M)) {
      GINGR_TRY(mc->fit_tgrid.ensure(ctx, M, m->T, true));
      mc->use_fit_tgrid = true;
    }
  }
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  g->keep_raw = true;
  drop_graph(g);   // the deterministic graph was captured without the raw copy
  return GINGR_OK;
}

// EvaluatorWrapper(probabilistic = true).logValue of a host state: out[0] = Prior (ModelEvaluator), out[1] = Distance
// (IndependentPointDistanceEvaluator); their sum is the product evaluator (Evaluator.scala:25-28).
int32_t gingr_evaluate_log_value(gingr_registration* g, const gingr_state* s, const double* alpha, double* out) {
  GINGR_TRY(mcmc_check(g, "gingr_evaluate_log_value: bad argument"));
  if (!s || !alpha || !out) return gingr_fail(g->ctx, GINGR_ERR_ARG, "gingr_evaluate_log_value: bad argument");
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  g->state_valid = false;
  mc->primed = false;
  GINGR_TRY(upload_state(g, s, alpha));
  GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R));
  GINGR_TRY(enqueue_log_value(g, g->fit.p, g->alpha.p, mc->md.p + MD_LP_PROP));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(out, mc->md.p + MD_LP_PROP, sizeof(double) * 2, cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GINGR_OK;
}

// GeneratorWrapperStochastic.logTransitionProbability(from, to) (GeneratorWrapperStochastic.scala:42-63): the informed
// generator alone (the mixture with the random generators is formed inside gingr_mcmc_chain).
int32_t gingr_log_transition_probability(gingr_registration* g, const gingr_state* from, const double* from_alpha,
                                         const gingr_state* to, const double* to_alpha, double* out) {
  GINGR_TRY(mcmc_check(g, "gingr_log_transition_probability: bad argument"));
  if (!from || !from_alpha || !to || !to_alpha || !out)
    return gingr_fail(g->ctx, GINGR_ERR_ARG, "gingr_log_transition_probability: bad argument");
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  const gingr_model* m = g->model;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  g->state_valid = false;
  mc->primed = false;
  GINGR_TRY(upload_state(g, from, from_alpha));
  GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R));
  g->keep_raw = true;
  GINGR_TRY(enqueue_posterior_phase(g));
  GINGR_TRY(enqueue_posterior_mean_coeffs(g, mc->cm_prop.p));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mc->s_alpha.p, to_alpha, sizeof(double) * m->r, cudaMemcpyHostToDevice, ctx->stream));
  const double* to_mesh = nullptr;
  GINGR_TRY(enqueue_to_mesh(g, from->step_length, g->fit.p, g->alpha.p, mc->s_alpha.p, &to_mesh));
  GINGR_TRY(enqueue_log_transition(g, g->Mx_raw.p, mc->cm_prop.p, g->ds.p, g->is.p, to_mesh, mc->md.p + MD_TINF_FW));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(out, mc->md.p + MD_TINF_FW, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GINGR_OK;
}

// `iters` Metropolis-Hastings steps of the chain that starts at the device-resident state (gingr_initialize_state /
// gingr_update / a previous gingr_mcmc_chain), without host round trips.
int32_t gingr_mcmc_chain(gingr_registration* g, int32_t iters, uint64_t seed) {
  GINGR_TRY(mcmc_check(g, "gingr_mcmc_chain: bad argument"));
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  if (iters < 0) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_chain: bad argument");
  if (!g->state_valid) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_chain: no device-resident state (call gingr_initialize_state first)");
  g->host_mirror_current = false;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (!mc->primed) GINGR_TRY(mcmc_prime(g));
  const bool graph = graphs_enabled(ctx);
  if (graph) GINGR_TRY(mcmc_capture(g, seed));
  for (int k = 0; k < iters; ++k) {
    if (graph) {
      GINGR_CUDA_TRY(ctx, cudaGraphLaunch(mc->graph_exec.h, ctx->stream));
      ctx->launches += mc->graph_launches;
    } else {
      GINGR_TRY(enqueue_mcmc_step(g, seed));
    }
  }
  return GINGR_OK;
}

// ---- the MH step of many chains as ONE kernel sequence (batch.cuh; the plan and its builder: update.cu) -------------------
static int32_t mcmc_batch_plan_build(gingr_ctx* ctx, gingr_registration** regs, int n, uint64_t seed, BatchPlan& bp) {
  GINGR_TRY(batch_cap_gram(ctx, regs, n));
  for (int k = 0; k < n; ++k)
    if (!regs[k]->mcmc->primed) GINGR_TRY(mcmc_prime(regs[k]));
  return batch_plan_build(ctx, regs, n, seed, /*kind=*/2, bp, [&](int k) { return enqueue_mcmc_step(regs[k], seed + (uint64_t)k); });
}

// Independent chains batched on one GPU (BASELINE config 5): chain k uses seed + k.  The chains' steps run as one
// batched kernel sequence (blockIdx.z = chain; a step that is not batchable: the captured per-chain step graphs
// replayed round-robin on a pool of streams, as gingr_update_batch does).
int32_t gingr_mcmc_batch(gingr_registration** regs, int32_t n, int32_t iters, uint64_t seed) {
  if (!regs || n <= 0 || iters < 0) return gingr_fail(nullptr, GINGR_ERR_ARG, "gingr_mcmc_batch: bad argument");
  gingr_ctx* ctx = regs[0] ? regs[0]->ctx : nullptr;
  for (int k = 0; k < n; ++k) {
    if (!regs[k] || regs[k]->ctx != ctx) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_batch: chains must share one ctx");
    GINGR_TRY(mcmc_check(regs[k], "gingr_mcmc_batch: bad argument"));
    if (!regs[k]->state_valid) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_batch: chain without device-resident state");
    regs[k]->host_mirror_current = false;
  }
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (n >= 2 && n <= 65535 && graphs_enabled(ctx)) {
    static thread_local BatchPlan& bp = *new BatchPlan();   // never deleted (BatchPlan)
    if (!batch_plan_current(bp, ctx, regs, n, seed, 2)) {
      const int32_t rc = mcmc_batch_plan_build(ctx, regs, n, seed, bp);
      if (rc < 0) { bp.drop(); return rc; }
    }
    if (!bp.unsupported) {
      for (int k = 0; k < n; ++k)
        if (!regs[k]->mcmc->primed) GINGR_TRY(mcmc_prime(regs[k]));
      for (int it = 0; it < iters; ++it) GINGR_CUDA_TRY(ctx, cudaGraphLaunch(bp.exec.h, ctx->stream));
      ctx->launches += (int64_t)iters * bp.nlaunch;
      return GINGR_OK;
    }
  }
  ChainStreamPool* sp = nullptr;
  GINGR_TRY(chain_stream_pool(ctx, &sp));
  for (int k = 0; k < n; ++k) {
    if (!regs[k]->mcmc->primed) GINGR_TRY(mcmc_prime(regs[k]));
    GINGR_TRY(mcmc_capture(regs[k], seed + (uint64_t)k));
  }
  GINGR_TRY(replay_chain_graphs(ctx, sp, n, iters, [&](int k) { return regs[k]->mcmc->graph_exec.h; }, [](int, cudaStream_t) {}));
  for (int k = 0; k < n; ++k) ctx->launches += (int64_t)iters * regs[k]->mcmc->graph_launches;
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// Sample collection of the chain (LogHelper.samplesFromLog, LogHelper.scala:29-43): the rule lives with the chain and the
// accumulators start from zero here and whenever the chain is primed afresh.  take_every_n = 0 switches it off.
int32_t gingr_mcmc_collect(gingr_registration* g, int32_t burn_in, int32_t take_every_n, int32_t total) {
  GINGR_TRY(mcmc_check(g, "gingr_mcmc_collect: bad argument"));
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  if (burn_in < 0 || take_every_n < 0 || total < 0)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_collect: burn_in, take_every_n and total must be >= 0");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  mc->col_burn_in = burn_in;
  mc->col_every = take_every_n;
  mc->col_total = total;
  if (take_every_n > 0) {
    const size_t M = (size_t)g->model->M;
    GINGR_CUDA_TRY(ctx, mc->col_acc.alloc(ACC_WORDS * M));
    GINGR_CUDA_TRY(ctx, mc->col_cnt.alloc(M));
    GINGR_TRY(collect_reset(g));
  }
  mc->graph_exec.reset();   // the captured step holds the rule and the accumulators
  ++g_batch_epoch;          // ... and so do batched plans that name this chain
  return GINGR_OK;
}

// The collected statistics of n chains pooled in the order regs[0], regs[1], ... (PosteriorHelper.scala:31-79 reduces
// them to the distance maps).  Chains share one ctx and one model and have collection on.  Outputs may be null.
int32_t gingr_mcmc_samples(gingr_registration** regs, int32_t n, int64_t* count, double* mean, double* cov, double* normal) {
  if (!regs || n <= 0 || !regs[0]) return gingr_fail(nullptr, GINGR_ERR_ARG, "gingr_mcmc_samples: bad argument");
  gingr_ctx* ctx = regs[0]->ctx;
  const gingr_model* m = regs[0]->model;
  std::vector<const double*> accs(n);
  std::vector<const long long*> cnts(n);
  for (int k = 0; k < n; ++k) {
    if (!regs[k] || regs[k]->ctx != ctx || regs[k]->model != m)
      return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_samples: chains must share one ctx and one model");
    GINGR_TRY(mcmc_check(regs[k], "gingr_mcmc_samples: bad argument"));
    const McmcState* mc = regs[k]->mcmc.get();
    if (mc->col_every <= 0) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_samples: sample collection is off (gingr_mcmc_collect)");
    accs[k] = mc->col_acc.p;
    cnts[k] = mc->col_cnt.p;
  }
  if (normal && m->T <= 0) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_samples: normals need the model triangles");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t M = (size_t)m->M;
  DevBuf<const double*> d_accs;
  DevBuf<const long long*> d_cnts;
  DevBuf<double> out;
  DevBuf<long long> d_count;
  GINGR_CUDA_TRY(ctx, d_accs.alloc(n));
  GINGR_CUDA_TRY(ctx, d_cnts.alloc(n));
  GINGR_CUDA_TRY(ctx, out.alloc(15 * M));
  GINGR_CUDA_TRY(ctx, d_count.alloc(1));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_accs.p, accs.data(), sizeof(const double*) * n, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_cnts.p, cnts.data(), sizeof(const long long*) * n, cudaMemcpyHostToDevice, st));
  mcmc_samples_pool_kernel<<<ceil_div(m->M, 256), 256, 0, st>>>(m->M, n, d_accs.p, d_cnts.p, out.p, out.p + 3 * M, out.p + 12 * M,
                                                              d_count.p);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  long long h_count = 0;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(&h_count, d_count.p, sizeof(long long), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (cov && h_count < 2) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_samples: the covariance needs at least 2 samples");
  if (count) *count = h_count;
  if (mean) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mean, out.p, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, st));
  if (cov) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(cov, out.p + 3 * M, sizeof(double) * 9 * M, cudaMemcpyDeviceToHost, st));
  if (normal) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(normal, out.p + 12 * M, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return GINGR_OK;
}

// Chain bookkeeping.  values[16]: 0/1 log value (prior, distance) of the current state, 2/3 of the last proposal,
// 4/5 informed transition log density current -> proposal / proposal -> current of the last step, 6 u_accept, 7 the MH
// log ratio a, 8 best log value, 9/10 mixture transition log densities of the last step.  counts[32]: 0 steps, 1 leaf of
// the last step, 2 last accept flag, 3 accepted, 5 NaN transitions, 8..17 proposals per generator leaf, 18..27 accepted
// per leaf (order: informed, yaw, pitch, roll, x, y, z, shape steps 0..2).
int32_t gingr_mcmc_stats(gingr_registration* g, double* values, int32_t* counts) {
  GINGR_TRY(mcmc_check(g, "gingr_mcmc_stats: bad argument"));
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (values) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(values, mc->md.p, sizeof(double) * MD_COUNT, cudaMemcpyDeviceToHost, ctx->stream));
  if (counts) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(counts, mc->mi.p, sizeof(int) * MI_COUNT, cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GINGR_OK;
}

// The best sample of the chain so far (BestAndCurrentSampleLogger.currentBestSample, GingrAlgorithm.scala:160-163).
int32_t gingr_mcmc_best(gingr_registration* g, gingr_state* out, double* alpha_out, double* fit_out) {
  GINGR_TRY(mcmc_check(g, "gingr_mcmc_best: bad argument"));
  gingr_ctx* ctx = g->ctx;
  McmcState* mc = g->mcmc.get();
  const gingr_model* m = g->model;
  if (!out) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_best: bad argument");
  if (!mc->primed) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_mcmc_best: the chain has not started");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  double* h = ctx->h_pinned;
  int* hi = reinterpret_cast<int*>(h + DS_COUNT);
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(h, mc->best_ds.p, sizeof(double) * DS_COUNT, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(hi, mc->best_is.p, sizeof(int) * IS_COUNT, cudaMemcpyDeviceToHost, st));
  if (alpha_out) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(alpha_out, mc->best_alpha.p, sizeof(double) * m->r, cudaMemcpyDeviceToHost, st));
  if (fit_out) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(fit_out, mc->best_fit.p, sizeof(double) * 3 * (size_t)m->M, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  out->scale = h[DS_SCALE];
  for (int d = 0; d < 3; ++d) { out->translation[d] = h[DS_T + d]; out->euler[d] = h[DS_EULER + d]; out->center[d] = h[DS_CENTER + d]; }
  out->sigma2 = h[DS_SIGMA2];
  out->step_length = h[DS_STEP];
  out->global_transformation = hi[IS_GT];
  out->iteration = hi[IS_ITER];
  out->status = hi[IS_STATUS];
  out->rank = m->r;
  return GINGR_OK;
}

}  // extern "C"
