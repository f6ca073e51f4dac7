// gingr.hpp -- header-only C++17 host mirror of the reference's registration interface over the C ABI of
// gingr_cuda.h.  The reference is compiled JVM code whose toolchain is absent here (no JVM / sbt / scalismo), so beside
// the Scala shim (scala/, source only) and the Python mirror the tests drive (gingr_b200/api.py) this header gives native
// callers the same surface: the case classes' names, fields and DEFAULTS, `initializeState`, `update`, `propose`, `run`
// with the reference's stopping rules and statuses.  Citations are relative to src/main/scala/gingr/ of the reference.
//
//   GeneralRegistrationState / ModelFittingParameters   api/GeneralRegistrationState.scala:28-41, api/ModelFittingParameters.scala:31-74
//   CpdConfiguration / IcpConfiguration                  api/registration/config/CPD.scala:105-115, ICP.scala:54-66
//   GingrAlgorithm::update / propose / run               api/GingrAlgorithm.scala:192-254, :115-175,
//                                                        api/sampling/generators/GingrGeneratorWrapper.scala:28-39
//
// Errors: negative C status codes become gingr::Error (with gingr_last_error's text); numerical failure is NOT an
// exception -- as in the reference it is the state's status ModelFlexibilityError.  There is no CPU fallback: without a
// CUDA device the Context constructor throws.
#pragma once

#include <array>
#include <cmath>
#include <cstdint>
#include <functional>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "gingr_cuda.h"

namespace gingr {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& msg) : std::runtime_error("libgingr_cuda error " + std::to_string(c) + ": " + msg), code(c) {}
};

// api/FittingStatuses.scala:20-23, api/GlobalTranformationType.scala:20-24, registration/config/ICP.scala:29-33
enum class FittingStatus : int32_t { None = GINGR_STATUS_NONE, MaxIteration = GINGR_STATUS_MAX_ITERATION,
                                     Converged = GINGR_STATUS_CONVERGED, ModelFlexibilityError = GINGR_STATUS_MODEL_FLEXIBILITY_ERROR };
enum class GlobalTransformationType : int32_t { SimilarityTransforms = GINGR_SIMILARITY_TRANSFORMS,
                                                RigidTransforms = GINGR_RIGID_TRANSFORMS, NoTransforms = GINGR_NO_TRANSFORMS };
enum class ICPCorrespondenceMethod : int32_t { TriangularClosestPoint = GINGR_TRIANGULAR_CLOSEST_POINT,
                                               AlongNormalClosestPoint = GINGR_ALONG_NORMAL_CLOSEST_POINT,
                                               PointcloudClosestPoint = GINGR_POINTCLOUD_CLOSEST_POINT };

class Context {
 public:
  explicit Context(int device = 0) {
    const int32_t rc = gingr_ctx_create(device, &h_);
    if (rc < 0) {
      const char* m = gingr_last_error(nullptr);
      throw Error(rc, m ? m : "");
    }
  }
  ~Context() { if (h_) gingr_ctx_destroy(h_); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  gingr_ctx* handle() const { return h_; }
  // negative -> exception; 0 / GINGR_MODEL_FLEXIBILITY are returned to the caller
  int32_t check(int32_t rc) const {
    if (rc < 0) {
      const char* m = gingr_last_error(h_);
      throw Error(rc, m ? m : "");
    }
    return rc;
  }
  void synchronize() const { check(gingr_ctx_synchronize(h_)); }
  int64_t launchCount() const { return gingr_ctx_launch_count(h_); }

 private:
  gingr_ctx* h_ = nullptr;
};

// api/ModelFittingParameters.scala:31-74 (scale; pose = translation + Euler rotation about the origin; shape)
struct ModelFittingParameters {
  double scale = 1.0;
  std::array<double, 3> translation{0.0, 0.0, 0.0};
  std::array<double, 3> euler{0.0, 0.0, 0.0};  // phi, theta, psi
  std::vector<double> shape;                   // alpha[rank]
};

// api/GeneralRegistrationState.scala:28-41 (model / target / landmarks live in the device handles)
struct GeneralRegistrationState {
  ModelFittingParameters modelParameters;
  std::vector<double> fit;  // [M][3]
  double sigma2 = 1.0;
  GlobalTransformationType globalTransformation = GlobalTransformationType::RigidTransforms;
  double stepLength = 1.0;
  std::string generatedBy;
  int iteration = 0;
  FittingStatus status = FittingStatus::None;

  gingr_state toPod() const {
    gingr_state s{};
    s.scale = modelParameters.scale;
    for (int d = 0; d < 3; ++d) {
      s.translation[d] = modelParameters.translation[d];
      s.euler[d] = modelParameters.euler[d];
      s.center[d] = 0.0;
    }
    s.sigma2 = sigma2;
    s.step_length = stepLength;
    s.global_transformation = static_cast<int32_t>(globalTransformation);
    s.iteration = iteration;
    s.status = static_cast<int32_t>(status);
    s.rank = static_cast<int32_t>(modelParameters.shape.size());
    return s;
  }
  void fromPod(const gingr_state& s) {
    modelParameters.scale = s.scale;
    for (int d = 0; d < 3; ++d) {
      modelParameters.translation[d] = s.translation[d];
      modelParameters.euler[d] = s.euler[d];
    }
    sigma2 = s.sigma2;
    stepLength = s.step_length;
    globalTransformation = static_cast<GlobalTransformationType>(s.global_transformation);
    iteration = s.iteration;
    status = static_cast<FittingStatus>(s.status);
  }
};

// registration/config/CPD.scala:105-115; converged: |sigma2_last - sigma2_current| < threshold (:106-110)
struct CpdConfiguration {
  int maxIterations = 100;
  double threshold = 1e-10;
  bool useLandmarkCorrespondence = true;
  std::optional<double> initialSigma;
  double w = 0.0;
  double lambda = 1.0;
  static constexpr const char* name = "CPD";

  bool converged(const GeneralRegistrationState& last, const GeneralRegistrationState& current, double thr) const {
    return std::fabs(last.sigma2 - current.sigma2) < thr;
  }
  gingr_config toPod() const {
    gingr_config c{};
    c.algorithm = GINGR_ALGO_CPD;
    c.max_iterations = maxIterations;
    c.threshold = threshold;
    c.use_landmark_correspondence = useLandmarkCorrespondence ? 1 : 0;
    c.has_initial_sigma = initialSigma ? 1 : 0;
    c.initial_sigma = initialSigma.value_or(0.0);
    c.w = w;
    c.lambda = lambda;
    return c;
  }
};

// registration/config/ICP.scala:54-66; converged: never (:57-58); sigma2 annealed linearly (:65)
struct IcpConfiguration {
  int maxIterations = 100;
  double threshold = 1e-10;
  bool useLandmarkCorrespondence = true;
  double initialSigma = 100.0;
  double endSigma = 1.0;
  bool reverseCorrespondenceDirection = false;
  ICPCorrespondenceMethod correspondenceMethod = ICPCorrespondenceMethod::TriangularClosestPoint;
  static constexpr const char* name = "ICP";

  double sigmaStep() const { return (initialSigma - endSigma) / static_cast<double>(maxIterations); }
  bool converged(const GeneralRegistrationState&, const GeneralRegistrationState&, double) const { return false; }
  gingr_config toPod() const {
    gingr_config c{};
    c.algorithm = GINGR_ALGO_ICP;
    c.max_iterations = maxIterations;
    c.threshold = threshold;
    c.use_landmark_correspondence = useLandmarkCorrespondence ? 1 : 0;
    c.has_initial_sigma = 1;
    c.initial_sigma = initialSigma;
    c.end_sigma = endSigma;
    c.reverse_correspondence_direction = reverseCorrespondenceDirection ? 1 : 0;
    c.correspondence_method = static_cast<int32_t>(correspondenceMethod);
    return c;
  }
};

// sampling/evaluators/IndependentPointDistanceEvaluator.scala:26-32
enum class EvaluationMode : int32_t { ModelToTargetEvaluation = GINGR_EVAL_MODEL_TO_TARGET,
                                      TargetToModelEvaluation = GINGR_EVAL_TARGET_TO_MODEL, SymmetricEvaluation = GINGR_EVAL_SYMMETRIC };

// ProbabilisticSettings(IndependentPoints(state, uncertainty, mode, evaluatedPoints), randomMixture)
// (api/GingrAlgorithm.scala:40-50, sampling/Evaluator.scala:43-60) with the widths of Generator.DefaultRandom
// (sampling/Generator.scala:27-83).  Empty id lists: all points are compared.
struct ProbabilisticSettings {
  double uncertainty = 1.0;
  EvaluationMode mode = EvaluationMode::ModelToTargetEvaluation;
  double randomMixture = 0.5;
  std::vector<int32_t> modelPointIds, targetPointIds;
  std::array<double, 3> rotationSdev{0.01, 0.01, 0.01};    // yaw, pitch, roll
  std::array<double, 3> translationSdev{0.1, 0.1, 0.1};
  std::array<double, 3> shapeSteps{1.0, 0.1, 0.01};

  gingr_mcmc_settings toPod() const {
    gingr_mcmc_settings m{};
    m.random_mixture = randomMixture;
    m.uncertainty = uncertainty;
    m.evaluation_mode = static_cast<int32_t>(mode);
    for (int d = 0; d < 3; ++d) {
      m.rot_sdev[d] = rotationSdev[d];
      m.trans_sdev[d] = translationSdev[d];
      m.shape_sdev[d] = shapeSteps[d];
    }
    return m;
  }
};

template <class Config>
class GingrAlgorithm;

// scalismo PointDistributionModel on the device
class Model {
 public:
  // basis: COLUMN-major [3M x r] with leading dimension ld (Breeze layout); tri may be empty (CPD only)
  Model(const Context& ctx, int M, int r, const double* ref, const double* mean, const double* basis, int64_t ld,
        const double* variance, const int32_t* tri = nullptr, int T = 0)
      : ctx_(&ctx), M_(M), r_(r) {
    ctx.check(gingr_model_upload(ctx.handle(), M, r, ref, mean, basis, ld, variance, tri, T, &h_));
  }
  // GPMMTriangleMesh3D(reference, relativeTolerance).GaussianMixture(pars), api/gpmm/GPMMHelper.scala:99-129, on the device
  static Model gaussianMixture(const Context& ctx, int M, const double* ref, const int32_t* tri, int T,
                               const std::vector<double>& sigma, const std::vector<double>& scaling,
                               double relativeTolerance = 0.01, int maxRank = 0) {
    if (sigma.size() != scaling.size() || sigma.empty()) throw Error(GINGR_ERR_ARG, "one scaling per sigma");
    Model m(ctx);
    int32_t rank = 0;
    ctx.check(gingr_gpmm_gaussian_mixture(ctx.handle(), M, ref, tri, T, static_cast<int32_t>(sigma.size()), sigma.data(),
                                          scaling.data(), relativeTolerance, maxRank, &m.h_, &rank));
    m.M_ = M;
    m.r_ = rank;
    return m;
  }
  // the mirror-symmetric Gaussian (mixture) kernel about the plane x = 0 (gingr_gpmm_gaussian_symmetric), on the device;
  // the caller centres the template on that plane
  static Model gaussianSymmetric(const Context& ctx, int M, const double* ref, const int32_t* tri, int T,
                                 const std::vector<double>& sigma, const std::vector<double>& scaling,
                                 double relativeTolerance = 0.01, int maxRank = 0) {
    if (sigma.size() != scaling.size() || sigma.empty()) throw Error(GINGR_ERR_ARG, "one scaling per sigma");
    Model m(ctx);
    int32_t rank = 0;
    ctx.check(gingr_gpmm_gaussian_symmetric(ctx.handle(), M, ref, tri, T, static_cast<int32_t>(sigma.size()), sigma.data(),
                                            scaling.data(), relativeTolerance, maxRank, &m.h_, &rank));
    m.M_ = M;
    m.r_ = rank;
    return m;
  }
  // the inverse-Laplacian look-up kernel scaling (L + gamma I)^-1 (pinv for gamma = 0) of the triangle graph
  // (gingr_gpmm_inverse_laplacian), on the device; at most 6000 vertices
  static Model inverseLaplacian(const Context& ctx, int M, const double* ref, const int32_t* tri, int T, double scaling,
                                double gamma, double relativeTolerance = 0.01, int maxRank = 0) {
    Model m(ctx);
    int32_t rank = 0;
    if (ctx.check(gingr_gpmm_inverse_laplacian(ctx.handle(), M, ref, tri, T, scaling, gamma, relativeTolerance, maxRank, &m.h_,
                                               &rank)) == GINGR_MODEL_FLEXIBILITY)
      throw Error(GINGR_MODEL_FLEXIBILITY, "L + gamma I is not numerically positive definite");
    m.M_ = M;
    m.r_ = rank;
    return m;
  }
  // model.newReference(newRef, NearestNeighborInterpolator()), registration/SimpleRegistrator.scala:90-92
  Model newReference(int M2, const double* ref, const int32_t* tri = nullptr, int T = 0) const {
    Model m(*ctx_);
    ctx_->check(gingr_model_new_reference(ctx_->handle(), h_, M2, ref, tri, T, &m.h_));
    m.M_ = M2;
    m.r_ = r_;
    return m;
  }
  // model.transform(R, t).posterior(trainingData) as a new model (GingrAlgorithm.scala:299-300; scalismo, SURVEY.md A3).
  // R row-major [9], t [3]; noiseKind 0: noise[n] isotropic variances, 1: noise[9n] covariances.  Throws Error with code
  // GINGR_MODEL_FLEXIBILITY where the posterior fails.
  Model posterior(const std::array<double, 9>& R, const std::array<double, 3>& t, const std::vector<int32_t>& pid,
                  const std::vector<double>& points, int noiseKind, const std::vector<double>& noise) const {
    const size_t n = pid.size();
    if (points.size() != 3 * n || noise.size() != (noiseKind == 0 ? n : 9 * n)) throw Error(GINGR_ERR_ARG, "observation array sizes");
    Model m(*ctx_);
    if (ctx_->check(gingr_model_posterior(ctx_->handle(), h_, R.data(), t.data(), static_cast<int32_t>(n), pid.data(), points.data(),
                                          noiseKind, noise.data(), &m.h_)) == GINGR_MODEL_FLEXIBILITY)
      throw Error(GINGR_MODEL_FLEXIBILITY, "posterior failed (ModelFlexibilityError)");
    m.M_ = M_;
    m.r_ = r_;
    return m;
  }
  // ModelFittingParameters.modelInstanceShapePoseScale, api/ModelFittingParameters.scala:130-143
  std::vector<double> instance(const ModelFittingParameters& p) const {
    GeneralRegistrationState s;
    s.modelParameters = p;
    const gingr_state pod = s.toPod();
    std::vector<double> fit(static_cast<size_t>(3) * M_);
    ctx_->check(gingr_model_instance(ctx_->handle(), h_, &pod, p.shape.data(), fit.data()));
    return fit;
  }
  ~Model() { if (h_) gingr_model_destroy(h_); }
  Model(Model&& o) noexcept : ctx_(o.ctx_), h_(o.h_), M_(o.M_), r_(o.r_) { o.h_ = nullptr; }
  Model(const Model&) = delete;
  Model& operator=(const Model&) = delete;
  gingr_model* handle() const { return h_; }
  int points() const { return M_; }
  int rank() const { return r_; }

 private:
  template <class Config>
  friend class GingrAlgorithm;
  explicit Model(const Context& ctx) : ctx_(&ctx) {}
  const Context* ctx_;
  gingr_model* h_ = nullptr;
  int M_ = 0, r_ = 0;
};

// target TriangleMesh (or point set) on the device
class Target {
 public:
  Target(const Context& ctx, int N, const double* pts, const int32_t* tri = nullptr, int T = 0) : N_(N) {
    ctx.check(gingr_target_upload(ctx.handle(), N, pts, tri, T, &h_));
  }
  ~Target() { if (h_) gingr_target_destroy(h_); }
  Target(Target&& o) noexcept : h_(o.h_), N_(o.N_) { o.h_ = nullptr; }
  Target(const Target&) = delete;
  Target& operator=(const Target&) = delete;
  gingr_target* handle() const { return h_; }
  int points() const { return N_; }

 private:
  gingr_target* h_ = nullptr;
  int N_ = 0;
};

// GingrAlgorithm[State, Config] (api/GingrAlgorithm.scala:65-302) for Config = CpdConfiguration / IcpConfiguration
template <class Config>
class GingrAlgorithm {
 public:
  using State = GeneralRegistrationState;
  GingrAlgorithm(const Context& ctx, const Model& model, const Target& target, Config config = Config())
      : ctx_(&ctx), model_(&model), config_(std::move(config)) {
    const gingr_config pod = config_.toPod();
    ctx.check(gingr_registration_create(ctx.handle(), model.handle(), target.handle(), &pod, &h_));
  }
  ~GingrAlgorithm() { if (h_) gingr_registration_destroy(h_); }
  GingrAlgorithm(const GingrAlgorithm&) = delete;
  GingrAlgorithm& operator=(const GingrAlgorithm&) = delete;

  const char* name() const { return Config::name; }
  const Config& config() const { return config_; }

  // GeneralRegistrationState.landmarkCorrespondences resolved by the caller (GeneralRegistrationState.scala:43-62)
  void setLandmarks(const std::vector<int32_t>& pid, const std::vector<double>& points, const std::vector<double>& cov) {
    if (points.size() != 3 * pid.size() || cov.size() != 9 * pid.size()) throw Error(GINGR_ERR_ARG, "landmark array sizes");
    ctx_->check(gingr_registration_set_landmarks(h_, static_cast<int32_t>(pid.size()), pid.data(), points.data(), cov.data()));
  }

  // GeneralRegistrationState.apply (:136-178) + initializeState (CPD.scala:92-103 / ICP.scala:74-86)
  State initializeState(GlobalTransformationType transform = GlobalTransformationType::RigidTransforms) const {
    State g;
    g.globalTransformation = transform;
    g.modelParameters.shape.assign(model_->rank(), 0.0);
    return initializeState(g);
  }
  State initializeState(State general) const {
    if (static_cast<int>(general.modelParameters.shape.size()) != model_->rank())
      throw Error(GINGR_ERR_ARG, "shape parameters must have the model's rank");
    gingr_state pod = general.toPod();
    general.fit.resize(static_cast<size_t>(3) * model_->points());
    ctx_->check(gingr_initialize_state(h_, &pod, general.modelParameters.shape.data(), general.fit.data()));
    general.fromPod(pod);
    return general;
  }

  // GingrAlgorithm.update (:192-254); the returned fit is already the refreshed one of GingrGeneratorWrapper.propose
  State update(const State& current, bool probabilistic = false, uint64_t seed = 0) const {
    const gingr_state in = current.toPod();
    gingr_state out{};
    State next = current;
    next.fit.resize(static_cast<size_t>(3) * model_->points());
    std::vector<double> alpha(current.modelParameters.shape.size());
    ctx_->check(gingr_update(h_, &in, current.modelParameters.shape.data(), probabilistic ? 1 : 0, seed, &out, alpha.data(),
                             next.fit.data()));
    next.fromPod(out);
    next.modelParameters.shape = std::move(alpha);
    return next;
  }

  // GingrAlgorithm.computePosterior(current) (:281-302): the posterior model of the configuration's correspondences,
  // uncertainties and landmarks at `current`.  Throws Error with code GINGR_MODEL_FLEXIBILITY where the posterior fails.
  Model computePosterior(const State& current) const {
    const gingr_state in = current.toPod();
    Model m(*ctx_);
    if (ctx_->check(gingr_registration_posterior_model(h_, &in, current.modelParameters.shape.data(), &m.h_)) == GINGR_MODEL_FLEXIBILITY)
      throw Error(GINGR_MODEL_FLEXIBILITY, "posterior failed (ModelFlexibilityError)");
    m.M_ = model_->points();
    m.r_ = model_->rank();
    return m;
  }

  // GingrGeneratorWrapper.propose (GingrGeneratorWrapper.scala:28-39): update, refreshed fit, iteration + 1, generatedBy
  State propose(const State& current, bool probabilistic = false, uint64_t seed = 0) const {
    State next = update(current, probabilistic, seed);
    next.iteration = current.iteration + 1;
    next.generatedBy = probabilistic ? "Stochastic" : "Deterministic";
    return next;
  }

  // Deterministic GingrAlgorithm.run (:115-175): the chain yields the initial state first, so maxIterations - 1 proposals
  // are made; stops on converged(last, current) or ModelFlexibilityError; a state still at status None ends as Converged /
  // MaxIteration (:165-171).
  State run(State state, const std::function<void(const State&)>& callBackLogger = nullptr) const {
    std::optional<State> last;
    FittingStatus final_status = FittingStatus::MaxIteration;
    for (int k = 0; k < config_.maxIterations; ++k) {
      if (k > 0) state = propose(state);
      if (callBackLogger) callBackLogger(state);
      const bool converged = last && config_.converged(*last, state, config_.threshold);
      const bool error = state.status == FittingStatus::ModelFlexibilityError;
      last = state;
      if (converged) {
        final_status = FittingStatus::Converged;
        break;
      }
      if (error) break;
    }
    if (state.status == FittingStatus::None) state.status = final_status;
    return state;
  }

  // ---- probabilistic registration (GingrAlgorithm.run with ProbabilisticSettings, :115-190) ----
  void configureProbabilistic(const ProbabilisticSettings& s) {
    const gingr_mcmc_settings pod = s.toPod();
    ctx_->check(gingr_mcmc_configure(h_, &pod, s.modelPointIds.empty() ? nullptr : s.modelPointIds.data(),
                                     static_cast<int32_t>(s.modelPointIds.size()),
                                     s.targetPointIds.empty() ? nullptr : s.targetPointIds.data(),
                                     static_cast<int32_t>(s.targetPointIds.size())));
  }
  // (Prior, Distance) log values of the evaluators (sampling/Evaluator.scala:43-60); their sum is the product evaluator.
  // Replaces the device-resident state: call before initializeState, not between it and a chain.
  std::pair<double, double> logValue(const State& state) const {
    const gingr_state pod = state.toPod();
    double out[2] = {0.0, 0.0};
    ctx_->check(gingr_evaluate_log_value(h_, &pod, state.modelParameters.shape.data(), out));
    return {out[0], out[1]};
  }
  // `iters` Metropolis-Hastings steps on the device from the device-resident state (initializeState / update first)
  void mcmcChain(int iters, uint64_t seed) { ctx_->check(gingr_mcmc_chain(h_, iters, seed)); }
  State downloadState() const { return download(&gingr_state_download); }
  State mcmcBest() const { return download(&gingr_mcmc_best); }
  // run(...) with probabilisticSettings: maxIterations - 1 steps, the best sample is returned (:160-171)
  State runProbabilistic(const State& initial, const ProbabilisticSettings& settings, uint64_t seed = 0) {
    configureProbabilistic(settings);
    initializeState(initial);
    mcmcChain(config_.maxIterations > 1 ? config_.maxIterations - 1 : 0, seed);
    State best = mcmcBest();
    if (best.status == FittingStatus::None) best.status = FittingStatus::MaxIteration;
    return best;
  }

  gingr_registration* handle() const { return h_; }

 private:
  State download(int32_t (*fn)(gingr_registration*, gingr_state*, double*, double*)) const {
    State s;
    gingr_state pod{};
    s.modelParameters.shape.resize(model_->rank());
    s.fit.resize(static_cast<size_t>(3) * model_->points());
    ctx_->check(fn(h_, &pod, s.modelParameters.shape.data(), s.fit.data()));
    s.fromPod(pod);
    return s;
  }
  const Context* ctx_;
  const Model* model_;
  Config config_;
  gingr_registration* h_ = nullptr;
};

using CpdRegistration = GingrAlgorithm<CpdConfiguration>;  // registration/config/CPD.scala:117-160
using IcpRegistration = GingrAlgorithm<IcpConfiguration>;  // registration/config/ICP.scala:84-110

}  // namespace gingr
