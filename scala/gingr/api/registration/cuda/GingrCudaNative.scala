/*
 * Panama FFM (JDK 22+) binding of libgingr_cuda.so -- the C ABI declared in include/gingr_cuda.h.
 * NOT COMPILED IN THIS REPOSITORY'S CI: the build image has no JVM / sbt / scalismo.  It is the reference-side
 * stub a GiNGR maintainer adds (see INTEGRATION.md).  Lives under package gingr.api so that it may call the
 * private[api] updaters of GeneralRegistrationState (api/GeneralRegistrationState.scala:75-102).
 */
package gingr.api.registration.cuda

import java.lang.foreign.*
import java.lang.foreign.ValueLayout.*
import java.lang.invoke.MethodHandle

object GingrCudaNative {
  private val linker = Linker.nativeLinker()
  private val arena  = Arena.global()
  private val lib    = SymbolLookup.libraryLookup(sys.props.getOrElse("gingr.cuda.lib", "libgingr_cuda.so"), arena)

  private def fn(name: String, ret: MemoryLayout, args: MemoryLayout*): MethodHandle =
    linker.downcallHandle(lib.find(name).orElseThrow(), FunctionDescriptor.of(ret, args*))

  /** struct gingr_state (include/gingr_cuda.h): 12 doubles then 4 int32 = 112 bytes. */
  val STATE: StructLayout = MemoryLayout.structLayout(
    JAVA_DOUBLE.withName("scale"),
    MemoryLayout.sequenceLayout(3, JAVA_DOUBLE).withName("translation"),
    MemoryLayout.sequenceLayout(3, JAVA_DOUBLE).withName("euler"),
    MemoryLayout.sequenceLayout(3, JAVA_DOUBLE).withName("center"),
    JAVA_DOUBLE.withName("sigma2"),
    JAVA_DOUBLE.withName("step_length"),
    JAVA_INT.withName("global_transformation"),
    JAVA_INT.withName("iteration"),
    JAVA_INT.withName("status"),
    JAVA_INT.withName("rank")
  )

  /** struct gingr_config: int32 x2, double, int32 x2, double x4, int32 x2 (natural alignment, 64 bytes). */
  val CONFIG: StructLayout = MemoryLayout.structLayout(
    JAVA_INT.withName("algorithm"),
    JAVA_INT.withName("max_iterations"),
    JAVA_DOUBLE.withName("threshold"),
    JAVA_INT.withName("use_landmark_correspondence"),
    JAVA_INT.withName("has_initial_sigma"),
    JAVA_DOUBLE.withName("initial_sigma"),
    JAVA_DOUBLE.withName("w"),
    JAVA_DOUBLE.withName("lambda"),
    JAVA_DOUBLE.withName("end_sigma"),
    JAVA_INT.withName("reverse_correspondence_direction"),
    JAVA_INT.withName("correspondence_method")
  )

  val ctxCreate      = fn("gingr_ctx_create", JAVA_INT, JAVA_INT, ADDRESS)
  val ctxDestroy     = fn("gingr_ctx_destroy", JAVA_INT, ADDRESS)
  val lastError      = fn("gingr_last_error", ADDRESS, ADDRESS)
  val modelUpload    = fn("gingr_model_upload", JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG,
                          ADDRESS, ADDRESS, JAVA_INT, ADDRESS)
  val modelDestroy   = fn("gingr_model_destroy", JAVA_INT, ADDRESS)
  val targetUpload   = fn("gingr_target_upload", JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS)
  val targetDestroy  = fn("gingr_target_destroy", JAVA_INT, ADDRESS)
  val regCreate      = fn("gingr_registration_create", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  val regDestroy     = fn("gingr_registration_destroy", JAVA_INT, ADDRESS)
  val regLandmarks   = fn("gingr_registration_set_landmarks", JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS)
  val initializeState = fn("gingr_initialize_state", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  val update         = fn("gingr_update", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS)
  val cpdEstep       = fn("gingr_cpd_estep", JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_DOUBLE, JAVA_DOUBLE, ADDRESS,
                          ADDRESS, ADDRESS)
  val icpClosest     = fn("gingr_icp_closest", JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT,
                          ADDRESS, ADDRESS, ADDRESS, ADDRESS)

  // probabilistic registration (SURVEY.md 8f-1) and multi-resolution hand-over (8f-2)
  /** struct gingr_mcmc_settings: double x2, int32 x2, double x9 = 96 bytes. */
  val MCMC_SETTINGS: StructLayout = MemoryLayout.structLayout(
    JAVA_DOUBLE.withName("random_mixture"),
    JAVA_DOUBLE.withName("uncertainty"),
    JAVA_INT.withName("evaluation_mode"),
    JAVA_INT.withName("reserved"),
    MemoryLayout.sequenceLayout(3, JAVA_DOUBLE).withName("rot_sdev"),
    MemoryLayout.sequenceLayout(3, JAVA_DOUBLE).withName("trans_sdev"),
    MemoryLayout.sequenceLayout(3, JAVA_DOUBLE).withName("shape_sdev")
  )
  val mcmcConfigure  = fn("gingr_mcmc_configure", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT)
  val evaluateLogValue = fn("gingr_evaluate_log_value", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  val logTransition  = fn("gingr_log_transition_probability", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  val mcmcChain      = fn("gingr_mcmc_chain", JAVA_INT, ADDRESS, JAVA_INT, JAVA_LONG)
  val mcmcBatch      = fn("gingr_mcmc_batch", JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_LONG)
  val mcmcStats      = fn("gingr_mcmc_stats", JAVA_INT, ADDRESS, ADDRESS, ADDRESS)
  val mcmcBest       = fn("gingr_mcmc_best", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  val stateDownload  = fn("gingr_state_download", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  val modelNewReference = fn("gingr_model_new_reference", JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS)
  // GPMM construction on the device (api/gpmm/GPMMHelper.scala:99-129) and the way back into scalismo's storage
  val gpmmGaussianMixture = fn("gingr_gpmm_gaussian_mixture", JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT,
                               ADDRESS, ADDRESS, JAVA_DOUBLE, JAVA_INT, ADDRESS, ADDRESS)
  // the mirror-symmetric kernel about x = 0 (scalismo's symmetrised Gaussian kernel), same arguments
  val gpmmGaussianSymmetric = fn("gingr_gpmm_gaussian_symmetric", JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT,
                                 ADDRESS, ADDRESS, JAVA_DOUBLE, JAVA_INT, ADDRESS, ADDRESS)
  // the inverse-Laplacian look-up kernel of the triangle graph (LaplacianHelper.scala:26-55)
  val gpmmInverseLaplacian = fn("gingr_gpmm_inverse_laplacian", JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_DOUBLE,
                                JAVA_DOUBLE, JAVA_DOUBLE, JAVA_INT, ADDRESS, ADDRESS)
  val modelDownload  = fn("gingr_model_download", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS)

  // the remaining entry points of include/gingr_cuda.h (every exported function has a handle here; tests/test_scala_shim.py
  // checks names, arity and argument classes against the header)
  val version        = fn("gingr_version", JAVA_INT)
  val ctxStream      = fn("gingr_ctx_stream", ADDRESS, ADDRESS)
  val ctxSynchronize = fn("gingr_ctx_synchronize", JAVA_INT, ADDRESS)
  val ctxLaunchCount = fn("gingr_ctx_launch_count", JAVA_LONG, ADDRESS)
  val commUniqueId   = fn("gingr_comm_unique_id", JAVA_INT, ADDRESS)
  val commInit       = fn("gingr_comm_init", JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS)
  // other/algorithms/cpd/BCPD.scala:167-184, :200-209 (nu, nu', N-hat, x-hat in one call)
  val bcpdEstep      = fn("gingr_bcpd_estep", JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_DOUBLE, JAVA_DOUBLE,
                          JAVA_DOUBLE, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  // CPD.scala:81-90 computeInitialSigma2
  val cpdInitialSigma2 = fn("gingr_cpd_initial_sigma2", JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS)
  // ClosestPointRegistrator.scala:34-45 closestPointCorrespondenceReversal
  val icpClosestReversal = fn("gingr_icp_closest_reversal", JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT,
                              ADDRESS, ADDRESS, ADDRESS)
  // GingrAlgorithm.scala:281-302 (model.transform(rigid).posterior(observations), mean only), :215 / :236 (coefficients), :93-95 (instance)
  val posteriorMean  = fn("gingr_posterior_mean", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT,
                          ADDRESS, ADDRESS, ADDRESS)
  // per-vertex 3 x 3 covariance of the same posterior (what PosteriorHelper colour-maps)
  val posteriorCov   = fn("gingr_posterior_covariance", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT,
                          ADDRESS, ADDRESS)
  // GingrAlgorithm.scala:299-300 model.transform(rigid).posterior(trainingData) as a new model handle, :281-302 computePosterior
  val modelPosterior = fn("gingr_model_posterior", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT,
                          ADDRESS, ADDRESS)
  val registrationPosteriorModel = fn("gingr_registration_posterior_model", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  val posteriorModelProfile = fn("gingr_posterior_model_profile", JAVA_INT, ADDRESS, ADDRESS, ADDRESS)
  val coefficients   = fn("gingr_coefficients", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  // the r x r solve of the regression alone (pinv(Mx) * rhs as a Cholesky solve): A, nrhs rows of B -> L, L^-1 B^T rows, A^-1 b_0
  val spdSolve       = fn("gingr_spd_solve", JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT,
                          ADDRESS)
  val modelInstance  = fn("gingr_model_instance", JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS)
  // device-resident loops: `iters` x update() without the host round trip (GingrAlgorithm.run's deterministic branch, :179-189)
  val updateChain    = fn("gingr_update_chain", JAVA_INT, ADDRESS, JAVA_INT)
  val updateChainSampled = fn("gingr_update_chain_sampled", JAVA_INT, ADDRESS, JAVA_INT, JAVA_LONG)
  val updateBatch    = fn("gingr_update_batch", JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_LONG)
  val setProfiling   = fn("gingr_registration_set_profiling", JAVA_INT, ADDRESS, JAVA_INT)
  val getProfile     = fn("gingr_registration_get_profile", JAVA_INT, ADDRESS, ADDRESS, ADDRESS)

  def check(code: Int, ctx: MemorySegment): Int = {
    if (code < 0) {
      val msg = lastError.invoke(ctx).asInstanceOf[MemorySegment].reinterpret(4096).getString(0)
      throw new RuntimeException(s"libgingr_cuda error $code: $msg")
    }
    code
  }
}
