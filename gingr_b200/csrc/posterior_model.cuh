// posterior_model.cuh -- the GP posterior as a new device model (included by update.cu behind gpmm.cuh).
//
// scalismo's model.transform(R, t).posterior(obs) (SURVEY.md A3; GingrAlgorithm.scala:68, :281-302) is again a low-rank
// model: reference R ref + t, mean R (mean + Phi D c), basis (I (x) R) Phi U, variance s with U diag(s) U^T = D Mx^-1 D.
// The system Mx = L L^T is factorised with the r rows sqrt(lambda_k) e_k riding along (posterior_core / the registration's
// raw system), which leaves B = D L^-T, B B^T = D Mx^-1 D.  One-sided Jacobi on the columns of B (gpmm_jacobi, the KL
// basis of the GPMM build) gives B V = [g_j] with orthogonal columns: s_j = |g_j|^2, U_j = g_j / |g_j|.  The basis
// Phi U is the one big product (3M x r x r) and runs on the FP64 tensor pipe (basis_rotate.cu) with the 1 / |g_j| and
// the pose in its epilogue.
// Zero variances: row and column k of B are exactly zero for lambda_k = 0 (Mx has the unit row / column k there, so L
// has too, and the Jacobi never rotates a zero column); such an index gets the unit vector e_k and variance 0.
#pragma once

namespace gingr {

// U[a][jj] = column src[jj] of G (column-major [r][r]), or e_k for src[jj] = -1 - k; zero padding to [rp][rp]
__global__ void posterior_u_kernel(int r, int rp, const double* __restrict__ G, const int* __restrict__ src, double* __restrict__ U) {
  const int a = blockIdx.y;
  for (int jj = blockIdx.x * blockDim.x + threadIdx.x; jj < rp; jj += gridDim.x * blockDim.x) {
    double v = 0.0;
    if (a < r && jj < r) {
      const int s = src[jj];
      v = s >= 0 ? G[(size_t)s * r + a] : (a == -1 - s ? 1.0 : 0.0);
    }
    U[(size_t)a * rp + jj] = v;
  }
}

// ref2_i = R ref_i + t,  mean2_i = R (mean_i + inst_i)  with inst = Phi D c
__global__ void posterior_mean_ref_kernel(int M, const double* __restrict__ ref, const double* __restrict__ mean,
                                          const double* __restrict__ inst, const double* __restrict__ ds,
                                          double* __restrict__ ref2, double* __restrict__ mean2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const double* R = ds + DS_R;
  double p[3], q[3];
  for (int d = 0; d < 3; ++d) {
    p[d] = ref[3 * i + d];
    q[d] = mean[3 * i + d] + inst[3 * i + d];
  }
  for (int d = 0; d < 3; ++d) {
    ref2[3 * i + d] = R[3 * d] * p[0] + R[3 * d + 1] * p[1] + R[3 * d + 2] * p[2] + ds[DS_T + d];
    mean2[3 * i + d] = R[3 * d] * q[0] + R[3 * d + 1] * q[1] + R[3 * d + 2] * q[2];
  }
}

}  // namespace gingr

static int32_t posterior_model_finish(gingr_ctx* ctx, const gingr_model* m, const double* d_B, const double* d_c,
                                      const double* d_ds, gingr::PosteriorModelEvents& ev, gingr_model** out) {
  const int M = m->M, r = m->r, rp = m->rp;
  cudaStream_t st = ctx->stream;
  // ---- eigenpairs of D Mx^-1 D: Jacobi on the columns of B (column-major copy, column length r)
  DevBuf<double> G, norm2, U, scale, inst;
  DevBuf<int> flag, src;
  GINGR_CUDA_TRY(ctx, G.alloc((size_t)r * r));
  GINGR_CUDA_TRY(ctx, norm2.alloc(r));
  GINGR_CUDA_TRY(ctx, flag.alloc(4));
  GINGR_CUDA_TRY(ctx, U.alloc((size_t)rp * rp));
  GINGR_CUDA_TRY(ctx, scale.alloc(rp));
  GINGR_CUDA_TRY(ctx, src.alloc(rp));
  GINGR_CUDA_TRY(ctx, inst.alloc((size_t)3 * M));
  GINGR_TRY(transpose_enqueue(ctx, r, d_B, rp, G.p, r));
  std::vector<double> n2;
  int sweeps = 0;
  GINGR_TRY(gpmm_jacobi(ctx, r, r, G.p, flag.p, norm2.p, &n2, &sweeps));
  std::vector<double> sl(rp);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(sl.data(), m->sqrt_lambda.p, sizeof(double) * rp, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  // columns by variance, descending (stable); the zero-variance indices last, as unit vectors
  std::vector<int> order, hsrc(rp, 0);
  for (int j = 0; j < r; ++j)
    if (sl[j] > 0.0) order.push_back(j);
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return n2[x] > n2[y]; });
  std::vector<double> hscale(rp, 0.0), sl2(rp, 0.0);
  int jj = 0;
  for (int j : order) {
    const double nrm = sqrt(n2[j]);
    hsrc[jj] = j;
    sl2[jj] = nrm;
    hscale[jj] = nrm > 0.0 ? 1.0 / nrm : 0.0;
    ++jj;
  }
  for (int k = 0; k < r; ++k)
    if (!(sl[k] > 0.0)) {
      hsrc[jj] = -1 - k;
      hscale[jj] = 1.0;
      ++jj;
    }
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(src.p, hsrc.data(), sizeof(int) * rp, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(scale.p, hscale.data(), sizeof(double) * rp, cudaMemcpyHostToDevice, st));
  gingr::posterior_u_kernel<<<dim3(ceil_div(rp, 256), rp), 256, 0, st>>>(r, rp, G.p, src.p, U.p);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(ev.record(ctx, 2));
  // ---- the new model: basis on DMMA, mean and reference, topology, regression constants
  std::unique_ptr<gingr_model> m2(new gingr_model());
  m2->ctx = ctx;
  m2->M = M; m2->r = r; m2->rp = rp; m2->m0 = 0; m2->Ml = M;
  GINGR_CUDA_TRY(ctx, m2->ref.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, m2->mean.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, m2->sqrt_lambda.alloc(rp));
  GINGR_CUDA_TRY(ctx, m2->phi.alloc((size_t)3 * M * rp));
  GINGR_TRY(basis_rotate_enqueue(ctx, 3 * M, rp, m->phi.p, U.p, scale.p, d_ds + DS_R, m2->phi.p));
  GINGR_TRY(ev.record(ctx, 3));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m2->sqrt_lambda.p, sl2.data(), sizeof(double) * rp, cudaMemcpyHostToDevice, st));
  GINGR_TRY(gemv_rows_enqueue(ctx, 3 * M, r, rp, m->phi.p, 1, d_c, nullptr, inst.p, nullptr, m->sqrt_lambda.p));
  gingr::posterior_mean_ref_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, m->ref.p, m->mean.p, inst.p, d_ds, m2->ref.p, m2->mean.p);
  GINGR_LAUNCHED(ctx);
  m2->T = m->T;
  if (m->T > 0) {
    GINGR_CUDA_TRY(ctx, m2->tri.alloc(m->tri.n));
    GINGR_CUDA_TRY(ctx, m2->adj_off.alloc(m->adj_off.n));
    GINGR_CUDA_TRY(ctx, m2->adj.alloc(m->adj.n));
    GINGR_CUDA_TRY(ctx, m2->boundary.alloc(m->boundary.n));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m2->tri.p, m->tri.p, sizeof(int32_t) * m->tri.n, cudaMemcpyDeviceToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m2->adj_off.p, m->adj_off.p, sizeof(int32_t) * m->adj_off.n, cudaMemcpyDeviceToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m2->adj.p, m->adj.p, sizeof(int32_t) * m->adj.n, cudaMemcpyDeviceToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m2->boundary.p, m->boundary.p, m->boundary.n, cudaMemcpyDeviceToDevice, st));
  }
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));   // sl2 is a host vector
  // not orthonormal in general (a re-referenced source basis): the constants are built as for an upload
  GINGR_TRY(model_build_constants(ctx, m2.get()));
  GINGR_TRY(ev.record(ctx, 4));
  GINGR_CUDA_TRY(ctx, cudaEventSynchronize(ev.e[4]));
  float ms[4];
  for (int k = 0; k < 4; ++k) GINGR_CUDA_TRY(ctx, cudaEventElapsedTime(&ms[k], ev.e[k], ev.e[k + 1]));
  float whole = 0.f;
  GINGR_CUDA_TRY(ctx, cudaEventElapsedTime(&whole, ev.e[0], ev.e[4]));
  for (int k = 0; k < 4; ++k) ctx->posterior_model_ms[k] = ms[k];
  ctx->posterior_model_ms[4] = whole;
  ctx->posterior_model_sweeps = sweeps;
  *out = m2.release();
  return GINGR_OK;
}

extern "C" {

// GingrAlgorithm.computePosterior(current) (GingrAlgorithm.scala:281-302): the posterior phase of the iteration at the
// given state (correspondences, uncertainties, landmarks) with the raw system kept, then the model as above.
int32_t gingr_registration_posterior_model(gingr_registration* g, const gingr_state* state, const double* alpha,
                                           gingr_model** out) {
  if (!g || !state || !alpha || !out) return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_registration_posterior_model: bad argument");
  *out = nullptr;
  gingr_ctx* ctx = g->ctx;
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_registration_posterior_model: single-GPU entry point");
  const gingr_model* m = g->model;
  const int r = m->r, rp = m->rp;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  gingr::PosteriorModelEvents ev;
  GINGR_TRY(ev.create(ctx));
  GINGR_TRY(ev.record(ctx, 0));
  mcmc_invalidate(g);
  g->state_valid = false;
  GINGR_TRY(upload_state(g, state, alpha));
  GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R));
  GINGR_CUDA_TRY(ctx, g->Mx_raw.alloc((size_t)(r + 1) * rp));
  const bool keep_raw = g->keep_raw;   // restored: the captured iteration graphs do not keep the raw system
  g->keep_raw = true;
  const int32_t rc = enqueue_posterior_phase(g);
  g->keep_raw = keep_raw;
  GINGR_TRY(rc);
  // [Mx ; rhs ; D] factorised once more: the raw system, the rows of D riding along
  cudaStream_t st = ctx->stream;
  DevBuf<double> sys, c;
  DevBuf<int> info, flags;
  CholWs cws;
  GINGR_CUDA_TRY(ctx, sys.alloc((size_t)(2 * r + 8) * rp));
  GINGR_CUDA_TRY(ctx, c.alloc(rp));
  GINGR_CUDA_TRY(ctx, info.alloc(4));
  GINGR_CUDA_TRY(ctx, flags.alloc((size_t)ceil_div(r, 64) + 8));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(flags.p, 0, sizeof(int) * flags.n, st));
  GINGR_TRY(cws.alloc(ctx, r, 2 * r + 1));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(sys.p, 0, sizeof(double) * (size_t)(2 * r + 8) * rp, st));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(info.p, 0, sizeof(int) * 4, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(sys.p, g->Mx_raw.p, sizeof(double) * (size_t)(r + 1) * rp, cudaMemcpyDeviceToDevice, st));
  gingr::posterior_model_rows_kernel<<<dim3(ceil_div(rp, 256), r), 256, 0, st>>>(r, rp, m->sqrt_lambda.p, sys.p + (size_t)(r + 1) * rp);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(cholesky_df_enqueue(ctx, r, 2 * r + 1, sys.p, rp, info.p, cws));
  GINGR_TRY(chol_backsolve_enqueue(ctx, r, sys.p, rp, sys.p + (size_t)r * rp, c.p, flags.p, &cws));
  GINGR_LAUNCH(ctx, check_finite_kernel, ceil_div(r, 256), 256, 0, st, r, c.p, info.p + 1);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(ev.record(ctx, 1));
  int hinfo[2] = {0, 0}, fail_post = 0;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(hinfo, info.p, sizeof(int) * 2, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(&fail_post, g->is.p + IS_FAIL_POST, sizeof(int), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (hinfo[0] || hinfo[1] || fail_post) return GINGR_MODEL_FLEXIBILITY;
  return posterior_model_finish(ctx, m, sys.p + (size_t)(r + 1) * rp, c.p, g->ds.p, ev, out);
}

// Test window on the iteration's posterior system (not in gingr_cuda.h): the same posterior phase as above at the given
// state, then sys [(r + 1) x r] = the kept raw system unpadded (rows 0 .. r-1 the full symmetric Mx as the MH chain reads
// it, row r the rhs) and, if non-null, wrow / u [3M] as obs_kernel wrote them.  max_cta > 0 schedules the Gram of this
// call on at most that many CTAs; the plan is rebuilt as it was afterwards and whatever captured the old plan is dropped.
GINGR_API int32_t gingr_debug_posterior_system(gingr_registration* g, const gingr_state* state, const double* alpha,
                                               int32_t max_cta, double* sys, double* wrow, double* u) {
  if (!g || !state || !alpha || !sys || max_cta < 0)
    return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_debug_posterior_system: bad argument");
  gingr_ctx* ctx = g->ctx;
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_debug_posterior_system: single-GPU entry point");
  const gingr_model* m = g->model;
  const int r = m->r, rp = m->rp, M = m->M;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int prev_cta = g->gram.ncta;
  if (max_cta > 0) {
    drop_graph(g);
    mcmc_invalidate(g);
    mcmc_drop_chain_graph(g);
    GINGR_TRY(g->gram.build(ctx, g->gram.rows, r, rp, max_cta));
  }
  static_assert(IS_FAIL_POST == IS_INFO + 1, "the posterior flags are copied as one pair");
  int hflags[2] = {0, 0};
  int32_t rc = [&]() -> int32_t {
    mcmc_invalidate(g);
    g->state_valid = false;
    GINGR_TRY(upload_state(g, state, alpha));
    GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R));
    GINGR_CUDA_TRY(ctx, g->Mx_raw.alloc((size_t)(r + 1) * rp));
    const bool keep_raw = g->keep_raw;
    g->keep_raw = true;
    const int32_t rc_post = enqueue_posterior_phase(g);
    g->keep_raw = keep_raw;
    GINGR_TRY(rc_post);
    cudaStream_t st = ctx->stream;
    GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(sys, sizeof(double) * r, g->Mx_raw.p, sizeof(double) * rp, sizeof(double) * r, r + 1,
                                          cudaMemcpyDeviceToHost, st));
    if (wrow) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(wrow, g->wrow.p, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, st));
    if (u) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(u, g->u.p, sizeof(double) * 3 * M, cudaMemcpyDeviceToHost, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(hflags, g->is.p + IS_INFO, sizeof(int) * 2, cudaMemcpyDeviceToHost, st));
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    return GINGR_OK;
  }();
  if (max_cta > 0) {   // the plan of the registration back, also after a failure
    const int32_t rb = g->gram.build(ctx, g->gram.rows, r, rp, prev_cta);
    if (rc >= 0) rc = rb;
  }
  GINGR_TRY(rc);
  return hflags[0] || hflags[1] ? GINGR_MODEL_FLEXIBILITY : GINGR_OK;
}

// Test window on the iteration's update phase (not in gingr_cuda.h): the posterior phase at the given state, then the update
// phase as an iteration runs it, with the inputs and results of every stage copied out.  Every output may be null:
//   L [r x r], z [r]     the factor and the forward-substituted rhs before the update phase (unpadded; upper triangle as stored)
//   z2 [r]               the rhs row after it: z plus the Philox normals when `probabilistic` is set
//   vec [6 x r]          c, S c, alpha*, alpha_c, q, alpha_new
//   inst_a, inst_b, newshape, u [3M]; pro_sums [10]; ds [DS_COUNT] and is [IS_COUNT] of the state block
//   alpha_out [r], fit [3M]   the committed coefficients and the refreshed fit
//   S, W0 [r x r]        the model's regression constants
// kept_factor = 1 takes the back substitution that needs the factor alone (the MH chain's kept factors).  The captured
// iteration graph and the MH memo are dropped afterwards.
GINGR_API int32_t gingr_debug_update_phase(gingr_registration* g, const gingr_state* state, const double* alpha,
                                           int32_t probabilistic, uint64_t seed, int32_t kept_factor, double* L, double* z,
                                           double* z2, double* vec, double* inst_a, double* inst_b, double* newshape,
                                           double* u, double* pro_sums, double* ds, int32_t* is, double* alpha_out,
                                           double* fit, double* S, double* W0) {
  if (!g || !state || !alpha) return gingr_fail(g ? g->ctx : nullptr, GINGR_ERR_ARG, "gingr_debug_update_phase: bad argument");
  gingr_ctx* ctx = g->ctx;
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_debug_update_phase: single-GPU entry point");
  const gingr_model* m = g->model;
  const int r = m->r, rp = m->rp, M = m->M;
  const size_t row = sizeof(double) * r, pitch = sizeof(double) * rp;
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  drop_graph(g);
  mcmc_invalidate(g);
  g->state_valid = false;
  g->host_mirror_current = false;
  GINGR_TRY(upload_state(g, state, alpha));
  GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R));
  GINGR_TRY(enqueue_posterior_phase(g));
  const double* Mx = g->Mx.p;
  if (L) GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(L, row, Mx, pitch, row, r, cudaMemcpyDeviceToHost, st));
  if (z) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(z, Mx + (size_t)r * rp, row, cudaMemcpyDeviceToHost, st));
  // the fit refresh writes inst_a again: it runs below, after the copies, as the update phase would have run it
  g->skip_fit_refresh = true;
  const int32_t rc = enqueue_update_phase(g, probabilistic, seed, /*fresh_factor=*/kept_factor == 0);
  g->skip_fit_refresh = false;
  GINGR_TRY(rc);
  if (z2) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(z2, Mx + (size_t)r * rp, row, cudaMemcpyDeviceToHost, st));
  if (vec) GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(vec, row, g->vec.p, pitch, row, 6, cudaMemcpyDeviceToHost, st));
  const size_t pts = sizeof(double) * 3 * M;
  if (inst_a) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(inst_a, g->inst_a.p, pts, cudaMemcpyDeviceToHost, st));
  if (inst_b) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(inst_b, g->inst_b.p, pts, cudaMemcpyDeviceToHost, st));
  if (newshape) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(newshape, g->newshape.p, pts, cudaMemcpyDeviceToHost, st));
  if (u) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(u, g->u.p, pts, cudaMemcpyDeviceToHost, st));
  if (pro_sums) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(pro_sums, g->pro_sums.p, sizeof(double) * 10, cudaMemcpyDeviceToHost, st));
  if (ds) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(ds, g->ds.p, sizeof(double) * DS_COUNT, cudaMemcpyDeviceToHost, st));
  if (is) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(is, g->is.p, sizeof(int) * IS_COUNT, cudaMemcpyDeviceToHost, st));
  if (alpha_out) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(alpha_out, g->alpha.p, row, cudaMemcpyDeviceToHost, st));
  GINGR_TRY(evaluate_fit(g, DS_SCALE, DS_T, DS_R2));
  if (fit) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(fit, g->fit.p, pts, cudaMemcpyDeviceToHost, st));
  if (S) GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(S, row, m->S.p, pitch, row, r, cudaMemcpyDeviceToHost, st));
  if (W0) GINGR_CUDA_TRY(ctx, cudaMemcpy2DAsync(W0, row, m->W0.p, pitch, row, r, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  drop_graph(g);
  mcmc_invalidate(g);
  return GINGR_OK;
}

int32_t gingr_posterior_model_profile(const gingr_ctx* ctx, double* ms, int32_t* sweeps) {
  if (!ctx || !ms) return gingr_fail(nullptr, GINGR_ERR_ARG, "gingr_posterior_model_profile: bad argument");
  for (int k = 0; k < 5; ++k) ms[k] = ctx->posterior_model_ms[k];
  if (sweeps) *sweeps = ctx->posterior_model_sweeps;
  return GINGR_OK;
}

}  // extern "C"
