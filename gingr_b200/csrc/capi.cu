// capi.cu -- extern "C" boundary of libgingr_cuda.so: context, uploads and the kernel-level entry
// points (K1 E-step, K2 closest point, K3 posterior).  The full iteration lives in update.cu.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <mutex>

#include "closest.cuh"
#include "common.cuh"
#include "estep.cuh"
#include "grid.cuh"
#include "nccl_dl.cuh"
#include "posterior.cuh"

static std::mutex g_err_mutex;
static std::string g_last_error;

void gingr_set_error(gingr_ctx* ctx, const char* msg) {
  if (ctx) ctx->last_error = msg;
  std::lock_guard<std::mutex> lock(g_err_mutex);
  g_last_error = msg;
}

int32_t gingr_fail(gingr_ctx* ctx, int32_t code, const char* msg) {
  gingr_set_error(ctx, msg);
  return code;
}

// per-ctx scratch for the kernel-level calls (the registration handle owns its own)
struct CtxScratch {
  gingr::EstepWorkspace estep;
  DevBuf<double> a, b, c, d;
  DevBuf<int32_t> ia;
  DevBuf<uint8_t> ua;
};

static CtxScratch* scratch_of(gingr_ctx* ctx);

struct gingr_ctx_full : gingr_ctx {
  CtxScratch scratch;
};

static CtxScratch* scratch_of(gingr_ctx* ctx) { return &static_cast<gingr_ctx_full*>(ctx)->scratch; }

extern "C" {

int32_t gingr_version(void) { return 100; }

int32_t gingr_ctx_create(int32_t device, gingr_ctx** out) {
  if (!out) return gingr_fail(nullptr, GINGR_ERR_ARG, "gingr_ctx_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    return gingr_fail(nullptr, GINGR_ERR_CUDA,
                      "gingr_ctx_create: no CUDA device (libgingr_cuda has no CPU fallback)");
  }
  if (device < 0 || device >= count) return gingr_fail(nullptr, GINGR_ERR_ARG, "gingr_ctx_create: bad device index");
  std::unique_ptr<gingr_ctx, decltype(&gingr_ctx_destroy)> ctx(new gingr_ctx_full(), gingr_ctx_destroy);
  ctx->device = device;
  GINGR_CUDA_TRY(nullptr, cudaSetDevice(device));
  cudaDeviceProp prop;
  GINGR_CUDA_TRY(nullptr, cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return gingr_fail(nullptr, GINGR_ERR_CUDA, "gingr_ctx_create: device is not sm_100 (Blackwell) -- unsupported");
  ctx->num_sms = prop.multiProcessorCount;
  int prio_lo = 0, prio_hi = 0;
  GINGR_CUDA_TRY(nullptr, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  GINGR_CUDA_TRY(nullptr, cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi));
  GINGR_CUDA_TRY(nullptr, cudaStreamCreateWithPriority(&ctx->side_stream, cudaStreamNonBlocking, prio_lo));
  GINGR_CUDA_TRY(nullptr, cudaMallocHost((void**)&ctx->h_pinned, ctx->h_pinned_count * sizeof(double)));
  *out = ctx.release();
  return GINGR_OK;
}

int32_t gingr_ctx_destroy(gingr_ctx* ctx) {
  if (!ctx) return GINGR_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  gingr::comm_destroy(ctx);
  if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
  for (auto& e : ctx->chol_events) cudaEventDestroy(e);
  if (ctx->side_stream) cudaStreamDestroy(ctx->side_stream);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete static_cast<gingr_ctx_full*>(ctx);   // frees the scratch buffers
  return GINGR_OK;
}

const char* gingr_last_error(const gingr_ctx* ctx) {
  if (ctx) return ctx->last_error.c_str();
  std::lock_guard<std::mutex> lock(g_err_mutex);
  return g_last_error.c_str();
}

void* gingr_ctx_stream(gingr_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int32_t gingr_ctx_synchronize(gingr_ctx* ctx) {
  if (!ctx) return GINGR_ERR_ARG;
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GINGR_OK;
}

int64_t gingr_ctx_launch_count(const gingr_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ---------------------------------------------------------------------------------------------
// uploads
// ---------------------------------------------------------------------------------------------
int32_t gingr_target_upload(gingr_ctx* ctx, int32_t N, const double* pts, const int32_t* tri, int32_t T,
                            gingr_target** out) {
  if (!ctx || !out || !pts || N <= 0 || T < 0 || (T > 0 && !tri))
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_target_upload: bad argument");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (T > 0)
    for (int k = 0; k < 3 * T; ++k)
      if (tri[k] < 0 || tri[k] >= N) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_target_upload: triangle index out of range");
  std::unique_ptr<gingr_target> t(new gingr_target());
  t->ctx = ctx;
  t->N_total = N;
  for (size_t k = 0; k < (size_t)3 * N; ++k) {
    if (!(fabs(pts[k]) < INFINITY)) { t->nonfinite = true; break; }
    t->maxabs = std::max(t->maxabs, fabs(pts[k]));
  }
  shard_range(N, ctx->nranks, ctx->rank, &t->n0, &t->N);
  // full vertex set (SoA) -- the ICP search and the single-GPU E-step use it; the E-step shard is a view
  // into a separately packed SoA when sharded.
  CtxScratch* s = scratch_of(ctx);
  GINGR_CUDA_TRY(ctx, s->a.alloc((size_t)3 * N));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(s->a.p, pts, sizeof(double) * 3 * (size_t)N, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_CUDA_TRY(ctx, t->verts.alloc((size_t)3 * N));
  GINGR_TRY(gingr::aos_to_soa_enqueue(ctx, N, s->a.p, t->verts.p));
  GINGR_CUDA_TRY(ctx, t->aos.alloc((size_t)3 * N));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(t->aos.p, s->a.p, sizeof(double) * 3 * (size_t)N, cudaMemcpyDeviceToDevice, ctx->stream));
  if (t->N > 0) {
    GINGR_CUDA_TRY(ctx, t->soa.alloc((size_t)3 * t->N));
    GINGR_TRY(gingr::aos_to_soa_enqueue(ctx, t->N, s->a.p + (size_t)3 * t->n0, t->soa.p));
  }
  t->T = T;
  if (T > 0) {
    GINGR_CUDA_TRY(ctx, t->tri.alloc((size_t)3 * T));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(t->tri.p, tri, sizeof(int32_t) * 3 * (size_t)T, cudaMemcpyHostToDevice, ctx->stream));
    GINGR_TRY(gingr::mesh_static_upload(ctx, N, pts, T, tri, &t->normals, &t->boundary));
  }
  if (gingr::grid_wanted(N) && !t->nonfinite) {
    gingr::VertexArray va;
    va.p = t->aos.p;
    t->pgrid = std::make_unique<gingr::SpatialGrid>();
    GINGR_TRY(t->pgrid->ensure(ctx, N, N, false));
    GINGR_TRY(gingr::grid_build_points_enqueue(ctx, *t->pgrid, N, va));
    if (T > 0) {
      t->tgrid = std::make_unique<gingr::SpatialGrid>();
      t->tgrid->entry_boxes = true;   // static grid, searched every iteration: boxes stored with the entries
      GINGR_TRY(t->tgrid->ensure(ctx, N, T, true));
      GINGR_TRY(gingr::grid_build_triangles_enqueue(ctx, *t->tgrid, N, va, T, t->tri.p));
    }
  }
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  *out = t.release();
  return GINGR_OK;
}

int32_t gingr_target_destroy(gingr_target* t) {
  if (!t) return GINGR_OK;
  cudaSetDevice(t->ctx->device);
  delete t;
  return GINGR_OK;
}

// ---------------------------------------------------------------------------------------------
// K1 entry points
// ---------------------------------------------------------------------------------------------
static bool host_nonfinite(const double* v, size_t n) {
  for (size_t k = 0; k < n; ++k)
    if (!(fabs(v[k]) < INFINITY)) return true;
  return false;
}

// upper bound of every squared pair distance from the coordinate ranges: |x - y|^2 <= 3 (max|x| + max|y|)^2
static double d2_bound(const gingr_target* target, const double* fit, size_t n3) {
  double m = 0.0;
  for (size_t k = 0; k < n3; ++k) m = std::max(m, fabs(fit[k]));
  const double s = m + target->maxabs;
  return 3.0 * s * s;
}

static void fill_nan(double* p, size_t n) {
  if (p)
    for (size_t k = 0; k < n; ++k) p[k] = NAN;
}

static int32_t estep_common(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* fit,
                            gingr::EstepWorkspace** ws_out) {
  CtxScratch* s = scratch_of(ctx);
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GINGR_TRY(s->estep.ensure(ctx, M, target->N));
  GINGR_CUDA_TRY(ctx, s->a.alloc((size_t)3 * std::max(M, 1)));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(s->a.p, fit, sizeof(double) * 3 * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_TRY(gingr::aos_to_soa_enqueue(ctx, M, s->a.p, s->estep.fit_soa.p));
  *ws_out = &s->estep;
  return GINGR_OK;
}

// rows [4][M] -> host P1[M], PX[M][3]; combines shards when nranks > 1
static int32_t estep_download(gingr_ctx* ctx, gingr::EstepWorkspace* ws, int M, int N, double* P1, double* Pt1,
                              double* PX, std::vector<double>* rows_host) {
  if (ctx->nranks > 1) GINGR_TRY(gingr::comm_allreduce_sum(ctx, ws->rows.p, (size_t)4 * M));
  rows_host->resize((size_t)4 * M);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(rows_host->data(), ws->rows.p, sizeof(double) * 4 * (size_t)M,
                                      cudaMemcpyDeviceToHost, ctx->stream));
  if (Pt1)
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(Pt1, ws->pt1.p, sizeof(double) * (size_t)N, cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const double* r = rows_host->data();
  if (P1) memcpy(P1, r, sizeof(double) * (size_t)M);
  if (PX)
    for (int i = 0; i < M; ++i) {
      PX[3 * i] = r[(size_t)M + i];
      PX[3 * i + 1] = r[(size_t)2 * M + i];
      PX[3 * i + 2] = r[(size_t)3 * M + i];
    }
  return GINGR_OK;
}

int32_t gingr_cpd_estep(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* fit, double sigma2,
                        double w, double* P1, double* Pt1, double* PX) {
  if (!ctx || !target || !fit || M <= 0) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_cpd_estep: bad argument");
  if (target->nonfinite || host_nonfinite(fit, (size_t)3 * M) || !(fabs(sigma2) < INFINITY)) {
    // a NaN coordinate makes every entry of the reference's P NaN (CPD.scala:54-75)
    fill_nan(P1, M); fill_nan(Pt1, target->N); fill_nan(PX, (size_t)3 * M);
    return GINGR_OK;
  }
  gingr::EstepWorkspace* ws = nullptr;
  GINGR_TRY(estep_common(ctx, target, M, fit, &ws));
  double* h = ctx->h_pinned;
  memset(h, 0, sizeof(double) * 16);
  h[0] = sigma2;
  h[3] = w;
  h[4] = (double)M / (double)target->N_total;
  h[7] = d2_bound(target, fit, (size_t)3 * M);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(ws->scal.p, h, sizeof(double) * 16, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_TRY(gingr::estep_cpd_scalars_enqueue(ctx, ws->scal.p));
  if (target->N > 0) GINGR_TRY(gingr::estep_enqueue(ctx, *ws, M, target->N, target->soa.p, false));
  std::vector<double> rows;
  return estep_download(ctx, ws, M, target->N, P1, Pt1, PX, &rows);
}

int32_t gingr_bcpd_estep(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* y,
                         const double* sigma_mm, const double* alpha, double sigma2, double s, double w, double* nu,
                         double* nu_prime, double* n_hat, double* x_hat) {
  if (!ctx || !target || !y || !sigma_mm || !alpha || M <= 0)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_bcpd_estep: bad argument");
  if (target->nonfinite || host_nonfinite(y, (size_t)3 * M) || host_nonfinite(sigma_mm, M) || host_nonfinite(alpha, M) ||
      !(fabs(sigma2) < INFINITY)) {
    fill_nan(nu, M); fill_nan(nu_prime, target->N); fill_nan(n_hat, 1); fill_nan(x_hat, (size_t)3 * M);
    return GINGR_OK;
  }
  gingr::EstepWorkspace* ws = nullptr;
  GINGR_TRY(estep_common(ctx, target, M, y, &ws));
  CtxScratch* sc = scratch_of(ctx);
  GINGR_CUDA_TRY(ctx, sc->b.alloc((size_t)2 * M));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(sc->b.p, sigma_mm, sizeof(double) * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(sc->b.p + M, alpha, sizeof(double) * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
  double* h = ctx->h_pinned;
  memset(h, 0, sizeof(double) * 16);
  h[0] = sigma2;
  h[3] = w;
  h[5] = s;
  h[6] = 1.0 / (double)target->N_total;
  h[7] = d2_bound(target, y, (size_t)3 * M);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(ws->scal.p, h, sizeof(double) * 16, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_TRY(gingr::estep_bcpd_rowf_enqueue(ctx, M, sc->b.p, sc->b.p + M, ws->scal.p, ws->rowf.p));
  if (target->N > 0) GINGR_TRY(gingr::estep_enqueue(ctx, *ws, M, target->N, target->soa.p, true));
  std::vector<double> rows;
  std::vector<double> nup((size_t)target->N);
  std::vector<double> nuv((size_t)M), px((size_t)3 * M);
  GINGR_TRY(estep_download(ctx, ws, M, target->N, nuv.data(), nup.data(), px.data(), &rows));
  if (nu) memcpy(nu, nuv.data(), sizeof(double) * (size_t)M);
  if (nu_prime) memcpy(nu_prime, nup.data(), sizeof(double) * (size_t)target->N);
  if (n_hat) {
    // Nhat = sum(nu')  BCPD.scala:204 ; across ranks the caller sums the shard values
    double sum = 0.0;
    for (int j = 0; j < target->N; ++j) sum += nup[j];
    *n_hat = sum;
  }
  if (x_hat)  // xhat = pinv(diag(nu (x) 1_3)) (P (x) I_3) X  BCPD.scala:209 : rows with nu == 0 map to 0
    for (int i = 0; i < M; ++i) {
      const double inv = nuv[i] != 0.0 ? 1.0 / nuv[i] : 0.0;
      for (int d = 0; d < 3; ++d) x_hat[3 * i + d] = px[3 * i + d] * inv;
    }
  return GINGR_OK;
}

int32_t gingr_cpd_initial_sigma2(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* pts,
                                 double* sigma2_out) {
  if (!ctx || !target || !pts || !sigma2_out || M <= 0)
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_cpd_initial_sigma2: bad argument");
  CtxScratch* s = scratch_of(ctx);
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  GINGR_CUDA_TRY(ctx, s->a.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, s->b.alloc(16));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(s->a.p, pts, sizeof(double) * 3 * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
  GINGR_TRY(gingr::initial_sigma2_enqueue(ctx, M, s->a.p, target->N_total, target->verts.p, s->b.p));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(sigma2_out, s->b.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return GINGR_OK;
}

// ---------------------------------------------------------------------------------------------
// K2 entry point
// ---------------------------------------------------------------------------------------------
// shared by the two K2 entry points: uploads the template, computes its normals / boundary flags
struct TemplateUpload {
  DevBuf<double> aos, soa, normals;
  DevBuf<int32_t> tri, off, adj;
  DevBuf<uint8_t> boundary;
  gingr::SpatialGrid pgrid, tgrid;
};

static int32_t upload_template(gingr_ctx* ctx, int M, const double* tpl, const int32_t* tpl_tri, int T, TemplateUpload* u,
                               gingr::MeshView* view, bool want_pgrid) {
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, u->aos.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, u->soa.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(u->aos.p, tpl, sizeof(double) * 3 * (size_t)M, cudaMemcpyHostToDevice, st));
  GINGR_TRY(gingr::aos_to_soa_enqueue(ctx, M, u->aos.p, u->soa.p));
  view->n = M;
  view->aos = u->aos.p;
  view->soa = u->soa.p;
  view->T = T;
  if (T > 0) {
    for (int k = 0; k < 3 * T; ++k)
      if (tpl_tri[k] < 0 || tpl_tri[k] >= M) return gingr_fail(ctx, GINGR_ERR_ARG, "template triangle index out of range");
    std::vector<int32_t> off, adj;
    std::vector<uint8_t> flags;
    gingr::build_vertex_adjacency(M, T, tpl_tri, &off, &adj);
    gingr::compute_boundary_flags(M, T, tpl_tri, &flags);
    GINGR_CUDA_TRY(ctx, u->tri.alloc((size_t)3 * T));
    GINGR_CUDA_TRY(ctx, u->off.alloc(off.size()));
    GINGR_CUDA_TRY(ctx, u->adj.alloc(adj.size()));
    GINGR_CUDA_TRY(ctx, u->normals.alloc((size_t)3 * M));
    GINGR_CUDA_TRY(ctx, u->boundary.alloc((size_t)M));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(u->tri.p, tpl_tri, sizeof(int32_t) * 3 * (size_t)T, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(u->off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(u->adj.p, adj.data(), adj.size() * 4, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(u->boundary.p, flags.data(), (size_t)M, cudaMemcpyHostToDevice, st));
    GINGR_TRY(gingr::vertex_normals_enqueue(ctx, M, u->aos.p, u->tri.p, u->off.p, u->adj.p, u->normals.p));
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));  // off / adj / flags are stack vectors
    view->tri = u->tri.p;
    view->normals = u->normals.p;
    view->boundary = u->boundary.p;
  }
  if (gingr::grid_wanted(M)) {
    gingr::VertexArray va;
    va.p = u->aos.p;
    if (want_pgrid) {
      GINGR_TRY(u->pgrid.ensure(ctx, M, M, false));
      GINGR_TRY(gingr::grid_build_points_enqueue(ctx, u->pgrid, M, va));
      view->pgrid = &u->pgrid;
    }
    if (T > 0) {
      GINGR_TRY(u->tgrid.ensure(ctx, M, T, true));
      GINGR_TRY(gingr::grid_build_triangles_enqueue(ctx, u->tgrid, M, va, T, u->tri.p));
      view->tgrid = &u->tgrid;
    }
  }
  return GINGR_OK;
}

static gingr::MeshView target_view(const gingr_target* t) {
  gingr::MeshView v;
  v.n = t->N_total;
  v.aos = t->aos.p;
  v.soa = t->verts.p;
  v.T = t->T;
  v.tri = t->tri.p;
  v.normals = t->normals.p;
  v.boundary = t->boundary.p;
  v.pgrid = t->pgrid.get();
  v.tgrid = t->tgrid.get();
  return v;
}

int32_t gingr_icp_closest(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* tpl,
                          const int32_t* tpl_tri, int32_t T, int32_t method, int32_t* idx, double* cp, uint8_t* w,
                          double* mean_distance) {
  if (!ctx || !target || !tpl || M <= 0 || T < 0 || (T > 0 && !tpl_tri))
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_icp_closest: bad argument");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  gingr::ClosestWorkspace ws;
  TemplateUpload up;
  gingr::MeshView tv;
  GINGR_TRY(ws.ensure(ctx, M, target->N_total, target->T, T));
  GINGR_TRY(upload_template(ctx, M, tpl, tpl_tri, T, &up, &tv, false));
  GINGR_TRY(gingr::icp_correspondence_enqueue(ctx, ws, tv, target_view(target), method));
  cudaStream_t st = ctx->stream;
  if (idx) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(idx, ws.idx.p, sizeof(int32_t) * (size_t)M, cudaMemcpyDeviceToHost, st));
  if (cp) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(cp, ws.cp.p, sizeof(double) * 3 * (size_t)M, cudaMemcpyDeviceToHost, st));
  if (w) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(w, ws.w.p, (size_t)M, cudaMemcpyDeviceToHost, st));
  if (mean_distance) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mean_distance, ws.mean_dist.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return GINGR_OK;
}

int32_t gingr_icp_closest_reversal(gingr_ctx* ctx, const gingr_target* target, int32_t M, const double* tpl,
                                   const int32_t* tpl_tri, int32_t T, int32_t method, int32_t* tpl_id, uint8_t* w,
                                   double* mean_distance) {
  if (!ctx || !target || !tpl || M <= 0 || T < 0 || (T > 0 && !tpl_tri))
    return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_icp_closest_reversal: bad argument");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int N = target->N_total;
  gingr::ClosestWorkspace ws;
  TemplateUpload up;
  gingr::MeshView tv;
  DevBuf<int32_t> tid;
  GINGR_TRY(ws.ensure(ctx, N, M, T, target->T));
  GINGR_TRY(upload_template(ctx, M, tpl, tpl_tri, T, &up, &tv, true));
  // corr = closestPointCorrespondence(target, template): the roles are swapped (:38)
  GINGR_TRY(gingr::icp_correspondence_enqueue(ctx, ws, target_view(target), tv, method));
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, tid.alloc((size_t)N));
  // templateId = template.pointSet.findClosestPoint(p).id for the corresponding point p (:40)
  GINGR_TRY(gingr::nn_vertex_enqueue(ctx, ws, N, ws.cp.p, M, up.soa.p, ws.d2.p, tid.p, tv.pgrid, ws.qorder.get()));
  if (tpl_id) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(tpl_id, tid.p, sizeof(int32_t) * (size_t)N, cudaMemcpyDeviceToHost, st));
  if (w) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(w, ws.w.p, (size_t)N, cudaMemcpyDeviceToHost, st));
  if (mean_distance) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mean_distance, ws.mean_dist.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return GINGR_OK;
}

}  // extern "C"
