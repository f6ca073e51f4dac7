// common.cuh -- context, handles and small helpers shared by the gingr_cuda translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <memory>
#include <string>
#include <vector>

#include "../../include/gingr_cuda.h"

#define GINGR_NUM_SMS_B200 148

struct NcclApi;  // nccl_dl.cu
struct LaunchRecorder;  // batch.cuh
namespace gingr { struct SpatialGrid; }  // grid.cuh

struct gingr_ctx {
  int device = 0;
  int num_sms = GINGR_NUM_SMS_B200;
  cudaStream_t stream = nullptr;       // all work of the ctx; highest priority
  cudaStream_t side_stream = nullptr;  // low priority: bulk trailing updates of the Cholesky lookahead (chol.cu)
  std::vector<cudaEvent_t> chol_events;  // 2 per block step, created on first use
  std::string last_error;
  int64_t launches = 0;
  LaunchRecorder* rec = nullptr;       // while set, batch-aware launches are recorded instead of issued (batch.cuh)
  // multi-GPU
  int nranks = 1, rank = 0;
  void* nccl_comm = nullptr;
  // small pinned staging buffer for scalars
  double* h_pinned = nullptr;  // 4096 doubles
  size_t h_pinned_count = 4096;
};

// Device buffer that owns its memory: freed when the owner goes away, moved but never copied.
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) {
      if (p) cudaFree(p);
      p = o.p; n = o.n;
      o.p = nullptr; o.n = 0;
    }
    return *this;
  }
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  // grows only: keeps the block when it holds count elements, else frees it before allocating the larger one
  cudaError_t alloc(size_t count) {
    if (p && n >= count) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    cudaError_t e = cudaMalloc((void**)&p, (count ? count : 1) * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
};

// Owner of an instantiated CUDA graph; reset() destroys it.
struct GraphExec {
  cudaGraphExec_t h = nullptr;
  GraphExec() = default;
  GraphExec(const GraphExec&) = delete;
  GraphExec& operator=(const GraphExec&) = delete;
  GraphExec(GraphExec&& o) noexcept : h(o.h) { o.h = nullptr; }
  GraphExec& operator=(GraphExec&& o) noexcept {
    if (this != &o) {
      reset();
      h = o.h;
      o.h = nullptr;
    }
    return *this;
  }
  ~GraphExec() { reset(); }
  void reset() {
    if (h) cudaGraphExecDestroy(h);
    h = nullptr;
  }
};

struct gingr_target {
  gingr_ctx* ctx = nullptr;
  int N_total = 0;      // number of target points in the whole target
  int n0 = 0, N = 0;    // this rank's shard [n0, n0 + N) for the E-step (== whole target when nranks == 1)
  double maxabs = 0.0;  // max |coordinate| (bounds the pair distances: gauss_exp2_tab<SAFE>)
  bool nonfinite = false;  // a NaN/Inf coordinate: every E-step on it fails like the reference's NaN-filled P
  DevBuf<double> soa;   // E-step shard, SoA [3][N] (x[], y[], z[]) in the k-d order of gingr::estep_target_order
  DevBuf<int32_t> soa_perm;  // [N] shard index (from n0) of soa position j
  // full mesh (ICP): vertices SoA [3][N_total], triangles, per-vertex normals and boundary flags
  DevBuf<double> verts; // [3][N_total]
  DevBuf<double> aos;   // [N_total][3] the same vertices, AoS (queries of the reversed ICP direction, line tests)
  int T = 0;
  DevBuf<int32_t> tri;      // [3T]
  DevBuf<double> normals;   // [3][N_total]
  DevBuf<uint8_t> boundary; // [N_total]
  // static uniform grids over the vertices / triangles (K2 at scale; null below the size where a scan wins)
  std::unique_ptr<gingr::SpatialGrid> pgrid, tgrid;
};

struct gingr_model {
  gingr_ctx* ctx = nullptr;
  int M = 0, r = 0, rp = 0;   // rp = r padded to a multiple of 8 (row pitch of phi)
  int m0 = 0, Ml = 0;         // this rank's point shard [m0, m0 + Ml)
  DevBuf<double> ref;         // [3M] AoS reference points (all points, replicated)
  DevBuf<double> mean;        // [3M] meanVector (all points)
  DevBuf<double> phi;         // [3*Ml][rp] ROW-major basis rows of this rank's shard
  DevBuf<double> sqrt_lambda; // [rp] sqrt(variance), zero padded
  int T = 0;
  DevBuf<int32_t> tri;        // [3T] reference triangles (ICP)
  DevBuf<int32_t> adj_off;    // [M+1] CSR vertex -> incident triangles (ascending triangle id)
  DevBuf<int32_t> adj;        // [3T]
  DevBuf<uint8_t> boundary;   // [M] pointIsOnBoundary of the reference topology (reversed ICP direction)
  // constants of the `coefficients` regression (noise 1e-5 on all M points):
  DevBuf<double> S;           // [rp][rp] S = D Phi^T Phi D, D = diag(sqrt(lambda))
  DevBuf<double> W0;          // [rp][rp] (1e-5 I + S)^-1
  bool has_regression_constants = false;
};

#define GINGR_CUDA_TRY(ctx, expr)                                                                   \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess) {                                                                        \
      char _b[512];                                                                                 \
      snprintf(_b, sizeof(_b), "%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      gingr_set_error((ctx), _b);                                                                   \
      return GINGR_ERR_CUDA;                                                                        \
    }                                                                                               \
  } while (0)

#define GINGR_TRY(expr)              \
  do {                               \
    int32_t _s = (expr);             \
    if (_s < 0) return _s;           \
  } while (0)

void gingr_set_error(gingr_ctx* ctx, const char* msg);
int32_t gingr_fail(gingr_ctx* ctx, int32_t code, const char* msg);

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Count a kernel launch on the ctx (bench.py reports gpu_launches from this).
#define GINGR_LAUNCHED(ctx) ((ctx)->launches++)

// shard [begin, end) of n items for rank of nranks (contiguous, remainder spread over first ranks)
static inline void shard_range(int n, int nranks, int rank, int* begin, int* count) {
  int base = n / nranks, rem = n % nranks;
  *begin = rank * base + (rank < rem ? rank : rem);
  *count = base + (rank < rem ? 1 : 0);
}
