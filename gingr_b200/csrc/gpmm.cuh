// gpmm.cuh -- GPMM construction on the device (included by update.cu; SURVEY.md 8f item 4).
//
// Replaces GPMMTriangleMesh3D(reference, relativeTolerance).Gaussian / GaussianMixture (api/gpmm/GPMMHelper.scala:99-129)
// -> GPMM.construct (:39-54) -> scalismo LowRankGaussianProcess.approximateGPCholesky (SURVEY.md A7):
//   pivoted Cholesky L (3M x k) of the matrix-valued kernel on the reference points until
//   trace(residual) <= relTol * trace(K);  (V, d) = svd(L^T L);  basis = L V diag(d^-1/2),  variance = d.
// The kernels of these constructors are DiagonalKernel(scalar kernel, 3), i.e. K = Ks (x) I3 with
//   ks(x, y) = sum_q scaling_q exp(-|x - y|^2 / sigma_q^2)          [scalismo GaussianKernel: sigma^2, not 2 sigma^2]
// so the 3M x 3M factorisation is the scalar M x M one taken three times: a pivot (point p, dimension 0) leaves the
// residual diagonal of (p, 1), (p, 2) untouched and maximal, so the columns come in triples of the same point, and after
// c columns of triple k the trace is 3 T(k) - c (T(k) - T(k+1)) with T the scalar traces -- which also reproduces a rank
// that is not a multiple of three (tests/test_oracle_gpmm.py proves this against the literal 3M x 3M algorithm).
// The mirror-symmetric kernel (scalismo's symmetrised kernel about x = 0, gingr_gpmm_gaussian_symmetric) is diagonal
// too, with two distinct blocks: ks - ks_m for dimension 0 and ks + ks_m for dimensions 1 and 2, ks_m(x, y) = ks(S x, y).
// The inverse-Laplacian kernel (gingr_gpmm_inverse_laplacian) is Ks (x) I3 with Ks a dense M x M matrix computed up
// front (Laplacian assembly, data-flow Cholesky with the identity riding along, DMMA Gram); its block reads Ks.
// All cases are one loop (gpmm_build): a scalar factorisation per block, merged on the host in the literal order.
//   pivoted Cholesky   one column per step: argmax of the residual diagonal (lowest index on ties), the kernel column
//                      minus the projection on the previous columns, diagonal update; all scalars stay on the device,
//                      the host looks at the trace history once per batch of steps
//   KL basis           instead of forming L^T L and its eigenvectors: one-sided Jacobi (Hestenes) on the tall factor
//                      itself, L = U Sigma V^T, so U is the orthonormal basis and Sigma^2 the variances -- rotations of
//                      column pairs in round-robin order, one CTA per pair, until no pair is rotated
// The degenerate (triple) eigenvalues make the basis unique only up to a rotation inside each eigenspace; what is
// defined -- and tested -- is the rank, the variances and the covariance basis diag(variance) basis^T = L L^T.
#pragma once

namespace gingr {

struct GaussKernelDev {
  int n;
  double inv_sigma2[8];
  double scaling[8];
};

__device__ __forceinline__ double gpmm_kernel(const GaussKernelDev& kp, double dx, double dy, double dz) {
  const double d2 = dx * dx + dy * dy + dz * dz;
  double s = 0.0;
  for (int q = 0; q < kp.n; ++q) s += kp.scaling[q] * exp(-d2 * kp.inv_sigma2[q]);
  return s;
}

// The scalar M x M block a factorisation works on: GPMM_PLAIN is ks itself; GPMM_MINUS / GPMM_PLUS are ks(x, y) -/+ ks(S x, y)
// with the mirror S = diag(-1, 1, 1) about the plane x = 0 (the blocks of the mirror-symmetric kernel, see
// gingr_gpmm_gaussian_symmetric); GPMM_LOOKUP reads a dense symmetric M x M matrix (pitch M) passed in place of the points
// (the inverse-Laplacian kernel, gingr_gpmm_inverse_laplacian).
enum GpmmBlockKind { GPMM_PLAIN = 0, GPMM_MINUS = 1, GPMM_PLUS = 2, GPMM_LOOKUP = 3 };

template <int KIND>
__device__ __forceinline__ double gpmm_entry(const GaussKernelDev& kp, const double* __restrict__ pts, int M, int i, int p) {
  if constexpr (KIND == GPMM_LOOKUP) {
    return pts[(size_t)p * M + i];   // row p = column p: coalesced over i
  } else if constexpr (KIND == GPMM_PLAIN) {
    return gpmm_kernel(kp, pts[3 * i] - pts[3 * p], pts[3 * i + 1] - pts[3 * p + 1], pts[3 * i + 2] - pts[3 * p + 2]);
  } else {
    const double dy = pts[3 * i + 1] - pts[3 * p + 1], dz = pts[3 * i + 2] - pts[3 * p + 2];
    const double k = gpmm_kernel(kp, pts[3 * i] - pts[3 * p], dy, dz);
    const double km = gpmm_kernel(kp, -pts[3 * i] - pts[3 * p], dy, dz);   // S x_i - x_p
    return KIND == GPMM_MINUS ? k - km : k + km;
  }
}

template <int KIND>
__global__ void gpmm_init_diag_kernel(int M, GaussKernelDev kp, const double* __restrict__ pts, double* __restrict__ d,
                                      uint8_t* __restrict__ done) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  if constexpr (KIND == GPMM_PLAIN) d[i] = gpmm_kernel(kp, 0.0, 0.0, 0.0);
  else d[i] = gpmm_entry<KIND>(kp, pts, M, i, i);
  done[i] = 0;
}

// per-block (max residual, lowest index) over the points not yet chosen, and the block's share of the residual trace
__global__ void __launch_bounds__(256) gpmm_argmax_partial_kernel(int M, const double* __restrict__ d, const uint8_t* __restrict__ done,
                                                                  double* __restrict__ pmax, int* __restrict__ pidx,
                                                                  double* __restrict__ psum) {
  __shared__ double smax[256], ssum[256];
  __shared__ int sidx[256];
  double best = -1.0, sum = 0.0;
  int bi = 0x7fffffff;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < M; i += gridDim.x * 256) {
    if (done[i]) continue;
    const double v = d[i];
    sum += v;
    if (v > best || (v == best && i < bi)) { best = v; bi = i; }
  }
  smax[threadIdx.x] = best; sidx[threadIdx.x] = bi; ssum[threadIdx.x] = sum;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const double v = smax[threadIdx.x + o];
      const int j = sidx[threadIdx.x + o];
      if (v > smax[threadIdx.x] || (v == smax[threadIdx.x] && j < sidx[threadIdx.x])) { smax[threadIdx.x] = v; sidx[threadIdx.x] = j; }
      ssum[threadIdx.x] += ssum[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { pmax[blockIdx.x] = smax[0]; pidx[blockIdx.x] = sidx[0]; psum[blockIdx.x] = ssum[0]; }
}

// pivot of step k, its residual, and T(k) = residual trace before the step (fixed block order: deterministic)
__global__ void gpmm_argmax_final_kernel(int nb, int k, const double* __restrict__ pmax, const int* __restrict__ pidx,
                                         const double* __restrict__ psum, int* __restrict__ pivots, double* __restrict__ dpiv,
                                         double* __restrict__ trace) {
  if (threadIdx.x != 0) return;
  double best = -1.0, sum = 0.0;
  int bi = 0x7fffffff;
  for (int b = 0; b < nb; ++b) {
    sum += psum[b];
    if (pmax[b] > best || (pmax[b] == best && pidx[b] < bi)) { best = pmax[b]; bi = pidx[b]; }
  }
  pivots[k] = bi;
  dpiv[k] = best;
  trace[k] = sum;
}

// column k of the scalar factor (column-major Ls[k][M]): (block(x_i, x_p) - sum_{j<k} Ls[j][i] Ls[j][p]) / sqrt(d_p) for the
// points not yet chosen, sqrt(d_p) at the pivot, 0 at earlier pivots; residual diagonal updated
template <int KIND>
__global__ void __launch_bounds__(256) gpmm_column_kernel(int M, int k, GaussKernelDev kp, const double* __restrict__ pts /*AoS*/,
                                                          const int* __restrict__ pivots, const double* __restrict__ dpiv,
                                                          double* __restrict__ Ls, double* __restrict__ d,
                                                          uint8_t* __restrict__ done) {
  extern __shared__ double lp[];   // Ls[j][p], j < k
  const int p = pivots[k];
  const double dp = dpiv[k];
  for (int j = threadIdx.x; j < k; j += 256) lp[j] = Ls[(size_t)j * M + p];
  __syncthreads();
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= M) return;
  double out = 0.0;
  if (dp > 0.0) {
    const double piv = sqrt(dp);
    if (i == p) {
      out = piv;
    } else if (!done[i]) {
      double v = gpmm_entry<KIND>(kp, pts, M, i, p);
      for (int j = 0; j < k; ++j) v -= Ls[(size_t)j * M + i] * lp[j];
      out = v / piv;
      d[i] -= out * out;
    }
  }
  Ls[(size_t)k * M + i] = out;
  if (i == p) done[i] = 1;
}

// ---- one-sided Jacobi on the columns of A (column-major [n][M]) --------------------------------------------------
// round-robin pairing (circle method) of n_even players, player n_even - 1 fixed
__device__ __forceinline__ void jacobi_pair(int n_even, int round, int m, int& a, int& b) {
  const int nm1 = n_even - 1;
  if (m == 0) { a = nm1; b = round % nm1; }
  else { a = (round + m) % nm1; b = (round - m + nm1) % nm1; }
  if (a > b) { const int t = a; a = b; b = t; }
}

__global__ void __launch_bounds__(256) gpmm_jacobi_round_kernel(int M, int n, int n_even, int round, double tol,
                                                                double* __restrict__ A, int* __restrict__ rotated) {
  __shared__ double red[3][256];
  __shared__ double cs[2];
  int a, b;
  jacobi_pair(n_even, round, blockIdx.x, a, b);
  if (b >= n) return;   // the dummy player of an odd n
  double* ca = A + (size_t)a * M;
  double* cb = A + (size_t)b * M;
  double saa = 0.0, sbb = 0.0, sab = 0.0;
  for (int i = threadIdx.x; i < M; i += 256) {
    const double x = ca[i], y = cb[i];
    saa = fma(x, x, saa); sbb = fma(y, y, sbb); sab = fma(x, y, sab);
  }
  red[0][threadIdx.x] = saa; red[1][threadIdx.x] = sbb; red[2][threadIdx.x] = sab;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o)
      for (int q = 0; q < 3; ++q) red[q][threadIdx.x] += red[q][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double alpha = red[0][0], beta = red[1][0], gamma = red[2][0];
    double c = 1.0, s = 0.0;
    if (fabs(gamma) > tol * sqrt(alpha * beta) && gamma != 0.0) {
      const double zeta = (beta - alpha) / (2.0 * gamma);
      const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
      c = 1.0 / sqrt(1.0 + t * t);
      s = c * t;
      atomicExch(rotated, 1);
    }
    cs[0] = c; cs[1] = s;
  }
  __syncthreads();
  const double c = cs[0], s = cs[1];
  if (s == 0.0) return;
  for (int i = threadIdx.x; i < M; i += 256) {
    const double x = ca[i], y = cb[i];
    ca[i] = c * x - s * y;
    cb[i] = s * x + c * y;
  }
}

__global__ void __launch_bounds__(256) gpmm_colnorm_kernel(int M, const double* __restrict__ A, double* __restrict__ norm2) {
  __shared__ double red[256];
  const double* c = A + (size_t)blockIdx.x * M;
  double s = 0.0;
  for (int i = threadIdx.x; i < M; i += 256) s = fma(c[i], c[i], s);
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) norm2[blockIdx.x] = red[0];
}

// model column c = (source set, scalar column j, dimension d):  phi[3 i + d][c] = A_set[j][i] / sqrt(norm2_set[j])
struct GpmmColumn { int set, j, d; };
__global__ void gpmm_assemble_kernel(int M, int r, int rp, const GpmmColumn* __restrict__ cols, const double* __restrict__ A0,
                                     const double* __restrict__ n0, const double* __restrict__ A1, const double* __restrict__ n1,
                                     const double* __restrict__ A2, const double* __restrict__ n2, double* __restrict__ phi) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (i >= M || c >= r) return;
  const GpmmColumn col = cols[c];
  const double* A = col.set == 0 ? A0 : col.set == 1 ? A1 : A2;
  const double* nn = col.set == 0 ? n0 : col.set == 1 ? n1 : n2;
  phi[((size_t)3 * i + col.d) * rp + c] = A[(size_t)col.j * M + i] / sqrt(nn[col.j]);
}

// ---- the inverse-Laplacian kernel: the system [L + gamma I (or L + P); I] for the data-flow Cholesky --------------------
// each edge of each triangle marks A[a][b] = A[b][a] = -1: one value stored, so duplicated edges and the triangle order do
// not change the result; self-edges of degenerate triangles are skipped
__global__ void lap_edges_kernel(int T, const int32_t* __restrict__ tri, int ld, double* __restrict__ A) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const int v[3] = {tri[3 * t], tri[3 * t + 1], tri[3 * t + 2]};
  for (int e = 0; e < 3; ++e) {
    const int a = v[e], b = v[(e + 1) % 3];
    if (a == b) continue;
    A[(size_t)a * ld + b] = -1.0;
    A[(size_t)b * ld + a] = -1.0;
  }
}

// row i: the degree (the marks of the row) + gamma on the diagonal; with project, P = sum_c 1_c 1_c^T / |c| added
// (comp: component of each vertex, inv_size: 1 / |c|); the identity row M + i rides along below the square part
__global__ void __launch_bounds__(256) lap_rows_kernel(int M, int ld, double gamma, int project, const int* __restrict__ comp,
                                                       const double* __restrict__ inv_size, double* __restrict__ A) {
  __shared__ int red[256];
  const int i = blockIdx.x;
  double* row = A + (size_t)i * ld;
  int deg = 0;
  for (int j = threadIdx.x; j < M; j += 256) deg += row[j] != 0.0;
  red[threadIdx.x] = deg;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  deg = red[0];
  const int ci = project ? comp[i] : 0;
  for (int j = threadIdx.x; j < M; j += 256) {
    double v = j == i ? deg + gamma : row[j];
    if (project && comp[j] == ci) v += inv_size[ci];
    row[j] = v;
  }
  if (threadIdx.x == 0) A[(size_t)(M + i) * ld + i] = 1.0;
}

// Ks = s (G - P) from G = A^-1 (pitch ld) into K (pitch M); *bad = 1 for a non-finite entry
__global__ void lap_scale_kernel(int M, int ld, double s, int project, const int* __restrict__ comp,
                                 const double* __restrict__ inv_size, const double* __restrict__ G, double* __restrict__ K,
                                 int* __restrict__ bad) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  if (j >= M) return;
  double g = G[(size_t)i * ld + j];
  if (project && comp[i] == comp[j]) g -= inv_size[comp[i]];
  const double v = s * g;
  K[(size_t)i * M + j] = v;
  if (!isfinite(v)) *bad = 1;
}

}  // namespace gingr

using namespace gingr;

// Hestenes sweeps until no pair is rotated; returns the squared column norms (host)
static int32_t gpmm_jacobi(gingr_ctx* ctx, int M, int n, double* d_A, int* d_flag, double* d_norm2, std::vector<double>* norm2,
                           int* sweeps_out) {
  cudaStream_t st = ctx->stream;
  const int n_even = (n + 1) & ~1;
  // a pair counts as orthogonal below the rounding level of its own dot product (length-M sums in FP64)
  const double tol = std::max(1e-14, 8.0 * 2.220446049250313e-16 * sqrt((double)M));
  int sweeps = 0;
  if (n >= 2) {
    for (; sweeps < 40; ++sweeps) {
      GINGR_CUDA_TRY(ctx, cudaMemsetAsync(d_flag, 0, sizeof(int), st));
      for (int round = 0; round < n_even - 1; ++round) {
        gpmm_jacobi_round_kernel<<<n_even / 2, 256, 0, st>>>(M, n, n_even, round, tol, d_A, d_flag);
        GINGR_LAUNCHED(ctx);
      }
      int h = 0;
      GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(&h, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
      GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
      if (!h) { ++sweeps; break; }
    }
  }
  gpmm_colnorm_kernel<<<n, 256, 0, st>>>(M, d_A, d_norm2);
  GINGR_LAUNCHED(ctx);
  norm2->resize(n);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(norm2->data(), d_norm2, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (sweeps_out) *sweeps_out = sweeps;
  return GINGR_OK;
}

namespace {

// One scalar pivoted Cholesky of an M x M block of K, run in batches of steps.  Its host history as of the last batch:
// htrace[k] = residual trace before step k, hdpiv[k] / hpiv[k] = pivot value / point of step k, for k <= steps done.
struct GpmmBlock {
  int kind = GPMM_PLAIN;
  int ncoord = 0;   // coordinates d of the 3M x 3M factor (rows 3 i + d) whose columns come from this block
  int kcap = 0;     // scalar columns it may compute
  int k = 0;        // scalar steps done
  int kalloc = 0;   // columns allocated in Ls
  DevBuf<double> d, Ls, dpiv, trace;
  DevBuf<int> pivots;
  DevBuf<uint8_t> done;
  std::vector<double> htrace, hdpiv;
  std::vector<int> hpiv;
};

using GpmmInitFn = void (*)(int, GaussKernelDev, const double*, double*, uint8_t*);
using GpmmColumnFn = void (*)(int, int, GaussKernelDev, const double*, const int*, const double*, double*, double*, uint8_t*);

void gpmm_kernels_of(int kind, GpmmInitFn* init, GpmmColumnFn* column) {
  *init = kind == GPMM_MINUS ? gpmm_init_diag_kernel<GPMM_MINUS> : kind == GPMM_PLUS ? gpmm_init_diag_kernel<GPMM_PLUS>
         : kind == GPMM_LOOKUP ? gpmm_init_diag_kernel<GPMM_LOOKUP> : gpmm_init_diag_kernel<GPMM_PLAIN>;
  *column = kind == GPMM_MINUS ? gpmm_column_kernel<GPMM_MINUS> : kind == GPMM_PLUS ? gpmm_column_kernel<GPMM_PLUS>
           : kind == GPMM_LOOKUP ? gpmm_column_kernel<GPMM_LOOKUP> : gpmm_column_kernel<GPMM_PLAIN>;
}

int32_t gpmm_block_init(gingr_ctx* ctx, int M, int kind, int ncoord, int kcap, const GaussKernelDev& kp, const double* pts,
                        GpmmBlock& b) {
  b.kind = kind; b.ncoord = ncoord; b.kcap = kcap;
  // the factor grows in chunks of columns so that a small rank does not allocate M x kcap
  b.kalloc = std::min(kcap, 256);
  GINGR_CUDA_TRY(ctx, b.d.alloc(M));
  GINGR_CUDA_TRY(ctx, b.done.alloc(M));
  GINGR_CUDA_TRY(ctx, b.Ls.alloc((size_t)b.kalloc * M));
  GINGR_CUDA_TRY(ctx, b.pivots.alloc(kcap + 1));
  GINGR_CUDA_TRY(ctx, b.dpiv.alloc(kcap + 1));
  GINGR_CUDA_TRY(ctx, b.trace.alloc(kcap + 2));
  GpmmInitFn init;
  GpmmColumnFn column;
  gpmm_kernels_of(kind, &init, &column);
  init<<<ceil_div(M, 256), 256, 0, ctx->stream>>>(M, kp, pts, b.d.p, b.done.p);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

// the block's next batch of steps (at most 32, never past kcap), then the pivot and trace of the step after it; the
// history is copied back
int32_t gpmm_block_batch(gingr_ctx* ctx, int M, int nb, const GaussKernelDev& kp, const double* pts, double* pmax, int* pidx,
                         double* psum, GpmmBlock& b) {
  cudaStream_t st = ctx->stream;
  const int batch = std::min(32, b.kcap - b.k);
  if (b.k + batch > b.kalloc) {   // grow the factor
    const int knew = std::min(b.kcap, std::max(b.kalloc * 2, b.k + batch));
    DevBuf<double> bigger;
    GINGR_CUDA_TRY(ctx, bigger.alloc((size_t)knew * M));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(bigger.p, b.Ls.p, sizeof(double) * (size_t)b.k * M, cudaMemcpyDeviceToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    b.Ls = std::move(bigger);
    b.kalloc = knew;
  }
  GpmmInitFn init;
  GpmmColumnFn column;
  gpmm_kernels_of(b.kind, &init, &column);
  for (int s = 0; s < batch; ++s) {
    const int k = b.k + s;
    gpmm_argmax_partial_kernel<<<nb, 256, 0, st>>>(M, b.d.p, b.done.p, pmax, pidx, psum);
    gpmm_argmax_final_kernel<<<1, 32, 0, st>>>(nb, k, pmax, pidx, psum, b.pivots.p, b.dpiv.p, b.trace.p);
    column<<<ceil_div(M, 256), 256, sizeof(double) * (size_t)std::max(k, 1), st>>>(M, k, kp, pts, b.pivots.p, b.dpiv.p, b.Ls.p,
                                                                                  b.d.p, b.done.p);
    ctx->launches += 3;
  }
  b.k += batch;
  gpmm_argmax_partial_kernel<<<nb, 256, 0, st>>>(M, b.d.p, b.done.p, pmax, pidx, psum);
  gpmm_argmax_final_kernel<<<1, 32, 0, st>>>(nb, b.k, pmax, pidx, psum, b.pivots.p, b.dpiv.p, b.trace.p);
  ctx->launches += 2;
  b.htrace.resize(b.k + 1);
  b.hdpiv.resize(b.k + 1);
  b.hpiv.resize(b.k + 1);
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(b.htrace.data(), b.trace.p, sizeof(double) * (b.k + 1), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(b.hdpiv.data(), b.dpiv.p, sizeof(double) * (b.k + 1), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(b.hpiv.data(), b.pivots.p, sizeof(int) * (b.k + 1), cudaMemcpyDeviceToHost, st));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// scalismo's approximateGPCholesky for a kernel that is diagonal in the coordinate index, with coordinate d taking the
// scalar block blk[g[d]] (rows 3 i + d of the 3M x 3M matrix).  The 3M x 3M algorithm picks the first maximal residual
// diagonal; a pivot in one coordinate leaves the others' residuals untouched and each block's pivot values never increase,
// so its column sequence is the merge of the blocks' scalar sequences: at each step the coordinate whose next pivot value
// is largest, ties to the lowest index 3 i + d.  Coordinates that share a block are at most one scalar step apart (on a
// tie the lagging one's pivot point has the lower index), which gives the residual trace before a step as, per block,
// n T(k) - c (T(k) - T(k + 1)) with k the lagging step and c the coordinates one step ahead.  The loop stops where the
// reference's does -- trace <= relTol * trace(K), or max_rank columns -- or where a block would need a column past kcap.
// The arguments are checked by the callers.  lookup (device, M x M, pitch M) non-null: the one block is that matrix
// (GPMM_LOOKUP) instead of the Gaussian kp.
int32_t gpmm_build(gingr_ctx* ctx, const char* fn, bool symmetric, int32_t M, const double* ref_pts, const int32_t* tri,
                   int32_t T, const GaussKernelDev& kp, const double* lookup, double rel_tol, int32_t max_rank,
                   gingr_model** out, int32_t* rank_out) {
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const long long full_cap = max_rank > 0 ? std::min<long long>(max_rank, 3LL * M) : 3LL * M;
  const int nblk = symmetric ? 2 : 1;
  const int g[3] = {0, symmetric ? 1 : 0, symmetric ? 1 : 0};
  const int nb = std::min(128, ceil_div(M, 256));
  std::unique_ptr<gingr_model> m;
  int r = 0;
  {   // the factors and their scratch are freed before the regression constants are built
    DevBuf<double> pts, pmax, psum;
    DevBuf<int> pidx, flag;
    GpmmBlock blk[2];
    GINGR_CUDA_TRY(ctx, pts.alloc((size_t)3 * M));
    GINGR_CUDA_TRY(ctx, pmax.alloc(nb));
    GINGR_CUDA_TRY(ctx, psum.alloc(nb));
    GINGR_CUDA_TRY(ctx, pidx.alloc(nb));
    GINGR_CUDA_TRY(ctx, flag.alloc(4));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(pts.p, ref_pts, sizeof(double) * 3 * (size_t)M, cudaMemcpyHostToDevice, st));
    const double* src = lookup ? lookup : pts.p;   // what the blocks' entries are computed from
    for (int b = 0; b < nblk; ++b) {
      const int ncoord = symmetric ? (b == 0 ? 1 : 2) : 3;
      const int kind = symmetric ? (b == 0 ? GPMM_MINUS : GPMM_PLUS) : lookup ? GPMM_LOOKUP : GPMM_PLAIN;
      // scalar columns that may be needed (6000: the previous columns' pivot row is staged in 48 KB of shared memory)
      const int kcap = (int)std::min<long long>(std::min<long long>((full_cap + ncoord - 1) / ncoord, M), 6000);
      GINGR_TRY(gpmm_block_init(ctx, M, kind, ncoord, kcap, kp, src, blk[b]));
    }
    for (int b = 0; b < nblk; ++b) GINGR_TRY(gpmm_block_batch(ctx, M, nb, kp, src, pmax.p, pidx.p, psum.p, blk[b]));
    // ---- the merge, batch by batch: a block runs its next batch when the merged sequence takes its first column not yet computed
    double tol = 0.0;
    for (int b = 0; b < nblk; ++b) tol += rel_tol * blk[b].ncoord * blk[b].htrace[0];
    int kd[3] = {0, 0, 0};   // scalar columns coordinate d has taken
    long long cols = 0;
    for (;;) {
      if (cols >= full_cap) break;
      double tr = 0.0;
      for (int b = 0; b < nblk; ++b) {
        int klag = M, ahead = 0;
        for (int dd = 0; dd < 3; ++dd)
          if (g[dd] == b) klag = std::min(klag, kd[dd]);
        for (int dd = 0; dd < 3; ++dd) ahead += g[dd] == b && kd[dd] > klag;
        const std::vector<double>& h = blk[b].htrace;
        tr += ahead ? blk[b].ncoord * h[klag] - ahead * (h[klag] - h[klag + 1]) : blk[b].ncoord * h[klag];
      }
      if (!(tr > tol)) break;
      int dn = -1;
      for (int dd = 0; dd < 3; ++dd) {
        if (kd[dd] >= M) continue;   // every point of this coordinate is a pivot
        if (dn < 0) { dn = dd; continue; }
        const GpmmBlock &a = blk[g[dd]], &c = blk[g[dn]];
        const double va = a.hdpiv[kd[dd]], vc = c.hdpiv[kd[dn]];
        if (va > vc || (va == vc && 3LL * a.hpiv[kd[dd]] + dd < 3LL * c.hpiv[kd[dn]] + dn)) dn = dd;
      }
      if (dn < 0) break;
      GpmmBlock& b = blk[g[dn]];
      if (kd[dn] >= b.k) {
        if (b.k >= b.kcap) break;
        GINGR_TRY(gpmm_block_batch(ctx, M, nb, kp, src, pmax.p, pidx.p, psum.p, b));
      }
      ++kd[dn];
      ++cols;
    }
    const int rank = (int)cols;
    if (rank <= 0) return gingr_fail(ctx, GINGR_ERR_ARG, (std::string(fn) + ": the tolerance leaves an empty model").c_str());
    // ---- KL basis: one-sided Jacobi on each block's factor; where the block's coordinates took different column counts
    // the lower count gets a truncated copy, rotated on its own
    DevBuf<double> Lt[2], norm2[3];
    std::vector<double> n2[3];
    const double* setA[3] = {nullptr, nullptr, nullptr};
    int set_of[3] = {0, 0, 0};
    int nset = 0;
    for (int b = 0; b < nblk; ++b) {
      int hi = 0, lo = M;
      for (int dd = 0; dd < 3; ++dd)
        if (g[dd] == b) { hi = std::max(hi, kd[dd]); lo = std::min(lo, kd[dd]); }
      const int shi = nset++;
      const int slo = lo < hi && lo > 0 ? nset++ : shi;
      for (int dd = 0; dd < 3; ++dd)
        if (g[dd] == b) set_of[dd] = kd[dd] == hi ? shi : slo;
      GINGR_CUDA_TRY(ctx, norm2[shi].alloc(std::max(hi, 1)));
      setA[shi] = blk[b].Ls.p;
      if (slo != shi) {
        GINGR_CUDA_TRY(ctx, norm2[slo].alloc(lo));
        GINGR_CUDA_TRY(ctx, Lt[b].alloc((size_t)lo * M));
        GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(Lt[b].p, blk[b].Ls.p, sizeof(double) * (size_t)lo * M, cudaMemcpyDeviceToDevice, st));
        setA[slo] = Lt[b].p;
      }
      if (hi > 0) GINGR_TRY(gpmm_jacobi(ctx, M, hi, blk[b].Ls.p, flag.p, norm2[shi].p, &n2[shi], nullptr));
      if (slo != shi) GINGR_TRY(gpmm_jacobi(ctx, M, lo, Lt[b].p, flag.p, norm2[slo].p, &n2[slo], nullptr));
    }
    for (int q = nset; q < 3; ++q) setA[q] = setA[0];
    // ---- columns of the model, sorted by variance (descending; ties: dimension, then scalar column)
    std::vector<GpmmColumn> cols_v;
    std::vector<double> lam;
    for (int dd = 0; dd < 3; ++dd)
      for (int j = 0; j < kd[dd]; ++j) {
        cols_v.push_back(GpmmColumn{set_of[dd], j, dd});
        lam.push_back(n2[set_of[dd]][j]);
      }
    std::vector<int> order(cols_v.size());
    for (size_t q = 0; q < order.size(); ++q) order[q] = (int)q;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return lam[x] > lam[y]; });
    r = (int)cols_v.size();
    std::vector<GpmmColumn> scols(r);
    std::vector<double> var(r);
    for (int q = 0; q < r; ++q) { scols[q] = cols_v[order[q]]; var[q] = lam[order[q]]; }
    // ---- the model handle
    DevBuf<GpmmColumn> dcols;
    m.reset(new gingr_model());
    m->ctx = ctx;
    m->M = M; m->r = r; m->rp = (r + 7) / 8 * 8; m->m0 = 0; m->Ml = M;
    GINGR_CUDA_TRY(ctx, m->ref.alloc((size_t)3 * M));
    GINGR_CUDA_TRY(ctx, m->mean.alloc((size_t)3 * M));
    GINGR_CUDA_TRY(ctx, m->sqrt_lambda.alloc(m->rp));
    GINGR_CUDA_TRY(ctx, m->phi.alloc((size_t)3 * M * m->rp));
    GINGR_CUDA_TRY(ctx, dcols.alloc(r));
    std::vector<double> sl(m->rp, 0.0);
    for (int q = 0; q < r; ++q) sl[q] = sqrt(var[q]);
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->ref.p, pts.p, sizeof(double) * 3 * (size_t)M, cudaMemcpyDeviceToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(m->mean.p, 0, sizeof(double) * 3 * (size_t)M, st));
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(m->phi.p, 0, sizeof(double) * (size_t)3 * M * m->rp, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(m->sqrt_lambda.p, sl.data(), sizeof(double) * m->rp, cudaMemcpyHostToDevice, st));
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(dcols.p, scols.data(), sizeof(GpmmColumn) * r, cudaMemcpyHostToDevice, st));
    const double* setn[3];
    for (int q = 0; q < 3; ++q) setn[q] = q < nset ? norm2[q].p : norm2[0].p;
    gpmm_assemble_kernel<<<dim3(ceil_div(M, 256), r), 256, 0, st>>>(M, r, m->rp, dcols.p, setA[0], setn[0], setA[1], setn[1],
                                                                    setA[2], setn[2], m->phi.p);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));   // sl / scols are host vectors
  }
  GINGR_TRY(model_upload_topology(ctx, m.get(), tri, T));
  GINGR_TRY(model_build_constants(ctx, m.get()));
  *out = m.release();
  if (rank_out) *rank_out = r;
  return GINGR_OK;
}

int32_t gpmm_build_gaussian(gingr_ctx* ctx, const char* fn, bool symmetric, int32_t M, const double* ref_pts, const int32_t* tri,
                            int32_t T, int32_t n_kernels, const double* sigma, const double* scaling, double rel_tol,
                            int32_t max_rank, gingr_model** out, int32_t* rank_out) {
  if (!ctx || !ref_pts || !out || M <= 0 || T < 0 || (T > 0 && !tri) || n_kernels <= 0 || n_kernels > 8 || !sigma || !scaling ||
      !(rel_tol >= 0.0) || max_rank < 0)
    return gingr_fail(ctx, GINGR_ERR_ARG, (std::string(fn) + ": bad argument (1..8 kernels, relTol >= 0)").c_str());
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, (std::string(fn) + ": single-GPU entry point (build before sharding)").c_str());
  GaussKernelDev kp;
  kp.n = n_kernels;
  for (int q = 0; q < n_kernels; ++q) {
    if (!(sigma[q] > 0.0) || !(scaling[q] > 0.0)) return gingr_fail(ctx, GINGR_ERR_ARG, (std::string(fn) + ": sigma and scaling must be positive").c_str());
    kp.inv_sigma2[q] = 1.0 / (sigma[q] * sigma[q]);
    kp.scaling[q] = scaling[q];
  }
  return gpmm_build(ctx, fn, symmetric, M, ref_pts, tri, T, kp, nullptr, rel_tol, max_rank, out, rank_out);
}

// The largest template of the inverse-Laplacian builder: its models are nearly full rank, and the pivoted Cholesky computes
// at most 6000 scalar columns (gpmm_build's kcap).
constexpr int LAP_MAX_M = 6000;

// Ks = scaling (L + gamma I)^-1, or for gamma = 0 scaling L^+ = scaling ((L + P)^-1 - P), into K (device, M x M, pitch M).
// The components behind P come from a union-find over the triangles on the host (O(T)); a vertex in no triangle is a
// component of its own.  The system [A; I] is factorised by the data-flow Cholesky, the identity rows come out as
// Y = L_A^-T, and A^-1 = Y Y^T is the DMMA Gram of Y^T.  *failed: A not numerically positive definite, or Ks not finite.
int32_t laplacian_inverse(gingr_ctx* ctx, int M, const int32_t* tri, int T, double scaling, double gamma, DevBuf<double>& K,
                          bool* failed) {
  cudaStream_t st = ctx->stream;
  const bool project = gamma == 0.0;
  std::vector<int> comp(M, 0);
  std::vector<double> inv_size(1, 0.0);
  if (project) {
    std::vector<int> parent(M);
    for (int i = 0; i < M; ++i) parent[i] = i;
    auto find = [&](int x) {
      while (parent[x] != x) x = parent[x] = parent[parent[x]];
      return x;
    };
    for (int t = 0; t < T; ++t)
      for (int e = 0; e < 3; ++e) {
        const int a = find(tri[3 * t + e]), b = find(tri[3 * t + (e + 1) % 3]);
        if (a != b) parent[std::max(a, b)] = std::min(a, b);
      }
    std::vector<int> label(M, -1), size;
    for (int i = 0; i < M; ++i) {
      const int root = find(i);
      if (label[root] < 0) { label[root] = (int)size.size(); size.push_back(0); }
      comp[i] = label[root];
      ++size[comp[i]];
    }
    inv_size.resize(size.size());
    for (size_t c = 0; c < size.size(); ++c) inv_size[c] = 1.0 / size[c];
  }
  const int ld = (M + 7) / 8 * 8;   // even pitch, 16-byte rows (chol_df), rp of the Gram
  DevBuf<double> G;
  DevBuf<int32_t> dtri, dcomp;
  DevBuf<double> dinv;
  DevBuf<int> info;
  GINGR_CUDA_TRY(ctx, dtri.alloc((size_t)3 * T));
  GINGR_CUDA_TRY(ctx, dcomp.alloc(M));
  GINGR_CUDA_TRY(ctx, dinv.alloc(inv_size.size()));
  GINGR_CUDA_TRY(ctx, info.alloc(4));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(dtri.p, tri, sizeof(int32_t) * 3 * (size_t)T, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(dcomp.p, comp.data(), sizeof(int) * (size_t)M, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(dinv.p, inv_size.data(), sizeof(double) * inv_size.size(), cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(info.p, 0, sizeof(int) * 4, st));
  {
    DevBuf<double> sys, Yt;
    CholWs cws;
    GramPlan plan;
    GINGR_CUDA_TRY(ctx, sys.alloc((size_t)(2 * M + 8) * ld));
    GINGR_CUDA_TRY(ctx, Yt.alloc((size_t)M * ld));
    GINGR_CUDA_TRY(ctx, G.alloc((size_t)M * ld));
    GINGR_TRY(cws.alloc(ctx, M, 2 * M));
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(sys.p, 0, sizeof(double) * (size_t)(2 * M + 8) * ld, st));
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(Yt.p, 0, sizeof(double) * (size_t)M * ld, st));
    lap_edges_kernel<<<ceil_div(T, 256), 256, 0, st>>>(T, dtri.p, ld, sys.p);
    GINGR_LAUNCHED(ctx);
    lap_rows_kernel<<<M, 256, 0, st>>>(M, ld, gamma, project ? 1 : 0, dcomp.p, dinv.p, sys.p);
    GINGR_LAUNCHED(ctx);
    GINGR_TRY(cholesky_df_enqueue(ctx, M, 2 * M, sys.p, ld, info.p, cws));
    GINGR_TRY(transpose_enqueue(ctx, M, sys.p + (size_t)M * ld, ld, Yt.p, ld));   // Y^T = L_A^-1, lower triangular
    GINGR_TRY(plan.build(ctx, M, M, ld));
    GINGR_TRY(gram_partials_enqueue(ctx, plan, Yt.p, nullptr));
    GINGR_TRY(gram_finish_enqueue(ctx, plan, plan.d_partial.p, nullptr, 0.0, 0, nullptr, nullptr, ld, G.p));
    GINGR_CUDA_TRY(ctx, K.alloc((size_t)M * M));
    lap_scale_kernel<<<dim3(ceil_div(M, 256), M), 256, 0, st>>>(M, ld, scaling, project ? 1 : 0, dcomp.p, dinv.p, G.p, K.p,
                                                                 info.p + 1);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    int h[2] = {0, 0};
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(h, info.p, sizeof(int) * 2, cudaMemcpyDeviceToHost, st));
    GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));   // also: the host vectors above were copied
    *failed = h[0] != 0 || h[1] != 0;
  }
  return GINGR_OK;
}

}  // namespace

extern "C" {

int32_t gingr_gpmm_gaussian_mixture(gingr_ctx* ctx, int32_t M, const double* ref_pts, const int32_t* tri, int32_t T,
                                    int32_t n_kernels, const double* sigma, const double* scaling, double rel_tol,
                                    int32_t max_rank, gingr_model** out, int32_t* rank_out) {
  return gpmm_build_gaussian(ctx, "gingr_gpmm_gaussian_mixture", false, M, ref_pts, tri, T, n_kernels, sigma, scaling, rel_tol,
                             max_rank, out, rank_out);
}

int32_t gingr_gpmm_gaussian_symmetric(gingr_ctx* ctx, int32_t M, const double* ref_pts, const int32_t* tri, int32_t T,
                                      int32_t n_kernels, const double* sigma, const double* scaling, double rel_tol,
                                      int32_t max_rank, gingr_model** out, int32_t* rank_out) {
  return gpmm_build_gaussian(ctx, "gingr_gpmm_gaussian_symmetric", true, M, ref_pts, tri, T, n_kernels, sigma, scaling, rel_tol,
                             max_rank, out, rank_out);
}

int32_t gingr_gpmm_inverse_laplacian(gingr_ctx* ctx, int32_t M, const double* ref_pts, const int32_t* tri, int32_t T,
                                     double scaling, double gamma, double rel_tol, int32_t max_rank, gingr_model** out,
                                     int32_t* rank_out) {
  const char* fn = "gingr_gpmm_inverse_laplacian";
  if (out) *out = nullptr;
  if (!ctx || !ref_pts || !out || M <= 0 || T <= 0 || !tri || !(scaling > 0.0) || !std::isfinite(scaling) || !(gamma >= 0.0) ||
      !std::isfinite(gamma) || !(rel_tol >= 0.0) || max_rank < 0)
    return gingr_fail(ctx, GINGR_ERR_ARG, (std::string(fn) + ": bad argument (T > 0, scaling > 0 and gamma >= 0 finite, relTol >= 0, "
                                                             "maxRank >= 0)").c_str());
  for (int64_t q = 0; q < 3 * (int64_t)T; ++q)
    if (tri[q] < 0 || tri[q] >= M) return gingr_fail(ctx, GINGR_ERR_ARG, (std::string(fn) + ": triangle index outside [0, M)").c_str());
  if (M > LAP_MAX_M)
    return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, (std::string(fn) + ": at most 6000 vertices (a dense, nearly full-rank model); "
                                                                     "decimate the template first").c_str());
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, (std::string(fn) + ": single-GPU entry point (build before sharding)").c_str());
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> K;
  bool failed = false;
  GINGR_TRY(laplacian_inverse(ctx, M, tri, T, scaling, gamma, K, &failed));
  if (failed) return gingr_fail(ctx, GINGR_MODEL_FLEXIBILITY, (std::string(fn) + ": L + gamma I is not numerically positive definite "
                                                                                 "or the kernel is not finite").c_str());
  GaussKernelDev kp{};
  return gpmm_build(ctx, fn, false, M, ref_pts, tri, T, kp, K.p, rel_tol, max_rank, out, rank_out);
}

// The model as scalismo stores it (SURVEY.md A1): meanVector [3M], basisMatrix column-major [3M x r] (leading dimension
// ld_basis >= 3M), variance [r].  Any output may be NULL.
int32_t gingr_model_download(gingr_ctx* ctx, const gingr_model* model, int32_t* M_out, int32_t* r_out, double* ref_pts,
                             double* mean, double* basis, int64_t ld_basis, double* variance) {
  if (!ctx || !model) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_download: bad argument");
  if (ctx->nranks != 1) return gingr_fail(ctx, GINGR_ERR_UNSUPPORTED, "gingr_model_download: single-GPU entry point");
  const int M = model->M, r = model->r, rp = model->rp;
  if (M_out) *M_out = M;
  if (r_out) *r_out = r;
  if (basis && ld_basis < 3 * (int64_t)M) return gingr_fail(ctx, GINGR_ERR_ARG, "gingr_model_download: ld_basis < 3 M");
  GINGR_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if (ref_pts) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(ref_pts, model->ref.p, sizeof(double) * 3 * (size_t)M, cudaMemcpyDeviceToHost, st));
  if (mean) GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(mean, model->mean.p, sizeof(double) * 3 * (size_t)M, cudaMemcpyDeviceToHost, st));
  std::vector<double> sl, rows;
  if (variance) {
    sl.resize(rp);
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(sl.data(), model->sqrt_lambda.p, sizeof(double) * rp, cudaMemcpyDeviceToHost, st));
  }
  if (basis) {
    rows.resize((size_t)3 * M * rp);
    GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(rows.data(), model->phi.p, sizeof(double) * rows.size(), cudaMemcpyDeviceToHost, st));
  }
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (variance)
    for (int a = 0; a < r; ++a) variance[a] = sl[a] * sl[a];
  if (basis)
    for (int a = 0; a < r; ++a)
      for (size_t k = 0; k < (size_t)3 * M; ++k) basis[(size_t)a * ld_basis + k] = rows[k * rp + a];
  return GINGR_OK;
}

}  // extern "C"
