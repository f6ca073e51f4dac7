// closest.cu -- K2: ICP closest-point correspondence for sm_100a.   COMPILED WITH -fmad=false.
//
// Replaces registration/utils/ClosestPointRegistrator.scala:
//   ClosestPointUnstructuredPointsDomain3D (:133-148)  nearest target vertex        -> nn_vertex_kernel
//   ClosestPointTriangleMesh3D (:74-96)                closest point on a triangle   -> surface_kernel
//     + findClosestPoint of that point (:83), isPointOnBoundary (:53-55), isNormalDirectionOpposite
//       (:57-60), isClosestPointIntersecting (:62-72)                                -> line_mesh_kernel,
//                                                                                       icp_weights_kernel
// Exactness: every distance is evaluated in FP64 with individually rounded operations in the order the
// JVM evaluates scalismo's `norm2` (x*x + y*y + z*z, no FMA contraction -- hence -fmad=false), the scan
// is in ascending index order with a strict `<`, and partial results of index ranges are merged lowest
// range first, so the argmin is exact with ties broken by the lowest index.
// The searches are tiled brute force (queries in registers, candidates staged through shared memory),
// FP64-pipe bound at 8 M N flop for the vertex search.
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "closest.cuh"
#include "closest_geom.cuh"
#include "batch.cuh"
#include "grid.cuh"

namespace gingr {

constexpr int QT = 128;    // queries (threads) per CTA
constexpr int PT = 256;    // candidate points per shared-memory tile
constexpr int TT = 64;     // candidate triangles per shared-memory tile

// ---------------------------------------------------------------------------------------------
// nearest vertex
// ---------------------------------------------------------------------------------------------
GINGR_KERNEL((QT), nn_vertex_kernel, int M, const double* __restrict__ q /*AoS [M][3]*/, int N,
                                                       const double* __restrict__ pts /*SoA [3][N]*/,
                                                       double* __restrict__ part_d2, int32_t* __restrict__ part_idx) {
  __shared__ double sx[PT], sy[PT], sz[PT];
  const int i = blockIdx.x * QT + threadIdx.x;
  const int per = (N + gridDim.y - 1) / gridDim.y;
  const int j_begin = blockIdx.y * per, j_end = min(N, j_begin + per);
  const int ii = min(i, M - 1);
  const double qx = q[3 * ii], qy = q[3 * ii + 1], qz = q[3 * ii + 2];
  double best = INFINITY;
  int32_t bi = -1;
  for (int j0 = j_begin; j0 < j_end; j0 += PT) {
    const int cnt = min(PT, j_end - j0);
    __syncthreads();
    for (int t = threadIdx.x; t < cnt; t += QT) {
      sx[t] = pts[j0 + t];
      sy[t] = pts[N + j0 + t];
      sz[t] = pts[2 * N + j0 + t];
    }
    __syncthreads();
#pragma unroll 4
    for (int t = 0; t < cnt; ++t) {
      const double dx = qx - sx[t], dy = qy - sy[t], dz = qz - sz[t];
      const double d = dx * dx + dy * dy + dz * dz;
      if (d < best) {
        best = d;
        bi = j0 + t;
      }
    }
  }
  if (i < M) {
    part_d2[(size_t)blockIdx.y * M + i] = best;
    part_idx[(size_t)blockIdx.y * M + i] = bi;
  }
}

GINGR_KERNEL_NB(nn_reduce_kernel, int M, int splits, const double* __restrict__ part_d2,
                                 const int32_t* __restrict__ part_idx, double* __restrict__ d2,
                                 int32_t* __restrict__ idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  double best = INFINITY;
  int32_t bi = -1;
  for (int k = 0; k < splits; ++k) {
    const double d = part_d2[(size_t)k * M + i];
    if (d < best) {
      best = d;
      bi = part_idx[(size_t)k * M + i];
    }
  }
  d2[i] = best;
  idx[i] = bi;
}

// part: [splits][M] d2, tri ; [splits][M][3] cp
GINGR_KERNEL((QT), surface_kernel, int M, const double* __restrict__ q, int N,
                                                     const double* __restrict__ verts /*SoA [3][N]*/, int T,
                                                     const int32_t* __restrict__ tri, double* __restrict__ part_d2,
                                                     int32_t* __restrict__ part_tri, double* __restrict__ part_cp) {
  __shared__ double st[TT][9];
  __shared__ double sb[TT][6];   // bounding box of the staged triangle (lo, hi)
  const int i = blockIdx.x * QT + threadIdx.x;
  const int per = (T + gridDim.y - 1) / gridDim.y;
  const int t_begin = blockIdx.y * per, t_end = min(T, t_begin + per);
  const int ii = min(i, M - 1);
  const double qx = q[3 * ii], qy = q[3 * ii + 1], qz = q[3 * ii + 2];
  double best = INFINITY, bx = 0, by = 0, bz = 0;
  int32_t bt = -1;
  for (int t0 = t_begin; t0 < t_end; t0 += TT) {
    const int cnt = min(TT, t_end - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * 9; e += QT) {
      const int t = e / 9, k = e % 9;
      const int v = tri[3 * (t0 + t) + k / 3];
      st[t][k] = verts[(size_t)(k % 3) * N + v];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * 3; e += QT) {
      const int t = e / 3, k = e % 3;
      const double a = st[t][k], b = st[t][3 + k], c = st[t][6 + k];
      sb[t][k] = fmin(a, fmin(b, c));
      sb[t][3 + k] = fmax(a, fmax(b, c));
    }
    __syncthreads();
    for (int t = 0; t < cnt; ++t) {
      // a triangle lies inside its box: it cannot beat the best (strict <, so it cannot replace an equal one either)
      // when the box is farther -- by more than the rounding of this bound
      const double ex = fmax(fmax(sb[t][0] - qx, qx - sb[t][3]), 0.0), ey = fmax(fmax(sb[t][1] - qy, qy - sb[t][4]), 0.0),
                   ez = fmax(fmax(sb[t][2] - qz, qz - sb[t][5]), 0.0);
      if ((ex * ex + ey * ey + ez * ez) * (1.0 - 1e-12) > best) continue;
      double cx, cy, cz;
      closest_on_triangle(qx, qy, qz, &st[t][0], &st[t][3], &st[t][6], cx, cy, cz);
      const double dx = qx - cx, dy = qy - cy, dz = qz - cz;
      const double d = dx * dx + dy * dy + dz * dz;
      if (d < best) { best = d; bt = t0 + t; bx = cx; by = cy; bz = cz; }
    }
  }
  if (i < M) {
    const size_t o = (size_t)blockIdx.y * M + i;
    part_d2[o] = best;
    part_tri[o] = bt;
    part_cp[3 * o] = bx;
    part_cp[3 * o + 1] = by;
    part_cp[3 * o + 2] = bz;
  }
}

GINGR_KERNEL_NB(surface_reduce_kernel, int M, int splits, const double* __restrict__ part_d2,
                                      const int32_t* __restrict__ part_tri, const double* __restrict__ part_cp,
                                      double* __restrict__ d2, int32_t* __restrict__ tri_out,
                                      double* __restrict__ cp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  double best = INFINITY;
  int bk = 0;
  for (int k = 0; k < splits; ++k) {
    const double d = part_d2[(size_t)k * M + i];
    if (d < best) { best = d; bk = k; }
  }
  const size_t o = (size_t)bk * M + i;
  d2[i] = best;
  if (tri_out) tri_out[i] = part_tri[o];
  cp[3 * i] = part_cp[3 * o];
  cp[3 * i + 1] = part_cp[3 * o + 1];
  cp[3 * i + 2] = part_cp[3 * o + 2];
}

// ---------------------------------------------------------------------------------------------
// Intersections of the infinite line o + s d with a mesh (scalismo getIntersectionPoints, SURVEY.md A6), hits
// equal to o dropped (`.filter(f => f != p)`), nearest hit kept (strict <, ascending triangle id: lowest id on
// ties).  Two users:
//   isClosestPointIntersecting (:62-72)   o = vertex i of the mesh itself, d = o - cp_i; triangles incident to
//                                         vertex i only touch the line at o and are skipped (SELF = true)
//   ClosestPointAlongNormal (:105-110)    o = template vertex, d = its normal, mesh = the target (SELF = false);
//                                         the hit point itself is needed (WITH_POINT = true)
// DIFF = true: the direction is o - other[i] (computed in registers), else other[i] is the direction.
// ---------------------------------------------------------------------------------------------
GINGR_KERNEL_T((bool SELF, bool DIFF, bool WITH_POINT), (SELF, DIFF, WITH_POINT), (QT), line_mesh_kernel, int M,
               const double* __restrict__ o /*AoS*/, const double* __restrict__ other /*AoS*/,
               const double* __restrict__ mesh /*AoS vertices*/, int T, const int32_t* __restrict__ tri,
               double* __restrict__ part_min, double* __restrict__ part_pt,
               int q0 /*vertex id of query 0 (SELF: a query range of the mesh)*/) {
  __shared__ double st[TT][9];
  __shared__ int32_t sv[TT][3];
  const int i = blockIdx.x * QT + threadIdx.x;
  const int per = (T + gridDim.y - 1) / gridDim.y;
  const int t_begin = blockIdx.y * per, t_end = min(T, t_begin + per);
  const int ii = min(i, M - 1);
  const double ox = o[3 * ii], oy = o[3 * ii + 1], oz = o[3 * ii + 2];
  double dx = other[3 * ii], dy = other[3 * ii + 1], dz = other[3 * ii + 2];
  if (DIFF) { dx = ox - dx; dy = oy - dy; dz = oz - dz; }
  double best = INFINITY, bx = ox, by = oy, bz = oz;
  for (int t0 = t_begin; t0 < t_end; t0 += TT) {
    const int cnt = min(TT, t_end - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * 9; e += QT) {
      const int t = e / 9, k = e % 9;
      const int v = tri[3 * (t0 + t) + k / 3];
      st[t][k] = mesh[3 * v + (k % 3)];
      if (k % 3 == 0) sv[t][k / 3] = v;
    }
    __syncthreads();
    for (int t = 0; t < cnt; ++t) {
      if (SELF && (sv[t][0] == q0 + ii || sv[t][1] == q0 + ii || sv[t][2] == q0 + ii)) continue;
      double d, ix, iy, iz;
      if (!line_triangle_hit(ox, oy, oz, dx, dy, dz, &st[t][0], &st[t][3], &st[t][6], d, ix, iy, iz)) continue;
      if (d < best) {
        best = d;
        if (WITH_POINT) { bx = ix; by = iy; bz = iz; }
      }
    }
  }
  if (i < M) {
    const size_t oidx = (size_t)blockIdx.y * M + i;
    part_min[oidx] = best;
    if (WITH_POINT) {
      part_pt[3 * oidx] = bx;
      part_pt[3 * oidx + 1] = by;
      part_pt[3 * oidx + 2] = bz;
    }
  }
}

// nearest hit over the triangle-range splits (lowest range first on ties); no hit: dist = 0, point = o, hit = 0
// (ClosestPointRegistrator.scala:127 "return p to avoid influencing the distance measure")
GINGR_KERNEL_NB(line_hit_reduce_kernel, int M, int splits, const double* __restrict__ o,
                                       const double* __restrict__ part_min, const double* __restrict__ part_pt,
                                       double* __restrict__ dist, double* __restrict__ pt, uint8_t* __restrict__ hit) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  double best = INFINITY;
  int bk = -1;
  for (int k = 0; k < splits; ++k) {
    const double d = part_min[(size_t)k * M + i];
    if (d < best) { best = d; bk = k; }
  }
  if (bk >= 0) {
    const size_t oidx = (size_t)bk * M + i;
    dist[i] = best;
    pt[3 * i] = part_pt[3 * oidx]; pt[3 * i + 1] = part_pt[3 * oidx + 1]; pt[3 * i + 2] = part_pt[3 * oidx + 2];
    hit[i] = 1;
  } else {
    dist[i] = 0.0;
    pt[3 * i] = o[3 * i]; pt[3 * i + 1] = o[3 * i + 1]; pt[3 * i + 2] = o[3 * i + 2];
    hit[i] = 0;
  }
}

// ---------------------------------------------------------------------------------------------
// vertex normals from a CSR vertex -> triangle adjacency (ascending triangle ids = the accumulation
// order of a triangle-ordered scatter).  verts AoS [n][3]; normals AoS [n][3].   SURVEY.md A6
// ---------------------------------------------------------------------------------------------
GINGR_KERNEL_NB(vertex_normals_kernel, int n, const double* __restrict__ v, const int32_t* __restrict__ tri,
                                      const int32_t* __restrict__ adj_off, const int32_t* __restrict__ adj,
                                      double* __restrict__ normals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double ax = 0, ay = 0, az = 0;
  const int b = adj_off[i], e = adj_off[i + 1];
  for (int k = b; k < e; ++k) {
    const int t = adj[k];
    const double* a = v + 3 * tri[3 * t];
    const double* bb = v + 3 * tri[3 * t + 1];
    const double* c = v + 3 * tri[3 * t + 2];
    const double ux = bb[0] - a[0], uy = bb[1] - a[1], uz = bb[2] - a[2];
    const double wx = c[0] - a[0], wy = c[1] - a[1], wz = c[2] - a[2];
    double nx = uy * wz - uz * wy, ny = uz * wx - ux * wz, nz = ux * wy - uy * wx;
    const double len = sqrt(nx * nx + ny * ny + nz * nz);
    nx /= len; ny /= len; nz /= len;
    ax += nx; ay += ny; az += nz;
  }
  const int cnt = e - b;
  if (cnt > 0) { ax /= cnt; ay /= cnt; az /= cnt; }
  const double len = sqrt(ax * ax + ay * ay + az * az);
  normals[3 * i] = ax / len;
  normals[3 * i + 1] = ay / len;
  normals[3 * i + 2] = az / len;
}

// w = 0 if target vertex on boundary, else 0 if normals opposite, else 0 if intersecting, else 1
// (ClosestPointRegistrator.scala:84-90).  min_part: [splits][M]
GINGR_KERNEL_NB(icp_weights_kernel, int M, const double* __restrict__ p, const double* __restrict__ cp,
                                   const int32_t* __restrict__ idx, const uint8_t* __restrict__ tgt_boundary,
                                   const double* __restrict__ n_tpl /*AoS*/, const double* __restrict__ n_tgt /*AoS*/,
                                   int splits, const double* __restrict__ min_part,
                                   const uint8_t* __restrict__ hit /*may be null*/, uint8_t* __restrict__ w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const int j = idx[i];
  uint8_t out = 1;
  if (hit && !hit[i]) {
    out = 0;  // no intersection along the normal (:127)
  } else if (tgt_boundary[j]) {
    out = 0;
  } else {
    const double dot = n_tpl[3 * i] * n_tgt[3 * j] + n_tpl[3 * i + 1] * n_tgt[3 * j + 1] + n_tpl[3 * i + 2] * n_tgt[3 * j + 2];
    if (dot < 0.0) {
      out = 0;
    } else {
      double md = INFINITY;
      for (int k = 0; k < splits; ++k) md = fmin(md, min_part[(size_t)k * M + i]);
      const double vx = p[3 * i] - cp[3 * i], vy = p[3 * i + 1] - cp[3 * i + 1], vz = p[3 * i + 2] - cp[3 * i + 2];
      if (md < sqrt(vx * vx + vy * vy + vz * vz)) out = 0;
    }
  }
  w[i] = out;
}

GINGR_KERNEL_NB(gather_points_kernel, int M, const int32_t* __restrict__ idx, int N, const double* __restrict__ soa,
                                     double* __restrict__ out /*AoS*/) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const int j = idx[i];
  out[3 * i] = soa[j];
  out[3 * i + 1] = soa[N + j];
  out[3 * i + 2] = soa[2 * N + j];
}

// deterministic mean of sqrt(d2) (squared = 1) or of d2 itself (squared = 0): fixed-order tree per block; large
// inputs use MEAN_BLOCKS blocks whose partial sums the last stage adds in block order
constexpr int MEAN_BLOCKS = 64;
GINGR_KERNEL((256), mean_sqrt_kernel, int M, const double* __restrict__ d2, double* __restrict__ out,
                                                        int squared, int final_stage) {
  __shared__ double red[256];
  double s = 0.0;
  if (final_stage == 2) {   // sum of the per-block partials (in d2), divided by M
    for (int i = threadIdx.x; i < MEAN_BLOCKS; i += 256) s += d2[i];
  } else {
    for (int i = blockIdx.x * 256 + threadIdx.x; i < M; i += gridDim.x * 256) s += squared ? sqrt(d2[i]) : d2[i];
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = final_stage ? red[0] / M : red[0];
}

static void mean_sqrt_enqueue(gingr_ctx* ctx, ClosestWorkspace& ws, int M, int squared, const double* d_d2 = nullptr) {
  cudaStream_t st = ctx->stream;
  if (!d_d2) d_d2 = ws.d2.p;
  if (M <= 0) return;
  if (M <= 16384) {
    GINGR_LAUNCH(ctx, mean_sqrt_kernel, 1, 256, 0, st, M, d_d2, ws.mean_dist.p, squared, 1);
    GINGR_LAUNCHED(ctx);
  } else {
    GINGR_LAUNCH(ctx, mean_sqrt_kernel, MEAN_BLOCKS, 256, 0, st, M, d_d2, ws.mean_part.p, squared, 0);
    GINGR_LAUNCHED(ctx);
    GINGR_LAUNCH(ctx, mean_sqrt_kernel, 1, 256, 0, st, M, ws.mean_part.p, ws.mean_dist.p, 0, 2);
    GINGR_LAUNCHED(ctx);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
void build_vertex_adjacency(int n, int T, const int32_t* tri, std::vector<int32_t>* off, std::vector<int32_t>* adj) {
  off->assign((size_t)n + 1, 0);
  for (int k = 0; k < 3 * T; ++k) (*off)[tri[k] + 1]++;
  for (int i = 0; i < n; ++i) (*off)[i + 1] += (*off)[i];
  adj->assign((size_t)3 * T, 0);
  std::vector<int32_t> cur(off->begin(), off->end() - 1);
  for (int t = 0; t < T; ++t)  // ascending triangle id per vertex
    for (int k = 0; k < 3; ++k) (*adj)[cur[tri[3 * t + k]]++] = t;
}

// pointIsOnBoundary for every vertex: a vertex touching an edge that belongs to exactly one triangle
void compute_boundary_flags(int n, int T, const int32_t* tri, std::vector<uint8_t>* flags) {
  flags->assign((size_t)n, 0);
  std::vector<uint64_t> edges;
  edges.reserve((size_t)3 * T);
  for (int t = 0; t < T; ++t)
    for (int k = 0; k < 3; ++k) {
      uint32_t a = (uint32_t)tri[3 * t + k], b = (uint32_t)tri[3 * t + (k + 1) % 3];
      if (a > b) std::swap(a, b);
      edges.push_back(((uint64_t)a << 32) | b);
    }
  std::sort(edges.begin(), edges.end());
  for (size_t i = 0; i < edges.size();) {
    size_t j = i + 1;
    while (j < edges.size() && edges[j] == edges[i]) ++j;
    if (j - i == 1) {
      (*flags)[edges[i] >> 32] = 1;
      (*flags)[edges[i] & 0xffffffffu] = 1;
    }
    i = j;
  }
}

int32_t vertex_normals_enqueue(gingr_ctx* ctx, int n, const double* d_verts_aos, const int32_t* d_tri,
                               const int32_t* d_adj_off, const int32_t* d_adj, double* d_normals) {
  GINGR_LAUNCH(ctx, vertex_normals_kernel, ceil_div(n, 128), 128, 0, ctx->stream, n, d_verts_aos, d_tri, d_adj_off, d_adj, d_normals);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// static per-mesh data for a target: vertex normals (AoS) and boundary flags
int32_t mesh_static_upload(gingr_ctx* ctx, int n, const double* verts_aos_host, int T, const int32_t* tri_host,
                           DevBuf<double>* normals, DevBuf<uint8_t>* boundary) {
  std::vector<int32_t> off, adj;
  build_vertex_adjacency(n, T, tri_host, &off, &adj);
  std::vector<uint8_t> flags;
  compute_boundary_flags(n, T, tri_host, &flags);
  DevBuf<int32_t> d_off, d_adj, d_tri;
  DevBuf<double> d_v;
  GINGR_CUDA_TRY(ctx, d_off.alloc(off.size()));
  GINGR_CUDA_TRY(ctx, d_adj.alloc(adj.size()));
  GINGR_CUDA_TRY(ctx, d_tri.alloc((size_t)3 * T));
  GINGR_CUDA_TRY(ctx, d_v.alloc((size_t)3 * n));
  GINGR_CUDA_TRY(ctx, normals->alloc((size_t)3 * n));
  GINGR_CUDA_TRY(ctx, boundary->alloc((size_t)n));
  cudaStream_t st = ctx->stream;
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_adj.p, adj.data(), adj.size() * 4, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_tri.p, tri_host, (size_t)3 * T * 4, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(d_v.p, verts_aos_host, (size_t)3 * n * 8, cudaMemcpyHostToDevice, st));
  GINGR_CUDA_TRY(ctx, cudaMemcpyAsync(boundary->p, flags.data(), (size_t)n, cudaMemcpyHostToDevice, st));
  GINGR_TRY(vertex_normals_enqueue(ctx, n, d_v.p, d_tri.p, d_off.p, d_adj.p, normals->p));
  GINGR_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return GINGR_OK;
}

static int pick_splits(const gingr_ctx* ctx, int M, int candidates, int tile) {
  const int qblocks = ceil_div(M, QT);
  const int want = ceil_div(ctx->num_sms * 4, qblocks);
  // small candidate sets: ranges shorter than a shared-memory tile (down to a quarter) so that a 100-vertex problem
  // is not a few CTAs looping over everything
  return std::max(1, std::min(want, ceil_div(candidates, std::max(tile / 4, 8))));
}

int32_t ClosestWorkspace::ensure(gingr_ctx* ctx, int nq, int n_search, int T_search, int T_query_mesh) {
  const int M = nq;
  s_nn = pick_splits(ctx, M, n_search, PT);
  s_surf = T_search > 0 ? pick_splits(ctx, M, T_search, TT) : 1;
  s_line = T_query_mesh > 0 ? pick_splits(ctx, M, T_query_mesh, TT) : 1;
  const int smax = std::max(s_nn, std::max(s_surf, s_line));
  GINGR_CUDA_TRY(ctx, part_d2.alloc((size_t)smax * M));
  GINGR_CUDA_TRY(ctx, part_idx.alloc((size_t)smax * M));
  GINGR_CUDA_TRY(ctx, part_cp.alloc((size_t)3 * std::max(s_surf, s_line) * M));
  GINGR_CUDA_TRY(ctx, d2.alloc((size_t)M));
  GINGR_CUDA_TRY(ctx, surf_d2.alloc((size_t)M));
  GINGR_CUDA_TRY(ctx, idx.alloc((size_t)M));
  GINGR_CUDA_TRY(ctx, cp.alloc((size_t)3 * M));
  GINGR_CUDA_TRY(ctx, w.alloc((size_t)M));
  GINGR_CUDA_TRY(ctx, hit.alloc((size_t)M));
  // a rank that searches only a query range never writes the other entries: keep them defined (weight 0, point 0)
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(w.p, 0, (size_t)M, ctx->stream));
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(cp.p, 0, sizeof(double) * 3 * (size_t)M, ctx->stream));
  GINGR_CUDA_TRY(ctx, mean_dist.alloc(1));
  GINGR_CUDA_TRY(ctx, mean_part.alloc(MEAN_BLOCKS));
  if (grid_wanted(std::max(n_search, std::max(T_search, T_query_mesh)))) {
    if (!qorder) qorder = std::make_unique<SpatialGrid>();
    GINGR_TRY(qorder->ensure(ctx, nq, nq, false));
  }
  return GINGR_OK;
}

// Nearest vertex (of a SoA point set) of arbitrary query points (AoS, device).
int32_t nn_vertex_enqueue(gingr_ctx* ctx, ClosestWorkspace& ws, int M, const double* d_q, int N,
                          const double* d_pts_soa, double* d_d2, int32_t* d_idx, const SpatialGrid* pgrid,
                          const SpatialGrid* order) {
  if (pgrid && pgrid->built) return grid_nn_enqueue(ctx, *pgrid, M, d_q, d_d2, d_idx, order);
  const int splits = std::min(ws.s_nn, std::max(1, ceil_div(N, PT / 4)));
  GINGR_LAUNCH(ctx, nn_vertex_kernel, dim3(ceil_div(M, QT), splits), QT, 0, ctx->stream, M, d_q, N, d_pts_soa, ws.part_d2.p,
                                                                          ws.part_idx.p);
  GINGR_LAUNCHED(ctx);
  GINGR_LAUNCH(ctx, nn_reduce_kernel, ceil_div(M, 128), 128, 0, ctx->stream, M, splits, ws.part_d2.p, ws.part_idx.p, d_d2, d_idx);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// closestPointCorrespondence(template, target) of one flavour (ClosestPointRegistrator.scala:74-160).  Both meshes
// are views; for the reversed direction (:34-45) the caller swaps them.  Needs: tpl.aos, (tpl.tri, tpl.normals for
// the mesh flavours); tgt.soa, (tgt.aos, tgt.tri, tgt.normals, tgt.boundary for the mesh flavours).
// Results for the tpl.n template vertices in ws.idx (nearest target vertex) / ws.cp / ws.w / ws.mean_dist.
int32_t icp_correspondence_enqueue(gingr_ctx* ctx, ClosestWorkspace& ws, const MeshView& tpl, const MeshView& tgt,
                                   int method, int q0, int qn) {
  cudaStream_t st = ctx->stream;
  // Query range [q0, q0 + qn) of the template vertices (SURVEY 8e: K2 splits the QUERIES across the GPUs; a rank
  // searches the vertices of its own basis shard, whose observation rows are the only ones it needs -- no gather).
  // All per-query outputs keep their global index; the template MESH (self-intersection test) stays whole.
  if (qn < 0) { q0 = 0; qn = tpl.n; }
  const int M = qn, N = tgt.n;
  if (M == 0) return GINGR_OK;
  const double* q_aos = tpl.aos + (size_t)3 * q0;
  const double* q_nrm = tpl.normals ? tpl.normals + (size_t)3 * q0 : nullptr;
  double* o_d2 = ws.d2.p + q0;
  int32_t* o_idx = ws.idx.p + q0;
  double* o_cp = ws.cp.p + (size_t)3 * q0;
  uint8_t* o_w = ws.w.p + q0;
  uint8_t* o_hit = ws.hit.p + q0;
  // any grid search ahead: sort the queries spatially once (a point grid over the template vertices)
  const SpatialGrid* order = nullptr;
  const bool any_grid = (tgt.pgrid && tgt.pgrid->built) || (tgt.tgrid && tgt.tgrid->built) || (tpl.tgrid && tpl.tgrid->built);
  if (any_grid && ws.qorder && ws.qorder->cap_items >= M) {
    VertexArray qa;
    qa.p = q_aos;
    GINGR_TRY(grid_build_points_enqueue(ctx, *ws.qorder, M, qa));
    order = ws.qorder.get();
  }
  if (method == GINGR_POINTCLOUD_CLOSEST_POINT) {
    GINGR_TRY(nn_vertex_enqueue(ctx, ws, M, q_aos, N, tgt.soa, o_d2, o_idx, tgt.pgrid, order));
    GINGR_LAUNCH(ctx, gather_points_kernel, ceil_div(M, 128), 128, 0, st, M, o_idx, N, tgt.soa, o_cp);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, gingr_fill_bytes(ctx, o_w, 1, (size_t)M, st));
    mean_sqrt_enqueue(ctx, ws, M, 1, o_d2);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    return GINGR_OK;
  }
  if (tgt.T <= 0 || tpl.T <= 0 || !tpl.normals || !tgt.normals || !tgt.boundary || !tgt.aos)
    return gingr_fail(ctx, GINGR_ERR_ARG, "the mesh flavours of the ICP correspondence need template and target triangles");
  // (chains batched in one launch fill the machine by themselves: long candidate ranges prune better, batch.cuh)
  const int s_surf = ctx->rec ? std::min(ws.s_surf, 2) : std::min(ws.s_surf, std::max(1, ceil_div(tgt.T, TT / 4)));
  int s_line = std::min(ws.s_line, std::max(1, ceil_div(tpl.T, TT / 4)));
  const bool tgt_grid = tgt.tgrid && tgt.tgrid->built, tpl_grid = tpl.tgrid && tpl.tgrid->built;
  double* o_sd2 = ws.surf_d2.p + q0;   // not o_d2: the nearest-vertex search below reuses that
  if (method == GINGR_TRIANGULAR_CLOSEST_POINT && tgt_grid) {
    GINGR_TRY(grid_surface_enqueue(ctx, *tgt.tgrid, M, q_aos, tgt.aos, tgt.tri, o_sd2, nullptr, o_cp, order));
    mean_sqrt_enqueue(ctx, ws, M, 1, o_sd2);
  } else if (method == GINGR_ALONG_NORMAL_CLOSEST_POINT && tgt_grid) {
    GINGR_TRY(grid_line_enqueue(ctx, *tgt.tgrid, M, q_aos, q_nrm, tgt.aos, tgt.tri, 0, ws.part_d2.p, ws.part_cp.p,
                                order));
    GINGR_LAUNCH(ctx, line_hit_reduce_kernel, ceil_div(M, 128), 128, 0, st, M, 1, q_aos, ws.part_d2.p, ws.part_cp.p, o_d2, o_cp, o_hit);
    GINGR_LAUNCHED(ctx);
    mean_sqrt_enqueue(ctx, ws, M, 0, o_d2);  // distance += (p - closestPoint).norm (:128)
  } else if (method == GINGR_TRIANGULAR_CLOSEST_POINT) {
    GINGR_LAUNCH(ctx, surface_kernel, dim3(ceil_div(M, QT), s_surf), QT, 0, st, M, q_aos, N, tgt.soa, tgt.T, tgt.tri, ws.part_d2.p,
                                                                 ws.part_idx.p, ws.part_cp.p);
    GINGR_LAUNCHED(ctx);
    GINGR_LAUNCH(ctx, surface_reduce_kernel, ceil_div(M, 128), 128, 0, st, M, s_surf, ws.part_d2.p, ws.part_idx.p, ws.part_cp.p,
                                                            o_sd2, nullptr, o_cp);
    GINGR_LAUNCHED(ctx);
    mean_sqrt_enqueue(ctx, ws, M, 1, o_sd2);
  } else if (method == GINGR_ALONG_NORMAL_CLOSEST_POINT) {
    // nearest intersection of the line (p, n_p) with the target mesh (:105-110)
    const int s_hit = s_surf;
    GINGR_LAUNCH_T(ctx, line_mesh_kernel, (false, false, true), dim3(ceil_div(M, QT), s_hit), QT, 0, st, M, q_aos, q_nrm, tgt.aos,
                   tgt.T, tgt.tri, ws.part_d2.p, ws.part_cp.p, 0);
    GINGR_LAUNCHED(ctx);
    GINGR_LAUNCH(ctx, line_hit_reduce_kernel, ceil_div(M, 128), 128, 0, st, M, s_hit, q_aos, ws.part_d2.p, ws.part_cp.p, o_d2, o_cp, o_hit);
    GINGR_LAUNCHED(ctx);
    mean_sqrt_enqueue(ctx, ws, M, 0, o_d2);  // distance += (p - closestPoint).norm (:128)
  } else {
    return gingr_fail(ctx, GINGR_ERR_ARG, "unknown ICP correspondence method");
  }
  // nearest target vertex of the corresponding point (:83 / :113); d2 of that search is not needed afterwards
  GINGR_TRY(nn_vertex_enqueue(ctx, ws, M, o_cp, N, tgt.soa, o_d2, o_idx, tgt.pgrid, order));
  // isClosestPointIntersecting on the template itself (:62-72): the lines of the query range against the WHOLE template
  if (tpl_grid) {
    GINGR_TRY(grid_line_enqueue(ctx, *tpl.tgrid, M, q_aos, o_cp, tpl.aos, tpl.tri, 1, ws.part_d2.p, nullptr, order, q0));
    s_line = 1;
  } else {
    GINGR_LAUNCH_T(ctx, line_mesh_kernel, (true, true, false), dim3(ceil_div(M, QT), s_line), QT, 0, st, M, q_aos, o_cp, tpl.aos,
                   tpl.T, tpl.tri, ws.part_d2.p, nullptr, q0);
    GINGR_LAUNCHED(ctx);
  }
  GINGR_LAUNCH(ctx, icp_weights_kernel, ceil_div(M, 128), 128, 0, st, M, q_aos, o_cp, o_idx, tgt.boundary, q_nrm, tgt.normals, s_line,
                                                       ws.part_d2.p,
                                                       method == GINGR_ALONG_NORMAL_CLOSEST_POINT ? o_hit : nullptr, o_w);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// Squared distance of nq arbitrary points (AoS) to the surface of a mesh: closestPointOnSurface(pt) of
// sampling/evaluators/IndependentPointDistanceEvaluator.scala:54-66, with the same kernels (and the same grid when the
// mesh view carries one) as the TriangularClosestPoint correspondence.  Result in ws.d2 [nq]; ws.cp holds the points.
int32_t surface_distance_enqueue(gingr_ctx* ctx, ClosestWorkspace& ws, int nq, const double* d_q, const MeshView& mesh) {
  cudaStream_t st = ctx->stream;
  if (mesh.T <= 0 || !mesh.tri || !mesh.soa || !mesh.aos)
    return gingr_fail(ctx, GINGR_ERR_ARG, "surface distance needs a triangle mesh (vertices AoS + SoA, triangles)");
  if (mesh.tgrid && mesh.tgrid->built) {
    GINGR_TRY(grid_surface_enqueue(ctx, *mesh.tgrid, nq, d_q, mesh.aos, mesh.tri, ws.d2.p, nullptr, ws.cp.p, nullptr));
    return GINGR_OK;
  }
  const int s_surf = ctx->rec ? std::min(ws.s_surf, 2) : std::min(ws.s_surf, std::max(1, ceil_div(mesh.T, TT / 4)));
  GINGR_LAUNCH(ctx, surface_kernel, dim3(ceil_div(nq, QT), s_surf), QT, 0, st, nq, d_q, mesh.n, mesh.soa, mesh.T, mesh.tri, ws.part_d2.p,
                                                                ws.part_idx.p, ws.part_cp.p);
  GINGR_LAUNCHED(ctx);
  GINGR_LAUNCH(ctx, surface_reduce_kernel, ceil_div(nq, 128), 128, 0, st, nq, s_surf, ws.part_d2.p, ws.part_idx.p, ws.part_cp.p, ws.d2.p,
                                                           nullptr, ws.cp.p);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// closestPointCorrespondenceReversal (:34-45), second half: the observations (templateId_j, target point x_j, w_j)
// of all target vertices j, folded per template vertex i in ascending j (deterministic, no atomics):
//   wcnt_i = #{j : tid_j = i, w_j = 1},  cp_i = mean of those x_j   (wcnt_i / sigma2 and the mean reproduce the
//   summed duplicate observations of the reference's regression exactly up to rounding)
__global__ void __launch_bounds__(128) reverse_fold_kernel(int M, int N, const int32_t* __restrict__ tid,
                                                           const uint8_t* __restrict__ w,
                                                           const double* __restrict__ x /*AoS target points*/,
                                                           double* __restrict__ cp, double* __restrict__ wcnt) {
  __shared__ int32_t s_tid[512];
  const int i = blockIdx.x * 128 + threadIdx.x;
  double sx = 0.0, sy = 0.0, sz = 0.0;
  int cnt = 0;
  for (int j0 = 0; j0 < N; j0 += 512) {
    const int c = min(512, N - j0);
    __syncthreads();
    for (int t = threadIdx.x; t < c; t += 128) s_tid[t] = w[j0 + t] ? tid[j0 + t] : -1;
    __syncthreads();
    for (int t = 0; t < c; ++t)
      if (s_tid[t] == i) {
        sx += x[3 * (j0 + t)]; sy += x[3 * (j0 + t) + 1]; sz += x[3 * (j0 + t) + 2];
        ++cnt;
      }
  }
  if (i < M) {
    wcnt[i] = (double)cnt;
    const double inv = cnt > 0 ? 1.0 / (double)cnt : 0.0;
    cp[3 * i] = sx * inv; cp[3 * i + 1] = sy * inv; cp[3 * i + 2] = sz * inv;
  }
}

// ---- the same fold in O(N + M) for large problems: lists of the target vertices per template vertex (integer atomics, then
// each list sorted ascending), summed in ascending j -- the order of the scan above, so the result is bit-identical
__global__ void rfold_count_kernel(int N, int M, const int32_t* __restrict__ tid, const uint8_t* __restrict__ w,
                                   int32_t* __restrict__ cnt) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < N && w[j] && tid[j] >= 0 && tid[j] < M) atomicAdd(&cnt[tid[j]], 1);
}

// exclusive scan of cnt[0..M) into start[0..M] by one CTA (M up to a few million: each thread owns a contiguous chunk)
__global__ void __launch_bounds__(1024) rfold_scan_kernel(int M, const int32_t* __restrict__ cnt, int32_t* __restrict__ start,
                                                          int32_t* __restrict__ fill) {
  __shared__ int sh[1024];
  const int per = (M + 1023) / 1024;
  const int b0 = threadIdx.x * per, b1 = min(M, b0 + per);
  int s = 0;
  for (int i = b0; i < b1; ++i) s += cnt[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int v = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
    __syncthreads();
    sh[threadIdx.x] += v;
    __syncthreads();
  }
  int run = sh[threadIdx.x] - s;
  for (int i = b0; i < b1; ++i) {
    start[i] = run;
    fill[i] = 0;
    run += cnt[i];
  }
  if (threadIdx.x == 1023) start[M] = sh[1023];
}

__global__ void rfold_scatter_kernel(int N, int M, const int32_t* __restrict__ tid, const uint8_t* __restrict__ w,
                                     const int32_t* __restrict__ start, int32_t* __restrict__ fill, int32_t* __restrict__ list) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < N && w[j] && tid[j] >= 0 && tid[j] < M) list[start[tid[j]] + atomicAdd(&fill[tid[j]], 1)] = j;
}

__global__ void rfold_sum_kernel(int M, const int32_t* __restrict__ start, int32_t* __restrict__ list,
                                 const double* __restrict__ x /*AoS target points*/, double* __restrict__ cp,
                                 double* __restrict__ wcnt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const int b = start[i], e = start[i + 1];
  for (int a = b + 1; a < e; ++a) {   // insertion sort: the lists are short (N / M on average)
    const int v = list[a];
    int k = a - 1;
    while (k >= b && list[k] > v) { list[k + 1] = list[k]; --k; }
    list[k + 1] = v;
  }
  double sx = 0.0, sy = 0.0, sz = 0.0;
  for (int a = b; a < e; ++a) {
    const int j = list[a];
    sx += x[3 * j]; sy += x[3 * j + 1]; sz += x[3 * j + 2];
  }
  const int cnt = e - b;
  wcnt[i] = (double)cnt;
  const double inv = cnt > 0 ? 1.0 / (double)cnt : 0.0;
  cp[3 * i] = sx * inv; cp[3 * i + 1] = sy * inv; cp[3 * i + 2] = sz * inv;
}

int32_t reverse_fold_enqueue(gingr_ctx* ctx, int M, int N, const int32_t* d_tid, const uint8_t* d_w,
                             const double* d_target_aos, double* d_cp, double* d_wcnt, int32_t* d_scratch) {
  cudaStream_t st = ctx->stream;
  const char* env = getenv("GINGR_RFOLD_LIST");   // 0 / 1: force the scan / the list form (tests); default: by size
  const int forced = (env && *env) ? atoi(env) : -1;
  const bool lists = forced >= 0 ? forced != 0 : (long long)M * (long long)N > (1LL << 24);
  if (d_scratch && lists) {
    // scratch: cnt [M], start [M + 1], fill [M], list [N]
    int32_t* cnt = d_scratch;
    int32_t* start = cnt + M;
    int32_t* fill = start + M + 1;
    int32_t* list = fill + M;
    GINGR_CUDA_TRY(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (size_t)M, st));
    rfold_count_kernel<<<ceil_div(N, 256), 256, 0, st>>>(N, M, d_tid, d_w, cnt);
    rfold_scan_kernel<<<1, 1024, 0, st>>>(M, cnt, start, fill);
    rfold_scatter_kernel<<<ceil_div(N, 256), 256, 0, st>>>(N, M, d_tid, d_w, start, fill, list);
    rfold_sum_kernel<<<ceil_div(M, 128), 128, 0, st>>>(M, start, list, d_target_aos, d_cp, d_wcnt);
    ctx->launches += 4;
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    return GINGR_OK;
  }
  reverse_fold_kernel<<<ceil_div(M, 128), 128, 0, st>>>(M, N, d_tid, d_w, d_target_aos, d_cp, d_wcnt);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

}  // namespace gingr
