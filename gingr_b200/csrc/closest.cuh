// closest.cuh -- host-side interface of the K2 closest-point kernels (closest.cu).
#pragma once
#include <memory>
#include <vector>

#include "common.cuh"

namespace gingr {

struct SpatialGrid;  // grid.cuh

// A mesh as the correspondence kernels see it: device pointers, any of which may be null when the flavour does
// not need it.  "template" = the mesh whose vertices are the queries, "target" = the mesh that is searched.
struct MeshView {
  int n = 0;                          // vertices
  const double* aos = nullptr;        // [n][3]
  const double* soa = nullptr;        // [3][n]
  int T = 0;                          // triangles
  const int32_t* tri = nullptr;       // [3T]
  const double* normals = nullptr;    // [n][3] vertex normals of THIS geometry
  const uint8_t* boundary = nullptr;  // [n] pointIsOnBoundary
  // optional uniform grids over THIS geometry (built by the owner, grid.cuh): when present the searches that scan
  // this mesh run on the grid instead of the brute-force scan, with bit-identical results
  const SpatialGrid* pgrid = nullptr;  // over the vertices
  const SpatialGrid* tgrid = nullptr;  // over the triangles (needs aos)
};

struct ClosestWorkspace {
  int s_nn = 1, s_surf = 1, s_line = 1;  // candidate-range splits of the three scans
  DevBuf<double> part_d2;     // [smax][nq]
  DevBuf<int32_t> part_idx;   // [smax][nq]
  DevBuf<double> part_cp;     // [max(s_surf, s_line)][nq][3]
  DevBuf<double> d2;          // [nq]
  DevBuf<double> surf_d2;     // [nq]   triangular flavour: squared distance to the target surface, kept after the search
                              //        (the point-distance evaluator of an MH step asks for exactly these, mcmc.cuh)
  DevBuf<int32_t> idx;        // [nq]   nearest target vertex
  DevBuf<double> cp;          // [nq][3] corresponding point
  DevBuf<uint8_t> w;          // [nq]   0/1 weight
  DevBuf<uint8_t> hit;        // [nq]   along-normal: the line met the target
  DevBuf<double> mean_dist;   // [1]
  DevBuf<double> mean_part;   // [64] per-block partial sums of the mean distance
  std::unique_ptr<SpatialGrid> qorder;  // point grid over the queries = their spatial sort (grid searches only)
  // nq queries against a mesh of n_search vertices / T_search triangles; T_query_mesh triangles of the query mesh
  int32_t ensure(gingr_ctx* ctx, int nq, int n_search, int T_search, int T_query_mesh);
};

void build_vertex_adjacency(int n, int T, const int32_t* tri, std::vector<int32_t>* off, std::vector<int32_t>* adj);
void compute_boundary_flags(int n, int T, const int32_t* tri, std::vector<uint8_t>* flags);
int32_t mesh_static_upload(gingr_ctx* ctx, int n, const double* verts_aos_host, int T, const int32_t* tri_host,
                           DevBuf<double>* normals, DevBuf<uint8_t>* boundary);
int32_t vertex_normals_enqueue(gingr_ctx* ctx, int n, const double* d_verts_aos, const int32_t* d_tri,
                               const int32_t* d_adj_off, const int32_t* d_adj, double* d_normals);
int32_t nn_vertex_enqueue(gingr_ctx* ctx, ClosestWorkspace& ws, int M, const double* d_q, int N,
                          const double* d_pts_soa, double* d_d2, int32_t* d_idx, const SpatialGrid* pgrid = nullptr,
                          const SpatialGrid* order = nullptr);
// q0 / qn: query range [q0, q0 + qn) of the template vertices (qn < 0: all).  Per-query outputs keep their global index.
int32_t icp_correspondence_enqueue(gingr_ctx* ctx, ClosestWorkspace& ws, const MeshView& tpl, const MeshView& tgt,
                                   int method, int q0 = 0, int qn = -1);
int32_t surface_distance_enqueue(gingr_ctx* ctx, ClosestWorkspace& ws, int nq, const double* d_q, const MeshView& mesh);
// d_scratch (optional): 3 M + N + 1 ints; with it, large problems (M N > 2^24) take the O(N + M) list form (same result)
int32_t reverse_fold_enqueue(gingr_ctx* ctx, int M, int N, const int32_t* d_tid, const uint8_t* d_w,
                             const double* d_target_aos, double* d_cp, double* d_wcnt, int32_t* d_scratch = nullptr);

}  // namespace gingr
