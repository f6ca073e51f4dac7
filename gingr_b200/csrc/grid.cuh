// grid.cuh -- uniform-grid acceleration of the K2 closest-point searches (grid.cu).
//
// The brute-force scans of closest.cu cost O(M N); at the sizes where K2 has a roofline at all (M, N >= 1e5,
// SURVEY.md 8d) a uniform grid over the searched geometry brings that to O(M * neighbourhood).  The grid only
// selects candidates: every candidate is evaluated with the shared arithmetic of closest_geom.cuh and winners are
// chosen by (value, lowest index), so results are bit-identical to the scans (tests/test_grid_gpu.py).
// Grids are built ON THE DEVICE with device-resident parameters (no host round trip), so the per-iteration rebuild
// over the moving fit is part of the captured iteration graph.
#pragma once
#include "common.cuh"

namespace gingr {

struct GridParams {     // lives in device memory
  double ox, oy, oz;    // origin = bounding-box minimum - margin
  double h, inv_h;      // cell edge
  double margin;        // safety margin of every conservative bound (1e-6 h)
  int nx, ny, nz;       // occupied cells per axis
  int bx2, by2;         // 16-cell blocks per axis (x, y): cells are numbered in nested 4x4x4 blocks, see cell_index
  int ncells;           // padded cell count (multiple of 4096)
  int overflow;         // triangle grid: entry capacity exceeded / oversized triangle -> queries scan everything
  int total;            // number of entries
};

struct SpatialGrid {
  int n_items = 0;      // points or triangles entered by the last build
  int cap_items = 0;    // what the buffers are sized for
  bool triangles = false;
  int cap_cells = 0, cap_entries = 0;
  DevBuf<GridParams> params;   // [1]
  DevBuf<int32_t> cell_start;  // [cap_cells + 1] exclusive prefix of the per-cell counts
  DevBuf<int32_t> fill;        // [cap_cells + 1] counts, then the scatter cursor
  DevBuf<int32_t> entries;     // triangle grid: [cap_entries] triangle ids, cell-major
  DevBuf<float4> tri_box;      // triangle grid: [T][2] bounding box of each triangle, rounded outward to float
  DevBuf<float4> entry_box;    // optional (entry_boxes, static grids): [cap_entries][2] the same box stored WITH each entry, so that
                               // the surface search streams boxes cell by cell instead of gathering them through the triangle id
  bool entry_boxes = false;    // set before ensure()
  DevBuf<double4> pts;         // point grid: [n] (x, y, z, original index as bits), cell-major
  DevBuf<double> bbox_part;    // [128][6]
  DevBuf<int32_t> block_sums;  // scan scratch
  bool built = false;
  int32_t ensure(gingr_ctx* ctx, int n_vertices, int n_items, bool triangles);
};

// point i, coordinate d of a vertex array = p[i * stride_pt + d * stride_dim]  (AoS: 3, 1;  SoA: 1, n)
struct VertexArray {
  const double* p = nullptr;
  int64_t stride_pt = 3, stride_dim = 1;
};

// Below these sizes of the searched geometry the brute-force scans are launch-bound and win; above, the grid.
// GINGR_K2_GRID=0 / 1 in the environment forces one or the other (tests).
bool grid_wanted(int n_search);

int32_t grid_build_points_enqueue(gingr_ctx* ctx, SpatialGrid& g, int n, VertexArray v);
int32_t grid_build_triangles_enqueue(gingr_ctx* ctx, SpatialGrid& g, int n, VertexArray v, int T, const int32_t* d_tri);

// nearest grid point of M queries (AoS): the grid twin of nn_vertex_kernel + nn_reduce_kernel
// `order` (all three): optional point grid built over (points near) the M queries; its cell-sorted point array is used
// as a spatial permutation so that the threads of a warp walk neighbouring cells
int32_t grid_nn_enqueue(gingr_ctx* ctx, const SpatialGrid& g, int M, const double* d_q, double* d_d2, int32_t* d_idx,
                        const SpatialGrid* order = nullptr);
// closest point on the gridded triangle mesh: twin of surface_kernel + surface_reduce_kernel
int32_t grid_surface_enqueue(gingr_ctx* ctx, const SpatialGrid& g, int M, const double* d_q, const double* d_verts_aos,
                             const int32_t* d_tri, double* d_d2, int32_t* d_tri_out, double* d_cp,
                             const SpatialGrid* order = nullptr);
// nearest intersection of the line o + s d with the gridded mesh: twin of line_mesh_kernel
//   self != 0: mesh is the query mesh itself, triangles incident to vertex i skipped, d = o - other, only hits
//              nearer than |d| can matter (isClosestPointIntersecting) -> bounded march, min distance only
//   self == 0: d = other (the vertex normal), unbounded march in both directions, hit point returned
int32_t grid_line_enqueue(gingr_ctx* ctx, const SpatialGrid& g, int M, const double* d_o, const double* d_other,
                          const double* d_mesh_aos, const int32_t* d_tri, int self, double* d_min, double* d_pt,
                          const SpatialGrid* order = nullptr, int q0 = 0 /*self: vertex id of query 0*/);

}  // namespace gingr
