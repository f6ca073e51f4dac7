// grid.cu -- uniform-grid twins of the K2 scans (closest.cu).   COMPILED WITH -fmad=false, like closest.cu.
//
// Replaces, at sizes where a scan is too slow, the spatial queries scalismo answers with a KD-tree / bounding-sphere
// tree behind registration/utils/ClosestPointRegistrator.scala: findClosestPoint (:83, :113, :143),
// closestPointOnSurface (:80), getIntersectionPoints (:65, :107).  See grid.cuh for the exactness argument.
//
// Build (all on the device, parameters stay in device memory so the rebuild over the moving fit can be captured in
// the iteration graph): bounding box -> cell edge h = 2 * diagonal / sqrt(n) (about 4 points per occupied cell for a
// surface sampling) -> per-cell counts (integer atomics; the order inside a cell is irrelevant because winners are
// chosen by (value, index)) -> exclusive scan -> scatter.  Triangles are entered in every cell their bounding box
// overlaps.
// Queries: one thread per query, expanding Chebyshev shells of cells around the query's cell until the best value is
// strictly below the distance to the unvisited region (minus a safety margin); lines march slab by slab along their
// major axis.
// Cells are numbered in nested 4x4x4 blocks (two levels: 64 and 4096 fine cells), so the entries of a coarse cell of
// edge 4h or 16h are ONE contiguous range of the same arrays: a query that is far from the surface (the normal case in
// the first ICP iterations) climbs to the coarser levels instead of walking thousands of empty fine cells.  A query
// that has not terminated after the last level's shells scans all items (bounded cost for outliers).
#include <algorithm>
#include <cstdlib>

#include "closest_geom.cuh"
#include "grid.cuh"

namespace gingr {

#ifdef GINGR_GRID_STATS
// tuning build only (tools/build_variant.sh stats grid.cu -DGINGR_GRID_STATS): event counters of the searches
__device__ unsigned long long grid_stats[24];   // 0-7 thread-per-query searches, 8-23 the warp-per-query surface search
#define GSTAT(k, n) atomicAdd(&grid_stats[k], (unsigned long long)(n))
#define GSTATW(k, n) do { if ((threadIdx.x & 31) == 0) atomicAdd(&grid_stats[8 + (k)], (unsigned long long)(n)); } while (0)
#else
#define GSTAT(k, n) ((void)0)
#define GSTATW(k, n) ((void)0)
#endif

constexpr int BB_BLOCKS = 128;
constexpr int SCAN_ITEMS = 4096;   // per block: 256 threads x 16
constexpr int LEVELS = 3;          // cell edges h, 4h, 16h
__constant__ int K_LEVEL[LEVELS] = {2, 2, 4};  // shells searched per level before climbing / falling back to the full scan
constexpr int MAX_TRI_CELLS = 512; // a triangle overlapping more cells than this marks the grid as overflowed

// ---------------------------------------------------------------------------------------------
// build
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grid_bbox_kernel(int n, VertexArray v, double* __restrict__ part /*[BB_BLOCKS][6]*/) {
  __shared__ double red[6][256];
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256)
    for (int d = 0; d < 3; ++d) {
      const double x = v.p[i * v.stride_pt + d * v.stride_dim];
      lo[d] = fmin(lo[d], x);
      hi[d] = fmax(hi[d], x);
    }
  for (int d = 0; d < 3; ++d) { red[d][threadIdx.x] = lo[d]; red[3 + d][threadIdx.x] = hi[d]; }
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o)
      for (int d = 0; d < 3; ++d) {
        red[d][threadIdx.x] = fmin(red[d][threadIdx.x], red[d][threadIdx.x + o]);
        red[3 + d][threadIdx.x] = fmax(red[3 + d][threadIdx.x], red[3 + d][threadIdx.x + o]);
      }
    __syncthreads();
  }
  if (threadIdx.x < 6) part[blockIdx.x * 6 + threadIdx.x] = red[threadIdx.x][0];
}

__global__ void grid_params_kernel(int n, int cap_cells, const double* __restrict__ part, GridParams* __restrict__ gp,
                                   double cell_scale /*cell edge = cell_scale * diagonal / sqrt(n)*/) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int b = 0; b < BB_BLOCKS; ++b)
    for (int d = 0; d < 3; ++d) {
      lo[d] = fmin(lo[d], part[b * 6 + d]);
      hi[d] = fmax(hi[d], part[b * 6 + 3 + d]);
    }
  GridParams g;
  double ext[3];
  bool ok = true;
  for (int d = 0; d < 3; ++d) {
    ext[d] = hi[d] - lo[d];
    ok = ok && isfinite(lo[d]) && isfinite(hi[d]);
  }
  const double diag = ok ? sqrt(ext[0] * ext[0] + ext[1] * ext[1] + ext[2] * ext[2]) : 0.0;
  if (!ok || !(diag > 0.0) || !isfinite(diag)) {
    // degenerate (one point, non-finite coordinates): a single cell holding everything
    g.ox = g.oy = g.oz = 0.0;
    g.h = 1.0; g.inv_h = 1.0; g.margin = 0.0;
    g.nx = g.ny = g.nz = 1;
  } else {
    double h = cell_scale * diag / sqrt((double)(n > 0 ? n : 1));
    int nx, ny, nz;
    for (;;) {
      const double m = 1e-6 * h;
      nx = (int)fmin(floor((ext[0] + 2.0 * m) / h) + 1.0, 1023.0);
      ny = (int)fmin(floor((ext[1] + 2.0 * m) / h) + 1.0, 1023.0);
      nz = (int)fmin(floor((ext[2] + 2.0 * m) / h) + 1.0, 1023.0);
      const double padded = (double)((nx + 15) & ~15) * (double)((ny + 15) & ~15) * (double)((nz + 15) & ~15);
      if (padded <= (double)cap_cells &&
          (double)nx * h >= ext[0] + 2.0 * m && (double)ny * h >= ext[1] + 2.0 * m && (double)nz * h >= ext[2] + 2.0 * m)
        break;
      h *= 1.25;
    }
    g.h = h; g.inv_h = 1.0 / h; g.margin = 1e-6 * h;
    g.ox = lo[0] - g.margin; g.oy = lo[1] - g.margin; g.oz = lo[2] - g.margin;
    g.nx = nx; g.ny = ny; g.nz = nz;
  }
  g.bx2 = (g.nx + 15) >> 4; g.by2 = (g.ny + 15) >> 4;
  g.ncells = g.bx2 * g.by2 * ((g.nz + 15) >> 4) * 4096;
  g.overflow = 0;
  g.total = 0;
  *gp = g;
}

__device__ __forceinline__ int cell_coord(double x, double o, double inv_h, int n) {
  const int c = __double2int_rd((x - o) * inv_h);   // saturating; NaN -> 0
  return min(max(c, 0), n - 1);
}
// nested 4x4x4 blocking: [16-blocks row-major][4-block within the 16-block][cell within the 4-block]
__device__ __forceinline__ int cell_index(const GridParams& g, int x, int y, int z) {
  const int b2 = ((z >> 4) * g.by2 + (y >> 4)) * g.bx2 + (x >> 4);
  return (b2 << 12) | (((z >> 2) & 3) << 10) | (((y >> 2) & 3) << 8) | (((x >> 2) & 3) << 6) | ((z & 3) << 4) |
         ((y & 3) << 2) | (x & 3);
}
__device__ __forceinline__ int cell_coord_raw(double x, double o, double inv_h) { return __double2int_rd((x - o) * inv_h); }

__global__ void __launch_bounds__(256) grid_point_count_kernel(int n, VertexArray v, const GridParams* __restrict__ gp,
                                                               int32_t* __restrict__ fill) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const GridParams g = *gp;
  const int cx = cell_coord(v.p[i * v.stride_pt], g.ox, g.inv_h, g.nx);
  const int cy = cell_coord(v.p[i * v.stride_pt + v.stride_dim], g.oy, g.inv_h, g.ny);
  const int cz = cell_coord(v.p[i * v.stride_pt + 2 * v.stride_dim], g.oz, g.inv_h, g.nz);
  atomicAdd(&fill[cell_index(g, cx, cy, cz)], 1);
}

__global__ void __launch_bounds__(256) grid_point_scatter_kernel(int n, VertexArray v, const GridParams* __restrict__ gp,
                                                                 const int32_t* __restrict__ cell_start,
                                                                 int32_t* __restrict__ fill, double4* __restrict__ pts) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const GridParams g = *gp;
  const double x = v.p[i * v.stride_pt], y = v.p[i * v.stride_pt + v.stride_dim], z = v.p[i * v.stride_pt + 2 * v.stride_dim];
  const int c = cell_index(g, cell_coord(x, g.ox, g.inv_h, g.nx), cell_coord(y, g.oy, g.inv_h, g.ny),
                           cell_coord(z, g.oz, g.inv_h, g.nz));
  const int pos = cell_start[c] + atomicAdd(&fill[c], 1);
  pts[pos] = make_double4(x, y, z, __longlong_as_double((long long)i));
}

struct TriCells {
  int x0, x1, y0, y1, z0, z1;
  bool too_big;
};

// bounding box of a triangle rounded OUTWARD to float: the 32-byte record the surface search rejects and
// de-duplicates candidates with, and -- so that both agree exactly -- also what the cell ranges are derived from
__device__ __forceinline__ void triangle_float_box(const double* __restrict__ va, int a, int b, int c, float4& lo, float4& hi) {
  const double* pa = va + 3 * (size_t)a; const double* pb = va + 3 * (size_t)b; const double* pc = va + 3 * (size_t)c;
  lo = make_float4(__double2float_rd(fmin(pa[0], fmin(pb[0], pc[0]))), __double2float_rd(fmin(pa[1], fmin(pb[1], pc[1]))),
                   __double2float_rd(fmin(pa[2], fmin(pb[2], pc[2]))), 0.f);
  hi = make_float4(__double2float_ru(fmax(pa[0], fmax(pb[0], pc[0]))), __double2float_ru(fmax(pa[1], fmax(pb[1], pc[1]))),
                   __double2float_ru(fmax(pa[2], fmax(pb[2], pc[2]))), 0.f);
}

__device__ __forceinline__ TriCells triangle_cells(const GridParams& g, const float4& lo, const float4& hi) {
  TriCells r;
  const double m = g.margin;
  r.x0 = cell_coord((double)lo.x - m, g.ox, g.inv_h, g.nx);
  r.x1 = cell_coord((double)hi.x + m, g.ox, g.inv_h, g.nx);
  r.y0 = cell_coord((double)lo.y - m, g.oy, g.inv_h, g.ny);
  r.y1 = cell_coord((double)hi.y + m, g.oy, g.inv_h, g.ny);
  r.z0 = cell_coord((double)lo.z - m, g.oz, g.inv_h, g.nz);
  r.z1 = cell_coord((double)hi.z + m, g.oz, g.inv_h, g.nz);
  r.too_big = (long long)(r.x1 - r.x0 + 1) * (r.y1 - r.y0 + 1) * (r.z1 - r.z0 + 1) > MAX_TRI_CELLS;
  return r;
}

// PASS 0: count, PASS 1: scatter
template <int PASS>
__global__ void __launch_bounds__(256) grid_tri_kernel(int T, const double* __restrict__ verts_aos, const int32_t* __restrict__ tri,
                                                       GridParams* __restrict__ gp, const int32_t* __restrict__ cell_start,
                                                       int32_t* __restrict__ fill, int32_t* __restrict__ entries, int cap_entries,
                                                       float4* __restrict__ tri_box, float4* __restrict__ entry_box /*may be null*/) {
  const int t = blockIdx.x * 256 + threadIdx.x;
  if (t >= T) return;
  const GridParams g = *gp;
  float4 blo, bhi;
  triangle_float_box(verts_aos, tri[3 * t], tri[3 * t + 1], tri[3 * t + 2], blo, bhi);
  if (PASS == 0) { tri_box[2 * t] = blo; tri_box[2 * t + 1] = bhi; }
  if (PASS == 1 && g.overflow) return;
  const TriCells r = triangle_cells(g, blo, bhi);
  if (r.too_big) {
    if (PASS == 0) atomicExch(&gp->overflow, 1);
    return;
  }
  for (int z = r.z0; z <= r.z1; ++z)
    for (int y = r.y0; y <= r.y1; ++y)
      for (int x = r.x0; x <= r.x1; ++x) {
        const int c = cell_index(g, x, y, z);
        if (PASS == 0) {
          atomicAdd(&fill[c], 1);
        } else {
          const int pos = cell_start[c] + atomicAdd(&fill[c], 1);
          if (pos < cap_entries) {
            entries[pos] = t;
            if (entry_box) { entry_box[2 * (size_t)pos] = blo; entry_box[2 * (size_t)pos + 1] = bhi; }
          }
        }
      }
}

// exclusive scan of fill[0 .. ncells] into cell_start, three kernels; blocks beyond ncells exit at once
__global__ void __launch_bounds__(256) grid_scan_sums_kernel(const GridParams* __restrict__ gp, const int32_t* __restrict__ in,
                                                             int32_t* __restrict__ block_sums) {
  const int n = gp->ncells + 1;
  const int base = blockIdx.x * SCAN_ITEMS;
  __shared__ int red[256];
  int s = 0;
  if (base < n)
    for (int k = threadIdx.x; k < SCAN_ITEMS; k += 256)
      if (base + k < n - 1) s += in[base + k];   // element ncells itself counts as 0 (it is only a sentinel)
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) block_sums[blockIdx.x] = red[0];
}

__global__ void __launch_bounds__(1024) grid_scan_blocks_kernel(int nblocks, int32_t* __restrict__ block_sums,
                                                                GridParams* __restrict__ gp, int cap_entries) {
  // one block: exclusive scan of up to 1024 * per block sums
  __shared__ int sh[1024];
  const int per = (nblocks + 1023) / 1024;
  const int b0 = threadIdx.x * per;
  int s = 0;
  for (int k = 0; k < per; ++k)
    if (b0 + k < nblocks) s += block_sums[b0 + k];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int v = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
    __syncthreads();
    sh[threadIdx.x] += v;
    __syncthreads();
  }
  int run = sh[threadIdx.x] - s;
  for (int k = 0; k < per; ++k)
    if (b0 + k < nblocks) {
      const int v = block_sums[b0 + k];
      block_sums[b0 + k] = run;
      run += v;
    }
  if (threadIdx.x == 1023) {
    gp->total = sh[1023];
    if (cap_entries > 0 && sh[1023] > cap_entries) gp->overflow = 1;
  }
}

__global__ void __launch_bounds__(256) grid_scan_write_kernel(const GridParams* __restrict__ gp, int32_t* __restrict__ fill,
                                                              const int32_t* __restrict__ block_sums,
                                                              int32_t* __restrict__ cell_start) {
  const int n = gp->ncells + 1;
  const int base = blockIdx.x * SCAN_ITEMS;
  if (base >= n) return;
  __shared__ int sh[256];
  // thread t owns the 16 consecutive items base + 16 t ...
  int v[16];
  int s = 0;
  const int i0 = base + threadIdx.x * 16;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    v[k] = (i0 + k < n - 1) ? fill[i0 + k] : 0;
    s += v[k];
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const int x = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
    __syncthreads();
    sh[threadIdx.x] += x;
    __syncthreads();
  }
  int run = block_sums[blockIdx.x] + sh[threadIdx.x] - s;
#pragma unroll
  for (int k = 0; k < 16; ++k)
    if (i0 + k < n) {
      cell_start[i0 + k] = run;
      fill[i0 + k] = 0;   // becomes the scatter cursor
      run += v[k];
    }
}

int32_t SpatialGrid::ensure(gingr_ctx* ctx, int nv, int items, bool tri) {
  cap_items = items;
  triangles = tri;
  const long long want = std::max(4096LL, 16LL * (long long)nv);
  cap_cells = (int)std::min(want, 1LL << 24);
  cap_entries = tri ? (int)std::min(16LL * (long long)items + 1024, (1LL << 30)) : 0;
  GINGR_CUDA_TRY(ctx, params.alloc(1));
  GINGR_CUDA_TRY(ctx, cell_start.alloc((size_t)cap_cells + 1));
  GINGR_CUDA_TRY(ctx, fill.alloc((size_t)cap_cells + 1));
  GINGR_CUDA_TRY(ctx, bbox_part.alloc((size_t)BB_BLOCKS * 6));
  GINGR_CUDA_TRY(ctx, block_sums.alloc((size_t)ceil_div(cap_cells + 1, SCAN_ITEMS)));
  if (tri) {
    GINGR_CUDA_TRY(ctx, entries.alloc((size_t)cap_entries));
    GINGR_CUDA_TRY(ctx, tri_box.alloc((size_t)2 * std::max(items, 1)));
    if (entry_boxes) GINGR_CUDA_TRY(ctx, entry_box.alloc((size_t)2 * cap_entries));
  } else {
    GINGR_CUDA_TRY(ctx, pts.alloc((size_t)std::max(items, 1)));
  }
  return GINGR_OK;
}

bool grid_wanted(int n_search) {
  // read on every call (not cached) so that a test process can run both paths on the same inputs
  const char* e = getenv("GINGR_K2_GRID");
  const int forced = (e && *e) ? atoi(e) : -1;
  if (forced == 0) return false;
  if (forced == 1) return true;
  return n_search >= 8192;
}

static int32_t grid_common_head(gingr_ctx* ctx, SpatialGrid& g, int n, VertexArray v) {
  cudaStream_t st = ctx->stream;
  grid_bbox_kernel<<<BB_BLOCKS, 256, 0, st>>>(n, v, g.bbox_part.p);
  GINGR_LAUNCHED(ctx);
  static const double cell_scale = [] { const char* e = getenv("GINGR_K2_CELL_SCALE"); return e && atof(e) > 0.0 ? atof(e) : 2.0; }();
  grid_params_kernel<<<1, 32, 0, st>>>(n, g.cap_cells, g.bbox_part.p, g.params.p, cell_scale);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaMemsetAsync(g.fill.p, 0, sizeof(int32_t) * ((size_t)g.cap_cells + 1), st));
  return GINGR_OK;
}

static int32_t grid_scan(gingr_ctx* ctx, SpatialGrid& g) {
  cudaStream_t st = ctx->stream;
  const int nb = ceil_div(g.cap_cells + 1, SCAN_ITEMS);
  grid_scan_sums_kernel<<<nb, 256, 0, st>>>(g.params.p, g.fill.p, g.block_sums.p);
  GINGR_LAUNCHED(ctx);
  grid_scan_blocks_kernel<<<1, 1024, 0, st>>>(nb, g.block_sums.p, g.params.p, g.cap_entries);
  GINGR_LAUNCHED(ctx);
  grid_scan_write_kernel<<<nb, 256, 0, st>>>(g.params.p, g.fill.p, g.block_sums.p, g.cell_start.p);
  GINGR_LAUNCHED(ctx);
  return GINGR_OK;
}

int32_t grid_build_points_enqueue(gingr_ctx* ctx, SpatialGrid& g, int n, VertexArray v) {
  if (g.triangles || n > g.cap_items) return gingr_fail(ctx, GINGR_ERR_ARG, "grid_build_points: grid not sized for this point set");
  cudaStream_t st = ctx->stream;
  GINGR_TRY(grid_common_head(ctx, g, n, v));
  grid_point_count_kernel<<<ceil_div(n, 256), 256, 0, st>>>(n, v, g.params.p, g.fill.p);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(grid_scan(ctx, g));
  grid_point_scatter_kernel<<<ceil_div(n, 256), 256, 0, st>>>(n, v, g.params.p, g.cell_start.p, g.fill.p, g.pts.p);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  g.n_items = n;
  g.built = true;
  return GINGR_OK;
}

int32_t grid_build_triangles_enqueue(gingr_ctx* ctx, SpatialGrid& g, int n, VertexArray v, int T, const int32_t* d_tri) {
  if (!g.triangles || T > g.cap_items || v.stride_pt != 3 || v.stride_dim != 1)
    return gingr_fail(ctx, GINGR_ERR_ARG, "grid_build_triangles: grid not sized for this mesh / vertices must be AoS");
  cudaStream_t st = ctx->stream;
  GINGR_TRY(grid_common_head(ctx, g, n, v));
  grid_tri_kernel<0><<<ceil_div(T, 256), 256, 0, st>>>(T, v.p, d_tri, g.params.p, g.cell_start.p, g.fill.p, g.entries.p,
                                                      g.cap_entries, g.tri_box.p, nullptr);
  GINGR_LAUNCHED(ctx);
  GINGR_TRY(grid_scan(ctx, g));
  grid_tri_kernel<1><<<ceil_div(T, 256), 256, 0, st>>>(T, v.p, d_tri, g.params.p, g.cell_start.p, g.fill.p, g.entries.p,
                                                      g.cap_entries, g.tri_box.p, g.entry_boxes ? g.entry_box.p : nullptr);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  g.n_items = T;
  g.built = true;
  return GINGR_OK;
}

// ---------------------------------------------------------------------------------------------
// shell iteration shared by the point and the surface query
// ---------------------------------------------------------------------------------------------
// squared distance from q to the (margin-inflated) box of level cell (x, y, z) with edge hl: a lower bound of the
// distance to every item entered in that cell
__device__ __forceinline__ double box_dist2(const GridParams& g, double qx, double qy, double qz, int x, int y, int z,
                                            double hl) {
  const double lx = g.ox + (double)x * hl - g.margin, ly = g.oy + (double)y * hl - g.margin, lz = g.oz + (double)z * hl - g.margin;
  const double w = hl + 2.0 * g.margin;
  const double dx = fmax(0.0, fmax(lx - qx, qx - (lx + w)));
  const double dy = fmax(0.0, fmax(ly - qy, qy - (ly + w)));
  const double dz = fmax(0.0, fmax(lz - qz, qz - (lz + w)));
  return dx * dx + dy * dy + dz * dz;
}

// Exact nearest-item search in two phases (the order a KD-tree query works in):
//   seed   an upper bound: the nearest OCCUPIED cell in the shells around the query's cell -- at the fine level
//          first, then at 4h and 16h for queries far from the surface -- descended to its nearest occupied fine
//          cell, whose entries are evaluated.  Sloppy by design; it only has to produce some candidate.
//   refine the fine cells around the candidate's own location (where()), which nearly always hold the true nearest
//   ball   the proof: every cell whose box is not farther than the current best (which shrinks as candidates are
//          evaluated) is visited, at the finest level where the ball spans at most 4096 cells.
// visit(e0, e1, x, y, z, sh) evaluates the entries [e0, e1) of the level-sh/2 cell (x, y, z) (sh < 0: seed phase,
// evaluate everything) with (value, lowest index) selection; best() returns the current best SQUARED distance.  Returns false when the caller must scan everything (no candidate near, or a ball too big).
template <typename V, typename B, typename W>
__device__ __forceinline__ bool grid_search(const GridParams& g, const int32_t* __restrict__ cell_start, double qx, double qy,
                                            double qz, V&& visit, B&& best, W&& where) {
  const int fx = cell_coord(qx, g.ox, g.inv_h, g.nx), fy = cell_coord(qy, g.oy, g.inv_h, g.ny),
            fz = cell_coord(qz, g.oz, g.inv_h, g.nz);
  // ---- seed ---------------------------------------------------------------------------------------
  bool seeded = false;
  for (int l = 0; l < LEVELS && !seeded; ++l) {
    const int sh = 2 * l;
    const int cx = fx >> sh, cy = fy >> sh, cz = fz >> sh;
    const int nx = ((g.nx - 1) >> sh) + 1, ny = ((g.ny - 1) >> sh) + 1, nz = ((g.nz - 1) >> sh) + 1;
    const double hl = g.h * (double)(1 << sh);
    const int span = 1 << (3 * sh);
    const int kmax = K_LEVEL[l];
    for (int k = 0; k <= kmax && !seeded; ++k) {
      double bd = INFINITY;
      int bx = 0, by = 0, bz = 0;
      const int z0 = max(cz - k, 0), z1 = min(cz + k, nz - 1);
      const int y0 = max(cy - k, 0), y1 = min(cy + k, ny - 1);
      const int x0 = max(cx - k, 0), x1 = min(cx + k, nx - 1);
      for (int z = z0; z <= z1; ++z) {
        const bool zb = (z == cz - k) || (z == cz + k);
        for (int y = y0; y <= y1; ++y) {
          auto cell = [&](int x) {
            const int c = cell_index(g, x << sh, y << sh, z << sh);
            GSTAT(1, 1);
            if (cell_start[c + span] > cell_start[c]) {
              const double d = box_dist2(g, qx, qy, qz, x, y, z, hl);
              if (d < bd) { bd = d; bx = x; by = y; bz = z; }
            }
          };
          if (zb || y == cy - k || y == cy + k) {
            for (int x = x0; x <= x1; ++x) cell(x);
          } else {  // interior rows of the shell only touch the two x faces
            if (cx - k >= 0) cell(cx - k);
            if (cx + k <= nx - 1) cell(cx + k);
          }
        }
      }
      if (bd < INFINITY) {
        // descend to the nearest occupied fine cell of the chosen cell
        for (int ll = l - 1; ll >= 0; --ll) {
          const int s2 = 2 * ll, sp2 = 1 << (3 * s2);
          const double h2 = g.h * (double)(1 << s2);
          double cd = INFINITY;
          int ux = bx << 2, uy = by << 2, uz = bz << 2;
          for (int c = 0; c < 64; ++c) {
            const int x = (bx << 2) + (c & 3), y = (by << 2) + ((c >> 2) & 3), z = (bz << 2) + (c >> 4);
            const int ci = cell_index(g, x << s2, y << s2, z << s2);   // consecutive in c: children are contiguous
            if (cell_start[ci + sp2] > cell_start[ci]) {
              const double d = box_dist2(g, qx, qy, qz, x, y, z, h2);
              if (d < cd) { cd = d; ux = x; uy = y; uz = z; }
            }
          }
          bx = ux; by = uy; bz = uz;
        }
        const int c = cell_index(g, bx, by, bz);
        visit(cell_start[c], cell_start[c + 1], bx, by, bz, -1);
        seeded = true;
      }
    }
  }
  GSTAT(0, 1);
  if (!seeded || !(best() < INFINITY)) { GSTAT(7, 1); return false; }
  // ---- refine: the true nearest item lies near the candidate's own location; the fine cells around it tighten the
  // bound to almost its final value before the ball is walked (two rounds: the location moves)
  for (int round = 0; round < 2; ++round) {
    double wx, wy, wz;
    where(wx, wy, wz);
    const int ux = cell_coord(wx, g.ox, g.inv_h, g.nx), uy = cell_coord(wy, g.oy, g.inv_h, g.ny),
              uz = cell_coord(wz, g.oz, g.inv_h, g.nz);
    for (int z = max(uz - 1, 0); z <= min(uz + 1, g.nz - 1); ++z)
      for (int y = max(uy - 1, 0); y <= min(uy + 1, g.ny - 1); ++y)
        for (int x = max(ux - 1, 0); x <= min(ux + 1, g.nx - 1); ++x) {
          const int c = cell_index(g, x, y, z);
          const int e0 = cell_start[c], e1 = cell_start[c + 1];
          if (e1 > e0 && !(box_dist2(g, qx, qy, qz, x, y, z, g.h) > best())) visit(e0, e1, x, y, z, 0);
        }
  }
  // ---- ball ---------------------------------------------------------------------------------------
  const double R = sqrt(best()) * (1.0 + 1e-12) + 2.0 * g.margin;
  const int rx0 = max(cell_coord_raw(qx - R, g.ox, g.inv_h), 0), rx1 = min(cell_coord_raw(qx + R, g.ox, g.inv_h), g.nx - 1);
  const int ry0 = max(cell_coord_raw(qy - R, g.oy, g.inv_h), 0), ry1 = min(cell_coord_raw(qy + R, g.oy, g.inv_h), g.ny - 1);
  const int rz0 = max(cell_coord_raw(qz - R, g.oz, g.inv_h), 0), rz1 = min(cell_coord_raw(qz + R, g.oz, g.inv_h), g.nz - 1);
  for (int l = 0; l < LEVELS; ++l) {
    const int sh = 2 * l;
    const int x0 = rx0 >> sh, x1 = rx1 >> sh, y0 = ry0 >> sh, y1 = ry1 >> sh, z0 = rz0 >> sh, z1 = rz1 >> sh;
    if ((long long)(x1 - x0 + 1) * (y1 - y0 + 1) * (z1 - z0 + 1) > 4096) continue;
    const double hl = g.h * (double)(1 << sh);
    const int span = 1 << (3 * sh);
    GSTAT(6, l);
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) {
        if (box_dist2(g, qx, qy, qz, min(max(fx >> sh, x0), x1), y, z, hl) > best()) continue;   // whole row too far
        for (int x = x0; x <= x1; ++x) {
          const int c = cell_index(g, x << sh, y << sh, z << sh);
          const int e0 = cell_start[c], e1 = cell_start[c + span];
          GSTAT(2, 1);
          if (e1 > e0 && !(box_dist2(g, qx, qy, qz, x, y, z, hl) > best())) { GSTAT(3, 1); GSTAT(4, e1 - e0); visit(e0, e1, x, y, z, sh); }
        }
      }
    return true;
  }
  GSTAT(7, 1);
  return false;
}

// a point grid built over the queries doubles as their spatial sort: slot -> original query id in pts[slot].w
static const double4* order_ptr(const SpatialGrid* order, int M) {
  return (order && order->built && !order->triangles && order->n_items == M) ? order->pts.p : nullptr;
}

// ---------------------------------------------------------------------------------------------
// nearest point
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) grid_nn_kernel(int M, const double4* __restrict__ order, const double* __restrict__ q, int n,
                                                      const GridParams* __restrict__ gp, const int32_t* __restrict__ cell_start,
                                                      const double4* __restrict__ pts, double* __restrict__ d2,
                                                      int32_t* __restrict__ idx) {
  const int slot = blockIdx.x * 128 + threadIdx.x;
  if (slot >= M) return;
  const int i = order ? (int)__double_as_longlong(order[slot].w) : slot;   // spatially sorted queries: coherent warps
  const double qx = q[3 * i], qy = q[3 * i + 1], qz = q[3 * i + 2];
  double best = INFINITY, bpx = 0, bpy = 0, bpz = 0;
  int bi = -1;
  auto consider = [&](int e) {
    const double4 p = pts[e];
    const double dx = qx - p.x, dy = qy - p.y, dz = qz - p.z;
    const double d = dx * dx + dy * dy + dz * dz;
    const int j = (int)__double_as_longlong(p.w);
    if (d < best || (d == best && j < bi)) { best = d; bi = j; bpx = p.x; bpy = p.y; bpz = p.z; }
  };
  if (isfinite(qx) && isfinite(qy) && isfinite(qz)) {
    const GridParams g = *gp;
    const bool done = grid_search(g, cell_start, qx, qy, qz,
                                  [&](int e0, int e1, int, int, int, int) { for (int e = e0; e < e1; ++e) consider(e); },
                                  [&]() { return best; }, [&](double& x, double& y, double& z) { x = bpx; y = bpy; z = bpz; });
    if (!done) {
      best = INFINITY; bi = -1;
      for (int e = 0; e < n; ++e) consider(e);
    }
  }
  d2[i] = best;
  idx[i] = bi;
}

int32_t grid_nn_enqueue(gingr_ctx* ctx, const SpatialGrid& g, int M, const double* d_q, double* d_d2, int32_t* d_idx,
                        const SpatialGrid* order) {
  if (!g.built || g.triangles) return gingr_fail(ctx, GINGR_ERR_ARG, "grid_nn: point grid not built");
  // thread per query: a candidate point is one distance evaluation, and the warp-per-query variant measured slower
  // (far queries 1015 vs 696 us, near queries 287 vs 83 us at 100k) -- unlike the surface search below
  grid_nn_kernel<<<ceil_div(M, 128), 128, 0, ctx->stream>>>(M, order_ptr(order, M), d_q, g.n_items, g.params.p, g.cell_start.p, g.pts.p, d_d2, d_idx);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// ---------------------------------------------------------------------------------------------
// closest point on the surface
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) grid_surface_kernel(int M, const double4* __restrict__ order, const double* __restrict__ q, int T,
                                                           const GridParams* __restrict__ gp,
                                                           const int32_t* __restrict__ cell_start,
                                                           const int32_t* __restrict__ entries,
                                                           const float4* __restrict__ tri_box,
                                                           const double* __restrict__ verts /*AoS*/,
                                                           const int32_t* __restrict__ tri, double* __restrict__ d2,
                                                           int32_t* __restrict__ tri_out, double* __restrict__ cp) {
  const int slot = blockIdx.x * 128 + threadIdx.x;
  if (slot >= M) return;
  const int i = order ? (int)__double_as_longlong(order[slot].w) : slot;   // spatially sorted queries: coherent warps
  const double qx = q[3 * i], qy = q[3 * i + 1], qz = q[3 * i + 2];
  double best = INFINITY, bx = 0, by = 0, bz = 0;
  int bt = -1;
  GridParams g;
  auto consider = [&](int t, int x, int y, int z, int sh) {
    {
      // quick reject: the triangle lies inside its (outward rounded) box, so it cannot beat or tie the best when
      // the box is strictly farther.  De-duplication: a triangle is entered in every cell its box overlaps; it is
      // evaluated only in the cell that holds the point of its box nearest to the query -- that cell is one of its
      // cells (same box, same monotone cell function as the build) and is never farther than the triangle itself, so
      // the ball walk reaches it whenever the triangle can win.
      const float4 lo = tri_box[2 * t], hi = tri_box[2 * t + 1];
      const double px = fmin(fmax(qx, (double)lo.x), (double)hi.x), py = fmin(fmax(qy, (double)lo.y), (double)hi.y),
                   pz = fmin(fmax(qz, (double)lo.z), (double)hi.z);
      const double ex = qx - px, ey = qy - py, ez = qz - pz;
      if ((ex * ex + ey * ey + ez * ez) * (1.0 - 1e-12) > best) return;
      if (sh >= 0 && ((cell_coord(px, g.ox, g.inv_h, g.nx) >> sh) != x || (cell_coord(py, g.oy, g.inv_h, g.ny) >> sh) != y ||
                      (cell_coord(pz, g.oz, g.inv_h, g.nz) >> sh) != z))
        return;
    }
    GSTAT(5, 1);
    const double* a = verts + 3 * (size_t)tri[3 * t];
    const double* b = verts + 3 * (size_t)tri[3 * t + 1];
    const double* c = verts + 3 * (size_t)tri[3 * t + 2];
    const double va[3] = {a[0], a[1], a[2]}, vb[3] = {b[0], b[1], b[2]}, vc[3] = {c[0], c[1], c[2]};
    double cx, cy, cz;
    closest_on_triangle(qx, qy, qz, va, vb, vc, cx, cy, cz);
    const double dx = qx - cx, dy = qy - cy, dz = qz - cz;
    const double d = dx * dx + dy * dy + dz * dz;
    if (d < best || (d == best && t < bt)) { best = d; bt = t; bx = cx; by = cy; bz = cz; }
  };
  if (isfinite(qx) && isfinite(qy) && isfinite(qz)) {
    g = *gp;
    bool done = false;
    if (!g.overflow) {
      done = grid_search(g, cell_start, qx, qy, qz,
                         [&](int e0, int e1, int x, int y, int z, int sh) {
                           for (int e = e0; e < e1; ++e) consider(entries[e], x, y, z, sh);
                         },
                         [&]() { return best; }, [&](double& x, double& y, double& z) { x = bx; y = by; z = bz; });
    }
    if (!done) {
      best = INFINITY; bt = -1; bx = by = bz = 0;
      for (int t = 0; t < T; ++t) consider(t, 0, 0, 0, -1);
    }
  }
  d2[i] = best;
  if (tri_out) tri_out[i] = bt;
  cp[3 * i] = bx; cp[3 * i + 1] = by; cp[3 * i + 2] = bz;
}


// ---------------------------------------------------------------------------------------------
// closest point on the surface, one WARP per query.
// The thread-per-query kernel above runs with 3-9 of 32 lanes active in its hot loops (profiles/r01s_ncu_grid_surface.md:
// every lane walks its own cells and takes its own branches of the exact triangle evaluation).  Here the 32 lanes share
// one query: cells of the seed cube / the refinement block / the ball are examined 32 at a time, the entries of a passing
// cell are box-tested 32 at a time, the survivors are COMPACTED into a per-warp queue and evaluated exactly 32 at a time.
// Same candidates' arithmetic, same conservative bounds, winners by (value, lowest triangle index) across lanes: the
// results are bit-identical to the scans.
// ---------------------------------------------------------------------------------------------
constexpr int WQ_WARPS = 4;      // queries (warps) per CTA
constexpr int WQ_CAP = 128;      // candidate queue per warp

struct WarpBest {
  double d, x, y, z;
  int t;
};

__device__ __forceinline__ void warp_best_reduce(WarpBest& b) {
  // lexicographic (d, t) minimum over the lanes, then the winner's point is broadcast
  double d = b.d;
  int t = b.t, who = threadIdx.x & 31;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, d, o);
    const int ot = __shfl_xor_sync(0xffffffffu, t, o);
    const int ow = __shfl_xor_sync(0xffffffffu, who, o);
    if (od < d || (od == d && (unsigned)ot < (unsigned)t)) { d = od; t = ot; who = ow; }
  }
  b.d = d; b.t = t;
  b.x = __shfl_sync(0xffffffffu, b.x, who);
  b.y = __shfl_sync(0xffffffffu, b.y, who);
  b.z = __shfl_sync(0xffffffffu, b.z, who);
}

#ifndef WQ_MINB
#define WQ_MINB 4   // 128 registers (a few spills in the cell walks); 3 (168, none) measured 11 % slower, 5 and 6 the same as 4
#endif
__global__ void __launch_bounds__(WQ_WARPS * 32, WQ_MINB) grid_surface_warp_kernel(
    int M, const double4* __restrict__ order, const double* __restrict__ q, int T, const GridParams* __restrict__ gp,
    const int32_t* __restrict__ cell_start, const int32_t* __restrict__ entries, const float4* __restrict__ tri_box,
    const double* __restrict__ verts /*AoS*/, const int32_t* __restrict__ tri, double* __restrict__ d2,
    int32_t* __restrict__ tri_out, double* __restrict__ cp, int descend /*GINGR_K2_DESCEND, A/B measurements*/,
    const float4* __restrict__ entry_box /*boxes stored with the entries (static grids), may be null*/) {
  __shared__ int s_queue[WQ_WARPS][WQ_CAP];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int slot = blockIdx.x * WQ_WARPS + w;
  if (slot >= M) return;   // whole warps leave: no partial-warp collectives below
  const int i = order ? (int)__double_as_longlong(order[slot].w) : slot;
  const double qx = q[3 * i], qy = q[3 * i + 1], qz = q[3 * i + 2];
  int* queue = s_queue[w];
  int qn = 0;   // warp-uniform
  WarpBest best;   // warp-uniform after every flush
  best.d = INFINITY; best.x = best.y = best.z = 0.0; best.t = 0x7fffffff;
  const GridParams g = *gp;

  // exact evaluation of the queued candidates, 32 at a time; the warp's best is re-established afterwards
  int phase = 0;   // statistics only: 0 seed, 1 refine, 2 ball
  (void)phase;
  GSTATW(0, 1);
  auto flush = [&]() {
    __syncwarp();
    GSTATW(8, 1); GSTATW(7, qn);
    WarpBest mine = best;
    for (int base = 0; base < qn; base += 32) {
      const int k = base + lane;
      if (k < qn) {
        const int t = queue[k];
        const double* a = verts + 3 * (size_t)tri[3 * t];
        const double* b = verts + 3 * (size_t)tri[3 * t + 1];
        const double* c = verts + 3 * (size_t)tri[3 * t + 2];
        const double va[3] = {a[0], a[1], a[2]}, vb[3] = {b[0], b[1], b[2]}, vc[3] = {c[0], c[1], c[2]};
        double cx, cy, cz;
        closest_on_triangle(qx, qy, qz, va, vb, vc, cx, cy, cz);
        const double dx = qx - cx, dy = qy - cy, dz = qz - cz;
        const double d = dx * dx + dy * dy + dz * dz;
        if (d < mine.d || (d == mine.d && (unsigned)t < (unsigned)mine.t)) { mine.d = d; mine.t = t; mine.x = cx; mine.y = cy; mine.z = cz; }
      }
    }
    warp_best_reduce(mine);
    best = mine;
    qn = 0;
    __syncwarp();
  };
  // box test (+ home-cell de-duplication for sh >= 0) of the triangles t = first + lane ... and compaction into the queue
  auto offer = [&](bool valid, int t, int x, int y, int z, int sh, int e) {   // e >= 0: position in `entries`
    bool pass = false;
    if (valid) {
      float4 lo, hi;
      if (entry_box != nullptr && e >= 0) { lo = entry_box[2 * (size_t)e]; hi = entry_box[2 * (size_t)e + 1]; }   // streams with entries[e]
      else { lo = tri_box[2 * t]; hi = tri_box[2 * t + 1]; }
      const double px = fmin(fmax(qx, (double)lo.x), (double)hi.x), py = fmin(fmax(qy, (double)lo.y), (double)hi.y),
                   pz = fmin(fmax(qz, (double)lo.z), (double)hi.z);
      const double ex = qx - px, ey = qy - py, ez = qz - pz;
      pass = !((ex * ex + ey * ey + ez * ez) * (1.0 - 1e-12) > best.d);
      if (pass && sh >= 0)
        pass = (cell_coord(px, g.ox, g.inv_h, g.nx) >> sh) == x && (cell_coord(py, g.oy, g.inv_h, g.ny) >> sh) == y &&
               (cell_coord(pz, g.oz, g.inv_h, g.nz) >> sh) == z;
    }
    const unsigned m = __ballot_sync(0xffffffffu, pass);
    if (pass) queue[qn + __popc(m & ((1u << lane) - 1u))] = t;
    qn += __popc(m);
    if (qn > WQ_CAP - 32) flush();
  };
  auto offer_entries = [&](int e0, int e1, int x, int y, int z, int sh) {
    GSTATW(phase == 0 ? 2 : (phase == 1 ? 3 : 6), e1 - e0);
    for (int base = e0; base < e1; base += 32) {
      const int e = base + lane;
      const bool valid = e < e1;
      offer(valid, valid ? entries[e] : 0, x, y, z, sh, e);
    }
  };

  int u1x = -9, u1y = -9, u1z = -9, u2x = -9, u2y = -9, u2z = -9;   // centres of the two refinement blocks (fine cells)
  auto refined = [&](int x, int y, int z) {
    return (abs(x - u1x) <= 1 && abs(y - u1y) <= 1 && abs(z - u1z) <= 1) || (abs(x - u2x) <= 1 && abs(y - u2y) <= 1 && abs(z - u2z) <= 1);
  };
  // a coarse cell of the ball walk that passed its box test: its 64 children (nested 4 x 4 x 4 blocking: contiguous in
  // cell_start), two per lane, are box-tested themselves and only the passing fine cells offer their entries -- a far
  // query's ball touches the surface in a cap that is a few FINE cells wide, a coarse cell holds ~16 occupied ones
  auto walk_fine = [&](int ci, int x, int y, int z) {   // (x, y, z) at level 1 (edge 4h), ci = index of its first fine cell
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const int c = lane + 32 * half;
      const int xx = (x << 2) | (c & 3), yy = (y << 2) | ((c >> 2) & 3), zz = (z << 2) | (c >> 4);
      int e0 = cell_start[ci + c], e1 = cell_start[ci + c + 1];
      if (e1 > e0 && (refined(xx, yy, zz) || box_dist2(g, qx, qy, qz, xx, yy, zz, g.h) > best.d)) e1 = e0;
      unsigned m = __ballot_sync(0xffffffffu, e1 > e0);
      GSTATW(10, __popc(m));
      while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        offer_entries(__shfl_sync(0xffffffffu, e0, src), __shfl_sync(0xffffffffu, e1, src), __shfl_sync(0xffffffffu, xx, src),
                      __shfl_sync(0xffffffffu, yy, src), __shfl_sync(0xffffffffu, zz, src), 0);
      }
    }
  };
  auto walk_mid = [&](int ci, int x, int y, int z) {    // (x, y, z) at level 2 (edge 16h): children at level 1
    const double h1 = g.h * 4.0;
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const int c = lane + 32 * half;
      const int xx = (x << 2) | (c & 3), yy = (y << 2) | ((c >> 2) & 3), zz = (z << 2) | (c >> 4);
      const int cc = ci + (c << 6);
      bool pass = cell_start[cc + 64] > cell_start[cc];
      if (pass && box_dist2(g, qx, qy, qz, xx, yy, zz, h1) > best.d) pass = false;
      unsigned m = __ballot_sync(0xffffffffu, pass);
      while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        walk_fine(__shfl_sync(0xffffffffu, cc, src), __shfl_sync(0xffffffffu, xx, src), __shfl_sync(0xffffffffu, yy, src),
                  __shfl_sync(0xffffffffu, zz, src));
      }
    }
  };

  bool done = false;
  const bool finite_q = isfinite(qx) && isfinite(qy) && isfinite(qz);
  if (finite_q && !g.overflow) {
    const int fx = cell_coord(qx, g.ox, g.inv_h, g.nx), fy = cell_coord(qy, g.oy, g.inv_h, g.ny),
              fz = cell_coord(qz, g.oz, g.inv_h, g.nz);
    // ---- seed: nearest occupied cell in the cubes around the query's cell, level by level ------------------------
    bool seeded = false;
    for (int l = 0; l < LEVELS && !seeded; ++l) {
      const int sh = 2 * l;
      const int cx = fx >> sh, cy = fy >> sh, cz = fz >> sh;
      const int nx = ((g.nx - 1) >> sh) + 1, ny = ((g.ny - 1) >> sh) + 1, nz = ((g.nz - 1) >> sh) + 1;
      const double hl = g.h * (double)(1 << sh);
      const int span = 1 << (3 * sh);
      for (int k = 0; k <= K_LEVEL[l] && !seeded; ++k) {
        const int side = 2 * k + 1, vol = side * side * side;
        GSTATW(1, vol);
        double bd = INFINITY;
        int bc = 0x7fffffff;   // packed (z, y, x) of the lane's nearest occupied cell, 10 bits each
        for (int c = lane; c < vol; c += 32) {
          const int x = cx - k + c % side, y = cy - k + (c / side) % side, z = cz - k + c / (side * side);
          if (x < 0 || y < 0 || z < 0 || x >= nx || y >= ny || z >= nz) continue;
          const int ci = cell_index(g, x << sh, y << sh, z << sh);
          if (cell_start[ci + span] > cell_start[ci]) {
            const double d = box_dist2(g, qx, qy, qz, x, y, z, hl);
            const int pc = (z << 20) | (y << 10) | x;
            if (d < bd || (d == bd && pc < bc)) { bd = d; bc = pc; }
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double od = __shfl_xor_sync(0xffffffffu, bd, o);
          const int oc = __shfl_xor_sync(0xffffffffu, bc, o);
          if (od < bd || (od == bd && oc < bc)) { bd = od; bc = oc; }
        }
        if (bd < INFINITY) {
          int bx = bc & 1023, by = (bc >> 10) & 1023, bz = bc >> 20;
          for (int ll = l - 1; ll >= 0; --ll) {   // descend to the nearest occupied child, 64 children: 2 per lane
            const int s2 = 2 * ll, sp2 = 1 << (3 * s2);
            const double h2 = g.h * (double)(1 << s2);
            double cd = INFINITY;
            int cc = 0x7fffffff;
            for (int c = lane; c < 64; c += 32) {
              const int x = (bx << 2) + (c & 3), y = (by << 2) + ((c >> 2) & 3), z = (bz << 2) + (c >> 4);
              const int ci = cell_index(g, x << s2, y << s2, z << s2);
              if (cell_start[ci + sp2] > cell_start[ci]) {
                const double d = box_dist2(g, qx, qy, qz, x, y, z, h2);
                const int pc = (z << 20) | (y << 10) | x;
                if (d < cd || (d == cd && pc < cc)) { cd = d; cc = pc; }
              }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              const double od = __shfl_xor_sync(0xffffffffu, cd, o);
              const int oc = __shfl_xor_sync(0xffffffffu, cc, o);
              if (od < cd || (od == cd && oc < cc)) { cd = od; cc = oc; }
            }
            bx = cc & 1023; by = (cc >> 10) & 1023; bz = cc >> 20;
          }
          const int ci = cell_index(g, bx, by, bz);
          offer_entries(cell_start[ci], cell_start[ci + 1], bx, by, bz, -1);
          flush();
          seeded = true;
        }
      }
    }
    if (seeded && best.d < INFINITY) {
      // ---- refine: the 27 fine cells around the candidate's own location, twice -----------------------------------
      // A cell examined here has had all the triangles it is the home cell of offered against a bound that was not
      // tighter than any later one: the second round and the ball walk below skip the cells of the earlier blocks
      // (their survivors would only be evaluated a second time).
      phase = 1;
      for (int round = 0; round < 2; ++round) {
        const int ux = cell_coord(best.x, g.ox, g.inv_h, g.nx), uy = cell_coord(best.y, g.oy, g.inv_h, g.ny),
                  uz = cell_coord(best.z, g.oz, g.inv_h, g.nz);
        if (round == 0) { u1x = ux; u1y = uy; u1z = uz; }
        u2x = ux; u2y = uy; u2z = uz;
        if (round == 1 && ux == u1x && uy == u1y && uz == u1z) break;
        int x = 0, y = 0, z = 0, e0 = 0, e1 = 0;
        if (lane < 27) {
          x = ux - 1 + lane % 3; y = uy - 1 + (lane / 3) % 3; z = uz - 1 + lane / 9;
          const bool seen = round == 1 && abs(x - u1x) <= 1 && abs(y - u1y) <= 1 && abs(z - u1z) <= 1;
          if (!seen && x >= 0 && y >= 0 && z >= 0 && x < g.nx && y < g.ny && z < g.nz) {
            const int c = cell_index(g, x, y, z);
            e0 = cell_start[c]; e1 = cell_start[c + 1];
            if (e1 > e0 && box_dist2(g, qx, qy, qz, x, y, z, g.h) > best.d) e1 = e0;
          }
        }
        unsigned m = __ballot_sync(0xffffffffu, e1 > e0);
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1;
          offer_entries(__shfl_sync(0xffffffffu, e0, src), __shfl_sync(0xffffffffu, e1, src), __shfl_sync(0xffffffffu, x, src),
                        __shfl_sync(0xffffffffu, y, src), __shfl_sync(0xffffffffu, z, src), 0);
        }
        flush();
      }
      // ---- ball: every cell whose box is not farther than the best, at the finest level with <= 4096 cells ---------
      const double R = sqrt(best.d) * (1.0 + 1e-12) + 2.0 * g.margin;
      const int rx0 = max(cell_coord_raw(qx - R, g.ox, g.inv_h), 0), rx1 = min(cell_coord_raw(qx + R, g.ox, g.inv_h), g.nx - 1);
      const int ry0 = max(cell_coord_raw(qy - R, g.oy, g.inv_h), 0), ry1 = min(cell_coord_raw(qy + R, g.oy, g.inv_h), g.ny - 1);
      const int rz0 = max(cell_coord_raw(qz - R, g.oz, g.inv_h), 0), rz1 = min(cell_coord_raw(qz + R, g.oz, g.inv_h), g.nz - 1);
      for (int l = 0; l < LEVELS && !done; ++l) {
        const int sh = 2 * l;
        const int x0 = rx0 >> sh, x1 = rx1 >> sh, y0 = ry0 >> sh, y1 = ry1 >> sh, z0 = rz0 >> sh, z1 = rz1 >> sh;
        const int sx = x1 - x0 + 1, sy = y1 - y0 + 1, sz = z1 - z0 + 1;
        if (sx < 1 || sy < 1 || sz < 1) { done = true; break; }   // cannot happen: the candidate lies inside the ball
        if ((long long)sx * sy * sz > 4096) continue;
        const int vol = sx * sy * sz;
        phase = 2;
        GSTATW(4, vol); GSTATW(9, l);
        const double hl = g.h * (double)(1 << sh);
        const int span = 1 << (3 * sh);
        // c -> (x, y, z) without integer divisions: c < 4096, so the float quotients (error < 1e-3 / n, the fraction of
        // (c + 0.5) / n is at least 0.5 / n from an integer) floor to the exact values
        const int sxy = sx * sy;
        const float inv_sx = 1.0f / (float)sx, inv_sxy = 1.0f / (float)sxy;
        for (int base = 0; base < vol; base += 32) {
          const int c = base + lane;
          int x = 0, y = 0, z = 0, e0 = 0, e1 = 0;
          if (c < vol) {
            const int zc = (int)(((float)c + 0.5f) * inv_sxy), rem = c - zc * sxy, yc = (int)(((float)rem + 0.5f) * inv_sx);
            x = x0 + rem - yc * sx; y = y0 + yc; z = z0 + zc;
            const int ci = cell_index(g, x << sh, y << sh, z << sh);
            e0 = cell_start[ci]; e1 = cell_start[ci + span];
            if (e1 > e0 && ((l == 0 && refined(x, y, z)) || box_dist2(g, qx, qy, qz, x, y, z, hl) > best.d)) e1 = e0;
          }
          int ci0 = 0;
          if (c < vol) ci0 = cell_index(g, x << sh, y << sh, z << sh);
          unsigned m = __ballot_sync(0xffffffffu, e1 > e0);
          GSTATW(5, __popc(m));
          while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const int xs = __shfl_sync(0xffffffffu, x, src), ys = __shfl_sync(0xffffffffu, y, src), zs = __shfl_sync(0xffffffffu, z, src);
            if (l == 0 || !descend)
              offer_entries(__shfl_sync(0xffffffffu, e0, src), __shfl_sync(0xffffffffu, e1, src), xs, ys, zs, sh);
            else if (l == 1)
              walk_fine(__shfl_sync(0xffffffffu, ci0, src), xs, ys, zs);
            else
              walk_mid(__shfl_sync(0xffffffffu, ci0, src), xs, ys, zs);
          }
        }
        flush();
        done = true;
      }
    }
  }
  if (finite_q && !done) {
    // everything (overflowed grid, nothing near, ball too big): all triangles, 32 at a time
    qn = 0;
    best.d = INFINITY; best.x = best.y = best.z = 0.0; best.t = 0x7fffffff;
    for (int base = 0; base < T; base += 32) offer(base + lane < T, base + lane, 0, 0, 0, -1, -1);
    flush();
  }
  if (lane == 0) {
    d2[i] = best.d;
    if (tri_out) tri_out[i] = best.t == 0x7fffffff ? -1 : best.t;
    cp[3 * i] = best.x; cp[3 * i + 1] = best.y; cp[3 * i + 2] = best.z;
  }
}


static bool warp_search_wanted() {
  const char* e = getenv("GINGR_K2_WARP");   // 0: thread-per-query surface search (A/B measurements); default: warp-per-query
  return !(e && *e && atoi(e) == 0);
}

int32_t grid_surface_enqueue(gingr_ctx* ctx, const SpatialGrid& g, int M, const double* d_q, const double* d_verts_aos,
                             const int32_t* d_tri, double* d_d2, int32_t* d_tri_out, double* d_cp, const SpatialGrid* order) {
  if (!g.built || !g.triangles) return gingr_fail(ctx, GINGR_ERR_ARG, "grid_surface: triangle grid not built");
  if (warp_search_wanted()) {
    static const int descend = [] { const char* e = getenv("GINGR_K2_DESCEND"); return e ? atoi(e) : 1; }();
    static const int use_entry_boxes = [] { const char* e = getenv("GINGR_K2_ENTRY_BOXES"); return e ? atoi(e) : 1; }();
    grid_surface_warp_kernel<<<ceil_div(M, WQ_WARPS), WQ_WARPS * 32, 0, ctx->stream>>>(
        M, order_ptr(order, M), d_q, g.n_items, g.params.p, g.cell_start.p, g.entries.p, g.tri_box.p, d_verts_aos, d_tri, d_d2,
        d_tri_out, d_cp, descend, (g.entry_boxes && use_entry_boxes) ? g.entry_box.p : nullptr);
    GINGR_LAUNCHED(ctx);
    GINGR_CUDA_TRY(ctx, cudaGetLastError());
    return GINGR_OK;
  }
  grid_surface_kernel<<<ceil_div(M, 128), 128, 0, ctx->stream>>>(M, order_ptr(order, M), d_q, g.n_items, g.params.p, g.cell_start.p, g.entries.p,
                                                                 g.tri_box.p, d_verts_aos, d_tri, d_d2, d_tri_out, d_cp);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

// ---------------------------------------------------------------------------------------------
// line vs mesh
// ---------------------------------------------------------------------------------------------
template <bool SELF>
__global__ void __launch_bounds__(128) grid_line_kernel(int M, const double4* __restrict__ order, const double* __restrict__ o, const double* __restrict__ other,
                                                        int T, const GridParams* __restrict__ gp,
                                                        const int32_t* __restrict__ cell_start,
                                                        const int32_t* __restrict__ entries,
                                                        const double* __restrict__ mesh /*AoS*/,
                                                        const int32_t* __restrict__ tri, double* __restrict__ out_min,
                                                        double* __restrict__ out_pt, int q0) {
  const int slot = blockIdx.x * 128 + threadIdx.x;
  if (slot >= M) return;
  const int i = order ? (int)__double_as_longlong(order[slot].w) : slot;   // spatially sorted queries: coherent warps
  const double ox = o[3 * i], oy = o[3 * i + 1], oz = o[3 * i + 2];
  double dx = other[3 * i], dy = other[3 * i + 1], dz = other[3 * i + 2];
  if (SELF) { dx = ox - dx; dy = oy - dy; dz = oz - dz; }
  double best = INFINITY, bx = ox, by = oy, bz = oz;
  int bt = 0x7fffffff;
  auto consider = [&](int t) {
    const int v0 = tri[3 * t], v1 = tri[3 * t + 1], v2 = tri[3 * t + 2];
    if (SELF && (v0 == q0 + i || v1 == q0 + i || v2 == q0 + i)) return;   // q0: vertex id of query 0 (query range of the mesh)
    const double* a = mesh + 3 * (size_t)v0;
    const double* b = mesh + 3 * (size_t)v1;
    const double* c = mesh + 3 * (size_t)v2;
    const double va[3] = {a[0], a[1], a[2]}, vb[3] = {b[0], b[1], b[2]}, vc[3] = {c[0], c[1], c[2]};
    double d, ix, iy, iz;
    if (!line_triangle_hit(ox, oy, oz, dx, dy, dz, va, vb, vc, d, ix, iy, iz)) return;
    if (d < best || (d == best && t < bt)) { best = d; bt = t; bx = ix; by = iy; bz = iz; }
  };
  const bool finite_in = isfinite(ox) && isfinite(oy) && isfinite(oz) && isfinite(dx) && isfinite(dy) && isfinite(dz);
  const GridParams g = *gp;
  if (finite_in && g.overflow) {
    for (int t = 0; t < T; ++t) consider(t);
  } else if (finite_in && !(dx == 0.0 && dy == 0.0 && dz == 0.0)) {
    // permute so that `a` is the major axis of the direction
    const double ax = fabs(dx), ay = fabs(dy), az = fabs(dz);
    double oa, ob, oc, da, db, dc, ga, gb, gc;
    int na, nb, nc, perm;
    if (ax >= ay && ax >= az) {
      oa = ox; ob = oy; oc = oz; da = dx; db = dy; dc = dz; ga = g.ox; gb = g.oy; gc = g.oz;
      na = g.nx; nb = g.ny; nc = g.nz; perm = 0;
    } else if (ay >= az) {
      oa = oy; ob = ox; oc = oz; da = dy; db = dx; dc = dz; ga = g.oy; gb = g.ox; gc = g.oz;
      na = g.ny; nb = g.nx; nc = g.nz; perm = 1;
    } else {
      oa = oz; ob = ox; oc = oy; da = dz; db = dx; dc = dy; ga = g.oz; gb = g.ox; gc = g.oy;
      na = g.nz; nb = g.nx; nc = g.ny; perm = 2;
    }
    const double dn = sqrt(dx * dx + dy * dy + dz * dz);
    const double inv_da = 1.0 / da;
    const double s_margin = fabs(g.margin * inv_da);
    const double s_limit = SELF ? 1.001 : INFINITY;   // SELF: only hits nearer than |d| (|s| < 1) can matter
    const int ja0 = cell_coord(oa, ga, g.inv_h, na);
    for (int dir = 1; dir >= -1; dir -= 2) {
      const int step = (da > 0.0) ? dir : -dir;
      for (int ja = ja0; ja >= 0 && ja < na; ja += step) {
        const double sA = ((ga + (double)ja * g.h) - oa) * inv_da, sB = ((ga + (double)(ja + 1) * g.h) - oa) * inv_da;
        double s_lo = fmin(sA, sB) - s_margin, s_hi = fmax(sA, sB) + s_margin;
        // the part of the slab on this half line, within the useful range
        if (dir > 0) { s_lo = fmax(s_lo, 0.0); s_hi = fmin(s_hi, s_limit); }
        else { s_hi = fmin(s_hi, 0.0); s_lo = fmax(s_lo, -s_limit); }
        if (s_lo > s_hi) {
          // empty: either the slab lies behind the origin (only possible for the first slabs when the origin is
          // outside the grid) or beyond the useful range (then every later slab is, too)
          const double s_near = dir > 0 ? fmin(sA, sB) : -fmax(sA, sB);
          if (s_near > s_limit) break;
          continue;
        }
        const double s_near = dir > 0 ? s_lo : -s_hi;
        if (s_near * dn - g.margin > best) break;   // every hit in this and later slabs is farther than the best
        const double b0 = ob + s_lo * db, b1 = ob + s_hi * db, c0 = oc + s_lo * dc, c1 = oc + s_hi * dc;
        int jb0 = cell_coord_raw(fmin(b0, b1) - g.margin, gb, g.inv_h), jb1 = cell_coord_raw(fmax(b0, b1) + g.margin, gb, g.inv_h);
        int jc0 = cell_coord_raw(fmin(c0, c1) - g.margin, gc, g.inv_h), jc1 = cell_coord_raw(fmax(c0, c1) + g.margin, gc, g.inv_h);
        if (jb1 < 0 || jb0 >= nb || jc1 < 0 || jc0 >= nc) continue;
        jb0 = max(jb0, 0); jb1 = min(jb1, nb - 1); jc0 = max(jc0, 0); jc1 = min(jc1, nc - 1);
        for (int jc = jc0; jc <= jc1; ++jc)
          for (int jb = jb0; jb <= jb1; ++jb) {
            const int c = perm == 0 ? cell_index(g, ja, jb, jc) : perm == 1 ? cell_index(g, jb, ja, jc) : cell_index(g, jb, jc, ja);
            const int e1 = cell_start[c + 1];
            for (int e = cell_start[c]; e < e1; ++e) consider(entries[e]);
          }
      }
    }
  }
  out_min[i] = best;
  if (out_pt) { out_pt[3 * i] = bx; out_pt[3 * i + 1] = by; out_pt[3 * i + 2] = bz; }
}

int32_t grid_line_enqueue(gingr_ctx* ctx, const SpatialGrid& g, int M, const double* d_o, const double* d_other,
                          const double* d_mesh_aos, const int32_t* d_tri, int self, double* d_min, double* d_pt,
                          const SpatialGrid* order, int q0) {
  if (!g.built || !g.triangles) return gingr_fail(ctx, GINGR_ERR_ARG, "grid_line: triangle grid not built");
  if (self)
    grid_line_kernel<true><<<ceil_div(M, 128), 128, 0, ctx->stream>>>(M, order_ptr(order, M), d_o, d_other, g.n_items, g.params.p, g.cell_start.p,
                                                                      g.entries.p, d_mesh_aos, d_tri, d_min, d_pt, q0);
  else
    grid_line_kernel<false><<<ceil_div(M, 128), 128, 0, ctx->stream>>>(M, order_ptr(order, M), d_o, d_other, g.n_items, g.params.p, g.cell_start.p,
                                                                       g.entries.p, d_mesh_aos, d_tri, d_min, d_pt, q0);
  GINGR_LAUNCHED(ctx);
  GINGR_CUDA_TRY(ctx, cudaGetLastError());
  return GINGR_OK;
}

}  // namespace gingr

#ifdef GINGR_GRID_STATS
extern "C" GINGR_API int32_t gingr_debug_grid_stats(unsigned long long* out, int32_t reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, gingr::grid_stats, sizeof(unsigned long long) * 24);
  if (reset) {
    unsigned long long z[24] = {0};
    cudaMemcpyToSymbol(gingr::grid_stats, z, sizeof(z));
  }
  return 0;
}
#endif
