// grid.cu — device-resident search surface: packs caller rows into float4, computes the bounding box
// and builds a dense uniform grid (counting sort by cell) on demand.
//
// This replaces pcl::search::KdTree / KdTreeFLANN<PointXYZRGBA>::setInputCloud, which every
// Feature::compute() of the reference builds implicitly (e.g. SHOT.cpp:305, 364; SHOT_demo.cpp:410).
// The searches on top of it are exact, so the answers equal the kd-tree's.
//
// Data layout in HBM: `raw` = N float4 in caller order (x, y, z, 1); per grid: `pts` = the finite
// points in cell-major order with w = original row index (so one 16-byte load yields coordinates
// and identity), `cell_start` = ncell + 1 ints.  Algorithmic traffic of a build: 16 B read +
// 4 B cell id write/read + 16 B reordered write per point (~40 B/point) plus the cell array.
#include <math.h>

#include <stdlib.h>

#include <algorithm>
#include <chrono>
#include <cstdlib>

#include "common.cuh"

namespace {

__device__ __forceinline__ unsigned enc_f32(float f) {
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
static inline float dec_f32(unsigned u) {
  unsigned v = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  float f;
  memcpy(&f, &v, 4);
  return f;
}

// rows (stride floats) → float4 (x, y, z, 1)
__global__ void pack_points_kernel(const float *__restrict__ xyz, int n, int stride, bool vec4,
                                   float4 *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float *p = xyz + (size_t)i * stride;
  float4 v;
  if (vec4) {
    v = *reinterpret_cast<const float4 *>(p);
  } else {
    v.x = p[0];
    v.y = p[1];
    v.z = p[2];
  }
  v.w = 1.0f;
  out[i] = v;
}

// bounding box of the finite points + their count.  box: 6 encoded uints (min xyz, max xyz), cnt.
__global__ void bbox_kernel(const float4 *__restrict__ pts, int n, unsigned *__restrict__ box, int *__restrict__ cnt) {
  unsigned mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u};
  int c = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = pts[i];
    if (!finite3(p.x, p.y, p.z)) continue;
    ++c;
    unsigned e[3] = {enc_f32(p.x), enc_f32(p.y), enc_f32(p.z)};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = min(mn[a], e[a]);
      mx[a] = max(mx[a], e[a]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  // one set of global atomics per CTA (one per warp — 66 000 atomics on seven addresses for a 1 M-point cloud — made
  // this kernel 49 us)
  __shared__ unsigned s_mn[3], s_mx[3];
  __shared__ int s_c;
  if (threadIdx.x == 0) {
    s_mn[0] = s_mn[1] = s_mn[2] = 0xffffffffu;
    s_mx[0] = s_mx[1] = s_mx[2] = 0u;
    s_c = 0;
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      atomicMin(&s_mn[a], mn[a]);
      atomicMax(&s_mx[a], mx[a]);
    }
    if (c) atomicAdd(&s_c, c);
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    atomicMin(&box[threadIdx.x], s_mn[threadIdx.x]);
    atomicMax(&box[3 + threadIdx.x], s_mx[threadIdx.x]);
  }
  if (threadIdx.x == 3 && s_c) atomicAdd(cnt, s_c);
}

__global__ void cell_count_kernel(const float4 *__restrict__ pts, int n, GridView g, int *__restrict__ cell_of,
                                  int *__restrict__ counts) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = pts[i];
  int c = -1;
  if (finite3(p.x, p.y, p.z)) {
    int cx = grid_coord(p.x, g.lox, g.inv_h, g.dx);
    int cy = grid_coord(p.y, g.loy, g.inv_h, g.dy);
    int cz = grid_coord(p.z, g.loz, g.inv_h, g.dz);
    c = cx + g.dx * (cy + g.dy * cz);
    atomicAdd(&counts[c], 1);
  }
  cell_of[i] = c;
}

// counts[c] still holds the population of cell c; it is consumed as a down-counter.
__global__ void cell_scatter_kernel(const float4 *__restrict__ pts, int n, const int *__restrict__ cell_of,
                                    const int *__restrict__ cell_start, int *__restrict__ counts,
                                    float4 *__restrict__ sorted) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = cell_of[i];
  if (c < 0) return;
  int slot = cell_start[c] + atomicSub(&counts[c], 1) - 1;
  float4 p = pts[i];
  p.w = __int_as_float(i);
  sorted[slot] = p;
}

int build_grid(b200_cloud *c, float cell, DeviceGrid &g) {
  HostTrace tr;
  b200_ctx *ctx = c->ctx;
  StageScope st_(ctx, ST_GRID);
  g.valid = false;
  const float requested = cell;
  // bound the dense cell array: <= 2^25 cells
  float ext[3] = {c->hi[0] - c->lo[0], c->hi[1] - c->lo[1], c->hi[2] - c->lo[2]};
  if (!(cell > 0.f) || !isfinite(cell)) cell = 1.0f;
  int dim[3];
  for (;;) {
    double cells = 1.0;
    float inv_h = 1.0f / cell;
    for (int a = 0; a < 3; ++a) {
      double d = floor((double)ext[a] * (double)inv_h) + 2.0;
      cells *= d;
    }
    if (cells <= (double)(1 << 25)) break;
    cell *= 1.25f;
  }
  GridView v;
  v.h = cell;
  v.inv_h = 1.0f / cell;
  v.lox = c->lo[0];
  v.loy = c->lo[1];
  v.loz = c->lo[2];
  for (int a = 0; a < 3; ++a) {
    // same expression as grid_coord(hi) + 1
    float f = floorf((c->hi[a] - c->lo[a]) * v.inv_h);
    dim[a] = (int)f + 1;
    if (dim[a] < 1) dim[a] = 1;
  }
  v.dx = dim[0];
  v.dy = dim[1];
  v.dz = dim[2];
  v.n = c->n_valid;
  float sc = 0.f;
  for (int a = 0; a < 3; ++a) sc = std::max(sc, std::max(fabsf(c->lo[a]), fabsf(c->hi[a])));
  v.coord_scale = sc;
  const size_t ncell = (size_t)dim[0] * dim[1] * dim[2];
  tr.tick("grid setup");
  B200_TRY(g.cell_start.alloc(ctx, ncell + 1));
  tr.tick("alloc cell_start");
  B200_TRY(g.pts.alloc(ctx, (size_t)std::max(c->n_valid, 1)));
  DevBuf<int> counts, cell_of;
  B200_TRY(counts.alloc(ctx, ncell + 1));
  tr.tick("alloc counts");
  B200_TRY(counts.zero());
  B200_TRY(cell_of.alloc(ctx, (size_t)std::max(c->n, 1)));
  tr.tick("memset + alloc cell_of");
  v.pts = g.pts.p;
  v.raw = c->raw.p;
  v.cell_start = g.cell_start.p;
  if (c->n > 0) {
    cell_count_kernel<<<ceil_div(c->n, 256), 256, 0, ctx->stream>>>(c->raw.p, c->n, v, cell_of.p, counts.p);
    B200_LAUNCHED(ctx);
  }
  B200_TRY(exclusive_scan_i32(ctx, counts.p, g.cell_start.p, (int)(ncell + 1), nullptr));
  if (c->n > 0) {
    cell_scatter_kernel<<<ceil_div(c->n, 256), 256, 0, ctx->stream>>>(c->raw.p, c->n, cell_of.p, g.cell_start.p,
                                                                     counts.p, g.pts.p);
    B200_LAUNCHED(ctx);
  }
  tr.tick("grid kernels enqueue");
  if (tr.on) fprintf(stderr, "[b200 trace] grid %d x %d x %d cells, h=%g\n", dim[0], dim[1], dim[2], (double)cell);
  g.view = v;
  g.cell = requested;
  g.valid = true;
  return B200_OK;
}

}  // namespace

int pack_points(b200_ctx *ctx, const float *d_xyz, int n, int stride, float4 *d_out) {
  if (n <= 0) return B200_OK;
  const bool vec4 = (stride % 4 == 0) && (((uintptr_t)d_xyz & 15u) == 0);
  pack_points_kernel<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(d_xyz, n, stride, vec4, d_out);
  B200_LAUNCHED(ctx);
  return B200_OK;
}

int cloud_upload(b200_ctx *ctx, const float *xyz, int n, int stride, bool on_device, std::unique_ptr<b200_cloud> &out) {
  if (n < 0 || stride < 3 || (n > 0 && !xyz)) return ctx->fail(B200_ERR_INVALID, "cloud_create: bad arguments");
  std::unique_ptr<b200_cloud> c(new (std::nothrow) b200_cloud());
  if (!c) return ctx->fail(B200_ERR_NOMEM, "cloud_create: out of host memory");
  c->ctx = ctx;
  c->n = n;
  B200_TRY(c->raw.alloc(ctx, (size_t)std::max(n, 1)));
  if (n > 0) {
    if (on_device) {
      B200_TRY(pack_points(ctx, xyz, n, stride, c->raw.p));
    } else {
      DevBuf<float> stage;
      B200_TRY(stage.alloc(ctx, (size_t)n * stride));
      B200_CUDA(ctx, cudaMemcpyAsync(stage.p, xyz, (size_t)n * stride * sizeof(float), cudaMemcpyHostToDevice,
                                     ctx->stream));
      B200_TRY(pack_points(ctx, stage.p, n, stride, c->raw.p));
    }
  }
  // bounding box + finite count (one 28-byte readback; the grid dimensions are sized on the host)
  DevBuf<unsigned> box;
  B200_TRY(box.alloc(ctx, 8));
  unsigned init[8] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u, 0u, 0u};
  B200_TRY(write_small(ctx, box.p, init, sizeof(init)));
  if (n > 0) {
    int blocks = std::min(ceil_div(n, 256), ctx->sm_count * 4);
    bbox_kernel<<<blocks, 256, 0, ctx->stream>>>(c->raw.p, n, box.p, reinterpret_cast<int *>(box.p + 6));
    B200_LAUNCHED(ctx);
  }
  unsigned hbox[8];
  B200_TRY(readback_small(ctx, box.p, hbox, sizeof(hbox)));
  c->n_valid = (int)hbox[6];
  if (c->n_valid > 0) {
    for (int a = 0; a < 3; ++a) {
      c->lo[a] = dec_f32(hbox[a]);
      c->hi[a] = dec_f32(hbox[3 + a]);
    }
  } else {
    for (int a = 0; a < 3; ++a) c->lo[a] = c->hi[a] = 0.f;
  }
  out = std::move(c);
  return B200_OK;
}

// Cell edge for k-nearest queries: non-empty cells should hold about k/2 points of a surface-like
// cloud, so that the 3x3x3 block around a query usually certifies the k nearest in one ring.
int cloud_grid_for_knn(b200_cloud *c, int k, const GridView **out) {
  if (!c->knn_grid.valid || c->knn_grid_k != k) {
    float ext[3] = {c->hi[0] - c->lo[0], c->hi[1] - c->lo[1], c->hi[2] - c->lo[2]};
    std::sort(ext, ext + 3);
    double area = std::max((double)ext[2] * (double)ext[1], 1e-12);
    // about k points per (flat-surface) cell: measured on the 1 M-point scene, k = 20: 0.5 k -> 1.95 ms, 0.7 k -> 1.42,
    // 1.0 k -> 1.35, 1.5 k -> 1.58, 3 k -> 1.89 (smaller cells need the second ring too often, larger ones scan more);
    // with the heap and the slab pruning of search.cuh: 0.5 k -> 1.24, 0.7 k -> 1.09, 1.0 k -> 1.03, 1.4 k -> 1.09,
    // 2 k -> 1.16, 3 k -> 1.28
    double target = std::max(2.0, 1.0 * k);
    float cell = (float)sqrt(area * target / std::max(c->n_valid, 1));
    B200_TRY(build_grid(c, cell, c->knn_grid));
    c->knn_grid_k = k;
  }
  *out = &c->knn_grid.view;
  return B200_OK;
}

// Cell edge for radius queries: the radius itself (27-cell stencil), but never so small that cells
// are mostly empty, nor so large that one cell holds the whole cloud when the radius is huge
// (SHOT_demo.cpp:498 uses radius 50 on a 0.6 m model: the support is the entire model).
int cloud_grid_for_radius(b200_cloud *c, double radius, const GridView **out) {
  float ext[3] = {c->hi[0] - c->lo[0], c->hi[1] - c->lo[1], c->hi[2] - c->lo[2]};
  std::sort(ext, ext + 3);
  double area = std::max((double)ext[2] * (double)ext[1], 1e-12);
  // edge at which a surface cell would hold ~8 points
  float dens_cell = (float)sqrt(area * 8.0 / std::max(c->n_valid, 1));
  // cell edge = radius (3 x 3 x 3 stencil).  Measured on the 1 M-point scene, r = 0.02: edge r / 1.5, r / 2, r / 3 scan
  // fewer candidates but more and shorter rows: SHOT 0.95 -> 0.98, 1.02, 1.16 ms.
  float cell = (float)radius;
  if (!(cell > 0.f)) cell = dens_cell;
  cell = std::max(cell, 0.5f * dens_cell);
  float maxext = std::max(ext[2], 1e-6f);
  cell = std::min(cell, std::max(maxext / 4.0f, dens_cell));
  if (!c->radius_grid.valid || fabsf(c->radius_grid.cell - cell) > 1e-3f * cell) {  // cell = requested edge
    B200_TRY(build_grid(c, cell, c->radius_grid));
  }
  *out = &c->radius_grid.view;
  return B200_OK;
}
