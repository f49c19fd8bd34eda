// normals.cu — per-point surface normals + curvature.
//
// Replaces pcl::NormalEstimationOMP<PointXYZRGBA, Normal>::compute as called at SHOT.cpp:302-308
// (k = 40), 6Dpose.cpp:275-278 (k = 10), SHOT_demo.cpp:405-411 (k = 50), SHOT_scenes.cpp:285-291
// (k = 20), CAD_desc.cpp:283-289 and, with setRadiusSearch, FPFH_demo.cpp:416-420 (r = 0.15) and
// FPFH_scenes_clustered.cpp:273-277 (r = 0.05).
//
// Arithmetic follows PCL 1.8: single-pass float32 mean/covariance with nine accumulators summed in
// neighbour order (nearest first), closed-form eigen33 for the smallest eigenvector, curvature =
// |lambda0 / trace|, flip towards the viewpoint.  The float32 sums are evaluated as the same
// mul/add sequence (the library is built with --fmad=false), so the covariance is bit-identical to
// the CPU evaluation; only the libm calls inside eigen33 (atan2f/cosf/sinf) can differ by an ulp.
//
// kNN mode: one query per thread, queries visited in cell order so a warp's threads share their
// candidate cells through L1; the k best candidates live in shared memory as a max-heap (search.cuh: 1.35 -> 1.17 ms
// against round 1's sorted list).  Radius mode: one query per
// CTA (gather → sort → accumulate).  Algorithmic HBM traffic: 16 B read + 16 B written per point.
//
// Round 2 measured three cooperative rewrites of the kNN kernel against this one on the 1 M-point scene, k = 20
// (all bit-identical to it; numbers in DESIGN.md section 4): a cell's candidate box staged once in shared memory and
// (a) a whole warp per query with a counted cut + rank sort: 1.83 ms, 909 M warp instructions; (b) 8-lane sub-groups
// with a bitonic sort: 2.45 ms, 1 331 M; (c) one query per thread with a density-estimated cut instead of the sorted
// insertion: 2.4-3.5 ms — against 1.35 ms and 893 M here.  The ballot/compaction bookkeeping of the cooperative
// forms costs about one warp instruction per candidate-query pair, more than the per-thread insertion they remove
// (62 % of this kernel's instructions, search.cuh), so the per-thread kernel stays.  A two-pass form of the search (the K
// smallest distances in registers, then a second pass collecting the winners) measured 1.45 ms against this kernel's
// 1.32 ms (DESIGN.md section 4).
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "pcl_eigen33.cuh"
#include "search.cuh"

namespace {

struct Normal4 {
  float nx, ny, nz, curv;
};

// accu: the nine sums already divided by the neighbour count.  PCL computePointNormal →
// solvePlaneParameters → eigen33 → flipNormalTowardsViewpoint.
__device__ inline Normal4 normal_from_accu(const float accu[9], float px, float py, float pz, float vpx, float vpy,
                                           float vpz) {
  float cov[9];
  cov[0] = accu[0] - accu[6] * accu[6];
  cov[1] = accu[1] - accu[6] * accu[7];
  cov[2] = accu[2] - accu[6] * accu[8];
  cov[4] = accu[3] - accu[7] * accu[7];
  cov[5] = accu[4] - accu[7] * accu[8];
  cov[8] = accu[5] - accu[8] * accu[8];
  cov[3] = cov[1];
  cov[6] = cov[2];
  cov[7] = cov[5];
  float scale = 0.0f;
#pragma unroll
  for (int i = 0; i < 9; ++i) scale = fmaxf(scale, fabsf(cov[i]));
  if (scale <= 1.17549435e-38f) scale = 1.0f;  // FLT_MIN
  float m[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) m[i] = cov[i] / scale;
  float roots[3];
  compute_roots(m, roots);
  const float eigenvalue = roots[0] * scale;
  m[0] -= roots[0];
  m[4] -= roots[0];
  m[8] -= roots[0];
  float v1[3], v2[3], v3[3];
  cross3(&m[0], &m[3], v1);
  cross3(&m[0], &m[6], v2);
  cross3(&m[3], &m[6], v3);
  const float l1 = v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2];
  const float l2 = v2[0] * v2[0] + v2[1] * v2[1] + v2[2] * v2[2];
  const float l3 = v3[0] * v3[0] + v3[1] * v3[1] + v3[2] * v3[2];
  float vx, vy, vz, l;
  if (l1 >= l2 && l1 >= l3) {
    vx = v1[0], vy = v1[1], vz = v1[2], l = l1;
  } else if (l2 >= l1 && l2 >= l3) {
    vx = v2[0], vy = v2[1], vz = v2[2], l = l2;
  } else {
    vx = v3[0], vy = v3[1], vz = v3[2], l = l3;
  }
  const float s = sqrtf(l);
  Normal4 r;
  r.nx = vx / s;
  r.ny = vy / s;
  r.nz = vz / s;
  const float eig_sum = cov[0] + cov[4] + cov[8];
  r.curv = (eig_sum != 0.0f) ? fabsf(eigenvalue / eig_sum) : 0.0f;
  const float dx = vpx - px, dy = vpy - py, dz = vpz - pz;
  const float cos_theta = (dx * r.nx + dy * r.ny + dz * r.nz);
  if (cos_theta < 0.0f) {
    r.nx *= -1.0f;
    r.ny *= -1.0f;
    r.nz *= -1.0f;
  }
  return r;
}

__global__ void fill_nan_kernel(float *p, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = nanf32();
}

// kNN mode.  q == nullptr: the queries are the indexed surface points themselves, visited in cell
// order (thread i takes g.pts[i]); results are scattered to the original row.
__global__ void normals_knn_kernel(GridView g, const float4 *__restrict__ q, int nq, int k, float vpx, float vpy,
                                   float vpz, float4 *__restrict__ out) {
  extern __shared__ unsigned char smem_raw[];
  const int T = blockDim.x;
  unsigned long long *sk = reinterpret_cast<unsigned long long *>(smem_raw) + threadIdx.x;
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= nq) return;
  float4 p;
  int dst;
  if (q) {
    p = q[i];
    dst = i;
  } else {
    p = g.pts[i];
    dst = orig_index(p);
  }
  float4 o = make_float4(nanf32(), nanf32(), nanf32(), nanf32());
  if (finite3(p.x, p.y, p.z)) {
    const int cnt = knn_query(g, p.x, p.y, p.z, k, sk, T);
    if (cnt >= 3) {
      float accu[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int j = 0; j < cnt; ++j) {
        const float4 n = g.raw[key_orig(sk[j * T])];
        accu[0] += n.x * n.x;
        accu[1] += n.x * n.y;
        accu[2] += n.x * n.z;
        accu[3] += n.y * n.y;
        accu[4] += n.y * n.z;
        accu[5] += n.z * n.z;
        accu[6] += n.x;
        accu[7] += n.y;
        accu[8] += n.z;
      }
      const float fn = (float)cnt;
#pragma unroll
      for (int a = 0; a < 9; ++a) accu[a] = accu[a] / fn;
      const Normal4 r = normal_from_accu(accu, p.x, p.y, p.z, vpx, vpy, vpz);
      o = make_float4(r.nx, r.ny, r.nz, r.curv);
    }
  }
  out[dst] = o;
}

// radius mode: one query per CTA.  The sorted neighbour list is walked by nine lanes, one per
// accumulator, so each sum keeps PCL's sequential order.
__global__ void __launch_bounds__(128) normals_radius_kernel(GridView g, const float4 *__restrict__ q, int nq,
                                                             float radius, float r2, int cap,
                                                             unsigned long long *glob_key, int *glob_pos, float vpx,
                                                             float vpy, float vpz, float4 *__restrict__ out,
                                                             const int *__restrict__ counts, int min_count) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_count;
  __shared__ float4 s_pts[128];
  unsigned long long *key;
  int *pos;
  cta_list(smem_raw, glob_key, glob_pos, cap, key, pos);
  for (int i = blockIdx.x; i < nq; i += gridDim.x) {
    if (counts[i] < min_count) continue;  // done by normals_radius_warp_kernel
    const float4 p = q[i];
    int n = gather_radius(g, p.x, p.y, p.z, radius, r2, key, pos, cap, &s_count);
    if (n > cap) n = cap;
    bitonic_sort(key, pos, n);
    // the nine float32 sums run sequentially in PCL's (d2, index) order, one lane each; the points are staged 128
    // at a time by the whole CTA so that their loads are in flight together instead of one per loop step
    float acc = 0.0f;
    for (int c0 = 0; c0 < n && n >= 3; c0 += 128) {
      const int m = min(128, n - c0);
      if ((int)threadIdx.x < m) s_pts[threadIdx.x] = g.pts[pos[c0 + threadIdx.x]];
      __syncthreads();
      if (threadIdx.x < 9) {
        const int lane = threadIdx.x;
        for (int j = 0; j < m; ++j) {
          const float4 v = s_pts[j];
          float a, b;
          switch (lane) {
            case 0: a = v.x, b = v.x; break;
            case 1: a = v.x, b = v.y; break;
            case 2: a = v.x, b = v.z; break;
            case 3: a = v.y, b = v.y; break;
            case 4: a = v.y, b = v.z; break;
            case 5: a = v.z, b = v.z; break;
            case 6: a = v.x, b = 1.0f; break;
            case 7: a = v.y, b = 1.0f; break;
            default: a = v.z, b = 1.0f; break;
          }
          acc += (lane < 6) ? a * b : a;
        }
      }
      __syncthreads();
    }
    if (threadIdx.x < 32) {
      const int lane = threadIdx.x;
      if (n >= 3 && lane < 9) acc = acc / (float)n;
      float accu[9];
#pragma unroll
      for (int a = 0; a < 9; ++a) accu[a] = __shfl_sync(0xffffffffu, acc, a);
      if (lane == 0) {
        float4 o = make_float4(nanf32(), nanf32(), nanf32(), nanf32());
        if (n >= 3) {
          const Normal4 r = normal_from_accu(accu, p.x, p.y, p.z, vpx, vpy, vpz);
          o = make_float4(r.nx, r.ny, r.nz, r.curv);
        }
        out[i] = o;
      }
    }
    __syncthreads();
  }
}


// radius mode, one query per WARP (neighbourhoods of up to CAP points; larger ones are left to the CTA kernel above).
// The CTA form spends most of a query's time with 119 of its 128 threads waiting: block-wide barriers between the
// 28-36 stages of the sort, and the nine sequential float32 sums at the end.  Here a warp gathers its query's
// neighbours into its own slice of shared memory (four 32-point chunks per trip, ballot compaction), orders the
// (d2, index) keys with a bitonic network synchronised by __syncwarp only, stages the points in that order and lets
// nine lanes run PCL's nine sums — each still strictly in (d2, index) order, so the covariance is the same bit for
// bit — while the SM's other warps work on their own queries.  Measured times: DESIGN.md section 4.
constexpr int NRW_WARPS = 8;
template <int CAP>
struct NrwSmem {
  unsigned long long key[CAP];
  float4 pts[CAP];
  int pos[CAP];
};

template <int CAP>
__global__ void __launch_bounds__(NRW_WARPS * 32)
    normals_radius_warp_kernel(GridView g, const float4 *__restrict__ q, int nq, float radius, float r2,
                               const int *__restrict__ counts, float vpx, float vpy, float vpz, float4 *__restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  NrwSmem<CAP> &sm = reinterpret_cast<NrwSmem<CAP> *>(smem_raw)[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * NRW_WARPS;
  const float4 *__restrict__ pts = g.pts;
  // which components of a staged point (x, y, z, 1) this lane multiplies: xx xy xz yy yz zz x y z
  const int ia = (lane < 3) ? 0 : (lane < 5) ? 1 : (lane == 5) ? 2 : (lane < 9 ? lane - 6 : 0);
  const int ib = (lane < 3) ? lane : (lane < 5) ? lane - 2 : (lane == 5) ? 2 : 3;
  for (int i = blockIdx.x * NRW_WARPS + (threadIdx.x >> 5); i < nq; i += nwarps) {
    const int cnt = counts[i];
    if (cnt > CAP) continue;  // the CTA kernel's
    const float4 c = q[i];
    if (cnt < 3) {  // search failure or computePointNormal: fewer than three neighbours
      if (lane == 0) out[i] = make_float4(nanf32(), nanf32(), nanf32(), nanf32());
      continue;
    }
    // ---- gather (cnt <= CAP neighbours), then order by (d2, index): FLANN's result order
    const int n = warp_gather_radius<CAP>(g, c, radius, r2, sm.key, sm.pos, lane);
    warp_bitonic_sort(sm.key, sm.pos, n, lane);
    // ---- the points in that order (w = 1: the plain sums read it as their second factor)
    for (int t = lane; t < n; t += 32) {
      const float4 v = pts[sm.pos[t]];
      sm.pts[t] = make_float4(v.x, v.y, v.z, 1.0f);
    }
    __syncwarp();
    // ---- nine sequential float32 sums, one lane each
    float acc = 0.0f;
    if (lane < 9) {
      const float *sp = reinterpret_cast<const float *>(sm.pts);
      for (int j = 0; j < n; ++j) {
        const float a = sp[4 * j + ia], b = sp[4 * j + ib];
        acc += (lane < 6) ? a * b : a;
      }
      acc = acc / (float)n;
    }
    float accu[9];
#pragma unroll
    for (int a = 0; a < 9; ++a) accu[a] = __shfl_sync(0xffffffffu, acc, a);
    if (lane == 0) {
      const Normal4 r = normal_from_accu(accu, c.x, c.y, c.z, vpx, vpy, vpz);
      out[i] = make_float4(r.nx, r.ny, r.nz, r.curv);
    }
    __syncwarp();
  }
}

template <int CAP>
int launch_normals_radius_warp(b200_ctx *ctx, const GridView &g, const float4 *d_q, int nq, float radius, float r2,
                               const int *d_counts, float vpx, float vpy, float vpz, float4 *out) {
  const size_t smem = sizeof(NrwSmem<CAP>) * NRW_WARPS;
  B200_CUDA(ctx, ensure_dyn_smem(normals_radius_warp_kernel<CAP>, smem));
  const int grid = std::min(ceil_div(nq, NRW_WARPS), ctx->sm_count * 16);
  normals_radius_warp_kernel<CAP><<<grid, NRW_WARPS * 32, smem, ctx->stream>>>(g, d_q, nq, radius, r2, d_counts, vpx, vpy, vpz,
                                                                              out);
  B200_LAUNCHED(ctx);
  return B200_OK;
}

}  // namespace

int dev_normals(b200_ctx *ctx, b200_cloud *c, const float4 *d_q, int nq, bool q_is_surface, int k, double radius,
                const float *vp, float *d_out) {
  // Feature::initCompute: exactly one of k / radius must be set
  if ((k != 0) == (radius != 0.0) || k < 0 || radius < 0.0)
    return ctx->fail(B200_ERR_INVALID, "normals: exactly one of k / radius must be non-zero");
  if (nq <= 0) return B200_OK;
  const float vpx = vp ? vp[0] : 0.f, vpy = vp ? vp[1] : 0.f, vpz = vp ? vp[2] : 0.f;
  float4 *out = reinterpret_cast<float4 *>(d_out);
  if (k) {
    if (k > 1024) return ctx->fail(B200_ERR_INVALID, "normals: k must be <= 1024");
    const GridView *g;
    B200_TRY(cloud_grid_for_knn(c, k, &g));
    size_t smem;
    const int T = knn_threads_for(k, &smem);
    if (smem > ctx->smem_optin) return ctx->fail(B200_ERR_INVALID, "normals: k too large for shared memory");
    B200_CUDA(ctx, ensure_dyn_smem(normals_knn_kernel, smem));
    StageScope st_(ctx, ST_NORMALS);
    if (q_is_surface) {
      // rows with non-finite coordinates are not in the grid: they keep NaN normals (PCL: is_dense=false)
      if (c->n_valid < c->n) {
        fill_nan_kernel<<<ceil_div((long long)c->n * 4, 256), 256, 0, ctx->stream>>>(d_out, (size_t)c->n * 4);
        B200_LAUNCHED(ctx);
      }
      if (c->n_valid > 0) {
        normals_knn_kernel<<<ceil_div(c->n_valid, T), T, smem, ctx->stream>>>(*g, nullptr, c->n_valid, k, vpx, vpy, vpz,
                                                                              out);
        B200_LAUNCHED(ctx);
      }
    } else {
      normals_knn_kernel<<<ceil_div(nq, T), T, smem, ctx->stream>>>(*g, d_q, nq, k, vpx, vpy, vpz, out);
      B200_LAUNCHED(ctx);
    }
    return B200_OK;
  }
  // radius mode
  const GridView *g;
  B200_TRY(cloud_grid_for_radius(c, radius, &g));
  DevBuf<int> counts;
  DevBuf<unsigned long long> stats;
  B200_TRY(counts.alloc(ctx, (size_t)nq));
  B200_TRY(stats.alloc(ctx, 8));
  B200_TRY(dev_radius_count(ctx, *g, d_q, nq, radius, counts.p, stats.p));
  unsigned long long hstats[2];
  B200_TRY(readback_small(ctx, stats.p, hstats, sizeof(hstats)));
  const int max_count = (int)hstats[0];
  ctx->last_max_nbrs = max_count;
  ctx->last_mean_nbrs = (double)hstats[1] / nq;
  const float r2 = (float)(radius * radius);
  StageScope st_(ctx, ST_NORMALS);
  // neighbourhoods of up to 256 points: one query per warp (B200_NORMALS_RADIUS=cta: everything by the CTA kernel)
  constexpr int WCAP = 256;
  const char *sel = getenv("B200_NORMALS_RADIUS");
  const bool warp_path = !(sel && !strcmp(sel, "cta"));
  if (warp_path) {
    if (max_count <= 64)
      B200_TRY(launch_normals_radius_warp<64>(ctx, *g, d_q, nq, (float)radius, r2, counts.p, vpx, vpy, vpz, out));
    else if (max_count <= 128)
      B200_TRY(launch_normals_radius_warp<128>(ctx, *g, d_q, nq, (float)radius, r2, counts.p, vpx, vpy, vpz, out));
    else
      B200_TRY(launch_normals_radius_warp<WCAP>(ctx, *g, d_q, nq, (float)radius, r2, counts.p, vpx, vpy, vpz, out));
    if (max_count <= WCAP) return B200_OK;
  }
  const int min_count = warp_path ? WCAP + 1 : 0;
  const int cap = next_pow2_host(std::max(max_count, 32));
  const size_t smem = (size_t)cap * 12;
  if (smem <= 96 * 1024) {
    B200_CUDA(ctx,
              ensure_dyn_smem(normals_radius_kernel, smem));
    const int grid = std::min(nq, ctx->sm_count * 8);
    normals_radius_kernel<<<grid, 128, smem, ctx->stream>>>(*g, d_q, nq, (float)radius, r2, cap, nullptr, nullptr, vpx,
                                                            vpy, vpz, out, counts.p, min_count);
    B200_LAUNCHED(ctx);
  } else {
    const int grid = std::min(nq, ctx->sm_count * 2);
    DevBuf<unsigned long long> gk;
    DevBuf<int> gp;
    B200_TRY(gk.alloc(ctx, (size_t)grid * cap));
    B200_TRY(gp.alloc(ctx, (size_t)grid * cap));
    normals_radius_kernel<<<grid, 128, 0, ctx->stream>>>(*g, d_q, nq, (float)radius, r2, cap, gk.p, gp.p, vpx, vpy,
                                                         vpz, out, counts.p, min_count);
    B200_LAUNCHED(ctx);
  }
  return B200_OK;
}
