// fpfh.cu — 33-bin Fast Point Feature Histograms.
//
// Replaces pcl::FPFHEstimation / FPFHEstimationOMP <PointXYZRGBA, Normal, FPFHSignature33>::compute
// (FPFH_demo.cpp:422-428 and 505-510, FPFH_scenes_clustered.cpp:287-293 and 379-387).
//
// Pass 1 (computeSPFHSignatures): for every surface point that is a neighbour of some query (all
// points when input == surface, as at every reference call site) the Darboux pair features
// (pcl::computePairFeatures, float32) of its neighbourhood are binned into 3 x 11 bins.  Each hit adds
// the same increment 100/(n-1), so the bins are counted as integers in shared memory (warp-level
// atomics, order independent) and the float32 value PCL reaches by repeated addition is rebuilt
// exactly from the count.
// Pass 2 (weightPointSPFHSignature): FPFH(p) = sum over neighbours (d2 != 0) of SPFH(q)/d2, walked in
// the (d2, index) order FLANN returns so each float32 bin sum keeps PCL's sequence (one lane per
// bin), then every 11-bin block is rescaled to sum 100 with the float64 running sums kept in PCL's
// order (one lane per block).
//
// Kernels: one point per WARP for neighbourhoods of up to 256 points (spfh_warp_kernel, fpfh_weight_warp_kernel: 1.38 ->
// 0.66 ms on the FPFH_demo configuration, 59 066 points with 97 neighbours on average), one point per CTA beyond that;
// the two forms are bit-identical (B200_FPFH=cta selects the CTA kernels for everything; the tests compare them).
//
// Algorithmic HBM traffic per descriptor (surface == keypoints): 32 B point+normal read, 132 B SPFH
// written and re-read, 132 B FPFH written: ~428 B (SURVEY.md §8(d)).
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "search.cuh"

namespace {

constexpr int FPFH_THREADS = 128;

__global__ void gather_normals_sorted_kernel(const float4 *__restrict__ sorted_pts, int n,
                                             const float4 *__restrict__ normals, float4 *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = normals[orig_index(sorted_pts[i])];
}

__global__ void fill_int_kernel(int *p, int n, int v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// mark every surface point that lies in the neighbourhood of a query
__global__ void __launch_bounds__(FPFH_THREADS)
    fpfh_mark_kernel(GridView g, const float4 *__restrict__ q, int nq, float radius, float r2, int *__restrict__ need) {
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= nq) return;
  const float4 c = q[w];
  int x0, x1, y0, y1, z0, z1;
  if (!finite3(c.x, c.y, c.z) || g.n == 0 || !ball_cell_range(g, c.x, c.y, c.z, radius, x0, x1, y0, y1, z0, z1)) return;
  for (int z = z0; z <= z1; ++z)
    for (int y = y0; y <= y1; ++y) {
      const int base = g.dx * (y + g.dy * z);
      const int s = g.cell_start[base + x0], e = g.cell_start[base + x1 + 1];
      for (int j = s + lane; j < e; j += 32) {
        const float4 p = g.pts[j];
        if (sqdist3(c.x, c.y, c.z, p.x, p.y, p.z) < r2) need[j] = 1;  // indexed by sorted position
      }
    }
}

// pcl::computePairFeatures (features/src/pfh.cpp), float32.  Degenerate pairs yield f1=f2=f3=0
// (FPFHEstimation::computePairFeatures ignores the return value and still bins them).
__device__ inline void pair_features(const float4 &p1, const float4 &n1, const float4 &p2, const float4 &n2,
                                     float &f1, float &f2, float &f3) {
  float dx = p2.x - p1.x, dy = p2.y - p1.y, dz = p2.z - p1.z;
  float s = dx * dx;
  s += dy * dy;
  s += dz * dz;
  const float f4 = sqrtf(s);
  if (f4 == 0.0f) {
    f1 = f2 = f3 = 0.0f;
    return;
  }
  float ax = n1.x, ay = n1.y, az = n1.z;  // n1_copy
  float bx = n2.x, by = n2.y, bz = n2.z;  // n2_copy
  float t = ax * dx;
  t += ay * dy;
  t += az * dz;
  const float angle1 = t / f4;
  t = bx * dx;
  t += by * dy;
  t += bz * dz;
  const float angle2 = t / f4;
  if (acos((double)fabsf(angle1)) > acos((double)fabsf(angle2))) {
    ax = n2.x, ay = n2.y, az = n2.z;
    bx = n1.x, by = n1.y, bz = n1.z;
    dx *= -1.0f;
    dy *= -1.0f;
    dz *= -1.0f;
    f3 = -angle2;
  } else {
    f3 = angle1;
  }
  // v = dp x n1
  float vx = dy * az - dz * ay;
  float vy = dz * ax - dx * az;
  float vz = dx * ay - dy * ax;
  s = vx * vx;
  s += vy * vy;
  s += vz * vz;
  const float v_norm = sqrtf(s);
  if (v_norm == 0.0f) {
    f1 = f2 = f3 = 0.0f;
    return;
  }
  vx /= v_norm;
  vy /= v_norm;
  vz /= v_norm;
  // w = n1 x v
  const float wx = ay * vz - az * vy;
  const float wy = az * vx - ax * vz;
  const float wz = ax * vy - ay * vx;
  t = vx * bx;
  t += vy * by;
  t += vz * bz;
  f2 = t;
  float wn = wx * bx;
  wn += wy * by;
  wn += wz * bz;
  float nn = ax * bx;
  nn += ay * by;
  nn += az * bz;
  f1 = (float)atan2((double)wn, (double)nn);  // correctly rounded stand-in for atan2f
}

__device__ __forceinline__ int clamp_bin(double x) {
  const double f = floor(x);
  int h;
  if (!(f == f) || f >= 2147483648.0 || f < -2147483648.0)
    h = -1;  // static_cast<int> of NaN / out of range gives INT_MIN on x86 → clamps to 0
  else
    h = (int)f;
  if (h < 0) h = 0;
  if (h >= 11) h = 10;
  return h;
}

// Pass 1: one surface point (in cell order) per CTA.  spfh is indexed by ORIGINAL row.
__global__ void __launch_bounds__(FPFH_THREADS)
    spfh_kernel(GridView g, const float4 *__restrict__ nrm, const int *__restrict__ need, float radius, float r2,
                int cap, unsigned long long *glob_key, int *glob_pos, float *__restrict__ spfh,
                const int *__restrict__ counts, int min_count) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_count;
  __shared__ int s_bins[33];
  unsigned long long *key;
  int *pos;
  cta_list(smem_raw, glob_key, glob_pos, cap, key, pos);
  const int tid = threadIdx.x;
  const double kPi = 3.14159265358979323846;
  const float d_pi = 1.0f / (2.0f * (float)kPi);
  for (int s = blockIdx.x; s < g.n; s += gridDim.x) {
    if (!need[s] || counts[s] < min_count) continue;  // block-uniform (smaller neighbourhoods: spfh_warp_kernel)
    const float4 p = g.pts[s];
    const float4 np = nrm[s];
    int n = gather_radius(g, p.x, p.y, p.z, radius, r2, key, pos, cap, &s_count);
    if (n > cap) n = cap;
    if (tid < 33) s_bins[tid] = 0;
    __syncthreads();
    for (int j = tid; j < n; j += FPFH_THREADS) {
      const int pj = pos[j];
      if (pj == s) continue;  // p_idx == indices[idx]
      float f1, f2, f3;
      pair_features(p, np, g.pts[pj], nrm[pj], f1, f2, f3);
      atomicAdd(&s_bins[clamp_bin(11 * (((double)f1 + kPi) * (double)d_pi))], 1);
      atomicAdd(&s_bins[11 + clamp_bin(11 * (((double)f2 + 1.0) * 0.5))], 1);
      atomicAdd(&s_bins[22 + clamp_bin(11 * (((double)f3 + 1.0) * 0.5))], 1);
    }
    __syncthreads();
    if (tid < 33) {
      // n == 0 cannot happen (the point finds itself); PCL would leave the row at zero
      const float hist_incr = 100.0f / (float)(n - 1);
      float v = 0.0f;
      const int cnt = s_bins[tid];
      for (int t = 0; t < cnt; ++t) v += hist_incr;
      spfh[(size_t)orig_index(p) * 33 + tid] = v;
    }
    __syncthreads();
  }
}

// Pass 2: one query per CTA.
__global__ void __launch_bounds__(FPFH_THREADS)
    fpfh_weight_kernel(GridView g, const float4 *__restrict__ q, int nq, float radius, float r2, int cap,
                       unsigned long long *glob_key, int *glob_pos, const float *__restrict__ spfh,
                       float *__restrict__ out, const int *__restrict__ counts, int min_count, int rows_by_w) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_count;
  __shared__ double s_sum[3];
  __shared__ double s_part[FPFH_THREADS / 32][3];
  __shared__ float s_tile[32 * 33];
  unsigned long long *key;
  int *pos;
  cta_list(smem_raw, glob_key, glob_pos, cap, key, pos);
  const int tid = threadIdx.x;
  for (int i = blockIdx.x; i < nq; i += gridDim.x) {
    if (counts[i] < min_count) continue;  // smaller neighbourhoods: fpfh_weight_warp_kernel
    const float4 c = q[i];
    const size_t row = rows_by_w ? (size_t)orig_index(c) : (size_t)i;  // surface mode: q is the cell-ordered surface
    int n = gather_radius(g, c.x, c.y, c.z, radius, r2, key, pos, cap, &s_count);
    if (n > cap) n = cap;
    bitonic_sort(key, pos, n);
    // Products spfh[neighbour][bin] * (1 / d2) are staged 32 neighbours at a time by the whole CTA (independent
    // loads in flight together), then
    //  - one lane per bin adds them in float32, sequentially in PCL's (d2, index) order (the weighted histogram);
    //  - every thread adds the products it staged into float64 partial sums of the three 11-bin blocks (PCL adds
    //    the same float products into a double neighbour by neighbour; the double sum is exact to ~1e-16 either
    //    way and only its float32 cast is used).
    double part[3] = {0.0, 0.0, 0.0};
    float acc = 0.0f;
    for (int c0 = 0; c0 < n; c0 += 32) {
      const int m = min(32, n - c0);
      for (int idx = tid; idx < m * 33; idx += FPFH_THREADS) {
        const int jj = idx / 33, b = idx - jj * 33;
        const unsigned long long kj = key[c0 + jj];
        const float d2 = key_d2(kj);
        float val = 0.0f;  // d2 == 0: PCL skips the neighbour (adding +0 leaves the non-negative sums unchanged)
        if (d2 != 0.0f) {
          const float weight = 1.0f / d2;
          val = spfh[(size_t)key_orig(kj) * 33 + b] * weight;
          part[b / 11] += (double)val;
        }
        s_tile[idx] = val;
      }
      __syncthreads();
      if (tid < 33)
        for (int jj = 0; jj < m; ++jj) acc += s_tile[jj * 33 + tid];
      __syncthreads();
    }
#pragma unroll
    for (int f = 0; f < 3; ++f) part[f] = warp_sum(part[f]);
    if ((tid & 31) == 0) {
#pragma unroll
      for (int f = 0; f < 3; ++f) s_part[tid >> 5][f] = part[f];
    }
    __syncthreads();
    if (tid < 3) {
      double sum = 0.0;
#pragma unroll
      for (int w = 0; w < FPFH_THREADS / 32; ++w) sum += s_part[w][tid];
      if (sum != 0) sum = 100.0 / sum;
      s_sum[tid] = sum;
    }
    __syncthreads();
    if (tid < 33) {
      float v = acc * (float)s_sum[tid / 11];
      if (n == 0) v = nanf32();  // searchForNeighbors == 0 → NaN row
      out[row * 33 + tid] = v;
    }
    __syncthreads();
  }
}


// ---- one point per WARP (neighbourhoods of up to FW_CAP points; larger ones stay with the CTA kernels above) --------
// The CTA kernels keep 128 threads on one point through block-wide barriers: around the gather, between the 28-36
// stages of the sort, and around the sequential float32 sums that a few lanes run while the rest wait.  Here a warp
// owns the point: ballot-compacted gather into its slice of shared memory, __syncwarp-only bitonic sort, the
// sequential sums on 11 lanes (three bins each: one per 11-bin block, so the lane's three float64 partial sums are
// the three block sums' shares) while the SM's other warps work on their own points.  Same arithmetic in the same
// order: the results are the CTA kernels' bit for bit.
constexpr int FW_CAP = 256;
constexpr int FW_WARPS = 8;
struct FwSmem {
  unsigned long long key[FW_CAP];
  int pos[FW_CAP];
  int bins[36];
};

// Pass 1 for surface points (cell order) with need[s] and at most FW_CAP neighbours
__global__ void __launch_bounds__(FW_WARPS * 32)
    spfh_warp_kernel(GridView g, const float4 *__restrict__ nrm, const int *__restrict__ need,
                     const int *__restrict__ counts, float radius, float r2, float *__restrict__ spfh) {
  __shared__ FwSmem s_all[FW_WARPS];
  FwSmem &sm = s_all[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * FW_WARPS;
  const double kPi = 3.14159265358979323846;
  const float d_pi = 1.0f / (2.0f * (float)kPi);
  for (int s = blockIdx.x * FW_WARPS + (threadIdx.x >> 5); s < g.n; s += nwarps) {
    if (!need[s] || counts[s] > FW_CAP) continue;
    const float4 p = g.pts[s];
    const float4 np = nrm[s];
    const int n = warp_gather_radius<FW_CAP>(g, p, radius, r2, nullptr, sm.pos, lane);
    sm.bins[lane] = 0;
    if (lane < 4) sm.bins[32 + lane] = 0;
    __syncwarp();
    for (int j = lane; j < n; j += 32) {
      const int pj = sm.pos[j];
      if (pj == s) continue;  // p_idx == indices[idx]
      float f1, f2, f3;
      pair_features(p, np, g.pts[pj], nrm[pj], f1, f2, f3);
      atomicAdd(&sm.bins[clamp_bin(11 * (((double)f1 + kPi) * (double)d_pi))], 1);
      atomicAdd(&sm.bins[11 + clamp_bin(11 * (((double)f2 + 1.0) * 0.5))], 1);
      atomicAdd(&sm.bins[22 + clamp_bin(11 * (((double)f3 + 1.0) * 0.5))], 1);
    }
    __syncwarp();
    // the float32 value PCL reaches by adding 100 / (n - 1) once per hit, rebuilt from the count
    const float hist_incr = 100.0f / (float)(n - 1);
    for (int b = lane; b < 33; b += 32) {
      float v = 0.0f;
      const int cnt = sm.bins[b];
      for (int t = 0; t < cnt; ++t) v += hist_incr;
      spfh[(size_t)orig_index(p) * 33 + b] = v;
    }
    __syncwarp();
  }
}

// Pass 2 for queries with at most FW_CAP neighbours.  rows_by_w: q is the cell-ordered surface, the output row is the
// point's original index.
__global__ void __launch_bounds__(FW_WARPS * 32)
    fpfh_weight_warp_kernel(GridView g, const float4 *__restrict__ q, int nq, const int *__restrict__ counts, float radius,
                            float r2, const float *__restrict__ spfh, float *__restrict__ out, int rows_by_w) {
  __shared__ FwSmem s_all[FW_WARPS];
  FwSmem &sm = s_all[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * FW_WARPS;
  for (int i = blockIdx.x * FW_WARPS + (threadIdx.x >> 5); i < nq; i += nwarps) {
    const int cnt = counts[i];
    if (cnt > FW_CAP) continue;
    const float4 c = q[i];
    const size_t row = rows_by_w ? (size_t)orig_index(c) : (size_t)i;
    if (cnt == 0) {  // searchForNeighbors == 0 -> NaN row
      for (int b = lane; b < 33; b += 32) out[row * 33 + b] = nanf32();
      continue;
    }
    const int n = warp_gather_radius<FW_CAP>(g, c, radius, r2, sm.key, nullptr, lane);
    warp_bitonic_sort(sm.key, nullptr, n, lane);
    // lane l < 11 owns bins l, l + 11, l + 22: float32 sums in (d2, index) order, float64 block sums beside them
    float acc[3] = {0.f, 0.f, 0.f};
    double part[3] = {0.0, 0.0, 0.0};
    if (lane < 11) {
      for (int j0 = 0; j0 < n; j0 += 4) {
        float val[4][3];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = j0 + u;
          val[u][0] = val[u][1] = val[u][2] = 0.0f;
          if (j < n) {
            const unsigned long long kj = sm.key[j];
            const float d2 = key_d2(kj);
            if (d2 != 0.0f) {  // d2 == 0: PCL skips the neighbour (adding +0 leaves the non-negative sums unchanged)
              const float weight = 1.0f / d2;
              const float *sp = spfh + (size_t)key_orig(kj) * 33 + lane;
#pragma unroll
              for (int f = 0; f < 3; ++f) val[u][f] = sp[11 * f] * weight;
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int f = 0; f < 3; ++f) {
            acc[f] += val[u][f];
            part[f] += (double)val[u][f];
          }
      }
    }
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      double sum = warp_sum(part[f]);
      if (sum != 0) sum = 100.0 / sum;
      if (lane < 11) out[row * 33 + 11 * f + lane] = acc[f] * (float)sum;
    }
    __syncwarp();
  }
}

__global__ void fill_nan_rows_kernel(float *p, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = nanf32();
}

}  // namespace

int dev_fpfh(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_q, int nq, bool q_is_surface,
             double radius, float *d_out) {
  if (!(radius > 0.0)) return ctx->fail(B200_ERR_INVALID, "fpfh: radius must be > 0");
  if (nq <= 0) return B200_OK;
  const GridView *g;
  B200_TRY(cloud_grid_for_radius(c, radius, &g));
  const int nv = c->n_valid;
  const float r2 = (float)(radius * radius);
  DevBuf<float4> nrm_sorted;
  B200_TRY(nrm_sorted.alloc(ctx, (size_t)std::max(nv, 1)));
  DevBuf<int> need, counts_s, counts_q;
  DevBuf<unsigned long long> stats;
  DevBuf<float> spfh;
  B200_TRY(need.alloc(ctx, (size_t)std::max(nv, 1)));
  B200_TRY(counts_s.alloc(ctx, (size_t)std::max(nv, 1)));
  B200_TRY(counts_q.alloc(ctx, (size_t)std::max(nq, 1)));
  B200_TRY(stats.alloc(ctx, 2));
  B200_TRY(spfh.alloc(ctx, (size_t)std::max(c->n, 1) * 33));
  B200_TRY(spfh.zero());
  if (nv > 0) {
    gather_normals_sorted_kernel<<<ceil_div(nv, 256), 256, 0, ctx->stream>>>(
        g->pts, nv, reinterpret_cast<const float4 *>(d_normals), nrm_sorted.p);
    B200_LAUNCHED(ctx);
    if (q_is_surface) {
      fill_int_kernel<<<ceil_div(nv, 256), 256, 0, ctx->stream>>>(need.p, nv, 1);
      B200_LAUNCHED(ctx);
    } else {
      B200_TRY(need.zero());
      fpfh_mark_kernel<<<ceil_div((long long)nq * 32, FPFH_THREADS), FPFH_THREADS, 0, ctx->stream>>>(
          *g, d_q, nq, (float)radius, r2, need.p);
      B200_LAUNCHED(ctx);
    }
  }
  // neighbourhood sizes of the surface points (pass 1, cell order) and of the queries (pass 2)
  unsigned long long hs[2], hq[2];
  B200_TRY(dev_radius_count(ctx, *g, g->pts, nv, radius, counts_s.p, stats.p));
  B200_CUDA(ctx, cudaMemcpyAsync(hs, stats.p, sizeof(hs), cudaMemcpyDeviceToHost, ctx->stream));
  B200_CUDA(ctx, ctx->sync());
  if (q_is_surface) {
    hq[0] = hs[0];
    hq[1] = hs[1];
  } else {
    B200_TRY(dev_radius_count(ctx, *g, d_q, nq, radius, counts_q.p, stats.p));
    B200_CUDA(ctx, cudaMemcpyAsync(hq, stats.p, sizeof(hq), cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(ctx, ctx->sync());
  }
  ctx->last_max_nbrs = (int)hq[0];
  ctx->last_mean_nbrs = (double)hq[1] / nq;
  // input == surface (every reference call site): pass 2 walks the cell-ordered surface and writes each row at the
  // point's original index, so the sizes of pass 1 serve both passes; rows that are not in the grid (non-finite
  // coordinates) are NaN rows
  const float4 *q2 = q_is_surface ? g->pts : d_q;
  const int nq2 = q_is_surface ? nv : nq;
  const int *cq2 = q_is_surface ? counts_s.p : counts_q.p;
  const int by_w = q_is_surface ? 1 : 0;
  const char *sel = getenv("B200_FPFH");  // "cta": everything by the one-point-per-CTA kernels
  const bool warp_path = !(sel && !strcmp(sel, "cta"));
  const int min_count = warp_path ? FW_CAP + 1 : 0;
  const bool cta1 = nv > 0 && (int)hs[0] >= min_count, cta2 = nq2 > 0 && (int)hq[0] >= min_count;
  const int max_count = (int)std::max(hs[0], hq[0]);
  const int cap = next_pow2_host(std::max(max_count, 32));
  const size_t smem = (size_t)cap * 12;
  const bool in_smem = smem <= 96 * 1024;
  DevBuf<unsigned long long> gk;
  DevBuf<int> gp;
  int grid1 = 1, grid2 = 1;
  if (cta1 || cta2) {
    if (in_smem) {
      B200_CUDA(ctx, ensure_dyn_smem(spfh_kernel, smem));
      B200_CUDA(ctx, ensure_dyn_smem(fpfh_weight_kernel, smem));
      grid1 = std::min(std::max(nv, 1), ctx->sm_count * 8);
      grid2 = std::min(std::max(nq2, 1), ctx->sm_count * 8);
    } else {
      grid1 = std::min(std::max(nv, 1), ctx->sm_count * 2);
      grid2 = std::min(std::max(nq2, 1), ctx->sm_count * 2);
      B200_TRY(gk.alloc(ctx, (size_t)std::max(grid1, grid2) * cap));
      B200_TRY(gp.alloc(ctx, (size_t)std::max(grid1, grid2) * cap));
    }
  }
  StageScope st_(ctx, ST_FPFH);
  if (q_is_surface && nv < c->n) {
    const size_t cells = (size_t)c->n * 33;
    fill_nan_rows_kernel<<<ceil_div((long long)cells, 256), 256, 0, ctx->stream>>>(d_out, cells);
    B200_LAUNCHED(ctx);
  }
  if (nv > 0) {
    if (warp_path) {
      spfh_warp_kernel<<<std::min(ceil_div(nv, FW_WARPS), ctx->sm_count * 16), FW_WARPS * 32, 0, ctx->stream>>>(
          *g, nrm_sorted.p, need.p, counts_s.p, (float)radius, r2, spfh.p);
      B200_LAUNCHED(ctx);
    }
    if (cta1) {
      spfh_kernel<<<grid1, FPFH_THREADS, in_smem ? smem : 0, ctx->stream>>>(*g, nrm_sorted.p, need.p, (float)radius, r2, cap,
                                                                           gk.p, gp.p, spfh.p, counts_s.p, min_count);
      B200_LAUNCHED(ctx);
    }
  }
  if (nq2 > 0) {
    if (warp_path) {
      fpfh_weight_warp_kernel<<<std::min(ceil_div(nq2, FW_WARPS), ctx->sm_count * 16), FW_WARPS * 32, 0, ctx->stream>>>(
          *g, q2, nq2, cq2, (float)radius, r2, spfh.p, d_out, by_w);
      B200_LAUNCHED(ctx);
    }
    if (cta2) {
      fpfh_weight_kernel<<<grid2, FPFH_THREADS, in_smem ? smem : 0, ctx->stream>>>(*g, q2, nq2, (float)radius, r2, cap, gk.p,
                                                                                  gp.p, spfh.p, d_out, cq2, min_count, by_w);
      B200_LAUNCHED(ctx);
    }
  }
  return B200_OK;
}
