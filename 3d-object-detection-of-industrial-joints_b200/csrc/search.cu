// search.cu — batched neighbour-search kernels behind b200_knn_search / b200_radius_search
// (KdTreeFLANN::nearestKSearch SHOT.cpp:163, Edge_detection.cpp:120; ::radiusSearch SHOT_VAR.cpp:356).
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "search.cuh"

namespace {

// one query per thread; lists in dynamic shared memory: float d[k][T], int p[k][T]
__global__ void knn_search_kernel(GridView g, const float4 *__restrict__ q, int nq, int k, int *__restrict__ idx,
                                  float *__restrict__ d2) {
  extern __shared__ unsigned char smem_raw[];
  const int T = blockDim.x;
  unsigned long long *sk = reinterpret_cast<unsigned long long *>(smem_raw) + threadIdx.x;
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= nq) return;
  const float4 p = q[i];
  int cnt = 0;
  if (finite3(p.x, p.y, p.z)) cnt = knn_query(g, p.x, p.y, p.z, k, sk, T);
  for (int j = 0; j < k; ++j) {
    const bool have = j < cnt;
    const unsigned long long key = have ? sk[j * T] : 0ull;
    idx[(size_t)i * k + j] = have ? key_orig(key) : -1;
    d2[(size_t)i * k + j] = have ? key_d2(key) : __int_as_float(0x7f800000);
  }
}

// one query per warp; counts + global max / sum
__global__ void radius_count_kernel(GridView g, const float4 *__restrict__ q, int nq, float radius, float r2,
                                    int *__restrict__ counts, unsigned long long *__restrict__ stats) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= nq) return;
  const float4 p = q[w];
  const int c = count_radius_warp(g, p.x, p.y, p.z, radius, r2);
  if ((threadIdx.x & 31) == 0) {
    counts[w] = c;
    if (stats) {
      atomicMax(&stats[0], (unsigned long long)c);
      atomicAdd(&stats[1], (unsigned long long)c);
    }
  }
}

// one query per CTA: gather, sort by (d2, index), write the CSR segment.
// list storage: shared (cap entries) or, when glob_key != nullptr, global scratch of cap entries per CTA.
__global__ void __launch_bounds__(128) radius_fill_kernel(GridView g, const float4 *__restrict__ q, int nq,
                                                          float radius, float r2, int cap,
                                                          unsigned long long *glob_key, int *glob_pos,
                                                          const long long *__restrict__ offsets,
                                                          int *__restrict__ idx, float *__restrict__ d2, int min_count) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_count;
  unsigned long long *key;
  int *pos;
  cta_list(smem_raw, glob_key, glob_pos, cap, key, pos);
  for (int i = blockIdx.x; i < nq; i += gridDim.x) {
    if (offsets[i + 1] - offsets[i] < (long long)min_count) continue;  // shorter lists: radius_fill_warp_kernel
    const float4 p = q[i];
    int n = gather_radius(g, p.x, p.y, p.z, radius, r2, key, pos, cap, &s_count);
    if (n > cap) n = cap;  // cannot happen: cap >= max count (host sized it)
    bitonic_sort(key, pos, n);
    const long long o = offsets[i];
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      idx[o + j] = key_orig(key[j]);
      d2[o + j] = key_d2(key[j]);
    }
    __syncthreads();
  }
}

// one query per warp for lists of up to RFW_CAP neighbours: ballot-compacted gather of the (d2, index) keys into the
// warp's slice of shared memory, bitonic sort synchronised by __syncwarp only, coalesced write of the CSR segment
constexpr int RFW_CAP = 512;
constexpr int RFW_WARPS = 8;
__global__ void __launch_bounds__(RFW_WARPS * 32)
    radius_fill_warp_kernel(GridView g, const float4 *__restrict__ q, int nq, float radius, float r2,
                            const long long *__restrict__ offsets, int *__restrict__ idx, float *__restrict__ d2) {
  __shared__ unsigned long long s_key[RFW_WARPS][RFW_CAP];
  unsigned long long *key = s_key[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * RFW_WARPS;
  for (int i = blockIdx.x * RFW_WARPS + (threadIdx.x >> 5); i < nq; i += nwarps) {
    const long long o = offsets[i];
    const long long cnt = offsets[i + 1] - o;
    if (cnt == 0 || cnt > RFW_CAP) continue;
    const int n = warp_gather_radius<RFW_CAP>(g, q[i], radius, r2, key, nullptr, lane);
    warp_bitonic_sort(key, nullptr, n, lane);
    for (int j = lane; j < n; j += 32) {
      idx[o + j] = key_orig(key[j]);
      d2[o + j] = key_d2(key[j]);
    }
    __syncwarp();
  }
}

__global__ void counts_to_i64_kernel(const int *__restrict__ ex, int n, const int *__restrict__ total,
                                     long long *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = ex[i];
  if (i == n) out[n] = *total;
}

}  // namespace

int knn_threads_for(int k, size_t *smem_bytes) {
  // keep the per-CTA candidate lists within ~96 KB
  int T = 128;
  while (T > 32 && (size_t)k * T * 8 > 96 * 1024) T >>= 1;
  *smem_bytes = (size_t)k * T * 8;
  return T;
}

int dev_knn_search(b200_ctx *ctx, b200_cloud *c, const float4 *d_q, int nq, int k, int *d_idx, float *d_d2,
                   int *k_found) {
  if (k <= 0 || k > 1024) return ctx->fail(B200_ERR_INVALID, "knn_search: k must be in [1, 1024]");
  const GridView *g;
  B200_TRY(cloud_grid_for_knn(c, k, &g));
  if (k_found) *k_found = std::min(k, c->n_valid);
  if (nq <= 0) return B200_OK;
  size_t smem;
  const int T = knn_threads_for(k, &smem);
  if (smem > ctx->smem_optin) return ctx->fail(B200_ERR_INVALID, "knn_search: k too large for shared memory");
  B200_CUDA(ctx, ensure_dyn_smem(knn_search_kernel, smem));
  knn_search_kernel<<<ceil_div(nq, T), T, smem, ctx->stream>>>(*g, d_q, nq, k, d_idx, d_d2);
  B200_LAUNCHED(ctx);
  return B200_OK;
}

int dev_radius_count(b200_ctx *ctx, const GridView &g, const float4 *d_q, int nq, double radius, int *d_counts,
                     unsigned long long *d_stats) {
  StageScope st_(ctx, ST_NBR_COUNT);
  if (d_stats) B200_CUDA(ctx, cudaMemsetAsync(d_stats, 0, 2 * sizeof(unsigned long long), ctx->stream));
  if (nq <= 0) return B200_OK;
  const float r2 = (float)(radius * radius);
  radius_count_kernel<<<ceil_div((long long)nq * 32, 256), 256, 0, ctx->stream>>>(g, d_q, nq, (float)radius, r2,
                                                                                 d_counts, d_stats);
  B200_LAUNCHED(ctx);
  return B200_OK;
}

// Radius search into caller CSR buffers.  max_count: the largest list (from dev_radius_count).
int dev_radius_fill_sized(b200_ctx *ctx, const GridView &g, const float4 *d_q, int nq, double radius, int max_count,
                          const long long *d_offsets, int *d_idx, float *d_d2) {
  if (nq <= 0 || max_count <= 0) return B200_OK;
  const float r2 = (float)(radius * radius);
  // lists of up to RFW_CAP neighbours: one query per warp (B200_RADIUS_FILL=cta: everything by the CTA kernel)
  const char *sel = getenv("B200_RADIUS_FILL");
  const bool warp_path = !(sel && !strcmp(sel, "cta"));
  if (warp_path) {
    radius_fill_warp_kernel<<<std::min(ceil_div(nq, RFW_WARPS), ctx->sm_count * 16), RFW_WARPS * 32, 0, ctx->stream>>>(
        g, d_q, nq, (float)radius, r2, d_offsets, d_idx, d_d2);
    B200_LAUNCHED(ctx);
    if (max_count <= RFW_CAP) return B200_OK;
  }
  const int min_count = warp_path ? RFW_CAP + 1 : 0;
  const int cap = next_pow2_host(std::max(max_count, 32));
  const size_t smem = (size_t)cap * 12;
  const int grid = std::min(nq, ctx->sm_count * 8);
  if (smem <= 96 * 1024) {
    B200_CUDA(ctx, ensure_dyn_smem(radius_fill_kernel, smem));
    radius_fill_kernel<<<grid, 128, smem, ctx->stream>>>(g, d_q, nq, (float)radius, r2, cap, nullptr, nullptr,
                                                         d_offsets, d_idx, d_d2, min_count);
    B200_LAUNCHED(ctx);
  } else {
    const int g2 = std::min(nq, ctx->sm_count * 2);
    DevBuf<unsigned long long> gk;
    DevBuf<int> gp;
    B200_TRY(gk.alloc(ctx, (size_t)g2 * cap));
    B200_TRY(gp.alloc(ctx, (size_t)g2 * cap));
    radius_fill_kernel<<<g2, 128, 0, ctx->stream>>>(g, d_q, nq, (float)radius, r2, cap, gk.p, gp.p, d_offsets, d_idx,
                                                    d_d2, min_count);
    B200_LAUNCHED(ctx);
  }
  return B200_OK;
}

int counts_to_offsets_i64(b200_ctx *ctx, const int *d_counts, int nq, long long *d_offsets) {
  DevBuf<int> ex, total;
  B200_TRY(ex.alloc(ctx, (size_t)nq + 1));
  B200_TRY(total.alloc(ctx, 1));
  B200_TRY(exclusive_scan_i32(ctx, d_counts, ex.p, nq, total.p));
  counts_to_i64_kernel<<<ceil_div(nq + 1, 256), 256, 0, ctx->stream>>>(ex.p, nq, total.p, d_offsets);
  B200_LAUNCHED(ctx);
  return B200_OK;
}
