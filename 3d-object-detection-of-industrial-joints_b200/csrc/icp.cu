// icp.cu — pcl::IterativeClosestPoint::align + getFitnessScore (SURVEY.md §8(f) rank 3: the refinement
// every reference program runs on the grouped poses — SHOT.cpp:177-192 (100 iterations), SHOT_demo.cpp:604-663,
// 6Dpose.cpp:572-609, FPFH_demo.cpp:611-668 (1 iteration)).
//
// pcl 1.8 registration/impl/icp.hpp with the defaults the reference leaves in place:
//   per iteration: determineCorrespondences (nearest target point of every source point, kept when
//   d2 <= max_dist^2; default unlimited) → at least 3 needed → TransformationEstimationSVD (Umeyama on the
//   corresponding points, no scaling) → transform the source → final = T * final → DefaultConvergenceCriteria:
//     1. iterations >= max_iterations                                   → converged
//     2. cos(angle) >= 1 - transformation_epsilon and |t|^2 <= transformation_epsilon (default 0: only an
//        exactly null motion)                                            → converged
//     3. |mse - previous mse| < 1e-12 (absolute; mse = mean d2 of this iteration's correspondences) → converged
//        relative threshold = euclidean_fitness_epsilon (default -DBL_MAX: never)
//   getFitnessScore: mean d2 from the aligned source points to their nearest target points.
// The nearest-neighbour search is the exact grid kNN (k = 1) of search.cuh; the Umeyama moments are
// float64 sums (PCL solves in float32: results agree to float32 rounding, not bit for bit); the
// convergence bookkeeping runs on the host from one small readback per iteration.
#include <algorithm>
#include <cfloat>
#include <cmath>

#include "linalg3.cuh"
#include "search.cuh"

namespace {

constexpr int ICP_THREADS = 128;

// nearest target point of every (finite) source point: original target row, d2; -1 = none within the distance gate
__global__ void __launch_bounds__(ICP_THREADS)
    icp_nn_kernel(GridView g, const float4 *__restrict__ src, int n, float max_d2, int *__restrict__ tgt_idx,
                  float *__restrict__ d2_out) {
  __shared__ unsigned long long sk[ICP_THREADS];
  const int i = blockIdx.x * ICP_THREADS + threadIdx.x;
  if (i >= n) return;
  const float4 p = src[i];
  int t = -1;
  float d2 = 0.f;
  if (finite3(p.x, p.y, p.z)) {
    const int cnt = knn_query(g, p.x, p.y, p.z, 1, sk + threadIdx.x, ICP_THREADS);
    if (cnt == 1 && !(key_d2(sk[threadIdx.x]) > max_d2)) {
      t = key_orig(sk[threadIdx.x]);  // original row of the target cloud
      d2 = key_d2(sk[threadIdx.x]);
    }
  }
  tgt_idx[i] = t;
  d2_out[i] = d2;
}

// sums[0..2] = sum src, [3..5] = sum dst, [6..14] = sum dst_r * src_c, [15] = sum d2, count[0] = pairs
__global__ void __launch_bounds__(256)
    icp_moments_kernel(GridView g, const float4 *__restrict__ src, int n, const int *__restrict__ tgt_idx,
                       const float *__restrict__ d2, double *__restrict__ sums, int *__restrict__ count) {
  double acc[16];
#pragma unroll
  for (int a = 0; a < 16; ++a) acc[a] = 0.0;
  int c = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int t = tgt_idx[i];
    if (t < 0) continue;
    const float4 s = src[i], q = g.raw[t];
    const double sv[3] = {s.x, s.y, s.z}, dv[3] = {q.x, q.y, q.z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      acc[a] += sv[a];
      acc[3 + a] += dv[a];
#pragma unroll
      for (int b = 0; b < 3; ++b) acc[6 + a * 3 + b] += dv[a] * sv[b];
    }
    acc[15] += (double)d2[i];
    ++c;
  }
#pragma unroll
  for (int a = 0; a < 16; ++a) acc[a] = warp_sum(acc[a]);
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 16; ++a) atomicAdd(&sums[a], acc[a]);
    if (c) atomicAdd(count, c);
  }
}

// p <- T p (Eigen: Matrix4f * homogeneous point, row by row, x y z then the translation)
__global__ void icp_transform_kernel(float4 *__restrict__ pts, int n, const float *__restrict__ T) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = pts[i];
  float o[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    float v = T[r * 4 + 0] * p.x;
    v += T[r * 4 + 1] * p.y;
    v += T[r * 4 + 2] * p.z;
    v += T[r * 4 + 3];
    o[r] = v;
  }
  pts[i] = make_float4(o[0], o[1], o[2], p.w);
}

void mat4_mul(const float *A, const float *B, float *C) {  // C = A * B, row-major
  float out[16];
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) {
      float v = A[r * 4 + 0] * B[0 * 4 + c];
      v += A[r * 4 + 1] * B[1 * 4 + c];
      v += A[r * 4 + 2] * B[2 * 4 + c];
      v += A[r * 4 + 3] * B[3 * 4 + c];
      out[r * 4 + c] = v;
    }
  memcpy(C, out, sizeof(out));
}

}  // namespace

// d_src: ns float4 source points (copied, the caller's buffer is not modified).  final_T: host, row-major 4x4.
// d_aligned (nullable): ns float4, the source under final_T.  Synchronises the stream.
int dev_icp_align(b200_ctx *ctx, const float4 *d_src, int ns, b200_cloud *target, int max_iterations, double max_corr_dist,
                  double transformation_epsilon, double euclidean_fitness_epsilon, const float *guess, float *final_T,
                  float4 *d_aligned, double *fitness, int *converged, int *iterations) {
  float fin[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  if (guess) memcpy(fin, guess, sizeof(fin));
  if (converged) *converged = 0;
  if (iterations) *iterations = 0;
  if (fitness) *fitness = DBL_MAX;
  memcpy(final_T, fin, sizeof(fin));
  if (ns <= 0 || target->n_valid <= 0) return B200_OK;
  const GridView *g;
  B200_TRY(cloud_grid_for_knn(target, 1, &g));
  DevBuf<float4> cur;
  DevBuf<int> tgt_idx, count;
  DevBuf<float> d2, dT;
  DevBuf<double> sums;
  B200_TRY(cur.alloc(ctx, (size_t)ns));
  B200_TRY(tgt_idx.alloc(ctx, (size_t)ns));
  B200_TRY(d2.alloc(ctx, (size_t)ns));
  B200_TRY(count.alloc(ctx, 1));
  B200_TRY(sums.alloc(ctx, 16));
  B200_TRY(dT.alloc(ctx, 16));
  B200_CUDA(ctx, cudaMemcpyAsync(cur.p, d_src, sizeof(float4) * (size_t)ns, cudaMemcpyDeviceToDevice, ctx->stream));
  const bool identity_guess = !guess || (memcmp(fin, (const float[16]){1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1}, 64) == 0);
  if (!identity_guess) {
    B200_CUDA(ctx, cudaMemcpyAsync(dT.p, fin, sizeof(fin), cudaMemcpyHostToDevice, ctx->stream));
    icp_transform_kernel<<<ceil_div(ns, 256), 256, 0, ctx->stream>>>(cur.p, ns, dT.p);
    B200_LAUNCHED(ctx);
  }
  const double md = (max_corr_dist > 0.0) ? max_corr_dist : std::sqrt(DBL_MAX);
  const double md2 = md * md;
  const float max_d2 = (md2 >= (double)FLT_MAX) ? FLT_MAX : (float)md2;
  // DefaultConvergenceCriteria as configured by IterativeClosestPoint::computeTransformation
  const double rotation_threshold = 1.0 - transformation_epsilon, translation_threshold = transformation_epsilon;
  const double mse_abs = 1e-12, mse_rel = euclidean_fitness_epsilon;
  double prev_mse = DBL_MAX;
  int it = 0;
  bool conv = false;
  const int nblocks = std::min(ceil_div(ns, 256), ctx->sm_count * 4);
  do {
    icp_nn_kernel<<<ceil_div(ns, ICP_THREADS), ICP_THREADS, 0, ctx->stream>>>(*g, cur.p, ns, max_d2, tgt_idx.p, d2.p);
    B200_LAUNCHED(ctx);
    B200_TRY(sums.zero());
    B200_TRY(count.zero());
    icp_moments_kernel<<<nblocks, 256, 0, ctx->stream>>>(*g, cur.p, ns, tgt_idx.p, d2.p, sums.p, count.p);
    B200_LAUNCHED(ctx);
    double h[16];
    int cnt = 0;
    B200_CUDA(ctx, cudaMemcpyAsync(h, sums.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(ctx, cudaMemcpyAsync(&cnt, count.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(ctx, ctx->sync());
    if (cnt < 3) {  // "Not enough correspondences found. Relax your threshold parameters."
      conv = false;
      break;
    }
    double ms[3], mdn[3], S[9], Td[16];
    for (int a = 0; a < 3; ++a) {
      ms[a] = h[a] / cnt;
      mdn[a] = h[3 + a] / cnt;
    }
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) S[a * 3 + b] = h[6 + a * 3 + b] / cnt - mdn[a] * ms[b];
    umeyama_from_moments(S, ms, mdn, Td);
    float T[16];
    for (int a = 0; a < 16; ++a) T[a] = (float)Td[a];
    B200_CUDA(ctx, cudaMemcpyAsync(dT.p, T, sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    icp_transform_kernel<<<ceil_div(ns, 256), 256, 0, ctx->stream>>>(cur.p, ns, dT.p);
    B200_LAUNCHED(ctx);
    B200_CUDA(ctx, ctx->sync());  // T is a stack buffer
    mat4_mul(T, fin, fin);
    ++it;
    // hasConverged()
    if (it >= max_iterations) {
      conv = true;
      break;
    }
    const double cos_angle = 0.5 * ((double)T[0] + (double)T[5] + (double)T[10] - 1.0);
    const double tr2 = (double)T[3] * T[3] + (double)T[7] * T[7] + (double)T[11] * T[11];
    if (cos_angle >= rotation_threshold && tr2 <= translation_threshold) {
      conv = true;
      break;
    }
    const double mse = h[15] / cnt;
    if (std::fabs(mse - prev_mse) < mse_abs) {
      conv = true;
      break;
    }
    if (std::fabs(mse - prev_mse) / prev_mse < mse_rel) {
      conv = true;
      break;
    }
    prev_mse = mse;
  } while (true);
  memcpy(final_T, fin, sizeof(fin));
  if (converged) *converged = conv ? 1 : 0;
  if (iterations) *iterations = it;
  // getFitnessScore (and the aligned cloud): the source under the final transformation
  B200_CUDA(ctx, cudaMemcpyAsync(cur.p, d_src, sizeof(float4) * (size_t)ns, cudaMemcpyDeviceToDevice, ctx->stream));
  B200_CUDA(ctx, cudaMemcpyAsync(dT.p, fin, sizeof(fin), cudaMemcpyHostToDevice, ctx->stream));
  icp_transform_kernel<<<ceil_div(ns, 256), 256, 0, ctx->stream>>>(cur.p, ns, dT.p);
  B200_LAUNCHED(ctx);
  if (d_aligned)
    B200_CUDA(ctx, cudaMemcpyAsync(d_aligned, cur.p, sizeof(float4) * (size_t)ns, cudaMemcpyDeviceToDevice, ctx->stream));
  if (fitness) {
    icp_nn_kernel<<<ceil_div(ns, ICP_THREADS), ICP_THREADS, 0, ctx->stream>>>(*g, cur.p, ns, FLT_MAX, tgt_idx.p, d2.p);
    B200_LAUNCHED(ctx);
    B200_TRY(sums.zero());
    B200_TRY(count.zero());
    icp_moments_kernel<<<nblocks, 256, 0, ctx->stream>>>(*g, cur.p, ns, tgt_idx.p, d2.p, sums.p, count.p);
    B200_LAUNCHED(ctx);
    double h[16];
    int cnt = 0;
    B200_CUDA(ctx, cudaMemcpyAsync(h, sums.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(ctx, cudaMemcpyAsync(&cnt, count.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(ctx, ctx->sync());
    *fitness = cnt > 0 ? h[15] / cnt : DBL_MAX;
  } else {
    B200_CUDA(ctx, ctx->sync());
  }
  return B200_OK;
}
