// hough.cu — pcl::Hough3DGrouping on the device (SURVEY.md §8(f) rank 1: the grouping every reference
// program uses by default — SHOT.cpp:433-470, SHOT_demo.cpp:540-577, FPFH_demo.cpp:548-585 — with the
// settings they make: setUseInterpolation(false), setUseDistanceWeight(true), setHoughBinSize,
// setHoughThreshold, reference frames given through setInputRf / setSceneRf).
//
// pcl 1.8 recognition/impl/cg/hough_3d.hpp:
//   train():        centroid = float32 running sum of the model keypoints / n; model_vote[i] = the offset
//                   (centroid - keypoint_i) expressed in keypoint i's reference frame (float32 dots).
//   houghVoting():  per correspondence, scene_vote = scene_rf^T * model_vote + scene point (float32, widened
//                   to double); the Hough space spans [min, max] of the votes with cubic bins of
//                   hough_bin_size; without interpolation a vote adds its weight to one bin.  The weight is
//                   1 - distance / max_distance, and max_distance is only tracked when interpolation is on
//                   (it stays -FLT_MAX), so every weight is exactly 1.0: a bin's value is its vote count.
//   findMaxima():   every bin with value >= threshold (threshold < 0: that fraction of the maximum) is an
//                   instance, in ascending bin index; its voters (ascending correspondence index) go to
//                   RANSAC (inlier threshold = bin size), exactly as in geometric-consistency grouping.
// Votes whose bin coordinate falls outside the space (a vote exactly on the upper bound) are dropped, as
// HoughSpace3D::vote does.  Correspondences with a non-finite reference frame are skipped.
//
// Everything stays on the device, with no host round trip: the correspondence count arrives as a device int,
// the vote bounds, the space and its 2^27-bin cap are computed by one thread, and the space is never
// materialised.  Instead the (bin, correspondence) pairs are sorted by bin with a stable LSD radix sort: a run of
// equal bins is that bin's vote count, the runs come in ascending bin order and the voters inside a run in
// ascending correspondence index.  Memory is O(correspondences), whatever the number of bins.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace {

constexpr long long HOUGH_MAX_BINS = 1ll << 27;
constexpr unsigned HOUGH_NO_BIN = 1u << 27;  // sort key of a skipped / dropped vote: after every bin
constexpr int HR_THREADS = 256;              // keys per radix-sort block
constexpr int HR_WARPS = HR_THREADS / 32;
constexpr int HR_BITS = 7;                   // 4 passes x 7 bits cover the 28-bit keys
constexpr int HR_DIGITS = 1 << HR_BITS;
constexpr int HR_PASSES = 4;

__device__ __forceinline__ unsigned enc_ordered(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec_ordered(unsigned e) {
  return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e);
}

// float32 running sum in row order (Eigen: centroid += p; centroid /= n), one thread per coordinate
__global__ void hough_centroid_kernel(const float4 *__restrict__ kp, int n, float *__restrict__ centroid) {
  const int a = threadIdx.x;
  if (a >= 3) return;
  float s = 0.f;
  for (int i = 0; i < n; ++i) {
    const float4 p = kp[i];
    s += (a == 0) ? p.x : (a == 1 ? p.y : p.z);
  }
  centroid[a] = s / (float)n;
}

__global__ void hough_model_votes_kernel(const float4 *__restrict__ kp, const float *__restrict__ rf, int n,
                                         const float *__restrict__ centroid, float *__restrict__ votes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = kp[i];
  const float dx = centroid[0] - p.x, dy = centroid[1] - p.y, dz = centroid[2] - p.z;
  const float *r = rf + (size_t)i * 9;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float v = r[a * 3 + 0] * dx;
    v += r[a * 3 + 1] * dy;
    v += r[a * 3 + 2] * dz;
    votes[(size_t)i * 3 + a] = v;
  }
}

__device__ __forceinline__ int hough_count(const int *d_C, int C_cap) { return min(*d_C, C_cap); }

// scene_votes (float32 values, as PCL computes them before widening) + their bounds
__global__ void hough_scene_votes_kernel(const b200_corr *__restrict__ corrs, const int *__restrict__ d_C, int C_cap,
                                         const float *__restrict__ mvotes, const float4 *__restrict__ scene_kp,
                                         const float *__restrict__ scene_rf, float *__restrict__ svotes,
                                         unsigned *__restrict__ box) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hough_count(d_C, C_cap)) return;
  const b200_corr c = corrs[i];
  const float *mv = mvotes + (size_t)c.index_query * 3;
  const float *r = scene_rf + (size_t)c.index_match * 9;
  const float4 sp = scene_kp[c.index_match];
  float v[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float t = r[0 * 3 + a] * mv[0];  // x axis component a
    t += r[1 * 3 + a] * mv[1];
    t += r[2 * 3 + a] * mv[2];
    t += (a == 0) ? sp.x : (a == 1 ? sp.y : sp.z);
    v[a] = t;
    svotes[(size_t)i * 3 + a] = t;
  }
  if (isfinite(v[0]) && isfinite(v[1]) && isfinite(v[2])) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      atomicMin(&box[a], enc_ordered(v[a]));
      atomicMax(&box[3 + a], enc_ordered(v[a]));
    }
  }
}

struct HoughSpace {
  double mn[3], bin;
  int cnt[3];
  int valid;  // at least one bin and no more than 2^27
};

// HoughSpace3D's constructor from the vote bounds (one thread): bin_count = ceil((max - min) / bin) per axis
__global__ void hough_space_kernel(const unsigned *__restrict__ box, double bin, HoughSpace *__restrict__ H,
                                   int *__restrict__ status) {
  HoughSpace h;
  h.bin = bin;
  h.valid = 0;
  if (box[0] <= box[3]) {  // otherwise no finite vote
    long long nbins = 1;
    bool over = false;
    for (int a = 0; a < 3 && !over; ++a) {
      h.mn[a] = (double)dec_ordered(box[a]);
      const double mx = (double)dec_ordered(box[3 + a]);
      h.cnt[a] = (int)ceil((mx - h.mn[a]) / bin);
      nbins *= max(h.cnt[a], 0);
      over = nbins > HOUGH_MAX_BINS;
    }
    if (over)
      *status = B200_ERR_CAPACITY;
    else
      h.valid = nbins > 0;  // a degenerate space (all votes on one coordinate of an axis) holds no bin
  }
  *H = h;
}

// sort keys: the bin of vote i (HOUGH_NO_BIN when it has none), values: i
__global__ void hough_keys_kernel(const float *__restrict__ svotes, const int *__restrict__ d_C, int C_cap,
                                  const HoughSpace *__restrict__ Hp, unsigned *__restrict__ keys,
                                  int *__restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C_cap) return;
  unsigned key = HOUGH_NO_BIN;
  const HoughSpace H = *Hp;
  if (H.valid && i < hough_count(d_C, C_cap)) {
    const float *v = svotes + (size_t)i * 3;
    if (isfinite(v[0]) && isfinite(v[1]) && isfinite(v[2])) {
      long long index = 0, mul = 1;
      bool in = true;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const int ci = (int)floor(((double)v[a] - H.mn[a]) / H.bin);
        if (ci < 0 || ci >= H.cnt[a]) in = false;
        index += mul * ci;
        mul *= H.cnt[a];
      }
      if (in) key = (unsigned)index;
    }
  }
  keys[i] = key;
  vals[i] = i;
}

// ---- stable LSD radix sort, HR_BITS per pass: per-block digit counts (digit-major, so that one exclusive scan
// gives every (digit, block) its output start), then a stable scatter (rank inside the warp by __match_any_sync,
// warps of the block in order)
__global__ void __launch_bounds__(HR_THREADS)
    hough_radix_count_kernel(const unsigned *__restrict__ keys, int n, int shift, int nblk, int *__restrict__ counts) {
  __shared__ int s_cnt[HR_DIGITS];
  if (threadIdx.x < HR_DIGITS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const int j = blockIdx.x * HR_THREADS + threadIdx.x;
  if (j < n) atomicAdd(&s_cnt[(keys[j] >> shift) & (HR_DIGITS - 1)], 1);
  __syncthreads();
  if (threadIdx.x < HR_DIGITS) counts[(size_t)threadIdx.x * nblk + blockIdx.x] = s_cnt[threadIdx.x];
}

__global__ void __launch_bounds__(HR_THREADS)
    hough_radix_scatter_kernel(const unsigned *__restrict__ keys, const int *__restrict__ vals, int n, int shift,
                               int nblk, const int *__restrict__ starts, unsigned *__restrict__ keys_out,
                               int *__restrict__ vals_out) {
  __shared__ int s_cnt[HR_WARPS][HR_DIGITS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = threadIdx.x; t < HR_WARPS * HR_DIGITS; t += HR_THREADS) (&s_cnt[0][0])[t] = 0;
  __syncthreads();
  const int j = blockIdx.x * HR_THREADS + threadIdx.x;
  const bool live = j < n;
  const unsigned k = live ? keys[j] : 0u;
  const int d = live ? (int)((k >> shift) & (HR_DIGITS - 1)) : HR_DIGITS + lane;  // padding lanes match nobody
  const unsigned peers = __match_any_sync(0xffffffffu, d);
  const int rank = __popc(peers & ((1u << lane) - 1u));
  if (live && rank == 0) s_cnt[warp][d] = __popc(peers);
  __syncthreads();
  if (threadIdx.x < HR_DIGITS) {  // exclusive prefix over the warps, per digit
    int run = 0;
    for (int w = 0; w < HR_WARPS; ++w) {
      const int c = s_cnt[w][threadIdx.x];
      s_cnt[w][threadIdx.x] = run;
      run += c;
    }
  }
  __syncthreads();
  if (!live) return;
  const int pos = starts[(size_t)d * nblk + blockIdx.x] + s_cnt[warp][d] + rank;
  keys_out[pos] = k;
  vals_out[pos] = vals[j];
}

// ---- runs of equal keys in the sorted array = the occupied bins, ascending
__global__ void hough_run_heads_kernel(const unsigned *__restrict__ keys, int n, int *__restrict__ head) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) head[j] = (j == 0 || keys[j] != keys[j - 1]) ? 1 : 0;
}

// run_start[r] = first position of run r; run_start[R] = n
__global__ void hough_run_starts_kernel(const int *__restrict__ head, const int *__restrict__ run_id, int n,
                                        const int *__restrict__ n_runs, int *__restrict__ run_start) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (head[j]) run_start[run_id[j]] = j;
  if (j == 0) run_start[*n_runs] = n;
}

// votes of every occupied bin (0 for the run of skipped votes) and their maximum
__global__ void hough_run_votes_kernel(const unsigned *__restrict__ keys, const int *__restrict__ run_start,
                                       const int *__restrict__ n_runs, int n, int *__restrict__ votes,
                                       int *__restrict__ vmax) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  int v = 0;
  if (r < *n_runs && keys[run_start[r]] != HOUGH_NO_BIN) v = run_start[r + 1] - run_start[r];
  votes[r] = v;
  if (v > 0) atomicMax(vmax, v);
}

// flags[r] = bin r is a maximum; sizes[r] = its vote count (0 otherwise)
__global__ void hough_flags_kernel(const int *__restrict__ votes, int n, double threshold, const int *__restrict__ vmax,
                                   int *__restrict__ flags, int *__restrict__ sizes) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  double thr = threshold;
  if (thr < 0) {  // HoughSpace3D::findMaxima: relative to the largest bin
    const double hmax = (double)*vmax;
    thr = (thr >= -1.0) ? -thr * hmax : hmax;
  }
  const int v = votes[r];
  const int f = (v > 0 && (double)v >= thr) ? 1 : 0;
  flags[r] = f;
  sizes[r] = f ? v : 0;
}

__global__ void hough_offsets_kernel(const int *__restrict__ flags, const int *__restrict__ slots,
                                     const int *__restrict__ starts, const int *__restrict__ sizes, int n, int max_inst,
                                     int *__restrict__ inst_offsets) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n || !flags[r]) return;
  const int s = slots[r];
  if (s < max_inst) inst_offsets[s + 1] = starts[r] + sizes[r];
}

// the voters of every instance, in the sorted (= ascending correspondence index) order of their run
__global__ void hough_members_kernel(const int *__restrict__ vals, const int *__restrict__ head,
                                     const int *__restrict__ run_id, const int *__restrict__ run_start,
                                     const int *__restrict__ flags, const int *__restrict__ starts, int n,
                                     int *__restrict__ members) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int r = run_id[j] + head[j] - 1;
  if (flags[r]) members[starts[r] + (j - run_start[r])] = vals[j];
}

__global__ void hough_gather_points_kernel(const b200_corr *__restrict__ corrs, const int *__restrict__ d_C, int C_cap,
                                           const float4 *__restrict__ model_kp, const float4 *__restrict__ scene_kp,
                                           float4 *__restrict__ mp, float4 *__restrict__ sp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hough_count(d_C, C_cap)) return;
  mp[i] = model_kp[corrs[i].index_query];
  sp[i] = scene_kp[corrs[i].index_match];
}

}  // namespace

// Hough3DGrouping::train(): d_votes (Km x 3) from the model keypoints and their frames
int dev_hough_model_votes(b200_ctx *ctx, const float4 *d_model_kp, const float *d_model_rf, int Km, float *d_votes) {
  if (Km <= 0) return B200_OK;
  DevBuf<float> centroid;
  B200_TRY(centroid.alloc(ctx, 3));
  hough_centroid_kernel<<<1, 32, 0, ctx->stream>>>(d_model_kp, Km, centroid.p);
  B200_LAUNCHED(ctx);
  hough_model_votes_kernel<<<ceil_div(Km, 256), 256, 0, ctx->stream>>>(d_model_kp, d_model_rf, Km, centroid.p, d_votes);
  B200_LAUNCHED(ctx);
  return B200_OK;
}

int dev_hough3d(b200_ctx *ctx, const float4 *d_model_kp, const float *d_model_votes, const float4 *d_scene_kp,
                const float *d_scene_rf, const b200_corr *d_corrs, const int *d_C, int C_cap, double bin_size,
                double threshold, float *d_T, int max_inst, int *d_inst_offsets, int *d_inst_counts,
                b200_corr *d_inst_corrs, int corr_cap, int *d_n_inst, int *d_status) {
  if (max_inst < 1) return ctx->fail(B200_ERR_INVALID, "hough3d: max_inst must be >= 1");
  if (!(bin_size > 0.0)) return ctx->fail(B200_ERR_INVALID, "hough3d: bin size must be > 0");
  B200_CUDA(ctx, cudaMemsetAsync(d_status, 0, sizeof(int), ctx->stream));
  B200_CUDA(ctx, cudaMemsetAsync(d_n_inst, 0, sizeof(int), ctx->stream));
  B200_CUDA(ctx, cudaMemsetAsync(d_inst_offsets, 0, sizeof(int) * ((size_t)max_inst + 1), ctx->stream));
  B200_CUDA(ctx, cudaMemsetAsync(d_inst_counts, 0, sizeof(int) * (size_t)max_inst, ctx->stream));
  if (C_cap <= 0) return B200_OK;
  const int n = C_cap, nb = ceil_div(n, 256);
  DevBuf<int> members;
  DevBuf<float4> mp, sp;
  B200_TRY(members.alloc(ctx, (size_t)n));
  B200_TRY(mp.alloc(ctx, (size_t)n));
  B200_TRY(sp.alloc(ctx, (size_t)n));
  {
    StageScope st_(ctx, ST_HOUGH);
    DevBuf<float> svotes;
    DevBuf<unsigned> box, keys, keys2;
    DevBuf<HoughSpace> space;
    DevBuf<int> vals, vals2;
    B200_TRY(svotes.alloc(ctx, (size_t)n * 3));
    B200_TRY(box.alloc(ctx, 6));
    B200_TRY(space.alloc(ctx, 1));
    B200_TRY(keys.alloc(ctx, (size_t)n));
    B200_TRY(keys2.alloc(ctx, (size_t)n));
    B200_TRY(vals.alloc(ctx, (size_t)n));
    B200_TRY(vals2.alloc(ctx, (size_t)n));
    const unsigned init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
    B200_TRY(write_small(ctx, box.p, init, sizeof(init)));
    hough_scene_votes_kernel<<<nb, 256, 0, ctx->stream>>>(d_corrs, d_C, n, d_model_votes, d_scene_kp, d_scene_rf,
                                                          svotes.p, box.p);
    B200_LAUNCHED(ctx);
    hough_space_kernel<<<1, 1, 0, ctx->stream>>>(box.p, bin_size, space.p, d_status);
    B200_LAUNCHED(ctx);
    hough_keys_kernel<<<nb, 256, 0, ctx->stream>>>(svotes.p, d_C, n, space.p, keys.p, vals.p);
    B200_LAUNCHED(ctx);
    // sort by bin
    const int nblk = ceil_div(n, HR_THREADS);
    DevBuf<int> counts;
    B200_TRY(counts.alloc(ctx, (size_t)nblk * HR_DIGITS));
    unsigned *kin = keys.p, *kout = keys2.p;
    int *vin = vals.p, *vout = vals2.p;
    for (int pass = 0; pass < HR_PASSES; ++pass) {
      const int shift = pass * HR_BITS;
      hough_radix_count_kernel<<<nblk, HR_THREADS, 0, ctx->stream>>>(kin, n, shift, nblk, counts.p);
      B200_LAUNCHED(ctx);
      B200_TRY(exclusive_scan_i32(ctx, counts.p, counts.p, nblk * HR_DIGITS, nullptr));
      hough_radix_scatter_kernel<<<nblk, HR_THREADS, 0, ctx->stream>>>(kin, vin, n, shift, nblk, counts.p, kout, vout);
      B200_LAUNCHED(ctx);
      std::swap(kin, kout);
      std::swap(vin, vout);
    }
    // runs -> bin votes -> maxima -> instances in ascending bin order, voters in ascending correspondence index
    DevBuf<int> head, run_id, n_runs, run_start, votes, vmax, flags, sizes, slots, starts;
    B200_TRY(head.alloc(ctx, (size_t)n));
    B200_TRY(run_id.alloc(ctx, (size_t)n));
    B200_TRY(n_runs.alloc(ctx, 1));
    B200_TRY(run_start.alloc(ctx, (size_t)n + 1));
    B200_TRY(votes.alloc(ctx, (size_t)n));
    B200_TRY(vmax.alloc(ctx, 1));
    B200_TRY(flags.alloc(ctx, (size_t)n));
    B200_TRY(sizes.alloc(ctx, (size_t)n));
    B200_TRY(slots.alloc(ctx, (size_t)n));
    B200_TRY(starts.alloc(ctx, (size_t)n));
    B200_TRY(vmax.zero());
    hough_run_heads_kernel<<<nb, 256, 0, ctx->stream>>>(kin, n, head.p);
    B200_LAUNCHED(ctx);
    B200_TRY(exclusive_scan_i32(ctx, head.p, run_id.p, n, n_runs.p));
    hough_run_starts_kernel<<<nb, 256, 0, ctx->stream>>>(head.p, run_id.p, n, n_runs.p, run_start.p);
    B200_LAUNCHED(ctx);
    hough_run_votes_kernel<<<nb, 256, 0, ctx->stream>>>(kin, run_start.p, n_runs.p, n, votes.p, vmax.p);
    B200_LAUNCHED(ctx);
    hough_flags_kernel<<<nb, 256, 0, ctx->stream>>>(votes.p, n, threshold, vmax.p, flags.p, sizes.p);
    B200_LAUNCHED(ctx);
    B200_TRY(exclusive_scan_i32(ctx, flags.p, slots.p, n, d_n_inst));
    B200_TRY(exclusive_scan_i32(ctx, sizes.p, starts.p, n, nullptr));
    hough_offsets_kernel<<<nb, 256, 0, ctx->stream>>>(flags.p, slots.p, starts.p, sizes.p, n, max_inst, d_inst_offsets);
    B200_LAUNCHED(ctx);
    hough_members_kernel<<<nb, 256, 0, ctx->stream>>>(vin, head.p, run_id.p, run_start.p, flags.p, starts.p, n,
                                                      members.p);
    B200_LAUNCHED(ctx);
    hough_gather_points_kernel<<<nb, 256, 0, ctx->stream>>>(d_corrs, d_C, n, d_model_kp, d_scene_kp, mp.p, sp.p);
    B200_LAUNCHED(ctx);
  }
  // what follows is RANSAC, one small CTA per instance: the next scene's wide stages may start beside it
  if (ctx->wide) ctx->wide->leave();
  return dev_ransac_instances(ctx, d_corrs, mp.p, sp.p, members.p, d_inst_offsets, d_n_inst, n, bin_size, d_T, max_inst,
                              d_inst_counts, d_inst_corrs, corr_cap);
}
