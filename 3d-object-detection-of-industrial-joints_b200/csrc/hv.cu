// hv.cu — hypothesis verification: pcl::GlobalHypothesesVerification as the reference drives it after ICP
// (SHOT_hypothesis.cpp:631-653: setSceneCloud :639, addModels(registered_instances, true) :640, the set* calls
// :642-648, verify :650, getMask :651).
//
// What runs where (DESIGN.md §7b):
//   set_scene   VoxelGrid(resolution) of the scene (keypoints.cu); the full-resolution scene stays resident for the
//               scene z-buffer.
//   add_models  ZBuffering (occlusion_reasoning.hpp): focal length from the cloud's |x/z|, |y/z| extent (ordered
//               atomics), depth maps by atomic minimum — one H x 75 x 75 stack for the hypotheses' self occlusion,
//               one 100 x 100 map for the scene — then one visibility pass and an order-preserving compaction.
//   verify      radius normals of the down-sampled scene + NaN compaction; per hypothesis VoxelGrid, radius
//               normals, compaction, radius search in the scene; per scene point the explaining model point is
//               selected with one 64-bit atomicMax (PCL keeps the pair with the LARGEST squared distance — its
//               comparison starts from numeric_limits<float>::min() — ties and all-zero lists to the lowest model
//               index); weights, outlier counts; occupancy cells of the complete models by stamping a grid; then
//               SAOptimize as ONE CTA (hv_anneal_kernel): every move evaluation updates the explained / occupancy
//               arrays in parallel (indices are unique within a hypothesis), integer duplicity sums by a block
//               reduction, the float32 running values by thread 0 in PCL's order.  std::random_shuffle's rand()
//               stream and the mt19937 acceptance stream do not depend on the data, so the host generates them.
// float32 sums that PCL evaluates sequentially (getTotalExplainedInformation, add_to_explained) are evaluated
// sequentially here too (one warp: coalesced loads, the adds in lane order).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <new>
#include <random>
#include <vector>

#include "common.cuh"

struct b200_hv {
  b200_ctx *ctx = nullptr;
  b200_hv_params P;
  // scene
  int n_scene = 0;
  DevBuf<float4> scene_raw;  // full resolution (z-buffer input)
  DevBuf<float> scene_ds;    // voxel centroids, n0 x 3
  int n0 = 0;
  // models
  int H = 0;
  std::vector<int> offsets;      // H + 1, points
  DevBuf<float4> models;         // complete models, concatenated
  DevBuf<float> visible;         // visible points (x, y, z), concatenated in model order
  std::vector<int> vis_offsets;  // H + 1
  // last verify
  int ns = 0, n_cells = 0;
  std::vector<b200_hv_info> info;
  std::vector<int> list_sizes;  // per valid hypothesis: explained, occupancy
  std::vector<int> h_expl_idx, h_occ_idx;
  std::vector<float> h_expl_w;
};

namespace {

constexpr int HV_MAX_HYPOTHESES = 4096;
constexpr long long HV_MAX_CELLS = 1ll << 27;

__host__ __device__ __forceinline__ unsigned hv_enc(float f) {  // monotone float -> unsigned
#ifdef __CUDA_ARCH__
  const unsigned b = __float_as_uint(f);
#else
  unsigned b;
  memcpy(&b, &f, 4);
#endif
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float hv_dec(unsigned u) {
  const unsigned b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  float f;
  memcpy(&f, &b, 4);
  return f;
#endif
}

// ---- ZBuffering::computeDepthMap, focal length part: max / min of x/z and y/z per cloud ---------------------
// ext: per cloud {max_u, min_u, max_v, min_v} as ordered unsigned, initialised to {-FLT_MAX, FLT_MAX, ...}
__global__ void hv_extent_kernel(const float4 *__restrict__ pts, const int *__restrict__ offsets, unsigned *__restrict__ ext) {
  const int h = blockIdx.y;
  const int lo = offsets[h], hi = offsets[h + 1];
  unsigned mxu = hv_enc(-3.402823466e38f), mnu = hv_enc(3.402823466e38f), mxv = mxu, mnv = mnu;
  for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (!finite3(p.x, p.y, p.z)) continue;
    const float bx = p.x / p.z, by = p.y / p.z;
    if (bx == bx) {  // a NaN fails both of PCL's comparisons
      mxu = max(mxu, hv_enc(bx));
      mnu = min(mnu, hv_enc(bx));
    }
    if (by == by) {
      mxv = max(mxv, hv_enc(by));
      mnv = min(mnv, hv_enc(by));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mxu = max(mxu, __shfl_xor_sync(0xffffffffu, mxu, o));
    mnu = min(mnu, __shfl_xor_sync(0xffffffffu, mnu, o));
    mxv = max(mxv, __shfl_xor_sync(0xffffffffu, mxv, o));
    mnv = min(mnv, __shfl_xor_sync(0xffffffffu, mnv, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&ext[4 * h + 0], mxu);
    atomicMin(&ext[4 * h + 1], mnu);
    atomicMax(&ext[4 * h + 2], mxv);
    atomicMin(&ext[4 * h + 3], mnv);
  }
}
__global__ void hv_extent_init_kernel(unsigned *ext, int H) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  ext[4 * h + 0] = ext[4 * h + 2] = hv_enc(-3.402823466e38f);
  ext[4 * h + 1] = ext[4 * h + 3] = hv_enc(3.402823466e38f);
}

// f_ = cx / max(max(|max_u|, |max_v|), max(|min_u|, |min_v|))
__device__ __forceinline__ float hv_focal(const unsigned *ext, int res) {
  const float cx = (float)res / 2.f - 0.5f;
  const float max_u = hv_dec(ext[0]), min_u = hv_dec(ext[1]), max_v = hv_dec(ext[2]), min_v = hv_dec(ext[3]);
  const float maxC = fmaxf(fmaxf(fabsf(max_u), fabsf(max_v)), fmaxf(fabsf(min_u), fabsf(min_v)));
  return cx / maxC;
}

// int u = static_cast<int>(f_ * x / z + cx) with the bounds test of computeDepthMap / filter; non-finite or
// out-of-range values fail it (cvttss2si gives INT_MIN on the reference's platform)
__device__ __forceinline__ bool hv_pixel(float f, int res, float x, float y, float z, int *pix) {
  const float c = (float)res / 2.f - 0.5f;
  const float fu = f * x / z + c;
  const float fv = f * y / z + c;
  if (!(fu > -2147483648.f && fu < 2147483648.f) || !(fv > -2147483648.f && fv < 2147483648.f)) return false;
  const int u = __float2int_rz(fu), v = __float2int_rz(fv);
  if (u >= res || v >= res || u < 0 || v < 0) return false;
  *pix = u + v * res;
  return true;
}

// depth maps: minimum z per pixel (ordered unsigned; 0xffffffff = no return, PCL's NaN)
__global__ void hv_depth_kernel(const float4 *__restrict__ pts, const int *__restrict__ offsets,
                                const unsigned *__restrict__ ext, int res, unsigned *__restrict__ depth) {
  const int h = blockIdx.y;
  const int lo = offsets[h], hi = offsets[h + 1];
  const float f = hv_focal(ext + 4 * h, res);
  unsigned *map = depth + (size_t)h * res * res;
  for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (!finite3(p.x, p.y, p.z)) continue;
    int pix;
    if (!hv_pixel(f, res, p.x, p.y, p.z, &pix)) continue;
    atomicMin(&map[pix], hv_enc(p.z));
  }
}

// ZBuffering::filter twice: against the hypothesis' own depth map (75 x 75, margin self_thr), then against the
// scene's (margin occ_thr); a pixel without a return removes the point
__global__ void hv_visible_kernel(const float4 *__restrict__ pts, const int *__restrict__ offsets,
                                  const unsigned *__restrict__ ext_self, int res_self, const unsigned *__restrict__ depth_self,
                                  float self_thr, const unsigned *__restrict__ ext_scene, int res_scene,
                                  const unsigned *__restrict__ depth_scene, float occ_thr, int *__restrict__ flags) {
  const int h = blockIdx.y;
  const int lo = offsets[h], hi = offsets[h + 1];
  const float fs = hv_focal(ext_self + 4 * h, res_self);
  const float fc = hv_focal(ext_scene, res_scene);
  const unsigned *map = depth_self + (size_t)h * res_self * res_self;
  for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    int keep = 0;
    if (finite3(p.x, p.y, p.z)) {
      int pix;
      if (hv_pixel(fs, res_self, p.x, p.y, p.z, &pix)) {
        const unsigned d = map[pix];
        if (d != 0xffffffffu && !((p.z - self_thr) > hv_dec(d))) {
          if (hv_pixel(fc, res_scene, p.x, p.y, p.z, &pix)) {
            const unsigned e = depth_scene[pix];
            if (e != 0xffffffffu && !((p.z - occ_thr) > hv_dec(e))) keep = 1;
          }
        }
      }
    }
    flags[i] = keep;
  }
}

__global__ void hv_all_finite_flags_kernel(const float4 *__restrict__ pts, int n, int *__restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = finite3(pts[i].x, pts[i].y, pts[i].z) ? 1 : 0;
}

__global__ void hv_compact_points_kernel(const float4 *__restrict__ pts, int n, const int *__restrict__ flags,
                                         const int *__restrict__ slots, float *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !flags[i]) return;
  const int s = slots[i];
  out[3 * (size_t)s + 0] = pts[i].x;
  out[3 * (size_t)s + 1] = pts[i].y;
  out[3 * (size_t)s + 2] = pts[i].z;
}

// visible offsets: the scan value at every model's first point (the total for empty models at the end)
__global__ void hv_gather_slots_kernel(const int *__restrict__ slots, const int *__restrict__ total, int n,
                                       const int *__restrict__ offsets, int H, int *__restrict__ out) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h > H) return;
  out[h] = (h == H || offsets[h] >= n) ? *total : slots[offsets[h]];
}

// ---- NaN-normal compaction (initialize / addModel: "check nans...") -----------------------------------------
__global__ void hv_normal_flags_kernel(const float4 *__restrict__ nrm, int n, int *__restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = finite3(nrm[i].x, nrm[i].y, nrm[i].z) ? 1 : 0;
}
__global__ void hv_compact_cloud_kernel(const float *__restrict__ xyz, const float4 *__restrict__ nrm, int n,
                                        const int *__restrict__ flags, const int *__restrict__ slots,
                                        float4 *__restrict__ out_pts, float4 *__restrict__ out_nrm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !flags[i]) return;
  const int s = slots[i];
  out_pts[s] = make_float4(xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], 1.f);
  out_nrm[s] = nrm[i];
}

// ---- addModel: outliers and the explaining model point of every scene point ----------------------------------
__global__ void hv_outlier_count_kernel(const int *__restrict__ counts, int nm, int *__restrict__ n_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = (i < nm && counts[i] == 0) ? 1 : 0;
  const int w = warp_sum(c);
  if ((threadIdx.x & 31) == 0 && w) atomicAdd(n_out, w);
}
// key = (squared distance if > FLT_MIN else 0) : (0xffffffff - model index): the maximum is PCL's "closest"
__global__ void hv_explain_kernel(const long long *__restrict__ offsets, const int *__restrict__ idx,
                                  const float *__restrict__ d2, int nm, unsigned long long *__restrict__ best) {
  const int i = blockIdx.x;
  if (i >= nm) return;
  const long long lo = offsets[i], hi = offsets[i + 1];
  for (long long k = lo + threadIdx.x; k < hi; k += blockDim.x) {
    const float d = d2[k];
    const unsigned hi32 = d > 1.17549435e-38f ? __float_as_uint(d) : 0u;
    const unsigned long long key = ((unsigned long long)hi32 << 32) | (unsigned long long)(0xffffffffu - (unsigned)i);
    atomicMax(&best[idx[k]], key);
  }
}
__global__ void hv_explained_flags_kernel(const unsigned long long *__restrict__ best, int ns, int *__restrict__ flags) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < ns) flags[j] = best[j] != 0ull ? 1 : 0;
}
// explained_ / explained_distances_ in ascending scene index (std::map order)
__global__ void hv_explained_emit_kernel(const unsigned long long *__restrict__ best, int ns, const int *__restrict__ flags,
                                         const int *__restrict__ slots, const float4 *__restrict__ scene_pts,
                                         const float4 *__restrict__ scene_nrm, const float4 *__restrict__ model_pts,
                                         const float4 *__restrict__ model_nrm, float inlier_thr, int *__restrict__ out_idx,
                                         float *__restrict__ out_w) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= ns || !flags[j]) return;
  const int i = (int)(0xffffffffu - (unsigned)(best[j] & 0xffffffffull));
  const float4 s = scene_pts[j], m = model_pts[i];
  const float d = sqdist3(m.x, m.y, m.z, s.x, s.y, s.z);  // the search's value for this pair
  const float d_weight = -(d * d / inlier_thr) + 1.f;
  const float4 sn = scene_nrm[j], mn = model_nrm[i];
  float dotp = ((sn.x * mn.x + sn.y * mn.y) + sn.z * mn.z) * 1.f;
  if (dotp < 0.f) dotp = 0.f;
  out_idx[slots[j]] = j;
  out_w[slots[j]] = d_weight * dotp;
}

// ---- occupancy grid of the complete models ---------------------------------------------------------------------
__global__ void hv_bounds_kernel(const float4 *__restrict__ pts, int lo, int hi, unsigned *__restrict__ box) {
  unsigned mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u};
  for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (!finite3(p.x, p.y, p.z)) continue;
    const unsigned e[3] = {hv_enc(p.x), hv_enc(p.y), hv_enc(p.z)};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = min(mn[a], e[a]);
      mx[a] = max(mx[a], e[a]);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&box[a], mn[a]);
      atomicMax(&box[3 + a], mx[a]);
    }
  }
}
// first point of hypothesis v (stamp v + 1) to reach a cell appends it to the hypothesis' list
__global__ void hv_occupancy_kernel(const float4 *__restrict__ pts, int lo, int hi, float mnx, float mny, float mnz, float res,
                                    int sx, int sy, int stamp_value, int *__restrict__ stamp, int *__restrict__ out_idx,
                                    int *__restrict__ out_count) {
  const int i = lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hi) return;
  const float4 p = pts[i];
  if (!finite3(p.x, p.y, p.z)) return;
  const int px = (int)floorf((p.x - mnx) / res);
  const int py = (int)floorf((p.y - mny) / res);
  const int pz = (int)floorf((p.z - mnz) / res);
  const int idx = pz * sx * sy + py * sx + px;
  if (atomicMax(&stamp[idx], stamp_value) < stamp_value) out_idx[atomicAdd(out_count, 1)] = idx;
}

// ---- SAOptimize ----------------------------------------------------------------------------------------------
struct HvExpl {
  const int *idx;
  const float *w;
  int n;
};
struct HvOcc {
  const int *idx;
  int n;
};
struct AnnealArgs {
  int H, ns;
  const HvExpl *expl;
  const HvOcc *occ;
  const float *outliers_weight;
  const int *bad_information;
  float w_cm;
  int *explained;     // ns, zero
  float *weighted;    // ns, zero
  int *occupancy;     // n_cells, zero
  float *seq_sum;     // H scratch: add_to_explained of every hypothesis
  float *compact;     // ns scratch: the weights of the explained points, in order
  const int *perms;   // n_iter x H: the move order of every iteration (std::random_shuffle, cumulative)
  const unsigned *mt; // n_iter x H raw mt19937 outputs
  int n_iter;         // iterations until the temperature falls to 1e-7
  int max_iterations; // noimprove_termination_criteria
  double initial_temp;
  int uniform_mode;
  unsigned char *active;  // H
  unsigned char *best;    // H
  double *out_cost;
  int *out_accepted;
};

constexpr int HV_SA_THREADS = 1024;

// sequential float32 sum of v[0..n) (optionally only where gate[i] > 0) by one warp: coalesced loads, the additions in
// index order on lane 0's accumulator
__device__ float hv_seq_sum_warp(const float *v, const int *gate, int n, float acc) {
  const int lane = threadIdx.x & 31;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    float x = 0.f;
    bool on = false;
    if (i < n) {
      on = gate ? gate[i] > 0 : true;
      x = v[i];
    }
    const unsigned m = __ballot_sync(0xffffffffu, on);
#pragma unroll 8
    for (int l = 0; l < 32; ++l) {
      const float y = __shfl_sync(0xffffffffu, x, l);
      if ((m >> l) & 1u) acc += y;
    }
  }
  return acc;
}

__device__ __forceinline__ int hv_dup_rule(int prev, int cur, int sgn) {
  const bool prev_dup = prev > 1;
  if (cur > 1 && prev_dup) return sgn;
  if (cur == 1 && prev_dup) return -2;
  if (cur > 1 && !prev_dup) return 2;
  return 0;
}

// block sum of two ints; result valid on thread 0; ends with a barrier
__device__ void hv_block_sum2(int a, int b, int *red, int *oa, int *ob) {
  a = warp_sum(a);
  b = warp_sum(b);
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    red[2 * w] = a;
    red[2 * w + 1] = b;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int sa = 0, sb = 0;
    for (int i = 0; i < HV_SA_THREADS / 32; ++i) {
      sa += red[2 * i];
      sb += red[2 * i + 1];
    }
    *oa = sa;
    *ob = sb;
  }
  __syncthreads();
}

// A move is evaluated without touching the arrays: the duplicity changes are integer functions of the current
// counts, the float32 running values live on thread 0, and PCL's explained_by_RM_distance_weighted is never read
// again after the initial total.  The counts only change when a move is accepted, and an accepted move ends the
// iteration — so all H moves are evaluated at once, and only after an accepted move (phase A); thread 0 replays
// PCL's sequence over the shuffled order on the running values: apply, test, unapply (the float32 round trip
// (v + a) - a is kept as PCL computes it; the unapply's duplicity changes are the exact negatives of the apply's) up
// to the first accepted move (phase B), and the block writes that move's counts (phase C).  An iteration that
// accepts nothing costs two barriers and H scalar evaluations.
__global__ void __launch_bounds__(HV_SA_THREADS) hv_anneal_kernel(AnnealArgs A) {
  __shared__ int red[2 * (HV_SA_THREADS / 32)];
  __shared__ int s_d0[HV_MAX_HYPOTHESES], s_d1[HV_MAX_HYPOTHESES];
  __shared__ int s_a, s_b, s_ctl, s_stop;
  // per-hypothesis scalars, the current iteration's move order and the mask live in shared memory: thread 0's replay
  // of an iteration is a chain of dependent reads, which through global memory cost more than its arithmetic
  extern __shared__ __align__(16) unsigned char s_dyn[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int H = A.H;
  float *s_seq = reinterpret_cast<float *>(s_dyn);  // add_to_explained of every hypothesis
  float *s_obad = s_seq + H;                         // outliers_weight_ * bad_information_
  int *s_perm = reinterpret_cast<int *>(s_obad + H);
  unsigned char *s_act = reinterpret_cast<unsigned char *>(s_perm + H);
  // ---- initial state: every hypothesis active
  for (int h = tid; h < H; h += HV_SA_THREADS) {
    s_act[h] = 1, A.best[h] = 1;
    s_obad[h] = A.outliers_weight[h] * (float)A.bad_information[h];
  }
  for (int h = 0; h < H; ++h) {
    const HvExpl e = A.expl[h];
    for (int k = tid; k < e.n; k += HV_SA_THREADS) {
      const int j = e.idx[k];
      A.explained[j] += 1;
      A.weighted[j] += e.w[k];
    }
    const HvOcc o = A.occ[h];
    for (int k = tid; k < o.n; k += HV_SA_THREADS) A.occupancy[o.idx[k]] += 1;
    __syncthreads();
  }
  // duplicity = sum of explained[i] over i with explained[i] > 1 = number of (hypothesis, point) entries on such
  // points; likewise the occupied-multiple count of the complete-model grid
  int dup = 0, cm = 0;
  for (int h = 0; h < H; ++h) {
    const HvExpl e = A.expl[h];
    for (int k = tid; k < e.n; k += HV_SA_THREADS) dup += A.explained[e.idx[k]] > 1 ? 1 : 0;
    const HvOcc o = A.occ[h];
    for (int k = tid; k < o.n; k += HV_SA_THREADS) cm += A.occupancy[o.idx[k]] > 1 ? 1 : 0;
  }
  hv_block_sum2(dup, cm, red, &s_a, &s_b);
  // getTotalExplainedInformation adds weighted[i] over the explained points in ascending i: the few explained points
  // (a few per cent of the scene) are first compacted in order by the whole block — every thread a contiguous chunk,
  // counts scanned across the block — so that the sequential float32 sum only walks those
  int n_compact = 0;
  {
    const int chunk = (A.ns + HV_SA_THREADS - 1) / HV_SA_THREADS;
    const int lo = min(tid * chunk, A.ns), hi = min(lo + chunk, A.ns);
    int c = 0;
    for (int i = lo; i < hi; ++i) c += A.explained[i] > 0 ? 1 : 0;
    int incl = c;  // inclusive scan over the block: warp scan, then the warp totals
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) red[tid >> 5] = incl;
    __syncthreads();
    int base = 0;
    for (int w = 0; w < (tid >> 5); ++w) base += red[w];
    for (int w = 0; w < HV_SA_THREADS / 32; ++w) n_compact += red[w];
    int o = base + incl - c;
    for (int i = lo; i < hi; ++i)
      if (A.explained[i] > 0) A.compact[o++] = A.weighted[i];
    __syncthreads();
  }
  // sequential sums (warp 0)
  float good_information = 0.f;
  if (tid < 32) {
    for (int h = 0; h < H; ++h) {
      const float s = hv_seq_sum_warp(A.expl[h].w, nullptr, A.expl[h].n, 0.f);
      if (tid == 0) s_seq[h] = s;
    }
    good_information = hv_seq_sum_warp(A.compact, nullptr, n_compact, 0.f);
  }
  __syncthreads();
  // thread 0 carries PCL's running values
  float previous_explained = 0.f, previous_bad = 0.f;
  const float previous_unexplained = 0.f;
  int previous_dup = 0, previous_cm = 0, n_active = H, accepted = 0;
  double cost = 0.0, best_cost = 0.0, crit_best = 1.7976931348623157e308, temp = A.initial_temp;
  int iterations_left = A.max_iterations, mt_pos = 0;
  if (tid == 0) {
    previous_explained = good_information;
    previous_dup = s_a;
    previous_cm = s_b;
    for (int h = 0; h < H; ++h) previous_bad += s_obad[h];
    cost = (double)((previous_explained - previous_bad - (float)previous_dup - (float)previous_cm * A.w_cm - (float)H -
                     previous_unexplained) *
                    -1.f);
    best_cost = cost;
  }
  // evaluateSolution's value from the running values (thread 0)
  auto scalar_flip = [&](int m, int sgn, int d0, int d1) {
    const float sign = (float)sgn;
    n_active += sgn;
    previous_explained += s_seq[m] * sign;
    previous_dup += d0;
    previous_cm += d1;
    const float bad_info = previous_bad + s_obad[m] * sign;
    previous_bad = bad_info;
    const float duplicity_cm = (float)previous_cm * A.w_cm;
    cost = (double)((previous_explained - bad_info - (float)previous_dup - previous_unexplained - duplicity_cm -
                     (float)n_active) *
                    -1.f);
  };
  bool dirty = true;  // the counts changed since the moves were last evaluated (uniform over the block)
  for (int it = 0; it < A.n_iter; ++it) {
    if (tid == 0) {  // noimprove_termination_criteria, then the temperature test
      int stop = 0;
      if (cost < crit_best - 1e-7) {
        crit_best = cost;
        iterations_left = A.max_iterations;
      }
      if (iterations_left <= 0) stop = 1;
      --iterations_left;
      if (!(temp > 1e-7)) stop = 1;
      s_stop = stop;
    }
    for (int h = tid; h < H; h += HV_SA_THREADS) s_perm[h] = A.perms[(size_t)it * H + h];
    __syncthreads();  // also orders the previous iteration's count writes before the reads below
    if (s_stop) break;
    // ---- phase A (only after the counts changed): duplicity changes of every move against the current counts; the
    // block strides over one list after the other, per-move sums by shared-memory atomics, no barrier in between
    if (dirty) {
      for (int h = tid; h < H; h += HV_SA_THREADS) s_d0[h] = 0, s_d1[h] = 0;
      __syncthreads();
      for (int m = 0; m < H; ++m) {
        const int sgn = s_act[m] ? -1 : 1;
        int d0 = 0, d1 = 0;
        const HvExpl e = A.expl[m];
        for (int k = tid; k < e.n; k += HV_SA_THREADS) {
          const int prev = A.explained[e.idx[k]];
          d0 += hv_dup_rule(prev, prev + sgn, sgn);
        }
        const HvOcc o = A.occ[m];
        for (int k = tid; k < o.n; k += HV_SA_THREADS) {
          const int prev = A.occupancy[o.idx[k]];
          d1 += hv_dup_rule(prev, prev + sgn, sgn);
        }
        d0 = warp_sum(d0);
        d1 = warp_sum(d1);
        if (lane == 0) {
          if (d0) atomicAdd(&s_d0[m], d0);
          if (d1) atomicAdd(&s_d1[m], d1);
        }
      }
      __syncthreads();
    }
    // ---- phase B: PCL's sequence over the shuffled moves, up to the first accepted one
    if (tid == 0) {
      const double actual_cost = cost;
      int taken = -1;
      for (int mi = 0; mi < H; ++mi) {
        const int m = s_perm[mi];
        const int sgn = s_act[m] ? -1 : 1;
        scalar_flip(m, sgn, s_d0[m], s_d1[m]);  // apply_and_evaluate
        const double delta = cost - actual_cost;
        bool take = delta < 0;
        if (!take) {
          const unsigned x = A.mt[mt_pos++];
          // u < exp(-2 delta / T).  Every non-zero variate is at least 2^-32 = 2.3e-10 > exp(-22): when the exponent
          // is below -25 (most evaluations once the temperature has fallen) the outcome is "rejected" without the
          // float64 division and exponential, which were most of an iteration's serial time
          if (x == 0u || !(2.0 * delta > 25.0 * temp)) {
            const double u = A.uniform_mode == 1 ? (double)x : (double)x / 4294967296.0;
            take = u < exp(2.0 * -delta / temp);
          }
        }
        if (take) {
          accepted++;
          s_act[m] = sgn > 0 ? 1 : 0;
          taken = m;
          if (cost < best_cost) {
            best_cost = cost;
            taken |= 0x40000000;  // also a new best
          }
          break;
        }
        scalar_flip(m, -sgn, -s_d0[m], -s_d1[m]);  // unapply
      }
      s_ctl = taken;
      temp *= 0.95;
    }
    __syncthreads();
    // ---- phase C: the accepted move's counts
    const int ctl = s_ctl;
    if (ctl >= 0) {
      const int m = ctl & 0x3fffffff;
      const int sgn = s_act[m] ? 1 : -1;  // the state after the flip
      const HvExpl e = A.expl[m];
      for (int k = tid; k < e.n; k += HV_SA_THREADS) A.explained[e.idx[k]] += sgn;
      const HvOcc o = A.occ[m];
      for (int k = tid; k < o.n; k += HV_SA_THREADS) A.occupancy[o.idx[k]] += sgn;
      if (ctl & 0x40000000)
        for (int h = tid; h < H; h += HV_SA_THREADS) A.best[h] = s_act[h];
    }
    dirty = ctl >= 0;
  }
  if (tid == 0) {
    *A.out_cost = best_cost;
    *A.out_accepted = accepted;
  }
}

// glibc rand() (TYPE_3): the stream std::random_shuffle draws from
struct GlibcRand {
  uint32_t st[31];
  explicit GlibcRand(unsigned seed) {
    if (seed == 0) seed = 1;
    std::vector<uint32_t> r(344);
    int32_t word = (int32_t)seed;
    r[0] = (uint32_t)word;
    for (int i = 1; i < 31; ++i) {
      const int64_t hi = word / 127773, lo = word % 127773;
      int64_t w = 16807 * lo - 2836 * hi;
      if (w < 0) w += 2147483647;
      word = (int32_t)w;
      r[i] = (uint32_t)word;
    }
    for (int i = 31; i < 34; ++i) r[i] = r[i - 31];
    for (int i = 34; i < 344; ++i) r[i] = r[i - 31] + r[i - 3];
    for (int i = 0; i < 31; ++i) st[i] = r[313 + i];
  }
  int next() {
    const uint32_t o = st[0] + st[28];
    for (int i = 0; i < 30; ++i) st[i] = st[i + 1];
    st[30] = o;
    return (int)(o >> 1);
  }
};

template <class T>
int hv_upload(b200_ctx *ctx, DevBuf<T> &buf, const T *host, size_t count) {
  B200_TRY(buf.alloc(ctx, count));
  if (count) B200_CUDA(ctx, cudaMemcpyAsync(buf.p, host, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return B200_OK;
}
template <class T>
int hv_download(b200_ctx *ctx, T *host, const T *dev, size_t count) {
  if (count) {
    B200_CUDA(ctx, ctx->sync());
    B200_CUDA(ctx, cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(ctx, ctx->sync());
  }
  return B200_OK;
}

// device lists -> the annealing kernel -> mask
int run_anneal(b200_ctx *ctx, int H, int ns, const std::vector<HvExpl> &expl, const std::vector<HvOcc> &occ, int n_cells,
               const float *h_outliers_weight, const int *h_bad, const b200_hv_params &P, unsigned char *mask,
               double *best_cost, int *accepted) {
  if (H > HV_MAX_HYPOTHESES) return ctx->fail(B200_ERR_CAPACITY, "hv: more than 4096 hypotheses");
  // iterations until the temperature reaches the stop value (linear_cooling: t *= 0.95; stop 1e-7)
  int n_iter = 0;
  for (double t = (double)P.initial_temp; t > 1e-7 && n_iter < (1 << 20); t *= 0.95) ++n_iter;
  if ((long long)n_iter * H > (1ll << 24)) return ctx->fail(B200_ERR_CAPACITY, "hv: annealing schedule too long");
  std::vector<int> perms((size_t)std::max(n_iter * H, 1)), moves((size_t)H);
  std::vector<unsigned> mt((size_t)std::max(n_iter * H, 1));
  for (int i = 0; i < H; ++i) moves[i] = i;
  GlibcRand rnd(P.rand_seed);
  for (int it = 0; it < n_iter; ++it) {
    for (int i = 1; i < H; ++i) {  // std::random_shuffle (libstdc++)
      const int j = rnd.next() % (i + 1);
      if (i != j) std::swap(moves[i], moves[j]);
    }
    memcpy(&perms[(size_t)it * H], moves.data(), sizeof(int) * (size_t)H);
  }
  std::mt19937 rng(P.mt_seed);
  for (auto &x : mt) x = (unsigned)rng();
  DevBuf<HvExpl> d_expl;
  DevBuf<HvOcc> d_occ;
  DevBuf<float> d_ow, d_weighted, d_seq, d_compact;
  DevBuf<int> d_bad, d_explained, d_occupancy, d_perms, d_acc;
  DevBuf<unsigned> d_mt;
  DevBuf<unsigned char> d_active, d_best;
  DevBuf<double> d_cost;
  B200_TRY(hv_upload(ctx, d_expl, expl.data(), (size_t)H));
  B200_TRY(hv_upload(ctx, d_occ, occ.data(), (size_t)H));
  B200_TRY(hv_upload(ctx, d_ow, h_outliers_weight, (size_t)H));
  B200_TRY(hv_upload(ctx, d_bad, h_bad, (size_t)H));
  B200_TRY(hv_upload(ctx, d_perms, perms.data(), perms.size()));
  B200_TRY(hv_upload(ctx, d_mt, mt.data(), mt.size()));
  B200_TRY(d_weighted.alloc(ctx, (size_t)std::max(ns, 1)));
  B200_TRY(d_explained.alloc(ctx, (size_t)std::max(ns, 1)));
  B200_TRY(d_occupancy.alloc(ctx, (size_t)std::max(n_cells, 1)));
  B200_TRY(d_seq.alloc(ctx, (size_t)H));
  B200_TRY(d_compact.alloc(ctx, (size_t)std::max(ns, 1)));
  B200_TRY(d_active.alloc(ctx, (size_t)H));
  B200_TRY(d_best.alloc(ctx, (size_t)H));
  B200_TRY(d_cost.alloc(ctx, 1));
  B200_TRY(d_acc.alloc(ctx, 1));
  B200_TRY(d_weighted.zero());
  B200_TRY(d_explained.zero());
  B200_TRY(d_occupancy.zero());
  AnnealArgs A;
  A.H = H, A.ns = ns, A.expl = d_expl.p, A.occ = d_occ.p, A.outliers_weight = d_ow.p, A.bad_information = d_bad.p;
  A.w_cm = P.w_occupied_multiple_cm, A.explained = d_explained.p, A.weighted = d_weighted.p, A.occupancy = d_occupancy.p;
  A.seq_sum = d_seq.p, A.compact = d_compact.p, A.perms = d_perms.p, A.mt = d_mt.p, A.n_iter = n_iter, A.max_iterations = P.max_iterations;
  A.initial_temp = (double)P.initial_temp, A.uniform_mode = P.sa_uniform_mode, A.active = d_active.p, A.best = d_best.p;
  A.out_cost = d_cost.p, A.out_accepted = d_acc.p;
  const size_t dyn = (size_t)H * 13 + 16;
  B200_CUDA(ctx, ensure_dyn_smem(hv_anneal_kernel, dyn));
  hv_anneal_kernel<<<1, HV_SA_THREADS, dyn, ctx->stream>>>(A);
  B200_LAUNCHED(ctx);
  B200_TRY(hv_download(ctx, mask, d_best.p, (size_t)H));
  double c;
  int a;
  B200_TRY(hv_download(ctx, &c, d_cost.p, 1));
  B200_TRY(hv_download(ctx, &a, d_acc.p, 1));
  if (best_cost) *best_cost = c;
  if (accepted) *accepted = a;
  return B200_OK;
}

int check_hv_params(b200_ctx *ctx, const b200_hv_params &P) {
  if (!(P.resolution > 0.f) || !(P.inlier_threshold > 0.f) || !(P.radius_normals > 0.f) || !(P.res_occupancy_grid > 0.f) ||
      !(P.initial_temp > 0.f) || P.zbuffer_scene_resolution < 1 || P.zbuffer_scene_resolution > 4096 ||
      P.zbuffer_self_resolution < 1 || P.zbuffer_self_resolution > 1024 || P.sa_uniform_mode < 0 || P.sa_uniform_mode > 1)
    return ctx->fail(B200_ERR_INVALID, "hv: bad parameters");
  return B200_OK;
}

// radius normals of a device cloud (xyz rows, n x 3) on itself, rows with a NaN normal dropped:
// out_pts / out_nrm hold *n_out compacted rows
int normals_and_compact(b200_ctx *ctx, const float *d_xyz, int n, double radius, DevBuf<float4> &out_pts,
                        DevBuf<float4> &out_nrm, int *n_out) {
  *n_out = 0;
  B200_TRY(out_pts.alloc(ctx, (size_t)std::max(n, 1)));
  B200_TRY(out_nrm.alloc(ctx, (size_t)std::max(n, 1)));
  if (n <= 0) return B200_OK;
  std::unique_ptr<b200_cloud> cloud;
  B200_TRY(cloud_upload(ctx, d_xyz, n, 3, true, cloud));
  DevBuf<float> nrm;
  DevBuf<int> flags, slots, total;
  B200_TRY(nrm.alloc(ctx, (size_t)n * 4));
  B200_TRY(flags.alloc(ctx, (size_t)n));
  B200_TRY(slots.alloc(ctx, (size_t)n));
  B200_TRY(total.alloc(ctx, 1));
  B200_TRY(dev_normals(ctx, cloud.get(), cloud->raw.p, n, true, 0, radius, nullptr, nrm.p));
  hv_normal_flags_kernel<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(reinterpret_cast<const float4 *>(nrm.p), n, flags.p);
  B200_LAUNCHED(ctx);
  B200_TRY(exclusive_scan_i32(ctx, flags.p, slots.p, n, total.p));
  hv_compact_cloud_kernel<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(d_xyz, reinterpret_cast<const float4 *>(nrm.p), n, flags.p,
                                                                    slots.p, out_pts.p, out_nrm.p);
  B200_LAUNCHED(ctx);
  B200_TRY(readback_small(ctx, total.p, n_out, sizeof(int)));
  return B200_OK;
}

}  // namespace

extern "C" {

void b200_hv_params_default(b200_hv_params *p) {
  if (!p) return;
  // HypothesisVerification / GlobalHypothesesVerification constructors
  p->resolution = 0.005f;
  p->inlier_threshold = 0.005f;
  p->occlusion_threshold = 0.005f;
  p->regularizer = 1.f;
  p->radius_normals = 0.01f;
  p->res_occupancy_grid = 0.01f;
  p->w_occupied_multiple_cm = 4.f;
  p->initial_temp = 1000.f;
  p->max_iterations = 5000;
  p->occlusion_reasoning = 0;
  p->zbuffer_scene_resolution = 100;
  p->zbuffer_self_resolution = 75;
  p->self_occlusion_threshold = 0.005f;
  p->detect_clutter = 1;
  p->radius_clutter = 0.03f;
  p->clutter_regularizer = 5.f;
  p->rand_seed = 1u;
  p->mt_seed = 5489u;
  p->sa_uniform_mode = 0;
}

int b200_hv_create(b200_ctx *ctx, const b200_hv_params *p, b200_hv **out) {
  if (!ctx || !out) return B200_ERR_INVALID;
  b200_hv *hv = new (std::nothrow) b200_hv();
  if (!hv) return ctx->fail(B200_ERR_NOMEM, "hv: out of host memory");
  hv->ctx = ctx;
  if (p)
    hv->P = *p;
  else
    b200_hv_params_default(&hv->P);
  *out = hv;
  return B200_OK;
}

int b200_hv_destroy(b200_hv *hv) {
  delete hv;
  return B200_OK;
}

int b200_hv_set_params(b200_hv *hv, const b200_hv_params *p) {
  if (!hv || !p) return B200_ERR_INVALID;
  hv->P = *p;
  return B200_OK;
}

int b200_hv_set_scene(b200_ctx *ctx, b200_hv *hv, const float *scene_xyz, int n, int stride) {
  if (!ctx || !hv || hv->ctx != ctx) return B200_ERR_INVALID;
  if (n < 0 || stride < 3 || (n > 0 && !scene_xyz)) return ctx->fail(B200_ERR_INVALID, "hv_set_scene: bad arguments");
  B200_CUDA(ctx, cudaSetDevice(ctx->device));
  B200_TRY(check_hv_params(ctx, hv->P));
  try {
    // setSceneCloud clears the models
    hv->H = 0;
    hv->offsets.clear();
    hv->vis_offsets.clear();
    hv->n_scene = n;
    hv->n0 = 0;
    DevBuf<float> stage;
    B200_TRY(hv_upload(ctx, stage, scene_xyz, (size_t)n * stride));
    B200_TRY(hv->scene_raw.alloc(ctx, (size_t)std::max(n, 1)));
    B200_TRY(hv->scene_ds.alloc(ctx, (size_t)std::max(n, 1) * 3));
    if (n == 0) return B200_OK;
    B200_TRY(pack_points(ctx, stage.p, n, stride, hv->scene_raw.p));
    DevBuf<int> cnt;
    B200_TRY(cnt.alloc(ctx, 1));
    B200_TRY(dev_voxel_grid(ctx, stage.p, n, stride, hv->P.resolution, hv->P.resolution, hv->P.resolution, hv->scene_ds.p,
                            cnt.p));
    B200_TRY(readback_small(ctx, cnt.p, &hv->n0, sizeof(int)));
  } catch (const std::bad_alloc &) {
    return ctx->fail(B200_ERR_NOMEM, "hv: out of host memory");
  }
  return B200_OK;
}

int b200_hv_add_models(b200_ctx *ctx, b200_hv *hv, const float *models_xyz, const int *model_offsets, int H, int stride,
                       int occlusion_reasoning) {
  if (!ctx || !hv || hv->ctx != ctx) return B200_ERR_INVALID;
  if (H < 0 || stride < 3 || !model_offsets || model_offsets[0] != 0)
    return ctx->fail(B200_ERR_INVALID, "hv_add_models: bad arguments");
  for (int h = 0; h < H; ++h)
    if (model_offsets[h + 1] < model_offsets[h]) return ctx->fail(B200_ERR_INVALID, "hv_add_models: offsets must not decrease");
  const int total = model_offsets[H];
  if (total > 0 && !models_xyz) return ctx->fail(B200_ERR_INVALID, "hv_add_models: null models");
  if (H > HV_MAX_HYPOTHESES) return ctx->fail(B200_ERR_CAPACITY, "hv: more than 4096 hypotheses");
  B200_CUDA(ctx, cudaSetDevice(ctx->device));
  B200_TRY(check_hv_params(ctx, hv->P));
  try {
    hv->H = H;
    hv->offsets.assign(model_offsets, model_offsets + H + 1);
    hv->vis_offsets.assign((size_t)H + 1, 0);
    B200_TRY(hv->models.alloc(ctx, (size_t)std::max(total, 1)));
    B200_TRY(hv->visible.alloc(ctx, (size_t)std::max(total, 1) * 3));
    if (H == 0 || total == 0) return B200_OK;
    {
      DevBuf<float> stage;
      B200_TRY(hv_upload(ctx, stage, models_xyz, (size_t)total * stride));
      B200_TRY(pack_points(ctx, stage.p, total, stride, hv->models.p));
    }
    DevBuf<int> d_off, flags, slots, tot, d_vis;
    B200_TRY(hv_upload(ctx, d_off, model_offsets, (size_t)H + 1));
    B200_TRY(flags.alloc(ctx, (size_t)total));
    B200_TRY(slots.alloc(ctx, (size_t)total));
    B200_TRY(tot.alloc(ctx, 1));
    B200_TRY(d_vis.alloc(ctx, (size_t)H + 1));
    int max_len = 0;
    for (int h = 0; h < H; ++h) max_len = std::max(max_len, model_offsets[h + 1] - model_offsets[h]);
    const dim3 grid((unsigned)std::max(1, std::min(ceil_div(max_len, 256), 64)), (unsigned)H);
    if (!occlusion_reasoning) {
      hv_all_finite_flags_kernel<<<ceil_div(total, 256), 256, 0, ctx->stream>>>(hv->models.p, total, flags.p);
      B200_LAUNCHED(ctx);
    } else {
      if (hv->n_scene <= 0) return ctx->fail(B200_ERR_INVALID, "hv_add_models: setSceneCloud must come first");
      const int rs = hv->P.zbuffer_scene_resolution, rm = hv->P.zbuffer_self_resolution;
      DevBuf<unsigned> ext_scene, ext_self, depth_scene, depth_self;
      DevBuf<int> scene_off;
      B200_TRY(ext_scene.alloc(ctx, 4));
      B200_TRY(ext_self.alloc(ctx, (size_t)H * 4));
      B200_TRY(depth_scene.alloc(ctx, (size_t)rs * rs));
      B200_TRY(depth_self.alloc(ctx, (size_t)H * rm * rm));
      const int so[2] = {0, hv->n_scene};
      B200_TRY(scene_off.alloc(ctx, 2));
      B200_TRY(write_small(ctx, scene_off.p, so, sizeof(so)));
      B200_CUDA(ctx, cudaMemsetAsync(depth_scene.p, 0xff, sizeof(unsigned) * (size_t)rs * rs, ctx->stream));
      B200_CUDA(ctx, cudaMemsetAsync(depth_self.p, 0xff, sizeof(unsigned) * (size_t)H * rm * rm, ctx->stream));
      hv_extent_init_kernel<<<1, 32, 0, ctx->stream>>>(ext_scene.p, 1);
      B200_LAUNCHED(ctx);
      hv_extent_init_kernel<<<ceil_div(H, 256), 256, 0, ctx->stream>>>(ext_self.p, H);
      B200_LAUNCHED(ctx);
      const dim3 sgrid((unsigned)std::min(ceil_div(hv->n_scene, 256), ctx->sm_count * 8), 1u);
      hv_extent_kernel<<<sgrid, 256, 0, ctx->stream>>>(hv->scene_raw.p, scene_off.p, ext_scene.p);
      B200_LAUNCHED(ctx);
      hv_depth_kernel<<<sgrid, 256, 0, ctx->stream>>>(hv->scene_raw.p, scene_off.p, ext_scene.p, rs, depth_scene.p);
      B200_LAUNCHED(ctx);
      hv_extent_kernel<<<grid, 256, 0, ctx->stream>>>(hv->models.p, d_off.p, ext_self.p);
      B200_LAUNCHED(ctx);
      hv_depth_kernel<<<grid, 256, 0, ctx->stream>>>(hv->models.p, d_off.p, ext_self.p, rm, depth_self.p);
      B200_LAUNCHED(ctx);
      hv_visible_kernel<<<grid, 256, 0, ctx->stream>>>(hv->models.p, d_off.p, ext_self.p, rm, depth_self.p,
                                                       hv->P.self_occlusion_threshold, ext_scene.p, rs, depth_scene.p,
                                                       hv->P.occlusion_threshold, flags.p);
      B200_LAUNCHED(ctx);
    }
    B200_TRY(exclusive_scan_i32(ctx, flags.p, slots.p, total, tot.p));
    hv_compact_points_kernel<<<ceil_div(total, 256), 256, 0, ctx->stream>>>(hv->models.p, total, flags.p, slots.p,
                                                                           hv->visible.p);
    B200_LAUNCHED(ctx);
    hv_gather_slots_kernel<<<ceil_div(H + 1, 256), 256, 0, ctx->stream>>>(slots.p, tot.p, total, d_off.p, H, d_vis.p);
    B200_LAUNCHED(ctx);
    B200_TRY(hv_download(ctx, hv->vis_offsets.data(), d_vis.p, (size_t)H + 1));
  } catch (const std::bad_alloc &) {
    return ctx->fail(B200_ERR_NOMEM, "hv: out of host memory");
  }
  return B200_OK;
}

int b200_hv_verify(b200_ctx *ctx, b200_hv *hv, unsigned char *mask, b200_hv_info *info, double *best_cost,
                   int *accepted_moves) {
  if (!ctx || !hv || hv->ctx != ctx) return B200_ERR_INVALID;
  const int H = hv->H;
  if (H > 0 && !mask) return ctx->fail(B200_ERR_INVALID, "hv_verify: null mask");
  B200_CUDA(ctx, cudaSetDevice(ctx->device));
  B200_TRY(check_hv_params(ctx, hv->P));
  const b200_hv_params &P = hv->P;
  if (P.detect_clutter)
    return ctx->fail(B200_ERR_INVALID, "hv_verify: the clutter cue (setDetectClutter(true)) is not implemented");
  if (best_cost) *best_cost = 0.0;
  if (accepted_moves) *accepted_moves = 0;
  try {
    hv->info.assign((size_t)H, b200_hv_info{});
    hv->list_sizes.clear();
    hv->h_expl_idx.clear(), hv->h_expl_w.clear(), hv->h_occ_idx.clear();
    hv->ns = 0, hv->n_cells = 0;
    for (int h = 0; h < H; ++h) {
      mask[h] = 0;
      hv->info[h].n_visible = hv->vis_offsets[h + 1] - hv->vis_offsets[h];
    }
    // ---- initialize(): scene normals, NaN compaction, the search structure over what is left
    DevBuf<float4> S, SN;
    int ns = 0;
    B200_TRY(normals_and_compact(ctx, hv->scene_ds.p, hv->n0, (double)P.radius_normals, S, SN, &ns));
    hv->ns = ns;
    std::unique_ptr<b200_cloud> scene_cloud;
    const GridView *sg = nullptr;
    if (ns > 0) {
      B200_TRY(cloud_upload(ctx, reinterpret_cast<const float *>(S.p), ns, 4, true, scene_cloud));
      B200_TRY(cloud_grid_for_radius(scene_cloud.get(), (double)P.inlier_threshold, &sg));
    }
    // ---- addModel per hypothesis
    std::vector<int> indices, bad_information;
    std::vector<float> outliers_weight;
    std::vector<std::unique_ptr<DevBuf<int>>> expl_idx;
    std::vector<std::unique_ptr<DevBuf<float>>> expl_w;
    std::vector<HvExpl> expl;
    DevBuf<unsigned long long> best;
    DevBuf<int> eflags, eslots;
    B200_TRY(best.alloc(ctx, (size_t)std::max(ns, 1)));
    B200_TRY(eflags.alloc(ctx, (size_t)std::max(ns, 1)));
    B200_TRY(eslots.alloc(ctx, (size_t)std::max(ns, 1)));
    for (int h = 0; h < H; ++h) {
      b200_hv_info &I = hv->info[h];
      const int nv = I.n_visible;
      if (nv <= 0) continue;  // "The model cloud has no points.."
      DevBuf<float> V;
      DevBuf<int> cnt;
      B200_TRY(V.alloc(ctx, (size_t)nv * 3));
      B200_TRY(cnt.alloc(ctx, 4));
      B200_TRY(dev_voxel_grid(ctx, hv->visible.p + 3 * (size_t)hv->vis_offsets[h], nv, 3, P.resolution, P.resolution,
                              P.resolution, V.p, cnt.p));
      int nvox = 0;
      B200_TRY(readback_small(ctx, cnt.p, &nvox, sizeof(int)));
      if (nvox <= 0) continue;
      DevBuf<float4> M, MN;
      int nm = 0;
      B200_TRY(normals_and_compact(ctx, V.p, nvox, (double)P.radius_normals, M, MN, &nm));
      I.valid = 1;
      I.n_points = nm;
      int n_out = 0, n_expl = 0;
      std::unique_ptr<DevBuf<int>> li(new DevBuf<int>());
      std::unique_ptr<DevBuf<float>> lw(new DevBuf<float>());
      if (nm > 0 && ns > 0) {
        DevBuf<int> counts;
        DevBuf<unsigned long long> stats;
        DevBuf<long long> offs;
        B200_TRY(counts.alloc(ctx, (size_t)nm));
        B200_TRY(stats.alloc(ctx, 2));
        B200_TRY(offs.alloc(ctx, (size_t)nm + 1));
        B200_TRY(dev_radius_count(ctx, *sg, M.p, nm, (double)P.inlier_threshold, counts.p, stats.p));
        B200_TRY(counts_to_offsets_i64(ctx, counts.p, nm, offs.p));
        B200_CUDA(ctx, cudaMemsetAsync(cnt.p, 0, sizeof(int) * 4, ctx->stream));
        hv_outlier_count_kernel<<<ceil_div(nm, 256), 256, 0, ctx->stream>>>(counts.p, nm, cnt.p);
        B200_LAUNCHED(ctx);
        unsigned long long hstats[2];
        B200_TRY(readback_small(ctx, stats.p, hstats, sizeof(hstats)));
        const long long pairs = (long long)hstats[1];
        if (pairs > 0) {
          DevBuf<int> nidx;
          DevBuf<float> nd2;
          B200_TRY(nidx.alloc(ctx, (size_t)pairs));
          B200_TRY(nd2.alloc(ctx, (size_t)pairs));
          B200_TRY(dev_radius_fill_sized(ctx, *sg, M.p, nm, (double)P.inlier_threshold, (int)hstats[0], offs.p, nidx.p, nd2.p));
          B200_CUDA(ctx, cudaMemsetAsync(best.p, 0, sizeof(unsigned long long) * (size_t)ns, ctx->stream));
          hv_explain_kernel<<<nm, 64, 0, ctx->stream>>>(offs.p, nidx.p, nd2.p, nm, best.p);
          B200_LAUNCHED(ctx);
          hv_explained_flags_kernel<<<ceil_div(ns, 256), 256, 0, ctx->stream>>>(best.p, ns, eflags.p);
          B200_LAUNCHED(ctx);
          B200_TRY(exclusive_scan_i32(ctx, eflags.p, eslots.p, ns, cnt.p + 1));
          int two[2];
          B200_TRY(readback_small(ctx, cnt.p, two, sizeof(two)));
          n_out = two[0], n_expl = two[1];
          B200_TRY(li->alloc(ctx, (size_t)std::max(n_expl, 1)));
          B200_TRY(lw->alloc(ctx, (size_t)std::max(n_expl, 1)));
          hv_explained_emit_kernel<<<ceil_div(ns, 256), 256, 0, ctx->stream>>>(best.p, ns, eflags.p, eslots.p, S.p, SN.p, M.p,
                                                                              MN.p, P.inlier_threshold, li->p, lw->p);
          B200_LAUNCHED(ctx);
        } else {
          n_out = nm;
        }
      } else {
        n_out = nm;  // no scene point can explain anything
      }
      if (!li->p) {
        B200_TRY(li->alloc(ctx, 1));
        B200_TRY(lw->alloc(ctx, 1));
      }
      // outliers_weight_: accumulate(o copies of regularizer_, 0.f) / o; 1 without outliers
      float acc = 0.f;
      for (int i = 0; i < n_out; ++i) acc += P.regularizer;
      float ow = acc / (float)n_out;
      if (n_out == 0) ow = 1.f;
      I.n_outliers = n_out;
      I.outliers_weight = ow;
      I.n_explained = n_expl;
      indices.push_back(h);
      outliers_weight.push_back(ow);
      bad_information.push_back(n_out);
      expl.push_back(HvExpl{li->p, lw->p, n_expl});
      expl_idx.push_back(std::move(li));
      expl_w.push_back(std::move(lw));
    }
    const int Hv = (int)indices.size();
    // ---- occupancy grid of the complete models of the valid hypotheses
    std::vector<HvOcc> occ;
    DevBuf<int> occ_idx, occ_cnt, stamp;
    int n_cells = 0;
    if (Hv > 0) {
      DevBuf<unsigned> box;
      B200_TRY(box.alloc(ctx, 8));
      const unsigned init[8] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u, 0u, 0u};
      B200_TRY(write_small(ctx, box.p, init, sizeof(init)));
      for (int v = 0; v < Hv; ++v) {
        const int lo = hv->offsets[indices[v]], hi = hv->offsets[indices[v] + 1];
        if (hi <= lo) continue;
        hv_bounds_kernel<<<std::min(ceil_div(hi - lo, 256), 64), 256, 0, ctx->stream>>>(hv->models.p, lo, hi, box.p);
        B200_LAUNCHED(ctx);
      }
      unsigned hb[8];
      B200_TRY(readback_small(ctx, box.p, hb, sizeof(hb)));
      float mn[3], mx[3];
      for (int a = 0; a < 3; ++a) {
        // PCL's initial values when no point was seen
        mn[a] = hb[a] == 0xffffffffu ? 3.402823466e38f : hv_dec(hb[a]);
        mx[a] = hb[3 + a] == 0u ? -3.402823466e38f : hv_dec(hb[3 + a]);
      }
      const float res = P.res_occupancy_grid;
      long long size[3];
      for (int a = 0; a < 3; ++a) {
        const float ext = std::ceil(std::abs(mx[a] - mn[a]) / res);
        if (!(ext < 2147483000.f)) return ctx->fail(B200_ERR_CAPACITY, "hv: occupancy grid too large");
        size[a] = (long long)static_cast<int>(ext) + 1;
      }
      if (size[0] * size[1] * size[2] > HV_MAX_CELLS) return ctx->fail(B200_ERR_CAPACITY, "hv: occupancy grid too large");
      n_cells = (int)(size[0] * size[1] * size[2]);
      hv->n_cells = n_cells;
      B200_TRY(stamp.alloc(ctx, (size_t)n_cells));
      B200_TRY(stamp.zero());
      B200_TRY(occ_idx.alloc(ctx, (size_t)std::max(hv->offsets[H], 1)));
      B200_TRY(occ_cnt.alloc(ctx, (size_t)Hv));
      B200_TRY(occ_cnt.zero());
      for (int v = 0; v < Hv; ++v) {
        const int lo = hv->offsets[indices[v]], hi = hv->offsets[indices[v] + 1];
        if (hi <= lo) continue;
        hv_occupancy_kernel<<<ceil_div(hi - lo, 256), 256, 0, ctx->stream>>>(hv->models.p, lo, hi, mn[0], mn[1], mn[2], res,
                                                                            (int)size[0], (int)size[1], v + 1, stamp.p,
                                                                            occ_idx.p + lo, occ_cnt.p + v);
        B200_LAUNCHED(ctx);
      }
      std::vector<int> h_cnt((size_t)Hv);
      B200_TRY(hv_download(ctx, h_cnt.data(), occ_cnt.p, (size_t)Hv));
      for (int v = 0; v < Hv; ++v) {
        occ.push_back(HvOcc{occ_idx.p + hv->offsets[indices[v]], h_cnt[v]});
        hv->info[indices[v]].n_occupancy = h_cnt[v];
      }
    }
    // ---- keep the cue lists for inspection (tests, diagnostics)
    for (int v = 0; v < Hv; ++v) {
      hv->list_sizes.push_back(expl[v].n);
      hv->list_sizes.push_back(occ[v].n);
      const size_t e0 = hv->h_expl_idx.size(), o0 = hv->h_occ_idx.size();
      hv->h_expl_idx.resize(e0 + expl[v].n);
      hv->h_expl_w.resize(e0 + expl[v].n);
      hv->h_occ_idx.resize(o0 + occ[v].n);
      B200_TRY(hv_download(ctx, hv->h_expl_idx.data() + e0, expl[v].idx, (size_t)expl[v].n));
      B200_TRY(hv_download(ctx, hv->h_expl_w.data() + e0, expl[v].w, (size_t)expl[v].n));
      B200_TRY(hv_download(ctx, hv->h_occ_idx.data() + o0, occ[v].idx, (size_t)occ[v].n));
      float s = 0.f;
      for (int k = 0; k < expl[v].n; ++k) s += hv->h_expl_w[e0 + k];
      hv->info[indices[v]].explained_sum = s;
    }
    if (info) memcpy(info, hv->info.data(), sizeof(b200_hv_info) * (size_t)H);
    if (Hv == 0) return B200_OK;
    // ---- SAOptimize
    std::vector<unsigned char> sub((size_t)Hv);
    B200_TRY(run_anneal(ctx, Hv, ns, expl, occ, n_cells, outliers_weight.data(), bad_information.data(), P, sub.data(),
                        best_cost, accepted_moves));
    for (int v = 0; v < Hv; ++v) mask[indices[v]] = sub[v];
  } catch (const std::bad_alloc &) {
    return ctx->fail(B200_ERR_NOMEM, "hv: out of host memory");
  }
  return B200_OK;
}

int b200_hv_last_size(const b200_hv *hv, int which) {
  if (!hv) return -1;
  switch (which) {
    case 0: return hv->ns;
    case 1: return hv->n_cells;
    case 2: return (int)hv->h_expl_idx.size();
    case 3: return (int)hv->h_expl_w.size();
    case 4: return (int)hv->h_occ_idx.size();
    case 5: return (int)hv->list_sizes.size();
  }
  return -1;
}

int b200_hv_last_copy(b200_ctx *ctx, const b200_hv *hv, int which, void *dst) {
  if (!ctx || !hv || !dst) return B200_ERR_INVALID;
  switch (which) {
    case 2: memcpy(dst, hv->h_expl_idx.data(), hv->h_expl_idx.size() * 4); return B200_OK;
    case 3: memcpy(dst, hv->h_expl_w.data(), hv->h_expl_w.size() * 4); return B200_OK;
    case 4: memcpy(dst, hv->h_occ_idx.data(), hv->h_occ_idx.size() * 4); return B200_OK;
    case 5: memcpy(dst, hv->list_sizes.data(), hv->list_sizes.size() * 4); return B200_OK;
  }
  return ctx->fail(B200_ERR_INVALID, "hv_last_copy: no such list");
}

int b200_hv_optimize(b200_ctx *ctx, int H, int ns, const int *expl_off, const int *expl_idx, const float *expl_w,
                     const int *occ_off, const int *occ_idx, int n_cells, const float *outliers_weight,
                     const int *bad_information, const b200_hv_params *p, unsigned char *mask, double *best_cost,
                     int *accepted_moves) {
  if (!ctx) return B200_ERR_INVALID;
  if (H < 0 || ns < 0 || n_cells < 0 || !p || (H > 0 && (!expl_off || !occ_off || !outliers_weight || !bad_information || !mask)))
    return ctx->fail(B200_ERR_INVALID, "hv_optimize: bad arguments");
  if (best_cost) *best_cost = 0.0;
  if (accepted_moves) *accepted_moves = 0;
  if (H == 0) return B200_OK;
  B200_CUDA(ctx, cudaSetDevice(ctx->device));
  B200_TRY(check_hv_params(ctx, *p));
  const int ne = expl_off[H], no = occ_off[H];
  for (int h = 0; h < H; ++h)
    if (expl_off[h + 1] < expl_off[h] || occ_off[h + 1] < occ_off[h] || expl_off[0] != 0 || occ_off[0] != 0)
      return ctx->fail(B200_ERR_INVALID, "hv_optimize: bad offsets");
  if ((ne > 0 && (!expl_idx || !expl_w)) || (no > 0 && !occ_idx)) return ctx->fail(B200_ERR_INVALID, "hv_optimize: null lists");
  for (int k = 0; k < ne; ++k)
    if (expl_idx[k] < 0 || expl_idx[k] >= ns) return ctx->fail(B200_ERR_INVALID, "hv_optimize: scene index out of range");
  for (int k = 0; k < no; ++k)
    if (occ_idx[k] < 0 || occ_idx[k] >= n_cells) return ctx->fail(B200_ERR_INVALID, "hv_optimize: cell index out of range");
  try {
    DevBuf<int> d_ei, d_oi;
    DevBuf<float> d_ew;
    B200_TRY(hv_upload(ctx, d_ei, expl_idx, (size_t)ne));
    B200_TRY(hv_upload(ctx, d_ew, expl_w, (size_t)ne));
    B200_TRY(hv_upload(ctx, d_oi, occ_idx, (size_t)no));
    std::vector<HvExpl> expl((size_t)H);
    std::vector<HvOcc> occ((size_t)H);
    for (int h = 0; h < H; ++h) {
      expl[h] = HvExpl{d_ei.p + expl_off[h], d_ew.p + expl_off[h], expl_off[h + 1] - expl_off[h]};
      occ[h] = HvOcc{d_oi.p + occ_off[h], occ_off[h + 1] - occ_off[h]};
    }
    return run_anneal(ctx, H, ns, expl, occ, n_cells, outliers_weight, bad_information, *p, mask, best_cost, accepted_moves);
  } catch (const std::bad_alloc &) {
    return ctx->fail(B200_ERR_NOMEM, "hv: out of host memory");
  }
}

}  // extern "C"
