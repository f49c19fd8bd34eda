// board.cu — pcl::BOARDLocalReferenceFrameEstimation::compute (SURVEY.md §8(f) rank 1: the frame source of the
// reference's Hough branch — SHOT.cpp:441-453, 6Dpose.cpp:497-509, FPFH_demo.cpp:556-568: setFindHoles(true),
// setRadiusSearch(rf_rad_), keypoints as input, the full cloud as search surface).
//
// pcl 1.8 features/impl/board.hpp computePointLRF, per keypoint:
//   support = radius search; fewer than 6 points → NaN frame
//   z   = direction of least variance of the support (planeFitting), sign by the mean support normal
//   x   : over the support points beyond margin_thresh * tangent_radius (tangent_radius_ stays 0 unless
//         setTangentRadius is called, which the reference never does: the ring is then every neighbour with
//         d2 > 0): the point whose normal deviates most from z; with find_holes the directions of the ring
//         points, measured from a random axis orthogonal to z, are binned into check_margin_array_size sectors
//         and the widest run of empty sectors that is plausible as a border (hole_size_prob_thresh, steep_thresh)
//         gives x instead.
//   y   = z × x
// The random axis comes from rand() in PCL (serial loop, two draws per keypoint with a full support); here the
// stream is glibc's generator carried by the context (b200_ctx_srand; a fresh context is srand(1)), drawn in
// keypoint order exactly like PCL's loop.
//
// One WARP per keypoint for supports of up to 512 points (board_warp_kernel), one CTA per keypoint beyond that
// (board_kernel): radius gather + sort into the (d2, index) order PCL iterates in, float64 sums for the plane fit,
// the sector table and the most different normal as order-independent reductions on packed (value, position) keys
// (BoardScan: PCL's sequential first-minimum / first-maximum scans are lexicographic minima), one thread for the hole
// analysis.  All float32 expressions keep PCL's operation order (--fmad=false).
// Measured (91 076 keypoints on the 1 M-point scene, r = 0.02, 279 support points on average, up to 1 874; host
// buffers in and out): 13.9 ms with one CTA per keypoint and one thread per sector walking the support; 8.0 ms with
// the reductions; 6.5 ms with the warp kernel for the supports it takes; 5.2 ms once the warp kernel's reductions
// break ties by the (d2, index) key themselves (BoardScan2) and its support is no longer sorted.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "linalg3.cuh"
#include "search.cuh"

namespace {

constexpr int BOARD_THREADS = 128;
constexpr int BOARD_MAX_SECTORS = 64;
constexpr float TWO_PI_F = 6.283185307179586f;  // 2 * static_cast<float>(M_PI)

__device__ __forceinline__ float dot3f(const float *a, const float *b) {
  float s = a[0] * b[0];
  s += a[1] * b[1];
  s += a[2] * b[2];
  return s;
}

__device__ __forceinline__ void normalize3f(float *v) {
  const float n = sqrtf(dot3f(v, v));
  v[0] /= n;
  v[1] /= n;
  v[2] /= n;
}

__device__ __forceinline__ void directed_orthogonal_axis(const float *axis, const float *origin, const float *point,
                                                         float *out) {
  const float xo[3] = {point[0] - origin[0], point[1] - origin[1], point[2] - origin[2]};
  const float t = dot3f(axis, xo);
  const float proj[3] = {point[0] - t * axis[0], point[1] - t * axis[1], point[2] - t * axis[2]};
  out[0] = proj[0] - origin[0];
  out[1] = proj[1] - origin[1];
  out[2] = proj[2] - origin[2];
  normalize3f(out);
}

__device__ __forceinline__ void cross3f(const float *a, const float *b, float *o) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}

__device__ __forceinline__ float angle_between_unit(const float *v1, const float *v2, const float *axis) {
  float o[3];
  cross3f(v1, v2, o);
  const float a = acosf(fmaxf(-1.0f, fminf(1.0f, dot3f(v1, v2))));
  return dot3f(o, axis) < 0.f ? (TWO_PI_F - a) : a;
}

__device__ __forceinline__ double block_sum(double v, double *s_red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < BOARD_THREADS / 32; ++w) t += s_red[w];
  return t;
}

struct BoardArgs {
  int second_search;  // tangent_radius != 0 and != search radius: the x axis uses its own support
  float tangent_r2;   // (float)(tangent_radius^2), the acceptance bound of that search
  int find_holes;
  float tangent_radius, margin_thresh;
  int sectors;
  float hole_size_prob_thresh, steep_thresh;
};

// z axis (eigenvector of the smallest eigenvalue of the support's scatter, sign by the mean support normal) and the
// random axis orthogonal to it (find_holes); one thread
__device__ void board_axes(const double *cv, const double *nm, const BoardArgs &a, int i, const int *__restrict__ rand_rank,
                           const int *__restrict__ rand_values, float *z_out, float *x_out) {
    const double A[9] = {cv[0], cv[1], cv[2], cv[1], cv[3], cv[4], cv[2], cv[4], cv[5]};
    double w[3], V[9];
    eigh3_f64(A, w, V);
    float z[3] = {(float)V[0], (float)V[3], (float)V[6]};
    // normalDisambiguation
    if (nm[0] != 0.0 || nm[1] != 0.0 || nm[2] != 0.0) {
      if ((double)z[0] * nm[0] + (double)z[1] * nm[1] + (double)z[2] * nm[2] < 0.0) {
        z[0] = -z[0];
        z[1] = -z[1];
        z[2] = -z[2];
      }
    }
    z_out[0] = z[0], z_out[1] = z[1], z_out[2] = z[2];
    float x[3] = {0.f, 0.f, 0.f};
    if (a.find_holes) {  // randomOrthogonalAxis
      const int r = rand_rank[i];
      const float r0 = ((float)rand_values[2 * r] / 2147483648.0f) * 2.0f - 1.0f;  // (float)RAND_MAX == 2^31
      const float r1 = ((float)rand_values[2 * r + 1] / 2147483648.0f) * 2.0f - 1.0f;
      if (!(fabsf(z[2] - 0.0f) < 1e-8f)) {
        x[0] = r0;
        x[1] = r1;
        x[2] = -(z[0] * x[0] + z[1] * x[1]) / z[2];
      } else if (!(fabsf(z[1] - 0.0f) < 1e-8f)) {
        x[0] = r0;
        x[2] = r1;
        x[1] = -(z[0] * x[0] + z[2] * x[2]) / z[1];
      } else if (!(fabsf(z[0] - 0.0f) < 1e-8f)) {
        x[1] = r0;
        x[2] = r1;
        x[0] = -(z[1] * x[1] + z[2] * x[2]) / z[0];
      }
      normalize3f(x);
    }
    x_out[0] = x[0], x_out[1] = x[1], x_out[2] = x[2];
}

struct BoardSectors {
  const int *check;
  const float *min_angle, *max_angle, *min_angle_normal, *max_angle_normal;
};

// hole analysis over the sector table and the x axis (one thread): the tail of computePointLRF
__device__ void board_finish(const BoardArgs &a, int S, const BoardSectors &sec, float min_normal_cos, int min_t,
                             int margin_found, const float *xr, const float *z, const float *c,
                             const float4 *__restrict__ pts, const int *pos, float *out) {
    float x[3] = {xr[0], xr[1], xr[2]};
    bool ok = true;
    bool use_min_normal = true;
    if (margin_found && a.find_holes) {
      bool hole_present = false;
      for (int k = 0; k < S; ++k)
        if (!sec.check[k]) {
          hole_present = true;
          break;
        }
      if (hole_present) {
        float angle = 0.f;
        int first_no_border = -1;
        if (sec.check[S - 1]) {
          first_no_border = 0;
        } else {
          for (int k = 0; k < S; ++k)
            if (sec.check[k]) {
              first_no_border = k;
              break;
            }
        }
        float max_hole_prob = -FLT_MAX;
        if (first_no_border >= 0)
          for (int ch = first_no_border; ch < S; ++ch) {
            if (sec.check[ch]) continue;
            const int hole_first = ch;
            int hole_end = hole_first + 1;
            while (!sec.check[hole_end % S]) ++hole_end;
            if (hole_end - hole_first > 0) {
              const int previous_hole = (((hole_first - 1) < 0) ? (hole_first - 1) + S : (hole_first - 1)) % S;
              const int following_hole = hole_end % S;
              float normal_begin = sec.max_angle_normal[previous_hole];
              float normal_end = sec.min_angle_normal[following_hole];
              normal_begin -= min_normal_cos;
              normal_end -= min_normal_cos;
              normal_begin = normal_begin / (1.0f - min_normal_cos);
              normal_end = normal_end / (1.0f - min_normal_cos);
              normal_begin = 1.0f - normal_begin;
              normal_end = 1.0f - normal_end;
              float hole_width;
              if (following_hole < previous_hole)
                hole_width = sec.min_angle[following_hole] + TWO_PI_F - sec.max_angle[previous_hole];
              else
                hole_width = sec.min_angle[following_hole] - sec.max_angle[previous_hole];
              const float hole_prob = hole_width / TWO_PI_F;
              const float steep_prob = (normal_end + normal_begin) / 2.0f;
              if (hole_prob > a.hole_size_prob_thresh && steep_prob > a.steep_thresh && hole_prob > max_hole_prob) {
                max_hole_prob = hole_prob;
                const float angle_weight = ((normal_end - normal_begin) + 1.0f) / 2.0f;
                if (following_hole < previous_hole)
                  angle = sec.max_angle[previous_hole] +
                          (sec.min_angle[following_hole] + TWO_PI_F - sec.max_angle[previous_hole]) * angle_weight;
                else
                  angle = sec.max_angle[previous_hole] +
                          (sec.min_angle[following_hole] - sec.max_angle[previous_hole]) * angle_weight;
              }
            }
            if (hole_end >= S) break;
            ch = hole_end - 1;
          }
        if (max_hole_prob > -FLT_MAX) {
          // x = Eigen::AngleAxisf(angle, z) * x
          const float sn = sinf(angle), cs = cosf(angle);
          const float sa[3] = {sn * z[0], sn * z[1], sn * z[2]};
          const float ca[3] = {(1.f - cs) * z[0], (1.f - cs) * z[1], (1.f - cs) * z[2]};
          float R[9];
          float tmp = ca[0] * z[1];
          R[1] = tmp - sa[2];
          R[3] = tmp + sa[2];
          tmp = ca[0] * z[2];
          R[2] = tmp + sa[1];
          R[6] = tmp - sa[1];
          tmp = ca[1] * z[2];
          R[5] = tmp - sa[0];
          R[7] = tmp + sa[0];
          R[0] = ca[0] * z[0] + cs;
          R[4] = ca[1] * z[1] + cs;
          R[8] = ca[2] * z[2] + cs;
          float nx[3];
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            float v = R[r * 3 + 0] * x[0];
            v += R[r * 3 + 1] * x[1];
            v += R[r * 3 + 2] * x[2];
            nx[r] = v;
          }
          x[0] = nx[0], x[1] = nx[1], x[2] = nx[2];
          use_min_normal = false;
        }
      }
    }
    if (use_min_normal) {
      if (min_t < 0) {
        ok = false;  // every support normal is NaN
      } else {
        const float4 p = pts[pos[min_t]];
        const float pv[3] = {p.x, p.y, p.z};
        directed_orthogonal_axis(z, c, pv, x);
      }
    }
    if (ok) {
      float y[3];
      cross3f(z, x, y);
      out[0] = x[0], out[1] = x[1], out[2] = x[2];
      out[3] = y[0], out[4] = y[1], out[5] = y[2];
      out[6] = z[0], out[7] = z[1], out[8] = z[2];
    } else {
      for (int k = 0; k < 9; ++k) out[k] = nanf32();
    }
}

// The sector table and the "most different normal" of computePointLRF are sequential scans in PCL — per sector the
// FIRST support point (in (d2, index) order) with the smallest / largest direction angle, and the first point with the
// smallest normal cosine — i.e. lexicographic minima of (value, position): order-independent reductions.  They are
// evaluated with 64-bit shared-memory atomics on packed keys (value bits : position), all lanes over the support at
// once, instead of one thread per sector walking the whole support (which bounded both kernels: S x n sequential
// steps per keypoint).  Angles are >= +0, so their bit patterns order like the values; cosines go through the usual
// sign flip; NaN cosines never win a comparison in PCL and are skipped here.
struct BoardScan {
  unsigned long long mnkey[BOARD_MAX_SECTORS], mxkey[BOARD_MAX_SECTORS];
  unsigned long long cos_in, cos_out;  // most different normal among the margin points / among the others
  int found;                           // any support point beyond the margin distance
};
__device__ __forceinline__ unsigned board_ord(float f) {  // monotone float -> unsigned
  const unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float board_unord(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
__device__ __forceinline__ void board_scan_init(BoardScan &sc, int idx, int S) {  // idx: the caller's thread / lane index
  if (idx < S) {
    sc.mnkey[idx] = ~0ull;
    sc.mxkey[idx] = 0ull;
  }
  if (idx == 0) {
    sc.cos_in = ~0ull;
    sc.cos_out = ~0ull;
    sc.found = 0;
  }
}
// support point t: d2, direction angle, normal cosine
__device__ __forceinline__ void board_scan_point(BoardScan &sc, int t, float d2, float ang, float nc, float margin_distance2,
                                                 float max_boundary_angle, int S, bool find_holes) {
  const bool in_margin = d2 > margin_distance2;
  if (in_margin) sc.found = 1;  // benign race: every writer stores 1
  if (nc == nc) {
    const unsigned long long k = ((unsigned long long)board_ord(nc) << 32) | (unsigned)t;
    atomicMin(in_margin ? &sc.cos_in : &sc.cos_out, k);
  }
  if (find_holes && in_margin && ang == ang) {  // PCL indexes out of range for a NaN direction (point on the axis)
    const int b = min((int)floorf(ang / max_boundary_angle), S - 1);
    const unsigned long long hi = (unsigned long long)__float_as_uint(ang) << 32;
    atomicMin(&sc.mnkey[b], hi | (unsigned)t);
    atomicMax(&sc.mxkey[b], hi | (0xffffffffu - (unsigned)t));
  }
}
// sector s of the table PCL's loop leaves behind
__device__ __forceinline__ void board_scan_sector(const BoardScan &sc, int s, const float *f_cos, int *check, float *min_angle,
                                                  float *max_angle, float *min_angle_normal, float *max_angle_normal) {
  const unsigned long long a = sc.mnkey[s], b = sc.mxkey[s];
  const bool chk = a != ~0ull;
  check[s] = chk ? 1 : 0;
  min_angle[s] = chk ? __uint_as_float((unsigned)(a >> 32)) : FLT_MAX;
  max_angle[s] = chk ? __uint_as_float((unsigned)(b >> 32)) : -FLT_MAX;
  min_angle_normal[s] = chk ? f_cos[(unsigned)(a & 0xffffffffull)] : -1.0f;
  max_angle_normal[s] = chk ? f_cos[0xffffffffu - (unsigned)(b & 0xffffffffull)] : -1.0f;
}
__device__ __forceinline__ void board_scan_min_cos(const BoardScan &sc, float *min_cos, int *min_t, int *margin_found) {
  const unsigned long long k = sc.found ? sc.cos_in : sc.cos_out;
  *margin_found = sc.found;
  if (k == ~0ull) {
    *min_cos = FLT_MAX;
    *min_t = -1;
  } else {
    *min_cos = board_unord((unsigned)(k >> 32));
    *min_t = (int)(unsigned)(k & 0xffffffffull);
  }
}

__global__ void board_flags_kernel(const int *__restrict__ counts, int K, int *__restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < K) flags[i] = counts[i] >= 6 ? 1 : 0;
}

__global__ void __launch_bounds__(BOARD_THREADS)
    board_kernel(GridView g, const float *__restrict__ normals, const float4 *__restrict__ kp, int K, float radius_f, float r2,
                 int cap, unsigned long long *glob_key, int *glob_pos, float *glob_f, BoardArgs a,
                 const int *__restrict__ rand_rank, const int *__restrict__ rand_values, float *__restrict__ rf_out,
                 const int *__restrict__ counts, int min_count) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_count;
  __shared__ double s_red[BOARD_THREADS / 32];
  __shared__ float s_z[3], s_x[3];
  __shared__ int s_check[BOARD_MAX_SECTORS];
  __shared__ float s_min_angle[BOARD_MAX_SECTORS], s_max_angle[BOARD_MAX_SECTORS], s_min_angle_normal[BOARD_MAX_SECTORS],
      s_max_angle_normal[BOARD_MAX_SECTORS];
  __shared__ float s_min_cos;
  __shared__ int s_min_t, s_margin_found;
  __shared__ BoardScan s_scan;

  unsigned long long *key;
  int *pos;
  float *f_cos, *f_ang;
  if (glob_key) {
    key = glob_key + (size_t)blockIdx.x * cap;
    pos = glob_pos + (size_t)blockIdx.x * cap;
    f_cos = glob_f + (size_t)blockIdx.x * cap * 2;
  } else {
    key = reinterpret_cast<unsigned long long *>(smem_raw);
    pos = reinterpret_cast<int *>(smem_raw + (size_t)cap * 8);
    f_cos = reinterpret_cast<float *>(smem_raw + (size_t)cap * 12);
  }
  f_ang = f_cos + cap;
  const int tid = threadIdx.x;
  const float4 *__restrict__ pts = g.pts;
  const int S = a.sectors;
  const float radius2 = a.tangent_radius * a.tangent_radius;
  const float margin_distance2 = a.margin_thresh * a.margin_thresh * radius2;
  const float max_boundary_angle = TWO_PI_F / (float)S;

  for (int i = blockIdx.x; i < K; i += gridDim.x) {
    if (counts[i] < min_count) continue;  // smaller supports: board_warp_kernel
    const float4 c4 = kp[i];
    const float c[3] = {c4.x, c4.y, c4.z};
    int n = gather_radius(g, c4.x, c4.y, c4.z, radius_f, r2, key, pos, cap, &s_count);
    if (n > cap) n = cap;
    float *out = rf_out + (size_t)i * 9;
    if (n < 6) {
      if (tid < 9) out[tid] = nanf32();
      __syncthreads();
      continue;
    }
    bitonic_sort(key, pos, n);
    // ---- planeFitting: float64 centroid and scatter, eigenvector of the smallest eigenvalue
    double m[3] = {0.0, 0.0, 0.0}, nm[3] = {0.0, 0.0, 0.0};
    for (int t = tid; t < n; t += BOARD_THREADS) {
      const float4 p = pts[pos[t]];
      m[0] += (double)p.x;
      m[1] += (double)p.y;
      m[2] += (double)p.z;
      const float *q = normals + (size_t)key_orig(key[t]) * 4;
      const float q0 = q[0], q1 = q[1], q2 = q[2];
      if (finite3(q0, q1, q2)) {
        nm[0] += (double)q0;
        nm[1] += (double)q1;
        nm[2] += (double)q2;
      }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      m[k] = block_sum(m[k], s_red) / n;
      nm[k] = block_sum(nm[k], s_red);
    }
    double cv[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int t = tid; t < n; t += BOARD_THREADS) {
      const float4 p = pts[pos[t]];
      const double d0 = (double)p.x - m[0], d1 = (double)p.y - m[1], d2 = (double)p.z - m[2];
      cv[0] += d0 * d0;
      cv[1] += d0 * d1;
      cv[2] += d0 * d2;
      cv[3] += d1 * d1;
      cv[4] += d1 * d2;
      cv[5] += d2 * d2;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) cv[k] = block_sum(cv[k], s_red);
    if (tid == 0) board_axes(cv, nm, a, i, rand_rank, rand_values, s_z, s_x);
    __syncthreads();
    const float z[3] = {s_z[0], s_z[1], s_z[2]};
    const float xr[3] = {s_x[0], s_x[1], s_x[2]};
    if (a.second_search) {  // "extract support points for Rx radius"
      n = gather_radius(g, c4.x, c4.y, c4.z, a.tangent_radius, a.tangent_r2, key, pos, cap, &s_count);
      if (n > cap) n = cap;
      bitonic_sort(key, pos, n);
    }
    // ---- per support point: cosine of its normal with z, direction angle from the random axis; sector table and
    // most different normal as order-independent reductions (BoardScan)
    board_scan_init(s_scan, tid, BOARD_MAX_SECTORS);
    __syncthreads();
    for (int t = tid; t < n; t += BOARD_THREADS) {
      const float *q = normals + (size_t)key_orig(key[t]) * 4;
      const float nv[3] = {q[0], q[1], q[2]};
      const float nc = dot3f(z, nv);
      f_cos[t] = nc;
      const float d2t = key_d2(key[t]);
      float ang = 0.f;
      if (a.find_holes && d2t > margin_distance2) {
        const float4 p = pts[pos[t]];
        const float pv[3] = {p.x, p.y, p.z};
        float ind[3];
        directed_orthogonal_axis(z, c, pv, ind);
        ang = angle_between_unit(xr, ind, z);
      }
      board_scan_point(s_scan, t, d2t, ang, nc, margin_distance2, max_boundary_angle, S, a.find_holes != 0);
    }
    __syncthreads();
    if (a.find_holes && tid < S)
      board_scan_sector(s_scan, tid, f_cos, s_check, s_min_angle, s_max_angle, s_min_angle_normal, s_max_angle_normal);
    if (tid == BOARD_MAX_SECTORS) board_scan_min_cos(s_scan, &s_min_cos, &s_min_t, &s_margin_found);
    __syncthreads();
    if (tid == 0) {
      const BoardSectors sec = {s_check, s_min_angle, s_max_angle, s_min_angle_normal, s_max_angle_normal};
      board_finish(a, S, sec, s_min_cos, s_min_t, s_margin_found, xr, z, c, pts, pos, out);
    }
    __syncthreads();
  }
}

// ---- one keypoint per WARP (supports of up to BW_CAP points, one search radius; the rest stays with board_kernel) ----
// Same steps as board_kernel with the warp in the CTA's place: ballot-compacted gather into the warp's slice of shared
// memory (left in gather order: no sort), float64 sums by lane partials + shuffles, the sector table and the most
// different normal by two-stage reductions (BoardScan2), the hole analysis by lane 0.  The CTA kernel
// keeps 128 threads on a keypoint through ~50 block-wide barriers and three single-thread phases; here the SM's other
// warps work on their own keypoints meanwhile.  The float64 sums are grouped differently (32 partials instead of
// 128), so they can differ from the CTA kernel's in the last bit; everything after the float32 cast of the z axis is
// the same float32 sequence.
constexpr int BW_CAP = 512;
constexpr int BW_WARPS = 4;
// Two-stage form of BoardScan for an UNSORTED support: the extreme value first (32-bit atomics), then — among the
// points that reach it — the smallest (d2, index) key, which is the point PCL's scan over the sorted support meets
// first.  The warp kernel therefore needs no sort at all (it was 45 of its stages for a 512-point support).
struct BoardScan2 {
  unsigned mnv[BOARD_MAX_SECTORS], mxv[BOARD_MAX_SECTORS];            // angle bits: smallest / largest per sector
  unsigned long long mnk[BOARD_MAX_SECTORS], mxk[BOARD_MAX_SECTORS];  // first point (key) reaching them
  unsigned cosv[2];                                                   // ordered cosine: margin points / the others
  unsigned long long cosk[2];
  int found;
};
struct BwSmem {
  unsigned long long key[BW_CAP];
  int pos[BW_CAP];
  float f_cos[BW_CAP], f_ang[BW_CAP];
  BoardScan2 scan;
  int check[BOARD_MAX_SECTORS];
  float min_angle[BOARD_MAX_SECTORS], max_angle[BOARD_MAX_SECTORS], min_angle_normal[BOARD_MAX_SECTORS],
      max_angle_normal[BOARD_MAX_SECTORS];
  float z[3], x[3];
  float min_cos;
  int min_t, margin_found;
};

__global__ void __launch_bounds__(BW_WARPS * 32)
    board_warp_kernel(GridView g, const float *__restrict__ normals, const float4 *__restrict__ kp, int K, float radius_f,
                      float r2, BoardArgs a, const int *__restrict__ counts, const int *__restrict__ rand_rank,
                      const int *__restrict__ rand_values, float *__restrict__ rf_out) {
  extern __shared__ __align__(16) unsigned char bw_raw[];
  BwSmem &sm = reinterpret_cast<BwSmem *>(bw_raw)[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * BW_WARPS;
  const float4 *__restrict__ pts = g.pts;
  const int *__restrict__ cs = g.cell_start;
  const int S = a.sectors;
  const float radius2 = a.tangent_radius * a.tangent_radius;
  const float margin_distance2 = a.margin_thresh * a.margin_thresh * radius2;
  const float max_boundary_angle = TWO_PI_F / (float)S;
  for (int i = blockIdx.x * BW_WARPS + (threadIdx.x >> 5); i < K; i += nwarps) {
    const int cnt = counts[i];
    if (cnt > BW_CAP) continue;  // board_kernel's
    float *out = rf_out + (size_t)i * 9;
    if (cnt < 6) {
      if (lane < 9) out[lane] = nanf32();
      continue;
    }
    const float4 c4 = kp[i];
    const float c[3] = {c4.x, c4.y, c4.z};
    // ---- gather (cnt neighbours: the count pass ran the same test on the same points)
    int n = 0;
    {
      int x0, x1, y0, y1, z0, z1;
      if (ball_cell_range(g, c4.x, c4.y, c4.z, radius_f, x0, x1, y0, y1, z0, z1)) {
        for (int zc = z0; zc <= z1; ++zc)
          for (int yc = y0; yc <= y1; ++yc) {
            const int base = g.dx * (yc + g.dy * zc);
            const int s0 = cs[base + x0], e = cs[base + x1 + 1];
            for (int j0 = s0; j0 < e; j0 += 128) {
              float4 p[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int j = j0 + 32 * u + lane;
                p[u] = (j < e) ? pts[j] : make_float4(0.f, 0.f, 0.f, 0.f);
              }
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int j = j0 + 32 * u + lane;
                const float d2 = sqdist3(c4.x, c4.y, c4.z, p[u].x, p[u].y, p[u].z);
                const bool hit = j < e && d2 < r2;
                const unsigned m = __ballot_sync(0xffffffffu, hit);
                if (hit) {
                  const int slot = n + __popc(m & ((1u << lane) - 1u));
                  if (slot < BW_CAP) {
                    sm.key[slot] = nbr_key(d2, orig_index(p[u]));
                    sm.pos[slot] = j;
                  }
                }
                n += __popc(m);
              }
            }
          }
      }
    }
    if (n > BW_CAP) n = BW_CAP;  // cannot happen
    __syncwarp();  // the support stays in gather order: nothing below depends on the order (BoardScan2)
    // ---- planeFitting: float64 centroid and scatter
    double m[3] = {0.0, 0.0, 0.0}, nm[3] = {0.0, 0.0, 0.0};
    for (int t = lane; t < n; t += 32) {
      const float4 p = pts[sm.pos[t]];
      m[0] += (double)p.x;
      m[1] += (double)p.y;
      m[2] += (double)p.z;
      const float *q = normals + (size_t)key_orig(sm.key[t]) * 4;
      const float q0 = q[0], q1 = q[1], q2 = q[2];
      if (finite3(q0, q1, q2)) {
        nm[0] += (double)q0;
        nm[1] += (double)q1;
        nm[2] += (double)q2;
      }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      m[k] = warp_sum(m[k]) / n;
      nm[k] = warp_sum(nm[k]);
    }
    double cv[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int t = lane; t < n; t += 32) {
      const float4 p = pts[sm.pos[t]];
      const double d0 = (double)p.x - m[0], d1 = (double)p.y - m[1], d2 = (double)p.z - m[2];
      cv[0] += d0 * d0;
      cv[1] += d0 * d1;
      cv[2] += d0 * d2;
      cv[3] += d1 * d1;
      cv[4] += d1 * d2;
      cv[5] += d2 * d2;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) cv[k] = warp_sum(cv[k]);
    if (lane == 0) board_axes(cv, nm, a, i, rand_rank, rand_values, sm.z, sm.x);
    __syncwarp();
    const float z[3] = {sm.z[0], sm.z[1], sm.z[2]};
    const float xr[3] = {sm.x[0], sm.x[1], sm.x[2]};
    // ---- per support point: cosine of its normal with z, direction angle from the random axis; sector table and
    // most different normal as order-independent reductions (BoardScan)
    for (int sct = lane; sct < BOARD_MAX_SECTORS; sct += 32) {
      sm.scan.mnv[sct] = 0xffffffffu;
      sm.scan.mxv[sct] = 0u;
      sm.scan.mnk[sct] = ~0ull;
      sm.scan.mxk[sct] = ~0ull;
      sm.min_angle_normal[sct] = -1.0f;
      sm.max_angle_normal[sct] = -1.0f;
    }
    if (lane < 2) {
      sm.scan.cosv[lane] = 0xffffffffu;
      sm.scan.cosk[lane] = ~0ull;
    }
    if (lane == 0) {
      sm.scan.found = 0;
      sm.min_t = -1;
    }
    __syncwarp();
    // stage 1: values
    for (int t = lane; t < n; t += 32) {
      const float *q = normals + (size_t)key_orig(sm.key[t]) * 4;
      const float nv[3] = {q[0], q[1], q[2]};
      const float nc = dot3f(z, nv);
      sm.f_cos[t] = nc;
      const bool in_margin = key_d2(sm.key[t]) > margin_distance2;
      float ang = 0.f;
      if (a.find_holes && in_margin) {
        const float4 p = pts[sm.pos[t]];
        const float pv[3] = {p.x, p.y, p.z};
        float ind[3];
        directed_orthogonal_axis(z, c, pv, ind);
        ang = angle_between_unit(xr, ind, z);
      }
      sm.f_ang[t] = ang;
      if (in_margin) sm.scan.found = 1;
      if (nc == nc) atomicMin(&sm.scan.cosv[in_margin ? 0 : 1], board_ord(nc));
      if (a.find_holes && in_margin && ang == ang) {  // PCL indexes out of range for a NaN direction
        const int b = min((int)floorf(ang / max_boundary_angle), S - 1);
        atomicMin(&sm.scan.mnv[b], __float_as_uint(ang));
        atomicMax(&sm.scan.mxv[b], __float_as_uint(ang));
      }
    }
    __syncwarp();
    // stage 2: among the points reaching an extreme, the smallest (d2, index) key
    for (int t = lane; t < n; t += 32) {
      const float nc = sm.f_cos[t], ang = sm.f_ang[t];
      const unsigned long long kt = sm.key[t];
      const bool in_margin = key_d2(kt) > margin_distance2;
      if (nc == nc && board_ord(nc) == sm.scan.cosv[in_margin ? 0 : 1]) atomicMin(&sm.scan.cosk[in_margin ? 0 : 1], kt);
      if (a.find_holes && in_margin && ang == ang) {
        const int b = min((int)floorf(ang / max_boundary_angle), S - 1);
        if (__float_as_uint(ang) == sm.scan.mnv[b]) atomicMin(&sm.scan.mnk[b], kt);
        if (__float_as_uint(ang) == sm.scan.mxv[b]) atomicMin(&sm.scan.mxk[b], kt);
      }
    }
    __syncwarp();
    // stage 3: the winners leave what the sequential scans would have kept
    const int cos_set = sm.scan.found ? 0 : 1;
    for (int t = lane; t < n; t += 32) {
      const float nc = sm.f_cos[t], ang = sm.f_ang[t];
      const unsigned long long kt = sm.key[t];
      const bool in_margin = key_d2(kt) > margin_distance2;
      if ((in_margin ? 0 : 1) == cos_set && kt == sm.scan.cosk[cos_set]) sm.min_t = t;
      if (a.find_holes && in_margin && ang == ang) {
        const int b = min((int)floorf(ang / max_boundary_angle), S - 1);
        if (kt == sm.scan.mnk[b]) sm.min_angle_normal[b] = nc;
        if (kt == sm.scan.mxk[b]) sm.max_angle_normal[b] = nc;
      }
    }
    if (a.find_holes)
      for (int sct = lane; sct < S; sct += 32) {
        const bool chk = sm.scan.mnv[sct] != 0xffffffffu;
        sm.check[sct] = chk ? 1 : 0;
        sm.min_angle[sct] = chk ? __uint_as_float(sm.scan.mnv[sct]) : FLT_MAX;
        sm.max_angle[sct] = chk ? __uint_as_float(sm.scan.mxv[sct]) : -FLT_MAX;
      }
    if (lane == 31) {
      sm.margin_found = sm.scan.found;
      const unsigned cv = sm.scan.cosv[cos_set];
      sm.min_cos = (sm.scan.cosk[cos_set] == ~0ull) ? FLT_MAX : board_unord(cv);
    }
    __syncwarp();
    if (lane == 0) {
      const BoardSectors sec = {sm.check, sm.min_angle, sm.max_angle, sm.min_angle_normal, sm.max_angle_normal};
      board_finish(a, S, sec, sm.min_cos, sm.min_t, sm.margin_found, xr, z, c, pts, sm.pos, out);
    }
    __syncwarp();
  }
}

// glibc rand(): TYPE_3 additive feedback generator (r[i] = r[i-3] + r[i-31], Lehmer-seeded, 310 values discarded)
void glibc_seed(unsigned seed, uint32_t st[31]) {
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

// the next `count` rand() values of the stream st (st[0] oldest), which is advanced past them
void glibc_fill(uint32_t st[31], int *out, int count) {
  uint32_t r[31];
  memcpy(r, st, sizeof(r));
  int h = 0;  // st[k] == r[(h + k) % 31]
  for (int i = 0; i < count; ++i) {
    const uint32_t o = r[h] + r[(h + 28) % 31];
    r[h] = o;
    h = (h + 1) % 31;
    out[i] = (int)(o >> 1);
  }
  for (int k = 0; k < 31; ++k) st[k] = r[(h + k) % 31];
}

}  // namespace

void board_rand_seed(b200_ctx *ctx, unsigned seed) {
  glibc_seed(seed, ctx->rand_state);
  ctx->rand_seeded = true;
}

// d_normals: one row of 4 floats per surface point, original order.  d_rf: K x 9.  The random axes draw from
// rand_state, which is advanced by exactly two values per keypoint with a full support.  Host waits: one
// readback_small (the support maxima, which size the CTA kernel's shared memory, and the number of full supports).
int dev_board_lrf_from(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_kp, int K, double radius,
                       const b200_board_params *p, uint32_t rand_state[31], float *d_rf) {
  if (!(radius > 0.0)) return ctx->fail(B200_ERR_INVALID, "board_lrf: radius must be > 0");
  if (p->check_margin_array_size < 1 || p->check_margin_array_size > BOARD_MAX_SECTORS)
    return ctx->fail(B200_ERR_INVALID, "board_lrf: check_margin_array_size must be in 1..64");
  const bool second = p->tangent_radius != 0.0f && (double)p->tangent_radius != radius;
  if (K <= 0) return B200_OK;
  StageScope st_(ctx, ST_BOARD);
  const GridView *g;
  B200_TRY(cloud_grid_for_radius(c, radius, &g));
  DevBuf<int> counts, counts2, flags, rank, rnd;
  DevBuf<unsigned long long> info;  // [0] support max, [2] x-axis support max (second search), [4] full supports
  B200_TRY(counts.alloc(ctx, (size_t)K));
  B200_TRY(flags.alloc(ctx, (size_t)K));
  B200_TRY(rank.alloc(ctx, (size_t)K));
  B200_TRY(info.alloc(ctx, 5));
  B200_TRY(info.zero());
  B200_TRY(dev_radius_count(ctx, *g, d_kp, K, radius, counts.p, info.p));
  if (second) {  // the x-axis support may be larger than the plane-fit support
    B200_TRY(counts2.alloc(ctx, (size_t)K));
    B200_TRY(dev_radius_count(ctx, *g, d_kp, K, (double)p->tangent_radius, counts2.p, info.p + 2));
  }
  board_flags_kernel<<<ceil_div(K, 256), 256, 0, ctx->stream>>>(counts.p, K, flags.p);
  B200_LAUNCHED(ctx);
  B200_TRY(exclusive_scan_i32(ctx, flags.p, rank.p, K, reinterpret_cast<int *>(info.p + 4)));
  unsigned long long hinfo[5];
  B200_TRY(readback_small(ctx, info.p, hinfo, sizeof(hinfo)));
  const int max_count = second ? (int)std::max(hinfo[0], hinfo[2]) : (int)hinfo[0];
  const int n_full = (int)(unsigned)hinfo[4];
  // two rand() values per keypoint with a full support, in keypoint order (PCL's serial loop), staged in the
  // context's pinned buffer.  Refilling it here is safe: the readback_small above drained the stream, so the copy
  // an earlier call enqueued from it has completed.
  B200_TRY(rnd.alloc(ctx, (size_t)std::max(2 * n_full, 1)));
  if (p->find_holes && n_full > 0) {
    const size_t need = (size_t)2 * n_full;
    if (ctx->board_draws_cap < need) {
      if (ctx->board_draws) cudaFreeHost(ctx->board_draws);
      ctx->board_draws = nullptr;
      ctx->board_draws_cap = 0;
      B200_CUDA(ctx, cudaHostAlloc((void **)&ctx->board_draws, need * sizeof(int), cudaHostAllocDefault));
      ctx->board_draws_cap = need;
    }
    glibc_fill(rand_state, ctx->board_draws, (int)need);
    B200_CUDA(ctx, cudaMemcpyAsync(rnd.p, ctx->board_draws, need * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  }
  BoardArgs a;
  a.second_search = second ? 1 : 0;
  a.tangent_r2 = (float)((double)p->tangent_radius * (double)p->tangent_radius);
  a.find_holes = p->find_holes ? 1 : 0;
  a.tangent_radius = p->tangent_radius;
  a.margin_thresh = p->margin_thresh;
  a.sectors = p->check_margin_array_size;
  a.hole_size_prob_thresh = p->hole_size_prob_thresh;
  a.steep_thresh = p->steep_thresh;
  const float r2 = (float)(radius * radius);
  // supports of up to BW_CAP points: one keypoint per warp (B200_BOARD=cta: everything by the CTA kernel); the
  // two-radius form (setTangentRadius, never used by the reference) stays with the CTA kernel
  const char *sel = getenv("B200_BOARD");
  const bool warp_path = !second && !(sel && !strcmp(sel, "cta"));
  if (warp_path) {
    const size_t smem_w = sizeof(BwSmem) * BW_WARPS;
    B200_CUDA(ctx, ensure_dyn_smem(board_warp_kernel, smem_w));
    board_warp_kernel<<<std::min(ceil_div(K, BW_WARPS), ctx->sm_count * 16), BW_WARPS * 32, smem_w, ctx->stream>>>(
        *g, d_normals, d_kp, K, (float)radius, r2, a, counts.p, rank.p, rnd.p, d_rf);
    B200_LAUNCHED(ctx);
  }
  const int min_count = warp_path ? BW_CAP + 1 : 0;
  const int cap = next_pow2_host(std::max(max_count, 32));
  const size_t smem = (size_t)cap * 20;
  if (max_count < min_count) {
    // every keypoint was the warp kernel's
  } else if (smem <= 160 * 1024) {
    B200_CUDA(ctx, ensure_dyn_smem(board_kernel, smem));
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 4096)));
    const int grid = std::min(K, ctx->sm_count * per_sm);
    board_kernel<<<grid, BOARD_THREADS, smem, ctx->stream>>>(*g, d_normals, d_kp, K, (float)radius, r2, cap, nullptr, nullptr,
                                                            nullptr, a, rank.p, rnd.p, d_rf, counts.p, min_count);
    B200_LAUNCHED(ctx);
  } else {
    const int grid = std::min(K, ctx->sm_count * 2);
    DevBuf<unsigned long long> gk;
    DevBuf<int> gp;
    DevBuf<float> gf;
    B200_TRY(gk.alloc(ctx, (size_t)grid * cap));
    B200_TRY(gp.alloc(ctx, (size_t)grid * cap));
    B200_TRY(gf.alloc(ctx, (size_t)grid * cap * 2));
    board_kernel<<<grid, BOARD_THREADS, 0, ctx->stream>>>(*g, d_normals, d_kp, K, (float)radius, r2, cap, gk.p, gp.p, gf.p, a,
                                                         rank.p, rnd.p, d_rf, counts.p, min_count);
    B200_LAUNCHED(ctx);
  }
  return B200_OK;
}

// b200_board_lrf: draws from the context's stream (srand(1) unless reseeded), which then continues after them
int dev_board_lrf(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_kp, int K, double radius,
                  const b200_board_params *p, float *d_rf) {
  if (p->find_holes && !ctx->rand_seeded) board_rand_seed(ctx, 1u);
  return dev_board_lrf_from(ctx, c, d_normals, d_kp, K, radius, p, ctx->rand_state, d_rf);
}
