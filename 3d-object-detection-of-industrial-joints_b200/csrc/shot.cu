// shot.cu — SHOT local reference frame + SHOT352 descriptor, fused.
//
// Two kernels share the arithmetic:
//   shot_warp_kernel  one keypoint per WARP (neighbourhoods up to 1024 points — every keypoint of the
//                     reference's parameter sets): the warp gathers its neighbour list into shared
//                     memory, accumulates the float64 covariance with shuffles, one lane solves the
//                     3x3 eigen-problem while the SM's other warps keep working, and the 352-bin
//                     histogram is a per-warp shared-memory array.  No sort: the distance order is
//                     only needed by PCL's tie rule, which selects five rows by rank on demand.
//                     Per-neighbour interpolation runs in float32 with explicit error bands around
//                     every discrete decision; a neighbour inside a band is re-evaluated with PCL's
//                     float64 expressions (shot_neighbor_exact), so the bins chosen are identical.
//   shot_kernel       one keypoint per CTA, sorted list in shared or global memory: neighbourhoods
//                     larger than that (SHOT_demo.cpp:498's radius 50 puts the whole model in one).
//
// Replaces pcl::SHOTEstimationOMP<PointXYZRGBA, Normal, SHOT352>::compute (SHOT.cpp:360-371,
// SHOT_demo.cpp:419-424 and 497-502, 6Dpose.cpp:450-461, CAD_desc.cpp:341-352), including the
// SHOTLocalReferenceFrameEstimationOMP pass that its initCompute runs first.  PCL searches the
// neighbourhood twice (once per pass, same radius); here the gathered list is reused.
//
// Per keypoint: radius gather (warp-aggregated append into shared memory) → sort by (d2, index) →
// weighted covariance in float64 (block reduction) → 3x3 eigen-solve → sign disambiguation by
// majority vote, with PCL's median rule on ties → per neighbour: 32-sector / 11-bin quadrilinear
// interpolation evaluated in float64 exactly as PCL does, accumulated into a 352-bin float32
// histogram in shared memory with atomics → L2 normalisation → one coalesced 1444-byte store.
// Discrete choices (sector, bin, sign votes) use the same float64 expressions as PCL; only the
// float32 accumulation order differs (atomics), which is far inside the 1e-4 L2 parity bound.
//
// Algorithmic HBM traffic per descriptor: 1444 B written + the neighbourhood's points and normals
// (32 B each) read once: 1444 + 32 * N/K bytes amortised (SURVEY.md §8(d)).
#include <algorithm>

#include "linalg3.cuh"
#include "search.cuh"

namespace {

constexpr int SHOT_THREADS = 128;
constexpr int SHOT_LEN = 352;

__global__ void gather_normals_kernel(const float4 *__restrict__ sorted_pts, int n, const float4 *__restrict__ normals,
                                      float4 *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = normals[orig_index(sorted_pts[i])];
}

// One neighbour of computePointSHOT (createBinDistanceShape + interpolateSingleChannel), evaluated
// with PCL's float64 expressions.  hist: 352 floats in shared memory; fr: frame rows x, y, z.
// Histogram accumulators.  FloatBins: float32 atomics (CTA kernel, several warps share the bins).
// FixedBins: fixed point in 32 bits — shared-memory integer adds are native while float (and 64-bit)
// adds are compare-and-swap loops.  Every contribution is >= 0 and <= 4, so with n neighbours a bin sum
// is at most 4 n: the scale is 2^20 for n <= 1024 and 2^19 up to SW_CAP = 2016 (the unsigned sum cannot
// wrap).  The quantisation (<= 4.8e-7 per contribution of order 1, same size as float32 rounding of the
// bin sums) is ~1e-7 of the histogram norm, far inside the 1e-4 parity bound.
struct FloatBins {
  float *h;
  __device__ __forceinline__ void add(int bin, float v) const { atomicAdd(&h[bin], v); }
};
struct FixedBins {
  int *h;
  float scale;
  __device__ __forceinline__ void add(int bin, float v) const { atomicAdd(&h[bin], __float2int_rn(v * scale)); }
};

template <class Bins>
__device__ __noinline__ void shot_neighbor_exact(Bins s_hist, const float4 nv, const float4 p, const float4 c,
                                                 const float d2, const float *fr, const double radius) {
  const float fxx = fr[0], fxy = fr[1], fxz = fr[2];
  const float fyx = fr[3], fyy = fr[4], fyz = fr[5];
  const float fzx = fr[6], fzy = fr[7], fzz = fr[8];
  const double radius3_4 = (radius * 3) / 4, radius1_4 = radius / 4, radius1_2 = radius / 2;
  const double RAD_45 = 0.78539816339744830961566084581988;
  const double RAD_90 = 1.5707963267948966192313216916398;
  const double RAD_135 = 2.3561944901923449288469825374596;
  const double RAD_PI_7_8 = 2.7488935718910690836548129603691;
  {
        // createBinDistanceShape
        float dotf = nv.x * fzx;
        dotf += nv.y * fzy;
        dotf += nv.z * fzz;
        double cosineDesc = (double)dotf;
        if (cosineDesc > 1.0) cosineDesc = 1.0;
        if (cosineDesc < -1.0) cosineDesc = -1.0;
        double binDistance = ((1.0 + cosineDesc) * 10) / 2;
        // interpolateSingleChannel
        const float dx = p.x - c.x, dy = p.y - c.y, dz = p.z - c.z;
        const double distance = sqrt((double)d2);
        if (fabs(distance) < 1E-15) return;
        float t;
        t = dx * fxx;
        t += dy * fxy;
        t += dz * fxz;
        double xInFeatRef = (double)t;
        t = dx * fyx;
        t += dy * fyy;
        t += dz * fyz;
        double yInFeatRef = (double)t;
        t = dx * fzx;
        t += dy * fzy;
        t += dz * fzz;
        double zInFeatRef = (double)t;
        if (fabs(yInFeatRef) < 1E-30) yInFeatRef = 0;
        if (fabs(xInFeatRef) < 1E-30) xInFeatRef = 0;
        if (fabs(zInFeatRef) < 1E-30) zInFeatRef = 0;

        const int bit4 = ((yInFeatRef > 0) || ((yInFeatRef == 0.0) && (xInFeatRef < 0))) ? 1 : 0;
        const int bit3 = (((xInFeatRef > 0) || ((xInFeatRef == 0.0) && (yInFeatRef > 0))) ? !bit4 : bit4) ? 1 : 0;
        int desc_index = (bit4 << 3) + (bit3 << 2);
        desc_index = desc_index << 1;
        if ((xInFeatRef * yInFeatRef > 0) || (xInFeatRef == 0.0))
          desc_index += (fabs(xInFeatRef) >= fabs(yInFeatRef)) ? 0 : 4;
        else
          desc_index += (fabs(xInFeatRef) > fabs(yInFeatRef)) ? 4 : 0;
        desc_index += zInFeatRef > 0 ? 1 : 0;
        desc_index += (distance > radius1_2) ? 2 : 0;

        const int step_index = (int)floor(binDistance + 0.5);
        const int volume_index = desc_index * 11;
        binDistance -= step_index;
        double intWeight = (1 - fabs(binDistance));
        if (binDistance > 0)
          s_hist.add(volume_index + ((step_index + 1) % 10), (float)binDistance);
        else
          s_hist.add(volume_index + ((step_index - 1 + 10) % 10), -(float)binDistance);

        if (distance > radius1_2) {
          const double radiusDistance = (distance - radius3_4) / radius1_2;
          if (distance > radius3_4)
            intWeight += 1 - radiusDistance;
          else {
            intWeight += 1 + radiusDistance;
            s_hist.add((desc_index - 2) * 11 + step_index, -(float)radiusDistance);
          }
        } else {
          const double radiusDistance = (distance - radius1_4) / radius1_2;
          if (distance < radius1_4)
            intWeight += 1 + radiusDistance;
          else {
            intWeight += 1 - radiusDistance;
            s_hist.add((desc_index + 2) * 11 + step_index, (float)radiusDistance);
          }
        }

        double inclinationCos = zInFeatRef / distance;
        if (inclinationCos < -1.0) inclinationCos = -1.0;
        if (inclinationCos > 1.0) inclinationCos = 1.0;
        const double inclination = acos(inclinationCos);
        if (inclination > RAD_90 || (fabs(inclination - RAD_90) < 1e-30 && zInFeatRef <= 0)) {
          const double inclinationDistance = (inclination - RAD_135) / RAD_90;
          if (inclination > RAD_135)
            intWeight += 1 - inclinationDistance;
          else {
            intWeight += 1 + inclinationDistance;
            s_hist.add((desc_index + 1) * 11 + step_index, -(float)inclinationDistance);
          }
        } else {
          const double inclinationDistance = (inclination - RAD_45) / RAD_90;
          if (inclination < RAD_45)
            intWeight += 1 + inclinationDistance;
          else {
            intWeight += 1 - inclinationDistance;
            s_hist.add((desc_index - 1) * 11 + step_index, (float)inclinationDistance);
          }
        }

        if (yInFeatRef != 0.0 || xInFeatRef != 0.0) {
          const double azimuth = atan2(yInFeatRef, xInFeatRef);
          const int sel = desc_index >> 2;
          double azimuthDistance = (azimuth - (-RAD_PI_7_8 + RAD_45 * sel)) / RAD_45;
          azimuthDistance = fmax(-0.5, fmin(azimuthDistance, 0.5));
          if (azimuthDistance > 0) {
            intWeight += 1 - azimuthDistance;
            const int interp_index = (desc_index + 4) % 32;
            s_hist.add(interp_index * 11 + step_index, (float)azimuthDistance);
          } else {
            const int interp_index = (desc_index - 4 + 32) % 32;
            intWeight += 1 + azimuthDistance;
            s_hist.add(interp_index * 11 + step_index, -(float)azimuthDistance);
          }
        }
        s_hist.add(volume_index + step_index, (float)intWeight);
  }
}

__global__ void __launch_bounds__(SHOT_THREADS)
    shot_kernel(GridView g, const float4 *__restrict__ nrm, const float4 *__restrict__ kp, int K, float radius_f,
                double radius, float r2, int cap, unsigned long long *glob_key, int *glob_pos,
                float *__restrict__ desc, float *__restrict__ rf_out, int lrf_only,
                const int *__restrict__ counts, int min_count) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ int s_count;
  __shared__ int s_votes[3];       // skipped, plusX, plusZ
  __shared__ double s_red[7][4];   // block reduction scratch
  __shared__ double s_axes[6];     // v1 (x axis), v3 (z axis) before disambiguation
  __shared__ float s_frame[9];     // x, y, z axes (float)
  __shared__ int s_ok;
  __shared__ float s_hist[SHOT_LEN];
  __shared__ double s_norm[4];

  unsigned long long *key;
  int *pos;
  cta_list(smem_raw, glob_key, glob_pos, cap, key, pos);
  const int tid = threadIdx.x;
  const float4 *__restrict__ pts = g.pts;

  for (int i = blockIdx.x; i < K; i += gridDim.x) {
    if (counts[i] < min_count) continue;  // handled by shot_warp_kernel
    const float4 c = kp[i];
    int n = gather_radius(g, c.x, c.y, c.z, radius_f, r2, key, pos, cap, &s_count);
    if (n > cap) n = cap;
    bitonic_sort(key, pos, n);
    if (tid < 3) s_votes[tid] = 0;
    for (int b = tid; b < SHOT_LEN; b += SHOT_THREADS) s_hist[b] = 0.0f;
    __syncthreads();

    // ---- local reference frame: weighted covariance (shot_lrf.hpp getLocalRF) ----
    double part[7] = {0, 0, 0, 0, 0, 0, 0};
    int skipped = 0;
    for (int j = tid; j < n; j += SHOT_THREADS) {
      const float4 p = pts[pos[j]];
      if (p.x == c.x && p.y == c.y && p.z == c.z) {
        ++skipped;
        continue;
      }
      const double vx = (double)(p.x - c.x), vy = (double)(p.y - c.y), vz = (double)(p.z - c.z);
      const double w = radius - sqrt((double)key_d2(key[j]));
      part[0] += w * (vx * vx);
      part[1] += w * (vx * vy);
      part[2] += w * (vx * vz);
      part[3] += w * (vy * vy);
      part[4] += w * (vy * vz);
      part[5] += w * (vz * vz);
      part[6] += w;
    }
#pragma unroll
    for (int a = 0; a < 7; ++a) part[a] = warp_sum(part[a]);
    skipped = warp_sum(skipped);
    if ((tid & 31) == 0) {
#pragma unroll
      for (int a = 0; a < 7; ++a) s_red[a][tid >> 5] = part[a];
      if (skipped) atomicAdd(&s_votes[0], skipped);
    }
    __syncthreads();
    const int n_skip = s_votes[0];
    const int valid = n - n_skip;
    if (tid == 0) {
      int ok = (valid >= 5) ? 1 : 0;
      if (ok) {
        double s[7];
#pragma unroll
        for (int a = 0; a < 7; ++a) s[a] = ((s_red[a][0] + s_red[a][1]) + s_red[a][2]) + s_red[a][3];
        double cov[9] = {s[0] / s[6], s[1] / s[6], s[2] / s[6], s[1] / s[6], s[3] / s[6],
                         s[4] / s[6], s[2] / s[6], s[4] / s[6], s[5] / s[6]};
        double w[3], V[9];
        eigh3_f64(cov, w, V);
        if (!isfinite(w[0]) || !isfinite(w[1]) || !isfinite(w[2])) ok = 0;
        s_axes[0] = V[0 * 3 + 2];
        s_axes[1] = V[1 * 3 + 2];
        s_axes[2] = V[2 * 3 + 2];
        s_axes[3] = V[0 * 3 + 0];
        s_axes[4] = V[1 * 3 + 0];
        s_axes[5] = V[2 * 3 + 0];
      }
      s_ok = ok;
    }
    __syncthreads();
    int ok = s_ok;
    if (ok) {
      // sign votes
      const double v1x = s_axes[0], v1y = s_axes[1], v1z = s_axes[2];
      const double v3x = s_axes[3], v3y = s_axes[4], v3z = s_axes[5];
      int px = 0, pz = 0;
      for (int j = tid; j < n; j += SHOT_THREADS) {
        const float4 p = pts[pos[j]];
        if (p.x == c.x && p.y == c.y && p.z == c.z) continue;
        const double vx = (double)(p.x - c.x), vy = (double)(p.y - c.y), vz = (double)(p.z - c.z);
        if (vx * v1x + vy * v1y + vz * v1z >= 0) ++px;
        if (vx * v3x + vy * v3y + vz * v3z >= 0) ++pz;
      }
      px = warp_sum(px);
      pz = warp_sum(pz);
      if ((tid & 31) == 0) {
        if (px) atomicAdd(&s_votes[1], px);
        if (pz) atomicAdd(&s_votes[2], pz);
      }
      __syncthreads();
      if (tid == 0) {
        double ax[2][3] = {{v1x, v1y, v1z}, {v3x, v3y, v3z}};
        for (int which = 0; which < 2; ++which) {
          int plus = 2 * s_votes[1 + which] - valid;
          double *a = ax[which];
          if (plus == 0) {
            // tie: look at the 5 valid rows around the median distance (rows are distance sorted;
            // the skipped rows are the d2 == 0 prefix of the list)
            const int med = valid / 2;
            for (int t = -2; t <= 2; ++t) {
              const float4 p = pts[pos[n_skip + med - t]];
              const double vx = (double)(p.x - c.x), vy = (double)(p.y - c.y), vz = (double)(p.z - c.z);
              if (vx * a[0] + vy * a[1] + vz * a[2] > 0) ++plus;
            }
            if (plus < 3) {
              a[0] = -a[0];
              a[1] = -a[1];
              a[2] = -a[2];
            }
          } else if (plus < 0) {
            a[0] = -a[0];
            a[1] = -a[1];
            a[2] = -a[2];
          }
        }
        const float x0 = (float)ax[0][0], x1 = (float)ax[0][1], x2 = (float)ax[0][2];
        const float z0 = (float)ax[1][0], z1 = (float)ax[1][1], z2 = (float)ax[1][2];
        s_frame[0] = x0;
        s_frame[1] = x1;
        s_frame[2] = x2;
        s_frame[3] = z1 * x2 - z2 * x1;  // y = z cross x (float)
        s_frame[4] = z2 * x0 - z0 * x2;
        s_frame[5] = z0 * x1 - z1 * x0;
        s_frame[6] = z0;
        s_frame[7] = z1;
        s_frame[8] = z2;
      }
      __syncthreads();
    }

    if (lrf_only) {
      if (tid < 9) rf_out[(size_t)i * 9 + tid] = ok ? s_frame[tid] : nanf32();
      __syncthreads();
      continue;
    }

    // SHOTEstimation::computeFeature: non-finite keypoint, NaN frame or empty search → NaN row;
    // computePointSHOT: fewer than 5 neighbours → NaN descriptor.
    const bool desc_ok = ok && n >= 5;
    if (desc_ok) {
      float fr[9];
#pragma unroll
      for (int a = 0; a < 9; ++a) fr[a] = s_frame[a];
      for (int j = tid; j < n; j += SHOT_THREADS) {
        const int pj = pos[j];
        const float4 nv = nrm[pj];
        if (!finite3(nv.x, nv.y, nv.z)) continue;
        shot_neighbor_exact(FloatBins{s_hist}, nv, pts[pj], c, key_d2(key[j]), fr, radius);
      }
      __syncthreads();
      // normalizeHistogram: acc_norm (double) += shot[j] * shot[j] (float product)
      double acc = 0.0;
      for (int b = tid; b < SHOT_LEN; b += SHOT_THREADS) {
        const float h = s_hist[b];
        acc += (double)(h * h);
      }
      acc = warp_sum(acc);
      if ((tid & 31) == 0) s_norm[tid >> 5] = acc;
      __syncthreads();
      const double acc_norm = sqrt(((s_norm[0] + s_norm[1]) + s_norm[2]) + s_norm[3]);
      const float fnorm = (float)acc_norm;
      for (int b = tid; b < SHOT_LEN; b += SHOT_THREADS) desc[(size_t)i * SHOT_LEN + b] = s_hist[b] / fnorm;
      if (rf_out && tid < 9) rf_out[(size_t)i * 9 + tid] = s_frame[tid];
    } else {
      for (int b = tid; b < SHOT_LEN; b += SHOT_THREADS) desc[(size_t)i * SHOT_LEN + b] = nanf32();
      // rf is NaN when the row is rejected by computeFeature (frame NaN / empty search); a valid frame
      // with 1..4 neighbours cannot occur (a valid frame needs >= 5 neighbours)
      if (rf_out && tid < 9) rf_out[(size_t)i * 9 + tid] = nanf32();
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// warp-per-keypoint kernel
// ------------------------------------------------------------------------------------------
constexpr int SW_WARPS = 8;
constexpr int SW_THREADS = SW_WARPS * 32;
constexpr int SW_CAP = 2016;  // neighbours per keypoint held in shared memory (three CTAs of 8 warps fit one SM)

// ---- local reference frame, pass 1: neighbour count + weighted covariance sums (shot_lrf.hpp getLocalRF) -----------
// One keypoint per warp, straight over the candidate cells (no list): n = #{d2 < r2}, the number of neighbours
// coinciding with the keypoint (PCL skips them), and the seven float64 sums  sum w v v^T (upper triangle), sum w  with
// w = r - |v|.  This pass doubles as the neighbour count every descriptor call needs (list sizing, n-bar statistics).
// The eigen-solve then runs one keypoint per THREAD (shot_eigen_kernel) instead of on one lane of a warp whose other
// 31 lanes idle, and the descriptor kernel's instruction footprint shrinks by the float64 Jacobi code (the fused
// kernel stalled on instruction fetch more than on anything else: 24 warps per SM in different phases of 64 KB of code).
__global__ void __launch_bounds__(256)
    shot_count_cov_kernel(GridView g, const float4 *__restrict__ kp, int K, float radius_f, double radius, float r2,
                          int *__restrict__ counts, double *__restrict__ acc, unsigned long long *__restrict__ stats) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= K) return;
  const float4 c = kp[i];
  double part[7] = {0, 0, 0, 0, 0, 0, 0};
  int n = 0, skipped = 0;
  int x0, x1, y0, y1, z0, z1;
  if (finite3(c.x, c.y, c.z) && g.n > 0 && ball_cell_range(g, c.x, c.y, c.z, radius_f, x0, x1, y0, y1, z0, z1)) {
    const float4 *__restrict__ pts = g.pts;
    const int *__restrict__ cs = g.cell_start;
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) {
        const int base = g.dx * (y + g.dy * z);
        const int e = cs[base + x1 + 1];
        for (int j0 = cs[base + x0] + lane; j0 < e; j0 += 128) {
         float4 pp[4];
#pragma unroll
         for (int u = 0; u < 4; ++u) pp[u] = (j0 + 32 * u < e) ? pts[j0 + 32 * u] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
         for (int u = 0; u < 4; ++u) {
          const float4 p = pp[u];
          const float d2 = (j0 + 32 * u < e) ? sqdist3(c.x, c.y, c.z, p.x, p.y, p.z) : 3.0e38f;
          if (d2 < r2) {
            ++n;
            if (p.x == c.x && p.y == c.y && p.z == c.z) {
              ++skipped;
            } else {
              const double vx = (double)(p.x - c.x), vy = (double)(p.y - c.y), vz = (double)(p.z - c.z);
              const double w = radius - sqrt((double)d2);
              part[0] += w * (vx * vx);
              part[1] += w * (vx * vy);
              part[2] += w * (vx * vz);
              part[3] += w * (vy * vy);
              part[4] += w * (vy * vz);
              part[5] += w * (vz * vz);
              part[6] += w;
            }
          }
         }
        }
      }
  }
#pragma unroll
  for (int a = 0; a < 7; ++a) part[a] = warp_sum(part[a]);
  n = warp_sum(n);
  skipped = warp_sum(skipped);
  if (lane < 7) {
    double v = part[0];
#pragma unroll
    for (int a = 1; a < 7; ++a)
      if (lane == a) v = part[a];
    acc[(size_t)i * 8 + lane] = v;
  }
  if (lane == 7) acc[(size_t)i * 8 + 7] = (double)skipped;
  if (lane == 0) {
    counts[i] = n;
    if (stats) {
      atomicMax(&stats[0], (unsigned long long)n);
      atomicAdd(&stats[1], (unsigned long long)n);
    }
  }
}

// ---- pass 2: 3x3 eigen-solve, one keypoint per thread.  axes: x axis (largest eigenvalue) and z axis (smallest)
// before the sign disambiguation, float64; flags: 1 = frame defined (>= 5 valid neighbours, finite eigenvalues) ----
__global__ void shot_eigen_kernel(const int *__restrict__ counts, const double *__restrict__ acc, int K,
                                  double *__restrict__ axes, int *__restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K) return;
  const double *s = acc + (size_t)i * 8;
  const int valid = counts[i] - (int)s[7];
  int ok = valid >= 5 ? 1 : 0;
  double ax[6] = {0, 0, 0, 0, 0, 0};
  if (ok) {
    const double cov[9] = {s[0] / s[6], s[1] / s[6], s[2] / s[6], s[1] / s[6], s[3] / s[6],
                           s[4] / s[6], s[2] / s[6], s[4] / s[6], s[5] / s[6]};
    double w[3], V[9];
    eigh3_f64(cov, w, V);
    if (!isfinite(w[0]) || !isfinite(w[1]) || !isfinite(w[2])) ok = 0;
    ax[0] = V[0 * 3 + 2], ax[1] = V[1 * 3 + 2], ax[2] = V[2 * 3 + 2];
    ax[3] = V[0 * 3 + 0], ax[4] = V[1 * 3 + 0], ax[5] = V[2 * 3 + 0];
  }
#pragma unroll
  for (int a = 0; a < 6; ++a) axes[(size_t)i * 6 + a] = ax[a];
  flags[i] = ok;
}

struct ShotWarpSmem {
  int pos[SW_CAP];     // position of the neighbour in the cell-ordered point array; its float32 squared
                       // distance (FLANN's L2_Simple value) is recomputed from the point when needed
  int hist[SHOT_LEN];  // fixed point (FixedBins), read back as unsigned
  int sel[8];          // rows picked by the tie rule
};

__global__ void __launch_bounds__(SW_THREADS, 3)
    shot_warp_kernel(GridView g, const float4 *__restrict__ nrm, const float4 *__restrict__ kp,
                     const int *__restrict__ counts, const double *__restrict__ acc, const double *__restrict__ axes,
                     const int *__restrict__ flags, int K, float radius_f, double radius, float r2,
                     int *__restrict__ work_counter, float *__restrict__ desc, float *__restrict__ rf_out,
                     int lrf_only) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  ShotWarpSmem &sm = reinterpret_cast<ShotWarpSmem *>(smem_raw)[warp];
  const float4 *__restrict__ pts = g.pts;

  const double radius3_4 = (radius * 3) / 4, radius1_4 = radius / 4, radius1_2 = radius / 2;
  const float r12f = (float)radius1_2, r34f = (float)radius3_4, r14f = (float)radius1_4;
  const float inv_r12f = 1.0f / r12f;
  const float m_r = 1e-6f * radius_f;  // band around the radial thresholds: covers sqrtf vs sqrt((double)d2)
  const float RAD_45f = 0.78539816339744830961566084581988f, RAD_90f = 1.5707963267948966192313216916398f;
  const float RAD_135f = 2.3561944901923449288469825374596f, RAD_PI_7_8f = 2.7488935718910690836548129603691f;
  const float INV_RAD_90f = 1.0f / RAD_90f, INV_RAD_45f = 1.0f / RAD_45f;
  const float COS_45f = 0.70710678118654752440f;

  while (true) {
    int i = 0;
    if (lane == 0) i = atomicAdd(work_counter, 1);
    i = __shfl_sync(0xffffffffu, i, 0);
    if (i >= K) break;
    if (counts[i] > SW_CAP) continue;  // left to shot_kernel
    const float4 c = kp[i];

    const int n = warp_gather_radius<SW_CAP>(g, c, radius_f, r2, nullptr, sm.pos, lane);
    for (int b = lane; b < SHOT_LEN; b += 32) sm.hist[b] = 0;
    __syncwarp();

    // ---- local reference frame: covariance sums and eigenvectors come from the two passes above ----
    const int n_skip = (int)acc[(size_t)i * 8 + 7];
    const int valid = n - n_skip;
    const int ok = flags[i];
    double ax[6];  // x axis (largest eigenvalue), z axis (smallest), before disambiguation
#pragma unroll
    for (int a = 0; a < 6; ++a) ax[a] = axes[(size_t)i * 6 + a];
    float fr[9];
    if (ok) {
      // sign votes: v . axis >= 0 in float64; a float32 estimate settles the clear cases
      const float a0 = (float)ax[0], a1 = (float)ax[1], a2 = (float)ax[2];
      const float b0 = (float)ax[3], b1 = (float)ax[4], b2 = (float)ax[5];
      int px = 0, pz = 0;
      for (int j = lane; j < n; j += 32) {
        const float4 p = pts[sm.pos[j]];
        if (p.x == c.x && p.y == c.y && p.z == c.z) continue;
        const float fx = p.x - c.x, fy = p.y - c.y, fz = p.z - c.z;
        const float band = 4e-6f * (fabsf(fx) + fabsf(fy) + fabsf(fz));
        const float ex = fx * a0 + fy * a1 + fz * a2, ez = fx * b0 + fy * b1 + fz * b2;
        if (fabsf(ex) > band)
          px += ex > 0.f;
        else
          px += ((double)fx * ax[0] + (double)fy * ax[1] + (double)fz * ax[2] >= 0) ? 1 : 0;
        if (fabsf(ez) > band)
          pz += ez > 0.f;
        else
          pz += ((double)fx * ax[3] + (double)fy * ax[4] + (double)fz * ax[5] >= 0) ? 1 : 0;
      }
      px = warp_sum(px);
      pz = warp_sum(pz);
      const int plus_x = 2 * px - valid, plus_z = 2 * pz - valid;
      if (plus_x == 0 || plus_z == 0) {
        // tie: PCL looks at the 5 valid rows around the median distance of the (d2, index)-sorted
        // list (the skipped rows are its d2 == 0 prefix): select them by rank
        const int r0 = n_skip + valid / 2 - 2;
        // squared distances: staged in the unused half of the list when it fits, else recomputed
        const bool staged = n <= SW_CAP / 2;
        float *d2s = reinterpret_cast<float *>(sm.pos + SW_CAP / 2);
        auto d2_at = [&](int a) -> float {
          if (staged) return d2s[a];
          const float4 q = pts[sm.pos[a]];
          return sqdist3(c.x, c.y, c.z, q.x, q.y, q.z);
        };
        if (staged) {
          for (int a = lane; a < n; a += 32) {
            const float4 q = pts[sm.pos[a]];
            d2s[a] = sqdist3(c.x, c.y, c.z, q.x, q.y, q.z);
          }
          __syncwarp();
        }
        // d2 values (as ordered bit patterns) of ranks r0 and r0 + 4 by bisection on the bits ...
        unsigned u_lo = 0, u_hi = 0;
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
          const int target = r0 + 4 * which + 1;  // smallest u with #{d2 <= u} >= target
          unsigned lo = 0, hi = 0x7f800000u;
          while (lo < hi) {
            const unsigned mid = lo + ((hi - lo) >> 1);
            int cnt = 0;
            for (int a = lane; a < n; a += 32) cnt += __float_as_uint(d2_at(a)) <= mid;
            cnt = __reduce_add_sync(0xffffffffu, cnt);
            if (cnt >= target)
              hi = mid;
            else
              lo = mid + 1;
          }
          if (which)
            u_hi = lo;
          else
            u_lo = lo;
        }
        // ... then exact (d2, index) ranks only for the few rows in that value range
        for (int a0 = 0; a0 < n; a0 += 32) {
          const int a = a0 + lane;
          const unsigned ua = (a < n) ? __float_as_uint(d2_at(a)) : 0xffffffffu;
          unsigned todo = __ballot_sync(0xffffffffu, a < n && ua >= u_lo && ua <= u_hi);
          while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int e = a0 + src;
            const float de = d2_at(e);
            const int pe = sm.pos[e];
            const int oe = orig_index(pts[pe]);
            int rank = 0;
            for (int b = lane; b < n; b += 32) {
              const float db = d2_at(b);
              if (db < de)
                ++rank;
              else if (db == de && b != e)
                rank += orig_index(pts[sm.pos[b]]) < oe;
            }
            rank = __reduce_add_sync(0xffffffffu, rank);
            if (lane == 0 && rank >= r0 && rank < r0 + 5) sm.sel[rank - r0] = pe;
          }
        }
        __syncwarp();
      }
      if (lane == 0) {
        for (int which = 0; which < 2; ++which) {
          int plus = which ? plus_z : plus_x;
          double *a = ax + 3 * which;
          if (plus == 0) {
            for (int t = 0; t < 5; ++t) {
              const float4 p = pts[sm.sel[t]];
              const double vx = (double)(p.x - c.x), vy = (double)(p.y - c.y), vz = (double)(p.z - c.z);
              if (vx * a[0] + vy * a[1] + vz * a[2] > 0) ++plus;
            }
            if (plus < 3) a[0] = -a[0], a[1] = -a[1], a[2] = -a[2];
          } else if (plus < 0) {
            a[0] = -a[0], a[1] = -a[1], a[2] = -a[2];
          }
        }
        const float x0 = (float)ax[0], x1 = (float)ax[1], x2 = (float)ax[2];
        const float z0 = (float)ax[3], z1 = (float)ax[4], z2 = (float)ax[5];
        fr[0] = x0, fr[1] = x1, fr[2] = x2;
        fr[3] = z1 * x2 - z2 * x1;  // y = z cross x (float)
        fr[4] = z2 * x0 - z0 * x2;
        fr[5] = z0 * x1 - z1 * x0;
        fr[6] = z0, fr[7] = z1, fr[8] = z2;
      }
#pragma unroll
      for (int a = 0; a < 9; ++a) fr[a] = __shfl_sync(0xffffffffu, fr[a], 0);
    }

    if (lrf_only) {
      if (lane < 9) {
        float v = nanf32();
#pragma unroll
        for (int a = 0; a < 9; ++a)
          if (lane == a && ok) v = fr[a];
        rf_out[(size_t)i * 9 + lane] = v;
      }
      continue;
    }

    // SHOTEstimation::computeFeature: non-finite keypoint, NaN frame or empty search → NaN row;
    // computePointSHOT: fewer than 5 neighbours → NaN descriptor.
    const bool desc_ok = ok && n >= 5;
    if (desc_ok) {
      const float fxx = fr[0], fxy = fr[1], fxz = fr[2];
      const float fyx = fr[3], fyy = fr[4], fyz = fr[5];
      const float fzx = fr[6], fzy = fr[7], fzz = fr[8];
      const float fx_scale = (n <= 1024) ? 1048576.0f : 524288.0f, fx_inv = 1.0f / fx_scale;
      const FixedBins hist{sm.hist, fx_scale};
      for (int j = lane; j < n; j += 32) {
        const int pj = sm.pos[j];
        const float4 nv = nrm[pj];
        if (!finite3(nv.x, nv.y, nv.z)) continue;
        const float4 p = pts[pj];
        const float d2 = sqdist3(c.x, c.y, c.z, p.x, p.y, p.z);
        // ---- float32 evaluation with error bands; `slow` → PCL's float64 expressions decide ----
        const float df = sqrtf(d2);
        bool slow = d2 < 1e-29f || fabsf(df - r12f) < m_r || fabsf(df - r34f) < m_r || fabsf(df - r14f) < m_r;
        const float dx = p.x - c.x, dy = p.y - c.y, dz = p.z - c.z;
        float xf = dx * fxx;
        xf += dy * fxy;
        xf += dz * fxz;
        float yf = dx * fyx;
        yf += dy * fyy;
        yf += dz * fyz;
        float zf = dx * fzx;
        zf += dy * fzy;
        zf += dz * fzz;
        // PCL zeroes |.| < 1e-30 (in float64): magnitudes this small go to the exact path
        slow = slow || fabsf(xf) < 1e-29f || fabsf(yf) < 1e-29f || fabsf(zf) < 1e-29f;
        const float cosv = zf / df;
        const float acv = fabsf(cosv);
        slow = slow || fabsf(acv - COS_45f) < 2e-6f;
        const float az = atan2f(yf, xf);
        // sector bits: sign and magnitude comparisons of float values are exact in float32
        const int bit4 = (yf > 0.f) ? 1 : 0;
        const int bit3 = ((xf > 0.f) ? !bit4 : bit4) ? 1 : 0;
        int desc_index = ((bit4 << 3) + (bit3 << 2)) << 1;
        if ((xf > 0.f) == (yf > 0.f))
          desc_index += (fabsf(xf) >= fabsf(yf)) ? 0 : 4;
        else
          desc_index += (fabsf(xf) > fabsf(yf)) ? 4 : 0;
        const int sel = desc_index >> 2;
        const float az0 = -RAD_PI_7_8f + RAD_45f * (float)sel;
        slow = slow || fabsf(az - az0) < 6e-6f;
        if (slow) {
          shot_neighbor_exact(hist, nv, p, c, d2, fr, radius);
          continue;
        }
        desc_index += zf > 0.f ? 1 : 0;
        desc_index += (df > r12f) ? 2 : 0;
        // createBinDistanceShape: the cosine bin is cheap in float64, exactly as PCL
        float dotf = nv.x * fzx;
        dotf += nv.y * fzy;
        dotf += nv.z * fzz;
        double cosineDesc = (double)dotf;
        if (cosineDesc > 1.0) cosineDesc = 1.0;
        if (cosineDesc < -1.0) cosineDesc = -1.0;
        double binDistance = ((1.0 + cosineDesc) * 10) / 2;
        const int step_index = (int)floor(binDistance + 0.5);
        const int volume_index = desc_index * 11;
        binDistance -= step_index;
        const float bd = (float)binDistance;
        float intWeight = (float)(1 - fabs(binDistance));
        if (binDistance > 0)
          hist.add(volume_index + ((step_index + 1) % 10), bd);
        else
          hist.add(volume_index + ((step_index - 1 + 10) % 10), -bd);
        // radial
        if (df > r12f) {
          const float rd = (df - r34f) * inv_r12f;
          if (df > r34f)
            intWeight += 1 - rd;
          else {
            intWeight += 1 + rd;
            hist.add((desc_index - 2) * 11 + step_index, -rd);
          }
        } else {
          const float rd = (df - r14f) * inv_r12f;
          if (df < r14f)
            intWeight += 1 + rd;
          else {
            intWeight += 1 - rd;
            hist.add((desc_index + 2) * 11 + step_index, rd);
          }
        }
        // elevation: acos(z/d) > 90 degrees <=> z <= 0 (PCL's tie clause covers z == 0)
        const float inc = acosf(fminf(1.0f, fmaxf(-1.0f, cosv)));
        if (zf < 0.f) {
          const float id = (inc - RAD_135f) * INV_RAD_90f;
          if (cosv < -COS_45f)
            intWeight += 1 - id;
          else {
            intWeight += 1 + id;
            hist.add((desc_index + 1) * 11 + step_index, -id);
          }
        } else {
          const float id = (inc - RAD_45f) * INV_RAD_90f;
          if (cosv > COS_45f)
            intWeight += 1 + id;
          else {
            intWeight += 1 - id;
            hist.add((desc_index - 1) * 11 + step_index, id);
          }
        }
        // azimuth (x and y are non-zero here)
        {
          float ad = (az - az0) * INV_RAD_45f;
          ad = fmaxf(-0.5f, fminf(ad, 0.5f));
          if (ad > 0) {
            intWeight += 1 - ad;
            hist.add(((desc_index + 4) % 32) * 11 + step_index, ad);
          } else {
            intWeight += 1 + ad;
            hist.add(((desc_index - 4 + 32) % 32) * 11 + step_index, -ad);
          }
        }
        hist.add(volume_index + step_index, intWeight);
      }
      __syncwarp();
      // normalizeHistogram: acc_norm (double) += shot[j] * shot[j] (float product)
      double acc = 0.0;
      for (int b = lane; b < SHOT_LEN; b += 32) {
        const float h = (float)(unsigned)sm.hist[b] * fx_inv;
        acc += (double)(h * h);
      }
      acc = warp_sum(acc);
      const float fnorm = (float)sqrt(acc);
      for (int b = lane; b < SHOT_LEN; b += 32)
        desc[(size_t)i * SHOT_LEN + b] = ((float)(unsigned)sm.hist[b] * fx_inv) / fnorm;
      if (rf_out && lane < 9) {
        float v = 0.f;
#pragma unroll
        for (int a = 0; a < 9; ++a)
          if (lane == a) v = fr[a];
        rf_out[(size_t)i * 9 + lane] = v;
      }
    } else {
      for (int b = lane; b < SHOT_LEN; b += 32) desc[(size_t)i * SHOT_LEN + b] = nanf32();
      if (rf_out && lane < 9) rf_out[(size_t)i * 9 + lane] = nanf32();
    }
    __syncwarp();
  }
}

}  // namespace

int dev_shot(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_kp, int K, double radius,
             float *d_desc, float *d_rf, bool lrf_only) {
  if (!(radius > 0.0)) return ctx->fail(B200_ERR_INVALID, "shot: radius must be > 0");
  if (K <= 0) return B200_OK;
  const GridView *g;
  B200_TRY(cloud_grid_for_radius(c, radius, &g));
  // pass 1: neighbour counts (list sizing, the bench's n-bar) + the frames' covariance sums; pass 2: eigen-solves
  DevBuf<int> counts, flags;
  DevBuf<double> acc, axes;
  DevBuf<unsigned long long> stats;
  B200_TRY(counts.alloc(ctx, (size_t)K));
  B200_TRY(flags.alloc(ctx, (size_t)K));
  B200_TRY(acc.alloc(ctx, (size_t)K * 8));
  B200_TRY(axes.alloc(ctx, (size_t)K * 6));
  B200_TRY(stats.alloc(ctx, 2));
  const float r2 = (float)(radius * radius);
  {
    StageScope stc_(ctx, ST_NBR_COUNT);
    B200_CUDA(ctx, cudaMemsetAsync(stats.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
    shot_count_cov_kernel<<<ceil_div((long long)K * 32, 256), 256, 0, ctx->stream>>>(*g, d_kp, K, (float)radius, radius,
                                                                                    r2, counts.p, acc.p, stats.p);
    B200_LAUNCHED(ctx);
    shot_eigen_kernel<<<ceil_div(K, 128), 128, 0, ctx->stream>>>(counts.p, acc.p, K, axes.p, flags.p);
    B200_LAUNCHED(ctx);
  }
  unsigned long long hstats[2];
  B200_TRY(readback_small(ctx, stats.p, hstats, sizeof(hstats)));
  const int max_count = (int)hstats[0];
  ctx->last_max_nbrs = max_count;
  ctx->last_mean_nbrs = (double)hstats[1] / K;

  StageScope st_(ctx, ST_SHOT);
  DevBuf<float4> nrm_sorted;
  if (!lrf_only) {
    B200_TRY(nrm_sorted.alloc(ctx, (size_t)std::max(c->n_valid, 1)));
    if (c->n_valid > 0) {
      gather_normals_kernel<<<ceil_div(c->n_valid, 256), 256, 0, ctx->stream>>>(
          g->pts, c->n_valid, reinterpret_cast<const float4 *>(d_normals), nrm_sorted.p);
      B200_LAUNCHED(ctx);
    }
  }
  // neighbourhoods up to SW_CAP points: one keypoint per warp, dynamic work distribution
  {
    DevBuf<int> work;
    B200_TRY(work.alloc(ctx, 1));
    B200_TRY(work.zero());
    const size_t smem_w = sizeof(ShotWarpSmem) * SW_WARPS;
    B200_CUDA(ctx, ensure_dyn_smem(shot_warp_kernel, smem_w));
    const int grid_w = std::min(ceil_div(K, SW_WARPS), ctx->sm_count * 3);
    shot_warp_kernel<<<grid_w, SW_THREADS, smem_w, ctx->stream>>>(*g, nrm_sorted.p, d_kp, counts.p, acc.p, axes.p, flags.p,
                                                                 K, (float)radius, radius, r2, work.p, d_desc, d_rf,
                                                                 lrf_only ? 1 : 0);
    B200_LAUNCHED(ctx);
  }
  if (max_count <= SW_CAP) return B200_OK;
  // larger neighbourhoods (e.g. SHOT_demo.cpp:498's radius 50): one keypoint per CTA, sorted list
  const int min_count = SW_CAP + 1;
  const int cap = next_pow2_host(std::max(max_count, 32));
  const size_t smem = (size_t)cap * 12;
  if (smem <= 96 * 1024) {
    B200_CUDA(ctx, ensure_dyn_smem(shot_kernel, smem));
    int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 4096)));
    const int grid = std::min(K, ctx->sm_count * per_sm);
    shot_kernel<<<grid, SHOT_THREADS, smem, ctx->stream>>>(*g, nrm_sorted.p, d_kp, K, (float)radius, radius, r2, cap,
                                                          nullptr, nullptr, d_desc, d_rf, lrf_only ? 1 : 0, counts.p, min_count);
    B200_LAUNCHED(ctx);
  } else {
    const int grid = std::min(K, ctx->sm_count * 2);
    DevBuf<unsigned long long> gk;
    DevBuf<int> gp;
    B200_TRY(gk.alloc(ctx, (size_t)grid * cap));
    B200_TRY(gp.alloc(ctx, (size_t)grid * cap));
    shot_kernel<<<grid, SHOT_THREADS, 0, ctx->stream>>>(*g, nrm_sorted.p, d_kp, K, (float)radius, radius, r2, cap,
                                                       gk.p, gp.p, d_desc, d_rf, lrf_only ? 1 : 0, counts.p, min_count);
    B200_LAUNCHED(ctx);
  }
  return B200_OK;
}
