// search.cuh — device-side exact neighbour search on the uniform grid.
//
//  nbr_key             a neighbour as one 64-bit key: float bits of d2 (non-negative, so the unsigned order is the
//                      float order) in the high word, ORIGINAL row index in the low word.  One unsigned compare is
//                      FLANN's (distance, index) order (RadiusResultSet is sorted with DistanceIndex::operator<);
//                      key_d2 / key_orig decode it.
//  knn_query           one query per thread, candidate list in shared memory; replaces
//                      KdTreeFLANN::nearestKSearch as used by NormalEstimationOMP with setKSearch
//                      (SHOT.cpp:302-308) and by the explicit calls (SHOT.cpp:163, Edge_detection.cpp:120).
//  Radius search replaces KdTreeFLANN::radiusSearch (SHOT_VAR.cpp:356; implicit in SHOT / FPFH / radius normals).
//  Acceptance is d2 < (float)(r*r), strict, on the float32 L2_Simple distance — bit-identical to FLANN's test.
//  cta_list            the list storage of a one-query-per-CTA kernel: shared memory or a slice of global scratch.
//  gather_radius       one query per CTA, neighbours appended to a list with warp-aggregated atomics.
//  count_radius_warp   one query per warp, the number of neighbours (sizes the lists of both gathers).
//  bitonic_sort        orders a CTA's list by key.
//  warp_gather_radius  one query per warp, neighbours appended in scan order to the warp's list by ballot compaction.
//  warp_bitonic_sort   orders a warp's list by key, synchronised by __syncwarp only.
#pragma once

#include <type_traits>

#include "common.cuh"

__device__ __forceinline__ unsigned long long nbr_key(float d2, int orig) {
  return ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)orig;
}
__device__ __forceinline__ float key_d2(unsigned long long k) { return __uint_as_float((unsigned)(k >> 32)); }
__device__ __forceinline__ int key_orig(unsigned long long k) { return (int)(unsigned)(k & 0xffffffffull); }

// Exact k nearest neighbours of (qx,qy,qz).  sk: this thread's column of a [k][T] shared array of nbr_key keys
// (element j at [j*T]): a shift of the sorted list moves one 8-byte word per step.  Returns the number found
// (min(k, g.n)), sorted ascending.  Coordinates of a neighbour: g.raw[key_orig(key)].
__device__ inline int knn_query(const GridView &g, float qx, float qy, float qz, int k, unsigned long long *sk, int T) {
  const float4 *__restrict__ pts = g.pts;
  const int *__restrict__ cs = g.cell_start;
  if (k > g.n) k = g.n;
  if (k <= 0) return 0;
  const int cx = grid_coord(qx, g.lox, g.inv_h, g.dx);
  const int cy = grid_coord(qy, g.loy, g.inv_h, g.dy);
  const int cz = grid_coord(qz, g.loz, g.inv_h, g.dz);
  int cnt = 0;
  const int maxR = max(g.dx, max(g.dy, g.dz));
  const float margin = 4e-6f * (g.coord_scale + fabsf(qx) + fabsf(qy) + fabsf(qz)) + 1e-5f * g.h;
  unsigned long long worst = ~0ull;  // key of the current k-th neighbour once the list is full

  // The k best keys are kept as a MAX-HEAP in the shared-memory column (root = current k-th): a candidate that beats
  // the root replaces it and sinks at most log2(k) levels.  A sorted list (round 1) shifted k / 2 entries on average —
  // and, one query per thread, a warp executes the LONGEST shift of its inserting lanes: with the heap the longest
  // path is 4 levels for k = 20.  The list is put in (distance, index) order once at the end.  (A 4-ary heap — two
// levels, independent child loads — measured the same: 1.173 against 1.168 ms.)
  auto sift_down = [&](int i, int n, unsigned long long key) {  // key sinks from slot i of a heap of n slots
    while (true) {
      int c = 2 * i + 1;
      if (c >= n) break;
      unsigned long long ck = sk[c * T];
      if (c + 1 < n) {
        const unsigned long long ck2 = sk[(c + 1) * T];
        if (ck2 > ck) {
          ck = ck2;
          ++c;
        }
      }
      if (ck <= key) break;
      sk[i * T] = ck;
      i = c;
    }
    sk[i * T] = key;
  };
  auto scan_run = [&](int c0, int c1) {
    const int s = cs[c0], e = cs[c1 + 1];
    for (int j = s; j < e; ++j) {
      const float4 p = pts[j];
      const float d = sqdist3(qx, qy, qz, p.x, p.y, p.z);
      const unsigned long long key = nbr_key(d, orig_index(p));
      if (key >= worst) continue;
      if (cnt < k) {
        sk[cnt * T] = key;
        if (++cnt == k) {
          for (int i = k / 2 - 1; i >= 0; --i) sift_down(i, k, sk[i * T]);
          worst = sk[0];
        }
      } else {
        sift_down(0, k, key);
        worst = sk[0];
      }
    }
  };

  // Slab pruning.  Every point of a cell row (y, z fixed) is at least the row's slab distance away from the query;
  // once the list is full, a row (or a single cell of it) that is STRICTLY farther than the current k-th neighbour
  // cannot change the result — (distance, index) ties included — and is skipped.  -DB200_KNN_NO_PRUNE restores the
  // unpruned scan (the result is the same by construction; the parity tests hold either way).
#ifndef B200_KNN_NO_PRUNE
  auto gap = [&](int c, int qc, float q, float lo) -> float {  // lower bound of |coordinate - q| inside cell index c
    float d = 0.f;
    if (c > qc) d = (lo + (float)c * g.h) - q;
    else if (c < qc) d = q - (lo + (float)(c + 1) * g.h);
    return fmaxf(d - margin, 0.f);
  };
  auto row_far = [&](int y, int z, float gx) -> bool {
    if (cnt < k) return false;
    const float gy = gap(y, cy, qy, g.loy), gz = gap(z, cz, qz, g.loz);
    return (gx * gx + gy * gy + gz * gz) * 0.99999f > key_d2(worst);
  };
  // a row's run of cells xa..xb (it spans the query's column): the end cells are dropped while they are too far
  auto scan_row = [&](int y, int z, int row, int xa, int xb) {
    if (cnt == k) {
      const float gy = gap(y, cy, qy, g.loy), gz = gap(z, cz, qz, g.loz);
      const float yz = gy * gy + gz * gz, w = key_d2(worst);
      if (yz * 0.99999f > w) return;
      while (xa < cx) {
        const float gx = gap(xa, cx, qx, g.lox);
        if (!((gx * gx + yz) * 0.99999f > w)) break;
        ++xa;
      }
      while (xb > cx) {
        const float gx = gap(xb, cx, qx, g.lox);
        if (!((gx * gx + yz) * 0.99999f > w)) break;
        --xb;
      }
    }
    scan_run(row + xa, row + xb);
  };
#else
  auto gap = [&](int, int, float, float) -> float { return 0.f; };
  auto row_far = [&](int, int, float) -> bool { return false; };
  auto scan_row = [&](int, int, int row, int xa, int xb) { scan_run(row + xa, row + xb); };
#endif
  for (int R = 0; R <= maxR; ++R) {
    const int z0 = max(cz - R, 0), z1 = min(cz + R, g.dz - 1);
    const int y0 = max(cy - R, 0), y1 = min(cy + R, g.dy - 1);
    const int x0 = max(cx - R, 0), x1 = min(cx + R, g.dx - 1);
    if (R == 1) {
      // the first shell, nearest rows first (|dz| + |dy| = 0, 1, 2): the list fills with close points
      // early, so that most later candidates fail the cheap "farther than the current k-th" test
      // instead of being inserted and displaced again (the result does not depend on the order).  Measured and dropped:
      // visiting, of each pair of opposite neighbours, the one on the query's side of its cell first — the lanes of a
      // warp then read different rows at the same step: 1.06 against 1.02 ms
#pragma unroll 1
      for (int t = 0; t < 9; ++t) {
        const int dz = (t == 3) ? -1 : (t == 4) ? 1 : (t >= 5) ? ((t & 1) ? -1 : 1) : 0;
        const int dy = (t == 1) ? -1 : (t == 2) ? 1 : (t >= 5) ? ((t < 7) ? -1 : 1) : 0;
        const int z = cz + dz, y = cy + dy;
        if (z < 0 || z >= g.dz || y < 0 || y >= g.dy) continue;
        const int row = g.dx * (y + g.dy * z);
        if (t == 0) {
          if (cx - 1 >= 0 && !row_far(y, z, gap(cx - 1, cx, qx, g.lox))) scan_run(row + cx - 1, row + cx - 1);
          if (cx + 1 <= g.dx - 1 && !row_far(y, z, gap(cx + 1, cx, qx, g.lox))) scan_run(row + cx + 1, row + cx + 1);
        } else {
          scan_row(y, z, row, x0, x1);
        }
      }
    } else
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) {
        const bool face = (abs(z - cz) == R) || (abs(y - cy) == R);
        const int row = g.dx * (y + g.dy * z);
        if (face) {
          scan_row(y, z, row, x0, x1);
        } else {
          if (cx - R >= 0 && !row_far(y, z, gap(cx - R, cx, qx, g.lox))) scan_run(row + cx - R, row + cx - R);
          // R > 0 here (R == 0 is a face row)
          if (cx + R <= g.dx - 1 && !row_far(y, z, gap(cx + R, cx, qx, g.lox))) scan_run(row + cx + R, row + cx + R);
        }
      }
    const bool whole = (z0 == 0 && z1 == g.dz - 1 && y0 == 0 && y1 == g.dy - 1 && x0 == 0 && x1 == g.dx - 1);
    if (whole) break;
    if (cnt == k) {
      // everything outside the scanned block is at least `cert` away from the query
      float cert = 3.0e38f;
      if (cx - R > 0) cert = fminf(cert, qx - (g.lox + (float)(cx - R) * g.h));
      if (cx + R < g.dx - 1) cert = fminf(cert, (g.lox + (float)(cx + R + 1) * g.h) - qx);
      if (cy - R > 0) cert = fminf(cert, qy - (g.loy + (float)(cy - R) * g.h));
      if (cy + R < g.dy - 1) cert = fminf(cert, (g.loy + (float)(cy + R + 1) * g.h) - qy);
      if (cz - R > 0) cert = fminf(cert, qz - (g.loz + (float)(cz - R) * g.h));
      if (cz + R < g.dz - 1) cert = fminf(cert, (g.loz + (float)(cz + R + 1) * g.h) - qz);
      cert -= margin;
      if (cert > 0.f && key_d2(worst) < cert * cert * 0.99999f) break;
    }
  }
  // ascending (distance, index) order: FLANN's result order
  if (cnt == k) {
    for (int n = k - 1; n > 0; --n) {  // heap sort: the maximum goes to the end, the former last key sinks from the root
      const unsigned long long last = sk[n * T];
      sk[n * T] = sk[0];
      sift_down(0, n, last);
    }
  } else {
    for (int i = 1; i < cnt; ++i) {  // fewer points than k in the whole grid: the list was only appended to
      const unsigned long long key = sk[i * T];
      int pos = i;
      while (pos > 0) {
        const unsigned long long pk = sk[(pos - 1) * T];
        if (pk < key) break;
        sk[pos * T] = pk;
        --pos;
      }
      sk[pos * T] = key;
    }
  }
  return cnt;
}

// A two-pass form of knn_query (the K smallest distances in registers by a min/max chain, then a second pass that
// collects the winners) executed 20 % fewer instructions but measured 1.45 ms against 1.32 ms on the 1 M-point scene,
// k = 20, because its candidate loop waits on its loads (DESIGN.md section 4).

// Cell range of the ball around q, padded so that float rounding can never exclude a point the
// distance test would accept.  Returns false if the ball misses the grid entirely.
// Measured and dropped (end of round 2): sphere-against-cell pruning inside this box (rows and end cells whose slab
// distance reaches the radius: a fifth of the corner rows, half of their end cells).  Identical results, but slower —
// neighbour count 0.29 -> 0.37 ms, SHOT 0.90 -> 1.01 ms: a warp reads a row of cells 128 points per trip, so dropping
// a cell rarely saves a trip while every row pays for the test.  (The same idea does pay in knn_query, one query per
// thread, where every skipped candidate is a skipped iteration.)
__device__ __forceinline__ bool ball_cell_range(const GridView &g, float qx, float qy, float qz, float radius,
                                                int &x0, int &x1, int &y0, int &y1, int &z0, int &z1) {
  const float rp = radius * 1.00001f;
  const float ex = rp + 2e-6f * (fabsf(qx) + g.coord_scale);
  const float ey = rp + 2e-6f * (fabsf(qy) + g.coord_scale);
  const float ez = rp + 2e-6f * (fabsf(qz) + g.coord_scale);
  const float hix = g.lox + (float)g.dx * g.h, hiy = g.loy + (float)g.dy * g.h, hiz = g.loz + (float)g.dz * g.h;
  if (qx + ex < g.lox || qx - ex > hix + g.h || qy + ey < g.loy || qy - ey > hiy + g.h || qz + ez < g.loz ||
      qz - ez > hiz + g.h)
    return false;
  x0 = grid_coord(qx - ex, g.lox, g.inv_h, g.dx);
  x1 = grid_coord(qx + ex, g.lox, g.inv_h, g.dx);
  y0 = grid_coord(qy - ey, g.loy, g.inv_h, g.dy);
  y1 = grid_coord(qy + ey, g.loy, g.inv_h, g.dy);
  z0 = grid_coord(qz - ez, g.loz, g.inv_h, g.dz);
  z1 = grid_coord(qz + ez, g.loz, g.inv_h, g.dz);
  return true;
}

// List storage of a one-query-per-CTA kernel: `cap` keys, then `cap` positions, in the dynamic shared memory smem; or,
// when glob_key is set (lists too long for shared memory), this CTA's slices of the global scratch glob_key / glob_pos.
__device__ __forceinline__ void cta_list(unsigned char *smem, unsigned long long *glob_key, int *glob_pos, int cap,
                                         unsigned long long *&key, int *&pos) {
  if (glob_key) {
    key = glob_key + (size_t)blockIdx.x * cap;
    pos = glob_pos + (size_t)blockIdx.x * cap;
  } else {
    key = reinterpret_cast<unsigned long long *>(smem);
    pos = reinterpret_cast<int *>(smem + (size_t)cap * sizeof(unsigned long long));
  }
}

// CTA-cooperative radius gather.  Every thread of the block must call it.  key/pos: list storage
// with room for `cap` entries (shared or global).  Returns the total number of neighbours; only the
// first `cap` (in arrival order) are stored.  s_count: one int of shared memory.
__device__ inline int gather_radius(const GridView &g, float qx, float qy, float qz, float radius, float r2,
                                    unsigned long long *key, int *pos, int cap, int *s_count) {
  if (threadIdx.x == 0) *s_count = 0;
  __syncthreads();
  int x0, x1, y0, y1, z0, z1;
  if (finite3(qx, qy, qz) && g.n > 0 && ball_cell_range(g, qx, qy, qz, radius, x0, x1, y0, y1, z0, z1)) {
    const float4 *__restrict__ pts = g.pts;
    const int *__restrict__ cs = g.cell_start;
    const int ny = y1 - y0 + 1;
    const int nrows = ny * (z1 - z0 + 1);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int row = warp; row < nrows; row += nw) {
      const int y = y0 + row % ny, z = z0 + row / ny;
      const int base = g.dx * (y + g.dy * z);
      const int s = cs[base + x0], e = cs[base + x1 + 1];
      for (int j0 = s; j0 < e; j0 += 32) {
        const int j = j0 + lane;
        bool hit = false;
        float d2 = 0.f;
        float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < e) {
          p = pts[j];
          d2 = sqdist3(qx, qy, qz, p.x, p.y, p.z);
          hit = d2 < r2;
        }
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (m) {
          int slot0 = 0;
          if (lane == 0) slot0 = atomicAdd(s_count, __popc(m));
          slot0 = __shfl_sync(0xffffffffu, slot0, 0);
          if (hit) {
            const int slot = slot0 + __popc(m & ((1u << lane) - 1u));
            if (slot < cap) {
              key[slot] = nbr_key(d2, orig_index(p));
              pos[slot] = j;
            }
          }
        }
      }
    }
  }
  __syncthreads();
  return *s_count;
}

// Count-only variant for one warp (used to size lists / CSR outputs).
__device__ inline int count_radius_warp(const GridView &g, float qx, float qy, float qz, float radius, float r2) {
  int x0, x1, y0, y1, z0, z1;
  int c = 0;
  if (finite3(qx, qy, qz) && g.n > 0 && ball_cell_range(g, qx, qy, qz, radius, x0, x1, y0, y1, z0, z1)) {
    const float4 *__restrict__ pts = g.pts;
    const int *__restrict__ cs = g.cell_start;
    const int lane = threadIdx.x & 31;
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) {
        const int base = g.dx * (y + g.dy * z);
        const int s = cs[base + x0], e = cs[base + x1 + 1];
        for (int j = s + lane; j < e; j += 32) {
          const float4 p = pts[j];
          c += (sqdist3(qx, qy, qz, p.x, p.y, p.z) < r2) ? 1 : 0;
        }
      }
  }
  return warp_sum(c);
}

// CTA-cooperative bitonic sort of n (key, pos) pairs, ascending key.  The arrays must have room for
// the next power of two >= n.  Every thread of the block must call it.
__device__ inline void bitonic_sort(unsigned long long *key, int *pos, int n) {
  int np = 1;
  while (np < n) np <<= 1;
  for (int i = n + threadIdx.x; i < np; i += blockDim.x) {
    key[i] = ~0ull;
    pos[i] = -1;
  }
  __syncthreads();
  for (int k = 2; k <= np; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (np >> 1); t += blockDim.x) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = i | j;
        const bool up = ((i & k) == 0);
        const unsigned long long a = key[i], b = key[l];
        if ((a > b) == up) {
          key[i] = b;
          key[l] = a;
          const int pa = pos[i];
          pos[i] = pos[l];
          pos[l] = pa;
        }
      }
      __syncthreads();
    }
}

// One-warp radius gather: the neighbours of c (the count pass's guard and test, so their number is what
// count_radius_warp returned) are appended to the warp's list in scan order — cell rows z-major, then y, each row's
// points in cell order — as keys and / or positions in g.pts; key or pos may be nullptr.  Returns min(count, CAP);
// only the first CAP are stored.  Every lane of the warp must call it.  BOARD's warp kernel adds its float64 sums in
// this order: changing the order changes its frames.  (A nullptr argument is told apart by its type, so the compiler
// drops the store; a run-time test of a pointer into shared memory is not folded away.)
template <int CAP, class KeyPtr, class PosPtr>
__device__ __forceinline__ int warp_gather_radius(const GridView &g, const float4 c, float radius, float r2, KeyPtr key,
                                                  PosPtr pos, int lane) {
  int n = 0;
  int x0, x1, y0, y1, z0, z1;
  if (finite3(c.x, c.y, c.z) && g.n > 0 && ball_cell_range(g, c.x, c.y, c.z, radius, x0, x1, y0, y1, z0, z1)) {
    const float4 *__restrict__ pts = g.pts;
    const int *__restrict__ cs = g.cell_start;
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) {
        const int base = g.dx * (y + g.dy * z);
        const int s0 = cs[base + x0], e = cs[base + x1 + 1];
        // four 32-point chunks per trip, their loads issued before the first ballot (a trip per chunk made every
        // chunk wait for its own L2 round trip: SHOT's largest stall)
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
            const float d2 = sqdist3(c.x, c.y, c.z, p[u].x, p[u].y, p[u].z);
            const bool hit = j < e && d2 < r2;
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (hit) {
              const int slot = n + __popc(m & ((1u << lane) - 1u));
              if (slot < CAP) {
                if constexpr (!std::is_null_pointer_v<KeyPtr>) key[slot] = nbr_key(d2, orig_index(p[u]));
                if constexpr (!std::is_null_pointer_v<PosPtr>) pos[slot] = j;
              }
            }
            n += __popc(m);
          }
        }
      }
  }
  return min(n, CAP);
}

// One-warp bitonic sort of n (key, pos) pairs, ascending key, synchronised by __syncwarp only; pos may be nullptr.
// The arrays must have room for the next power of two >= max(n, 32).  Every lane of the warp must call it.
template <class PosPtr>
__device__ __forceinline__ void warp_bitonic_sort(unsigned long long *key, PosPtr pos, int n, int lane) {
  int np = 32;
  while (np < n) np <<= 1;
  for (int t = n + lane; t < np; t += 32) {
    key[t] = ~0ull;
    if constexpr (!std::is_null_pointer_v<PosPtr>) pos[t] = -1;
  }
  __syncwarp();
  for (int k = 2; k <= np; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = lane; t < (np >> 1); t += 32) {
        const int a = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int b = a | j;
        const bool up = ((a & k) == 0);
        const unsigned long long ka = key[a], kb = key[b];
        if ((ka > kb) == up) {
          key[a] = kb;
          key[b] = ka;
          if constexpr (!std::is_null_pointer_v<PosPtr>) {
            const int pa = pos[a];
            pos[a] = pos[b];
            pos[b] = pa;
          }
        }
      }
      __syncwarp();
    }
}

static inline int next_pow2_host(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}
