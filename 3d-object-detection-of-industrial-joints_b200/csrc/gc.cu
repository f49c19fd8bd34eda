// gc.cu — geometric-consistency grouping of correspondences + RANSAC pose, on the device.
//
// Replaces pcl::GeometricConsistencyGrouping<PointXYZRGBA, PointXYZRGBA>::recognize (SHOT.cpp:473-482,
// 6Dpose.cpp:529-538, SHOT_scenes.cpp:413-425): clusterCorrespondences (sort by distance, greedy
// seed-and-grow consensus sets under the pairwise distance-preservation test, sets larger than the
// threshold are taken) followed per set by CorrespondenceRejectorSampleConsensus (RANSAC on
// SampleConsensusModelRegistration, Umeyama on 3-samples, mt19937 seeded 12345).
//
// The greedy order is kept exactly.  A seed's consensus set depends on earlier seeds only through
// the `taken` flags, and only successful seeds change those; moreover a set computed against an
// older (smaller) set of flags is still exact as long as none of its members has been taken since
// (rejected candidates never influence later decisions).  So:
//   1. gc_adjacency_kernel evaluates the pairwise test once for all pairs into a C x C bitmap
//      (all SMs; this is the O(C^2) part).
//   2. gc_group_cluster_kernel (one 8-CTA thread-block cluster) takes the next 8 untaken seeds, one per
//      CTA, and grows each set speculatively against the current flags: candidates = row(seed) & ~taken,
//      the lowest candidate is admitted and its row ANDed in, and the last 64 or fewer candidates are
//      finished in registers.  Every CTA then walks the 8 results in the same order: the first seed whose
//      set touches an element committed earlier in the walk is inexact, everything before it commits,
//      and the next window restarts there.  On the benchmark scene (25 k correspondences, 3 770
//      instances) that is 678 rounds instead of 4 276 sequential seed scans.
// RANSAC runs afterwards, one CTA per instance in two size classes (32 threads up to 96 members, 128
// threads above): thread 0 draws the sample sequence (the RNG stream is inherently serial), the threads
// fit and score one sample each, thread 0 then replays the adaptive termination logic in order and
// discards the samples past the stopping point.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "linalg3.cuh"
#include "pcl_eigen33.cuh"

namespace {

// ---- sort by (distance, original position): rank by counting -----------------------------------
// A CTA ranks RANK_ITEMS correspondences: lane = item, warp = one eighth of every 256-key tile, partial counts
// merged in shared memory (32 items per CTA give ~800 CTAs for the 25 k correspondences of the target scene; one
// item per thread and 256 per CTA left two thirds of the SMs idle).
constexpr int RANK_ITEMS = 32;
constexpr int RANK_TILE = 2048;  // keys staged per barrier pair
__global__ void __launch_bounds__(256)
    gc_rank_kernel(const b200_corr *__restrict__ corrs, const int *__restrict__ d_C, int C_cap,
                   const float4 *__restrict__ model_kp, const float4 *__restrict__ scene_kp,
                   b200_corr *__restrict__ sorted, float4 *__restrict__ mp, float4 *__restrict__ sp,
                   const int *__restrict__ gate) {
  __shared__ unsigned long long tile[RANK_TILE];
  __shared__ int s_rank[RANK_ITEMS];
  if (gate && *gate == 0) return;  // the bucket sort below has done it
  const int C = min(*d_C, C_cap);
  if (blockIdx.x * RANK_ITEMS >= C) return;
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int i = blockIdx.x * RANK_ITEMS + lane;
  unsigned long long mykey = 0;
  if (i < C) mykey = ((unsigned long long)__float_as_uint(corrs[i].distance) << 32) | (unsigned)i;
  if (threadIdx.x < RANK_ITEMS) s_rank[threadIdx.x] = 0;
  int rank = 0;
  for (int base = 0; base < C; base += RANK_TILE) {
    __syncthreads();
#pragma unroll
    for (int u = 0; u < RANK_TILE / 256; ++u) {
      const int j = base + u * 256 + threadIdx.x;
      tile[u * 256 + threadIdx.x] =
          (j < C) ? (((unsigned long long)__float_as_uint(corrs[j].distance) << 32) | (unsigned)j) : ~0ull;
    }
    __syncthreads();
    const unsigned long long *mine = tile + slice * (RANK_TILE / 8);
#pragma unroll 16
    for (int t = 0; t < RANK_TILE / 8; ++t) rank += (mine[t] < mykey) ? 1 : 0;
  }
  atomicAdd(&s_rank[lane], rank);
  __syncthreads();
  if (slice == 0 && i < C) {
    const b200_corr mine = corrs[i];
    const int r = s_rank[lane];
    sorted[r] = mine;
    mp[r] = model_kp[mine.index_query];
    sp[r] = scene_kp[mine.index_match];
  }
}

// ---- the same order by buckets ------------------------------------------------------------------------
// Ranking by counting is O(C^2) (0.14 ms for the 25 k correspondences of the target scene).  The key's top 13 bits
// (sign, exponent, 4 mantissa bits of the distance) are a monotone bucket index: histogram -> one-CTA scan ->
// scatter -> rank inside the bucket (a hundred or two keys).  Four small launches; if a bucket holds more than
// SORT_BIG_BUCKET keys (many equal or nearly equal distances) a flag hands the scene to gc_rank_kernel instead —
// on the device, no host round trip.  Same keys, same total order: the output is gc_rank_kernel's bit for bit.
constexpr int SORT_BUCKETS = 8192;
constexpr int SORT_SHIFT = 19;       // bucket = sign, exponent, 4 mantissa bits of the distance (measured: 6 bits = 32 768
                                     // buckets make the one-CTA scan cost more than the rank kernel gains: 0.125 ms)
constexpr int SORT_BIG_BUCKET = 4096;

__device__ __forceinline__ unsigned long long corr_key(const b200_corr &c, int i) {
  return ((unsigned long long)__float_as_uint(c.distance) << 32) | (unsigned)i;
}

__global__ void __launch_bounds__(256)
    gc_sort_hist_kernel(const b200_corr *__restrict__ corrs, const int *__restrict__ d_C, int C_cap, int *__restrict__ hist) {
  const int C = min(*d_C, C_cap);
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < C) atomicAdd(&hist[__float_as_uint(corrs[i].distance) >> SORT_SHIFT], 1);
}

// one CTA: start[b] = number of keys in buckets before b; hist is cleared (it becomes the scatter cursor);
// *fallback = 1 when a bucket is too large for the per-key scan of gc_sort_rank_kernel
__global__ void __launch_bounds__(1024) gc_sort_scan_kernel(int *__restrict__ hist, int *__restrict__ start, int *__restrict__ fallback) {
  __shared__ int s_warp[32];
  __shared__ int s_big;
  constexpr int PER = SORT_BUCKETS / 1024;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_big = 0;
  __syncthreads();
  int sum = 0, mx = 0;
#pragma unroll 8
  for (int u = 0; u < PER; ++u) {
    const int v = hist[tid * PER + u];
    sum += v;
    mx = max(mx, v);
  }
  if (mx > SORT_BIG_BUCKET) s_big = 1;
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    s_warp[lane] = w;
  }
  __syncthreads();
  int run = incl - sum + (warp ? s_warp[warp - 1] : 0);
#pragma unroll 8
  for (int u = 0; u < PER; ++u) {
    const int v = hist[tid * PER + u];
    start[tid * PER + u] = run;
    run += v;
    hist[tid * PER + u] = 0;
  }
  if (tid == 1023) start[SORT_BUCKETS] = run;
  if (tid == 0) *fallback = s_big;
}

__global__ void __launch_bounds__(256)
    gc_sort_scatter_kernel(const b200_corr *__restrict__ corrs, const int *__restrict__ d_C, int C_cap,
                           const int *__restrict__ start, int *__restrict__ cursor, unsigned long long *__restrict__ keys,
                           const int *__restrict__ fallback) {
  if (*fallback) return;
  const int C = min(*d_C, C_cap);
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= C) return;
  const b200_corr c = corrs[i];
  const int b = (int)(__float_as_uint(c.distance) >> SORT_SHIFT);
  keys[start[b] + atomicAdd(&cursor[b], 1)] = corr_key(c, i);
}

__global__ void __launch_bounds__(256)
    gc_sort_rank_kernel(const b200_corr *__restrict__ corrs, const int *__restrict__ d_C, int C_cap,
                        const float4 *__restrict__ model_kp, const float4 *__restrict__ scene_kp,
                        const int *__restrict__ start, const unsigned long long *__restrict__ keys,
                        b200_corr *__restrict__ sorted, float4 *__restrict__ mp, float4 *__restrict__ sp,
                        const int *__restrict__ fallback) {
  if (*fallback) return;
  const int C = min(*d_C, C_cap);
  const int p = blockIdx.x * 256 + threadIdx.x;  // a position of the bucket-ordered key array: the threads of a
  if (p >= C) return;                            // warp mostly share a bucket, so they read the same keys
  const unsigned long long key = keys[p];
  const b200_corr mine = corrs[(int)(unsigned)(key & 0xffffffffull)];
  const int b = (int)((unsigned)(key >> 32) >> SORT_SHIFT);
  const int s = start[b], e = start[b + 1];
  int r = s;
  for (int j = s; j < e; ++j) r += (keys[j] < key) ? 1 : 0;
  sorted[r] = mine;
  mp[r] = model_kp[mine.index_query];
  sp[r] = scene_kp[mine.index_match];
}

// ---- pairwise consistency bitmap ------------------------------------------------------------------
// adj[i][j] = 1 iff correspondences i and j (sorted positions) pass the distance-preservation test,
// i != j.  Rows are row_words 32-bit words (a multiple of 8, so a row starts on a 32-byte sector).
// The decision is PCL's float expression; a MUFU-based estimate settles every pair that is not within
// a rigorous error band of the threshold and only the rest evaluate the IEEE square roots.
constexpr int ADJ_ROWS = 128;
constexpr int ADJ_WORDS = 32;  // words per CTA tile (1024 columns)
constexpr int ADJ_THREADS = 256;
#ifndef ADJ_UNROLL
#define ADJ_UNROLL 8  // pair tests inlined per word (measured: 4 -> 0.545 ms, 8 -> 0.521 ms once the ballot transposes were gone)
#endif
constexpr int ADJ_UNROLL_N = ADJ_UNROLL;

__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ float dist2f(const float4 &a, const float4 &b) {
  const float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z;
  float s = d0 * d0;
  s += d1 * d1;
  s += d2 * d2;
  return s;
}

// PCL's float expression itself (taken by the pairs inside the estimate's error band: out of line, the IEEE square
// roots are most of the test's code and it is inlined at every test site)
__device__ __noinline__ bool gc_fits_exact(float a, float c, double gc_size) {
  return !((double)fabsf(sqrtf(a) - sqrtf(c)) > gc_size);
}

// The grouping test with a fast path: `fits` <=> !gc_rejects.  sqrt.approx has a relative error of at
// most 2^-22, so |estimate - float expression| < 1e-6 (sa + sc); pairs outside that band around the
// threshold are decided by the estimate, the others evaluate the exact expression.
__device__ __forceinline__ bool gc_fits(const float4 &mk, const float4 &sk, const float4 &mj, const float4 &sj,
                                        float g_lo, float g_hi, double gc_size) {
  const float a = dist2f(sk, sj);
  const float c = dist2f(mk, mj);
  const float sa = sqrt_approx(a), sc = sqrt_approx(c);
  const float diff = fabsf(sa - sc);
  const float tol = 1e-6f * (sa + sc) + 1e-15f;
  if (diff > g_hi + tol) return false;
  if (diff < g_lo - tol) return true;
  return gc_fits_exact(a, c, gc_size);
}

__device__ __forceinline__ int gc_row_words(int C) { return (((C + 31) >> 5) + 127) & ~127; }

// 32 x 32 bit transpose across a warp: lane r holds row r (bit c = element (r, c)); returns, in lane c, column c
// (bit r = element (r, c)).  Five block-swap steps (blocks of 16, 8, 4, 2, 1) with one shuffle each — 32 ballots,
// each wrapped in the compiler's convergence guards, were 40 % of the kernel's code and a third of a mirrored word's
// instructions.
__device__ __forceinline__ unsigned transpose32(unsigned x, int lane) {
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const int j = 16 >> s;
    const unsigned m = (s == 0) ? 0x0000ffffu : (s == 1) ? 0x00ff00ffu : (s == 2) ? 0x0f0f0f0fu : (s == 3) ? 0x33333333u : 0x55555555u;
    const unsigned y = __shfl_xor_sync(0xffffffffu, x, j);
    const bool upper = (lane & j) == 0;             // this lane holds the upper row of the pair
    const unsigned a = upper ? x : y, b = upper ? y : x;
    const unsigned t = ((a >> j) ^ b) & m;          // upper-right block of a against lower-left block of b
    x ^= upper ? (t << j) : t;
  }
  return x;
}

__global__ void __launch_bounds__(ADJ_THREADS)
    gc_adjacency_kernel(const float4 *__restrict__ mp, const float4 *__restrict__ sp, const int *__restrict__ d_C,
                        int C_cap, double gc_size, float g_lo, float g_hi, unsigned *__restrict__ adj) {
  __shared__ float4 s_m[ADJ_WORDS * 32];
  __shared__ float4 s_s[ADJ_WORDS * 32];
  __shared__ unsigned s_t[2][4][ADJ_ROWS];  // mirror staging: [half][32-row block][column]
  const int C = min(*d_C, C_cap);
  const int row_words = gc_row_words(C);
  const int w0 = blockIdx.x * ADJ_WORDS;
  const int i0 = blockIdx.y * ADJ_ROWS;
  if (w0 >= row_words || i0 >= C) return;
  // The relation is symmetric (gc_fits is bit-for-bit symmetric in its two correspondences): a CTA evaluates only
  // the 128-column groups on or right of its 128-row block and writes the groups strictly right of it a second time
  // transposed (32 x 32 bit blocks turned by ballots), which fills the skipped groups of the rows below.
  if ((w0 + ADJ_WORDS) * 32 <= i0) return;
  const int tid = threadIdx.x;
  for (int t = tid; t < ADJ_WORDS * 32; t += ADJ_THREADS) {
    const int j = w0 * 32 + t;
    const bool in = j < C;
    s_m[t] = in ? mp[j] : make_float4(0.f, 0.f, 0.f, 0.f);
    s_s[t] = in ? sp[j] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  const int lane = tid & 31;
  const int i = i0 + (tid & (ADJ_ROWS - 1));
  const int half = tid / ADJ_ROWS, wr = (tid & (ADJ_ROWS - 1)) >> 5;  // column half of the tile, 32-row block
  const int wbase = (tid / ADJ_ROWS) * (ADJ_WORDS / 2);           // 16 words per thread
  const bool valid = i < C;
  const float4 mi = valid ? mp[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  const float4 si = valid ? sp[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  unsigned *row = adj + (size_t)(valid ? i : 0) * row_words + w0 + wbase;
#pragma unroll 1
  for (int wq = 0; wq < ADJ_WORDS / 2; wq += 4) {
    const int gw0 = w0 + wbase + wq;  // first of four words = 128 aligned columns
    if (gw0 >= row_words) break;
    const int jg = gw0 * 32;
    if (jg + 128 <= i0) continue;  // left of the row block: written by the transposed stores of the rows above
    const bool mirror = jg >= i0 + ADJ_ROWS;
    unsigned out[4];
#pragma unroll
    for (int w4 = 0; w4 < 4; ++w4) {
      const int w = wq + w4;
      unsigned bits = 0;
      const int t0 = (wbase + w) * 32;
#pragma unroll ADJ_UNROLL_N
      for (int b = 0; b < 32; ++b) {
        const bool ok = gc_fits(mi, si, s_m[t0 + b], s_s[t0 + b], g_lo, g_hi, gc_size);
        bits |= (ok ? 1u : 0u) << b;
      }
      const int gw = gw0 + w4;  // global word index
      const int j0 = gw * 32;
      if (j0 + 32 > C) bits &= (j0 >= C) ? 0u : ((1u << (C - j0)) - 1u);
      if ((i >> 5) == gw) bits &= ~(1u << (i & 31));
      if (!valid) bits = 0u;
      out[w4] = bits;
      if (mirror)  // uniform over the half CTA
        s_t[half][wr][w4 * 32 + lane] = transpose32(bits, lane);  // column j0 + lane, rows of this warp
    }
    if (mirror) {
      // the four warps of the half hold the same 128 columns for four consecutive 32-row blocks: one 16-byte
      // store per column instead of four scattered words
      asm volatile("bar.sync %0, %1;" ::"r"(1 + half), "r"(ADJ_ROWS) : "memory");
      const int col = tid & (ADJ_ROWS - 1);
      if (jg + col < C)
        *reinterpret_cast<uint4 *>(adj + (size_t)(jg + col) * row_words + (i0 >> 5)) =
            make_uint4(s_t[half][0][col], s_t[half][1][col], s_t[half][2][col], s_t[half][3][col]);
      asm volatile("bar.sync %0, %1;" ::"r"(1 + half), "r"(ADJ_ROWS) : "memory");
    }
    if (valid) *reinterpret_cast<uint4 *>(row + wq) = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// ---- greedy grouping on a thread-block cluster ----------------------------------------------------
// The whole greedy growth of a seed runs on bitmaps: candidates = row(seed) & ~taken; the lowest
// candidate j is admitted (it fits every member so far by construction) and candidates &= row(j);
// repeat until at most G_LIST candidates are left, which are listed in ascending position and
// finished in registers.  Rows are padded to a multiple of 128 words.
// A round evaluates the next GCL untaken seeds speculatively, one per CTA of the cluster: CTA r
// evaluates window seed r with all of its 128 threads (thread t handles the 16-byte pieces t,
// t + 128, ... of a bitmap row).  Every CTA keeps its own copy of the `taken` bitmap and of the
// running totals; after the evaluation each CTA writes its result (size + members) into every CTA's
// shared memory through DSMEM, one cluster barrier later all CTAs walk the window identically, so the
// copies never diverge and one barrier per round suffices (results are double-buffered by round parity).
constexpr int GCL = 8;            // cluster size = seeds per round
constexpr int GCL_THREADS = 128;
constexpr int G_MC = 64;          // member indices kept in shared memory per seed
constexpr int G_LIST = 64;        // candidates finished in registers

struct GroupArgs {
  const unsigned *adj;
  const float4 *mp;
  const float4 *sp;
  int *overflow;      // [GCL][C_cap] member indices past G_MC
  int *members;       // [C_cap] committed member lists, concatenated
  int *inst_offsets;  // [max_inst + 1]
  int *n_inst_out;
  long long *dbg;     // nullable (B200_GC_TIMING builds): per CTA [window, first row, admissions, list,
                      // list + greedy, cluster sync, commit] cycles and the round count
};

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// lowest set position of a 128-bit group that starts at position base, or INT_MAX
__device__ __forceinline__ int first_bit128(const uint4 &w, int base) {
  if (w.x) return base + __ffs(w.x) - 1;
  if (w.y) return base + 32 + __ffs(w.y) - 1;
  if (w.z) return base + 64 + __ffs(w.z) - 1;
  if (w.w) return base + 96 + __ffs(w.w) - 1;
  return 0x7fffffff;
}

__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned cluster_cta_rank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// address of the same shared-memory variable in CTA `rank` of the cluster
__device__ __forceinline__ unsigned dsmem_addr(const void *p, unsigned rank) {
  unsigned local = (unsigned)__cvta_generic_to_shared(p), remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(rank));
  return remote;
}
__device__ __forceinline__ void dsmem_store(unsigned addr, int v) {
  asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

__global__ void __cluster_dims__(GCL, 1, 1) __launch_bounds__(GCL_THREADS, 1)
    gc_group_cluster_kernel(GroupArgs ga, const int *__restrict__ d_C, int C_cap, double gc_size, float g_lo, float g_hi,
                            int gc_threshold, int max_inst) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  __shared__ int s_res[2][GCL][1 + G_MC];  // published results by round parity: [0] size, then members
  __shared__ int s_seed[GCL];
  __shared__ int s_nwin;
  __shared__ int s_list[64];
  __shared__ int s_redf[4], s_redc[4];
  __shared__ int s_mine[G_MC];
  __shared__ int s_state[4];  // cur, n_inst, total after a sequential commit walk
  __shared__ float4 s_newm, s_news;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rank = (int)cluster_cta_rank();
  const int C = min(*d_C, C_cap);
  const int row_words = gc_row_words(C);
  const int n4 = row_words >> 2;
  const int wpt = row_words / GCL_THREADS;
  uint4 *s_taken4 = reinterpret_cast<uint4 *>(s_raw);
  unsigned *s_taken = reinterpret_cast<unsigned *>(s_raw);
  uint4 *my_cb4 = s_taken4 + n4;
  const unsigned *my_cb = reinterpret_cast<const unsigned *>(my_cb4);
  int *my_over = ga.overflow + (size_t)rank * C_cap;

  for (int w = tid; w < row_words; w += GCL_THREADS) {
    const int j0 = w * 32;
    s_taken[w] = (j0 + 32 <= C) ? 0u : ((j0 >= C) ? ~0u : ~((1u << (C - j0)) - 1u));  // padding counts as taken
  }
  if (rank == 0 && tid == 0) ga.inst_offsets[0] = 0;
  int cur = 0, n_inst = 0, total = 0;  // identical in every thread of every CTA
  __syncthreads();
  cluster_sync_all();  // every CTA's shared memory exists before the first remote store

#ifdef B200_GC_TIMING
  long long tc_[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define CT(v) const long long v = clock64()
#define CA(i, e) tc_[i] += (e)
#else
#define CT(v)
#define CA(i, e)
#endif
  for (int round = 0;; ++round) {
    const int par = round & 1;
    CT(q0);
    // ---- window: the next GCL untaken positions at or after cur (warp 0 of every CTA, same result) ----
    if (warp == 0) {
      int n = 0;
      for (int wb = cur >> 5; wb < row_words && n < GCL; wb += 32) {
        const int wi = wb + lane;
        unsigned bits = (wi < row_words) ? ~s_taken[wi] : 0u;
        if (wi == (cur >> 5)) bits &= ~((1u << (cur & 31)) - 1u);
        const int cnt = __popc(bits);
        const int incl = warp_incl_scan(cnt, lane);
        int o = n + incl - cnt;
        while (bits && o < GCL) {
          const int b = __ffs(bits) - 1;
          bits &= bits - 1;
          s_seed[o++] = wi * 32 + b;
        }
        n += __shfl_sync(0xffffffffu, incl, 31);
      }
      if (lane == 0) s_nwin = min(n, GCL);
    }
    __syncthreads();
    const int nwin = s_nwin;
    if (nwin == 0) break;
    CT(q1);
    CA(0, q1 - q0);

    // ---- evaluate seed `rank` ----
    int size = 0;
    if (rank < nwin) {
      const int seed = s_seed[rank];
      size = 1;
      if (tid == 0) s_mine[0] = seed;
      int first = 0x7fffffff, cnt = 0;
      {
        const uint4 *row4 = reinterpret_cast<const uint4 *>(ga.adj + (size_t)seed * row_words);
        for (int u0 = tid; u0 < n4; u0 += 4 * GCL_THREADS) {  // loads of a block are issued before the first use
          uint4 x[4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (u0 + i * GCL_THREADS < n4) x[i] = __ldg(row4 + u0 + i * GCL_THREADS);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int u = u0 + i * GCL_THREADS;
            if (u < n4) {
              const uint4 t = s_taken4[u];
              const uint4 w = make_uint4(x[i].x & ~t.x, x[i].y & ~t.y, x[i].z & ~t.z, x[i].w & ~t.w);
              my_cb4[u] = w;
              if (w.x | w.y | w.z | w.w) {
                cnt += __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
                if (first == 0x7fffffff) first = first_bit128(w, u * 128);
              }
            }
          }
        }
      }
      first = __reduce_min_sync(0xffffffffu, first);
      cnt = __reduce_add_sync(0xffffffffu, cnt);
      if (lane == 0) {
        s_redf[warp] = first;
        s_redc[warp] = cnt;
      }
      __syncthreads();
      first = min(min(s_redf[0], s_redf[1]), min(s_redf[2], s_redf[3]));
      int n_cand = s_redc[0] + s_redc[1] + s_redc[2] + s_redc[3];
      CT(q2);
      CA(1, q2 - q1);
      // bitmap admissions while many candidates remain (each costs one row read)
      while (n_cand > G_LIST) {
        __syncthreads();  // everybody has read s_red* of the previous pass
        const int j = first;
        if (tid == 0) {
          if (size < G_MC)
            s_mine[size] = j;
          else
            my_over[size] = j;
        }
        ++size;
        const uint4 *rowj4 = reinterpret_cast<const uint4 *>(ga.adj + (size_t)j * row_words);
        first = 0x7fffffff;
        cnt = 0;
        const int ufirst = j >> 7;  // pieces before j's hold no candidates any more
        for (int u0 = (ufirst & ~(GCL_THREADS - 1)) + tid; u0 < n4; u0 += 4 * GCL_THREADS) {
          uint4 y[4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (u0 + i * GCL_THREADS < n4) y[i] = __ldg(rowj4 + u0 + i * GCL_THREADS);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int u = u0 + i * GCL_THREADS;
            if (u < n4) {
              uint4 w = my_cb4[u];
              if (w.x | w.y | w.z | w.w) {
                w.x &= y[i].x, w.y &= y[i].y, w.z &= y[i].z, w.w &= y[i].w;
                my_cb4[u] = w;
                cnt += __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
                if (first == 0x7fffffff) first = first_bit128(w, u * 128);
              }
            }
          }
        }
        first = __reduce_min_sync(0xffffffffu, first);
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0) {
          s_redf[warp] = first;
          s_redc[warp] = cnt;
        }
        __syncthreads();
        first = min(min(s_redf[0], s_redf[1]), min(s_redf[2], s_redf[3]));
        n_cand = s_redc[0] + s_redc[1] + s_redc[2] + s_redc[3];
      }
      CT(q3);
      CA(2, q3 - q2);
      if (n_cand > 0) {
        // at most 64 candidates left: list them in ascending position (thread t expands words
        // [t * wpt, (t + 1) * wpt) of the bitmap), fetch their points once and let warp 0 finish the
        // greedy growth in registers
        __syncthreads();
        int c = 0;
        const int w_lo = tid * wpt, w_min = first >> 5;
        for (int w = max(w_lo, w_min); w < w_lo + wpt; ++w) c += __popc(my_cb[w]);
        const int incl = warp_incl_scan(c, lane);
        if (lane == 31) s_redc[warp] = incl;
        __syncthreads();
        if (c) {
          int o = incl - c;
          for (int k = 0; k < warp; ++k) o += s_redc[k];
          for (int w = max(w_lo, w_min); w < w_lo + wpt; ++w) {
            unsigned bits = my_cb[w];
            while (bits) {
              s_list[o++] = w * 32 + __ffs(bits) - 1;
              bits &= bits - 1;
            }
          }
        }
        __syncthreads();
        CT(q4);
        CA(3, q4 - q3);
        if (warp == 0) {
          int j[2];
          float4 mj[2], sj[2];
          unsigned alive = 0;
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int idx = u * 32 + lane;
            if (idx < n_cand) {
              j[u] = s_list[idx];
              mj[u] = ga.mp[j[u]];
              sj[u] = ga.sp[j[u]];
              alive |= 1u << u;
            }
          }
          while (true) {
            unsigned bal = __ballot_sync(0xffffffffu, alive & 1u);
            int usel = 0;
            if (!bal) {
              bal = __ballot_sync(0xffffffffu, alive & 2u);
              usel = 1;
              if (!bal) break;
            }
            const int owner = __ffs(bal) - 1;
            // the admitted candidate's index and points go to every lane by shuffle
            const float4 am = usel ? mj[1] : mj[0], as = usel ? sj[1] : sj[0];
            const int jj = __shfl_sync(0xffffffffu, usel ? j[1] : j[0], owner);
            float4 mk, sk;
            mk.x = __shfl_sync(0xffffffffu, am.x, owner);
            mk.y = __shfl_sync(0xffffffffu, am.y, owner);
            mk.z = __shfl_sync(0xffffffffu, am.z, owner);
            sk.x = __shfl_sync(0xffffffffu, as.x, owner);
            sk.y = __shfl_sync(0xffffffffu, as.y, owner);
            sk.z = __shfl_sync(0xffffffffu, as.z, owner);
            mk.w = sk.w = 0.f;
            if (lane == owner) alive &= ~(1u << usel);
            if (lane == 0) {
              if (size < G_MC)
                s_mine[size] = jj;
              else
                my_over[size] = jj;
            }
            ++size;
#pragma unroll
            for (int u = 0; u < 2; ++u)
              if (((alive >> u) & 1u) && !gc_fits(mk, sk, mj[u], sj[u], g_lo, g_hi, gc_size)) alive &= ~(1u << u);
          }
          if (lane == 0) s_redc[0] = size;
        }
        __syncthreads();
        size = s_redc[0];
      }
      CT(q5);
      CA(4, q5 - q3);
      // ---- publish (size, members) into every CTA of the cluster ----
      const int msz = min(size, G_MC);
      for (int idx = tid; idx < GCL * (1 + msz); idx += GCL_THREADS) {
        const int t = idx / (1 + msz), k = idx % (1 + msz);
        dsmem_store(dsmem_addr(&s_res[par][rank][k], (unsigned)t), k == 0 ? size : s_mine[k - 1]);
      }
    }
    CT(q6);
    cluster_sync_all();
    CT(q7);
    CA(5, q7 - q6);

    // ---- commit (warp 0 of every CTA, identically): walk the window in order with the members held in
    // registers (lane l holds members l and l + 32 of every seed); a seed whose set touches an element
    // taken earlier in the walk is the first inexact one, everything before it commits.  Sets beyond the
    // shared-memory list are read from the owners' overflow arrays. ----
    if (warp == 0) {
      int szs = (lane < nwin) ? s_res[par][lane][0] : 0;
      int m0[GCL], m1[GCL];
#pragma unroll
      for (int r = 0; r < GCL; ++r) {
        const int sz = __shfl_sync(0xffffffffu, szs, r);
        m0[r] = (r < nwin && lane < sz) ? s_res[par][r][1 + lane] : -1;
        m1[r] = (r < nwin && lane + 32 < sz && lane + 32 < G_MC) ? s_res[par][r][1 + lane + 32] : -1;
      }
      int pstar = nwin;
#pragma unroll
      for (int r = 0; r < GCL; ++r) {
        if (r < nwin && pstar == nwin) {
          const int sz = __shfl_sync(0xffffffffu, szs, r);
          bool hit = (m0[r] >= 0 && ((s_taken[m0[r] >> 5] >> (m0[r] & 31)) & 1u)) ||
                     (m1[r] >= 0 && ((s_taken[m1[r] >> 5] >> (m1[r] & 31)) & 1u));
          for (int kk = G_MC + lane; kk < sz; kk += 32) {  // oversize set: the rest from global memory
            const int m = __ldcg(ga.overflow + (size_t)r * C_cap + kk);
            hit = hit || ((s_taken[m >> 5] >> (m & 31)) & 1u);
          }
          if (__any_sync(0xffffffffu, hit)) {
            pstar = r;
          } else if (sz > gc_threshold) {
            if (m0[r] >= 0) atomicOr(&s_taken[m0[r] >> 5], 1u << (m0[r] & 31));
            if (m1[r] >= 0) atomicOr(&s_taken[m1[r] >> 5], 1u << (m1[r] & 31));
            if (r == rank) {  // the owner writes the instance out
              if (m0[r] >= 0) ga.members[total + lane] = m0[r];
              if (m1[r] >= 0) ga.members[total + lane + 32] = m1[r];
              if (lane == 0 && n_inst < max_inst) ga.inst_offsets[n_inst + 1] = total + sz;
            }
            for (int kk = G_MC + lane; kk < sz; kk += 32) {
              const int m = __ldcg(ga.overflow + (size_t)r * C_cap + kk);
              atomicOr(&s_taken[m >> 5], 1u << (m & 31));
              if (r == rank) ga.members[total + kk] = m;
            }
            total += sz;
            ++n_inst;
            __syncwarp();
          }
        }
      }
      if (lane == 0) {
        s_state[0] = (pstar < nwin) ? s_seed[pstar] : s_seed[nwin - 1] + 1;
        s_state[1] = n_inst;
        s_state[2] = total;
      }
    }
    __syncthreads();
    cur = s_state[0];
    n_inst = s_state[1];
    total = s_state[2];
    CA(6, clock64() - q7);
    CA(7, 1);
  }
#ifdef B200_GC_TIMING
  if (ga.dbg && tid == 0)
    for (int i = 0; i < 8; ++i) ga.dbg[rank * 8 + i] = tc_[i];
#endif
  if (rank == 0 && tid == 0) *ga.n_inst_out = n_inst;
}

// ---- RANSAC pose per instance -------------------------------------------------------------------
// boost::mt19937 seeded 12345 (RandomSampleConsensus, non-random mode).  Every instance restarts the
// same stream, so the generator state after seeding and the first twist is computed once on the host
// and copied into shared memory per warp; later twists are done by the whole warp.
void mt19937_twisted_state(unsigned seed, unsigned out[624]) {
  out[0] = seed;
  for (int i = 1; i < 624; ++i) out[i] = 1812433253u * (out[i - 1] ^ (out[i - 1] >> 30)) + (unsigned)i;
  for (int i = 0; i < 624; ++i) {
    const unsigned y = (out[i] & 0x80000000u) | (out[(i + 1) % 624] & 0x7fffffffu);
    out[i] = out[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
  }
}

__device__ __forceinline__ unsigned mt_twist_word(unsigned a, unsigned b, unsigned c) {
  const unsigned y = (a & 0x80000000u) | (b & 0x7fffffffu);
  return c ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

// In-place regeneration of the 624-word state by one warp.  Word i needs s[i], s[i+1] (old) and
// s[(i+397) % 624]: old for i < 227, already regenerated for i >= 227 — so ranges of at most 227
// words are independent.
__device__ void mt_twist_warp(unsigned *s, int lane) {
  // every lane runs the same trip counts, so the __syncwarp calls are convergent; a step reads its
  // inputs before the barrier and writes after it (s[i + 1] belongs to the neighbouring lane)
  for (int base = 0; base < 227; base += 32) {
    const int i = base + lane;
    const bool on = i < 227;
    unsigned v = 0;
    if (on) v = mt_twist_word(s[i], s[i + 1], s[i + 397]);
    __syncwarp();
    if (on) s[i] = v;
    __syncwarp();
  }
  for (int base = 227; base < 623; base += 32) {  // s[i - 227] was regenerated at least 195 words earlier
    const int i = base + lane;
    const bool on = i < 623;
    unsigned v = 0;
    if (on) v = mt_twist_word(s[i], s[i + 1], s[i - 227]);
    __syncwarp();
    if (on) s[i] = v;
    __syncwarp();
  }
  if (lane == 0) s[623] = mt_twist_word(s[623], s[0], s[396]);
  __syncwarp();
}

__device__ __forceinline__ unsigned mt_temper(unsigned y) {
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= y >> 18;
  return y;
}

struct RansacBuffers {
  const b200_corr *sorted;
  const float4 *mp;
  const float4 *sp;
  const int *members;
  const int *inst_offsets;
  const int *n_inst;
  const unsigned *mt_init;  // [624] twisted state for seed 12345
  int *shuffled;   // [C_cap]
  int *last_pos;   // [C_cap]
  int *flags;      // [C_cap]
  float *T_out;    // [max_inst][16]
  int *inst_counts;
  b200_corr *inst_corrs;
};

// One CTA per instance, in two size classes (the instance sizes are only known on the device, so both kernels are
// launched over all instances and a CTA returns at once when the instance is not of its class): instances of up to
// RS_ONE_WARP_MAX members by ONE warp — the kernel waits most of the time for the thread that draws the samples, and
// with one-warp CTAs four times as many instances share an SM (0.55 -> 0.44 ms for the 3 770 small instances of the
// target scene) —, larger ones by four warps (the inlier counts of a sample loop over all members).
constexpr int RS_ONE_WARP_MAX = 96;
constexpr int RS_EXHAUST_AFTER = 165;   // samples (1 + 4 + 32 + 128) before the exhaustive bound is computed
constexpr int RS_EXHAUST_MAX_N = 18;    // ... for instances of at most this size (<= 4896 ordered samples)
constexpr int RS_SMALL = 128;          // instances up to this size keep shuffle array / pair matrix in shared memory

// squared residual of correspondence (s → g) under the row-major 4x4 float transform T
// The float64 fit of a 3-point sample (Jacobi eigen-solve with double divisions and square roots: ~20 KB of SASS
// per inlined copy).  Out of line: the kernel was 139 KB of code against a 32 KB instruction cache.
__device__ __noinline__ void umeyama3_sample(const double *src, const double *dst, float *T) {
  double Td[16];
  umeyama3(src, dst, 3, Td);
#pragma unroll
  for (int i = 0; i < 16; ++i) T[i] = (float)Td[i];
}

__device__ __forceinline__ float residual2(const float *T, const float4 &s, const float4 &g) {
  float e[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    float v = T[r * 4 + 0] * s.x;
    v += T[r * 4 + 1] * s.y;
    v += T[r * 4 + 2] * s.z;
    v += T[r * 4 + 3];
    e[r] = v - (r == 0 ? g.x : (r == 1 ? g.y : g.z));
  }
  float d = e[0] * e[0];
  d += e[1] * e[1];
  d += e[2] * e[2];
  return d;
}

__device__ __forceinline__ float sqdiff3(const float4 &u, const float4 &v) {
  const float dx = u.x - v.x, dy = u.y - v.y, dz = u.z - v.z;
  return dx * dx + dy * dy + dz * dz;
}

// r % d for 32-bit operands through a precomputed 64-bit reciprocal (Lemire's fastmod): exact.
__device__ __forceinline__ unsigned fastmod_u32(unsigned r, unsigned long long magic, unsigned d) {
  return (unsigned)__umul64hi(magic * r, d);
}

// One CTA per instance.  The sample sequence is inherently serial (one mt19937 stream, a partial
// Fisher-Yates shuffle whose state carries over between draws), so thread 0 draws; everything that
// does not depend on the shuffle state is taken out of that loop: the swap partners of a whole
// 624-word generator block are computed by all threads at once, isSampleGood is a table lookup,
// positions 0..2 of the shuffle array live in registers.  Models (double-precision Umeyama) are
// fitted and scored one sample per thread, in batches of 1, 4, 32, 128, 128, ...; thread 0 then
// replays the adaptive termination rule in order and discards the samples past the stopping point.
template <int RS_THREADS>
__global__ void __launch_bounds__(RS_THREADS, (RS_THREADS == 32) ? 20 : 5)
    gc_ransac_kernel(RansacBuffers rb, int max_inst, int corr_cap, double threshold, int max_iterations) {
  constexpr int RS_BATCH = RS_THREADS;  // samples fitted per batch (one per thread)
  __shared__ unsigned s_mt[624];
  __shared__ unsigned short s_jx[624];  // swap partner of draw t (valid when n <= 65536)
  __shared__ float s_Tb[RS_BATCH][17];  // padded rows: one sample per thread
  __shared__ int s_sel[RS_BATCH][3];
  __shared__ int s_cnt[RS_BATCH];
  __shared__ float s_bestT[16];
  __shared__ float s_acc[9];
  __shared__ int s_shuf[RS_SMALL];
  __shared__ unsigned s_pg[RS_SMALL][RS_SMALL / 32];  // pair (p, q) far enough apart for isSampleGood
  __shared__ int s_ctrl[8];  // 0 nb, 1 draw_failed, 2 need_twist, 3 stop, 4 any_good, 5 have_best, 6 cmax, 7 iterations
  __shared__ int s_warp_cnt[RS_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_inst = min(*rb.n_inst, max_inst);
  const int b = blockIdx.x;
  if (b >= n_inst) return;
  const int off = rb.inst_offsets[b];
  const int n = rb.inst_offsets[b + 1] - off;
  if ((n <= RS_ONE_WARP_MAX) != (RS_THREADS == 32)) return;  // the other size class
  const int *mem = rb.members + off;
  const bool small = n <= RS_SMALL;
  int *shuffled = small ? s_shuf : rb.shuffled + off;  // drawn from by thread 0 only
  int *last_pos = rb.last_pos + off;
  int *flags = rb.flags + off;

  for (int i = tid; i < 624; i += RS_THREADS) s_mt[i] = rb.mt_init[i];
  if (tid < 8) s_ctrl[tid] = (tid == 6) ? -1 : 0;  // [6]: best count over ALL admissible ordered samples, once known
  // index maps keyed by the model index: the last correspondence with a given index_query wins
  // (std::map in computeOriginalIndexMapping, unordered_map index_to_correspondence)
  for (int t = tid; t < n; t += RS_THREADS) {
    const int q = rb.sorted[mem[t]].index_query;
    int last = t;
    for (int u = t + 1; u < n; ++u)
      if (rb.sorted[mem[u]].index_query == q) last = u;
    last_pos[t] = last;
    shuffled[t] = t;
  }
  // computeSampleDistanceThreshold: float32 single-pass covariance of the source (model) points in
  // list order, one thread per accumulator
  if (tid < 9) {
    float acc = 0.0f;
    for (int t = 0; t < n; ++t) {
      const float4 v = rb.mp[mem[t]];
      float a, c;
      switch (tid) {
        case 0: a = v.x, c = v.x; break;
        case 1: a = v.x, c = v.y; break;
        case 2: a = v.x, c = v.z; break;
        case 3: a = v.y, c = v.y; break;
        case 4: a = v.y, c = v.z; break;
        case 5: a = v.z, c = v.z; break;
        case 6: a = v.x, c = 1.0f; break;
        case 7: a = v.y, c = 1.0f; break;
        default: a = v.z, c = 1.0f; break;
      }
      acc += (tid < 6) ? a * c : a;
    }
    s_acc[tid] = acc / (float)n;
  }
  __syncthreads();

  double sample_dist_thresh;
  {
    const float *a = s_acc;  // every thread evaluates the same scalar expression
    float cov[9];
    cov[0] = a[0] - a[6] * a[6];
    cov[1] = a[1] - a[6] * a[7];
    cov[2] = a[2] - a[6] * a[8];
    cov[4] = a[3] - a[7] * a[7];
    cov[5] = a[4] - a[7] * a[8];
    cov[8] = a[5] - a[8] * a[8];
    cov[3] = cov[1];
    cov[6] = cov[2];
    cov[7] = cov[5];
    float ev[3];
    eigen33_values(cov, ev);
    sample_dist_thresh = ((double)(sqrtf(ev[0]) + sqrtf(ev[1]) + sqrtf(ev[2]))) / 3.0;
    sample_dist_thresh *= sample_dist_thresh;
  }

  const double thresh2 = threshold * threshold;
  // isSampleGood needs three members whose pairwise squared (model) distances all exceed the
  // threshold.  For small instances the pair predicate is tabulated once; when no good triple
  // exists at all (typical: several scene points matched to one model point) every one of
  // getSamples' 1000 redraws fails and RANSAC ends without a model whatever the random stream is —
  // detected here instead of replaying 3000 draws on one thread.
  if (small && n >= 3) {
    const int nw = (n + 31) >> 5;
    for (int e = tid; e < n * nw; e += RS_THREADS) {
      const int p = e / nw, w = e % nw;
      const float4 a = rb.mp[mem[p]];
      unsigned bits = 0;
      for (int q = w * 32; q < min(n, w * 32 + 32); ++q)
        if (q != p && (double)sqdiff3(rb.mp[mem[q]], a) > sample_dist_thresh) bits |= 1u << (q & 31);
      s_pg[p][w] = bits;  // symmetric bit for bit: the coordinate differences only change sign
    }
    __syncthreads();
    int any_good = 0;
    for (int pq = tid; pq < n * n && !any_good; pq += RS_THREADS) {
      const int p = pq / n, q = pq % n;
      if (q <= p || !((s_pg[p][q >> 5] >> (q & 31)) & 1u)) continue;
      for (int w = 0; w < nw; ++w)
        if (s_pg[p][w] & s_pg[q][w]) any_good = 1;
    }
    if (any_good) s_ctrl[4] = 1;
    __syncthreads();
    if (tid == 0 && !s_ctrl[4]) s_ctrl[3] = 1;  // "no samples could be selected"
  }
  unsigned long long magic[3] = {0, 0, 0};
  if (n >= 3)
    for (int i = 0; i < 3; ++i) magic[i] = 0xFFFFFFFFFFFFFFFFull / (unsigned)(n - i) + 1ull;
  const bool use_jx = n >= 3 && n <= 65536;
  auto fill_jx = [&]() {  // swap partners for the 208 redraws of the current generator block
    if (use_jx)
      for (int t = tid; t < 624; t += RS_THREADS) {
        const int i = t % 3;
        s_jx[t] = (unsigned short)(i + (int)fastmod_u32(mt_temper(s_mt[t]) >> 1, magic[i], (unsigned)(n - i)));
      }
  };
  fill_jx();
  __syncthreads();

  // thread-0 state
  int mt_idx = 0;
  int iterations = 0, n_best = -2147483647;
  double k = 1.0;
  const unsigned skipped = 0;  // computeModelCoefficients cannot fail for a 3-sample
  const unsigned max_skip = (unsigned)max_iterations * 10u;
  const double log_probability = log(1.0 - 0.99);
  const double one_over_indices = 1.0 / (double)n;
  int sh0 = 0, sh1 = 1, sh2 = 2;  // shuffled[0..2]
  int attempts = 0;               // redraws of the sample under construction (survives a twist)
  int nb_local = 0;

  int batch_cap = 1;
  while (true) {
    // ---- draw phase ----
    if (tid == 0) {
      nb_local = 0;
      s_ctrl[1] = 0;
      attempts = 0;
    }
    while (true) {
      if (tid == 0) {
        s_ctrl[2] = 0;
        const bool active = !s_ctrl[3] && (double)iterations < k && skipped < max_skip && n >= 3;
        while (active && nb_local < batch_cap && !s_ctrl[1]) {
          bool good = false;
          while (!good && attempts < 1000 && mt_idx < 624) {  // SampleConsensusModel::getSamples
            int j0, j1, j2;
            if (use_jx) {
              j0 = s_jx[mt_idx], j1 = s_jx[mt_idx + 1], j2 = s_jx[mt_idx + 2];
            } else {
              j0 = (int)((mt_temper(s_mt[mt_idx]) >> 1) % (unsigned)n);
              j1 = 1 + (int)((mt_temper(s_mt[mt_idx + 1]) >> 1) % (unsigned)(n - 1));
              j2 = 2 + (int)((mt_temper(s_mt[mt_idx + 2]) >> 1) % (unsigned)(n - 2));
            }
            mt_idx += 3;
            // drawIndexSample: swap(shuffled[i], shuffled[i + r % (n - i)]) for i = 0, 1, 2
            int t;
            if (j0 == 1) { t = sh0, sh0 = sh1, sh1 = t; }
            else if (j0 == 2) { t = sh0, sh0 = sh2, sh2 = t; }
            else if (j0 > 2) { t = shuffled[j0], shuffled[j0] = sh0, sh0 = t; }
            if (j1 == 2) { t = sh1, sh1 = sh2, sh2 = t; }
            else if (j1 > 2) { t = shuffled[j1], shuffled[j1] = sh1, sh1 = t; }
            if (j2 > 2) { t = shuffled[j2], shuffled[j2] = sh2, sh2 = t; }
            if (small) {
              good = ((s_pg[sh0][sh1 >> 5] >> (sh1 & 31)) & (s_pg[sh0][sh2 >> 5] >> (sh2 & 31)) &
                      (s_pg[sh1][sh2 >> 5] >> (sh2 & 31)) & 1u) != 0;
            } else {
              const float4 p0 = rb.mp[mem[sh0]], p1 = rb.mp[mem[sh1]], p2 = rb.mp[mem[sh2]];
              good = (double)sqdiff3(p1, p0) > sample_dist_thresh && (double)sqdiff3(p2, p0) > sample_dist_thresh &&
                     (double)sqdiff3(p2, p1) > sample_dist_thresh;  // isSampleGood
            }
            ++attempts;
          }
          if (good) {
            s_sel[nb_local][0] = sh0;
            s_sel[nb_local][1] = sh1;
            s_sel[nb_local][2] = sh2;
            ++nb_local;
            attempts = 0;
          } else if (attempts >= 1000) {
            s_ctrl[1] = 1;  // "No samples could be selected": the loop ends when it gets here
          } else {
            s_ctrl[2] = 1;  // generator block used up (624 = 3 x 208: falls between redraws)
            break;
          }
        }
        s_ctrl[0] = nb_local;
      }
      __syncthreads();
      if (!s_ctrl[2]) break;
      if (warp == 0) mt_twist_warp(s_mt, lane);
      __syncthreads();
      fill_jx();
      if (tid == 0) mt_idx = 0;
      __syncthreads();
    }
    const int nb = s_ctrl[0];
    if (nb == 0) break;
    // ---- thread t: model from sample t (computeModelCoefficients), then countWithinDistance ----
    if (tid < nb) {
      double src[9], dst[9];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const int t = s_sel[tid][i];
        const float4 s = rb.mp[mem[t]];
        const float4 g = rb.sp[mem[last_pos[t]]];
        src[i * 3 + 0] = s.x;
        src[i * 3 + 1] = s.y;
        src[i * 3 + 2] = s.z;
        dst[i * 3 + 0] = g.x;
        dst[i * 3 + 1] = g.y;
        dst[i * 3 + 2] = g.z;
      }
      umeyama3_sample(src, dst, s_Tb[tid]);
    }
    __syncthreads();
    if (nb >= 32 && n <= 256) {
      if (tid < nb) {
        int cnt = 0;
        for (int t = 0; t < n; ++t)
          cnt += ((double)residual2(s_Tb[tid], rb.mp[mem[t]], rb.sp[mem[t]]) < thresh2) ? 1 : 0;
        s_cnt[tid] = cnt;
      }
    } else {
      for (int sidx = warp; sidx < nb; sidx += RS_THREADS / 32) {
        int cnt = 0;
        for (int t = lane; t < n; t += 32)
          cnt += ((double)residual2(s_Tb[sidx], rb.mp[mem[t]], rb.sp[mem[t]]) < thresh2) ? 1 : 0;
        cnt = warp_sum(cnt);
        if (lane == 0) s_cnt[sidx] = cnt;
      }
    }
    __syncthreads();
    // ---- thread 0: replay the sequential loop over the batch ----
    if (tid == 0) {
      bool stop = false;
      for (int i = 0; i < nb; ++i) {
        if (i > 0 && !((double)iterations < k && skipped < max_skip)) {
          stop = true;
          break;
        }
        const int c = s_cnt[i];
        if (c > n_best) {
          n_best = c;
          s_ctrl[5] = 1;
          for (int e = 0; e < 16; ++e) s_bestT[e] = s_Tb[i][e];
          const double w = (double)n_best * one_over_indices;
          double p_no_outliers = 1.0 - pow(w, 3.0);
          p_no_outliers = fmax(2.220446049250313e-16, p_no_outliers);
          p_no_outliers = fmin(1.0 - 2.220446049250313e-16, p_no_outliers);
          k = log_probability / log(p_no_outliers);
        }
        ++iterations;
        if (iterations > max_iterations) {
          stop = true;  // "RANSAC reached the maximum number of trials"
          break;
        }
        if (s_ctrl[6] >= 0 && n_best >= s_ctrl[6]) {
          stop = true;  // no later sample can replace the best model (see below): the remaining iterations are idle
          break;
        }
      }
      if (s_ctrl[1] || stop) s_ctrl[3] = 1;
      s_ctrl[7] = iterations;
    }
    __syncthreads();
    // A small instance that is still iterating after RS_EXHAUST_AFTER samples (typically one whose
    // models fit few of its members, so the adaptive bound stays near the 10 000-iteration limit):
    // evaluate every admissible ORDERED sample once, with the same arithmetic, to learn the largest
    // inlier count any sample can reach.  A later sample replaces the best model only with a strictly
    // larger count, so once n_best equals that maximum the outcome is final and the (serial) drawing of
    // the remaining samples is skipped.  Exact: the best model is the one the full loop would keep.
    if (s_ctrl[6] < 0 && !s_ctrl[3] && small && n <= RS_EXHAUST_MAX_N && s_ctrl[7] >= RS_EXHAUST_AFTER) {
      __syncthreads();
      if (tid == 0) s_ctrl[6] = 0;
      __syncthreads();
      const int n_ord = n * (n - 1) * (n - 2);
      for (int e = tid; e < n_ord; e += RS_THREADS) {
        const int t0 = e / ((n - 1) * (n - 2));
        const int rem = e % ((n - 1) * (n - 2));
        int t1 = rem / (n - 2), t2 = rem % (n - 2);
        t1 += (t1 >= t0) ? 1 : 0;                       // skip t0
        const int lo = min(t0, t1), hi = max(t0, t1);  // skip both
        t2 += (t2 >= lo) ? 1 : 0;
        t2 += (t2 >= hi) ? 1 : 0;
        const bool good = ((s_pg[t0][t1 >> 5] >> (t1 & 31)) & (s_pg[t0][t2 >> 5] >> (t2 & 31)) &
                           (s_pg[t1][t2 >> 5] >> (t2 & 31)) & 1u) != 0;
        if (!good) continue;
        const int sel[3] = {t0, t1, t2};
        double src[9], dst[9];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int t = sel[i];
          const float4 sv = rb.mp[mem[t]];
          const float4 gv = rb.sp[mem[last_pos[t]]];
          src[i * 3 + 0] = sv.x, src[i * 3 + 1] = sv.y, src[i * 3 + 2] = sv.z;
          dst[i * 3 + 0] = gv.x, dst[i * 3 + 1] = gv.y, dst[i * 3 + 2] = gv.z;
        }
        float Tf[16];
        umeyama3_sample(src, dst, Tf);
        int cnt = 0;
        for (int t = 0; t < n; ++t) cnt += ((double)residual2(Tf, rb.mp[mem[t]], rb.sp[mem[t]]) < thresh2) ? 1 : 0;
        atomicMax(&s_ctrl[6], cnt);
      }
      __syncthreads();
      if (tid == 0 && n_best >= s_ctrl[6]) s_ctrl[3] = 1;
      __syncthreads();
    }
    batch_cap = (batch_cap == 1) ? 4 : (batch_cap == 4 ? 32 : RS_BATCH);
  }
  // ---- result: inliers of the best model, filtered correspondences ----
  __syncthreads();
  const bool ok = s_ctrl[5] != 0;
  int n_inl = 0;
  if (ok) {
    // ordered compaction of the inlier positions (block-wide, chunked); flags[] receives the list
    for (int base = 0; base < n; base += RS_THREADS) {
      const int t = base + tid;
      int f = 0;
      if (t < n) f = ((double)residual2(s_bestT, rb.mp[mem[t]], rb.sp[mem[t]]) < thresh2) ? 1 : 0;
      const unsigned m = __ballot_sync(0xffffffffu, f);
      if (lane == 0) s_warp_cnt[warp] = __popc(m);
      __syncthreads();
      int before = n_inl, chunk_total = 0;
      for (int w = 0; w < RS_THREADS / 32; ++w) {
        if (w < warp) before += s_warp_cnt[w];
        chunk_total += s_warp_cnt[w];
      }
      if (f) flags[before + __popc(m & ((1u << lane) - 1u))] = t;
      n_inl += chunk_total;
      __syncthreads();
    }
  }
  __syncthreads();
  const bool use_model = ok && n_inl >= 3;
  float *T = rb.T_out + (size_t)b * 16;
  if (tid < 16) T[tid] = use_model ? s_bestT[tid] : ((tid % 5 == 0) ? 1.0f : 0.0f);
  const int out_n = use_model ? n_inl : n;
  for (int i = tid; i < out_n; i += RS_THREADS) {
    const int t = use_model ? last_pos[flags[i]] : i;
    if (off + i < corr_cap) rb.inst_corrs[off + i] = rb.sorted[mem[t]];
  }
  if (tid == 0) rb.inst_counts[b] = out_n;
}

}  // namespace

int dev_gc(b200_ctx *ctx, const float4 *d_model_kp, const float4 *d_scene_kp, const b200_corr *d_corrs,
           const int *d_C, int C_cap, double gc_size, int gc_threshold, const InstanceOut &out) {
  if (out.max_inst < 1) return ctx->fail(B200_ERR_INVALID, "gc: max_inst must be >= 1");
  B200_TRY(out.clear(ctx));
  if (C_cap <= 0) return B200_OK;
  // The consistency bitmap is C x C bits.  Up to GC_ASYNC_CAP correspondences it is sized for the
  // capacity and the whole stage stays asynchronous; above that the actual count is read back first, so that the
  // bitmap follows the real number of correspondences (typically a quarter of the scene keypoints: 88 MB instead
  // of 1.07 GB for the 91 k-keypoint scenes of the benchmark) at the price of one small readback per scene.
  constexpr int GC_ASYNC_CAP = 32768;           // 128 MiB bitmap
  constexpr long long GC_MAX_C = 524288;        // 32 GiB bitmap
  int C_eff = C_cap;
  if (C_cap > GC_ASYNC_CAP) {
    int C_now = 0;
    B200_TRY(readback_small(ctx, d_C, &C_now, sizeof(int)));
    C_eff = std::max(1, std::min(C_now, C_cap));
    if (C_eff > GC_MAX_C) return ctx->fail(B200_ERR_CAPACITY, "gc: more than 524288 correspondences");
  }
  const int row_words_cap = ((((C_eff + 31) >> 5) + 127) & ~127);
  const float g_lo = nextafterf((float)gc_size, -INFINITY), g_hi = nextafterf((float)gc_size, INFINITY);
  DevBuf<b200_corr> sorted;
  DevBuf<float4> mp, sp;
  DevBuf<unsigned> adj;
  DevBuf<int> overflow, members, sort_fb;
  B200_TRY(sorted.alloc(ctx, (size_t)C_eff));
  B200_TRY(sort_fb.alloc(ctx, 1));
  B200_TRY(mp.alloc(ctx, (size_t)C_eff));
  B200_TRY(sp.alloc(ctx, (size_t)C_eff));
  B200_TRY(adj.alloc(ctx, (size_t)C_eff * row_words_cap));
  {
    StageScope st_(ctx, ST_GC_SORT);
    const char *sel = getenv("B200_GC_SORT");  // "count": the O(C^2) counting kernel alone
    const int *gate = nullptr;
    if (!(sel && !strcmp(sel, "count"))) {
      DevBuf<int> hist, start;
      DevBuf<unsigned long long> keys;
      B200_TRY(hist.alloc(ctx, SORT_BUCKETS));
      B200_TRY(start.alloc(ctx, SORT_BUCKETS + 1));
      B200_TRY(keys.alloc(ctx, (size_t)C_eff));
      B200_TRY(hist.zero());
      const int nblk = ceil_div(C_eff, 256);
      gc_sort_hist_kernel<<<nblk, 256, 0, ctx->stream>>>(d_corrs, d_C, C_eff, hist.p);
      B200_LAUNCHED(ctx);
      gc_sort_scan_kernel<<<1, 1024, 0, ctx->stream>>>(hist.p, start.p, sort_fb.p);
      B200_LAUNCHED(ctx);
      gc_sort_scatter_kernel<<<nblk, 256, 0, ctx->stream>>>(d_corrs, d_C, C_eff, start.p, hist.p, keys.p, sort_fb.p);
      B200_LAUNCHED(ctx);
      gc_sort_rank_kernel<<<nblk, 256, 0, ctx->stream>>>(d_corrs, d_C, C_eff, d_model_kp, d_scene_kp, start.p, keys.p,
                                                        sorted.p, mp.p, sp.p, sort_fb.p);
      B200_LAUNCHED(ctx);
      gate = sort_fb.p;
    }
    gc_rank_kernel<<<ceil_div(C_eff, RANK_ITEMS), 256, 0, ctx->stream>>>(d_corrs, d_C, C_eff, d_model_kp, d_scene_kp,
                                                                 sorted.p, mp.p, sp.p, gate);
    B200_LAUNCHED(ctx);
  }
  {
    StageScope st_(ctx, ST_GC_ADJ);
    dim3 grid(ceil_div(row_words_cap, ADJ_WORDS), ceil_div(C_eff, ADJ_ROWS));
    gc_adjacency_kernel<<<grid, ADJ_THREADS, 0, ctx->stream>>>(mp.p, sp.p, d_C, C_eff, gc_size, g_lo, g_hi, adj.p);
    B200_LAUNCHED(ctx);
  }
  B200_TRY(overflow.alloc(ctx, (size_t)GCL * C_eff));
  B200_TRY(members.alloc(ctx, (size_t)C_eff));
  GroupArgs ga;
  ga.adj = adj.p;
  ga.mp = mp.p;
  ga.sp = sp.p;
  ga.overflow = overflow.p;
  ga.members = members.p;
  ga.inst_offsets = out.offsets;
  ga.n_inst_out = out.n;
  DevBuf<long long> dbg;
  const bool debug = getenv("B200_GC_DEBUG") != nullptr;
  ga.dbg = nullptr;
  if (debug) {
    B200_TRY(dbg.alloc(ctx, GCL * 8));
    B200_TRY(dbg.zero());
    ga.dbg = dbg.p;
  }
  // everything up to here keeps the whole GPU busy; the grouping kernel is one cluster: the next scene's wide
  // stages may start beside it
  if (ctx->wide) ctx->wide->leave();
  {
    StageScope st_(ctx, ST_GC_GROUP);
    // one 8-CTA cluster: a seed per CTA; shared memory = taken bitmap + candidate bitmap (at most 2 x 64 KiB: GC_MAX_C
    // caps a row at 16 384 words)
    const size_t smem = 2 * (size_t)row_words_cap * sizeof(unsigned);
    B200_CUDA(ctx, ensure_dyn_smem(gc_group_cluster_kernel, smem));
    gc_group_cluster_kernel<<<GCL, GCL_THREADS, smem, ctx->stream>>>(ga, d_C, C_eff, gc_size, g_lo, g_hi, gc_threshold,
                                                                    out.max_inst);
    B200_LAUNCHED(ctx);
  }
  if (debug) {
    long long h[GCL * 8];
    B200_CUDA(ctx, cudaMemcpyAsync(h, dbg.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(ctx, ctx->sync());
    for (int w = 0; w < GCL; ++w)
      fprintf(stderr, "gc_group cta %d: window %lld init %lld and %lld list %lld list+greedy %lld cluster-sync %lld commit %lld rounds %lld\n",
              w, h[w * 8], h[w * 8 + 1], h[w * 8 + 2], h[w * 8 + 3], h[w * 8 + 4], h[w * 8 + 5], h[w * 8 + 6], h[w * 8 + 7]);
  }

  return dev_ransac_instances(ctx, sorted.p, mp.p, sp.p, members.p, C_eff, gc_size, out);
}

// RANSAC pose + correspondence filtering for a set of instances (shared by geometric-consistency and
// Hough grouping).  corrs: the correspondence records the member indices refer to; mp / sp: model and
// scene keypoint of every correspondence; members: concatenated member lists, inst_offsets[i]..[i+1].
int dev_ransac_instances(b200_ctx *ctx, const b200_corr *d_corrs, const float4 *d_mp, const float4 *d_sp,
                         const int *d_members, int C_cap, double threshold, const InstanceOut &out) {
  DevBuf<int> shuffled, last_pos, flags;
  if (!ctx->mt_state) {
    unsigned host_state[624];
    mt19937_twisted_state(12345u, host_state);
    B200_CUDA(ctx, cudaMalloc(&ctx->mt_state, sizeof(host_state)));
    B200_CUDA(ctx, cudaMemcpyAsync(ctx->mt_state, host_state, sizeof(host_state), cudaMemcpyHostToDevice, ctx->stream));
    B200_CUDA(ctx, ctx->sync());
  }
  B200_TRY(shuffled.alloc(ctx, (size_t)C_cap));
  B200_TRY(last_pos.alloc(ctx, (size_t)C_cap));
  B200_TRY(flags.alloc(ctx, (size_t)C_cap));
  RansacBuffers rb;
  rb.sorted = d_corrs;
  rb.mp = d_mp;
  rb.sp = d_sp;
  rb.members = d_members;
  rb.inst_offsets = out.offsets;
  rb.n_inst = out.n;
  rb.mt_init = ctx->mt_state;
  rb.shuffled = shuffled.p;
  rb.last_pos = last_pos.p;
  rb.flags = flags.p;
  rb.T_out = out.T;
  rb.inst_counts = out.counts;
  rb.inst_corrs = out.corrs;
  StageScope st_(ctx, ST_GC_RANSAC);
  gc_ransac_kernel<32><<<out.max_inst, 32, 0, ctx->stream>>>(rb, out.max_inst, out.corr_cap, threshold, 10000);
  B200_LAUNCHED(ctx);
  gc_ransac_kernel<128><<<out.max_inst, 128, 0, ctx->stream>>>(rb, out.max_inst, out.corr_cap, threshold, 10000);
  B200_LAUNCHED(ctx);
  return B200_OK;
}
