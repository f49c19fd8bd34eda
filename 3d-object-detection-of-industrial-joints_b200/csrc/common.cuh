// common.cuh — context, stream-ordered scratch buffers, launch accounting and small device helpers
// shared by every kernel file of libb200reg.so.  Compiled with --fmad=false: float32 sums that
// PCL/FLANN evaluate as plain mul/add sequences must not be contracted into FMAs.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>
#include <array>
#include <mutex>
#include <map>
#include <memory>
#include <utility>
#include <vector>
#include <cstdio>
#include <cstdlib>
#include <chrono>

#include "../../include/b200reg.h"

// pipeline stages timed with CUDA events on the context's stream when profiling is enabled
enum b200_stage {
  ST_GRID = 0,
  ST_NORMALS,
  ST_NBR_COUNT,
  ST_SHOT,
  ST_FPFH,
  ST_MATCH,
  ST_GC_SORT,
  ST_GC_ADJ,
  ST_GC_GROUP,
  ST_GC_RANSAC,
  ST_MATCH_FILTER,  // nested inside ST_MATCH: the tcgen05 pre-filter kernel alone
  ST_BOARD,         // BOARD reference frames (board.cu)
  ST_HOUGH,         // Hough voting and maxima (hough.cu); its RANSAC is ST_GC_RANSAC
  ST_COUNT
};

struct StageEvent {
  cudaEvent_t a, b;
  int stage;
};

// Device scratch arena.  Every buffer of a context is used on the context's single stream, so a
// block can be handed to the next user as soon as the previous owner releases it (stream order makes
// the reuse safe) — no driver call in steady state.  cudaMallocAsync was measured to stall the host
// for 0.2-0.7 s per step here (it waits for in-flight work before reusing large freed blocks).
struct ArenaBlock {
  void *p;
  size_t size;
  bool used;
};

struct WideSection;

struct b200_ctx {
  WideSection *wide = nullptr;  // set while this context is inside the wide-stage gate (see WideGate)
  std::vector<ArenaBlock> arena;
  size_t arena_bytes = 0;
  void *arena_alloc(size_t bytes, cudaError_t *err) {
    const size_t gran = bytes >= (1u << 20) ? (1u << 20) : 512;
    bytes = ((bytes + gran - 1) / gran) * gran;
    int best = -1;
    for (int i = 0; i < (int)arena.size(); ++i)
      if (!arena[i].used && arena[i].size >= bytes && (best < 0 || arena[i].size < arena[best].size)) best = i;
    if (best >= 0 && arena[best].size <= 2 * bytes + (1u << 20)) {
      arena[best].used = true;
      *err = cudaSuccess;
      return arena[best].p;
    }
    // high-water cap: before growing past it, give the idle blocks back to the driver (a long-running service that
    // sees scenes of very different sizes would otherwise keep every size class it ever needed)
    static const size_t cap = []() {
      const char *e = getenv("B200_ARENA_CAP_MB");
      return (size_t)(e ? atoll(e) : 4096) << 20;
    }();
    if (arena_bytes + bytes > cap) arena_trim();
    void *p = nullptr;
    *err = cudaMalloc(&p, bytes);
    if (*err == cudaErrorMemoryAllocation) {  // out of memory: release what is idle and retry once
      cudaGetLastError();
      arena_trim();
      *err = cudaMalloc(&p, bytes);
    }
    if (*err != cudaSuccess) return nullptr;
    arena.push_back({p, bytes, true});
    arena_bytes += bytes;
    return p;
  }
  void arena_free(void *p) {
    for (auto &b : arena)
      if (b.p == p) {
        b.used = false;
        return;
      }
  }
  void arena_trim() {  // frees every idle block (cudaFree synchronises the device: only on the growth path)
    size_t w = 0;
    for (size_t i = 0; i < arena.size(); ++i) {
      if (arena[i].used) {
        arena[w++] = arena[i];
      } else {
        cudaFree(arena[i].p);
        arena_bytes -= arena[i].size;
      }
    }
    arena.resize(w);
  }
  void arena_destroy() {
    for (auto &b : arena) cudaFree(b.p);
    arena.clear();
    arena_bytes = 0;
  }
  bool profiling = false;
  std::vector<StageEvent> stage_events;
  std::vector<cudaEvent_t> event_pool;
  double stage_ms[ST_COUNT] = {0};
  int stage_n[ST_COUNT] = {0};
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 148;
  size_t smem_optin = 0;
  int64_t launches = 0;
  // Host waits.  Spinning (cudaStreamSynchronize) has the lowest latency; with more lanes than host cores the
  // contexts are switched to a blocking event wait instead (b200_ctx_set_blocking_sync), which sleeps the thread.
  bool blocking_sync = false;
  cudaEvent_t sync_ev = nullptr;
  cudaError_t sync() {
    if (!blocking_sync) return cudaStreamSynchronize(stream);
    cudaError_t e = cudaSuccess;
    if (!sync_ev) e = cudaEventCreateWithFlags(&sync_ev, cudaEventBlockingSync | cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(sync_ev, stream);
    if (e == cudaSuccess) e = cudaEventSynchronize(sync_ev);
    return e;
  }
  // small device->host readbacks go through mapped pinned memory written by a kernel, not through the copy engine
  // (see readback_small in api.cu)
  void *mailbox_host = nullptr;
  void *mailbox_dev = nullptr;
  uint32_t rand_state[31] = {0};  // glibc rand() stream for BOARD's random axis (board.cu)
  bool rand_seeded = false;
  int *board_draws = nullptr;  // pinned staging of BOARD's rand() draws (board.cu)
  size_t board_draws_cap = 0;
  double last_mean_nbrs = 0.0;
  int last_max_nbrs = 0;
  float last_match_err_ratio = 0.f;  // max observed approximation error / assumed bound (profiling only)
  int last_match_fallback = -1;  // rows the tensor-core filter could not certify (valid after a sync)
  int last_match_pass1_fail = -1;  // rows the one-term pass left to the three-term pass (profiling only)
  std::string err;
  void *nccl_comm = nullptr;  // ncclComm_t once b200_comm_init has run (comm.cu)
  int comm_rank = 0, comm_world = 1;
  void *pinned = nullptr;  // small pinned staging block for tiny readbacks
  unsigned *mt_state = nullptr;  // mt19937 state after seeding with 12345 and the first twist (gc.cu)
  int fail(int code, const char *msg) {
    err = msg;
    return code;
  }
  int fail_cuda(cudaError_t e, const char *what, const char *file, int line) {
    char buf[512];
    snprintf(buf, sizeof(buf), "CUDA error %s (%s) at %s:%d in %s", cudaGetErrorName(e), cudaGetErrorString(e),
             file, line, what);
    err = buf;
    return B200_ERR_CUDA;
  }
};

#define B200_CUDA(ctx, expr)                                                        \
  do {                                                                              \
    cudaError_t e__ = (expr);                                                       \
    if (e__ != cudaSuccess) return (ctx)->fail_cuda(e__, #expr, __FILE__, __LINE__); \
  } while (0)

#define B200_TRY(expr)          \
  do {                          \
    int rc__ = (expr);          \
    if (rc__ != B200_OK) return rc__; \
  } while (0)

// After a kernel launch: count it and surface launch-configuration errors.
#define B200_LAUNCHED(ctx)                                                           \
  do {                                                                               \
    (ctx)->launches++;                                                               \
    cudaError_t e__ = cudaGetLastError();                                            \
    if (e__ != cudaSuccess) return (ctx)->fail_cuda(e__, "kernel launch", __FILE__, __LINE__); \
  } while (0)

// Device buffer from the context's arena (see ArenaBlock).
template <class T>
struct DevBuf {
  b200_ctx *ctx = nullptr;
  T *p = nullptr;
  size_t n = 0;
  DevBuf() {}
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p) ctx->arena_free(p);
    p = nullptr;
    n = 0;
  }
  int alloc(b200_ctx *c, size_t count) {
    release();
    ctx = c;
    n = count;
    if (count == 0) count = 1;
    cudaError_t e;
    p = (T *)c->arena_alloc(count * sizeof(T), &e);
    if (e != cudaSuccess) {
      p = nullptr;
      c->fail_cuda(e, "cudaMalloc (arena)", __FILE__, __LINE__);
      return e == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA;
    }
    return B200_OK;
  }
  int zero() {
    cudaError_t e = cudaMemsetAsync(p, 0, (n ? n : 1) * sizeof(T), ctx->stream);
    if (e != cudaSuccess) return ctx->fail_cuda(e, "cudaMemsetAsync", __FILE__, __LINE__);
    return B200_OK;
  }
};

// Records a CUDA-event pair around a stage (only when profiling is on; otherwise free).
struct StageScope {
  b200_ctx *ctx;
  StageEvent ev;
  bool on;
  StageScope(b200_ctx *c, int stage) : ctx(c), on(c->profiling) {
    if (!on) return;
    auto get = [&]() {
      cudaEvent_t e;
      if (!ctx->event_pool.empty()) {
        e = ctx->event_pool.back();
        ctx->event_pool.pop_back();
      } else {
        cudaEventCreate(&e);
      }
      return e;
    };
    ev.a = get();
    ev.b = get();
    ev.stage = stage;
    cudaEventRecord(ev.a, ctx->stream);
  }
  ~StageScope() {
    if (!on) return;
    cudaEventRecord(ev.b, ctx->stream);
    ctx->stage_events.push_back(ev);
  }
};

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Opt-in dynamic shared memory of a kernel.  The attribute is per function and device, shared by every context
// (lane) of the process: it only ever grows here, so a launch on another thread that asked for less stays valid
// (setting it to each call's own size let one lane shrink it under another lane's launch).
template <class F>
static inline cudaError_t ensure_dyn_smem(F *func, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void *>, size_t> cur;  // (device, kernel) -> bytes granted so far
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(mu);
  size_t &c = cur[std::make_pair(dev, reinterpret_cast<const void *>(func))];
  if (bytes <= c) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) c = bytes;
  return e;
}

// ------------------------------------------------------------------------------------------
// Uniform grid over a search surface (grid.cu builds it).
// pts: points in cell-major order, w = original row index (bit pattern of an int).
// ------------------------------------------------------------------------------------------
struct GridView {
  const float4 *pts;
  const float4 *raw;  // the cloud in caller order (x, y, z, 1): neighbour coordinates by original index
  const int *cell_start;  // ncell + 1 entries
  float lox, loy, loz;
  float h, inv_h;
  int dx, dy, dz;
  int n;              // number of indexed (finite) points
  float coord_scale;  // max |coordinate| of the bounding box (for conservative float margins)
};

__host__ __device__ __forceinline__ int grid_coord(float v, float lo, float inv_h, int dim) {
  float f = floorf((v - lo) * inv_h);
  if (!(f >= 0.0f)) return 0;
  if (f >= (float)dim) return dim - 1;
  return (int)f;
}

// FLANN L2_Simple<float> over x, y, z: ((dx*dx + dy*dy) + dz*dz), no FMA (--fmad=false keeps it so).
__device__ __forceinline__ float sqdist3(float ax, float ay, float az, float bx, float by, float bz) {
  float d0 = ax - bx;
  float r = __fmul_rn(d0, d0);
  float d1 = ay - by;
  r = __fadd_rn(r, __fmul_rn(d1, d1));
  float d2 = az - bz;
  r = __fadd_rn(r, __fmul_rn(d2, d2));
  return r;
}

__device__ __forceinline__ int orig_index(const float4 &p) { return __float_as_int(p.w); }

__device__ __forceinline__ float nanf32() { return __int_as_float(0x7fc00000); }

__device__ __forceinline__ bool finite3(float x, float y, float z) {
  return isfinite(x) && isfinite(y) && isfinite(z);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------
// internal entry points implemented across the .cu files (all asynchronous on ctx->stream unless
// noted; every pointer is a device pointer)
// ------------------------------------------------------------------------------------------
struct DeviceGrid {
  DevBuf<float4> pts;
  DevBuf<int> cell_start;
  GridView view;
  float cell = 0.f;
  bool valid = false;
};

struct b200_cloud {
  b200_ctx *ctx = nullptr;
  int n = 0;
  int n_valid = 0;
  DevBuf<float4> raw;  // original order, w = 1 (pad)
  float lo[3], hi[3];  // bounding box of the finite points (host copy)
  DeviceGrid knn_grid;     // cell sized for k-nearest queries
  int knn_grid_k = 0;
  DeviceGrid radius_grid;  // cell sized for fixed-radius queries
};

// Model side of the tensor-core correspondence filter (match_tc.cu), prepared once per resident model: the fp16
// split operands, |b|^2, the power-of-two scale and the row-validity flags do not change between scenes.
struct TcModelPrep {
  bool ready = false;
  int Km = 0, D = 0, rowsB = 0;
  DevBuf<unsigned short> B1, B3;  // fp16 bits: one-term [b1] and three-term [b1|b2|b1] rows, zero padded
  DevBuf<float> nb;               // |b_j|^2 (+inf for padding / invalid rows)
  DevBuf<float> scaleB;           // [0] = 2^s, [1] = max |b|
  DevBuf<unsigned> bits;          // [0] = bits of max |b|, [1] = bits of max |b|^2
  DevBuf<unsigned char> mvalid;   // row has only finite values
  DevBuf<int> nmv;                // number of valid rows
};

struct b200_model {
  b200_ctx *ctx = nullptr;
  int K = 0;
  int D = 352;
  DevBuf<float> desc;  // K x D
  DevBuf<float4> kp;   // K keypoints
  TcModelPrep tc;      // filled by match_prepare_model for libraries large enough for the tensor-core path
  // Hough branch (b200_model_create_shot_hough)
  bool has_frames = false;
  DevBuf<float> rf;             // K x 9 BOARD frames of the keypoints
  DevBuf<float> votes;          // K x 3 Hough3DGrouping::train() votes
  uint32_t rand_state[31] = {0};  // the creating context's rand() stream right after the frames
};

struct b200_library {
  b200_ctx *ctx = nullptr;
  std::vector<b200_model *> views;
  std::vector<std::array<float, 16>> poses;  // per view: row-major 4x4 (view -> CAD pose table), identity by default
};

// B200_TRACE=1: host-side wall time between ticks (debugging aid)
struct HostTrace {
  bool on;
  std::chrono::steady_clock::time_point t;
  HostTrace() : on(getenv("B200_TRACE") != nullptr), t(std::chrono::steady_clock::now()) {}
  void tick(const char *what) {
    if (!on) return;
    auto n = std::chrono::steady_clock::now();
    double ms = std::chrono::duration<double, std::milli>(n - t).count();
    if (ms > 0.3) fprintf(stderr, "[b200 trace] %s: %.3f ms host\n", what, ms);
    t = n;
  }
};

// Wide-stage gate.  A scene registration is a run of GPU-wide stages (normals, descriptors, matching, the
// consistency bitmap: every SM busy) followed by the grouping kernel, a latency-bound chain on one 8-CTA cluster.
// With several scenes in flight on one device (one context + stream + host thread each) the step rate is best when
// the wide runs of different scenes do not overlap each other but do overlap the grouping of the previous scenes —
// and worst when the lanes fall into lockstep (all in their wide run, then all in grouping with 140 SMs idle).  The
// gate makes the good schedule deterministic: contexts take turns for the wide run, in arrival order; a turn ends
// when the grouping kernel is about to be enqueued, by recording an event the next turn's stream waits on.
// Measured (target workload): gated 9.4 ms/scene with any number of lanes >= 2; free-running lanes 9.9 (2 lanes),
// 8.0 (4 lanes) once nothing small goes through the copy engines (readback_small).  Free running is therefore the
// default and the gate is opt-in (B200_WIDE_GATE=1) for deployments that can afford only two lanes of memory.
struct WideGate {
  std::mutex mu;
  cudaEvent_t ev = nullptr;
  bool recorded = false;
};
WideGate *wide_gate(int device);  // api.cu; nullptr unless B200_WIDE_GATE=1

struct WideSection {
  b200_ctx *ctx = nullptr;
  WideGate *g = nullptr;
  bool held = false;
  int enter(b200_ctx *c) {
    ctx = c;
    g = wide_gate(c->device);
    if (!g) return B200_OK;
    g->mu.lock();
    held = true;
    c->wide = this;
    if (!g->ev) {
      cudaError_t e = cudaEventCreateWithFlags(&g->ev, cudaEventDisableTiming);
      if (e != cudaSuccess) {
        g->ev = nullptr;
        leave();
        return c->fail_cuda(e, "cudaEventCreate (wide gate)", __FILE__, __LINE__);
      }
    }
    if (g->recorded) {
      cudaError_t e = cudaStreamWaitEvent(c->stream, g->ev, 0);
      if (e != cudaSuccess) {
        leave();
        return c->fail_cuda(e, "cudaStreamWaitEvent (wide gate)", __FILE__, __LINE__);
      }
    }
    return B200_OK;
  }
  void leave() {
    if (!held) return;
    if (g->ev && cudaEventRecord(g->ev, ctx->stream) == cudaSuccess) g->recorded = true;
    ctx->wide = nullptr;
    held = false;
    g->mu.unlock();
  }
  ~WideSection() { leave(); }
};

// api.cu — small transfers that stay off the copy engines.  The copy-engine queues are shared by all streams and run
// in order: a tiny D2H readback enqueued behind another context's pending result download (which waits for that
// context's whole scene) stalls this context's host for the length of the other scene.  readback_small: up to 256
// bytes device -> host through a kernel writing mapped pinned memory, then a stream synchronise.  write_small: up
// to 64 bytes host -> device as kernel arguments.
constexpr size_t B200_MAILBOX_BYTES = 256;
int readback_small(b200_ctx *ctx, const void *d_src, void *h_dst, size_t bytes);
int write_small(b200_ctx *ctx, void *d_dst, const void *h_src, size_t bytes);

// scan.cu
int exclusive_scan_i32(b200_ctx *ctx, const int *d_in, int *d_out, int n, int *d_total /*nullable*/);
// grid.cu
int cloud_upload(b200_ctx *ctx, const float *xyz, int n, int stride, bool on_device, std::unique_ptr<b200_cloud> &out);
int cloud_grid_for_knn(b200_cloud *c, int k, const GridView **out);
int cloud_grid_for_radius(b200_cloud *c, double radius, const GridView **out);
int pack_points(b200_ctx *ctx, const float *d_xyz, int n, int stride, float4 *d_out);
// search.cu
int dev_knn_search(b200_ctx *ctx, b200_cloud *c, const float4 *d_q, int nq, int k, int *d_idx, float *d_d2,
                   int *k_found);
int dev_radius_count(b200_ctx *ctx, const GridView &g, const float4 *d_q, int nq, double radius, int *d_counts,
                     unsigned long long *d_stats /* [0]=max, [1]=sum */);
int dev_radius_fill_sized(b200_ctx *ctx, const GridView &g, const float4 *d_q, int nq, double radius, int max_count,
                          const long long *d_offsets, int *d_idx, float *d_d2);
int counts_to_offsets_i64(b200_ctx *ctx, const int *d_counts, int nq, long long *d_offsets);
int knn_threads_for(int k, size_t *smem_bytes);
// normals.cu
int dev_normals(b200_ctx *ctx, b200_cloud *c, const float4 *d_q, int nq, bool q_is_surface, int k, double radius,
                const float *vp, float *d_out);
// shot.cu
int dev_shot(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_kp, int K, double radius,
             float *d_desc, float *d_rf, bool lrf_only);
// fpfh.cu
int dev_fpfh(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_q, int nq, bool q_is_surface,
             double radius, float *d_out);
// match.cu
int dev_match(b200_ctx *ctx, const float *d_model, int Km, const float *d_scene, int Ks, int D, int mode, float thr,
              b200_corr *d_out, int *d_count, const TcModelPrep *prep = nullptr);
int match_prepare_model(b200_ctx *ctx, b200_model *m);  // no-op for small libraries
int match_prepare_rows(b200_ctx *ctx, const float *d_desc, int K, int D, TcModelPrep *t);
int dev_nearest1(b200_ctx *ctx, const float *d_model, int Km, const unsigned char *mvalid_p, const TcModelPrep *prep,
                 const float *d_q, int nq, int D, int *d_idx, float *d_d2);

// Device result of one grouping run (dev_gc, dev_hough3d): per instance its 4x4 pose (T, max_inst x 16), the start of
// its correspondences (offsets, max_inst + 1) and how many RANSAC kept (counts, max_inst); the kept correspondences
// (corrs, corr_cap entries) and the number of instances found (*n, which may exceed max_inst).
struct InstanceOut {
  float *T;
  int max_inst;
  int *offsets;
  int *counts;
  b200_corr *corrs;
  int corr_cap;
  int *n;
  // the zero count, offsets and counts every grouping run starts from
  int clear(b200_ctx *ctx) const {
    B200_CUDA(ctx, cudaMemsetAsync(n, 0, sizeof(int), ctx->stream));
    B200_CUDA(ctx, cudaMemsetAsync(offsets, 0, sizeof(int) * ((size_t)max_inst + 1), ctx->stream));
    B200_CUDA(ctx, cudaMemsetAsync(counts, 0, sizeof(int) * (size_t)max_inst, ctx->stream));
    return B200_OK;
  }
};

int dev_ransac_instances(b200_ctx *ctx, const b200_corr *d_corrs, const float4 *d_mp, const float4 *d_sp,
                         const int *d_members, int C_cap, double threshold, const InstanceOut &out);
// hough.cu
int dev_hough_model_votes(b200_ctx *ctx, const float4 *d_model_kp, const float *d_model_rf, int Km, float *d_votes);
// correspondence count: *d_C (at most C_cap); *d_status = B200_ERR_CAPACITY when the space has more than 2^27 bins
int dev_hough3d(b200_ctx *ctx, const float4 *d_model_kp, const float *d_model_votes, const float4 *d_scene_kp,
                const float *d_scene_rf, const b200_corr *d_corrs, const int *d_C, int C_cap, double bin_size,
                double threshold, const InstanceOut &out, int *d_status);
// board.cu
void board_rand_seed(b200_ctx *ctx, unsigned seed);
int dev_board_lrf_from(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_kp, int K, double radius,
                       const b200_board_params *p, uint32_t rand_state[31], float *d_rf);
int dev_board_lrf(b200_ctx *ctx, b200_cloud *c, const float *d_normals, const float4 *d_kp, int K, double radius,
                  const b200_board_params *p, float *d_rf);
// icp.cu
int dev_icp_align(b200_ctx *ctx, const float4 *d_src, int ns, b200_cloud *target, int max_iterations, double max_corr_dist,
                  double transformation_epsilon, double euclidean_fitness_epsilon, const float *guess, float *final_T,
                  float4 *d_aligned, double *fitness, int *converged, int *iterations);
// keypoints.cu
int dev_remove_nan(b200_ctx *ctx, const float *d_xyz, int n, int stride, float *d_out_xyz, int *d_out_index, int *d_count);
int dev_transform_points(b200_ctx *ctx, const float *d_xyz, int n, int stride, const float *T16, float *d_out_xyz);
int dev_uniform_sampling(b200_ctx *ctx, const float *d_xyz, int n, int stride, float leaf, float *d_out_xyz,
                         int *d_out_index, int *d_count);
int dev_voxel_grid(b200_ctx *ctx, const float *d_xyz, int n, int stride, float lx, float ly, float lz,
                   float *d_out_xyz, int *d_count);
// comm.cu
int comm_unique_id(void *id128, size_t bytes, std::string *err);
int comm_init(b200_ctx *ctx, const void *id128, int rank, int world);
int comm_destroy(b200_ctx *ctx);
int comm_broadcast(b200_ctx *ctx, void *d_buf, size_t bytes, int root);
int comm_allgather(b200_ctx *ctx, const void *d_send, void *d_recv, size_t bytes_per_rank);
int dev_gather_correspondences(b200_ctx *ctx, const b200_corr *d_corrs, const int *d_count, int cap,
                               b200_corr *d_gathered, int *d_counts);
int dev_concat_lists(b200_ctx *ctx, const b200_corr *d_gathered, const int *d_counts, int world, int cap,
                     b200_corr *d_out, int out_cap, int *d_n_out);
int dev_offset_scene_index(b200_ctx *ctx, b200_corr *d_corrs, const int *d_n, int cap, int offset);
// gc.cu
int dev_gc(b200_ctx *ctx, const float4 *d_model_kp, const float4 *d_scene_kp, const b200_corr *d_corrs,
           const int *d_C, int C_cap, double gc_size, int gc_threshold, const InstanceOut &out);
