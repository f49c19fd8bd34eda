// api.cu — the C ABI of libb200reg.so (include/b200reg.h): argument checking, host<->device staging
// and the resident SHOT registration pipeline.  No torch types, no exceptions across the boundary.
#include <algorithm>
#include <functional>
#include <initializer_list>
#include <mutex>
#include <thread>
#include <array>
#include <string>
#include <cstdio>
#include <cstring>
#include <exception>
#include <new>
#include <vector>

#include "common.cuh"

WideGate *wide_gate(int device) {
  static WideGate gates[64];
  static const bool on = [] {
    const char *e = getenv("B200_WIDE_GATE");
    return e && e[0] == '1';
  }();
  if (!on || device < 0 || device >= 64) return nullptr;
  return &gates[device];
}

namespace {
__global__ void mailbox_publish_kernel(const unsigned *__restrict__ src, unsigned *__restrict__ dst, int words) {
  if ((int)threadIdx.x < words) dst[threadIdx.x] = src[threadIdx.x];
}
struct SmallWords {
  unsigned w[16];
};
__global__ void write_small_kernel(unsigned *__restrict__ dst, SmallWords v, int words) {
  if ((int)threadIdx.x < words) dst[threadIdx.x] = v.w[threadIdx.x];
}
}  // namespace

int readback_small(b200_ctx *ctx, const void *d_src, void *h_dst, size_t bytes) {
  if (bytes == 0) return B200_OK;
  if (bytes > B200_MAILBOX_BYTES || (bytes & 3)) return ctx->fail(B200_ERR_INVALID, "readback_small: bad size");
  if (!ctx->mailbox_host) {
    B200_CUDA(ctx, cudaHostAlloc(&ctx->mailbox_host, B200_MAILBOX_BYTES, cudaHostAllocMapped));
    B200_CUDA(ctx, cudaHostGetDevicePointer(&ctx->mailbox_dev, ctx->mailbox_host, 0));
  }
  mailbox_publish_kernel<<<1, 64, 0, ctx->stream>>>((const unsigned *)d_src, (unsigned *)ctx->mailbox_dev, (int)(bytes / 4));
  B200_LAUNCHED(ctx);
  B200_CUDA(ctx, ctx->sync());
  memcpy(h_dst, ctx->mailbox_host, bytes);
  return B200_OK;
}

int write_small(b200_ctx *ctx, void *d_dst, const void *h_src, size_t bytes) {
  if (bytes == 0) return B200_OK;
  if (bytes > sizeof(SmallWords) || (bytes & 3)) return ctx->fail(B200_ERR_INVALID, "write_small: bad size");
  SmallWords v;
  memcpy(v.w, h_src, bytes);
  write_small_kernel<<<1, 32, 0, ctx->stream>>>((unsigned *)d_dst, v, (int)(bytes / 4));
  B200_LAUNCHED(ctx);
  return B200_OK;
}

namespace {

thread_local std::string g_error = "";  // per thread: the batch API's lane threads write it too

int set_device(b200_ctx *ctx) {
  cudaError_t e = cudaSetDevice(ctx->device);
  if (e != cudaSuccess) return ctx->fail_cuda(e, "cudaSetDevice", __FILE__, __LINE__);
  return B200_OK;
}

#define API_ENTER(ctx)                        \
  if (!(ctx)) {                               \
    g_error = "null context";                 \
    return B200_ERR_INVALID;                  \
  }                                           \
  B200_TRY(set_device(ctx))

template <class T>
int upload(b200_ctx *ctx, DevBuf<T> &buf, const T *host, size_t count) {
  B200_TRY(buf.alloc(ctx, count));
  if (count)
    B200_CUDA(ctx, cudaMemcpyAsync(buf.p, host, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return B200_OK;
}

// Result downloads are enqueued only once the stream has drained: a D2H copy waiting in the (shared, in-order)
// copy-engine queue for its own stream's kernels would hold up the copies and memsets of every other context.
template <class T>
int download(b200_ctx *ctx, T *host, const T *dev, size_t count) {
  if (count) {
    B200_CUDA(ctx, ctx->sync());
    B200_CUDA(ctx, cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  }
  return B200_OK;
}

// host rows (stride floats) → device float4
int upload_points(b200_ctx *ctx, const float *xyz, int n, int stride, DevBuf<float4> &out) {
  if (n < 0 || stride < 3 || (n > 0 && !xyz)) return ctx->fail(B200_ERR_INVALID, "bad point array");
  B200_TRY(out.alloc(ctx, (size_t)std::max(n, 1)));
  if (n == 0) return B200_OK;
  DevBuf<float> stage;
  B200_TRY(upload(ctx, stage, xyz, (size_t)n * stride));
  return pack_points(ctx, stage.p, n, stride, out.p);
}

int pack_device_points(b200_ctx *ctx, const float *d_xyz, int n, int stride, DevBuf<float4> &out) {
  if (n < 0 || stride < 3 || (n > 0 && !d_xyz)) return ctx->fail(B200_ERR_INVALID, "bad point array");
  B200_TRY(out.alloc(ctx, (size_t)std::max(n, 1)));
  return pack_points(ctx, d_xyz, n, stride, out.p);
}

// b200_cloud_create / b200_dev_cloud_create
int cloud_create(b200_ctx *ctx, const float *xyz, int n, int stride, bool on_device, b200_cloud **out) {
  if (!out) return ctx->fail(B200_ERR_INVALID, "cloud_create: bad arguments");
  std::unique_ptr<b200_cloud> cloud;
  B200_TRY(cloud_upload(ctx, xyz, n, stride, on_device, cloud));
  *out = cloud.release();
  return B200_OK;
}

int check_params(b200_ctx *ctx, const b200_shot_params *p) {
  if (!p) return ctx->fail(B200_ERR_INVALID, "null params");
  if ((p->normal_k != 0) == (p->normal_radius != 0.0))
    return ctx->fail(B200_ERR_INVALID, "params: exactly one of normal_k / normal_radius must be non-zero");
  if (!(p->descr_radius > 0.0)) return ctx->fail(B200_ERR_INVALID, "params: descr_radius must be > 0");
  if (p->match_mode != 1 && p->match_mode != 2) return ctx->fail(B200_ERR_INVALID, "params: match_mode must be 1 or 2");
  if (p->max_instances < 1) return ctx->fail(B200_ERR_INVALID, "params: max_instances must be >= 1");
  return B200_OK;
}

int check_hough_params(b200_ctx *ctx, const b200_hough_params *h) {
  if (!h) return ctx->fail(B200_ERR_INVALID, "null Hough params");
  if (!(h->rf_radius > 0.0)) return ctx->fail(B200_ERR_INVALID, "hough params: rf_radius must be > 0");
  if (!(h->bin_size > 0.0)) return ctx->fail(B200_ERR_INVALID, "hough params: bin_size must be > 0");
  return B200_OK;
}

// the checks the SHOT scene registrations (host and device buffers, lanes) make of the parameters and of a non-null
// model; a model of another descriptor length (FPFH: 33) would have dev_match read K x 352 floats from K x 33
int check_registration(b200_ctx *ctx, const b200_model *model, const b200_shot_params *p, const b200_hough_params *h) {
  B200_TRY(check_params(ctx, p));
  if (model->D != 352)
    return ctx->fail(B200_ERR_INVALID, "register_scene_shot: the model is not a SHOT352 model (b200_model_create_shot)");
  if (!h) return B200_OK;
  B200_TRY(check_hough_params(ctx, h));
  if (!model->has_frames)
    return ctx->fail(B200_ERR_INVALID, "register_scene_hough: the model has no frames (b200_model_create_shot_hough)");
  return B200_OK;
}

// The dense cloud a BOARD frame estimation searches (setSearchSurface) and the normal estimation run on it
// (setKSearch / setRadiusSearch): the FPFH Hough branch's surface, which is not the keypoint cloud its descriptors use.
struct DenseSurface {
  const float *xyz;
  int n, stride;
  int normal_k;
  double normal_radius;
  int check(b200_ctx *ctx) const {
    if ((normal_k != 0) == (normal_radius != 0.0) || normal_k < 0 || normal_radius < 0.0)
      return ctx->fail(B200_ERR_INVALID, "exactly one of surface_normal_k / surface_normal_radius must be positive");
    return B200_OK;
  }
  // the cloud on the device and its normals (cloud->n x 4)
  int upload(b200_ctx *ctx, std::unique_ptr<b200_cloud> &cloud, DevBuf<float> &normals) const {
    B200_TRY(cloud_upload(ctx, xyz, n, stride, false, cloud));
    B200_TRY(normals.alloc(ctx, (size_t)std::max(cloud->n, 1) * 4));
    return dev_normals(ctx, cloud.get(), cloud->raw.p, cloud->n, true, normal_k, normal_radius, nullptr, normals.p);
  }
};

// Device result of a scene registration: the correspondence list (cap entries) and, per view, its correspondence
// count and one grouping result for max_inst instances and cap instance correspondences (out(v)).
struct ResultBufs {
  int cap = 0, max_inst = 0;
  DevBuf<b200_corr> corrs, inst_corrs;
  DevBuf<int> offsets, counts, n_inst, n_corrs;
  DevBuf<float> T;
  int alloc(b200_ctx *ctx, int corr_cap, int instances, int views = 1) {
    cap = corr_cap;
    max_inst = instances;
    const size_t v = (size_t)std::max(views, 1);
    B200_TRY(corrs.alloc(ctx, (size_t)cap));
    B200_TRY(inst_corrs.alloc(ctx, (size_t)cap * v));
    B200_TRY(offsets.alloc(ctx, ((size_t)max_inst + 1) * v));
    B200_TRY(counts.alloc(ctx, (size_t)max_inst * v));
    B200_TRY(n_inst.alloc(ctx, v));
    B200_TRY(n_corrs.alloc(ctx, v));
    return T.alloc(ctx, (size_t)max_inst * 16 * v);
  }
  InstanceOut out(int v = 0) const {
    return {T.p + (size_t)v * max_inst * 16, max_inst, offsets.p + (size_t)v * (max_inst + 1),
            counts.p + (size_t)v * max_inst, inst_corrs.p + (size_t)v * cap, cap, n_inst.p + v};
  }
};

// a caller's correspondence list (C > 0 entries) and its count into r
int upload_corrs(b200_ctx *ctx, ResultBufs &r, const b200_corr *corrs, int C) {
  B200_CUDA(ctx, cudaMemcpyAsync(r.corrs.p, corrs, (size_t)C * sizeof(b200_corr), cudaMemcpyHostToDevice, ctx->stream));
  B200_CUDA(ctx, cudaMemcpyAsync(r.n_corrs.p, &C, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  return B200_OK;
}

// normals of the whole scene, then SHOT352 at the keypoints d_kp[0, K)
int scene_descriptors(b200_ctx *ctx, b200_cloud *scene, const b200_shot_params *p, const float4 *d_kp, int K,
                      float *d_normals, float *d_desc) {
  B200_TRY(dev_normals(ctx, scene, scene->raw.p, scene->n, true, p->normal_k, p->normal_radius, nullptr, d_normals));
  return dev_shot(ctx, scene, d_normals, d_kp, K, p->descr_radius, d_desc, nullptr, false);
}

// The Hough branch after the correspondence search (SHOT and FPFH pipelines): BOARD frames of the scene keypoints
// over `surface` and its normals, drawn from the model's recorded rand() state, then Hough3DGrouping with the model's
// votes.  d_rf_out nullable; d_status: see dev_hough3d.
int hough_branch(b200_ctx *ctx, const b200_model *model, b200_cloud *surface, const float *d_normals,
                 const float4 *d_kp, int Ks, const b200_hough_params *h, const b200_corr *d_corrs, const int *d_n_corrs,
                 const InstanceOut &out, float *d_rf_out, int *d_status) {
  DevBuf<float> rf_tmp;
  float *d_rf = d_rf_out;
  if (!d_rf) {
    B200_TRY(rf_tmp.alloc(ctx, (size_t)std::max(Ks, 1) * 9));
    d_rf = rf_tmp.p;
  }
  uint32_t stream_state[31];  // every scene starts from the model's recorded rand() state
  memcpy(stream_state, model->rand_state, sizeof(stream_state));
  B200_TRY(dev_board_lrf_from(ctx, surface, d_normals, d_kp, Ks, h->rf_radius, &h->board, stream_state, d_rf));
  return dev_hough3d(ctx, model->kp.p, model->votes.p, d_kp, d_rf, d_corrs, d_n_corrs, Ks, h->bin_size, h->threshold,
                     out, d_status);
}

// scene side of the pipeline on resident buffers: normals -> SHOT352 -> correspondence search, then
// geometric-consistency grouping (h == nullptr) or the Hough branch (BOARD frames of the scene keypoints ->
// Hough3DGrouping; d_rf_out nullable, d_status: see dev_hough3d)
int scene_pipeline(b200_ctx *ctx, const b200_model *model, b200_cloud *scene, const float4 *d_kp, int Ks,
                   const b200_shot_params *p, const InstanceOut &out, b200_corr *d_corrs, int *d_n_corrs,
                   float *d_desc_out, const b200_hough_params *h = nullptr, float *d_rf_out = nullptr,
                   int *d_status = nullptr) {
  DevBuf<float> normals, desc_tmp;
  B200_TRY(normals.alloc(ctx, (size_t)std::max(scene->n, 1) * 4));
  float *d_desc = d_desc_out;
  if (!d_desc) {
    B200_TRY(desc_tmp.alloc(ctx, (size_t)std::max(Ks, 1) * 352));
    d_desc = desc_tmp.p;
  }
  // this scene's turn for the GPU-wide stages; dev_gc / dev_hough3d end it before the latency-bound part
  WideSection wide;
  B200_TRY(wide.enter(ctx));
  B200_TRY(scene_descriptors(ctx, scene, p, d_kp, Ks, normals.p, d_desc));
  B200_TRY(dev_match(ctx, model->desc.p, model->K, d_desc, Ks, 352, p->match_mode, p->match_thr, d_corrs, d_n_corrs,
                     &model->tc));
  if (!h) return dev_gc(ctx, model->kp.p, d_kp, d_corrs, d_n_corrs, Ks, p->gc_size, p->gc_threshold, out);
  return hough_branch(ctx, model, scene, normals.p, d_kp, Ks, h, d_corrs, d_n_corrs, out, d_rf_out, d_status);
}

__global__ void unpack_points_kernel(const float4 *__restrict__ in, int n, float *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 v = in[i];
  out[(size_t)i * 3 + 0] = v.x;
  out[(size_t)i * 3 + 1] = v.y;
  out[(size_t)i * 3 + 2] = v.z;
}


int download_instances(b200_ctx *ctx, const InstanceOut &o, float *transforms, int *inst_offsets, b200_corr *inst_corrs,
                       int corr_cap, int *n_inst) {
  int found = 0;
  B200_TRY(download(ctx, &found, o.n, 1));
  B200_CUDA(ctx, ctx->sync());
  *n_inst = found;
  const int m = std::min(found, o.max_inst);
  if (inst_offsets) inst_offsets[0] = 0;
  if (m > 0) {
    std::vector<int> offs((size_t)m + 1), cnts((size_t)m);
    B200_TRY(download(ctx, offs.data(), o.offsets, (size_t)m + 1));
    B200_TRY(download(ctx, cnts.data(), o.counts, (size_t)m));
    if (transforms) B200_TRY(download(ctx, transforms, o.T, (size_t)m * 16));
    B200_CUDA(ctx, ctx->sync());
    const int used = std::min(offs[m], o.corr_cap);
    std::vector<b200_corr> all((size_t)std::max(used, 1));
    B200_TRY(download(ctx, all.data(), o.corrs, (size_t)used));
    B200_CUDA(ctx, ctx->sync());
    int w = 0;
    bool overflow = false;
    for (int i = 0; i < m; ++i) {
      for (int j = 0; j < cnts[i]; ++j) {
        if (inst_corrs && w < corr_cap)
          inst_corrs[w] = all[(size_t)offs[i] + j];
        else if (inst_corrs)
          overflow = true;
        ++w;
      }
      if (inst_offsets) inst_offsets[i + 1] = std::min(w, corr_cap);
    }
    if (overflow) return ctx->fail(B200_ERR_CAPACITY, "gc: inst_corrs capacity too small");
  }
  if (found > o.max_inst) return ctx->fail(B200_ERR_CAPACITY, "gc: more instances than max_inst");
  return B200_OK;
}

// An optional per-keypoint output of a scene registration (frames, descriptors): n floats, skipped when host is null.
struct ExtraOut {
  float *host;
  const float *dev;
  size_t n;
};

// Host side of a scene registration: the correspondence count (with d_status, the Hough status too) and one wait,
// then the correspondence list, the per-keypoint outputs, and the instances.
int download_result(b200_ctx *ctx, const ResultBufs &r, const int *d_status, std::initializer_list<ExtraOut> extras,
                    float *transforms, int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int *n_inst,
                    b200_corr *corrs_out, int *n_corrs) {
  int nc = 0, status = B200_OK;
  B200_TRY(download(ctx, &nc, r.n_corrs.p, 1));
  if (d_status) B200_TRY(download(ctx, &status, d_status, 1));
  B200_CUDA(ctx, ctx->sync());
  if (n_corrs) *n_corrs = nc;
  if (corrs_out) B200_TRY(download(ctx, corrs_out, r.corrs.p, (size_t)nc));
  for (const ExtraOut &x : extras)
    if (x.host) B200_TRY(download(ctx, x.host, x.dev, x.n));
  if (status == B200_ERR_CAPACITY) {
    B200_CUDA(ctx, ctx->sync());  // the downloads above land before the call returns
    return ctx->fail(B200_ERR_CAPACITY, "hough3d: more than 2^27 bins (bin size too small)");
  }
  return download_instances(ctx, r.out(), transforms, inst_offsets, inst_corrs, corr_cap, n_inst);
}


}  // namespace

extern "C" {

int b200_abi_version(void) { return B200REG_ABI_VERSION; }

const char *b200_last_error(const b200_ctx *ctx) { return ctx ? ctx->err.c_str() : g_error.c_str(); }

int b200_ctx_create(b200_ctx **out, int device, void *stream) {
  if (!out) {
    g_error = "b200_ctx_create: null output";
    return B200_ERR_INVALID;
  }
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    g_error = std::string("no CUDA device available (") + cudaGetErrorString(e) + "); libb200reg has no CPU fallback";
    return B200_ERR_NODEVICE;
  }
  if (device < 0 || device >= count) {
    g_error = "b200_ctx_create: device index out of range";
    return B200_ERR_INVALID;
  }
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    g_error = std::string("cudaSetDevice/cudaGetDeviceProperties failed: ") + cudaGetErrorString(e);
    return B200_ERR_CUDA;
  }
  if (prop.major != 10) {
    g_error = "libb200reg is built for sm_100a only; device is " + std::string(prop.name);
    return B200_ERR_NODEVICE;
  }
  b200_ctx *ctx = new (std::nothrow) b200_ctx();
  if (!ctx) return B200_ERR_NOMEM;
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  if (stream) {
    ctx->stream = (cudaStream_t)stream;
  } else {
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
      g_error = std::string("cudaStreamCreate failed: ") + cudaGetErrorString(e);
      delete ctx;
      return B200_ERR_CUDA;
    }
    ctx->own_stream = true;
  }
  *out = ctx;
  return B200_OK;
}

int b200_ctx_destroy(b200_ctx *ctx) {
  if (!ctx) return B200_OK;
  cudaSetDevice(ctx->device);
  ctx->sync();
  for (auto &ev : ctx->stage_events) {
    cudaEventDestroy(ev.a);
    cudaEventDestroy(ev.b);
  }
  for (auto e : ctx->event_pool) cudaEventDestroy(e);
  comm_destroy(ctx);
  ctx->arena_destroy();
  if (ctx->mt_state) cudaFree(ctx->mt_state);
  if (ctx->mailbox_host) cudaFreeHost(ctx->mailbox_host);
  if (ctx->board_draws) cudaFreeHost(ctx->board_draws);
  if (ctx->sync_ev) cudaEventDestroy(ctx->sync_ev);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return B200_OK;
}

int b200_ctx_set_blocking_sync(b200_ctx *ctx, int enable) {
  API_ENTER(ctx);
  ctx->blocking_sync = enable != 0;
  return B200_OK;
}

int b200_ctx_sync(b200_ctx *ctx) {
  API_ENTER(ctx);
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

int64_t b200_ctx_launch_count(const b200_ctx *ctx) { return ctx ? ctx->launches : 0; }

static int resolve_stage_events(b200_ctx *ctx) {
  B200_CUDA(ctx, ctx->sync());
  for (auto &ev : ctx->stage_events) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) {
      ctx->stage_ms[ev.stage] += ms;
      ctx->stage_n[ev.stage] += 1;
    }
    ctx->event_pool.push_back(ev.a);
    ctx->event_pool.push_back(ev.b);
  }
  ctx->stage_events.clear();
  return B200_OK;
}

int b200_ctx_set_profiling(b200_ctx *ctx, int enable) {
  API_ENTER(ctx);
  ctx->profiling = enable != 0;
  return B200_OK;
}

int b200_ctx_reset_profiling(b200_ctx *ctx) {
  API_ENTER(ctx);
  B200_TRY(resolve_stage_events(ctx));
  for (int i = 0; i < ST_COUNT; ++i) {
    ctx->stage_ms[i] = 0.0;
    ctx->stage_n[i] = 0;
  }
  return B200_OK;
}

int b200_ctx_stage_count(void) { return ST_COUNT; }

const char *b200_ctx_stage_name(int stage) {
  static const char *names[ST_COUNT] = {"grid_build", "normals", "neighbor_count", "shot", "fpfh",
                                        "match",      "gc_sort", "gc_adjacency",   "gc_group", "gc_ransac",
                                        "match_filter", "board", "hough"};
  return (stage >= 0 && stage < ST_COUNT) ? names[stage] : "";
}

int b200_ctx_stage_time(b200_ctx *ctx, int stage, double *total_ms, int *calls) {
  API_ENTER(ctx);
  if (stage < 0 || stage >= ST_COUNT) return ctx->fail(B200_ERR_INVALID, "stage out of range");
  B200_TRY(resolve_stage_events(ctx));
  if (total_ms) *total_ms = ctx->stage_ms[stage];
  if (calls) *calls = ctx->stage_n[stage];
  return B200_OK;
}

int b200_last_match_fallback(b200_ctx *ctx, int *rows) {
  API_ENTER(ctx);
  B200_CUDA(ctx, ctx->sync());
  if (rows) *rows = ctx->last_match_fallback;
  return B200_OK;
}

int b200_last_match_pass1_rows(b200_ctx *ctx, int *rows) {
  API_ENTER(ctx);
  B200_CUDA(ctx, ctx->sync());
  if (rows) *rows = ctx->last_match_pass1_fail;
  return B200_OK;
}

int b200_last_match_error_ratio(b200_ctx *ctx, float *ratio) {
  API_ENTER(ctx);
  B200_CUDA(ctx, ctx->sync());
  if (ratio) *ratio = ctx->last_match_err_ratio;
  return B200_OK;
}

int b200_last_neighbor_stats(const b200_ctx *ctx, double *mean_nbrs, int *max_nbrs) {
  if (!ctx) return B200_ERR_INVALID;
  if (mean_nbrs) *mean_nbrs = ctx->last_mean_nbrs;
  if (max_nbrs) *max_nbrs = ctx->last_max_nbrs;
  return B200_OK;
}

/* ------------------------------------------------------------------ surface */
int b200_cloud_create(b200_ctx *ctx, const float *xyz, int n, int stride, b200_cloud **out) {
  API_ENTER(ctx);
  return cloud_create(ctx, xyz, n, stride, false, out);
}

int b200_dev_cloud_create(b200_ctx *ctx, const float *d_xyz, int n, int stride, b200_cloud **out) {
  API_ENTER(ctx);
  return cloud_create(ctx, d_xyz, n, stride, true, out);
}

int b200_cloud_destroy(b200_cloud *cloud) {
  if (!cloud) return B200_OK;
  cudaSetDevice(cloud->ctx->device);
  delete cloud;
  return B200_OK;
}

int b200_cloud_size(const b200_cloud *cloud) { return cloud ? cloud->n : 0; }

int b200_radius_search(b200_ctx *ctx, b200_cloud *surf, const float *q, int nq, int qstride, double radius,
                       int64_t *offsets, int *idx, float *d2, int64_t cap, int64_t *total) {
  API_ENTER(ctx);
  if (!surf || !offsets || !total || nq < 0 || !(radius > 0.0))
    return ctx->fail(B200_ERR_INVALID, "radius_search: bad arguments");
  DevBuf<float4> dq;
  B200_TRY(upload_points(ctx, q, nq, qstride, dq));
  const GridView *g;
  B200_TRY(cloud_grid_for_radius(surf, radius, &g));
  DevBuf<int> counts;
  DevBuf<unsigned long long> stats;
  DevBuf<long long> offs;
  B200_TRY(counts.alloc(ctx, (size_t)std::max(nq, 1)));
  B200_TRY(stats.alloc(ctx, 2));
  B200_TRY(offs.alloc(ctx, (size_t)nq + 1));
  B200_TRY(dev_radius_count(ctx, *g, dq.p, nq, radius, counts.p, stats.p));
  if (nq > 0) {
    B200_TRY(counts_to_offsets_i64(ctx, counts.p, nq, offs.p));
  } else {
    B200_CUDA(ctx, cudaMemsetAsync(offs.p, 0, sizeof(long long), ctx->stream));
  }
  unsigned long long hstats[2];
  B200_TRY(download(ctx, hstats, stats.p, 2));
  B200_TRY(download(ctx, reinterpret_cast<long long *>(offsets), offs.p, (size_t)nq + 1));
  B200_CUDA(ctx, ctx->sync());
  *total = offsets[nq];
  if (cap < *total || !idx || !d2) {
    if (cap == 0) return B200_OK; /* sizing call */
    return ctx->fail(B200_ERR_CAPACITY, "radius_search: output capacity too small");
  }
  if (*total == 0) return B200_OK;
  DevBuf<int> didx;
  DevBuf<float> dd2;
  B200_TRY(didx.alloc(ctx, (size_t)*total));
  B200_TRY(dd2.alloc(ctx, (size_t)*total));
  B200_TRY(dev_radius_fill_sized(ctx, *g, dq.p, nq, radius, (int)hstats[0], offs.p, didx.p, dd2.p));
  B200_TRY(download(ctx, idx, didx.p, (size_t)*total));
  B200_TRY(download(ctx, d2, dd2.p, (size_t)*total));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

int b200_knn_search(b200_ctx *ctx, b200_cloud *surf, const float *q, int nq, int qstride, int k, int *idx, float *d2,
                    int *k_found) {
  API_ENTER(ctx);
  if (!surf || nq < 0 || (nq > 0 && (!idx || !d2))) return ctx->fail(B200_ERR_INVALID, "knn_search: bad arguments");
  DevBuf<float4> dq;
  B200_TRY(upload_points(ctx, q, nq, qstride, dq));
  DevBuf<int> didx;
  DevBuf<float> dd2;
  B200_TRY(didx.alloc(ctx, (size_t)std::max(nq, 1) * std::max(k, 1)));
  B200_TRY(dd2.alloc(ctx, (size_t)std::max(nq, 1) * std::max(k, 1)));
  B200_TRY(dev_knn_search(ctx, surf, dq.p, nq, k, didx.p, dd2.p, k_found));
  B200_TRY(download(ctx, idx, didx.p, (size_t)nq * k));
  B200_TRY(download(ctx, d2, dd2.p, (size_t)nq * k));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

/* ------------------------------------------------------------------ normals */
int b200_dev_normals(b200_ctx *ctx, b200_cloud *surf, const float *d_q, int nq, int qstride, int k, double radius,
                     const float *viewpoint, float *d_out) {
  API_ENTER(ctx);
  if (!surf || !d_out) return ctx->fail(B200_ERR_INVALID, "normals: bad arguments");
  if (!d_q) return dev_normals(ctx, surf, surf->raw.p, surf->n, true, k, radius, viewpoint, d_out);
  DevBuf<float4> dq;
  B200_TRY(pack_device_points(ctx, d_q, nq, qstride, dq));
  return dev_normals(ctx, surf, dq.p, nq, false, k, radius, viewpoint, d_out);
}

int b200_normals(b200_ctx *ctx, b200_cloud *surf, const float *q, int nq, int qstride, int k, double radius,
                 const float *viewpoint, float *out) {
  API_ENTER(ctx);
  if (!surf || !out) return ctx->fail(B200_ERR_INVALID, "normals: bad arguments");
  DevBuf<float> dout;
  if (!q) {
    nq = surf->n;
    B200_TRY(dout.alloc(ctx, (size_t)std::max(nq, 1) * 4));
    B200_TRY(dev_normals(ctx, surf, surf->raw.p, nq, true, k, radius, viewpoint, dout.p));
  } else {
    DevBuf<float4> dq;
    B200_TRY(upload_points(ctx, q, nq, qstride, dq));
    B200_TRY(dout.alloc(ctx, (size_t)std::max(nq, 1) * 4));
    B200_TRY(dev_normals(ctx, surf, dq.p, nq, false, k, radius, viewpoint, dout.p));
  }
  B200_TRY(download(ctx, out, dout.p, (size_t)nq * 4));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

/* ------------------------------------------------------------------ SHOT */
int b200_shot_lrf(b200_ctx *ctx, b200_cloud *surf, const float *kp, int K, int kstride, double radius, float *out) {
  API_ENTER(ctx);
  if (!surf || (K > 0 && !out)) return ctx->fail(B200_ERR_INVALID, "shot_lrf: bad arguments");
  DevBuf<float4> dkp;
  B200_TRY(upload_points(ctx, kp, K, kstride, dkp));
  DevBuf<float> drf;
  B200_TRY(drf.alloc(ctx, (size_t)std::max(K, 1) * 9));
  B200_TRY(dev_shot(ctx, surf, nullptr, dkp.p, K, radius, nullptr, drf.p, true));
  B200_TRY(download(ctx, out, drf.p, (size_t)K * 9));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

int b200_dev_shot352(b200_ctx *ctx, b200_cloud *surf, const float *d_normals, const float *d_kp, int K, int kstride,
                     double radius, float *d_desc, float *d_rf) {
  API_ENTER(ctx);
  if (!surf || !d_normals || (K > 0 && !d_desc)) return ctx->fail(B200_ERR_INVALID, "shot352: bad arguments");
  DevBuf<float4> dkp;
  B200_TRY(pack_device_points(ctx, d_kp, K, kstride, dkp));
  return dev_shot(ctx, surf, d_normals, dkp.p, K, radius, d_desc, d_rf, false);
}

int b200_shot352(b200_ctx *ctx, b200_cloud *surf, const float *normals, const float *kp, int K, int kstride,
                 double radius, float *desc, float *rf) {
  API_ENTER(ctx);
  if (!surf || !normals || (K > 0 && !desc)) return ctx->fail(B200_ERR_INVALID, "shot352: bad arguments");
  DevBuf<float4> dkp;
  B200_TRY(upload_points(ctx, kp, K, kstride, dkp));
  DevBuf<float> dn, ddesc, drf;
  B200_TRY(upload(ctx, dn, normals, (size_t)surf->n * 4));
  B200_TRY(ddesc.alloc(ctx, (size_t)std::max(K, 1) * 352));
  B200_TRY(drf.alloc(ctx, (size_t)std::max(K, 1) * 9));
  B200_TRY(dev_shot(ctx, surf, dn.p, dkp.p, K, radius, ddesc.p, drf.p, false));
  B200_TRY(download(ctx, desc, ddesc.p, (size_t)K * 352));
  if (rf) B200_TRY(download(ctx, rf, drf.p, (size_t)K * 9));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

/* ------------------------------------------------------------------ FPFH */
int b200_dev_fpfh33(b200_ctx *ctx, b200_cloud *surf, const float *d_normals, const float *d_q, int nq, int qstride,
                    double radius, float *d_out) {
  API_ENTER(ctx);
  if (!surf || !d_normals || !d_out) return ctx->fail(B200_ERR_INVALID, "fpfh33: bad arguments");
  if (!d_q) return dev_fpfh(ctx, surf, d_normals, surf->raw.p, surf->n, true, radius, d_out);
  DevBuf<float4> dq;
  B200_TRY(pack_device_points(ctx, d_q, nq, qstride, dq));
  return dev_fpfh(ctx, surf, d_normals, dq.p, nq, false, radius, d_out);
}

int b200_fpfh33(b200_ctx *ctx, b200_cloud *surf, const float *normals, const float *q, int nq, int qstride,
                double radius, float *out) {
  API_ENTER(ctx);
  if (!surf || !normals || !out) return ctx->fail(B200_ERR_INVALID, "fpfh33: bad arguments");
  DevBuf<float> dn, dout;
  B200_TRY(upload(ctx, dn, normals, (size_t)surf->n * 4));
  if (!q) {
    nq = surf->n;
    B200_TRY(dout.alloc(ctx, (size_t)std::max(nq, 1) * 33));
    B200_TRY(dev_fpfh(ctx, surf, dn.p, surf->raw.p, nq, true, radius, dout.p));
  } else {
    DevBuf<float4> dq;
    B200_TRY(upload_points(ctx, q, nq, qstride, dq));
    B200_TRY(dout.alloc(ctx, (size_t)std::max(nq, 1) * 33));
    B200_TRY(dev_fpfh(ctx, surf, dn.p, dq.p, nq, false, radius, dout.p));
  }
  B200_TRY(download(ctx, out, dout.p, (size_t)nq * 33));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

/* ------------------------------------------------------------------ matching */
int b200_dev_match(b200_ctx *ctx, const float *d_model, int Km, const float *d_scene, int Ks, int D, int mode,
                   float thr, b200_corr *d_out, int *d_count) {
  API_ENTER(ctx);
  if (!d_count || (Ks > 0 && !d_out)) return ctx->fail(B200_ERR_INVALID, "match: bad arguments");
  return dev_match(ctx, d_model, Km, d_scene, Ks, D, mode, thr, d_out, d_count);
}

int b200_match(b200_ctx *ctx, const float *model, int Km, const float *scene, int Ks, int D, int mode, float thr,
               b200_corr *out, int *count) {
  API_ENTER(ctx);
  if (!count || Km < 0 || Ks < 0 || D <= 0 || (Ks > 0 && (!out || !scene)) || (Km > 0 && !model))
    return ctx->fail(B200_ERR_INVALID, "match: bad arguments");
  DevBuf<float> dm, ds;
  DevBuf<b200_corr> dout;
  DevBuf<int> dcount;
  B200_TRY(upload(ctx, dm, model, (size_t)Km * D));
  B200_TRY(upload(ctx, ds, scene, (size_t)Ks * D));
  B200_TRY(dout.alloc(ctx, (size_t)std::max(Ks, 1)));
  B200_TRY(dcount.alloc(ctx, 1));
  B200_TRY(dev_match(ctx, dm.p, Km, ds.p, Ks, D, mode, thr, dout.p, dcount.p));
  B200_TRY(download(ctx, count, dcount.p, 1));
  B200_CUDA(ctx, ctx->sync());
  B200_TRY(download(ctx, out, dout.p, (size_t)*count));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

/* ------------------------------------------------------------------ keypoints */
int b200_dev_uniform_sampling(b200_ctx *ctx, const float *d_xyz, int n, int stride, double leaf, float *d_out_xyz,
                              int *d_out_index, int *d_count) {
  API_ENTER(ctx);
  if (n < 0 || stride < 3 || !d_count || (n > 0 && (!d_xyz || !d_out_xyz)))
    return ctx->fail(B200_ERR_INVALID, "uniform_sampling: bad arguments");
  return dev_uniform_sampling(ctx, d_xyz, n, stride, (float)leaf, d_out_xyz, d_out_index, d_count);
}

int b200_uniform_sampling(b200_ctx *ctx, const float *xyz, int n, int stride, double leaf, float *out_xyz,
                          int *out_index, int *count) {
  API_ENTER(ctx);
  if (n < 0 || stride < 3 || !count || (n > 0 && (!xyz || !out_xyz)))
    return ctx->fail(B200_ERR_INVALID, "uniform_sampling: bad arguments");
  *count = 0;
  if (n == 0) return B200_OK;
  DevBuf<float> din, dout;
  DevBuf<int> didx, dcount;
  B200_TRY(upload(ctx, din, xyz, (size_t)n * stride));
  B200_TRY(dout.alloc(ctx, (size_t)n * 3));
  B200_TRY(didx.alloc(ctx, (size_t)n));
  B200_TRY(dcount.alloc(ctx, 1));
  B200_TRY(dev_uniform_sampling(ctx, din.p, n, stride, (float)leaf, dout.p, didx.p, dcount.p));
  B200_TRY(download(ctx, count, dcount.p, 1));
  B200_CUDA(ctx, ctx->sync());
  B200_TRY(download(ctx, out_xyz, dout.p, (size_t)*count * 3));
  if (out_index) B200_TRY(download(ctx, out_index, didx.p, (size_t)*count));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

int b200_remove_nan(b200_ctx *ctx, const float *xyz, int n, int stride, float *out_xyz, int *out_index, int *count) {
  API_ENTER(ctx);
  if (n < 0 || stride < 3 || !count || (n > 0 && (!xyz || !out_xyz)))
    return ctx->fail(B200_ERR_INVALID, "remove_nan: bad arguments");
  *count = 0;
  if (n == 0) return B200_OK;
  DevBuf<float> din, dout;
  DevBuf<int> didx, dcount;
  B200_TRY(upload(ctx, din, xyz, (size_t)n * stride));
  B200_TRY(dout.alloc(ctx, (size_t)n * 3));
  B200_TRY(didx.alloc(ctx, (size_t)n));
  B200_TRY(dcount.alloc(ctx, 1));
  B200_TRY(dev_remove_nan(ctx, din.p, n, stride, dout.p, didx.p, dcount.p));
  B200_TRY(readback_small(ctx, dcount.p, count, sizeof(int)));
  B200_TRY(download(ctx, out_xyz, dout.p, (size_t)*count * 3));
  if (out_index) B200_TRY(download(ctx, out_index, didx.p, (size_t)*count));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

int b200_transform_points(b200_ctx *ctx, const float *xyz, int n, int stride, const float *transform, float *out_xyz) {
  API_ENTER(ctx);
  if (n < 0 || stride < 3 || !transform || (n > 0 && (!xyz || !out_xyz)))
    return ctx->fail(B200_ERR_INVALID, "transform_points: bad arguments");
  if (n == 0) return B200_OK;
  DevBuf<float> din, dout;
  B200_TRY(upload(ctx, din, xyz, (size_t)n * stride));
  B200_TRY(dout.alloc(ctx, (size_t)n * 3));
  B200_TRY(dev_transform_points(ctx, din.p, n, stride, transform, dout.p));
  B200_TRY(download(ctx, out_xyz, dout.p, (size_t)n * 3));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

int b200_dev_voxel_grid(b200_ctx *ctx, const float *d_xyz, int n, int stride, float lx, float ly, float lz,
                        float *d_out_xyz, int *d_count) {
  API_ENTER(ctx);
  if (n < 0 || stride < 3 || !d_count || (n > 0 && (!d_xyz || !d_out_xyz)))
    return ctx->fail(B200_ERR_INVALID, "voxel_grid: bad arguments");
  return dev_voxel_grid(ctx, d_xyz, n, stride, lx, ly, lz, d_out_xyz, d_count);
}

int b200_voxel_grid(b200_ctx *ctx, const float *xyz, int n, int stride, float lx, float ly, float lz, float *out_xyz,
                    int *count) {
  API_ENTER(ctx);
  if (n < 0 || stride < 3 || !count || (n > 0 && (!xyz || !out_xyz)))
    return ctx->fail(B200_ERR_INVALID, "voxel_grid: bad arguments");
  *count = 0;
  if (n == 0) return B200_OK;
  DevBuf<float> din, dout;
  DevBuf<int> dcount;
  B200_TRY(upload(ctx, din, xyz, (size_t)n * stride));
  B200_TRY(dout.alloc(ctx, (size_t)n * 3));
  B200_TRY(dcount.alloc(ctx, 1));
  B200_TRY(dev_voxel_grid(ctx, din.p, n, stride, lx, ly, lz, dout.p, dcount.p));
  B200_TRY(download(ctx, count, dcount.p, 1));
  B200_CUDA(ctx, ctx->sync());
  B200_TRY(download(ctx, out_xyz, dout.p, (size_t)*count * 3));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

/* ------------------------------------------------------------------ grouping */
int b200_gc_recognize(b200_ctx *ctx, const float *model_kp, int Km, int mstride, const float *scene_kp, int Ks,
                      int sstride, const b200_corr *corrs, int C, double gc_size, int gc_threshold, float *transforms,
                      int max_inst, int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int *n_inst) {
  API_ENTER(ctx);
  if (!n_inst || C < 0 || max_inst < 1 || (C > 0 && !corrs))
    return ctx->fail(B200_ERR_INVALID, "gc_recognize: bad arguments");
  *n_inst = 0;
  if (inst_offsets) inst_offsets[0] = 0;
  if (C == 0) {
    // PCL: "no correspondences" → recognize() returns without instances
    return B200_OK;
  }
  for (int i = 0; i < C; ++i)
    if (corrs[i].index_query < 0 || corrs[i].index_query >= Km || corrs[i].index_match < 0 ||
        corrs[i].index_match >= Ks)
      return ctx->fail(B200_ERR_INVALID, "gc_recognize: correspondence index out of range");
  DevBuf<float4> dm, ds;
  B200_TRY(upload_points(ctx, model_kp, Km, mstride, dm));
  B200_TRY(upload_points(ctx, scene_kp, Ks, sstride, ds));
  ResultBufs r;
  B200_TRY(r.alloc(ctx, C, max_inst));
  B200_TRY(upload_corrs(ctx, r, corrs, C));
  B200_TRY(dev_gc(ctx, dm.p, ds.p, r.corrs.p, r.n_corrs.p, C, gc_size, gc_threshold, r.out()));
  return download_instances(ctx, r.out(), transforms, inst_offsets, inst_corrs, corr_cap, n_inst);
}

int b200_hough3d_recognize(b200_ctx *ctx, const float *model_kp, const float *model_rf, int Km, int mstride,
                           const float *scene_kp, const float *scene_rf, int Ks, int sstride, const b200_corr *corrs, int C,
                           double bin_size, double threshold, float *transforms, int max_inst, int *inst_offsets,
                           b200_corr *inst_corrs, int corr_cap, int *n_inst) {
  API_ENTER(ctx);
  if (!n_inst || C < 0 || max_inst < 1 || (C > 0 && (!corrs || !model_rf || !scene_rf)))
    return ctx->fail(B200_ERR_INVALID, "hough3d_recognize: bad arguments");
  *n_inst = 0;
  if (inst_offsets) inst_offsets[0] = 0;
  if (C == 0) return B200_OK;
  for (int i = 0; i < C; ++i)
    if (corrs[i].index_query < 0 || corrs[i].index_query >= Km || corrs[i].index_match < 0 ||
        corrs[i].index_match >= Ks)
      return ctx->fail(B200_ERR_INVALID, "hough3d_recognize: correspondence index out of range");
  if (!(bin_size > 0.0)) return ctx->fail(B200_ERR_INVALID, "hough3d: bin size must be > 0");
  DevBuf<float4> dm, ds;
  DevBuf<float> dmrf, dsrf, dvotes;
  B200_TRY(upload_points(ctx, model_kp, Km, mstride, dm));
  B200_TRY(upload_points(ctx, scene_kp, Ks, sstride, ds));
  B200_TRY(upload(ctx, dmrf, model_rf, (size_t)Km * 9));
  B200_TRY(upload(ctx, dsrf, scene_rf, (size_t)Ks * 9));
  B200_TRY(dvotes.alloc(ctx, (size_t)std::max(Km, 1) * 3));
  B200_TRY(dev_hough_model_votes(ctx, dm.p, dmrf.p, Km, dvotes.p));
  ResultBufs r;
  DevBuf<int> dstatus;
  B200_TRY(r.alloc(ctx, C, max_inst));
  B200_TRY(upload_corrs(ctx, r, corrs, C));
  B200_TRY(dstatus.alloc(ctx, 1));
  B200_TRY(dev_hough3d(ctx, dm.p, dvotes.p, ds.p, dsrf.p, r.corrs.p, r.n_corrs.p, C, bin_size, threshold, r.out(),
                       dstatus.p));
  int status = B200_OK;
  B200_TRY(readback_small(ctx, dstatus.p, &status, sizeof(int)));
  if (status == B200_ERR_CAPACITY) return ctx->fail(B200_ERR_CAPACITY, "hough3d: more than 2^27 bins (bin size too small)");
  return download_instances(ctx, r.out(), transforms, inst_offsets, inst_corrs, corr_cap, n_inst);
}

/* ------------------------------------------------------------------ BOARD frames */
void b200_board_params_default(b200_board_params *p) {
  if (!p) return;
  p->find_holes = 0;
  p->tangent_radius = 0.0f;
  p->margin_thresh = 0.85f;
  p->check_margin_array_size = 24;
  p->hole_size_prob_thresh = 0.2f;
  p->steep_thresh = 0.1f;
}

int b200_ctx_srand(b200_ctx *ctx, unsigned seed) {
  API_ENTER(ctx);
  board_rand_seed(ctx, seed);
  return B200_OK;
}

int b200_board_lrf(b200_ctx *ctx, b200_cloud *surface, const float *normals, const float *kp, int K, int kstride,
                   double radius, const b200_board_params *p, float *rf) {
  API_ENTER(ctx);
  if (!surface || !normals || !p || K < 0 || (K > 0 && !rf)) return ctx->fail(B200_ERR_INVALID, "board_lrf: bad arguments");
  DevBuf<float4> dkp;
  B200_TRY(upload_points(ctx, kp, K, kstride, dkp));
  DevBuf<float> dn, drf;
  B200_TRY(upload(ctx, dn, normals, (size_t)surface->n * 4));
  B200_TRY(drf.alloc(ctx, (size_t)std::max(K, 1) * 9));
  B200_TRY(dev_board_lrf(ctx, surface, dn.p, dkp.p, K, radius, p, drf.p));
  B200_TRY(download(ctx, rf, drf.p, (size_t)K * 9));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

/* ------------------------------------------------------------------ pose refinement */
int b200_icp_align(b200_ctx *ctx, const float *source, int ns, int sstride, b200_cloud *target, int max_iterations,
                   double max_corr_dist, double transformation_epsilon, double euclidean_fitness_epsilon,
                   const float *guess, float *final_transform, float *aligned, double *fitness, int *converged,
                   int *iterations) {
  API_ENTER(ctx);
  if (!target || !final_transform || ns < 0 || max_iterations < 0)
    return ctx->fail(B200_ERR_INVALID, "icp_align: bad arguments");
  DevBuf<float4> dsrc, dal;
  B200_TRY(upload_points(ctx, source, ns, sstride, dsrc));
  if (aligned) B200_TRY(dal.alloc(ctx, (size_t)std::max(ns, 1)));
  B200_TRY(dev_icp_align(ctx, dsrc.p, ns, target, max_iterations, max_corr_dist, transformation_epsilon,
                         euclidean_fitness_epsilon, guess, final_transform, aligned ? dal.p : nullptr, fitness, converged,
                         iterations));
  if (aligned && ns > 0) {
    std::vector<float4> h((size_t)ns);
    B200_TRY(download(ctx, h.data(), dal.p, (size_t)ns));
    B200_CUDA(ctx, ctx->sync());
    for (int i = 0; i < ns; ++i) {
      aligned[3 * i + 0] = h[i].x;
      aligned[3 * i + 1] = h[i].y;
      aligned[3 * i + 2] = h[i].z;
    }
  }
  return B200_OK;
}

/* ------------------------------------------------------------------ resident pipeline */
}  // extern "C"

namespace {
// The Hough side of a model (SHOT and FPFH): the BOARD frames of its keypoints over `surface` and its normals, drawn
// from ctx's rand() stream (a context never seeded is srand(1)), the stream's state after them, and
// Hough3DGrouping::train()'s votes.
int model_frames(b200_ctx *ctx, b200_model *m, b200_cloud *surface, const float *d_normals, const b200_hough_params *h) {
  if (!ctx->rand_seeded) board_rand_seed(ctx, 1u);
  B200_TRY(m->rf.alloc(ctx, (size_t)std::max(m->K, 1) * 9));
  B200_TRY(m->votes.alloc(ctx, (size_t)std::max(m->K, 1) * 3));
  B200_TRY(dev_board_lrf(ctx, surface, d_normals, m->kp.p, m->K, h->rf_radius, &h->board, m->rf.p));
  B200_TRY(dev_hough_model_votes(ctx, m->kp.p, m->rf.p, m->K, m->votes.p));
  memcpy(m->rand_state, ctx->rand_state, sizeof(m->rand_state));
  m->has_frames = true;
  return B200_OK;
}

// normals + SHOT352 of the model keypoints; with h, also their BOARD frames and the Hough votes (model_frames)
int model_create(b200_ctx *ctx, const float *xyz, int n, int stride, const float *kp, int K, int kstride,
                 const b200_shot_params *p, const b200_hough_params *h, b200_model **out) {
  if (!out) return ctx->fail(B200_ERR_INVALID, "model_create: null output");
  B200_TRY(check_params(ctx, p));
  if (h) B200_TRY(check_hough_params(ctx, h));
  std::unique_ptr<b200_cloud> cloud;
  B200_TRY(cloud_upload(ctx, xyz, n, stride, false, cloud));
  std::unique_ptr<b200_model> m(new (std::nothrow) b200_model());
  if (!m) return ctx->fail(B200_ERR_NOMEM, "model_create: out of host memory");
  m->ctx = ctx;
  m->K = K;
  DevBuf<float> normals;
  B200_TRY(normals.alloc(ctx, (size_t)std::max(n, 1) * 4));
  B200_TRY(dev_normals(ctx, cloud.get(), cloud->raw.p, n, true, p->normal_k, p->normal_radius, nullptr, normals.p));
  B200_TRY(upload_points(ctx, kp, K, kstride, m->kp));
  B200_TRY(m->desc.alloc(ctx, (size_t)std::max(K, 1) * 352));
  B200_TRY(dev_shot(ctx, cloud.get(), normals.p, m->kp.p, K, p->descr_radius, m->desc.p, nullptr, false));
  B200_TRY(match_prepare_model(ctx, m.get()));
  if (h) B200_TRY(model_frames(ctx, m.get(), cloud.get(), normals.p, h));
  B200_CUDA(ctx, ctx->sync());
  *out = m.release();
  return B200_OK;
}
}  // namespace

extern "C" {

int b200_model_create_shot(b200_ctx *ctx, const float *xyz, int n, int stride, const float *kp, int K, int kstride,
                           const b200_shot_params *p, b200_model **out) {
  API_ENTER(ctx);
  return model_create(ctx, xyz, n, stride, kp, K, kstride, p, nullptr, out);
}

int b200_model_create_shot_hough(b200_ctx *ctx, const float *xyz, int n, int stride, const float *kp, int K, int kstride,
                                 const b200_shot_params *p, const b200_hough_params *h, b200_model **out) {
  API_ENTER(ctx);
  return model_create(ctx, xyz, n, stride, kp, K, kstride, p, h, out);
}

int b200_model_download_frames(b200_ctx *ctx, const b200_model *m, float *rf) {
  API_ENTER(ctx);
  if (!m || !m->has_frames) return ctx->fail(B200_ERR_INVALID, "model_download_frames: the model has no frames");
  if (m->K > 0 && !rf) return ctx->fail(B200_ERR_INVALID, "model_download_frames: null output");
  B200_TRY(download(ctx, rf, m->rf.p, (size_t)m->K * 9));
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

int b200_model_destroy(b200_model *m) {
  if (!m) return B200_OK;
  cudaSetDevice(m->ctx->device);
  delete m;
  return B200_OK;
}

int b200_model_size(const b200_model *m) { return m ? m->K : 0; }

int b200_model_download(b200_ctx *ctx, const b200_model *m, float *desc, float *kp) {
  API_ENTER(ctx);
  if (!m) return ctx->fail(B200_ERR_INVALID, "model_download: null model");
  if (desc) B200_TRY(download(ctx, desc, m->desc.p, (size_t)m->K * m->D));
  DevBuf<float> tmp;
  if (kp && m->K > 0) {
    B200_TRY(tmp.alloc(ctx, (size_t)m->K * 3));
    unpack_points_kernel<<<ceil_div(m->K, 256), 256, 0, ctx->stream>>>(m->kp.p, m->K, tmp.p);
    B200_LAUNCHED(ctx);
    B200_TRY(download(ctx, kp, tmp.p, (size_t)m->K * 3));
  }
  B200_CUDA(ctx, ctx->sync());
  return B200_OK;
}

}  // extern "C"

namespace {
// b200_dev_register_scene_shot (h == nullptr) / b200_dev_register_scene_shot_hough
int dev_register_scene(b200_ctx *ctx, const b200_model *model, const float *d_scene_xyz, int n, int stride,
                       const float *d_scene_kp, int Ks, int kstride, const b200_shot_params *p, float *d_transforms,
                       int *d_inst_offsets, int *d_inst_counts, b200_corr *d_inst_corrs, int corr_cap, int *d_n_inst,
                       b200_corr *d_corrs_out, int *d_n_corrs, float *d_desc_out, const b200_hough_params *h,
                       float *d_rf_out, int *d_status) {
  if (!model || !d_transforms || !d_inst_offsets || !d_inst_counts || !d_inst_corrs || !d_n_inst || !d_corrs_out ||
      !d_n_corrs || Ks < 0 || (h && !d_status))
    return ctx->fail(B200_ERR_INVALID, "register_scene: bad arguments");
  B200_TRY(check_registration(ctx, model, p, h));
  const InstanceOut out = {d_transforms, p->max_instances, d_inst_offsets, d_inst_counts, d_inst_corrs, corr_cap,
                           d_n_inst};
  std::unique_ptr<b200_cloud> scene;
  B200_TRY(cloud_upload(ctx, d_scene_xyz, n, stride, true, scene));
  DevBuf<float4> dkp;
  B200_TRY(pack_device_points(ctx, d_scene_kp, Ks, kstride, dkp));
  return scene_pipeline(ctx, model, scene.get(), dkp.p, Ks, p, out, d_corrs_out, d_n_corrs, d_desc_out, h, d_rf_out,
                        d_status);
}

// b200_register_scene_shot (h == nullptr) / b200_register_scene_shot_hough
int register_scene(b200_ctx *ctx, const b200_model *model, const float *scene_xyz, int n, int stride,
                   const float *scene_kp, int Ks, int kstride, const b200_shot_params *p, float *transforms,
                   int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int *n_inst, b200_corr *corrs_out,
                   int *n_corrs, const b200_hough_params *h, float *rf_out) {
  if (!model || !n_inst || Ks < 0) return ctx->fail(B200_ERR_INVALID, "register_scene: bad arguments");
  B200_TRY(check_registration(ctx, model, p, h));
  *n_inst = 0;
  if (n_corrs) *n_corrs = 0;
  HostTrace tr;
  std::unique_ptr<b200_cloud> scene;
  B200_TRY(cloud_upload(ctx, scene_xyz, n, stride, false, scene));
  tr.tick("e2e cloud_upload");
  DevBuf<float4> dkp;
  B200_TRY(upload_points(ctx, scene_kp, Ks, kstride, dkp));
  const int cap = std::max(Ks, 1);
  ResultBufs r;
  DevBuf<int> dstatus;
  DevBuf<float> drf;
  B200_TRY(r.alloc(ctx, cap, p->max_instances));
  if (h) {
    B200_TRY(dstatus.alloc(ctx, 1));
    B200_TRY(drf.alloc(ctx, (size_t)cap * 9));
  }
  B200_TRY(scene_pipeline(ctx, model, scene.get(), dkp.p, Ks, p, r.out(), r.corrs.p, r.n_corrs.p, nullptr, h, drf.p,
                          dstatus.p));
  tr.tick("e2e pipeline issue");
  B200_TRY(download_result(ctx, r, dstatus.p, {{rf_out, drf.p, (size_t)Ks * 9}}, transforms, inst_offsets, inst_corrs,
                           corr_cap, n_inst, corrs_out, n_corrs));
  tr.tick("e2e download");
  return B200_OK;
}
}  // namespace

extern "C" {

int b200_dev_register_scene_shot(b200_ctx *ctx, const b200_model *model, const float *d_scene_xyz, int n, int stride,
                                 const float *d_scene_kp, int Ks, int kstride, const b200_shot_params *p,
                                 float *d_transforms, int *d_inst_offsets, int *d_inst_counts,
                                 b200_corr *d_inst_corrs, int corr_cap, int *d_n_inst, b200_corr *d_corrs_out,
                                 int *d_n_corrs, float *d_desc_out) {
  API_ENTER(ctx);
  return dev_register_scene(ctx, model, d_scene_xyz, n, stride, d_scene_kp, Ks, kstride, p, d_transforms, d_inst_offsets,
                            d_inst_counts, d_inst_corrs, corr_cap, d_n_inst, d_corrs_out, d_n_corrs, d_desc_out, nullptr,
                            nullptr, nullptr);
}
int b200_dev_register_scene_shot_hough(b200_ctx *ctx, const b200_model *model, const float *d_scene_xyz, int n,
                                       int stride, const float *d_scene_kp, int Ks, int kstride,
                                       const b200_shot_params *p, const b200_hough_params *h, float *d_transforms,
                                       int *d_inst_offsets, int *d_inst_counts, b200_corr *d_inst_corrs, int corr_cap,
                                       int *d_n_inst, b200_corr *d_corrs_out, int *d_n_corrs, float *d_desc_out,
                                       float *d_rf_out, int *d_status) {
  API_ENTER(ctx);
  if (!h) return ctx->fail(B200_ERR_INVALID, "null Hough params");
  return dev_register_scene(ctx, model, d_scene_xyz, n, stride, d_scene_kp, Ks, kstride, p, d_transforms, d_inst_offsets,
                            d_inst_counts, d_inst_corrs, corr_cap, d_n_inst, d_corrs_out, d_n_corrs, d_desc_out, h,
                            d_rf_out, d_status);
}

int b200_register_scene_shot(b200_ctx *ctx, const b200_model *model, const float *scene_xyz, int n, int stride,
                             const float *scene_kp, int Ks, int kstride, const b200_shot_params *p, float *transforms,
                             int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int *n_inst, b200_corr *corrs_out,
                             int *n_corrs) {
  API_ENTER(ctx);
  return register_scene(ctx, model, scene_xyz, n, stride, scene_kp, Ks, kstride, p, transforms, inst_offsets, inst_corrs,
                        corr_cap, n_inst, corrs_out, n_corrs, nullptr, nullptr);
}

int b200_register_scene_shot_hough(b200_ctx *ctx, const b200_model *model, const float *scene_xyz, int n, int stride,
                                   const float *scene_kp, int Ks, int kstride, const b200_shot_params *p,
                                   const b200_hough_params *h, float *transforms, int *inst_offsets,
                                   b200_corr *inst_corrs, int corr_cap, int *n_inst, b200_corr *corrs_out, int *n_corrs,
                                   float *rf_out) {
  API_ENTER(ctx);
  if (!h) return ctx->fail(B200_ERR_INVALID, "null Hough params");
  return register_scene(ctx, model, scene_xyz, n, stride, scene_kp, Ks, kstride, p, transforms, inst_offsets, inst_corrs,
                        corr_cap, n_inst, corrs_out, n_corrs, h, rf_out);
}

/* ------------------------------------------------------------------ resident FPFH pipeline */
// FPFH_demo.cpp:405-538 with the model side resident: the reference estimates normals ON the keypoint clouds by radius
// (:416-420, :486-492) and runs FPFHEstimation with input = surface = the keypoint cloud (:422-428, :505-510).
namespace {
int fpfh_side(b200_ctx *ctx, b200_cloud *cloud, const b200_shot_params *p, DevBuf<float> &desc) {
  DevBuf<float> normals;
  B200_TRY(normals.alloc(ctx, (size_t)std::max(cloud->n, 1) * 4));
  B200_TRY(desc.alloc(ctx, (size_t)std::max(cloud->n, 1) * 33));
  B200_TRY(dev_normals(ctx, cloud, cloud->raw.p, cloud->n, true, p->normal_k, p->normal_radius, nullptr, normals.p));
  return dev_fpfh(ctx, cloud, normals.p, cloud->raw.p, cloud->n, true, p->descr_radius, desc.p);
}

// b200_model_create_fpfh (h == nullptr) / b200_model_create_fpfh_hough: with h, also the BOARD frames of the
// keypoints over the dense cloud `surface` and the Hough votes (model_frames)
int model_create_fpfh(b200_ctx *ctx, const float *kp, int K, int kstride, const b200_shot_params *p,
                      const DenseSurface *surface, const b200_hough_params *h, b200_model **out) {
  if (!out) return ctx->fail(B200_ERR_INVALID, "model_create_fpfh: null output");
  B200_TRY(check_params(ctx, p));
  if (h) {
    B200_TRY(check_hough_params(ctx, h));
    B200_TRY(surface->check(ctx));
  }
  std::unique_ptr<b200_cloud> cloud;
  B200_TRY(cloud_upload(ctx, kp, K, kstride, false, cloud));
  std::unique_ptr<b200_model> m(new (std::nothrow) b200_model());
  if (!m) return ctx->fail(B200_ERR_NOMEM, "model_create_fpfh: out of host memory");
  m->ctx = ctx;
  m->K = K;
  m->D = 33;
  B200_TRY(fpfh_side(ctx, cloud.get(), p, m->desc));
  B200_TRY(m->kp.alloc(ctx, (size_t)std::max(K, 1)));
  if (K > 0)
    B200_CUDA(ctx, cudaMemcpyAsync(m->kp.p, cloud->raw.p, (size_t)K * sizeof(float4), cudaMemcpyDeviceToDevice,
                                   ctx->stream));
  B200_TRY(match_prepare_model(ctx, m.get()));
  if (h) {
    std::unique_ptr<b200_cloud> dense;
    DevBuf<float> normals;
    B200_TRY(surface->upload(ctx, dense, normals));
    B200_TRY(model_frames(ctx, m.get(), dense.get(), normals.p, h));
  }
  B200_CUDA(ctx, ctx->sync());
  *out = m.release();
  return B200_OK;
}

// b200_register_scene_fpfh (h == nullptr: GC grouping) / b200_register_scene_fpfh_hough (the Hough branch over the
// dense scene cloud `surface`; rf_out nullable)
int register_scene_fpfh(b200_ctx *ctx, const b200_model *model, const float *scene_kp, int Ks, int kstride,
                        const b200_shot_params *p, const DenseSurface *surface, const b200_hough_params *h,
                        float *transforms, int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int *n_inst,
                        b200_corr *corrs_out, int *n_corrs, float *desc_out, float *rf_out) {
  if (!model || model->D != 33 || !n_inst || Ks < 0)
    return ctx->fail(B200_ERR_INVALID, "register_scene_fpfh: bad arguments (the model must come from b200_model_create_fpfh)");
  B200_TRY(check_params(ctx, p));
  if (h) {
    B200_TRY(check_hough_params(ctx, h));
    if (!model->has_frames)
      return ctx->fail(B200_ERR_INVALID, "register_scene_fpfh_hough: the model has no frames (b200_model_create_fpfh_hough)");
    B200_TRY(surface->check(ctx));
  }
  *n_inst = 0;
  if (n_corrs) *n_corrs = 0;
  std::unique_ptr<b200_cloud> scene;
  B200_TRY(cloud_upload(ctx, scene_kp, Ks, kstride, false, scene));
  DevBuf<float> desc;
  ResultBufs r;
  B200_TRY(fpfh_side(ctx, scene.get(), p, desc));
  B200_TRY(r.alloc(ctx, std::max(Ks, 1), p->max_instances));
  B200_TRY(dev_match(ctx, model->desc.p, model->K, desc.p, Ks, 33, p->match_mode, p->match_thr, r.corrs.p, r.n_corrs.p,
                     &model->tc));
  std::unique_ptr<b200_cloud> dense;
  DevBuf<float> normals, rf;
  DevBuf<int> status;
  if (!h) {
    B200_TRY(dev_gc(ctx, model->kp.p, scene->raw.p, r.corrs.p, r.n_corrs.p, Ks, p->gc_size, p->gc_threshold, r.out()));
  } else {
    B200_TRY(surface->upload(ctx, dense, normals));
    B200_TRY(rf.alloc(ctx, (size_t)std::max(Ks, 1) * 9));
    B200_TRY(status.alloc(ctx, 1));
    B200_TRY(hough_branch(ctx, model, dense.get(), normals.p, scene->raw.p, Ks, h, r.corrs.p, r.n_corrs.p, r.out(),
                          rf.p, status.p));
  }
  return download_result(ctx, r, status.p, {{desc_out, desc.p, (size_t)Ks * 33}, {rf_out, rf.p, (size_t)Ks * 9}},
                         transforms, inst_offsets, inst_corrs, corr_cap, n_inst, corrs_out, n_corrs);
}
}  // namespace

int b200_model_create_fpfh(b200_ctx *ctx, const float *kp, int K, int kstride, const b200_shot_params *p,
                           b200_model **out) {
  API_ENTER(ctx);
  return model_create_fpfh(ctx, kp, K, kstride, p, nullptr, nullptr, out);
}

int b200_model_create_fpfh_hough(b200_ctx *ctx, const float *xyz, int n, int stride, const float *kp, int K,
                                 int kstride, const b200_shot_params *p, int surface_normal_k,
                                 double surface_normal_radius, const b200_hough_params *h, b200_model **out) {
  API_ENTER(ctx);
  if (!h) return ctx->fail(B200_ERR_INVALID, "null Hough params");
  const DenseSurface surface = {xyz, n, stride, surface_normal_k, surface_normal_radius};
  return model_create_fpfh(ctx, kp, K, kstride, p, &surface, h, out);
}

int b200_model_descriptor_length(const b200_model *m) { return m ? m->D : 0; }

int b200_register_scene_fpfh(b200_ctx *ctx, const b200_model *model, const float *scene_kp, int Ks, int kstride,
                             const b200_shot_params *p, float *transforms, int *inst_offsets, b200_corr *inst_corrs,
                             int corr_cap, int *n_inst, b200_corr *corrs_out, int *n_corrs, float *desc_out) {
  API_ENTER(ctx);
  return register_scene_fpfh(ctx, model, scene_kp, Ks, kstride, p, nullptr, nullptr, transforms, inst_offsets,
                             inst_corrs, corr_cap, n_inst, corrs_out, n_corrs, desc_out, nullptr);
}

int b200_register_scene_fpfh_hough(b200_ctx *ctx, const b200_model *model, const float *scene_xyz, int n, int stride,
                                   const float *scene_kp, int Ks, int kstride, const b200_shot_params *p,
                                   int surface_normal_k, double surface_normal_radius, const b200_hough_params *h,
                                   float *transforms, int *inst_offsets, b200_corr *inst_corrs, int corr_cap,
                                   int *n_inst, b200_corr *corrs_out, int *n_corrs, float *desc_out, float *rf_out) {
  API_ENTER(ctx);
  if (!h) return ctx->fail(B200_ERR_INVALID, "null Hough params");
  const DenseSurface surface = {scene_xyz, n, stride, surface_normal_k, surface_normal_radius};
  return register_scene_fpfh(ctx, model, scene_kp, Ks, kstride, p, &surface, h, transforms, inst_offsets, inst_corrs,
                             corr_cap, n_inst, corrs_out, n_corrs, desc_out, rf_out);
}

/* ------------------------------------------------------------------ multi-GPU (comm.cu) */
int b200_comm_unique_id(void *id128, size_t bytes) {
  std::string err;
  const int rc = comm_unique_id(id128, bytes, &err);
  if (rc != B200_OK) g_error = err;
  return rc;
}

int b200_comm_init(b200_ctx *ctx, const void *id128, int rank, int world) {
  API_ENTER(ctx);
  return comm_init(ctx, id128, rank, world);
}

int b200_comm_destroy(b200_ctx *ctx) {
  API_ENTER(ctx);
  return comm_destroy(ctx);
}

int b200_comm_rank(const b200_ctx *ctx) { return ctx ? ctx->comm_rank : 0; }
int b200_comm_size(const b200_ctx *ctx) { return ctx ? ctx->comm_world : 1; }

int b200_gather_correspondences(b200_ctx *ctx, const b200_corr *d_corrs, const int *d_count, int cap,
                                b200_corr *d_gathered, int *d_counts) {
  API_ENTER(ctx);
  if (!d_corrs || !d_count || !d_gathered || !d_counts)
    return ctx->fail(B200_ERR_INVALID, "gather_correspondences: null buffer");
  return dev_gather_correspondences(ctx, d_corrs, d_count, cap, d_gathered, d_counts);
}

// One scene over all ranks of the communicator (north star: "scene keypoints are sharded across the GPUs, the model
// library replicated, correspondences gathered with NCCL"; SURVEY.md 8(e) single-large-scene mode).  Collective:
// every rank calls it; the scene and the outputs are the root's (other ranks may pass null buffers).
//   root: upload -> broadcast xyz + keypoints (NCCL) -> every rank: grid + normals of the whole scene (replicated:
//   1 M points cost about a millisecond) -> SHOT352 + correspondence search for the rank's contiguous keypoint slab
//   [Ks r / G, Ks (r + 1) / G) -> all-gather of the slab lists -> root: concatenation in rank order (= ascending scene
//   index, exactly the single-GPU list) -> grouping + RANSAC -> download.
// Every per-keypoint / per-row computation is independent of the partition, so the result is the single-GPU one
// bit for bit.
int b200_register_scene_shot_sharded(b200_ctx *ctx, const b200_model *model, int root, const float *scene_xyz, int n,
                                     int stride, const float *scene_kp, int Ks, int kstride, const b200_shot_params *p,
                                     float *transforms, int *inst_offsets, b200_corr *inst_corrs, int corr_cap,
                                     int *n_inst, b200_corr *corrs_out, int *n_corrs) {
  API_ENTER(ctx);
  const int G = ctx->comm_world, r = ctx->comm_rank;
  if (!model || root < 0 || root >= G) return ctx->fail(B200_ERR_INVALID, "register_scene_sharded: bad arguments");
  if (model->D != 352)
    return ctx->fail(B200_ERR_INVALID, "register_scene_sharded: the model is not a SHOT352 model (b200_model_create_shot)");
  B200_TRY(check_params(ctx, p));
  const bool is_root = r == root;
  if (is_root && (!n_inst || Ks < 0 || n < 0)) return ctx->fail(B200_ERR_INVALID, "register_scene_sharded: bad arguments");
  if (n_inst) *n_inst = 0;
  if (n_corrs) *n_corrs = 0;
  // sizes from the root
  DevBuf<int> dh;
  B200_TRY(dh.alloc(ctx, 4));
  int hdr[4] = {n, Ks, 0, 0};
  if (is_root) B200_TRY(write_small(ctx, dh.p, hdr, sizeof(hdr)));
  B200_TRY(comm_broadcast(ctx, dh.p, sizeof(hdr), root));
  if (!is_root) B200_TRY(readback_small(ctx, dh.p, hdr, sizeof(hdr)));
  n = hdr[0];
  Ks = hdr[1];
  DevBuf<float4> raw, dkp;
  if (is_root) {
    B200_TRY(upload_points(ctx, scene_xyz, n, stride, raw));
    B200_TRY(upload_points(ctx, scene_kp, Ks, kstride, dkp));
  } else {
    B200_TRY(raw.alloc(ctx, (size_t)std::max(n, 1)));
    B200_TRY(dkp.alloc(ctx, (size_t)std::max(Ks, 1)));
  }
  B200_TRY(comm_broadcast(ctx, raw.p, (size_t)n * sizeof(float4), root));
  B200_TRY(comm_broadcast(ctx, dkp.p, (size_t)Ks * sizeof(float4), root));
  std::unique_ptr<b200_cloud> scene;
  B200_TRY(cloud_upload(ctx, reinterpret_cast<const float *>(raw.p), n, 4, true, scene));
  const int k0 = (int)((long long)Ks * r / G), k1 = (int)((long long)Ks * (r + 1) / G);
  const int slab = k1 - k0, cap = (Ks + G - 1) / G + 1;
  DevBuf<float> normals, desc;
  DevBuf<b200_corr> dslab, dall;
  DevBuf<int> dcnt, dcounts;
  ResultBufs res;
  B200_TRY(normals.alloc(ctx, (size_t)std::max(n, 1) * 4));
  B200_TRY(desc.alloc(ctx, (size_t)std::max(slab, 1) * 352));
  B200_TRY(dslab.alloc(ctx, (size_t)cap));
  B200_TRY(dall.alloc(ctx, (size_t)cap * G));
  B200_TRY(dcnt.alloc(ctx, 1));
  B200_TRY(dcounts.alloc(ctx, (size_t)G));
  B200_TRY(scene_descriptors(ctx, scene.get(), p, dkp.p + k0, slab, normals.p, desc.p));
  B200_TRY(dev_match(ctx, model->desc.p, model->K, desc.p, slab, 352, p->match_mode, p->match_thr, dslab.p, dcnt.p,
                     &model->tc));
  B200_TRY(dev_offset_scene_index(ctx, dslab.p, dcnt.p, cap, k0));
  B200_TRY(dev_gather_correspondences(ctx, dslab.p, dcnt.p, cap, dall.p, dcounts.p));
  if (!is_root) {
    B200_CUDA(ctx, ctx->sync());
    return B200_OK;
  }
  B200_TRY(res.alloc(ctx, std::max(Ks, 1), p->max_instances));
  B200_TRY(dev_concat_lists(ctx, dall.p, dcounts.p, G, cap, res.corrs.p, res.cap, res.n_corrs.p));
  B200_TRY(dev_gc(ctx, model->kp.p, dkp.p, res.corrs.p, res.n_corrs.p, Ks, p->gc_size, p->gc_threshold, res.out()));
  return download_result(ctx, res, nullptr, {}, transforms, inst_offsets, inst_corrs, corr_cap, n_inst, corrs_out,
                         n_corrs);
}

/* ------------------------------------------------------------------ lanes */
namespace {
// contexts kept per device for b200_register_scene_batch_shot (their arenas stay warm between batches)
struct LanePool {
  std::mutex mu;
  std::vector<b200_ctx *> ctxs;
  int grow(int device, int lanes) {  // at least `lanes` contexts; the caller holds mu
    while ((int)ctxs.size() < lanes) {
      b200_ctx *c = nullptr;
      B200_TRY(b200_ctx_create(&c, device, nullptr));
      ctxs.push_back(c);
    }
    return B200_OK;
  }
};
LanePool &lane_pool(int device) {
  static LanePool pools[64];
  return pools[(device >= 0 && device < 64) ? device : 0];
}

// The lane driver of the batch calls: `lanes` pooled contexts of `device`, one host thread each; lane l registers
// scenes l, l + lanes, ... through scene(ctx, s), whose return code goes to status[s].  Returns the first status
// other than B200_OK / B200_ERR_CAPACITY (with that lane's error text), else B200_OK.
int run_lanes(int device, int n_scenes, int lanes, int *status, const std::function<int(b200_ctx *, int)> &scene) {
  if (n_scenes == 0) return B200_OK;
  lanes = std::min(lanes, n_scenes);
  LanePool &pool = lane_pool(device);
  std::lock_guard<std::mutex> hold(pool.mu);  // one batch at a time per device
  B200_TRY(pool.grow(device, lanes));
  // more lanes than host cores: sleep in the host waits instead of spinning
  const unsigned hw = std::thread::hardware_concurrency();
  for (int l = 0; l < lanes; ++l) pool.ctxs[(size_t)l]->blocking_sync = hw != 0 && (unsigned)lanes > hw;
  auto work = [&](int lane) {
    b200_ctx *c = pool.ctxs[(size_t)lane];
    for (int s = lane; s < n_scenes; s += lanes) status[s] = scene(c, s);
  };
  std::vector<std::thread> threads;
  for (int l = 1; l < lanes; ++l) threads.emplace_back(work, l);
  work(0);
  for (std::thread &t : threads) t.join();
  for (int s = 0; s < n_scenes; ++s)
    if (status[s] != B200_OK && status[s] != B200_ERR_CAPACITY) {
      g_error = std::string("register_scene_batch: scene ") + std::to_string(s) + ": " +
                b200_last_error(pool.ctxs[(size_t)(s % lanes)]);
      return status[s];
    }
  return B200_OK;
}

bool batch_args_ok(const b200_model *model, int n_scenes, const float *const *scene_xyz, const int *n_points,
                   const float *const *scene_kp, const int *n_kp, const b200_shot_params *p, int lanes, int *n_inst,
                   int *status) {
  return model && n_scenes >= 0 && lanes >= 1 && lanes <= 16 && p &&
         !(n_scenes > 0 && (!scene_xyz || !n_points || !scene_kp || !n_kp || !n_inst || !status));
}

// both batch calls: register_scene per scene, with h == nullptr for geometric-consistency grouping
int register_batch(int device, const b200_model *model, int n_scenes, const float *const *scene_xyz,
                   const int *n_points, int stride, const float *const *scene_kp, const int *n_kp, int kstride,
                   const b200_shot_params *p, const b200_hough_params *h, int lanes, float *const *transforms,
                   int *const *inst_offsets, b200_corr *const *inst_corrs, const int *corr_cap, int *n_inst,
                   b200_corr *const *corrs_out, int *n_corrs, int *status) {
  return run_lanes(device, n_scenes, lanes, status, [&](b200_ctx *c, int s) {
    int nc = 0;
    int rc = set_device(c);
    if (rc == B200_OK)
      rc = register_scene(c, model, scene_xyz[s], n_points[s], stride, scene_kp[s], n_kp[s], kstride, p,
                          transforms ? transforms[s] : nullptr, inst_offsets ? inst_offsets[s] : nullptr,
                          inst_corrs ? inst_corrs[s] : nullptr, corr_cap ? corr_cap[s] : 0, &n_inst[s],
                          corrs_out ? corrs_out[s] : nullptr, &nc, h, nullptr);
    if (n_corrs) n_corrs[s] = nc;
    return rc;
  });
}
}  // namespace

int b200_register_scene_batch_shot(int device, const b200_model *model, int n_scenes, const float *const *scene_xyz,
                                   const int *n_points, int stride, const float *const *scene_kp, const int *n_kp,
                                   int kstride, const b200_shot_params *p, int lanes, float *const *transforms,
                                   int *const *inst_offsets, b200_corr *const *inst_corrs, const int *corr_cap,
                                   int *n_inst, b200_corr *const *corrs_out, int *n_corrs, int *status) {
  if (!batch_args_ok(model, n_scenes, scene_xyz, n_points, scene_kp, n_kp, p, lanes, n_inst, status)) {
    g_error = "register_scene_batch: bad arguments";
    return B200_ERR_INVALID;
  }
  return register_batch(device, model, n_scenes, scene_xyz, n_points, stride, scene_kp, n_kp, kstride, p, nullptr, lanes,
                        transforms, inst_offsets, inst_corrs, corr_cap, n_inst, corrs_out, n_corrs, status);
}

int b200_register_scene_batch_shot_hough(int device, const b200_model *model, int n_scenes,
                                         const float *const *scene_xyz, const int *n_points, int stride,
                                         const float *const *scene_kp, const int *n_kp, int kstride,
                                         const b200_shot_params *p, const b200_hough_params *h, int lanes,
                                         float *const *transforms, int *const *inst_offsets,
                                         b200_corr *const *inst_corrs, const int *corr_cap, int *n_inst,
                                         b200_corr *const *corrs_out, int *n_corrs, int *status) {
  if (!batch_args_ok(model, n_scenes, scene_xyz, n_points, scene_kp, n_kp, p, lanes, n_inst, status) || !h) {
    g_error = "register_scene_batch_hough: bad arguments";
    return B200_ERR_INVALID;
  }
  return register_batch(device, model, n_scenes, scene_xyz, n_points, stride, scene_kp, n_kp, kstride, p, h, lanes,
                        transforms, inst_offsets, inst_corrs, corr_cap, n_inst, corrs_out, n_corrs, status);
}

int b200_lanes_release(int device) {
  LanePool &pool = lane_pool(device);
  std::lock_guard<std::mutex> hold(pool.mu);
  for (b200_ctx *c : pool.ctxs) b200_ctx_destroy(c);
  pool.ctxs.clear();
  return B200_OK;
}

/* ------------------------------------------------------------------ multi-view library */
static const std::array<float, 16> kIdentityPose = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
int b200_library_create(b200_ctx *ctx, b200_library **out) {
  API_ENTER(ctx);
  if (!out) return ctx->fail(B200_ERR_INVALID, "library_create: null output");
  b200_library *lib = new b200_library();
  lib->ctx = ctx;
  *out = lib;
  return B200_OK;
}

int b200_library_destroy(b200_library *lib) {
  if (!lib) return B200_OK;
  for (b200_model *m : lib->views) b200_model_destroy(m);
  delete lib;
  return B200_OK;
}

int b200_library_add_view(b200_ctx *ctx, b200_library *lib, const float *xyz, int n, int stride, const float *kp, int K,
                          int kstride, const b200_shot_params *p, int *view_id) {
  API_ENTER(ctx);
  if (!lib) return ctx->fail(B200_ERR_INVALID, "library_add_view: null library");
  b200_model *m = nullptr;
  B200_TRY(b200_model_create_shot(ctx, xyz, n, stride, kp, K, kstride, p, &m));
  lib->views.push_back(m);
  lib->poses.push_back(kIdentityPose);
  if (view_id) *view_id = (int)lib->views.size() - 1;
  return B200_OK;
}

int b200_library_add_view_descriptors(b200_ctx *ctx, b200_library *lib, const float *desc, const float *kp, int K,
                                      int kstride, int *view_id) {
  API_ENTER(ctx);
  if (!lib || K < 0 || (K > 0 && (!desc || !kp))) return ctx->fail(B200_ERR_INVALID, "library_add_view_descriptors: bad arguments");
  std::unique_ptr<b200_model> m(new (std::nothrow) b200_model());
  if (!m) return ctx->fail(B200_ERR_NOMEM, "library_add_view_descriptors: out of host memory");
  m->ctx = ctx;
  m->K = K;
  B200_TRY(upload(ctx, m->desc, desc, (size_t)K * 352));
  B200_TRY(upload_points(ctx, kp, K, kstride, m->kp));
  B200_TRY(match_prepare_model(ctx, m.get()));
  B200_CUDA(ctx, ctx->sync());
  lib->views.push_back(m.release());
  lib->poses.push_back(kIdentityPose);
  if (view_id) *view_id = (int)lib->views.size() - 1;
  return B200_OK;
}

int b200_library_set_view_pose(b200_library *lib, int view, const float *pose16) {
  if (!lib || !pose16 || view < 0 || view >= (int)lib->views.size()) return B200_ERR_INVALID;
  memcpy(lib->poses[(size_t)view].data(), pose16, sizeof(float) * 16);
  return B200_OK;
}

int b200_library_get_view_pose(const b200_library *lib, int view, float *pose16) {
  if (!lib || !pose16 || view < 0 || view >= (int)lib->views.size()) return B200_ERR_INVALID;
  memcpy(pose16, lib->poses[(size_t)view].data(), sizeof(float) * 16);
  return B200_OK;
}

/* On-disk form (little endian): "B200LIB1", uint32 n_views, uint32 D (352), then per view: uint32 K, 16 float pose,
 * K x 3 float keypoints, K x D float descriptors; the file ends with a uint64 FNV-1a hash of everything before it. */
namespace {
const char kLibMagic[8] = {'B', '2', '0', '0', 'L', 'I', 'B', '1'};
struct Fnv {
  uint64_t h = 1469598103934665603ull;
  void add(const void *p, size_t n) {
    const unsigned char *b = (const unsigned char *)p;
    for (size_t i = 0; i < n; ++i) {
      h ^= b[i];
      h *= 1099511628211ull;
    }
  }
};
bool put(FILE *f, Fnv &h, const void *p, size_t n) {
  h.add(p, n);
  return n == 0 || fwrite(p, 1, n, f) == n;
}
bool get(FILE *f, Fnv &h, void *p, size_t n) {
  if (n && fread(p, 1, n, f) != n) return false;
  h.add(p, n);
  return true;
}
}  // namespace

int b200_library_save(b200_ctx *ctx, const b200_library *lib, const char *path) {
  API_ENTER(ctx);
  if (!lib || !path) return ctx->fail(B200_ERR_INVALID, "library_save: bad arguments");
  FILE *f = fopen(path, "wb");
  if (!f) return ctx->fail(B200_ERR_INVALID, (std::string("library_save: cannot open ") + path).c_str());
  Fnv h;
  const uint32_t nv = (uint32_t)lib->views.size(), D = 352;
  bool ok = put(f, h, kLibMagic, 8) && put(f, h, &nv, 4) && put(f, h, &D, 4);
  int rc = B200_OK;
  for (uint32_t v = 0; ok && rc == B200_OK && v < nv; ++v) {
    const b200_model *m = lib->views[v];
    const uint32_t K = (uint32_t)m->K;
    std::vector<float> desc((size_t)K * D), kp((size_t)K * 3);
    rc = b200_model_download(ctx, m, desc.data(), kp.data());
    if (rc == B200_OK)
      ok = put(f, h, &K, 4) && put(f, h, lib->poses[v].data(), 64) && put(f, h, kp.data(), kp.size() * 4) &&
           put(f, h, desc.data(), desc.size() * 4);
  }
  const uint64_t sum = h.h;
  ok = ok && fwrite(&sum, 8, 1, f) == 1;
  ok = (fclose(f) == 0) && ok;
  if (rc != B200_OK) return rc;
  if (!ok) return ctx->fail(B200_ERR_INVALID, (std::string("library_save: write error on ") + path).c_str());
  return B200_OK;
}

int b200_library_load(b200_ctx *ctx, const char *path, b200_library **out) {
  API_ENTER(ctx);
  if (!path || !out) return ctx->fail(B200_ERR_INVALID, "library_load: bad arguments");
  *out = nullptr;
  FILE *f = fopen(path, "rb");
  if (!f) return ctx->fail(B200_ERR_INVALID, (std::string("library_load: cannot open ") + path).c_str());
  Fnv h;
  char magic[8];
  uint32_t nv = 0, D = 0;
  // what is left of the file bounds every allocation below (a corrupt count must not turn into a 94 GB vector)
  long long file_left = 0;
  if (fseek(f, 0, SEEK_END) == 0) {
    file_left = ftell(f);
    rewind(f);
  }
  b200_library *lib = new (std::nothrow) b200_library();
  if (!lib) {
    fclose(f);
    return ctx->fail(B200_ERR_NOMEM, "library_load: out of host memory");
  }
  lib->ctx = ctx;
  int rc = B200_OK;
  const char *why = nullptr;
  try {
  if (!get(f, h, magic, 8) || memcmp(magic, kLibMagic, 8) != 0) why = "not a B200LIB1 file";
  if (!why && (!get(f, h, &nv, 4) || !get(f, h, &D, 4) || D != 352 || nv > (1u << 20))) why = "bad header";
  for (uint32_t v = 0; !why && rc == B200_OK && v < nv; ++v) {
    uint32_t K = 0;
    std::array<float, 16> pose;
    if (!get(f, h, &K, 4) || K > (1u << 26) || !get(f, h, pose.data(), 64)) {
      why = "truncated view header";
      break;
    }
    if ((long long)K * (3 + D) * 4 > file_left - ftell(f)) {
      why = "view larger than the file";
      break;
    }
    std::vector<float> kp((size_t)K * 3), desc((size_t)K * D);
    if (!get(f, h, kp.data(), kp.size() * 4) || !get(f, h, desc.data(), desc.size() * 4)) {
      why = "truncated view data";
      break;
    }
    int id = -1;
    rc = b200_library_add_view_descriptors(ctx, lib, desc.data(), kp.data(), (int)K, 3, &id);
    if (rc == B200_OK) lib->poses[(size_t)id] = pose;
  }
  uint64_t sum = 0;
  if (!why && rc == B200_OK && (fread(&sum, 8, 1, f) != 1 || sum != h.h)) why = "checksum mismatch";
  } catch (const std::exception &) {  // std::bad_alloc from the staging vectors: no exception crosses the C ABI
    rc = B200_ERR_NOMEM;
    ctx->fail(rc, "library_load: out of host memory");
  }
  fclose(f);
  if (why || rc != B200_OK) {
    b200_library_destroy(lib);
    return why ? ctx->fail(B200_ERR_INVALID, (std::string("library_load: ") + why).c_str()) : rc;
  }
  *out = lib;
  return B200_OK;
}

int b200_library_views(const b200_library *lib) { return lib ? (int)lib->views.size() : 0; }

int b200_library_view_size(const b200_library *lib, int view) {
  return (lib && view >= 0 && view < (int)lib->views.size()) ? lib->views[view]->K : 0;
}

int b200_library_download_view(b200_ctx *ctx, const b200_library *lib, int view, float *desc, float *kp) {
  API_ENTER(ctx);
  if (!lib || view < 0 || view >= (int)lib->views.size()) return ctx->fail(B200_ERR_INVALID, "library: bad view index");
  return b200_model_download(ctx, lib->views[view], desc, kp);
}

int b200_register_scene_library(b200_ctx *ctx, const b200_library *lib, const float *scene_xyz, int n, int stride,
                                const float *scene_kp, int Ks, int kstride, const b200_shot_params *p, float *transforms,
                                int *inst_view, int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int max_inst,
                                int *n_inst, int *view_n_corrs) {
  API_ENTER(ctx);
  if (!lib || !n_inst || Ks < 0 || max_inst < 1) return ctx->fail(B200_ERR_INVALID, "register_scene_library: bad arguments");
  B200_TRY(check_params(ctx, p));
  *n_inst = 0;
  if (inst_offsets) inst_offsets[0] = 0;
  std::unique_ptr<b200_cloud> scene;
  B200_TRY(cloud_upload(ctx, scene_xyz, n, stride, false, scene));
  // scene side once: normals + SHOT352 at the keypoints (the reference recomputes both per view)
  DevBuf<float4> dkp;
  DevBuf<float> normals, desc;
  B200_TRY(upload_points(ctx, scene_kp, Ks, kstride, dkp));
  B200_TRY(normals.alloc(ctx, (size_t)std::max(scene->n, 1) * 4));
  B200_TRY(desc.alloc(ctx, (size_t)std::max(Ks, 1) * 352));
  B200_TRY(scene_descriptors(ctx, scene.get(), p, dkp.p, Ks, normals.p, desc.p));
  // Every view's matching + grouping is enqueued first (per-view slices of the output buffers, no host wait in
  // between), then ONE synchronisation and a handful of bulk downloads; the per-view instance lists are put
  // together on the host.  (Round 1 waited and downloaded view by view: 2 ms per view, 0.38 s for 192 views.)
  const int cap = std::max(Ks, 1), mi = p->max_instances;
  const int V = (int)lib->views.size();
  ResultBufs res;  // per view: its correspondence count and instances (its correspondence list is a lane's)
  B200_TRY(res.alloc(ctx, cap, mi, V));
  // The per-view kernels are small (a view has a few hundred descriptors; its grouping runs on one 8-CTA cluster), so
  // the views go round-robin over a few lane contexts of this device (own stream + scratch arena each, the pool of
  // b200_register_scene_batch_shot) and overlap on the GPU; one host thread enqueues everything.
  {
    const int L = std::max(1, std::min(V, 8));
    LanePool &pool = lane_pool(ctx->device);
    std::lock_guard<std::mutex> hold(pool.mu);
    B200_TRY(pool.grow(ctx->device, L));
    int rc = B200_OK;
    cudaEvent_t ready = nullptr;
    cudaError_t e = cudaEventCreateWithFlags(&ready, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(ready, ctx->stream);   // scene descriptors + keypoints are on the device
    std::vector<DevBuf<b200_corr>> lane_corrs((size_t)L);
    for (int l = 0; l < L && e == cudaSuccess && rc == B200_OK; ++l) {
      b200_ctx *lc = pool.ctxs[(size_t)l];
      e = cudaStreamWaitEvent(lc->stream, ready, 0);
      if (e == cudaSuccess) rc = lane_corrs[(size_t)l].alloc(lc, (size_t)cap);
    }
    for (int v = 0; v < V && rc == B200_OK && e == cudaSuccess; ++v) {
      const b200_model *m = lib->views[v];
      b200_ctx *lc = pool.ctxs[(size_t)(v % L)];
      b200_corr *vc = lane_corrs[(size_t)(v % L)].p;
      rc = dev_match(lc, m->desc.p, m->K, desc.p, Ks, 352, p->match_mode, p->match_thr, vc, res.n_corrs.p + v, &m->tc);
      if (rc == B200_OK)
        rc = dev_gc(lc, m->kp.p, dkp.p, vc, res.n_corrs.p + v, Ks, p->gc_size, p->gc_threshold, res.out(v));
      if (rc != B200_OK) ctx->err = lc->err;
    }
    for (int l = 0; l < L; ++l) {   // all lanes drained before their scratch is released and the results are read
      const cudaError_t es = pool.ctxs[(size_t)l]->sync();
      if (es != cudaSuccess && e == cudaSuccess) e = es;
    }
    if (ready) cudaEventDestroy(ready);
    if (e != cudaSuccess && rc == B200_OK) rc = ctx->fail_cuda(e, "register_scene_library lanes", __FILE__, __LINE__);
    B200_TRY(rc);
  }
  int total_inst = 0;
  bool overflow = false;
  try {  // host staging vectors: std::bad_alloc must not cross the C ABI
    std::vector<int> hn((size_t)std::max(V, 1)), hnc((size_t)std::max(V, 1));
    B200_TRY(download(ctx, hn.data(), res.n_inst.p, (size_t)V));
    B200_TRY(download(ctx, hnc.data(), res.n_corrs.p, (size_t)V));
    B200_CUDA(ctx, ctx->sync());
    if (view_n_corrs)
      for (int v = 0; v < V; ++v) view_n_corrs[v] = hnc[(size_t)v];
    std::vector<int> hoffs(((size_t)mi + 1) * std::max(V, 1)), hcnts((size_t)mi * std::max(V, 1));
    std::vector<float> hT((size_t)mi * 16 * std::max(V, 1));
    std::vector<b200_corr> hic((size_t)cap * std::max(V, 1));
    if (V > 0) {
      B200_TRY(download(ctx, hoffs.data(), res.offsets.p, hoffs.size()));
      B200_TRY(download(ctx, hcnts.data(), res.counts.p, hcnts.size()));
      B200_TRY(download(ctx, hT.data(), res.T.p, hT.size()));
      B200_TRY(download(ctx, hic.data(), res.inst_corrs.p, hic.size()));
      B200_CUDA(ctx, ctx->sync());
    }
    int total_corr = 0;
    for (int v = 0; v < V && !overflow; ++v) {
      if (hn[(size_t)v] > mi) overflow = true;  // more than max_instances in this view: the first ones are kept
      const int kept = std::min(hn[(size_t)v], mi);
      const int *offs = hoffs.data() + (size_t)v * (mi + 1);
      const int *cnts = hcnts.data() + (size_t)v * mi;
      for (int i = 0; i < kept; ++i) {
        const int cnt = cnts[i];
        if (total_inst >= max_inst || total_corr + cnt > corr_cap) {
          overflow = true;
          break;
        }
        if (transforms)
          memcpy(transforms + (size_t)total_inst * 16, hT.data() + ((size_t)v * mi + i) * 16, sizeof(float) * 16);
        if (inst_view) inst_view[total_inst] = v;
        if (inst_corrs && cnt > 0)
          memcpy(inst_corrs + total_corr, hic.data() + (size_t)v * cap + offs[i], sizeof(b200_corr) * (size_t)cnt);
        total_corr += cnt;
        ++total_inst;
        if (inst_offsets) inst_offsets[total_inst] = total_corr;
      }
    }
  } catch (const std::exception &) {
    return ctx->fail(B200_ERR_NOMEM, "register_scene_library: out of host memory");
  }
  *n_inst = total_inst;
  if (overflow) return ctx->fail(B200_ERR_CAPACITY, "register_scene_library: output capacity too small");
  return B200_OK;
}

} /* extern "C" */
