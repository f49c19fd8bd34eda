/*
 * b200reg.h — C ABI of libb200reg.so, the B200 (sm_100a) implementation of the SHOT/FPFH
 * recognition hot path of Merium88/3D-Object-Detection-of-Industrial-Joints.
 *
 * The reference reaches this path through PCL classes (SURVEY.md §8(b)); each entry point below
 * names the reference call site (file:line under /root/reference) whose PCL call it replaces.
 * The PCL-style C++ adapters in include/pcl_b200/ flatten clouds and call these functions;
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions
 *  - plain pointers and sizes only; every function returns 0 (B200_OK) or a negative b200_status;
 *    no exceptions cross the boundary; b200_last_error() gives the text of the last failure.
 *  - points are float rows with a caller-given stride in floats (>= 3; x, y, z first), so
 *    pcl::PointXYZRGBA (stride 8), float4 (4) and packed xyz (3) are all accepted without a copy
 *    on the caller's side.  Normals are rows of 4 floats (nx, ny, nz, curvature) — the first 16
 *    bytes of pcl::Normal are nx, ny, nz, pad; the shim copies curvature into slot 3.
 *  - `b200_*`      : HOST pointers; the call uploads, computes on the GPU, downloads and
 *                    synchronises (this is the drop-in form the PCL-style adapters use).
 *  - `b200_dev_*`  : DEVICE pointers; asynchronous on the context's stream, no host sync unless
 *                    stated.  Used for resident pipelines and by the torch-based harness.
 *  - there is no CPU fallback: every function fails with B200_ERR_NODEVICE / B200_ERR_CUDA when
 *    no sm_100 device is usable.
 *  - NaN semantics follow PCL: degenerate points yield NaN rows, not errors.
 */
#ifndef B200REG_H_
#define B200REG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200REG_ABI_VERSION 1

#if defined(__GNUC__)
#define B200_API __attribute__((visibility("default")))
#else
#define B200_API
#endif

typedef enum {
  B200_OK = 0,
  B200_ERR_INVALID = -1,   /* bad argument (e.g. both k and radius set, like Feature::initCompute) */
  B200_ERR_CUDA = -2,      /* CUDA runtime error; see b200_last_error */
  B200_ERR_NOMEM = -3,
  B200_ERR_CAPACITY = -4,  /* caller-provided output capacity too small; required size reported */
  B200_ERR_NODEVICE = -5
} b200_status;

typedef struct b200_ctx b200_ctx;     /* device, stream, scratch pool; one per host thread */
typedef struct b200_cloud b200_cloud; /* device-resident search surface (+ uniform grids) */
typedef struct b200_model b200_model; /* device-resident model descriptor library + keypoints */

/* pcl::Correspondence (SHOT.cpp:420): index_query = model index, index_match = scene index,
 * distance = squared L2 descriptor distance. */
typedef struct {
  int index_query;
  int index_match;
  float distance;
} b200_corr;

/* ---------------------------------------------------------------- context ---------------- */
/* stream: a cudaStream_t to run on (e.g. torch's current stream), or NULL to create one. */
B200_API int b200_ctx_create(b200_ctx **out, int device, void *stream);
B200_API int b200_ctx_destroy(b200_ctx *ctx);
/* Host waits of this context: 0 (default) spin on the stream (lowest latency), 1 sleep on a blocking event — for
 * deployments with more contexts (lanes) than host cores. */
B200_API int b200_ctx_set_blocking_sync(b200_ctx *ctx, int enable);
B200_API int b200_ctx_sync(b200_ctx *ctx);
B200_API const char *b200_last_error(const b200_ctx *ctx); /* never NULL; ctx may be NULL (global error) */
B200_API int b200_abi_version(void);
/* Number of this library's kernel launches on the context since creation (bench gpu_launches). */
B200_API int64_t b200_ctx_launch_count(const b200_ctx *ctx);

/* Per-stage device timing (CUDA events on the context's stream) for bench.py's roofline line.
 * Stages: 0 grid build, 1 normals, 2 neighbour count, 3 SHOT (LRF + descriptor), 4 FPFH, 5 matching,
 * 6 GC sort, 7 GC grouping, 8 GC RANSAC.  b200_ctx_stage_time synchronises the stream. */
B200_API int b200_ctx_set_profiling(b200_ctx *ctx, int enable);
B200_API int b200_ctx_reset_profiling(b200_ctx *ctx);
B200_API int b200_ctx_stage_count(void);
B200_API const char *b200_ctx_stage_name(int stage);
B200_API int b200_ctx_stage_time(b200_ctx *ctx, int stage, double *total_ms, int *calls);

/* ---------------------------------------------------------------- search surface --------- */
/* Replaces pcl::search::KdTree / KdTreeFLANN<PointXYZRGBA>::setInputCloud (built implicitly by
 * Feature::initCompute for every compute(); explicit at SHOT_VAR.cpp:350, Edge_detection.cpp:117).
 * Rows with a non-finite coordinate are dropped from the index but keep their position. */
B200_API int b200_cloud_create(b200_ctx *ctx, const float *xyz, int n, int stride, b200_cloud **out);     /* host rows */
B200_API int b200_dev_cloud_create(b200_ctx *ctx, const float *d_xyz, int n, int stride, b200_cloud **out); /* device rows */
B200_API int b200_cloud_destroy(b200_cloud *cloud);
B200_API int b200_cloud_size(const b200_cloud *cloud);

/* KdTreeFLANN::radiusSearch (SHOT_VAR.cpp:356, 434).  CSR result: offsets[nq+1]; neighbours with
 * d2 < (float)(radius*radius), each list sorted by (d2, index).  Two-call sizing: pass cap = 0 (idx,
 * d2 may be NULL) to obtain *total, then call again with buffers of that capacity. */
B200_API int b200_radius_search(b200_ctx *ctx, b200_cloud *surf, const float *q, int nq, int qstride, double radius,
                       int64_t *offsets, int *idx, float *d2, int64_t cap, int64_t *total);
/* KdTreeFLANN::nearestKSearch (SHOT.cpp:163, Edge_detection.cpp:120).  idx/d2: nq x k, sorted by
 * (d2, index); k is clamped to the number of indexed points (*k_found), unused slots are -1/+inf. */
B200_API int b200_knn_search(b200_ctx *ctx, b200_cloud *surf, const float *q, int nq, int qstride, int k, int *idx,
                    float *d2, int *k_found);

/* ---------------------------------------------------------------- keypoints -------------- */
/* pcl::UniformSampling<PointT>::filter (SHOT.cpp:314-323, SHOT_demo.cpp:246-249, 6Dpose.cpp:281-284,
 * CAD_desc.cpp:295-304; setRadiusSearch(leaf)): per occupied leaf of the lattice ijk = floor(p / leaf) the
 * input point closest to the leaf's integer index vector (PCL's own test), first point on ties.  Output
 * order: ascending leaf index (PCL's is hash-map order).  out_xyz: capacity n x 3 floats; out_index
 * (nullable): original row of every kept point; *count = number kept.  Non-finite rows are skipped.
 * B200_ERR_CAPACITY when the lattice has more than 2^26 leaves (PCL: "leaf size is too small"). */
B200_API int b200_uniform_sampling(b200_ctx *ctx, const float *xyz, int n, int stride, double leaf, float *out_xyz,
                                   int *out_index, int *count);
B200_API int b200_dev_uniform_sampling(b200_ctx *ctx, const float *d_xyz, int n, int stride, double leaf,
                                       float *d_out_xyz, int *d_out_index, int *d_count);
/* pcl::VoxelGrid<PointT>::filter (SHOT_demo.cpp:413-417, 489-491; FPFH_demo.cpp:412-415, 494;
 * setLeafSize(lx, ly, lz)): centroid of the points of every occupied voxel, ascending voxel index.  Only
 * x, y, z are averaged (the hot path never reads colour).  out_xyz: capacity n x 3 floats. */
B200_API int b200_voxel_grid(b200_ctx *ctx, const float *xyz, int n, int stride, float lx, float ly, float lz,
                             float *out_xyz, int *count);
B200_API int b200_dev_voxel_grid(b200_ctx *ctx, const float *d_xyz, int n, int stride, float lx, float ly, float lz,
                                 float *d_out_xyz, int *d_count);

/* pcl::removeNaNFromPointCloud (SHOT.cpp:298-299, first statement of the callback): rows with finite x, y, z, in
 * order; out_xyz n x 3, out_index (nullable) n: the kept rows' original positions. */
B200_API int b200_remove_nan(b200_ctx *ctx, const float *xyz, int n, int stride, float *out_xyz, int *out_index,
                             int *count);
/* pcl::transformPointCloud(cloud_in, cloud_out, Eigen::Matrix4f) (the model placed by a grouped pose before ICP and for
 * display: SHOT.cpp, SHOT_demo.cpp:590-663): transform = row-major 4x4; out_xyz n x 3; rows with a non-finite
 * coordinate are copied unchanged, like PCL's non-dense branch. */
B200_API int b200_transform_points(b200_ctx *ctx, const float *xyz, int n, int stride, const float *transform,
                                   float *out_xyz);

/* ---------------------------------------------------------------- normals ---------------- */
/* pcl::NormalEstimationOMP::compute — setKSearch(k) (SHOT.cpp:302-308, 6Dpose.cpp:275-278,
 * SHOT_demo.cpp:405-411, CAD_desc.cpp:283-289) or setRadiusSearch(r) (FPFH_demo.cpp:416-420,
 * FPFH_scenes_clustered.cpp:273-277).  Exactly one of k / radius non-zero.  q == NULL: the input
 * cloud is the surface itself.  viewpoint: 3 floats or NULL for (0,0,0).  out: nq x 4. */
B200_API int b200_normals(b200_ctx *ctx, b200_cloud *surf, const float *q, int nq, int qstride, int k, double radius,
                 const float *viewpoint, float *out);
B200_API int b200_dev_normals(b200_ctx *ctx, b200_cloud *surf, const float *d_q, int nq, int qstride, int k,
                     double radius, const float *viewpoint, float *d_out);

/* ---------------------------------------------------------------- SHOT ------------------- */
/* pcl::SHOTLocalReferenceFrameEstimationOMP (implicit in SHOTEstimationOMP::initCompute,
 * SHOT.cpp:360-366).  out: K x 9 (x, y, z axes). */
B200_API int b200_shot_lrf(b200_ctx *ctx, b200_cloud *surf, const float *kp, int K, int kstride, double radius, float *out);
/* pcl::SHOTEstimationOMP<PointXYZRGBA, Normal, SHOT352>::compute (SHOT.cpp:360-371,
 * SHOT_demo.cpp:419-424, 497-502, 6Dpose.cpp:450-461, CAD_desc.cpp:341-352).
 * normals: n x 4 for the search surface (setInputNormals); desc: K x 352; rf: K x 9 (may be NULL). */
B200_API int b200_shot352(b200_ctx *ctx, b200_cloud *surf, const float *normals, const float *kp, int K, int kstride,
                 double radius, float *desc, float *rf);
B200_API int b200_dev_shot352(b200_ctx *ctx, b200_cloud *surf, const float *d_normals, const float *d_kp, int K,
                     int kstride, double radius, float *d_desc, float *d_rf);

/* ---------------------------------------------------------------- FPFH ------------------- */
/* pcl::FPFHEstimation / FPFHEstimationOMP ::compute (FPFH_demo.cpp:422-428, 505-510;
 * FPFH_scenes_clustered.cpp:287-293, 379-387).  q == NULL: input == surface.  out: nq x 33. */
B200_API int b200_fpfh33(b200_ctx *ctx, b200_cloud *surf, const float *normals, const float *q, int nq, int qstride,
                double radius, float *out);
B200_API int b200_dev_fpfh33(b200_ctx *ctx, b200_cloud *surf, const float *d_normals, const float *d_q, int nq,
                    int qstride, double radius, float *d_out);

/* ---------------------------------------------------------------- matching --------------- */
/* pcl::KdTreeFLANN<SHOT352 / FPFHSignature33>::setInputCloud + nearestKSearch + the user
 * threshold loop.  mode 1: k = 1, accept d2 < thr (SHOT.cpp:405-423, SHOT_scenes.cpp:359-365,
 * 6Dpose.cpp:464-482).  mode 2: k = 2, accept d0/d1 <= 1 (SHOT_demo.cpp:508-530,
 * FPFH_demo.cpp:516-538).  D = 352 or 33 (any D accepted).  out: capacity Ks; ascending scene index. */
B200_API int b200_match(b200_ctx *ctx, const float *model, int Km, const float *scene, int Ks, int D, int mode, float thr,
               b200_corr *out, int *count);
B200_API int b200_dev_match(b200_ctx *ctx, const float *d_model, int Km, const float *d_scene, int Ks, int D, int mode,
                   float thr, b200_corr *d_out, int *d_count);

/* Resident descriptor index for the reference's per-query loop: KdTreeFLANN<Descriptor>::setInputCloud
 * (SHOT.cpp:405-406, SHOT_demo.cpp:508-509, FPFH_demo.cpp:516-517) followed by nearestKSearch per scene
 * descriptor (SHOT.cpp:417 k=1, SHOT_demo.cpp:521 k=2).  Rows with a non-finite value are dropped from
 * the index (their positions are kept).  idx/d2: nq x k in (distance, index) order; 1 <= k <= 16;
 * *k_found = min(k, indexed rows); unused slots are -1 / +inf. */
typedef struct b200_desc_index b200_desc_index;
B200_API int b200_desc_index_create(b200_ctx *ctx, const float *desc, int K, int D, b200_desc_index **out);
B200_API int b200_desc_index_destroy(b200_desc_index *index);
B200_API int b200_desc_index_size(const b200_desc_index *index);
B200_API int b200_desc_index_knn(b200_ctx *ctx, const b200_desc_index *index, const float *queries, int nq, int k,
                                 int *idx, float *d2, int *k_found);

/* ---------------------------------------------------------------- BOARD frames ----------- */
/* pcl::BOARDLocalReferenceFrameEstimation::compute — the reference frames of the Hough branch (SHOT.cpp:441-453,
 * 6Dpose.cpp:497-509, FPFH_demo.cpp:556-568: setFindHoles(true), setRadiusSearch(rf_rad_), setInputCloud(keypoints),
 * setInputNormals(cloud normals), setSearchSurface(cloud)).  Parameters = the PCL setters; b200_board_params_default
 * fills PCL's constructor defaults (tangent_radius 0, find_holes 0, margin_thresh 0.85, check_margin_array_size 24,
 * hole_size_prob_thresh 0.2, steep_thresh 0.1).  normals: one row of 4 floats per surface point.  rf: K x 9
 * (x, y, z axes); NaN rows for keypoints with fewer than 6 support points.  With find_holes PCL draws two rand()
 * values per keypoint with a full support, in keypoint order, from the process-wide stream; here the stream
 * (glibc's generator) belongs to the context: a new context is srand(1), b200_ctx_srand reseeds it, and successive
 * calls continue it (model frames, then scene frames, like the reference's two compute() calls).  The resident Hough
 * branch (b200_model_create_shot_hough) instead fixes the scene frames' stream per model: see there. */
typedef struct b200_board_params {
  int find_holes;
  float tangent_radius; /* 0: PCL's code path when setTangentRadius is never called */
  float margin_thresh;
  int check_margin_array_size; /* 1..64 */
  float hole_size_prob_thresh;
  float steep_thresh;
} b200_board_params;
B200_API void b200_board_params_default(b200_board_params *p);
B200_API int b200_ctx_srand(b200_ctx *ctx, unsigned seed);
B200_API int b200_board_lrf(b200_ctx *ctx, b200_cloud *surface, const float *normals, const float *kp, int K, int kstride,
                            double radius, const b200_board_params *p, float *rf);

/* ---------------------------------------------------------------- grouping --------------- */
/* pcl::GeometricConsistencyGrouping::recognize (SHOT.cpp:473-482, 6Dpose.cpp:529-538,
 * SHOT_scenes.cpp:413-425).  transforms: max_inst x 16 (row-major 4x4, model -> scene);
 * inst_offsets: max_inst + 1; inst_corrs: capacity corr_cap (>= C is always enough).
 * *n_inst is the number found (B200_ERR_CAPACITY if it exceeds max_inst; the first max_inst are valid). */
B200_API int b200_gc_recognize(b200_ctx *ctx, const float *model_kp, int Km, int mstride, const float *scene_kp, int Ks,
                      int sstride, const b200_corr *corrs, int C, double gc_size, int gc_threshold,
                      float *transforms, int max_inst, int *inst_offsets, b200_corr *inst_corrs, int corr_cap,
                      int *n_inst);

/* pcl::Hough3DGrouping::recognize (the reference's default grouping: SHOT.cpp:433-470, SHOT_demo.cpp:540-577,
 * FPFH_demo.cpp:548-585) with the reference's settings — setUseInterpolation(false), setUseDistanceWeight(true)
 * — and the reference frames given by the caller (setInputRf / setSceneRf; K x 9 floats: x, y, z axes, e.g.
 * from b200_shot_lrf).  bin_size = setHoughBinSize, threshold = setHoughThreshold (negative: fraction of the
 * largest bin).  Every Hough bin reaching the threshold is an instance (ascending bin index); its voters go
 * through the same RANSAC as in b200_gc_recognize (inlier threshold = bin size).  Outputs as b200_gc_recognize. */
B200_API int b200_hough3d_recognize(b200_ctx *ctx, const float *model_kp, const float *model_rf, int Km, int mstride,
                                    const float *scene_kp, const float *scene_rf, int Ks, int sstride,
                                    const b200_corr *corrs, int C, double bin_size, double threshold, float *transforms,
                                    int max_inst, int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int *n_inst);

/* ---------------------------------------------------------------- pose refinement -------- */
/* pcl::IterativeClosestPoint::align + getFitnessScore with the settings the reference uses: setMaximumIterations
 * only (SHOT.cpp:177-192: 100; SHOT_demo.cpp:604-663, FPFH_demo.cpp:611-668: 1; 6Dpose.cpp:572-609), everything
 * else PCL's default — pass max_corr_dist <= 0 for "unlimited", transformation_epsilon = 0,
 * euclidean_fitness_epsilon = -DBL_MAX.  source: the cloud that is moved (setInputSource: the rotated model);
 * target: a b200_cloud (setInputTarget: the scene).  guess (nullable): row-major 4x4 initial transform.
 * final_transform: row-major 4x4 (getFinalTransformation); aligned (nullable): ns x 3 = the source under it
 * (the cloud align() fills); *fitness = getFitnessScore() (mean squared distance to the nearest target point);
 * *converged = hasConverged(); *iterations = iterations run.  Per iteration: exact nearest target point of
 * every source point (kept when d2 <= max_corr_dist^2), Umeyama (no scale) on the pairs, stop on: iteration
 * cap, null motion within transformation_epsilon, |mse - previous mse| < 1e-12, relative mse change below
 * euclidean_fitness_epsilon; fewer than 3 pairs ends the loop unconverged. */
B200_API int b200_icp_align(b200_ctx *ctx, const float *source, int ns, int sstride, b200_cloud *target,
                            int max_iterations, double max_corr_dist, double transformation_epsilon,
                            double euclidean_fitness_epsilon, const float *guess, float *final_transform, float *aligned,
                            double *fitness, int *converged, int *iterations);

/* ---------------------------------------------------------------- resident pipeline ------ */
typedef struct {
  int normal_k;          /* NormalEstimationOMP::setKSearch; 0 if radius is used */
  double normal_radius;  /* NormalEstimationOMP::setRadiusSearch; 0 if k is used */
  double descr_radius;   /* SHOTEstimationOMP::setRadiusSearch (descr_rad_, SHOT.cpp:52) */
  int match_mode;        /* 1 or 2, see b200_match */
  float match_thr;       /* 0.25f SHOT_scenes.cpp:360 / 0.20f SHOT.cpp:418 */
  double gc_size;        /* cg_size_   (SHOT.cpp:53) */
  int gc_threshold;      /* cg_thresh_ (SHOT.cpp:54; passed as float, truncated) */
  int max_instances;
} b200_shot_params;

/* Model side of SHOT.cpp:302-371 / CAD_desc.cpp:283-352: normals + SHOT352 of the model keypoints,
 * kept on the device as the (replicated) descriptor library. */
B200_API int b200_model_create_shot(b200_ctx *ctx, const float *xyz, int n, int stride, const float *kp, int K,
                           int kstride, const b200_shot_params *p, b200_model **out);
B200_API int b200_model_destroy(b200_model *m);
B200_API int b200_model_size(const b200_model *m);
/* copy the library out (host): desc K x 352 (K x 33 for an FPFH model), kp K x 3 (either may be NULL) */
B200_API int b200_model_download(b200_ctx *ctx, const b200_model *m, float *desc, float *kp);

/* FPFH_demo.cpp:405-538 with the model side resident.  The reference estimates the normals ON the keypoint clouds by
 * radius (FPFH_demo.cpp:416-420, 486-492) and runs FPFHEstimation with input = surface = keypoints (:422-428,
 * :505-510); params: normal_radius (or normal_k), descr_radius = the FPFH radius, match_mode = 2 (the k = 2 ratio test
 * of :516-538), gc_size / gc_threshold.  The model's descriptors are K x 33 (b200_model_descriptor_length). */
B200_API int b200_model_create_fpfh(b200_ctx *ctx, const float *kp, int K, int kstride, const b200_shot_params *p,
                                    b200_model **out);
B200_API int b200_model_descriptor_length(const b200_model *m);
/* Scene side in one call (host buffers): normals + FPFH33 of the scene keypoint cloud, correspondence search against
 * the resident model, GC grouping + poses.  desc_out (Ks x 33) may be NULL; other outputs as b200_register_scene_shot. */
B200_API int b200_register_scene_fpfh(b200_ctx *ctx, const b200_model *model, const float *scene_kp, int Ks, int kstride,
                                      const b200_shot_params *p, float *transforms, int *inst_offsets,
                                      b200_corr *inst_corrs, int corr_cap, int *n_inst, b200_corr *corrs_out,
                                      int *n_corrs, float *desc_out);

/* Scene side of SHOT.cpp:305-483 in one call (host buffers in, host results out): normals →
 * SHOT352 at the keypoints → correspondence search against the resident model → GC grouping.
 * corrs_out (capacity Ks) / n_corrs receive the model-scene correspondences; may be NULL. */
B200_API int b200_register_scene_shot(b200_ctx *ctx, const b200_model *model, const float *scene_xyz, int n, int stride,
                             const float *scene_kp, int Ks, int kstride, const b200_shot_params *p,
                             float *transforms, int *inst_offsets, b200_corr *inst_corrs, int corr_cap,
                             int *n_inst, b200_corr *corrs_out, int *n_corrs);

/* Same pipeline with every buffer already resident (device pointers), asynchronous, no host
 * synchronisation; d_n_inst / d_n_corrs are device ints.  d_desc_out (Ks x 352) may be NULL. */
B200_API int b200_dev_register_scene_shot(b200_ctx *ctx, const b200_model *model, const float *d_scene_xyz, int n,
                                 int stride, const float *d_scene_kp, int Ks, int kstride,
                                 const b200_shot_params *p, float *d_transforms, int *d_inst_offsets,
                                 int *d_inst_counts, b200_corr *d_inst_corrs, int corr_cap, int *d_n_inst,
                                 b200_corr *d_corrs_out, int *d_n_corrs, float *d_desc_out);

/* A batch of scenes against one model with several scenes in flight (BASELINE config 5 on one GPU; the per-rank part
 * of the sharded batch).  The reference's programs register one frame per callback; for throughput the scenes are
 * independent, and `lanes` contexts (each with its own stream, arena and host thread, created and kept by the library
 * for `device`) work through the batch concurrently so that the latency-bound grouping kernel of one scene (8 SMs)
 * runs beside the GPU-wide stages of the others.  Scene s is handled by lane s mod lanes.  Per scene s: inputs
 * scene_xyz[s] (n_points[s] x stride), scene_kp[s] (n_kp[s] x kstride); outputs as b200_register_scene_shot into
 * transforms[s] (p->max_instances x 16), inst_offsets[s] (p->max_instances + 1), inst_corrs[s] (capacity corr_cap[s]),
 * n_inst[s], corrs_out[s] (capacity n_kp[s]; the array or any entry may be NULL), n_corrs[s], status[s] (the scene's
 * own return code).  Results are bit-identical to calling b200_register_scene_shot scene by scene.  Returns the
 * first non-OK status other than B200_ERR_CAPACITY, else B200_OK.  lanes: 1..16 (4 to 6 saturate a B200). */
B200_API int b200_register_scene_batch_shot(int device, const b200_model *model, int n_scenes,
                                            const float *const *scene_xyz, const int *n_points, int stride,
                                            const float *const *scene_kp, const int *n_kp, int kstride,
                                            const b200_shot_params *p, int lanes, float *const *transforms,
                                            int *const *inst_offsets, b200_corr *const *inst_corrs, const int *corr_cap,
                                            int *n_inst, b200_corr *const *corrs_out, int *n_corrs, int *status);

/* The lane contexts of b200_register_scene_batch_shot (streams, arenas: about 1.3 GB each for a 1 M-point scene) stay
 * alive between batches; this frees the ones of `device`. */
B200_API int b200_lanes_release(int device);

/* ---------------------------------------------------------------- resident Hough branch -- */
/* The reference's default branch (use_hough_ = true: SHOT.cpp:433-470, SHOT_demo.cpp:540-577): BOARD frames of the
 * model and scene keypoints, then Hough3DGrouping, on the resident pipeline. */
typedef struct {
  double rf_radius;          /* BOARDLocalReferenceFrameEstimation::setRadiusSearch (rf_rad_) */
  b200_board_params board;   /* the reference sets find_holes = 1 */
  double bin_size;           /* Hough3DGrouping::setHoughBinSize (cg_size_) */
  double threshold;          /* setHoughThreshold (cg_thresh_; negative = fraction of the largest bin) */
} b200_hough_params;

/* What b200_model_create_shot builds (identical descriptors), plus, kept on the device: the BOARD frames of the model
 * keypoints (over the model cloud and the normals computed there) and Hough3DGrouping::train()'s votes.
 * The rand() stream: the model's frames draw from ctx's stream exactly as b200_board_lrf does (ctx's stream then
 * continues after them), and the model records the stream's state after its frames.  EVERY scene registered against
 * the model draws its frames from that recorded state, so a registration gives what a fresh process doing
 * srand(seed) -> model frames -> scene frames computes, whatever the scene order, lane count or context.  (A
 * long-running PCL process instead keeps one stream going across its callbacks; b200_board_lrf offers that.) */
B200_API int b200_model_create_shot_hough(b200_ctx *ctx, const float *xyz, int n, int stride, const float *kp, int K,
                                          int kstride, const b200_shot_params *p, const b200_hough_params *h,
                                          b200_model **out);
/* rf: K x 9.  B200_ERR_INVALID for a model without frames (not made by b200_model_create_shot_hough). */
B200_API int b200_model_download_frames(b200_ctx *ctx, const b200_model *m, float *rf);

/* Scene side of the Hough branch in one call: normals -> SHOT352 -> correspondence search (as in
 * b200_register_scene_shot) -> BOARD frames of the scene keypoints over the scene cloud and its normals ->
 * Hough3DGrouping -> RANSAC poses.  Outputs as b200_register_scene_shot; p->gc_size / p->gc_threshold are not read.
 * rf_out (Ks x 9, nullable): the scene frames.  B200_ERR_CAPACITY when the Hough space would exceed 2^27 bins (no
 * instance; the correspondences are still returned) or there are more than p->max_instances instances (the first
 * ones are kept).  B200_ERR_INVALID for a model without frames. */
B200_API int b200_register_scene_shot_hough(b200_ctx *ctx, const b200_model *model, const float *scene_xyz, int n,
                                            int stride, const float *scene_kp, int Ks, int kstride,
                                            const b200_shot_params *p, const b200_hough_params *h, float *transforms,
                                            int *inst_offsets, b200_corr *inst_corrs, int corr_cap, int *n_inst,
                                            b200_corr *corrs_out, int *n_corrs, float *rf_out);

/* Device-pointer, asynchronous form (as b200_dev_register_scene_shot).  d_rf_out (Ks x 9) may be NULL; *d_status (a
 * device int) receives B200_OK, or B200_ERR_CAPACITY when the Hough space would exceed 2^27 bins. */
B200_API int b200_dev_register_scene_shot_hough(b200_ctx *ctx, const b200_model *model, const float *d_scene_xyz, int n,
                                                int stride, const float *d_scene_kp, int Ks, int kstride,
                                                const b200_shot_params *p, const b200_hough_params *h,
                                                float *d_transforms, int *d_inst_offsets, int *d_inst_counts,
                                                b200_corr *d_inst_corrs, int corr_cap, int *d_n_inst,
                                                b200_corr *d_corrs_out, int *d_n_corrs, float *d_desc_out,
                                                float *d_rf_out, int *d_status);

/* Lanes form, arguments and outputs as b200_register_scene_batch_shot plus h.  Results are those of
 * b200_register_scene_shot_hough scene by scene: the rand() draws and every grouping step are the same.  One exception:
 * a BOARD frame can differ in its last bit between two builds of the same scene cloud.  This happens for about 1 row in
 * 50 000 on 1 M-point scenes (DESIGN §7). */
B200_API int b200_register_scene_batch_shot_hough(int device, const b200_model *model, int n_scenes,
                                                  const float *const *scene_xyz, const int *n_points, int stride,
                                                  const float *const *scene_kp, const int *n_kp, int kstride,
                                                  const b200_shot_params *p, const b200_hough_params *h, int lanes,
                                                  float *const *transforms, int *const *inst_offsets,
                                                  b200_corr *const *inst_corrs, const int *corr_cap, int *n_inst,
                                                  b200_corr *const *corrs_out, int *n_corrs, int *status);

/* ---------------------------------------------------------------- multi-view library ----- */
/* The reference recognises against a set of rendered partial views of the CAD models: CAD_desc.cpp:231-370
 * builds one SHOT descriptor set per view, and SHOT.cpp:243-483 / 6Dpose.cpp / SHOT_demo.cpp:430-663 loop over
 * the views, recomputing the SCENE normals and descriptors inside the loop (6Dpose.cpp:458-461).  A library
 * keeps every view's descriptors + keypoints resident; b200_register_scene_library computes the scene side
 * once and then runs correspondence search + geometric-consistency grouping per view. */
typedef struct b200_library b200_library;
B200_API int b200_library_create(b200_ctx *ctx, b200_library **out);
B200_API int b200_library_destroy(b200_library *lib);
/* one view = body of the CAD_desc.cpp loop (normals, SHOT352 at the keypoints); *view_id = its index */
B200_API int b200_library_add_view(b200_ctx *ctx, b200_library *lib, const float *xyz, int n, int stride, const float *kp,
                                   int K, int kstride, const b200_shot_params *p, int *view_id);
B200_API int b200_library_views(const b200_library *lib);
B200_API int b200_library_view_size(const b200_library *lib, int view);
B200_API int b200_library_download_view(b200_ctx *ctx, const b200_library *lib, int view, float *desc, float *kp);
/* A view from descriptors computed elsewhere (K x 352) and their keypoints — e.g. the reference's own
 * Partial_View<l>.txt dumps (CAD_desc.cpp:354-370: one float per line, 352 per keypoint). */
B200_API int b200_library_add_view_descriptors(b200_ctx *ctx, b200_library *lib, const float *desc, const float *kp, int K,
                                               int kstride, int *view_id);
/* view -> CAD pose table (the reference keeps it in pose.txt, SHOT_demo.cpp:206-239): row-major 4x4 per view,
 * identity until set; carried by the library file. */
B200_API int b200_library_set_view_pose(b200_library *lib, int view, const float *pose16);
B200_API int b200_library_get_view_pose(const b200_library *lib, int view, float *pose16);
/* Binary library file replacing the text dumps: "B200LIB1", uint32 views, uint32 D, per view {uint32 K, 16 float pose,
 * K x 3 float keypoints, K x D float descriptors}, uint64 FNV-1a of the preceding bytes; little endian.
 * b200_library_load rejects a wrong magic, a truncated file or a checksum mismatch (B200_ERR_INVALID). */
B200_API int b200_library_save(b200_ctx *ctx, const b200_library *lib, const char *path);
B200_API int b200_library_load(b200_ctx *ctx, const char *path, b200_library **out);
/* Instances of all views, concatenated in view order: inst_view[i] = view of instance i; transforms, inst_offsets
 * (max_inst + 1) and inst_corrs (index_query = keypoint index WITHIN the view) as in b200_gc_recognize;
 * view_n_corrs (nullable, one per view) = correspondences found for that view.  p->max_instances bounds the
 * instances kept per view, max_inst the total. */
B200_API int b200_register_scene_library(b200_ctx *ctx, const b200_library *lib, const float *scene_xyz, int n, int stride,
                                         const float *scene_kp, int Ks, int kstride, const b200_shot_params *p,
                                         float *transforms, int *inst_view, int *inst_offsets, b200_corr *inst_corrs,
                                         int corr_cap, int max_inst, int *n_inst, int *view_n_corrs);

/* ---------------------------------------------------------------------------------------------------------------
 * Multi-GPU (SURVEY.md 8(e)): one context per GPU, each driven by its own host thread or process; the context owns
 * an NCCL communicator (NCCL is bound at run time: libnccl.so.2).  The reference's callbacks process one scene at a
 * time (SHOT.cpp:204, per-keypoint SHOT at :360-371, the matching loop :409-423): the sharded call splits exactly
 * those two loops over the GPUs.
 * ------------------------------------------------------------------------------------------------------------- */
/* 128-byte rendezvous token (ncclUniqueId).  Call on one rank, hand the bytes to the others (pipe, file, MPI ...). */
B200_API int b200_comm_unique_id(void *id128, size_t bytes);
/* Collective over the `world` contexts that share the token. */
B200_API int b200_comm_init(b200_ctx *ctx, const void *id128, int rank, int world);
B200_API int b200_comm_destroy(b200_ctx *ctx);
B200_API int b200_comm_rank(const b200_ctx *ctx);
B200_API int b200_comm_size(const b200_ctx *ctx);
/* Device buffers, asynchronous on the context's stream.  Every rank contributes *d_count (<= cap) correspondences;
 * afterwards d_gathered holds rank r's list at [r * cap, r * cap + d_counts[r]) on every rank (multi-scene batches:
 * gather of the lists of the scenes registered in this step). */
B200_API int b200_gather_correspondences(b200_ctx *ctx, const b200_corr *d_corrs, const int *d_count, int cap,
                                         b200_corr *d_gathered, int *d_counts);
/* One scene over all ranks: keypoint slabs per rank, model library replicated, correspondence lists gathered on
 * `root`, grouping + poses there.  Collective (every rank calls it with its own resident copy of the model);
 * host buffers; the scene and the outputs are the root's, other ranks may pass NULL.  Same outputs as
 * b200_register_scene_shot, bit for bit. */
B200_API int b200_register_scene_shot_sharded(b200_ctx *ctx, const b200_model *model, int root, const float *scene_xyz,
                                              int n, int stride, const float *scene_kp, int Ks, int kstride,
                                              const b200_shot_params *p, float *transforms, int *inst_offsets,
                                              b200_corr *inst_corrs, int corr_cap, int *n_inst, b200_corr *corrs_out,
                                              int *n_corrs);

/* ---------------------------------------------------------------------------------------------------------------
 * Hypothesis verification: pcl::GlobalHypothesesVerification<PointT, PointT> as SHOT_hypothesis.cpp:631-653 drives
 * it after ICP — setSceneCloud (:639), addModels(registered_instances, true) (:640), setInlierThreshold /
 * setOcclusionThreshold / setRegularizer / setRadiusClutter / setClutterRegularizer / setDetectClutter /
 * setRadiusNormals (:642-648), verify (:650), getMask (:651).  The object mirrors that call order, because PCL's
 * results depend on it: the scene is voxelised with the resolution in force at setSceneCloud, the models are
 * occlusion-filtered with the occlusion threshold in force at addModels (the reference sets its own value only
 * afterwards, so the constructor default 0.005 applies), everything else is read at verify.
 *
 * On the device: the scene voxel grid, the scene and per-hypothesis z-buffers (focal length from the cloud's
 * extent, depth maps by atomic minimum), the visibility filter, the hypotheses' voxel grids and radius normals, the
 * radius search of every hypothesis point in the scene (explained points, their weights, the outliers), the
 * occupancy grid of the complete models, and the simulated-annealing search over the hypothesis mask (one CTA; the
 * shuffle and acceptance streams — glibc rand() and mt19937, both never seeded by PCL — are generated on the host
 * and consumed in order).  Only detect_clutter = 0 (the reference's setting) is implemented; B200_ERR_INVALID
 * otherwise.  Input points must be finite (the reference removes NaNs first, SHOT.cpp:298-299): non-finite rows are
 * skipped.  See DESIGN.md for the recalled PCL details this rests on.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct b200_hv b200_hv;
typedef struct {
  float resolution;               /* HypothesisVerification::resolution_, 0.005: voxel size of scene and hypotheses */
  float inlier_threshold;         /* setInlierThreshold (hv_inlier_th_, SHOT_hypothesis.cpp:59) */
  float occlusion_threshold;      /* setOcclusionThreshold; read when the models are added */
  float regularizer;              /* setRegularizer (hv_regularizer_) */
  float radius_normals;           /* setRadiusNormals (hv_rad_normals_) */
  float res_occupancy_grid;       /* 0.01 */
  float w_occupied_multiple_cm;   /* 4 */
  float initial_temp;             /* 1000 */
  int max_iterations;             /* 5000: annealing stops after this many iterations without improvement */
  int occlusion_reasoning;        /* unused by the object API (addModels' argument); kept for layout parity with tests */
  int zbuffer_scene_resolution;   /* 100 */
  int zbuffer_self_resolution;    /* 75 */
  float self_occlusion_threshold; /* 0.005 */
  int detect_clutter;             /* setDetectClutter; must be 0 at verify */
  float radius_clutter;           /* setRadiusClutter: accepted, unused without the clutter cue */
  float clutter_regularizer;      /* setClutterRegularizer: accepted, unused without the clutter cue */
  unsigned rand_seed;             /* srand() state std::random_shuffle draws from (1: never seeded) */
  unsigned mt_seed;               /* 5489: default-constructed mt19937 */
  int sa_uniform_mode;            /* 0: x / 2^32; 1: the raw 32-bit value (uphill moves never accepted) */
} b200_hv_params;
typedef struct {
  int valid;           /* addModel succeeded (the visible cloud has points) */
  int n_visible;       /* points left by the self- and scene-occlusion filters */
  int n_points;        /* after VoxelGrid and the NaN-normal compaction */
  int n_outliers;      /* points with no scene point within the inlier threshold (bad_information_) */
  int n_explained;     /* scene points explained by the hypothesis */
  int n_occupancy;     /* occupancy-grid cells of the complete model */
  float outliers_weight;
  float explained_sum; /* float32 sum of the explained weights, in scene order */
} b200_hv_info;
B200_API void b200_hv_params_default(b200_hv_params *p); /* PCL's constructor defaults */
B200_API int b200_hv_create(b200_ctx *ctx, const b200_hv_params *p /* nullable: defaults */, b200_hv **out);
B200_API int b200_hv_destroy(b200_hv *hv);
B200_API int b200_hv_set_params(b200_hv *hv, const b200_hv_params *p);                       /* the set* calls */
B200_API int b200_hv_set_scene(b200_ctx *ctx, b200_hv *hv, const float *scene_xyz, int n, int stride); /* setSceneCloud */
/* addModels: H clouds concatenated (host rows), model_offsets[H + 1] in points.  Replaces earlier models. */
B200_API int b200_hv_add_models(b200_ctx *ctx, b200_hv *hv, const float *models_xyz, const int *model_offsets, int H,
                                int stride, int occlusion_reasoning);
/* verify + getMask.  mask: H bytes (1 = the hypothesis survives).  info (nullable): H entries.  best_cost /
 * accepted_moves (nullable): the annealing's best cost and its number of accepted moves. */
B200_API int b200_hv_verify(b200_ctx *ctx, b200_hv *hv, unsigned char *mask, b200_hv_info *info, double *best_cost,
                            int *accepted_moves);
/* Sizes / contents of the last verify: which = 0 scene points after the NaN-normal compaction (size only), 1
 * occupancy cells (size only), 2 explained scene indices, 3 explained weights (float), 4 occupancy cell indices
 * (order within a hypothesis unspecified), 5 per valid hypothesis: list lengths (explained, occupancy) pairs. */
B200_API int b200_hv_last_size(const b200_hv *hv, int which);
B200_API int b200_hv_last_copy(b200_ctx *ctx, const b200_hv *hv, int which, void *dst);
/* The annealing alone on given cue lists (CSR over H hypotheses, host arrays): SAOptimize. */
B200_API int b200_hv_optimize(b200_ctx *ctx, int H, int ns, const int *expl_off, const int *expl_idx, const float *expl_w,
                              const int *occ_off, const int *occ_idx, int n_cells, const float *outliers_weight,
                              const int *bad_information, const b200_hv_params *p, unsigned char *mask,
                              double *best_cost, int *accepted_moves);

/* Statistics of the last descriptor call on this context (for bench records): mean / max number of
 * radius neighbours per keypoint. */
B200_API int b200_last_neighbor_stats(const b200_ctx *ctx, double *mean_nbrs, int *max_nbrs);

/* Rows of the last b200_match / pipeline call that the tensor-core pre-filter could not certify and
 * that were re-evaluated by the exact float32 kernel (-1: the filter was not used).  Recorded only while
 * profiling is enabled; synchronises the stream. */
B200_API int b200_last_match_fallback(b200_ctx *ctx, int *rows);
/* Rows the one-term first pass of the filter left to the three-term second pass (-1: no such pass ran). */
B200_API int b200_last_match_pass1_rows(b200_ctx *ctx, int *rows);
/* Largest observed |approximate - exact| candidate distance of the last filtered match, divided by the
 * error bound the certificate assumes (must stay well below 1).  Profiling only; synchronises. */
B200_API int b200_last_match_error_ratio(b200_ctx *ctx, float *ratio);

#ifdef __cplusplus
}
#endif
#endif /* B200REG_H_ */
