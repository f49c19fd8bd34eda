"""ctypes mirror of include/b200reg.h (the C ABI of libb200reg.so).

Tests and bench.py call the CUDA path through this module, i.e. through the same entry points the
PCL-style C++ adapters (include/pcl_b200/) bind.  Nothing here computes anything: if the shared
library is missing or no B200 is present the calls raise — there is no CPU fallback.
"""
import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200reg.so")
_LIB = None

CORR_DTYPE = np.dtype([("index_query", "<i4"), ("index_match", "<i4"), ("distance", "<f4")])

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_CAPACITY, ERR_NODEVICE = 0, -1, -2, -3, -4, -5

EXPORTS = [
    "b200_ctx_create", "b200_ctx_destroy", "b200_ctx_sync", "b200_last_error", "b200_abi_version",
    "b200_ctx_launch_count", "b200_cloud_create", "b200_dev_cloud_create", "b200_cloud_destroy", "b200_cloud_size",
    "b200_radius_search", "b200_knn_search", "b200_normals", "b200_dev_normals", "b200_shot_lrf", "b200_shot352",
    "b200_dev_shot352", "b200_fpfh33", "b200_dev_fpfh33", "b200_match", "b200_dev_match", "b200_gc_recognize",
    "b200_model_create_shot", "b200_model_destroy", "b200_model_size", "b200_model_download",
    "b200_register_scene_shot", "b200_dev_register_scene_shot", "b200_last_neighbor_stats",
    "b200_ctx_set_blocking_sync", "b200_ctx_set_profiling", "b200_ctx_reset_profiling", "b200_ctx_stage_count", "b200_ctx_stage_name",
    "b200_ctx_stage_time", "b200_last_match_fallback", "b200_last_match_error_ratio", "b200_last_match_pass1_rows", "b200_comm_unique_id", "b200_comm_init", "b200_comm_destroy",
    "b200_comm_rank", "b200_comm_size", "b200_model_create_fpfh", "b200_model_descriptor_length",
    "b200_register_scene_fpfh", "b200_gather_correspondences", "b200_register_scene_shot_sharded",
    "b200_desc_index_create", "b200_desc_index_destroy", "b200_desc_index_size", "b200_desc_index_knn",
    "b200_uniform_sampling", "b200_dev_uniform_sampling", "b200_voxel_grid", "b200_dev_voxel_grid",
    "b200_library_create", "b200_library_destroy", "b200_library_add_view", "b200_library_views",
    "b200_library_add_view_descriptors", "b200_library_set_view_pose", "b200_library_get_view_pose",
    "b200_library_save", "b200_library_load", "b200_register_scene_batch_shot", "b200_lanes_release",
    "b200_library_view_size", "b200_library_download_view", "b200_register_scene_library",
    "b200_hough3d_recognize",
    "b200_icp_align",
    "b200_remove_nan",
    "b200_transform_points",
    "b200_board_params_default",
    "b200_ctx_srand",
    "b200_board_lrf",
    "b200_model_create_shot_hough", "b200_model_download_frames", "b200_register_scene_shot_hough",
    "b200_dev_register_scene_shot_hough", "b200_register_scene_batch_shot_hough",
    "b200_hv_params_default", "b200_hv_create", "b200_hv_destroy", "b200_hv_set_params", "b200_hv_set_scene",
    "b200_hv_add_models", "b200_hv_verify", "b200_hv_last_size", "b200_hv_last_copy", "b200_hv_optimize",
]


class B200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libb200reg error %d: %s" % (code, msg))
        self.code = code


class Corr(C.Structure):
    _fields_ = [("index_query", C.c_int), ("index_match", C.c_int), ("distance", C.c_float)]


class ShotParams(C.Structure):
    _fields_ = [("normal_k", C.c_int), ("normal_radius", C.c_double), ("descr_radius", C.c_double),
                ("match_mode", C.c_int), ("match_thr", C.c_float), ("gc_size", C.c_double),
                ("gc_threshold", C.c_int), ("max_instances", C.c_int)]


def shot_params(normal_k=10, normal_radius=0.0, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02,
                gc_threshold=2, max_instances=256):
    return ShotParams(int(normal_k), float(normal_radius), float(descr_radius), int(match_mode), float(match_thr),
                      float(gc_size), int(gc_threshold), int(max_instances))


class BoardParams(C.Structure):
    _fields_ = [("find_holes", C.c_int), ("tangent_radius", C.c_float), ("margin_thresh", C.c_float),
                ("check_margin_array_size", C.c_int), ("hole_size_prob_thresh", C.c_float), ("steep_thresh", C.c_float)]


def board_params(find_holes=True, tangent_radius=0.0, margin_thresh=0.85, check_margin_array_size=24,
                 hole_size_prob_thresh=0.2, steep_thresh=0.1):
    """PCL's constructor defaults, with find_holes as the reference sets it (SHOT.cpp:442)."""
    return BoardParams(int(find_holes), float(tangent_radius), float(margin_thresh), int(check_margin_array_size),
                       float(hole_size_prob_thresh), float(steep_thresh))


class HoughParams(C.Structure):
    """b200_hough_params: BOARD frames + Hough3DGrouping of the resident Hough branch."""
    _fields_ = [("rf_radius", C.c_double), ("board", BoardParams), ("bin_size", C.c_double), ("threshold", C.c_double)]


def hough_params(rf_radius=0.02, bin_size=0.02, threshold=2.0, **board):
    """The reference's Hough branch (SHOT_scenes.cpp:54-55: rf_rad_ / cg_size_ 0.02, cg_thresh_ 2); keyword
    arguments go to board_params (find_holes on)."""
    return HoughParams(float(rf_radius), board_params(**board), float(bin_size), float(threshold))


class HvParams(C.Structure):
    """b200_hv_params (pcl::GlobalHypothesesVerification's members; SHOT_hypothesis.cpp:58-64, 642-648)."""
    _fields_ = [("resolution", C.c_float), ("inlier_threshold", C.c_float), ("occlusion_threshold", C.c_float),
                ("regularizer", C.c_float), ("radius_normals", C.c_float), ("res_occupancy_grid", C.c_float),
                ("w_occupied_multiple_cm", C.c_float), ("initial_temp", C.c_float), ("max_iterations", C.c_int),
                ("occlusion_reasoning", C.c_int), ("zbuffer_scene_resolution", C.c_int),
                ("zbuffer_self_resolution", C.c_int), ("self_occlusion_threshold", C.c_float),
                ("detect_clutter", C.c_int), ("radius_clutter", C.c_float), ("clutter_regularizer", C.c_float),
                ("rand_seed", C.c_uint), ("mt_seed", C.c_uint), ("sa_uniform_mode", C.c_int)]


HV_INFO_DTYPE = np.dtype([("valid", "<i4"), ("n_visible", "<i4"), ("n_points", "<i4"), ("n_outliers", "<i4"),
                          ("n_explained", "<i4"), ("n_occupancy", "<i4"), ("outliers_weight", "<f4"),
                          ("explained_sum", "<f4")])


def hv_params(**kw):
    """PCL's constructor defaults, overridden by keyword."""
    p = HvParams()
    lib().b200_hv_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError("unknown hypothesis-verification parameter %r" % k)
        setattr(p, k, v)
    return p


def lib():
    """Loads libb200reg.so; raises (loudly) if it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libb200reg.so is missing (%s): build it with __graft_entry__.build(); "
                               "there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, fp, ip = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)
        i, d, f = C.c_int, C.c_double, C.c_float
        sig = {
            "b200_ctx_create": [C.POINTER(vp), i, vp],
            "b200_ctx_destroy": [vp],
            "b200_ctx_sync": [vp],
            "b200_cloud_create": [vp, fp, i, i, C.POINTER(vp)],
            "b200_dev_cloud_create": [vp, vp, i, i, C.POINTER(vp)],
            "b200_cloud_destroy": [vp],
            "b200_cloud_size": [vp],
            "b200_radius_search": [vp, vp, fp, i, i, d, C.POINTER(C.c_int64), ip, fp, C.c_int64,
                                   C.POINTER(C.c_int64)],
            "b200_knn_search": [vp, vp, fp, i, i, i, ip, fp, ip],
            "b200_normals": [vp, vp, fp, i, i, i, d, fp, fp],
            "b200_dev_normals": [vp, vp, vp, i, i, i, d, fp, vp],
            "b200_shot_lrf": [vp, vp, fp, i, i, d, fp],
            "b200_shot352": [vp, vp, fp, fp, i, i, d, fp, fp],
            "b200_dev_shot352": [vp, vp, vp, vp, i, i, d, vp, vp],
            "b200_fpfh33": [vp, vp, fp, fp, i, i, d, fp],
            "b200_dev_fpfh33": [vp, vp, vp, vp, i, i, d, vp],
            "b200_match": [vp, fp, i, fp, i, i, i, f, C.POINTER(Corr), ip],
            "b200_dev_match": [vp, vp, i, vp, i, i, i, f, vp, vp],
            "b200_gc_recognize": [vp, fp, i, i, fp, i, i, C.POINTER(Corr), i, d, i, fp, i, ip, C.POINTER(Corr), i, ip],
            "b200_model_create_shot": [vp, fp, i, i, fp, i, i, C.POINTER(ShotParams), C.POINTER(vp)],
            "b200_model_destroy": [vp],
            "b200_model_size": [vp],
            "b200_model_download": [vp, vp, fp, fp],
            "b200_register_scene_shot": [vp, vp, fp, i, i, fp, i, i, C.POINTER(ShotParams), fp, ip, C.POINTER(Corr), i,
                                         ip, C.POINTER(Corr), ip],
            "b200_dev_register_scene_shot": [vp, vp, vp, i, i, vp, i, i, C.POINTER(ShotParams), vp, vp, vp, vp, i, vp,
                                             vp, vp, vp],
            "b200_last_neighbor_stats": [vp, C.POINTER(d), ip],
            "b200_ctx_set_blocking_sync": [vp, i],
            "b200_ctx_set_profiling": [vp, i],
            "b200_ctx_reset_profiling": [vp],
            "b200_ctx_stage_count": [],
            "b200_ctx_stage_time": [vp, i, C.POINTER(d), ip],
            "b200_last_match_fallback": [vp, ip],
            "b200_last_match_pass1_rows": [vp, ip],
            "b200_model_create_fpfh": [vp, fp, i, i, C.POINTER(ShotParams), C.POINTER(vp)],
            "b200_model_descriptor_length": [vp],
            "b200_register_scene_fpfh": [vp, vp, fp, i, i, C.POINTER(ShotParams), fp, ip, C.POINTER(Corr), i, ip,
                                         C.POINTER(Corr), ip, fp],
            "b200_comm_unique_id": [vp, C.c_size_t],
            "b200_comm_init": [vp, vp, i, i],
            "b200_comm_destroy": [vp],
            "b200_comm_rank": [vp],
            "b200_comm_size": [vp],
            "b200_gather_correspondences": [vp, vp, vp, i, vp, vp],
            "b200_register_scene_shot_sharded": [vp, vp, i, fp, i, i, fp, i, i, C.POINTER(ShotParams), fp, ip,
                                                 C.POINTER(Corr), i, ip, C.POINTER(Corr), ip],
            "b200_last_match_error_ratio": [vp, fp],
            "b200_desc_index_create": [vp, fp, i, i, C.POINTER(vp)],
            "b200_desc_index_destroy": [vp],
            "b200_desc_index_size": [vp],
            "b200_desc_index_knn": [vp, vp, fp, i, i, ip, fp, ip],
            "b200_uniform_sampling": [vp, fp, i, i, d, fp, ip, ip],
            "b200_dev_uniform_sampling": [vp, vp, i, i, d, vp, vp, vp],
            "b200_voxel_grid": [vp, fp, i, i, f, f, f, fp, ip],
            "b200_dev_voxel_grid": [vp, vp, i, i, f, f, f, vp, vp],
            "b200_hough3d_recognize": [vp, fp, fp, i, i, fp, fp, i, i, C.POINTER(Corr), i, d, d, fp, i, ip, C.POINTER(Corr),
                                       i, ip],
            "b200_board_params_default": [C.POINTER(BoardParams)],
            "b200_ctx_srand": [vp, C.c_uint],
            "b200_board_lrf": [vp, vp, fp, fp, i, i, d, C.POINTER(BoardParams), fp],
            "b200_model_create_shot_hough": [vp, fp, i, i, fp, i, i, C.POINTER(ShotParams), C.POINTER(HoughParams),
                                             C.POINTER(vp)],
            "b200_model_download_frames": [vp, vp, fp],
            "b200_register_scene_shot_hough": [vp, vp, fp, i, i, fp, i, i, C.POINTER(ShotParams), C.POINTER(HoughParams),
                                               fp, ip, C.POINTER(Corr), i, ip, C.POINTER(Corr), ip, fp],
            "b200_dev_register_scene_shot_hough": [vp, vp, vp, i, i, vp, i, i, C.POINTER(ShotParams),
                                                   C.POINTER(HoughParams), vp, vp, vp, vp, i, vp, vp, vp, vp, vp, vp],
            "b200_register_scene_batch_shot_hough": [i, vp, i, C.POINTER(fp), ip, i, C.POINTER(fp), ip, i,
                                                     C.POINTER(ShotParams), C.POINTER(HoughParams), i, C.POINTER(fp),
                                                     C.POINTER(ip), C.POINTER(C.POINTER(Corr)), ip, ip,
                                                     C.POINTER(C.POINTER(Corr)), ip, ip],
            "b200_remove_nan": [vp, fp, i, i, fp, ip, ip],
            "b200_transform_points": [vp, fp, i, i, fp, fp],
            "b200_icp_align": [vp, fp, i, i, vp, i, d, d, d, fp, fp, fp, C.POINTER(d), ip, ip],
            "b200_library_create": [vp, C.POINTER(vp)],
            "b200_library_destroy": [vp],
            "b200_library_add_view": [vp, vp, fp, i, i, fp, i, i, C.POINTER(ShotParams), ip],
            "b200_library_add_view_descriptors": [vp, vp, fp, fp, i, i, ip],
            "b200_library_set_view_pose": [vp, i, fp],
            "b200_library_get_view_pose": [vp, i, fp],
            "b200_library_save": [vp, vp, C.c_char_p],
            "b200_library_load": [vp, C.c_char_p, C.POINTER(vp)],
            "b200_register_scene_batch_shot": [i, vp, i, C.POINTER(fp), ip, i, C.POINTER(fp), ip, i, C.POINTER(ShotParams), i,
                                               C.POINTER(fp), C.POINTER(ip), C.POINTER(C.POINTER(Corr)), ip, ip,
                                               C.POINTER(C.POINTER(Corr)), ip, ip],
            "b200_lanes_release": [i],
            "b200_library_views": [vp],
            "b200_library_view_size": [vp, i],
            "b200_library_download_view": [vp, vp, i, fp, fp],
            "b200_register_scene_library": [vp, vp, fp, i, i, fp, i, i, C.POINTER(ShotParams), fp, ip, ip,
                                            C.POINTER(Corr), i, i, ip, ip],
            "b200_hv_create": [vp, C.POINTER(HvParams), C.POINTER(vp)],
            "b200_hv_destroy": [vp],
            "b200_hv_set_params": [vp, C.POINTER(HvParams)],
            "b200_hv_set_scene": [vp, vp, fp, i, i],
            "b200_hv_add_models": [vp, vp, fp, ip, i, i, i],
            "b200_hv_verify": [vp, vp, C.POINTER(C.c_ubyte), vp, C.POINTER(d), ip],
            "b200_hv_last_size": [vp, i],
            "b200_hv_last_copy": [vp, vp, i, vp],
            "b200_hv_optimize": [vp, i, i, ip, ip, fp, ip, ip, i, fp, ip, C.POINTER(HvParams), C.POINTER(C.c_ubyte),
                                 C.POINTER(d), ip],
        }
        for name, args in sig.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = C.c_int
        L.b200_board_params_default.restype = None
        L.b200_hv_params_default.restype = None
        L.b200_hv_params_default.argtypes = [C.POINTER(HvParams)]
        L.b200_last_error.argtypes = [vp]
        L.b200_last_error.restype = C.c_char_p
        L.b200_ctx_stage_name.argtypes = [i]
        L.b200_ctx_stage_name.restype = C.c_char_p
        L.b200_abi_version.argtypes = []
        L.b200_abi_version.restype = C.c_int
        L.b200_ctx_launch_count.argtypes = [vp]
        L.b200_ctx_launch_count.restype = C.c_int64
        _LIB = L
    return _LIB


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _i(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _c(a):
    return a.ctypes.data_as(C.POINTER(Corr))


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("points must be (n, >=3) float32")
    return a


def _dptr(t):
    """Device pointer of a torch CUDA tensor (or a raw int)."""
    if t is None:
        return None
    if isinstance(t, int):
        return C.c_void_p(t)
    return C.c_void_p(t.data_ptr())


class InstanceList:
    """Per-instance correspondence lists as views into the flat output buffer (pcl's
    std::vector<pcl::Correspondences>): nothing is copied or sliced until an item is asked for."""

    def __init__(self, flat, offsets, n):
        self.flat, self.offsets, self.n = flat, offsets, int(n)

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(self.n))]
        if i < 0:
            i += self.n
        if not 0 <= i < self.n:
            raise IndexError(i)
        return self.flat[self.offsets[i]:self.offsets[i + 1]]

    def __iter__(self):
        return (self[i] for i in range(self.n))


class Cloud:
    def __init__(self, ctx, handle, n):
        self.ctx, self.h, self.n = ctx, handle, n
        ctx._children.add(self)

    def close(self):
        if self.h and self.ctx.h:      # clouds / models must be destroyed before their context
            lib().b200_cloud_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Model:
    def __init__(self, ctx, handle):
        self.ctx, self.h = ctx, handle
        ctx._children.add(self)

    @property
    def size(self):
        return lib().b200_model_size(self.h)

    def download(self):
        K = self.size
        desc = np.zeros((K, lib().b200_model_descriptor_length(self.h)), dtype=np.float32)
        kp = np.zeros((K, 3), dtype=np.float32)
        self.ctx._chk(lib().b200_model_download(self.ctx.h, self.h, _f(desc), _f(kp)))
        return desc, kp

    def download_frames(self):
        """K x 9 BOARD frames of a model from Context.model_create_shot_hough (b200_model_download_frames)."""
        rf = np.zeros((max(self.size, 1), 9), dtype=np.float32)
        self.ctx._chk(lib().b200_model_download_frames(self.ctx.h, self.h, _f(rf)))
        return rf[:self.size]

    def close(self):
        if self.h and self.ctx.h:
            lib().b200_model_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DescIndex:
    def __init__(self, ctx, handle, D):
        self.ctx, self.h, self.D = ctx, handle, D
        ctx._children.add(self)

    @property
    def size(self):
        return lib().b200_desc_index_size(self.h)

    def knn(self, queries, k):
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.D)
        idx = np.zeros((len(q), k), dtype=np.int32)
        d2 = np.zeros((len(q), k), dtype=np.float32)
        kf = C.c_int()
        self.ctx._chk(lib().b200_desc_index_knn(self.ctx.h, self.h, _f(q), len(q), int(k), _i(idx), _f(d2),
                                                C.byref(kf)))
        return idx, d2, kf.value

    def close(self):
        if self.h and self.ctx.h:
            lib().b200_desc_index_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Library:
    """b200_library: descriptor library over the views of the CAD models (CAD_desc.cpp:231-370)."""

    def __init__(self, ctx, handle=None):
        self.ctx = ctx
        h = handle
        if h is None:
            h = C.c_void_p()
            ctx._chk(lib().b200_library_create(ctx.h, C.byref(h)))
        self.h = h
        ctx._children.add(self)

    @classmethod
    def load(cls, ctx, path):
        """Reads a B200LIB1 file written by save() (b200_library_load)."""
        h = C.c_void_p()
        ctx._chk(lib().b200_library_load(ctx.h, os.fsencode(path), C.byref(h)))
        return cls(ctx, h)

    def save(self, path):
        self.ctx._chk(lib().b200_library_save(self.ctx.h, self.h, os.fsencode(path)))

    def add_view_descriptors(self, desc, kp):
        """A view from precomputed descriptors (K x 352) and keypoints, e.g. the reference's text dumps."""
        desc = np.ascontiguousarray(desc, dtype=np.float32).reshape(-1, 352)
        kp = _pts(kp)
        assert len(desc) == len(kp)
        v = C.c_int()
        self.ctx._chk(lib().b200_library_add_view_descriptors(self.ctx.h, self.h, _f(desc), _f(kp), len(kp), kp.shape[1],
                                                              C.byref(v)))
        return v.value

    def set_view_pose(self, v, pose):
        pose = np.ascontiguousarray(pose, dtype=np.float32).reshape(16)
        if lib().b200_library_set_view_pose(self.h, int(v), _f(pose)) != OK:
            raise B200Error(ERR_INVALID, "library: bad view index")

    def view_pose(self, v):
        pose = np.zeros(16, dtype=np.float32)
        if lib().b200_library_get_view_pose(self.h, int(v), _f(pose)) != OK:
            raise B200Error(ERR_INVALID, "library: bad view index")
        return pose.reshape(4, 4)

    def add_view(self, xyz, kp, params):
        xyz, kp = _pts(xyz), _pts(kp)
        v = C.c_int()
        self.ctx._chk(lib().b200_library_add_view(self.ctx.h, self.h, _f(xyz), len(xyz), xyz.shape[1], _f(kp), len(kp),
                                                  kp.shape[1], C.byref(params), C.byref(v)))
        return v.value

    @property
    def views(self):
        return lib().b200_library_views(self.h)

    def view_size(self, v):
        return lib().b200_library_view_size(self.h, int(v))

    def download_view(self, v):
        K = self.view_size(v)
        desc = np.zeros((K, 352), dtype=np.float32)
        kp = np.zeros((K, 3), dtype=np.float32)
        self.ctx._chk(lib().b200_library_download_view(self.ctx.h, self.h, int(v), _f(desc), _f(kp)))
        return desc, kp

    def register_scene(self, scene_xyz, scene_kp, params, max_inst=4096):
        scene_xyz, scene_kp = _pts(scene_xyz), _pts(scene_kp)
        Ks, nv = len(scene_kp), self.views
        cap = max(Ks, 1) * max(nv, 1)
        T = np.empty((max_inst, 16), dtype=np.float32)
        view = np.empty(max_inst, dtype=np.int32)
        off = np.empty(max_inst + 1, dtype=np.int32)
        ic = np.empty(cap, dtype=CORR_DTYPE)
        ncorr = np.zeros(max(nv, 1), dtype=np.int32)
        n = C.c_int()
        rc = lib().b200_register_scene_library(self.ctx.h, self.h, _f(scene_xyz), len(scene_xyz), scene_xyz.shape[1],
                                               _f(scene_kp), Ks, scene_kp.shape[1], C.byref(params), _f(T), _i(view),
                                               _i(off), _c(ic), cap, max_inst, C.byref(n), _i(ncorr))
        if rc not in (OK, ERR_CAPACITY):
            self.ctx._chk(rc)
        m = n.value
        if rc == ERR_CAPACITY:
            import warnings
            warnings.warn("b200_register_scene_library: output capacity exceeded, results truncated", RuntimeWarning,
                          stacklevel=2)
        return {"transforms": T[:m].reshape(m, 4, 4), "view": view[:m], "instances": InstanceList(ic, off, m),
                "n_instances": m, "view_n_corrs": ncorr[:nv], "truncated": rc == ERR_CAPACITY}

    def close(self):
        if self.h and self.ctx.h:
            lib().b200_library_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HypothesisVerification:
    """b200_hv: pcl::GlobalHypothesesVerification in the reference's call order (SHOT_hypothesis.cpp:631-653)."""

    def __init__(self, ctx, params=None):
        self.ctx = ctx
        h = C.c_void_p()
        ctx._chk(lib().b200_hv_create(ctx.h, C.byref(params) if params is not None else None, C.byref(h)))
        self.h = h
        self.H = 0
        ctx._children.add(self)

    def set_params(self, params):
        self.ctx._chk(lib().b200_hv_set_params(self.h, C.byref(params)))

    def set_scene(self, scene_xyz):
        xyz = _pts(scene_xyz)
        self.ctx._chk(lib().b200_hv_set_scene(self.ctx.h, self.h, _f(xyz), len(xyz), xyz.shape[1]))

    def add_models(self, models, occlusion_reasoning=False):
        models = [_pts(m) for m in models]
        offs = np.zeros(len(models) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([len(m) for m in models])
        flat = np.ascontiguousarray(np.concatenate([m[:, :3] for m in models]) if models and offs[-1] > 0
                                    else np.zeros((1, 3), np.float32), dtype=np.float32)
        self.H = len(models)
        self.ctx._chk(lib().b200_hv_add_models(self.ctx.h, self.h, _f(flat), _i(offs), self.H, 3,
                                               1 if occlusion_reasoning else 0))

    def verify(self):
        """verify + getMask.  Returns a dict: mask, info, best_cost, accepted_moves, n_scene_points, n_cells and the cue lists (CSR over the valid hypotheses)."""
        H = self.H
        mask = np.zeros(max(H, 1), dtype=np.uint8)
        info = np.zeros(max(H, 1), dtype=HV_INFO_DTYPE)
        cost, acc = C.c_double(0.0), C.c_int(0)
        self.ctx._chk(lib().b200_hv_verify(self.ctx.h, self.h, mask.ctypes.data_as(C.POINTER(C.c_ubyte)),
                                           info.ctypes.data, C.byref(cost), C.byref(acc)))
        out = {"mask": mask[:H].astype(bool), "info": info[:H], "best_cost": cost.value, "accepted_moves": acc.value,
               "n_scene_points": lib().b200_hv_last_size(self.h, 0), "n_cells": lib().b200_hv_last_size(self.h, 1)}
        arrs = {}
        for which, (name, dt) in {2: ("expl_idx", np.int32), 3: ("expl_w", np.float32), 4: ("occ_idx", np.int32),
                                  5: ("sizes", np.int32)}.items():
            n = lib().b200_hv_last_size(self.h, which)
            a = np.zeros(max(n, 1), dtype=dt)
            if n > 0:
                self.ctx._chk(lib().b200_hv_last_copy(self.ctx.h, self.h, which, a.ctypes.data))
            arrs[name] = a[:n]
        sizes = arrs.pop("sizes").reshape(-1, 2)
        out.update(arrs)
        out["expl_off"] = np.concatenate([[0], np.cumsum(sizes[:, 0])]).astype(np.int32)
        out["occ_off"] = np.concatenate([[0], np.cumsum(sizes[:, 1])]).astype(np.int32)
        return out

    def close(self):
        if self.h and self.ctx.h:
            lib().b200_hv_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """b200_ctx: one per host thread.  stream: a raw cudaStream_t (int), e.g.
    torch.cuda.current_stream().cuda_stream, or None for a private stream."""

    def __init__(self, device=0, stream=None):
        h = C.c_void_p()
        rc = lib().b200_ctx_create(C.byref(h), int(device), C.c_void_p(stream) if stream else None)
        if rc != OK:
            raise B200Error(rc, lib().b200_last_error(None).decode())
        self.h = h
        self._children = weakref.WeakSet()

    def _chk(self, rc):
        if rc != OK:
            raise B200Error(rc, lib().b200_last_error(self.h).decode())

    def close(self):
        if self.h:
            for ch in list(self._children):
                ch.close()
            lib().b200_ctx_destroy(self.h)
            self.h = None

    def set_blocking_sync(self, on=True):
        """Host waits sleep on a blocking event instead of spinning (more lanes than host cores)."""
        self._chk(lib().b200_ctx_set_blocking_sync(self.h, 1 if on else 0))

    def sync(self):
        self._chk(lib().b200_ctx_sync(self.h))

    @property
    def launches(self):
        return int(lib().b200_ctx_launch_count(self.h))

    def set_profiling(self, on=True):
        self._chk(lib().b200_ctx_set_profiling(self.h, 1 if on else 0))

    def reset_profiling(self):
        self._chk(lib().b200_ctx_reset_profiling(self.h))

    def stage_times(self):
        """{stage name: (total ms, calls)} since the last reset (synchronises the stream)."""
        out = {}
        for s in range(lib().b200_ctx_stage_count()):
            ms, n = C.c_double(), C.c_int()
            self._chk(lib().b200_ctx_stage_time(self.h, s, C.byref(ms), C.byref(n)))
            out[lib().b200_ctx_stage_name(s).decode()] = (ms.value, n.value)
        return out

    def match_fallback_rows(self):
        n = C.c_int()
        self._chk(lib().b200_last_match_fallback(self.h, C.byref(n)))
        return n.value

    def match_pass1_rows(self):
        n = C.c_int()
        self._chk(lib().b200_last_match_pass1_rows(self.h, C.byref(n)))
        return n.value

    def match_error_ratio(self):
        r = C.c_float()
        self._chk(lib().b200_last_match_error_ratio(self.h, C.byref(r)))
        return r.value

    def neighbor_stats(self):
        m, mx = C.c_double(), C.c_int()
        lib().b200_last_neighbor_stats(self.h, C.byref(m), C.byref(mx))
        return m.value, mx.value

    # ---- surface ------------------------------------------------------------------------------
    def cloud(self, xyz):
        xyz = _pts(xyz)
        h = C.c_void_p()
        self._chk(lib().b200_cloud_create(self.h, _f(xyz), len(xyz), xyz.shape[1], C.byref(h)))
        return Cloud(self, h, len(xyz))

    def dev_cloud(self, t, n=None, stride=None):
        n = t.shape[0] if n is None else n
        stride = t.shape[1] if stride is None else stride
        h = C.c_void_p()
        self._chk(lib().b200_dev_cloud_create(self.h, _dptr(t), int(n), int(stride), C.byref(h)))
        return Cloud(self, h, n)

    def radius_search(self, cloud, q, radius):
        q = _pts(q)
        off = np.zeros(len(q) + 1, dtype=np.int64)
        total = C.c_int64()
        op = off.ctypes.data_as(C.POINTER(C.c_int64))
        self._chk(lib().b200_radius_search(self.h, cloud.h, _f(q), len(q), q.shape[1], float(radius), op, None, None, 0,
                                           C.byref(total)))
        t = total.value
        idx = np.zeros(max(t, 1), dtype=np.int32)
        d2 = np.zeros(max(t, 1), dtype=np.float32)
        if t:
            self._chk(lib().b200_radius_search(self.h, cloud.h, _f(q), len(q), q.shape[1], float(radius), op, _i(idx),
                                               _f(d2), t, C.byref(total)))
        return off, idx[:t], d2[:t]

    def knn_search(self, cloud, q, k):
        q = _pts(q)
        idx = np.zeros((len(q), k), dtype=np.int32)
        d2 = np.zeros((len(q), k), dtype=np.float32)
        kf = C.c_int()
        self._chk(lib().b200_knn_search(self.h, cloud.h, _f(q), len(q), q.shape[1], int(k), _i(idx), _f(d2),
                                        C.byref(kf)))
        return idx, d2, kf.value

    # ---- features -----------------------------------------------------------------------------
    def normals(self, cloud, q=None, k=0, radius=0.0, viewpoint=None):
        vp = None if viewpoint is None else _f(np.ascontiguousarray(viewpoint, dtype=np.float32))
        if q is None:
            out = np.zeros((cloud.n, 4), dtype=np.float32)
            self._chk(lib().b200_normals(self.h, cloud.h, None, 0, 0, int(k), float(radius), vp, _f(out)))
        else:
            q = _pts(q)
            out = np.zeros((len(q), 4), dtype=np.float32)
            self._chk(lib().b200_normals(self.h, cloud.h, _f(q), len(q), q.shape[1], int(k), float(radius), vp,
                                         _f(out)))
        return out

    def shot_lrf(self, cloud, kp, radius):
        kp = _pts(kp)
        out = np.zeros((len(kp), 9), dtype=np.float32)
        self._chk(lib().b200_shot_lrf(self.h, cloud.h, _f(kp), len(kp), kp.shape[1], float(radius), _f(out)))
        return out

    def shot352(self, cloud, normals, kp, radius):
        kp = _pts(kp)
        normals = np.ascontiguousarray(normals, dtype=np.float32)
        assert normals.shape == (cloud.n, 4)
        desc = np.zeros((len(kp), 352), dtype=np.float32)
        rf = np.zeros((len(kp), 9), dtype=np.float32)
        self._chk(lib().b200_shot352(self.h, cloud.h, _f(normals), _f(kp), len(kp), kp.shape[1], float(radius),
                                     _f(desc), _f(rf)))
        return desc, rf

    def fpfh33(self, cloud, normals, radius, q=None):
        normals = np.ascontiguousarray(normals, dtype=np.float32)
        assert normals.shape == (cloud.n, 4)
        if q is None:
            out = np.zeros((cloud.n, 33), dtype=np.float32)
            self._chk(lib().b200_fpfh33(self.h, cloud.h, _f(normals), None, 0, 0, float(radius), _f(out)))
        else:
            q = _pts(q)
            out = np.zeros((len(q), 33), dtype=np.float32)
            self._chk(lib().b200_fpfh33(self.h, cloud.h, _f(normals), _f(q), len(q), q.shape[1], float(radius),
                                        _f(out)))
        return out

    # ---- hypothesis verification (GlobalHypothesesVerification, SHOT_hypothesis.cpp:631-653) -------
    def hypothesis_verification(self, params=None):
        return HypothesisVerification(self, params)

    def hv_optimize(self, ns, expl_off, expl_idx, expl_w, occ_off, occ_idx, n_cells, outliers_weight,
                    bad_information, params):
        """SAOptimize alone on given cue lists.  Returns (mask, best_cost, accepted_moves)."""
        H = len(expl_off) - 1
        eo = np.ascontiguousarray(expl_off, dtype=np.int32)
        ei = np.ascontiguousarray(np.append(expl_idx, 0), dtype=np.int32)
        ew = np.ascontiguousarray(np.append(expl_w, 0), dtype=np.float32)
        oo = np.ascontiguousarray(occ_off, dtype=np.int32)
        oi = np.ascontiguousarray(np.append(occ_idx, 0), dtype=np.int32)
        ow = np.ascontiguousarray(outliers_weight, dtype=np.float32)
        bi = np.ascontiguousarray(bad_information, dtype=np.int32)
        mask = np.zeros(max(H, 1), dtype=np.uint8)
        cost, acc = C.c_double(0.0), C.c_int(0)
        self._chk(lib().b200_hv_optimize(self.h, H, int(ns), _i(eo), _i(ei), _f(ew), _i(oo), _i(oi), int(n_cells),
                                         _f(ow), _i(bi), C.byref(params), mask.ctypes.data_as(C.POINTER(C.c_ubyte)),
                                         C.byref(cost), C.byref(acc)))
        return mask[:H].astype(bool), cost.value, acc.value

    # ---- per-query descriptor index (KdTreeFLANN<Descriptor> drop-in) -------------------------------
    def desc_index(self, desc):
        desc = np.ascontiguousarray(desc, dtype=np.float32)
        h = C.c_void_p()
        self._chk(lib().b200_desc_index_create(self.h, _f(desc), desc.shape[0], desc.shape[1], C.byref(h)))
        return DescIndex(self, h, desc.shape[1])

    # ---- keypoints ------------------------------------------------------------------------------
    def uniform_sampling(self, xyz, leaf, return_index=False):
        xyz = _pts(xyz)
        out = np.empty((max(len(xyz), 1), 3), dtype=np.float32)
        idx = np.empty(max(len(xyz), 1), dtype=np.int32)
        n = C.c_int()
        self._chk(lib().b200_uniform_sampling(self.h, _f(xyz), len(xyz), xyz.shape[1], float(leaf), _f(out), _i(idx),
                                              C.byref(n)))
        return (out[:n.value].copy(), idx[:n.value].copy()) if return_index else out[:n.value].copy()

    def voxel_grid(self, xyz, leaf):
        xyz = _pts(xyz)
        lx, ly, lz = (leaf, leaf, leaf) if np.isscalar(leaf) else leaf
        out = np.empty((max(len(xyz), 1), 3), dtype=np.float32)
        n = C.c_int()
        self._chk(lib().b200_voxel_grid(self.h, _f(xyz), len(xyz), xyz.shape[1], float(lx), float(ly), float(lz),
                                        _f(out), C.byref(n)))
        return out[:n.value].copy()

    # ---- matching / grouping ------------------------------------------------------------------
    def match(self, model, scene, mode=1, thr=0.25):
        model = np.ascontiguousarray(model, dtype=np.float32)
        scene = np.ascontiguousarray(scene, dtype=np.float32)
        assert model.ndim == 2 and scene.ndim == 2 and model.shape[1] == scene.shape[1]
        out = np.zeros(max(len(scene), 1), dtype=CORR_DTYPE)
        cnt = C.c_int()
        self._chk(lib().b200_match(self.h, _f(model), len(model), _f(scene), len(scene), model.shape[1], int(mode),
                                   float(thr), _c(out), C.byref(cnt)))
        return out[:cnt.value].copy()

    def gc_recognize(self, model_kp, scene_kp, corrs, gc_size, gc_threshold, max_inst=256):
        model_kp, scene_kp = _pts(model_kp), _pts(scene_kp)
        corrs = np.ascontiguousarray(corrs, dtype=CORR_DTYPE)
        T = np.zeros((max_inst, 16), dtype=np.float32)
        off = np.zeros(max_inst + 1, dtype=np.int32)
        cap = max(len(corrs), 1)
        oc = np.zeros(cap, dtype=CORR_DTYPE)
        n = C.c_int()
        rc = lib().b200_gc_recognize(self.h, _f(model_kp), len(model_kp), model_kp.shape[1], _f(scene_kp),
                                     len(scene_kp), scene_kp.shape[1], _c(corrs), len(corrs), float(gc_size),
                                     int(gc_threshold), _f(T), max_inst, _i(off), _c(oc), cap, C.byref(n))
        if rc not in (OK, ERR_CAPACITY):
            self._chk(rc)
        m = min(n.value, max_inst)
        return T[:m].reshape(m, 4, 4).copy(), [oc[off[i]:off[i + 1]].copy() for i in range(m)], n.value

    def hough3d_recognize(self, model_kp, model_rf, scene_kp, scene_rf, corrs, bin_size, threshold, max_inst=256):
        model_kp, scene_kp = _pts(model_kp), _pts(scene_kp)
        model_rf = np.ascontiguousarray(model_rf, dtype=np.float32).reshape(len(model_kp), 9)
        scene_rf = np.ascontiguousarray(scene_rf, dtype=np.float32).reshape(len(scene_kp), 9)
        corrs = np.ascontiguousarray(corrs, dtype=CORR_DTYPE)
        T = np.zeros((max_inst, 16), dtype=np.float32)
        off = np.zeros(max_inst + 1, dtype=np.int32)
        cap = max(len(corrs), 1)
        oc = np.zeros(cap, dtype=CORR_DTYPE)
        n = C.c_int()
        rc = lib().b200_hough3d_recognize(self.h, _f(model_kp), _f(model_rf), len(model_kp), model_kp.shape[1],
                                          _f(scene_kp), _f(scene_rf), len(scene_kp), scene_kp.shape[1], _c(corrs),
                                          len(corrs), float(bin_size), float(threshold), _f(T), max_inst, _i(off), _c(oc),
                                          cap, C.byref(n))
        if rc not in (OK, ERR_CAPACITY):
            self._chk(rc)
        m = min(n.value, max_inst)
        return T[:m].reshape(m, 4, 4).copy(), [oc[off[i]:off[i + 1]].copy() for i in range(m)], n.value

    def remove_nan(self, xyz):
        """pcl::removeNaNFromPointCloud (b200_remove_nan).  Returns (kept rows n x 3, their original indices)."""
        xyz = _pts(xyz)
        out = np.zeros((max(len(xyz), 1), 3), dtype=np.float32)
        idx = np.zeros(max(len(xyz), 1), dtype=np.int32)
        n = C.c_int()
        self._chk(lib().b200_remove_nan(self.h, _f(xyz), len(xyz), xyz.shape[1], _f(out), _i(idx), C.byref(n)))
        return out[:n.value], idx[:n.value]

    def transform_points(self, xyz, transform):
        """pcl::transformPointCloud with a 4x4 matrix (b200_transform_points)."""
        xyz = _pts(xyz)
        T = np.ascontiguousarray(transform, dtype=np.float32).reshape(16)
        out = np.zeros((max(len(xyz), 1), 3), dtype=np.float32)
        self._chk(lib().b200_transform_points(self.h, _f(xyz), len(xyz), xyz.shape[1], _f(T), _f(out)))
        return out[:len(xyz)]

    def srand(self, seed):
        """Reseeds the context's rand() stream (BOARD's random axis), like srand(seed) for PCL."""
        self._chk(lib().b200_ctx_srand(self.h, int(seed)))

    def board_lrf(self, cloud, normals, kp, radius, params=None):
        """pcl::BOARDLocalReferenceFrameEstimation::compute (b200_board_lrf).  Returns K x 9 frames."""
        kp = _pts(kp)
        normals = np.ascontiguousarray(normals, dtype=np.float32).reshape(cloud.n, 4)
        params = params or board_params()
        out = np.zeros((max(len(kp), 1), 9), dtype=np.float32)
        self._chk(lib().b200_board_lrf(self.h, cloud.h, _f(normals), _f(kp), len(kp), kp.shape[1], float(radius),
                                       C.byref(params), _f(out)))
        return out[:len(kp)]

    def icp_align(self, source, target, max_iterations=10, max_corr_dist=0.0, transformation_epsilon=0.0,
                  euclidean_fitness_epsilon=-1.7976931348623157e308, guess=None):
        """pcl::IterativeClosestPoint::align (b200_icp_align).  target: a Cloud.  Returns a dict with
        final_transform (4x4), aligned (ns x 3), fitness, converged, iterations."""
        source = _pts(source)
        T = np.zeros(16, dtype=np.float32)
        al = np.zeros((max(len(source), 1), 3), dtype=np.float32)
        g = None if guess is None else np.ascontiguousarray(guess, dtype=np.float32).reshape(16)
        fit, conv, it = C.c_double(), C.c_int(), C.c_int()
        self._chk(lib().b200_icp_align(self.h, _f(source), len(source), source.shape[1], target.h, int(max_iterations),
                                       float(max_corr_dist), float(transformation_epsilon),
                                       float(euclidean_fitness_epsilon), None if g is None else _f(g), _f(T), _f(al),
                                       C.byref(fit), C.byref(conv), C.byref(it)))
        return {"final_transform": T.reshape(4, 4), "aligned": al[:len(source)], "fitness": fit.value,
                "converged": bool(conv.value), "iterations": it.value}

    # ---- resident pipeline --------------------------------------------------------------------
    def model_create_shot(self, xyz, kp, params):
        xyz, kp = _pts(xyz), _pts(kp)
        h = C.c_void_p()
        self._chk(lib().b200_model_create_shot(self.h, _f(xyz), len(xyz), xyz.shape[1], _f(kp), len(kp), kp.shape[1],
                                               C.byref(params), C.byref(h)))
        return Model(self, h)

    def register_scene_shot(self, model, scene_xyz, scene_kp, params):
        """Host buffers in, host results out (b200_register_scene_shot)."""
        scene_xyz, scene_kp = _pts(scene_xyz), _pts(scene_kp)
        mi = params.max_instances
        Ks = len(scene_kp)
        T = np.empty((mi, 16), dtype=np.float32)       # filled by the library (no zero-fill on the caller's clock)
        off = np.empty(mi + 1, dtype=np.int32)
        ic = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        corrs = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        n_inst, n_corr = C.c_int(), C.c_int()
        rc = lib().b200_register_scene_shot(self.h, model.h, _f(scene_xyz), len(scene_xyz), scene_xyz.shape[1],
                                            _f(scene_kp), Ks, scene_kp.shape[1], C.byref(params), _f(T), _i(off),
                                            _c(ic), max(Ks, 1), C.byref(n_inst), _c(corrs), C.byref(n_corr))
        if rc not in (OK, ERR_CAPACITY):
            self._chk(rc)
        m = min(n_inst.value, mi)
        if rc == ERR_CAPACITY:
            import warnings
            warnings.warn("b200_register_scene_shot: output capacity exceeded (%d instances found, %d kept): %s"
                          % (n_inst.value, m, lib().b200_last_error(self.h).decode()), RuntimeWarning, stacklevel=2)
        return {"transforms": T[:m].reshape(m, 4, 4), "instances": InstanceList(ic, off, m),
                "n_instances": n_inst.value, "corrs": corrs[:n_corr.value], "truncated": rc == ERR_CAPACITY}

    # ---- resident Hough branch (BOARD frames + Hough3DGrouping) ------------------------------------
    def model_create_shot_hough(self, xyz, kp, params, hough):
        """b200_model_create_shot_hough: the SHOT model plus its BOARD frames (drawn from this context's rand()
        stream) and Hough votes."""
        xyz, kp = _pts(xyz), _pts(kp)
        h = C.c_void_p()
        self._chk(lib().b200_model_create_shot_hough(self.h, _f(xyz), len(xyz), xyz.shape[1], _f(kp), len(kp),
                                                     kp.shape[1], C.byref(params), C.byref(hough), C.byref(h)))
        return Model(self, h)

    def register_scene_shot_hough(self, model, scene_xyz, scene_kp, params, hough):
        """Host buffers in, host results out (b200_register_scene_shot_hough).  As register_scene_shot, plus the scene
        frames ("rf", Ks x 9) and the return code ("status": 0, or ERR_CAPACITY when the instances were truncated or
        the Hough space would exceed 2^27 bins)."""
        scene_xyz, scene_kp = _pts(scene_xyz), _pts(scene_kp)
        mi, Ks = params.max_instances, len(scene_kp)
        T = np.empty((mi, 16), dtype=np.float32)
        off = np.zeros(mi + 1, dtype=np.int32)
        ic = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        corrs = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        rf = np.empty((max(Ks, 1), 9), dtype=np.float32)
        n_inst, n_corr = C.c_int(), C.c_int()
        rc = lib().b200_register_scene_shot_hough(self.h, model.h, _f(scene_xyz), len(scene_xyz), scene_xyz.shape[1],
                                                  _f(scene_kp), Ks, scene_kp.shape[1], C.byref(params), C.byref(hough),
                                                  _f(T), _i(off), _c(ic), max(Ks, 1), C.byref(n_inst), _c(corrs),
                                                  C.byref(n_corr), _f(rf))
        if rc not in (OK, ERR_CAPACITY):
            self._chk(rc)
        m = min(n_inst.value, mi)
        return {"transforms": T[:m].reshape(m, 4, 4), "instances": InstanceList(ic, off, m),
                "n_instances": n_inst.value, "corrs": corrs[:n_corr.value], "rf": rf[:Ks], "status": rc}

    def dev_register_scene_shot_hough(self, model, d_xyz, n, stride, d_kp, Ks, kstride, params, hough, out):
        """All buffers resident (torch CUDA tensors in `out`, as dev_register_scene_shot, plus the device int
        out["status"] and optionally out["rf"]), asynchronous (b200_dev_register_scene_shot_hough)."""
        self._chk(lib().b200_dev_register_scene_shot_hough(
            self.h, model.h, _dptr(d_xyz), int(n), int(stride), _dptr(d_kp), int(Ks), int(kstride), C.byref(params),
            C.byref(hough), _dptr(out["transforms"]), _dptr(out["inst_offsets"]), _dptr(out["inst_counts"]),
            _dptr(out["inst_corrs"]), int(out["corr_cap"]), _dptr(out["n_inst"]), _dptr(out["corrs"]),
            _dptr(out["n_corrs"]), _dptr(out.get("desc")), _dptr(out.get("rf")), _dptr(out["status"])))

    # ---- resident FPFH pipeline (FPFH_demo.cpp:405-538) -------------------------------------------
    def model_create_fpfh(self, kp, params):
        kp = _pts(kp)
        h = C.c_void_p()
        self._chk(lib().b200_model_create_fpfh(self.h, _f(kp), len(kp), kp.shape[1], C.byref(params), C.byref(h)))
        return Model(self, h)

    def register_scene_fpfh(self, model, scene_kp, params, want_desc=False):
        scene_kp = _pts(scene_kp)
        mi, Ks = params.max_instances, len(scene_kp)
        T = np.empty((mi, 16), dtype=np.float32)
        off = np.empty(mi + 1, dtype=np.int32)
        ic = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        corrs = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        desc = np.empty((max(Ks, 1), 33), dtype=np.float32) if want_desc else None
        n_inst, n_corr = C.c_int(), C.c_int()
        rc = lib().b200_register_scene_fpfh(self.h, model.h, _f(scene_kp), Ks, scene_kp.shape[1], C.byref(params), _f(T),
                                            _i(off), _c(ic), max(Ks, 1), C.byref(n_inst), _c(corrs), C.byref(n_corr),
                                            _f(desc) if want_desc else None)
        if rc not in (OK, ERR_CAPACITY):
            self._chk(rc)
        m = min(n_inst.value, mi)
        out = {"transforms": T[:m].reshape(m, 4, 4), "instances": InstanceList(ic, off, m),
               "n_instances": n_inst.value, "corrs": corrs[:n_corr.value], "truncated": rc == ERR_CAPACITY}
        if want_desc:
            out["desc"] = desc[:Ks]
        return out

    # ---- multi-GPU (the library's own NCCL communicator) -----------------------------------------
    def comm_init(self, unique_id, rank, world):
        """Collective over the `world` contexts sharing `unique_id` (bytes from comm_unique_id() on one rank)."""
        buf = (C.c_char * 128).from_buffer_copy(bytes(unique_id))
        self._chk(lib().b200_comm_init(self.h, buf, int(rank), int(world)))

    def comm_destroy(self):
        self._chk(lib().b200_comm_destroy(self.h))

    @property
    def comm_rank(self):
        return lib().b200_comm_rank(self.h)

    @property
    def comm_size(self):
        return lib().b200_comm_size(self.h)

    def register_scene_shot_sharded(self, model, params, scene_xyz=None, scene_kp=None, root=0):
        """One scene over all ranks (b200_register_scene_shot_sharded).  Collective; the root passes the scene and
        gets the result dict, the other ranks pass nothing and get None."""
        is_root = self.comm_rank == root
        if not is_root:
            self._chk(lib().b200_register_scene_shot_sharded(self.h, model.h, int(root), None, 0, 3, None, 0, 3,
                                                             C.byref(params), None, None, None, 0, None, None, None))
            return None
        scene_xyz, scene_kp = _pts(scene_xyz), _pts(scene_kp)
        mi, Ks = params.max_instances, len(scene_kp)
        T = np.empty((mi, 16), dtype=np.float32)
        off = np.empty(mi + 1, dtype=np.int32)
        ic = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        corrs = np.empty(max(Ks, 1), dtype=CORR_DTYPE)
        n_inst, n_corr = C.c_int(), C.c_int()
        rc = lib().b200_register_scene_shot_sharded(
            self.h, model.h, int(root), _f(scene_xyz), len(scene_xyz), scene_xyz.shape[1], _f(scene_kp), Ks,
            scene_kp.shape[1], C.byref(params), _f(T), _i(off), _c(ic), max(Ks, 1), C.byref(n_inst), _c(corrs),
            C.byref(n_corr))
        if rc not in (OK, ERR_CAPACITY):
            self._chk(rc)
        m = min(n_inst.value, mi)
        return {"transforms": T[:m].reshape(m, 4, 4), "instances": InstanceList(ic, off, m),
                "n_instances": n_inst.value, "corrs": corrs[:n_corr.value], "truncated": rc == ERR_CAPACITY}

    def dev_register_scene_shot(self, model, d_xyz, n, stride, d_kp, Ks, kstride, params, out):
        """All buffers resident (torch CUDA tensors in `out`), asynchronous (b200_dev_register_scene_shot)."""
        self._chk(lib().b200_dev_register_scene_shot(
            self.h, model.h, _dptr(d_xyz), int(n), int(stride), _dptr(d_kp), int(Ks), int(kstride), C.byref(params),
            _dptr(out["transforms"]), _dptr(out["inst_offsets"]), _dptr(out["inst_counts"]), _dptr(out["inst_corrs"]),
            int(out["corr_cap"]), _dptr(out["n_inst"]), _dptr(out["corrs"]), _dptr(out["n_corrs"]),
            _dptr(out.get("desc"))))

    def dev_normals(self, cloud, d_out, k=0, radius=0.0):
        self._chk(lib().b200_dev_normals(self.h, cloud.h, None, 0, 0, int(k), float(radius), None, _dptr(d_out)))

    def dev_shot352(self, cloud, d_normals, d_kp, K, kstride, radius, d_desc, d_rf=None):
        self._chk(lib().b200_dev_shot352(self.h, cloud.h, _dptr(d_normals), _dptr(d_kp), int(K), int(kstride),
                                         float(radius), _dptr(d_desc), _dptr(d_rf)))

    def dev_match(self, d_model, Km, d_scene, Ks, D, mode, thr, d_out, d_count):
        self._chk(lib().b200_dev_match(self.h, _dptr(d_model), int(Km), _dptr(d_scene), int(Ks), int(D), int(mode),
                                       float(thr), _dptr(d_out), _dptr(d_count)))


def comm_unique_id():
    """128-byte NCCL rendezvous token (b200_comm_unique_id): create on one rank, send to the others."""
    buf = (C.c_char * 128)()
    rc = lib().b200_comm_unique_id(buf, 128)
    if rc != OK:
        raise B200Error(rc, lib().b200_last_error(None).decode())
    return bytes(buf)


def register_scene_batch(model, scenes, keypoints, params, lanes=4, device=0, hough=None):
    """b200_register_scene_batch_shot: a batch of scenes against one resident model, `lanes` scenes in flight on
    `device` (contexts and host threads live inside the library).  Returns one result dict per scene, like
    Context.register_scene_shot.  With `hough` (HoughParams), b200_register_scene_batch_shot_hough: the Hough branch
    against a model from Context.model_create_shot_hough."""
    n = len(scenes)
    scenes = [_pts(x) for x in scenes]
    keypoints = [_pts(k) for k in keypoints]
    stride = scenes[0].shape[1] if n else 3
    kstride = keypoints[0].shape[1] if n else 3
    assert all(x.shape[1] == stride for x in scenes) and all(k.shape[1] == kstride for k in keypoints)
    mi = params.max_instances
    fp, ip, cp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(Corr)
    T = [np.empty((mi, 16), dtype=np.float32) for _ in range(n)]
    off = [np.empty(mi + 1, dtype=np.int32) for _ in range(n)]
    ic = [np.empty(max(len(k), 1), dtype=CORR_DTYPE) for k in keypoints]
    co = [np.empty(max(len(k), 1), dtype=CORR_DTYPE) for k in keypoints]
    npts = np.array([len(x) for x in scenes], dtype=np.int32)
    nkp = np.array([len(k) for k in keypoints], dtype=np.int32)
    cap = np.array([len(a) for a in ic], dtype=np.int32)
    n_inst = np.zeros(max(n, 1), dtype=np.int32)
    n_corr = np.zeros(max(n, 1), dtype=np.int32)
    status = np.zeros(max(n, 1), dtype=np.int32)
    inputs = (int(device), model.h, n, (fp * n)(*[_f(x) for x in scenes]), _i(npts), stride,
              (fp * n)(*[_f(k) for k in keypoints]), _i(nkp), kstride, C.byref(params))
    outputs = (int(lanes), (fp * n)(*[_f(t) for t in T]), (ip * n)(*[_i(o) for o in off]),
               (cp * n)(*[_c(a) for a in ic]), _i(cap), _i(n_inst), (cp * n)(*[_c(a) for a in co]), _i(n_corr),
               _i(status))
    if hough is None:
        rc = lib().b200_register_scene_batch_shot(*inputs, *outputs)
    else:
        rc = lib().b200_register_scene_batch_shot_hough(*inputs, C.byref(hough), *outputs)
    if rc != OK:
        raise B200Error(rc, lib().b200_last_error(None).decode())
    out = []
    for s in range(n):
        m = min(int(n_inst[s]), mi)
        out.append({"transforms": T[s][:m].reshape(m, 4, 4), "instances": InstanceList(ic[s], off[s], m),
                    "n_instances": int(n_inst[s]), "corrs": co[s][:int(n_corr[s])], "status": int(status[s])})
    return out


def lanes_release(device=0):
    """Frees the contexts b200_register_scene_batch_shot keeps for `device`."""
    lib().b200_lanes_release(int(device))


# ---- the reference's text dump of a view's descriptors (CAD_desc.cpp:354-370) ----------------------------------
def read_partial_view_text(path):
    """Partial_View<l>.txt: one float per line (std::ostream default formatting, 6 significant digits), 352 per
    keypoint.  Returns (K, 352) float32.  Feed it to Library.add_view_descriptors with the view's keypoints."""
    vals = np.loadtxt(path, dtype=np.float64, ndmin=1)
    if len(vals) % 352:
        raise ValueError("%s: %d values is not a multiple of 352" % (path, len(vals)))
    return vals.astype(np.float32).reshape(-1, 352)


def write_partial_view_text(path, desc):
    """Writes descriptors the way CAD_desc.cpp does (`myfile << value << std::endl`, i.e. %g)."""
    desc = np.asarray(desc, dtype=np.float32).reshape(-1, 352)
    with open(path, "w") as f:
        for v in desc.reshape(-1):
            f.write("%g\n" % v)
