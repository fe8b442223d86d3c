"""ctypes binding of libb200ppf.so (include/b200ppf.h) — the only way Python reaches the kernels.

There is no CPU fallback: loading fails loudly when the library has not been built, and
Context() fails loudly when no sm_100 GPU is usable.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

from . import build as _build

FEATURE_PCL_PFH, FEATURE_DROST_COS, FEATURE_DROST_ANGLE = 0, 1, 2
ALPHA_MODE_A, ALPHA_MODE_B = 0, 1
NALPHA_CEIL, NALPHA_FLOOR_DROP, NALPHA_FLOOR_CLAMP = 0, 1, 2

HYP_DTYPE = np.dtype(
    [("pose", np.float32, (12,)), ("votes", np.uint32), ("model_index", np.uint32),
     ("alpha_bin", np.uint32), ("scene_index", np.uint32)]
)
SIG_DTYPE = np.dtype([("f1", np.float32), ("f2", np.float32), ("f3", np.float32), ("f4", np.float32),
                      ("alpha_m", np.float32)])
assert HYP_DTYPE.itemsize == 64 and SIG_DTYPE.itemsize == 20


class TableInfo(C.Structure):
    _fields_ = [("n_model", C.c_uint64), ("n_entries", C.c_uint64), ("n_keys", C.c_uint64),
                ("key_space", C.c_uint64), ("n_slices", C.c_uint32), ("slice_rows", C.c_uint32),
                ("n_alpha", C.c_uint32), ("key_bits", C.c_uint32), ("lo", C.c_int32 * 4),
                ("size", C.c_int32 * 4), ("angle_step", C.c_float), ("dist_step", C.c_float),
                ("max_dist", C.c_float), ("phase_cells", C.c_uint32), ("nalpha_rule", C.c_uint32), ("reserved", C.c_uint32),
                ("n_merged", C.c_uint64)]


class Timings(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("upload_ms", "features_ms", "keys_ms", "sort_ms", "csr_ms", "grid_ms",
                                         "vote_ms", "pose_ms", "cluster_ms", "transform_ms", "icp_ms", "prep_ms")]


class IcpParams(C.Structure):
    _fields_ = [("max_iterations", C.c_int), ("tolerance", C.c_float), ("rejection_scale", C.c_float),
                ("num_levels", C.c_int)]


class IcpJob(C.Structure):
    _fields_ = [("model", C.c_void_p), ("scene", C.c_void_p), ("poses16", C.c_void_p), ("n_poses", C.c_size_t),
                ("residuals", C.c_void_p)]


class ObjectParams(C.Structure):
    _fields_ = [("leaf", C.c_float), ("sor_mean_k", C.c_int), ("sor_stddev_mul", C.c_double), ("normal_k", C.c_int),
                ("edge_curvature", C.c_float), ("ref_rate", C.c_uint32), ("pos_thr", C.c_float), ("rot_thr", C.c_float),
                ("icp_poses", C.c_int), ("icp", IcpParams)]


class ObjectResult(C.Structure):
    _fields_ = [("pose", C.c_double * 16), ("residual", C.c_double), ("votes", C.c_uint32), ("n_poses", C.c_uint32),
                ("n_cropped", C.c_uint32), ("n_sampled", C.c_uint32), ("n_filtered", C.c_uint32), ("n_edges", C.c_uint32)] + \
               [(n, C.c_float) for n in ("crop_ms", "voxel_ms", "outlier_ms", "normals_ms", "edges_ms", "match_ms", "icp_ms",
                                         "total_wall_ms")]


class CvObjectParams(C.Structure):
    _fields_ = [("leaf", C.c_float), ("sor_mean_k", C.c_int), ("sor_stddev_mul", C.c_double), ("normal_k", C.c_int),
                ("edge_curvature", C.c_float), ("use_edges", C.c_int), ("relative_scene_sample_step", C.c_double),
                ("relative_scene_distance", C.c_double), ("icp_poses", C.c_int), ("icp", IcpParams)]


class VerifyParams(C.Structure):
    _fields_ = [("inlier_dist", C.c_float), ("normal_angle", C.c_float)]


class PoseFit(C.Structure):
    _fields_ = [("inliers", C.c_uint32), ("visible", C.c_uint32), ("fit", C.c_float), ("rms", C.c_float)]


class Candidate(C.Structure):
    _fields_ = [("pose", C.c_double * 16), ("residual", C.c_double), ("votes", C.c_uint32), ("rank", C.c_uint32), ("fit", PoseFit)]


CANDIDATE_UNUSED = 0xFFFFFFFF  # rank of an unused candidate slot

CV_POSE_DTYPE = np.dtype([("pose", np.float64, (16,)), ("alpha", np.float64), ("residual", np.float64), ("angle", np.float64),
                          ("t", np.float64, (3,)), ("q", np.float64, (4,)), ("model_index", np.uint32), ("num_votes", np.uint32),
                          ("alpha_index", np.uint32), ("reference_index", np.uint32)])
assert CV_POSE_DTYPE.itemsize == 224


class CvInfo(C.Structure):
    _fields_ = [("n_sampled", C.c_uint64), ("table_size", C.c_uint64), ("n_nodes", C.c_uint64), ("n_scene_sampled", C.c_uint64),
                ("n_second_sampled", C.c_uint64), ("angle_step", C.c_double), ("distance_step", C.c_double),
                ("position_threshold", C.c_double), ("rotation_threshold", C.c_double), ("num_angles", C.c_int32),
                ("reserved", C.c_int32)]


# every symbol include/b200ppf.h declares: (name, restype, argtypes)
_vp, _sz, _f, _i = C.c_void_p, C.c_size_t, C.c_float, C.c_int
SYMBOLS = {
    "b200ppf_create": (_i, [_i, C.POINTER(_vp)]),
    "b200ppf_destroy": (None, [_vp]),
    "b200ppf_last_error": (C.c_char_p, [_vp]),
    "b200ppf_version": (_i, []),
    "b200ppf_set_feature_mode": (_i, [_vp, _i]),
    "b200ppf_set_alpha_mode": (_i, [_vp, _i]),
    "b200ppf_set_nalpha_rule": (_i, [_vp, _i]),
    "b200ppf_get_device": (_i, [_vp]),
    "b200ppf_get_stream": (_vp, [_vp]),
    "b200ppf_synchronize": (_i, [_vp]),
    "b200ppf_get_timings": (_i, [_vp, C.POINTER(Timings)]),
    "b200ppf_launch_count": (C.c_uint64, [_vp]),
    "b200ppf_cloud_upload": (_i, [_vp, _vp, _sz, _sz, _sz, C.POINTER(_vp)]),
    "b200ppf_cloud_size": (_sz, [_vp]),
    "b200ppf_cloud_free": (None, [_vp]),
    "b200ppf_features_compute": (_i, [_vp, _vp, C.POINTER(_vp)]),
    "b200ppf_features_upload": (_i, [_vp, _vp, _sz, C.POINTER(_vp)]),
    "b200ppf_features_download": (_i, [_vp, _vp, _sz, _sz, _vp]),
    "b200ppf_features_count": (_sz, [_vp]),
    "b200ppf_features_free": (None, [_vp]),
    "b200ppf_table_build": (_i, [_vp, _vp, _f, _f, C.POINTER(_vp)]),
    "b200ppf_table_build_from_cloud": (_i, [_vp, _vp, _f, _f, C.POINTER(_vp)]),
    "b200ppf_table_get_info": (_i, [_vp, C.POINTER(TableInfo)]),
    "b200ppf_table_query": (_i, [_vp, _vp, _f, _f, _f, _f, _vp, _sz, C.POINTER(_sz)]),
    "b200ppf_table_query_key": (_i, [_vp, _vp, _vp, _vp, _sz, C.POINTER(_sz)]),
    "b200ppf_table_alpha_m": (_i, [_vp, _vp, _vp]),
    "b200ppf_table_export": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "b200ppf_table_clone": (_i, [_vp, _vp, C.POINTER(_vp)]),
    "b200ppf_table_free": (None, [_vp]),
    "b200ppf_table_save": (_i, [_vp, _vp, C.c_char_p]),
    "b200ppf_table_load": (_i, [_vp, C.c_char_p, C.POINTER(_vp)]),
    "b200ppf_vote": (_i, [_vp, _vp, _vp, _vp, _sz, _sz, _sz, _vp]),
    "b200ppf_vote_device": (_i, [_vp, _vp, _vp, _vp, _sz, _sz, _sz, _vp]),
    "b200ppf_vote_scatter_device": (_i, [_vp, _vp, _vp, _vp, _sz, _sz, _sz, _vp, _i, _sz, _sz]),
    "b200ppf_hyp_buffer_create": (_i, [_vp, _sz, C.POINTER(_vp), _vp]),
    "b200ppf_hyp_buffer_open": (_i, [_vp, _vp, C.POINTER(_vp)]),
    "b200ppf_hyp_buffer_download": (_i, [_vp, _vp, _sz, _sz, _vp]),
    "b200ppf_hyp_buffer_release": (_i, [_vp, _vp, _i]),
    "b200ppf_group_create": (_i, [_vp, _i, _i, _sz, C.POINTER(_vp), _vp]),
    "b200ppf_group_connect": (_i, [_vp, _vp]),
    "b200ppf_group_destroy": (None, [_vp]),
    "b200ppf_group_vote": (_i, [_vp, _vp, _vp, _vp, _sz]),
    "b200ppf_group_cluster": (_i, [_vp, _vp, _vp, _vp, _sz, _f, _f, _vp, _vp, _vp, C.POINTER(_sz)]),
    "b200ppf_group_register": (_i, [_vp, _vp, _vp, _vp, _sz, _f, _f, _vp, _vp, _vp, C.POINTER(_sz)]),
    "b200ppf_group_records": (_vp, [_vp]),
    "b200ppf_multi_create": (_i, [_vp, _i, C.POINTER(_vp)]),
    "b200ppf_multi_destroy": (None, [_vp]),
    "b200ppf_multi_size": (_i, [_vp]),
    "b200ppf_multi_context": (_vp, [_vp, _i]),
    "b200ppf_multi_table": (_vp, [_vp, _i]),
    "b200ppf_multi_last_error": (C.c_char_p, [_vp]),
    "b200ppf_multi_train": (_i, [_vp, _vp, _sz, _sz, _sz, _f, _f]),
    "b200ppf_multi_adopt": (_i, [_vp, _vp, _sz, _sz, _sz, _vp]),
    "b200ppf_multi_load": (_i, [_vp, _vp, _sz, _sz, _sz, C.c_char_p]),
    "b200ppf_multi_scene": (_i, [_vp, _vp, _sz, _sz, _sz]),
    "b200ppf_multi_register": (_i, [_vp, _sz, _f, _f, _vp, _vp, _vp, C.POINTER(_sz)]),
    "b200ppf_vote_stats": (_i, [_vp, _vp]),
    "b200ppf_vote_debug_pairs": (_i, [_vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "b200ppf_vote_debug_accumulator": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "b200ppf_debug_alpha_bins": (_i, [_vp, _f, _i, _i, _vp, _vp, _sz, _vp, _vp]),
    "b200ppf_debug_radix_sort": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, C.c_uint64, _i, C.POINTER(_i)]),
    "b200ppf_debug_lower_bounds": (_i, [_vp, _vp, C.c_uint32, C.c_int64, C.c_uint32, C.c_uint32, _vp, _sz]),
    "b200ppf_debug_flag_scan": (_i, [_vp, _vp, C.c_uint32, _vp, _sz, _i, C.POINTER(C.c_uint32)]),
    "b200ppf_debug_scan_rows": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, _sz, _vp, _sz]),
    "b200ppf_debug_run_heads": (_i, [_vp, _vp, C.c_uint32, _vp, _sz]),
    "b200ppf_microbench_atoms": (_i, [_vp, _i, C.POINTER(C.c_double)]),
    "b200ppf_cluster": (_i, [_vp, _vp, _sz, _f, _f, _vp, _vp, C.POINTER(_sz)]),
    "b200ppf_cluster_device": (_i, [_vp, _vp, _sz, _f, _f, _vp, _vp, C.POINTER(_sz)]),
    "b200ppf_cluster_assignment": (_i, [_vp, _vp, _sz, C.POINTER(_sz)]),
    "b200ppf_icp_refine": (_i, [_vp, _vp, _vp, C.POINTER(IcpParams), _vp, _sz, _vp, C.POINTER(C.c_uint64)]),
    "b200ppf_icp_refine_batch": (_i, [_vp, C.POINTER(IcpJob), _sz, C.POINTER(IcpParams), C.POINTER(C.c_uint64)]),
    "b200ppf_transform": (_i, [_vp, _vp, _vp, _vp, _sz]),
    "b200ppf_cloud_upload_xyz": (_i, [_vp, _vp, _sz, _sz, C.POINTER(_vp)]),
    "b200ppf_cloud_download": (_i, [_vp, _vp, _vp, _sz, _sz, _sz]),
    "b200ppf_voxel_grid": (_i, [_vp, _vp, _vp, C.POINTER(_vp)]),
    "b200ppf_knn": (_i, [_vp, _vp, _i, _vp, _vp]),
    "b200ppf_statistical_outlier_removal": (_i, [_vp, _vp, _i, C.c_double, C.POINTER(_vp), _vp, _vp,
                                                 C.POINTER(C.c_double)]),
    "b200ppf_normal_estimation": (_i, [_vp, _vp, _i, _vp, _i]),
    "b200ppf_curvature_edges": (_i, [_vp, _vp, _f, C.POINTER(_vp)]),
    "b200ppf_normalize_normals": (_i, [_vp, _vp]),
    "b200ppf_frustum_corners": (_i, [_vp, _i, _i, _i, _i, _i, _i, C.c_double, C.c_double, C.c_double, C.c_double, _vp]),
    "b200ppf_crop_pyramid": (_i, [_vp, _vp, _vp, C.POINTER(_vp), _vp]),
    "b200ppf_crop_pyramids": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "b200ppf_debug_knn_host": (_i, [_vp, _sz, _sz, _i, _i, _f, _vp, _i, _vp, _vp, _vp, _vp]),
    "b200ppf_object_params_default": (None, [C.POINTER(ObjectParams)]),
    "b200ppf_match_object": (_i, [_vp, _vp, _vp, _vp, _vp, C.POINTER(ObjectParams), C.POINTER(ObjectResult), C.POINTER(_vp),
                                  C.POINTER(_vp)]),
    "b200ppf_match_frame": (_i, [_vp, _vp, _sz, _vp, _vp, _vp, C.POINTER(ObjectParams), C.POINTER(ObjectResult), _vp]),
    "b200ppf_verify_params_default": (None, [C.POINTER(VerifyParams)]),
    "b200ppf_score_poses": (_i, [_vp, C.POINTER(IcpJob), _sz, C.POINTER(VerifyParams), C.POINTER(PoseFit)]),
    "b200ppf_match_frame_verified": (_i, [_vp, _vp, _sz, _vp, _vp, _vp, C.POINTER(ObjectParams), C.POINTER(VerifyParams),
                                          C.POINTER(ObjectResult), _vp, C.POINTER(Candidate)]),
    "b200cv_match_frame_verified": (_i, [_vp, _vp, _sz, _vp, _vp, _vp, C.POINTER(CvObjectParams), C.POINTER(VerifyParams),
                                         C.POINTER(ObjectResult), _vp, C.POINTER(Candidate)]),
    "b200ppf_register": (_i, [_vp, _vp, _vp, _vp, _sz, _f, _f, _vp, _vp, _vp, C.POINTER(_sz)]),
    "b200cv_detector_create": (_i, [_vp, C.c_double, C.c_double, C.c_double, C.POINTER(_vp)]),
    "b200cv_detector_free": (None, [_vp]),
    "b200cv_detector_set_search_params": (_i, [_vp, C.c_double, C.c_double]),
    "b200cv_detector_train": (_i, [_vp, _vp, _sz, _sz]),
    "b200cv_detector_get_info": (_i, [_vp, C.POINTER(CvInfo)]),
    "b200cv_detector_model_points": (_i, [_vp, _vp]),
    "b200cv_detector_scene_points": (_i, [_vp, _vp]),
    "b200cv_detector_match": (_i, [_vp, _vp, _sz, _sz, C.c_double, C.c_double, _vp, _sz, C.POINTER(_sz)]),
    "b200cv_detector_match_s2b": (_i, [_vp, _vp, _sz, _sz, _vp, _sz, _sz, C.c_double, C.c_double, _vp, _sz, C.POINTER(_sz)]),
    "b200cv_detector_match_cloud": (_i, [_vp, _vp, _vp, C.c_double, C.c_double, _vp, _sz, C.POINTER(_sz)]),
    "b200cv_object_params_default": (None, [C.POINTER(CvObjectParams)]),
    "b200cv_match_object": (_i, [_vp, _vp, _vp, _vp, C.POINTER(CvObjectParams), C.POINTER(ObjectResult), C.POINTER(_vp),
                                 C.POINTER(_vp)]),
    "b200cv_match_frame": (_i, [_vp, _vp, _sz, _vp, _vp, _vp, C.POINTER(CvObjectParams), C.POINTER(ObjectResult), _vp]),
    "b200cv_detector_bucket": (_i, [_vp, _sz, _vp, _sz, C.POINTER(_sz)]),
    "b200cv_detector_table_export": (_i, [_vp, _vp, _vp, _vp]),
    "b200cv_detector_raw_poses": (_i, [_vp, _vp, _sz, C.POINTER(_sz)]),
    "b200cv_detector_debug_accumulator": (_i, [_vp, _vp, _sz, _sz, _vp, _sz, _sz, C.c_double, C.c_double, _sz, _vp]),
}

_lib = None


class B200PPFError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b200ppf error {code}: {msg}")
        self.code = code


def lib() -> C.CDLL:
    """Load libb200ppf.so from the in-tree build directory (never from site-packages)."""
    global _lib
    if _lib is None:
        path = os.environ.get("B200PPF_LIB", _build.LIB_PATH)  # override = tuning variants of the same library
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: run `python -m yolo_ppf_pose_estimation_b200.build` "
                "(or __graft_entry__.build()). There is no CPU fallback.")
        L = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError here == missing export
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _alive(ctx) -> bool:
    return bool(getattr(ctx, "_h", None) and ctx._h.value)


def _as_ptr(x):
    """numpy array, int address (e.g. torch.Tensor.data_ptr()) or None -> c_void_p"""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return _p(x)
    return C.c_void_p(int(x))


class Context:
    """One GPU, one stream.  One context per process/rank."""

    def __init__(self, device: int = 0, feature_mode: int = FEATURE_PCL_PFH, alpha_mode: int = ALPHA_MODE_A,
                 nalpha_rule: int = NALPHA_CEIL):
        self._h = C.c_void_p()
        # the handles made on this context (clouds, tables, detectors, ...): the library needs them freed before the
        # context is destroyed, which garbage collection of a reference cycle holding both would not guarantee
        self._owned = weakref.WeakSet()
        rc = lib().b200ppf_create(device, C.byref(self._h))
        if rc != 0:
            raise B200PPFError(rc, lib().b200ppf_last_error(None).decode())
        self.check(lib().b200ppf_set_feature_mode(self._h, feature_mode))
        self.check(lib().b200ppf_set_alpha_mode(self._h, alpha_mode))
        self.check(lib().b200ppf_set_nalpha_rule(self._h, nalpha_rule))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            for obj in list(self._owned):
                obj.close()
            lib().b200ppf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != 0:
            raise B200PPFError(rc, lib().b200ppf_last_error(self._h).decode())

    @property
    def device(self):
        return lib().b200ppf_get_device(self._h)

    @property
    def stream(self):
        return lib().b200ppf_get_stream(self._h)

    @property
    def launch_count(self):
        return int(lib().b200ppf_launch_count(self._h))

    def set_alpha_mode(self, mode):
        self.check(lib().b200ppf_set_alpha_mode(self._h, mode))

    def set_nalpha_rule(self, rule):
        """alpha columns of the accumulator: NALPHA_CEIL (default) | NALPHA_FLOOR_DROP | NALPHA_FLOOR_CLAMP; read at table build"""
        self.check(lib().b200ppf_set_nalpha_rule(self._h, rule))

    def set_feature_mode(self, mode):
        self.check(lib().b200ppf_set_feature_mode(self._h, mode))

    def synchronize(self):
        self.check(lib().b200ppf_synchronize(self._h))

    def timings(self):
        t = Timings()
        self.check(lib().b200ppf_get_timings(self._h, C.byref(t)))
        return {n: getattr(t, n) for n, _ in Timings._fields_}

    # ---- clouds -------------------------------------------------------------------------------
    def upload_cloud(self, cloud, stride=None, normal_offset=None):
        """cloud: (N, 6) [x y z nx ny nz] float32 (the reference's cv::Mat layout) or (N, 12) PointNormal."""
        if isinstance(cloud, np.ndarray):
            cloud = np.ascontiguousarray(cloud, np.float32)
            n = cloud.shape[0]
            stride = cloud.shape[1] if stride is None else stride
            ptr = _p(cloud)
        else:  # raw (pinned) host address
            ptr, n = cloud
            ptr = C.c_void_p(int(ptr))
        if normal_offset is None:
            normal_offset = 4 if stride == 12 else 3
        h = C.c_void_p()
        self.check(lib().b200ppf_cloud_upload(self._h, ptr, n, stride, normal_offset, C.byref(h)))
        return Cloud(self, h)

    # ---- scene pre-processing (reference CloudProcessing.h:340-427) --------------------------------
    def upload_xyz(self, xyz):
        """(N, >=3) float32 rows starting with x y z -> device cloud with zero normals"""
        xyz = np.ascontiguousarray(xyz, np.float32)
        h = C.c_void_p()
        self.check(lib().b200ppf_cloud_upload_xyz(self._h, _p(xyz), xyz.shape[0], xyz.shape[1], C.byref(h)))
        return Cloud(self, h)

    def crop_pyramid(self, cloud: "Cloud", corners):
        """CloudProcessor::SceneCropping's ConvexHull + CropHull for one box: -> (cropped Cloud, kept indices)"""
        c12 = np.ascontiguousarray(corners, np.float32).reshape(12)
        kept = np.zeros(cloud.size, np.uint32)
        h = C.c_void_p()
        self.check(lib().b200ppf_crop_pyramid(self._h, cloud._h, _p(c12), C.byref(h), _p(kept)))
        out = Cloud(self, h)
        return out, kept[:out.size].copy()

    def crop_pyramids(self, cloud: "Cloud", corners):
        """SceneCropping for K boxes in one pass over the frame: corners (K, 4, 3) or (K, 12) -> K Clouds, cloud k as
        crop_pyramid(cloud, corners[k]) makes it"""
        c12 = np.ascontiguousarray(corners, np.float32).reshape(-1, 12)
        out = (C.c_void_p * max(1, c12.shape[0]))()
        self.check(lib().b200ppf_crop_pyramids(self._h, cloud._h, _p(c12), c12.shape[0], out))
        return [Cloud(self, C.c_void_p(out[k])) for k in range(c12.shape[0])]

    def voxel_grid(self, cloud: "Cloud", leaf) -> "Cloud":
        """pcl::VoxelGrid<PointXYZ>::filter (Subsampling)"""
        leaf3 = np.ascontiguousarray(np.broadcast_to(np.asarray(leaf, np.float32), (3,)))
        h = C.c_void_p()
        self.check(lib().b200ppf_voxel_grid(self._h, cloud._h, _p(leaf3), C.byref(h)))
        return Cloud(self, h)

    def knn(self, cloud: "Cloud", k):
        """parity hook: (idx (N,k) uint32, d2 (N,k) float32), rows sorted by (d2, index), self included"""
        idx = np.zeros((cloud.size, k), np.uint32)
        d2 = np.zeros((cloud.size, k), np.float32)
        self.check(lib().b200ppf_knn(self._h, cloud._h, k, _p(idx), _p(d2)))
        return idx, d2

    def statistical_outlier_removal(self, cloud: "Cloud", mean_k=50, stddev_mul=1.0):
        """pcl::StatisticalOutlierRemoval<PointXYZ>::filter (OutlierProcessing):
        -> (filtered Cloud, kept indices, mean distances, threshold)"""
        n = cloud.size
        kept = np.zeros(n, np.uint32)
        dist = np.zeros(n, np.float32)
        thr = C.c_double(0.0)
        h = C.c_void_p()
        self.check(lib().b200ppf_statistical_outlier_removal(self._h, cloud._h, mean_k, float(stddev_mul), C.byref(h),
                                                             _p(kept), _p(dist), C.byref(thr)))
        out = Cloud(self, h)
        return out, kept[:out.size].copy(), dist, thr.value

    def normal_estimation(self, cloud: "Cloud", k=30, viewpoint=None, covariance_mode=0):
        """pcl::NormalEstimationOMP::compute with setKSearch(k), in place (normals + curvature)"""
        vp3 = None if viewpoint is None else np.ascontiguousarray(viewpoint, np.float32)
        self.check(lib().b200ppf_normal_estimation(self._h, cloud._h, k, _p(vp3), covariance_mode))

    def curvature_edges(self, cloud: "Cloud", threshold) -> "Cloud":
        """CloudProcessor::EdgeExtraction: points with curvature > threshold"""
        h = C.c_void_p()
        self.check(lib().b200ppf_curvature_edges(self._h, cloud._h, np.float32(threshold), C.byref(h)))
        return Cloud(self, h)

    def normalize_normals(self, cloud: "Cloud"):
        """CloudProcessor::PointCloudXYZNormalToMat's re-normalisation, in place"""
        self.check(lib().b200ppf_normalize_normals(self._h, cloud._h))

    @staticmethod
    def _params(params_cls, default_fn, overrides):
        """defaults, then overrides (fields of params_cls; icp_* for the ICP)"""
        prm = params_cls()
        default_fn(C.byref(prm))
        for k, v in overrides.items():
            if k.startswith("icp_") and k != "icp_poses":
                setattr(prm.icp, k[4:], v)
            else:
                setattr(prm, k, v)
        return prm

    @staticmethod
    def _result(res):
        out = {n: getattr(res, n) for n, _ in ObjectResult._fields_ if n != "pose"}
        out["pose"] = np.array(res.pose, np.float64).reshape(4, 4)
        return out

    def _object_call(self, params_cls, default_fn, call, overrides):
        """the per-object calls: -> (result dict, object Cloud, edges Cloud or None)"""
        prm = self._params(params_cls, default_fn, overrides)
        res = ObjectResult()
        obj, edg = C.c_void_p(), C.c_void_p()
        self.check(call(C.byref(prm), C.byref(res), C.byref(obj), C.byref(edg)))
        return self._result(res), Cloud(self, obj), (Cloud(self, edg) if edg.value else None)

    def _frame_call(self, params_cls, default_fn, call, corners, overrides):
        """the frame calls: -> (result dicts, one per box, int32 status per box)"""
        c12 = np.ascontiguousarray(corners, np.float32).reshape(-1, 12)
        prm = self._params(params_cls, default_fn, overrides)
        res = (ObjectResult * max(1, c12.shape[0]))()
        status = np.zeros(max(1, c12.shape[0]), np.int32)
        self.check(call(c12.shape[0], _p(c12), C.byref(prm), res, _p(status)))
        return [self._result(res[k]) for k in range(c12.shape[0])], status[:c12.shape[0]]

    @staticmethod
    def verify_params(**overrides):
        """VerifyParams: the defaults (inlier_dist 0.01 m, normal_angle 30 degrees), then overrides"""
        prm = VerifyParams()
        lib().b200ppf_verify_params_default(C.byref(prm))
        for k, v in overrides.items():
            setattr(prm, k, v)
        return prm

    @staticmethod
    def _fit(f):
        return {"inliers": f.inliers, "visible": f.visible, "fit": f.fit, "rms": f.rms}

    def _verified_frame_call(self, params_cls, default_fn, call, corners, overrides):
        """the verified frame calls: -> (result dicts, int32 status per box, candidate dicts per box (used slots only,
        best first))"""
        c12 = np.ascontiguousarray(corners, np.float32).reshape(-1, 12)
        K = c12.shape[0]
        vover = {k: overrides.pop(k) for k in ("inlier_dist", "normal_angle") if k in overrides}
        prm = self._params(params_cls, default_fn, overrides)
        vp = self.verify_params(**vover)
        slots = max(prm.icp_poses, 1)
        res = (ObjectResult * max(1, K))()
        status = np.zeros(max(1, K), np.int32)
        cand = (Candidate * max(1, K * slots))()
        self.check(call(K, _p(c12), C.byref(prm), C.byref(vp), res, _p(status), cand))
        per_box = []
        for b in range(K):
            cs = [cand[b * slots + i] for i in range(slots)]
            per_box.append([{"pose": np.array(c.pose, np.float64).reshape(4, 4), "residual": c.residual, "votes": c.votes,
                             "rank": c.rank, "fit": self._fit(c.fit)} for c in cs if c.rank != CANDIDATE_UNUSED])
        return [self._result(res[k]) for k in range(K)], status[:K], per_box

    def score_poses(self, jobs, inlier_dist=None, normal_angle=None):
        """b200ppf_score_poses: jobs = [(model, scene, poses (P,4,4)), ...] -> [list of P fit dicts per job]
        (inliers, visible, fit, rms); None keeps a default (0.01 m, 30 degrees)"""
        over = {k: v for k, v in (("inlier_dist", inlier_dist), ("normal_angle", normal_angle)) if v is not None}
        vp = self.verify_params(**over)
        arrays = [np.ascontiguousarray(np.asarray(p, np.float64).reshape(-1, 4, 4)) for _, _, p in jobs]
        js = (IcpJob * max(1, len(jobs)))()
        for k, ((m, s, _), P) in enumerate(zip(jobs, arrays)):
            js[k] = IcpJob(m._h, s._h, P.ctypes.data, P.shape[0], None)
        total = sum(P.shape[0] for P in arrays)
        fits = (PoseFit * max(1, total))()
        self.check(lib().b200ppf_score_poses(self._h, js, len(jobs), C.byref(vp), fits))
        out, at = [], 0
        for P in arrays:
            out.append([self._fit(fits[at + i]) for i in range(P.shape[0])])
            at += P.shape[0]
        return out

    def cv_match_frame_verified(self, scene: "Cloud", corners, detectors, models, **overrides):
        """cv_match_frame with every candidate pose scored (b200cv_match_frame_verified) and the best one returned ->
        (result dicts, status per box, candidates per box sorted by fit).  overrides: fields of CvObjectParams (icp_* for
        the ICP), inlier_dist and normal_angle for the scoring."""
        n = len(detectors)
        dets, mods = self._handles(detectors, n), self._handles(models, n)
        return self._verified_frame_call(
            CvObjectParams, lib().b200cv_object_params_default,
            lambda k, c, *a: lib().b200cv_match_frame_verified(self._h, scene._h, k, c, dets, mods, *a), corners, dict(overrides))

    def match_frame_verified(self, scene: "Cloud", corners, models, tables, **overrides):
        """match_frame with every candidate pose scored (b200ppf_match_frame_verified), as cv_match_frame_verified"""
        n = len(models)
        mods, tabs = self._handles(models, n), self._handles(tables, n)
        return self._verified_frame_call(
            ObjectParams, lib().b200ppf_object_params_default,
            lambda k, c, *a: lib().b200ppf_match_frame_verified(self._h, scene._h, k, c, mods, tabs, *a), corners, dict(overrides))

    @staticmethod
    def _handles(objs, n):
        return (C.c_void_p * max(1, n))(*[None if o is None else o._h for o in objs])

    def match_object(self, scene: "Cloud", corners, model: "Cloud", table: "Table", **overrides):
        """One YOLO box start to finish (src/YOLO_cropping_ppf_test.cpp:91-122) on device handles:
        -> (result dict, object Cloud, edges Cloud or None).  overrides: fields of ObjectParams (icp_* for the ICP)."""
        c12 = np.ascontiguousarray(corners, np.float32).reshape(12)
        return self._object_call(ObjectParams, lib().b200ppf_object_params_default,
                                 lambda *a: lib().b200ppf_match_object(self._h, scene._h, _p(c12), model._h, table._h, *a), overrides)

    def cv_match_object(self, detector: "CvDetector", scene: "Cloud", corners, model: "Cloud", **overrides):
        """match_object with the engine the reference calls (b200cv_match_object): pre-processing -> Matching_S2B
        (use_edges=0: Matching) with a trained CvDetector -> ICP of the best clusters against model (the full model).
        overrides: fields of CvObjectParams (icp_* for the ICP)."""
        c12 = np.ascontiguousarray(corners, np.float32).reshape(12)
        return self._object_call(CvObjectParams, lib().b200cv_object_params_default,
                                 lambda *a: lib().b200cv_match_object(detector._h, scene._h, _p(c12), model._h, *a), overrides)

    def cv_match_frame(self, scene: "Cloud", corners, detectors, models, **overrides):
        """every box of a frame in one call (b200cv_match_frame): corners (K, 4, 3), detectors / models one per box ->
        (K result dicts as cv_match_object gives them, status per box: 0 or the per-object call's error code).
        crop_ms, icp_ms and total_wall_ms are the frame's, repeated in every result."""
        n = len(detectors)
        dets, mods = self._handles(detectors, n), self._handles(models, n)
        return self._frame_call(CvObjectParams, lib().b200cv_object_params_default,
                                lambda k, c, *a: lib().b200cv_match_frame(self._h, scene._h, k, c, dets, mods, *a), corners, overrides)

    def match_frame(self, scene: "Cloud", corners, models, tables, **overrides):
        """match_object for every box of a frame in one call (b200ppf_match_frame), as cv_match_frame"""
        n = len(models)
        mods, tabs = self._handles(models, n), self._handles(tables, n)
        return self._frame_call(ObjectParams, lib().b200ppf_object_params_default,
                                lambda k, c, *a: lib().b200ppf_match_frame(self._h, scene._h, k, c, mods, tabs, *a), corners, overrides)

    # ---- K1 / K2 -------------------------------------------------------------------------------
    def features_compute(self, model: "Cloud") -> "Features":
        h = C.c_void_p()
        self.check(lib().b200ppf_features_compute(self._h, model._h, C.byref(h)))
        return Features(self, h)

    def features_upload(self, feats) -> "Features":
        feats = np.ascontiguousarray(feats, np.float32).reshape(-1, 5)
        h = C.c_void_p()
        self.check(lib().b200ppf_features_upload(self._h, _p(feats), feats.shape[0], C.byref(h)))
        return Features(self, h)

    def table_build(self, feats: "Features", angle_step, dist_step) -> "Table":
        h = C.c_void_p()
        self.check(lib().b200ppf_table_build(self._h, feats._h, np.float32(angle_step), np.float32(dist_step),
                                             C.byref(h)))
        return Table(self, h)

    def table_build_from_cloud(self, model: "Cloud", angle_step, dist_step) -> "Table":
        h = C.c_void_p()
        self.check(lib().b200ppf_table_build_from_cloud(self._h, model._h, np.float32(angle_step),
                                                        np.float32(dist_step), C.byref(h)))
        return Table(self, h)

    def icp_refine(self, model: "Cloud", scene: "Cloud", poses, max_iterations=100, tolerance=0.005,
                   rejection_scale=2.5, num_levels=8):
        """ICP::registerModelToScene(model, scene, poses): -> (refined (P,4,4) float64, residuals, iterations)"""
        P = np.ascontiguousarray(np.asarray(poses, np.float64).reshape(-1, 4, 4)).copy()
        res = np.zeros(P.shape[0], np.float64)
        it = C.c_uint64(0)
        prm = IcpParams(max_iterations, tolerance, rejection_scale, num_levels)
        self.check(lib().b200ppf_icp_refine(self._h, model._h, scene._h, C.byref(prm), _p(P), P.shape[0], _p(res),
                                            C.byref(it)))
        return P, res, int(it.value)

    def icp_refine_batch(self, jobs, max_iterations=100, tolerance=0.005, rejection_scale=2.5, num_levels=8):
        """several registerModelToScene problems in one call: jobs = [(model, scene, poses), ...] ->
        ([(refined (P,4,4), residuals) per job], total iterations)"""
        arrays = []
        for _, _, p in jobs:
            P = np.ascontiguousarray(np.asarray(p, np.float64).reshape(-1, 4, 4)).copy()
            arrays.append((P, np.zeros(P.shape[0], np.float64)))
        js = (IcpJob * max(1, len(jobs)))()
        for k, ((m, s, _), (P, r)) in enumerate(zip(jobs, arrays)):
            js[k] = IcpJob(m._h, s._h, P.ctypes.data, P.shape[0], r.ctypes.data)
        it = C.c_uint64(0)
        prm = IcpParams(max_iterations, tolerance, rejection_scale, num_levels)
        self.check(lib().b200ppf_icp_refine_batch(self._h, js, len(jobs), C.byref(prm), C.byref(it)))
        return arrays, int(it.value)

    def table_load(self, path) -> "Table":
        """LoadTrainedDetector: rebuild a saved table on this context's device (no K1/K2)."""
        h = C.c_void_p()
        self.check(lib().b200ppf_table_load(self._h, os.fsencode(path), C.byref(h)))
        return Table(self, h)

    # ---- K3 -----------------------------------------------------------------------------------
    def vote(self, model, table, scene, ref_first=0, ref_step=1, ref_count=None):
        if ref_count is None:
            ref_count = (scene.size - ref_first + ref_step - 1) // ref_step
        hyps = np.zeros(ref_count, HYP_DTYPE)
        self.check(lib().b200ppf_vote(self._h, model._h, table._h, scene._h, ref_first, ref_step, ref_count,
                                      _p(hyps)))
        return hyps

    def vote_device(self, model, table, scene, ref_first, ref_step, ref_count, hyps_device_ptr):
        """Asynchronous on the context stream; hyps_device_ptr is a device address (64 B per reference)."""
        self.check(lib().b200ppf_vote_device(self._h, model._h, table._h, scene._h, ref_first, ref_step,
                                             ref_count, _as_ptr(hyps_device_ptr)))

    def hyp_buffer_create(self, n_records):
        """-> (device address, 64-byte IPC handle) of a record buffer peers can map"""
        ptr = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        self.check(lib().b200ppf_hyp_buffer_create(self._h, n_records, C.byref(ptr), handle))
        return ptr.value, bytes(handle)

    def hyp_buffer_open(self, handle: bytes):
        ptr = C.c_void_p()
        buf = (C.c_ubyte * 64).from_buffer_copy(handle)
        self.check(lib().b200ppf_hyp_buffer_open(self._h, buf, C.byref(ptr)))
        return ptr.value

    def hyp_buffer_release(self, ptr, opened_from_handle):
        self.check(lib().b200ppf_hyp_buffer_release(self._h, C.c_void_p(ptr), 1 if opened_from_handle else 0))

    def vote_scatter_device(self, model, table, scene, ref_first, ref_step, ref_count, peer_ptrs, slot_first, slot_step):
        """vote + pose; record k goes to slot slot_first + k*slot_step of every buffer in peer_ptrs (device addresses)"""
        arr = (C.c_void_p * len(peer_ptrs))(*peer_ptrs)
        self.check(lib().b200ppf_vote_scatter_device(self._h, model._h, table._h, scene._h, ref_first, ref_step, ref_count,
                                                     arr, len(peer_ptrs), slot_first, slot_step))

    def download_hypotheses(self, ptr, n):
        """records of a device buffer -> numpy (synchronises the context stream)"""
        out = np.zeros(n, HYP_DTYPE)
        self.check(lib().b200ppf_hyp_buffer_download(self._h, C.c_void_p(ptr), 0, n, _p(out)))
        return out

    def vote_stats(self):
        s = np.zeros(4, np.uint64)
        self.check(lib().b200ppf_vote_stats(self._h, _p(s)))
        return dict(zip(("pairs_examined", "pairs_in_radius", "nonempty_lookups", "votes"), (int(x) for x in s)))

    def vote_debug_pairs(self, table, scene, s_r):
        n = scene.size
        inr = np.zeros(n, np.uint8)
        d = np.zeros((n, 4), np.int32)
        a = np.zeros(n, np.float32)
        self.check(lib().b200ppf_vote_debug_pairs(self._h, table._h, scene._h, s_r, _p(inr), _p(d), _p(a)))
        return inr, d, a

    def vote_debug_accumulator(self, table, scene, s_r):
        info = table.info
        acc = np.zeros((info.n_model, info.n_alpha), np.uint32)
        self.check(lib().b200ppf_vote_debug_accumulator(self._h, table._h, scene._h, s_r, _p(acc)))
        return acc

    def microbench_atoms(self, pattern=1):
        """measured shared-memory reduction rate (atomics/s): 0 conflict-free, 1 random words, 2 one word"""
        v = C.c_double(0.0)
        self.check(lib().b200ppf_microbench_atoms(self._h, pattern, C.byref(v)))
        return v.value

    # ---- sorted-key primitives: parity hooks (copies in, one run, whole arrays back) ------------------
    def debug_radix_sort(self, keys, max_key, v0=None, v1=None, v0_iota=False):
        """radix_sort_u32 -> (keys, v0, v1, result_in_alt): the arrays holding the sorted data, None for a payload not
        given.  v0_iota: the sort takes v0 to be 0..n-1 and never reads the v0 given."""
        sets = [None if a is None else np.array(a, np.uint32).reshape(-1) for a in (keys, v0, v1)]
        if any(a is not None and a.size != sets[0].size for a in sets):
            raise ValueError("payloads must have one word per key")
        alts = [None if a is None else np.zeros_like(a) for a in sets]
        alt = C.c_int(0)
        self.check(lib().b200ppf_debug_radix_sort(self._h, _p(sets[0]), _p(alts[0]), _p(sets[1]), _p(alts[1]), _p(sets[2]),
                                                  _p(alts[2]), sets[0].size, int(max_key), int(bool(v0_iota)), C.byref(alt)))
        out = alts if alt.value else sets
        return out[0], out[1], out[2], bool(alt.value)

    def debug_lower_bounds(self, sorted_keys, n_keys, shift, dev_len=None, offsets=None):
        """lower_bounds -> offsets, the whole array (default n_keys + 1 zeros; words past n_keys are the caller's canary).
        dev_len: the list length, read from device memory (None: len(sorted_keys), passed by value)"""
        s = np.ascontiguousarray(sorted_keys, np.uint32).reshape(-1)
        off = np.zeros(n_keys + 1, np.uint32) if offsets is None else np.array(offsets, np.uint32).reshape(-1)
        self.check(lib().b200ppf_debug_lower_bounds(self._h, _p(s), s.size, -1 if dev_len is None else int(dev_len), n_keys,
                                                    shift, _p(off), off.size))
        return off

    def debug_flag_scan(self, flags, rank=None, host_total=False, total=0):
        """flag_scan (host_total: flag_scan_host) -> (rank, total): rank the whole array (default len(flags) zeros), total
        the device total's value before the call"""
        f = np.ascontiguousarray(flags, np.uint32).reshape(-1)
        r = np.zeros(f.size, np.uint32) if rank is None else np.array(rank, np.uint32).reshape(-1)
        t = C.c_uint32(total)
        self.check(lib().b200ppf_debug_flag_scan(self._h, _p(f), f.size, _p(r), r.size, int(bool(host_total)), C.byref(t)))
        return r, t.value

    def debug_scan_rows(self, data, n_rows, row_len, totals=None):
        """scan_rows -> (data, totals), whole arrays: data is n_rows * row_len words and whatever follows them, totals
        n_rows words by default"""
        d = np.array(data, np.uint32).reshape(-1)
        t = np.zeros(n_rows, np.uint32) if totals is None else np.array(totals, np.uint32).reshape(-1)
        self.check(lib().b200ppf_debug_scan_rows(self._h, _p(d), n_rows, row_len, d.size, _p(t), t.size))
        return d, t

    def debug_run_heads(self, sorted_keys, head=None):
        """run_heads -> head, the whole array (default len(sorted_keys) zeros)"""
        s = np.ascontiguousarray(sorted_keys, np.uint32).reshape(-1)
        h = np.zeros(s.size, np.uint32) if head is None else np.array(head, np.uint32).reshape(-1)
        self.check(lib().b200ppf_debug_run_heads(self._h, _p(s), s.size, _p(h), h.size))
        return h

    # ---- K4 / K5 / align ------------------------------------------------------------------------
    def cluster(self, hyps, pos_thr=0.01, rot_thr=20.0 / 180.0 * np.pi, device_ptr=None, n=None):
        poses = np.zeros((3, 16), np.float32)
        votes = np.zeros(3, np.uint32)
        k = C.c_size_t(0)
        if device_ptr is not None:
            self.check(lib().b200ppf_cluster_device(self._h, _as_ptr(device_ptr), n, np.float32(pos_thr),
                                                    np.float32(rot_thr), _p(poses), _p(votes), C.byref(k)))
        else:
            hyps = np.ascontiguousarray(hyps, HYP_DTYPE)
            self.check(lib().b200ppf_cluster(self._h, _p(hyps), hyps.shape[0], np.float32(pos_thr),
                                             np.float32(rot_thr), _p(poses), _p(votes), C.byref(k)))
        return poses[:k.value].reshape(-1, 4, 4), votes[:k.value]

    def cluster_assignment(self, n):
        a = np.zeros(n, np.uint32)
        ncl = C.c_size_t(0)
        self.check(lib().b200ppf_cluster_assignment(self._h, _p(a), n, C.byref(ncl)))
        return a, int(ncl.value)

    def transform(self, cloud, pose16):
        M = np.ascontiguousarray(pose16, np.float32).reshape(16)
        out = np.zeros((cloud.size, 3), np.float32)
        self.check(lib().b200ppf_transform(self._h, cloud._h, _p(M), _p(out), 3))
        return out

    def register(self, model, table, scene, ref_rate=5, pos_thr=0.01, rot_thr=20.0 / 180.0 * np.pi):
        final = np.zeros(16, np.float32)
        poses = np.zeros((3, 16), np.float32)
        votes = np.zeros(3, np.uint32)
        k = C.c_size_t(0)
        self.check(lib().b200ppf_register(self._h, model._h, table._h, scene._h, ref_rate, np.float32(pos_thr),
                                          np.float32(rot_thr), _p(final), _p(poses), _p(votes), C.byref(k)))
        return final.reshape(4, 4), poses[:k.value].reshape(-1, 4, 4), votes[:k.value]


class CvDetector:
    """cv::ppf_match_3d::PPF3DDetector(relativeSamplingStep, relativeDistanceStep = 0.05, numAngles = 30) on the device
    (b200cv_*; reference include/CloudProcessing.h:205-236, :442, :495)."""

    def __init__(self, ctx: "Context", relative_sampling_step, relative_distance_step=0.05, num_angles=30):
        self.ctx = ctx
        self._h = C.c_void_p()
        ctx.check(lib().b200cv_detector_create(ctx._h, float(relative_sampling_step), float(relative_distance_step),
                                               float(num_angles), C.byref(self._h)))
        ctx._owned.add(self)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            if _alive(self.ctx):  # a detector whose context is gone went with it
                lib().b200cv_detector_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_search_params(self, position_threshold=-1.0, rotation_threshold=-1.0):
        self.ctx.check(lib().b200cv_detector_set_search_params(self._h, float(position_threshold), float(rotation_threshold)))

    def train_model(self, model):
        m = np.ascontiguousarray(model, np.float32)
        self.ctx.check(lib().b200cv_detector_train(self._h, _p(m), m.shape[0], m.shape[1]))
        return self

    @property
    def info(self) -> CvInfo:
        ci = CvInfo()
        self.ctx.check(lib().b200cv_detector_get_info(self._h, C.byref(ci)))
        return ci

    def model_points(self):
        out = np.zeros((self.info.n_sampled, 6), np.float32)
        self.ctx.check(lib().b200cv_detector_model_points(self._h, _p(out)))
        return out

    def scene_points(self):
        out = np.zeros((self.info.n_scene_sampled, 6), np.float32)
        self.ctx.check(lib().b200cv_detector_scene_points(self._h, _p(out)))
        return out

    def _match(self, scene, edge, sample_step, distance, max_poses):
        s = np.ascontiguousarray(scene, np.float32)
        res = np.zeros(max_poses, CV_POSE_DTYPE)
        k = C.c_size_t(0)
        if edge is None:
            self.ctx.check(lib().b200cv_detector_match(self._h, _p(s), s.shape[0], s.shape[1], float(sample_step), float(distance),
                                                       _p(res), max_poses, C.byref(k)))
        else:
            e = np.ascontiguousarray(edge, np.float32)
            self.ctx.check(lib().b200cv_detector_match_s2b(self._h, _p(s), s.shape[0], s.shape[1], _p(e), e.shape[0], e.shape[1],
                                                           float(sample_step), float(distance), _p(res), max_poses, C.byref(k)))
        return res[:min(k.value, max_poses)], int(k.value)

    def match_cloud(self, scene: "Cloud", edge: "Cloud | None" = None, relative_scene_sample_step=1.0 / 5.0,
                    relative_scene_distance=0.03, max_poses=16):
        """match (edge None) / match_S2B on device clouds of the detector's context; returns what match returns"""
        res = np.zeros(max_poses, CV_POSE_DTYPE)
        k = C.c_size_t(0)
        self.ctx.check(lib().b200cv_detector_match_cloud(self._h, scene._h, None if edge is None else edge._h, float(relative_scene_sample_step),
                                                         float(relative_scene_distance), _p(res), max_poses, C.byref(k)))
        return res[:min(k.value, max_poses)], int(k.value)

    def match(self, scene, relative_scene_sample_step=1.0 / 5.0, relative_scene_distance=0.03, max_poses=16):
        """-> (pose clusters best first as CV_POSE_DTYPE records, number of clusters)"""
        return self._match(scene, None, relative_scene_sample_step, relative_scene_distance, max_poses)

    def match_s2b(self, scene, edge, relative_scene_sample_step=1.0 / 5.0, relative_scene_distance=0.03, max_poses=16):
        return self._match(scene, edge, relative_scene_sample_step, relative_scene_distance, max_poses)

    def raw_poses(self):
        """the per-reference poses of the last match, before clustering"""
        k = C.c_size_t(0)
        self.ctx.check(lib().b200cv_detector_raw_poses(self._h, None, 0, C.byref(k)))
        out = np.zeros(k.value, CV_POSE_DTYPE)
        self.ctx.check(lib().b200cv_detector_raw_poses(self._h, _p(out), k.value, C.byref(k)))
        return out

    def bucket(self, b):
        k = C.c_size_t(0)
        self.ctx.check(lib().b200cv_detector_bucket(self._h, int(b), None, 0, C.byref(k)))
        out = np.zeros(k.value, np.uint32)
        if k.value:
            self.ctx.check(lib().b200cv_detector_bucket(self._h, int(b), _p(out), k.value, C.byref(k)))
        return out

    def table_export(self):
        ci = self.info
        off = np.zeros(ci.table_size + 1, np.uint32)
        nodes = np.zeros(ci.n_nodes, np.uint32)
        alpha = np.zeros(ci.n_sampled * ci.n_sampled, np.float32)
        self.ctx.check(lib().b200cv_detector_table_export(self._h, _p(off), _p(nodes), _p(alpha)))
        return off, nodes, alpha

    def accumulator(self, scene, reference, relative_scene_sample_step, relative_scene_distance, edge=None):
        """accumulator (M, numAngles) of reference point number `reference` (the reference-th of the sampled references)"""
        s = np.ascontiguousarray(scene, np.float32)
        ci = self.info
        acc = np.zeros((ci.n_sampled, ci.num_angles), np.uint32)
        e = None if edge is None else np.ascontiguousarray(edge, np.float32)
        self.ctx.check(lib().b200cv_detector_debug_accumulator(self._h, _p(s), s.shape[0], s.shape[1], _p(e), 0 if e is None else e.shape[0],
                                                               0 if e is None else e.shape[1], float(relative_scene_sample_step),
                                                               float(relative_scene_distance), int(reference), _p(acc)))
        return acc


GROUP_HANDLE_BYTES = 192


class Group:
    """One rank of a multi-process group (one process / context per GPU): b200ppf_group_*."""

    def __init__(self, ctx: "Context", rank: int, world: int, n_records: int):
        self.ctx, self.rank, self.world = ctx, rank, world
        self._h = C.c_void_p()
        self.handles = np.zeros(GROUP_HANDLE_BYTES, np.uint8)
        ctx.check(lib().b200ppf_group_create(ctx._h, rank, world, n_records, C.byref(self._h), _p(self.handles)))
        ctx._owned.add(self)

    def connect(self, all_handles):
        """all_handles: the `handles` blobs of every rank, in rank order (world x 192 bytes)"""
        blob = np.ascontiguousarray(np.concatenate([np.asarray(h, np.uint8).reshape(-1) for h in all_handles]))
        assert blob.size == self.world * GROUP_HANDLE_BYTES
        self.ctx.check(lib().b200ppf_group_connect(self._h, _p(blob)))

    def vote(self, model, table, scene, ref_rate=1):
        self.ctx.check(lib().b200ppf_group_vote(self._h, model._h, table._h, scene._h, ref_rate))

    def cluster(self, model, table, scene, ref_rate=1, pos_thr=0.01, rot_thr=20.0 / 180.0 * np.pi):
        final = np.zeros(16, np.float32)
        poses = np.zeros((3, 16), np.float32)
        votes = np.zeros(3, np.uint32)
        k = C.c_size_t(0)
        self.ctx.check(lib().b200ppf_group_cluster(self._h, model._h, table._h, scene._h, ref_rate, np.float32(pos_thr),
                                                   np.float32(rot_thr), _p(final), _p(poses), _p(votes), C.byref(k)))
        return poses[:k.value].reshape(-1, 4, 4), votes[:k.value]

    def register(self, model, table, scene, ref_rate=1, pos_thr=0.01, rot_thr=20.0 / 180.0 * np.pi):
        self.vote(model, table, scene, ref_rate)
        return self.cluster(model, table, scene, ref_rate, pos_thr, rot_thr)

    def records(self, n):
        """the complete hypothesis set of the last step (synchronises)"""
        return self.ctx.download_hypotheses(lib().b200ppf_group_records(self._h), n)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            if _alive(self.ctx):
                lib().b200ppf_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Multi:
    """Several GPUs driven by this process: b200ppf_multi_* (what the PCL-shaped shim uses for B200PPF_DEVICES=0,1,..)."""

    def __init__(self, devices):
        dev = np.ascontiguousarray(devices, np.int32)
        self._h = C.c_void_p()
        rc = lib().b200ppf_multi_create(_p(dev), len(dev), C.byref(self._h))
        if rc != 0:
            raise B200PPFError(rc, lib().b200ppf_last_error(None).decode())

    def check(self, rc):
        if rc != 0:
            raise B200PPFError(rc, lib().b200ppf_multi_last_error(self._h).decode())

    @property
    def size(self):
        return lib().b200ppf_multi_size(self._h)

    def train(self, model, angle_step, dist_step):
        m = np.ascontiguousarray(model, np.float32)
        self.check(lib().b200ppf_multi_train(self._h, _p(m), m.shape[0], m.shape[1], 3, np.float32(angle_step), np.float32(dist_step)))

    def scene(self, scene):
        s = np.ascontiguousarray(scene, np.float32)
        self.check(lib().b200ppf_multi_scene(self._h, _p(s), s.shape[0], s.shape[1], 3))

    def register(self, ref_rate=5, pos_thr=0.01, rot_thr=20.0 / 180.0 * np.pi):
        final = np.zeros(16, np.float32)
        poses = np.zeros((3, 16), np.float32)
        votes = np.zeros(3, np.uint32)
        k = C.c_size_t(0)
        self.check(lib().b200ppf_multi_register(self._h, ref_rate, np.float32(pos_thr), np.float32(rot_thr), _p(final), _p(poses),
                                                _p(votes), C.byref(k)))
        return final.reshape(4, 4), poses[:k.value].reshape(-1, 4, 4), votes[:k.value]

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().b200ppf_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def debug_alpha_bins(alpha_m, alpha_s, angle_step, alpha_mode=ALPHA_MODE_A, ctx: "Context | None" = None,
                     nalpha_rule=NALPHA_CEIL):
    """(fast, exact) alpha bins; host build of the inline functions when ctx is None, device otherwise."""
    am = np.ascontiguousarray(alpha_m, np.float32)
    as_ = np.ascontiguousarray(alpha_s, np.float32)
    fast = np.zeros(am.shape[0], np.uint32)
    exact = np.zeros(am.shape[0], np.uint32)
    rc = lib().b200ppf_debug_alpha_bins(ctx._h if ctx else None, np.float32(angle_step), alpha_mode, nalpha_rule, _p(am),
                                        _p(as_), am.shape[0], _p(fast), _p(exact))
    if rc != 0:
        raise B200PPFError(rc, lib().b200ppf_last_error(ctx._h if ctx else None).decode())
    return fast, exact


def frustum_corners(depth, box, intrinsics):
    """SceneCropping's four far corners for box = (x, y, w, h), intrinsics = (fx, fy, ppx, ppy): (4, 3) float32"""
    depth = np.ascontiguousarray(depth, np.float32)
    out = np.zeros((4, 3), np.float32)
    fx, fy, ppx, ppy = (float(v) for v in intrinsics)
    rc = lib().b200ppf_frustum_corners(_p(depth), depth.shape[0], depth.shape[1], int(box[0]), int(box[1]), int(box[2]),
                                       int(box[3]), fx, fy, ppx, ppy, _p(out))
    if rc != 0:
        raise B200PPFError(rc, lib().b200ppf_last_error(None).decode())
    return out


def debug_knn_host(xyz, k, mode=0, cell_edge=0.0, viewpoint=None, covariance_mode=0):
    """The device kernels' neighbour query (one __host__ __device__ function) run on the CPU: a test hook.
    mode 0 -> (idx, d2); 1 -> mean distances to the k-1 nearest other points; 2 -> (N, 4) normals + curvature."""
    xyz = np.ascontiguousarray(xyz, np.float32)
    n = xyz.shape[0]
    idx = np.zeros((n, k), np.uint32) if mode == 0 else None
    d2 = np.zeros((n, k), np.float32) if mode == 0 else None
    dist = np.zeros(n, np.float32) if mode == 1 else None
    nrm = np.zeros((n, 4), np.float32) if mode == 2 else None
    vp3 = None if viewpoint is None else np.ascontiguousarray(viewpoint, np.float32)
    rc = lib().b200ppf_debug_knn_host(_p(xyz), n, xyz.shape[1], k, mode, np.float32(cell_edge), _p(vp3), covariance_mode,
                                      _p(idx), _p(d2), _p(dist), _p(nrm))
    if rc != 0:
        raise B200PPFError(rc, lib().b200ppf_last_error(None).decode())
    return (idx, d2) if mode == 0 else (dist if mode == 1 else nrm)


class _Handle:
    _free = None

    def __init__(self, ctx, h):
        self.ctx, self._h = ctx, h
        ctx._owned.add(self)

    def free(self):
        if self._h is not None and self._h.value:
            if _alive(self.ctx):  # a handle whose context is gone went with it
                getattr(lib(), self._free)(self._h)
            self._h = None

    close = free  # what Context.close calls on everything it owns

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Cloud(_Handle):
    _free = "b200ppf_cloud_free"

    @property
    def size(self):
        return int(lib().b200ppf_cloud_size(self._h))

    def download(self, curvature=False):
        """-> (N, 6) [x y z nx ny nz] (the reference's cv::Mat layout), or (N, 7) with the curvature last"""
        stride = 7 if curvature else 6
        out = np.zeros((self.size, stride), np.float32)
        self.ctx.check(lib().b200ppf_cloud_download(self.ctx._h, self._h, _p(out), stride, 3, 6 if curvature else 0))
        return out


class Features(_Handle):
    _free = "b200ppf_features_free"

    @property
    def count(self):
        return int(lib().b200ppf_features_count(self._h))

    def download(self, first=0, count=None):
        count = self.count - first if count is None else count
        out = np.zeros((count, 5), np.float32)
        self.ctx.check(lib().b200ppf_features_download(self.ctx._h, self._h, first, count, _p(out)))
        return out


class Table(_Handle):
    _free = "b200ppf_table_free"

    @property
    def info(self) -> TableInfo:
        ti = TableInfo()
        self.ctx.check(lib().b200ppf_table_get_info(self._h, C.byref(ti)))
        return ti

    def save(self, path):
        self.ctx.check(lib().b200ppf_table_save(self.ctx._h, self._h, os.fsencode(path)))

    def query(self, f1, f2, f3, f4):
        cap = 4096
        while True:
            out = np.zeros((cap, 2), np.uint64)
            n = C.c_size_t(0)
            self.ctx.check(lib().b200ppf_table_query(self.ctx._h, self._h, f1, f2, f3, f4, _p(out), cap, C.byref(n)))
            if n.value <= cap:
                return out[:n.value]
            cap = n.value

    def query_key(self, d):
        d = np.ascontiguousarray(d, np.int32)
        cap = 4096
        while True:
            out = np.zeros((cap, 2), np.uint64)
            n = C.c_size_t(0)
            self.ctx.check(lib().b200ppf_table_query_key(self.ctx._h, self._h, _p(d), _p(out), cap, C.byref(n)))
            if n.value <= cap:
                return out[:n.value]
            cap = n.value

    def alpha_m(self):
        n = self.info.n_model
        out = np.zeros((n, n), np.float32)
        self.ctx.check(lib().b200ppf_table_alpha_m(self.ctx._h, self._h, _p(out)))
        return out

    def export(self):
        """-> offsets (n_slices*key_space+1), entry_i, entry_j, entry_alpha_m"""
        ti = self.info
        off = np.zeros(ti.n_slices * ti.key_space + 1, np.uint32)
        ei = np.zeros(ti.n_entries, np.uint32)
        ej = np.zeros(ti.n_entries, np.uint32)
        ea = np.zeros(ti.n_entries, np.float32)
        self.ctx.check(lib().b200ppf_table_export(self.ctx._h, self._h, _p(off), _p(ei), _p(ej), _p(ea)))
        return off, ei, ej, ea

    def unpack_key(self, packed):
        """packed key (within one slice) -> the four quantised components PCL hashes"""
        ti = self.info
        packed = np.asarray(packed, np.int64)
        c = packed % ti.size[2]
        r = packed // ti.size[2]
        b = r % ti.size[1]
        r = r // ti.size[1]
        a = r % ti.size[0]
        e = r // ti.size[0]
        return np.stack([a + ti.lo[0], b + ti.lo[1], c + ti.lo[2], e + ti.lo[3]], axis=-1).astype(np.int32)
