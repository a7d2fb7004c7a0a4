"""ctypes binding of libmoped_cuda.so (include/moped_cuda.h) — the product's only compute path.

There is no CPU fallback: if the library is missing it is built with nvcc (moped_b200.build), and if
no B200 is visible `Context()` raises. Python here is plumbing for tests and bench.py; C/C++ hosts bind
the same symbols directly (see INTEGRATION.md).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")

MATCH_TENSOR = 0
MATCH_EXACT = 1


class PoseParams(C.Structure):
    _fields_ = [("max_ransac_tests", C.c_int32), ("max_lm_tests", C.c_int32), ("max_objects_per_cluster", C.c_int32),
                ("n_pts_align", C.c_int32), ("min_npts_object", C.c_int32), ("error_threshold", C.c_float), ("seed", C.c_uint64)]

    @classmethod
    def of(cls, params, seed=1):
        """params = (MaxRANSACTests, MaxLMTests, MaxObjectsPerCluster, NPtsAlign, MinNPtsObject, ErrorThreshold)"""
        return cls(int(params[0]), int(params[1]), int(params[2]), int(params[3]), int(params[4]), float(params[5]), int(seed))


class PipelineParams(C.Structure):
    _fields_ = [("match_ratio", C.c_float), ("match_mode", C.c_int32),
                ("cluster_radius", C.c_float), ("cluster_merge", C.c_float), ("cluster_min_pts", C.c_int32), ("cluster_max_iterations", C.c_int32),
                ("pose", PoseParams), ("filter_min_points", C.c_int32), ("filter_feature_distance", C.c_float), ("filter_min_score", C.c_float),
                ("pose2", PoseParams), ("filter2_min_points", C.c_int32), ("filter2_feature_distance", C.c_float), ("filter2_min_score", C.c_float)]


class RigCamera(C.Structure):
    """mc_rig_camera: camera c's image of frame f is height x width bytes at gray + f * frame_stride."""
    _fields_ = [("gray", C.c_void_p), ("frame_stride", C.c_int64), ("height", C.c_int32), ("width", C.c_int32)]


class DepthPipelineParams(C.Structure):
    """mc_depth_pipeline_params: moped3d's CLUSTER_LINKAGE -> POSE -> FILTER -> POSE2 -> FILTER2."""
    _fields_ = [("variant", C.c_int32),
                ("cluster_cutoff", C.c_float), ("cluster_min_pts", C.c_int32), ("cluster_use_3d_filter", C.c_int32), ("cluster_linkage_type", C.c_int32),
                ("cluster_sigma_2d", C.c_float), ("cluster_sigma_3d", C.c_float),
                ("pose", PoseParams), ("pose_alpha", C.c_float),
                ("filter_min_points", C.c_int32), ("filter_feature_distance", C.c_float), ("filter_min_score", C.c_float),
                ("pose2", PoseParams), ("pose2_alpha", C.c_float),
                ("filter2_min_points", C.c_int32), ("filter2_feature_distance", C.c_float), ("filter2_min_score", C.c_float)]


class DepthFilterParams(C.Structure):
    """mc_depth_filter_params: FILTER_PROJECTION_DEPTH's own parameters and the depth camera, for one filter step of the moped3d chain."""
    _fields_ = [("plausible_sq_distance", C.c_float), ("depth_fraction", C.c_float), ("min_keypoint_fraction", C.c_float),
                ("depth_K", C.c_float * 4), ("depth_pose", C.c_float * 7)]

    @classmethod
    def of(cls, plausible_sq_distance, depth_fraction, min_keypoint_fraction, depth_K, depth_pose):
        return cls(float(plausible_sq_distance), float(depth_fraction), float(min_keypoint_fraction), (C.c_float * 4)(*_f32(depth_K).reshape(4)),
                   (C.c_float * 7)(*_f32(depth_pose).reshape(7)))


# every symbol include/moped_cuda.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "mc_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "mc_destroy": (None, [C.c_void_p]),
    "mc_last_error": (C.c_char_p, [C.c_void_p]),
    "mc_version": (C.c_char_p, []),
    "mc_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mc_synchronize": (C.c_int, [C.c_void_p]),
    "mc_db_upload": (C.c_int, [C.c_void_p, _f32p, _f32p, _i32p, C.c_int64, C.c_int, C.c_int, C.c_int64]),
    "mc_db_rows": (C.c_int64, [C.c_void_p]),
    "mc_db_set_global_tables": (C.c_int, [C.c_void_p, _f32p, _i32p, C.c_int64, C.c_int]),
    "mc_set_cameras": (C.c_int, [C.c_void_p, _f32p, _f32p, C.c_int]),
    "mc_match": (C.c_int, [C.c_void_p, _f32p, C.c_int, C.c_float, C.c_int, _i32p, _f32p, _u8p, C.c_void_p]),
    "mc_match_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_match_merge_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_cluster_meanshift": (C.c_int, [C.c_void_p, _i32p, _i32p, _f32p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int,
                                       C.POINTER(C.c_int32), _i32p, _i32p, _i32p]),
    "mc_pose_hypotheses": (C.c_int, [C.c_void_p, _i32p, C.c_int, _f32p, _f32p, _i32p, _i32p, _i32p, _f32p, C.c_int, C.POINTER(PoseParams),
                                     _i32p, _f32p, _f32p, _f32p, C.c_void_p]),
    "mc_pose_hypotheses_dev": (C.c_int, [C.c_void_p] + [C.c_void_p] * 7 + [C.c_int, C.POINTER(PoseParams)] + [C.c_void_p] * 4),
    "mc_pose_ransac": (C.c_int, [C.c_void_p, _i32p, C.c_int, _f32p, _f32p, _i32p, C.POINTER(PoseParams), _u8p, _f32p, _i32p]),
    "mc_pose_depth_hypotheses": (C.c_int, [C.c_void_p, C.c_int, _i32p, C.c_int, _f32p, _f32p, _f32p, _f32p, _i32p, _i32p, _i32p, _f32p, C.c_int,
                                           C.POINTER(PoseParams), C.c_float, _i32p, _f32p, _f32p, _f32p, C.c_void_p]),
    "mc_pose_depth_hypotheses_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 8 + [C.c_int, C.POINTER(PoseParams), C.c_float]
                                     + [C.c_void_p] * 4),
    "mc_pose_depth_ransac": (C.c_int, [C.c_void_p, C.c_int, _i32p, C.c_int, _f32p, _f32p, _f32p, _f32p, _i32p, C.c_void_p, C.POINTER(PoseParams),
                                       C.c_float, _u8p, _f32p, _i32p]),
    "mc_filter_projection": (C.c_int, [C.c_void_p, _i32p, _i32p, _f32p, _f32p, C.c_int, _i32p, _f32p, C.c_int, C.c_int, C.c_float, C.c_float,
                                       _u8p, _f32p, C.POINTER(C.c_int32), _i32p, _i32p]),
    "mc_filter_projection_depth": (C.c_int, [C.c_void_p, _i32p, _i32p, _f32p, _f32p, C.c_int, _i32p, _f32p, C.c_int, C.c_int, C.c_float, C.c_float,
                                             C.c_float, C.c_float, C.c_float, _i32p, _f32p, _f32p, _f32p, C.c_int, C.c_int, _f32p, _f32p,
                                             _u8p, _f32p, C.POINTER(C.c_int32), _i32p, _i32p]),
    "mc_model_db_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "mc_model_db_destroy": (None, [C.c_void_p]),
    "mc_model_db_last_error": (C.c_char_p, [C.c_void_p]),
    "mc_model_db_add_xml_file": (C.c_int, [C.c_void_p, C.c_char_p]),
    "mc_model_db_add_xml_files": (C.c_int, [C.c_void_p, C.POINTER(C.c_char_p), C.c_int, C.c_int]),
    "mc_model_db_add_xml_buffer": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "mc_model_db_remove": (C.c_int, [C.c_void_p, C.c_char_p]),
    "mc_model_db_n_models": (C.c_int, [C.c_void_p]),
    "mc_model_db_model_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "mc_model_db_model_bbox": (C.c_int, [C.c_void_p, C.c_int, _f32p]),
    "mc_model_db_pack": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "mc_model_db_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]),
    "mc_model_db_save": (C.c_int, [C.c_void_p, C.c_char_p]),
    "mc_model_db_load": (C.c_int, [C.c_void_p, C.c_char_p]),
    "mc_cluster_linkage": (C.c_int, [C.c_void_p, _f32p, _f32p, _f32p, C.c_int, _f32p, _f32p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int,
                                     C.c_float, C.c_float, C.POINTER(C.c_int32), _i32p, _i32p, C.c_void_p]),
    "mc_linkage_agglomerate": (C.c_int, [C.c_void_p, _f32p, C.c_int, C.c_float, C.c_int, C.c_int, C.POINTER(C.c_int32), _i32p, _i32p]),
    "mc_depth_pipeline_default_params": (None, [C.POINTER(DepthPipelineParams)]),
    "mc_process_depth_frames": (C.c_int, [C.c_void_p, _i32p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _f32p, _f32p,
                                          C.c_int, C.c_int, C.POINTER(DepthPipelineParams), C.c_int, _i32p, _i32p, _f32p, _f32p, _i32p, C.c_void_p]),
    "mc_process_depth_frames_dev": (C.c_int, [C.c_void_p, _i32p, C.c_int, C.c_int] + [C.c_void_p] * 7 + [C.c_int, C.c_int, C.POINTER(DepthPipelineParams),
                                              C.c_int, _i32p, _i32p, _f32p, _f32p, _i32p, C.c_void_p]),
    "mc_sift_extract": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _i32p, _f32p, C.c_void_p, _f32p]),
    "mc_sift_extract_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_process_images": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(PipelineParams), C.c_int, _i32p, _i32p,
                                    _f32p, _f32p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_process_rig_images": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(PipelineParams), C.c_int,
                                        _i32p, _i32p, _f32p, _f32p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_process_rig_cameras": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(PipelineParams), C.c_int, _i32p, _i32p,
                                         _f32p, _f32p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_process_rig_cameras_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(PipelineParams), C.c_int, _i32p,
                                             _i32p, _f32p, _f32p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_extract_rig_cameras": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 3 + [_i32p, C.c_void_p,
                                                                                                                    C.c_void_p]),
    "mc_extract_rig_cameras_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 3 + [_i32p, C.c_void_p,
                                                                                                                        C.c_void_p]),
    "mc_sift_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double)]),
    "mc_sift_read_plane": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "mc_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "mc_pipeline_default_params": (None, [C.POINTER(PipelineParams)]),
    "mc_process_frame": (C.c_int, [C.c_void_p, _f32p, _f32p, _i32p, C.c_int, C.POINTER(PipelineParams), C.c_int, C.POINTER(C.c_int32),
                                   _i32p, _f32p, _f32p, C.c_void_p]),
    "mc_process_frame_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(PipelineParams), C.c_int,
                                       C.POINTER(C.c_int32), _i32p, _f32p, _f32p, C.c_void_p]),
    "mc_process_matched_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(PipelineParams), C.c_int,
                                         C.POINTER(C.c_int32), _i32p, _f32p, _f32p, C.c_void_p]),
    "mc_process_frames": (C.c_int, [C.c_void_p, _f32p, _f32p, _i32p, _i32p, C.c_int, C.POINTER(PipelineParams), C.c_int,
                                    _i32p, _i32p, _f32p, _f32p, C.c_void_p, C.c_void_p]),
    "mc_process_frames_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _i32p, C.c_int, C.POINTER(PipelineParams), C.c_int,
                                        _i32p, _i32p, _f32p, _f32p, C.c_void_p, C.c_void_p]),
    "mc_process_frames_matched_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _i32p, C.c_int, C.c_int, C.c_int,
                                                C.POINTER(PipelineParams), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_frame_shard_slot_bytes": (C.c_size_t, [C.c_int, C.POINTER(PipelineParams)]),
    "mc_process_frame_sharded_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(PipelineParams),
                                               C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_set_tuning": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "mc_kernel_launches": (C.c_int64, [C.c_void_p]),
    "mc_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "mc_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "mc_match_last_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mc_match_tier_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mc_sm_partition": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mc_match_merge_packed_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_join_lanes": (C.c_int, [C.c_void_p]),
    "mc_adaptive_model_init": (None, [C.c_void_p, _f32p, _f32p, _f32p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]),
    "mc_match_adaptive": (C.c_int, [C.c_void_p, _f32p, _f32p, C.c_int, _f32p, _f32p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_float,
                                    C.c_float, _i32p, _f32p, _u8p]),
    "mc_match_adaptive_frames": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _i32p, C.c_int, _f32p, _f32p, C.c_int, C.c_int, C.c_void_p,
                                           C.c_int, C.c_float, C.c_float, C.c_float, _i32p] + [C.c_void_p] * 8),
    "mc_match_adaptive_frames_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _i32p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                               C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float, _i32p] + [C.c_void_p] * 8),
    "mc_match_adaptive_frames_merged_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, _i32p, C.c_int, C.c_int, C.c_int,
                                                      C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float,
                                                      _i32p] + [C.c_void_p] * 8),
    "mc_process_depth_queries": (C.c_int, [C.c_void_p] * 6 + [_i32p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_float,
                                           C.c_float, C.c_float, C.POINTER(DepthPipelineParams), C.c_int, _i32p, _i32p, _f32p, _f32p, _i32p, C.c_void_p]),
    "mc_process_depth_queries_dev": (C.c_int, [C.c_void_p] * 6 + [_i32p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                               C.c_float, C.c_float, C.c_float, C.POINTER(DepthPipelineParams), C.c_int, _i32p, _i32p, _f32p, _f32p,
                                               _i32p, C.c_void_p]),
    "mc_process_depth_queries_merged_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [_i32p, C.c_int, C.c_int, C.c_int,
                                                      C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float,
                                                      C.POINTER(DepthPipelineParams), C.c_int, _i32p, _i32p, _f32p, _f32p, _i32p, C.c_void_p]),
    "mc_set_depth_filter": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(DepthFilterParams), C.c_void_p, C.c_void_p, C.c_int]),
    "mc_set_undistortion": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "mc_undistort": (C.c_int, [C.c_void_p, C.c_int, _u8p, C.c_int, C.c_int, C.c_int, _u8p]),
    "mc_undistort_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

MC_ERR_ARG = -2
MC_ERR_CAPACITY = -4

# mc_adaptive_model: one moped3d ratio curve per database model
ADAPTIVE_MODEL = np.dtype([("depth_peak", np.float32), ("depth_fade", np.float32), ("ratio_low", np.float32), ("ratio_high", np.float32)])
# MATCH_ADAPTIVE_FLANN_CPU's constructor values in moped3d's pipeline (MinRatioMin .. MaxRatioMax, DimensionPeak, DimensionFade)
ADAPTIVE_DEFAULTS = (0.6, 0.75, 0.65, 0.8, 150.0, 50.0)
# MaximumDepth, DefaultDepth, CauchyScale as the stage sets them
ADAPTIVE_DEPTHS = (4.0, 1.0, 0.1)


def adaptive_model_init(bbox_min, bbox_max, K, n_features, params=ADAPTIVE_DEFAULTS):
    """mc_adaptive_model_init per model: bbox_min / bbox_max [n_models, 3], K = (fx, fy, cx, cy), n_features [n_models] (database rows
    of each model), params = (MinRatioMin, MinRatioMax, MaxRatioMin, MaxRatioMax, DimensionPeak, DimensionFade).
    Returns a structured array of ADAPTIVE_MODEL records (host computation; no device needed)."""
    lo, hi = _f32(bbox_min).reshape(-1, 3), _f32(bbox_max).reshape(-1, 3)
    nf = np.asarray(n_features, np.int64).reshape(-1)
    Kf = _f32(K).reshape(4)
    lib = load()
    out = np.zeros(len(lo), ADAPTIVE_MODEL)
    for m in range(len(lo)):
        lib.mc_adaptive_model_init(out[m:m + 1].ctypes.data, np.ascontiguousarray(lo[m]), np.ascontiguousarray(hi[m]), Kf, int(nf[m]),
                                   *[float(p) for p in params])
    return out

_lib = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Load (building first if needed) libmoped_cuda.so and type every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path):
        _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class MopedCudaError(RuntimeError):
    pass


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


class Context:
    """One GPU context: device-resident model database + cameras + scratch."""

    def __init__(self, device: int = 0):
        self.L = load()
        h = C.c_void_p()
        st = self.L.mc_create(C.byref(h), device)
        if st != 0:
            raise MopedCudaError(f"mc_create failed ({st}): {self.L.mc_last_error(None).decode()}")
        self.h = h
        self.D = 128
        self.n_models = 0

    def _check(self, st, what):
        if st != 0:
            raise MopedCudaError(f"{what} failed ({st}): {self.L.mc_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.L.mc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, stream_handle):
        self._check(self.L.mc_set_stream(self.h, C.c_void_p(stream_handle) if stream_handle else None), "mc_set_stream")

    def synchronize(self):
        self._check(self.L.mc_synchronize(self.h), "mc_synchronize")

    @property
    def launches(self) -> int:
        return int(self.L.mc_kernel_launches(self.h))

    def set_profiling(self, on: bool):
        self._check(self.L.mc_set_profiling(self.h, 1 if on else 0), "mc_set_profiling")

    def coarse_kernel_ms(self) -> float:
        v = C.c_float(0)
        self._check(self.L.mc_profile_read(self.h, C.byref(v)), "mc_profile_read")
        return float(v.value)

    def match_last_stats(self):
        """{certified, fallback, candidates per query, DB splits} of the last matching pass on this context."""
        st = np.zeros(4, np.int32)
        self._check(self.L.mc_match_last_stats(self.h, st.ctypes.data), "mc_match_last_stats")
        return st

    def match_tier_stats(self):
        """{queries, certified by the 8-bit pass, certified by the fp16 pass, exhaustive exact scan} of the last matching pass."""
        st = np.zeros(4, np.int32)
        self._check(self.L.mc_match_tier_stats(self.h, st.ctypes.data), "mc_match_tier_stats")
        return st

    def sm_partition(self):
        """(SMs of the coarse matching kernel, SMs of the stage partition or 0)"""
        st = np.zeros(2, np.int32)
        self._check(self.L.mc_sm_partition(self.h, st.ctypes.data), "mc_sm_partition")
        return int(st[0]), int(st[1])

    # ---- database / cameras
    def db_upload(self, desc, xyz, model_of_row, n_models, row_base=0):
        desc, xyz, model_of_row = _f32(desc), _f32(xyz), _i32(model_of_row)
        self.D = desc.shape[1]
        self.n_models = int(n_models)
        self._check(self.L.mc_db_upload(self.h, desc, xyz, model_of_row, desc.shape[0], desc.shape[1], int(n_models), int(row_base)), "mc_db_upload")

    def db_set_global_tables(self, xyz_all, model_of_row_all, n_models_all):
        xyz_all, model_of_row_all = _f32(xyz_all), _i32(model_of_row_all)
        self.n_models = int(n_models_all)
        self._check(self.L.mc_db_set_global_tables(self.h, xyz_all, model_of_row_all, len(model_of_row_all), int(n_models_all)), "mc_db_set_global_tables")

    def set_cameras(self, K, cam_pose):
        K, cam_pose = _f32(K).reshape(-1, 4), _f32(cam_pose).reshape(-1, 7)
        self.n_images = len(K)
        self._check(self.L.mc_set_cameras(self.h, K, cam_pose, len(K)), "mc_set_cameras")

    # ---- MATCH
    def match(self, q_desc, ratio=0.8, mode=MATCH_TENSOR):
        q = _f32(q_desc)
        Q = len(q)
        nn_row = np.full((Q, 2), -1, np.int32)
        nn_dist = np.zeros((Q, 2), np.float32)
        acc = np.zeros(Q, np.uint8)
        stats = np.zeros(4, np.int32)
        self._check(self.L.mc_match(self.h, q, Q, ratio, mode, nn_row, nn_dist, acc, stats.ctypes.data), "mc_match")
        return nn_row, nn_dist, acc.astype(bool), stats

    def match_dev(self, q_ptr, Q, ratio, mode, nn_row_ptr, nn_dist_ptr, acc_ptr):
        self._check(self.L.mc_match_dev(self.h, q_ptr, Q, ratio, mode, nn_row_ptr, nn_dist_ptr, acc_ptr), "mc_match_dev")

    def match_merge_dev(self, rows_all_ptr, dist_all_ptr, n_shards, Q, ratio, nn_row_ptr, nn_dist_ptr, acc_ptr):
        self._check(self.L.mc_match_merge_dev(self.h, rows_all_ptr, dist_all_ptr, n_shards, Q, ratio, nn_row_ptr, nn_dist_ptr, acc_ptr),
                    "mc_match_merge_dev")

    def match_merge_packed_dev(self, packed_all_ptr, n_shards, Q, ratio, nn_row_ptr, nn_dist_ptr, acc_ptr):
        self._check(self.L.mc_match_merge_packed_dev(self.h, packed_all_ptr, n_shards, Q, ratio, nn_row_ptr, nn_dist_ptr, acc_ptr),
                    "mc_match_merge_packed_dev")

    def join_lanes(self):
        self._check(self.L.mc_join_lanes(self.h), "mc_join_lanes")

    # ---- MATCH, moped3d's depth-adaptive variant
    @staticmethod
    def _curves(models):
        return np.ascontiguousarray(models, dtype=ADAPTIVE_MODEL)

    def match_adaptive(self, q_desc, q_xy, depth, fill_distance, models, depths=ADAPTIVE_DEPTHS):
        """One frame: q_desc [Q, D] normalised, q_xy [Q, 2], depth / fill_distance [H, W], models = ADAPTIVE_MODEL records (one per database
        model), depths = (maximum_depth, default_depth, cauchy_scale). Returns (nn_row [Q, 2], nn_dist [Q, 2], accepted [Q] bool)."""
        q, xy = _f32(q_desc).reshape(-1, self.D), _f32(q_xy).reshape(-1, 2)
        d, fd = _f32(depth), _f32(fill_distance)
        cv = self._curves(models)
        Q = len(q)
        nn_row = np.full((Q, 2), -1, np.int32)
        nn_dist = np.zeros((Q, 2), np.float32)
        acc = np.zeros(Q, np.uint8)
        if Q == 0:
            q, xy = np.zeros((1, self.D), np.float32), np.zeros((1, 2), np.float32)
        self._check(self.L.mc_match_adaptive(self.h, q, xy, Q, d.reshape(-1), fd.reshape(-1), d.shape[1], d.shape[0], cv.ctypes.data, len(cv),
                                             *[float(v) for v in depths], nn_row.reshape(-1) if Q else np.zeros(2, np.int32),
                                             nn_dist.reshape(-1) if Q else np.zeros(2, np.float32), acc if Q else np.zeros(1, np.uint8)),
                    "mc_match_adaptive")
        return nn_row, nn_dist, acc.astype(bool)

    def _adaptive_frames_result(self, st, what, partial, out, partial_status=(MC_ERR_CAPACITY,)):
        if st != 0 and not (partial and st in partial_status):
            self._check(st, what)
        out["status"] = int(st)
        if st != 0:
            out["error"] = self.L.mc_last_error(self.h).decode()
        return out

    def match_adaptive_frames(self, q_desc, q_xy, q_image, frame_offsets, depth, fill_distance, models, depths=ADAPTIVE_DEPTHS, partial=False):
        """A batch of frames in one matching pass (mc_match_adaptive_frames). q_desc [Q, D], q_xy [Q, 2], q_image [Q] or None,
        frame_offsets [n_frames + 1], depth / fill_distance [n_frames, H, W]. Returns dict(match_offsets [n_frames, n_models + 1] global,
        match_feature / match_image / match_xy / match_xyz with capacity Q (frame f's matches from frame_offsets[f] on), nn_row, nn_dist,
        accepted, frame_info [n_frames, 3], status). partial=True returns a capacity error (a frame with more than 8192 accepted matches)
        as status -4 with the results instead of raising."""
        fo = _i32(frame_offsets).reshape(-1)
        nf = len(fo) - 1
        cv = self._curves(models)
        d, fd = _f32(depth), _f32(fill_distance)
        H, W = d.shape[-2], d.shape[-1]
        q, xy = _f32(q_desc).reshape(-1, self.D), _f32(q_xy).reshape(-1, 2)
        img = _i32(q_image).reshape(-1) if q_image is not None else None
        Q = len(q)
        n = max(Q, 1)
        out = dict(match_offsets=np.zeros((nf, len(cv) + 1), np.int32), match_feature=np.zeros(n, np.int32), match_image=np.zeros(n, np.int32),
                   match_xy=np.zeros((n, 2), np.float32), match_xyz=np.zeros((n, 3), np.float32), nn_row=np.full((n, 2), -1, np.int32),
                   nn_dist=np.zeros((n, 2), np.float32), accepted=np.zeros(n, np.uint8), frame_info=np.zeros((nf, 3), np.int32))
        p = lambda a: a.ctypes.data if a is not None and a.size else None
        st = self.L.mc_match_adaptive_frames(self.h, p(q), p(xy), p(img), fo, nf, d.reshape(-1), fd.reshape(-1), W, H, cv.ctypes.data,
                                             len(cv), *[float(v) for v in depths], out["match_offsets"].reshape(-1),
                                             *[out[k].ctypes.data for k in ("match_feature", "match_image", "match_xy", "match_xyz", "nn_row", "nn_dist",
                                                                            "accepted", "frame_info")])
        out["accepted"] = out["accepted"].astype(bool)
        for k in ("match_feature", "match_image", "match_xy", "match_xyz", "nn_row", "nn_dist", "accepted"):
            out[k] = out[k][:Q]
        return self._adaptive_frames_result(st, "mc_match_adaptive_frames", partial, out)

    def match_adaptive_frames_dev(self, q_ptr, xy_ptr, img_ptr, frame_offsets, depth_ptr, fill_ptr, width, height, models, match_feature_ptr,
                                  match_image_ptr, match_xy_ptr, match_xyz_ptr, nn_row_ptr=None, nn_dist_ptr=None, acc_ptr=None, depths=ADAPTIVE_DEPTHS,
                                  partial=False):
        """mc_match_adaptive_frames_dev: the same with device pointers for the queries, the planes and the per-match / per-feature outputs
        (img_ptr, nn_row_ptr, nn_dist_ptr, acc_ptr may be None). Returns dict(match_offsets, frame_info, status) (host arrays)."""
        fo = _i32(frame_offsets).reshape(-1)
        nf = len(fo) - 1
        cv = self._curves(models)
        out = dict(match_offsets=np.zeros((nf, len(cv) + 1), np.int32), frame_info=np.zeros((nf, 3), np.int32))
        st = self.L.mc_match_adaptive_frames_dev(self.h, q_ptr, xy_ptr, img_ptr, fo, nf, depth_ptr, fill_ptr, int(width), int(height), cv.ctypes.data,
                                                 len(cv), *[float(v) for v in depths], out["match_offsets"].reshape(-1), match_feature_ptr,
                                                 match_image_ptr, match_xy_ptr, match_xyz_ptr, nn_row_ptr, nn_dist_ptr, acc_ptr,
                                                 out["frame_info"].ctypes.data)
        return self._adaptive_frames_result(st, "mc_match_adaptive_frames_dev", partial, out)

    def match_adaptive_frames_merged_dev(self, packed_all_ptr, n_shards, xy_ptr, img_ptr, frame_offsets, frame_begin, frame_end, depth_ptr, fill_ptr,
                                         width, height, models, match_feature_ptr, match_image_ptr, match_xy_ptr, match_xyz_ptr, nn_row_ptr=None,
                                         nn_dist_ptr=None, acc_ptr=None, depths=ADAPTIVE_DEPTHS, partial=False):
        """mc_match_adaptive_frames_merged_dev: frames [frame_begin, frame_end) of the batch from the n_shards gathered packed blocks at
        packed_all_ptr (device, n_shards x 16 Q bytes). depth_ptr / fill_ptr hold the range's planes only; the per-feature and per-match
        outputs use global feature indices (nn_row_ptr, nn_dist_ptr, acc_ptr may be None). Returns dict(match_offsets
        [frame_end - frame_begin, n_models + 1], frame_info [frame_end - frame_begin, 3], status). partial=True returns a capacity error
        (frame_info status 1) or a row outside the tables (status 2, MC_ERR_ARG) as status with the results instead of raising."""
        fo = _i32(frame_offsets).reshape(-1)
        nf, nr = len(fo) - 1, int(frame_end) - int(frame_begin)
        cv = self._curves(models)
        out = dict(match_offsets=np.zeros((max(nr, 1), len(cv) + 1), np.int32), frame_info=np.zeros((max(nr, 1), 3), np.int32))
        st = self.L.mc_match_adaptive_frames_merged_dev(self.h, packed_all_ptr, int(n_shards), xy_ptr, img_ptr, fo, nf, int(frame_begin), int(frame_end),
                                                        depth_ptr, fill_ptr, int(width), int(height), cv.ctypes.data, len(cv),
                                                        *[float(v) for v in depths], out["match_offsets"].reshape(-1), match_feature_ptr, match_image_ptr,
                                                        match_xy_ptr, match_xyz_ptr, nn_row_ptr, nn_dist_ptr, acc_ptr, out["frame_info"].ctypes.data)
        out["match_offsets"], out["frame_info"] = out["match_offsets"][:max(nr, 0)], out["frame_info"][:max(nr, 0)]
        return self._adaptive_frames_result(st, "mc_match_adaptive_frames_merged_dev", partial, out, (MC_ERR_CAPACITY, MC_ERR_ARG))

    # ---- CLUSTER
    def cluster(self, matches, n_images=1, radius=200.0, merge=20.0, minpts=7, maxiter=100):
        off = _i32(matches["offsets"])
        M = int(off[-1])
        n = C.c_int32(0)
        cm = np.zeros(M + 2, np.int32)
        co = np.zeros(M + 2, np.int32)
        mem = np.zeros(M + 2, np.int32)
        img = _i32(matches["image"]) if M else np.zeros(1, np.int32)
        xy = _f32(matches["xy"]) if M else np.zeros((1, 2), np.float32)
        self._check(self.L.mc_cluster_meanshift(self.h, off, img, xy, len(off) - 1, n_images, radius, merge, minpts, maxiter,
                                                C.byref(n), cm, co, mem), "mc_cluster_meanshift")
        c = n.value
        return dict(model=cm[:c].copy(), offsets=co[:c + 1].copy(), members=mem[:co[c]].copy())

    # ---- POSE
    def pose_hypotheses(self, cluster_offsets, pt_xy, pt_xyz, pt_image, hyp_cluster, sample_pos, init_quat, params, want_mask=True):
        co = _i32(cluster_offsets)
        hc, sp, iq = _i32(hyp_cluster), _i32(sample_pos), _f32(init_quat)
        n_hyp = len(hc)
        pp = params if isinstance(params, PoseParams) else PoseParams.of(params)
        n_in = np.zeros(n_hyp, np.int32)
        pose_lm = np.zeros((n_hyp, 7), np.float32)
        pose_refit = np.zeros((n_hyp, 7), np.float32)
        err = np.zeros((n_hyp, 2), np.float32)
        sizes = (co[1:] - co[:-1])[hc]
        mask = np.zeros(int(sizes.sum()) + 1, np.uint8) if want_mask else None
        self._check(self.L.mc_pose_hypotheses(self.h, co, len(co) - 1, _f32(pt_xy), _f32(pt_xyz), _i32(pt_image), hc, sp, iq, n_hyp, C.byref(pp),
                                              n_in, pose_lm, pose_refit, err, mask.ctypes.data if want_mask else None), "mc_pose_hypotheses")
        masks = None
        if want_mask:
            o = np.concatenate([[0], np.cumsum(sizes)])
            masks = [mask[o[h]:o[h + 1]].astype(bool) for h in range(n_hyp)]
        return n_in, pose_lm, pose_refit, err, masks

    def pose_hypotheses_dev(self, co_ptr, xy_ptr, xyz_ptr, img_ptr, hc_ptr, sp_ptr, iq_ptr, n_hyp, params, n_in_ptr, pose_lm_ptr, pose_refit_ptr, err_ptr):
        """Device-pointer variant (asynchronous on the context's stream)."""
        pp = params if isinstance(params, PoseParams) else PoseParams.of(params)
        self._check(self.L.mc_pose_hypotheses_dev(self.h, co_ptr, xy_ptr, xyz_ptr, img_ptr, hc_ptr, sp_ptr, iq_ptr, n_hyp, C.byref(pp),
                                                  n_in_ptr, pose_lm_ptr, pose_refit_ptr, err_ptr), "mc_pose_hypotheses_dev")

    def pose_ransac(self, cluster_offsets, pt_xy, pt_xyz, pt_image, params, seed=1):
        co = _i32(cluster_offsets)
        pp = params if isinstance(params, PoseParams) else PoseParams.of(params, seed)
        n_tasks = (len(co) - 1) * pp.max_objects_per_cluster
        found = np.zeros(n_tasks, np.uint8)
        pose = np.zeros((n_tasks, 7), np.float32)
        n_tests = np.zeros(n_tasks, np.int32)
        self._check(self.L.mc_pose_ransac(self.h, co, len(co) - 1, _f32(pt_xy), _f32(pt_xyz), _i32(pt_image), C.byref(pp), found, pose, n_tests),
                    "mc_pose_ransac")
        return found.astype(bool), pose, n_tests

    # ---- POSE, moped3d depth-aware variants (0 = back-projection, 1 = reprojection + depth)
    def pose_depth_hypotheses(self, variant, cluster_offsets, pt_xy, pt_xyz, pt_world, pt_cauchy, pt_image, hyp_cluster, sample_pos, init_quat,
                              params, alpha, want_mask=True):
        co = _i32(cluster_offsets)
        hc, sp, iq = _i32(hyp_cluster), _i32(sample_pos), _f32(init_quat)
        n_hyp = len(hc)
        pp = params if isinstance(params, PoseParams) else PoseParams.of(params)
        n_in = np.zeros(n_hyp, np.int32)
        pose_lm = np.zeros((n_hyp, 7), np.float32)
        pose_refit = np.zeros((n_hyp, 7), np.float32)
        err = np.zeros((n_hyp, 2), np.float32)
        sizes = (co[1:] - co[:-1])[hc]
        mask = np.zeros(int(sizes.sum()) + 1, np.uint8) if want_mask else None
        self._check(self.L.mc_pose_depth_hypotheses(self.h, int(variant), co, len(co) - 1, _f32(pt_xy), _f32(pt_xyz), _f32(pt_world), _f32(pt_cauchy),
                                                    _i32(pt_image), hc, sp, iq, n_hyp, C.byref(pp), float(alpha), n_in, pose_lm, pose_refit, err,
                                                    mask.ctypes.data if want_mask else None), "mc_pose_depth_hypotheses")
        masks = None
        if want_mask:
            o = np.concatenate([[0], np.cumsum(sizes)])
            masks = [mask[o[h]:o[h + 1]].astype(bool) for h in range(n_hyp)]
        return n_in, pose_lm, pose_refit, err, masks

    def pose_depth_hypotheses_dev(self, variant, co_ptr, max_cluster_size, xy_ptr, xyz_ptr, world_ptr, cauchy_ptr, img_ptr, hc_ptr, sp_ptr, iq_ptr,
                                  n_hyp, params, alpha, n_in_ptr, pose_lm_ptr, pose_refit_ptr, err_ptr):
        """Device-pointer variant (asynchronous on the context's stream); world_ptr / cauchy_ptr may be None for variant 2."""
        pp = params if isinstance(params, PoseParams) else PoseParams.of(params)
        self._check(self.L.mc_pose_depth_hypotheses_dev(self.h, int(variant), co_ptr, int(max_cluster_size), xy_ptr, xyz_ptr, world_ptr, cauchy_ptr,
                                                        img_ptr, hc_ptr, sp_ptr, iq_ptr, n_hyp, C.byref(pp), float(alpha), n_in_ptr, pose_lm_ptr,
                                                        pose_refit_ptr, err_ptr), "mc_pose_depth_hypotheses_dev")

    def pose_depth_ransac(self, variant, cluster_offsets, pt_xy, pt_xyz, pt_world, pt_cauchy, pt_image, params, alpha, seed=1, pt_tie=None):
        co = _i32(cluster_offsets)
        pp = params if isinstance(params, PoseParams) else PoseParams.of(params, seed)
        n_tasks = (len(co) - 1) * pp.max_objects_per_cluster
        found = np.zeros(n_tasks, np.uint8)
        pose = np.zeros((n_tasks, 7), np.float32)
        n_tests = np.zeros(n_tasks, np.int32)
        tie = _i32(pt_tie) if pt_tie is not None else None
        self._check(self.L.mc_pose_depth_ransac(self.h, int(variant), co, len(co) - 1, _f32(pt_xy), _f32(pt_xyz), _f32(pt_world), _f32(pt_cauchy),
                                                _i32(pt_image), tie.ctypes.data if tie is not None else None, C.byref(pp), float(alpha), found, pose,
                                                n_tests), "mc_pose_depth_ransac")
        return found.astype(bool), pose, n_tests

    def filter_depth(self, matches, obj_model, obj_pose, params, test_offsets, test_xyz, depth_K, depth_pose, depth, fill_distance):
        """moped3d's FILTER_PROJECTION_DEPTH. params = (MinPoints, FeatureDistance, PlausibleSqDistance, MinScore, DepthFraction,
        MinKeypointFraction); depth / fill_distance: H x W float planes."""
        off = _i32(matches["offsets"])
        M = int(off[-1])
        om, op = _i32(obj_model), _f32(obj_pose).reshape(-1, 7)
        n = len(om)
        keep = np.zeros(n + 1, np.uint8)
        score = np.zeros(n + 1, np.float32)
        ns = C.c_int32(0)
        co = np.zeros(n + 2, np.int32)
        mem = np.zeros(M + 2, np.int32)
        img = _i32(matches["image"]) if M else np.zeros(1, np.int32)
        xy = _f32(matches["xy"]) if M else np.zeros((1, 2), np.float32)
        xyz = _f32(matches["xyz"]) if M else np.zeros((1, 3), np.float32)
        if n == 0:
            om, op = np.zeros(1, np.int32), np.zeros((1, 7), np.float32)
        to = _i32(test_offsets)
        tx = _f32(test_xyz).reshape(-1, 3) if int(to[-1]) else np.zeros((1, 3), np.float32)
        d, f = _f32(depth), _f32(fill_distance)
        self._check(self.L.mc_filter_projection_depth(self.h, off, img, xy, xyz, len(off) - 1, om, op, n, int(params[0]), float(params[1]),
                                                      float(params[2]), float(params[3]), float(params[4]), float(params[5]), to, tx, _f32(depth_K),
                                                      _f32(depth_pose), d.shape[1], d.shape[0], d, f, keep, score, C.byref(ns), co, mem),
                    "mc_filter_projection_depth")
        s = ns.value
        return dict(keep=keep[:n].astype(bool), score=score[:n].copy(), offsets=co[:s + 1].copy(), members=mem[:co[s]].copy())

    # ---- FILTER
    def filter(self, matches, obj_model, obj_pose, params=(5, 4096.0, 2.0)):
        off = _i32(matches["offsets"])
        M = int(off[-1])
        om, op = _i32(obj_model), _f32(obj_pose).reshape(-1, 7)
        n = len(om)
        keep = np.zeros(n + 1, np.uint8)
        score = np.zeros(n + 1, np.float32)
        ns = C.c_int32(0)
        co = np.zeros(n + 2, np.int32)
        mem = np.zeros(M + 2, np.int32)
        img = _i32(matches["image"]) if M else np.zeros(1, np.int32)
        xy = _f32(matches["xy"]) if M else np.zeros((1, 2), np.float32)
        xyz = _f32(matches["xyz"]) if M else np.zeros((1, 3), np.float32)
        if n == 0:
            om, op = np.zeros(1, np.int32), np.zeros((1, 7), np.float32)
        self._check(self.L.mc_filter_projection(self.h, off, img, xy, xyz, len(off) - 1, om, op, n, int(params[0]), float(params[1]), float(params[2]),
                                                keep, score, C.byref(ns), co, mem), "mc_filter_projection")
        s = ns.value
        return dict(keep=keep[:n].astype(bool), score=score[:n].copy(), offsets=co[:s + 1].copy(), members=mem[:co[s]].copy())

    # ---- whole frame
    def default_params(self) -> PipelineParams:
        p = PipelineParams()
        self.L.mc_pipeline_default_params(C.byref(p))
        return p

    def cluster_linkage(self, xy, xyz, world, depth, distance, cutoff=0.1, min_pts=7, use3d_filter=2, linkage_type=1, sigma2d=-1.0, sigma3d=-1.0,
                        want_similarity=False):
        """moped3d CLUSTER_LINKAGE on one model's matches -> (offsets, members[, K])."""
        xy, xyz, world, depth, distance = _f32(xy), _f32(xyz), _f32(world), _f32(depth), _f32(distance)
        n = len(xy)
        nc = C.c_int32(0)
        off = np.zeros(n + 2, np.int32)
        mem = np.zeros(n + 1, np.int32)
        K = np.zeros((n, n), np.float32) if want_similarity else None
        self._check(self.L.mc_cluster_linkage(self.h, xy.reshape(-1), xyz.reshape(-1), world.reshape(-1), n, depth.reshape(-1), distance.reshape(-1),
                                              depth.shape[1], depth.shape[0], cutoff, min_pts, use3d_filter, linkage_type, sigma2d, sigma3d,
                                              C.byref(nc), off, mem, K.ctypes.data if K is not None else None), "mc_cluster_linkage")
        out = (off[:nc.value + 1].copy(), mem[:off[nc.value]].copy())
        return out + (K,) if want_similarity else out

    def linkage_agglomerate(self, K, cutoff=0.1, min_pts=7, linkage_type=1):
        K = _f32(K)
        n = len(K)
        nc = C.c_int32(0)
        off = np.zeros(n + 2, np.int32)
        mem = np.zeros(n + 1, np.int32)
        self._check(self.L.mc_linkage_agglomerate(self.h, K.reshape(-1), n, cutoff, min_pts, linkage_type, C.byref(nc), off, mem), "mc_linkage_agglomerate")
        return off[:nc.value + 1].copy(), mem[:off[nc.value]].copy()

    def sift(self, gray, double_size=True, max_keypoints=8192):
        """FEAT step on a batch of equally sized grayscale images [B,H,W] (or one [H,W]) -> list of (xy, scale_ori, desc)."""
        g = np.ascontiguousarray(gray, dtype=np.uint8)
        single = g.ndim == 2
        if single:
            g = g[None]
        B, H, W = g.shape
        counts = np.zeros(B, np.int32)
        xy = np.zeros((B, max_keypoints, 2), np.float32)
        so = np.zeros((B, max_keypoints, 2), np.float32)
        desc = np.zeros((B, max_keypoints, 128), np.float32)
        self._check(self.L.mc_sift_extract(self.h, g.reshape(-1), B, H, W, 1 if double_size else 0, max_keypoints, counts, xy.reshape(-1),
                                           so.ctypes.data, desc.reshape(-1)), "mc_sift_extract")
        out = [(xy[f, :counts[f]].copy(), so[f, :counts[f]].copy(), desc[f, :counts[f]].copy()) for f in range(B)]
        return out[0] if single else out

    def process_images(self, gray, double_size=True, max_keypoints=4096, params=None, max_objects=64, want_times=False):
        """FEAT..FILTER2 for a batch of single-camera frames [B,H,W] uint8 -> list of dicts (model, pose, score, n_features)."""
        g = np.ascontiguousarray(gray, dtype=np.uint8)
        if g.ndim == 2:
            g = g[None]
        B, H, W = g.shape
        p = params or self.default_params()
        n = np.zeros(B, np.int32)
        om = np.zeros((B, max_objects), np.int32)
        op = np.zeros((B, max_objects, 7), np.float32)
        os_ = np.zeros((B, max_objects), np.float32)
        nf = np.zeros(B, np.int32)
        info = np.zeros((B, 4), np.int32)
        ms = np.zeros(3, np.float32)
        self._check(self.L.mc_process_images(self.h, g.reshape(-1), B, H, W, 1 if double_size else 0, max_keypoints, C.byref(p), max_objects, n,
                                             om.reshape(-1), op.reshape(-1), os_.reshape(-1), nf.ctypes.data, info.ctypes.data,
                                             ms.ctypes.data if want_times else None), "mc_process_images")
        out = [dict(model=om[f, :n[f]].copy(), pose=op[f, :n[f]].copy(), score=os_[f, :n[f]].copy(), n_features=int(nf[f]), info=info[f].copy())
               for f in range(B)]
        if want_times:
            out[0]["stage_ms"] = ms
        return out

    def process_rig_images(self, gray, double_size=True, max_keypoints=4096, params=None, max_objects=64, want_times=False):
        """FEAT..FILTER2 for a batch of camera-rig frames [B,C,H,W] uint8, image c of a frame from camera c -> list of dicts (model,
        pose, score, n_features = keypoints per camera, info)."""
        g = np.ascontiguousarray(gray, dtype=np.uint8)
        B, Cn, H, W = g.shape
        p = params or self.default_params()
        n = np.zeros(B, np.int32)
        om = np.zeros((B, max_objects), np.int32)
        op = np.zeros((B, max_objects, 7), np.float32)
        os_ = np.zeros((B, max_objects), np.float32)
        nf = np.zeros((B, Cn), np.int32)
        info = np.zeros((B, 4), np.int32)
        ms = np.zeros(3, np.float32)
        self._check(self.L.mc_process_rig_images(self.h, g.reshape(-1), B, Cn, H, W, 1 if double_size else 0, max_keypoints, C.byref(p),
                                                 max_objects, n, om.reshape(-1), op.reshape(-1), os_.reshape(-1), nf.ctypes.data, info.ctypes.data,
                                                 ms.ctypes.data if want_times else None), "mc_process_rig_images")
        out = [dict(model=om[f, :n[f]].copy(), pose=op[f, :n[f]].copy(), score=os_[f, :n[f]].copy(), n_features=nf[f].copy(), info=info[f].copy())
               for f in range(B)]
        if want_times:
            out[0]["stage_ms"] = ms
        return out

    def process_rig_cameras(self, images, double_size=True, max_keypoints=4096, params=None, max_objects=64, want_times=False):
        """mc_process_rig_cameras: FEAT..FILTER2 for camera-rig frames whose cameras may differ in size; images = one uint8 array
        (n_frames, H_c, W_c) per camera c -> the per-frame dicts of process_rig_images."""
        ims = [np.ascontiguousarray(g, dtype=np.uint8) for g in images]
        cams = (RigCamera * len(ims))(*[RigCamera(g.ctypes.data, g.shape[1] * g.shape[2], g.shape[1], g.shape[2]) for g in ims])
        return self._rig_cameras("mc_process_rig_cameras", cams, len(ims[0]), double_size, max_keypoints, params, max_objects, want_times)

    def process_rig_cameras_dev(self, ptrs, strides, sizes, n_frames, double_size=True, max_keypoints=4096, params=None, max_objects=64,
                                want_times=False):
        """mc_process_rig_cameras_dev: camera c's image of frame f is sizes[c] = (H, W) bytes at device address ptrs[c] + f * strides[c]
        -> the per-frame dicts of process_rig_images."""
        cams = (RigCamera * len(ptrs))(*[RigCamera(int(p), int(st), int(h), int(w)) for p, st, (h, w) in zip(ptrs, strides, sizes)])
        return self._rig_cameras("mc_process_rig_cameras_dev", cams, n_frames, double_size, max_keypoints, params, max_objects, want_times)

    def _rig_cameras(self, fn, cams, B, double_size, max_keypoints, params, max_objects, want_times):
        Cn = len(cams)
        p = params or self.default_params()
        n = np.zeros(B, np.int32)
        om = np.zeros((B, max_objects), np.int32)
        op = np.zeros((B, max_objects, 7), np.float32)
        os_ = np.zeros((B, max_objects), np.float32)
        nf = np.zeros((B, Cn), np.int32)
        info = np.zeros((B, 4), np.int32)
        ms = np.zeros(3, np.float32)
        self._check(getattr(self.L, fn)(self.h, C.cast(cams, C.c_void_p), Cn, B, 1 if double_size else 0, max_keypoints, C.byref(p), max_objects,
                                        n, om.reshape(-1), op.reshape(-1), os_.reshape(-1), nf.ctypes.data, info.ctypes.data,
                                        ms.ctypes.data if want_times else None), fn)
        out = [dict(model=om[f, :n[f]].copy(), pose=op[f, :n[f]].copy(), score=os_[f, :n[f]].copy(), n_features=nf[f].copy(), info=info[f].copy())
               for f in range(B)]
        if want_times:
            out[0]["stage_ms"] = ms
        return out

    def extract_rig_cameras(self, images, desc, xy, image, double_size=True, max_keypoints=4096, want_times=False, partial=False):
        """mc_extract_rig_cameras: FEAT of process_rig_cameras alone; images = one uint8 array (n_frames, H_c, W_c) per camera c. The query
        arrays go to the contiguous CUDA tensors desc (float32, rows of 128), xy (float32, rows of 2) and image (int32), each with room for
        n_frames x n_cameras x max_keypoints rows. Returns (frame_offsets [n_frames + 1], n_features [n_frames, n_cameras], feat_ms or
        None); partial=True appends the status and returns it for any failure of the call instead of raising."""
        ims = [np.ascontiguousarray(g, dtype=np.uint8) for g in images]
        cams = (RigCamera * len(ims))(*[RigCamera(g.ctypes.data, g.shape[1] * g.shape[2], g.shape[1], g.shape[2]) for g in ims])
        return self._extract_rig("mc_extract_rig_cameras", cams, len(ims[0]), desc, xy, image, double_size, max_keypoints, want_times, partial)

    def extract_rig_cameras_dev(self, ptrs, strides, sizes, n_frames, desc, xy, image, double_size=True, max_keypoints=4096,
                                want_times=False, partial=False):
        """mc_extract_rig_cameras_dev: the images as process_rig_cameras_dev takes them, the outputs as extract_rig_cameras."""
        cams = (RigCamera * len(ptrs))(*[RigCamera(int(p), int(st), int(h), int(w)) for p, st, (h, w) in zip(ptrs, strides, sizes)])
        return self._extract_rig("mc_extract_rig_cameras_dev", cams, n_frames, desc, xy, image, double_size, max_keypoints, want_times, partial)

    @staticmethod
    def _check_outputs(fn, rows, desc, xy, image):
        """the output tensors hold rows rows of their kind on the device; the kernels store desc rows as float4 (16-byte aligned)"""
        import torch
        for name, t, dtype, width in (("desc", desc, torch.float32, 128), ("xy", xy, torch.float32, 2), ("image", image, torch.int32, 1)):
            if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != dtype or not t.is_contiguous():
                raise ValueError(f"{fn}: {name} must be a contiguous CUDA tensor of {dtype}")
            if t.numel() < rows * width:
                raise ValueError(f"{fn}: {name} holds {t.numel() // width} rows, {rows} needed (n_frames x n_cameras x max_keypoints)")
        if desc.data_ptr() % 16 or xy.data_ptr() % 8:
            raise ValueError(f"{fn}: desc must be 16-byte and xy 8-byte aligned")

    def _extract_rig(self, fn, cams, B, desc, xy, image, double_size, max_keypoints, want_times, partial):
        self._check_outputs(fn, max(B, 0) * len(cams) * max(max_keypoints, 0), desc, xy, image)
        fo = np.zeros(max(B, 0) + 1, np.int32)
        nf = np.zeros((max(B, 1), len(cams)), np.int32)
        ms = np.zeros(1, np.float32)
        st = getattr(self.L, fn)(self.h, C.cast(cams, C.c_void_p), len(cams), B, 1 if double_size else 0, max_keypoints, desc.data_ptr(),
                                 xy.data_ptr(), image.data_ptr(), fo, nf.ctypes.data, ms.ctypes.data if want_times else None)
        if st != 0 and not partial:
            self._check(st, fn)
        out = (fo, nf[:B], float(ms[0]) if want_times else None)
        return out + (int(st),) if partial else out

    def set_undistortion(self, camera, K, kc, height, width):
        """mc_set_undistortion: UNDISTORTED_IMAGE for camera `camera` (K = (fx, fy, cx, cy), kc = (k1, k2, p1, p2[, k3])) on
        height x width images; kc=None clears the camera's table."""
        if kc is None:
            self._check(self.L.mc_set_undistortion(self.h, int(camera), None, None, 0, int(height), int(width)), "mc_set_undistortion")
            return
        Kf, kf = _f32(K).reshape(-1), _f32(kc).reshape(-1)
        self._check(self.L.mc_set_undistortion(self.h, int(camera), Kf.ctypes.data, kf.ctypes.data, len(kf), int(height), int(width)),
                    "mc_set_undistortion")

    def undistort(self, gray, camera=0):
        """mc_undistort: a batch [B,H,W] (or one [H,W]) of uint8 images of `camera` -> the undistorted images, same shape"""
        g = np.ascontiguousarray(gray, dtype=np.uint8)
        b = g.reshape((-1,) + g.shape[-2:])
        out = np.empty_like(b)
        self._check(self.L.mc_undistort(self.h, int(camera), b.reshape(-1), b.shape[0], b.shape[1], b.shape[2], out.reshape(-1)), "mc_undistort")
        return out.reshape(g.shape)

    def undistort_dev(self, gray_ptr, B, H, W, out_ptr, camera=0):
        self._check(self.L.mc_undistort_dev(self.h, int(camera), gray_ptr, B, H, W, out_ptr), "mc_undistort_dev")

    def sift_dev(self, gray_ptr, B, H, W, double_size, max_keypoints, xy_ptr, so_ptr, desc_ptr, counts_ptr):
        self._check(self.L.mc_sift_extract_dev(self.h, gray_ptr, B, H, W, 1 if double_size else 0, max_keypoints, xy_ptr, so_ptr, desc_ptr,
                                               counts_ptr), "mc_sift_extract_dev")

    def sift_profile_read(self):
        ms, by = C.c_float(0), C.c_double(0)
        self._check(self.L.mc_sift_profile_read(self.h, C.byref(ms), C.byref(by)), "mc_sift_profile_read")
        return float(ms.value), float(by.value)

    def sift_plane(self, frame, octave, stack, index):
        r, c = C.c_int32(0), C.c_int32(0)
        self._check(self.L.mc_sift_read_plane(self.h, frame, octave, stack, index, None, C.byref(r), C.byref(c)), "mc_sift_read_plane")
        out = np.zeros((r.value, c.value), np.float32)
        self._check(self.L.mc_sift_read_plane(self.h, frame, octave, stack, index, out.ctypes.data, None, None), "mc_sift_read_plane")
        return out

    def process_frame(self, q_desc, q_xy, q_image, params=None, max_objects=256, want_times=False):
        p = params or self.default_params()
        q = _f32(q_desc)
        n = C.c_int32(0)
        om = np.zeros(max_objects, np.int32)
        op = np.zeros((max_objects, 7), np.float32)
        os_ = np.zeros(max_objects, np.float32)
        ms = np.zeros(6, np.float32)
        self._check(self.L.mc_process_frame(self.h, q, _f32(q_xy), _i32(q_image), len(q), C.byref(p), max_objects, C.byref(n), om, op, os_,
                                            ms.ctypes.data if want_times else None), "mc_process_frame")
        k = n.value
        out = dict(model=om[:k].copy(), pose=op[:k].copy(), score=os_[:k].copy())
        if want_times:
            out["stage_ms"] = ms
        return out

    def process_matched_dev(self, nn_row_ptr, acc_ptr, xy_ptr, img_ptr, Q, params=None, max_objects=256, times=None):
        p = params or self.default_params()
        n = C.c_int32(0)
        om = np.zeros(max_objects, np.int32)
        op = np.zeros((max_objects, 7), np.float32)
        os_ = np.zeros(max_objects, np.float32)
        self._check(self.L.mc_process_matched_dev(self.h, nn_row_ptr, acc_ptr, xy_ptr, img_ptr, Q, C.byref(p), max_objects, C.byref(n), om, op, os_,
                                                  times.ctypes.data if times is not None else None), "mc_process_matched_dev")
        k = n.value
        return dict(model=om[:k].copy(), pose=op[:k].copy(), score=os_[:k].copy())

    def process_frame_dev(self, q_ptr, xy_ptr, img_ptr, Q, params=None, max_objects=256, times=None):
        p = params or self.default_params()
        n = C.c_int32(0)
        om = np.zeros(max_objects, np.int32)
        op = np.zeros((max_objects, 7), np.float32)
        os_ = np.zeros(max_objects, np.float32)
        self._check(self.L.mc_process_frame_dev(self.h, q_ptr, xy_ptr, img_ptr, Q, C.byref(p), max_objects, C.byref(n), om, op, os_,
                                                times.ctypes.data if times is not None else None), "mc_process_frame_dev")
        k = n.value
        return dict(model=om[:k].copy(), pose=op[:k].copy(), score=os_[:k].copy())

    # ---- frame batches
    def set_option(self, key: str, value: int):
        self._check(self.L.mc_set_option(self.h, key.encode(), int(value)), "mc_set_option")

    def set_tuning(self, frame_lanes=0, pose_warps_per_task=0, match_chunks=0):
        self._check(self.L.mc_set_tuning(self.h, int(frame_lanes), int(pose_warps_per_task), int(match_chunks)), "mc_set_tuning")

    @staticmethod
    def _unpack_frames(n_frames, max_objects, n_obj, om, op, os_, info):
        out = []
        for f in range(n_frames):
            k = int(n_obj[f])
            out.append(dict(model=om[f, :k].copy(), pose=op[f, :k].copy(), score=os_[f, :k].copy(), info=info[f].copy()))
        return out

    def process_frames(self, q_desc, q_xy, q_image, frame_offsets, params=None, max_objects=64, times=None):
        """Host-buffer batch call: list of per-frame dict(model, pose, score, info)."""
        p = params or self.default_params()
        fo = _i32(frame_offsets)
        nf = len(fo) - 1
        n_obj = np.zeros(nf, np.int32)
        om = np.zeros((nf, max_objects), np.int32)
        op = np.zeros((nf, max_objects, 7), np.float32)
        os_ = np.zeros((nf, max_objects), np.float32)
        info = np.zeros((nf, 4), np.int32)
        q = _f32(q_desc).reshape(-1, self.D)
        xy = _f32(q_xy).reshape(-1, 2)
        img = _i32(q_image).reshape(-1)
        if len(q) == 0:
            q, xy, img = np.zeros((1, self.D), np.float32), np.zeros((1, 2), np.float32), np.zeros(1, np.int32)
        self._check(self.L.mc_process_frames(self.h, q, xy, img, fo, nf, C.byref(p), max_objects, n_obj, om.reshape(-1), op.reshape(-1), os_.reshape(-1),
                                             info.ctypes.data, times.ctypes.data if times is not None else None), "mc_process_frames")
        return self._unpack_frames(nf, max_objects, n_obj, om, op, os_, info)

    def process_frames_dev(self, q_ptr, xy_ptr, img_ptr, frame_offsets, params=None, max_objects=64, times=None):
        p = params or self.default_params()
        fo = _i32(frame_offsets)
        nf = len(fo) - 1
        n_obj = np.zeros(nf, np.int32)
        om = np.zeros((nf, max_objects), np.int32)
        op = np.zeros((nf, max_objects, 7), np.float32)
        os_ = np.zeros((nf, max_objects), np.float32)
        info = np.zeros((nf, 4), np.int32)
        self._check(self.L.mc_process_frames_dev(self.h, q_ptr, xy_ptr, img_ptr, fo, nf, C.byref(p), max_objects, n_obj, om.reshape(-1), op.reshape(-1),
                                                 os_.reshape(-1), info.ctypes.data, times.ctypes.data if times is not None else None),
                    "mc_process_frames_dev")
        return self._unpack_frames(nf, max_objects, n_obj, om, op, os_, info)

    # ---- moped3d frames
    def default_depth_params(self) -> DepthPipelineParams:
        p = DepthPipelineParams()
        self.L.mc_depth_pipeline_default_params(C.byref(p))
        return p

    def _depth_frames(self, fn, what, match_offsets, n_models, arrays, params, max_objects, times):
        p = params or self.default_depth_params()
        mo = _i32(match_offsets).reshape(-1)
        nf = len(mo) // (int(n_models) + 1)
        n_obj = np.zeros(nf, np.int32)
        om = np.zeros((nf, max_objects), np.int32)
        op = np.zeros((nf, max_objects, 7), np.float32)
        os_ = np.zeros((nf, max_objects), np.float32)
        info = np.zeros((nf, 4), np.int32)
        st = fn(self.h, mo, nf, int(n_models), *arrays, C.byref(p), int(max_objects), n_obj, om.reshape(-1), op.reshape(-1), os_.reshape(-1),
                info.reshape(-1), times.ctypes.data if times is not None else None)
        self._check(st, what)
        return self._unpack_frames(nf, max_objects, n_obj, om, op, os_, info)

    def process_depth_frames(self, match_offsets, n_models, match_image, match_xy, match_xyz, match_world, match_fill, depth, fill_distance,
                             params=None, max_objects=64, times=None):
        """moped3d CLUSTER..FILTER2 on host arrays. match_offsets: [n_frames, n_models + 1] global CSR rows; depth / fill_distance:
        [n_frames, H, W] (or [H, W] for one frame). `times` (optional float32[5]) receives the per-step device time.
        Returns a list of per-frame dict(model, pose, score, info)."""
        d, fd = _f32(depth), _f32(fill_distance)
        H, W = d.shape[-2], d.shape[-1]
        keep = [_i32(match_image).reshape(-1), _f32(match_xy).reshape(-1), _f32(match_xyz).reshape(-1), _f32(match_world).reshape(-1),
                _f32(match_fill).reshape(-1)]
        arrays = [a.ctypes.data if a.size else None for a in keep] + [d.reshape(-1), fd.reshape(-1), W, H]
        return self._depth_frames(self.L.mc_process_depth_frames, "mc_process_depth_frames", match_offsets, n_models, arrays, params, max_objects,
                                  times)

    def process_depth_frames_dev(self, match_offsets, n_models, image_ptr, xy_ptr, xyz_ptr, world_ptr, fill_ptr, depth_ptr, fill_distance_ptr,
                                 width, height, params=None, max_objects=64, times=None):
        """The same with the per-match arrays and maps on the device (pointers); match_offsets stays a host array."""
        arrays = [image_ptr, xy_ptr, xyz_ptr, world_ptr, fill_ptr, depth_ptr, fill_distance_ptr, int(width), int(height)]
        return self._depth_frames(self.L.mc_process_depth_frames_dev, "mc_process_depth_frames_dev", match_offsets, n_models, arrays, params,
                                  max_objects, times)

    def set_depth_filter(self, step, params, test_offsets=None, test_xyz=None):
        """mc_set_depth_filter: step 0 = FILTER, 1 = FILTER2 of the moped3d chain runs FILTER_PROJECTION_DEPTH with `params`
        (DepthFilterParams) and the test points test_offsets [n_models + 1] / test_xyz [n, 3] (copied to the device now);
        params=None puts the step back to FILTER_PROJECTION."""
        if params is None:
            self._check(self.L.mc_set_depth_filter(self.h, int(step), None, None, None, 0), "mc_set_depth_filter")
            return
        to = _i32(test_offsets).reshape(-1)
        tx = _f32(test_xyz).reshape(-1) if test_xyz is not None else None
        self._check(self.L.mc_set_depth_filter(self.h, int(step), C.byref(params), to.ctypes.data, tx.ctypes.data if tx is not None and tx.size else None,
                                               len(to) - 1), "mc_set_depth_filter")

    def _depth_queries(self, fn, what, n_frames, n_models, args, params, max_objects, times, partial):
        p = params or self.default_depth_params()
        n_obj = np.zeros(n_frames, np.int32)
        om = np.zeros((max(n_frames, 1), max_objects), np.int32)
        op = np.zeros((max(n_frames, 1), max_objects, 7), np.float32)
        os_ = np.zeros((max(n_frames, 1), max_objects), np.float32)
        info = np.zeros((max(n_frames, 1), 4), np.int32)
        st = fn(self.h, *args, C.byref(p), int(max_objects), n_obj if n_frames else np.zeros(1, np.int32), om.reshape(-1), op.reshape(-1),
                os_.reshape(-1), info.reshape(-1), times.ctypes.data if times is not None else None)
        if st != 0 and not (partial and st in (MC_ERR_ARG, MC_ERR_CAPACITY)):
            self._check(st, what)
        n_obj = np.where((info[:n_frames, 1] != 0) | (n_obj > max_objects), 0, n_obj)   # a failed frame has no objects; info keeps its counts
        frames = self._unpack_frames(n_frames, max_objects, n_obj, om, op, os_, info)
        return (frames, int(st)) if partial else frames

    def process_depth_queries(self, q_desc, q_xy, q_image, q_world, q_fill, frame_offsets, depth, fill_distance, models, depths=ADAPTIVE_DEPTHS,
                              params=None, max_objects=64, times=None, partial=False):
        """moped3d from features to objects on host arrays (mc_process_depth_queries): MATCH, the per-match gather of DEPTHPROP's q_world
        [Q, 3] / q_fill [Q], CLUSTER..FILTER2. q_desc [Q, D], q_xy [Q, 2], q_image [Q] or None, frame_offsets [n_frames + 1],
        depth / fill_distance [n_frames, H, W], models = ADAPTIVE_MODEL records. `times` (optional float32[2]) receives the device time
        of MATCH and of CLUSTER..FILTER2. Returns the per-frame dict(model, pose, score, info) of process_depth_frames; info = {objects,
        status, accepted matches, clusters}. partial=True returns (frames, status) and does not raise for a frame that failed (MC_ERR_ARG,
        MC_ERR_CAPACITY)."""
        fo = _i32(frame_offsets).reshape(-1)
        cv = self._curves(models)
        d, fd = _f32(depth), _f32(fill_distance)
        keep = [_f32(q_desc).reshape(-1, self.D), _f32(q_xy).reshape(-1, 2), _i32(q_image).reshape(-1) if q_image is not None else None,
                _f32(q_world).reshape(-1, 3) if q_world is not None else None, _f32(q_fill).reshape(-1) if q_fill is not None else None]
        ptrs = [a.ctypes.data if a is not None and a.size else None for a in keep]
        args = ptrs + [fo, len(fo) - 1, d.ctypes.data, fd.ctypes.data, d.shape[-1], d.shape[-2], cv.ctypes.data, len(cv), *[float(v) for v in depths]]
        return self._depth_queries(self.L.mc_process_depth_queries, "mc_process_depth_queries", len(fo) - 1, len(cv), args, params, max_objects,
                                   times, partial)

    def process_depth_queries_dev(self, q_ptr, xy_ptr, img_ptr, world_ptr, fill_ptr, frame_offsets, depth_ptr, fill_distance_ptr, width, height,
                                  models, depths=ADAPTIVE_DEPTHS, params=None, max_objects=64, times=None, partial=False):
        """mc_process_depth_queries_dev: the same with the per-feature arrays and the planes on the device (pointers)."""
        fo = _i32(frame_offsets).reshape(-1)
        cv = self._curves(models)
        args = [q_ptr, xy_ptr, img_ptr, world_ptr, fill_ptr, fo, len(fo) - 1, depth_ptr, fill_distance_ptr, int(width), int(height), cv.ctypes.data,
                len(cv), *[float(v) for v in depths]]
        return self._depth_queries(self.L.mc_process_depth_queries_dev, "mc_process_depth_queries_dev", len(fo) - 1, len(cv), args, params,
                                   max_objects, times, partial)

    def process_depth_queries_merged_dev(self, packed_all_ptr, n_shards, xy_ptr, img_ptr, world_ptr, fill_ptr, frame_offsets, frame_begin, frame_end,
                                         depth_ptr, fill_distance_ptr, width, height, models, depths=ADAPTIVE_DEPTHS, params=None, max_objects=64,
                                         times=None, partial=False):
        """mc_process_depth_queries_merged_dev: frames [frame_begin, frame_end) from the n_shards gathered packed blocks; the per-feature
        arrays hold the whole batch, depth_ptr / fill_distance_ptr the range's planes only. One dict per frame of the range."""
        fo = _i32(frame_offsets).reshape(-1)
        cv = self._curves(models)
        args = [packed_all_ptr, int(n_shards), xy_ptr, img_ptr, world_ptr, fill_ptr, fo, len(fo) - 1, int(frame_begin), int(frame_end), depth_ptr,
                fill_distance_ptr, int(width), int(height), cv.ctypes.data, len(cv), *[float(v) for v in depths]]
        return self._depth_queries(self.L.mc_process_depth_queries_merged_dev, "mc_process_depth_queries_merged_dev",
                                   max(int(frame_end) - int(frame_begin), 0), len(cv), args, params, max_objects, times, partial)

    def process_frames_matched_dev(self, nn_row_ptr, acc_ptr, xy_ptr, img_ptr, frame_offsets, frame_begin, frame_end, params, max_objects,
                                   info_ptr, model_ptr, pose_ptr, score_ptr):
        fo = _i32(frame_offsets)
        self._check(self.L.mc_process_frames_matched_dev(self.h, nn_row_ptr, acc_ptr, xy_ptr, img_ptr, fo, len(fo) - 1, int(frame_begin), int(frame_end),
                                                         C.byref(params), int(max_objects), info_ptr, model_ptr, pose_ptr, score_ptr),
                    "mc_process_frames_matched_dev")


    def frame_shard_slot_bytes(self, n_features, params):
        """bytes of one rank's exchange record of mc_process_frame_sharded_dev (the exchange buffer holds shard_world of them)"""
        return int(self.L.mc_frame_shard_slot_bytes(int(n_features), C.byref(params)))

    def process_frame_sharded_dev(self, phase, nn_row_ptr, acc_ptr, xy_ptr, img_ptr, n_features, params, shard_rank, shard_world, exchange_ptr,
                                  max_objects, info_ptr, model_ptr, pose_ptr, score_ptr):
        """One phase (0, 1, 2) of a frame whose RANSAC tasks are distributed by cluster over shard_world ranks; the caller all-gathers the
        exchange buffer in place between the phases. Asynchronous on the context's stream."""
        self._check(self.L.mc_process_frame_sharded_dev(self.h, int(phase), nn_row_ptr, acc_ptr, xy_ptr, img_ptr, int(n_features), C.byref(params),
                                                        int(shard_rank), int(shard_world), exchange_ptr, int(max_objects), info_ptr, model_ptr,
                                                        pose_ptr, score_ptr), "mc_process_frame_sharded_dev")


class ModelDB:
    """ctypes view of the model-database loader (mc_model_db_*): `.moped.xml` files -> packed rows -> device."""

    def __init__(self):
        self.L = load()
        h = C.c_void_p()
        st = self.L.mc_model_db_create(C.byref(h))
        if st != 0:
            raise MopedCudaError("mc_model_db_create failed")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.mc_model_db_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st, what):
        if st != 0:
            raise MopedCudaError(f"{what}: status {st}: {self.L.mc_model_db_last_error(self.h).decode()}")

    def add_xml_file(self, path):
        self._check(self.L.mc_model_db_add_xml_file(self.h, os.fsencode(path)), "mc_model_db_add_xml_file")

    def add_xml_files(self, paths, n_threads=0):
        arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
        self._check(self.L.mc_model_db_add_xml_files(self.h, arr, len(paths), n_threads), "mc_model_db_add_xml_files")

    def add_xml_buffer(self, data: bytes):
        self._check(self.L.mc_model_db_add_xml_buffer(self.h, data, len(data)), "mc_model_db_add_xml_buffer")

    def remove(self, name):
        self._check(self.L.mc_model_db_remove(self.h, name.encode()), "mc_model_db_remove")

    def names(self):
        return [self.L.mc_model_db_model_name(self.h, i).decode() for i in range(self.L.mc_model_db_n_models(self.h))]

    def bbox(self, i):
        b = np.zeros(6, np.float32)
        self._check(self.L.mc_model_db_model_bbox(self.h, i, b), "mc_model_db_model_bbox")
        return b

    def pack(self, desc_type="SIFT", desc_size=128, normalise=True):
        """Copies of the packed rows: dict(desc[N,D], xyz[N,3], model_of_row[N], n_pts[n_models])."""
        n = C.c_int64()
        pd, px, pm, pn = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(self.L.mc_model_db_pack(self.h, desc_type.encode(), desc_size, 1 if normalise else 0, C.byref(n), C.byref(pd), C.byref(px),
                                            C.byref(pm), C.byref(pn)), "mc_model_db_pack")
        N, M = n.value, self.L.mc_model_db_n_models(self.h)

        def view(ptr, ctype, count, shape):
            if count == 0:
                return np.zeros(shape, dtype=np.dtype(ctype))
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(count,)).reshape(shape).copy()
        return dict(desc=view(pd, C.c_float, N * desc_size, (N, desc_size)), xyz=view(px, C.c_float, N * 3, (N, 3)),
                    model_of_row=view(pm, C.c_int32, N, (N,)), n_pts=view(pn, C.c_int32, M, (M,)))

    def upload(self, ctx: "Context", desc_type="SIFT", desc_size=128):
        self._check(self.L.mc_model_db_upload(self.h, ctx.h, desc_type.encode(), desc_size), "mc_model_db_upload")

    def save(self, path):
        self._check(self.L.mc_model_db_save(self.h, os.fsencode(path)), "mc_model_db_save")

    def load(self, path):
        self._check(self.L.mc_model_db_load(self.h, os.fsencode(path)), "mc_model_db_load")
