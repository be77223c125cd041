"""ctypes binding of include/gm_capi.h (the C-ABI of csrc/libgm_b200.so).

This is the only way Python reaches the product: there is no CPU implementation to fall back
to.  A missing library is built with nvcc if possible (cross-compiles without a GPU), otherwise
the import raises; a missing CUDA device makes `Context()` raise GmError(GM_ERR_NO_DEVICE).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

GM_OK = 0
GM_ERR_INVALID_ARG = 1
GM_ERR_NO_DEVICE = 2
GM_ERR_CUDA = 3
GM_ERR_CAPACITY = 4
GM_ERR_STAGE_ORDER = 5
GM_WARN_VOXEL_OVERFLOW = 6
GM_ERR_NN_INDEX_RANGE = 7
GM_ERR_INTERNAL = 8
GM_ERR_NO_MODEL = 9

GM_MODEL_PLANE = 0
GM_MODEL_CYLINDER = 1


class gm_params(C.Structure):
    _fields_ = [
        ("boxFilterBound", C.c_double),
        ("voxelGridLeafSize", C.c_double),
        ("neighborRadius", C.c_double),
        ("weightingFactor", C.c_double),
        ("displayCloud", C.c_int32),
        ("displayNormals", C.c_int32),
        ("displayCenterAxis", C.c_int32),
        ("usePCLViz", C.c_int32),
        ("is_dense", C.c_int32),
        ("nn_index_mode", C.c_int32),
        ("ransacThreshold", C.c_double),
        ("cylinderRadiusMin", C.c_double),
        ("cylinderRadiusMax", C.c_double),
        ("refitIterations", C.c_int32),
        ("maxSlices", C.c_int32),
        ("sliceLength", C.c_double),
        ("weight_mode", C.c_int32),
        ("arrow_mode", C.c_int32),
    ]


class gm_counts(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_input", "n_cropped", "n_valid", "n_voxels", "n_cells", "voxel_overflow", "nn_out_of_range", "device_error")]


class gm_frame(C.Structure):
    _fields_ = [("vals", C.c_float * 3), ("vecs", C.c_float * 9), ("scatter", C.c_float * 9)]


class gm_arrow(C.Structure):
    _fields_ = [("start", C.c_float * 3), ("end", C.c_float * 3), ("scale", C.c_float * 3),
                ("color_argb", C.c_float * 4), ("id", C.c_int32)]


class gm_model(C.Structure):
    _fields_ = [("kind", C.c_int32), ("best_id", C.c_int32), ("best_count", C.c_int32), ("refit_count", C.c_int32),
                ("hyp", C.c_float * 8), ("coef", C.c_float * 8), ("rms", C.c_float), ("pad_", C.c_float)]


class gm_slice(C.Structure):
    _fields_ = [("center", C.c_float * 3), ("dir", C.c_float * 3), ("radius", C.c_float), ("rms", C.c_float),
                ("t_mid", C.c_float), ("count", C.c_int32)]


class gm_compression(C.Structure):
    _fields_ = [("n_points", C.c_int32), ("n_plane", C.c_int32), ("n_cylinder", C.c_int32), ("n_residual", C.c_int32),
                ("n_residual_voxels", C.c_int32), ("n_slices", C.c_int32), ("plane_coef", C.c_float * 4),
                ("plane_u", C.c_float * 3), ("plane_v", C.c_float * 3), ("plane_bounds", C.c_float * 4), ("plane_rms", C.c_float),
                ("cyl_coef", C.c_float * 7), ("cyl_t_range", C.c_float * 2), ("cyl_rms", C.c_float), ("residual_rms", C.c_float),
                ("total_rms", C.c_float), ("leaf", C.c_float), ("ratio", C.c_float), ("bytes_in", C.c_uint64),
                ("bytes_out", C.c_uint64)]


class gm_primitive(C.Structure):
    _fields_ = [("model", gm_model), ("n_remaining", C.c_int32), ("pad_", C.c_int32)]


class gm_primitive_compression(C.Structure):
    _fields_ = [("n_points", C.c_int32), ("n_primitives", C.c_int32), ("n_residual", C.c_int32), ("n_residual_voxels", C.c_int32),
                ("leaf", C.c_float), ("residual_rms", C.c_float), ("total_rms", C.c_float), ("ratio", C.c_float),
                ("bytes_in", C.c_uint64), ("bytes_out", C.c_uint64)]


class gm_icp_params(C.Structure):
    _fields_ = [("init_pose34", C.c_float * 12), ("max_correspondence_distance", C.c_double), ("max_iterations", C.c_int32),
                ("pad_", C.c_int32), ("min_rotation_step", C.c_double), ("min_translation_step", C.c_double),
                ("degeneracy_ratio", C.c_double)]


class gm_registration(C.Structure):
    _fields_ = [("pose34", C.c_float * 12), ("iterations", C.c_int32), ("converged", C.c_int32), ("n_source", C.c_int32),
                ("n_correspondences", C.c_int32), ("rmse", C.c_float), ("fitness", C.c_float), ("n_degenerate", C.c_int32),
                ("pad_", C.c_int32), ("eigenvalues", C.c_double * 6), ("eigenvectors", C.c_double * 36)]


class gm_odometry_params(C.Structure):
    _fields_ = [("icp", gm_icp_params), ("max_planarity", C.c_double), ("min_fitness", C.c_double), ("register_first", C.c_int32),
                ("max_steps", C.c_int32)]


class gm_odometry_record(C.Structure):
    _fields_ = [("pose34", C.c_float * 12), ("guess34", C.c_float * 12), ("accepted", C.c_int32), ("registered", C.c_int32),
                ("iterations", C.c_int32), ("converged", C.c_int32), ("n_source", C.c_int32), ("n_correspondences", C.c_int32),
                ("n_degenerate", C.c_int32), ("rmse", C.c_float), ("fitness", C.c_float), ("pad_", C.c_int32)]


GM_MAX_ICP_ITERATIONS = 64
GM_MAX_PRIMITIVES = 64
PRIMITIVE_RECORD_DTYPE = np.dtype([("kind", "<i4"), ("count", "<i4"), ("coef", "<f4", 7), ("extents", "<f4", 4), ("rms", "<f4")])


class gm_scan_summary(C.Structure):
    _fields_ = [("counts", gm_counts), ("frame", gm_frame), ("plane", gm_model), ("cylinder", gm_model),
                ("n_slices", C.c_int32), ("pad_", C.c_int32)]


class gm_host_outputs(C.Structure):
    _fields_ = [("summary", C.c_void_p), ("cloud_xyzw", C.c_void_p), ("cloud_capacity", C.c_size_t),
                ("normals8", C.c_void_p), ("normals_capacity", C.c_size_t), ("labels", C.c_void_p),
                ("labels_capacity", C.c_size_t), ("slices", C.c_void_p), ("slices_capacity", C.c_int32),
                ("centroids_xyzw", C.c_void_p), ("nn_normal8", C.c_void_p), ("voxel_capacity", C.c_size_t)]


SLICE_DTYPE = np.dtype([("center", "<f4", 3), ("dir", "<f4", 3), ("radius", "<f4"), ("rms", "<f4"),
                        ("t_mid", "<f4"), ("count", "<i4")])
ARROW_DTYPE = np.dtype([("start", "<f4", 3), ("end", "<f4", 3), ("scale", "<f4", 3), ("color_argb", "<f4", 4),
                        ("id", "<i4")])


class GmError(RuntimeError):
    def __init__(self, status: int, where: str, detail: str = ""):
        self.status = status
        msg = f"{where}: gm_status {status} ({_lib().gm_status_string(status).decode()})"
        if detail:
            msg += f": {detail}"
        super().__init__(msg)


_LIB = None

# every symbol include/gm_capi.h declares; tests/test_abi.py checks the list against the header
SYMBOLS = [
    "gm_params_default", "gm_create", "gm_destroy", "gm_set_params", "gm_get_params", "gm_markers_normals_mode", "gm_set_stream", "gm_last_error",
    "gm_status_string", "gm_version", "gm_launch_count", "gm_reset_launch_count", "gm_synchronize",
    "gm_upload_scan", "gm_set_scan_device", "gm_crop", "gm_normals", "gm_voxel", "gm_local_frame", "gm_ransac",
    "gm_ransac_key_device_ptr", "gm_ransac_select", "gm_label", "gm_axis_polyline", "gm_process_scan",
    "gm_get_counts", "gm_download_cloud", "gm_download_normals", "gm_download_neighbor_counts",
    "gm_download_valid_map", "gm_download_voxel_assignment", "gm_download_voxels", "gm_get_voxel_grid",
    "gm_get_frame", "gm_download_hypotheses", "gm_get_model", "gm_download_labels", "gm_download_polyline",
    "gm_inject_compacted", "gm_markers_eigen", "gm_markers_normals", "gm_fetch_async", "gm_profile_enable",
    "gm_profile_num_segments", "gm_profile_segment_name", "gm_profile_read", "gm_compress", "gm_get_compression",
    "gm_download_compressed", "gm_upload_pointcloud2", "gm_ransac_export_key", "gm_ransac_import_key", "gm_set_count_mode", "gm_set_grid_box", "gm_set_owned_range", "gm_get_voxel_bbox", "gm_set_voxel_bbox",
    "gm_get_search_stats", "gm_set_voxel_mode", "gm_ransac_pair", "gm_ransac_select_pair", "gm_ransac_export_keys",
    "gm_ransac_import_keys", "gm_map_create", "gm_map_destroy", "gm_map_clear", "gm_map_insert", "gm_map_stats", "gm_map_download", "gm_map_save",
    "gm_map_load", "gm_map_leaf", "gm_set_normals_mode", "gm_set_graph_mode", "gm_get_graph_stats",
    "gm_comm_create", "gm_comm_handle", "gm_comm_connect", "gm_comm_mailbox", "gm_comm_connect_local", "gm_comm_destroy", "gm_comm_rank", "gm_comm_world", "gm_comm_last_error", "gm_set_comm", "gm_ransac_sharded", "gm_allreduce_voxel_bbox", "gm_allreduce_frame", "gm_set_voxel_bbox_hint", "gm_set_knn", "gm_download_knn_indices", "gm_set_knn_max_radius", "gm_pointcloud2_size", "gm_encode_pointcloud2", "gm_marker_array_size",
    "gm_extract_primitives", "gm_get_primitives", "gm_download_primitive_ids", "gm_compress_primitives",
    "gm_download_compressed_primitives", "gm_icp_params_default", "gm_register", "gm_get_registration",
    "gm_download_correspondences", "gm_register_map", "gm_download_map_correspondences", "gm_map_download_planes",
    "gm_odometry_params_default", "gm_odometry_create", "gm_odometry_destroy", "gm_odometry_step", "gm_odometry_steps", "gm_odometry_get",
    "gm_map_evict", "gm_map_merge", "gm_odometry_set_window",
    "gm_upload_pointcloud2_timed", "gm_download_point_times", "gm_deskew", "gm_odometry_deskew",
    "gm_encode_marker_array", "gm_store_open", "gm_store_close", "gm_store_append", "gm_store_append_blob", "gm_store_count", "gm_store_info", "gm_store_read",
]


def library_path() -> str:
    return _build.LIB


def _lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB
    if not os.path.exists(path):
        _build.build()  # raises if nvcc is missing: no CPU fallback
    lib = C.CDLL(path)
    vp, i32, i64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
    sig = {
        "gm_params_default": (None, [C.POINTER(gm_params)]),
        "gm_create": (i32, [C.POINTER(gm_params), sz, i32, C.POINTER(vp)]),
        "gm_destroy": (None, [vp]),
        "gm_set_params": (i32, [vp, C.POINTER(gm_params)]),
        "gm_get_params": (i32, [vp, C.POINTER(gm_params)]),
        "gm_markers_normals_mode": (None, [vp, vp, i32, i32, vp]),
        "gm_set_stream": (i32, [vp, vp]),
        "gm_last_error": (C.c_char_p, [vp]),
        "gm_status_string": (C.c_char_p, [i32]),
        "gm_version": (i32, []),
        "gm_launch_count": (i64, [vp]),
        "gm_reset_launch_count": (None, [vp]),
        "gm_synchronize": (i32, [vp]),
        "gm_upload_scan": (i32, [vp, vp, sz, sz]),
        "gm_set_scan_device": (i32, [vp, vp, sz]),
        "gm_crop": (i32, [vp]),
        "gm_normals": (i32, [vp]),
        "gm_voxel": (i32, [vp]),
        "gm_local_frame": (i32, [vp]),
        "gm_ransac": (i32, [vp, i32, vp, i32, i32, i32]),
        "gm_ransac_key_device_ptr": (i32, [vp, i32, C.POINTER(vp)]),
        "gm_ransac_select": (i32, [vp, i32]),
        "gm_label": (i32, [vp]),
        "gm_axis_polyline": (i32, [vp]),
        "gm_process_scan": (i32, [vp, vp, i32, vp, i32]),
        "gm_get_counts": (i32, [vp, C.POINTER(gm_counts)]),
        "gm_download_cloud": (i32, [vp, i32, vp, sz]),
        "gm_download_normals": (i32, [vp, i32, vp, sz]),
        "gm_download_neighbor_counts": (i32, [vp, vp, sz]),
        "gm_download_valid_map": (i32, [vp, vp, sz]),
        "gm_download_voxel_assignment": (i32, [vp, vp, vp, sz]),
        "gm_download_voxels": (i32, [vp, vp, vp, vp, vp, vp, sz]),
        "gm_get_voxel_grid": (i32, [vp, C.POINTER(i32 * 6)]),
        "gm_get_frame": (i32, [vp, C.POINTER(gm_frame)]),
        "gm_download_hypotheses": (i32, [vp, i32, vp, vp, vp, i32]),
        "gm_get_model": (i32, [vp, i32, C.POINTER(gm_model)]),
        "gm_download_labels": (i32, [vp, vp, sz]),
        "gm_download_polyline": (i32, [vp, vp, i32, C.POINTER(i32)]),
        "gm_inject_compacted": (i32, [vp, vp, vp, sz]),
        "gm_markers_eigen": (None, [C.POINTER(gm_frame), vp]),
        "gm_markers_normals": (None, [vp, vp, i32, vp]),
        "gm_fetch_async": (i32, [vp, C.POINTER(gm_host_outputs)]),
        "gm_profile_enable": (i32, [vp, i32]),
        "gm_profile_num_segments": (i32, []),
        "gm_profile_segment_name": (C.c_char_p, [i32]),
        "gm_profile_read": (i32, [vp, vp, vp]),
        "gm_compress": (i32, [vp]),
        "gm_get_compression": (i32, [vp, C.POINTER(gm_compression)]),
        "gm_download_compressed": (i32, [vp, vp, sz, C.POINTER(sz)]),
        "gm_upload_pointcloud2": (i32, [vp, vp, sz, sz, sz, sz, sz]),
        "gm_ransac_export_key": (i32, [vp, i32, vp]),
        "gm_ransac_import_key": (i32, [vp, i32, vp]),
        "gm_set_count_mode": (i32, [vp, i32]),
        "gm_set_normals_mode": (i32, [vp, i32]),
        "gm_set_graph_mode": (i32, [vp, i32]),
        "gm_get_graph_stats": (i32, [vp, C.POINTER(i64), C.POINTER(i64)]),
        "gm_comm_create": (i32, [i32, i32, C.POINTER(vp)]),
        "gm_comm_handle": (i32, [vp, vp]),
        "gm_comm_connect": (i32, [vp, vp]),
        "gm_comm_mailbox": (i32, [vp, C.POINTER(vp)]),
        "gm_comm_connect_local": (i32, [vp, C.POINTER(vp)]),
        "gm_comm_destroy": (None, [vp]),
        "gm_comm_rank": (i32, [vp]),
        "gm_comm_world": (i32, [vp]),
        "gm_comm_last_error": (C.c_char_p, [vp]),
        "gm_set_comm": (i32, [vp, vp]),
        "gm_ransac_sharded": (i32, [vp, vp, i32, vp, i32]),
        "gm_allreduce_voxel_bbox": (i32, [vp]),
        "gm_allreduce_frame": (i32, [vp]),
        "gm_set_voxel_bbox_hint": (i32, [vp, vp, vp]),
        "gm_set_knn": (i32, [vp, i32, i32]),
        "gm_download_knn_indices": (i32, [vp, vp, sz]),
        "gm_set_knn_max_radius": (i32, [vp, C.c_double]),
        "gm_pointcloud2_size": (sz, [sz, C.c_char_p]),
        "gm_encode_pointcloud2": (i32, [vp, sz, C.c_char_p, C.c_uint32, C.c_uint64, i32, vp, sz, C.POINTER(sz)]),
        "gm_marker_array_size": (sz, [i32, C.c_char_p, C.c_char_p]),
        "gm_encode_marker_array": (i32, [vp, i32, C.c_char_p, C.c_char_p, C.c_uint64, vp, sz, C.POINTER(sz)]),
        "gm_store_open": (i32, [C.c_char_p, i32, C.POINTER(vp)]),
        "gm_store_close": (None, [vp]),
        "gm_store_append": (i32, [vp, vp, C.c_uint64, C.c_uint64, vp]),
        "gm_store_append_blob": (i32, [vp, C.c_uint64, C.c_uint64, vp, vp, sz]),
        "gm_store_count": (i64, [vp]),
        "gm_store_info": (i32, [vp, i64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), vp, C.POINTER(C.c_uint64)]),
        "gm_store_read": (i32, [vp, i64, vp, sz, C.POINTER(sz)]),
        "gm_set_grid_box": (i32, [vp, vp, vp]),
        "gm_set_owned_range": (i32, [vp, i32, C.c_float, C.c_float]),
        "gm_get_voxel_bbox": (i32, [vp, vp, vp]),
        "gm_set_voxel_bbox": (i32, [vp, vp, vp]),
        "gm_get_search_stats": (i32, [vp, C.POINTER(i64), C.POINTER(i64)]),
        "gm_set_voxel_mode": (i32, [vp, i32]),
        "gm_ransac_pair": (i32, [vp, vp, i32, i32, i32, vp, i32, i32, i32]),
        "gm_ransac_select_pair": (i32, [vp]),
        "gm_ransac_export_keys": (i32, [vp, vp]),
        "gm_ransac_import_keys": (i32, [vp, vp]),
        "gm_map_create": (i32, [C.c_double, sz, C.POINTER(vp)]),
        "gm_map_destroy": (None, [vp]),
        "gm_map_clear": (i32, [vp]),
        "gm_map_insert": (i32, [vp, vp, vp, i32]),
        "gm_map_stats": (i32, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "gm_map_download": (i32, [vp, vp, vp, vp, sz, C.POINTER(sz)]),
        "gm_map_save": (i32, [vp, C.c_char_p]),
        "gm_map_load": (i32, [C.c_char_p, sz, C.POINTER(vp)]),
        "gm_map_leaf": (C.c_double, [vp]),
        "gm_extract_primitives": (i32, [vp, i32, i32, vp, i32, vp, i32]),
        "gm_get_primitives": (i32, [vp, vp, i32, C.POINTER(i32)]),
        "gm_download_primitive_ids": (i32, [vp, vp, sz]),
        "gm_compress_primitives": (i32, [vp]),
        "gm_download_compressed_primitives": (i32, [vp, vp, sz, C.POINTER(sz)]),
        "gm_icp_params_default": (None, [C.POINTER(gm_icp_params)]),
        "gm_register": (i32, [vp, vp, C.POINTER(gm_icp_params)]),
        "gm_get_registration": (i32, [vp, C.POINTER(gm_registration)]),
        "gm_download_correspondences": (i32, [vp, vp, vp, sz]),
        "gm_register_map": (i32, [vp, vp, C.POINTER(gm_icp_params), C.c_double]),
        "gm_download_map_correspondences": (i32, [vp, vp, vp, sz]),
        "gm_map_download_planes": (i32, [vp, C.c_double, vp, sz, C.POINTER(sz)]),
        "gm_odometry_params_default": (None, [C.POINTER(gm_odometry_params)]),
        "gm_odometry_create": (i32, [vp, C.POINTER(gm_odometry_params), C.POINTER(vp)]),
        "gm_odometry_destroy": (None, [vp]),
        "gm_odometry_step": (i32, [vp, vp, vp]),
        "gm_odometry_steps": (i32, [vp]),
        "gm_odometry_get": (i32, [vp, vp, i32, C.POINTER(i32)]),
        "gm_map_evict": (i32, [vp, vp, vp, vp, i32]),
        "gm_map_merge": (i32, [vp, vp]),
        "gm_odometry_set_window": (i32, [vp, i32, vp]),
        "gm_upload_pointcloud2_timed": (i32, [vp, vp, sz, sz, sz, sz, sz, sz]),
        "gm_download_point_times": (i32, [vp, vp, sz]),
        "gm_deskew": (i32, [vp, vp, C.c_double, C.c_double]),
        "gm_odometry_deskew": (i32, [vp, vp, C.c_double, C.c_double]),
    }
    assert set(sig) == set(SYMBOLS)
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


def default_params(**overrides) -> gm_params:
    p = gm_params()
    _lib().gm_params_default(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise AttributeError(f"gm_params has no field {k}")
        setattr(p, k, v)
    return p


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _as_xyzw(points: np.ndarray) -> np.ndarray:
    a = np.ascontiguousarray(points, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("points must be n x 3 or n x 4 float32")
    if a.shape[1] == 3:
        a = np.concatenate([a, np.ones((a.shape[0], 1), np.float32)], axis=1)
    return a


class Context:
    """Owns one gm_ctx.  All heavy lifting happens in the CUDA library."""

    def __init__(self, params: gm_params | None = None, max_points: int = 1 << 20, max_hypotheses: int = 4096):
        lib = _lib()
        self.params = params if params is not None else default_params()
        self.max_points = int(max_points)
        self.max_hypotheses = int(max_hypotheses)
        h = C.c_void_p()
        st = lib.gm_create(C.byref(self.params), self.max_points, self.max_hypotheses, C.byref(h))
        if st != GM_OK:
            raise GmError(st, "gm_create")
        self._h = h
        self._keepalive = None

    # -- plumbing ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            _lib().gm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, st: int, where: str, ok=(GM_OK,)):
        if st not in ok:
            raise GmError(st, where, _lib().gm_last_error(self._h).decode())
        return st

    def set_params(self, params: gm_params):
        self._ck(_lib().gm_set_params(self._h, C.byref(params)), "gm_set_params")
        self.params = params

    def set_stream(self, cuda_stream: int | None):
        """cuda_stream: a cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream); None = the
        context's own stream.  The handle 0 names CUDA's legacy default stream (what torch's default
        stream is), which the C-ABI spells cudaStreamLegacy (0x1) because NULL means "own stream" there."""
        if cuda_stream is None:
            h = 0
        elif cuda_stream == 0:
            h = 1  # cudaStreamLegacy
        else:
            h = cuda_stream
        self._ck(_lib().gm_set_stream(self._h, C.c_void_p(h)), "gm_set_stream")

    def set_count_mode(self, mode: int):
        """0 = tile-culled inlier counting (default), 1 = brute-force FP32 kernels; identical counts."""
        self._ck(_lib().gm_set_count_mode(self._h, mode), "gm_set_count_mode")

    def set_normals_mode(self, mode: int):
        """0 = neighbourhood sums in grid order (fast, default); 1 = in FLANN's (d2, index) order: normals bit-identical
        to the CPU oracle (verification mode, slow)."""
        self._ck(_lib().gm_set_normals_mode(self._h, mode), "gm_set_normals_mode")

    def set_comm(self, comm: "PeerComm | None"):
        """Attach a connected PeerComm: ransac_sharded / allreduce_voxel_bbox / allreduce_frame then run over NVLink peer memory."""
        self._ck(_lib().gm_set_comm(self._h, comm._h if comm is not None else None), "gm_set_comm")
        self._comm = comm

    def ransac_sharded(self, plane_samples: np.ndarray, cyl_samples: np.ndarray):
        ps = np.ascontiguousarray(plane_samples, np.int32)
        cs = np.ascontiguousarray(cyl_samples, np.int32)
        self._keepalive = (ps, cs)
        self._ck(_lib().gm_ransac_sharded(self._h, _ptr(ps), ps.shape[0], _ptr(cs), cs.shape[0]), "gm_ransac_sharded")

    def allreduce_voxel_bbox(self):
        self._ck(_lib().gm_allreduce_voxel_bbox(self._h), "gm_allreduce_voxel_bbox")

    def allreduce_frame(self):
        self._ck(_lib().gm_allreduce_frame(self._h), "gm_allreduce_frame")

    def set_voxel_bbox_hint(self, mn=None, mx=None):
        if mn is None:
            self._ck(_lib().gm_set_voxel_bbox_hint(self._h, None, None), "gm_set_voxel_bbox_hint")
        else:
            a, b = np.ascontiguousarray(mn, np.float32), np.ascontiguousarray(mx, np.float32)
            self._ck(_lib().gm_set_voxel_bbox_hint(self._h, _ptr(a), _ptr(b)), "gm_set_voxel_bbox_hint")

    def set_knn(self, k: int, keep_indices: bool = False, max_radius: float = 0.0):
        """k > 0: k-nearest-neighbour normals (setKSearch) instead of the radius search; 0 = radius mode.
        max_radius > 0: only neighbours nearer than that count (the k nearest within the radius)."""
        self._ck(_lib().gm_set_knn(self._h, k, 1 if keep_indices else 0), "gm_set_knn")
        self._ck(_lib().gm_set_knn_max_radius(self._h, float(max_radius)), "gm_set_knn_max_radius")
        self._knn = k

    def download_knn_indices(self) -> np.ndarray:
        m = max(self.counts().n_cropped, 0)
        out = np.empty((m, self._knn), np.int32)
        self._ck(_lib().gm_download_knn_indices(self._h, _ptr(out), m), "gm_download_knn_indices")
        return out

    def set_graph_mode(self, mode: int):
        """2 = auto (default: graphs for scans up to 524288 points), 1 = always replay a captured CUDA graph, 0 = plain launches."""
        self._ck(_lib().gm_set_graph_mode(self._h, mode), "gm_set_graph_mode")

    def graph_stats(self):
        """-> (graphs captured, graph launches) of process_scan since the context was created"""
        a, b = C.c_int64(0), C.c_int64(0)
        self._ck(_lib().gm_get_graph_stats(self._h, C.byref(a), C.byref(b)), "gm_get_graph_stats")
        return int(a.value), int(b.value)

    def set_grid_box(self, mn=None, mx=None):
        """Neighbour grid over [mn, mx] instead of the crop cube (map slabs); None clears."""
        if mn is None:
            self._ck(_lib().gm_set_grid_box(self._h, None, None), "gm_set_grid_box")
        else:
            a, b = np.ascontiguousarray(mn, np.float32), np.ascontiguousarray(mx, np.float32)
            self._ck(_lib().gm_set_grid_box(self._h, _ptr(a), _ptr(b)), "gm_set_grid_box")

    def set_owned_range(self, axis: int = -1, lo: float = 0.0, hi: float = 0.0):
        """Points with coord[axis] outside [lo, hi) are halo: searched, then dropped with the NaN normals."""
        self._ck(_lib().gm_set_owned_range(self._h, axis, lo, hi), "gm_set_owned_range")

    def set_voxel_mode(self, mode: int):
        """0 = sort-free dense VoxelGrid when the lattice fits (default), 1 = always sort-based; identical results."""
        self._ck(_lib().gm_set_voxel_mode(self._h, mode), "gm_set_voxel_mode")

    def search_stats(self):
        """-> (distance tests executed, neighbours found) of the last normals()"""
        a, b = C.c_int64(0), C.c_int64(0)
        self._ck(_lib().gm_get_search_stats(self._h, C.byref(a), C.byref(b)), "gm_get_search_stats")
        return int(a.value), int(b.value)

    def voxel_bbox(self):
        a, b = np.empty(3, np.float32), np.empty(3, np.float32)
        self._ck(_lib().gm_get_voxel_bbox(self._h, _ptr(a), _ptr(b)), "gm_get_voxel_bbox")
        return a, b

    def set_voxel_bbox(self, mn=None, mx=None):
        """Override pcl::getMinMax3D before voxel() (global lattice of a multi-slab map); None clears."""
        if mn is None:
            self._ck(_lib().gm_set_voxel_bbox(self._h, None, None), "gm_set_voxel_bbox")
        else:
            a, b = np.ascontiguousarray(mn, np.float32), np.ascontiguousarray(mx, np.float32)
            self._ck(_lib().gm_set_voxel_bbox(self._h, _ptr(a), _ptr(b)), "gm_set_voxel_bbox")

    def synchronize(self):
        self._ck(_lib().gm_synchronize(self._h), "gm_synchronize")

    @property
    def launch_count(self) -> int:
        return int(_lib().gm_launch_count(self._h))

    def reset_launch_count(self):
        _lib().gm_reset_launch_count(self._h)

    # -- input ------------------------------------------------------------------------------
    def upload_scan(self, points: np.ndarray):
        a = _as_xyzw(points)
        self._keepalive = a
        self._ck(_lib().gm_upload_scan(self._h, _ptr(a), a.shape[0], 16), "gm_upload_scan")

    def upload_scan_raw(self, host_ptr: int, n: int, stride: int = 16):
        self._ck(_lib().gm_upload_scan(self._h, C.c_void_p(host_ptr), n, stride), "gm_upload_scan")

    def upload_pointcloud2(self, data: np.ndarray, n: int, point_step: int, offset_x: int, offset_y: int, offset_z: int):
        """data: contiguous uint8 payload of a sensor_msgs/PointCloud2 (n * point_step bytes)."""
        raw = np.ascontiguousarray(data, dtype=np.uint8)
        self._keepalive = raw
        self._ck(_lib().gm_upload_pointcloud2(self._h, _ptr(raw), n, point_step, offset_x, offset_y, offset_z), "gm_upload_pointcloud2")

    def upload_pointcloud2_raw(self, host_ptr: int, n: int, point_step: int, offset_x: int, offset_y: int, offset_z: int):
        """Same from a raw host address (e.g. a pinned torch tensor); the caller keeps the buffer alive."""
        self._ck(_lib().gm_upload_pointcloud2(self._h, C.c_void_p(host_ptr), n, point_step, offset_x, offset_y, offset_z), "gm_upload_pointcloud2")

    def upload_pointcloud2_timed(self, data: np.ndarray, n: int, point_step: int, offset_x: int, offset_y: int, offset_z: int,
                                 offset_t: int):
        """upload_pointcloud2 plus the float32 per-point time (seconds) at byte offset offset_t, e.g. PointXYZIRT::time."""
        raw = np.ascontiguousarray(data, dtype=np.uint8)
        self._keepalive = raw
        self._ck(_lib().gm_upload_pointcloud2_timed(self._h, _ptr(raw), n, point_step, offset_x, offset_y, offset_z, offset_t),
                 "gm_upload_pointcloud2_timed")

    def point_times(self) -> np.ndarray:
        """The n decoded times of the timed scan (float32)."""
        out = np.empty(max(self.counts().n_input, 0), np.float32)
        self._ck(_lib().gm_download_point_times(self._h, _ptr(out), out.shape[0]), "gm_download_point_times")
        return out

    def deskew(self, delta34, t_ref: float, period: float):
        """Express every point of the timed scan in the sensor frame at t_ref, the sensor moving by delta34 (3x4 or 4x4, the
        previous scan's frame to this one's) over `period` seconds (include/gm_capi.h, gm_deskew).  Before crop()."""
        d = np.ascontiguousarray(np.asarray(delta34, np.float32)[:3, :4].reshape(12))
        self._ck(_lib().gm_deskew(self._h, _ptr(d), C.c_double(t_ref), C.c_double(period)), "gm_deskew")

    def set_scan_device(self, device_ptr: int, n: int):
        self._ck(_lib().gm_set_scan_device(self._h, C.c_void_p(device_ptr), n), "gm_set_scan_device")

    # -- stages -----------------------------------------------------------------------------
    def crop(self):
        self._ck(_lib().gm_crop(self._h), "gm_crop")

    def normals(self):
        self._ck(_lib().gm_normals(self._h), "gm_normals")

    def voxel(self):
        self._ck(_lib().gm_voxel(self._h), "gm_voxel")

    def local_frame(self):
        self._ck(_lib().gm_local_frame(self._h), "gm_local_frame")

    def ransac(self, kind: int, samples: np.ndarray, h_begin: int = 0, h_end: int | None = None):
        s = np.ascontiguousarray(samples, dtype=np.int32)
        H = s.shape[0]
        self._ck(_lib().gm_ransac(self._h, kind, _ptr(s), H, h_begin, H if h_end is None else h_end), "gm_ransac")

    def ransac_key_device_ptr(self, kind: int) -> int:
        p = C.c_void_p()
        self._ck(_lib().gm_ransac_key_device_ptr(self._h, kind, C.byref(p)), "gm_ransac_key_device_ptr")
        return int(p.value)

    def ransac_export_key(self, kind: int, dst_device_ptr: int):
        self._ck(_lib().gm_ransac_export_key(self._h, kind, C.c_void_p(dst_device_ptr)), "gm_ransac_export_key")

    def ransac_import_key(self, kind: int, src_device_ptr: int):
        self._ck(_lib().gm_ransac_import_key(self._h, kind, C.c_void_p(src_device_ptr)), "gm_ransac_import_key")

    def ransac_pair(self, plane_samples, cyl_samples, p_range=None, c_range=None):
        """gm_ransac for both primitives side by side; ranges = (begin, end) hypothesis shards (default: all)."""
        ps = np.ascontiguousarray(plane_samples, dtype=np.int32)
        cs = np.ascontiguousarray(cyl_samples, dtype=np.int32)
        pb, pe = p_range if p_range is not None else (0, ps.shape[0])
        cb, ce = c_range if c_range is not None else (0, cs.shape[0])
        self._ck(_lib().gm_ransac_pair(self._h, _ptr(ps), ps.shape[0], pb, pe, _ptr(cs), cs.shape[0], cb, ce), "gm_ransac_pair")

    def ransac_select_pair(self):
        self._ck(_lib().gm_ransac_select_pair(self._h), "gm_ransac_select_pair")

    def ransac_export_keys(self, dst_device_ptr: int):
        self._ck(_lib().gm_ransac_export_keys(self._h, C.c_void_p(dst_device_ptr)), "gm_ransac_export_keys")

    def ransac_import_keys(self, src_device_ptr: int):
        self._ck(_lib().gm_ransac_import_keys(self._h, C.c_void_p(src_device_ptr)), "gm_ransac_import_keys")

    def ransac_select(self, kind: int):
        self._ck(_lib().gm_ransac_select(self._h, kind), "gm_ransac_select")

    def label(self):
        self._ck(_lib().gm_label(self._h), "gm_label")

    def axis_polyline(self):
        self._ck(_lib().gm_axis_polyline(self._h), "gm_axis_polyline")

    def process_scan(self, plane_samples: np.ndarray | None, cyl_samples: np.ndarray | None):
        ps = None if plane_samples is None else np.ascontiguousarray(plane_samples, dtype=np.int32)
        cs = None if cyl_samples is None else np.ascontiguousarray(cyl_samples, dtype=np.int32)
        self._ck(_lib().gm_process_scan(self._h, _ptr(ps), 0 if ps is None else ps.shape[0], _ptr(cs),
                                        0 if cs is None else cs.shape[0]), "gm_process_scan")

    def inject_compacted(self, points: np.ndarray, normals8: np.ndarray | None = None):
        a = _as_xyzw(points)
        nr = None if normals8 is None else np.ascontiguousarray(normals8, dtype=np.float32)
        if nr is not None and nr.shape != (a.shape[0], 8):
            raise ValueError("normals8 must be n x 8")
        self._ck(_lib().gm_inject_compacted(self._h, _ptr(a), _ptr(nr), a.shape[0]), "gm_inject_compacted")

    # -- results ----------------------------------------------------------------------------
    def counts(self) -> gm_counts:
        c = gm_counts()
        self._ck(_lib().gm_get_counts(self._h, C.byref(c)), "gm_get_counts")
        return c

    def download_cloud(self, which: int = 1) -> np.ndarray:
        c = self.counts()
        n = c.n_cropped if which == 0 else c.n_valid
        out = np.empty((max(n, 0), 4), np.float32)
        self._ck(_lib().gm_download_cloud(self._h, which, _ptr(out), out.shape[0]), "gm_download_cloud")
        return out

    def download_normals(self, which: int = 1) -> np.ndarray:
        c = self.counts()
        n = c.n_cropped if which == 0 else c.n_valid
        out = np.empty((max(n, 0), 8), np.float32)
        self._ck(_lib().gm_download_normals(self._h, which, _ptr(out), out.shape[0]), "gm_download_normals")
        return out

    def download_neighbor_counts(self) -> np.ndarray:
        out = np.empty(max(self.counts().n_cropped, 0), np.int32)
        self._ck(_lib().gm_download_neighbor_counts(self._h, _ptr(out), out.shape[0]), "gm_download_neighbor_counts")
        return out

    def download_valid_map(self) -> np.ndarray:
        out = np.empty(max(self.counts().n_cropped, 0), np.int32)
        self._ck(_lib().gm_download_valid_map(self._h, _ptr(out), out.shape[0]), "gm_download_valid_map")
        return out

    def download_voxel_assignment(self):
        n = max(self.counts().n_valid, 0)
        keys, assign = np.empty(n, np.int32), np.empty(n, np.int32)
        st = self._ck(_lib().gm_download_voxel_assignment(self._h, _ptr(keys), _ptr(assign), n),
                      "gm_download_voxel_assignment", ok=(GM_OK, GM_WARN_VOXEL_OVERFLOW))
        return keys, assign, st

    def download_voxels(self, with_nn: bool = True):
        V = max(self.counts().n_voxels, 0)
        cen = np.empty((V, 4), np.float32)
        keys, cnt = np.empty(V, np.int32), np.empty(V, np.int32)
        nn = np.empty(V, np.int32) if with_nn else None
        nnn = np.empty((V, 8), np.float32) if with_nn else None
        st = self._ck(_lib().gm_download_voxels(self._h, _ptr(cen), _ptr(keys), _ptr(cnt), _ptr(nn), _ptr(nnn), V),
                      "gm_download_voxels", ok=(GM_OK, GM_WARN_VOXEL_OVERFLOW, GM_ERR_NN_INDEX_RANGE))
        return {"centroids": cen, "keys": keys, "counts": cnt, "nn_index": nn, "nn_normal": nnn, "status": st}

    def voxel_grid(self) -> np.ndarray:
        g = (C.c_int32 * 6)()
        self._ck(_lib().gm_get_voxel_grid(self._h, C.byref(g)), "gm_get_voxel_grid")
        return np.array(list(g), np.int32)

    def frame(self):
        f = gm_frame()
        self._ck(_lib().gm_get_frame(self._h, C.byref(f)), "gm_get_frame")
        return {"vals": np.array(f.vals, np.float32), "vecs": np.array(f.vecs, np.float32).reshape(3, 3),
                "scatter": np.array(f.scatter, np.float32).reshape(3, 3), "_struct": f}

    def download_hypotheses(self, kind: int, H: int):
        coef = np.empty((H, 4 if kind == GM_MODEL_PLANE else 7), np.float32)
        test = np.empty((H, 12), np.float32) if kind == GM_MODEL_CYLINDER else None
        counts = np.empty(H, np.int32)
        self._ck(_lib().gm_download_hypotheses(self._h, kind, _ptr(coef), _ptr(test), _ptr(counts), H), "gm_download_hypotheses")
        return coef, test, counts

    def model(self, kind: int):
        m = gm_model()
        st = self._ck(_lib().gm_get_model(self._h, kind, C.byref(m)), "gm_get_model", ok=(GM_OK, GM_ERR_NO_MODEL))
        k = 4 if kind == GM_MODEL_PLANE else 7
        return {"kind": m.kind, "best_id": m.best_id, "best_count": m.best_count, "refit_count": m.refit_count,
                "hyp": np.array(m.hyp[:k], np.float32), "coef": np.array(m.coef[:k], np.float32), "rms": float(m.rms),
                "status": st}

    def download_labels(self) -> np.ndarray:
        out = np.empty(max(self.counts().n_valid, 0), np.uint8)
        self._ck(_lib().gm_download_labels(self._h, _ptr(out), out.shape[0]), "gm_download_labels")
        return out

    def download_polyline(self) -> np.ndarray:
        cap = int(self.params.maxSlices)
        out = np.zeros(cap, SLICE_DTYPE)
        n = C.c_int32(0)
        self._ck(_lib().gm_download_polyline(self._h, _ptr(out), cap, C.byref(n)), "gm_download_polyline")
        return out[: n.value].copy()


def _ctx_fetch_async(self, outputs: gm_host_outputs):
    self._ck(_lib().gm_fetch_async(self._h, C.byref(outputs)), "gm_fetch_async")


def _ctx_profile_enable(self, on: bool = True):
    self._ck(_lib().gm_profile_enable(self._h, 1 if on else 0), "gm_profile_enable")


def _ctx_profile_read(self) -> dict:
    """{segment: (ms_sum, calls)} since the last read."""
    k = _lib().gm_profile_num_segments()
    ms, calls = np.zeros(k, np.float32), np.zeros(k, np.int32)
    self._ck(_lib().gm_profile_read(self._h, _ptr(ms), _ptr(calls)), "gm_profile_read")
    return {_lib().gm_profile_segment_name(i).decode(): (float(ms[i]), int(calls[i])) for i in range(k)}


def _ctx_compress(self):
    self._ck(_lib().gm_compress(self._h), "gm_compress")


def _ctx_compression(self) -> gm_compression:
    c = gm_compression()
    self._ck(_lib().gm_get_compression(self._h, C.byref(c)), "gm_get_compression")
    return c


def _ctx_download_compressed(self) -> bytes:
    n = C.c_size_t(0)
    self._ck(_lib().gm_download_compressed(self._h, None, 0, C.byref(n)), "gm_download_compressed")
    buf = np.empty(n.value, np.uint8)
    self._ck(_lib().gm_download_compressed(self._h, _ptr(buf), buf.shape[0], C.byref(n)), "gm_download_compressed")
    return buf.tobytes()


def _ctx_extract_primitives(self, plane_draws: np.ndarray | None, cyl_draws: np.ndarray | None, max_primitives: int,
                            min_inliers: int):
    """Sequential multi-primitive extraction (gm_extract_primitives).  plane_draws: max_primitives x Hp x 3 uint32,
    cyl_draws: max_primitives x Hc x 2 uint32 (None = no hypotheses of that kind)."""
    draws = []
    for d, per in ((plane_draws, 3), (cyl_draws, 2)):
        if d is None:
            draws.append((None, 0))
            continue
        a = np.ascontiguousarray(d, dtype=np.uint32)
        if a.ndim != 3 or a.shape[0] != max_primitives or a.shape[2] != per:
            raise ValueError(f"draws must be max_primitives x H x {per}")
        draws.append((a, a.shape[1]))
    (pd, hp), (cd, hc) = draws
    self._ck(_lib().gm_extract_primitives(self._h, int(max_primitives), int(min_inliers), _ptr(pd), hp, _ptr(cd), hc),
             "gm_extract_primitives")


def _ctx_primitives(self) -> list:
    """The extracted primitives in extraction order: dicts of gm_primitive (hyp / coef trimmed to 4 or 7 values)."""
    n = C.c_int32(0)
    self._ck(_lib().gm_get_primitives(self._h, None, 0, C.byref(n)), "gm_get_primitives")
    out = (gm_primitive * max(n.value, 1))()
    self._ck(_lib().gm_get_primitives(self._h, out, n.value, C.byref(n)), "gm_get_primitives")
    res = []
    for p in out[: n.value]:
        m = p.model
        k = 4 if m.kind == GM_MODEL_PLANE else 7
        res.append({"kind": m.kind, "best_id": m.best_id, "best_count": m.best_count, "refit_count": m.refit_count,
                    "hyp": np.array(m.hyp[:k], np.float32), "coef": np.array(m.coef[:k], np.float32), "rms": float(m.rms),
                    "n_remaining": p.n_remaining})
    return res


def _ctx_download_primitive_ids(self) -> np.ndarray:
    out = np.empty(max(self.counts().n_valid, 0), np.uint8)
    self._ck(_lib().gm_download_primitive_ids(self._h, _ptr(out), out.shape[0]), "gm_download_primitive_ids")
    return out


def _ctx_compress_primitives(self):
    self._ck(_lib().gm_compress_primitives(self._h), "gm_compress_primitives")


def _ctx_download_compressed_primitives(self) -> bytes:
    n = C.c_size_t(0)
    self._ck(_lib().gm_download_compressed_primitives(self._h, None, 0, C.byref(n)), "gm_download_compressed_primitives")
    buf = np.empty(n.value, np.uint8)
    self._ck(_lib().gm_download_compressed_primitives(self._h, _ptr(buf), buf.shape[0], C.byref(n)), "gm_download_compressed_primitives")
    return buf.tobytes()


def parse_compressed_primitives(blob: bytes) -> dict:
    """GMP1 blob -> {"header": gm_primitive_compression, "records": PRIMITIVE_RECORD_DTYPE array, "residual": V x 3 float32}."""
    magic, version = np.frombuffer(blob, "<u4", 2)
    if magic != 0x31504D47 or version != 1:
        raise ValueError("not a GMP1 blob")
    hs = C.sizeof(gm_primitive_compression)
    h = gm_primitive_compression.from_buffer_copy(blob[8:8 + hs])
    off = 8 + hs
    rec = np.frombuffer(blob, PRIMITIVE_RECORD_DTYPE, h.n_primitives, off).copy()
    off += h.n_primitives * PRIMITIVE_RECORD_DTYPE.itemsize
    res = np.frombuffer(blob, "<f4", 3 * h.n_residual_voxels, off).reshape(-1, 3).copy()
    if off + res.nbytes != len(blob):
        raise ValueError("GMP1 blob size does not match its header")
    return {"header": h, "records": rec, "residual": res}


def icp_params(init_pose34=None, **overrides) -> gm_icp_params:
    """gm_icp_params with the library defaults, the initial guess (3x4 or 4x4 row-major [R|t], None = identity) and
    any field overridden by keyword."""
    p = gm_icp_params()
    _lib().gm_icp_params_default(C.byref(p))
    if init_pose34 is not None:
        p.init_pose34[:] = [float(v) for v in np.asarray(init_pose34, np.float32)[:3, :4].reshape(12)]
    for k, v in overrides.items():
        if not hasattr(p, k) or k == "pad_":
            raise AttributeError(f"gm_icp_params has no field {k}")
        setattr(p, k, v)
    return p


def _registration_dict(r: gm_registration) -> dict:
    return {"pose": np.array(r.pose34, np.float32).reshape(3, 4), "iterations": r.iterations, "converged": r.converged,
            "n_source": r.n_source, "n_correspondences": r.n_correspondences, "rmse": float(r.rmse), "fitness": float(r.fitness),
            "n_degenerate": r.n_degenerate, "eigenvalues": np.array(r.eigenvalues, np.float64),
            "eigenvectors": np.array(r.eigenvectors, np.float64).reshape(6, 6), "_struct": r}


def _ctx_register_async(self, target: "Context", init_pose34=None, **params):
    """Enqueue gm_register(self = source, target) without waiting; read the result with registration()."""
    p = icp_params(init_pose34, **params)
    self._ck(_lib().gm_register(self._h, target._h, C.byref(p)), "gm_register")


def _ctx_registration(self) -> dict:
    r = gm_registration()
    self._ck(_lib().gm_get_registration(self._h, C.byref(r)), "gm_get_registration")
    return _registration_dict(r)


def _ctx_register(self, target: "Context", init_pose34=None, **params) -> dict:
    """Point-to-plane ICP of this context's voxel centroids (after voxel()) against `target`'s compacted cloud and normals
    (after normals()).  Keywords: the fields of gm_icp_params.  -> {"pose": 3x4 float32 source -> target, "iterations",
    "converged", "n_source", "n_correspondences", "rmse", "fitness", "n_degenerate", "eigenvalues" (6, ascending),
    "eigenvectors" (6x6, column k = eigenvector k over (wx, wy, wz, vx, vy, vz))}."""
    _ctx_register_async(self, target, init_pose34, **params)
    return _ctx_registration(self)


def _ctx_download_correspondences(self):
    """-> (target_index int32 V: compacted target index or -1, residual float32 V: float(r) or NaN) of the last executed
    iteration of the last register()."""
    V = _ctx_registration(self)["n_source"]
    idx, res = np.empty(max(V, 0), np.int32), np.empty(max(V, 0), np.float32)
    self._ck(_lib().gm_download_correspondences(self._h, _ptr(idx), _ptr(res), idx.shape[0]), "gm_download_correspondences")
    return idx, res


def _ctx_register_map_async(self, vmap: "VoxelMap", init_pose34=None, max_planarity: float = 0.1, **params):
    """Enqueue gm_register_map(self = source, vmap) without waiting; read the result with registration()."""
    p = icp_params(init_pose34, **params)
    self._ck(_lib().gm_register_map(self._h, vmap._h, C.byref(p), C.c_double(max_planarity)), "gm_register_map")


def _ctx_register_map(self, vmap: "VoxelMap", init_pose34=None, max_planarity: float = 0.1, **params) -> dict:
    """Point-to-plane ICP of this context's voxel centroids (after voxel()) against the planes of the voxel map `vmap`
    (include/gm_capi.h, gm_register_map): init_pose34 and the result's pose are source -> map frame.  Keywords: the
    fields of gm_icp_params.  -> the dict of register()."""
    _ctx_register_map_async(self, vmap, init_pose34, max_planarity, **params)
    return _ctx_registration(self)


def _ctx_download_map_correspondences(self):
    """-> (ijk int32 V x 3: the matched map voxel's cell or INT32_MIN x 3, residual float32 V: float(r) or NaN) of the
    last executed iteration of the last register_map()."""
    V = _ctx_registration(self)["n_source"]
    ijk, res = np.empty((max(V, 0), 3), np.int32), np.empty(max(V, 0), np.float32)
    self._ck(_lib().gm_download_map_correspondences(self._h, _ptr(ijk), _ptr(res), ijk.shape[0]), "gm_download_map_correspondences")
    return ijk, res


Context.register = _ctx_register
Context.register_map = _ctx_register_map
Context.register_map_async = _ctx_register_map_async
Context.download_map_correspondences = _ctx_download_map_correspondences
Context.register_async = _ctx_register_async
Context.registration = _ctx_registration
Context.download_correspondences = _ctx_download_correspondences
Context.extract_primitives = _ctx_extract_primitives
Context.primitives = _ctx_primitives
Context.download_primitive_ids = _ctx_download_primitive_ids
Context.compress_primitives = _ctx_compress_primitives
Context.download_compressed_primitives = _ctx_download_compressed_primitives
Context.compress = _ctx_compress
Context.compression = _ctx_compression
Context.download_compressed = _ctx_download_compressed
Context.fetch_async = _ctx_fetch_async
Context.profile_enable = _ctx_profile_enable
Context.profile_read = _ctx_profile_read


def markers_eigen(frame_struct: gm_frame) -> np.ndarray:
    out = np.zeros(3, ARROW_DTYPE)
    _lib().gm_markers_eigen(C.byref(frame_struct), _ptr(out))
    return out


def markers_normals(centroids: np.ndarray, nn_normal8: np.ndarray, arrow_mode: int = 0) -> np.ndarray:
    """arrow_mode 0 = the reference's arrows (end point = the normal itself, quirk B.4), 1 = end = centroid + normal."""
    cen = np.ascontiguousarray(centroids, np.float32)
    nn = np.ascontiguousarray(nn_normal8, np.float32)
    out = np.zeros(cen.shape[0], ARROW_DTYPE)
    _lib().gm_markers_normals_mode(_ptr(cen), _ptr(nn), cen.shape[0], arrow_mode, _ptr(out))
    return out


class VoxelMap:
    """Aggregated voxel map across scans (gm_map_*, SURVEY 8f.3): insertion-order independent."""

    def __init__(self, leaf: float = 0.1, capacity_voxels: int = 1 << 20, _handle=None):
        if _handle is not None:
            self._h = _handle
            return
        h = C.c_void_p()
        st = _lib().gm_map_create(C.c_double(leaf), capacity_voxels, C.byref(h))
        if st != GM_OK:
            raise GmError(st, "gm_map_create")
        self._h = h

    @classmethod
    def load(cls, path: str, min_capacity_voxels: int = 0) -> "VoxelMap":
        h = C.c_void_p()
        st = _lib().gm_map_load(path.encode(), min_capacity_voxels, C.byref(h))
        if st != GM_OK:
            raise GmError(st, "gm_map_load")
        return cls(_handle=h)

    def _ck(self, st, where, ok=(GM_OK,)):
        if st not in ok:
            raise GmError(st, where)
        return st

    @property
    def leaf(self) -> float:
        return float(_lib().gm_map_leaf(self._h))

    def insert(self, ctx: "Context", pose34=None, label_filter: int = -1):
        pose = None if pose34 is None else np.ascontiguousarray(np.asarray(pose34, np.float32).reshape(12))
        self._ck(_lib().gm_map_insert(self._h, ctx._h, _ptr(pose) if pose is not None else None, label_filter), "gm_map_insert")

    def stats(self):
        """-> (n_voxels, n_points, n_out_of_range, full) ; full = an insert found the table full"""
        a, b, c = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        st = self._ck(_lib().gm_map_stats(self._h, C.byref(a), C.byref(b), C.byref(c)), "gm_map_stats", ok=(GM_OK, GM_ERR_CAPACITY))
        return int(a.value), int(b.value), int(c.value), st == GM_ERR_CAPACITY

    def download(self):
        n = C.c_size_t(0)
        self._ck(_lib().gm_map_download(self._h, None, None, None, 0, C.byref(n)), "gm_map_download", ok=(GM_OK, GM_ERR_CAPACITY))
        V = int(n.value)
        ijk, cnt, cen = np.empty((V, 3), np.int32), np.empty(V, np.int32), np.empty((V, 4), np.float32)
        self._ck(_lib().gm_map_download(self._h, _ptr(ijk), _ptr(cnt), _ptr(cen), V, C.byref(n)), "gm_map_download", ok=(GM_OK, GM_ERR_CAPACITY))
        return {"ijk": ijk, "counts": cnt, "centroids": cen}

    def planes(self, max_planarity: float = 0.1) -> np.ndarray:
        """V x 4 float32 in download() order: {normal, 1} of each voxel with a plane, {NaN, NaN, NaN, 0} without."""
        n = C.c_size_t(0)
        self._ck(_lib().gm_map_download_planes(self._h, C.c_double(max_planarity), None, 0, C.byref(n)), "gm_map_download_planes")
        out = np.empty((int(n.value), 4), np.float32)
        self._ck(_lib().gm_map_download_planes(self._h, C.c_double(max_planarity), _ptr(out), out.shape[0], C.byref(n)),
                 "gm_map_download_planes")
        return out

    def evict(self, ctx: "Context", center, half_cells: int, archive: "VoxelMap | None" = None):
        """Keep the voxels whose cell is within half_cells (Chebyshev, in cells) of center's cell; move the others into
        `archive` (None = drop them).  Asynchronous on ctx's stream (include/gm_capi.h, gm_map_evict)."""
        c = np.ascontiguousarray(np.asarray(center, np.float32).reshape(3))
        ctx._ck(_lib().gm_map_evict(self._h, ctx._h, archive._h if archive is not None else None, _ptr(c), int(half_cells)),
                "gm_map_evict")

    def merge(self, src: "VoxelMap") -> bool:
        """self += src (gm_map_merge; synchronises the device).  -> full: this map found its table full and dropped voxels."""
        st = self._ck(_lib().gm_map_merge(self._h, src._h), "gm_map_merge", ok=(GM_OK, GM_ERR_CAPACITY))
        return st == GM_ERR_CAPACITY

    def clear(self):
        self._ck(_lib().gm_map_clear(self._h), "gm_map_clear")

    def save(self, path: str):
        self._ck(_lib().gm_map_save(self._h, path.encode()), "gm_map_save")

    def close(self):
        if getattr(self, "_h", None):
            _lib().gm_map_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def odometry_params(init_pose34=None, **overrides) -> gm_odometry_params:
    """gm_odometry_params with the library defaults, the first scan's pose (or its guess) as init_pose34 (3x4 or 4x4, None
    = identity) and any field overridden by keyword: those of gm_odometry_params and of its gm_icp_params."""
    p = gm_odometry_params()
    _lib().gm_odometry_params_default(C.byref(p))
    icp = {k: v for k, v in overrides.items() if k not in ("max_planarity", "min_fitness", "register_first", "max_steps")}
    p.icp = icp_params(init_pose34, **icp)
    for k, v in overrides.items():
        if k not in icp:
            setattr(p, k, v)
    return p


class Odometry:
    """Map odometry on the device (include/gm_capi.h, gm_odometry_*): each step() predicts the scan's pose, registers it to
    `vmap`, gates the result and inserts the scan at the accepted pose, without a host synchronisation.  Keywords: the
    fields of gm_odometry_params and of its gm_icp_params.  Close it before the map."""

    def __init__(self, vmap: VoxelMap, init_pose34=None, **params):
        self.params = odometry_params(init_pose34, **params)
        h = C.c_void_p()
        st = _lib().gm_odometry_create(vmap._h, C.byref(self.params), C.byref(h))
        if st != GM_OK:
            raise GmError(st, "gm_odometry_create")
        self._h = h
        self.map = vmap

    def step(self, ctx: "Context", delta34=None):
        """One step with ctx after voxel(); delta34 (3x4 or 4x4) = the sensor's motion since the previous scan in its
        frame, None = constant velocity."""
        d = None if delta34 is None else np.ascontiguousarray(np.asarray(delta34, np.float32)[:3, :4].reshape(12))
        ctx._ck(_lib().gm_odometry_step(self._h, ctx._h, _ptr(d)), "gm_odometry_step")

    def deskew(self, ctx: "Context", t_ref: float, period: float):
        """Deskew ctx's timed scan, the one the next step() takes, with the trajectory's constant-velocity increment (the
        identity before step 2).  Waits on ctx's stream for the previous step (include/gm_capi.h, gm_odometry_deskew)."""
        ctx._ck(_lib().gm_odometry_deskew(self._h, ctx._h, C.c_double(t_ref), C.c_double(period)), "gm_odometry_deskew")

    def set_window(self, half_cells: int, archive: VoxelMap | None = None):
        """From the next step on, end each step by evicting the map's voxels outside half_cells cells of the step's pose
        into `archive` (None = drop them); 0 = no window (include/gm_capi.h, gm_odometry_set_window)."""
        st = _lib().gm_odometry_set_window(self._h, int(half_cells), archive._h if archive is not None else None)
        if st != GM_OK:
            raise GmError(st, "gm_odometry_set_window")
        self.archive = archive                                   # the archive must outlive the odometry

    @property
    def steps(self) -> int:
        return int(_lib().gm_odometry_steps(self._h))

    def records(self):
        """-> the gm_odometry_record array of every step issued so far (waits for them)."""
        n = C.c_int32(0)
        _lib().gm_odometry_get(self._h, None, 0, C.byref(n))
        recs = (gm_odometry_record * max(n.value, 1))()
        st = _lib().gm_odometry_get(self._h, recs, n.value, C.byref(n))
        if st != GM_OK:
            raise GmError(st, "gm_odometry_get")
        return recs[:n.value]

    def trajectory(self) -> dict:
        """-> numpy arrays over the steps: poses and guesses (k x 3 x 4 float32), accepted, registered, iterations, converged,
        n_source, n_correspondences, n_degenerate (int32), rmse, fitness (float32)."""
        recs = self.records()
        out = {"poses": np.array([r.pose34[:] for r in recs], np.float32).reshape(-1, 3, 4),
               "guesses": np.array([r.guess34[:] for r in recs], np.float32).reshape(-1, 3, 4)}
        for f in ("accepted", "registered", "iterations", "converged", "n_source", "n_correspondences", "n_degenerate"):
            out[f] = np.array([getattr(r, f) for r in recs], np.int32)
        for f in ("rmse", "fitness"):
            out[f] = np.array([getattr(r, f) for r in recs], np.float32)
        return out

    def close(self):
        if getattr(self, "_h", None):
            _lib().gm_odometry_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PeerComm:
    """Mailbox of one rank for the peer-memory collectives (include/gm_capi.h: gm_comm_*).  world = 1 needs no peers;
    otherwise exchange `handle()` (64 bytes) between the ranks and call `connect(all_handles)` (world x 64 bytes)."""

    def __init__(self, rank: int = 0, world: int = 1):
        h = C.c_void_p()
        st = _lib().gm_comm_create(rank, world, C.byref(h))
        if st != GM_OK:
            raise GmError(st, "gm_comm_create")
        self._h, self.rank, self.world = h, rank, world

    def handle(self) -> bytes:
        buf = (C.c_ubyte * 64)()
        st = _lib().gm_comm_handle(self._h, buf)
        if st != GM_OK:
            raise GmError(st, "gm_comm_handle", _lib().gm_comm_last_error(self._h).decode())
        return bytes(buf)

    def connect(self, handles: bytes):
        if len(handles) != 64 * self.world:
            raise ValueError("handles must be world x 64 bytes")
        buf = (C.c_ubyte * len(handles)).from_buffer_copy(handles)
        st = _lib().gm_comm_connect(self._h, buf)
        if st != GM_OK:
            raise GmError(st, "gm_comm_connect", _lib().gm_comm_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            _lib().gm_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def encode_pointcloud2(xyzw: np.ndarray, frame_id: str = "/velodyne", seq: int = 0, stamp_ns: int = 0, is_dense: bool = True) -> bytes:
    """sensor_msgs/PointCloud2 (ROS 1 wire format) of an n x 4 float32 cloud, as pcl::toROSMsg lays it out."""
    a = _as_xyzw(xyzw)
    f = frame_id.encode()
    buf = (C.c_ubyte * _lib().gm_pointcloud2_size(a.shape[0], f))()
    n = C.c_size_t(0)
    st = _lib().gm_encode_pointcloud2(_ptr(a), a.shape[0], f, seq, stamp_ns, 1 if is_dense else 0, buf, len(buf), C.byref(n))
    if st != GM_OK:
        raise GmError(st, "gm_encode_pointcloud2")
    return bytes(buf[: n.value])


def encode_marker_array(arrows: np.ndarray, ns: str, frame_id: str = "/velodyne", stamp_ns: int = 0) -> bytes:
    """visualization_msgs/MarkerArray (ROS 1 wire format) of ARROW_DTYPE arrows (markers_eigen / markers_normals)."""
    a = np.ascontiguousarray(arrows, ARROW_DTYPE)
    f, s_ = frame_id.encode(), ns.encode()
    buf = (C.c_ubyte * _lib().gm_marker_array_size(len(a), f, s_))()
    n = C.c_size_t(0)
    st = _lib().gm_encode_marker_array(_ptr(a), len(a), f, s_, stamp_ns, buf, len(buf), C.byref(n))
    if st != GM_OK:
        raise GmError(st, "gm_encode_marker_array")
    return bytes(buf[: n.value])


class PrimitiveStore:
    """Append-only on-disk store of per-scan compressed primitives (include/gm_capi.h: gm_store_*)."""

    def __init__(self, path: str, create: bool = True):
        h = C.c_void_p()
        st = _lib().gm_store_open(path.encode(), 1 if create else 0, C.byref(h))
        if st != GM_OK:
            raise GmError(st, "gm_store_open")
        self._h = h

    def append(self, ctx: "Context", scan_id: int, stamp_ns: int = 0, pose34=None):
        pose = None if pose34 is None else np.ascontiguousarray(np.asarray(pose34, np.float32).reshape(12))
        st = _lib().gm_store_append(self._h, ctx._h, scan_id, stamp_ns, _ptr(pose))
        if st != GM_OK:
            raise GmError(st, "gm_store_append")

    def append_blob(self, blob: bytes, scan_id: int, stamp_ns: int = 0, pose34=None):
        pose = None if pose34 is None else np.ascontiguousarray(np.asarray(pose34, np.float32).reshape(12))
        buf = (C.c_ubyte * max(len(blob), 1)).from_buffer_copy(blob if blob else b"\0")
        st = _lib().gm_store_append_blob(self._h, scan_id, stamp_ns, _ptr(pose), buf, len(blob))
        if st != GM_OK:
            raise GmError(st, "gm_store_append_blob")

    def __len__(self):
        return int(_lib().gm_store_count(self._h))

    def info(self, i: int):
        a, b, n = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        pose = np.zeros(12, np.float32)
        st = _lib().gm_store_info(self._h, i, C.byref(a), C.byref(b), _ptr(pose), C.byref(n))
        if st != GM_OK:
            raise GmError(st, "gm_store_info")
        return {"scan_id": int(a.value), "stamp_ns": int(b.value), "pose": pose.reshape(3, 4), "bytes": int(n.value)}

    def read(self, i: int) -> bytes:
        n = C.c_size_t(0)
        st = _lib().gm_store_read(self._h, i, None, 0, C.byref(n))
        if st != GM_OK:
            raise GmError(st, "gm_store_read")
        buf = (C.c_ubyte * max(n.value, 1))()
        st = _lib().gm_store_read(self._h, i, buf, n.value, C.byref(n))
        if st != GM_OK:
            raise GmError(st, "gm_store_read")
        return bytes(buf[: n.value])

    def close(self):
        if getattr(self, "_h", None):
            _lib().gm_store_close(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
