"""ctypes binding of liblocreg.so (include/locreg.h).  Fails loudly when the library is missing:
there is no CPU fallback anywhere in this package."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, os.environ.get("LOCREG_SO", "liblocreg.so"))  # LOCREG_SO: experiment builds only

ICP_P2P, ICP_P2LINE, ICP_P2PLANE, NDT_DIRECT, NDT_INCREMENTAL = 0, 1, 2, 3, 4
NEARBY_CENTER, NEARBY6 = 0, 1
LOOP_PERSISTENT, LOOP_GRAPH = 0, 1

# every symbol include/locreg.h declares (tests/test_cabi.py checks the library exports them all)
SYMBOLS = [
    "locreg_default_options", "locreg_create", "locreg_destroy", "locreg_set_stream", "locreg_set_target",
    "locreg_set_target_device", "locreg_align", "locreg_compute_hb", "locreg_knn", "locreg_debug_points",
    "locreg_align_batch", "locreg_align_batch_device", "locreg_relocalise", "locreg_pack_score",
    "locreg_transform_cloud", "locreg_ndt_num_voxels", "locreg_ndt_get_voxels", "locreg_last_timing",
    "locreg_profile", "locreg_last_error", "locreg_version", "locreg_filter_remove_nan", "locreg_filter_crop_box",
    "locreg_filter_voxel_grid", "locreg_set_global_map", "locreg_reset_local_map",
    "locreg_local_map_add_keyframe", "locreg_local_map_get", "locreg_local_map_clear",
    "locreg_comm_unique_id", "locreg_comm_init", "locreg_comm_destroy", "locreg_comm_info", "locreg_shard_range",
    "locreg_relocalise_sharded", "locreg_align_batch_sharded", "locreg_index_info", "locreg_align_loam",
    "locreg_align_loam_batch", "locreg_relocalise_loam", "locreg_relocalise_loam_sharded", "locreg_relocalise_staged",
    "locreg_relocalise_staged_sharded", "locreg_relocalise_loam_staged", "locreg_relocalise_loam_staged_sharded",
]


class Options(C.Structure):
    _fields_ = [("method", C.c_int32), ("max_iteration", C.c_int32), ("min_effective_pts", C.c_int32),
                ("use_ann", C.c_int32), ("eps", C.c_double), ("max_nn_distance", C.c_double),
                ("max_plane_distance", C.c_double), ("max_line_distance", C.c_double), ("voxel_size", C.c_double),
                ("res_outlier_th", C.c_double), ("min_pts_in_voxel", C.c_int32), ("nearby_type", C.c_int32),
                ("knn_cell_size", C.c_double), ("loop_mode", C.c_int32), ("knn_lists", C.c_int32),
                ("ndt_capacity", C.c_int32), ("zero_initial_translation", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("iters", C.c_int32), ("updates", C.c_int32), ("converged", C.c_int32), ("degenerate", C.c_int32),
                ("n_effective", C.c_int64), ("n_inlier", C.c_int64), ("sum_sq_res", C.c_double),
                ("pose_written", C.c_int32), ("pad_", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "pad_"}


_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(_SO):
            raise RuntimeError(f"{_SO} is missing — build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
                               "loc_lib_b200 has no CPU fallback")
        L = C.CDLL(_SO)
        vp, sz, i32, i64 = C.c_void_p, C.c_size_t, C.c_int32, C.c_int64
        L.locreg_default_options.argtypes = [C.POINTER(Options), i32]
        L.locreg_create.argtypes = [C.POINTER(Options), i32, C.POINTER(vp)]
        L.locreg_destroy.argtypes = [vp]
        L.locreg_set_stream.argtypes = [vp, vp]
        L.locreg_set_target.argtypes = [vp, vp, sz, sz]
        L.locreg_set_target_device.argtypes = [vp, vp, sz, sz]
        L.locreg_align.argtypes = [vp, vp, sz, sz, vp, vp, vp, C.POINTER(Result)]
        L.locreg_compute_hb.argtypes = [vp, vp, sz, sz, vp, vp, vp, C.POINTER(Result)]
        L.locreg_align_loam.argtypes = [vp, vp, vp, sz, vp, sz, sz, vp, i32, C.c_double, vp, vp]
        L.locreg_align_loam_batch.argtypes = [vp, vp, vp, vp, vp, vp, sz, vp, sz, i32, C.c_double, vp, vp]
        L.locreg_relocalise_loam.argtypes = [vp, vp, vp, sz, vp, sz, sz, vp, sz, i32, C.c_double, vp, vp, vp, vp, vp]
        L.locreg_relocalise_loam_sharded.argtypes = [vp, vp, vp, sz, vp, sz, sz, vp, sz, i32, C.c_double, vp, vp, vp]
        L.locreg_relocalise_loam_staged.argtypes = [vp, vp, vp, sz, vp, sz, sz, vp, sz, vp, vp, i32, C.c_double, vp, vp, vp,
                                                    vp, vp, vp]
        L.locreg_relocalise_loam_staged_sharded.argtypes = L.locreg_relocalise_loam_staged.argtypes
        L.locreg_knn.argtypes = [vp, vp, sz, sz, i32, vp]
        L.locreg_debug_points.argtypes = [vp, vp, sz, sz, vp, vp, vp]
        L.locreg_align_batch.argtypes = [vp, vp, vp, sz, vp, sz, vp, vp]
        L.locreg_align_batch_device.argtypes = [vp, vp, vp, vp, sz, sz, vp, vp]
        L.locreg_relocalise.argtypes = [vp, vp, sz, sz, vp, sz, vp, vp, vp, vp, vp]
        L.locreg_relocalise_staged.argtypes = [vp, vp, sz, sz, vp, sz, vp, vp, i32, vp, vp, vp, vp, vp, vp]
        L.locreg_relocalise_staged_sharded.argtypes = [vp, vp, sz, sz, vp, sz, vp, vp, i32, vp, vp, vp, vp, vp, vp]
        L.locreg_pack_score.restype = C.c_uint64
        L.locreg_pack_score.argtypes = [C.c_double, C.c_uint32]
        L.locreg_transform_cloud.argtypes = [vp, vp, sz, sz, vp, vp]
        L.locreg_ndt_num_voxels.argtypes = [vp, C.POINTER(sz)]
        L.locreg_ndt_get_voxels.argtypes = [vp, vp, vp, vp, vp]
        L.locreg_last_timing.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i64)]
        L.locreg_index_info.argtypes = [vp, C.POINTER(sz), C.POINTER(sz), C.POINTER(sz)]
        L.locreg_profile.argtypes = [vp, i32, vp, vp]
        L.locreg_set_global_map.argtypes = [vp, vp, sz, sz]
        L.locreg_reset_local_map.argtypes = [vp, vp, vp, C.POINTER(sz)]
        L.locreg_local_map_add_keyframe.argtypes = [vp, vp, sz, sz, vp, i32, C.c_float, C.POINTER(sz)]
        L.locreg_local_map_get.argtypes = [vp, vp, sz, C.POINTER(sz), C.POINTER(sz)]
        L.locreg_local_map_clear.argtypes = [vp]
        L.locreg_filter_remove_nan.argtypes = [vp, vp, sz, sz, vp, C.POINTER(sz)]
        L.locreg_filter_crop_box.argtypes = [vp, vp, sz, sz, vp, vp, vp, C.POINTER(sz)]
        L.locreg_filter_voxel_grid.argtypes = [vp, vp, sz, sz, C.c_float, vp, C.POINTER(sz)]
        L.locreg_comm_unique_id.argtypes = [vp]
        L.locreg_comm_init.argtypes = [vp, vp, i32, i32]
        L.locreg_comm_destroy.argtypes = [vp]
        L.locreg_comm_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
        L.locreg_shard_range.argtypes = [sz, i32, i32, C.POINTER(sz), C.POINTER(sz)]
        L.locreg_relocalise_sharded.argtypes = [vp, vp, sz, sz, vp, sz, vp, vp, vp]
        L.locreg_align_batch_sharded.argtypes = [vp, vp, vp, sz, vp, sz, sz, vp, vp]
        L.locreg_last_error.restype = C.c_char_p
        L.locreg_version.restype = C.c_char_p
        _LIB = L
    return _LIB


class LocregError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise LocregError(f"locreg error {rc}: {lib().locreg_last_error().decode()}")
