"""ctypes binding of libotslam_b200.so (the C ABI declared in include/otslam_b200.h).

There is no CPU fallback: if the CUDA library is missing this module raises at import, and every
compute entry point raises RuntimeError when no B200 is usable.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libotslam_b200.so")

OK, ERR_INVALID, ERR_FORMAT, ERR_CUDA, ERR_NOMEM, ERR_OVERFLOW = 0, -1, -2, -3, -4, -5
MEM_HOST, MEM_DEVICE = 0, 1
COLOR_NONE, COLOR_RGB8 = 0, 1


class SlabSpec(C.Structure):
    _fields_ = [("axis", C.c_int32), ("thickness", C.c_int32), ("n_ranks", C.c_int32), ("rank", C.c_int32),
                ("halo", C.c_int32)]


if not os.path.exists(SO_PATH):
    raise ImportError(
        f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(otslam_b200 has no CPU fallback)")

lib = C.CDLL(SO_PATH)

_vp, _i, _i64, _d, _u64 = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_uint64
_SIGS = {
    "otslam_last_error": (C.c_char_p, []),
    "otslam_version": (_i, []),
    "otslam_launch_count": (_i64, []),
    "otslam_last_op_device_ms": (_d, []),
    "otslam_trim_scratch": (_i, []),
    "otslam_host_alloc": (_i, [_u64, C.POINTER(_vp)]),
    "otslam_host_free": (_i, [_vp]),
    "otslam_selftest_division": (_i, [_u64, _u64, C.POINTER(_u64), _i]),
    "otslam_selftest_ordered_sum": (_i, [_i64, _u64, _i, C.POINTER(_u64), _i]),
    "otslam_volume_create": (_i, [_d, _d, _i, _i, C.POINTER(SlabSpec), C.POINTER(_vp)]),
    "otslam_volume_destroy": (_i, [_vp]),
    "otslam_volume_reset": (_i, [_vp]),
    "otslam_volume_set_stream": (_i, [_vp, _vp]),
    "otslam_volume_set_batch": (_i, [_vp, _i]),
    "otslam_volume_set_zsplit": (_i, [_vp, _i]),
    "otslam_volume_profile": (_i, [_vp, _i, _vp, _vp]),
    "otslam_volume_integrate_u16": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _d, _d]),
    "otslam_volume_integrate_f32": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "otslam_volume_integrate_batch": (_i, [_vp, _i, _vp, _vp, _i, _i, _vp, _vp, _d, _d, _i]),
    "otslam_volume_set_objects": (_i, [_vp, _i]),
    "otslam_volume_select_object": (_i, [_vp, _i]),
    "otslam_volume_integrate_batch_objects": (_i, [_vp, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _d, _d, _i]),
    "otslam_volume_num_blocks": (_i, [_vp, C.POINTER(_i64)]),
    "otslam_volume_export_blocks": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "otslam_volume_stats": (_i, [_vp, C.POINTER(_i64), C.POINTER(_u64), C.POINTER(_u64)]),
    "otslam_volume_save": (_i, [_vp, C.c_char_p]),
    "otslam_volume_load": (_i, [_vp, C.c_char_p, C.POINTER(_i64)]),
    "otslam_checkpoint_info": (_i, [C.c_char_p, C.POINTER(_d), C.POINTER(_d), C.POINTER(C.c_int32), C.POINTER(_i64), C.POINTER(_i64)]),
    "otslam_checkpoint_profile": (_i, [_vp]),
    "otslam_volume_halo_export":(_i, [_vp, C.POINTER(_i64), _vp, _vp, _vp]),
    "otslam_volume_halo_import": (_i, [_vp, _i64, _vp, _vp]),
    "otslam_volume_halo_pack": (_i, [_vp, C.POINTER(_i64), _vp]),
    "otslam_volume_halo_fetch": (_i, [_vp, _vp, _vp]),
    "otslam_volume_wait_stream": (_i, [_vp, _vp]),
    "otslam_volume_extract_mesh": (_i, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "otslam_volume_mesh_copy": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "otslam_volume_mesh_sample": (_i, [_vp, _i64, _u64, _vp, _vp, _vp]),
    "otslam_volume_extract_points": (_i, [_vp, C.POINTER(_i64)]),
    "otslam_volume_points_copy": (_i, [_vp, _vp, _vp, _vp]),
    "otslam_volume_points_normals": (_i, [_vp, _vp]),
    "otslam_volume_raycast": (_i, [_vp, _i, _i, _i, _vp, _vp, _d, _d, _vp, _vp, _vp, _vp, C.POINTER(_i64)]),
    "otslam_volume_track": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp, _d, _d, _d, _d, _i, _vp, _vp, _vp, _vp, _vp, _i]),
    "otslam_volume_track_pyramid": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp, _d, _d, _d, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "otslam_depth_convert": (_i, [_vp, _i64, _d, _d, _vp, _i]),
    "otslam_backproject_rgbd": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, C.POINTER(_i64), _i]),
    "otslam_mesh_vertex_normals": (_i, [_vp, _i64, _vp, _i64, _vp, _i]),
    "otslam_mesh_sample_uniform": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _u64, _vp, _vp, _vp, _i]),
    "otslam_cloud_zfilter": (_i, [_vp, _vp, _i64, _d, _vp, _vp, C.POINTER(_i64), _i]),
    "otslam_cloud_voxel_down_sample": (_i, [_vp, _vp, _i64, _d, _vp, _vp, _vp, _vp, C.POINTER(_i64), _i]),
    "otslam_cloud_remove_statistical_outlier": (_i, [_vp, _i64, _i, _d, _vp, C.POINTER(_i64), _vp, _i]),
    "otslam_cloud_nn_distance": (_i, [_vp, _i64, _vp, _i64, _vp, _i]),
    "otslam_cloud_nn_within": (_i, [_vp, _i64, _vp, _i64, _d, _vp, _vp, _i]),
    "otslam_cloud_estimate_normals": (_i, [_vp, _i64, _vp, _d, _i, _vp, _i]),
    "otslam_cloud_icp_point_to_plane": (_i, [_vp, _i64, _vp, _vp, _i64, _d, _vp, _d, _d, _i, _vp, _vp, _vp, _vp, _vp, _i]),
    "otslam_cloud_cluster_dbscan": (_i, [_vp, _i64, _d, _i64, _vp, _vp, _i]),
    "otslam_cloud_segment_plane": (_i, [_vp, _i64, _d, _i, _i, _d, _u64, _vp, _vp, _vp, _vp, _i]),
    "otslam_grid_to_points": (_i, [_vp, _i, _i, _d, _d, _d, _i, _vp, C.POINTER(_i64), _i]),
    "otslam_cloud_transform": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _i]),
    "otslam_cloud_center": (_i, [_vp, _i64, _vp, _i]),
    "otslam_cloud_rotate": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _i]),
    "otslam_grid_smart_paste": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "otslam_cloud_merge_pack": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _i]),
    "otslam_decoder_create": (_i, [_i, _i, _i, _i, C.POINTER(_vp)]),
    "otslam_decoder_destroy": (_i, [_vp]),
    "otslam_decoder_decode_files": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "otslam_decoder_decode": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "otslam_decoder_put": (_i, [_vp, _i, _vp, _vp]),
    "otslam_decoder_fetch": (_i, [_vp, _i, _i, _vp, _vp]),
    "otslam_decoder_integrate": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _d, _d, _vp]),
    "otslam_decoder_profile": (_i, [_vp, _vp]),
    "otslam_read_pose_files": (_i, [_i, _vp, _vp, _vp]),
}
EXPORTS = tuple(_SIGS)
MISSING = []                        # tests assert this is empty: the .so must export the whole header
for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name, None)
    if _fn is None:
        MISSING.append(_name)
        continue
    _fn.restype = _res
    _fn.argtypes = _args


def last_error():
    return lib.otslam_last_error().decode(errors="replace")


def check(status):
    """Turn a C status into the exception the reference's `except Exception` paths expect
    (Open3D LogError -> RuntimeError; /root/reference/3d_model/reconstruct_rgbd_filter.py:108-109)."""
    if status != OK:
        if status == ERR_NOMEM:
            raise MemoryError(last_error())
        raise RuntimeError(last_error())


def ptr(a):
    """Raw address of a numpy array / torch tensor / None / int."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))


def launch_count():
    return int(lib.otslam_launch_count())


def last_op_device_ms():
    return float(lib.otslam_last_op_device_ms())


def pinned_empty(shape, dtype):
    """NumPy array over page-locked host memory (freed with the array); ordinary pageable memory when no CUDA
    device is usable (only the copy speed differs)."""
    import weakref
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) * dt.itemsize
    p = C.c_void_p()
    if lib.otslam_host_alloc(n, C.byref(p)) != OK or not p.value:
        return np.empty(shape, dt)
    buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)
    weakref.finalize(buf, lib.otslam_host_free, C.c_void_p(p.value))
    return arr
