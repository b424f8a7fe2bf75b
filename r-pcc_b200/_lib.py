"""ctypes loader for librpcc_b200.so (the C ABI declared in include/rpcc_b200.h).

Every type that crosses the boundary is declared here once: the signature of each entry point (SIGNATURES) and
the mirrors of the header's structures and constants.  tests/test_abi_bindings.py holds them to the header.

There is no CPU fallback anywhere in this package: if the library is missing, or a compute
entry point is called without a CUDA device, the call raises."""
import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RPCC_B200_LIB") or os.path.join(_PKG, "lib", "librpcc_b200.so")  # env: A/B builds
_lib = None


class RpccError(RuntimeError):
    pass


# name -> (restype, argtypes) of every RPCC_API function, in the header's order.  Pointers, handles and
# out-parameters are c_void_p: ptr() returns one for numpy and torch alike, and byref(), ctypes arrays and None
# pass as well.  Scalars take their exact C type, so a missing argument or a float where an int is declared
# raises, and 64-bit sizes and seeds are passed whole.
_v, _s = C.c_void_p, C.c_char_p
_i, _f, _d, _z = C.c_int, C.c_float, C.c_double, C.c_size_t
_i64, _u64, _ll = C.c_int64, C.c_uint64, C.c_longlong
SIGNATURES = {
    "rpcc_last_error": (_s, ()),
    "rpcc_version": (_i, ()),
    "rpcc_launch_count": (_ll, ()),
    "rpcc_device_count": (_i, ()),
    "rpcc_transform_map": (_i, (_i, _i, _d, _d, _d, _v)),
    "rpcc_project_batch": (_i, (_v, _i, _v, _i, _i, _i, _f, _f, _f, _v, _v, _v)),
    "rpcc_intensity_owner_batch": (_i, (_v, _v, _i, _i, _i, _f, _f, _f, _v, _v, _v, _v, _v)),
    "rpcc_range_to_xyz_batch": (_i, (_v, _v, _i, _i, _v, _v)),
    "rpcc_ground_fit_batch": (_i, (_v, _v, _i, _i, _i, _u64, _v, _v, _v)),
    "rpcc_fps_batch": (_i, (_v, _i, _i, _i, _v, _v, _v)),
    "rpcc_segment_fps_batch": (_i, (_v, _v, _v, _i, _i, _i, _i, _f, _v, _v, _v)),
    "rpcc_dbscan_workspace_bytes": (_z, (_i, _i, _i)),
    "rpcc_dbscan_segment_batch": (_i, (_v, _v, _v, _i, _i, _i, _d, _d, _d, _d, _i, _i, _f, _v, _v, _v)),
    "rpcc_book_bytes": (_z, (_i, _i, _i, _i)),
    "rpcc_assign_labels_batch": (_i, (_v, _v, _v, _v, _i, _i, _i, _i, _v, _v, _v)),
    "rpcc_label_stats_batch": (_i, (_v, _v, _i, _i, _i, _i, _v, _v)),
    "rpcc_point_model_batch": (_i, (_v, _v, _v, _v, _i, _i, _i, _i, _v, _v, _v)),
    "rpcc_label_order_batch": (_i, (_v, _v, _i, _i, _i, _i, _v, _z, _v)),
    "rpcc_plane_model_batch": (_i, (_v, _v, _v, _z, _v, _i, _i, _i, _i, _i, _f, _i, _i, _f, _u64, _v, _v, _v)),
    "rpcc_quantize_pack_batch": (_i, (_v, _v, _v, _v, _v, _v, _f, _i, _i, _i, _i, _v, _z, _v, _v, _z, _v, _v, _v)),
    "rpcc_frame_offsets_batch": (_i, (_v, _i, _v, _v, _v)),
    "rpcc_intensity_pack_batch": (_i, (_v, _v, _i, _i, _i, _d, _v, _v, _v, _v)),
    "rpcc_keypoints_salience_batch": (_i, (_v, _v, _v, _i, _i, _i, _i, _i, _i, _i, _i, _i, _v, _v, _i, _i,
                                           _v, _v, _v, _v, _v, _v)),
    "rpcc_decode_batch": (_i, (_v, _v, _z, _v, _v, _z, _v, _v, _v, _v, _i, _i, _i, _i, _v, _v, _v, _v, _v, _v)),
    "rpcc_decode_packed_batch": (_i, (_v, _v, _v, _v, _v, _v, _v, _v, _i, _i, _i, _i, _v, _v, _v, _v, _v, _v)),
    "rpcc_points_workspace_bytes": (_z, (_i, _i, _i)),
    "rpcc_points_out_batch": (_i, (_v, _v, _i, _i, _i, _v, _v, _v, _v)),
    "rpcc_points_out_intensity_batch": (_i, (_v, _v, _v, _i, _i, _i, _v, _v, _v, _v)),
    "rpcc_intensity_unpack_batch": (_i, (_v, _v, _v, _i, _i, _i, _d, _v, _v)),
    "rpcc_dequantize_batch": (_i, (_v, _v, _z, _v, _v, _v, _v, _i, _i, _i, _i, _v, _v, _v, _v, _i, _v)),
    "rpcc_chamfer_batch": (_i, (_v, _i, _v, _i, _v, _v, _v, _v, _v, _v)),
    "rpcc_chamfer_stats": (_i, (_v, _i, _v, _i, _f, _v, _v)),
    "rpcc_eval_workspace_bytes": (_z, (_i, _i, _i)),
    "rpcc_eval_batch": (_i, (_v, _v, _v, _v, _v, _i, _i, _i, _d, _d, _d, _f, _v, _v, _v, _v, _v)),
    "rpcc_eval_steps_batch": (_i, (_v, _i, _i, _d, _v, _v, _v)),
    "rpcc_normals_workspace_bytes": (_z, (_i, _i, _i)),
    "rpcc_normals_batch": (_i, (_v, _v, _i, _i, _i, _d, _d, _d, _i, _f, _v, _v, _v)),
    "rpcc_p2plane_workspace_bytes": (_z, (_i, _i, _i)),
    "rpcc_p2plane_batch": (_i, (_v, _v, _v, _v, _v, _i, _i, _i, _d, _d, _d, _v, _v, _v)),
    "rpcc_op_point_cloud_to_range_image_even": (_i, (_v, _i64, _i, _i, _i, _f, _f, _f, _v)),
    "rpcc_op_point_modeling": (_i, (_v, _v, _i, _i, _v, _i, _v)),
    "rpcc_op_intra_predict": (_i, (_v, _v, _i, _v, _i, _i, _v)),
    "rpcc_op_uniform_quantize": (_i, (_v, _v, _i, _i, _f, _v, _v)),
    "rpcc_op_extract_features_with_segment": (_i, (_v, _v, _i, _i, _i, _i, _i, _i, _i, _v, _v)),
    "rpcc_op_nonuniform_quantize": (_i, (_v, _v, _v, _i, _i, _v, _v, _i, _i, _v, _v, _v, _v)),
    "rpcc_op_extract_contour": (_i, (_v, _i, _i, _v, _v, _v)),
    "rpcc_op_recover_map": (_i, (_v, _v, _i64, _i, _i, _v)),
    "rpcc_op_furthest_point_sample": (_i, (_v, _i, _i, _i, _v)),
    "rpcc_op_segment": (_i, (_v, _v, _v, _i, _i, _i, _f, _v, _v)),
    "rpcc_op_segment_dbscan": (_i, (_v, _v, _v, _i, _i, _d, _d, _d, _d, _i, _i, _f, _v, _v, _v)),
    "rpcc_op_chamfer": (_i, (_v, _i, _v, _i, _v, _v, _v, _v)),
    "rpcc_op_plane_modeling": (_i, (_v, _v, _v, _i, _i, _f, _u64, _v, _i, _v)),
    "rpcc_op_range_to_xyz": (_i, (_v, _v, _i, _i, _v)),
    "rpcc_op_ground_fit": (_i, (_v, _v, _i, _i, _u64, _v)),
    "rpcc_op_dequantize": (_i, (_v, _i64, _v, _i, _i, _v, _i, _v, _v)),
    "rpcc_op_intensity_owner": (_i, (_v, _i64, _i, _i, _f, _f, _f, _v, _v)),
    "rpcc_op_intensity_pack": (_i, (_v, _v, _i, _i, _d, _v, _v, _v)),
    "rpcc_op_intensity_unpack": (_i, (_v, _i64, _v, _i, _i, _d, _v)),
    "rpcc_encoder_create": (_i, (_v, _v)),
    "rpcc_encoder_destroy": (None, (_v,)),
    "rpcc_encoder_slots": (_i, ()),
    "rpcc_encoder_encode_device": (_i, (_v, _i, _v, _i, _v, _i, _v, _v)),
    "rpcc_encoder_encode_host": (_i, (_v, _v, _i, _v, _i, _v, _v, _v, _v, _v, _z, _v, _z, _v, _v, _v)),
    "rpcc_encoder_encode_host_intensity": (_i, (_v, _v, _i, _v, _i, _v, _v, _v, _v, _v, _z, _v, _z, _v, _v, _v, _v)),
    "rpcc_encoder_sync": (_i, (_v,)),
    "rpcc_encoder_profile": (_i, (_v, _i)),
    "rpcc_encoder_stage_times": (_i, (_v, _v, _v, _v)),
    "rpcc_encoder_stream": (_v, (_v, _i)),
    "rpcc_encoder_device_buffer": (_v, (_v, _i, _s)),
    "rpcc_packer_create": (_i, (_i, _s, _v)),
    "rpcc_packer_destroy": (None, (_v,)),
    "rpcc_packer_submit": (_i, (_v, _i, _i, _i, _i, _v, _v, _v, _v, _v, _v, _v, _v, _v, _v, _z, _v)),
    "rpcc_packer_submit_intensity": (_i, (_v, _i, _i, _i, _i, _v, _v, _v, _v, _v, _v, _v, _v, _v, _v, _v, _z, _v)),
    "rpcc_packer_wait": (_i, (_v, _ll)),
    "rpcc_bz2_compress": (_i, (_v, _z, _v, _z, _v)),
    "rpcc_bz2_decompress": (_i, (_v, _z, _v, _z, _v)),
    "rpcc_read_bin_xyz": (_i, (_s, _v, _i64, _v)),
    "rpcc_read_bin_rows": (_i, (_s, _v, _i64, _v)),
    "rpcc_unpack_rpcc": (_i, (_v, _z, _i, _v, _z, _v)),
    "rpcc_unpack_rpcc_intensity": (_i, (_v, _z, _i, _v, _z, _v)),
}


class EncoderConfig(C.Structure):
    """rpcc_encoder_config."""
    _fields_ = [("H", C.c_int), ("W", C.c_int), ("hfov", C.c_double), ("vmax", C.c_double), ("vmin", C.c_double),
                ("cluster_num", C.c_int), ("ground_threshold", C.c_float), ("step", C.c_double),
                ("nonuniform", C.c_int), ("level_num", C.c_int), ("level_kp_num", C.c_int * 8),
                ("level_dacc", C.c_double * 8), ("ground_level", C.c_int), ("feature_region", C.c_int),
                ("segments", C.c_int), ("sharp_num", C.c_int), ("less_sharp_num", C.c_int), ("flat_num", C.c_int),
                ("max_batch", C.c_int), ("max_points", C.c_int64), ("device", C.c_int),
                ("model_method", C.c_int), ("plane_angle_threshold", C.c_float), ("host_chunk", C.c_int),
                ("eval", C.c_int), ("eval_threshold_sq", C.c_float), ("segment_method", C.c_int),
                ("dbscan_eps", C.c_double), ("dbscan_min_points", C.c_int), ("intensity_step", C.c_double)]


# rpcc_frame_result
RESULT_DTYPE = np.dtype([("sym_count", np.uint32), ("seq_count", np.uint32), ("model_rows", np.uint32),
                         ("flags", np.uint32)])
FLAG_INTENSITY_CLAMPED = 8   # rpcc_frame_result.flags bit3

EVAL_COLS = 12   # RPCC_EVAL_COLS
P2PLANE_COLS = 7  # RPCC_P2PLANE_COLS
NORMAL_KNN, NORMAL_RADIUS = 16, 1.0   # RPCC_NORMAL_KNN, RPCC_NORMAL_RADIUS


def build(verbose=False):
    """Compile every CUDA source for sm_100a into lib/librpcc_b200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_PKG, "csrc"), "-j", str(min(16, os.cpu_count() or 4))]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RpccError("building librpcc_b200.so failed:\n" + res.stdout)
    if verbose:
        print(res.stdout)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RpccError("%s not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)" % LIB_PATH)
        dll = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            try:
                fn = getattr(dll, name)
            except AttributeError as e:  # an incomplete build must not go unnoticed
                raise RpccError("librpcc_b200.so does not export %s (stale build?)" % name) from e
            fn.restype, fn.argtypes = restype, argtypes
        _lib = dll
    return _lib


def check(rc):
    if rc != 0:
        raise RpccError("librpcc_b200 error %d: %s" % (rc, lib().rpcc_last_error().decode()))
    return rc


def ptr(a):
    """Address of a numpy array or torch tensor (or None)."""
    if a is None:
        return C.c_void_p(0)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    return a.ctypes.data_as(C.c_void_p)


def launch_count():
    return int(lib().rpcc_launch_count())
