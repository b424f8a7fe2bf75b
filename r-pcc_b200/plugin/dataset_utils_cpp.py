"""dataset_utils_cpp (cpp_modules.cpp:631-636)."""
from ._np import np, _lib, check, ptr, f32


def point_cloud_to_range_image_even(point_cloud, H, W, horizontal_FOV, vertical_max, vertical_min):
    """(N,3) f32 -> (H,W) f32, cpp_modules.cpp:427-467.  (N,4) KITTI rows are accepted as well."""
    pc = f32(point_cloud)
    if pc.ndim != 2 or pc.shape[1] not in (3, 4):
        raise ValueError("point_cloud must be (N,3) or (N,4)")
    out = np.empty((H, W), np.float32)
    check(_lib.lib().rpcc_op_point_cloud_to_range_image_even(
        ptr(pc), pc.shape[0], pc.shape[1], int(H), int(W), horizontal_FOV, vertical_max, vertical_min, ptr(out)))
    return out
