"""model_method='plane' of PointCloudSegment.cluster_modeling (reference utils/segment_utils.py:188-216) on the
GPU: per-cluster deterministic RANSAC planes with the reference's grazing-angle validation (csrc/plane.cu).
open3d's segment_plane -- third-party, randomised, absent here -- is not reproduced bit for bit; what the
codec guarantees with these planes is the error bound and the bitstream size (DESIGN.md section 7)."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import check, ptr


def plane_modeling(transform_map, range_image, seg_idx, angle_threshold, seed=0x5EED):
    """-> cluster_models (K-1, 4) float64: rows for labels 1 .. K-1, as the reference returns them."""
    lut = np.ascontiguousarray(transform_map, dtype=np.float32)
    H, W = lut.shape[:2]
    ri = np.ascontiguousarray(range_image, dtype=np.float32).reshape(H, W)
    seg = np.ascontiguousarray(seg_idx, dtype=np.int32).reshape(H, W)
    rows = np.empty((256, 4), np.float32)
    n = C.c_int(0)
    check(_lib.lib().rpcc_op_plane_modeling(ptr(ri), ptr(seg), ptr(lut), H, W, angle_threshold, seed, ptr(rows),
                                            rows.shape[0], C.byref(n)))
    return rows[:n.value].astype(np.float64)
