"""Mirror of utils/segment_utils.py:12-233 (PointCloudSegment) for the FPS and DBSCAN + point/plane paths.

segment() always follows the reference's default GPU branch (`cpu=False`,
utils/segment_utils.py:132-148): the `--cpu` branch is a different algorithm (f64, compacted FPS
input, the norm bug of :45-47) and still needs CUDA for FPS, so it is not reproduced.  The ground
plane comes from the device RANSAC (csrc/ground.cu) unless `ground_model` is injected -- open3d,
which the reference calls here, is third-party, randomised and not pinned.  The DBSCAN branch follows this project's
own definition (csrc/dbscan.cu, DESIGN.md §4) in place of open3d's cluster_dbscan."""
import numpy as np

from . import _lib
from ._lib import check, ptr
from .config import DEFAULT_COMPRESSOR_CFG
from .plugin import segment_utils_cpp


class PointCloudSegment:
    def __init__(self, transform_map, plane_num=1):
        self.plane_num = plane_num
        self.transform_map = np.ascontiguousarray(transform_map, dtype=np.float32)
        self.ground_seed = 0x5EED

    def ransac_plane_segmentation(self, range_image, seed=None):
        """Ground plane [a,b,c,d] (f32) of one frame, deterministic (csrc/ground.cu)."""
        H, W = self.transform_map.shape[:2]
        ri = np.ascontiguousarray(range_image, dtype=np.float32).reshape(H, W)
        g = np.empty(4, np.float32)
        check(_lib.lib().rpcc_op_ground_fit(ptr(ri), ptr(self.transform_map), H, W,
                                            self.ground_seed if seed is None else seed, ptr(g)))
        return g

    def segment(self, point_cloud, range_image, segment_cfg, cpu=False, ground_model=None, return_centers=False):
        assert self.transform_map is not None, "Must set transform_map first."
        segment_method = segment_cfg["segment_method"]
        assert segment_method in ["FPS", "DBSCAN"]
        H, W = self.transform_map.shape[:2]
        ri = np.ascontiguousarray(range_image, dtype=np.float32).reshape(H, W)
        if ground_model is None:
            ground_model = self.ransac_plane_segmentation(ri)
        g32 = np.ascontiguousarray(ground_model, dtype=np.float32)  # torch.from_numpy(ground_model).float()
        m = int(segment_cfg["cluster_num"])
        if segment_method == "DBSCAN":
            return self._segment_dbscan(ri, g32, segment_cfg, m), g32
        seg = np.empty((H, W), np.int32)
        cidx = np.empty(m, np.int32)
        check(_lib.lib().rpcc_op_segment(ptr(ri), ptr(self.transform_map), ptr(g32), H, W, m,
                                         segment_cfg["ground_vertical_threshold"], ptr(seg), ptr(cidx)))
        seg = seg.astype(np.int64)  # torch.max indices
        if return_centers:
            return seg, g32, cidx
        return seg, g32

    def _angles(self):
        """(hfov, vmax, vmin) of the ray table: row 0 looks along vmin, the last row along vmax
        (dataset/transformer.py:41-54); the window search of the DBSCAN kernels bounds angles with a margin far above
        the f32 rounding of the table."""
        z = self.transform_map[:, 0, 2].astype(np.float64)
        return 2 * np.pi, float(np.arcsin(z[-1])), float(np.arcsin(z[0]))

    def _segment_dbscan(self, ri, g32, segment_cfg, m):
        H, W = self.transform_map.shape[:2]
        hfov, vmax, vmin = self._angles()
        seg = np.empty((H, W), np.int32)
        check(_lib.lib().rpcc_op_segment_dbscan(ptr(ri), ptr(self.transform_map), ptr(g32), H, W, hfov, vmax, vmin,
                                                float(segment_cfg["DBSCAN_eps"]),
                                                int(segment_cfg.get("DBSCAN_min_points", DEFAULT_COMPRESSOR_CFG["DBSCAN_min_points"])), m,
                                                segment_cfg["ground_vertical_threshold"], ptr(seg), None, None))
        return seg.astype(np.int64)

    def cluster_modeling(self, point_cloud, range_image, seg_idx, model_cfg):
        model_method = model_cfg["model_method"]
        assert model_method in ["point", "plane"]
        if model_method == "point":
            cluster_models = segment_utils_cpp.point_modeling(range_image, seg_idx)
            cluster_models = np.concatenate((np.zeros((cluster_models.shape[0], 3)), np.expand_dims(cluster_models, -1)), -1)
            return cluster_models[1:]
        from .plane_model import plane_modeling
        return plane_modeling(self.transform_map, range_image, seg_idx, model_cfg["angle_threshold"])

    def intra_predict(self, seg_idx, model_param):
        return segment_utils_cpp.intra_predict(seg_idx, model_param, self.transform_map)
