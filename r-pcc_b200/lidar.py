"""LiDAR tables (reference dataset/lidar_cfg/*.yaml, dataset/__init__.py:39-43) and the ray LUT
(dataset/transformer.py:26-54)."""
import math

import numpy as np

from . import _lib

# name -> (HORIZONTAL_FOV, VERTICAL_ANGLE_MAX, VERTICAL_ANGLE_MIN, RANGE_IMAGE_HEIGHT, RANGE_IMAGE_WIDTH)
LIDAR_TABLE = {
    "Velodyne64E": (360, 2.0, -24.9, 64, 2000),        # Velodyne_HDL_64E.yaml
    "Velodyne32E": (360, 10.67, -30.67, 32, 2250),     # Velodyne_HDL_32E.yaml
    "VelodyneVLP16": (360, 15.0, -15.0, 16, 1800),     # Velodyne_VLP_16.yaml
    "Velodyne64E_unofficial": (360, 2.5, -23.6, 80, 2000),
}


class LidarConfig:
    """Angles are kept as the Python doubles dataset/transformer.py:32-34 computes
    (deg * (np.pi / 180)); the kernels receive them narrowed to f32 exactly like the pybind
    call narrows them (cpp_modules.cpp:427-428)."""

    def __init__(self, name=None, hfov_deg=None, vmax_deg=None, vmin_deg=None, H=None, W=None):
        if name is not None:
            hfov_deg, vmax_deg, vmin_deg, H, W = LIDAR_TABLE[name]
        self.name = name
        self.H, self.W = int(H), int(W)
        self.horizontal_FOV = hfov_deg * (np.pi / 180)
        self.vertical_max = vmax_deg * (np.pi / 180)
        self.vertical_min = vmin_deg * (np.pi / 180)
        self.vertical_FOV = self.vertical_max - self.vertical_min
        self._lut = None

    @property
    def HW(self):
        return self.H * self.W

    def transform_map(self):
        """(H,W,3) f32 unit ray directions, bit-identical to create_transform_map."""
        if self._lut is None:
            lut = np.empty((self.H, self.W, 3), np.float32)
            _lib.check(_lib.lib().rpcc_transform_map(self.H, self.W, self.horizontal_FOV, self.vertical_max,
                                                     self.vertical_min, _lib.ptr(lut)))
            self._lut = lut
        return self._lut
