"""Mirror of the reference's dataset layer for this path: PCTransformer
(dataset/transformer.py:11-101), DatasetTemplate (dataset/dataset.py:7-107) and build_dataset
(dataset/__init__.py:52-69).  Arithmetic runs on the GPU through the plugin ops."""
import struct

import numpy as np
import yaml

from . import _lib
from ._lib import check, ptr
from .lidar import LIDAR_TABLE, LidarConfig
from .plugin import dataset_utils_cpp


class PCTransformer:
    def __init__(self, lidar_cfg=None, channel_distribute_csv=None):
        """lidar_cfg: a lidar name ('Velodyne64E', ...), a LidarConfig, or the path of a yaml file
        with the reference's keys (dataset/lidar_cfg/*.yaml)."""
        if channel_distribute_csv is not None:
            raise NotImplementedError("uneven beam tables are outside this path (every reference lidar entry has csv=None)")
        self.even_dist = True
        if isinstance(lidar_cfg, LidarConfig):
            cfg = lidar_cfg
        elif lidar_cfg in LIDAR_TABLE:
            cfg = LidarConfig(lidar_cfg)
        else:
            with open(lidar_cfg, "r") as f:
                y = yaml.safe_load(f)
            cfg = LidarConfig(None, y["HORIZONTAL_FOV"], y["VERTICAL_ANGLE_MAX"], y["VERTICAL_ANGLE_MIN"],
                              y["RANGE_IMAGE_HEIGHT"], y["RANGE_IMAGE_WIDTH"])
        self.cfg = cfg
        self.horizontal_FOV = cfg.horizontal_FOV
        self.vertical_max = cfg.vertical_max
        self.vertical_min = cfg.vertical_min
        self.vertical_FOV = cfg.vertical_FOV
        self.H, self.W = cfg.H, cfg.W
        self.transform_map = self.create_transform_map()

    def create_transform_map(self):
        return self.cfg.transform_map()

    def point_cloud_to_range_image(self, point_cloud):
        return dataset_utils_cpp.point_cloud_to_range_image_even(np.asarray(point_cloud).astype(np.float32), self.H, self.W,
                                                                 self.horizontal_FOV, self.vertical_max, self.vertical_min)

    def range_image_to_point_cloud(self, range_image):
        ri = np.ascontiguousarray(range_image, dtype=np.float32)
        if ri.ndim not in (2, 3):
            assert False
        xyz = np.empty((self.H, self.W, 3), np.float32)
        check(_lib.lib().rpcc_op_range_to_xyz(ptr(ri), ptr(self.transform_map), self.H, self.W, ptr(xyz)))
        return xyz


class DatasetTemplate:
    def __init__(self, datalist, dataset_cfg, channel_distribute_csv=None, use_radius_outlier_removal=False):
        self.data_list = []
        if datalist is not None:
            for line in open(datalist, "r"):
                if line.strip():
                    self.data_list.append(line.strip())
        if dataset_cfg is not None:
            self.dataset_cfg = dataset_cfg
            self.PCTransformer = PCTransformer(dataset_cfg, channel_distribute_csv)
            self.transform_map = self.PCTransformer.transform_map
        if use_radius_outlier_removal:
            raise NotImplementedError("radius outlier removal needs open3d (outside this path)")

    def __len__(self):
        return len(self.data_list)

    def __getitem__(self, index):
        file_name = self.data_list[index]
        original_point_cloud = self.load_data(file_name)
        range_image = self.PCTransformer.point_cloud_to_range_image(original_point_cloud)
        range_image = np.expand_dims(range_image, -1)
        point_cloud = self.PCTransformer.range_image_to_point_cloud(range_image)
        return point_cloud, range_image, original_point_cloud, file_name

    def load_data(self, file):
        data_type = file.split(".")[-1]
        if data_type == "txt":
            point_cloud = np.loadtxt(file)
        elif data_type == "bin":
            point_cloud = np.fromfile(file, dtype=np.float32).reshape((-1, 4))
        elif data_type in ("npy", "npz"):
            point_cloud = np.load(file)
        else:
            assert False, "File type not correct: " + file  # .ply/.pcd need open3d (outside this path)
        return point_cloud[:, :3]

    def load_range_image_points_from_file(self, file):
        original_point_cloud = self.load_data(file)
        range_image = self.PCTransformer.point_cloud_to_range_image(original_point_cloud)
        range_image = np.expand_dims(range_image, -1)
        point_cloud = self.PCTransformer.range_image_to_point_cloud(range_image)
        return point_cloud, range_image, original_point_cloud

    def save_point_cloud_to_file(self, file, point_cloud, color=None, intensity=None):
        """intensity: (H,W) or (H,W,1) image of the decoded intensities for the fourth column (None: zeros)."""
        data_type = file.split(".")[-1]
        valid_idx = np.where(np.sum(point_cloud, -1) != 0)
        grid = point_cloud.shape[:-1]
        point_cloud = point_cloud[valid_idx]
        if intensity is None:
            fourth = np.zeros((point_cloud.shape[0], 1))
        else:
            fourth = np.asarray(intensity).reshape(grid)[valid_idx][:, None]
        if data_type == "txt":
            np.savetxt(file, np.concatenate((point_cloud, fourth), -1))
        elif data_type == "bin":
            np.concatenate((point_cloud, fourth), -1).astype(np.float32).tofile(file)
        elif data_type in ("npy", "npz"):
            np.save(file, np.concatenate((point_cloud, fourth), -1))
        elif data_type == "ply":
            with open(file, "wb") as fid:
                fid.write(b"ply\nformat binary_little_endian 1.0\n")
                fid.write(bytes("element vertex %d\n" % point_cloud.shape[0], "utf-8"))
                fid.write(b"property float x\nproperty float y\nproperty float z\nend_header\n")
                fid.write(np.ascontiguousarray(point_cloud[:, :3], dtype="<f4").tobytes())
        else:
            assert False, "File type not correct."


__lidar_cfg__ = {k: k for k in ("VelodyneVLP16", "Velodyne32E", "Velodyne64E")}
__dataset_cfg__ = {"KITTI": "Velodyne64E", "KITTI_test": "Velodyne64E_unofficial", "NCLT": "Velodyne32E",
                   "Oxford": "Velodyne32E", "HKUSTCampus": "VelodyneVLP16"}


def build_dataset(datalist=None, dataset_name=None, lidar_type=None, use_radius_outlier_removal=False):
    """dataset/__init__.py:52-69 (the dataset-specific subclasses are offline converters, not on the path)."""
    if dataset_name is not None:
        return DatasetTemplate(datalist, __dataset_cfg__[dataset_name], None, use_radius_outlier_removal)
    if lidar_type is not None:
        return DatasetTemplate(datalist, __lidar_cfg__[lidar_type], None, use_radius_outlier_removal)
    return DatasetTemplate(datalist, dataset_cfg=None, use_radius_outlier_removal=use_radius_outlier_removal)
