"""Codec parameters: the values of the reference's cfgs/compressor.yaml and its loader
(utils/utils.py:18-25).  A plain dict with attribute access stands in for EasyDict."""
import copy

import yaml

# cfgs/compressor.yaml:1-36
DEFAULT_COMPRESSOR_CFG = {
    "compress_framework": "uniform",
    "accuracy": 0.02,
    "level_key_point_num": [30, 10, 3, 0],
    "level_delta_acc": [0, 0.02, 0.04, 0.06],
    "ground_salience_level": 2,
    "feature_region": 3,
    "segments": 8,
    "sharp_num": 4,
    "less_sharp_num": 8,
    "flat_num": 6,
    "segment_method": "FPS",
    "ground_threshold": 0.1,
    "cluster_num": 100,
    "DBSCAN_eps": 1.5,
    # neighbours of a DBSCAN core point, itself included; the reference hard-codes its own value inside its DBSCAN
    # branch, which is not available to check, so this default is this project's choice
    "DBSCAN_min_points": 10,
    "modeling_method": "point",
    "plane_angle_threshold": 75,
    "basic_compressor": "bzip2",
    # this project's intensity section (DESIGN.md §4): maximum error of the decoded intensity, None = no section
    "intensity_accuracy": None,
}


class AttrDict(dict):
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


def load_compressor_cfg(yaml_file=None):
    """utils/utils.py:18-25; with no file, the shipped defaults."""
    if yaml_file is None:
        return AttrDict(copy.deepcopy(DEFAULT_COMPRESSOR_CFG))
    with open(yaml_file, "r") as f:
        cfg = yaml.safe_load(f)
    out = AttrDict(copy.deepcopy(DEFAULT_COMPRESSOR_CFG))
    out.update(cfg or {})
    return out
