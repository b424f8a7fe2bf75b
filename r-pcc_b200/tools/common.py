"""Argument handling shared by the drivers (reference tools/compress.py:18-85)."""
import argparse

from ..config import load_compressor_cfg


def base_parser(single):
    p = argparse.ArgumentParser()
    if single:
        p.add_argument("--input", help="single frame input.")
        p.add_argument("--output", help="output file.")
    else:
        p.add_argument("--datalist", help="text file, one input path per line.")
        p.add_argument("--output_dir", help="output directory.")
        p.add_argument("--workers", type=int, default=4, help="host entropy-coder threads.")
        p.add_argument("--output", action="store_true", help="print per-frame information.")
        p.add_argument("--batch", type=int, default=256, help="frames per GPU launch.")
    p.add_argument("--lidar", help="lidar type of this point cloud collection.")
    p.add_argument("--compressor_yaml", default=None)
    p.add_argument("--basic_compressor", type=str, default=None)
    p.add_argument("--accuracy", type=float, default=None)
    p.add_argument("--segment_method", type=str, default=None)
    p.add_argument("--cluster_num", type=int, default=None)
    p.add_argument("--DBSCAN_eps", type=float, default=None)
    p.add_argument("--DBSCAN_min_points", type=int, default=None, help="neighbours of a DBSCAN core point, itself included.")
    p.add_argument("--model_method", type=str, default=None)
    p.add_argument("--angle_threshold", type=float, default=None)
    p.add_argument("--nonuniform", action="store_true")
    p.add_argument("--eval", action="store_true")
    p.add_argument("--intensity_accuracy", type=float, default=None,
                   help="carry the intensity column in an extra section, to within this maximum error (default: the "
                        "yaml's intensity_accuracy; unset = no intensity).")
    p.add_argument("--cpu", action="store_true", help="accepted for compatibility; the GPU branch semantics are always used.")
    return p


def resolve(args):
    """-> (cfg, accuracy(step), segment_cfg, model_cfg, uniform, method) as tools/compress.py:44-85."""
    cfg = load_compressor_cfg(args.compressor_yaml)
    accuracy = cfg["accuracy"] * 2
    segment_cfg = {"segment_method": cfg["segment_method"], "ground_vertical_threshold": cfg["ground_threshold"],
                   "cluster_num": cfg["cluster_num"], "DBSCAN_eps": cfg["DBSCAN_eps"],
                   "DBSCAN_min_points": cfg["DBSCAN_min_points"]}
    model_cfg = {"model_method": cfg["modeling_method"], "angle_threshold": cfg["plane_angle_threshold"]}
    method = cfg["basic_compressor"]
    if args.basic_compressor is not None:
        method = args.basic_compressor
    if args.accuracy is not None:
        accuracy = args.accuracy * 2
    if args.segment_method is not None:
        segment_cfg["segment_method"] = args.segment_method
    if args.cluster_num is not None:
        segment_cfg["cluster_num"] = args.cluster_num
    if args.DBSCAN_eps is not None:
        segment_cfg["DBSCAN_eps"] = args.DBSCAN_eps
    if args.DBSCAN_min_points is not None:
        segment_cfg["DBSCAN_min_points"] = args.DBSCAN_min_points
    if segment_cfg["segment_method"] == "DBSCAN" and not (float(segment_cfg["DBSCAN_eps"]) > 0
                                                          and int(segment_cfg["DBSCAN_min_points"]) >= 1):
        raise SystemExit("DBSCAN needs --DBSCAN_eps > 0 and --DBSCAN_min_points >= 1")
    if args.model_method is not None:
        model_cfg["model_method"] = args.model_method
    if args.angle_threshold is not None:
        model_cfg["angle_threshold"] = args.angle_threshold
    uniform = False if args.nonuniform else cfg["compress_framework"] == "uniform"
    if not 1 <= int(segment_cfg["cluster_num"]) <= 252:
        # labels are bytes on the device (0 ground, 1 empty, 2.. clusters; RPCC_MAX_LABELS in include/rpcc_b200.h); the
        # reference's uint16 idx_sequence would allow more
        raise SystemExit("--cluster_num must be in [1, 252] on this path (got %s)" % segment_cfg["cluster_num"])
    return cfg, accuracy, segment_cfg, model_cfg, uniform, method


def intensity_accuracy(args, cfg):
    """--intensity_accuracy, else the yaml's intensity_accuracy; None = no intensity section."""
    a = args.intensity_accuracy if getattr(args, "intensity_accuracy", None) is not None else cfg.get("intensity_accuracy")
    if a is not None and not float(a) > 0:
        raise SystemExit("--intensity_accuracy must be positive (got %s)" % a)
    return None if a is None else float(a)


def warn_clamped(flags, names):
    """The frames whose intensity section had to clamp a value to [0, 255] steps (rpcc_frame_result.flags bit 3)."""
    from .._lib import FLAG_INTENSITY_CLAMPED
    for f, n in zip(flags, names):
        if int(f) & FLAG_INTENSITY_CLAMPED:
            print("WARNING: %s: intensities outside [0, 255 * 2 * intensity_accuracy] were clamped" % n)
