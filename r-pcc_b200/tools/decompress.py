"""python -m rpcc_b200.tools.decompress --input X.rpcc --output X.bin --lidar Velodyne64E
Mirror of the reference's tools/decompress.py:45-150.  --intensity_accuracy A reads the intensity section too and writes
the decoded intensities as the fourth column (the file must have the section)."""
import os

import numpy as np

from .. import _lib
from .._lib import check, ptr
from ..compress_utils import BasicCompressor, decompress_point_cloud, read_compressed_bitstream
from ..dataset import build_dataset
from ..evaluate_metrics import calc_chamfer_distance
from ..segment_utils import PointCloudSegment
from .common import base_parser, intensity_accuracy, resolve
from .compress import quantizer


def decompress(args):
    cfg, accuracy, segment_cfg, model_cfg, uniform, method = resolve(args)
    basic_compressor = BasicCompressor(method_name=method)
    dataset = build_dataset(lidar_type=args.lidar)
    model_num = segment_cfg["cluster_num"] + 1
    H, W = dataset.transform_map.shape[:2]
    inten = intensity_accuracy(args, cfg)
    compressed_data = read_compressed_bitstream(args.input, uniform=uniform, intensity=inten is not None)
    q = None
    if inten is not None:
        q = np.frombuffer(basic_compressor.decompress(compressed_data.pop("intensity")), np.uint8)
    residual_quantized, seg_idx, salience_level, plane_param = decompress_point_cloud(compressed_data, basic_compressor,
                                                                                      model_num, H, W)
    QM = quantizer(cfg, accuracy, uniform)
    residual = QM.dequantize_residual(residual_quantized, seg_idx, salience_level)
    pc_seg = PointCloudSegment(dataset.transform_map)
    range_image_rec = pc_seg.intra_predict(seg_idx, plane_param) + residual
    point_cloud_rec = dataset.PCTransformer.range_image_to_point_cloud(range_image_rec)
    intensity = None
    if q is not None:
        intensity = np.empty((H, W), np.float32)
        seg = np.ascontiguousarray(seg_idx, np.int32)
        check(_lib.lib().rpcc_op_intensity_unpack(ptr(q), q.size, ptr(seg), H, W, 2 * inten, ptr(intensity)))
    dataset.save_point_cloud_to_file(args.output, point_cloud_rec, intensity=intensity)
    print("\nDecompression finished.")
    print(args.output.split(".")[-1], "file save in ", args.output)
    result = {}
    if args.eval:
        assert args.original_point_cloud is not None, \
            "If want to evaluate the reconstruction quality, must set the original point cloud file path first."
        point_cloud, range_image, _ = dataset.load_range_image_points_from_file(args.original_point_cloud)
        n_points = np.where(range_image != 0)[0].shape[0]
        range_dif = np.abs(range_image_rec - range_image)
        chamfer = calc_chamfer_distance(point_cloud, point_cloud_rec, out=False)
        bits = os.path.getsize(args.input) * 8
        print("\nCompared with ", args.original_point_cloud)
        print("    BPP: ", bits / n_points)
        print("    Compression Ratio: ", (n_points * 32 * 3) / bits)
        print("    Depth Error (mean): ", np.mean(range_dif))
        print("    Depth Error (max): ", np.max(range_dif))
        print("    Chamfer Distance (mean): ", chamfer["mean"])
        print("    F1 score (threshold=0.02): ", chamfer["f_score"])
        result.update(max_depth_error=float(np.max(range_dif)), chamfer_mean=chamfer["mean"])
    return result


def main(argv=None):
    p = base_parser(single=True)
    p.add_argument("--original_point_cloud", default=None)
    args = p.parse_args(argv)
    return decompress(args)


if __name__ == "__main__":
    main()
