"""TEST INFRASTRUCTURE: the reference's torch lines, run by torch itself on the GPU box.

/root/reference cannot travel to the GPU box, and its segment() needs CUDA, so the dozen torch
statements of PointCloudSegment.segment's GPU branch (utils/segment_utils.py:133-148,168-169 and
the helpers at :18-27,38-52,54-72) are restated here verbatim in torch; the arithmetic is torch's
own.  FPS inside it is the reference's own compiled kernel (oracle/_ref/libref_fps.so) when
present, else the oracle's C restatement.
"""
import numpy as np
import torch

import oracle
from oracle import ref


def ref_fps_gpu(points, m):
    """points (B,n,3) cuda f32 -> (B,m) int32, via the reference kernel (ops/fps/fps_utils.py:25-29)."""
    B, n, _ = points.shape
    temp = torch.full((B, n), 1e10, dtype=torch.float32, device=points.device)
    idx = torch.zeros((B, m), dtype=torch.int32, device=points.device)
    torch.cuda.synchronize()
    rc = ref.fps().ref_fps_launch(B, n, m, points.data_ptr(), temp.data_ptr(), idx.data_ptr())
    assert rc == 0
    return idx


def torch_segment(range_image, lut, ground_model, cluster_num=100, thr=0.1, fps="ref"):
    """range_image (H,W) f32 np, lut (H,W,3) f32 np, ground_model (4,) f64 -> seg_idx (H,W) int64 np,
    center_idx (M,) int32 np, nonground_points (HW,3) f32 np."""
    H, W = lut.shape[:2]
    point_cloud = torch.from_numpy((range_image.reshape(H, W, 1) * lut)).float().cuda()  # numpy f32 mul, as dataset.py
    gm = torch.from_numpy(np.asarray(ground_model)).float().cuda()
    # calc_plane_residual_vertical
    pp = gm.unsqueeze(0).unsqueeze(0)
    depth_dif = torch.abs(torch.sum(point_cloud * pp[..., :3], -1) + pp[..., 3]) / torch.norm(pp[..., :3], 2, -1)
    nonground_mask = depth_dif > thr
    nonground_points = (point_cloud * nonground_mask.unsqueeze(-1)).view(-1, 3)
    if fps == "ref" and ref.have_cuda():
        center_idx = ref_fps_gpu(nonground_points.unsqueeze(0).contiguous(), cluster_num)
    else:
        center_idx = torch.from_numpy(oracle.fps(nonground_points.cpu().numpy(), cluster_num)).cuda().unsqueeze(0)
    cluster_centers = nonground_points[center_idx[0].long()]
    seg_idx = torch_labels(range_image, lut, ground_model, cluster_centers)
    return seg_idx, center_idx[0].cpu().numpy(), nonground_points.cpu().numpy()


def torch_labels(range_image, lut, ground_model, centers):
    """The label lines of segment() (utils/segment_utils.py:142-148,168-169) for GIVEN cluster centres:
    range_image (H,W) f32 np, lut (H,W,3) f32 np, ground_model (4,), centers (M,3) f32 np or cuda tensor
    -> seg_idx (H,W) int64 np."""
    H, W = lut.shape[:2]
    range_image_cuda = torch.from_numpy(range_image.reshape(H, W, 1)).float().cuda()
    transform_map = torch.from_numpy(lut).float().cuda()
    point_cloud = torch.from_numpy((range_image.reshape(H, W, 1) * lut)).float().cuda()
    pp = torch.from_numpy(np.asarray(ground_model)).float().cuda().unsqueeze(0).unsqueeze(0)
    cluster_centers = centers if isinstance(centers, torch.Tensor) else torch.from_numpy(np.asarray(centers, np.float32))
    cluster_centers = cluster_centers.float().cuda()
    # calc_plane_residual_depth
    r_plane = -pp[..., 3] / torch.sum(pp[..., :3] * transform_map, -1)
    ground_residual = range_image_cuda[..., 0] - r_plane
    # calc_cluster_residual_radius
    diff = point_cloud.view(H, W, 1, 3) - cluster_centers.unsqueeze(0).unsqueeze(0)
    cluster_residual_radius = torch.norm(diff, 2, -1)
    distance = torch.cat((ground_residual.unsqueeze(-1), cluster_residual_radius), -1)
    _, seg_idx = torch.max(-distance.abs(), -1)
    seg_idx = seg_idx.cpu().numpy()
    seg_idx[np.where(seg_idx > 0)] += 1
    seg_idx[np.where(range_image.reshape(H, W) == 0)] = 1
    return seg_idx
