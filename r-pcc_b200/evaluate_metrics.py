"""Mirror of utils/evaluate_metrics.py:9-45 (calc_chamfer_distance) on the device chamfer kernels, and point-to-plane
PSNR for range images (calc_point_to_plane_psnr) on the device normals of csrc/normals.cu.  The reference's own PSNR
helper (:48-72, normals from open3d) is not reproduced bit for bit: open3d is absent, parity unpinned (DESIGN.md)."""
import time

import numpy as np
import torch

from . import _lib
from ._lib import NORMAL_KNN, NORMAL_RADIUS, check, ptr


def calc_chamfer_distance(points1, points2, f1_threshold=0.02, out=True):
    t = time.time()
    pc_1 = points1[np.where(np.sum(points1, -1) != 0)]
    pc_2 = points2[np.where(np.sum(points2, -1) != 0)]
    a = torch.from_numpy(np.ascontiguousarray(pc_1, dtype=np.float32)).cuda()
    b = torch.from_numpy(np.ascontiguousarray(pc_2, dtype=np.float32)).cuda()
    n, m = a.shape[0], b.shape[0]
    dist1 = torch.empty(n, dtype=torch.float32, device=a.device)
    dist2 = torch.empty(m, dtype=torch.float32, device=a.device)
    idx1 = torch.empty(n, dtype=torch.int32, device=a.device)
    idx2 = torch.empty(m, dtype=torch.int32, device=a.device)
    scratch = torch.empty(n + m, dtype=torch.int64, device=a.device)
    stats = torch.empty(4, dtype=torch.float64, device=a.device)
    st = torch.cuda.current_stream().cuda_stream
    check(_lib.lib().rpcc_chamfer_batch(ptr(a), n, ptr(b), m, ptr(dist1), ptr(idx1), ptr(dist2), ptr(idx2), ptr(scratch), st))
    check(_lib.lib().rpcc_chamfer_stats(ptr(dist1), n, ptr(dist2), m, f1_threshold ** 2, ptr(stats), st))
    s = stats.cpu().numpy()
    cham_dist1 = float(s[0] / max(n, 1))
    cham_dist2 = float(s[2] / max(m, 1))
    # fscore.py:12-16 (float32 means of the indicator)
    precision = float(np.float32(s[1]) / np.float32(max(n, 1)))
    recall = float(np.float32(s[3]) / np.float32(max(m, 1)))
    f_score = 2 * precision * recall / (precision + recall) if (precision + recall) > 0 else 0.0
    result = {
        "max": max(cham_dist1, cham_dist2),
        "mean": (cham_dist1 + cham_dist2) / 2,
        "sum": cham_dist1 + cham_dist2,
        "cd1": cham_dist1,
        "cd2": cham_dist2,
        "f_score": f_score,
        "precision": precision,
        "recall": recall,
        "chamfer_dist_info": {
            "dist1": dist1.cpu().numpy(),
            "dist2": dist2.cpu().numpy(),
            "idx1": idx1.cpu().numpy(),
            "idx2": idx2.cpu().numpy(),
        },
    }
    if out:
        for key, value in result.items():
            print(key, value)
        print("time cost: ", time.time() - t)
    return result


def calc_point_to_plane_psnr(range_ref, range_rec, lidar, knn=NORMAL_KNN, radius=NORMAL_RADIUS, r=59.7):
    """Point-to-plane PSNR of two range images over one lidar's ray table (DESIGN.md, "Point-to-plane PSNR"): each
    point's error is its offset from its nearest neighbour in the other cloud projected on that neighbour's k-NN normal
    (point-to-point where the neighbour has none); psnr = 10 log10(3 r^2 / mse) per direction, "psnr" their mean.
    range_ref / range_rec: (H,W) or (B,H,W) f32, numpy or torch (host or device).  -> dict of floats for one frame, of
    lists for a batch."""
    from . import device
    from .batch import p2plane_summary
    from .lidar import LidarConfig
    cfg = lidar if isinstance(lidar, LidarConfig) else LidarConfig(lidar)

    def dev(a):
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.asarray(a, dtype=np.float32))
        return t.to(device="cuda", dtype=torch.float32).reshape(-1, cfg.H, cfg.W).contiguous()

    a, b = dev(range_ref), dev(range_rec)
    if a.shape != b.shape:
        raise ValueError("range_ref and range_rec differ in shape")
    lut = torch.from_numpy(cfg.transform_map()).to(a.device)
    na, _ = device.normals_batch(a, lut, cfg, knn, radius)
    nb, _ = device.normals_batch(b, lut, cfg, knn, radius)
    m = device.p2plane_batch(a, b, lut, cfg, na, nb).cpu().numpy()
    rows = []
    for row in m:
        s = p2plane_summary(row)
        mse1, mse2 = s["p2plane_mse1"], s["p2plane_mse2"]
        with np.errstate(divide="ignore"):
            p = [10 * np.log10(3 * r * r / x) if x > 0 else float("inf") for x in (mse1, mse2)]
        rows.append({"psnr": (p[0] + p[1]) / 2, "psnr1": p[0], "psnr2": p[1], "mse1": mse1, "mse2": mse2,
                     "no_normal_points": s["no_normal_points"], "exhaustive_points": int(row[6])})
    if (range_ref.dim() if isinstance(range_ref, torch.Tensor) else np.ndim(range_ref)) == 2:
        return rows[0]
    return {k: [x[k] for x in rows] for k in rows[0]}
