"""Mirror of utils/evaluate_metrics.py:9-45 (calc_chamfer_distance) on the device chamfer kernels.
The PSNR helpers of that file need open3d normals and a cKDTree and are outside this path."""
import time

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr


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
