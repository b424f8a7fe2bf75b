"""TEST INFRASTRUCTURE -- numpy / scipy restatement of this project's DBSCAN segmentation (DESIGN.md §4, "DBSCAN (this
project's definition)"; csrc/dbscan.cu).  NOT product code.

  points     pixels with range != 0 and |sum(pc*g) + g3| / |g0..2| > ground_threshold, in f32 as the FPS mask
             (torch's size-3 association: (t0 + t2) + t1)
  neighbour  cham_d(p, q) <= e2, e2 = f32(eps * eps) (eps * eps in double); p is its own neighbour
  core       at least min_points neighbours; clusters = connected components of the cores
  border     a non-core point with a core neighbour joins the cluster of its nearest core: smallest cham_d, then
             smallest flat pixel index
  noise      every other point
  labels     0 ground, 1 empty; clusters ranked by size (cores + borders; on equal size the smaller first core pixel
             first), the first cluster_num - 1 kept and numbered 2 .. in order of their first core pixel; noise and
             the other clusters share cluster_num + 1

Candidates come from scipy's cKDTree at a radius slightly above eps and are filtered with the exact f32 distance.
compress_frame encodes a frame with these labels in place of FPS's, so that whole `.rpcc` sections can be compared.
"""
import numpy as np

from . import (extract_features, intra_predict, lidar_params, model_param_point, nonuniform_quantize, pack_sections,
               plane_models_device, project, transform_map, uniform_quantize)
from .normals import cham_d

F32, F64 = np.float32, np.float64


def points_mask(range_image, lut, ground, thr=0.1):
    """-> (pts (HW,3) f32, point (HW,) bool): the pixels DBSCAN clusters."""
    ri = np.asarray(range_image, F32).reshape(-1)
    pts = (ri[:, None] * np.asarray(lut, F32).reshape(-1, 3)).astype(F32)
    g = np.asarray(ground, F32).reshape(4)
    s = (pts[:, 0] * g[0] + pts[:, 2] * g[2]) + pts[:, 1] * g[1]
    gn = np.sqrt((g[0] * g[0] + g[2] * g[2]) + g[1] * g[1])
    with np.errstate(divide="ignore", invalid="ignore"):
        dif = np.abs(s + g[3]) / gn
    return pts, (ri != 0) & (dif > F32(thr))


def graph(range_image, lut, ground, eps, thr=0.1):
    """The neighbour relation of a frame -> dict(vid (n,) flat pixel indices of the points, ascending; i, j (e,) edges
    i < j as positions in vid; d (e,) their f32 distances; HW; ri)."""
    ri = np.asarray(range_image, F32).reshape(-1)
    pts, point = points_mask(ri, lut, ground, thr)
    e2 = F32(float(eps) * float(eps))
    vid = np.flatnonzero(point)
    P = pts[vid]
    i = j = np.zeros(0, np.int64)
    d = np.zeros(0, F32)
    if vid.size > 1:
        from scipy.spatial import cKDTree
        r = float(np.sqrt(F64(e2))) * (1 + 1e-5) + 1e-30
        pairs = cKDTree(P.astype(F64)).query_pairs(r, output_type="ndarray")
        if pairs.size:
            i, j = pairs[:, 0].astype(np.int64), pairs[:, 1].astype(np.int64)
            swap = i > j
            i, j = np.where(swap, j, i), np.where(swap, i, j)
            d = cham_d(P[i], P[j])
            keep = d <= e2
            i, j, d = i[keep], j[keep], d[keep]
    return dict(vid=vid, i=i, j=j, d=d, HW=ri.size, ri=ri)


def labels_from_graph(G, min_points, cluster_num):
    """-> (labels (HW,) int32, clusters found)."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    vid, i, j, d = G["vid"], G["i"], G["j"], G["d"]
    n = vid.size
    lab = np.where(G["ri"] == 0, 1, 0).astype(np.int32)
    if n == 0:
        return lab, 0
    deg = 1 + np.bincount(i, minlength=n) + np.bincount(j, minlength=n)
    core = deg >= min_points
    root = np.full(n, -1, np.int64)
    cpos = np.flatnonzero(core)
    if cpos.size:
        cc = core[i] & core[j]
        A = coo_matrix((np.ones(int(cc.sum()), np.int8), (i[cc], j[cc])), shape=(n, n))
        _, comp = connected_components(A, directed=False)
        first = np.full(comp.max() + 1, n, np.int64)
        np.minimum.at(first, comp[cpos], cpos)               # positions ascend with the pixel index
        root[cpos] = first[comp[cpos]]
        # borders: a non-core end of an edge whose other end is core
        a = core[i] & ~core[j]
        b = core[j] & ~core[i]
        bp = np.concatenate((j[a], i[b]))
        cp = np.concatenate((i[a], j[b]))
        bd = np.concatenate((d[a], d[b]))
        if bp.size:
            o = np.lexsort((cp, bd, bp))                      # by border, then distance, then core pixel
            bp, cp = bp[o], cp[o]
            lead = np.ones(bp.size, bool)
            lead[1:] = bp[1:] != bp[:-1]
            root[bp[lead]] = root[cp[lead]]
    pts_lab = np.full(n, cluster_num + 1, np.int32)
    member = root >= 0
    roots, sizes = np.unique(root[member], return_counts=True)
    kept = np.sort(roots[np.lexsort((roots, -sizes))[:max(cluster_num - 1, 0)]])
    lab_of = np.full(n, cluster_num + 1, np.int32)
    lab_of[kept] = 2 + np.arange(kept.size, dtype=np.int32)
    pts_lab[member] = lab_of[root[member]]
    lab[vid] = pts_lab
    return lab, int(roots.size)


def segment(range_image, lut, ground, eps=1.5, min_points=10, cluster_num=100, thr=0.1):
    """-> (H,W) int32 labels of one frame."""
    lut = np.asarray(lut, F32)
    lab, _ = labels_from_graph(graph(range_image, lut, ground, eps, thr), min_points, cluster_num)
    return lab.reshape(lut.shape[:2])


def compress_frame(points, lidar, ground_model, seg, accuracy=0.02, nonuniform=False, model_method="point",
                   angle_threshold=75.0, frame=0):
    """tools/compress.py:44-133 with the labels `seg` (H,W) (e.g. segment()'s) instead of FPS's, and the device's own
    per-cluster planes for model_method 'plane' (oracle.plane_models_device) -> dict(seg_idx, model_param, symbols,
    sections).  The steps are oracle.compress_frame's after its segmentation, with the same defaults."""
    H, W, hfov, vmax, vmin = lidar_params(lidar)
    lut = transform_map(H, W, hfov, vmax, vmin)
    step = accuracy * 2
    ri = project(points, H, W, hfov, vmax, vmin)
    seg = np.ascontiguousarray(seg, np.int32).reshape(H, W)
    mp = model_param_point(ri, seg, ground_model)
    if model_method == "plane":
        mp = plane_models_device(ri, lut, seg, mp, frame=frame, angle_threshold=float(angle_threshold))
    res = ri - intra_predict(seg, mp, lut)
    sal = None
    if not nonuniform:
        sym = uniform_quantize(seg, res, step)
    else:
        c = dict(level_kp_num=(30, 10, 3, 0), level_dacc=(0, 0.02, 0.04, 0.06), ground_level=2,
                 region=3, segments=8, sharp_num=4, less_sharp_num=8, flat_num=6)
        _, kp = extract_features(ri, seg, c["region"], c["segments"], c["sharp_num"], c["less_sharp_num"], c["flat_num"])
        acc = np.array([step] * len(c["level_kp_num"])) + np.array(c["level_dacc"])
        sym, sal = nonuniform_quantize(seg, res, kp, c["level_kp_num"], acc, c["ground_level"])
    return dict(seg_idx=seg, model_param=mp, symbols=sym, sections=pack_sections(mp, seg, sym, sal))
