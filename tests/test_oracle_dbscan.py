"""oracle.dbscan (the restatement of this project's DBSCAN definition, DESIGN.md §4) against known answers on hand-built
frames.  A frame here is one row of pixels whose ray table holds the points themselves (range 1), so that every
coordinate and every f32 distance is chosen exactly.  No GPU."""
import numpy as np
import pytest

from oracle import dbscan
from oracle.normals import cham_d

F32 = np.float32
GROUND = np.array([0, 0, 1, 100], F32)        # every point near z = 0 lies 100 m off this plane: not ground


def frame(points, empty=()):
    """points (n,3) -> (range (1,W), lut (1,W,3)); pixels listed in `empty` are left empty."""
    pts = np.asarray(points, F32).reshape(-1, 3)
    ri = np.ones((1, pts.shape[0]), F32)
    ri[0, list(empty)] = 0
    return ri, pts.reshape(1, -1, 3).copy()


def labels(points, eps, min_points, cluster_num=100, empty=()):
    ri, lut = frame(points, empty)
    return dbscan.segment(ri, lut, GROUND, eps, min_points, cluster_num)[0]


def line(x0, n, step=0.1, y=0.0):
    return [(x0 + k * step, y, 0.0) for k in range(n)]


def test_two_blobs_noise_ground_and_empty():
    blob_a = [(0.1 * i, 0.1 * j, 0.0) for i in range(4) for j in range(3)]
    blob_b = [(10 + 0.1 * i, 0.1 * j, 0.0) for i in range(4) for j in range(3)]
    pts = blob_a + [(5.0, 5.0, 0.0)] + blob_b + [(20.0, 20.0, 0.0), (3.0, 0.0, -100.0), (7.0, 0.0, 0.0)]
    lab = labels(pts, eps=0.5, min_points=5, empty=[len(pts) - 1])
    assert (lab[:12] == 2).all() and (lab[13:25] == 3).all()
    assert lab[12] == 101 and lab[25] == 101           # noise: the rest label cluster_num + 1
    assert lab[26] == 0                                # on the ground plane
    assert lab[27] == 1                                # empty pixel


def _boundary_steps(e2):
    """f32 steps dx with cham_d((0,0,0), (dx,0,0)) == e2 and the smallest one above e2."""
    cand = [F32(np.sqrt(np.float64(e2)))]
    for _ in range(4):
        cand = [np.nextafter(cand[0], F32(0))] + cand + [np.nextafter(cand[-1], F32(np.inf))]
    cand = np.array(cand, F32)
    d = cham_d(np.zeros(3, F32), np.stack([cand, np.zeros_like(cand), np.zeros_like(cand)], -1))
    on = cand[d == e2]
    over = cand[d > e2]
    assert on.size and over.size
    return on[-1], over[0]


@pytest.mark.parametrize("eps", [0.3, 1.5])
def test_chain_on_the_f32_e2_boundary(eps):
    e2 = F32(eps * eps)                                # eps * eps in double, then rounded once
    on, over = _boundary_steps(e2)
    pts = [(0.0, 0.0, 0.0), (on, 0.0, 0.0),            # exactly e2 apart: neighbours
           (0.0, 50.0, 0.0), (over, 50.0, 0.0),        # one f32 step farther: not
           (0.0, 90.0, 0.0), (F32(eps) * F32(0.5), 90.0, 0.0), (F32(eps), 90.0, 0.0)]  # a chain of half-eps links
    lab = labels(pts, eps, min_points=1)
    assert lab[0] == lab[1]
    assert lab[2] != lab[3]
    assert lab[4] == lab[5] == lab[6]
    # with min_points = 2 the pair that is one step too far apart is noise, the linked pair a cluster
    lab2 = labels(pts, eps, min_points=2)
    assert lab2[0] == lab2[1] != 101
    assert lab2[2] == lab2[3] == 101


@pytest.mark.parametrize("right_first", [True, False])
def test_border_equidistant_from_two_clusters_goes_to_the_smaller_pixel(right_first):
    left = [(-0.5, 0.0, 0.0), (-0.6, 0.0, 0.0), (-0.7, 0.0, 0.0), (-0.8, 0.0, 0.0)]
    right = [(0.5, 0.0, 0.0), (0.6, 0.0, 0.0), (0.7, 0.0, 0.0), (0.8, 0.0, 0.0)]
    border = [(0.0, 0.0, 0.0)]                           # 0.25 from both x = -0.5 and x = 0.5; 3 neighbours: not core
    pts = (right + left if right_first else left + right) + border
    lab = labels(pts, eps=0.55, min_points=4)
    assert lab[0] == 2 and lab[4] == 3 and lab[:4].tolist() == [2] * 4 and lab[4:8].tolist() == [3] * 4
    assert lab[8] == 2                                   # nearest cores tie; the one at the smaller pixel wins


def test_more_clusters_than_labels_size_ties_and_rest_label():
    sizes = [4, 5, 4, 2]
    pts = []
    for c, n in enumerate(sizes):
        pts += line(10.0 * c, n)
    first = np.cumsum([0] + sizes)
    lab = labels(pts, eps=0.15, min_points=1, cluster_num=3)     # two kept clusters
    got = [lab[first[c]:first[c + 1]] for c in range(4)]
    assert all((g == g[0]).all() for g in got)
    # kept: the 5 and, of the two 4s, the one with the smaller first pixel; numbered by first pixel
    assert [int(g[0]) for g in got] == [2, 3, 4, 4]
    ri, lut = frame(pts)
    _, found = dbscan.labels_from_graph(dbscan.graph(ri, lut, GROUND, 0.15), 1, 3)
    assert found == 4
    # cluster_num = 1: no cluster is kept, every point takes label 2
    assert (labels(pts, eps=0.15, min_points=1, cluster_num=1) == 2).all()
    # more labels than clusters: all kept, in pixel order
    assert [int(lab[f]) for lab in [labels(pts, eps=0.15, min_points=1, cluster_num=10)] for f in first[:4]] == [2, 3, 4, 5]


def _brute(pts, eps, min_points, cluster_num):
    """The definition of DESIGN.md §4 by brute force: all pairs, union-find, explicit loops."""
    n = len(pts)
    e2 = F32(eps * eps)
    D = np.stack([cham_d(pts[a], pts) for a in range(n)])
    nb = D <= e2
    core = nb.sum(1) >= min_points
    par = list(range(n))

    def find(x):
        while par[x] != x:
            x = par[x]
        return x
    for a in range(n):
        for b in range(n):
            if core[a] and core[b] and nb[a, b]:
                ra, rb = find(a), find(b)
                if ra != rb:
                    par[max(ra, rb)] = min(ra, rb)
    root = [find(a) if core[a] else -1 for a in range(n)]
    for a in range(n):
        if not core[a]:
            c = [(D[a, b], b) for b in range(n) if core[b] and nb[a, b]]
            if c:
                root[a] = find(min(c)[1])
    size = {}
    for r in root:
        if r >= 0:
            size[r] = size.get(r, 0) + 1
    ranked = sorted(size, key=lambda r: (-size[r], r))[:cluster_num - 1]
    name = {r: 2 + k for k, r in enumerate(sorted(ranked))}
    return np.array([name.get(r, cluster_num + 1) for r in root])


@pytest.mark.parametrize("min_points,cluster_num", [(1, 252), (1, 6), (4, 8), (6, 100)])
def test_random_cloud_against_brute_force(min_points, cluster_num):
    rng = np.random.default_rng(7 + min_points)
    centres = rng.uniform(-20, 20, (12, 3))
    pts = np.concatenate([c + rng.normal(0, 0.6, (int(rng.integers(3, 40)), 3)) for c in centres])
    pts = np.concatenate([pts, rng.uniform(-25, 25, (40, 3))]).astype(F32)
    pts[:, 2] = np.clip(pts[:, 2], -50, 50)
    lab = labels(pts, eps=0.9, min_points=min_points, cluster_num=cluster_num)
    assert (lab == _brute(pts, 0.9, min_points, cluster_num)).all()
    if min_points == 1:                                  # plain connected components: nothing is noise
        assert cluster_num < 252 or (lab != 253).all()


@pytest.mark.parametrize("model_method,nonuniform", [("point", False), ("point", True), ("plane", False)])
def test_compress_frame_with_given_labels_equals_the_fps_pipeline(model_method, nonuniform):
    """dbscan.compress_frame is oracle.compress_frame after its segmentation: fed FPS's own labels, the same sections."""
    import oracle
    from rpcc_b200 import synthetic
    p, g = synthetic.frame(3, "VelodyneVLP16")
    kw = dict(nonuniform=nonuniform, model_method=model_method)
    want = oracle.compress_frame(p, "VelodyneVLP16", g, plane_impl="device", **kw)
    got = dbscan.compress_frame(p, "VelodyneVLP16", g, want["seg_idx"], **kw)
    assert got["sections"] == want["sections"]
