"""CPU pins of oracle/normals.py, the numpy restatement of the point-to-plane definition (DESIGN.md, "Point-to-plane
PSNR") that tests/test_gpu_p2plane.py holds csrc/normals.cu to.  The clouds here are given directly as ray tables with
range 1 (points = lut), so that they lie exactly on the analytic shapes."""
import numpy as np

from oracle import normals as N


def _plane_grid(H=12, W=40, step=0.125):
    """Points of z = 0.25 x - 0.5 y - 2 on a dyadic grid: exact in f32 and in f64."""
    x, y = np.meshgrid(np.arange(W) * step - 2.0, np.arange(H) * step + 10.0)   # x + y + z > 0: all points valid
    z = 0.25 * x - 0.5 * y - 2.0
    return np.stack([x, y, z], -1).astype(np.float32)


def test_fmaf_is_exactly_rounded():
    rng = np.random.default_rng(0)
    a = rng.standard_normal(20000).astype(np.float32)
    c = rng.standard_normal(20000).astype(np.float32)
    want = np.array([float(np.float32(_exact_fma(float(x), float(x), float(z)))) for x, z in zip(a, c)], np.float32)
    assert np.array_equal(N.fmaf(a, a, c).view(np.uint32), want.view(np.uint32))


def _exact_fma(a, b, c):
    from fractions import Fraction
    v = Fraction(a) * Fraction(b) + Fraction(c)
    # round the exact rational to the nearest f32, ties to even
    f = np.float32(float(v))
    lo, hi = (np.nextafter(f, np.float32(-np.inf)), f) if Fraction(float(f)) > v else (f, np.nextafter(f, np.float32(np.inf)))
    dl, dh = v - Fraction(float(lo)), Fraction(float(hi)) - v
    if dl != dh:
        return lo if dl < dh else hi
    return lo if (lo.view(np.uint32) & 1) == 0 else hi


def test_plane_gives_its_normal():
    lut = _plane_grid()
    rng = np.ones(lut.shape[:2], np.float32)
    for brute in (True, False):
        out = N.normals(rng, lut, knn=16, radius=1.0, brute=brute)
        assert out["has"].sum() == rng.size                    # every point of the plane has a normal
        want = np.array([-0.25, 0.5, 1.0]) / np.linalg.norm([0.25, 0.5, 1.0])   # oriented so that n . p <= 0
        assert np.abs(out["normals"][out["has"]] - want).max() <= 1e-9
        p = lut.reshape(-1, 3).astype(np.float64)
        assert ((out["normals"] * p).sum(1) <= 0).all()


def test_single_scan_line_has_no_normal():
    lut = np.zeros((4, 64, 3), np.float32)
    t = np.arange(64) * 0.0625
    lut[2] = np.stack([t, 0.5 * t + 1.0, np.full(64, -2.0)], -1)   # one straight line of points, the other rows empty
    rng = np.ones((4, 64), np.float32)
    out = N.normals(rng, lut, knn=16, radius=1.0)
    assert out["count"][2 * 64:3 * 64].min() >= 3
    assert not out["has"].any()


def test_fewer_than_three_neighbours_within_radius_have_no_normal():
    lut = _plane_grid(H=4, W=8, step=2.0)                    # neighbours 2 m apart: only the point itself within 1 m
    rng = np.ones(lut.shape[:2], np.float32)
    out = N.normals(rng, lut, knn=16, radius=1.0)
    assert (out["count"] == 1).all() and not out["has"].any()
    lut2 = lut.copy()
    lut2[0, 1] = lut2[0, 0] + np.float32(0.25)               # a pair: two neighbours, still no normal
    out = N.normals(rng, lut2, knn=16, radius=1.0)
    assert out["count"][0] == 2 and not out["has"].any()
    out = N.normals(rng, lut, knn=16, radius=3.0)            # a larger radius reaches the grid neighbours
    assert out["has"].all()


def test_knn_sets_tree_equals_brute_force():
    from rpcc_b200 import synthetic
    import oracle
    lidar = "VelodyneVLP16"
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    img = oracle.project(synthetic.frame(5, lidar)[0], H, W, hf, vmax, vmin)
    img[:, ::3] = 0
    for knn, radius in ((16, 1.0), (3, 0.3), (32, 5.0)):
        a = N.knn_sets(img, lut, knn, radius, brute=True)
        b = N.knn_sets(img, lut, knn, radius, brute=False)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_p2plane_error_definition():
    """Two parallel planes 0.25 apart vertically: every error is their distance squared; a point whose neighbour has no normal counts its squared
    distance."""
    lut = _plane_grid(step=0.25)
    a = np.ones(lut.shape[:2], np.float32)
    lut2 = lut.copy()
    lut2[..., 2] -= np.float32(0.25)
    both = np.concatenate([lut, lut2], 0)
    ref = np.concatenate([a, np.zeros_like(a)], 0)
    rec = np.concatenate([np.zeros_like(a), a], 0)
    n = np.zeros(both.shape[:2] + (3,), np.float32)
    n[...] = np.array([-0.25, 0.5, 1.0]) / np.linalg.norm([0.25, 0.5, 1.0])
    m = N.p2plane(ref, rec, both, n, n)
    dz = 0.25 / np.linalg.norm([0.25, 0.5, 1.0])              # distance between the planes along their normal
    assert m[0] == m[3] == a.size and m[2] == m[5] == 0
    assert abs(m[1] / m[0] - dz * dz) <= 1e-6 * dz * dz and abs(m[4] / m[3] - dz * dz) <= 1e-6 * dz * dz
    m0 = N.p2plane(ref, rec, both, np.zeros_like(n), np.zeros_like(n))
    assert m0[2] == m0[5] == a.size and m0[1] > m[1]
    e = N.p2plane(ref, np.zeros_like(rec), both, n, n)
    assert e[0] == a.size and np.isinf(e[1]) and e[3] == 0 and e[4] == 0
