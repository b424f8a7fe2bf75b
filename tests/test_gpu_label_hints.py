"""GPU parity tests for the encoder's label assignment from FPS owner hints.  The FPS rounds leave, per pixel, the
centre that gave its smallest running distance when no other centre comes within a relative 4e-6 (eps) of it, and the
assignment evaluates that one centre; every other pixel takes the bounded search.  Each scene runs through the encoder
(injected ground planes) and its labels are compared with torch's own segment() lines for the encoder's own range
images and centres (tests/refimpl.py).  The scenes count, with a numpy restatement of the distances, the pixels whose
two nearest centres lie within eps (the fallback) and just outside it (hints near the margin); the mirror and bisector
scenes assert a minimum of both, so that they show both sides of the margin were reached, and the others assert the
condition they are built for (far pixels, duplicate centres)."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

LIDARS = ["Velodyne64E", "Velodyne32E", "VelodyneVLP16"]
EPS = 4e-6
GROUND = np.array([0.0057, -0.0445, -0.9990, -1.7938], np.float32)


@pytest.fixture(scope="module")
def T():
    import torch
    return torch


@pytest.fixture(scope="module")
def R():
    import rpcc_b200
    return rpcc_b200


def _sum3(a, b, c):
    return (np.float32(a) + np.float32(c)) + np.float32(b)


def _points_of(ri, lut):
    """Points r * ray (f32) of the non-empty pixels, raster order: they project back onto (about) the same pixels."""
    m = ri != 0
    xyz = (ri[..., None] * lut)[m]
    return np.concatenate([xyz, np.zeros((xyz.shape[0], 1), np.float32)], 1).astype(np.float32)


def _margins(ri, lut, g, cents):
    """numpy restatement: among the pixels the assignment resolves by a hint or by the search (valid, above the ground
    threshold, residual not below the ground-skip threshold), how many have their two nearest centres (squared FPS-style
    distances) within eps, and how many between eps and 5 eps."""
    ri, lut = ri.reshape(-1), lut.reshape(-1, 3)
    g = g.astype(np.float32)
    xyz = ri[:, None] * lut
    gn = np.sqrt(_sum3(g[0] * g[0], g[1] * g[1], g[2] * g[2]))
    keep = np.abs(_sum3(xyz[:, 0] * g[0], xyz[:, 1] * g[1], xyz[:, 2] * g[2]) + g[3]) / gn > np.float32(0.1)
    rp = (-g[3]) / _sum3(g[0] * lut[:, 0], g[1] * lut[:, 1], g[2] * lut[:, 2])
    res = np.abs(ri - rp)
    dpl = np.min(np.abs(_sum3(cents[:, 0] * g[0], cents[:, 1] * g[1], cents[:, 2] * g[2]) + g[3]))
    skip = np.float32(0.5) * (dpl / np.sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2])) * np.float32(0.99) - np.float32(2e-4)
    sel = (ri != 0) & keep & ~(res < skip)
    p = xyz[sel]
    d = np.empty((p.shape[0], cents.shape[0]), np.float32)
    for c in range(cents.shape[0]):
        dd = p - cents[c]
        d[:, c] = _sum3(dd[:, 0] * dd[:, 0], dd[:, 1] * dd[:, 1], dd[:, 2] * dd[:, 2])
    ds = np.sort(d, 1)
    d0, d1 = ds[:, 0].astype(np.float64), ds[:, 1].astype(np.float64)
    amb = d1 <= d0 * (1 + EPS)
    near = ~amb & (d1 <= d0 * (1 + 5 * EPS))
    return int(amb.sum()), int(near.sum())


def _encode_and_check(T, R, lidar, images, grounds):
    """Encode the range images' points with the given ground planes; labels against torch for the encoder's own range
    images and centres.  -> (pixels within eps, pixels within (eps, 5 eps]) summed over the frames"""
    import refimpl
    from rpcc_b200.batch import BatchEncoder
    cfg = lidar if isinstance(lidar, R.LidarConfig) else R.LidarConfig(lidar)
    lut = cfg.transform_map()
    H, W = cfg.H, cfg.W
    per = [_points_of(ri, lut) for ri in images]
    pts = np.concatenate(per, 0)
    off = np.cumsum([0] + [p.shape[0] for p in per]).astype(np.int64)
    B = len(images)
    grounds = np.asarray(grounds, np.float32)
    with BatchEncoder(cfg, accuracy=0.02, max_batch=B, max_points=max(pts.shape[0], 1), host_chunk=B) as enc:
        enc.encode_host(pts, off, grounds)
        m = enc.K - 2
        rng = enc.device_buffer(0, "range", (B, H, W), T.float32).cpu().numpy().copy()
        labels = enc.device_buffer(0, "labels", (B, H, W), T.uint8).cpu().numpy().astype(np.int64)
        cents = enc.device_buffer(0, "centers", (B, m, 3), T.float32).cpu().numpy().copy()
    amb = near = 0
    for b in range(B):
        want = refimpl.torch_labels(rng[b], lut, grounds[b], cents[b])
        assert np.array_equal(labels[b], want), (cfg.name, b, int(np.sum(labels[b] != want)))
        a, n = _margins(rng[b], lut, grounds[b], cents[b])
        amb += a
        near += n
    return amb, near, rng, cents


def _base(lidar, i):
    from rpcc_b200 import synthetic
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    pts, _ = synthetic.frame(900 + i, lidar)
    return oracle.project(pts, H, W, hf, vmax, vmin)


def _mirror(ri, rel=None, g=None):
    """The image made symmetric about the vertical plane through azimuth 0 (the ray table is: column w and column
    -w mod W hold (x, y, z) and (x, -y, z) bit for bit); rel: the mirrored half scaled by 1 + rel * U(0.5, 1) per row."""
    W = ri.shape[1]
    out = ri.copy()
    w = np.arange(1, W // 2)
    half = ri[:, w]
    if rel is not None:
        half = (half * (1 + rel * g.uniform(0.5, 1.0, (ri.shape[0], 1)))).astype(np.float32)
    out[:, (-w) % W] = half
    return out


def _bisectors(ri, lut, cents, g):
    """ri with one pixel per pair of neighbouring centres moved onto (or next to) the pair's bisector: the pixel whose
    ray passes nearest to the pair's midpoint gets the range at which the ray crosses the bisector, times 1 + delta, with
    delta from a ladder of 0 and +-1e-8 ... 1e-5 -- so that the pixel's two nearest centres differ by anything from an
    exact tie to some 1e-5 relative.  (Centres of a first encoding of ri: the moved pixels are close to two centres and
    rarely change the seeds; the check uses the centres of the encoding that is checked.)"""
    out = ri.copy()
    l = lut.reshape(-1, 3).astype(np.float64)
    ln = l / np.linalg.norm(l, axis=1, keepdims=True)
    c = cents.astype(np.float64)
    live = np.flatnonzero(np.any(cents != 0, 1))
    ladder = [0.0, 1e-8, -1e-8, 1e-7, -1e-7, 5e-7, -5e-7, 2e-6, -2e-6, 5e-6, -5e-6, 1e-5, -1e-5]
    used = set()
    for k, i in enumerate(live):
        d = np.sum((c[live] - c[i]) ** 2, 1)
        d[live == i] = np.inf
        j = live[int(np.argmin(d))]
        mid = 0.5 * (c[i] + c[j])
        px = int(np.argmax(ln @ (mid / np.linalg.norm(mid))))
        den = 2.0 * (l[px] @ (c[i] - c[j]))
        if px in used or den == 0:
            continue
        r = (c[i] @ c[i] - c[j] @ c[j]) / den
        if not (0.5 < r < 200) or np.linalg.norm(r * l[px] - mid) > 0.25 * np.sqrt(d.min()):
            continue
        used.add(px)
        out.reshape(-1)[px] = np.float32(r * (1 + ladder[k % len(ladder)]))
    return out


@pytest.mark.parametrize("lidar", LIDARS)
def test_hints_on_mirror_and_bisector_scenes(T, R, lidar):
    """Mirror-symmetric frames (where FPS picks mirrored centres, pixels on the symmetry plane are tied exactly), the
    same frames with the mirrored half moved by 1e-7 ... 2e-5 relative, frames with pixels placed at and around the
    bisectors of neighbouring centres (pixels on both sides of eps), and a frame whose seed 0 is a real point (the
    origin points' running distances are not zero: the hints' origin rule matters)."""
    g = np.random.default_rng(21)
    base = [_base(lidar, i) for i in range(3)]
    imgs = [_mirror(base[0]), _mirror(base[1])]
    for k, rel in enumerate((1e-7, 1e-6, 3e-6, 6e-6, 2e-5)):
        imgs.append(_mirror(base[k % 3], rel, g))
    seed0 = base[2].copy()
    seed0[0, 0] = np.float32(12.5)                       # row 0 looks up: far above the ground plane
    imgs.append(seed0)
    grounds = np.tile(GROUND, (len(imgs), 1))
    _, _, rng, cents = _encode_and_check(T, R, lidar, imgs, grounds)
    assert rng[-1, 0, 0] != 0 and not np.all(cents[-1, 0] == 0), "seed 0 should be a real point"
    lut = R.LidarConfig(lidar).transform_map()
    bis = [_bisectors(rng[b], lut, cents[b], g) for b in (0, 2, 7)]
    amb, near, _, _ = _encode_and_check(T, R, lidar, imgs + bis, np.tile(GROUND, (len(imgs) + len(bis), 1)))
    print(lidar, "pixels with two centres within eps:", amb, "| within (eps, 5 eps]:", near)
    assert amb >= 10 and near >= 10, (lidar, amb, near)


def test_hints_far_points_and_duplicate_centres(T, R):
    """Points beyond 1e5 m (the first pass's running distances clamp at 1e10: no hint from seed 0), and a frame with
    fewer live points than centres (every live point becomes a centre, then all running distances are zero and seed 0
    repeats: duplicate centres)."""
    lidar = "Velodyne64E"
    g = np.random.default_rng(22)
    H, W = oracle.LIDARS[lidar]["H"], oracle.LIDARS[lidar]["W"]
    far = _base(lidar, 5)
    idx = g.choice(H * W, 3000, replace=False)
    far.reshape(-1)[idx] = g.uniform(1.2e5, 4e5, idx.size).astype(np.float32)
    few = _base(lidar, 6)
    lut = R.LidarConfig(lidar).transform_map()
    xyz = few[..., None] * lut
    live = (np.abs(_sum3(xyz[..., 0] * GROUND[0], xyz[..., 1] * GROUND[1], xyz[..., 2] * GROUND[2]) + GROUND[3])
            / np.float32(np.linalg.norm(GROUND[:3])) > 0.08) & (few != 0)
    keep = np.flatnonzero(live.reshape(-1))
    drop = keep[g.permutation(keep.size)[40:]]
    few.reshape(-1)[drop] = 0.0                          # at most 40 points above the ground are left
    few[0, 0] = 0.0                                      # seed 0 an empty pixel
    amb, near, rng, cents = _encode_and_check(T, R, lidar, [far, few], np.tile(GROUND, (2, 1)))
    n_far = int(np.sum(rng[0] > 1e5))
    dup = cents[1][np.all(cents[1] == 0, 1)].shape[0]
    print("far pixels:", n_far, "| centres at the origin in the sparse frame:", dup, "| within eps:", amb)
    assert n_far >= 1000 and dup >= 2


@pytest.mark.parametrize("shape", [(11, 101), (18, 57)])
def test_hints_on_odd_images(T, R, shape):
    """A 1111-pixel and a 1026-pixel image (not multiples of 4: staged into padded copies, and the FPS of a staged image
    leaves every hint at 255), mirror-symmetric as above, through the encoder."""
    H, W = shape
    cfg = R.LidarConfig(hfov_deg=360.0, vmax_deg=10.0, vmin_deg=-25.0, H=H, W=W)
    g = np.random.default_rng(23)
    imgs = []
    for i in range(4):
        ri = (3.0 + 40.0 * g.random((H, W))).astype(np.float32)
        ri[g.random((H, W)) < 0.1] = 0.0
        imgs.append(_mirror(ri) if i % 2 == 0 else ri)
    amb, near, _, _ = _encode_and_check(T, R, cfg, imgs, np.tile(GROUND, (len(imgs), 1)))
    print(shape, "pixels with two centres within eps:", amb)
