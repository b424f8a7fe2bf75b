"""GPU parity tests, stage by stage, through the C ABI (rpcc_*_batch) against the oracle
(oracle/liborc.so), the reference's own compiled code (oracle/_ref, when shipped) and torch's own
arithmetic for the segment() lines (tests/refimpl.py).  Integer/index/byte results: bit-exact."""
import hashlib
import os

import numpy as np
import pytest

import oracle
from oracle import ref
from conftest import EXAMPLE_GROUND

pytestmark = pytest.mark.gpu

LIDARS = ["Velodyne64E", "Velodyne32E", "VelodyneVLP16"]


@pytest.fixture(scope="module")
def T():
    import torch
    return torch


@pytest.fixture(scope="module")
def R():
    import rpcc_b200
    from rpcc_b200 import device, synthetic
    rpcc_b200.device_mod = device
    rpcc_b200.synth = synthetic
    return rpcc_b200


def _frames(R, lidar, seeds):
    pts, off, g = R.synth.batch(seeds, lidar)
    return pts, off, g


def _project_dev(T, R, pts, off, lidar_name):
    cfg = R.LidarConfig(lidar_name)
    d_pts = T.from_numpy(pts).cuda()
    d_off = T.from_numpy(off).cuda()
    rng = R.device_mod.project_batch(d_pts, d_off, cfg)
    T.cuda.synchronize()
    return cfg, rng


# ----------------------------------------------------------------------------- stage 1
def test_project_example_bit_exact(T, R, example_points):
    off = np.array([0, example_points.shape[0]], np.int64)
    cfg, rng = _project_dev(T, R, example_points, off, "Velodyne64E")
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    want = oracle.project(example_points, H, W, hf, vmax, vmin)
    got = rng[0].cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert (got != 0).sum() == 94053
    # the reference's own range image of this frame (point_cloud_to_range_image_even), stored by tests/golden/make_golden.py
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "example_golden.npz"))
    assert hashlib.sha256(got.tobytes()).hexdigest() == str(gold["u_range_sha"])


@pytest.mark.parametrize("lidar", LIDARS)
def test_project_synthetic_batch(T, R, lidar):
    pts, off, _ = _frames(R, lidar, range(6))
    cfg, rng = _project_dev(T, R, pts, off, lidar)
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    got = rng.cpu().numpy()
    for b in range(6):
        want = oracle.project(pts[off[b]:off[b + 1]], H, W, hf, vmax, vmin)
        assert np.array_equal(got[b].view(np.uint32), want.view(np.uint32)), (lidar, b)


def test_project_stride3_empty_and_zero_points(T, R):
    cfg = R.LidarConfig("Velodyne64E")
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    p0, _ = R.synth.frame(3)
    rs = np.random.default_rng(0)
    # frame 1: exact-zero points sprinkled in (SURVEY C9: they re-open their pixel), frame 2: empty
    p1 = p0[:5000].copy()
    zrow = int(round((0 - np.float32(vmin)) / ((np.float32(vmax) - np.float32(vmin)) / 63)))
    # points that land on the zero-depth pixel (row zrow, col 0), before and after the zeros
    dirv = oracle.transform_map(H, W, hf, vmax, vmin)[zrow, 0]
    hits = np.stack([dirv * d for d in (7.0, 5.0, 9.0, 8.0)]).astype(np.float32)
    seqs = [hits[0], hits[1], np.zeros(3, np.float32), hits[2], np.array([-0.0, 0.0, 0.0], np.float32), hits[3]]
    ins = sorted(rs.choice(5000, len(seqs), replace=False))
    for i, s in zip(ins, seqs):
        p1[i, :3] = s
    frames = [p0[:, :3].copy(), p1[:, :3].copy(), np.zeros((0, 3), np.float32), p0[:100, :3].copy()]
    pts = np.ascontiguousarray(np.concatenate(frames, 0))
    off = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int64)
    rng = R.device_mod.project_batch(T.from_numpy(pts).cuda(), T.from_numpy(off).cuda(), cfg)
    got = rng.cpu().numpy()
    for b, fr in enumerate(frames):
        want = oracle.project(fr, H, W, hf, vmax, vmin)
        assert np.array_equal(got[b].view(np.uint32), want.view(np.uint32)), b
    assert got[2].max() == 0


def test_project_rounding_boundary_stress(T, R):
    """The kernel derives most pixels with a fast atan2 and only re-derives with the exact libm sequence
    when the continuous coordinate is near a rounding boundary; aim points AT the boundaries (column
    k+0.5 and row k+0.5, offsets from 1e-7 to 1e-2 px, both sides, all quadrants) and demand the
    reference's image bit for bit."""
    g = np.random.default_rng(11)
    for lidar in LIDARS:
        cfg = R.LidarConfig(lidar)
        H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
        n = 300000
        deltas = np.concatenate([[0.0], 10.0 ** np.arange(-7, -1.9, 0.25)])
        d = g.choice(deltas, n) * g.choice([-1.0, 1.0], n)
        on_col = g.random(n) < 0.6
        colf = g.integers(0, W, n) + np.where(on_col, 0.5 + d, g.random(n))
        rowf = g.integers(0, H, n) + np.where(~on_col, 0.5 + d, g.random(n) - 0.5)
        az = colf * (hf / W)
        el = vmin + rowf * ((vmax - vmin) / (H - 1))
        r = g.uniform(1.0, 90.0, n)
        pts = np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el), np.zeros(n)], -1).astype(np.float32)
        # axis-aligned and degenerate directions
        extra = np.array([[5, 0, 0, 0], [-5, 0, 0, 0], [0, 5, 0, 0], [0, -5, 0, 0], [0, 0, 5, 0], [0, 0, -5, 0], [1, 1, 0, 0],
                          [-1, -1, 0, 0], [1e-20, 0, 0, 0], [0, 1e-20, 1e-20, 0], [3, -0.0, -1, 0], [-3, -0.0, -1, 0],
                          [1, 2, -0.0, 0]], np.float32)
        pts = np.concatenate([pts, extra], 0)
        off = np.array([0, pts.shape[0]], np.int64)
        rng = R.device_mod.project_batch(T.from_numpy(pts).cuda(), T.from_numpy(off).cuda(), cfg)
        want = oracle.project(pts, H, W, hf, vmax, vmin)
        got = rng[0].cpu().numpy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (lidar, int((got != want).sum()))


def test_project_random_cloud_stress(T, R):
    """2M random points per lidar table: directions well outside the vertical field of view (row clamp,
    the exact-path elevations), all ranges from millimetres to kilometres, many collisions per pixel."""
    g = np.random.default_rng(5)
    for lidar in LIDARS:
        cfg = R.LidarConfig(lidar)
        H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
        n = 2000000
        az = g.uniform(-np.pi, np.pi, n)
        el = np.where(g.random(n) < 0.8, g.uniform(vmin - 0.05, vmax + 0.05, n), g.uniform(-1.55, 1.55, n))
        r = 10.0 ** g.uniform(-3, 3.5, n)
        pts = np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el), g.random(n)], -1).astype(np.float32)
        off = np.array([0, n // 3, n // 3, n], np.int64)   # three frames, the middle one empty
        rng = R.device_mod.project_batch(T.from_numpy(pts).cuda(), T.from_numpy(off).cuda(), cfg)
        got = rng.cpu().numpy()
        for b in range(3):
            want = oracle.project(pts[off[b]:off[b + 1]], H, W, hf, vmax, vmin)
            assert np.array_equal(got[b].view(np.uint32), want.view(np.uint32)), (lidar, b, int((got[b] != want).sum()))


def test_project_many_synthetic_frames(T, R):
    pts, off, _ = _frames(R, "Velodyne64E", range(100, 140))
    cfg, rng = _project_dev(T, R, pts, off, "Velodyne64E")
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    got = rng.cpu().numpy()
    for b in range(40):
        want = oracle.project(pts[off[b]:off[b + 1]], H, W, hf, vmax, vmin)
        assert np.array_equal(got[b].view(np.uint32), want.view(np.uint32)), b


# ----------------------------------------------------------------------------- torch semantics (H2)
def test_torch_size3_reduction_association(T):
    """Pins the float32 association of torch.sum / torch.norm over a size-3 last dim on this box:
    the device kernels assume (t0 + t2) + t1 (common.cuh torch_sum3)."""
    g = np.random.default_rng(7)
    n = 1 << 22
    v = (g.standard_normal((n, 3)) * g.uniform(0.01, 80, (n, 1))).astype(np.float32)
    tv = T.from_numpy(v).cuda()
    got_sum = T.sum(tv * tv, -1).cpu().numpy()
    got_norm = T.norm(tv, 2, -1).cpu().numpy()
    sq = v * v
    a02_1 = (sq[:, 0] + sq[:, 2]) + sq[:, 1]
    a01_2 = (sq[:, 0] + sq[:, 1]) + sq[:, 2]
    m_sum = {"(0+2)+1": np.mean(got_sum != a02_1), "(0+1)+2": np.mean(got_sum != a01_2)}
    m_norm = {"(0+2)+1": np.mean(got_norm != np.sqrt(a02_1)), "(0+1)+2": np.mean(got_norm != np.sqrt(a01_2))}
    print("sum mismatch rates", m_sum, "norm mismatch rates", m_norm)
    assert m_sum["(0+2)+1"] == 0.0, m_sum
    assert m_norm["(0+2)+1"] == 0.0, m_norm
    # 4-D broadcast shape used by calc_cluster_residual_radius (H,W,100,3) and the (1,1,3) plane norm
    pc = tv[: 64 * 500].view(64, 500, 1, 3)
    c = tv[100000:100100].view(1, 1, 100, 3)
    d = T.norm(pc - c, 2, -1).cpu().numpy()
    dn = (v[: 64 * 500].reshape(64, 500, 1, 3) - v[100000:100100].reshape(1, 1, 100, 3))
    dq = dn * dn
    assert np.array_equal(d, np.sqrt((dq[..., 0] + dq[..., 2]) + dq[..., 1]))
    g3 = T.norm(tv[:1].view(1, 1, 3), 2, -1).cpu().numpy().ravel()[0]
    assert g3 == np.sqrt((sq[0, 0] + sq[0, 2]) + sq[0, 1])
    # comparison against the python scalar is done in float32; max returns the first index on ties
    x = T.tensor([np.float32(0.1)], dtype=T.float32).cuda()
    assert not bool((x > 0.1).item())
    t = T.tensor([[-1.0, -1.0, -2.0, -1.0]]).cuda()
    assert int(T.max(t, -1)[1].item()) == 0


# ----------------------------------------------------------------------------- stage 2: FPS
def test_fps_generic_vs_reference_kernel(T, R):
    g = np.random.default_rng(1)
    for n, m, dup in [(5000, 64, False), (1024, 32, True), (777, 20, True), (40000, 100, False), (33, 8, False)]:
        pts = g.standard_normal((2, n, 3)).astype(np.float32) * 10
        if dup:  # exact ties: many identical points (the masked origin points of segment())
            pts[:, g.choice(n, n // 2, replace=False)] = 0.0
            pts[1, :, :] = np.round(pts[1], 0)
        got = R.device_mod.fps_batch(T.from_numpy(pts).cuda(), m).cpu().numpy()
        for b in range(2):
            want = oracle.fps(pts[b], m)
            assert np.array_equal(got[b], want), (n, m, b)
        if ref.have_cuda():
            import refimpl
            r = refimpl.ref_fps_gpu(T.from_numpy(pts).cuda(), m).cpu().numpy()
            assert np.array_equal(got, r), (n, m)


@pytest.mark.parametrize("lidar", LIDARS)
def test_segment_fps_and_labels(T, R, lidar):
    import refimpl
    seeds = [0, 1, 2]
    pts, off, grounds = _frames(R, lidar, seeds)
    cfg, rng = _project_dev(T, R, pts, off, lidar)
    lut = cfg.transform_map()
    d_lut = T.from_numpy(lut).cuda()
    d_g = T.from_numpy(grounds.astype(np.float32)).cuda()
    cidx, centers = R.device_mod.segment_fps_batch(rng, d_lut, d_g, 100, 0.1)
    labels, book = R.device_mod.assign_labels_batch(rng, d_lut, d_g, centers)
    T.cuda.synchronize()
    ri = rng.cpu().numpy()
    for b in range(len(seeds)):
        seg_o, cidx_o, cent_o = oracle.segment(ri[b], lut, grounds[b], 100)
        seg_t, cidx_t, ng_t = refimpl.torch_segment(ri[b], lut, grounds[b], 100)
        # the oracle restatement and torch's own arithmetic (+ the reference FPS kernel) agree ...
        assert np.array_equal(cidx_o, cidx_t), (lidar, b)
        assert np.array_equal(seg_o, seg_t), (lidar, b, int((seg_o != seg_t).sum()))
        # ... and the device path reproduces both
        assert np.array_equal(cidx[b].cpu().numpy(), cidx_t), (lidar, b)
        assert np.array_equal(centers[b].cpu().numpy(), ng_t[cidx_t]), (lidar, b)
        assert np.array_equal(labels[b].cpu().numpy().astype(np.int64), seg_t), (lidar, b)


@pytest.mark.parametrize("lidar,count", [("Velodyne64E", 64), ("Velodyne32E", 48)])
def test_segment_fps_many_frames_against_the_reference_kernel(T, R, lidar, count):
    """Seeds of many distinct frames in one launch against the reference's own kernel (one launch as well): the rare
    paths of the round kernel -- ties, buckets that die, frames that take several CTAs' worth of time -- get their
    chance to show up."""
    import refimpl
    if not ref.have_cuda():
        pytest.skip("oracle/_ref/libref_fps.so not shipped")
    pts, off, grounds = _frames(R, lidar, list(range(300, 300 + count)))
    cfg, rng = _project_dev(T, R, pts, off, lidar)
    d_lut = T.from_numpy(cfg.transform_map()).cuda()
    d_g = T.from_numpy(grounds.astype(np.float32)).cuda()
    cidx, centers = R.device_mod.segment_fps_batch(rng, d_lut, d_g, 100, 0.1)
    # the reference's masked cloud (utils/segment_utils.py:137-141), torch's own arithmetic
    pc = rng.unsqueeze(-1) * d_lut.unsqueeze(0)                                  # (B, H, W, 3)
    pp = d_g.view(-1, 1, 1, 4)
    dif = T.abs(T.sum(pc * pp[..., :3], -1) + pp[..., 3]) / T.norm(pp[..., :3], 2, -1)
    masked = (pc * (dif > 0.1).unsqueeze(-1)).reshape(count, -1, 3).contiguous()
    want = refimpl.ref_fps_gpu(masked, 100)
    T.cuda.synchronize()
    assert T.equal(cidx, want), [int(b) for b in T.nonzero((cidx != want).any(1)).flatten()[:8]]
    assert T.equal(centers, T.gather(masked, 1, want.long().unsqueeze(-1).expand(-1, -1, 3)))


def test_segment_fps_when_seed_zero_is_a_real_point(T, R):
    """The FPS kernel has two update paths: the usual one (pixel 0 is a ground / empty pixel, so every masked point sits
    at distance zero from seed 0 for good) and the general one, taken when pixel 0 survives the ground mask -- then the
    masked points are live candidates, tie among themselves across the whole image, and can be chosen.  A ground model
    far from every point masks nothing; the empty pixels still are origin points."""
    import refimpl
    lidar = "VelodyneVLP16"
    pts, off, grounds = _frames(R, lidar, [7, 8])
    cfg, rng = _project_dev(T, R, pts, off, lidar)
    lut = cfg.transform_map()
    ri = rng.cpu().numpy()
    assert (ri[:, 0, 0] != 0).all()                     # pixel 0 holds a point in these frames
    g = np.tile(np.array([[0.0, 0.0, 1.0, 100.0]], np.float32), (2, 1))
    d_lut, d_g = T.from_numpy(lut).cuda(), T.from_numpy(g).cuda()
    cidx, centers = R.device_mod.segment_fps_batch(rng, d_lut, d_g, 100, 0.1)
    labels, _ = R.device_mod.assign_labels_batch(rng, d_lut, d_g, centers)
    T.cuda.synchronize()
    for b in range(2):
        seg_t, cidx_t, ng_t = refimpl.torch_segment(ri[b], lut, g[b], 100)
        assert np.array_equal(cidx[b].cpu().numpy(), cidx_t), b
        assert np.array_equal(centers[b].cpu().numpy(), ng_t[cidx_t]), b
        assert np.array_equal(labels[b].cpu().numpy().astype(np.int64), seg_t), b


@pytest.mark.parametrize("lidar", LIDARS)
def test_segment_fps_with_exact_ties_between_buckets(T, R, lidar):
    """The round kernel keeps one maximum per 64-pixel bucket and finds a round's winner inside the single bucket that holds
    the frame's maximum; when several buckets hold the very same value every warp scans its candidates for the smallest
    tie key.  Range images that force that path: a sphere (every ray the same length: symmetric distances all over the
    image), ranges rounded to whole metres, and an empty frame; ground far away (nothing masked) and a real one."""
    import refimpl
    pts, off, grounds = _frames(R, lidar, [3])
    cfg, rng = _project_dev(T, R, pts, off, lidar)
    lut = cfg.transform_map()
    real = rng[0].cpu().numpy()
    H, W = real.shape
    images = [np.full((H, W), 10.0, np.float32), np.round(real), np.zeros((H, W), np.float32)]
    half = np.full((H, W), 7.0, np.float32)
    half[:, W // 2:] = 0.0                                 # half of the image empty
    images.append(half)
    ri = np.stack(images).astype(np.float32)
    for g4 in ([0.0, 0.0, 1.0, 100.0], list(grounds[0])):
        g = np.tile(np.array([g4], np.float32), (len(images), 1))
        d_r, d_lut, d_g = T.from_numpy(ri).cuda(), T.from_numpy(lut).cuda(), T.from_numpy(g).cuda()
        cidx, centers = R.device_mod.segment_fps_batch(d_r, d_lut, d_g, 100, 0.1)
        T.cuda.synchronize()
        for b in range(len(images)):
            _, cidx_t, ng_t = refimpl.torch_segment(ri[b], lut, g[b], 100)
            assert np.array_equal(cidx[b].cpu().numpy(), cidx_t), (lidar, b, g4)
            assert np.array_equal(centers[b].cpu().numpy(), ng_t[cidx_t]), (lidar, b, g4)


def test_segment_fps_odd_image_takes_the_generic_kernels(T, R):
    """Images whose pixel count is 1, 2 or 3 modulo 4 (3 x 343, 18 x 57, 11 x 101; no lidar of the reference has one) are
    staged into copies padded to a multiple of 4 pixels, every pad pixel a copy of pixel 0.  Seed 0 is an origin point in
    one frame and a real point in two others; in the last one it lies 150 m from every other point, so the origin points
    hold the largest distance and round 1 is decided by the tie rule among them, which a pad pixel would join if it were
    one of them.  Seeds and labels against the oracle."""
    for H, W in ((3, 343), (18, 57), (11, 101)):
        g = np.random.default_rng(5)
        az = np.linspace(0, 2 * np.pi, W, endpoint=False)[None, :]
        el = np.linspace(-0.4, 0.1, H)[:, None]
        lut = np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el) * np.ones_like(az)], -1).astype(np.float32)
        ri = (5.0 + 20.0 * g.random((4, H, W))).astype(np.float32)
        ri[g.random((4, H, W)) < 0.1] = 0.0
        ri[1, 0, 0] = 0.0
        ri[2, 0, 0] = 9.0
        ri[3][:, (az[0] > np.pi / 3) & (az[0] < 5 * np.pi / 3)] = 0.0   # points within 60 degrees of pixel 0's azimuth only
        ri[3, 0, 0] = 150.0
        xyz = ri[3][..., None].astype(np.float64) * lut
        p0 = xyz[0, 0]
        assert np.all(np.linalg.norm(xyz - p0, axis=-1)[ri[3] != 0][1:] < 0.99 * np.linalg.norm(p0)), (H, W)
        ground = np.tile(np.array([[0.0, 0.0, 1.0, 1.7]], np.float32), (4, 1))
        d_r, d_lut, d_g = T.from_numpy(ri).cuda(), T.from_numpy(lut).cuda(), T.from_numpy(ground).cuda()
        cidx, centers = R.device_mod.segment_fps_batch(d_r, d_lut, d_g, 40, 0.1)
        labels, _ = R.device_mod.assign_labels_batch(d_r, d_lut, d_g, centers)
        T.cuda.synchronize()
        for b in range(4):
            seg_o, cidx_o, cent_o = oracle.segment(ri[b], lut, ground[b], 40)
            assert b != 3 or not cent_o[1].any(), (H, W)     # round 1 picked an origin point
            assert np.array_equal(cidx[b].cpu().numpy(), cidx_o), (H, W, b)
            assert np.array_equal(labels[b].cpu().numpy().astype(np.int64), seg_o), (H, W, b)


def test_segment_example_frame(T, R, example_points):
    import refimpl
    off = np.array([0, example_points.shape[0]], np.int64)
    cfg, rng = _project_dev(T, R, example_points, off, "Velodyne64E")
    lut = cfg.transform_map()
    d_lut = T.from_numpy(lut).cuda()
    d_g = T.tensor([EXAMPLE_GROUND], dtype=T.float32).cuda()
    cidx, centers = R.device_mod.segment_fps_batch(rng, d_lut, d_g, 100, 0.1)
    labels, _ = R.device_mod.assign_labels_batch(rng, d_lut, d_g, centers)
    seg_t, cidx_t, _ = refimpl.torch_segment(rng[0].cpu().numpy(), lut, np.array(EXAMPLE_GROUND), 100)
    assert np.array_equal(cidx[0].cpu().numpy(), cidx_t)
    assert np.array_equal(labels[0].cpu().numpy().astype(np.int64), seg_t)


# ----------------------------------------------------------------------------- stages 3+4
@pytest.mark.parametrize("lidar", LIDARS)
def test_model_quantize_pack(T, R, lidar):
    seeds = [4, 5]
    pts, off, grounds = _frames(R, lidar, seeds)
    cfg, rng = _project_dev(T, R, pts, off, lidar)
    lut = cfg.transform_map()
    d_lut = T.from_numpy(lut).cuda()
    d_g = T.from_numpy(grounds.astype(np.float32)).cuda()
    cidx, centers = R.device_mod.segment_fps_batch(rng, d_lut, d_g, 100, 0.1)
    labels, book = R.device_mod.assign_labels_batch(rng, d_lut, d_g, centers)
    model, results = R.device_mod.point_model_batch(rng, labels, d_g, book, 102)
    step = 0.04
    symbols, contour, seq = R.device_mod.quantize_pack_batch(rng, labels, model, d_lut, book, step)
    T.cuda.synchronize()
    res = results.cpu().numpy().view(np.uint32)
    for b in range(len(seeds)):
        want = oracle.compress_frame(pts[off[b]:off[b + 1]], lidar, grounds[b])
        sec = want["sections"]
        nsym, nseq, rows = int(res[b, 0]), int(res[b, 1]), int(res[b, 2])
        assert np.array_equal(labels[b].cpu().numpy().astype(np.int32), want["seg_idx"])
        assert rows == want["model_param"].shape[0]
        assert model[b, :rows].cpu().numpy().tobytes() == sec["plane_param"]
        assert symbols[b, :nsym].cpu().numpy().tobytes() == sec["residual_quantized"]
        assert contour[b].cpu().numpy().tobytes() == sec["contour_map"]
        assert seq[b, :nseq].cpu().numpy().tobytes() == sec["idx_sequence"]


# ----------------------------------------------------------------------------- ground plane (the product's own RANSAC)
@pytest.mark.parametrize("lidar", LIDARS)
def test_ground_fit_matches_its_restatement(T, R, lidar):
    """open3d's segment_plane cannot be pinned (absent, and the reference feeds it an unseeded subsample), so the
    ground plane is the product's own deterministic RANSAC; the oracle restates it (same counter-based samples, same
    summation orders) and the device planes must equal it bit for bit -- single-frame op and batched kernel (frame
    keys), plus the reference's fallback when fewer than 800 pixels lie below -1.5 m (every pixel is a candidate)."""
    from rpcc_b200.segment_utils import PointCloudSegment
    seeds = [81, 82, 83, 84, 85]
    pts, off, _ = _frames(R, lidar, seeds)
    cfg, rng = _project_dev(T, R, pts, off, lidar)
    lut = cfg.transform_map()
    seg = PointCloudSegment(lut)
    ris = rng.cpu().numpy().reshape(len(seeds), cfg.H, cfg.W)
    for b in range(len(seeds)):
        for seed in (0x5EED, 7):
            got = seg.ransac_plane_segmentation(ris[b], seed=seed)
            want = oracle.ground_fit(ris[b], lut, seed=seed, frame=0)
            assert got.tobytes() == want.tobytes(), (lidar, b, seed, got, want)
    # batched kernel: without frame keys every frame is keyed 0 (its plane depends on its content alone); with
    # caller-supplied keys frame b is keyed seed + keys[b]
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    d_lut = T.from_numpy(lut).cuda()
    d_g = T.empty((len(seeds), 4), dtype=T.float32, device="cuda")
    keys = np.array([0, 11, 5, 1 << 40, 3], np.uint64)
    d_keys = T.from_numpy(keys.view(np.int64)).cuda()
    for dk, hk in ((None, np.zeros(len(seeds), np.uint64)), (d_keys, keys)):
        check(_lib.lib().rpcc_ground_fit_batch(ptr(rng), ptr(d_lut), len(seeds), cfg.H, cfg.W, 0x5EED,
                                               ptr(dk) if dk is not None else None, ptr(d_g),
                                               T.cuda.current_stream().cuda_stream))
        T.cuda.synchronize()
        got = d_g.cpu().numpy()
        for b in range(len(seeds)):
            assert got[b].tobytes() == oracle.ground_fit(ris[b], lut, seed=0x5EED, frame=int(hk[b])).tobytes(), (lidar, b)
    # no ground below the sensor: fewer than 800 candidates -> all pixels (utils/segment_utils.py:105-106)
    bare = np.where(ris[0] * lut[..., 2] < -1.5, 0.0, ris[0]).astype(np.float32)
    assert seg.ransac_plane_segmentation(bare).tobytes() == oracle.ground_fit(bare, lut).tobytes()
