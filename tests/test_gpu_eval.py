"""GPU tests of the range-image evaluation stage (csrc/evalq.cu): its window search must return, bit for bit, the squared
nearest-neighbour distances of the exact O(N*M) chamfer kernel (rpcc_chamfer_batch, pinned to the oracle's restatement
oracle.chamfer_nn in test_gpu_pipeline.py::test_plugin_fps_and_chamfer_drop_in) -- on encode->decode pairs, on unrelated frame pairs, with holes, and with the
negative ranges that force the exhaustive path."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu
LIDARS = ["Velodyne64E", "Velodyne32E", "VelodyneVLP16"]


def _brute(T, a_img, b_img, lut):
    """(H,W) range images -> dist1, dist2 over the compacted clouds, like calc_chamfer_distance
    (utils/evaluate_metrics.py:14-19)."""
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    pa = (a_img[..., None] * lut).reshape(-1, 3)
    pb = (b_img[..., None] * lut).reshape(-1, 3)
    va, vb = np.sum(pa, -1) != 0, np.sum(pb, -1) != 0
    a = T.from_numpy(np.ascontiguousarray(pa[va])).cuda()
    b = T.from_numpy(np.ascontiguousarray(pb[vb])).cuda()
    n, m = a.shape[0], b.shape[0]
    if n == 0 or m == 0:       # an empty cloud on the other side: +inf everywhere (rpcc_chamfer_batch's convention)
        return va, vb, np.full(n, np.inf, np.float32), np.full(m, np.inf, np.float32)
    d1 = T.empty(n, dtype=T.float32, device="cuda"); d2 = T.empty(m, dtype=T.float32, device="cuda")
    i1 = T.empty(n, dtype=T.int32, device="cuda"); i2 = T.empty(m, dtype=T.int32, device="cuda")
    scratch = T.empty(n + m, dtype=T.int64, device="cuda")
    check(_lib.lib().rpcc_chamfer_batch(ptr(a), n, ptr(b), m, ptr(d1), ptr(i1), ptr(d2), ptr(i2), ptr(scratch),
                                        T.cuda.current_stream().cuda_stream))
    T.cuda.synchronize()
    return va, vb, d1.cpu().numpy(), d2.cpu().numpy()


def _check_pair(T, R, lidar, a_img, b_img, expect_exhaustive=None):
    from rpcc_b200 import device
    cfg = R.LidarConfig(lidar)
    lut = cfg.transform_map()
    A = T.from_numpy(np.ascontiguousarray(a_img[None])).cuda()
    Bm = T.from_numpy(np.ascontiguousarray(b_img[None])).cuda()
    m, d1, d2 = device.eval_batch(A, Bm, T.from_numpy(lut).cuda(), cfg, want_dist=True)
    T.cuda.synchronize()
    m = m.cpu().numpy()[0]
    d1, d2 = d1.cpu().numpy()[0], d2.cpu().numpy()[0]
    va, vb, w1, w2 = _brute(T, a_img, b_img, lut)
    assert np.array_equal(d1.reshape(-1)[va.reshape(-1)].view(np.uint32), w1.view(np.uint32)), lidar
    assert np.array_equal(d2.reshape(-1)[vb.reshape(-1)].view(np.uint32), w2.view(np.uint32)), lidar
    assert (d1.reshape(-1)[~va.reshape(-1)] == -1).all()
    assert m[2] == va.sum() and m[6] == vb.sum()
    if np.isfinite(w1).all():
        assert abs(m[3] - np.sqrt(w1).astype(np.float64).sum()) <= 1e-9 * max(m[3], 1)    # torch.sqrt(dist1): f32 roots
    assert m[4] == (w1 < np.float32(0.0004)).sum() and m[8] == (w2 < np.float32(0.0004)).sum()
    dif = np.abs(b_img - a_img)
    assert m[0] == float(dif.max()) and abs(m[1] - dif.astype(np.float64).sum()) <= 1e-9 * max(m[1], 1)
    if expect_exhaustive is not None:
        assert (m[10] > 0) == expect_exhaustive
    return m


@pytest.fixture(scope="module")
def T():
    import torch
    return torch


@pytest.fixture(scope="module")
def R():
    import rpcc_b200
    return rpcc_b200


@pytest.mark.parametrize("lidar", LIDARS)
def test_window_search_equals_brute_force_on_decoded_frames(T, R, lidar):
    from rpcc_b200 import synthetic
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    p, g = synthetic.frame(31, lidar)
    o = oracle.compress_frame(p, lidar, g)
    rec, _, _ = oracle.decompress_sections(o["sections"], lidar, 0.02)
    m = _check_pair(T, R, lidar, o["range_image"], rec.reshape(H, W).astype(np.float32), expect_exhaustive=False)
    assert m[0] <= 0.02 + 1e-5


def test_window_search_on_unrelated_and_damaged_pairs(T, R):
    from rpcc_b200 import synthetic
    lidar = "VelodyneVLP16"          # small image: the exact O(N*M) check stays cheap even when windows grow
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    a = oracle.project(synthetic.frame(41, lidar)[0], H, W, hf, vmax, vmin)
    b = oracle.project(synthetic.frame(42, lidar)[0], H, W, hf, vmax, vmin)
    _check_pair(T, R, lidar, a, b)                       # two different scenes: windows of many pixels
    rng = np.random.default_rng(3)
    holes = b.copy()
    holes[rng.random(b.shape) < 0.6] = 0                 # most neighbours missing
    holes[:, 200:700] = 0                                # and a 500-column gap: beyond the tabulated window
    _check_pair(T, R, lidar, a, holes, expect_exhaustive=True)
    _check_pair(T, R, lidar, a, np.zeros_like(a))        # an empty cloud on one side
    shifted = np.roll(a, 3, axis=1) * np.float32(1.01)
    _check_pair(T, R, lidar, a, shifted)
    neg = a.copy()
    neg[5, 100] = -neg[5, 100] if neg[5, 100] != 0 else -3.0   # a point behind the sensor: exhaustive search for the frame
    _check_pair(T, R, lidar, a, neg, expect_exhaustive=True)


def test_encoder_eval_stage_matches_the_standalone_kernels(T, R):
    """cfg.eval: the chain decodes what it wrote (packed streams) and evaluates it; same table as decoding the blobs
    with BatchDecoder and calling rpcc_eval_batch, and no label mismatches."""
    from rpcc_b200 import device, synthetic
    from rpcc_b200.batch import BatchDecoder, BatchEncoder, eval_summary
    for nonuniform in (False, True):
        pts, off, grounds = synthetic.batch([51, 52, 53], "Velodyne64E")
        with BatchEncoder("Velodyne64E", accuracy=0.02, nonuniform=nonuniform, max_batch=3, max_points=pts.shape[0],
                          eval=True, host_chunk=2) as enc:
            out = enc.encode_host(pts, off, grounds)
            ev = out["eval"].copy()
            blobs = enc.compress(pts, off, grounds)
            cfg = enc.lidar
            rng = enc.device_buffer(0, "range", (2, cfg.H, cfg.W), T.float32).clone()     # chunk 0 = frames 0, 1
        dec = BatchDecoder("Velodyne64E", accuracy=0.02, nonuniform=nonuniform)
        d = dec.decode(blobs[:2], want_xyz=False)
        m, _, _ = device.eval_batch(rng, d["range"].contiguous(), T.from_numpy(cfg.transform_map()).cuda(), cfg)
        T.cuda.synchronize()
        assert np.array_equal(m.cpu().numpy()[:, :10], ev[:2, :10])
        assert (ev[:, 11] == 0).all() and (ev[:, 10] == 0).all()
        s = eval_summary(ev[0], cfg.HW)
        assert s["depth_max"] <= (0.02 if not nonuniform else 0.05) + 1e-5 and 0.3 < s["f_score"] <= 1.0
