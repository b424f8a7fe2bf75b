"""GPU tests of point-to-plane PSNR (csrc/normals.cu): the k-NN normals against oracle/normals.py on synthetic frames of
three lidars, with holes, a wide gap, a negative range and the knn / radius edges; the point-to-plane table against the
oracle and against its analytic properties; the encoder's eval = 2 stage; and the --p2plane column of compress_datalist."""
import os
import re

import numpy as np
import pytest

import oracle
from oracle import normals as N

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIDARS = ["VelodyneVLP16", "Velodyne32E", "Velodyne64E"]


@pytest.fixture(scope="module")
def T():
    import torch
    return torch


def _lut(lidar):
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    return oracle.transform_map(H, W, hf, vmax, vmin)


def _dev_normals(T, lidar, imgs, knn=16, radius=1.0):
    from rpcc_b200 import LidarConfig, device
    cfg = LidarConfig(lidar)
    t = T.from_numpy(np.ascontiguousarray(np.stack(imgs), dtype=np.float32)).cuda()
    n, fb = device.normals_batch(t, T.from_numpy(cfg.transform_map()).cuda(), cfg, knn, radius)
    T.cuda.synchronize()
    return n.cpu().numpy().reshape(len(imgs), -1, 3), fb.cpu().numpy()


def _check_normals(img, lut, got, knn, radius):
    """Device normals (HW,3) f32 against the oracle: same "no normal" set away from the eigen-gap threshold, and within
    1e-6 rad elsewhere (up to sign only where n . p is within rounding of 0)."""
    want = N.normals(img, lut, knn, radius)
    pts, valid = N.cloud(img, lut)
    has = np.any(got != 0, 1)
    assert not has[~valid].any()
    lam = want["lam"]
    gap = (lam[:, 1] - lam[:, 0]) - 1e-6 * lam[:, 2]
    clear = (want["count"] < 3) | (np.abs(gap) > 1e-4 * lam[:, 2]) | (lam[:, 2] == 0)
    assert np.array_equal(has[clear & valid], want["has"][clear & valid])
    both = has & want["has"]
    g = got[both].astype(np.float64)
    w = want["normals"][both]
    assert np.abs(np.linalg.norm(g, axis=1) - 1).max() <= 1e-6
    cos = np.abs((g * w).sum(1)) / np.linalg.norm(g, axis=1)
    ang = np.arccos(np.minimum(cos, 1.0))
    assert ang.max() <= 1e-6, ang.max()
    p = pts[both].astype(np.float64)
    side = (g * p).sum(1)
    ambiguous = np.abs((w * p).sum(1)) <= 1e-6 * np.linalg.norm(p, axis=1)
    assert (side[~ambiguous] <= 0).all() and ((g * w).sum(1)[~ambiguous] > 0).all()
    return want


@pytest.mark.parametrize("lidar", LIDARS)
def test_normals_match_the_oracle(T, lidar):
    from rpcc_b200 import synthetic
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = _lut(lidar)
    imgs = [oracle.project(synthetic.frame(s, lidar)[0], H, W, hf, vmax, vmin) for s in (61, 62)]
    got, fb = _dev_normals(T, lidar, imgs)
    for b in range(2):
        want = _check_normals(imgs[b], lut, got[b], 16, 1.0)
        assert want["has"].mean() > 0.5                      # most points of a scene have a normal


def test_normals_on_damaged_frames_and_at_the_parameter_edges(T):
    from rpcc_b200 import synthetic
    lidar = "VelodyneVLP16"
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = _lut(lidar)
    a = oracle.project(synthetic.frame(71, lidar)[0], H, W, hf, vmax, vmin)
    rng = np.random.default_rng(5)
    holes = a.copy()
    holes[rng.random(a.shape) < 0.6] = 0
    holes[:, 200:700] = 0
    holes[8, 400:405] = 2.0                 # a few near points alone in the gap: too few within the radius, whole scan
    got, fb = _dev_normals(T, lidar, [a, holes])
    _check_normals(a, lut, got[0], 16, 1.0)
    _check_normals(holes, lut, got[1], 16, 1.0)
    assert fb[0] == 0 and fb[1] > 0
    neg = a.copy()
    neg[5, 100] = -3.0                      # a point behind the sensor: the frame is searched exhaustively
    got, fb = _dev_normals(T, lidar, [neg])
    _check_normals(neg, lut, got[0], 16, 1.0)
    assert fb[0] == np.count_nonzero(N.cloud(neg, lut)[1])
    for knn, radius in ((3, 1.0), (32, 1.0), (16, 0.05)):
        got, _ = _dev_normals(T, lidar, [a], knn, radius)
        want = _check_normals(a, lut, got[0], knn, radius)
        if radius < 0.1:
            pts, valid = N.cloud(a, lut)
            far = valid & (np.linalg.norm(pts, axis=1) > 20)
            assert (~want["has"][far]).mean() > 0.5          # far points have no normal at a 5 cm radius


def test_normals_argument_checks(T):
    from rpcc_b200 import LidarConfig, _lib, device
    cfg = LidarConfig("VelodyneVLP16")
    t = T.zeros((1, cfg.H, cfg.W), dtype=T.float32, device="cuda")
    lut = T.from_numpy(cfg.transform_map()).cuda()
    for knn, radius in ((2, 1.0), (33, 1.0), (16, 0.0), (16, -1.0)):
        with pytest.raises(_lib.RpccError):
            device.normals_batch(t, lut, cfg, knn, radius)
    n, _ = device.normals_batch(t, lut, cfg)
    assert not n.any()


def _pair(lidar, seed, accuracy=0.02):
    from rpcc_b200 import synthetic
    H, W = oracle.lidar_params(lidar)[:2]
    p, g = synthetic.frame(seed, lidar)
    o = oracle.compress_frame(p, lidar, g, accuracy=accuracy)
    rec, _, _ = oracle.decompress_sections(o["sections"], lidar, accuracy)
    return o["range_image"].astype(np.float32), rec.reshape(H, W).astype(np.float32)


def _dev_p2plane(T, lidar, refs, recs, knn=16, radius=1.0):
    from rpcc_b200 import LidarConfig, device
    cfg = LidarConfig(lidar)
    lut = T.from_numpy(cfg.transform_map()).cuda()
    a = T.from_numpy(np.ascontiguousarray(np.stack(refs), dtype=np.float32)).cuda()
    b = T.from_numpy(np.ascontiguousarray(np.stack(recs), dtype=np.float32)).cuda()
    na, _ = device.normals_batch(a, lut, cfg, knn, radius)
    nb, _ = device.normals_batch(b, lut, cfg, knn, radius)
    m = device.p2plane_batch(a, b, lut, cfg, na, nb)
    e, _, _ = device.eval_batch(a, b, lut, cfg)
    T.cuda.synchronize()
    B = len(refs)
    return (m.cpu().numpy(), na.cpu().numpy().reshape(B, -1, 3), nb.cpu().numpy().reshape(B, -1, 3), e.cpu().numpy())


@pytest.mark.parametrize("lidar", LIDARS)
def test_p2plane_matches_the_oracle_on_decoded_frames(T, lidar):
    ref, rec = _pair(lidar, 81)
    m, na, nb, e = _dev_p2plane(T, lidar, [ref], [rec])
    want = N.p2plane(ref, rec, _lut(lidar), na[0], nb[0])
    m = m[0]
    assert m[0] == want[0] and m[3] == want[3] and m[2] == want[2] and m[5] == want[5]
    assert abs(m[1] - want[1]) <= 1e-9 * want[1] and abs(m[4] - want[4]) <= 1e-9 * want[4]
    assert m[6] == 0
    assert m[0] == e[0, 2] and m[3] == e[0, 6]
    # per point the plane error is at most the point-to-point one, so the same holds for the sums (f32 normals: 1e-6)
    assert m[1] <= e[0, 5] * (1 + 1e-6) and m[4] <= e[0, 9] * (1 + 1e-6)
    assert m[1] < 0.5 * e[0, 5]


def test_p2plane_on_damaged_pairs(T):
    from rpcc_b200 import synthetic
    lidar = "VelodyneVLP16"
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = _lut(lidar)
    a = oracle.project(synthetic.frame(41, lidar)[0], H, W, hf, vmax, vmin)
    b = oracle.project(synthetic.frame(42, lidar)[0], H, W, hf, vmax, vmin)
    rng = np.random.default_rng(3)
    holes = b.copy()
    holes[rng.random(b.shape) < 0.6] = 0
    holes[:, 200:700] = 0
    neg = a.copy()
    neg[5, 100] = -3.0
    pairs = [(a, b), (a, holes), (a, neg)]
    m, na, nb, e = _dev_p2plane(T, lidar, [p[0] for p in pairs], [p[1] for p in pairs])
    for k, (x, y) in enumerate(pairs):
        want = N.p2plane(x, y, lut, na[k], nb[k])
        assert np.array_equal(m[k, [0, 2, 3, 5]], want[[0, 2, 3, 5]]), k
        assert np.allclose(m[k, [1, 4]], want[[1, 4]], rtol=1e-9, atol=0), k
        assert m[k, 6] == e[k, 10], k                        # the same searches as the chamfer's fall back
    assert m[1, 6] > 0 and m[2, 6] > 0
    # an empty cloud on the other side: +inf one way, nothing the other
    m, _, _, _ = _dev_p2plane(T, lidar, [a], [np.zeros_like(a)])
    assert m[0, 0] > 0 and np.isinf(m[0, 1]) and m[0, 3] == 0 and m[0, 4] == 0


def test_p2plane_of_parallel_and_coplanar_ground_planes(T):
    """A horizontal ground plane against the same plane lowered by d: mse = d^2 (within 1e-6 relative).  Against a
    sparser sampling of the same plane, whose points sit elsewhere in the plane: mse <= 1e-10."""
    lidar = "Velodyne64E"
    lut = _lut(lidar)
    lz = lut[..., 2]
    down = lz < -0.03

    def ground(h):
        img = np.zeros(lz.shape, np.float32)
        img[down] = (np.float64(h) / -lz[down].astype(np.float64)).astype(np.float32)
        return img

    ref = ground(1.75)
    d = 0.5
    sparse = ref.copy()
    sparse[:, 1::2] = 0
    m, _, _, e = _dev_p2plane(T, lidar, [ref, ref], [ground(1.75 + d), sparse])
    assert abs(m[0, 1] / m[0, 0] - d * d) <= 1e-6 * d * d and abs(m[0, 4] / m[0, 3] - d * d) <= 1e-6 * d * d
    assert m[1, 1] / m[1, 0] <= 1e-10 and m[1, 4] / m[1, 3] <= 1e-10
    assert e[1, 5] / e[1, 2] > 1e-4                            # the point-to-point error is not small there
    assert m[:, [2, 5]].sum() < 0.01 * m[:, [0, 3]].sum()


def test_calc_point_to_plane_psnr_host_and_device(T):
    from rpcc_b200.batch import p2plane_summary
    from rpcc_b200.evaluate_metrics import calc_point_to_plane_psnr
    lidar = "Velodyne32E"
    ref, rec = _pair(lidar, 91)
    m, _, _, _ = _dev_p2plane(T, lidar, [ref], [rec])
    s = p2plane_summary(m[0])
    host = calc_point_to_plane_psnr(ref, rec, lidar)
    dev = calc_point_to_plane_psnr(T.from_numpy(ref).cuda(), T.from_numpy(rec).cuda(), lidar)
    assert host["psnr"] == dev["psnr"] == s["psnr_p2plane"]
    mse1 = m[0, 1] / m[0, 0]
    assert host["mse1"] == mse1 and abs(host["psnr1"] - 10 * np.log10(3 * 59.7 ** 2 / mse1)) <= 1e-12
    batch = calc_point_to_plane_psnr(np.stack([ref, ref]), np.stack([rec, ref]), lidar)
    assert batch["psnr"][0] == host["psnr"] and batch["psnr"][1] == float("inf")


def test_encoder_p2plane_stage_matches_the_standalone_kernels(T):
    """eval = 2: columns 0-11 are those of eval = 1 bit for bit, 12-18 those of the standalone calls on the slot's range
    images and the BatchDecoder reconstruction."""
    from rpcc_b200 import LidarConfig, device, synthetic
    from rpcc_b200._lib import EVAL_COLS, P2PLANE_COLS
    from rpcc_b200.batch import BatchDecoder, BatchEncoder, eval_summary
    for nonuniform in (False, True):
        pts, off, grounds = synthetic.batch([51, 52, 53], "Velodyne64E")
        kw = dict(accuracy=0.02, nonuniform=nonuniform, max_batch=3, max_points=pts.shape[0], eval=True, host_chunk=2)
        with BatchEncoder("Velodyne64E", **kw) as enc:
            ev1 = enc.encode_host(pts, off, grounds)["eval"].copy()
        with BatchEncoder("Velodyne64E", p2plane=True, **kw) as enc:
            out = enc.encode_host(pts, off, grounds)
            ev = out["eval"].copy()
            blobs = enc.compress(pts, off, grounds)
            cfg = enc.lidar
            rng = enc.device_buffer(0, "range", (2, cfg.H, cfg.W), T.float32).clone()
        assert ev.shape == (3, EVAL_COLS + P2PLANE_COLS)
        assert np.array_equal(ev[:, :EVAL_COLS].view(np.uint64), ev1.view(np.uint64))
        dec = BatchDecoder("Velodyne64E", accuracy=0.02, nonuniform=nonuniform)
        d = dec.decode(blobs[:2], want_xyz=False)
        lut = T.from_numpy(cfg.transform_map()).cuda()
        rec = d["range"].contiguous()
        na, _ = device.normals_batch(rng, lut, LidarConfig("Velodyne64E"))
        nb, _ = device.normals_batch(rec, lut, LidarConfig("Velodyne64E"))
        m = device.p2plane_batch(rng, rec, lut, cfg, na, nb)
        T.cuda.synchronize()
        assert np.array_equal(m.cpu().numpy().view(np.uint64), ev[:2, EVAL_COLS:].view(np.uint64))
        s = eval_summary(ev[0], cfg.HW)
        assert np.isfinite(s["psnr_p2plane"]) and s["psnr_p2plane"] >= s["psnr_p2p"]
        assert s["no_normal_points"] == int(ev[0, EVAL_COLS + 2] + ev[0, EVAL_COLS + 5])
        assert "psnr_p2plane" not in eval_summary(ev1[0], cfg.HW)


def test_compress_datalist_p2plane_column(T, tmp_path, capsys):
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchEncoder, eval_summary
    from rpcc_b200.tools import compress_datalist
    from rpcc_b200.tools.compress_datalist import M_PSNR_P2PLANE, output_path_for
    lidar = "Velodyne64E"
    names, frames = [], []
    os.makedirs(tmp_path / "in")
    for i in range(3):
        p, _ = synthetic.frame(9100 + i, lidar)
        path = str(tmp_path / "in" / ("%06d.bin" % i))
        p.tofile(path)
        names.append(path)
        frames.append(p)
    lst = str(tmp_path / "list.txt")
    open(lst, "w").write("\n".join(names) + "\n")

    def run(outdir, *flags):
        a = compress_datalist.parser().parse_args(["--datalist", lst, "--output_dir", str(tmp_path / outdir), "--lidar",
                                                   lidar, "--workers", "2", "--batch", "2", "--output", *flags])
        table = compress_datalist.compress(a)
        return table, capsys.readouterr().out, [open(output_path_for(str(tmp_path / outdir), n), "rb").read() for n in names]

    t0, out0, blobs0 = run("plain")
    t1, out1, blobs1 = run("p2", "--p2plane")
    assert blobs1 == blobs0
    assert "Point-to-Plane" not in out0 and not t0[:, M_PSNR_P2PLANE].any()
    lines = re.findall(r"Point-to-Plane PSNR \(r=59.7\):\s+(\S+)", out1)
    assert len(lines) == 3 and "Point-to-Plane PSNR (mean over frames)" in out1
    assert "Point-to-Point PSNR" in out1                     # --p2plane implies --eval
    pts = np.concatenate(frames)
    off = np.concatenate(([0], np.cumsum([f.shape[0] for f in frames]))).astype(np.int64)
    with BatchEncoder(lidar, eval=True, p2plane=True, max_batch=3, max_points=pts.shape[0]) as enc:
        ev = enc.encode_host(pts, off)["eval"]
        want = [eval_summary(ev[i], enc.lidar.HW)["psnr_p2plane"] for i in range(3)]
    assert list(t1[:, M_PSNR_P2PLANE]) == want
    assert [float(x) for x in lines] == want


def test_p2plane_cols_match_header():
    from rpcc_b200._lib import NORMAL_KNN, NORMAL_RADIUS, P2PLANE_COLS
    src = open(os.path.join(ROOT, "include", "rpcc_b200.h")).read()
    m = re.search(r"^#define\s+RPCC_P2PLANE_COLS\s+(\d+)\b", src, re.M)
    assert m and P2PLANE_COLS == int(m.group(1))
    assert NORMAL_KNN == int(re.search(r"^#define\s+RPCC_NORMAL_KNN\s+(\d+)\b", src, re.M).group(1))
    assert NORMAL_RADIUS == float(re.search(r"^#define\s+RPCC_NORMAL_RADIUS\s+([0-9.]+)f?\b", src, re.M).group(1))
