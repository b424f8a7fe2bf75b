"""Pins the CPU oracle (oracle/liborc.so) BEFORE it is trusted as a checker:
  * against tests/golden/example_golden.npz, produced by the reference's own Python + C++ on
    assets/example_data/example.bin (tests/golden/make_golden.py);
  * against the reference's compiled C++ (oracle/_ref) on synthetic frames of every lidar, when present;
  * against the only known-answer vector the reference holds (ContourExtractor docstring);
  * its restated glibc atan2f against the libm of the machine the test runs on."""
import hashlib
import os

import numpy as np
import pytest

import oracle
from oracle import ref

GOLD = os.path.join(os.path.dirname(__file__), "golden", "example_golden.npz")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.mark.parametrize("tag,nonuniform", [("u", False), ("n", True)])
def test_oracle_matches_reference_golden(example_points, gold, tag, nonuniform):
    out = oracle.compress_frame(example_points, "Velodyne64E", gold["ground"], accuracy=0.02, nonuniform=nonuniform)
    g = lambda k: gold[tag + "_" + k]  # noqa: E731
    assert sha(out["range_image"]) == str(g("range_sha"))
    assert int((out["range_image"] != 0).sum()) == int(g("valid")) == 94053
    assert np.array_equal(out["seg_idx"].astype(np.uint8), g("seg_u8"))
    assert np.array_equal(out["center_idx"], g("center_idx"))
    assert out["model_param"].tobytes() == g("model_param").tobytes()
    assert sha(out["pred"]) == str(g("pred_sha"))
    assert np.array_equal(out["symbols"].astype(np.int16), g("symbols"))
    sec = out["sections"]
    assert sec["contour_map"] == g("contour_bits").tobytes()
    assert sec["idx_sequence"] == g("idx_sequence").tobytes()
    if nonuniform:
        assert np.array_equal(out["key_point_map"].astype(np.uint8), g("key_points_u8"))
        assert np.array_equal(out["salience_level"].astype(np.uint8), g("salience"))
    # the .rpcc file, byte for byte (bz2 level 9 is deterministic)
    assert oracle.write_rpcc(sec, "bzip2") == g("rpcc").tobytes()
    rec, xyz, seg = oracle.decompress_sections(sec, "Velodyne64E", 0.02)
    assert sha(rec[..., None]) == str(g("rec_sha"))
    assert sha(xyz) == str(g("xyz_sha"))
    bound = 0.02 if not nonuniform else 0.02 + 0.03
    assert float(np.abs(rec - out["range_image"]).max()) <= bound + 1e-5


def test_contour_known_answer(gold):
    contour, seq = oracle.extract_contour(gold["kat_idx_map"])
    assert np.array_equal(contour, gold["kat_contour"])
    assert np.array_equal(seq, gold["kat_seq"])
    assert np.array_equal(oracle.recover_map(contour, seq), gold["kat_idx_map"])


@pytest.mark.skipif(not ref.have_cpp(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("lidar", ["Velodyne64E", "Velodyne32E", "VelodyneVLP16", "64x31", "4x1025"])
def test_oracle_matches_compiled_reference(lidar):
    """Also at two shapes no lidar has (a sensor of +10 / -25 degrees): W < 32, and W > 1024 with H*W % 32 != 0."""
    from rpcc_b200 import LidarConfig, synthetic
    if "x" in lidar:
        H, W = map(int, lidar.split("x"))
        lidar = LidarConfig(hfov_deg=360.0, vmax_deg=10.0, vmin_deg=-25.0, H=H, W=W)
    d, s, q, c, f = (ref.cpp(n) for n in ("dataset_utils_cpp", "segment_utils_cpp", "quantization_utils_cpp",
                                          "contour_utils_cpp", "feature_extractor_cpp"))
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    for seed in (11, 12):
        pts, ground = synthetic.frame(seed, lidar)
        ri = oracle.project(pts, H, W, hf, vmax, vmin)
        assert np.array_equal(ri.view(np.uint32), d.point_cloud_to_range_image_even(
            np.ascontiguousarray(pts[:, :3]), H, W, hf, vmax, vmin).view(np.uint32))
        assert np.array_equal(ri, oracle.project(pts, H, W, hf, vmax, vmin, restated_atan2=True))
        seg, _, _ = oracle.segment(ri, lut, ground, 100)
        pm = oracle.point_modeling(ri, seg)
        assert pm.tobytes() == s.point_modeling(ri[..., None], seg).tobytes()
        mp = oracle.model_param_point(ri, seg, ground)
        pred = oracle.intra_predict(seg, mp, lut)
        assert pred.tobytes() == s.intra_predict(seg, mp, lut).tobytes()
        res = ri - pred
        assert np.array_equal(oracle.uniform_quantize(seg, res, 0.04), q.uniform_quantize(seg, res[..., None], 0.04))
        _, kp = oracle.extract_features(ri, seg)
        kp_r = _ref_keypoints_zeroed_heap(ri, seg)
        assert np.array_equal(kp, kp_r)
        acc = np.array([0.04] * 4) + np.array([0, 0.02, 0.04, 0.06])
        sy, sl = oracle.nonuniform_quantize(seg, res, kp, (30, 10, 3, 0), acc, 2)
        sy_r, sl_r = q.nonuniform_quantize(seg, res[..., None], kp, np.array((30, 10, 3, 0)), acc, 2)
        assert np.array_equal(sy, sy_r) and np.array_equal(sl, sl_r)
        ct, sq = oracle.extract_contour(seg)
        ct_r, sq_r = c.extract_contour(seg)
        assert np.array_equal(ct, ct_r) and np.array_equal(sq, sq_r)
        assert np.array_equal(oracle.recover_map(ct, sq), c.recover_map(ct_r, sq_r))


def _ref_keypoints_zeroed_heap(ri, seg):
    """The reference's extract_features_with_segment never zero-fills its output (SURVEY C7), so it is
    run in a child process whose malloc zero-fills (glibc MALLOC_PERTURB_=255): the deterministic reading."""
    import subprocess
    import sys
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as d:
        np.savez(os.path.join(d, "in.npz"), ri=ri, seg=seg)
        code = ("import sys, numpy as np; sys.path.insert(0, %r); from oracle import ref; "
                "z = np.load(%r); f = ref.cpp('feature_extractor_cpp'); "
                "_, kp = f.extract_features_with_segment(z['ri'], z['seg'], 3, 8, 4, 8, 6); np.save(%r, kp)"
                % (root, os.path.join(d, "in.npz"), os.path.join(d, "kp.npy")))
        subprocess.check_call([sys.executable, "-c", code], env=dict(os.environ, MALLOC_PERTURB_="255"))
        return np.load(os.path.join(d, "kp.npy"))


def test_restated_atan2f_matches_libm():
    g = np.random.default_rng(5)
    n = 2_000_000
    x = (g.standard_normal(n) * 40).astype(np.float32)
    y = (g.standard_normal(n) * 40).astype(np.float32)
    a, b = oracle.atan2f_pair(y, x)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    # vertical-angle style inputs (z, planar distance), axis-aligned and signed-zero cases
    z = (g.standard_normal(n) * 3).astype(np.float32)
    d = np.abs(x) + np.float32(0.5)
    a, b = oracle.atan2f_pair(z, d)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    sp_y = np.array([0.0, -0.0, 0.0, -0.0, 1.0, -1.0, 0.0, 5.0, -5.0, 1e-30, 3.0], np.float32)
    sp_x = np.array([0.0, 0.0, -0.0, -0.0, 0.0, 0.0, 1.0, 1.0, 1.0, 1.0, -1e-30], np.float32)
    a, b = oracle.atan2f_pair(sp_y, sp_x)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_fps_tie_rule_matches_tree_order():
    """All-identical points: the reference tree picks min bit-reversed (k mod 1024), then min k (SURVEY A.2)."""
    pts = np.zeros((3000, 3), np.float32)
    idx = oracle.fps(pts, 4)
    assert idx.tolist() == [0, 0, 0, 0]
    pts[5:] = 1.0  # points 0..4 at the origin, the rest identical and tied: residue class 0 wins
    idx = oracle.fps(pts, 3)   # (bit-reversed thread id 0), and inside it the lowest k that is not an origin point
    assert idx[1] == 1024
    pts[1024] = 0.0            # take that one out: class 0 still wins through k = 2048
    assert oracle.fps(pts, 3)[1] == 2048
    pts[2048] = 0.0            # class 0 exhausted: next is thread 512 (bit-reversed id 1)
    assert oracle.fps(pts, 3)[1] == 512


def test_plane_oracle_restatement_properties():
    """oracle.plane (the reference's plane branch with a seeded stand-in for open3d, PARITY UNPINNED):
    the pieces that ARE pinned by the reference's own text -- the < 30 pixel rule, the angle test's
    expression, the row layout -- and the codec's error bound through the full oracle pipeline."""
    from oracle import plane as oplane
    import rpcc_b200  # noqa: F401  (registers the package alias; synthetic frames are plain numpy)
    from rpcc_b200 import synthetic
    pts, g = synthetic.frame(7, "Velodyne64E")
    out = oracle.compress_frame(pts, "Velodyne64E", g, accuracy=0.02, model_method="plane", plane_seed=3)
    ri, seg, mp, lut = out["range_image"], out["seg_idx"], out["model_param"], out["lut"]
    cnt = np.bincount(seg.ravel(), minlength=mp.shape[0])
    is_plane = np.abs(mp[:, :3]).sum(1) > 0
    assert is_plane[0] and not is_plane[1]
    assert not is_plane[2:][cnt[2:] < 30].any()
    assert is_plane[2:].sum() > 20
    rec, _, seg2 = oracle.decompress_sections(out["sections"], "Velodyne64E", 0.02)
    assert np.array_equal(seg2, seg)
    assert float(np.abs(rec - ri)[ri > 0].max()) <= 0.02 + 1e-5
    # angle test: a plane facing the sensor passes, a grazing one is rejected, a NaN-poisoned one is kept
    idx = np.where(seg == int(np.argmax(cnt[2:]) + 2))
    s = lut[idx].astype(np.float64).mean(0)
    s /= np.linalg.norm(s)
    assert oplane.plane_angle_validation(lut, np.array([s[0], s[1], s[2], -10.0]), idx, 75)
    t = np.cross(s, [0, 0, 1.0])
    t /= np.linalg.norm(t)
    assert not oplane.plane_angle_validation(lut, np.array([t[0], t[1], t[2], -1.0]), idx, 75)
    # least-squares plane of exact coplanar points
    q = np.random.default_rng(0).normal(size=(50, 3))
    q[:, 2] = 0.25 * q[:, 0] - 0.5 * q[:, 1] + 3.0
    pl = oplane.get_plane_from_points(q)
    assert np.abs(q @ pl[:3] + pl[3]).max() < 1e-9 and abs(np.linalg.norm(pl[:3]) - 1) < 1e-12


def test_oracle_ransac_restatements_behave():
    """orc_ground_fit / orc_plane_models restate the PRODUCT's deterministic RANSACs (open3d cannot be pinned): on the
    CPU they are checked by what the codec guarantees -- a unit ground normal near the synthetic scene's true plane,
    reproducible, keyed by seed and frame; plane-model rows that are unit normals or point rows, a smaller stream than
    with point models and the error bound of the codec after decoding."""
    from rpcc_b200 import synthetic
    pts, g_true = synthetic.frame(77, "Velodyne64E")
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    ri = oracle.project(pts, H, W, hf, vmax, vmin)
    g = oracle.ground_fit(ri, lut)
    assert abs(float(np.linalg.norm(g[:3])) - 1.0) < 1e-5
    t = np.asarray(g_true, np.float64) * np.sign(g_true[2]) * np.sign(g[2])
    assert float(np.abs(g[:3] - t[:3]).max()) < 0.02 and abs(float(g[3] - t[3])) < 0.1
    assert oracle.ground_fit(ri, lut).tobytes() == g.tobytes()
    assert oracle.ground_fit(ri, lut, frame=1).tobytes() != g.tobytes() or oracle.ground_fit(ri, lut, seed=9).tobytes() != g.tobytes()
    point = oracle.compress_frame(pts, "Velodyne64E", g)
    plane = oracle.compress_frame(pts, "Velodyne64E", g, model_method="plane", plane_impl="device")
    mp = plane["model_param"]
    rows = mp[2:]
    is_plane = np.abs(rows[:, :3]).sum(1) > 0
    assert is_plane.sum() >= 10
    assert np.all(np.abs(np.linalg.norm(rows[is_plane, :3].astype(np.float64), axis=1) - 1.0) < 1e-5)
    assert np.array_equal(rows[~is_plane].view(np.uint32), point["model_param"][2:][~is_plane].view(np.uint32))
    assert len(oracle.write_rpcc(plane["sections"], "bzip2")) < len(oracle.write_rpcc(point["sections"], "bzip2"))
    rec, _, seg = oracle.decompress_sections(plane["sections"], "Velodyne64E", 0.02)
    assert np.array_equal(seg, plane["seg_idx"])
    valid = ri > 0
    assert float(np.abs(rec - ri)[valid].max()) <= 0.02 + 1e-5


def test_example_frame_with_fitted_ground_golden(example_points):
    """The reference's example frame with nothing injected: the oracle (ground RANSAC restatement included) must keep
    producing the committed bytes; tests/test_gpu_pipeline.py holds the device to the same hashes."""
    import hashlib
    import json
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "example_fitted.json")))
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    g = oracle.ground_fit(oracle.project(example_points, H, W, hf, vmax, vmin), lut)
    assert g.tobytes().hex() == gold["ground_f32_hex"]
    for name, kw in (("point", {}), ("plane", dict(model_method="plane", plane_impl="device"))):
        blob = oracle.write_rpcc(oracle.compress_frame(example_points, "Velodyne64E", g, **kw)["sections"], "bzip2")
        assert len(blob) == gold[name]["rpcc_bytes"] and hashlib.sha256(blob).hexdigest() == gold[name]["sha256"], name
