"""GPU parity tests of the drop-in plugin ops, the batched encoder/decoder and the L3 mirror,
against the oracle, the committed reference goldens and (when shipped) the reference's compiled code."""
import hashlib
import os

import numpy as np
import pytest

import oracle
from oracle import ref
from conftest import EXAMPLE_GROUND

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "example_golden.npz")
LIDARS = ["Velodyne64E", "Velodyne32E", "VelodyneVLP16"]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def R():
    import rpcc_b200
    return rpcc_b200


# ------------------------------------------------------------------------------------ plugin ops
def test_plugin_ops_match_reference_modules(R, example_points, gold):
    from rpcc_b200.plugin import (contour_utils_cpp, dataset_utils_cpp, feature_extractor_cpp, quantization_utils_cpp,
                                  segment_utils_cpp)
    cfg = R.LidarConfig("Velodyne64E")
    lut = cfg.transform_map()
    H, W = cfg.H, cfg.W
    ri = dataset_utils_cpp.point_cloud_to_range_image_even(example_points[:, :3], H, W, cfg.horizontal_FOV,
                                                           cfg.vertical_max, cfg.vertical_min)
    assert sha(ri) == str(gold["u_range_sha"])
    seg = gold["u_seg_u8"].astype(np.int64)       # what torch.max hands the reference: int64
    pm = segment_utils_cpp.point_modeling(ri[..., None], seg)
    assert pm.shape == (102,) and pm.tobytes() == oracle.point_modeling(ri, seg).tobytes()
    mp = gold["u_model_param"]
    pred = segment_utils_cpp.intra_predict(seg, mp.astype(np.float64), lut)   # f64 model: forcecast like pybind
    assert pred.shape == (H, W, 1) and sha(pred) == str(gold["u_pred_sha"])
    res = ri[..., None] - pred
    sym = quantization_utils_cpp.uniform_quantize(seg, res, 0.04)
    assert sym.dtype == np.int32 and np.array_equal(sym.astype(np.int16), gold["u_symbols"])
    feat, kp = feature_extractor_cpp.extract_features_with_segment(ri, seg, 3, 8, 4, 8, 6)
    assert np.array_equal(kp.astype(np.uint8), gold["n_key_points_u8"])
    feat_o, _ = oracle.extract_features(ri, seg)
    assert np.array_equal(feat.view(np.uint32), feat_o.view(np.uint32))
    acc = np.array([0.04] * 4) + np.array([0, 0.02, 0.04, 0.06])
    symn, sal = quantization_utils_cpp.nonuniform_quantize(seg, res, kp, np.array((30, 10, 3, 0)), acc, 2)
    assert np.array_equal(symn.astype(np.int16), gold["n_symbols"]) and np.array_equal(sal.astype(np.uint8), gold["n_salience"])
    contour, seq = contour_utils_cpp.extract_contour(seg)
    assert np.packbits(contour.astype(bool), axis=None).tobytes() == gold["u_contour_bits"].tobytes()
    assert np.array_equal(seq.astype(np.uint16), gold["u_idx_sequence"])
    assert np.array_equal(contour_utils_cpp.recover_map(contour, seq), seg)
    # the reference's only known-answer vector (utils/contour_utils.py:182-195), a 4x5 map
    c, s = contour_utils_cpp.extract_contour(gold["kat_idx_map"])
    assert np.array_equal(c, gold["kat_contour"]) and np.array_equal(s, gold["kat_seq"])
    assert np.array_equal(contour_utils_cpp.recover_map(c, s), gold["kat_idx_map"])


def test_plugin_ops_random_label_maps(R):
    """Ragged / adversarial inputs: random labels (many tiny runs), big symbols, empty clusters, tiny images."""
    from rpcc_b200.plugin import contour_utils_cpp, quantization_utils_cpp, segment_utils_cpp
    g = np.random.default_rng(3)
    for (H, W, K) in [(64, 2000, 102), (7, 333, 5), (1, 40, 3), (16, 1800, 254), (33, 1031, 60), (40, 31, 20),
                      (3, 1023, 102)]:
        seg = g.integers(0, K, (H, W)).astype(np.int32)
        seg[g.random((H, W)) < 0.3] = 1
        if K > 10:
            seg[seg == 7] = 8                      # an empty cluster -> NaN mean, as the reference
        ri = (g.random((H, W)) * 79 + 1).astype(np.float32)
        ri[seg == 1] = 0
        res = (g.standard_normal((H, W)) * 3).astype(np.float32)
        res.ravel()[:5] = [2000.0, -2000.0, 0.02, -0.02, 0.06]   # |q| > 32767: int32 result must not wrap
        pm = segment_utils_cpp.point_modeling(ri, seg)
        assert pm.tobytes() == oracle.point_modeling(ri, seg).tobytes()
        sym = quantization_utils_cpp.uniform_quantize(seg, res, 0.04)
        assert np.array_equal(sym, oracle.uniform_quantize(seg, res, 0.04))
        c, s = contour_utils_cpp.extract_contour(seg)
        co, so = oracle.extract_contour(seg)
        assert np.array_equal(c, co) and np.array_equal(s, so)
        assert np.array_equal(contour_utils_cpp.recover_map(c, s), seg)
    # exact means outside the fast path's [2^-5, 256) window: sequential double accumulation fallback
    seg = g.integers(2, 6, (8, 256)).astype(np.int32)
    ri = (g.random((8, 256)) * 1e-3 + 1e-6).astype(np.float32)
    ri[0, :10] = 300.0
    assert segment_utils_cpp.point_modeling(ri, seg).tobytes() == oracle.point_modeling(ri, seg).tobytes()


def test_plugin_fps_and_chamfer_drop_in(R):
    import torch
    from rpcc_b200.plugin import chamfer_3D, furthest_point_sampling_cuda as fps
    g = np.random.default_rng(9)
    xyz = torch.from_numpy(g.standard_normal((2, 3000, 3)).astype(np.float32)).cuda()
    idx = fps.furthest_point_sample(xyz, 50)
    assert idx.dtype == torch.int32 and idx.shape == (2, 50)
    for b in range(2):
        assert np.array_equal(idx[b].cpu().numpy(), oracle.fps(xyz[b].cpu().numpy(), 50))
    a = g.standard_normal((1, 2000, 3)).astype(np.float32)
    bb = (a[:, :1500] + g.standard_normal((1, 1500, 3)).astype(np.float32) * 0.01)
    bb[0, 10] = bb[0, 11]                        # duplicate target: first index must win
    d1, d2, i1, i2 = chamfer_3D.chamfer_3DDist()(torch.from_numpy(a).cuda(), torch.from_numpy(bb).cuda())
    od1, oi1 = oracle.chamfer_nn(a[0], bb[0], fma_mode=1)
    od2, oi2 = oracle.chamfer_nn(bb[0], a[0], fma_mode=1)
    assert np.array_equal(i1[0].cpu().numpy(), oi1) and np.array_equal(i2[0].cpu().numpy(), oi2)
    assert np.array_equal(d1[0].cpu().numpy(), od1) and np.array_equal(d2[0].cpu().numpy(), od2)
    if ref.have_cuda():
        ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(bb).cuda()
        rd1 = torch.zeros(1, 2000, device="cuda"); rd2 = torch.zeros(1, 1500, device="cuda")
        ri1 = torch.zeros(1, 2000, dtype=torch.int32, device="cuda"); ri2 = torch.zeros(1, 1500, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        assert ref.chamfer().ref_chamfer_launch(1, 2000, ta.data_ptr(), 1500, tb.data_ptr(), rd1.data_ptr(), ri1.data_ptr(),
                                                rd2.data_ptr(), ri2.data_ptr()) == 0
        assert torch.equal(rd1, d1) and torch.equal(rd2, d2) and torch.equal(ri1, i1) and torch.equal(ri2, i2)


# ------------------------------------------------------------------------------------ batched encoder
def test_encoder_example_frame_is_byte_exact(R, example_points, gold):
    """BASELINE configs[0]: example.bin, 64E, uniform, FPS, point modelling, accuracy 0.02, bzip2 ->
    the .rpcc bytes of the reference's own tools/compress.py pipeline (given the same ground model)."""
    from rpcc_b200.batch import BatchEncoder
    off = np.array([0, example_points.shape[0]], np.int64)
    with BatchEncoder("Velodyne64E", accuracy=0.02, max_batch=1, max_points=example_points.shape[0]) as enc:
        blobs = enc.compress(example_points, off, np.array([EXAMPLE_GROUND]))
        assert blobs[0] == gold["u_rpcc"].tobytes()
        assert len(blobs[0]) == 36460
    with BatchEncoder("Velodyne64E", accuracy=0.02, nonuniform=True, max_batch=1, max_points=example_points.shape[0]) as enc:
        out = enc.encode_host(example_points, off, np.array([EXAMPLE_GROUND]))
        sec = BatchEncoder.frame_sections(out, 0)
        assert sec["salience_level"] == gold["n_salience"].tobytes()
        assert sec["residual_quantized"] == gold["n_symbols"].tobytes()
        assert enc.compress(example_points, off, np.array([EXAMPLE_GROUND]))[0] == gold["n_rpcc"].tobytes()


@pytest.mark.parametrize("lidar,nonuniform", [("Velodyne64E", False), ("Velodyne64E", True), ("Velodyne32E", False),
                                               ("VelodyneVLP16", False), ("VelodyneVLP16", True)])
def test_encoder_batches_match_oracle_and_roundtrip(R, lidar, nonuniform):
    """Several chunks through the pipelined host path (max_batch 3, 8 frames: ragged last chunk), every
    section byte-exact against the oracle, then decoded again on the GPU: decode == oracle decode bit for
    bit, |range_rec - range| <= step/2 (+ level delta)."""
    import torch
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchDecoder, BatchEncoder
    seeds = list(range(20, 28))
    pts, off, grounds = synthetic.batch(seeds, lidar)
    with BatchEncoder(lidar, accuracy=0.02, nonuniform=nonuniform, max_batch=3) as enc:
        out = enc.encode_host(pts, off, grounds)
        secs = [BatchEncoder.frame_sections(out, b) for b in range(len(seeds))]
        blobs = enc.compress(pts, off, grounds)
    wants = []
    for b in range(len(seeds)):
        want = oracle.compress_frame(pts[off[b]:off[b + 1]], lidar, grounds[b], nonuniform=nonuniform)
        wants.append(want)
        for k, v in want["sections"].items():
            assert secs[b][k] == v, (lidar, b, k)
        assert blobs[b] == oracle.write_rpcc(want["sections"], "bzip2")
    dec = BatchDecoder(lidar, accuracy=0.02, nonuniform=nonuniform)
    d = dec.decode(blobs)
    for b in range(len(seeds)):
        rec, xyz, seg = oracle.decompress_sections(wants[b]["sections"], lidar, 0.02)
        assert np.array_equal(d["labels"][b].cpu().numpy().astype(np.int32), seg)
        assert np.array_equal(d["range"][b].cpu().numpy().view(np.uint32), rec.view(np.uint32))
        assert np.array_equal(d["xyz"][b].cpu().numpy().view(np.uint32), xyz.view(np.uint32))
        bound = 0.02 + (0.03 if nonuniform else 0.0)
        assert float(np.abs(rec - wants[b]["range_image"]).max()) <= bound + 1e-5


@pytest.mark.parametrize("lidar,accuracy,clusters,nonuniform", [
    ("Velodyne64E", 0.005, 20, False), ("Velodyne64E", 0.05, 250, False), ("Velodyne64E", 0.01, 37, True),
    ("VelodyneVLP16", 0.05, 250, True), ("Velodyne32E", 0.005, 64, False)])
def test_encoder_other_accuracies_and_cluster_counts(R, lidar, accuracy, clusters, nonuniform):
    """Off the default configuration: --accuracy 0.005 ... 0.05 and --cluster_num 20 ... 250 (the u8 label limit is 252):
    other centre counts per lane in the label kernel, other table sizes in the quantiser, int16 symbols near their
    range at the fine step.  Every section byte-exact against the oracle, ground injected and fitted on the device."""
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchEncoder
    from rpcc_b200.config import load_compressor_cfg
    cfg = load_compressor_cfg()
    cfg["cluster_num"] = clusters
    seeds = [40, 41, 42]
    pts, off, grounds = synthetic.batch(seeds, lidar)
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    with BatchEncoder(lidar, accuracy=accuracy, nonuniform=nonuniform, compressor_cfg=cfg, max_batch=2) as enc:
        for inject in (True, False):
            out = enc.encode_host(pts, off, grounds if inject else None)
            for b in range(len(seeds)):
                p = pts[off[b]:off[b + 1]]
                g = grounds[b] if inject else oracle.ground_fit(oracle.project(p, H, W, hf, vmax, vmin), lut)
                want = oracle.compress_frame(p, lidar, g, accuracy=accuracy, nonuniform=nonuniform, cluster_num=clusters)
                got = BatchEncoder.frame_sections(out, b)
                for k, v in want["sections"].items():
                    assert got[k] == v, (lidar, accuracy, clusters, nonuniform, inject, b, k)


@pytest.mark.parametrize("lidar,nonuniform,B", [("Velodyne64E", False, 700), ("VelodyneVLP16", True, 1300)])
def test_long_launch_every_cta_takes_several_frames(R, lidar, nonuniform, B):
    """BASELINE full size and beyond: one launch of B frames (more than the 2 x 148 CTAs of the one-CTA-per-frame
    kernels, so the FPS frame queue, the persistent projection teams and the ground fit all take several frames per
    CTA).  The B slots are copies of 6 distinct frames in a scrambled order: every copy must produce the bytes of its
    source frame, the distinct ones the oracle's, with the ground plane fitted on the device and injected alike."""
    import torch
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchEncoder
    nd = 6
    per = [synthetic.frame(60 + i, lidar) for i in range(nd)]
    order = [(i * 7 + i // 5) % nd for i in range(B)]
    pts = np.concatenate([per[k][0] for k in order], 0)
    off = np.cumsum([0] + [per[k][0].shape[0] for k in order]).astype(np.int64)
    grounds = np.stack([per[k][1] for k in order]).astype(np.float32)
    with BatchEncoder(lidar, accuracy=0.02, nonuniform=nonuniform, max_batch=B, max_points=pts.shape[0], host_chunk=B) as enc:
        out = enc.encode_host(pts, off, grounds)
        first = {}
        for b in range(B):
            sec = BatchEncoder.frame_sections(out, b)
            k = order[b]
            if k not in first:
                first[k] = sec
                want = oracle.compress_frame(per[k][0], lidar, per[k][1], nonuniform=nonuniform)["sections"]
                for name, v in want.items():
                    assert sec[name] == v, (lidar, b, name)
            else:
                assert sec == first[k], (lidar, b, k)
        # device-fitted ground: deterministic per frame content + position-independent except for the RANSAC key
        d_pts, d_off = torch.from_numpy(pts).cuda(), torch.from_numpy(off).cuda()
        enc.encode_device(0, d_pts, d_off, B, None)
        enc.sync()
        sb = enc.device_buffer(0, "sym_base", (B + 1,), torch.int64).cpu().numpy()
        sym1 = enc.device_buffer(0, "symbols", (int(sb[-1]),), torch.int16).cpu().numpy().copy()
        g1 = enc.device_buffer(0, "ground", (B, 4), torch.float32).cpu().numpy().copy()
        enc.encode_device(0, d_pts, d_off, B, None)
        enc.sync()
        sb2 = enc.device_buffer(0, "sym_base", (B + 1,), torch.int64).cpu().numpy()
        assert np.array_equal(sb, sb2)
        assert np.array_equal(sym1, enc.device_buffer(0, "symbols", (int(sb[-1]),), torch.int16).cpu().numpy())
        assert np.array_equal(g1.view(np.uint32), enc.device_buffer(0, "ground", (B, 4), torch.float32).cpu().numpy().view(np.uint32))
        assert np.isfinite(g1).all() and (np.abs(np.linalg.norm(g1[:, :3], axis=1) - 1.0) < 1e-4).all()


@pytest.mark.parametrize("lidar", ["Velodyne64E", "VelodyneVLP16"])
def test_encoder_with_device_ground_is_byte_exact_against_the_oracle(R, lidar):
    """No ground model injected anywhere: the device fits the plane (keyed by the frame's index within the call, across
    the pipeline stages of encode_host) and the oracle fits its restatement of the same RANSAC -- every section of
    every frame must still come out byte for byte."""
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchEncoder
    seeds = list(range(90, 97))
    pts, off, _ = synthetic.batch(seeds, lidar)
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    with BatchEncoder(lidar, accuracy=0.02, max_batch=3, host_chunk=3) as enc:
        out = enc.encode_host(pts, off, None)
        for b in range(len(seeds)):
            p = pts[off[b]:off[b + 1]]
            g = oracle.ground_fit(oracle.project(p, H, W, hf, vmax, vmin), lut, seed=0x5EED)
            want = oracle.compress_frame(p, lidar, g)["sections"]
            got = BatchEncoder.frame_sections(out, b)
            for k, v in want.items():
                assert got[k] == v, (lidar, b, k)


@pytest.mark.parametrize("method", ["point", "plane"])
def test_example_frame_with_fitted_ground_matches_the_golden_hash(R, example_points, method):
    """BASELINE configs[0] with nothing injected: example.bin through the batched encoder (device ground fit, host
    bzip2) must give the committed .rpcc bytes of tests/golden/example_fitted.json (written by the oracle)."""
    import json
    from rpcc_b200.batch import BatchEncoder
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "example_fitted.json")))
    off = np.array([0, example_points.shape[0]], np.int64)
    with BatchEncoder("Velodyne64E", accuracy=0.02, max_batch=1, max_points=example_points.shape[0], model_method=method) as enc:
        blob = enc.compress(example_points, off, None)[0]
    assert len(blob) == gold[method]["rpcc_bytes"]
    assert hashlib.sha256(blob).hexdigest() == gold[method]["sha256"]


def test_encoder_device_path_and_ground_fit(R):
    """Device-resident inputs, ground fitted on the device: deterministic, close to the true plane, and the
    rest of the chain is byte-exact against the oracle GIVEN that fitted plane."""
    import torch
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchEncoder
    pts, off, grounds = synthetic.batch([40, 41, 42, 43], "Velodyne64E")
    d_pts, d_off = torch.from_numpy(pts).cuda(), torch.from_numpy(off).cuda()
    with BatchEncoder("Velodyne64E", accuracy=0.02, max_batch=4) as enc:
        fitted = []
        for rep in range(2):
            # same absolute frame keys on both passes: the plane must be bit-reproducible
            enc2 = BatchEncoder("Velodyne64E", accuracy=0.02, max_batch=4)
            enc2.encode_device(0, d_pts, d_off, 4, None)
            enc2.sync()
            fitted.append(enc2.device_buffer(0, "ground", (4, 4), torch.float32).cpu().numpy().copy())
            if rep == 1:
                res = enc2.device_buffer(0, "results", (4, 4), torch.int32).cpu().numpy().view(np.uint32)
                model = enc2.device_buffer(0, "model", (4, 102, 4), torch.float32).cpu().numpy()
                sym_base = enc2.device_buffer(0, "sym_base", (5,), torch.int64).cpu().numpy()
                symbols = enc2.device_buffer(0, "symbols", (int(sym_base[-1]),), torch.int16).cpu().numpy()
            enc2.close()
        assert np.array_equal(fitted[0], fitted[1])
        for b in range(4):
            g = fitted[0][b].astype(np.float64)
            t = grounds[b] * np.sign(grounds[b][2]) * np.sign(g[2])
            assert abs(np.linalg.norm(g[:3]) - 1) < 1e-5
            assert np.abs(g[:3] - t[:3]).max() < 2e-2 and abs(g[3] - t[3]) < 0.1, (g, t)
            want = oracle.compress_frame(pts[off[b]:off[b + 1]], "Velodyne64E", fitted[0][b])
            assert model[b, :int(res[b, 2])].tobytes() == want["sections"]["plane_param"]
            assert symbols[sym_base[b]:sym_base[b + 1]].tobytes() == want["sections"]["residual_quantized"]


def test_degenerate_frames_in_a_batch(R):
    """An empty frame, a five-point frame and a frame whose points all lie on the ground (every pixel masked: FPS runs on
    a cloud of identical origin points and the tie rule alone picks the seeds) between two ordinary frames: every section
    equals the oracle's, and the streams decode."""
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchDecoder, BatchEncoder
    lidar = "VelodyneVLP16"
    a, ga = synthetic.frame(90, lidar)
    b, gb = synthetic.frame(91, lidar)
    flat = a[np.abs(a[:, :3] @ ga[:3] + ga[3]) < 0.05][:4000]          # ground returns only
    frames = [a, np.zeros((0, 4), np.float32), b[:5].copy(), flat, b]
    grounds = np.stack([ga, ga, gb, ga, gb])
    pts = np.concatenate(frames, 0)
    off = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int64)
    with BatchEncoder(lidar, accuracy=0.02, max_batch=8, max_points=max(pts.shape[0], 1), host_chunk=2) as enc:
        out = enc.encode_host(pts, off, grounds)
        for i, f in enumerate(frames):
            want = oracle.compress_frame(f, lidar, grounds[i])["sections"]
            got = BatchEncoder.frame_sections(out, i)
            for k in want:
                assert got[k] == want[k], (i, k)
        blobs = enc.compress(pts, off, grounds)
    d = BatchDecoder(lidar, accuracy=0.02).decode(blobs, want_xyz=False, want_points=True)
    assert d["points"][1].shape[0] == 0 and d["points"][2].shape[0] <= 5 and d["points"][0].shape[0] > 10000


def test_encode_host_is_independent_of_the_pipeline_chunking(R):
    """encode_host cuts a call into host_chunk-frame pipeline stages; every section (including the ground
    plane fitted on the device, keyed by the frame's index within the call) must not depend on the cut."""
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchEncoder
    pts, off, _ = synthetic.batch(list(range(60, 67)), "Velodyne64E")
    got = []
    for chunk in (7, 2, 3):
        with BatchEncoder("Velodyne64E", accuracy=0.02, max_batch=7, host_chunk=chunk) as enc:
            out = enc.encode_host(pts, off, None)
            got.append([BatchEncoder.frame_sections(out, b) for b in range(7)])
    assert got[0] == got[1] == got[2]


# ------------------------------------------------------------------------------------ L3 mirror + tools
def test_l3_mirror_single_frame_compress_decompress_eval(R, example_points, gold, tmp_path):
    """The reference's single-frame flow (tools/compress.py --eval, tools/decompress.py) through the mirrored
    classes: same .rpcc bytes, same reconstruction, chamfer within 1e-5 relative of the oracle's."""
    from rpcc_b200.tools import compress as tc, decompress as td
    inp = os.path.join(os.path.dirname(__file__), "golden", "example.bin")
    outp = str(tmp_path / "example.rpcc")
    args = tc.base_parser(single=True).parse_args(["--input", inp, "--output", outp, "--lidar", "Velodyne64E", "--eval"])
    r = tc.compress(args, ground_model=np.array(EXAMPLE_GROUND))
    assert open(outp, "rb").read() == gold["u_rpcc"].tobytes()
    assert r["max_depth_error"] <= 0.02 + 1e-5
    binp = str(tmp_path / "rec.bin")
    p = td.base_parser(single=True)
    p.add_argument("--original_point_cloud", default=None)
    td.decompress(p.parse_args(["--input", outp, "--output", binp, "--lidar", "Velodyne64E"]))
    rec = np.fromfile(binp, np.float32).reshape(-1, 4)
    assert rec.shape[0] == 94053 and np.all(rec[:, 3] == 0)
    # chamfer against a CPU brute-force on a subsample (tolerance stated by north_star: 1e-5 relative)
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    ri = oracle.project(example_points, H, W, hf, vmax, vmin)
    orig = (ri[..., None] * lut).reshape(-1, 3)
    orig = orig[np.sum(orig, -1) != 0]
    from rpcc_b200.evaluate_metrics import calc_chamfer_distance
    res = calc_chamfer_distance(orig, rec[:, :3], out=False)
    sub = np.arange(0, orig.shape[0], 97)
    od, oi = oracle.chamfer_nn(orig[sub], rec[:, :3], fma_mode=1)
    assert np.array_equal(res["chamfer_dist_info"]["idx1"][sub], oi)
    assert np.array_equal(res["chamfer_dist_info"]["dist1"][sub], od)
    d1 = res["chamfer_dist_info"]["dist1"].astype(np.float64)
    assert abs(res["cd1"] - np.sqrt(d1).mean()) <= 1e-5 * res["cd1"]
    assert 0.0 < res["mean"] < 0.02 and res["f_score"] > 0.95


def test_segment_mirror_signature(R, example_points, gold):
    from rpcc_b200.dataset import build_dataset
    from rpcc_b200.segment_utils import PointCloudSegment
    ds = build_dataset(lidar_type="Velodyne64E")
    pc, ri, orig = ds.load_range_image_points_from_file(os.path.join(os.path.dirname(__file__), "golden", "example.bin"))
    assert pc.shape == (64, 2000, 3) and ri.shape == (64, 2000, 1)
    assert np.array_equal(pc, ri * ds.transform_map)
    seg_cfg = {"segment_method": "FPS", "ground_vertical_threshold": 0.1, "cluster_num": 100, "DBSCAN_eps": 1.5}
    seg, gm = PointCloudSegment(ds.transform_map).segment(pc, ri, seg_cfg, ground_model=np.array(EXAMPLE_GROUND))
    assert seg.dtype == np.int64 and gm.dtype == np.float32
    assert np.array_equal(seg.astype(np.uint8), gold["u_seg_u8"])
    seg2, gm2 = PointCloudSegment(ds.transform_map).segment(pc, ri, seg_cfg)     # device RANSAC ground
    assert abs(np.linalg.norm(gm2[:3]) - 1) < 1e-5 and abs(abs(gm2[2]) - 1) < 0.02 and 1.5 < abs(gm2[3]) < 2.0
