"""DBSCAN segmentation on the GPU (csrc/dbscan.cu) against oracle.dbscan, this project's definition restated in numpy
and scipy (DESIGN.md §4): labels bit for bit, `.rpcc` bytes through BatchEncoder, the decoder's round trip, and the
independence of the bytes from batching and from the tool that wrote them."""
import os

import numpy as np
import pytest

import oracle
from oracle import dbscan

pytestmark = pytest.mark.gpu
THR = 0.1


def _geometry(lidar):
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    return H, W, hf, vmax, vmin, oracle.transform_map(H, W, hf, vmax, vmin)


def _device(ri, grounds, lidar, eps, min_points, cluster_num=100):
    """ri (B,H,W) f32, grounds (B,4) -> (labels (B,H,W) u8, exhaustive-scan counts (B,), clusters found (B,))."""
    import torch
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    H, W, hf, vmax, vmin, lut = _geometry(lidar)
    B = ri.shape[0]
    dev = torch.device("cuda", 0)
    r = torch.from_numpy(np.ascontiguousarray(ri, np.float32)).to(dev)
    lt = torch.from_numpy(lut).to(dev)
    g = torch.from_numpy(np.ascontiguousarray(grounds, np.float32)).to(dev)
    lab = torch.empty((B, H * W), dtype=torch.uint8, device=dev)
    ws = torch.empty((_lib.lib().rpcc_dbscan_workspace_bytes(B, H, W),), dtype=torch.uint8, device=dev)
    check(_lib.lib().rpcc_dbscan_segment_batch(ptr(r), ptr(lt), ptr(g), B, H, W, hf, vmax, vmin, float(eps),
                                               int(min_points), int(cluster_num), THR, ptr(lab), ptr(ws), None))
    torch.cuda.synchronize()
    cnt = ws[:8 * B].cpu().numpy().view(np.uint32)
    return lab.cpu().numpy().reshape(B, H, W), cnt[:B].copy(), cnt[B:2 * B].copy()


def _frames(lidar, seeds):
    from rpcc_b200 import synthetic
    H, W, hf, vmax, vmin, lut = _geometry(lidar)
    out = []
    for s in seeds:
        p, g = synthetic.frame(s, lidar)
        out.append((p, g, oracle.project(p, H, W, hf, vmax, vmin)))
    return out


@pytest.mark.parametrize("lidar", ["Velodyne64E", "Velodyne32E", "VelodyneVLP16"])
@pytest.mark.parametrize("eps", [0.5, 1.5])
def test_labels_equal_the_oracle(lidar, eps):
    H, W, hf, vmax, vmin, lut = _geometry(lidar)
    (p, g, ri), = _frames(lidar, [11])
    G = dbscan.graph(ri, lut, g, eps, THR)
    for min_points in (1, 10):
        want, found = dbscan.labels_from_graph(G, min_points, 100)
        got, exh, clusters = _device(ri[None], g[None], lidar, eps, min_points)
        assert np.array_equal(got[0].reshape(-1), want), (lidar, eps, min_points,
                                                           int((got[0].reshape(-1) != want).sum()))
        assert clusters[0] == found
        if eps < 1.5:
            assert exh[0] == 0                 # synthetic points are >= 1.5 m away: the window settles every query


def test_several_frames_in_one_launch_and_small_cluster_num():
    lidar = "VelodyneVLP16"
    H, W, hf, vmax, vmin, lut = _geometry(lidar)
    fr = _frames(lidar, [21, 22, 23, 24, 25])
    ri = np.stack([f[2] for f in fr])
    gs = np.stack([f[1] for f in fr])
    for cluster_num, min_points in ((100, 4), (3, 10), (1, 1)):
        got, _, clusters = _device(ri, gs, lidar, 0.5, min_points, cluster_num)
        for b in range(len(fr)):
            want, found = dbscan.labels_from_graph(dbscan.graph(ri[b], lut, gs[b], 0.5, THR), min_points, cluster_num)
            assert np.array_equal(got[b].reshape(-1), want), (b, cluster_num, min_points)
            assert clusters[b] == found
        # each frame alone gives the same labels as in the batch
        alone, _, _ = _device(ri[2:3], gs[2:3], lidar, 0.5, min_points, cluster_num)
        assert np.array_equal(alone[0], got[2])


def test_points_nearer_than_eps_and_negative_ranges_take_the_exhaustive_scan():
    lidar = "VelodyneVLP16"
    H, W, hf, vmax, vmin, lut = _geometry(lidar)
    (p, g, ri), (p2, g2, ri2) = _frames(lidar, [31, 32])
    near = ri.copy()
    near[7:10, 400:460] = np.float32(1.0) + np.arange(60, dtype=np.float32) * np.float32(0.005)  # an object at 1.0-1.3 m
    neg = ri2.copy()
    neg[12, 5] = np.float32(-3.0)                           # a point behind the sensor: the whole frame is exhaustive
    got, exh, _ = _device(np.stack([near, neg]), np.stack([g, g2]), lidar, 1.5, 10)
    for b, (r, gg) in enumerate(((near, g), (neg, g2))):
        want = dbscan.segment(r, lut, gg, 1.5, 10, 100, THR)
        assert np.array_equal(got[b], want), b
    assert exh[0] >= 180                                    # at least the 180 pixels nearer than eps
    pts, mask = dbscan.points_mask(neg, lut, g2, THR)
    assert exh[1] == mask.sum()


def test_bad_arguments_are_refused():
    from rpcc_b200 import _lib
    H, W, hf, vmax, vmin, lut = _geometry("VelodyneVLP16")
    ri = np.zeros((H, W), np.float32)
    seg = np.empty((H, W), np.int32)
    g = np.array([0, 0, 1, 1.7], np.float32)
    L = _lib.lib()
    for eps, mp in ((0.0, 10), (-1.0, 10), (1.5, 0)):
        rc = L.rpcc_op_segment_dbscan(_lib.ptr(ri), _lib.ptr(lut), _lib.ptr(g), H, W, hf, vmax, vmin, eps, mp, 100, THR,
                                      _lib.ptr(seg), None, None)
        assert rc == -1, (eps, mp)                          # RPCC_ERR_ARG


def _cfg(**kw):
    from rpcc_b200.config import load_compressor_cfg
    cfg = load_compressor_cfg()
    cfg["segment_method"] = "DBSCAN"
    cfg.update(kw)
    return cfg


@pytest.fixture(scope="module")
def coded():
    """Two VLP16 frames and one 32E frame with the oracle's DBSCAN labels (eps 1.5, min_points 10, injected ground)."""
    out = {}
    for lidar, seeds in (("VelodyneVLP16", [41, 42]), ("Velodyne32E", [43])):
        H, W, hf, vmax, vmin, lut = _geometry(lidar)
        out[lidar] = [(p, g, dbscan.segment(ri, lut, g, 1.5, 10, 100, THR)) for p, g, ri in _frames(lidar, seeds)]
    return out


@pytest.mark.parametrize("model_method", ["point", "plane"])
@pytest.mark.parametrize("nonuniform", [False, True])
def test_encoder_bytes_equal_the_oracle_pipeline(coded, model_method, nonuniform):
    from rpcc_b200.batch import BatchEncoder
    for lidar, frames in coded.items():
        pts = np.concatenate([f[0] for f in frames])
        off = np.concatenate([[0], np.cumsum([f[0].shape[0] for f in frames])]).astype(np.int64)
        gs = np.stack([f[1] for f in frames])
        with BatchEncoder(lidar, accuracy=0.02, nonuniform=nonuniform, compressor_cfg=_cfg(), max_batch=len(frames),
                          max_points=pts.shape[0], model_method=model_method) as enc:
            out = enc.encode_host(pts, off, gs)
            for b, (p, g, seg) in enumerate(frames):
                want = dbscan.compress_frame(p, lidar, g, seg, nonuniform=nonuniform,
                                             model_method=model_method)["sections"]
                got = BatchEncoder.frame_sections(out, b)
                for k in want:
                    assert got[k] == want[k], (lidar, b, k)


@pytest.mark.parametrize("nonuniform", [False, True])
def test_decoder_round_trip(coded, nonuniform):
    from rpcc_b200.batch import BatchDecoder, BatchEncoder
    lidar = "VelodyneVLP16"
    frames = coded[lidar]
    pts = np.concatenate([f[0] for f in frames])
    off = np.concatenate([[0], np.cumsum([f[0].shape[0] for f in frames])]).astype(np.int64)
    gs = np.stack([f[1] for f in frames])
    H, W, hf, vmax, vmin, lut = _geometry(lidar)
    acc = 0.02
    with BatchEncoder(lidar, accuracy=acc, nonuniform=nonuniform, compressor_cfg=_cfg(), max_batch=len(frames),
                      max_points=pts.shape[0]) as enc:
        blobs = enc.compress(pts, off, gs)
    with BatchDecoder(lidar, accuracy=acc, nonuniform=nonuniform, compressor_cfg=_cfg()) as dec:
        rec = dec.decode(blobs)
        rng, labs = rec["range"].cpu().numpy(), rec["labels"].cpu().numpy()
    bound = acc + (0.06 if nonuniform else 0.0) + 1e-5
    for b, (p, g, seg) in enumerate(frames):
        ri = oracle.project(p, H, W, hf, vmax, vmin)
        assert np.abs(rng[b] - ri).max() <= bound
        assert np.array_equal(labs[b], seg)


def _write_bins(tmp, lidar, seeds):
    from rpcc_b200 import synthetic
    names = []
    for i, s in enumerate(seeds):
        p, _ = synthetic.frame(s, lidar)
        path = "%s/in/%06d.bin" % (tmp, i)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        p.tofile(path)
        names.append(path)
    lst = tmp + "/list.txt"
    open(lst, "w").write("\n".join(names) + "\n")
    return names, lst


def test_tools_write_identical_files_independent_of_batching(tmp_path, capsys):
    from rpcc_b200.tools import compress, compress_datalist, decompress
    from rpcc_b200.tools.common import base_parser
    from rpcc_b200.tools.compress_datalist import output_path_for
    lidar = "VelodyneVLP16"
    root = str(tmp_path)
    names, lst = _write_bins(root, lidar, [51, 52, 53, 51, 54])    # frame 51 twice, at positions 0 and 3
    flags = ["--lidar", lidar, "--segment_method", "DBSCAN", "--DBSCAN_eps", "1.5", "--DBSCAN_min_points", "10"]
    outs = {}
    for batch in (2, 5):
        a = base_parser(single=False).parse_args(["--datalist", lst, "--output_dir", "%s/o%d" % (root, batch),
                                                  "--workers", "2", "--batch", str(batch)] + flags)
        compress_datalist.compress(a)
        outs[batch] = [open(output_path_for("%s/o%d" % (root, batch), n), "rb").read() for n in names]
    assert outs[2] == outs[5]
    assert outs[2][0] == outs[2][3]
    for i in (0, 2):
        single = "%s/single_%d.rpcc" % (root, i)
        compress.compress(base_parser(single=True).parse_args(["--input", names[i], "--output", single] + flags))
        assert open(single, "rb").read() == outs[2][i], i
    # the oracle's bytes, with the ground plane the device fits (restated by oracle.ground_fit, frame key 0)
    H, W, hf, vmax, vmin, lut = _geometry(lidar)
    p = np.fromfile(names[1], np.float32).reshape(-1, 4)
    ri = oracle.project(p, H, W, hf, vmax, vmin)
    g = oracle.ground_fit(ri, lut)
    seg = dbscan.segment(ri, lut, g, 1.5, 10, 100, THR)
    want = oracle.write_rpcc(dbscan.compress_frame(p, lidar, g, seg)["sections"])
    assert outs[2][1] == want
    # decoding needs nothing new: decompress.py turns the file back into points within the accuracy
    rec = root + "/rec.bin"
    res = decompress.main(["--input", output_path_for(root + "/o2", names[1]), "--output", rec, "--eval",
                           "--original_point_cloud", names[1]] + flags)
    assert res["max_depth_error"] <= 0.02 + 1e-5
    assert os.path.getsize(rec) > 0
    capsys.readouterr()
