"""Bit-exact encode and decode against the oracle at range-image shapes no reference lidar has.

The three lidars of the reference (64 x 2000, 32 x 2250, 16 x 1800) share every property the kernels choose a code path
by: W >= 1024, H*W a multiple of 32 and of 16 * 8 bits, far from the encoder's 1024-pixel minimum and the FPS's
131 072-pixel capacity.  A sensor described by a lidar yaml or a LidarConfig can have any H >= 2, W >= 1 with
1024 <= H*W <= 131 072, and there the quantiser, the label decoder, the key-point sort, the window searches and the
tile loops take branches the lidars never reach.  SHAPES lists one image per such branch with the reason beside it;
test_shape_table_reaches_every_branch recomputes each reason from H and W, so that an edit cannot empty the table of
its purpose.  The GPU tests run three synthetic frames of each shape per launch through the encoder, the decoder, the
intensity stages and the window stages, and compare every output with the oracle bit for bit."""
import functools

import numpy as np
import pytest

import oracle
from oracle import dbscan
from oracle import intensity as oi

TILE = 1024            # RPCC_TILE: pixels per rank tile of the quantiser, the label decoder and the points writer
FPS_CAPACITY = 131072  # pixels the FPS rounds keep on chip
WINDOW_HALF = 48       # kEvR (window.cuh): the largest window half-width of the eval / normals / DBSCAN searches
THR = 0.1
SEEDS = (0, 1, 2)


def _keypoint_alloc(W, region=3, segments=8):
    """N of rpcc_keypoints_salience_batch: the per-segment sort allocation, a power of two >= (W - 2 region) / segments."""
    per_max = max((W - 2 * region) // segments, 1)
    N = 2
    while N < per_max:
        N <<= 1
    return N


# name -> predicate of (H, W, hfov_deg): the shape-selected branches (kernel: condition)
BRANCHES = {
    "encoder minimum (H*W = 1024, one tile)": lambda H, W, f: H * W == TILE,
    "quantiser narrow kernel with H*W % 16 == 0 (not staged although it could be)":
        lambda H, W, f: W < TILE and H * W % 16 == 0,
    "row starts by p % W (W < 32): up to two per 32-pixel slice": lambda H, W, f: W < 32,
    "key points: shared-memory network for N < 32": lambda H, W, f: _keypoint_alloc(W) < 32,
    "window wider than the ring (2 dc + 1 >= W reachable)": lambda H, W, f: W <= 2 * WINDOW_HALF + 1,
    "FPS staging: H*W % 4 != 0": lambda H, W, f: H * W % 4 != 0,
    "contour words: cbytes % 4 == 3": lambda H, W, f: (H * W + 7) // 8 % 4 == 3,
    "contour words: cbytes % 4 == 1": lambda H, W, f: (H * W + 7) // 8 % 4 == 1,
    "last tile partial and not whole 32-pixel slices": lambda H, W, f: H * W % 32 != 0,
    "W = 32: first width of the next_row walk": lambda H, W, f: W == 32,
    "W = 33": lambda H, W, f: W == 33,
    "widest narrow image: row starts at pixels 0 and W of tile 0": lambda H, W, f: W == TILE - 1,
    "narrowest WIDE image: a row start at every tile start, staged":
        lambda H, W, f: W == TILE and H * W % 16 == 0,
    "WIDE but unstaged: H*W % 16 != 0": lambda H, W, f: W >= TILE and H * W % 16 != 0,
    "row window clipped on both sides: H <= 3": lambda H, W, f: H <= 3,
    "FPS capacity: 131072 pixels, Q = 2, T = 128":
        lambda H, W, f: H * W == FPS_CAPACITY and (H * W + 63) // 64 > 1024 and (H * W + TILE - 1) // TILE == 128,
    "key points: shared-memory network for per > 512 (N = 1024)": lambda H, W, f: _keypoint_alloc(W) > 512,
    "not 360 degrees: points outside the FOV": lambda H, W, f: f != 360,
}

# (H, W, hfov_deg, reasons).  Sensor: +10 / -25 degrees.
SHAPES = [
    (2, 512, 360, ["encoder minimum (H*W = 1024, one tile)", "row window clipped on both sides: H <= 3",
                   "quantiser narrow kernel with H*W % 16 == 0 (not staged although it could be)"]),
    (64, 31, 360, ["row starts by p % W (W < 32): up to two per 32-pixel slice",
                   "key points: shared-memory network for N < 32", "window wider than the ring (2 dc + 1 >= W reachable)"]),
    (37, 29, 360, ["row starts by p % W (W < 32): up to two per 32-pixel slice", "FPS staging: H*W % 4 != 0",
                   "contour words: cbytes % 4 == 3", "last tile partial and not whole 32-pixel slices"]),
    (33, 32, 360, ["W = 32: first width of the next_row walk"]),
    (32, 33, 360, ["W = 33"]),
    (3, 1023, 360, ["widest narrow image: row starts at pixels 0 and W of tile 0", "row window clipped on both sides: H <= 3"]),
    (3, 1024, 360, ["narrowest WIDE image: a row start at every tile start, staged",
                    "row window clipped on both sides: H <= 3"]),
    (4, 1025, 360, ["WIDE but unstaged: H*W % 16 != 0", "contour words: cbytes % 4 == 1", "last tile partial and not whole 32-pixel slices"]),
    (128, 1024, 360, ["FPS capacity: 131072 pixels, Q = 2, T = 128"]),
    (16, 8192, 360, ["FPS capacity: 131072 pixels, Q = 2, T = 128",
                     "key points: shared-memory network for per > 512 (N = 1024)"]),
    (20, 700, 120, ["not 360 degrees: points outside the FOV"]),
]
EMPTY_FRAME_AT = {(37, 29): 1, (128, 1024): 3}     # shape -> position of an empty frame in the launch
PLANE_SHAPES = [(2, 512), (64, 31), (4, 1025), (128, 1024)]
DBSCAN_MAX_PIXELS = 4100                            # the oracle's DBSCAN at eps 1.5 needs tens of GB at 131072 pixels

ALL = [s[:3] for s in SHAPES]
FULL = [s for s in ALL if s[2] == 360]


def _id(s):
    return "%dx%d" % s[:2] + ("" if s[2] == 360 else "_%ddeg" % s[2])


def _cfg(shape):
    from rpcc_b200 import LidarConfig
    H, W, fov = shape
    return LidarConfig(hfov_deg=float(fov), vmax_deg=10.0, vmin_deg=-25.0, H=H, W=W)


@functools.lru_cache(maxsize=None)
def _frames(shape, empty=True):
    """-> (points per frame, ground per frame): the synthetic frames of the shape, with an empty frame where
    EMPTY_FRAME_AT puts one (its ground is its neighbour's)."""
    from rpcc_b200 import synthetic
    cfg = _cfg(shape)
    fr = []
    with np.errstate(invalid="ignore"):
        fr = [synthetic.frame(s, cfg) for s in SEEDS]
    pos = EMPTY_FRAME_AT.get(shape[:2]) if empty else None
    if pos is not None:
        fr.insert(pos, (np.zeros((0, 4), np.float32), fr[min(pos, len(fr) - 1)][1]))
    return [f[0] for f in fr], [np.asarray(f[1], np.float64) for f in fr]


def _geometry(shape):
    H, W, hf, vmax, vmin = oracle.lidar_params(_cfg(shape))
    return H, W, hf, vmax, vmin, oracle.transform_map(H, W, hf, vmax, vmin)


# ----------------------------------------------------------------------------------------------- the table (no GPU)
def test_shape_table_reaches_every_branch():
    rows = {}
    for H, W, fov, reasons in SHAPES:
        assert H >= 2 and W >= 1 and TILE <= H * W <= FPS_CAPACITY, (H, W)
        assert reasons, (H, W)
        for r in reasons:
            assert BRANCHES[r](H, W, fov), (H, W, r)
            rows.setdefault(r, []).append((H, W))
    assert set(rows) == set(BRANCHES), set(BRANCHES) - set(rows)
    # the lidars of the reference reach none of them
    from rpcc_b200.lidar import LIDAR_TABLE
    for name in ("Velodyne64E", "Velodyne32E", "VelodyneVLP16"):
        fov, _, _, H, W = LIDAR_TABLE[name]
        assert not any(p(H, W, fov) for p in BRANCHES.values()), name
    assert set(EMPTY_FRAME_AT) <= {s[:2] for s in ALL} and set(PLANE_SHAPES) <= {s[:2] for s in ALL}


def test_wide_rows_reach_the_large_keypoint_sort():
    """At 16 x 8192 some row of every frame holds more than 8 * 512 + 6 non-ground pixels: per > 512."""
    shape = (16, 8192, 360)
    H, W, hf, vmax, vmin, lut = _geometry(shape)
    pts, grounds = _frames(shape, empty=False)
    for p, g in zip(pts, grounds):
        seg, _, _ = oracle.segment(oracle.project(p, H, W, hf, vmax, vmin), lut, g)
        per = ((seg >= 2).sum(1) - 2 * 3) // 8
        assert per.max() > 512, per.max()


@pytest.mark.parametrize("shape", ALL, ids=_id)
def test_oracle_round_trips_every_shape(shape):
    """The oracle itself at the shape: decompress_sections gives back the labels, and the ranges within the bound."""
    pts, grounds = _frames(shape)
    for nonuniform in (False, True):
        for p, g in zip(pts, grounds):
            out = oracle.compress_frame(p, _cfg(shape), g, nonuniform=nonuniform)
            rec, _, seg = oracle.decompress_sections(out["sections"], _cfg(shape), 0.02)
            assert np.array_equal(seg, out["seg_idx"])
            ri = out["range_image"]
            bound = np.float32(0.02 + (0.03 if nonuniform else 0.0)) + np.spacing(np.abs(ri))
            assert np.all(np.abs(rec - ri) <= bound), (shape, nonuniform)


# ----------------------------------------------------------------------------------------------- GPU helpers
def _compressor_cfg(segment_method="FPS"):
    from rpcc_b200.config import load_compressor_cfg
    cfg = load_compressor_cfg()
    cfg["segment_method"] = segment_method
    return cfg


def _want(coding, shape, p, g, lut):
    """The oracle's frame for one coding -> dict(sections, seg_idx, range_image, key_point_map?)."""
    cfg = _cfg(shape)
    if coding == "dbscan":
        H, W, hf, vmax, vmin = oracle.lidar_params(cfg)
        c = _compressor_cfg("DBSCAN")
        ri = oracle.project(p, H, W, hf, vmax, vmin)
        seg = dbscan.segment(ri, lut, g, c["DBSCAN_eps"], c["DBSCAN_min_points"], c["cluster_num"], THR)
        out = dbscan.compress_frame(p, cfg, g, seg)
        out["range_image"] = ri
        return out
    kw = dict(nonuniform=coding == "nonuniform")
    if coding == "plane":
        kw.update(model_method="plane", plane_impl="device")
    return oracle.compress_frame(p, cfg, g, **kw)


def _tile0_row_start_pairs(segs, W):
    """Row starts inside tile 0 other than pixel 0 whose left neighbour has the same label, over the frames: only there
    does the contour bit come from the row start alone."""
    n = 0
    for seg in segs:
        flat = seg.reshape(-1)
        starts = np.arange(W, min(TILE, flat.size), W)
        n += int(np.sum(flat[starts] == flat[starts - 1]))
    return n


def _encode_decode(coding, shape):
    """Every frame of the shape through BatchEncoder with the ground injected and fitted on the device: every section
    and the `.rpcc` bytes against the oracle; the streams through BatchDecoder against oracle.decompress_sections."""
    from rpcc_b200.batch import BatchDecoder, BatchEncoder
    cfg = _cfg(shape)
    H, W, hf, vmax, vmin, lut = _geometry(shape)
    frames, grounds = _frames(shape)
    pts = np.concatenate(frames, 0)
    off = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int64)
    B = len(frames)
    nonuniform = coding == "nonuniform"
    ccfg = _compressor_cfg("DBSCAN" if coding == "dbscan" else "FPS")
    model_method = "plane" if coding == "plane" else "point"
    segs = []
    with BatchEncoder(cfg, accuracy=0.02, nonuniform=nonuniform, compressor_cfg=ccfg, max_batch=B,
                      max_points=pts.shape[0], model_method=model_method) as enc:
        for inject in (True, False):
            gs = np.stack(grounds) if inject else None
            out = enc.encode_host(pts, off, gs)
            wants = []
            for b in range(B):
                g = grounds[b] if inject else oracle.ground_fit(oracle.project(frames[b], H, W, hf, vmax, vmin), lut)
                want = _want(coding, shape, frames[b], g, lut)
                wants.append(want)
                segs.append(want["seg_idx"])
                got = BatchEncoder.frame_sections(out, b)
                assert set(got) == set(want["sections"]), (shape, coding)
                for k, v in want["sections"].items():
                    assert got[k] == v, (shape, coding, b, inject, k)
            blobs = enc.compress(pts, off, gs)
            for b in range(B):
                assert blobs[b] == oracle.write_rpcc(wants[b]["sections"]), (shape, coding, b, inject)
            with BatchDecoder(cfg, accuracy=0.02, nonuniform=nonuniform, compressor_cfg=ccfg) as dec:
                d = dec.decode(blobs, want_xyz=True, want_points=True)
                labels, rng, xyz = (d[k].cpu().numpy() for k in ("labels", "range", "xyz"))
                res = d["results"]
                rows = [r.copy() for r in d["points"]]
            for b in range(B):
                sec = wants[b]["sections"]
                rec, wxyz, seg = oracle.decompress_sections(sec, cfg, 0.02)
                assert np.array_equal(labels[b].astype(np.int32), seg), (shape, coding, b, inject)
                assert np.array_equal(rng[b].view(np.uint32), rec.view(np.uint32)), (shape, coding, b, inject)
                assert np.array_equal(xyz[b].view(np.uint32), wxyz.view(np.uint32)), (shape, coding, b, inject)
                flat = wxyz.reshape(-1, 3)
                keep = (flat[:, 0] + flat[:, 1]) + flat[:, 2] != 0          # np.sum(point_cloud, -1) != 0
                assert rows[b].shape == (int(keep.sum()), 4), (shape, coding, b)
                assert np.array_equal(rows[b][:, :3].view(np.uint32), flat[keep].view(np.uint32)), (shape, coding, b)
                assert not rows[b][:, 3].any()
                assert int(res["sym_count"][b]) == len(sec["residual_quantized"]) // 2
                assert int(res["seq_count"][b]) == len(sec["idx_sequence"]) // 2
                assert int(res["flags"][b]) == 0, (shape, coding, b, int(res["flags"][b]))
                # the accuracy holds unless a symbol wrapped: a ground plane fitted on a 3-row image can pass near the
                # sensor, and its prediction then misses by kilometres (the int16 stream wraps like the reference's)
                if np.all(np.abs(np.asarray(wants[b]["symbols"], np.int64)) <= 32767):
                    ri = wants[b]["range_image"]
                    bound = np.float32(0.02 + (0.03 if nonuniform else 0.0)) + np.spacing(np.abs(ri))
                    assert np.all(np.abs(rec - ri) <= bound), (shape, coding, b)
            if nonuniform:
                _check_keypoints(wants)
    return segs


def _check_keypoints(wants):
    """The plugin's extract_features_with_segment (keypoints_kernel) against the oracle's key-point and feature maps: a key
    point that moves within its label changes no section."""
    from rpcc_b200.plugin import feature_extractor_cpp
    for w in wants:
        feat, kp = feature_extractor_cpp.extract_features_with_segment(w["range_image"], w["seg_idx"], 3, 8, 4, 8, 6)
        feat_o, kp_o = oracle.extract_features(w["range_image"], w["seg_idx"])
        assert np.array_equal(kp, kp_o) and np.array_equal(kp, w["key_point_map"])
        assert np.array_equal(feat.view(np.uint32), feat_o.view(np.uint32))


CODINGS = ([pytest.param(c, s, id="%s-%s" % (c, _id(s))) for c in ("uniform", "nonuniform") for s in ALL]
           + [pytest.param("plane", s, id="plane-" + _id(s)) for s in ALL if s[:2] in PLANE_SHAPES]
           + [pytest.param("dbscan", s, id="dbscan-" + _id(s)) for s in FULL if s[0] * s[1] <= DBSCAN_MAX_PIXELS])


# ----------------------------------------------------------------------------------------------- encode and decode
@pytest.mark.gpu
@pytest.mark.parametrize("coding,shape", CODINGS)
def test_encode_and_decode_match_the_oracle(coding, shape):
    segs = _encode_decode(coding, shape)
    H, W = shape[:2]
    if W < TILE and H > 2 and coding != "dbscan":
        # the row starts of tile 0 after pixel 0 decide a contour bit in some frame (3 x 1023: pixel 1023).  At H = 2
        # the one such pixel joins the two rings' ends, which these scenes never give one label.
        assert _tile0_row_start_pairs(segs, W) > 0, shape


# ----------------------------------------------------------------------------------------------- intensity
INTENSITY_SHAPES = [s for s in ALL if s[0] * s[1] % 32 != 0 or s[0] * s[1] == FPS_CAPACITY]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", INTENSITY_SHAPES, ids=_id)
def test_intensity_matches_the_oracle(shape):
    """Owners and the intensity image (project.cu) against oracle.intensity's sequential loop, the section bytes of the
    encoder (intensity.cu) against its quantiser, and the decoded `.bin` intensities against its inverse."""
    import torch
    from rpcc_b200 import device
    from rpcc_b200.batch import BatchDecoder, BatchEncoder
    cfg = _cfg(shape)
    H, W, hf, vmax, vmin, lut = _geometry(shape)
    frames, grounds = _frames(shape)
    acc = 0.01
    pts = np.concatenate(frames, 0)
    off = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int64)
    B = len(frames)
    rng, own, inten = device.intensity_owner_batch(torch.from_numpy(pts).cuda(), torch.from_numpy(off).cuda(), cfg)
    rng, own, inten = rng.cpu().numpy(), own.cpu().numpy(), inten.cpu().numpy()
    with BatchEncoder(cfg, accuracy=0.02, max_batch=B, max_points=pts.shape[0], intensity_accuracy=acc) as enc:
        out = enc.encode_host(pts, off, np.stack(grounds))
        secs = [BatchEncoder.frame_sections(out, b) for b in range(B)]
        blobs = enc.compress(pts, off, np.stack(grounds))
    with BatchDecoder(cfg, accuracy=0.02, intensity_accuracy=acc) as dec:
        d = dec.decode(blobs, want_xyz=False, want_points=True)
        rows = [r.copy() for r in d["points"]]
        rec = d["range"].cpu().numpy()
    for b, f in enumerate(frames):
        ri, owner = oi.project_owner(f, H, W, hf, vmax, vmin)
        img = oi.intensity_image(f, owner)
        assert np.array_equal(rng[b], ri) and np.array_equal(own[b], owner), (shape, b)
        assert np.array_equal(inten[b].view(np.uint32), img.view(np.uint32)), (shape, b)
        q, _ = oi.intensity_pack(img, ri, 2 * acc)
        assert secs[b]["intensity"] == q.tobytes(), (shape, b)
        back = oi.intensity_unpack(q, np.where(ri != 0, 0, 1), 2 * acc).reshape(-1)
        xyz = rec[b].reshape(-1, 1) * lut.reshape(-1, 3)
        keep = (xyz[:, 0] + xyz[:, 1]) + xyz[:, 2] != 0
        assert np.array_equal(rows[b][:, 3].view(np.uint32), back[keep].view(np.uint32)), (shape, b)


# ----------------------------------------------------------------------------------------------- window stages
def _dbscan_eps(shape):
    return 1.5 if shape[0] * shape[1] <= DBSCAN_MAX_PIXELS else 0.3


def _device_dbscan(ri, grounds, shape, eps, min_points=10, cluster_num=100):
    import torch
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    H, W, hf, vmax, vmin, lut = _geometry(shape)
    B = ri.shape[0]
    r = torch.from_numpy(np.ascontiguousarray(ri, np.float32)).cuda()
    lt = torch.from_numpy(lut).cuda()
    g = torch.from_numpy(np.ascontiguousarray(grounds, np.float32)).cuda()
    lab = torch.empty((B, H * W), dtype=torch.uint8, device="cuda")
    ws = torch.empty((_lib.lib().rpcc_dbscan_workspace_bytes(B, H, W),), dtype=torch.uint8, device="cuda")
    check(_lib.lib().rpcc_dbscan_segment_batch(ptr(r), ptr(lt), ptr(g), B, H, W, hf, vmax, vmin, float(eps),
                                               int(min_points), int(cluster_num), THR, ptr(lab), ptr(ws), None))
    torch.cuda.synchronize()
    return lab.cpu().numpy().reshape(B, H, W)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", FULL, ids=_id)
def test_window_stages_match_the_oracle(shape):
    """eval_batch against the exact chamfer kernel on decoded and on unrelated pairs, normals_batch against
    oracle.normals, and DBSCAN labels against oracle.dbscan, one launch per stage."""
    import torch
    from test_gpu_eval import _brute
    from test_gpu_p2plane import _check_normals
    from rpcc_b200 import device
    from rpcc_b200._lib import NORMAL_KNN, NORMAL_RADIUS
    cfg = _cfg(shape)
    H, W, hf, vmax, vmin, lut = _geometry(shape)
    frames, grounds = _frames(shape, empty=False)
    ris, recs = [], []
    for p, g in zip(frames, grounds):
        o = oracle.compress_frame(p, cfg, g)
        ris.append(o["range_image"])
        recs.append(oracle.decompress_sections(o["sections"], cfg, 0.02)[0].astype(np.float32))
    n = len(ris)
    a_imgs = ris + ris
    b_imgs = recs + [ris[(k + 1) % n] for k in range(n)]
    d_lut = torch.from_numpy(lut).cuda()
    A = torch.from_numpy(np.stack(a_imgs)).cuda()
    Bm = torch.from_numpy(np.stack(b_imgs)).cuda()
    m, d1, d2 = device.eval_batch(A, Bm, d_lut, cfg, want_dist=True)
    torch.cuda.synchronize()
    d1, d2 = d1.cpu().numpy(), d2.cpu().numpy()
    for k in range(2 * n):
        va, vb, w1, w2 = _brute(torch, a_imgs[k], b_imgs[k], lut)
        assert np.array_equal(d1[k].reshape(-1)[va.reshape(-1)].view(np.uint32), w1.view(np.uint32)), (shape, k)
        assert np.array_equal(d2[k].reshape(-1)[vb.reshape(-1)].view(np.uint32), w2.view(np.uint32)), (shape, k)
        assert (d1[k].reshape(-1)[~va.reshape(-1)] == -1).all()
    normals, _ = device.normals_batch(A[:n].contiguous(), d_lut, cfg)
    torch.cuda.synchronize()
    normals = normals.cpu().numpy().reshape(n, -1, 3)
    for k in range(n):
        _check_normals(ris[k], lut, normals[k], NORMAL_KNN, NORMAL_RADIUS)
    eps = _dbscan_eps(shape)
    got = _device_dbscan(np.stack(ris), np.stack(grounds), shape, eps)
    for k in range(n):
        want = dbscan.segment(ris[k], lut, grounds[k], eps, 10, 100, THR)
        assert np.array_equal(got[k], want), (shape, k, int((got[k] != want).sum()))


@pytest.mark.gpu
def test_window_stages_refuse_a_sensor_that_is_not_360_degrees():
    import torch
    from rpcc_b200 import RpccError, device
    shape = next(s for s in ALL if s[2] != 360)
    cfg = _cfg(shape)
    H, W, hf, vmax, vmin, lut = _geometry(shape)
    r = torch.ones((1, H, W), dtype=torch.float32, device="cuda")
    d_lut = torch.from_numpy(lut).cuda()
    with pytest.raises(RpccError, match="360-degree"):
        device.eval_batch(r, r, d_lut, cfg)
    with pytest.raises(RpccError, match="360-degree"):
        device.normals_batch(r, d_lut, cfg)
    with pytest.raises(RpccError, match="360-degree"):
        _device_dbscan(np.ones((1, H, W), np.float32), np.array([[0, 0, 1, 1.7]], np.float32), shape, 1.5)
