"""GPU parity tests aimed at the encoder's exactness guards.  Each fast path of the hot kernels is guarded by an error
argument and has an exact fallback; these tests build inputs that trip the guards (ranges outside the synthetic
1.5-80 m band, values on the decision thresholds, the FPS launch shapes ordinary frames never take) and demand the
results of references that share none of the kernels' shortcuts: the C oracle, torch's own f32 arithmetic for the
segment() lines (tests/refimpl.py), and plain IEEE arithmetic in numpy.  Each test prints how many inputs fell inside
the guard's band and asserts a minimum, so that it shows the fallback was really reached."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

LIDARS = ["Velodyne64E", "Velodyne32E", "VelodyneVLP16"]
F32_TENTH = np.float32(0.1)


@pytest.fixture(scope="module")
def T():
    import torch
    return torch


@pytest.fixture(scope="module")
def R():
    import rpcc_b200
    from rpcc_b200 import device
    rpcc_b200.device_mod = device
    return rpcc_b200


def _lut(lidar):
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    return oracle.transform_map(H, W, hf, vmax, vmin)


def _f32_steps(x, k):
    """x (f32 array) moved by k ulps (k an int array or scalar), for positive finite x."""
    x = np.asarray(x, np.float32)
    return (x.view(np.int32) + np.asarray(k, np.int32)).view(np.float32)


def _round_half_away(t):
    t = np.asarray(t, np.float64)
    return (np.sign(t) * np.floor(np.abs(t) + 0.5)).astype(np.int64)


def _sum3(a, b, c):
    """torch.sum over a size-3 last dim in f32: (t0 + t2) + t1 (pinned by test_torch_size3_reduction_association)."""
    return (np.float32(a) + np.float32(c)) + np.float32(b)


def _ground_dif(r, t, g):
    """torch's |sum(p * g[:3]) + g3| / norm(g[:3]) for p = r * t, in f32 (utils/segment_utils.py:137-139).
    -> (dif, a, gnorm)"""
    g = np.asarray(g, np.float32)
    r = np.asarray(r, np.float32)
    x, y, z = r * t[..., 0], r * t[..., 1], r * t[..., 2]
    a = np.abs(_sum3(x * g[0], y * g[1], z * g[2]) + g[3])
    gn = np.sqrt(_sum3(g[0] * g[0], g[1] * g[1], g[2] * g[2]))
    return a / gn, a, gn


def _rplane(t, g):
    g = np.asarray(g, np.float32)
    return (-g[3]) / _sum3(g[0] * t[..., 0], g[1] * t[..., 1], g[2] * t[..., 2])


# ----------------------------------------------------------------------------------------------- 1. scenes, end to end
def _points_of(ri, lut):
    """Points whose projection gives back (within an ulp or so) the range image ri: r * ray in f32, raster order."""
    m = ri != 0
    xyz = (ri[..., None] * lut)[m]
    return np.concatenate([xyz, np.zeros((xyz.shape[0], 1), np.float32)], 1).astype(np.float32)


def scene(lidar, kind, seed=0):
    """A synthetic frame with pixels moved outside the 1.5-80 m band.  kind:
      'far'   whole clusters at 250-3000 m on the rows looking up, far ground returns on the two rows nearest to
              horizontal (residual computed with the most cancellation);
      'edges' 32- and 64-pixel buckets whose x (or y) straddles +-250 m and -256 m ulp by ulp, sub-millimetre
              clusters at +-250 m, ranges below 2^-5 m, exactly 2^-5 m and exactly 256 m (and their neighbours);
      'wrap'  far clusters at 1400-2600 m that, in a frame coded with one cluster, leave the int16 symbol range.
    -> (points (N,4) f32, ground (4,) f64)"""
    from rpcc_b200 import synthetic
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = _lut(lidar)
    pts, ground = synthetic.frame(500 + seed + {"far": 0, "edges": 100, "wrap": 200}[kind], lidar)
    ri = oracle.project(pts, H, W, hf, vmax, vmin)
    g = np.random.default_rng(77 + seed)
    tz = lut[:, W // 8, 2]
    up = np.nonzero(tz > 0.01)[0]
    down = np.nonzero(tz < 0)[0]
    if kind in ("far", "wrap"):
        lo, hi = (250.0, 3000.0) if kind == "far" else (1400.0, 2600.0)
        for k in range(8):
            h = int(g.choice(up))
            w0 = int(g.integers(0, W - 48))
            base = g.uniform(lo, hi)
            ri[h, w0:w0 + 48] = (base * (1 + 2e-3 * g.random(48))).astype(np.float32)
    if kind == "far":
        rows = down[np.argsort(-tz[down])[:2]]               # the downward rows nearest to horizontal
        for h in rows:
            rp = _rplane(lut[h], ground)
            ok = (rp > 0) & (rp < 5000)
            noise = (1 + g.normal(0, 2e-5, W)).astype(np.float32)
            ri[h, ok] = (rp * noise)[ok]
    if kind == "edges":
        hs = int(up[0]) if len(up) else H - 1
        hd = int(down[len(down) // 2])
        for h in (hs, hd):
            for (w0, comp, target) in ((0, 0, 250.0), (W // 2 - 32, 0, -250.0), (W // 4 - 32, 1, 250.0),
                                       (W // 2 + 64, 0, -256.0)):
                w = np.arange(w0, w0 + 64) % W
                t = lut[h, w, comp]
                r0 = np.float32(target) / t
                k = (np.arange(64) % 9) - 4                      # -4 .. +4 ulps around the crossing
                ri[h, w] = _f32_steps(r0, k)
            # a sub-millimetre cluster on the 250 m crossing (one 32-pixel slice)
            w = np.arange(96, 128)
            ri[h, w] = (np.float32(250.0) / lut[h, w, 0] + g.uniform(0, 4e-4, 32)).astype(np.float32)
        near = np.array([0.004, 0.01, 0.02, 0.03, np.float32(2.0 ** -5), _f32_steps(np.float32(2.0 ** -5), -1),
                         _f32_steps(np.float32(2.0 ** -5), 1), 0.04, 256.0, _f32_steps(np.float32(256.0), -1),
                         _f32_steps(np.float32(256.0), 1), 256.0], np.float32)
        for i, h in enumerate(up[:3] if len(up) else [H - 1]):
            w0 = 3 * W // 4 + 40 * i
            ri[h, w0:w0 + 32] = np.resize(near, 32)
    return _points_of(ri, lut), ground


def _wrapped(symbols):
    return int(np.sum(np.abs(np.asarray(symbols, np.int64)) > 32767))


def _encode_and_check(lidar, frames, grounds, *, nonuniform=False, model_method="point", cluster_num=100, eval=False):
    """Every frame through BatchEncoder.encode_host with the ground injected and fitted on the device; every section
    against the oracle; the streams decoded by BatchDecoder against oracle.decompress_sections.
    -> per frame of the injected-ground pass: dict(want=oracle.compress_frame output, flags=results flags, eval=row)"""
    from rpcc_b200.batch import BatchDecoder, BatchEncoder
    from rpcc_b200.config import load_compressor_cfg
    cfg = load_compressor_cfg()
    cfg["cluster_num"] = cluster_num
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = _lut(lidar)
    pts = np.concatenate(frames, 0)
    off = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int64)
    B = len(frames)
    okw = dict(nonuniform=nonuniform, cluster_num=cluster_num, model_method=model_method)
    if model_method == "plane":
        okw["plane_impl"] = "device"
    report = []
    with BatchEncoder(lidar, accuracy=0.02, compressor_cfg=cfg, max_batch=B, max_points=pts.shape[0],
                      model_method=model_method, eval=eval, nonuniform=nonuniform) as enc:
        for inject in (True, False):
            out = enc.encode_host(pts, off, np.stack(grounds) if inject else None)
            wants = []
            for b in range(B):
                g = grounds[b] if inject else oracle.ground_fit(oracle.project(frames[b], H, W, hf, vmax, vmin), lut)
                want = oracle.compress_frame(frames[b], lidar, g, **okw)
                wants.append(want)
                got = BatchEncoder.frame_sections(out, b)
                for k, v in want["sections"].items():
                    assert got[k] == v, (lidar, b, inject, nonuniform, model_method, k)
                if inject:
                    report.append(dict(want=want, flags=int(out["results"][b]["flags"]),
                                       eval=None if out["eval"] is None else out["eval"][b].copy()))
            blobs = enc.compress(pts, off, np.stack(grounds) if inject else None)
            dec = BatchDecoder(lidar, accuracy=0.02, nonuniform=nonuniform, compressor_cfg=cfg)
            d = dec.decode(blobs)
            for b in range(B):
                rec, xyz, seg = oracle.decompress_sections(wants[b]["sections"], lidar, 0.02)
                assert np.array_equal(d["labels"][b].cpu().numpy().astype(np.int32), seg), (lidar, b, inject)
                assert np.array_equal(d["range"][b].cpu().numpy().view(np.uint32), rec.view(np.uint32)), (lidar, b)
                assert np.array_equal(d["xyz"][b].cpu().numpy().view(np.uint32), xyz.view(np.uint32)), (lidar, b)
                if _wrapped(wants[b]["symbols"]) == 0:
                    ri = wants[b]["range_image"]
                    bound = 0.02 + (0.03 if nonuniform else 0.0)
                    assert np.all(np.abs(rec - ri) <= np.float32(bound) + np.spacing(np.abs(ri))), (lidar, b)
    return report


def _guard_flag(want):
    """flag bit 0 of the label kernel: a pixel with a label >= 2 and a range outside [2^-5, 256)."""
    ri, seg = want["range_image"], want["seg_idx"]
    return bool(np.any((seg >= 2) & ((ri < np.float32(2.0 ** -5)) | (ri >= np.float32(256.0)))))


@pytest.mark.parametrize("lidar", LIDARS)
def test_far_near_and_edge_scenes_uniform(R, lidar):
    frames, grounds = zip(*[scene(lidar, k) for k in ("far", "edges")])
    rep = _encode_and_check(lidar, list(frames), list(grounds))
    for b, r in enumerate(rep):
        want_flag = _guard_flag(r["want"])
        ri = r["want"]["range_image"]
        print(lidar, ("far", "edges")[b], "flag", r["flags"] & 1, "pixels >= 256 m", int((ri >= 256).sum()),
              "pixels < 2^-5 m", int(((ri > 0) & (ri < 2.0 ** -5)).sum()))
        assert want_flag, (lidar, ("far", "edges")[b])                    # the scene reaches the exact-sum fallback ...
        assert (r["flags"] & 1) == 1, (lidar, ("far", "edges")[b])       # ... and the kernel raised its flag


@pytest.mark.parametrize("nonuniform,method", [(True, "point"), (False, "plane")])
def test_far_near_and_edge_scenes_other_codings(R, nonuniform, method):
    lidar = "Velodyne64E"
    frames, grounds = zip(*[scene(lidar, k, seed=1) for k in ("far", "edges")])
    _encode_and_check(lidar, list(frames), list(grounds), nonuniform=nonuniform, model_method=method)


@pytest.mark.parametrize("lidar", LIDARS)
def test_one_cluster_frames_wrap_their_symbols(R, lidar):
    """cluster_num = 1: one centre (the masked pixel 0), so one cluster holds ranges from metres to kilometres and its
    residuals leave the int16 range: the symbols wrap like astype(np.int16), the decoded ranges go negative and the
    eval window search falls back to its exhaustive scan.  Also FPS with one seed (m = 1) through the encoder."""
    frames, grounds = zip(*[scene(lidar, k) for k in ("far", "edges", "wrap")])
    rep = _encode_and_check(lidar, list(frames), list(grounds), cluster_num=1, eval=True)
    wrapped = [_wrapped(r["want"]["symbols"]) for r in rep]
    fallbacks = [float(r["eval"][10]) for r in rep]
    print(lidar, "wrapped symbols per frame", wrapped, "exhaustive eval points per frame", fallbacks)
    assert wrapped[2] > 0 and fallbacks[2] > 0
    for b, r in enumerate(rep):
        assert (r["flags"] & 1) == int(_guard_flag(r["want"])), (lidar, b)


# ----------------------------------------------------------------------------------------------- 2. decision thresholds
def _quantiser_inputs(lidar, B, K, g):
    """Labels, constant / plane model rows and ranges whose residual / step lies within 1e-7 .. 1e-3 of k + 0.5 (both
    sides and exactly on it), plus |q| > 32767.  -> ri (B,H,W) f32, seg (B,H,W) i32, model (B,K,4) f32, steps (B,K) f32"""
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    lut = _lut(lidar)
    ris, segs, models, steps = [], [], [], []
    for b in range(B):
        seg = np.repeat(g.integers(0, K, (H, W // 8)), 8, axis=1)[:, :W].astype(np.int32)
        seg[g.random((H, W)) < 0.05] = 1
        model = np.zeros((K, 4), np.float32)
        model[0] = [0.01, -0.02, 0.9997, 1.73]                          # ground row: a plane
        model[2:, 3] = g.uniform(5, 80, K - 2)                          # point-model rows: constants
        model[2:12:3, 3] = 3000.0                                       # room below for q < -32767
        pl = np.arange(3, K, 7)                                         # some plane rows
        model[pl, :3] = g.normal(0, 1, (len(pl), 3))
        model[pl, 3] = -np.abs(g.uniform(5, 30, len(pl))) * np.sign(model[pl, 2] + 1e-9)
        st = g.uniform(0.005, 0.05, K).astype(np.float32)
        seg[np.abs(oracle.intra_predict(seg, model, lut)) > 1e4] = 1     # plane rows nearly parallel to the ray
        pred = oracle.intra_predict(seg, model, lut)
        kk = g.integers(-3000, 3000, (H, W)).astype(np.float64)
        big = g.random((H, W)) < 0.01
        kk[big] = np.where(g.random(int(big.sum())) < 0.5, 1, -1) * g.integers(32768, 40000, int(big.sum()))
        delta = g.choice(np.concatenate([[0.0] * 6, 10.0 ** np.arange(-7, -2.9, 0.5)]), (H, W)) * g.choice([-1.0, 1.0], (H, W))
        s = st[seg].astype(np.float64)
        tt = kk + 0.5 + delta
        r0 = (pred.astype(np.float64) + tt * s).astype(np.float32)
        # scan the f32 neighbours of the target range for the residual closest to the target quotient
        cand = np.stack([_f32_steps(np.abs(r0), j) * np.sign(r0) for j in range(-6, 7)], -1).astype(np.float32)
        res = cand - pred[..., None]
        tq = res / st[seg][..., None]
        pick = np.argmin(np.abs(tq.astype(np.float64) - tt[..., None]), -1)
        ri = np.take_along_axis(cand, pick[..., None], -1)[..., 0]
        ri[seg == 1] = 0.0
        ris.append(ri); segs.append(seg); models.append(model); steps.append(st)
    return np.stack(ris), np.stack(segs), np.stack(models), np.stack(steps)


def _want_symbols(ri, seg, model, lut, step):
    """q = roundf((r - pred) / step) (cpp_modules.cpp:318), label-major stream, -> (int64 q, f32 quotients)"""
    pred = oracle.intra_predict(seg, model, lut)
    st = np.asarray(step, np.float32)
    s = st[seg] if st.ndim else np.full(seg.shape, st, np.float32)
    res = (ri - pred).astype(np.float32)
    t = res / s
    q = _round_half_away(t)
    order = np.argsort(seg.ravel(), kind="stable")
    keep = seg.ravel()[order] != 1
    return q.ravel()[order][keep], t.ravel()[order][keep], res.ravel()[order][keep], s.ravel()[order][keep]


def test_quantiser_on_the_rounding_boundaries(T, R):
    """The quantiser rounds a reciprocal product and redoes the division only when the quotient is within 1e-6 of
    k + 0.5 (both the staged and the plain kernel); residuals aimed at the boundaries, per-label and scalar steps,
    constant and plane rows, and symbols that wrap."""
    from rpcc_b200.plugin import quantization_utils_cpp
    lidar = "Velodyne64E"
    lut = _lut(lidar)
    H, W = lut.shape[:2]
    B, K = 2, 60
    g = np.random.default_rng(21)
    ri, seg, model, steps = _quantiser_inputs(lidar, B, K, g)
    d_lut = T.from_numpy(lut).cuda()
    d_ri = T.from_numpy(ri).cuda()
    d_seg = T.from_numpy(seg.astype(np.uint8)).cuda()
    d_model = T.from_numpy(model).cuda()
    d_g = T.from_numpy(model[:, 0].copy()).cuda()
    book = R.device_mod.label_stats_batch(d_ri, d_seg, K)
    _, results = R.device_mod.point_model_batch(d_ri, d_seg, d_g, book, K)     # tile offsets of the book
    nsym = results[:, 0].cpu().numpy()
    odd = T.empty(B * H * W + 1, dtype=T.float32, device="cuda")[1:].view(B, H, W)
    odd.copy_(d_ri)
    band = flips = wraps = 0
    for scalar in (0.005, 0.01, 0.04, 0.05, None):
        spl = None if scalar is not None else T.from_numpy(steps).cuda()
        for rng in (d_ri, odd):                         # 16-byte aligned (staged kernel), 4-byte offset (plain kernel)
            sym, _, _ = R.device_mod.quantize_pack_batch(rng, d_seg, d_model, d_lut, book, scalar or 0.0, spl)
            T.cuda.synchronize()
            for b in range(B):
                q, t, res, s = _want_symbols(ri[b], seg[b], model[b], lut, steps[b] if scalar is None else scalar)
                assert int(nsym[b]) == q.size
                got = sym[b, :q.size].cpu().numpy()
                assert np.array_equal(got, q.astype(np.int16)), (scalar, b, int(np.sum(got != q.astype(np.int16))))
                if rng is d_ri:
                    t64 = t.astype(np.float64)
                    band += int(np.sum(np.abs(np.abs(t64 - np.floor(t64)) - 0.5) <= 1e-6 * np.abs(t64)))
                    # the reciprocal product alone (no fallback) rounds these otherwise -- and not from exactly k + 0.5
                    tf = (res * (np.float32(1) / s).astype(np.float32)).astype(np.float32).astype(np.float64)
                    flips += int(np.sum((np.rint(tf) != q) & (np.abs(tf - np.floor(tf)) != 0.5)))
                    wraps += int(np.sum(np.abs(q) > 32767))
    # the drop-in op (int32 symbols, no wrap)
    for b in range(B):
        q, _, _, _ = _want_symbols(ri[b], seg[b], model[b], lut, 0.04)
        pred = oracle.intra_predict(seg[b], model[b], lut)
        got = quantization_utils_cpp.uniform_quantize(seg[b].astype(np.int64), (ri[b] - pred)[..., None], 0.04)
        assert np.array_equal(np.asarray(got).astype(np.int64), q), b
    print("quantiser: quotients within 1e-6 of k+0.5:", band, "| reciprocal product rounds otherwise:", flips,
          "| wrapped:", wraps)
    assert band >= 1000 and flips >= 20 and wraps >= 100


def _same_bits(a, b):
    """Bit-exact f32 comparison up to the sign of zero (torch's masked points are r * lut * 0, so -0.0 where the
    coordinate is negative; the kernels store +0.0, and the two are the same point to every later stage)."""
    return np.array_equal((a + np.float32(0)).view(np.uint32), (b + np.float32(0)).view(np.uint32))


def _mask_images(lut, grounds, n_live, g):
    """Range images whose live pixels sit within a few ulps of the ground threshold (torch's f32 arithmetic), the
    rest empty: -> (ri (B,H,W) f32, ulp offsets of the live pixels from f32(0.1))"""
    H, W = lut.shape[:2]
    B = len(grounds)
    ri = np.zeros((B, H, W), np.float32)
    offs = []
    flat = lut.reshape(-1, 3)
    for b in range(B):
        gm = np.asarray(grounds[b], np.float32)
        gn = float(np.sqrt(np.sum(gm[:3].astype(np.float64) ** 2)))
        gd = flat.astype(np.float64) @ gm[:3].astype(np.float64)
        cand_px = np.nonzero(np.abs(gd) > 1e-3)[0]
        px = g.choice(cand_px, n_live, replace=False)
        side = g.choice([-1.0, 1.0], n_live)
        side = np.where((side * 0.1 * gn - gm[3]) / gd[px] > 0, side, -side)    # the side in front of the sensor
        r0 = ((side * 0.1 * gn - gm[3]) / gd[px]).astype(np.float32)
        want = g.integers(-3, 4, n_live)
        want[: n_live // 4] = 0                                            # exactly on 0.1
        cands = np.stack([_f32_steps(r0, j) for j in range(-48, 49)], -1)
        dif, _, _ = _ground_dif(cands, flat[px][:, None, :], gm)
        ud = dif.view(np.int32).astype(np.int64) - np.int64(F32_TENTH.view(np.int32))
        pick = np.argmin(np.abs(ud - want[:, None]), -1)
        # and for some pixels the numerators |sum + g3| whose reciprocal product lands on the other side of 0.1
        _, a, gn = _ground_dif(cands, flat[px][:, None, :], gm)
        grid = ((F32_TENTH * gn).view(np.int32) + np.arange(-64, 65, dtype=np.int32)).view(np.float32)
        qa = grid * (np.float32(1) / gn)
        cross = grid[((grid / gn > F32_TENTH) != (qa > F32_TENTH)) & (qa != F32_TENTH)]
        hit = np.isin(a, cross)
        pick = np.where((g.random(n_live) < 0.4) & hit.any(-1), hit.argmax(-1), pick)
        ri[b].reshape(-1)[px] = np.take_along_axis(cands, pick[:, None], -1)[:, 0]
        offs.append(np.take_along_axis(ud, pick[:, None], -1)[:, 0])
    return ri, np.concatenate(offs)


def _torch_mask_fps(T, rng, lut, grounds, m):
    """utils/segment_utils.py:137-141 in torch, then oracle.fps per frame -> (cidx (B,m), centres (B,m,3))"""
    d_lut = T.from_numpy(lut).cuda() if isinstance(lut, np.ndarray) else lut
    d_g = T.from_numpy(np.asarray(grounds, np.float32)).cuda().view(-1, 1, 1, 4)
    pc = rng.unsqueeze(-1) * d_lut.unsqueeze(0)
    dif = T.abs(T.sum(pc * d_g[..., :3], -1) + d_g[..., 3]) / T.norm(d_g[..., :3], 2, -1)
    masked = (pc * (dif > 0.1).unsqueeze(-1)).reshape(rng.shape[0], -1, 3).cpu().numpy()
    cidx = np.stack([oracle.fps(masked[b], m) for b in range(masked.shape[0])])
    cent = np.stack([masked[b][cidx[b]] for b in range(masked.shape[0])])
    return cidx, cent


def _odd_lut():
    return _grid_lut(11, 101, -0.4, 0.1)                          # 1111 pixels: staged into a padded copy


def test_ground_mask_on_the_threshold(T, R):
    """FPS's first pass masks the ground with a reciprocal product and redoes the division for lanes within 1e-6 of
    the threshold; pixels a few ulps around f32(0.1) (exactly 0.1 is masked: strict '>'), planes of non-unit norm,
    fewer live points than seeds (every kept point becomes a centre, then the dmax == 0 rounds).  Planes through or
    near the sensor keep |sum(p * g) + g3| small, so that its f32 grid is as fine as 0.1's and every ulp can be hit."""
    g = np.random.default_rng(8)
    grounds = np.array([[0.01, -0.02, 0.9997, 1.73], [0.548, -0.921, -1.836, 0.0], [1.43, -1.866, 0.919, 0.0],
                        [-0.2, 0.11, 0.37, 0.02]], np.float32)
    near = exact = flips = 0
    for name, lut in [(l, _lut(l)) for l in LIDARS] + [("odd", _odd_lut())]:
        n_live = 200 if name != "odd" else 120
        ri, ud = _mask_images(lut, grounds, n_live, g)
        d_r, d_lut, d_g = T.from_numpy(ri).cuda(), T.from_numpy(lut).cuda(), T.from_numpy(grounds).cuda()
        cidx, centers = R.device_mod.segment_fps_batch(d_r, d_lut, d_g, 252, 0.1)
        T.cuda.synchronize()
        w_idx, w_cent = _torch_mask_fps(T, d_r, d_lut, grounds, 252)
        assert np.array_equal(cidx.cpu().numpy(), w_idx), name
        assert _same_bits(centers.cpu().numpy(), w_cent), name
        near += int(np.sum(np.abs(ud) <= 4))
        exact += int(np.sum(ud == 0))
        for b in range(len(grounds)):
            live = ri[b] != 0
            dif, a, gn = _ground_dif(ri[b][live], lut[live], grounds[b])
            qa = a * (np.float32(1) / gn)                 # the reciprocal product alone decides otherwise, off 0.1 itself
            flips += int(np.sum(((qa > F32_TENTH) != (dif > F32_TENTH)) & (qa != F32_TENTH)))
    print("ground mask: pixels within 4 ulps of 0.1:", near, "| exactly 0.1:", exact,
          "| reciprocal product decides otherwise:", flips)
    assert near >= 1500 and exact >= 300 and flips >= 100


def _label_scene(lidar, g):
    """A range image and centres with exact ties (mirror-image centres about a pixel at azimuth 90 or 270 degrees;
    a centre at exactly the pixel's ground residual), slices whose residuals sit around the whole-slice ground-skip
    threshold, and far pixels.  -> (ri (H,W) f32, ground (4,) f32, centres (M,3) f32)"""
    H, W = oracle.LIDARS[lidar]["H"], oracle.LIDARS[lidar]["W"]
    lut = _lut(lidar)
    gm = np.array([0.0, 0.0, 1.0, 1.73], np.float32)
    ri = np.zeros((H, W), np.float32)
    cents = []
    # (a) mirror ties: at azimuth 0 and 180 degrees y of the pixel is 0 or ~1e-16, so y - a and y + a round to -a and
    #     a exactly and the two centres are at exactly the same distance
    for i, h in enumerate(range(0, H, max(1, H // 16))):
        for col in (0, W // 2):
            r = np.float32(6.0 + 2.5 * i + (col > 0))
            ri[h, col] = r
            p = r * lut[h, col]
            a = np.float32(0.25)
            pair = [np.array([p[0], a, p[2]], np.float32), np.array([p[0], -a, p[2]], np.float32)]
            cents += pair if (i + col) % 2 else pair[::-1]
    # (b) ground-channel ties: a centre straight below the pixel at exactly its ground residual
    for j in range(80):
        h, col = int(g.integers(0, H)), int(g.integers(0, W))
        if ri[h, col] != 0 or col < 3 or col > W - 3 or abs(col - W // 2) < 3:
            continue
        r = np.float32(g.uniform(3, 40))
        t = lut[h, col]
        best = np.abs(r - _rplane(t, gm))
        p = r * t
        cz = np.float32(p[2] - best)
        for k in range(-4, 5):
            c = _f32_steps(np.abs(cz), k) * np.sign(cz) if cz != 0 else cz
            if np.float32(p[2] - c) == best:
                ri[h, col] = r
                cents.append(np.array([p[0], p[1], c], np.float32))
                break
    # (c) a centre high above the plane sets the skip threshold; slices of pixels whose residual is just around it
    cents.append(np.array([5.0, 5.0, 30.0], np.float32))
    dpl = min(abs(float(c[2]) + 1.73) for c in cents)
    skip = 0.5 * dpl * 0.99 - 2e-4
    down = np.nonzero(lut[:, 0, 2] < -0.05)[0]
    for s, h in enumerate(down[:6]):
        w0 = 64 * (5 + s)
        rp = _rplane(lut[h, w0:w0 + 64], gm)
        f = np.where(np.arange(64) < 32, 1 - 1e-4, 1 + 1e-4) if s % 2 else np.full(64, 1 - 1e-6)
        ri[h, w0:w0 + 64] = (rp + skip * f).astype(np.float32)
    # (d) far pixels, ground and not
    far = g.choice(H * W, 400, replace=False)
    far = far[ri.reshape(-1)[far] == 0]
    ri.reshape(-1)[far] = g.uniform(250, 3000, far.size).astype(np.float32)
    M = len(cents)
    assert M <= 252
    return ri, gm, np.stack(cents).astype(np.float32)


def _torch_like_ties(ri, lut, gm, cents):
    """numpy restatement of the distance table: how many pixels have two channels at the smallest |distance|."""
    live = ri != 0
    t = lut[live]
    r = ri[live]
    p = r[:, None] * t
    gr = np.abs(r - _rplane(t, gm))
    d = p[:, None, :] - cents[None]
    dd = np.sqrt(_sum3(d[..., 0] * d[..., 0], d[..., 1] * d[..., 1], d[..., 2] * d[..., 2]))
    allc = np.concatenate([gr[:, None], dd], 1)
    mn = allc.min(1, keepdims=True)
    n_at = (allc == mn).sum(1)
    return int(np.sum((n_at > 1) & (allc[:, 0] != mn[:, 0]))), int(np.sum((n_at > 1) & (allc[:, 0] == mn[:, 0])))


def test_labels_with_ties_skip_threshold_and_far_pixels(T, R):
    import refimpl
    g = np.random.default_rng(4)
    for lidar in LIDARS:
        lut = _lut(lidar)
        ri, gm, cents = _label_scene(lidar, g)
        d_r, d_lut = T.from_numpy(ri[None]).cuda(), T.from_numpy(lut).cuda()
        d_g, d_c = T.from_numpy(gm[None]).cuda(), T.from_numpy(cents[None]).cuda()
        M = cents.shape[0]
        labels, book = R.device_mod.assign_labels_batch(d_r, d_lut, d_g, d_c)
        model, results = R.device_mod.point_model_batch(d_r, labels, d_g, book, M + 2)
        T.cuda.synchronize()
        want = refimpl.torch_labels(ri, lut, gm, cents)
        got = labels[0].cpu().numpy().astype(np.int64)
        assert np.array_equal(got, want), (lidar, int(np.sum(got != want)))
        rows = int(results[0, 2].item())
        mp = oracle.model_param_point(ri, want.astype(np.int32), gm)
        assert rows == mp.shape[0]
        assert model[0, :rows].cpu().numpy().tobytes() == mp.tobytes(), lidar
        assert (int(results[0, 3].item()) & 1) == 1                    # far pixels with labels >= 2
        cc, gc = _torch_like_ties(ri, lut, gm, cents)
        print(lidar, "pixels tied between two centres:", cc, "| between the ground and a centre:", gc)
        assert cc >= 10 and gc >= 5, (lidar, cc, gc)


def test_point_model_means_outside_the_exact_sum_window(T, R):
    """The per-label means come from an exact u64 sum of range * 2^28, which truncates below 2^-5 m and is only
    proven up to 256 m; a frame with such a range under a label >= 2 is flagged and its means redone by the
    reference's own double loop.  Labels of tiny ranges only (where the truncation would show in the f32 mean), of
    ranges at and beyond 256 m, and mixed ones, through label_stats_batch + point_model_batch against the oracle."""
    lidar = "VelodyneVLP16"
    lut = _lut(lidar)
    H, W = lut.shape[:2]
    K = 40
    g = np.random.default_rng(31)
    seg = np.repeat(g.integers(2, K, (3, H, W // 4)), 4, axis=2).astype(np.int32)
    ri = (g.random((3, H, W)) * 60 + 2).astype(np.float32)
    tiny = (seg >= 2) & (seg < 12)
    ri[tiny] = (g.random(int(tiny.sum())) * 0.03 + 1e-4).astype(np.float32)
    far = (seg >= 12) & (seg < 18)
    ri[far] = np.where(g.random(int(far.sum())) < 0.3, np.float32(256.0),
                       g.uniform(256, 3000, int(far.sum()))).astype(np.float32)
    ri[2] = np.where(seg[2] < 12, np.float32(2.0 ** -5), ri[2])          # exactly 2^-5: inside the window
    ri[2][seg[2] >= 12] = np.minimum(ri[2][seg[2] >= 12], _f32_steps(np.float32(256.0), -1))
    seg[g.random(seg.shape) < 0.05] = 1
    ri[seg == 1] = 0.0
    gm = np.array([[0.0, 0.0, 1.0, 1.73]] * 3, np.float32)
    d_r, d_seg, d_g = T.from_numpy(ri).cuda(), T.from_numpy(seg.astype(np.uint8)).cuda(), T.from_numpy(gm).cuda()
    book = R.device_mod.label_stats_batch(d_r, d_seg, K)
    model, results = R.device_mod.point_model_batch(d_r, d_seg, d_g, book, K)
    T.cuda.synchronize()
    res = results.cpu().numpy()
    inexact = 0
    for b in range(3):
        want = oracle.model_param_point(ri[b], seg[b], gm[b])
        rows = int(res[b, 2])
        assert rows == want.shape[0]
        assert model[b, :rows].cpu().numpy().tobytes() == want.tobytes(), b
        assert (int(res[b, 3]) & 1) == (0 if b == 2 else 1), b
        # labels whose mean the truncated u64 sum would get wrong
        for l in range(2, K):
            r = ri[b][seg[b] == l].astype(np.float64)
            if r.size:
                trunc = np.sum(np.floor(r * 268435456.0)) / 268435456.0
                inexact += int(np.float32(trunc / r.size) != np.float32(np.sum(r) / r.size))
    print("labels whose mean the window's u64 sum would round otherwise:", inexact)
    assert inexact >= 3


# ----------------------------------------------------------------------------------------------- 3. FPS launch shapes
def _images(T, R, lidar, n_distinct, B, g):
    """B distinct range images of one lidar: n_distinct synthetic frames, each copy scaled and thinned at random."""
    from rpcc_b200 import synthetic
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    fr = [synthetic.frame(700 + i, lidar) for i in range(n_distinct)]
    base = [oracle.project(p, H, W, hf, vmax, vmin) for p, _ in fr]
    grounds = np.stack([gr for _, gr in fr]).astype(np.float32)
    ri = np.empty((B, H, W), np.float32)
    gs = np.empty((B, 4), np.float32)
    for b in range(B):
        k = b % n_distinct
        ri[b] = base[k] * np.float32(1 + 0.02 * g.random()) * (g.random((H, W)) > 0.05 * g.random())
        gs[b] = grounds[k]
    return ri, gs


def test_fps_many_distinct_frames_one_launch(T, R):
    """More frames than twice the SM count, every one distinct, so the longest-first frame queue really reorders;
    seeds against torch's mask and the oracle's FPS (the twin of the reference-kernel test, which needs oracle/_ref)."""
    g = np.random.default_rng(12)
    sms = T.cuda.get_device_properties(0).multi_processor_count
    for lidar, B in (("VelodyneVLP16", 2 * sms + 9), ("Velodyne64E", 2 * sms + 3)):
        ri, gs = _images(T, R, lidar, 12, B, g)
        lut = _lut(lidar)
        d_r, d_lut, d_g = T.from_numpy(ri).cuda(), T.from_numpy(lut).cuda(), T.from_numpy(gs).cuda()
        cidx, centers = R.device_mod.segment_fps_batch(d_r, d_lut, d_g, 100, 0.1)
        w_idx, w_cent = _torch_mask_fps(T, d_r, d_lut, gs, 100)
        got = cidx.cpu().numpy()
        assert np.array_equal(got, w_idx), (lidar, np.nonzero((got != w_idx).any(1))[0][:8])
        assert _same_bits(centers.cpu().numpy(), w_cent), lidar


def test_fps_index_order_queue_beyond_8192_frames(T, R):
    """More than 8192 frames of a 1024-pixel image: the frame queue is taken in index order."""
    g = np.random.default_rng(13)
    H, W = 8, 128
    lut = _grid_lut(H, W, -0.35, 0.05)
    B = 8200
    ri = (2.0 + 40.0 * g.random((B, H, W))).astype(np.float32)
    ri[g.random((B, H, W)) < 0.1] = 0.0
    gs = np.tile(np.array([[0.0, 0.0, 1.0, 1.7]], np.float32), (B, 1))
    gs[:, 3] += g.uniform(-0.3, 0.3, B).astype(np.float32)
    d_r, d_lut, d_g = T.from_numpy(ri).cuda(), T.from_numpy(lut).cuda(), T.from_numpy(gs).cuda()
    cidx, centers = R.device_mod.segment_fps_batch(d_r, d_lut, d_g, 24, 0.1)
    w_idx, w_cent = _torch_mask_fps(T, d_r, d_lut, gs, 24)
    got = cidx.cpu().numpy()
    assert np.array_equal(got, w_idx), np.nonzero((got != w_idx).any(1))[0][:8]
    assert _same_bits(centers.cpu().numpy(), w_cent)


def _grid_lut(H, W, lo, hi):
    az = np.linspace(0, 2 * np.pi, W, endpoint=False)[None, :]
    el = np.linspace(lo, hi, H)[:, None]
    return np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el) * np.ones_like(az)], -1).astype(np.float32)


@pytest.mark.parametrize("table", LIDARS + ["32x1500"])
def test_fps_one_seed_and_unaligned_range_buffer(T, R, table):
    """m = 1 on aligned buffers; m = 100 and m = 1 with a range buffer 4 bytes off a 16-byte boundary, and m = 100 with
    such a LUT, both staged into aligned copies (Q = 2 for the 64E and 32E tables, 1 for the VLP16 and a 32 x 1500
    table).  Seeds and centres against torch's mask and the oracle's FPS."""
    g = np.random.default_rng(14)
    if table in LIDARS:
        ri, gs = _images(T, R, table, 3, 3, g)
        lut = _lut(table)
    else:
        lut = _grid_lut(32, 1500, -0.4, 0.1)
        ri = (3.0 + 50.0 * g.random((3, 32, 1500))).astype(np.float32)
        ri[g.random(ri.shape) < 0.1] = 0.0
        gs = np.tile(np.array([[0.01, 0.0, 1.0, 1.7]], np.float32), (3, 1))
    d_r, d_lut, d_g = T.from_numpy(ri).cuda(), T.from_numpy(lut).cuda(), T.from_numpy(gs).cuda()
    odd = T.empty(ri.size + 1, dtype=T.float32, device="cuda")[1:].view(ri.shape)
    odd.copy_(d_r)
    odd_lut = T.empty(d_lut.numel() + 1, dtype=T.float32, device="cuda")[1:].view(d_lut.shape)
    odd_lut.copy_(d_lut)
    for rng, lut_in, m in ((d_r, d_lut, 1), (odd, d_lut, 100), (odd, d_lut, 1), (d_r, odd_lut, 100)):
        cidx, centers = R.device_mod.segment_fps_batch(rng, lut_in, d_g, m, 0.1)
        w_idx, w_cent = _torch_mask_fps(T, d_r, d_lut, gs, m)
        assert np.array_equal(cidx.cpu().numpy(), w_idx), (table, m)
        assert _same_bits(centers.cpu().numpy(), w_cent), (table, m)


def test_fps_refuses_images_beyond_131072_pixels(T, R):
    """A 2 x 65 540 image (131 080 pixels) holds more 64-pixel buckets than the round kernel keeps on chip: the launch is
    refused, for m = 100 and m = 1, through an aligned range buffer and through one 4 bytes off a 16-byte boundary
    (which would be staged)."""
    H, W = 2, 65540
    d_lut = T.from_numpy(_grid_lut(H, W, -0.1, 0.1)).cuda()
    d_g = T.tensor([[0.0, 0.0, 1.0, 1.7]], dtype=T.float32, device="cuda")
    d_r = T.full((1, H, W), 10.0, dtype=T.float32, device="cuda")
    odd = T.empty(d_r.numel() + 1, dtype=T.float32, device="cuda")[1:].view(d_r.shape)
    odd.copy_(d_r)
    for rng in (d_r, odd):
        for m in (100, 1):
            with pytest.raises(R.RpccError, match="131072 pixels"):
                R.device_mod.segment_fps_batch(rng, d_lut, d_g, m, 0.1)
