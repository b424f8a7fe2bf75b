"""The range-image window searches held to brute force where their pruning bound binds.

rpcc_eval_batch (evalq.cu), rpcc_normals_batch / rpcc_p2plane_batch (normals.cu) and rpcc_dbscan_segment_batch
(dbscan.cu) grow a window around the query's pixel and stop once everything outside it is provably farther than what
they still need.  On natural frames the nearest neighbour sits 1 to 5 pixels away, far inside that bound, so a bound a
little too high goes unnoticed.  The images here are sparse: every query sits alone in an otherwise empty neighbourhood
with a candidate k rows or columns away at the foot of the perpendicular from the query point to the candidate's ray
(the closest that ray comes, within a few f32 ulps), which is where the bound is tight, and a decoy on the query's own
pixel whose distance is the smallest one above the candidate's, ideally also below the stop bound of tables without the
angular slack.  A search that stops on a bound above the candidate's distance returns the decoy.  Every angle comes
from the f32 ray table, as the kernels see it.

The CPU test restates the bound (oracle/window.py) and checks it against such candidates at every k the tables hold;
the GPU tests compare each stage with the brute-force references of oracle/ bit for bit."""
import functools

import numpy as np
import pytest

import oracle
from oracle import dbscan as odb
from oracle import normals as N
from oracle import window as OW

F32, F64 = np.float32, np.float64
KEVR = OW.KEVR
THR = 0.1
MAX_CASES = 3000          # per image: at most 6000 valid points, so the references stay on their brute-force paths

# id -> LidarConfig arguments; the shapes without a name are +10 / -25 degree sensors unless they say otherwise
SHAPES = {
    "64E": dict(name="Velodyne64E"),
    "32E": dict(name="Velodyne32E"),
    "VLP16": dict(name="VelodyneVLP16"),
    "2x65536": dict(H=2, W=65536),            # the FPS capacity in two rings: column pitch 8.7e-5 rad at -25 degrees
    "4x32768": dict(H=4, W=32768),
    "8192x16": dict(H=8192, W=16),            # row pitch 7.5e-5 rad
    "16384x8": dict(H=16384, W=8),            # row pitch 3.7e-5 rad
    "64x2048_1deg": dict(H=64, W=2048, vmax_deg=1.0, vmin_deg=-1.0),   # a fine row pitch at a small image
    "2x262144": dict(H=2, W=262144),          # rpcc_eval_batch only: past the encoder's 131 072 pixels
}
ENCODER_SHAPES = [s for s in SHAPES if s != "2x262144"]


def _cfg(sid):
    from rpcc_b200 import LidarConfig
    s = SHAPES[sid]
    if "name" in s:
        return LidarConfig(s["name"])
    return LidarConfig(hfov_deg=360.0, vmax_deg=s.get("vmax_deg", 10.0), vmin_deg=s.get("vmin_deg", -25.0), H=s["H"],
                       W=s["W"])


@functools.lru_cache(maxsize=None)
def _geometry(sid):
    """-> (cfg, H, W, hfov, vmax, vmin, lut (H*W, 3) f32)."""
    cfg = _cfg(sid)
    H, W, hf, vmax, vmin = oracle.lidar_params(cfg)
    return cfg, H, W, hf, vmax, vmin, oracle.transform_map(H, W, hf, vmax, vmin).reshape(-1, 3)


def _foot_row(sid):
    """The row of largest |elevation|, where the column bound (cmin) is tight."""
    _, H, _, _, vmax, vmin, _ = _geometry(sid)
    return 0 if abs(vmin) >= abs(vmax) else H - 1


def _kmax(sid, direction):
    """Largest k whose table entry the walk reads: columns while 2 dc + 1 < W, rows while the window is not every row."""
    _, H, W = _geometry(sid)[:3]
    return min(KEVR + 1, W // 2 if direction == "col" else H - 1)


def _ks(sid, direction):
    """k = 1, 2, a middle value and kEvR - 1, as far as the shape has them."""
    km = min(_kmax(sid, direction), KEVR - 1)
    return sorted({k for k in (1, 2, max(1, km // 2), km) if 1 <= k <= km})


# ----------------------------------------------------------------------------------------------- generator
def _ulps(x, n):
    """Positive f32 x moved by n ulps."""
    return (np.asarray(x, F32).view(np.int32) + np.asarray(n, np.int32)).view(F32)


def _points(r, rays):
    return (np.asarray(r, F32)[..., None] * rays).astype(F32)          # image_point: r * ray in f32


def _hug(lut, qp, rq, cp, span=3):
    """The candidate range on ray cp closest to the query point rq * ray(qp): the f32 foot of the perpendicular +- span
    ulps, the one with the smallest cham_d -> (range, cham_d), each shaped like rq.  Past 90 degrees the foot is
    behind the sensor, and the closest positive range is a tiny one."""
    q = _points(rq, lut[qp])
    lc = lut[cp].astype(F64)
    foot = np.maximum((q.astype(F64) * lc).sum(-1) / (lc * lc).sum(-1), 1e-6 * rq).astype(F32)
    rc = _ulps(foot[..., None], np.arange(-span, span + 1))
    d = N.cham_d(q[..., None, :], _points(rc, lut[cp][..., None, :]))
    j = np.argmin(d, -1)[..., None]
    return np.take_along_axis(rc, j, -1)[..., 0], np.take_along_axis(d, j, -1)[..., 0]


def _decoy(lut, qp, rq, above, span=10):
    """The range on the query's own ray whose cham_d is the smallest one above `above` (inf if none in reach)."""
    q = _points(rq, lut[qp])
    s = np.sqrt(np.asarray(above, F64))
    x0 = np.stack([(rq + s).astype(F32), np.maximum(rq - s, 1e-3).astype(F32)], -1)
    x = _ulps(x0[..., None], np.arange(-span, span + 1)).reshape(x0.shape[:-1] + (-1,))
    d = N.cham_d(q[..., None, :], _points(x, lut[qp][..., None, :]))
    d = np.where(d > np.asarray(above, F32)[..., None], d, np.inf)
    j = np.argmin(d, -1)[..., None]
    return np.take_along_axis(x, j, -1)[..., 0], np.take_along_axis(d, j, -1)[..., 0]


def _tight_pairs(sid, direction, k, n, rng):
    """n random (query pixel, candidate pixel) pairs k columns apart in the foot row, or k rows apart in one column."""
    _, H, W = _geometry(sid)[:3]
    s = rng.choice(np.array([-1, 1]), n)
    if direction == "col":
        h = _foot_row(sid)
        w = rng.integers(0, W, n)
        return h * W + w, h * W + (w + s * k) % W
    h = rng.integers(0, H - k, n)
    w = rng.integers(0, W, n)
    hq = np.where(s > 0, h, h + k)
    return hq * W + w, (hq + s * k) * W + w


def _layout(sid, direction, k, rng, max_cases=MAX_CASES):
    """Case footprints whose points are farther from each other's queries than their own candidate -> (query pixels,
    candidate pixels).  Columns: in the foot row, random side, the last case's candidate across column W-1 -> 0 (the
    wrap).  Rows: stacked from row 0 to row H-1, so the extreme rows and the middle ones all hold queries, in columns
    further apart than k rows."""
    _, H, W, hf, vmax, vmin, _ = _geometry(sid)
    if direction == "col":
        h, L = _foot_row(sid), 2 * k + 3
        n = max(1, min(max_cases, (W - 2 * k - 2) // L))
        j = int(rng.integers(0, k))
        o = W - 1 - j - (n - 1) * L - k - 1                  # the last query at W-1-j
        w = (o + np.arange(n) * L + k + 1) % W
        s = rng.choice(np.array([-1, 1]), n)
        s[-1] = 1
        return h * W + w, h * W + (w + s * k) % W
    period = 2 * k + 2
    col_pitch = np.cos(max(abs(vmax), abs(vmin))) * hf / W
    cols = np.arange(0, W, max(1, int(np.ceil(1.5 * k * (vmax - vmin) / (H - 1) / col_pitch))))
    starts = np.arange(0, H - k, period)
    if starts[-1] + k < H - 1:
        starts = np.append(starts, H - 1 - k)              # a case ending on the last row
    if starts.size > 1 and starts[-1] - starts[-2] < period:
        starts = np.delete(starts, -2)
    hh, ww = np.meshgrid(starts, cols, indexing="ij")
    hh, ww = hh.reshape(-1), ww.reshape(-1)
    if hh.size > max_cases:
        keep = np.sort(rng.choice(hh.size, max_cases, replace=False))
        hh, ww = hh[keep], ww[keep]
    up = rng.random(hh.size) < 0.5
    hq = np.where(up, hh, hh + k)
    return hq * W + ww, np.where(up, hh + k, hh) * W + ww


def _hugging_pair(sid, direction, k, seed, trials=16):
    """-> (A, B) (H,W) f32 range images and dict(qp, cp, trap): A holds the queries, B the candidates and the decoys.
    Per case `trials` query ranges are drawn; a trial whose decoy lies between the candidate's distance and the stop
    bound of the tables without slack (a search with that bound returns the decoy) is taken when there is one."""
    _, H, W, hf, vmax, vmin, lut = _geometry(sid)
    rng = np.random.default_rng(seed)
    qp, cp = _layout(sid, direction, k, rng)
    n = qp.size
    rq = rng.uniform(0.5, 120.0, (n, trials)).astype(F32)
    Q, C = np.repeat(qp[:, None], trials, 1), np.repeat(cp[:, None], trials, 1)
    rc, dc = _hug(lut, Q, rq, C)
    x, dd = _decoy(lut, Q, rq, dc)
    row, col = OW.eval_geom(H, W, hf, vmax, vmin, tau=0.0)
    old = OW.stop_bound(rq, (col if direction == "col" else row)[k])
    trap = np.isfinite(dd) & (dd < old)
    t = np.where(trap.any(1), np.argmax(trap, 1), 0)
    pick = (np.arange(n), t)
    A = np.zeros(H * W, F32)
    B = np.zeros(H * W, F32)
    A[qp] = rq[pick]
    B[cp] = rc[pick]
    B[qp] = np.where(np.isfinite(dd[pick]), x[pick], 0)
    return A.reshape(H, W), B.reshape(H, W), dict(qp=qp, cp=cp, trap=trap[pick])


# ----------------------------------------------------------------------------------------------- the bound (no GPU)
def _bound_misses(sid, tau, n=1500, seed=0):
    """[(direction, k, misses)] where a candidate's exact f32 cham_d lies below the stop bound of its table entry."""
    _, H, W, hf, vmax, vmin, lut = _geometry(sid)
    row, col = OW.eval_geom(H, W, hf, vmax, vmin, tau)
    rng = np.random.default_rng(seed)
    out = []
    for direction, table in (("col", col), ("row", row)):
        for k in range(1, _kmax(sid, direction) + 1):
            qp, cp = _tight_pairs(sid, direction, k, n, rng)
            rq = rng.uniform(0.5, 120.0, n).astype(F32)
            _, d = _hug(lut, qp, rq, cp)
            bad = int((d < OW.stop_bound(rq, table[k])).sum())
            if bad:
                out.append((direction, k, bad))
    return out


@pytest.mark.parametrize("sid", list(SHAPES))
def test_stop_bound_holds_at_bound_hugging_candidates(sid):
    """For every k the tables hold (up to kEvR + 1), in both directions: no candidate at the foot of the perpendicular,
    +- 3 ulps of range, is nearer than the bound the device compares with."""
    assert _bound_misses(sid, OW.TAU) == []


def test_tables_without_the_angular_slack_miss_at_fine_pitches():
    """The generator has teeth: the tables as they were before the absolute slack (a relative margin alone) put the
    bound above real candidates at 2 x 65536 (columns) and 16384 x 8 (rows), and nowhere at the reference lidars."""
    assert any(d == "col" for d, _, _ in _bound_misses("2x65536", 0.0))
    assert any(d == "row" for d, _, _ in _bound_misses("16384x8", 0.0))
    for sid in ("64E", "32E", "VLP16"):
        assert _bound_misses(sid, 0.0) == [], sid


def test_slack_costs_less_than_the_margin_at_the_lidars():
    """At the reference lidars the angular slack lowers no table entry by as much as the relative margin does, so
    their windows stay as they were; the tables stay non-decreasing in k."""
    for sid in ("64E", "32E", "VLP16"):
        _, H, W, hf, vmax, vmin, _ = _geometry(sid)
        row, col = OW.eval_geom(H, W, hf, vmax, vmin)
        row0, col0 = OW.eval_geom(H, W, hf, vmax, vmin, tau=0.0)
        for a, b in ((row, row0), (col, col0)):
            assert a[0] == 0 and np.all(a <= b) and np.all(a[1:] > b[1:] * F32(1 - 2e-3))
            assert np.all(np.diff(a.astype(F64)) >= 0)


def test_generator_places_traps_where_the_old_bound_fails():
    """At 2 x 65536, k = 1, some decoys sit between the candidate's distance and the old stop bound; every decoy is
    farther than its candidate, so the candidate is the nearest point of B."""
    _, H, W, hf, vmax, vmin, lut = _geometry("2x65536")
    A, B, c = _hugging_pair("2x65536", "col", 1, seed=11)
    assert c["trap"].sum() >= 3
    q = _points(A.reshape(-1)[c["qp"]], lut[c["qp"]])
    dc = N.cham_d(q, _points(B.reshape(-1)[c["cp"]], lut[c["cp"]]))
    dd = N.cham_d(q, _points(B.reshape(-1)[c["qp"]], lut[c["qp"]]))
    assert np.all(dc < dd)


# ----------------------------------------------------------------------------------------------- GPU: eval
def _t(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _eval(sid, As, Bs):
    from rpcc_b200 import device
    import torch
    cfg, *_, lut = _geometry(sid)
    m, d1, d2 = device.eval_batch(_t(np.stack(As)), _t(np.stack(Bs)), _t(lut), cfg, want_dist=True)
    torch.cuda.synchronize()
    return m.cpu().numpy(), d1.cpu().numpy().reshape(len(As), -1), d2.cpu().numpy().reshape(len(As), -1)


def _check_eval(sid, A, B, m, d1, d2):
    """dist1 / dist2 bit for bit against oracle.chamfer_nn (the chamfer kernel's FMA order), columns 2-9 recomputed from
    them."""
    lut = _geometry(sid)[-1]
    pa, va = N.cloud(A, lut)
    pb, vb = N.cloud(B, lut)
    w1, _ = oracle.chamfer_nn(pa[va], pb[vb], fma_mode=1)
    w2, _ = oracle.chamfer_nn(pb[vb], pa[va], fma_mode=1)
    assert np.array_equal(d1[va].view(np.uint32), w1.view(np.uint32)), (sid, int((d1[va] != w1).sum()))
    assert np.array_equal(d2[vb].view(np.uint32), w2.view(np.uint32)), (sid, int((d2[vb] != w2).sum()))
    assert (d1[~va] == -1).all() and (d2[~vb] == -1).all()
    thr = F32(0.02 ** 2)
    for c, w in ((2, w1), (6, w2)):
        assert m[c] == w.size and m[c + 2] == (w < thr).sum()
        assert abs(m[c + 1] - np.sqrt(w).astype(F64).sum()) <= 1e-9 * m[c + 1]
        assert abs(m[c + 3] - w.astype(F64).sum()) <= 1e-9 * m[c + 3]


def _hugging_frames(sid):
    return [(d, k) + _hugging_pair(sid, d, k, seed=1000 * k + (d == "row"))
            for d in ("col", "row") for k in _ks(sid, d)]


@pytest.mark.gpu
@pytest.mark.parametrize("sid", list(SHAPES))
def test_eval_distances_at_bound_hugging_pairs(sid):
    """Column feet at k = 1, 2, a middle k and kEvR - 1 (one across the wrap), row feet likewise from the first to the
    last row: all pairs of a shape in one launch."""
    fr = _hugging_frames(sid)
    m, d1, d2 = _eval(sid, [f[2] for f in fr], [f[3] for f in fr])
    lut = _geometry(sid)[-1]
    hits = total = 0
    for b, (d, k, A, B, c) in enumerate(fr):
        _check_eval(sid, A, B, m[b], d1[b], d2[b])
        q = _points(A.reshape(-1)[c["qp"]], lut[c["qp"]])
        dc = N.cham_d(q, _points(B.reshape(-1)[c["cp"]], lut[c["cp"]]))
        hits, total = hits + int((d1[b][c["qp"]] == dc).sum()), total + dc.size
    # the candidate is the query's nearest point, bar the odd wide-angle case whose neighbour case is nearer
    assert hits >= 0.95 * total, (sid, hits, total)


EDGE = [("64E", "col"), ("2x65536", "col"), ("8192x16", "row")]


@pytest.mark.gpu
@pytest.mark.parametrize("sid,direction", EDGE)
def test_eval_at_the_window_edge(sid, direction):
    """The only candidate exactly kEvR away is found inside the tabulated window (no whole-image scan); at kEvR + 1
    the walk scans the whole image, and the distances are the brute force's in both cases."""
    frames = []
    for k in (KEVR, KEVR + 1):
        _, H, W, *_ = _geometry(sid)
        rng = np.random.default_rng(k)
        qp, cp = _layout(sid, direction, k, rng, max_cases=400)
        if direction == "col":                               # slots wider than the window: nothing else in reach
            qp, cp = qp[::2], cp[::2]
        rq = rng.uniform(0.5, 120.0, qp.size).astype(F32)
        rc, _ = _hug(_geometry(sid)[-1], qp, rq, cp)
        A, B = np.zeros(H * W, F32), np.zeros(H * W, F32)
        A[qp], B[cp] = rq, rc
        frames.append((A.reshape(H, W), B.reshape(H, W)))
    m, d1, d2 = _eval(sid, [f[0] for f in frames], [f[1] for f in frames])
    for b, (A, B) in enumerate(frames):
        _check_eval(sid, A, B, m[b], d1[b], d2[b])
    assert m[0, 10] == 0 and m[1, 10] > 0, m[:, 10]


# ----------------------------------------------------------------------------------------------- GPU: p2plane, normals
def _random_normals(img, rng):
    """(HW,3) f32: a unit normal at about half of the image's points, (0,0,0) elsewhere."""
    n = rng.normal(size=(img.size, 3))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    n[(img.reshape(-1) == 0) | (rng.random(img.size) < 0.5)] = 0
    return n.astype(F32)


def _p2plane(sid, As, Bs, NA, NB):
    from rpcc_b200 import device
    import torch
    cfg, *_, lut = _geometry(sid)
    m = device.p2plane_batch(_t(np.stack(As)), _t(np.stack(Bs)), _t(lut), cfg, _t(np.stack(NA)), _t(np.stack(NB)))
    torch.cuda.synchronize()
    return m.cpu().numpy()


def _check_p2plane(sid, A, B, na, nb, m):
    want = N.p2plane(A, B, _geometry(sid)[-1], na, nb)
    assert np.array_equal(m[[0, 2, 3, 5]], want[[0, 2, 3, 5]]), (sid, m, want)
    assert np.allclose(m[[1, 4]], want[[1, 4]], rtol=1e-9, atol=0), (sid, m, want)


@pytest.mark.gpu
@pytest.mark.parametrize("sid", ENCODER_SHAPES)
def test_p2plane_at_bound_hugging_pairs(sid):
    """The search that returns an index, on the same pairs: a normal at half of the points, so picking the decoy
    changes the no-normal count or the error."""
    fr = _hugging_frames(sid)
    rng = np.random.default_rng(7)
    NA = [_random_normals(f[2], rng) for f in fr]
    NB = [_random_normals(f[3], rng) for f in fr]
    m = _p2plane(sid, [f[2] for f in fr], [f[3] for f in fr], NA, NB)
    for b, f in enumerate(fr):
        _check_p2plane(sid, f[2], f[3], NA[b], NB[b], m[b])


def _tie_cases(sid, k, rng):
    """Queries at the azimuths where the ray table is mirror-symmetric (0, 90, 180, 270 degrees), two candidates at
    columns w - k and w + k with bit-identical cham_d (column 0: across the wrap) and a near point at column w + 1 off
    the line -> (img, qp, lo, hi, near): the tied pair is the query's 2nd and 3rd nearest, so with knn = 3 the first
    of them in raster order takes the last slot."""
    _, H, W, *_, lut = _geometry(sid)
    cols = [c for c in (0, W // 4, W // 2, 3 * W // 4) if 4 * c % W == 0]
    img = np.zeros(H * W, F32)
    out = []
    for h in range(H):
        base = 2.0 * 1.1 ** h                            # 10 % apart from row to row: out of each other's reach
        for w in cols:
            qp, a, b, near = h * W + w, h * W + (w - k) % W, h * W + (w + k) % W, h * W + (w + 1) % W
            for _ in range(20):
                rq = F32(base + rng.uniform(0, 1))
                ra, da = _hug(lut, np.array([qp]), np.array([rq]), np.array([a]), span=0)
                rb, db = _hug(lut, np.array([qp]), np.array([rq]), np.array([b]), span=0)
                if da[0] == db[0]:
                    break
            else:
                continue
            rn, dn = _hug(lut, np.array([qp]), np.array([rq]), np.array([near]), span=0)
            rn = F32(rn[0] * F32(1.0 + 0.3 * (k - 1) * (2.0 * np.pi / W)))        # off the line through the others
            if not N.cham_d(_points(rq, lut[qp]), _points(rn, lut[near])) < da[0]:
                continue
            img[[qp, a, b, near]] = rq, ra[0], rb[0], rn
            out.append((qp, min(a, b), max(a, b), near))
    return img.reshape(H, W), np.array(out)


TIE_SHAPES = ["64E", "VLP16", "2x65536", "4x32768", "64x2048_1deg"]


@pytest.mark.gpu
@pytest.mark.parametrize("sid", TIE_SHAPES)
def test_index_ties_go_to_the_first_pixel_in_raster_order(sid):
    """normals with knn = 3 (the tied pair in the last slot) against oracle.normals, and p2plane with a normal on one
    of the tied pair only: the neighbour is the pair's first pixel in raster order, also where the walk visits the
    other one first (the query in column 0, the pair across the wrap)."""
    from rpcc_b200 import device
    import torch
    cfg, H, W, *_, lut = _geometry(sid)
    rng = np.random.default_rng(3)
    imgs, cases = zip(*[_tie_cases(sid, k, rng) for k in (2, 3, 7)])
    for img, c in zip(imgs, cases):
        assert len(c) >= 4 and (c[:, 0] % W == 0).any(), (sid, len(c))
    radius = 1e4                                         # every neighbourhood is its 3 nearest points
    got, _ = device.normals_batch(_t(np.stack(imgs)), _t(lut), cfg, 3, radius)
    torch.cuda.synchronize()
    got = got.cpu().numpy().reshape(len(imgs), -1, 3)
    from test_gpu_p2plane import _check_normals
    for b, (img, c) in enumerate(zip(imgs, cases)):
        want = _check_normals(img, lut, got[b], 3, radius)
        assert want["has"][c[:, 0]].all(), sid
        idx, cnt = N.knn_sets(img, lut, 3, radius)
        lo, hi = (idx[c[:, 0]] == c[:, 1:2]).any(1), (idx[c[:, 0]] == c[:, 2:3]).any(1)
        assert not hi.any() and lo.mean() >= 0.9, sid       # mostly the tie is the last slot, never the later pixel
    # p2plane: A holds the queries alone, B the tied pairs; the normal sits on the raster-first one
    As, Bs, NB = [], [], []
    for img, c in zip(imgs, cases):
        a, bimg = np.zeros(H * W, F32), np.zeros(H * W, F32)
        a[c[:, 0]] = img.reshape(-1)[c[:, 0]]
        bimg[c[:, 1:3].reshape(-1)] = img.reshape(-1)[c[:, 1:3].reshape(-1)]
        nb = np.zeros((H * W, 3), F32)
        nb[c[:, 1]] = (0.0, 0.6, 0.8)
        As.append(a.reshape(H, W)); Bs.append(bimg.reshape(H, W)); NB.append(nb)
    NA = [np.zeros((H * W, 3), F32) for _ in As]
    m = _p2plane(sid, As, Bs, NA, NB)
    for b in range(len(As)):
        _check_p2plane(sid, As[b], Bs[b], NA[b], NB[b], m[b])
        assert m[b, 2] == 0, (sid, m[b])                   # every query took the neighbour that has the normal


# ----------------------------------------------------------------------------------------------- GPU: DBSCAN
GROUND = np.array([0.0, 0.0, 1.0, 1.0e4], F32)          # a plane 10 km below: every point is a DBSCAN point
EPS = 0.5


def _eps_pairs(sid, direction, e2, rng, max_cases=240):
    """Pairs (query, neighbour) whose cham_d is exactly e2, at eps / r from 1e-4 to 1e-1: the neighbour k rows or
    columns away with r sin(t_k) = eps, i.e. at the last row / column of db_window's window -> (img, list of (qp, cp))."""
    _, H, W, hf, vmax, vmin, lut = _geometry(sid)
    h0 = _foot_row(sid)
    pitch = (np.cos(max(abs(vmax), abs(vmin))) * hf / W) if direction == "col" else (vmax - vmin) / (H - 1)
    kmax = (W - 1) // 2 - 1 if direction == "col" else H - 1
    ks = sorted({int(k) for k in np.geomspace(1e-4, 1e-1, 12) / pitch if 1 <= k <= kmax})
    img = np.zeros(H * W, F32)
    out = []
    nxt = 0                                                  # next free column (col)
    free = np.zeros(W, np.int64)                             # next free row per column (row)
    # row pairs of one k sit in columns more than 0.25 rad apart: further than eps from each other
    cols = np.arange(0, W, max(1, int(np.ceil(0.25 / (np.cos(max(abs(vmax), abs(vmin))) * hf / W)))))
    for i in range(10 * max_cases):
        if len(out) >= max_cases or not ks:
            break
        k = ks[i % len(ks)]
        if direction == "col":
            if nxt + 2 * k + 3 > W:
                break
            qp, cp = h0 * W + nxt, h0 * W + nxt + k
            nxt += 2 * k + 3
        else:
            w = cols[(i // len(ks)) % cols.size]
            if free[w] + k >= H:
                continue
            qp, cp = free[w] * W + w, (free[w] + k) * W + w
            free[w] += k + 2
        a, b = lut[qp].astype(F64), lut[cp].astype(F64)
        r0 = np.sqrt(F64(e2)) / (np.linalg.norm(np.cross(a, b)) / np.linalg.norm(a) / np.linalg.norm(b))
        rq = _ulps(F32(r0), np.arange(-6, 7))
        rc, d = _hug(lut, np.full(rq.size, qp), rq, np.full(rq.size, cp), span=6)
        hit = np.flatnonzero(d == e2)
        if hit.size:
            img[[qp, cp]] = rq[hit[0]], rc[hit[0]]
            out.append((qp, cp))
    return img.reshape(H, W), out


def _device_dbscan(sid, imgs, eps, min_points, cluster_num):
    import torch
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    _, H, W, hf, vmax, vmin, lut = _geometry(sid)
    B = len(imgs)
    lab = torch.empty((B, H * W), dtype=torch.uint8, device="cuda")
    ws = torch.empty((_lib.lib().rpcc_dbscan_workspace_bytes(B, H, W),), dtype=torch.uint8, device="cuda")
    rg, lt, g = _t(np.stack(imgs)), _t(lut), _t(np.tile(GROUND, (B, 1)))      # held until the launch has run
    check(_lib.lib().rpcc_dbscan_segment_batch(ptr(rg), ptr(lt), ptr(g), B, H, W, hf, vmax, vmin, float(eps),
                                               int(min_points), int(cluster_num), THR, ptr(lab), ptr(ws), None))
    torch.cuda.synchronize()
    return lab.cpu().numpy().reshape(B, H, W)


def _eps_of(e2):
    """A double eps with (float)(eps * eps) == e2."""
    eps = float(np.sqrt(F64(e2)))
    for _ in range(64):
        got = F32(eps * eps)
        if got == e2:
            return eps
        eps = float(np.nextafter(eps, np.inf if got < e2 else -np.inf))
    raise AssertionError(e2)


@pytest.mark.gpu
@pytest.mark.parametrize("sid", ENCODER_SHAPES)
def test_dbscan_at_the_eps_edge(sid):
    """Pairs at exactly eps, with e2 one ulp below, at and one ulp above their distance, and min_points 1 and 2: the
    one edge neighbour decides whether both are core (2) and whether they share a cluster (1).  Labels against
    oracle.dbscan.segment."""
    rng = np.random.default_rng(5)
    e2 = F32(EPS * EPS)
    frames = [_eps_pairs(sid, d, e2, rng) for d in ("col", "row")]
    frames = [f for f in frames if f[1]]
    assert sum(len(f[1]) for f in frames) >= 12, sid
    imgs = [f[0] for f in frames]
    lut = _geometry(sid)[-1].reshape(_geometry(sid)[1], _geometry(sid)[2], 3)
    for step in (-1, 0, 1):
        eps = _eps_of(_ulps(e2, step))
        for min_points in (1, 2):
            got = _device_dbscan(sid, imgs, eps, min_points, 252)
            for b, (img, pairs) in enumerate(frames):
                want = odb.segment(img, lut, GROUND, eps, min_points, 252, THR)
                assert np.array_equal(got[b], want), (sid, step, min_points, b, int((got[b] != want).sum()))
                q, c = np.array(pairs).T
                lq, lc = want.reshape(-1)[q], want.reshape(-1)[c]
                if step >= 0:                                # linked: one kept cluster per pair
                    assert np.all(lq == lc) and lq.max() <= 252, (sid, step, min_points)
                elif min_points == 2:                        # not linked: neither is core
                    assert np.all(lq == 253) and np.all(lc == 253), (sid, step, min_points)


@pytest.mark.gpu
def test_encoder_with_dbscan_at_2x65536():
    """The eps-edge pairs through BatchEncoder with DBSCAN, and the same ranges moved by a third of the ring: every
    section and the `.rpcc` bytes equal the oracle's."""
    from rpcc_b200.batch import BatchEncoder
    from rpcc_b200.config import load_compressor_cfg
    sid = "2x65536"
    cfg, H, W, hf, vmax, vmin, lut = _geometry(sid)
    rng = np.random.default_rng(9)
    e2 = F32(EPS * EPS)
    frames = []
    img, pairs = _eps_pairs(sid, "col", e2, rng)            # two rings: no row pairs at this pitch
    for flat in (img.reshape(-1), np.roll(img, W // 3, 1).reshape(-1)):   # and the same ranges on other rays
        sel = np.flatnonzero(flat)
        sel = sel[(sel % W > 2) & (sel % W < W - 3)]          # away from the column seam of the projection
        pts = np.zeros((sel.size, 4), F32)
        pts[:, :3] = _points(flat[sel], lut[sel])
        frames.append(pts)
    ccfg = load_compressor_cfg()
    ccfg.update(segment_method="DBSCAN", DBSCAN_eps=EPS, DBSCAN_min_points=2, cluster_num=252)
    pts = np.concatenate(frames)
    off = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int64)
    g = np.tile(GROUND.astype(F64), (len(frames), 1))
    with BatchEncoder(cfg, accuracy=0.02, compressor_cfg=ccfg, max_batch=len(frames), max_points=pts.shape[0]) as enc:
        out = enc.encode_host(pts, off, g)
        blobs = enc.compress(pts, off, g)
        for b, p in enumerate(frames):
            ri = oracle.project(p, H, W, hf, vmax, vmin)
            seg = odb.segment(ri, lut.reshape(H, W, 3), g[b], EPS, 2, 252, THR)
            assert len(np.unique(seg)) > 5, b                # several pairs linked into clusters
            want = odb.compress_frame(p, cfg, g[b], seg)["sections"]
            got = BatchEncoder.frame_sections(out, b)
            assert set(got) == set(want)
            for key, v in want.items():
                assert got[key] == v, (b, key)
            assert blobs[b] == oracle.write_rpcc(want), b
