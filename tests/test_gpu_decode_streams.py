"""The decoder on streams this package's encoder never writes, and on damaged or mismatched `.rpcc` files.

The decoder is the one part of the codec that reads data from outside the program: files of other writers (a plane
`.rpcc` of the reference carries open3d rows our encoder never produces) and files run with other settings (another
lidar, the other framework).  Every other decoder test decodes what the encoder just wrote, so its label maps, model
rows and symbols all satisfy the encoder's invariants.  Here `_stream` builds canonical streams from arbitrary label
maps, rows and symbols (oracle.extract_contour gives the contour map and idx_sequence), one KIND per decoder code
path, and the tests hold every decode entry point to oracle.decompress_sections bit for bit; then each damage of
DAMAGES must be refused with a ValueError naming the frame, whatever else is in the batch and whatever the decoder
decoded before."""
import functools

import numpy as np
import pytest

import oracle

TILE = 1024            # RPCC_TILE: pixels per tile of the label decoder, the dequantiser and the points writer
MAX_TILES = 1024       # the largest range image rpcc_decode_packed_batch accepts, in tiles
ACC = 0.02
STEP = 2 * ACC
LEVEL_DACC = (0, 0.02, 0.04, 0.06)          # the default yaml's level_delta_acc
LEVEL_ACC = STEP + np.array(LEVEL_DACC)
F32_MIN_NORMAL = np.float32(1.17549435e-38)

# kind -> the code path it is there for
KINDS = {
    "dense": "a run at every pixel: idx_sequence holds H*W entries, a sequence read per pixel",
    "many_labels": "all 254 labels inside tile 0: the per-warp bins of match_any leaders, K = 254",
    "last_tile_only": "labels whose only pixels are in the last tile: offsets carried over every earlier tile",
    "empty": "all label 1 and no symbols: nothing to dequantise, row 1 predicts every pixel",
    "all_ground": "label 0 only: one model row (K padded to 2)",
    "plane_rows": "plane rows for label 0 and some labels >= 2, point rows between, a non-zero row 1",
    "sum_quirk": "rows where (x+y)+z and x+(y+z) disagree about zero: the point-model test's association",
    "subnormal_dot": "rows of subnormal components: subnormal dot products with the rays (built with -ftz=false)",
    "near_parallel": "rows whose dot with some ray is exactly 0 or a few ulps from it (one NaN prediction)",
    "extreme_symbols": "symbols at -32768, -32767, 0 and 32767, every salience level in use",
}


def _cfg(H, W):
    from rpcc_b200 import LidarConfig
    return LidarConfig(hfov_deg=360.0, vmax_deg=10.0, vmin_deg=-25.0, H=H, W=W)


@functools.lru_cache(maxsize=None)
def _lut(H, W):
    return oracle.transform_map(*oracle.lidar_params(_cfg(H, W)))


def _runs(rng, n, lo, hi, max_run):
    """n labels in runs of 1..max_run pixels, each run's label drawn from [lo, hi)."""
    lens = rng.integers(1, max_run + 1, n)
    lens = lens[:np.searchsorted(np.cumsum(lens), n) + 1]
    return np.repeat(rng.integers(lo, hi, lens.size), lens)[:n].astype(np.int32)


def _dot(row, t):
    """The prediction's denominator as the kernel and the oracle round it: ((x*t0) + (y*t1)) + (z*t2) in f32."""
    r = np.asarray(row, np.float32)
    t = np.asarray(t, np.float32)
    return (r[0] * t[..., 0] + r[1] * t[..., 1]) + r[2] * t[..., 2]


def _point_rows(rng, n):
    m = np.zeros((n, 4), np.float32)
    m[:, 3] = rng.uniform(1.0, 80.0, n)
    if n:
        m[0] = (0.0057, -0.0445, -0.999, -1.7938) + rng.normal(0, 1e-3, 4)
    if n > 1:
        m[1] = 0
    return m


def _stream(rng, H, W, kind, nonuniform=False):
    """-> dict(kind, H, W, seg (H,W) i32, model (rows,4) f32, symbols i16, salience u8 | None, sections), canonical:
    rows = highest label + 1 (as model.cu writes), one symbol per pixel of a label other than 1, the contour map and
    idx_sequence from oracle.extract_contour."""
    HW = H * W
    T = (HW + TILE - 1) // TILE
    lut = _lut(H, W).reshape(-1, 3)
    seg = _runs(rng, HW, 0, 20, 40)
    if kind == "dense":
        n = 60
        seg = (np.cumsum(rng.integers(1, n, (H, W)), axis=1) % n).astype(np.int32).ravel()
    elif kind == "many_labels":
        seg[:TILE] = rng.permutation(np.tile(np.arange(254), 5)[:TILE])
    elif kind == "last_tile_only":
        last = (T - 1) * TILE
        seg[last:] = _runs(rng, HW - last, 20, 40, 6)
        seg[last] = 39
    elif kind == "empty":
        seg[:] = 1
    elif kind == "all_ground":
        seg[:] = 0
    elif kind == "extreme_symbols":
        seg = _runs(rng, HW, 0, 10, 40)
        seg[-1] = 9
    rows = int(seg.max()) + 1
    model = _point_rows(rng, rows)
    if kind == "plane_rows":
        for l in [0] + [l for l in range(2, rows) if l % 3 == 0]:
            model[l, :3] = rng.normal(0, 1, 3)
            model[l, 3] = rng.uniform(-20, 20)
        model[1, 3] = rng.uniform(1, 10)
    elif kind == "sum_quirk":
        for l in range(2, rows):
            s = np.float32(rng.uniform(0.5, 4))
            if l % 2:
                model[l, :3] = (np.float32(1e-8) * s, s, -s)      # (x+y)+z == 0 != x+(y+z): a point model
            else:
                model[l, :3] = (s, -s, np.float32(1e-8) * s)      # (x+y)+z != 0 == x+(y+z): a plane
            model[l, 3] = rng.uniform(-30, 30)
    elif kind == "subnormal_dot":
        for l in range(2, rows):
            model[l, :3] = rng.uniform(-3, 3, 3) * 1e-39
            model[l, 3] = -rng.uniform(5, 50) * 1e-39
    elif kind == "near_parallel":
        nan_done = False
        for l in range(2, rows):
            at = np.flatnonzero(seg == l)
            if at.size == 0:
                continue
            t = lut[at[rng.integers(at.size)]]
            if t[1] == t[0]:
                continue
            n = np.array([t[1], -t[0], 0.0], np.float32)       # n . t == 0 exactly: t1*t0 - t0*t1
            if not nan_done:
                model[l] = (n[0], n[1], n[2], 0.0)              # the one NaN: -0 / 0
                nan_done = True
                continue
            if l % 2:
                n[0] = n[0] + 2 * np.spacing(n[0])              # a few ulps off the ray
            model[l] = (n[0], n[1], n[2], rng.uniform(-5, 5))
    seg = seg.reshape(H, W)
    nsym = int((seg != 1).sum())
    if kind == "extreme_symbols":
        symbols = rng.choice(np.array([-32768, -32767, 0, 32767], np.int16), nsym)
    else:
        symbols = rng.integers(-3000, 3000, nsym).astype(np.int16)
    sal = None
    if nonuniform:
        sal = rng.integers(0, len(LEVEL_DACC), rows).astype(np.uint8)
        if kind == "extreme_symbols":
            sal = rng.permutation(np.arange(rows) % len(LEVEL_DACC)).astype(np.uint8)
    sections = oracle.pack_sections(model, seg, symbols, sal)
    _, seq = oracle.extract_contour(seg)
    return dict(kind=kind, H=H, W=W, seg=seg, model=model, symbols=symbols, salience=sal, seq=seq.astype(np.uint16),
                sections=sections, nonuniform=nonuniform)


def _steps(s):
    """Per-label f64 steps of the stream (acc[salience_level[m]] non-uniform, the uniform step otherwise)."""
    return LEVEL_ACC[s["salience"]] if s["salience"] is not None else np.full(len(s["model"]), STEP)


@functools.lru_cache(maxsize=None)
def _streams(H, W, seed=0):
    """Every kind in both frameworks at one shape."""
    rng = np.random.default_rng(seed * 7919 + H * 65537 + W)
    return tuple(_stream(rng, H, W, k, nu) for nu in (False, True) for k in KINDS)


def _want(s):
    """oracle.decompress_sections (and intra_predict inside it) -> (labels, range, xyz) of one stream."""
    rec, xyz, seg = oracle.decompress_sections(s["sections"], _cfg(s["H"], s["W"]), ACC, LEVEL_DACC)
    return seg, rec, xyz


def _same(got, want, what):
    """Bit for bit, except that NaN matches NaN (payloads are not pinned: the x86 oracle's 0.0/0 is 0xFFC00000, the GPU's
    0x7FFFFFFF)."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, what
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), (what, int((np.isnan(got) != nan).sum()))
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32)), (
        what, int((got[~nan].view(np.uint32) != want[~nan].view(np.uint32)).sum()))


# ----------------------------------------------------------------------------------------------- the generator (no GPU)
GEN_SHAPES = [(64, 2000), (40, 31), (3, 1023), (16, 300)]


def _reaches(s):
    """The property each kind is there for, recomputed from the arrays."""
    seg, model, HW = s["seg"], s["model"], s["H"] * s["W"]
    flat = seg.ravel()
    lut = _lut(s["H"], s["W"]).reshape(-1, 3)
    present = np.unique(flat)
    k = s["kind"]
    if k == "dense":
        return s["seq"].size == HW
    if k == "many_labels":
        return len(np.unique(flat[:TILE])) == 254 and len(model) == 254
    if k == "last_tile_only":
        last = (HW - 1) // TILE * TILE
        return bool(set(np.unique(flat[last:]).tolist()) - set(np.unique(flat[:last]).tolist()))
    if k == "empty":
        return bool((flat == 1).all()) and s["symbols"].size == 0
    if k == "all_ground":
        return bool((flat == 0).all()) and len(model) == 1
    if k == "plane_rows":
        planes = [l for l in present if model[l, :3].any()]
        points = [l for l in present if l >= 2 and not model[l, :3].any()]
        return 0 in planes and any(l >= 2 for l in planes) and len(points) > 0 and model[1, 3] != 0
    if k == "sum_quirk":
        m = model[present]
        left = (m[:, 0] + m[:, 1]) + m[:, 2]
        right = m[:, 0] + (m[:, 1] + m[:, 2])
        return bool(((left == 0) & (right != 0)).any() and ((left != 0) & (right == 0)).any())
    if k == "subnormal_dot":
        d = np.concatenate([_dot(model[l], lut[flat == l]) for l in present if l >= 2])
        return bool(((d != 0) & (np.abs(d) < F32_MIN_NORMAL)).any())
    if k == "near_parallel":
        zero_nan = tiny = False
        for l in present:
            if l < 2:
                continue
            t = lut[flat == l]
            d = _dot(model[l], t)
            terms = np.abs(model[l, :3] * t).max(1)
            zero_nan |= bool(((d == 0) & (model[l, 3] == 0)).any())
            tiny |= bool(((d != 0) & (np.abs(d) <= 4 * np.spacing(terms))).any())
        return zero_nan and tiny
    if k == "extreme_symbols":
        ok = {-32768, -32767, 0, 32767} <= set(s["symbols"].tolist())
        if s["salience"] is not None:
            ok &= set(s["salience"].tolist()) == set(range(len(LEVEL_DACC)))
        return ok
    raise KeyError(k)


@pytest.mark.parametrize("shape", GEN_SHAPES, ids=lambda s: "%dx%d" % s)
def test_every_kind_reaches_its_property(shape):
    for s in _streams(*shape):
        assert _reaches(s), (shape, s["kind"], s["nonuniform"])
        assert len(s["model"]) == int(s["seg"].max()) + 1
        assert s["symbols"].size == int((s["seg"] != 1).sum())


@pytest.mark.parametrize("shape", GEN_SHAPES, ids=lambda s: "%dx%d" % s)
def test_every_kind_round_trips_through_the_oracle(shape):
    """recover_map gives the label map back, dequantize consumes every symbol and puts f32(q * step) at the pixels of
    the label-major order."""
    for s in _streams(*shape):
        H, W = shape
        contour = np.unpackbits(np.frombuffer(s["sections"]["contour_map"], np.uint8))[:H * W].reshape(H, W)
        seg = oracle.recover_map(contour, s["seq"])
        assert np.array_equal(seg, s["seg"]), (shape, s["kind"])
        steps = _steps(s)
        res = oracle.dequantize(s["symbols"], seg, steps).ravel()
        flat = seg.ravel()
        order = np.flatnonzero(flat != 1)
        order = order[np.argsort(flat[order], kind="stable")]
        want = (s["symbols"].astype(np.float64) * steps[flat[order]]).astype(np.float32)
        assert np.array_equal(res[order].view(np.uint32), want.view(np.uint32)), (shape, s["kind"])
        assert not res[flat == 1].any()


def test_oracle_dequantize_wants_a_step_per_label():
    seg = np.array([[0, 2, 3]], np.int32)
    with pytest.raises(AssertionError):
        oracle.dequantize(np.zeros(3, np.int16), seg, np.full(3, STEP))
    oracle.dequantize(np.zeros(3, np.int16), seg, np.full(4, STEP))


# ----------------------------------------------------------------------------------------------- kernels, called directly
PACKED_SHAPES = [
    ((64, 2000), "the 64E image"),
    ((40, 31), "W < 32: row starts by p % W"),
    ((3, 1023), "a row start inside tile 0"),
    ((16, 8192), "131 072 pixels, 128 tiles"),
]
LIMIT_SHAPE = (256, 4096)   # 1024 tiles: decode_impl's limit, eight times what the encoder accepts


def _torch():
    import torch
    return torch


def _packed_inputs(streams):
    torch = _torch()
    H, W = streams[0]["H"], streams[0]["W"]
    B = len(streams)
    K = max(max(len(s["model"]) for s in streams), 2)
    contour = np.stack([np.frombuffer(s["sections"]["contour_map"], np.uint8) for s in streams])
    seq = np.concatenate([s["seq"] for s in streams] + [np.zeros(1, np.uint16)])
    sym = np.concatenate([s["symbols"] for s in streams] + [np.zeros(1, np.int16)])
    seq_base = np.concatenate(([0], np.cumsum([s["seq"].size for s in streams]))).astype(np.uint64)
    sym_base = np.concatenate(([0], np.cumsum([s["symbols"].size for s in streams]))).astype(np.uint64)
    model = np.zeros((B, K, 4), np.float32)
    steps = np.full((B, K), STEP)
    for b, s in enumerate(streams):
        model[b, :len(s["model"])] = s["model"]
        steps[b, :len(s["model"])] = _steps(s)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return dict(H=H, W=W, B=B, K=K, contour=dev(contour), seq=dev(seq.view(np.int16)), sym=dev(sym),
                seq_base=dev(seq_base.view(np.int64)), sym_base=dev(sym_base.view(np.int64)), model=dev(model),
                steps=dev(steps), lut=dev(_lut(H, W)), seq_host=seq, sym_host=sym)


def _outputs(x, K=None):
    torch = _torch()
    from rpcc_b200 import _lib
    B, HW = x["B"], x["H"] * x["W"]
    K = K or x["K"]
    return dict(labels=torch.full((B, HW), 0xAB, dtype=torch.uint8, device="cuda"),
                range=torch.full((B, HW), 7.0, dtype=torch.float32, device="cuda"),
                xyz=torch.full((B, HW, 3), 7.0, dtype=torch.float32, device="cuda"),
                book=torch.empty((_lib.lib().rpcc_book_bytes(B, x["H"], x["W"], K),), dtype=torch.uint8, device="cuda"),
                results=torch.zeros((B, 4), dtype=torch.int32, device="cuda"))


def _host(o):
    from rpcc_b200._lib import RESULT_DTYPE
    B = o["results"].shape[0]
    return dict(labels=o["labels"].cpu().numpy(), range=o["range"].cpu().numpy(), xyz=o["xyz"].cpu().numpy(),
                results=o["results"].cpu().numpy().view(np.uint32).copy().view(RESULT_DTYPE).reshape(B))


def _decode_packed(x):
    torch = _torch()
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    o = _outputs(x)
    check(_lib.lib().rpcc_decode_packed_batch(ptr(x["contour"]), ptr(x["seq"]), ptr(x["seq_base"]), ptr(x["sym"]),
                                              ptr(x["sym_base"]), ptr(x["model"]), ptr(x["steps"]), ptr(x["lut"]), x["B"],
                                              x["H"], x["W"], x["K"], ptr(o["labels"]), ptr(o["range"]), ptr(o["xyz"]),
                                              ptr(o["book"]), ptr(o["results"]), None))
    torch.cuda.synchronize()
    return _host(o)


def _check_against_oracle(got, streams, skip=()):
    H, W = streams[0]["H"], streams[0]["W"]
    for b, s in enumerate(streams):
        if b in skip:
            continue
        what = ((H, W), b, s["kind"], s["nonuniform"])
        seg, rec, xyz = _want(s)
        assert np.array_equal(got["labels"][b].reshape(H, W).astype(np.int32), seg), what
        _same(got["range"][b].reshape(H, W), rec, what + ("range",))
        _same(got["xyz"][b].reshape(H, W, 3), xyz, what + ("xyz",))
        # NaN only where the deliberate zero dot with w = 0 is
        assert not np.isnan(rec).any() or s["kind"] == "near_parallel", what
        r = got["results"][b]
        assert int(r["sym_count"]) == len(s["sections"]["residual_quantized"]) // 2, what
        assert int(r["seq_count"]) == len(s["sections"]["idx_sequence"]) // 2, what
        assert int(r["model_rows"]) == len(s["model"]), what
        assert int(r["flags"]) == 0, what


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [p[0] for p in PACKED_SHAPES], ids=[p[1] for p in PACKED_SHAPES])
def test_packed_batch_of_every_kind_matches_the_oracle(shape):
    """One launch of every kind in both frameworks, with a different row count per frame."""
    streams = _streams(*shape)
    assert len({len(s["model"]) for s in streams}) > 5
    got = _decode_packed(_packed_inputs(streams))
    _check_against_oracle(got, streams)
    assert any(np.isnan(_want(s)[1]).any() for s in streams)


@pytest.mark.gpu
def test_packed_batch_at_the_tile_limit():
    """One frame of 1024 tiles (H*W = 1 048 576) decodes; at 1025 tiles the call is refused."""
    torch = _torch()
    from rpcc_b200 import RpccError, _lib
    from rpcc_b200._lib import check, ptr
    H, W = LIMIT_SHAPE
    assert H * W == MAX_TILES * TILE
    s = _stream(np.random.default_rng(5), H, W, "dense")
    x = _packed_inputs([s])
    _check_against_oracle(_decode_packed(x), [s])
    del x
    # 1025 tiles: refused before any launch (the buffers are never touched)
    d = torch.zeros(64, dtype=torch.int64, device="cuda")
    with pytest.raises(RpccError, match="range image too large"):
        check(_lib.lib().rpcc_decode_packed_batch(ptr(d), ptr(d), ptr(d), ptr(d), ptr(d), ptr(d), ptr(d), ptr(d), 1,
                                                  1025, TILE, 2, ptr(d), ptr(d), ptr(d), ptr(d), ptr(d), None))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(40, 31), (3, 1023)], ids=lambda s: "%dx%d" % s)
def test_strided_batch_matches_the_packed_batch(shape):
    """rpcc_decode_batch with seq_stride / sym_stride past every stream, poison after each frame's end, with counts and
    with NULL counts (trusted streams): the same bytes as the packed form."""
    torch = _torch()
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    streams = _streams(*shape)
    x = _packed_inputs(streams)
    want = _decode_packed(x)
    _check_against_oracle(want, streams)
    B = len(streams)
    seq_stride = max(s["seq"].size for s in streams) + 37
    sym_stride = max(s["symbols"].size for s in streams) + 41
    seq = np.full((B, seq_stride), 0xFFFF, np.uint16)       # a label no frame has a row for
    sym = np.full((B, sym_stride), -32768, np.int16)
    for b, s in enumerate(streams):
        seq[b, :s["seq"].size] = s["seq"]
        sym[b, :s["symbols"].size] = s["symbols"]
    seq_n = torch.from_numpy(np.array([s["seq"].size for s in streams], np.int32)).cuda()
    sym_n = torch.from_numpy(np.array([s["symbols"].size for s in streams], np.int32)).cuda()
    d_seq = torch.from_numpy(seq.view(np.int16)).cuda()
    d_sym = torch.from_numpy(sym).cuda()
    for counts in (True, False):
        o = _outputs(x)
        check(_lib.lib().rpcc_decode_batch(ptr(x["contour"]), ptr(d_seq), seq_stride, ptr(seq_n) if counts else None,
                                           ptr(d_sym), sym_stride, ptr(sym_n) if counts else None, ptr(x["model"]),
                                           ptr(x["steps"]), ptr(x["lut"]), B, x["H"], x["W"], x["K"], ptr(o["labels"]),
                                           ptr(o["range"]), ptr(o["xyz"]), ptr(o["book"]), ptr(o["results"]), None))
        torch.cuda.synchronize()
        got = _host(o)
        for k in ("labels", "range", "xyz", "results"):
            assert got[k].tobytes() == want[k].tobytes(), (shape, counts, k)


def _count_bits(contour_bytes, HW):
    """c(p): contour bits in pixels 1..p (pixel 0 always takes seq[0])."""
    bits = np.unpackbits(np.frombuffer(contour_bytes, np.uint8))[:HW].astype(np.int64)
    bits[0] = 0
    return np.cumsum(bits)


@pytest.mark.gpu
def test_packed_batch_on_damaged_sequences():
    """Damaged seqs next to intact frames of the same launch: labels are seq[c(p)] if c(p) < L else 1, then >= K -> 1;
    flag bit 2 exactly where some c(p) >= L, bit 1 exactly where some label >= K; the intact frames as the oracle."""
    H, W = 3, 1023
    HW = H * W
    streams = list(_streams(H, W))
    K = max(len(s["model"]) for s in streams)
    rng = np.random.default_rng(11)
    damaged = {}
    for b in (1, 4, 9, 12, 15):
        s = dict(streams[b])
        seq = s["seq"].astype(np.int64)
        if b == 1:
            seq = seq[:-3]                                        # short: the last pixels run past L
        elif b == 4:
            seq = seq.copy(); seq[rng.integers(seq.size)] = 300   # a label >= K
        elif b == 9:
            seq = np.concatenate((seq, [2, 3]))                   # long: entries no pixel reads
        elif b == 12:
            seq = seq[:seq.size // 2].copy(); seq[0] = K + 1      # both flags
        else:
            seq = seq.copy(); seq[-1] = 253 if K <= 253 else 1
        s["seq"] = seq.astype(np.uint16)
        damaged[b] = s
        streams[b] = s
    got = _decode_packed(_packed_inputs(streams))
    _check_against_oracle(got, streams, skip=damaged)
    for b, s in damaged.items():
        c = _count_bits(s["sections"]["contour_map"], HW)
        L = s["seq"].size
        lab = np.where(c < L, s["seq"][np.minimum(c, max(L - 1, 0))].astype(np.int64), 1)
        want_k = lab >= K
        lab[want_k] = 1
        assert np.array_equal(got["labels"][b].astype(np.int64), lab), b
        flags = int(got["results"][b]["flags"])
        assert bool(flags & 4) == bool((c >= L).any()), (b, flags)
        assert bool(flags & 2) == bool(want_k.any()), (b, flags)
    assert {b for b in damaged if int(got["results"][b]["flags"]) & 4} == {1, 12}
    assert {b for b in damaged if int(got["results"][b]["flags"]) & 2} == {4, 12}


@pytest.mark.gpu
@pytest.mark.parametrize("stats_ready", [0, 1])
def test_dequantize_caller_labels_past_k(stats_ready):
    """rpcc_dequantize_batch on caller label maps with labels >= K: those pixels decode as empty (label 1: no symbol,
    row 1's prediction), flags bit 1 is set for exactly those frames, and every other pixel -- label K-1's in the tiles
    after them too -- takes the symbols the oracle gives it; stats_ready 0 (histograms here) and 1 (rpcc_label_stats_batch
    first) agree."""
    torch = _torch()
    from rpcc_b200 import _lib
    from rpcc_b200._lib import RESULT_DTYPE, check, ptr
    H, W = 3, 1023
    HW = H * W
    rng = np.random.default_rng(3)
    K = 40
    segs = []
    for b in range(3):
        s = _stream(rng, H, W, "dense")
        seg = s["seg"] if b != 1 else s["seg"] % K             # frame 1 has no label >= K
        segs.append(seg.astype(np.int32))
    mapped = [np.where(s >= K, 1, s) for s in segs]
    nsym = [int((m != 1).sum()) for m in mapped]
    symbols = [rng.integers(-32768, 32768, n).astype(np.int16) for n in nsym]
    model = _point_rows(rng, K)[None].repeat(3, 0)
    model[:, 1, 3] = 2.5                                      # row 1 predicts the empty pixels
    model[2, 5] = (0.3, -0.2, 0.9, -4.0)
    steps = np.stack([LEVEL_ACC[rng.integers(0, 4, K)] for _ in range(3)])
    lut = _lut(H, W)
    sym_stride = max(nsym) + 5
    sym = np.zeros((3, sym_stride), np.int16)
    for b in range(3):
        sym[b, :nsym[b]] = symbols[b]
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    labels = dev(np.stack([s.ravel() for s in segs]).astype(np.uint8))
    d_sym, d_n = dev(sym), dev(np.array(nsym, np.int32))
    d_model, d_steps, d_lut = dev(model), dev(steps), dev(lut)
    rng_out = torch.ones((3, HW), dtype=torch.float32, device="cuda")    # ranges in [2^-5, 256): flag bit 0 stays clear
    xyz = torch.empty((3, HW, 3), dtype=torch.float32, device="cuda")
    book = torch.empty((_lib.lib().rpcc_book_bytes(3, H, W, K),), dtype=torch.uint8, device="cuda")
    results = torch.zeros((3, 4), dtype=torch.int32, device="cuda")
    if stats_ready:
        ones = torch.ones((3, HW), dtype=torch.float32, device="cuda")
        check(_lib.lib().rpcc_label_stats_batch(ptr(ones), ptr(labels), 3, H, W, K, ptr(book), None))
    check(_lib.lib().rpcc_dequantize_batch(ptr(labels), ptr(d_sym), sym_stride, ptr(d_n), ptr(d_model), ptr(d_steps),
                                           ptr(d_lut), 3, H, W, K, ptr(rng_out), ptr(xyz), ptr(book), ptr(results),
                                           stats_ready, None))
    torch.cuda.synchronize()
    rec_got, xyz_got = rng_out.cpu().numpy(), xyz.cpu().numpy()
    res = results.cpu().numpy().view(np.uint32).copy().view(RESULT_DTYPE).reshape(3)
    for b in range(3):
        m = mapped[b]
        assert (segs[b] >= K).any() == (b != 1)
        # label K-1 has pixels in a tile after a tile with labels >= K: the case a miscounted histogram shifts
        assert b == 1 or (segs[b].ravel()[:TILE] >= K).any() and (m.ravel()[TILE:] == K - 1).any()
        want = oracle.intra_predict(m, model[b], lut) + oracle.dequantize(symbols[b], m, steps[b])
        _same(rec_got[b].reshape(H, W), want, ("range", b, stats_ready))
        _same(xyz_got[b].reshape(H, W, 3), want[..., None] * lut, ("xyz", b, stats_ready))
        assert int(res["sym_count"][b]) == nsym[b], (b, int(res["sym_count"][b]), nsym[b])
        assert int(res["model_rows"][b]) == int(m.max()) + 1, b
        assert int(res["flags"][b]) == (2 if b != 1 else 0), (b, int(res["flags"][b]))


# ----------------------------------------------------------------------------------------------- the points writer
def _crafted_points(B=1100, H=2, W=512, seed=4):
    """Range images and a lut with rays where (x+y)+z and x+(y+z) disagree about zero, ranges at +-0, NaN, +-inf and
    below zero, every seventh frame with no points; B > 1024 frames carry the row base across points_base_kernel's
    chunks."""
    rng = np.random.default_rng(seed)
    HW = H * W
    lut = _lut(H, W).reshape(-1, 3).copy()
    special = np.array([(1e-8, 1, -1), (1, -1, 1e-8), (1, -1, 0), (0, 0, 0), (-0.5, 0.25, 0.25), (3e-39, 0, 0)],
                       np.float32)
    at = rng.choice(HW, 200, replace=False)
    lut[at] = special[np.arange(at.size) % len(special)]
    r = rng.uniform(0.5, 90, (B, HW)).astype(np.float32)
    pick = rng.random((B, HW))
    r[pick < 0.05] = 0.0
    r[(pick >= 0.05) & (pick < 0.08)] = -0.0
    r[(pick >= 0.08) & (pick < 0.09)] = np.nan
    r[(pick >= 0.09) & (pick < 0.10)] = np.inf
    r[(pick >= 0.10) & (pick < 0.11)] = -np.inf
    r[(pick >= 0.11) & (pick < 0.15)] *= -1
    r[::7] = 0.0
    r[3::7] = -0.0
    inten = rng.uniform(0, 1, (B, HW)).astype(np.float32)
    return r, lut.reshape(H, W, 3), inten


def _points_restated(r, lut, inten):
    with np.errstate(invalid="ignore", over="ignore"):
        xyz = r[..., None] * lut.reshape(1, -1, 3)
        keep = (xyz[..., 0] + xyz[..., 1]) + xyz[..., 2] != 0             # np.sum(point_cloud, -1) != 0
    rows = np.concatenate((xyz, (inten if inten is not None else np.zeros_like(r))[..., None]), -1)
    return rows[keep], np.concatenate(([0], np.cumsum(keep.sum(1)))).astype(np.int64), keep


def test_crafted_points_reach_every_case():
    r, lut, inten = _crafted_points()
    _, base, keep = _points_restated(r, lut, inten)
    t = lut.reshape(-1, 3)
    assert ((t[:, 0] + t[:, 1]) + t[:, 2] == 0).any() and (t[:, 0] + (t[:, 1] + t[:, 2]) != 0).any()
    l, rt = (t[:, 0] + t[:, 1]) + t[:, 2], t[:, 0] + (t[:, 1] + t[:, 2])
    assert ((l == 0) != (rt == 0)).sum() >= 2
    assert (keep.sum(1) == 0).sum() > 100 and r.shape[0] > 1024 and base[-1] > 0
    for v in (np.nan, np.inf, -np.inf):
        assert (np.isnan(r) if v != v else r == v).any()
    assert (np.signbit(r) & (r == 0)).any() and (r < 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("with_intensity", [False, True], ids=["points", "intensity"])
def test_points_out_on_crafted_range_images(with_intensity):
    torch = _torch()
    from rpcc_b200 import _lib
    from rpcc_b200._lib import check, ptr
    r, lut, inten = _crafted_points()
    B, HW = r.shape
    H, W = lut.shape[:2]
    rows = torch.full((B * HW, 4), 7.0, dtype=torch.float32, device="cuda")
    base = torch.zeros((B + 1,), dtype=torch.int64, device="cuda")
    ws = torch.empty((_lib.lib().rpcc_points_workspace_bytes(B, H, W),), dtype=torch.uint8, device="cuda")
    d_r, d_lut, d_i = (torch.from_numpy(a).cuda() for a in (r, np.ascontiguousarray(lut), inten))
    if with_intensity:
        check(_lib.lib().rpcc_points_out_intensity_batch(ptr(d_r), ptr(d_lut), ptr(d_i), B, H, W, ptr(rows), ptr(base),
                                                         ptr(ws), None))
    else:
        check(_lib.lib().rpcc_points_out_batch(ptr(d_r), ptr(d_lut), B, H, W, ptr(rows), ptr(base), ptr(ws), None))
    torch.cuda.synchronize()
    want_rows, want_base, _ = _points_restated(r, lut, inten if with_intensity else None)
    got_base = base.cpu().numpy()
    assert np.array_equal(got_base, want_base)
    _same(rows[:int(got_base[-1])].cpu().numpy(), want_rows, "rows")


# ----------------------------------------------------------------------------------------------- BatchDecoder on files
DEC_SHAPE = (16, 300)       # 4800 pixels: five tiles, the last one partial


def _decoder(nonuniform, method="bzip2", shape=DEC_SHAPE, lidar=None):
    from rpcc_b200.batch import BatchDecoder
    return BatchDecoder(lidar or _cfg(*shape), accuracy=ACC, nonuniform=nonuniform, basic_compressor=method, workers=2)


def _decoded(d):
    return dict(labels=d["labels"].cpu().numpy(), range=d["range"].cpu().numpy(), xyz=d["xyz"].cpu().numpy(),
                points=[p.copy() for p in d["points"]], results=d["results"].copy())


def _check_decoded(got, streams, what):
    for b, s in enumerate(streams):
        w = what + (b, s["kind"])
        seg, rec, xyz = _want(s)
        assert np.array_equal(got["labels"][b].astype(np.int32), seg), w
        _same(got["range"][b], rec, w + ("range",))
        _same(got["xyz"][b], xyz, w + ("xyz",))
        flat = xyz.reshape(-1, 3)
        with np.errstate(invalid="ignore"):
            keep = (flat[:, 0] + flat[:, 1]) + flat[:, 2] != 0
        _same(got["points"][b], np.concatenate((flat[keep], np.zeros((int(keep.sum()), 1), np.float32)), 1),
              w + ("points",))


def _frame_bytes(got, b):
    return b"".join(np.ascontiguousarray(got[k][b]).tobytes() for k in ("labels", "range", "xyz", "points"))


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["bzip2", "deflate"])
@pytest.mark.parametrize("nonuniform", [False, True], ids=["uniform", "nonuniform"])
def test_batch_decoder_on_foreign_files(nonuniform, method):
    """`.rpcc` files written by oracle.write_rpcc from every kind: bit-exact against the oracle, and every frame's bytes
    the same decoded alone, inside the mixed batch (both buffer sets), and alone after that batch of 254 rows."""
    streams = [s for s in _streams(*DEC_SHAPE) if s["nonuniform"] == nonuniform]
    blobs = [oracle.write_rpcc(s["sections"], method) for s in streams]
    alone = []
    for s, blob in zip(streams, blobs):
        with _decoder(nonuniform, method) as dec:
            got = _decoded(dec.decode([blob], want_xyz=True, want_points=True))
            _check_decoded(got, [s], ("alone", method))
            alone.append(_frame_bytes(got, 0))
    with _decoder(nonuniform, method) as dec:
        for buf_set in (0, 1):
            got = _decoded(dec.decode(blobs, want_xyz=True, want_points=True, buf_set=buf_set))
            _check_decoded(got, streams, ("batch", method, buf_set))
            for b in range(len(streams)):
                assert _frame_bytes(got, b) == alone[b], ("batch", buf_set, b)
        for b, blob in enumerate(blobs):
            got = _decoded(dec.decode([blob], want_xyz=True, want_points=True, buf_set=b % 2))
            assert _frame_bytes(got, 0) == alone[b], ("after a 254-row batch", b)


# ----------------------------------------------------------------------------------------------- damaged files
def _damage_frames(nonuniform, shape=DEC_SHAPE, seed=21):
    """Three frames: a plane-row frame and the 254-row frame around one with fewer rows than either."""
    rng = np.random.default_rng(seed)
    a = _stream(rng, *shape, "plane_rows", nonuniform)
    c = _stream(rng, *shape, "many_labels", nonuniform)
    seg = (np.cumsum(rng.integers(1, 12, shape), axis=1) % 12).astype(np.int32)    # a run at every pixel, 12 labels
    rows = int(seg.max()) + 1
    model = _point_rows(rng, rows)
    sym = rng.integers(-3000, 3000, int((seg != 1).sum())).astype(np.int16)
    sal = rng.integers(0, 4, rows).astype(np.uint8) if nonuniform else None
    _, seq = oracle.extract_contour(seg)
    d = dict(kind="dense12", H=shape[0], W=shape[1], seg=seg, model=model, symbols=sym, salience=sal,
             seq=seq.astype(np.uint16), sections=oracle.pack_sections(model, seg, sym, sal), nonuniform=nonuniform)
    assert len(d["model"]) < min(len(a["model"]), len(c["model"]))
    return [a, d, c]


def _relabel(sec, s, value):
    """idx_sequence with one run (of a label other than 1, between neighbours other than `value`) relabelled: the run
    count and the symbol count stay those of the contour map."""
    seq = s["seq"].copy()
    i = next(i for i in range(1, seq.size - 1) if seq[i] != 1 and seq[i - 1] != value and seq[i + 1] != value)
    seq[i] = value
    sec["idx_sequence"] = seq.tobytes()


def _damage(name, s):
    """-> the sections of stream s with the damage applied."""
    sec = dict(s["sections"])
    rows = len(s["model"])
    if name == "label_in_rows_to_K":
        _relabel(sec, s, rows)
    elif name == "label_ge_254":
        _relabel(sec, s, 300)
    elif name == "seq_short":
        sec["idx_sequence"] = sec["idx_sequence"][:-2]
    elif name == "seq_long":
        sec["idx_sequence"] += np.uint16([2]).tobytes()
    elif name == "symbols_short":
        sec["residual_quantized"] = sec["residual_quantized"][:-2]
    elif name == "symbols_long":
        sec["residual_quantized"] += np.int16([5]).tobytes()
    elif name == "contour_short":
        sec["contour_map"] = sec["contour_map"][:-1]
    elif name == "contour_long":
        sec["contour_map"] += b"\x00"
    elif name == "seq_odd":
        sec["idx_sequence"] += b"\x00"
    elif name == "symbols_odd":
        sec["residual_quantized"] += b"\x00"
    elif name == "plane_param_tail":
        sec["plane_param"] += np.float32([1.0]).tobytes()
    elif name == "rows_255":
        sec["plane_param"] = np.concatenate((s["model"], _point_rows(np.random.default_rng(0), 255)[rows:])).tobytes()
        if "salience_level" in sec:
            sec["salience_level"] = np.concatenate((s["salience"], np.zeros(255 - rows, np.uint8))).tobytes()
    elif name == "salience_short":
        sec["salience_level"] = sec["salience_level"][:-1]
    elif name == "salience_long":
        sec["salience_level"] += b"\x00"
    elif name == "salience_level_too_high":
        sal = bytearray(sec["salience_level"])
        sal[len(sal) // 2] = len(LEVEL_DACC)
        sec["salience_level"] = bytes(sal)
    else:
        raise KeyError(name)
    return sec


DAMAGES = ["label_in_rows_to_K", "label_ge_254", "seq_short", "seq_long", "symbols_short", "symbols_long",
           "contour_short", "contour_long", "seq_odd", "symbols_odd", "plane_param_tail", "rows_255"]
SALIENCE_DAMAGES = ["salience_short", "salience_long", "salience_level_too_high"]
DAMAGE_CASES = ([pytest.param(False, d, id="uniform-" + d) for d in DAMAGES]
                + [pytest.param(True, d, id="nonuniform-" + d) for d in DAMAGES + SALIENCE_DAMAGES])


def _refused_in_every_context(dec_factory, good, bad_blob, want_index_re, also=()):
    """The damaged frame 1 of [good0, bad, good2]: in that batch on a fresh decoder, alone on a fresh decoder, and in that
    batch after a batch with more rows on the same decoder; then the decoder still decodes the valid batch bit-exact."""
    blobs, streams = good
    batch = [blobs[0], bad_blob, blobs[2]]
    with dec_factory() as dec:
        with pytest.raises((ValueError,) + tuple(also), match=want_index_re(1)):
            dec.decode(batch, want_xyz=True, want_points=True)
        _check_decoded(_decoded(dec.decode(blobs, want_xyz=True, want_points=True)), streams, ("after",))
    with dec_factory() as dec:
        with pytest.raises((ValueError,) + tuple(also), match=want_index_re(0)):
            dec.decode([bad_blob], want_xyz=True, want_points=True)
        _check_decoded(_decoded(dec.decode(blobs, want_xyz=True, want_points=True)), streams, ("after alone",))
    with dec_factory() as dec:
        dec.decode(blobs + [blobs[2]], want_xyz=True, want_points=True)
        with pytest.raises((ValueError,) + tuple(also), match=want_index_re(1)):
            dec.decode(batch, want_xyz=True, want_points=True)
        _check_decoded(_decoded(dec.decode(blobs, want_xyz=True, want_points=True)), streams, ("after larger K",))


def _index_re(i):
    return r"batch index \[%d\]" % i


@pytest.mark.gpu
@pytest.mark.parametrize("nonuniform,damage", DAMAGE_CASES)
def test_damaged_file_is_refused_whatever_the_batch(nonuniform, damage):
    streams = _damage_frames(nonuniform)
    blobs = [oracle.write_rpcc(s["sections"]) for s in streams]
    bad = oracle.write_rpcc(_damage(damage, streams[1]))
    _refused_in_every_context(lambda: _decoder(nonuniform), (blobs, streams), bad, _index_re)


@pytest.mark.gpu
def test_file_of_another_lidar_is_refused():
    """A 64E file among 32E files given to a 32E decoder (RpccError from the section parser is accepted too)."""
    from rpcc_b200 import RpccError
    rng = np.random.default_rng(8)
    streams = [_stream(rng, 32, 2250, k) for k in ("plane_rows", "dense", "many_labels")]
    blobs = [oracle.write_rpcc(s["sections"]) for s in streams]
    bad = oracle.write_rpcc(_stream(rng, 64, 2000, "plane_rows")["sections"])
    _refused_in_every_context(lambda: _decoder(False, lidar=_cfg(32, 2250)), (blobs, streams), bad,
                              lambda i: r"batch index \[%d\]|librpcc_b200 error" % i, also=(RpccError,))


@pytest.mark.gpu
def test_uniform_file_is_refused_by_a_nonuniform_decoder():
    from rpcc_b200 import RpccError
    streams = _damage_frames(True)
    blobs = [oracle.write_rpcc(s["sections"]) for s in streams]
    uni = dict(streams[1]["sections"])
    del uni["salience_level"]
    _refused_in_every_context(lambda: _decoder(True), (blobs, streams), oracle.write_rpcc(uni),
                              lambda i: r"batch index \[%d\]|librpcc_b200 error" % i, also=(RpccError,))
