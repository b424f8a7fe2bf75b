"""CPU-side checks: the C ABI library builds, loads and exports every symbol the header declares;
compute entry points fail loudly without a GPU (no fallback); bitstream / entropy / config /
sharding host logic."""
import os
import re

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import rpcc_b200
    lib = rpcc_b200.lib()
    hdr = open(os.path.join(ROOT, "include", "rpcc_b200.h")).read()
    names = sorted(set(re.findall(r"RPCC_API[^;(]*?\b(rpcc_\w+)\s*\(", hdr)))
    assert len(names) >= 40
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert lib.rpcc_version() >= 100
    assert isinstance(rpcc_b200.launch_count(), int)


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import rpcc_b200
    from rpcc_b200.plugin import dataset_utils_cpp
    pts = np.random.rand(100, 3).astype(np.float32)
    with pytest.raises(rpcc_b200.RpccError):
        dataset_utils_cpp.point_cloud_to_range_image_even(pts, 64, 2000, 6.28, 0.03, -0.43)
    from rpcc_b200.batch import BatchEncoder
    with pytest.raises((rpcc_b200.RpccError, RuntimeError, AssertionError)):
        BatchEncoder("Velodyne64E", max_batch=1, device=0)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "r-pcc_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", src, re.M), f
                assert "liborc" not in src, f


def test_transform_map_identical_to_reference_formula():
    import rpcc_b200
    for name in ("Velodyne64E", "Velodyne32E", "VelodyneVLP16"):
        cfg = rpcc_b200.LidarConfig(name)
        H, W, hf, vmax, vmin = oracle.lidar_params(name)
        assert (cfg.H, cfg.W) == (H, W)
        assert np.array_equal(cfg.transform_map(), oracle.transform_map(H, W, hf, vmax, vmin))


def test_bitstream_layout_roundtrip():
    from rpcc_b200.compress_utils import BasicCompressor, pack_bitstream, parse_bitstream
    g = np.random.default_rng(0)
    raw = {"salience_level": g.integers(0, 4, 102).astype(np.uint8).tobytes(),
           "contour_map": g.integers(0, 255, 16000).astype(np.uint8).tobytes(),
           "idx_sequence": g.integers(0, 102, 6000).astype(np.uint16).tobytes(),
           "plane_param": g.standard_normal(408).astype(np.float32).tobytes(),
           "residual_quantized": g.integers(-100, 100, 94000).astype(np.int16).tobytes()}
    for method in ("bzip2", "gzip", "deflate", "lz4"):
        bc = BasicCompressor(method_name=method, gzip_mtime=0)
        for uniform in (True, False):
            comp = bc.compress_dict(raw)
            blob = pack_bitstream(comp, uniform=uniform)
            back = bc.decompress_dict(parse_bitstream(blob, uniform=uniform))
            for k in raw:
                if k == "salience_level" and uniform:
                    assert k not in back
                else:
                    assert back[k] == raw[k], (method, k)
    # same bytes as the oracle's writer (which restates utils/compress_utils.py:167-179)
    bc = BasicCompressor(method_name="bzip2")
    sec = {k: v for k, v in raw.items() if k != "salience_level"}
    assert pack_bitstream(bc.compress_dict(sec), uniform=True) == oracle.write_rpcc(sec, "bzip2")


def test_config_defaults_and_overrides(tmp_path):
    from rpcc_b200.config import load_compressor_cfg
    cfg = load_compressor_cfg()
    assert cfg.accuracy == 0.02 and cfg.cluster_num == 100 and cfg.basic_compressor == "bzip2"
    assert cfg["level_key_point_num"] == [30, 10, 3, 0]
    p = tmp_path / "c.yaml"
    p.write_text("accuracy: 0.05\nbasic_compressor: 'deflate'\n")
    cfg = load_compressor_cfg(str(p))
    assert cfg.accuracy == 0.05 and cfg.basic_compressor == "deflate" and cfg.cluster_num == 100


def test_synthetic_frames_deterministic_and_in_spec():
    from rpcc_b200 import synthetic
    a, ga = synthetic.frame(7)
    b, gb = synthetic.frame(7)
    assert np.array_equal(a, b) and np.array_equal(ga, gb)
    assert a.dtype == np.float32 and a.shape[1] == 4 and 90000 < a.shape[0] < 140000
    r = np.linalg.norm(a[:, :3], axis=1)
    assert r.min() >= 1.49 and r.max() <= 80.01
    assert (a[:, 2] < -1.5).sum() >= 800
    assert not np.any(np.all(a[:, :3] == 0, axis=1))
    assert abs(np.linalg.norm(ga[:3]) - 1) < 1e-12


def test_shard_ranges_partition():
    from rpcc_b200.shard import shard_range
    for n in (0, 1, 7, 8192, 8193):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_output_path_rule_matches_reference_quirk():
    from rpcc_b200.tools.compress_datalist import output_path_for
    # str.replace of the extension text anywhere in the path (reference tools/compress_datalist.py:140, SURVEY C12)
    assert output_path_for("out", "/data/kitti/000001.bin") == "out/data/kitti/000001.rpcc"
    assert output_path_for("out", "/data/bin_files/000001.bin") == "out/data/rpcc_files/000001.rpcc"


def test_bzip2_work_factor_does_not_change_the_bytes():
    """The label-sequence section is sent to libbz2 with its own work factor (host entropy stage, DESIGN.md): the bytes
    must be bz2.compress's -- on repetitive sequences long enough to take the tuned path, on short ones, on empty input."""
    import bz2
    from rpcc_b200.compress_utils import BasicCompressor
    bc = BasicCompressor(method_name="bzip2")
    rng = np.random.default_rng(7)
    runs = np.repeat(rng.integers(0, 102, 6000), rng.integers(1, 4, 6000)).astype(np.uint16)
    cases = [np.tile(np.array([0, 5, 0, 7], np.uint16), 20000), runs, np.tile(runs, 4), np.arange(3000, dtype=np.uint16),
             np.zeros(0, np.uint16)]
    for c in cases:
        raw = c.tobytes()
        assert bc.compress(raw, section="idx_sequence") == bz2.compress(raw)
        assert bc.compress(c, section="idx_sequence") == bz2.compress(raw)
        assert bc.compress(raw, section="residual_quantized") == bz2.compress(raw)
        assert bc.compress(raw) == bz2.compress(raw)
    assert BasicCompressor.bzip2_compress(cases[0].tobytes(), 1) == bz2.compress(cases[0].tobytes())
    assert BasicCompressor.bzip2_compress(cases[0].tobytes(), 250) == bz2.compress(cases[0].tobytes())


def test_default_workers_split_the_cores_over_the_local_ranks(monkeypatch):
    """Host entropy-coder threads: all cores but one for a single process, an even share under torchrun."""
    from rpcc_b200 import batch
    monkeypatch.setattr(os, "cpu_count", lambda: 32)
    monkeypatch.delenv("LOCAL_WORLD_SIZE", raising=False)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    assert batch.default_workers() == 31
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "8")
    assert batch.default_workers() == 3
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "64")
    assert batch.default_workers() == 1
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "junk")
    assert batch.default_workers() == 31


def test_native_packer_writes_the_bytes_python_bz2_would(tmp_path):
    """csrc/hostio.cu (host-only code: runs without a GPU): the native entropy pool must write, for every frame of an
    encode_host-shaped result, exactly save_compressed_bitstream(compress_dict(...)) of utils/compress_utils.py:167-179,
    255-310 -- uniform and non-uniform, to files and to memory -- and rpcc_unpack_rpcc / rpcc_read_bin_xyz must invert /
    match numpy."""
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import RESULT_DTYPE
    from rpcc_b200.hostio import Packer, read_bin_xyz, unpack_rpcc
    B, K = 3, 102
    frames = [synthetic.frame(60 + i, "VelodyneVLP16") for i in range(B)]
    secs = [oracle.compress_frame(p, "VelodyneVLP16", g, nonuniform=True)["sections"] for p, g in frames]
    cb = len(secs[0]["contour_map"])
    res = np.zeros(B, RESULT_DTYPE)
    model, contour, sal = np.zeros((B, K, 4), np.float32), np.zeros((B, cb), np.uint8), np.zeros((B, K), np.uint8)
    seq, sym = [], []
    for b, s in enumerate(secs):
        rows = len(s["plane_param"]) // 16
        res[b] = (len(s["residual_quantized"]) // 2, len(s["idx_sequence"]) // 2, rows, 0)
        model[b, :rows] = np.frombuffer(s["plane_param"], np.float32).reshape(-1, 4)
        contour[b] = np.frombuffer(s["contour_map"], np.uint8)
        sal[b, :rows] = np.frombuffer(s["salience_level"], np.uint8)
        seq.append(np.frombuffer(s["idx_sequence"], np.uint16))
        sym.append(np.frombuffer(s["residual_quantized"], np.int16))
    enc = dict(results=res, model=model, contour=contour, seq=np.concatenate(seq), symbols=np.concatenate(sym), salience=sal)
    pk = Packer(3)
    paths = [str(tmp_path / ("%d.rpcc" % b)) for b in range(B)]
    sizes, blobs = pk.wait(pk.submit(enc, K, False, paths, keep=True))
    for b in range(B):
        want = oracle.write_rpcc(secs[b])
        assert open(paths[b], "rb").read() == want and blobs[b, :sizes[b]].tobytes() == want
        back = unpack_rpcc(want, False, 1 << 20)
        assert all(back[k].tobytes() == secs[b][k] for k in secs[b])
    enc["salience"] = None
    sizes, blobs = pk.wait(pk.submit(enc, K, True, None, keep=True))
    for b in range(B):
        s = {k: v for k, v in secs[b].items() if k != "salience_level"}
        assert blobs[b, :sizes[b]].tobytes() == oracle.write_rpcc(s)
    with pytest.raises(Exception):
        pk.wait(pk.submit(enc, K, True, [str(tmp_path / "no_such_dir" / "x.rpcc")] * B))
    pk.close()
    f = tmp_path / "a.bin"
    frames[0][0].tofile(str(f))
    dst = np.zeros((frames[0][0].shape[0] + 5, 3), np.float32)
    assert read_bin_xyz(str(f), dst) == frames[0][0].shape[0]
    assert np.array_equal(dst[:frames[0][0].shape[0]], frames[0][0][:, :3])
    with pytest.raises(Exception):
        read_bin_xyz(str(f), dst[:10])


def _own_bz2(raw):
    import ctypes as C
    import rpcc_b200
    raw = bytes(raw)
    cap = len(raw) + len(raw) // 100 + 700
    dst = C.create_string_buffer(cap)
    n = C.c_size_t(0)
    rc = rpcc_b200.lib().rpcc_bz2_compress(raw, len(raw), dst, cap, C.byref(n))
    return rc, dst.raw[:n.value]


def test_own_bzip2_encoder_writes_libbz2_bytes():
    """csrc/bz2enc.cu must write exactly what bz2.compress (libbz2, level 9) writes -- the reference's coder,
    utils/compress_utils.py:296-298 -- or decline (1): edge cases of the run-length pass and of the table-count thresholds,
    random / low-entropy / int16 / run-heavy inputs of many sizes, every section of real frames, and the inputs it must
    leave to libbz2 (blocks that repeat a shorter string, more than one block)."""
    import bz2
    from rpcc_b200 import synthetic
    rng = np.random.default_rng(11)
    cases = [b"", b"a", b"ab", b"abc", b"aaaa", b"aaaab", b"aaaaa" * 3 + b"b", b"abracadabra", bytes(range(256)),
             bytes(range(256)) * 3 + b"x", b"\x00" * 70000 + b"\x01"]
    for L in (3, 4, 5, 254, 255, 256, 258, 259, 260, 510, 511, 600, 1020):
        cases.append(b"x" * L + b"y")
        cases.append(b"y" + b"x" * L)
    for n in (5, 50, 199, 200, 201, 599, 600, 1199, 1200, 2399, 2400, 10000, 70000):     # nMTF thresholds: 200/600/1200/2400
        cases.append(rng.integers(0, 256, n).astype(np.uint8).tobytes())
        cases.append(rng.integers(0, 3, n).astype(np.uint8).tobytes())
        cases.append(rng.integers(-30, 30, n // 2 + 1).astype(np.int16).tobytes())
        cases.append(np.repeat(rng.integers(0, 100, n // 7 + 1), rng.integers(1, 600, n // 7 + 1)).astype(np.uint8).tobytes()[:n])
        cases.append(rng.integers(0, 102, n // 2 + 1).astype(np.uint16).tobytes())
    for lidar in ("Velodyne64E", "VelodyneVLP16"):
        for nu in (False, True):
            p, g = synthetic.frame(5, lidar)
            cases.extend(oracle.compress_frame(p, lidar, g, nonuniform=nu)["sections"].values())
    done = 0
    for c in cases:
        rc, out = _own_bz2(c)
        assert rc in (0, 1), rc
        if rc == 0:
            assert out == bz2.compress(bytes(c)), (len(c), bytes(c[:16]))
            done += 1
    assert done >= len(cases) - 2
    # declined: whole repetitions of a shorter string (identical rotations: libbz2's order among them is its own), two blocks
    assert _own_bz2(b"abcabcabc")[0] == 1 and _own_bz2(b"ab" * 5000)[0] == 1
    assert _own_bz2(bytes(1020))[0] == 1                    # 4 x 255 zeros: the run-length pass makes a period of five of them
    assert _own_bz2(bytes(1000))[0] == 0 and _own_bz2(bytes(1000))[1] == bz2.compress(bytes(1000))
    assert _own_bz2(rng.integers(0, 256, 950000).astype(np.uint8).tobytes())[0] == 1


def _own_unbz2(stream, cap):
    import ctypes as C
    import rpcc_b200
    dst = C.create_string_buffer(max(cap, 1))
    n = C.c_size_t(0)
    rc = rpcc_b200.lib().rpcc_bz2_decompress(bytes(stream), len(stream), dst, cap, C.byref(n))
    return rc, dst.raw[:n.value]


def test_own_bzip2_decoder_inverts_libbz2():
    """csrc/bz2dec.cu must return what bz2.decompress returns (the reference's decoder, utils/compress_utils.py:300-302)
    for every stream bz2.compress writes: all levels, empty input, run-length edge cases, several blocks, every section of
    real frames; it must refuse (1, the caller then asks libbz2) a damaged stream or a bad CRC, and report a short
    destination."""
    import bz2
    from rpcc_b200 import synthetic
    rng = np.random.default_rng(12)
    cases = [b"", b"a", b"aaaa", b"aaaaa", b"a" * 259, b"a" * 260, b"a" * 1000, bytes(range(256)) * 10, b"ab" * 5000,
             b"\x00" * 70000 + b"\x01"]
    for n in (5, 199, 600, 2400, 10000, 70000):
        cases.append(rng.integers(0, 256, n).astype(np.uint8).tobytes())
        cases.append(rng.integers(0, 3, n).astype(np.uint8).tobytes())
        cases.append(rng.integers(-30, 30, n // 2 + 1).astype(np.int16).tobytes())
        cases.append(np.repeat(rng.integers(0, 100, n // 7 + 1), rng.integers(1, 600, n // 7 + 1)).astype(np.uint8).tobytes()[:n])
    cases.append(rng.normal(0, 20, 1_100_000).round().astype(np.int16).tobytes())            # three blocks at level 9
    for lidar in ("Velodyne64E", "VelodyneVLP16"):
        p, g = synthetic.frame(6, lidar)
        cases.extend(bytes(v) for v in oracle.compress_frame(p, lidar, g, nonuniform=True)["sections"].values())
    for i, c in enumerate(cases):
        for level in ((9, 1 + i % 8) if len(c) < 200000 else (9,)):
            rc, out = _own_unbz2(bz2.compress(c, level), len(c) + 8)
            assert rc == 0 and out == c, (i, len(c), level, rc)
    good = bz2.compress(cases[-1])
    assert _own_unbz2(good, len(cases[-1]) - 1)[0] < 0                         # destination too small
    bad = bytearray(good)
    bad[len(bad) // 2] ^= 0x10
    assert _own_unbz2(bytes(bad), len(cases[-1]) + 8)[0] != 0                  # damaged: declined, never "ok"
    assert _own_unbz2(good[:len(good) // 2], len(cases[-1]) + 8)[0] == 1       # truncated
    assert _own_unbz2(b"BZh9" + b"\x00" * 20, 100)[0] == 1 and _own_unbz2(b"not a stream", 100)[0] == 1


@pytest.mark.parametrize("coder", ["auto", "own", "libbz2"])
def test_packer_coders_agree(tmp_path, monkeypatch, coder):
    """The entropy pool may use libbz2, the library's own encoder, or whichever it measures as cheaper per section: the
    files are the same."""
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import RESULT_DTYPE
    from rpcc_b200.hostio import Packer
    monkeypatch.setenv("RPCC_BZ2_CODER", coder)
    B, K = 6, 102
    secs = []
    for i in range(B):
        p, g = synthetic.frame(80 + i % 3, "VelodyneVLP16")
        secs.append(oracle.compress_frame(p, "VelodyneVLP16", g)["sections"])
    cb = len(secs[0]["contour_map"])
    res = np.zeros(B, RESULT_DTYPE)
    model, contour = np.zeros((B, K, 4), np.float32), np.zeros((B, cb), np.uint8)
    seq, sym = [], []
    for b, s in enumerate(secs):
        rows = len(s["plane_param"]) // 16
        res[b] = (len(s["residual_quantized"]) // 2, len(s["idx_sequence"]) // 2, rows, 0)
        model[b, :rows] = np.frombuffer(s["plane_param"], np.float32).reshape(-1, 4)
        contour[b] = np.frombuffer(s["contour_map"], np.uint8)
        seq.append(np.frombuffer(s["idx_sequence"], np.uint16))
        sym.append(np.frombuffer(s["residual_quantized"], np.int16))
    enc = dict(results=res, model=model, contour=contour, seq=np.concatenate(seq), symbols=np.concatenate(sym), salience=None)
    pk = Packer(1, "bzip2")                                  # one worker: frames 0, 1, 2.. go through the probing sequence
    sizes, blobs = pk.wait(pk.submit(enc, K, True, None, keep=True))
    pk.close()
    for b in range(B):
        assert blobs[b, :sizes[b]].tobytes() == oracle.write_rpcc(secs[b]), (coder, b)


def test_cpulist_parsing_and_numa_binding_is_harmless_without_topology(tmp_path):
    """shard.bind_to_gpu_numa: the kernel's cpulist format, and no effect (and no exception) where the GPU's sysfs node
    is missing -- this container has neither a GPU nor a NUMA topology."""
    from rpcc_b200.shard import bind_to_gpu_numa, parse_cpulist
    assert parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert parse_cpulist("") == set()
    before = os.sched_getaffinity(0)
    assert bind_to_gpu_numa(0, sysfs=str(tmp_path)) is None
    assert os.sched_getaffinity(0) == before
