"""The intensity section on the GPU (DESIGN.md §4, "Intensity"): the owner pass and gather (project.cu) against
oracle/intensity.py's sequential owner loop, the section's bytes against its quantiser, the five geometry sections
unchanged by it, the round trip through BatchEncoder / BatchDecoder and the tools, the readers that skip the section,
and the errors."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from oracle import intensity as oi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXAMPLE = os.path.join(ROOT, "tests", "golden", "example.bin")
GEOMETRY = ("contour_map", "idx_sequence", "plane_param", "residual_quantized")


def _example():
    return np.fromfile(EXAMPLE, np.float32).reshape(-1, 4)


def _device_owner(frames, lidar):
    import torch
    from rpcc_b200 import device
    from rpcc_b200.lidar import LidarConfig
    pts = torch.from_numpy(np.ascontiguousarray(np.concatenate(frames, 0), np.float32)).cuda()
    off = torch.from_numpy(np.concatenate(([0], np.cumsum([len(f) for f in frames]))).astype(np.int64)).cuda()
    rng, own, inten = device.intensity_owner_batch(pts, off, LidarConfig(lidar))
    torch.cuda.synchronize()
    return rng.cpu().numpy(), own.cpu().numpy(), inten.cpu().numpy()


def _check_owner(frames, lidar):
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    rng, own, inten = _device_owner(frames, lidar)
    for b, f in enumerate(frames):
        ri, want = oi.project_owner(f, H, W, hf, vmax, vmin)
        assert np.array_equal(rng[b], ri)
        assert np.array_equal(own[b], want), (lidar, b, int((own[b] != want).sum()))
        assert np.array_equal(inten[b].view(np.uint32), oi.intensity_image(f, want).view(np.uint32))


def _crafted():
    """Duplicates with different intensities, equal sqrtf(d2) from different d2, and the zero-depth cases."""
    rs = np.random.default_rng(5)
    base = rs.normal(0, 15, (4000, 4)).astype(np.float32)
    base[:, 3] = rs.random(4000, dtype=np.float32)
    dup = base[:500].copy()
    dup[:, 3] = rs.random(500, dtype=np.float32)
    ulp = base[500:900].copy()
    ulp[:, 2] = np.nextafter(ulp[:, 2], np.float32(1e9))          # a different square, mostly the same depth
    ulp[:, 3] += 1
    zero = np.zeros((1, 4), np.float32)
    tiny = np.asarray([[1e-30, 2e-30, 0, 0.5]], np.float32)     # zero depth off column 0
    col0 = np.asarray([[7.0, 0.0, 0.0, 0.1], [6.0, 0.0, 0.0, 0.2]], np.float32)   # (0,0,0)'s pixel
    return [np.concatenate((zero, col0, base, dup, ulp), 0),             # zero before
            np.concatenate((col0[:1], base, zero, col0[1:], dup), 0),   # zero between
            np.concatenate((base, col0, ulp, zero), 0),                 # zero after
            np.concatenate((tiny, base, tiny * 2, np.asarray([[1e-30, 2e-30, 1e-3, 0.7]], np.float32), dup), 0)]


def test_owner_example_and_lidars():
    from rpcc_b200 import synthetic
    _check_owner([_example()], "Velodyne64E")
    for lidar in ("Velodyne64E", "Velodyne32E", "VelodyneVLP16"):
        _check_owner([synthetic.frame(s, lidar)[0] for s in (3, 4)], lidar)


def test_owner_crafted_ties_and_zero_depth():
    _check_owner(_crafted(), "VelodyneVLP16")


def test_owner_uneven_batch():
    from rpcc_b200 import synthetic
    fr = [synthetic.frame(9, "Velodyne64E")[0], _example()[:1000], _example(), np.zeros((0, 4), np.float32),
          synthetic.frame(10, "Velodyne64E")[0][:77777]]
    _check_owner(fr, "Velodyne64E")


def test_pack_bytes_and_flag():
    import torch
    from rpcc_b200 import device
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    rng, own, inten = _device_owner([_example()], "Velodyne64E")
    special = np.asarray([0.005, 0.015, 0.025, -0.005, -0.004, -1, 2.55, 2.555, 2.56, 9, np.nan, np.inf], np.float32)
    im = inten.copy()
    full = np.flatnonzero(rng[0].reshape(-1) != 0)
    im.reshape(-1)[full[:special.size * 5]] = np.tile(special, 5)
    for acc in (0.005, 0.01, 0.025):
        q, base, clamped = device.intensity_pack_batch(torch.from_numpy(np.concatenate((im, inten))).cuda(),
                                                       torch.from_numpy(np.concatenate((rng, rng))).cuda(), 2 * acc)
        q = q.cpu().numpy()
        want0, c0 = oi.intensity_pack(im[0], rng[0], 2 * acc)
        want1, c1 = oi.intensity_pack(inten[0], rng[0], 2 * acc)
        assert np.array_equal(q, np.concatenate((want0, want1)))
        assert clamped.cpu().tolist() == [c0, c1] and c0 and not c1
        # and back, against the oracle's inverse
        labels = torch.from_numpy(np.where(np.concatenate((rng, rng)) != 0, 0, 1).astype(np.uint8)).cuda()
        back = device.intensity_unpack_batch(labels, torch.from_numpy(q).cuda(), base, 2 * acc).cpu().numpy()
        seg = np.where(rng[0] != 0, 0, 1).astype(np.int32)
        assert np.array_equal(back[0], oi.intensity_unpack(want0, seg, 2 * acc))
        assert np.array_equal(back[1], oi.intensity_unpack(want1, seg, 2 * acc))


def _frames():
    from rpcc_b200 import synthetic
    return [_example()] + [synthetic.frame(s, "Velodyne64E")[0] for s in (31, 32)]


def _encode(frames, intensity, **kw):
    from rpcc_b200.batch import BatchEncoder
    pts = np.concatenate(frames, 0)
    off = np.concatenate(([0], np.cumsum([len(f) for f in frames]))).astype(np.int64)
    with BatchEncoder("Velodyne64E", max_batch=4, intensity_accuracy=intensity, **kw) as enc:
        return enc.compress(pts, off)


def _parse(blob, uniform=True, intensity=False):
    from rpcc_b200.compress_utils import parse_bitstream
    return parse_bitstream(blob, uniform=uniform, intensity=intensity)


@pytest.mark.parametrize("kw", [dict(), dict(nonuniform=True), dict(model_method="plane"),
                                dict(compressor_cfg=dict(__import__("rpcc_b200.config", fromlist=["x"]).DEFAULT_COMPRESSOR_CFG,
                                                         segment_method="DBSCAN")),
                                dict(basic_compressor="gzip")])
def test_geometry_sections_unchanged(kw):
    fr = _frames()
    off_ = _encode(fr, None, **kw)
    on = _encode(fr, 0.01, **kw)
    uniform = not kw.get("nonuniform", False)
    for a, b in zip(off_, on):
        assert b.startswith(a)                               # the first five sections are the same bytes
        assert _parse(a, uniform) == _parse(b, uniform)
        assert "intensity" in _parse(b, uniform, True)


def _decode(blobs, intensity):
    from rpcc_b200.batch import BatchDecoder
    with BatchDecoder("Velodyne64E", intensity_accuracy=intensity) as dec:
        out = dec.decode(blobs, want_xyz=False, want_points=True)
        return [p.copy() for p in out["points"]], out["range"].cpu().numpy()


def test_round_trip_and_compatibility():
    fr = _frames()
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    lut = oracle.transform_map(H, W, hf, vmax, vmin)
    plain = _encode(fr, None)
    for acc in (0.005, 0.01, 0.025):
        blobs = _encode(fr, acc)
        rows, rng = _decode(blobs, acc)
        rows0, rng0 = _decode(plain, None)
        rows_skip, rng_skip = _decode(blobs, None)            # geometry only from an intensity file
        assert np.array_equal(rng, rng0) and np.array_equal(rng_skip, rng0)
        for b, f in enumerate(fr):
            assert np.array_equal(rows[b][:, :3], rows0[b][:, :3]) and np.array_equal(rows_skip[b], rows0[b])
            assert not rows0[b][:, 3].any()
            # every row's intensity vs its pixel's owner
            _, own = oi.project_owner(f, H, W, hf, vmax, vmin)
            xyz = rng[b].reshape(-1, 1) * lut.reshape(-1, 3)
            keep = np.flatnonzero((xyz[:, 0] + xyz[:, 1]) + xyz[:, 2] != 0)
            want = oi.intensity_image(f, own).reshape(-1)[keep]
            got = rows[b][:, 3]
            if b == 0 and acc == 0.005:
                assert np.array_equal(got, want)                  # KITTI's 0.01 grid: lossless
            ok = (want >= 0) & (want <= np.float32(255 * 2 * acc))
            assert np.all(np.abs(got[ok].astype(np.float64) - want[ok]) <= acc + 1e-7), acc


def test_errors():
    from rpcc_b200 import _lib
    from rpcc_b200.batch import BatchDecoder, BatchEncoder
    from rpcc_b200.compress_utils import pack_bitstream
    ex = _example()
    plain, with_i = _encode([ex], None)[0], _encode([ex], 0.01)[0]
    for method in ("bzip2", "gzip"):
        with BatchDecoder("Velodyne64E", intensity_accuracy=0.01, basic_compressor=method) as dec:
            with pytest.raises((ValueError, _lib.RpccError), match="intensity"):
                dec.decode([plain], want_xyz=False, want_points=True)
            with pytest.raises((ValueError, _lib.RpccError)):
                dec.decode([with_i[:-7]], want_xyz=False, want_points=True)
    # an intensity section of the wrong length
    secs = _parse(with_i, True, True)
    import bz2
    secs["intensity"] = bz2.compress(bz2.decompress(secs["intensity"])[:-1])
    with BatchDecoder("Velodyne64E", intensity_accuracy=0.01) as dec:
        with pytest.raises(ValueError, match="intensity"):
            dec.decode([pack_bitstream(secs)], want_xyz=False, want_points=True)
    with BatchEncoder("Velodyne64E", max_batch=2, intensity_accuracy=0.01) as enc:
        with pytest.raises(ValueError):
            enc.encode_host(ex[:, :3].copy(), np.asarray([0, len(ex)], np.int64))
        import ctypes as C
        z = np.zeros(1 << 20, np.uint8)
        p = _lib.ptr(z)
        rc = _lib.lib().rpcc_encoder_encode_host(enc._h, _lib.ptr(ex), 4, _lib.ptr(np.asarray([0, len(ex)], np.int64)), 1,
                                                 None, p, p, p, p, 1000, p, 1000, None, None, None)
        assert rc == -1 and b"intensity" in _lib.lib().rpcc_last_error()
        pts3 = np.ascontiguousarray(ex[:, :3])
        rc = _lib.lib().rpcc_encoder_encode_host_intensity(enc._h, _lib.ptr(pts3), 3,
                                                           _lib.ptr(np.asarray([0, len(ex)], np.int64)), 1, None, p, p, p,
                                                           p, 1000, p, 1000, None, None, None, p)
        assert rc == -1 and b"stride" in _lib.lib().rpcc_last_error()


def _run(mod, *args):
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "rpcc_b200.tools." + mod] + list(args), cwd=ROOT, env=env,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


def test_tools_end_to_end(tmp_path):
    from rpcc_b200 import synthetic
    d = tmp_path / "frames"
    d.mkdir()
    names = []
    for i, f in enumerate([_example(), synthetic.frame(41, "Velodyne64E")[0], _example()]):
        n = str(d / ("%02d.bin" % i))
        f.tofile(n)
        names.append(n)
    lst = tmp_path / "list.txt"
    lst.write_text("\n".join(names) + "\n")
    outs = {}
    for batch in ("1", "3"):
        o = tmp_path / ("out%s" % batch)
        _run("compress_datalist", "--datalist", str(lst), "--output_dir", str(o), "--lidar", "Velodyne64E", "--batch", batch,
             "--intensity_accuracy", "0.005")
        from rpcc_b200.tools.compress_datalist import output_path_for
        outs[batch] = [open(output_path_for(str(o), n), "rb").read() for n in names]
    assert outs["1"] == outs["3"]
    single = str(tmp_path / "single.rpcc")
    txt = _run("compress", "--input", names[0], "--output", single, "--lidar", "Velodyne64E", "--intensity_accuracy", "0.005")
    assert "Intensity section" in txt
    assert open(single, "rb").read() == outs["1"][0]
    # decompress.py: with the flag the rows carry the owners' intensities, without it the geometry of the plain file
    rows_i, rows_0 = str(tmp_path / "i.bin"), str(tmp_path / "z.bin")
    _run("decompress", "--input", single, "--output", rows_i, "--lidar", "Velodyne64E", "--intensity_accuracy", "0.005")
    _run("decompress", "--input", single, "--output", rows_0, "--lidar", "Velodyne64E")
    plain = str(tmp_path / "plain.rpcc")
    _run("compress", "--input", names[0], "--output", plain, "--lidar", "Velodyne64E")
    rows_p = str(tmp_path / "p.bin")
    _run("decompress", "--input", plain, "--output", rows_p, "--lidar", "Velodyne64E")
    a, z, p = (np.fromfile(x, np.float32).reshape(-1, 4) for x in (rows_i, rows_0, rows_p))
    assert np.array_equal(z, p) and np.array_equal(a[:, :3], p[:, :3])
    # decompress_datalist writes the same rows as decompress.py
    lst2 = tmp_path / "list2.txt"
    from rpcc_b200.tools.compress_datalist import output_path_for
    lst2.write_text(output_path_for(str(tmp_path / "out1"), names[0]) + "\n")
    od = tmp_path / "dec"
    _run("decompress_datalist", "--datalist", str(lst2), "--output_dir", str(od), "--lidar", "Velodyne64E",
         "--intensity_accuracy", "0.005")
    from rpcc_b200.tools.decompress_datalist import output_path_for as dec_path
    got = np.fromfile(dec_path(str(od), str(lst2.read_text().strip())), np.float32).reshape(-1, 4)
    assert np.array_equal(got, a)
    H, W, hf, vmax, vmin = oracle.lidar_params("Velodyne64E")
    ex = _example()
    _, own = oi.project_owner(ex, H, W, hf, vmax, vmin)
    assert set(np.unique(a[:, 3])) <= set(np.unique(ex[:, 3]))
    assert a[:, 3].any()


def test_reference_decoder_reads_the_geometry(tmp_path):
    """Where the reference is staged, its own tools/decompress.py decodes an intensity file to the plain file's rows."""
    runner = os.path.join(ROOT, "baseline", "run_reference_tool.py")
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "R-PCC", "tools")):
        pytest.skip("baseline/_ref/R-PCC not staged (python baseline/stage_reference.py where /root/reference exists)")
    ex = str(tmp_path / "f.bin")
    _example().tofile(ex)
    blobs = {}
    for name, extra in (("i", ["--intensity_accuracy", "0.01"]), ("p", [])):
        out = str(tmp_path / (name + ".rpcc"))
        _run("compress", "--input", ex, "--output", out, "--lidar", "Velodyne64E", *extra)
        dec = str(tmp_path / (name + ".bin"))
        r = subprocess.run([sys.executable, runner, "--ops", "b200", "--tool", "decompress", "--", "--input", out, "--output",
                            dec, "--lidar", "Velodyne64E"], cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT),
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        blobs[name] = open(dec, "rb").read()
    assert blobs["i"] == blobs["p"]
