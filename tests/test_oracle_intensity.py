"""The intensity definition (DESIGN.md §4, "Intensity") as oracle/intensity.py restates it: its projection against the C
oracle's, its sequential owner loop against the closed form of the owner rule on small hand-built point lists (ties,
equal depths from different squared depths, zero-depth re-openings), and the quantiser (half-points, negatives,
clamping, NaN).  No GPU."""
import math

import numpy as np
import pytest

import oracle
from oracle import intensity

LIDAR = "VelodyneVLP16"


def _geo():
    return oracle.lidar_params(LIDAR)


def _pixel(p):
    """The pixel a point lands on and its depth bits: orc_project on the point alone, and for a zero-depth point the
    reference's expressions restated in float32 (it leaves no trace in the image)."""
    H, W, hf, vmax, vmin = _geo()
    ri = oracle.project(np.asarray([p], np.float32), H, W, hf, vmax, vmin)
    x, y, z = (np.float32(v) for v in p[:3])
    d = np.sqrt(np.float32(x * x + y * y) + np.float32(z * z), dtype=np.float32)
    if d != 0:
        pix = int(np.flatnonzero(ri.reshape(-1) != 0)[0])
        return pix, d.view(np.uint32)
    ha = np.float32(math.atan2(float(y), float(x)))
    if ha < 0:
        ha = np.float32(float(ha) + 2 * 3.14159265)
    va = np.float32(math.atan2(float(z), float(np.sqrt(np.float32(x * x + y * y), dtype=np.float32))))
    col = int(np.round(np.float32(np.float32(ha / np.float32(hf)) * np.float32(W)))) % W
    vres = np.float32(np.float32(np.float32(vmax) - np.float32(vmin)) / np.float32(H - 1))
    row = min(max(int(np.round(np.float32(np.float32(va - np.float32(vmin)) / vres))), 0), H - 1)
    return row * W + col, np.uint32(0)


def _owner_by_rule(points):
    """Owner = smallest index after the pixel's last zero-depth point whose depth has the pixel's final range bits."""
    H, W, hf, vmax, vmin = _geo()
    ri = oracle.project(points, H, W, hf, vmax, vmin).reshape(-1)
    owner = np.full(H * W, -1, np.int64)
    last_zero = {}
    per_pix = {}
    for i, p in enumerate(points):
        pix, bits = _pixel(p)
        if bits == 0:
            last_zero[pix] = i
        per_pix.setdefault(pix, []).append((i, bits))
    for pix, lst in per_pix.items():
        if ri[pix] == 0:
            continue
        z = last_zero.get(pix, -1)
        owner[pix] = min(i for i, b in lst if i > z and b == ri[pix:pix + 1].view(np.uint32)[0])
    return owner


def _pt(px, r, it, jitter=0.0):
    """A point at range r towards a fixed direction (azimuth px * 0.02 rad, elevation 0), intensity it."""
    a = px * 0.02
    return [r * math.cos(a) + jitter, r * math.sin(a), 0.0, it]


CASES = {
    "ties_go_to_the_earlier_point": [_pt(1, 10, 0.1), _pt(1, 10, 0.2), _pt(1, 9, 0.3), _pt(1, 9, 0.4), _pt(1, 11, 0.5)],
    "first_store_then_smaller": [_pt(2, 12, 0.1), _pt(2, 11, 0.2), _pt(2, 13, 0.3), _pt(3, 5, 0.4)],
    "zero_before": [[0, 0, 0, 0.9], _pt(0, 7, 0.1), _pt(0, 6, 0.2)],
    "zero_between": [_pt(0, 5, 0.1), [0, 0, 0, 0.9], _pt(0, 7, 0.2), _pt(0, 8, 0.3)],
    "zero_after": [_pt(0, 5, 0.1), _pt(0, 4, 0.2), [0, 0, 0, 0.9]],
    "tiny_zero_depth_off_column_0": [[1e-30, 1e-30, 0, 0.5], [3.0, 3.0, 0.0, 0.1], [1e-30, 1e-30, 0, 0.6],
                                     [4.0, 4.0, 0.0, 0.2]],
}


@pytest.mark.parametrize("lidar", ["Velodyne64E", "Velodyne32E", "VelodyneVLP16"])
def test_range_image_equals_the_c_oracle(lidar):
    """The restated pixel derivation puts every point where orc_project does: the two range images are bit-equal."""
    import os
    from rpcc_b200 import synthetic
    H, W, hf, vmax, vmin = oracle.lidar_params(lidar)
    frames = [synthetic.frame(5, lidar)[0]]
    if lidar == "Velodyne64E":
        frames.append(np.fromfile(os.path.join(os.path.dirname(__file__), "golden", "example.bin"),
                                  np.float32).reshape(-1, 4))
    for f in frames:
        ri, own = intensity.project_owner(f, H, W, hf, vmax, vmin)
        assert np.array_equal(ri.view(np.uint32), oracle.project(f, H, W, hf, vmax, vmin).view(np.uint32))
        assert np.array_equal(own >= 0, ri != 0)


@pytest.mark.parametrize("name", sorted(CASES))
def test_owner_rule(name):
    pts = np.asarray(CASES[name], np.float32)
    H, W, hf, vmax, vmin = _geo()
    ri, own = intensity.project_owner(pts, H, W, hf, vmax, vmin)
    assert np.array_equal(ri, oracle.project(pts, H, W, hf, vmax, vmin))
    assert np.array_equal(own.reshape(-1), _owner_by_rule(pts)), name


def test_equal_depth_from_different_squares_is_a_tie():
    """Two points whose x*x+y*y+z*z differ by an ulp but whose sqrtf agrees: the earlier one owns the pixel, even when the
    later one has the smaller square."""
    base = np.float32(10.0)
    found = None
    for z in np.linspace(1e-3, 4e-3, 64, dtype=np.float32):
        d2a = np.float32(np.float32(base * base) + np.float32(z * z))
        if d2a != np.float32(base * base) and np.sqrt(d2a, dtype=np.float32) == base:
            found = z
            break
    assert found is not None
    pts = np.asarray([[base, 0, found, 0.25], [base, 0, 0, 0.75]], np.float32)   # the later point has the smaller square
    H, W, hf, vmax, vmin = _geo()
    _, own = intensity.project_owner(pts, H, W, hf, vmax, vmin)
    assert own.reshape(-1).max() == 0 and np.array_equal(own.reshape(-1), _owner_by_rule(pts))


def _q_by_rule(v, step):
    if math.isnan(v):
        return 0, False
    q = math.copysign(float(np.floor(abs(v / step) + 0.5)), v)     # round half away from zero, in f64
    return min(max(q, 0), 255), q < 0 or q > 255


@pytest.mark.parametrize("acc", [0.005, 0.01, 0.025, 0.5])
def test_quantiser(acc):
    step = 2 * acc
    vals = [0.0, step / 2, 1.5 * step, 2.5 * step, -step / 2, -0.4 * step, -3 * step, 255 * step, 255.5 * step,
            300 * step, float("nan"), float("inf"), 0.37, 0.99]
    vals = np.asarray(vals, np.float32)
    ri = np.ones(vals.size, np.float32)
    ri[3] = 0                                             # an empty pixel: no byte
    q, clamped = intensity.intensity_pack(vals, ri, step)
    want = [_q_by_rule(float(v), step) for i, v in enumerate(vals) if ri[i] != 0]
    assert q.tolist() == [w[0] for w in want]
    assert clamped == any(w[1] for w in want) and clamped
    seg = np.where(ri != 0, 2, 1).astype(np.int32)
    back = intensity.intensity_unpack(q, seg, step)
    assert np.array_equal(back[ri != 0], np.asarray([np.float32(float(k) * step) for k in q], np.float32))
    assert back[3] == 0
    with pytest.raises(ValueError):
        intensity.intensity_unpack(q[:-1], seg, step)


def test_kitti_grid_is_lossless_at_0_005():
    """KITTI stores reflectance on a 0.01 grid: at intensity_accuracy 0.005 every value of the golden frame comes back
    bit for bit."""
    import os
    p = np.fromfile(os.path.join(os.path.dirname(__file__), "golden", "example.bin"), np.float32).reshape(-1, 4)
    v = np.unique(p[:, 3])
    q, clamped = intensity.intensity_pack(v, np.ones_like(v), 0.01)
    assert not clamped
    assert np.array_equal(intensity.intensity_unpack(q, np.zeros(v.size, np.int32), 0.01), v)
