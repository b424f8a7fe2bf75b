"""TEST INFRASTRUCTURE -- the intensity section (DESIGN.md §4, "Intensity") restated in numpy.  NOT product code.

The reference discards the intensity column (dataset/dataset.py:62), so there is nothing of it to pin against; this
module states the project's own definition once, independently of the CUDA path:

* project_owner: the reference's sequential z-buffer loop (cpp_modules.cpp:427-467, as orc_project restates it) run
  point by point, recording which input row made each store.  The pixel of a point follows cpp_modules.cpp:443-458 in
  float32 numpy arithmetic (every operation rounded, no FMA) with the box's libm atan2f (orc_libm_atan2f);
  tests/test_oracle_intensity.py checks that the range image equals oracle.project's.
* intensity_pack / intensity_unpack: the quantiser and its inverse, in float64 as the definition states them.
"""
import numpy as np

from . import atan2f_pair

F32 = np.float32


def _roundf(v):
    """C roundf of float32 values (half away from zero), exactly: the fraction of an f32 is exact in f64."""
    d = np.asarray(v, np.float64)
    t = np.trunc(d)
    return t + np.where(np.abs(d - t) >= 0.5, np.sign(d), 0.0)


def pixels(points, H, W, hfov, vmax, vmin):
    """-> (flat pixel index int64 (N,), depth f32 (N,)) of every point, as the reference's projection derives them."""
    p = np.ascontiguousarray(points, np.float32)
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    depth = np.sqrt((x * x + y * y) + z * z)
    _, ha = atan2f_pair(y, x)
    ha = np.where(ha < 0, (ha.astype(np.float64) + 2 * 3.14159265).astype(F32), ha)
    planar = np.sqrt(x * x + y * y)
    _, va = atan2f_pair(z, planar)
    # the pybind boundary narrows hfov / vmax / vmin to float (cpp_modules.cpp:427-428)
    col = _roundf(ha / F32(hfov) * F32(W)).astype(np.int64) % W
    vres = (F32(vmax) - F32(vmin)) / F32(H - 1)
    row = np.clip(_roundf((va - F32(vmin)) / vres).astype(np.int64), 0, H - 1)
    return row * W + col, depth


def project_owner(points, H, W, hfov, vmax, vmin):
    """-> ((H,W) f32 range image, (H,W) int64 owner: the row of the last store into the pixel, -1 where it ends empty)."""
    pix, depth = pixels(points, H, W, hfov, vmax, vmin)
    ri = [0.0] * (H * W)
    owner = [-1] * (H * W)
    for i, (q, d) in enumerate(zip(pix.tolist(), depth.tolist())):   # f32 values compare exactly as Python floats
        if ri[q] == 0 or d < ri[q]:
            ri[q] = d
            owner[q] = i
    ri = np.asarray(ri, np.float32).reshape(H, W)
    owner = np.asarray(owner, np.int64).reshape(H, W)
    owner[ri == 0] = -1
    return ri, owner


def intensity_image(points, owner):
    """The owners' intensities (H,W) f32, 0 at pixels without an owner."""
    p = np.asarray(points, np.float32)
    out = np.zeros(owner.shape, np.float32)
    has = owner >= 0
    out[has] = p[owner[has], 3]
    return out


def intensity_pack(intensity, ri, step):
    """-> (the section: u8 per pixel with ri != 0, raster order; whether the clamp acted).
    q = clamp(round half away from zero of (double)i / step, 0, 255), NaN -> 0."""
    v = np.asarray(intensity, np.float32).reshape(-1)[np.asarray(ri, np.float32).reshape(-1) != 0]
    with np.errstate(invalid="ignore"):
        d = v.astype(np.float64) / float(step)
        t = np.trunc(d)
        r = t + np.where(np.abs(d - t) >= 0.5, np.sign(d), 0.0)
        nan = np.isnan(r)
        clamped = bool(np.any((r < 0) | (r > 255)))
    return np.where(nan, 0, np.clip(np.nan_to_num(r), 0, 255)).astype(np.uint8), clamped


def intensity_unpack(q, seg, step):
    """-> (H,W) f32: (float)((double)q * step) at pixels whose label is not 1 (empty), 0 elsewhere; raises when the
    section does not hold one byte per such pixel."""
    q = np.asarray(q, np.uint8).reshape(-1)
    seg = np.asarray(seg)
    full = seg.reshape(-1) != 1
    if q.size != int(full.sum()):
        raise ValueError("intensity section holds %d bytes, the label map needs %d" % (q.size, int(full.sum())))
    out = np.zeros(seg.size, np.float32)
    out[full] = (q.astype(np.float64) * float(step)).astype(np.float32)
    return out.reshape(seg.shape)
