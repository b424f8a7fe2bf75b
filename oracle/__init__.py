"""TEST INFRASTRUCTURE -- the CPU oracle for the R-PCC hot path.  NOT product code.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs may import this package; nothing under ``r-pcc_b200/``
does, and the product fails loudly without its CUDA library.

``oracle.*`` functions are numpy-facing wrappers over ``liborc.so`` (the plain-C
restatement in ``rpcc_oracle.c``; each C function cites the reference file:line it
follows).  ``oracle.ref`` exposes the reference's OWN compiled code
(``oracle/_ref``, built by ``oracle/Makefile`` from /root/reference in the dev
container and shipped prebuilt to the GPU box) when it is present.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
_LIB = None

# name -> (restype, argtypes) of every ORC_API function of rpcc_oracle.c, in the file's order; the types follow
# r-pcc_b200/_lib.py (pointers c_void_p, scalars their exact C type).  tests/test_abi_bindings.py holds them to the C.
_v, _i, _f, _d = C.c_void_p, C.c_int, C.c_float, C.c_double
_i64, _u64 = C.c_int64, C.c_uint64
SIGNATURES = {
    "orc_atanf": (_f, (_f,)),
    "orc_atan2f": (_f, (_f, _f)),
    "orc_libm_atan2f": (_f, (_f, _f)),
    "orc_atan2f_array": (None, (_v, _v, _i64, _v, _v)),
    "orc_transform_map": (None, (_i, _i, _d, _d, _d, _v)),
    "orc_project": (None, (_v, _i, _i64, _i, _i, _f, _f, _f, _i, _v)),
    "orc_range_to_xyz": (None, (_v, _v, _i64, _v)),
    "orc_fps": (None, (_v, _i, _i, _i, _v, _v)),
    "orc_nonground_points": (None, (_v, _v, _i64, _f, _i, _v)),
    "orc_assign_labels": (None, (_v, _v, _v, _v, _v, _i, _i64, _i, _v)),
    "orc_point_modeling": (_i, (_v, _v, _i64, _v, _i)),
    "orc_intra_predict": (None, (_v, _v, _v, _i64, _v)),
    "orc_uniform_quantize": (_i64, (_v, _v, _i64, _f, _v)),
    "orc_extract_features": (None, (_v, _v, _i, _i, _i, _i, _i, _i, _i, _v, _v)),
    "orc_nonuniform_quantize": (_i64, (_v, _v, _v, _i64, _v, _v, _i, _i, _v, _v, _v)),
    "orc_extract_contour": (_i64, (_v, _i, _i, _v, _v)),
    "orc_recover_map": (None, (_v, _v, _i64, _i64, _v)),
    "orc_dequantize": (_i64, (_v, _v, _i64, _v, _i, _v)),
    "orc_chamfer_nn": (None, (_v, _i64, _v, _i64, _i, _v, _v)),
    "orc_ground_fit": (None, (_v, _v, _i64, _u64, _u64, _i, _v)),
    "orc_plane_models": (None, (_v, _v, _v, _i64, _i, _u64, _u64, _i, _f, _i, _i, _f, _i, _v)),
}


def build(force=False):
    """Compile liborc.so (and oracle/_ref when /root/reference is present)."""
    so = os.path.join(_DIR, "liborc.so")
    src = os.path.join(_DIR, "rpcc_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _DIR, "liborc.so"], stdout=subprocess.DEVNULL)
    if os.path.exists("/root/reference/ops/cpp_modules/src/cpp_modules.cpp"):
        subprocess.check_call(["make", "-C", _DIR, "ref"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_DIR, "liborc.so")
        if not os.path.exists(so):
            build()
        dll = C.CDLL(so)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(dll, name)
            fn.restype, fn.argtypes = restype, argtypes
        _LIB = dll
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


# --------------------------------------------------------------------------- lidar tables
# dataset/lidar_cfg/*.yaml (values only)
LIDARS = {
    "Velodyne64E": dict(H=64, W=2000, hfov_deg=360.0, vmax_deg=2.0, vmin_deg=-24.9),
    "Velodyne32E": dict(H=32, W=2250, hfov_deg=360.0, vmax_deg=10.67, vmin_deg=-30.67),
    "VelodyneVLP16": dict(H=16, W=1800, hfov_deg=360.0, vmax_deg=15.0, vmin_deg=-15.0),
}


def lidar_params(spec):
    """(H, W, hfov, vmax, vmin) as the Python doubles dataset/transformer.py:32-37 computes.  spec: a name of LIDARS,
    or any sensor object with H, W and the angles in radians as horizontal_FOV, vertical_max, vertical_min (such as
    rpcc_b200's LidarConfig, which computes them the same way)."""
    if isinstance(spec, str):
        c = LIDARS[spec]
        return (c["H"], c["W"], c["hfov_deg"] * (np.pi / 180), c["vmax_deg"] * (np.pi / 180),
                c["vmin_deg"] * (np.pi / 180))
    return (int(spec.H), int(spec.W), float(spec.horizontal_FOV), float(spec.vertical_max), float(spec.vertical_min))


# --------------------------------------------------------------------------- stages
def atan2f_pair(y, x):
    y, x = _f32(y).ravel(), _f32(x).ravel()
    a, b = np.empty_like(y), np.empty_like(y)
    lib().orc_atan2f_array(_p(y), _p(x), y.size, _p(a), _p(b))
    return a, b


def transform_map(H, W, hfov, vmax, vmin):
    lut = np.empty((H, W, 3), np.float32)
    lib().orc_transform_map(H, W, hfov, vmax, vmin, _p(lut))
    return lut


def project(points, H, W, hfov, vmax, vmin, restated_atan2=False):
    """points: (N,3) or (N,4) f32 -> (H,W) f32 range image."""
    pts = _f32(points)
    ri = np.empty((H, W), np.float32)
    lib().orc_project(_p(pts), pts.shape[1], pts.shape[0], H, W, hfov, vmax, vmin, int(restated_atan2), _p(ri))
    return ri


def range_to_xyz(ri, lut):
    ri = _f32(ri).reshape(-1)
    lut = _f32(lut)
    xyz = np.empty(lut.shape, np.float32)
    lib().orc_range_to_xyz(_p(ri), _p(lut), ri.size, _p(xyz))
    return xyz


def fps(points, m, fma_mode=0):
    pts = _f32(points).reshape(-1, 3)
    temp = np.empty(pts.shape[0], np.float32)
    idx = np.zeros(m, np.int32)
    lib().orc_fps(_p(pts), pts.shape[0], m, fma_mode, _p(temp), _p(idx))
    return idx


def ground_fit(range_image, lut, seed=0x5EED, frame=0, threads=512):
    """The PRODUCT's deterministic ground RANSAC restated (rpcc_oracle.c: orc_ground_fit) -- open3d's segment_plane,
    which the reference calls on an unseeded subsample (utils/segment_utils.py:74-82,101-108), cannot be pinned."""
    ri = _f32(range_image).reshape(-1)
    lut = _f32(lut)
    g = np.empty(4, np.float32)
    lib().orc_ground_fit(_p(ri), _p(lut), ri.size, seed, frame, int(threads), _p(g))
    return g


def nonground_points(xyz, ground_model, thr=0.1, assoc=0):
    xyz = _f32(xyz)
    g = _f32(ground_model)
    out = np.empty((xyz.size // 3, 3), np.float32)
    lib().orc_nonground_points(_p(xyz), _p(g), xyz.size // 3, thr, assoc, _p(out))
    return out


def segment(range_image, lut, ground_model, cluster_num=100, thr=0.1, assoc=0, fma_mode=0):
    """utils/segment_utils.py:133-148,168-169 given the ground model.
    Returns (seg_idx (H,W) int32, center_idx (M,) int32, centers (M,3) f32)."""
    lut = _f32(lut)
    H, W = lut.shape[:2]
    ri = _f32(range_image).reshape(H, W)
    g = _f32(ground_model)
    xyz = range_to_xyz(ri, lut)
    ng = nonground_points(xyz, g, thr, assoc)
    cidx = fps(ng, cluster_num, fma_mode)
    centers = np.ascontiguousarray(ng[cidx])
    seg = np.empty((H, W), np.int32)
    lib().orc_assign_labels(_p(ri), _p(xyz), _p(lut), _p(g), _p(centers), cluster_num, H * W, assoc, _p(seg))
    return seg, cidx, centers


def point_modeling(range_image, seg):
    ri = _f32(range_image).ravel()
    seg = _i32(seg).ravel()
    out = np.empty(70000, np.float32)
    K = lib().orc_point_modeling(_p(ri), _p(seg), seg.size, _p(out), out.size)
    assert K > 0
    return out[:K].copy()


def model_param_point(range_image, seg, ground_model):
    """tools/compress.py:101-102 for model_method='point': (K,4) f32 rows as they reach the bitstream."""
    pm = point_modeling(range_image, seg)
    cm = np.concatenate((np.zeros((pm.shape[0], 3)), pm[:, None].astype(np.float64)), -1)[1:]
    mp = np.concatenate((np.asarray(ground_model, np.float64).reshape(1, 4), cm), 0)
    return mp.astype(np.float32)


PLANE_SEED = 0x5EED ^ 0x9E3779B97F4A7C15      # the encoder's key for the per-cluster planes (csrc/encoder.cu)


def plane_models_device(range_image, lut, seg, model_point, seed=PLANE_SEED, frame=0, angle_threshold=75.0,
                        min_pixels=30, dist_thr=0.1, ransac_n=4, iters=10, threads=128):
    """The PRODUCT's deterministic per-cluster RANSAC restated (rpcc_oracle.c: orc_plane_models): the point-model rows
    `model_point` (K,4) with the rows of the accepted planes replaced.  (oracle.plane restates the REFERENCE's branch
    with a seeded stand-in for open3d instead.)"""
    ri = _f32(range_image).reshape(-1)
    mp = _f32(model_point).copy()
    lib().orc_plane_models(_p(ri), _p(_f32(lut)), _p(_i32(seg)), ri.size, int(mp.shape[0]), seed, frame,
                           int(min_pixels), dist_thr, int(ransac_n), int(iters), angle_threshold, int(threads), _p(mp))
    return mp


def intra_predict(seg, model_param, lut):
    seg = _i32(seg)
    mp = _f32(model_param)
    lut = _f32(lut)
    pred = np.empty(seg.shape, np.float32)
    lib().orc_intra_predict(_p(seg), _p(mp), _p(lut), seg.size, _p(pred))
    return pred


def uniform_quantize(seg, residual, step):
    seg = _i32(seg).ravel()
    res = _f32(residual).ravel()
    out = np.empty(seg.size, np.int32)
    n = lib().orc_uniform_quantize(_p(seg), _p(res), seg.size, step, _p(out))
    return out[:n].copy()


def extract_features(range_image, seg, region=3, segments=8, sharp_num=4, less_sharp_num=8, flat_num=6):
    seg = _i32(seg)
    H, W = seg.shape
    ri = _f32(range_image).reshape(H, W)
    feat = np.empty((H, W), np.float32)
    kp = np.empty((H, W), np.int32)
    lib().orc_extract_features(_p(ri), _p(seg), H, W, region, segments, sharp_num, less_sharp_num,
                               flat_num, _p(feat), _p(kp))
    return feat, kp


def nonuniform_quantize(seg, residual, kp, level_kp_num, level_acc, ground_level):
    seg = _i32(seg).ravel()
    res = _f32(residual).ravel()
    kp = _i32(kp).ravel()
    lk = _i32(level_kp_num)
    la = _f32(level_acc)
    out = np.empty(seg.size, np.int32)
    sal = np.empty(70000, np.int32)
    K = C.c_int(0)
    n = lib().orc_nonuniform_quantize(_p(seg), _p(res), _p(kp), seg.size, _p(lk), _p(la),
                                      la.size, ground_level, _p(out), _p(sal), C.byref(K))
    return out[:n].copy(), sal[:K.value].copy()


def extract_contour(seg):
    seg = _i32(seg)
    H, W = seg.shape
    contour = np.empty((H, W), np.int32)
    seq = np.empty(H * W, np.int32)
    L = lib().orc_extract_contour(_p(seg), H, W, _p(contour), _p(seq))
    return contour, seq[:L].copy()


def recover_map(contour, seq):
    contour = _i32(contour)
    seq = _i32(seq)
    seg = np.zeros(contour.shape, np.int32)
    lib().orc_recover_map(_p(contour), _p(seq), seq.size, contour.size, _p(seg))
    return seg


def dequantize(q, seg, steps):
    """steps: scalar (uniform) or per-label f64 array (acc[salience_level[m]])."""
    seg = _i32(seg)
    q = np.ascontiguousarray(q, np.int16)
    K = int(seg.max()) + 1
    st = np.full(K, steps, np.float64) if np.isscalar(steps) else np.ascontiguousarray(steps, np.float64)
    assert st.ndim == 1 and st.size >= K, "per-label steps must cover labels 0 .. %d" % (K - 1)
    res = np.empty(seg.shape, np.float32)
    n = lib().orc_dequantize(_p(q), _p(seg), seg.size, _p(st), K, _p(res))
    assert n == q.size, (n, q.size)
    return res


def chamfer_nn(a, b, fma_mode=0):
    a, b = _f32(a).reshape(-1, 3), _f32(b).reshape(-1, 3)
    dist = np.empty(a.shape[0], np.float32)
    idx = np.empty(a.shape[0], np.int32)
    lib().orc_chamfer_nn(_p(a), a.shape[0], _p(b), b.shape[0], fma_mode, _p(dist), _p(idx))
    return dist, idx


# --------------------------------------------------------------------------- whole-frame restatement
def pack_sections(model_param, seg, symbols, salience=None):
    """utils/compress_utils.py:138-161: the uncompressed sections in file order."""
    contour, seq = extract_contour(seg)
    sec = {}
    if salience is not None:
        sec["salience_level"] = np.asarray(salience).astype(np.uint8).tobytes()
    sec["contour_map"] = np.packbits(contour.astype(bool), axis=None).astype(np.uint8).tobytes()
    sec["idx_sequence"] = seq.astype(np.uint16).tobytes()
    sec["plane_param"] = np.asarray(model_param).astype(np.float32).tobytes()
    sec["residual_quantized"] = np.asarray(symbols).astype(np.int16).tobytes()
    return sec


SECTION_ORDER = ("salience_level", "contour_map", "idx_sequence", "plane_param", "residual_quantized")


def write_rpcc(sections, method="bzip2"):
    """utils/compress_utils.py:167-179 + BasicCompressor :255-310 (bz2 level 9 / gzip level 9)."""
    import bz2
    import gzip
    import struct
    out = b""
    for k in SECTION_ORDER:
        if k not in sections:
            continue
        raw = sections[k]
        if method == "bzip2":
            c = bz2.compress(raw)
        elif method in ("gzip", "deflate"):
            c = gzip.compress(raw, mtime=0)
        else:
            raise ValueError(method)
        out += struct.pack("i", len(c)) + c
    return out


def compress_frame(points, lidar="Velodyne64E", ground_model=None, accuracy=0.02, nonuniform=False,
                   cluster_num=100, assoc=0, fma_mode=0, cfg=None, model_method="point", plane_seed=0,
                   angle_threshold=75, plane_impl="reference", frame=0):
    """tools/compress.py:44-133 given the ground model; returns a dict of every intermediate (the parity
    tests compare the CUDA path stage by stage).  model_method='plane' uses oracle.plane (open3d stand-in)."""
    H, W, hfov, vmax, vmin = lidar_params(lidar)
    lut = transform_map(H, W, hfov, vmax, vmin)
    step = accuracy * 2
    ri = project(points, H, W, hfov, vmax, vmin)
    seg, cidx, centers = segment(ri, lut, ground_model, cluster_num, 0.1, assoc, fma_mode)
    if model_method == "plane" and plane_impl == "device":
        mp = plane_models_device(ri, lut, seg, model_param_point(ri, seg, ground_model), frame=frame,
                                 angle_threshold=float(angle_threshold))
    elif model_method == "plane":
        from . import plane as _plane
        cm = _plane.cluster_modeling_plane(lut, ri, seg, angle_threshold, plane_seed)
        mp = np.concatenate((np.asarray(ground_model, np.float64).reshape(1, 4), cm), 0).astype(np.float32)
    else:
        mp = model_param_point(ri, seg, ground_model)
    pred = intra_predict(seg, mp, lut)
    res = ri - pred
    out = dict(range_image=ri, seg_idx=seg, center_idx=cidx, model_param=mp, pred=pred, lut=lut)
    if not nonuniform:
        sym = uniform_quantize(seg, res, step)
        sal = None
    else:
        c = dict(level_kp_num=(30, 10, 3, 0), level_dacc=(0, 0.02, 0.04, 0.06), ground_level=2,
                 region=3, segments=8, sharp_num=4, less_sharp_num=8, flat_num=6)
        c.update(cfg or {})
        _, kp = extract_features(ri, seg, c["region"], c["segments"], c["sharp_num"],
                                 c["less_sharp_num"], c["flat_num"])
        acc = np.array([step] * len(c["level_kp_num"])) + np.array(c["level_dacc"])
        sym, sal = nonuniform_quantize(seg, res, kp, c["level_kp_num"], acc, c["ground_level"])
        out.update(key_point_map=kp, salience_level=sal, level_acc=acc)
    out["symbols"] = sym
    out["sections"] = pack_sections(mp, seg, sym, sal)
    return out


def decompress_sections(sections, lidar="Velodyne64E", accuracy=0.02, level_dacc=(0, 0.02, 0.04, 0.06)):
    """tools/decompress.py:88-110: sections -> (range_rec (H,W), xyz (H,W,3))."""
    H, W, hfov, vmax, vmin = lidar_params(lidar)
    lut = transform_map(H, W, hfov, vmax, vmin)
    step = accuracy * 2
    contour = np.unpackbits(np.frombuffer(sections["contour_map"], np.uint8))[:H * W].reshape(H, W)
    seq = np.frombuffer(sections["idx_sequence"], np.uint16)
    seg = recover_map(contour, seq)
    mp = np.frombuffer(sections["plane_param"], np.float32).reshape(-1, 4)
    q = np.frombuffer(sections["residual_quantized"], np.int16)
    if "salience_level" in sections:
        sal = np.frombuffer(sections["salience_level"], np.uint8)
        acc = np.array([step] * len(level_dacc)) + np.array(level_dacc)
        K = int(seg.max()) + 1
        steps = acc[sal[:K]]
    else:
        steps = step
    res = dequantize(q, seg, steps)
    pred = intra_predict(seg, mp, lut)
    rec = pred + res
    return rec, rec[..., None] * lut, seg
