"""Batched encoder / decoder: many frames per kernel launch, host entropy coding on threads.

This is the re-plumbed tools/compress_datalist.py (reference :48-206: a ThreadPoolExecutor over a
per-frame closure that holds the GIL in every native call): frames go to the GPU in batches
(rpcc_encoder_encode_host pipelines upload / kernels / download over stream slots), the five
`.rpcc` sections come back packed, and bz2/deflate -- sequential by nature -- run on a host
thread pool while the next batch is on the device.
"""
import concurrent.futures as futures
import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from ._lib import EVAL_COLS, P2PLANE_COLS, RESULT_DTYPE, EncoderConfig, check, ptr
from .compress_utils import BasicCompressor, pack_bitstream, parse_bitstream
from .config import load_compressor_cfg
from .lidar import LidarConfig


def _psnr(mse):
    with np.errstate(divide="ignore"):
        return 10 * np.log10(3 * 59.7 * 59.7 / mse) if mse > 0 else float("inf")


def p2plane_summary(m):
    """One row of rpcc_p2plane_batch's table (7 columns) -> point-to-plane mse both ways and their mean PSNR (r = 59.7,
    the convention of psnr_p2p).  An empty cloud on the other side gives an infinite mse and a PSNR of -inf."""
    mse1, mse2 = m[1] / max(m[0], 1.0), m[4] / max(m[3], 1.0)
    return {"psnr_p2plane": (_psnr(mse1) + _psnr(mse2)) / 2, "p2plane_mse1": float(mse1), "p2plane_mse2": float(mse2),
            "no_normal_points": int(m[2] + m[5])}


def eval_summary(m, HW):
    """One row of rpcc_eval_batch's table -> the figures tools/compress_datalist.py:180-199 prints
    (utils/evaluate_metrics.py:20-31, fscore.py:12-16; point-to-point PSNR as :57-72 with r = 59.7).  A row with
    rpcc_p2plane_batch's columns after the 12 (an encoder with p2plane=True) adds psnr_p2plane, p2plane_mse1/2 and
    no_normal_points (p2plane_summary)."""
    n1, n2 = max(m[2], 1.0), max(m[6], 1.0)
    cd1, cd2 = m[3] / n1, m[7] / n2
    p1, p2 = float(np.float32(m[4]) / np.float32(n1)), float(np.float32(m[8]) / np.float32(n2))
    f = 2 * p1 * p2 / (p1 + p2) if (p1 + p2) > 0 else 0.0
    mse1, mse2 = m[5] / n1, m[9] / n2
    with np.errstate(divide="ignore"):
        psnr = [10 * np.log10(3 * 59.7 * 59.7 / x) if x > 0 else float("inf") for x in (mse1, mse2)]
    out = {"depth_max": float(m[0]), "depth_mean": float(m[1] / HW), "cd1": cd1, "cd2": cd2, "mean": (cd1 + cd2) / 2,
           "max": max(cd1, cd2), "sum": cd1 + cd2, "f_score": f, "precision": p1, "recall": p2,
           "psnr_p2p": (psnr[0] + psnr[1]) / 2, "label_mismatches": int(m[11]), "exhaustive_points": int(m[10])}
    if len(m) >= EVAL_COLS + P2PLANE_COLS:
        out.update(p2plane_summary(m[EVAL_COLS:EVAL_COLS + P2PLANE_COLS]))
    return out


def _pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype, pin_memory=True)


def default_workers():
    """Host entropy-coder threads of one process: the box's cores split evenly over the ranks of a torchrun launch
    (LOCAL_WORLD_SIZE), one left for the thread that feeds the GPU."""
    n = os.cpu_count() or 2
    try:
        ranks = int(os.environ.get("LOCAL_WORLD_SIZE") or os.environ.get("WORLD_SIZE") or 1)
    except ValueError:
        ranks = 1
    return max(1, n // max(ranks, 1) - 1)


class BatchEncoder:
    """project -> ground fit -> FPS -> labels (segment_method 'DBSCAN': DBSCAN -> label statistics) -> (key points) ->
    point (or plane) models -> quantise + pack for batches of frames.  `accuracy` is the yaml value (step = 2 * accuracy, tools/compress.py:46).  eval=True also
    decodes every frame and fills the --eval table (encode_host's "eval", 12 columns); p2plane=True (with eval) adds
    the normals of both clouds and the 7 point-to-plane columns after them.  intensity_accuracy (default: the yaml's
    `intensity_accuracy`, None = off) adds the intensity section (DESIGN.md §4): points must then be (N,4) rows, and
    encode_host returns "intensity" and frame_sections the sixth section."""

    def __init__(self, lidar="Velodyne64E", accuracy=None, nonuniform=None, compressor_cfg=None, max_batch=256,
                 max_points=None, device=None, basic_compressor=None, workers=None, model_method=None, host_chunk=0,
                 eval=False, f1_threshold=0.02, p2plane=False, intensity_accuracy=None):
        cfg = load_compressor_cfg(compressor_cfg) if not isinstance(compressor_cfg, dict) else compressor_cfg
        self.cfg = cfg
        self.model_method = model_method or cfg["modeling_method"]
        self.lidar = lidar if isinstance(lidar, LidarConfig) else LidarConfig(lidar)
        if cfg["segment_method"] not in ("FPS", "DBSCAN"):
            raise ValueError("segment_method must be 'FPS' or 'DBSCAN'")
        if self.model_method not in ("point", "plane"):
            raise ValueError("model_method must be 'point' or 'plane'")
        self.accuracy = cfg["accuracy"] if accuracy is None else accuracy
        self.step = self.accuracy * 2
        self.uniform = (cfg["compress_framework"] == "uniform") if nonuniform is None else (not nonuniform)
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.max_batch = int(max_batch)
        self.max_points = int(max_points) if max_points else self.max_batch * 140000
        self.K = int(cfg["cluster_num"]) + 2
        self.method = basic_compressor or cfg["basic_compressor"]
        self.workers = workers or default_workers()
        c = EncoderConfig()
        c.H, c.W = self.lidar.H, self.lidar.W
        c.hfov, c.vmax, c.vmin = self.lidar.horizontal_FOV, self.lidar.vertical_max, self.lidar.vertical_min
        c.cluster_num = int(cfg["cluster_num"])
        c.ground_threshold = float(cfg["ground_threshold"])
        c.step = float(self.step)
        c.nonuniform = 0 if self.uniform else 1
        lk, ld = list(cfg["level_key_point_num"]), list(cfg["level_delta_acc"])
        c.level_num = len(lk)
        for i in range(len(lk)):
            c.level_kp_num[i] = int(lk[i])
            c.level_dacc[i] = float(ld[i])
        c.ground_level = int(cfg["ground_salience_level"])
        c.feature_region = int(cfg["feature_region"])
        c.segments = int(cfg["segments"])
        c.sharp_num = int(cfg["sharp_num"])
        c.less_sharp_num = int(cfg["less_sharp_num"])
        c.flat_num = int(cfg["flat_num"])
        c.max_batch = self.max_batch
        c.max_points = self.max_points
        c.device = self.device
        c.model_method = 1 if self.model_method == "plane" else 0
        c.plane_angle_threshold = float(cfg["plane_angle_threshold"])
        c.host_chunk = int(host_chunk)
        self.eval = bool(eval)
        self.p2plane = bool(p2plane)
        if self.p2plane and not self.eval:
            raise ValueError("p2plane=True needs eval=True")
        self.eval_cols = EVAL_COLS + (P2PLANE_COLS if self.p2plane else 0)
        c.eval = (2 if self.p2plane else 1) if self.eval else 0
        c.eval_threshold_sq = float(f1_threshold ** 2)
        if cfg["segment_method"] == "DBSCAN":
            c.segment_method = 1
            c.dbscan_eps = float(cfg["DBSCAN_eps"])
            c.dbscan_min_points = int(cfg["DBSCAN_min_points"])
        ia = cfg.get("intensity_accuracy") if intensity_accuracy is None else intensity_accuracy
        if ia is not None and not float(ia) > 0:
            raise ValueError("intensity_accuracy must be positive")
        self.intensity_accuracy = None if ia is None else float(ia)
        self.intensity = self.intensity_accuracy is not None
        c.intensity_step = 2 * self.intensity_accuracy if self.intensity else 0.0
        self._c = c
        self._h = C.c_void_p(0)
        check(_lib.lib().rpcc_encoder_create(C.byref(c), C.byref(self._h)))
        self._pool = None
        self._packer = None
        self._host = {}
        self._in = {}

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if self._packer is not None:
            self._packer.close()
            self._packer = None
        if self._h:
            _lib.lib().rpcc_encoder_destroy(self._h)
            self._h = C.c_void_p(0)
        if self._pool is not None:
            self._pool.shutdown()
            self._pool = None
        self._host, self._in = {}, {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ------------------------------------------------------------------ device path
    @property
    def slots(self):
        return int(_lib.lib().rpcc_encoder_slots())

    def encode_device(self, slot, points, offsets, B, ground=None, keys=None):
        """points (N,3|4) f32 cuda, offsets (B+1,) int64 cuda, ground (B,4) f32 cuda or None, keys (B,) int64 cuda
        or None (every frame keyed 0: its bytes depend on its points alone).  Asynchronous."""
        check(_lib.lib().rpcc_encoder_encode_device(self._h, int(slot), ptr(points), int(points.shape[1]), ptr(offsets),
                                                    int(B), ptr(ground) if ground is not None else None,
                                                    ptr(keys) if keys is not None else None))

    def sync(self):
        check(_lib.lib().rpcc_encoder_sync(self._h))

    STAGES = ("project", "ground", "fps", "assign", "keypoints", "model", "quantize", "eval")

    def profile(self, enable=True):
        """Start (or stop) recording CUDA events between the stages of every chain call."""
        check(_lib.lib().rpcc_encoder_profile(self._h, 1 if enable else 0))

    def stage_times(self):
        """-> ({stage: summed ms}, frames covered, chain calls) since profile(True)."""
        ms = (C.c_double * 8)()
        frames = C.c_longlong(0)
        calls = C.c_int(0)
        check(_lib.lib().rpcc_encoder_stage_times(self._h, ms, C.byref(frames), C.byref(calls)))
        return dict(zip(self.STAGES, list(ms))), int(frames.value), int(calls.value)

    def stream(self, slot):
        return _lib.lib().rpcc_encoder_stream(self._h, int(slot))

    def device_buffer(self, slot, name, shape, dtype):
        """A torch view of one of the slot's device buffers (tests / chaining)."""
        p = _lib.lib().rpcc_encoder_device_buffer(self._h, int(slot), name.encode())
        if not p:
            raise KeyError(name)
        n = int(np.prod(shape))
        itemsize = torch.empty((), dtype=dtype).element_size()
        # wrap the raw device pointer without copying
        iface = {"shape": (n * itemsize,), "typestr": "|u1", "data": (p, False), "version": 3}
        holder = type("_Dev", (), {"__cuda_array_interface__": iface})()
        return torch.as_tensor(holder, device="cuda:%d" % self.device).view(dtype).view(*shape)

    # ------------------------------------------------------------------ host path
    def _host_buffers(self, B, which=0):
        """Pinned output buffers for B frames; `which` selects one of several independent sets, so that the host
        entropy stage can still be reading set 0 while the GPU fills set 1 (pinned double-buffering)."""
        HW, K = self.lidar.HW, self.K
        h = self._host.get(which)
        if h is None or h["B"] < B:
            cap = max(B, self.max_batch)
            h = dict(B=cap,
                     results=_pinned((cap, 4), torch.int32),
                     model=_pinned((cap, K, 4), torch.float32),
                     contour=_pinned((cap, (HW + 7) // 8), torch.uint8),
                     seq=_pinned((cap * HW,), torch.int16),
                     symbols=_pinned((cap * HW,), torch.int16),
                     salience=_pinned((cap, K), torch.uint8),
                     eval=_pinned((cap, self.eval_cols), torch.float64),
                     intensity=_pinned((cap * HW,), torch.uint8) if self.intensity else None)
            self._host[which] = h
        return h

    def input_buffer(self, rows, which=0):
        """A pinned (rows, 3) f32 staging buffer for the points of one batch (readers fill it, encode_host uploads
        from it), (rows, 4) for an intensity encoder; `which` as in _host_buffers."""
        t = self._in.get(which)
        if t is None or t.shape[0] < rows:
            t = _pinned((max(int(rows), 1), 4 if self.intensity else 3), torch.float32)
            self._in[which] = t
        return t

    def encode_host(self, points, offsets, grounds=None, keys=None, out_set=0):
        """points: (N,3|4) f32 numpy or pinned torch tensor (all frames back to back); offsets (B+1,) int64;
        grounds (B,4) or None (fit on device); keys (B,) uint64 or None -- the per-frame keys of the deterministic
        RANSACs (None: key 0 for every frame, so a frame's bytes do not depend on how it is batched).  Returns a dict of numpy views (valid until the next call):
        results (structured: sym_count, seq_count, model_rows, flags), model (B,K,4) f32, contour (B,HW/8) u8,
        seq (sum,) u16, symbols (sum,) i16, salience (B,K) u8 | None, intensity (sum,) u8 | None (the intensity
        sections, at sym_off like the symbols), plus sym_off / seq_off (B+1,)."""
        pts = points if isinstance(points, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(points, dtype=np.float32))
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        B = off.size - 1
        h = self._host_buffers(B, out_set)
        g = None
        if grounds is not None:
            g = np.ascontiguousarray(grounds, dtype=np.float32)
        k = None if keys is None else np.ascontiguousarray(keys, dtype=np.uint64)
        if k is not None and k.size != B:
            raise ValueError("keys must hold one entry per frame")
        HW = self.lidar.HW
        if self.intensity and pts.shape[1] != 4:
            raise ValueError("an intensity encoder needs (N,4) points: x, y, z, intensity")
        check(_lib.lib().rpcc_encoder_encode_host_intensity(
            self._h, ptr(pts), int(pts.shape[1]), ptr(off), B, ptr(g) if g is not None else None, ptr(h["results"]),
            ptr(h["model"]), ptr(h["contour"]), ptr(h["seq"]), h["B"] * HW, ptr(h["symbols"]), h["B"] * HW,
            ptr(h["salience"]) if not self.uniform else None, ptr(k) if k is not None else None,
            ptr(h["eval"]) if self.eval else None, ptr(h["intensity"]) if self.intensity else None))
        res = h["results"].numpy()[:B].view(np.uint32).copy().view(RESULT_DTYPE).reshape(B)
        sym_off = np.concatenate(([0], np.cumsum(res["sym_count"], dtype=np.int64)))
        seq_off = np.concatenate(([0], np.cumsum(res["seq_count"], dtype=np.int64)))
        return dict(results=res, model=h["model"].numpy()[:B], contour=h["contour"].numpy()[:B],
                    seq=h["seq"].numpy()[:max(int(seq_off[-1]), 1)].view(np.uint16)[:seq_off[-1]],
                    symbols=h["symbols"].numpy()[:max(int(sym_off[-1]), 1)][:sym_off[-1]],
                    salience=None if self.uniform else h["salience"].numpy()[:B], sym_off=sym_off, seq_off=seq_off,
                    eval=h["eval"].numpy()[:B] if self.eval else None,
                    intensity=h["intensity"].numpy()[:sym_off[-1]] if self.intensity else None)

    @staticmethod
    def frame_sections(enc, b):
        """The five uncompressed sections of frame b, as compress_point_cloud builds them
        (utils/compress_utils.py:141-161), and the intensity section when the encoder has one."""
        r = enc["results"][b]
        rows = int(r["model_rows"])
        sec = {}
        if enc["salience"] is not None:
            sec["salience_level"] = enc["salience"][b, :rows].tobytes()
        sec["contour_map"] = enc["contour"][b].tobytes()
        sec["idx_sequence"] = enc["seq"][enc["seq_off"][b]:enc["seq_off"][b + 1]].tobytes()
        sec["plane_param"] = enc["model"][b, :rows].tobytes()
        sec["residual_quantized"] = enc["symbols"][enc["sym_off"][b]:enc["sym_off"][b + 1]].tobytes()
        if enc.get("intensity") is not None:
            sec["intensity"] = enc["intensity"][enc["sym_off"][b]:enc["sym_off"][b + 1]].tobytes()
        return sec

    def _entropy(self, sections):
        bc = BasicCompressor(method_name=self.method, gzip_mtime=0)
        return pack_bitstream({k: bc.compress(v, section=k) for k, v in sections.items()}, uniform=self.uniform)

    def packer(self):
        """The native entropy-coder pool (bzip2 only; csrc/hostio.cu), created on first use."""
        if self._packer is None:
            from .hostio import Packer
            self._packer = Packer(self.workers, self.method)
        return self._packer

    def compress(self, points, offsets, grounds=None, keys=None):
        """-> list of B `.rpcc` byte strings (GPU stages, then the host entropy coder: the native pool for bzip2, a
        Python thread pool for deflate / lz4)."""
        enc = self.encode_host(points, offsets, grounds, keys)
        B = len(enc["results"])
        if self.method == "bzip2":
            pk = self.packer()
            sizes, blobs = pk.wait(pk.submit(enc, self.K, self.uniform, None, keep=True))
            return [blobs[b, :sizes[b]].tobytes() for b in range(B)]
        if self._pool is None:
            self._pool = futures.ThreadPoolExecutor(self.workers)
        secs = [self.frame_sections(enc, b) for b in range(B)]
        return list(self._pool.map(self._entropy, secs))


class BatchDecoder:
    """.rpcc byte strings -> reconstructed range images / point clouds, B frames per launch
    (tools/decompress.py:88-112 for many frames).

    The sections are decompressed on host threads (libbz2 through the C ABI for bzip2: no GIL) straight into pinned
    staging buffers, with the frames' sequences and symbols packed back to back; one asynchronous upload per array,
    rpcc_decode_packed_batch, and -- with want_points -- the rows of the output `.bin` files compacted on the device, so
    that one download brings back exactly the bytes that go to disk.  All buffers (pinned and device) are allocated
    once per capacity and reused; two independent sets (`buf_set`) let a caller overlap the host work of one batch
    with the device work of another.

    intensity_accuracy (default: the yaml's `intensity_accuracy`, None = off) reads the intensity section as well (every
    file must have it) and puts the decoded intensities into the fourth column of `points`; without it a file's intensity
    section is skipped."""

    def __init__(self, lidar="Velodyne64E", accuracy=None, nonuniform=None, compressor_cfg=None, basic_compressor=None,
                 workers=None, device=None, intensity_accuracy=None):
        cfg = load_compressor_cfg(compressor_cfg) if not isinstance(compressor_cfg, dict) else compressor_cfg
        self.cfg = cfg
        self.lidar = lidar if isinstance(lidar, LidarConfig) else LidarConfig(lidar)
        self.accuracy = cfg["accuracy"] if accuracy is None else accuracy
        self.step = self.accuracy * 2
        self.uniform = (cfg["compress_framework"] == "uniform") if nonuniform is None else (not nonuniform)
        self.method = basic_compressor or cfg["basic_compressor"]
        self.level_acc = np.array([self.step] * len(cfg["level_key_point_num"])) + np.array(cfg["level_delta_acc"])
        self.workers = workers or default_workers()
        self.device = torch.cuda.current_device() if device is None else int(device)
        ia = cfg.get("intensity_accuracy") if intensity_accuracy is None else intensity_accuracy
        if ia is not None and not float(ia) > 0:
            raise ValueError("intensity_accuracy must be positive")
        self.intensity_accuracy = None if ia is None else float(ia)
        self.intensity = self.intensity_accuracy is not None
        self._lut = None
        self._pool = futures.ThreadPoolExecutor(self.workers)
        self._host = {}
        self._dev = {}
        self._streams = {}

    def close(self):
        if self._pool is not None:
            self._pool.shutdown()
            self._pool = None
        self._host, self._dev = {}, {}

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---------------------------------------------------------------- host side: files -> sections
    def _unpack(self, blob):
        """-> dict of raw sections (numpy uint8 views / bytes)"""
        if self.method == "bzip2":
            from .hostio import unpack_rpcc
            HW = self.lidar.HW
            return unpack_rpcc(blob, self.uniform, (HW + 7) // 8 + 5 * HW + 16 * 256 + 256 + 64, self.intensity)
        bc = BasicCompressor(method_name=self.method)
        return {k: np.frombuffer(v, np.uint8)
                for k, v in bc.decompress_dict(parse_bitstream(blob, uniform=self.uniform, intensity=self.intensity)).items()}

    def _section_error(self, s, cb, HW):
        """-> why the sections of one file cannot be a frame of this decoder's lidar and framework, or None."""
        if len(s["contour_map"]) != cb:
            return "contour_map holds %d bytes, not ceil(H*W / 8) = %d" % (len(s["contour_map"]), cb)
        for k in ("idx_sequence", "residual_quantized"):
            if len(s[k]) % 2:
                return "%s has an odd length (%d bytes)" % (k, len(s[k]))
            if len(s[k]) > 2 * HW:
                return "%s holds more than H*W entries" % k
        rows, tail = divmod(len(s["plane_param"]), 16)
        if tail or not 1 <= rows <= 254:
            return "plane_param holds %d bytes, not 1 to 254 rows of 16" % len(s["plane_param"])
        if not self.uniform:
            sal = np.frombuffer(s["salience_level"], np.uint8)
            if sal.size != rows:
                return "salience_level has %d entries for %d model rows" % (sal.size, rows)
            if sal.size and int(sal.max()) >= len(self.level_acc):
                return "salience level %d with %d levels configured" % (int(sal.max()), len(self.level_acc))
        if self.intensity and len(s["intensity"]) != len(s["residual_quantized"]) // 2:
            return "the intensity section does not hold one byte per symbol"
        return None

    def _buffers(self, B, K, which):
        HW = self.lidar.HW
        cb = (HW + 7) // 8
        h = self._host.get(which)
        if h is None or h["B"] < B or h["K"] < K:
            capB, capK = max(B, h["B"] if h else 0), max(K, h["K"] if h else 0)
            dev = torch.device("cuda", self.device)
            h = dict(B=capB, K=capK,
                     contour=_pinned((capB, cb), torch.uint8), model=_pinned((capB, capK, 4), torch.float32),
                     steps=_pinned((capB, capK), torch.float64), seq=_pinned((capB * HW,), torch.int16),
                     sym=_pinned((capB * HW,), torch.int16), base=_pinned((2, capB + 1), torch.int64),
                     results=_pinned((capB, 4), torch.int32), row_base=_pinned((capB + 1,), torch.int64),
                     rows=None, inten=_pinned((capB * HW,), torch.uint8) if self.intensity else None)
            d = dict(contour=torch.empty((capB, cb), dtype=torch.uint8, device=dev),
                     model=torch.empty((capB, capK, 4), dtype=torch.float32, device=dev),
                     steps=torch.empty((capB, capK), dtype=torch.float64, device=dev),
                     seq=torch.empty((capB * HW,), dtype=torch.int16, device=dev),
                     sym=torch.empty((capB * HW,), dtype=torch.int16, device=dev),
                     base=torch.empty((2, capB + 1), dtype=torch.int64, device=dev),
                     labels=torch.empty((capB, HW), dtype=torch.uint8, device=dev),
                     range=torch.empty((capB, HW), dtype=torch.float32, device=dev),
                     results=torch.empty((capB, 4), dtype=torch.int32, device=dev),
                     book=torch.empty((_lib.lib().rpcc_book_bytes(capB, self.lidar.H, self.lidar.W, capK),), dtype=torch.uint8, device=dev),
                     xyz=None, rows=None, row_base=None, pws=None,
                     inten=torch.empty((capB * HW,), dtype=torch.uint8, device=dev) if self.intensity else None,
                     inten_img=torch.empty((capB, HW), dtype=torch.float32, device=dev) if self.intensity else None)
            self._host[which], self._dev[which] = h, d
        return self._host[which], self._dev[which]

    def decode(self, blobs, want_xyz=True, want_points=False, buf_set=0):
        """-> dict(range (B,H,W) f32 cuda, xyz (B,H,W,3) f32 cuda | None, labels (B,H,W) u8 cuda, results,
        points: list of B (n,4) f32 numpy views of a pinned buffer | None).  The returned tensors and views belong to
        buffer set `buf_set` and are overwritten by the next decode() on that set."""
        B = len(blobs)
        H, W, HW = self.lidar.H, self.lidar.W, self.lidar.HW
        cb = (HW + 7) // 8
        secs = list(self._pool.map(self._unpack, blobs))
        # every frame is checked on its own before the upload, so that whether a file is refused does not depend on
        # the other frames of the batch or on the buffers' capacity left by earlier batches
        why = [self._section_error(s, cb, HW) for s in secs]
        bad = [b for b in range(B) if why[b]]
        if bad:
            raise ValueError("malformed .rpcc stream(s) at batch index %s: %s (wrong lidar / framework settings?)"
                             % (bad[:8], why[bad[0]]))
        rows = [len(s["plane_param"]) // 16 for s in secs]
        K = max(max(rows), 2)
        h, d = self._buffers(B, K, buf_set)
        Kc = h["K"]
        seq_n = np.array([len(s["idx_sequence"]) // 2 for s in secs], np.int64)
        sym_n = np.array([len(s["residual_quantized"]) // 2 for s in secs], np.int64)
        base = h["base"].numpy()
        base[0, 0] = base[1, 0] = 0
        np.cumsum(seq_n, out=base[0, 1:B + 1])
        np.cumsum(sym_n, out=base[1, 1:B + 1])
        contour, model, steps = h["contour"].numpy(), h["model"].numpy(), h["steps"].numpy()
        inten = h["inten"].numpy() if self.intensity else None
        seq, sym = h["seq"].numpy().view(np.uint8), h["sym"].numpy().view(np.uint8)
        model[:B] = 0
        steps[:B] = self.step

        def fill(b):
            s = secs[b]
            contour[b] = np.frombuffer(s["contour_map"], np.uint8)
            seq[2 * base[0, b]:2 * base[0, b + 1]] = np.frombuffer(s["idx_sequence"], np.uint8)
            sym[2 * base[1, b]:2 * base[1, b + 1]] = np.frombuffer(s["residual_quantized"], np.uint8)
            if self.intensity:
                inten[base[1, b]:base[1, b + 1]] = np.frombuffer(s["intensity"], np.uint8)
            model[b, :rows[b]] = np.frombuffer(s["plane_param"], np.uint8).view(np.float32).reshape(-1, 4)
            if not self.uniform:
                steps[b, :rows[b]] = self.level_acc[np.frombuffer(s["salience_level"], np.uint8)]

        list(self._pool.map(fill, range(B)))
        dev = torch.device("cuda", self.device)
        if self._lut is None:
            self._lut = torch.from_numpy(self.lidar.transform_map()).to(dev)
        # the caller's current stream carries the uploads, the kernels and the downloads in order
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream().cuda_stream
            d["contour"][:B].copy_(h["contour"][:B], non_blocking=True)
            d["model"][:B].copy_(h["model"][:B], non_blocking=True)
            d["steps"][:B].copy_(h["steps"][:B], non_blocking=True)
            d["base"].copy_(h["base"], non_blocking=True)
            nseq, nsym = int(base[0, B]), int(base[1, B])
            d["seq"][:nseq].copy_(h["seq"][:nseq], non_blocking=True)
            d["sym"][:nsym].copy_(h["sym"][:nsym], non_blocking=True)
            if self.intensity:
                d["inten"][:nsym].copy_(h["inten"][:nsym], non_blocking=True)
            xyz = None
            if want_xyz:
                if d["xyz"] is None:
                    d["xyz"] = torch.empty((h["B"], HW, 3), dtype=torch.float32, device=dev)
                xyz = d["xyz"]
            # model rows are strided by the buffers' K capacity: decode with that K (unused rows are zero = "no model")
            check(_lib.lib().rpcc_decode_packed_batch(ptr(d["contour"]), ptr(d["seq"]), ptr(d["base"][0]), ptr(d["sym"]),
                                                      ptr(d["base"][1]), ptr(d["model"]), ptr(d["steps"]), ptr(self._lut),
                                                      B, H, W, Kc, ptr(d["labels"]), ptr(d["range"]),
                                                      ptr(xyz) if want_xyz else None, ptr(d["book"]), ptr(d["results"]), st))
            h["results"][:B].copy_(d["results"][:B], non_blocking=True)
            points = None
            if want_points:
                if d["rows"] is None:
                    d["rows"] = torch.empty((h["B"] * HW, 4), dtype=torch.float32, device=dev)
                    d["row_base"] = torch.empty((h["B"] + 1,), dtype=torch.int64, device=dev)
                    d["pws"] = torch.empty((_lib.lib().rpcc_points_workspace_bytes(h["B"], H, W),), dtype=torch.uint8, device=dev)
                    h["rows"] = _pinned((h["B"] * HW, 4), torch.float32)
                if self.intensity:
                    # the symbols' offsets are the intensity section's: one byte per symbol
                    check(_lib.lib().rpcc_intensity_unpack_batch(ptr(d["labels"]), ptr(d["inten"]), ptr(d["base"][1]), B, H,
                                                                 W, 2 * self.intensity_accuracy, ptr(d["inten_img"]), st))
                check(_lib.lib().rpcc_points_out_intensity_batch(ptr(d["range"]), ptr(self._lut),
                                                                 ptr(d["inten_img"]) if self.intensity else None, B, H, W,
                                                                 ptr(d["rows"]), ptr(d["row_base"]), ptr(d["pws"]), st))
                h["row_base"][:B + 1].copy_(d["row_base"][:B + 1], non_blocking=True)
                torch.cuda.current_stream().synchronize()
                rb = h["row_base"].numpy()[:B + 1]
                total = int(rb[B])
                h["rows"][:total].copy_(d["rows"][:total], non_blocking=True)
                torch.cuda.current_stream().synchronize()
                hr = h["rows"].numpy()
                points = [hr[rb[b]:rb[b + 1]] for b in range(B)]
            else:
                torch.cuda.current_stream().synchronize()
        res = h["results"].numpy()[:B].view(np.uint32).copy().view(RESULT_DTYPE).reshape(B)
        # model_rows is the decoded map's highest label + 1: a label past the frame's own rows would otherwise read the
        # zero rows that pad it to the buffers' K
        bad = [b for b in range(B) if res["sym_count"][b] != sym_n[b] or res["seq_count"][b] != seq_n[b]
               or (res["flags"][b] & 6) or res["model_rows"][b] > rows[b]]
        if bad:
            raise ValueError("malformed .rpcc stream(s) at batch index %s (section lengths do not match the label map, or "
                             "a label has no model row; wrong lidar / framework settings?)" % bad[:8])
        return dict(range=d["range"][:B].view(B, H, W), xyz=None if xyz is None else xyz[:B].view(B, H, W, 3),
                    labels=d["labels"][:B].view(B, H, W), results=res, points=points)
