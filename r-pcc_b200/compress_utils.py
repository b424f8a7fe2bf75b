"""Mirror of utils/compress_utils.py: QuantizationModule (:35-132), compress_point_cloud (:138-164),
save/read_compressed_bitstream (:167-196), decompress_point_cloud (:199-214), BasicCompressor (:232-310).

The `.rpcc` layout is the reference's: no header; per section a native-endian int32 length then the
entropy-coded bytes, in the order [salience_level (non-uniform only)], contour_map, idx_sequence,
plane_param, residual_quantized (SURVEY App. B), optionally followed by this project's intensity section (DESIGN.md
§4), which every reader of the first five skips.  The entropy coder itself (bz2 / gzip / lz4) stays
on the host, as in the reference."""
import bz2
import copy
import ctypes as C
import ctypes.util as ctypes_util
import gzip
import struct

import numpy as np

from . import _lib
from ._lib import check, ptr
from .config import load_compressor_cfg
from .contour_utils import ContourExtractor
from .plugin import feature_extractor_cpp, quantization_utils_cpp


def extract_features_without_ground(range_image, seg_idx, feature_region=3, segments=8, sharp_num=4, less_sharp_num=8,
                                    flat_num=6):
    return feature_extractor_cpp.extract_features_with_segment(range_image, seg_idx, feature_region, segments,
                                                               sharp_num, less_sharp_num, flat_num)


class QuantizationModule:
    def __init__(self, base_accuracy, level_kp_num=(30, 10, 3, 0), level_dacc=(0, 0.02, 0.04, 0.06),
                 ground_salience_level=2, feature_region=3, segments=8, sharp_num=4, less_sharp_num=8, flat_num=6,
                 uniform=True):
        self.uniform = uniform
        if uniform:
            self.acc = base_accuracy
        else:
            self.level_kp_num = np.array(level_kp_num)
            self.acc = np.array([base_accuracy] * len(self.level_kp_num)) + np.array(level_dacc)
            self.ground_level = ground_salience_level
            self.feature_region = feature_region
            self.segments = segments
            self.sharp_num = sharp_num
            self.less_sharp_num = less_sharp_num
            self.flat_num = flat_num

    def quantize_residual(self, residual, seg_idx, point_cloud=None, range_image=None):
        if self.uniform:
            residual_quantized = quantization_utils_cpp.uniform_quantize(seg_idx, residual, self.acc)
            salience_level = None
            key_point_map = None
        else:
            feature_map, key_point_map = extract_features_without_ground(range_image, seg_idx, self.feature_region,
                                                                         self.segments, self.sharp_num,
                                                                         self.less_sharp_num, self.flat_num)
            residual_quantized, salience_level = quantization_utils_cpp.nonuniform_quantize(
                seg_idx, residual, key_point_map, self.level_kp_num, self.acc, self.ground_level)
        return residual_quantized, salience_level, key_point_map

    def dequantize_residual(self, quantized_residual, seg_idx, salience_level=None):
        """-> (H,W,1) f32: f32((double)q * step) scattered back label-major (utils/compress_utils.py:114-132,
        numpy >= 2 promotion); the reference's Python loop of np.where scans is one device pass here."""
        seg = np.ascontiguousarray(seg_idx, dtype=np.int32)
        H, W = seg.shape
        q = np.ascontiguousarray(quantized_residual, dtype=np.int16)
        K = max(int(seg.max()) + 1, 2)
        if self.uniform:
            steps = np.full(K, self.acc, np.float64)
        else:
            sal = np.asarray(salience_level)
            steps = np.asarray(self.acc, np.float64)[sal[:K].astype(np.int64)]
            if steps.size < K:
                steps = np.concatenate((steps, np.full(K - steps.size, self.acc[-1])))
        steps = np.ascontiguousarray(steps, np.float64)
        residual = np.empty((H, W), np.float32)
        consumed = C.c_int64(0)
        check(_lib.lib().rpcc_op_dequantize(ptr(q), q.size, ptr(seg), H, W, ptr(steps), K, ptr(residual),
                                            C.byref(consumed)))
        if consumed.value != q.shape[0]:
            raise ValueError("residual stream has %d symbols but the label map needs %d" % (q.shape[0], consumed.value))
        return np.expand_dims(residual, -1)


def compress_point_cloud(basic_compressor, plane_param, cluster_idx, salience_level, nonzero_residual_quantized,
                         ground_residual_quantized=None, cluster_residual_quantized=None,
                         point_cloud=None, range_image=None, full=False):
    original_data = {}
    original_data["residual_quantized"] = nonzero_residual_quantized.astype(np.int16)
    if full:
        if point_cloud is not None:
            original_data["point_cloud"] = point_cloud.astype(np.float32)
        if range_image is not None:
            original_data["range_image"] = range_image.astype(np.float32)
        if ground_residual_quantized is not None:
            original_data["ground_residual"] = ground_residual_quantized.astype(np.int16)
        if cluster_residual_quantized is not None:
            original_data["cluster_residual"] = cluster_residual_quantized.astype(np.int16)
    if salience_level is not None:
        original_data["salience_level"] = salience_level.astype(np.uint8)
    contour_map, idx_sequence = ContourExtractor.extract_contour(cluster_idx)
    contour_map = np.packbits(contour_map.astype(bool), axis=None)
    original_data["contour_map"] = contour_map.astype(np.uint8)
    original_data["idx_sequence"] = idx_sequence.astype(np.uint16)
    original_data["plane_param"] = plane_param.astype(np.float32)
    compressed_data = basic_compressor.compress_dict(original_data)
    return original_data, compressed_data


SECTION_ORDER = ("salience_level", "contour_map", "idx_sequence", "plane_param", "residual_quantized")
INTENSITY_SECTION = "intensity"     # optional, after residual_quantized


def pack_bitstream(compressed_data, uniform=True):
    """The bytes save_compressed_bitstream writes (utils/compress_utils.py:167-179), then the intensity section when
    `compressed_data` has one."""
    out = []
    keys = SECTION_ORDER + ((INTENSITY_SECTION,) if INTENSITY_SECTION in compressed_data else ())
    for key in keys:
        if key == "salience_level" and uniform:
            continue
        out.append(struct.pack("i", len(compressed_data[key])))
        out.append(bytes(compressed_data[key]))
    return b"".join(out)


def save_compressed_bitstream(file, compressed_data, uniform=True):
    with open(file, "wb") as f:
        f.write(pack_bitstream(compressed_data, uniform))


def parse_bitstream(buf, uniform=True, intensity=False):
    """The sections of a `.rpcc`; a trailing intensity section is skipped unless `intensity`, which requires it."""
    compressed_data = {}
    pos = 0
    keys = SECTION_ORDER + ((INTENSITY_SECTION,) if intensity else ())
    for key in keys:
        if key == "salience_level" and uniform:
            continue
        if key == INTENSITY_SECTION:
            if pos == len(buf):
                raise ValueError("the .rpcc has no intensity section (written without --intensity_accuracy)")
            if pos + 4 > len(buf) or not 0 <= struct.unpack_from("i", buf, pos)[0] <= len(buf) - pos - 4:
                raise ValueError("truncated .rpcc: the intensity section is shorter than its length")
        length = struct.unpack_from("i", buf, pos)[0]
        pos += 4
        compressed_data[key] = buf[pos:pos + length]
        pos += length
    return compressed_data


def read_compressed_bitstream(file, uniform=True, intensity=False):
    with open(file, "rb") as f:
        return parse_bitstream(f.read(), uniform, intensity)


def decompress_point_cloud(compressed_data, basic_compressor, model_num, H, W):
    """-> (residual_quantized i16, idx_map (H,W), salience_level | None, plane_param (rows,4)).
    `model_num` is accepted for signature parity; the row count comes from the section length (the
    reference declares cluster_num+1 rows although cluster_num+2 are stored, SURVEY App. B / C1)."""
    decompressed_data = basic_compressor.decompress_dict(compressed_data)
    plane_param = np.frombuffer(decompressed_data["plane_param"], dtype=np.float32).reshape(-1, 4)
    contour_map = np.unpackbits(np.frombuffer(decompressed_data["contour_map"], dtype=np.uint8))[:H * W]
    contour_map = np.reshape(contour_map, (H, W))
    idx_sequence = np.frombuffer(decompressed_data["idx_sequence"], dtype=np.uint16)
    idx_map = ContourExtractor.recover_map(contour_map, idx_sequence)
    if "salience_level" in decompressed_data.keys():
        salience_level = np.frombuffer(decompressed_data["salience_level"], dtype=np.uint8)
    else:
        salience_level = None
    residual_quantized = np.frombuffer(decompressed_data["residual_quantized"], dtype=np.int16)
    return residual_quantized, idx_map, salience_level, plane_param


_LZ4 = None


def _lz4():
    global _LZ4
    if _LZ4 is None:
        lib = C.CDLL("liblz4.so.1")
        lib.LZ4_compressBound.restype = C.c_int
        lib.LZ4_compress_default.restype = C.c_int
        lib.LZ4_decompress_safe.restype = C.c_int
        _LZ4 = lib
    return _LZ4


_BZ2 = False      # False: not tried yet; None: libbz2 not loadable (bz2.compress is used)
# libbz2's workFactor only decides how long the main block sort may struggle with repetitive data before the fallback sort
# takes over; the bytes written are the same either way (bzip2 manual, BZ2_bzCompressInit).  The label sequence is exactly
# that kind of input: sending it to the fallback sort at once halves its time (21 -> 11 ms for a 64E frame), which is a
# quarter of the whole host entropy stage; short sequences (the 12 KB of a KITTI frame) sort quickly either way and keep
# the default.  Sections not listed keep the library default (30, what bz2.compress passes).
_BZ2_WORK_FACTOR = {"idx_sequence": (32768, 1)}     # section -> (minimum length in bytes, work factor)


def _bz2lib():
    global _BZ2
    if _BZ2 is False:
        _BZ2 = None
        for name in (ctypes_util.find_library("bz2"), "libbz2.so.1.0", "libbz2.so.1"):
            if not name:
                continue
            try:
                lib = C.CDLL(name)
                lib.BZ2_bzBuffToBuffCompress.argtypes = [C.c_char_p, C.POINTER(C.c_uint), C.c_char_p, C.c_uint, C.c_int,
                                                         C.c_int, C.c_int]
                lib.BZ2_bzBuffToBuffCompress.restype = C.c_int
                _BZ2 = lib
                break
            except (OSError, AttributeError):
                continue
    return _BZ2


class BasicCompressor:
    """utils/compress_utils.py:232-310.  bzip2 = bz2.compress (level 9), gzip/deflate = gzip.compress
    (level 9; pass mtime for reproducible bytes, the reference leaves it at "now"), lz4 = the
    python-lz4 0.7 `dumps` framing (4-byte LE size + one LZ4 block) through liblz4."""

    def __init__(self, compressor_yaml=None, method_name=None, gzip_mtime=None):
        self.method_name = None
        self.gzip_mtime = gzip_mtime
        if compressor_yaml is not None:
            self.method_name = load_compressor_cfg(compressor_yaml)["basic_compressor"]
        if method_name is not None:
            self.method_name = method_name
        if self.method_name is not None:
            assert self.method_name in ["lz4", "bzip2", "gzip", "deflate"], \
                "Compression method is not existed. (lz4, bzip2, gzip, deflate)"

    def set_method(self, method_name):
        self.method_name = method_name
        assert self.method_name in ["lz4", "bzip2", "gzip", "deflate"], \
            "Compression method is not existed. (lz4, bzip2, gzip, deflate)"

    def compress_dict(self, data_dict):
        return {key: self.compress(val, section=key) for key, val in data_dict.items()}

    def decompress_dict(self, data_dict):
        return {key: self.decompress(val) for key, val in data_dict.items()}

    def compress(self, np_array, section=None):
        """`section` (the .rpcc section name) only tunes how the coder is driven, never the bytes it writes."""
        if self.method_name == "lz4":
            return self.lz4_compress(np_array)
        if self.method_name == "bzip2":
            min_len, wf = _BZ2_WORK_FACTOR.get(section, (0, 0))
            nbytes = len(np_array) if isinstance(np_array, (bytes, bytearray)) else np.asarray(np_array).nbytes
            return self.bzip2_compress(np_array, wf if nbytes >= min_len else 0)
        if self.method_name in ("gzip", "deflate"):
            return self.gzip_compress(np_array, self.gzip_mtime)

    def decompress(self, bitstream):
        if self.method_name == "lz4":
            return self.lz4_decompress(bitstream)
        if self.method_name == "bzip2":
            return self.bzip2_decompress(bitstream)
        if self.method_name in ("gzip", "deflate"):
            return self.gzip_decompress(bitstream)

    def calc_compressed_bytes(self, np_array):
        return len(self.compress(np_array))

    @staticmethod
    def lz4_compress(np_array):
        raw = bytes(memoryview(np.ascontiguousarray(np_array)).cast("B")) if not isinstance(np_array, (bytes, bytearray)) else bytes(np_array)
        lib = _lz4()
        cap = lib.LZ4_compressBound(len(raw))
        dst = C.create_string_buffer(cap)
        n = lib.LZ4_compress_default(raw, dst, len(raw), cap)
        if n <= 0 and len(raw) > 0:
            raise RuntimeError("LZ4 compression failed")
        return struct.pack("<I", len(raw)) + dst.raw[:n]

    @staticmethod
    def lz4_decompress(data):
        size = struct.unpack_from("<I", data, 0)[0]
        dst = C.create_string_buffer(max(size, 1))
        n = _lz4().LZ4_decompress_safe(bytes(data[4:]), dst, len(data) - 4, size)
        if n != size:
            raise RuntimeError("LZ4 decompression failed")
        return dst.raw[:size]

    @staticmethod
    def bzip2_compress(np_array, work_factor=0):
        """bz2.compress(x) of utils/compress_utils.py:296-298 (level 9).  With a work factor, the same libbz2 is called
        through ctypes (the GIL is released for the call) -- byte-identical output, see _BZ2_WORK_FACTOR."""
        lib = _bz2lib() if work_factor else None
        if lib is None:
            return bz2.compress(np_array)
        raw = np_array if isinstance(np_array, bytes) else bytes(memoryview(np.ascontiguousarray(np_array)).cast("B")) \
            if not isinstance(np_array, bytearray) else bytes(np_array)
        cap = len(raw) + len(raw) // 100 + 600          # bzlib: 1 % larger than the input plus 600 bytes always suffices
        dst = C.create_string_buffer(cap)
        n = C.c_uint(cap)
        if lib.BZ2_bzBuffToBuffCompress(dst, C.byref(n), raw, len(raw), 9, 0, int(work_factor)) != 0:
            return bz2.compress(raw)
        return dst.raw[:n.value]

    @staticmethod
    def bzip2_decompress(data):
        return bz2.decompress(data)

    @staticmethod
    def gzip_compress(np_array, mtime=None):
        return gzip.compress(np_array, mtime=mtime)

    @staticmethod
    def gzip_decompress(data):
        return gzip.decompress(data)
