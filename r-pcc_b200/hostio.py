"""The native host stage of the batch tools: `.bin` reader and the entropy-coder pool (csrc/hostio.cu).

`Packer` is BasicCompressor.compress_dict + save_compressed_bitstream (reference utils/compress_utils.py:167-179,
255-310) for every frame of an encode_host result, run by C++ threads straight out of the pinned buffers the GPU
wrote into; the GIL is not involved.  Only bzip2 (the reference default) runs there; the other coders keep the
Python path in batch.py."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import check, ptr


class Packer:
    def __init__(self, threads, method="bzip2"):
        self._h = C.c_void_p(0)
        check(_lib.lib().rpcc_packer_create(int(threads), method.encode(), C.byref(self._h)))
        self._keep = {}

    def close(self):
        if self._h:
            _lib.lib().rpcc_packer_destroy(self._h)
            self._h = C.c_void_p(0)
        self._keep.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def submit(self, enc, K, uniform, paths=None, keep=False):
        """enc: the dict BatchEncoder.encode_host returned (its arrays must stay untouched until wait()).
        paths: list of output files or None; keep=True returns every file in memory too.
        -> ticket; wait(ticket) returns (sizes (B,) uint32, blobs (B, stride) uint8 | None)."""
        res = enc["results"]
        B = len(res)
        res_c = np.ascontiguousarray(res)
        sizes = np.zeros(B, np.uint32)
        status = np.zeros(B, np.int32)
        blob_stride = 0
        if keep and B:
            # bzip2 never expands a section by more than 1 % + 600 bytes (bzlib manual); 4 length bytes per section
            raw = (int(enc["contour"].shape[1]) + 2 * int(res["seq_count"].max()) + 17 * int(K) + 3 * int(res["sym_count"].max()))
            blob_stride = raw + raw // 100 + 6 * 604
        blobs = np.empty((B, blob_stride), np.uint8) if blob_stride else None
        arr = None
        if paths is not None:
            arr = (C.c_char_p * B)(*[p.encode() if p else None for p in paths])
        sal = enc.get("salience")
        inten = enc.get("intensity")
        ticket = C.c_longlong(0)
        check(_lib.lib().rpcc_packer_submit_intensity(
            self._h, B, int(K), int(enc["contour"].shape[1]), 1 if uniform else 0, ptr(res_c), ptr(enc["model"]),
            ptr(enc["contour"]), ptr(enc["seq"]), ptr(enc["symbols"]), ptr(sal) if sal is not None else None,
            ptr(inten) if inten is not None else None, arr, ptr(sizes), ptr(status),
            ptr(blobs) if blobs is not None else None, blob_stride, C.byref(ticket)))
        self._keep[ticket.value] = (res_c, sizes, status, blobs, arr, enc)
        return ticket.value

    def wait(self, ticket):
        rc = _lib.lib().rpcc_packer_wait(self._h, ticket)
        res_c, sizes, status, blobs, arr, enc = self._keep.pop(ticket)
        check(rc)
        return sizes, blobs


def read_bin_xyz(path, dst):
    """KITTI .bin -> the xyz columns into dst ((cap, 3) f32 numpy view, e.g. of a pinned tensor); returns the rows."""
    rows = C.c_int64(0)
    check(_lib.lib().rpcc_read_bin_xyz(path.encode(), ptr(dst), dst.shape[0], C.byref(rows)))
    return int(rows.value)


def read_bin_rows(path, dst):
    """KITTI .bin -> whole rows (x, y, z, intensity) into dst ((cap, 4) f32 numpy view); returns the rows."""
    rows = C.c_int64(0)
    check(_lib.lib().rpcc_read_bin_rows(path.encode(), ptr(dst), dst.shape[0], C.byref(rows)))
    return int(rows.value)


def unpack_rpcc(blob, uniform, cap, intensity=False):
    """One bzip2 `.rpcc` -> dict of decompressed sections (bytes), as BasicCompressor.decompress_dict over
    read_compressed_bitstream; intensity=True also the intensity section, which the file must have."""
    names = ("contour_map", "idx_sequence", "plane_param", "residual_quantized")
    if not uniform:
        names = ("salience_level",) + names
    dst = np.empty(cap, np.uint8)
    lens = np.zeros(6, np.uint32)
    src = np.frombuffer(blob, np.uint8)
    fn = _lib.lib().rpcc_unpack_rpcc_intensity if intensity else _lib.lib().rpcc_unpack_rpcc
    check(fn(ptr(src), src.size, 1 if uniform else 0, ptr(dst), cap, ptr(lens)))
    out, at = {}, 0
    for i, k in enumerate(names):
        out[k] = dst[at:at + int(lens[i])]
        at += int(lens[i])
    if intensity:
        out["intensity"] = dst[at:at + int(lens[5])]
    return out
