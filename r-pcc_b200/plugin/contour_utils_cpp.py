"""contour_utils_cpp (cpp_modules.cpp:623-629)."""
from ._np import C, np, _lib, check, ptr, i32, hw


def extract_contour(idx_map):
    """-> (contour_map (H,W) int32, idx_sequence (L,) int32), cpp_modules.cpp:521-558."""
    seg = i32(idx_map)
    H, W = hw(seg)
    contour = np.empty((H, W), np.int32)
    seq = np.empty(H * W, np.int32)
    L = C.c_int64(0)
    check(_lib.lib().rpcc_op_extract_contour(ptr(seg), H, W, ptr(contour), ptr(seq), C.byref(L)))
    return contour, seq[:L.value].copy()


def recover_map(contour_map, idx_sequence):
    """-> (H,W) int32, cpp_modules.cpp:561-593."""
    cm = i32(contour_map)
    H, W = hw(cm)
    seq = i32(idx_sequence)
    out = np.empty((H, W), np.int32)
    check(_lib.lib().rpcc_op_recover_map(ptr(cm), ptr(seq), seq.size, H, W, ptr(out)))
    return out
