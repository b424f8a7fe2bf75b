"""quantization_utils_cpp (cpp_modules.cpp:615-621)."""
from ._np import C, np, _lib, check, ptr, f32, i32, hw


def uniform_quantize(seg_idx, residual, acc):
    """-> (n,) int32 label-major symbols, cpp_modules.cpp:288-334."""
    seg = i32(seg_idx)
    H, W = hw(seg)
    res = f32(residual)
    out = np.empty(H * W, np.int32)
    n = C.c_int64(0)
    check(_lib.lib().rpcc_op_uniform_quantize(ptr(seg), ptr(res), H, W, acc, ptr(out), C.byref(n)))
    return out[:n.value].copy()


def nonuniform_quantize(seg_idx, residual, key_point_map, level_kp_num, level_acc, ground_level):
    """-> ((n,) int32 symbols, (K,) int32 salience levels), cpp_modules.cpp:337-424."""
    seg = i32(seg_idx)
    H, W = hw(seg)
    res = f32(residual)
    kp = i32(key_point_map)
    lk = i32(level_kp_num)
    la = f32(level_acc)
    out = np.empty(H * W, np.int32)
    sal = np.empty(256, np.int32)
    n = C.c_int64(0)
    K = C.c_int(0)
    check(_lib.lib().rpcc_op_nonuniform_quantize(ptr(seg), ptr(res), ptr(kp), H, W, ptr(lk), ptr(la), la.size,
                                                 int(ground_level), ptr(out), C.byref(n), ptr(sal), C.byref(K)))
    return out[:n.value].copy(), sal[:K.value].copy()
