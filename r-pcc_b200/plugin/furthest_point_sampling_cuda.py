"""furthest_point_sampling_cuda (ops/fps/src/fps_api.cpp:7-9) and the autograd-free equivalent of
ops/fps/fps_utils.py:10-36."""
import torch

from .. import _lib
from .._lib import check, ptr


def furthest_point_sampling_wrapper(b, n, m, points_tensor, temp_tensor, idx_tensor):
    """Same contract as ops/fps/src/sampling.cpp:24-37: CUDA, contiguous tensors; writes idx in place;
    returns 1.  Errors raise instead of exit(-1)."""
    for t in (points_tensor, temp_tensor, idx_tensor):
        if not t.is_cuda or not t.is_contiguous():
            raise _lib.RpccError("furthest_point_sampling_wrapper needs contiguous CUDA tensors")
    st = torch.cuda.current_stream().cuda_stream
    check(_lib.lib().rpcc_fps_batch(ptr(points_tensor), int(b), int(n), int(m), ptr(temp_tensor), ptr(idx_tensor), st))
    return 1


def furthest_point_sample(xyz, npoint):
    """(B,N,3) f32 cuda -> (B,npoint) int32 cuda (ops/fps/fps_utils.py:12-29)."""
    assert xyz.is_contiguous()
    B, N, _ = xyz.size()
    output = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
    temp = torch.empty((B, N), dtype=torch.float32, device=xyz.device)
    furthest_point_sampling_wrapper(B, N, npoint, xyz, temp, output)
    return output
