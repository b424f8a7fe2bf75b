"""chamfer_3D (chamfer3D/chamfer_cuda.cpp:28-31) forward only, and chamfer_3DDist
(chamfer3D/dist_chamfer_3D.py:29-80) without autograd (R-PCC never differentiates through it)."""
import torch

from .. import _lib
from .._lib import check, ptr


def forward(xyz1, xyz2, dist1, dist2, idx1, idx2):
    """(B,N,3),(B,M,3) f32 cuda; fills dist1 (B,N), dist2 (B,M) f32 and idx1, idx2 int32; returns 1."""
    B, n, _ = xyz1.shape
    m = xyz2.shape[1]
    st = torch.cuda.current_stream().cuda_stream
    scratch = torch.empty((n + m,), dtype=torch.int64, device=xyz1.device)
    for b in range(B):
        check(_lib.lib().rpcc_chamfer_batch(ptr(xyz1[b]), n, ptr(xyz2[b]), m, ptr(dist1[b]), ptr(idx1[b]),
                                            ptr(dist2[b]), ptr(idx2[b]), ptr(scratch), st))
    return 1


class chamfer_3DDist(torch.nn.Module):
    def forward(self, input1, input2):
        input1 = input1.contiguous().float()
        input2 = input2.contiguous().float()
        B, n, _ = input1.shape
        m = input2.shape[1]
        dist1 = torch.empty((B, n), dtype=torch.float32, device=input1.device)
        dist2 = torch.empty((B, m), dtype=torch.float32, device=input1.device)
        idx1 = torch.empty((B, n), dtype=torch.int32, device=input1.device)
        idx2 = torch.empty((B, m), dtype=torch.int32, device=input1.device)
        forward(input1, input2, dist1, dist2, idx1, idx2)
        return dist1, dist2, idx1, idx2
