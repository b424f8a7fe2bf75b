"""Stream-ordered batch stages over torch CUDA tensors (torch is plumbing: device memory and
streams; every kernel is in librpcc_b200.so).  One function per `rpcc_*_batch` entry point."""
import torch

from . import _lib
from ._lib import EVAL_COLS, NORMAL_KNN, NORMAL_RADIUS, P2PLANE_COLS, check, ptr


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.RpccError("expected CUDA tensors (no CPU fallback)")
        if t is not None and not t.is_contiguous():
            raise _lib.RpccError("expected contiguous tensors")


def project_batch(points, offsets, lidar, out=None):
    """points (N,3|4) f32 cuda, offsets (B+1,) int64 cuda -> range (B,H,W) f32."""
    _need_cuda(points, offsets)
    B = offsets.numel() - 1
    rng = out if out is not None else torch.empty((B, lidar.H, lidar.W), dtype=torch.float32, device=points.device)
    scratch = torch.empty((max(B, 1) * 4,), dtype=torch.int32, device=points.device)
    check(_lib.lib().rpcc_project_batch(ptr(points), points.shape[1], ptr(offsets), B, lidar.H, lidar.W,
                                        lidar.horizontal_FOV, lidar.vertical_max, lidar.vertical_min, ptr(rng),
                                        ptr(scratch), _stream()))
    return rng


def range_to_xyz_batch(rng, lut):
    _need_cuda(rng, lut)
    B = rng.shape[0]
    HW = lut.numel() // 3
    xyz = torch.empty((B,) + tuple(lut.shape), dtype=torch.float32, device=rng.device)
    check(_lib.lib().rpcc_range_to_xyz_batch(ptr(rng), ptr(lut), B, HW, ptr(xyz), _stream()))
    return xyz


def fps_batch(points, m):
    """points (B,n,3) f32 cuda -> idx (B,m) int32 (reference furthest_point_sample)."""
    _need_cuda(points)
    B, n, _ = points.shape
    temp = torch.empty((B, n), dtype=torch.float32, device=points.device)
    idx = torch.empty((B, m), dtype=torch.int32, device=points.device)
    check(_lib.lib().rpcc_fps_batch(ptr(points), B, n, m, ptr(temp), ptr(idx), _stream()))
    return idx


def segment_fps_batch(rng, lut, ground, m, thr=0.1):
    _need_cuda(rng, lut, ground)
    B, H, W = rng.shape[0], lut.shape[0], lut.shape[1]
    cidx = torch.empty((B, m), dtype=torch.int32, device=rng.device)
    centers = torch.empty((B, m, 3), dtype=torch.float32, device=rng.device)
    check(_lib.lib().rpcc_segment_fps_batch(ptr(rng), ptr(lut), ptr(ground), B, H, W, m, thr,
                                            ptr(cidx), ptr(centers), _stream()))
    return cidx, centers


def new_book(B, H, W, K, device):
    n = _lib.lib().rpcc_book_bytes(B, H, W, K)
    return torch.empty((n,), dtype=torch.uint8, device=device)


def assign_labels_batch(rng, lut, ground, centers, book=None):
    _need_cuda(rng, lut, ground, centers)
    B, H, W = rng.shape[0], lut.shape[0], lut.shape[1]
    m = centers.shape[1]
    labels = torch.empty((B, H, W), dtype=torch.uint8, device=rng.device)
    if book is None:
        book = new_book(B, H, W, m + 2, rng.device)
    check(_lib.lib().rpcc_assign_labels_batch(ptr(rng), ptr(lut), ptr(ground), ptr(centers), B, H, W, m,
                                              ptr(labels), ptr(book), _stream()))
    return labels, book


def label_stats_batch(rng, labels, K, book=None):
    _need_cuda(rng, labels)
    B, H, W = labels.shape
    if book is None:
        book = new_book(B, H, W, K, rng.device)
    check(_lib.lib().rpcc_label_stats_batch(ptr(rng), ptr(labels), B, H, W, K, ptr(book), _stream()))
    return book


def point_model_batch(rng, labels, ground, book, K):
    _need_cuda(rng, labels, ground, book)
    B, H, W = labels.shape
    model = torch.empty((B, K, 4), dtype=torch.float32, device=rng.device)
    results = torch.empty((B, 4), dtype=torch.int32, device=rng.device)
    check(_lib.lib().rpcc_point_model_batch(ptr(rng), ptr(labels), ptr(ground), ptr(book), B, H, W, K,
                                            ptr(model), ptr(results), _stream()))
    return model, results


def quantize_pack_batch(rng, labels, model, lut, book, step, step_per_label=None):
    _need_cuda(rng, labels, model, lut, book, step_per_label)
    B, H, W = labels.shape
    K = model.shape[1]
    HW = H * W
    symbols = torch.empty((B, HW), dtype=torch.int16, device=rng.device)
    contour = torch.empty((B, (HW + 7) // 8), dtype=torch.uint8, device=rng.device)
    seq = torch.empty((B, HW), dtype=torch.int16, device=rng.device)  # uint16 payload
    check(_lib.lib().rpcc_quantize_pack_batch(ptr(rng), ptr(labels), ptr(model), ptr(lut), ptr(book),
                                              ptr(step_per_label), step, B, H, W, K, ptr(symbols), HW, ptr(contour),
                                              ptr(seq), HW, None, None, _stream()))
    return symbols, contour, seq


def eval_batch(range_ref, range_rec, lut, lidar, labels_ref=None, labels_rec=None, f1_threshold=0.02, want_dist=False):
    """The --eval figures for B pairs of range images over one ray table (rpcc_eval_batch, csrc/evalq.cu).
    -> (metrics (B, 12) f64 cuda, dist1 (B,H,W) f32 | None, dist2 | None); dist* are the squared nearest-neighbour
    distances of the reference's chamfer kernel, -1 at pixels that are not points."""
    _need_cuda(range_ref, range_rec, lut, labels_ref, labels_rec)
    B = range_ref.shape[0]
    H, W = lidar.H, lidar.W
    metrics = torch.empty((B, EVAL_COLS), dtype=torch.float64, device=range_ref.device)
    ws = torch.empty((_lib.lib().rpcc_eval_workspace_bytes(B, H, W),), dtype=torch.uint8, device=range_ref.device)
    d1 = torch.empty((B, H, W), dtype=torch.float32, device=range_ref.device) if want_dist else None
    d2 = torch.empty((B, H, W), dtype=torch.float32, device=range_ref.device) if want_dist else None
    check(_lib.lib().rpcc_eval_batch(ptr(range_ref), ptr(range_rec), ptr(lut), ptr(labels_ref), ptr(labels_rec), B, H, W,
                                     lidar.horizontal_FOV, lidar.vertical_max, lidar.vertical_min, f1_threshold ** 2,
                                     ptr(d1), ptr(d2), ptr(metrics), ptr(ws), _stream()))
    return metrics, d1, d2


def normals_batch(rng, lut, lidar, knn=NORMAL_KNN, radius=NORMAL_RADIUS):
    """k-NN PCA normals of B range images over one ray table (rpcc_normals_batch, csrc/normals.cu).
    -> (normals (B,H,W,3) f32 cuda, (0,0,0) where there is no normal; whole-image scans per frame (B,) int32 cuda)."""
    _need_cuda(rng, lut)
    B = rng.shape[0]
    H, W = lidar.H, lidar.W
    normals = torch.empty((B, H, W, 3), dtype=torch.float32, device=rng.device)
    ws = torch.empty((_lib.lib().rpcc_normals_workspace_bytes(B, H, W),), dtype=torch.uint8, device=rng.device)
    check(_lib.lib().rpcc_normals_batch(ptr(rng), ptr(lut), B, H, W, lidar.horizontal_FOV, lidar.vertical_max,
                                        lidar.vertical_min, int(knn), float(radius), ptr(normals), ptr(ws), _stream()))
    return normals, ws[:4 * B].view(torch.int32)


def p2plane_batch(range_ref, range_rec, lut, lidar, normals_ref, normals_rec):
    """Point-to-plane error of B pairs of range images with their normals (rpcc_p2plane_batch, csrc/normals.cu).
    -> metrics (B, 7) f64 cuda: n1, sum err1, no-normal count 1, n2, sum err2, no-normal count 2, whole-image scans."""
    _need_cuda(range_ref, range_rec, lut, normals_ref, normals_rec)
    B = range_ref.shape[0]
    H, W = lidar.H, lidar.W
    metrics = torch.empty((B, P2PLANE_COLS), dtype=torch.float64, device=range_ref.device)
    ws = torch.empty((_lib.lib().rpcc_p2plane_workspace_bytes(B, H, W),), dtype=torch.uint8, device=range_ref.device)
    check(_lib.lib().rpcc_p2plane_batch(ptr(range_ref), ptr(range_rec), ptr(lut), ptr(normals_ref), ptr(normals_rec), B, H,
                                        W, lidar.horizontal_FOV, lidar.vertical_max, lidar.vertical_min, ptr(metrics),
                                        ptr(ws), _stream()))
    return metrics


def intensity_owner_batch(points, offsets, lidar):
    """points (N,4) f32 cuda (x, y, z, intensity), offsets (B+1,) int64 cuda -> (range (B,H,W) f32, owner (B,H,W) int32
    in-frame row of the pixel's owner, -1 at empty pixels, intensity (B,H,W) f32): the projection, then the owner pass
    and the gather (DESIGN.md §4, "Intensity")."""
    _need_cuda(points, offsets)
    if points.dim() != 2 or points.shape[1] != 4:
        raise _lib.RpccError("intensity needs (N,4) points")
    B = offsets.numel() - 1
    dev = points.device
    rng = torch.empty((B, lidar.H, lidar.W), dtype=torch.float32, device=dev)
    scratch = torch.empty((max(B, 1) * 4,), dtype=torch.int32, device=dev)
    owner = torch.empty((B, lidar.H, lidar.W), dtype=torch.int32, device=dev)
    inten = torch.empty((B, lidar.H, lidar.W), dtype=torch.float32, device=dev)
    args = (lidar.H, lidar.W, lidar.horizontal_FOV, lidar.vertical_max, lidar.vertical_min)
    check(_lib.lib().rpcc_project_batch(ptr(points), 4, ptr(offsets), B, *args, ptr(rng), ptr(scratch), _stream()))
    check(_lib.lib().rpcc_intensity_owner_batch(ptr(points), ptr(offsets), B, *args, ptr(rng), ptr(scratch), ptr(owner),
                                                ptr(inten), _stream()))
    return rng, owner, inten


def intensity_pack_batch(intensity, rng, step):
    """intensity, range (B,H,W) f32 cuda -> (the frames' sections back to back (n,) u8, base (B+1,) int64,
    clamped (B,) bool)."""
    _need_cuda(intensity, rng)
    B = rng.shape[0]
    counts = (rng.reshape(B, -1) != 0).sum(1)
    base = torch.zeros((B + 1,), dtype=torch.int64, device=rng.device)
    torch.cumsum(counts, 0, out=base[1:])
    out = torch.empty((max(int(base[-1]), 1),), dtype=torch.uint8, device=rng.device)
    res = torch.zeros((B, 4), dtype=torch.int32, device=rng.device)
    check(_lib.lib().rpcc_intensity_pack_batch(ptr(intensity), ptr(rng), B, rng.shape[1], rng.shape[2], float(step),
                                               ptr(base), ptr(out), ptr(res), _stream()))
    return out[:int(base[-1])], base, (res[:, 3] & _lib.FLAG_INTENSITY_CLAMPED) != 0


def intensity_unpack_batch(labels, stream, base, step):
    """labels (B,H,W) u8 cuda (1 = empty), the sections back to back, base (B+1,) int64 -> intensity (B,H,W) f32."""
    _need_cuda(labels, stream, base)
    B, H, W = labels.shape
    out = torch.empty((B, H, W), dtype=torch.float32, device=labels.device)
    check(_lib.lib().rpcc_intensity_unpack_batch(ptr(labels), ptr(stream), ptr(base), B, H, W, float(step), ptr(out),
                                                 _stream()))
    return out
