#!/usr/bin/env python
"""Measurements of the SURVEY section-8 rows that are not on bench.py's headline metric, each beside the
reference's own implementation of the row timed on the same box:
   a5  FPS drop-in (rpcc_fps_batch)          vs the reference's CUDA kernel (oracle/_ref/libref_fps.so, same GPU)
   a11 decode (rpcc_decode_batch)            vs the oracle's restatement of recover_map + dequantize + predict (1 host core)
   a12 chamfer (rpcc_chamfer_batch)          vs the reference's CUDA kernel (oracle/_ref/libref_chamfer.so, same GPU)
   python scripts/bench_rows.py [frames]     (prints one JSON object; CUDA events, warm-up first)"""
import json
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import oracle  # noqa: E402  (the checker / CPU baseline only)
from oracle import ref  # noqa: E402
from rpcc_b200 import _lib, device, synthetic  # noqa: E402
from rpcc_b200._lib import check, ptr  # noqa: E402
from rpcc_b200.batch import BatchEncoder  # noqa: E402
from rpcc_b200.lidar import LidarConfig  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 296
LIDAR = "Velodyne64E"
cfg = LidarConfig(LIDAR)
H, W, HW = cfg.H, cfg.W, cfg.HW
dev = torch.device("cuda", 0)
out = {}


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


nd = 16
per = [synthetic.frame(100 + i, LIDAR) for i in range(nd)]
pts = np.concatenate([per[i % nd][0] for i in range(B)], 0)
off = np.cumsum([0] + [per[i % nd][0].shape[0] for i in range(B)]).astype(np.int64)
grounds = np.stack([per[i % nd][1] for i in range(B)]).astype(np.float32)

# ---------------------------------------------------------------------------------- encode once (inputs of the decoder)
with BatchEncoder(LIDAR, accuracy=0.02, max_batch=B, max_points=pts.shape[0], host_chunk=B) as enc:
    o = enc.encode_host(pts, off, grounds)
    res = o["results"].copy()
    K = o["model"].shape[1]
    contour = torch.from_numpy(o["contour"].copy()).to(dev)
    model = torch.from_numpy(o["model"].copy()).to(dev)
    seq_n = res["seq_count"].astype(np.uint32)
    sym_n = res["sym_count"].astype(np.uint32)
    seq_stride, sym_stride = int(seq_n.max()), int(sym_n.max())
    seq = np.zeros((B, seq_stride), np.uint16)
    sym = np.zeros((B, sym_stride), np.int16)
    for b in range(B):
        seq[b, :seq_n[b]] = o["seq"][o["seq_off"][b]:o["seq_off"][b + 1]]
        sym[b, :sym_n[b]] = o["symbols"][o["sym_off"][b]:o["sym_off"][b + 1]]
    sections0 = BatchEncoder.frame_sections(o, 0)
lut = torch.from_numpy(cfg.transform_map()).to(dev)

# ---------------------------------------------------------------------------------- a11 decode
d_seq, d_sym = torch.from_numpy(seq.view(np.int16)).to(dev), torch.from_numpy(sym).to(dev)
d_seq_n, d_sym_n = torch.from_numpy(seq_n.view(np.int32)).to(dev), torch.from_numpy(sym_n.view(np.int32)).to(dev)
steps = torch.full((B, K), 0.04, dtype=torch.float64, device=dev)
labels = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
rng = torch.empty((B, H, W), dtype=torch.float32, device=dev)
xyz = torch.empty((B, H, W, 3), dtype=torch.float32, device=dev)
book = torch.empty((_lib.lib().rpcc_book_bytes(B, H, W, K),), dtype=torch.uint8, device=dev)
results = torch.empty((B, 4), dtype=torch.int32, device=dev)
st = torch.cuda.current_stream().cuda_stream


def decode(with_xyz=True):
    check(_lib.lib().rpcc_decode_batch(ptr(contour), ptr(d_seq), seq_stride, ptr(d_seq_n), ptr(d_sym), sym_stride,
                                       ptr(d_sym_n), ptr(model), ptr(steps), ptr(lut), B, H, W, K,
                                       ptr(labels), ptr(rng), ptr(xyz) if with_xyz else None, ptr(book), ptr(results), st))


ms = timed(decode, 10)
v_mean, l_mean = float(sym_n.mean()), float(seq_n.mean())
alg = HW / 8 + 2 * l_mean + 2 * v_mean + HW + 4 * HW + 12 * HW      # in: bits, sequence, symbols; out: labels, range, xyz
t0 = time.perf_counter()
n_cpu = 4
for _ in range(n_cpu):
    rec0, xyz0, seg0 = oracle.decompress_sections(sections0, LIDAR, 0.02)
cpu_ms = (time.perf_counter() - t0) / n_cpu * 1e3
ok = bool(np.array_equal(rng[0].cpu().numpy().view(np.uint32), rec0.reshape(H, W).view(np.uint32)) and
          np.array_equal(xyz[0].cpu().numpy().view(np.uint32), xyz0.reshape(H, W, 3).view(np.uint32)))
peak = float(json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"]) if __import__("os").path.exists("MEASURED_PEAKS.json") else 6650.0
out["a11_decode"] = {"frames_per_launch": B, "ms_per_launch": ms, "frames_per_s": B / ms * 1e3,
                     "algorithmic_bytes_per_frame": alg, "achieved_gbs": alg * B / ms / 1e6, "frac_of_hbm_peak": alg * B / ms / 1e6 / peak,
                     "bit_exact_vs_oracle_frame0": ok,
                     "cpu_baseline": {"kind": "port", "cores": 1, "ms_per_frame": cpu_ms, "frames_per_s": 1e3 / cpu_ms,
                                      "sample": "%d decodes of one frame by the oracle's C restatement (recover_map, dequantize, "
                                                "intra_predict, range x LUT)" % n_cpu}}

# ---------------------------------------------------------------------------------- a5 FPS drop-in vs the reference kernel
ri = oracle.project(per[0][0], H, W, cfg.horizontal_FOV, cfg.vertical_max, cfg.vertical_min) if hasattr(cfg, "horizontal_FOV") else None
if ri is None:
    Hh, Ww, hf, vmax, vmin = oracle.lidar_params(LIDAR)
    ri = oracle.project(per[0][0], Hh, Ww, hf, vmax, vmin)
ng = oracle.nonground_points(oracle.range_to_xyz(ri, cfg.transform_map()), per[0][1])
FB = 8
p_fps = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(ng, (FB,) + ng.shape))).to(dev)
ours = device.fps_batch(p_fps, 100)
ms_ours = timed(lambda: device.fps_batch(p_fps, 100), 5)
fps_ref = {"available": ref.have_cuda()}
if ref.have_cuda():
    temp = torch.full((FB, HW), 1e10, dtype=torch.float32, device=dev)
    idx = torch.zeros((FB, 100), dtype=torch.int32, device=dev)
    lib = ref.fps()

    def run_ref():
        temp.fill_(1e10)
        assert lib.ref_fps_launch(FB, HW, 100, p_fps.data_ptr(), temp.data_ptr(), idx.data_ptr()) == 0
    ms_ref = timed(run_ref, 3)
    fps_ref.update({"ms_per_launch": ms_ref, "frames_per_s": FB / ms_ref * 1e3, "identical_seeds": bool(torch.equal(idx, ours))})
out["a5_fps_dropin"] = {"batch": FB, "n": HW, "m": 100, "ms_per_launch": ms_ours, "frames_per_s": FB / ms_ours * 1e3,
                        "reference_kernel_same_gpu": fps_ref,
                        "note": "generic (B,n,3) entry point with the caller's temp buffer; the pipeline uses the fused pruned kernel"}

# ---------------------------------------------------------------------------------- a12 chamfer vs the reference kernel
a = np.ascontiguousarray(oracle.range_to_xyz(ri, cfg.transform_map()).reshape(-1, 3))
a = a[a.sum(-1) != 0]
bpts = xyz[0].reshape(-1, 3).cpu().numpy()
bpts = np.ascontiguousarray(bpts[bpts.sum(-1) != 0])
ta, tb = torch.from_numpy(a).to(dev), torch.from_numpy(bpts).to(dev)
n, m = ta.shape[0], tb.shape[0]
d1, d2 = torch.empty(n, device=dev), torch.empty(m, device=dev)
i1, i2 = torch.empty(n, dtype=torch.int32, device=dev), torch.empty(m, dtype=torch.int32, device=dev)
scratch = torch.empty(n + m, dtype=torch.int64, device=dev)


def run_ch():
    check(_lib.lib().rpcc_chamfer_batch(ptr(ta), n, ptr(tb), m, ptr(d1), ptr(i1), ptr(d2), ptr(i2), ptr(scratch), st))


ms_ch = timed(run_ch, 5)
ch_ref = {"available": ref.have_cuda()}
if ref.have_cuda():
    rd1, rd2 = torch.empty(n, device=dev), torch.empty(m, device=dev)
    ri1, ri2 = torch.empty(n, dtype=torch.int32, device=dev), torch.empty(m, dtype=torch.int32, device=dev)
    libc = ref.chamfer()

    def run_chref():
        assert libc.ref_chamfer_launch(1, n, ta.data_ptr(), m, tb.data_ptr(), rd1.data_ptr(), ri1.data_ptr(), rd2.data_ptr(),
                                       ri2.data_ptr()) == 0
    ms_chref = timed(run_chref, 2)
    ch_ref.update({"ms_per_pair": ms_chref, "identical": bool(torch.equal(rd1, d1) and torch.equal(rd2, d2) and
                                                               torch.equal(ri1, i1) and torch.equal(ri2, i2))})
pairs = 2.0 * n * m
out["a12_chamfer"] = {"n": n, "m": m, "ms_per_pair": ms_ch, "pair_evaluations_per_s": pairs / ms_ch * 1e3,
                      "fp32_flops_per_s": pairs * 8 / ms_ch * 1e3, "reference_kernel_same_gpu": ch_ref,
                      "mean_sqrt_dist": [float(d1.sqrt().mean()), float(d2.sqrt().mean())]}
print(json.dumps(out))
