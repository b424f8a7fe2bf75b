"""DBSCAN encode chain on one GPU: frames/s with device-resident points, whole-image scans, clusters per frame, and the
bits per point of DBSCAN against FPS on the same frames.

    python scripts/dbscan_rate.py [--frames 1184] [--distinct 64] [--eps 1.5] [--min-points 10] [--out FILE]

`--distinct` synthetic 64E frames are tiled to `--frames` slots (each its own copy on the device), all in one launch of
the chain (project -> ground fit -> DBSCAN -> label statistics -> point models -> quantise + pack).  Times are CUDA
events around encode_device calls after a warm-up call; the ground plane is fitted on the device, as in bench.py's
`value`.  Bits per point are taken on the `--distinct` frames through encode + bzip2, against the default FPS chain.
Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

LIDAR = "Velodyne64E"


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=10).stdout.strip()
    except Exception:
        out = ""
    return out or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1184)
    ap.add_argument("--distinct", type=int, default=64)
    ap.add_argument("--eps", type=float, default=1.5)
    ap.add_argument("--min-points", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dbscan_rate.py needs a CUDA device")
    from rpcc_b200 import synthetic
    from rpcc_b200.batch import BatchEncoder
    from rpcc_b200.config import load_compressor_cfg
    torch.cuda.set_device(0)
    per = [synthetic.frame(i, LIDAR) for i in range(a.distinct)]
    rows = [per[i % a.distinct][0] for i in range(a.frames)]
    off = np.concatenate([[0], np.cumsum([p.shape[0] for p in rows])]).astype(np.int64)
    pts_d = torch.from_numpy(np.concatenate(rows)).cuda()
    off_d = torch.from_numpy(off).cuda()
    B = a.frames
    cfg = load_compressor_cfg()
    cfg.update(segment_method="DBSCAN", DBSCAN_eps=a.eps, DBSCAN_min_points=a.min_points)
    res = {"gpu": gpu_info(), "lidar": LIDAR, "frames_per_launch": B, "distinct_frames": a.distinct, "eps": a.eps,
           "min_points": a.min_points, "cluster_num": int(cfg["cluster_num"])}
    with BatchEncoder(LIDAR, compressor_cfg=cfg, max_batch=B, max_points=int(off[-1])) as enc:
        enc.encode_device(0, pts_d, off_d, B)              # warm-up
        enc.sync()
        ws = enc.device_buffer(0, "dbscan_workspace", (2 * B,), torch.int32).cpu().numpy()
        exh, clusters = ws[:B], ws[B:]
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        st = torch.cuda.ExternalStream(enc.stream(0))
        times = []
        for _ in range(a.reps):
            s.record(st)
            enc.encode_device(0, pts_d, off_d, B)
            e.record(st)
            e.synchronize()
            times.append(s.elapsed_time(e))
        enc.profile(True)
        enc.encode_device(0, pts_d, off_d, B)
        stages, _, _ = enc.stage_times()
        ms = float(np.median(times))
        res.update(ms_per_launch=ms, launch_ms_all=times, frames_per_s=B / (ms / 1e3), stage_ms=stages,
                   exhaustive_points_per_frame=float(exh.mean()), exhaustive_points_total=int(exh.sum()),
                   clusters_per_frame_mean=float(clusters.mean()), clusters_per_frame_min=int(clusters.min()),
                   clusters_per_frame_max=int(clusters.max()))
    pts_h = np.concatenate([p for p, _ in per])
    off_h = np.concatenate([[0], np.cumsum([p.shape[0] for p, _ in per])]).astype(np.int64)
    bits = {}
    for name, c in (("DBSCAN", cfg), ("FPS", load_compressor_cfg())):
        with BatchEncoder(LIDAR, compressor_cfg=c, max_batch=a.distinct, max_points=int(off_h[-1])) as enc:
            blobs = enc.compress(pts_h, off_h)
            npts = enc.encode_host(pts_h, off_h)["results"]["sym_count"].astype(np.int64).sum()
        bits[name] = 8.0 * sum(len(b) for b in blobs) / float(npts)
    res.update(bpp_dbscan=bits["DBSCAN"], bpp_fps=bits["FPS"])
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
