"""The intensity section on one GPU: kernel times of the owner pass, the gather, the pack and the unpack, the encode
chain's frames/s with intensity off and on, and the section's size on the golden KITTI frame.

    python scripts/intensity_rate.py [--frames 1184] [--distinct 64] [--reps 5] [--out FILE]

`--distinct` synthetic 64E frames are tiled to `--frames` slots (each its own copy on the device), all in one launch.
Kernel times come from torch.profiler (CUDA activities) over `--reps` launches of each stage after a warm-up, summed per
kernel name and divided by the launches; the projection kernel is listed for scale.  The chain's rate is CUDA events
around encode_device calls (device-resident points, ground plane fitted on the device, as bench.py's `value`),
alternating intensity off and on.  The section's size is taken on tests/golden/example.bin: the synthetic frames'
intensities are uniform noise and say nothing about compression.  Prints one JSON object (and writes it to --out)."""
import argparse
import bz2
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

LIDAR = "Velodyne64E"
KERNELS = ("project_kernel", "intensity_owner_kernel", "intensity_gather_kernel", "intensity_pack_kernel",
           "intensity_unpack_kernel")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=10).stdout.strip()
    except Exception:
        out = ""
    return out or torch.cuda.get_device_name(0)


def kernel_ms(fn, reps):
    """ms per call of every kernel in KERNELS, from one profiled run of `reps` calls of fn."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                out[k] = out.get(k, 0.0) + ev.device_time_total / 1e3 / reps
    return out


def chain_ms(enc, pts, off, B):
    st = torch.cuda.ExternalStream(enc.stream(0))
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(st)
    enc.encode_device(0, pts, off, B)
    e.record(st)
    e.synchronize()
    return s.elapsed_time(e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1184)
    ap.add_argument("--distinct", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("intensity_rate.py needs a CUDA device")
    from rpcc_b200 import device, synthetic
    from rpcc_b200.batch import BatchEncoder
    from rpcc_b200.lidar import LidarConfig
    torch.cuda.set_device(0)
    lidar = LidarConfig(LIDAR)
    per = [synthetic.frame(i, LIDAR)[0] for i in range(a.distinct)]
    rows = [per[i % a.distinct] for i in range(a.frames)]
    off = np.concatenate([[0], np.cumsum([p.shape[0] for p in rows])]).astype(np.int64)
    pts_d = torch.from_numpy(np.concatenate(rows)).cuda()
    off_d = torch.from_numpy(off).cuda()
    B = a.frames
    res = {"gpu": gpu_info(), "lidar": LIDAR, "frames_per_launch": B, "distinct_frames": a.distinct,
           "points_per_launch": int(off[-1])}

    rng, own, inten = device.intensity_owner_batch(pts_d, off_d, lidar)
    step = 0.02
    q, base, _ = device.intensity_pack_batch(inten, rng, step)
    labels = (rng == 0).to(torch.uint8)              # 1 = empty, as the decoder's labels
    ms = {}
    ms.update(kernel_ms(lambda: device.intensity_owner_batch(pts_d, off_d, lidar), a.reps))
    ms.update({k: v for k, v in kernel_ms(lambda: device.intensity_pack_batch(inten, rng, step), a.reps).items()
               if k == "intensity_pack_kernel"})
    ms.update({k: v for k, v in kernel_ms(lambda: device.intensity_unpack_batch(labels, q, base, step), a.reps).items()
               if k == "intensity_unpack_kernel"})
    res["kernel_ms_per_launch"] = ms

    encs = {name: BatchEncoder(LIDAR, max_batch=B, max_points=int(off[-1]), intensity_accuracy=acc)
            for name, acc in (("off", None), ("on", 0.01))}
    times = {"off": [], "on": []}
    for name in encs:
        chain_ms(encs[name], pts_d, off_d, B)        # warm-up
    for _ in range(a.reps):
        for name in ("off", "on"):
            times[name].append(chain_ms(encs[name], pts_d, off_d, B))
    for name, enc in encs.items():
        m = float(np.median(times[name]))
        res["chain_%s" % name] = {"ms_per_launch": m, "all_ms": times[name], "frames_per_s": B / (m / 1e3)}
        enc.close()

    ex = np.fromfile(os.path.join(ROOT, "tests", "golden", "example.bin"), np.float32).reshape(-1, 4)
    rate = {}
    for acc in (0.005, 0.01, 0.025):
        with BatchEncoder(LIDAR, max_batch=1, intensity_accuracy=acc) as enc:
            out = enc.encode_host(ex, np.asarray([0, ex.shape[0]], np.int64))
            geom = len(enc.compress(ex, np.asarray([0, ex.shape[0]], np.int64))[0])
        n = int(out["results"]["sym_count"][0])
        sec = len(bz2.compress(out["intensity"].tobytes())) + 4
        rate[str(acc)] = {"section_bytes": sec, "bits_per_point": 8.0 * sec / n, "points": n, "file_bytes": geom}
    res["example_bin"] = rate
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
