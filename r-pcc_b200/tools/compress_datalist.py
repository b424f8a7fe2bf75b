"""python -m rpcc_b200.tools.compress_datalist --datalist L.txt --output_dir OUT --lidar Velodyne64E
   torchrun --nproc-per-node 8 -m rpcc_b200.tools.compress_datalist ...          (one rank per GPU)

The reference's tools/compress_datalist.py:48-206 re-plumbed.  There, a ThreadPoolExecutor maps a per-frame closure
(load -> segment -> model -> predict -> quantise -> entropy-code -> save) that holds the GIL in every native call.
Here the datalist is sharded contiguously across ranks (no collective on the hot path) and each rank runs a three-stage
pipeline over batches of `--batch` frames, every stage on its own threads:

  readers   KITTI .bin -> xyz rows, straight into a pinned staging buffer (csrc/hostio.cu; 12 bytes per point cross
            PCIe, the intensity column never does -- dataset/dataset.py:62 drops it as well); with
            --intensity_accuracy whole 16-byte rows, and the intensity section is written after the five others
  GPU       BatchEncoder.encode_host: project -> ground fit -> FPS -> labels (or DBSCAN, --segment_method DBSCAN) ->
            models -> quantise + pack, and with
            --eval the decode + depth-error / chamfer / F-score stage (--p2plane, which implies --eval, adds the k-NN
            normals and point-to-plane PSNR); sections land in one of two pinned output sets
  packer    native bzip2 pool + file writes out of that pinned set while the GPU fills the other one

A frame's `.rpcc` bytes depend on its points alone: not on --batch, on its place in the datalist, on the number of
ranks, nor on which tool wrote it (tools/compress.py gives the same file; tests/test_gpu_datalist.py).
Output paths follow the reference: output_dir + input path with the extension text replaced by 'rpcc'
(compress_datalist.py:136-141, including its replace-everywhere quirk).  NCCL is used once, to gather the per-frame
metrics table."""
import concurrent.futures as futures
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from ..batch import BatchEncoder, eval_summary
from ..compress_utils import BasicCompressor, pack_bitstream
from ..hostio import read_bin_rows, read_bin_xyz
from ..shard import bind_to_gpu_numa, gather_metrics, shard_range
from .common import base_parser, intensity_accuracy, resolve, warn_clamped

# columns of the per-frame metrics table that the ranks all-gather
M_BYTES, M_POINTS, M_SECONDS, M_DEPTH_MAX, M_DEPTH_MEAN, M_CD_MEAN, M_FSCORE, M_PSNR, M_CD1, M_CD2, M_PSNR_P2PLANE = range(11)
METRIC_COLS = 11   # M_PSNR_P2PLANE is filled with --p2plane only


def output_path_for(output_dir, file_name):
    file_name = file_name.strip()
    if file_name[0] == "/":
        file_name = file_name[1:]
    output_path = os.path.join(output_dir, file_name)
    return output_path.replace(output_path.split(".")[-1], "rpcc")


def load_points(path, cols=3):
    """dataset/dataset.py:57-68 for the formats that are not KITTI .bin -> (N,3) f32; cols=4 keeps the intensity
    column, which the file must then have."""
    ext = path.split(".")[-1]
    if ext == "bin":
        return np.ascontiguousarray(np.fromfile(path, dtype=np.float32).reshape(-1, 4)[:, :cols])
    if ext in ("npy", "npz"):
        a = np.load(path)
    elif ext == "txt":
        a = np.loadtxt(path)
    else:
        raise ValueError("File type not correct: " + path)
    if a.ndim != 2 or a.shape[1] < cols:
        raise ValueError("%s has no intensity column (--intensity_accuracy needs x, y, z, intensity rows)" % path)
    return np.ascontiguousarray(a[:, :cols], dtype=np.float32)


def _rows_of(path):
    """Points in a file without reading it (.bin: 16 bytes per row); None when the file has to be parsed."""
    return os.path.getsize(path) // 16 if path.split(".")[-1] == "bin" else None


class _Batches:
    """Cuts a rank's files into batches and fills pinned staging buffers with their xyz rows on reader threads."""

    def __init__(self, enc, files, batch, readers, cols=3):
        self.enc, self.files, self.B, self.cols = enc, files, batch, cols
        self.pool = futures.ThreadPoolExecutor(max(1, readers))
        self.rows = [_rows_of(f) for f in files]
        self.parsed = {}
        for i, r in enumerate(self.rows):          # the rare non-.bin inputs are parsed up front (sizes unknown until then)
            if r is None:
                self.parsed[i] = load_points(files[i], cols)
                self.rows[i] = self.parsed[i].shape[0]
        self.n = (len(files) + batch - 1) // batch
        self.max_rows = max([sum(self.rows[k * batch:(k + 1) * batch]) for k in range(self.n)] or [1])

    def start(self, k):
        """Begin reading batch k into staging buffer k % 2 -> (offsets, futures)."""
        lo, hi = k * self.B, min(len(self.files), (k + 1) * self.B)
        off = np.zeros(hi - lo + 1, np.int64)
        np.cumsum(self.rows[lo:hi], out=off[1:])
        buf = self.enc.input_buffer(self.max_rows, k % 2).numpy()

        read = read_bin_rows if self.cols == 4 else read_bin_xyz

        def one(i):
            dst = buf[off[i - lo]:off[i - lo + 1]]
            if i in self.parsed:
                dst[...] = self.parsed.pop(i)
            elif read(self.files[i], dst) != dst.shape[0]:
                raise IOError("%s changed size while the datalist was being processed" % self.files[i])

        return off, [self.pool.submit(one, i) for i in range(lo, hi)]

    def close(self):
        self.pool.shutdown()


def compress(args, rank=None, world=None, collective=True):
    """rank / world default to the torchrun environment.  collective=False runs one rank's shard without a process
    group (tests: the union of the shards must equal the single-rank output); the returned table then holds this
    rank's rows only."""
    cfg, accuracy, segment_cfg, model_cfg, uniform, method = resolve(args)
    inten = intensity_accuracy(args, cfg)
    p2plane = bool(getattr(args, "p2plane", False))
    do_eval = bool(args.eval) or p2plane
    if model_cfg["model_method"] not in ("point", "plane"):
        raise NotImplementedError("the batched driver covers point and plane modelling")
    world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else int(world)
    rank = int(os.environ.get("RANK", "0")) if rank is None else int(rank)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:       # a rank of a torchrun job: stay next to its GPU
        bind_to_gpu_numa(local)
    if collective and world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    files = [l.strip() for l in open(args.datalist) if l.strip()]
    lo, hi = shard_range(len(files), rank, world)
    mine = files[lo:hi]
    cfg = dict(cfg)
    cfg["cluster_num"] = segment_cfg["cluster_num"]
    cfg["segment_method"] = segment_cfg["segment_method"]
    cfg["DBSCAN_eps"] = segment_cfg["DBSCAN_eps"]
    cfg["DBSCAN_min_points"] = segment_cfg["DBSCAN_min_points"]
    cfg["ground_threshold"] = segment_cfg["ground_vertical_threshold"]
    cfg["plane_angle_threshold"] = model_cfg["angle_threshold"]
    B = max(1, min(args.batch, max(len(mine), 1)))
    batches = _Batches(None, mine, B, readers=min(8, max(2, args.workers)), cols=4 if inten is not None else 3)
    enc = BatchEncoder(args.lidar, accuracy=accuracy / 2, nonuniform=not uniform, compressor_cfg=cfg, max_batch=B,
                       max_points=batches.max_rows, device=local, basic_compressor=method, workers=args.workers,
                       model_method=model_cfg["model_method"], eval=do_eval, p2plane=p2plane, intensity_accuracy=inten)
    batches.enc = enc
    HW = enc.lidar.HW
    metrics = np.zeros((len(mine), METRIC_COLS), np.float64)
    outs = [output_path_for(args.output_dir, f) for f in mine]
    for d in sorted({os.path.dirname(o) for o in outs}):
        os.makedirs(d, exist_ok=True)
    native = method == "bzip2"
    packer = enc.packer() if native else None
    pypool = None if native else futures.ThreadPoolExecutor(args.workers)
    bc = BasicCompressor(method_name=method)
    inflight = [None, None]        # per pinned output set: what is still being entropy-coded out of it

    def collect(slot):
        job = inflight[slot]
        if job is None:
            return
        inflight[slot] = None
        f0, n, handle = job
        if native:
            sizes, _ = packer.wait(handle)
            metrics[f0:f0 + n, M_BYTES] = sizes
        else:
            for j, fut in enumerate(handle):
                metrics[f0 + j, M_BYTES] = fut.result()

    def entropy_and_save(i, sections):
        blob = pack_bitstream({k: bc.compress(v, section=k) for k, v in sections.items()}, uniform=uniform)
        with open(outs[i], "wb") as f:
            f.write(blob)
        return len(blob)

    t0 = time.time()
    t_gpu = 0.0
    pending = batches.start(0) if batches.n else None
    for k in range(batches.n):
        off, futs = pending
        for fu in futs:
            fu.result()
        # the next batch is read into the other staging buffer while this one is on the GPU (encode_host has returned
        # from batch k-1, so that buffer is free)
        pending = batches.start(k + 1) if k + 1 < batches.n else None
        slot = k % 2
        collect(slot)              # the packer must be done with this output set before the GPU overwrites it
        f0, n = k * B, off.size - 1
        tg = time.time()
        out = enc.encode_host(enc.input_buffer(batches.max_rows, slot)[:off[-1]], off, None, out_set=slot)
        t_gpu += time.time() - tg
        res = out["results"]
        metrics[f0:f0 + n, M_POINTS] = res["sym_count"]
        if inten is not None:
            warn_clamped(res["flags"], mine[f0:f0 + n])
        if do_eval:
            for j in range(n):
                s = eval_summary(out["eval"][j], HW)
                metrics[f0 + j, M_DEPTH_MAX:M_CD2 + 1] = (s["depth_max"], s["depth_mean"], s["mean"], s["f_score"],
                                                          s["psnr_p2p"], s["cd1"], s["cd2"])
                if p2plane:
                    metrics[f0 + j, M_PSNR_P2PLANE] = s["psnr_p2plane"]
        if native:
            inflight[slot] = (f0, n, packer.submit(out, enc.K, uniform, outs[f0:f0 + n]))
        else:
            handle = [pypool.submit(entropy_and_save, f0 + j, BatchEncoder.frame_sections(out, j)) for j in range(n)]
            inflight[slot] = (f0, n, handle)
    collect(0)
    collect(1)
    batches.close()
    if pypool is not None:
        pypool.shutdown()
    dt = time.time() - t0
    metrics[:, M_SECONDS] = dt / max(len(mine), 1)
    enc.close()
    if not collective:
        return metrics
    table = gather_metrics(metrics, len(files), device=torch.device("cuda", local) if world > 1 else None)
    if rank == 0:
        report(args, files, table, world, dt, t_gpu, method, uniform, accuracy)
    if world > 1:
        dist.barrier()
    return table


def report(args, files, table, world, dt, t_gpu, method, uniform, accuracy):
    """What the reference prints per frame under --output / --eval (tools/compress_datalist.py:143-199), per frame and
    as a summary, plus the point-to-plane PSNR under --p2plane.  Times are amortised: frames are processed in batches,
    there is no per-frame stage time."""
    p2plane = bool(getattr(args, "p2plane", False))
    do_eval = bool(args.eval) or p2plane
    if args.output:
        for i, f in enumerate(files):
            bits, pts = table[i, M_BYTES] * 8, max(table[i, M_POINTS], 1)
            print("\nCompression finished.")
            print("binary bitstream save in ", output_path_for(args.output_dir, f))
            print("\nTime Cost:")
            print("    Total time cost (amortised over the batch): ", table[i, M_SECONDS])
            print("\nCompression Results: ")
            print("    Compression ratio: ", (pts * 32 * 3) / max(bits, 1))
            print("    BPP: ", bits / pts)
            print("\n")
            if do_eval:
                print("\nReconstruction quality: ")
                print("    Depth Error (mean): ", table[i, M_DEPTH_MEAN])
                print("    Depth Error (max): ", table[i, M_DEPTH_MAX])
                print("    Chamfer Distance (mean): ", table[i, M_CD_MEAN])
                print("    F1 score (threshold=0.02): ", table[i, M_FSCORE])
                print("    Point-to-Point PSNR (r=59.7): ", table[i, M_PSNR])
                if p2plane:
                    print("    Point-to-Plane PSNR (r=59.7): ", table[i, M_PSNR_P2PLANE])
    total_bytes, total_pts = table[:, M_BYTES].sum(), table[:, M_POINTS].sum()
    print("\nCompressed %d frames on %d GPU(s) in %.2f s (%.1f frames/s incl. file I/O and %s; rank 0 spent %.2f s in "
          "the GPU call)." % (len(files), world, dt, len(files) / dt if dt > 0 else 0.0, method, t_gpu))
    print("    mean BPP: ", 8.0 * total_bytes / max(total_pts, 1))
    print("    mean compression ratio: ", (total_pts * 96.0) / max(8.0 * total_bytes, 1))
    if do_eval and len(files):
        limit = accuracy + (0.0 if uniform else 0.06) + 0.00001      # compress_datalist.py:184-189
        worst = float(table[:, M_DEPTH_MAX].max())
        print("    Depth Error (max over frames): ", worst)
        print("    Chamfer Distance (mean over frames): ", float(table[:, M_CD_MEAN].mean()))
        print("    F1 score (mean over frames): ", float(table[:, M_FSCORE].mean()))
        if p2plane:
            print("    Point-to-Plane PSNR (mean over frames): ", float(table[:, M_PSNR_P2PLANE].mean()))
        if worst > limit:
            print("    WARNING: reconstruction error above the configured accuracy (%g > %g) -- a residual wrapped int16 "
                  "or a model row is not finite." % (worst, limit))


def parser():
    p = base_parser(single=False)
    p.add_argument("--p2plane", action="store_true",
                   help="also report point-to-plane PSNR (k-NN normals on the GPU; implies --eval).")
    return p


def main(argv=None):
    args = parser().parse_args(argv)
    return compress(args)


if __name__ == "__main__":
    main()
