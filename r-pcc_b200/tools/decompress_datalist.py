"""python -m rpcc_b200.tools.decompress_datalist --datalist L.txt --output_dir OUT --lidar Velodyne64E
   torchrun --nproc-per-node 8 -m rpcc_b200.tools.decompress_datalist ...        (one rank per GPU)

Batched mirror of the reference's tools/decompress_datalist.py:48-134; datalist lines are .rpcc files, outputs are
.bin files under output_dir (the extension text replaced as the reference does, :129).  Per batch: the files are read
and entropy-decoded on host threads, BatchDecoder runs recover_map / dequantise / predict / range x LUT on the device and
compacts the rows of every output file there (save_point_cloud_to_file's `x + y + z != 0` filter and zero intensity,
dataset/dataset.py:72-81; with --intensity_accuracy the decoded intensities instead), and writer threads put the pinned rows on disk while the next batch is decoded into the other
buffer set.  Frames are sharded contiguously across ranks; there is no collective."""
import concurrent.futures as futures
import os
import time

import torch

from ..batch import BatchDecoder
from ..shard import bind_to_gpu_numa, shard_range
from .common import base_parser, intensity_accuracy, resolve


def output_path_for(output_dir, file_name):
    fn = file_name[1:] if file_name[0] == "/" else file_name
    path = os.path.join(output_dir, fn)
    return path.replace(path.split(".")[-1], "bin")


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def decompress(args, rank=None, world=None):
    cfg, accuracy, segment_cfg, model_cfg, uniform, method = resolve(args)
    world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else int(world)
    rank = int(os.environ.get("RANK", "0")) if rank is None else int(rank)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:       # a rank of a torchrun job: stay next to its GPU
        bind_to_gpu_numa(local)
    files = [l.strip() for l in open(args.datalist) if l.strip()]
    for f in files:
        assert f.split(".")[-1] == "rpcc", f           # decompress_datalist.py:96
    lo, hi = shard_range(len(files), rank, world)
    mine = files[lo:hi]
    outs = [output_path_for(args.output_dir, f) for f in mine]
    for d in sorted({os.path.dirname(o) for o in outs}):
        os.makedirs(d, exist_ok=True)
    dec = BatchDecoder(args.lidar, accuracy=accuracy / 2, nonuniform=not uniform, compressor_cfg=dict(cfg),
                       basic_compressor=method, workers=args.workers, device=local,
                       intensity_accuracy=intensity_accuracy(args, cfg))
    io = futures.ThreadPoolExecutor(max(2, min(16, args.workers)))
    B = max(1, args.batch)
    nb = (len(mine) + B - 1) // B
    t0 = time.time()
    writes = [[], []]                 # per buffer set: the writer futures that still read its pinned rows
    reads = [io.submit(_read, f) for f in mine[:B]]
    for k in range(nb):
        blobs = [r.result() for r in reads]
        reads = [io.submit(_read, f) for f in mine[(k + 1) * B:(k + 2) * B]]     # next batch's files, in the background
        s = k % 2
        for w in writes[s]:
            w.result()
        out = dec.decode(blobs, want_xyz=False, want_points=True, buf_set=s)
        writes[s] = [io.submit(out["points"][j].tofile, outs[k * B + j]) for j in range(len(blobs))]
    for s in (0, 1):
        for w in writes[s]:
            w.result()
    io.shutdown()
    dec.close()
    dt = time.time() - t0
    if rank == 0:
        print("Decompressed %d frames in %.2f s (%.1f frames/s on this rank incl. file I/O)" %
              (len(mine), dt, len(mine) / dt if dt > 0 else 0.0))
    return len(mine), dt


def main(argv=None):
    args = base_parser(single=False).parse_args(argv)
    return decompress(args)


if __name__ == "__main__":
    main()
