#!/usr/bin/env python
"""Per-stage CUDA-event times of the encoder chain (296 frames per launch, one stream slot), quickly:
   [RPCC_B200_LIB=...] python scripts/stage_times.py [frames] [reps] [uniform|nonuniform] [point|plane] [off|eval|p2plane]
The last argument turns on the encoder's eval stage: "eval" = decode + chamfer figures, "p2plane" = also the normals
of both clouds and the point-to-plane table."""
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from rpcc_b200 import synthetic  # noqa: E402
from rpcc_b200.batch import BatchEncoder  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 296
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
nonuniform = len(sys.argv) > 3 and sys.argv[3] == "nonuniform"
method = sys.argv[4] if len(sys.argv) > 4 else "point"
ev = sys.argv[5] if len(sys.argv) > 5 else "off"
per = [synthetic.frame(i) for i in range(min(B, 32))]
pts = np.concatenate([per[i % len(per)][0] for i in range(B)], 0)
off = np.cumsum([0] + [per[i % len(per)][0].shape[0] for i in range(B)]).astype(np.int64)
enc = BatchEncoder("Velodyne64E", accuracy=0.02, nonuniform=nonuniform, max_batch=B, max_points=pts.shape[0], model_method=method,
                   eval=ev != "off", p2plane=ev == "p2plane")
d_pts, d_off = torch.from_numpy(pts).cuda(), torch.from_numpy(off).cuda()
for r in range(3):
    enc.encode_device(0, d_pts, d_off, B, None)
enc.sync()
enc.profile(True)
for r in range(reps):
    enc.encode_device(0, d_pts, d_off, B, None)
ms, frames, calls = enc.stage_times()
print(" ".join("%s=%.4f" % (k, v / calls) for k, v in ms.items()), "total=%.4f ms/launch" % (sum(ms.values()) / calls))
