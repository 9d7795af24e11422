#!/usr/bin/env python
"""Per-stage device times of the extraction (+ match) on B synthetic VGA frames, without the rest of bench.py.
  python tools/stage_times.py [B] [reps]        (ORBX_LIB=<path> times another build of the library)"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from rgbd_visualodometry_b200 import orb  # noqa: E402
from rgbd_visualodometry_b200.synth import synth_descriptors  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
frames = bench.make_frames(B, 0)
ctx = orb.Context(bench.NFEAT, bench.SCALE, bench.NLEVELS, bench.W, bench.H, B)
d_in = torch.from_numpy(frames).cuda()
d_k = torch.zeros((B, bench.CAP, 7), dtype=torch.float32, device="cuda")
d_d = torch.zeros((B, bench.CAP, 32), dtype=torch.uint8, device="cuda")
d_n = torch.zeros(B, dtype=torch.int32, device="cuda")
d_map = torch.from_numpy(synth_descriptors(bench.MAP_M, 3)).cuda()
d_best = torch.zeros((B, bench.MAP_M, 4), dtype=torch.int32, device="cuda")
torch.cuda.synchronize()


def step():
    ctx.detect_and_compute_device(d_in.data_ptr(), B, bench.W, bench.H, bench.W * 3, bench.H * bench.W * 3, 3, d_k.data_ptr(), d_d.data_ptr(), bench.CAP, d_n.data_ptr())
    ctx.match_device_ragged(d_map.data_ptr(), bench.MAP_M, d_d.data_ptr(), bench.CAP, d_n.data_ptr(), B, d_best.data_ptr())


for _ in range(5):
    step()
ctx.synchronize()
ctx.set_profiling(True)
acc = {}
for _ in range(reps):
    step()
    for k, v in ctx.stage_times().items():
        acc.setdefault(k, []).append(v)
ctx.set_profiling(False)
ctx.synchronize()
print(" ".join(f"{k}={np.median(v):.4f}" for k, v in acc.items()), "sum=%.4f" % sum(np.median(v) for v in acc.values()),
      "kp=%.1f" % d_n.float().mean().item(), "env=" + ",".join(f"{k}={v}" for k, v in os.environ.items() if k.startswith("ORBX_")))
