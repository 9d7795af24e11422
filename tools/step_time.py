#!/usr/bin/env python
"""Device time of the whole extraction step (and of extraction + 2 matches) on B synthetic VGA frames with the library's
normal stream layout (stage timers off, so the side-stream overlaps are active) -- wall clock over many asynchronous steps.
  python tools/step_time.py [B] [reps]        (ORBX_LIB=<path> times another build of the library)"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from rgbd_visualodometry_b200 import orb  # noqa: E402
from rgbd_visualodometry_b200.synth import synth_descriptors  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 50
frames = bench.make_frames(B, 0)
ctx = orb.Context(bench.NFEAT, bench.SCALE, bench.NLEVELS, bench.W, bench.H, B)
d_in = torch.from_numpy(frames).cuda()
d_k = torch.zeros((B, bench.CAP, 7), dtype=torch.float32, device="cuda")
d_d = torch.zeros((B, bench.CAP, 32), dtype=torch.uint8, device="cuda")
d_n = torch.zeros(B, dtype=torch.int32, device="cuda")
d_map = torch.from_numpy(synth_descriptors(bench.MAP_M, 3)).cuda()
d_best = torch.zeros((B, bench.MAP_M, 4), dtype=torch.int32, device="cuda")
torch.cuda.synchronize()


def extract():
    ctx.detect_and_compute_device(d_in.data_ptr(), B, bench.W, bench.H, bench.W * 3, bench.H * bench.W * 3, 3, d_k.data_ptr(), d_d.data_ptr(), bench.CAP, d_n.data_ptr())


def match():
    ctx.match_device_ragged(d_map.data_ptr(), bench.MAP_M, d_d.data_ptr(), bench.CAP, d_n.data_ptr(), B, d_best.data_ptr())


def timed(fn):
    for _ in range(5):
        fn()
    ctx.synchronize()
    best = 1e9
    for _ in range(3):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        ctx.synchronize()
        best = min(best, (time.perf_counter() - t0) / reps * 1e3)
    return best


t_e = timed(extract)
t_em = timed(lambda: (extract(), match(), match()))
print(f"extract={t_e:.4f} ms  extract+2match={t_em:.4f} ms  ({B / t_em:.1f} k frames/s)  kp={d_n.float().mean().item():.1f}",
      "env=" + ",".join(f"{k}={v}" for k, v in os.environ.items() if k.startswith("ORBX_")))
