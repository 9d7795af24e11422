#!/usr/bin/env python
"""k-nearest-neighbour matching (orbx_match_hamming_device_knn / _device_pairwise_knn, the top-k kernels) against the knn2
kernels (orbx_match_hamming_device_ragged / _device_pairwise with d_second), device-resident and CUDA-event timed on the
context's stream after a warm-up.  Per shape: the knn2 call, then the top-k call at k = 2, 3, 4, 8, 16 and 32.  Shapes:
  vo_1500x500           one VO call: 1500 map candidates against one 500-row frame
  bench_2048x1000x256   the bench's batch: 2048 map rows against 256 sets of 1000 rows
  map_100kx2000x32      100 000 map rows against 32 sets of 2000 rows
  frame_to_frame        255 pairs of extracted 640x480 / 1000-feature frames (pairwise calls)
  insert_heavy_k32      2048 identical query rows against 256 sets of 1000 rows in decreasing distance (every column
                        enters the list), top-k at k = 32 only
and cv2's BFMatcher.knnMatch on the host for the VO call.  Every top-k output's first two records per query are compared
with the knn2 output of the same run (the k-NN lists are prefixes of one another); `prefix_mismatches` must be 0.  Prints
the card, its power limit and SM clock with the numbers and writes them as JSON.

  python tools/knn_sweep.py [--out profiles/knn_sweep_b200.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from crosscheck_sweep import card  # noqa: E402
from pairwise_sweep import extract  # noqa: E402
from rgbd_visualodometry_b200 import orb  # noqa: E402
from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries, synth_sequence  # noqa: E402

KS = (2, 3, 4, 8, 16, 32)


def time_call(fn, st, window_s=0.25, windows=3):
    """us per call: median (min, max) over `windows` windows of about window_s seconds (at least 2 calls each)."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st); fn(); e1.record(st); e1.synchronize()
    first = e0.elapsed_time(e1)
    reps = max(2, int(window_s * 1e3 / max(first, 1e-3)))
    windows = windows if first < 100 else 1                 # (second-long calls: one window of two calls)
    us = []
    for _ in range(windows):
        e0.record(st)
        for _ in range(reps):
            fn()
        e1.record(st)
        e1.synchronize()
        us.append(e0.elapsed_time(e1) * 1e3 / reps)
    return {"us": float(np.median(us)), "min": float(min(us)), "max": float(max(us)), "reps": reps, "windows": windows}


class Shape:
    """Device-resident operands of one workload: shared-query ragged sets, or pairwise sets when dqc is given."""

    def __init__(self, name, dq, nq, dt, stride, dtc, nsets, dqc=None, keep=()):
        self.name, self.dq, self.nq, self.dt, self.stride, self.dtc, self.nsets, self.dqc = name, dq, nq, dt, stride, dtc, nsets, dqc
        self.keep = keep

    def knn2(self, ctx, best, second):
        if self.dqc is None:
            return lambda: ctx.match_device_ragged(self.dq, self.nq, self.dt, self.stride, self.dtc, self.nsets, best.data_ptr(), second.data_ptr())
        return lambda: ctx.match_device_pairwise(self.dq, self.nq, self.dqc, self.dt, self.stride, self.dtc, self.nsets, best.data_ptr(),
                                                 second.data_ptr())

    def topk(self, ctx, k, out):
        if self.dqc is None:
            return lambda: ctx.match_device_knn(self.dq, self.nq, self.dt, self.stride, self.dtc, self.nsets, k, out.data_ptr())
        return lambda: ctx.match_device_pairwise_knn(self.dq, self.nq, self.dqc, self.dt, self.stride, self.dtc, self.nsets, k, out.data_ptr())


def measure(ctx, st, s, ks=KS):
    best = torch.zeros((s.nsets, s.nq, 4), dtype=torch.int32, device="cuda")
    second = torch.zeros_like(best)
    k2 = s.knn2(ctx, best, second)
    k2(); ctx.synchronize()
    ref = torch.stack([best, second], 2)                    # [nsets, nq, 2, 4]
    qn = None
    if s.dqc is not None:                                   # pairwise: only records below each pair's query count are written
        qn = torch.arange(s.nq, device="cuda")[None, :] < torch.clamp(s.keep[-1][: s.nsets], 0, s.nq)[:, None]
    rows = []
    row = {"shape": s.name, "call": "knn2_kernel", "nq": s.nq, "stride": s.stride, "nsets": s.nsets, "time": time_call(k2, st)}
    rows.append(row); print(json.dumps(row), flush=True)
    for k in ks:
        out = torch.zeros((s.nsets, s.nq, k, 4), dtype=torch.int32, device="cuda")
        fn = s.topk(ctx, k, out)
        fn(); ctx.synchronize()
        n = min(k, 2)
        diff = (out[:, :, :n] != ref[:, :, :n]).any(-1).any(-1)
        if qn is not None:
            diff &= qn
        row = {"shape": s.name, "call": f"topk_k{k}", "k": k, "nq": s.nq, "stride": s.stride, "nsets": s.nsets, "time": time_call(fn, st),
               "prefix_mismatches": int(diff.sum())}
        row["over_knn2"] = row["time"]["us"] / rows[0]["time"]["us"]
        rows.append(row); print(json.dumps(row), flush=True)
        del out
    return rows


def shared(name, q, trains, counts):
    dq, dt = torch.from_numpy(np.ascontiguousarray(q)).cuda(), torch.from_numpy(np.ascontiguousarray(trains)).cuda()
    dc = torch.tensor(counts, dtype=torch.int32, device="cuda")
    return Shape(name, dq.data_ptr(), len(q), dt.data_ptr(), trains.shape[1], dc.data_ptr(), trains.shape[0], keep=(dq, dt, dc))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "knn_sweep.json"))
    args = ap.parse_args()
    info = card()
    print(info, flush=True)
    ctx = orb.Context(1, 1.2, 1, 64, 64, 1)
    st = torch.cuda.ExternalStream(ctx.stream)
    rows = []

    # 1. one VO call, and cv2 on the host for it
    t = synth_descriptors(500, 1)
    q = synth_map_queries(t, 1500, 2)
    rows += measure(ctx, st, shared("vo_1500x500", q, t[None], [500]))
    try:
        import cv2
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)
        for k in KS:
            bf.knnMatch(q, t, k=k)
            t0 = time.perf_counter(); reps = 5
            for _ in range(reps):
                bf.knnMatch(q, t, k=k)
            row = {"shape": "vo_1500x500", "call": f"cv2_host_k{k}", "k": k, "time": {"us": (time.perf_counter() - t0) * 1e6 / reps, "reps": reps},
                   "cv2": cv2.__version__, "threads": cv2.getNumThreads()}
            rows.append(row); print(json.dumps(row), flush=True)
    except ImportError:
        print("cv2 not importable: no host timing", flush=True)

    # 2. the bench's batch
    trains = np.stack([synth_descriptors(1000, 10 + s) for s in range(256)])
    q = synth_map_queries(trains[0], 2048, 9)
    rows += measure(ctx, st, shared("bench_2048x1000x256", q, trains, [1000] * 256))

    # 3. a large map against a few frames
    trains = np.stack([synth_descriptors(2000, 400 + s) for s in range(32)])
    q = synth_map_queries(trains[0], 100000, 8)
    rows += measure(ctx, st, shared("map_100kx2000x32", q, trains, [2000] * 32))
    del trains, q
    torch.cuda.empty_cache()

    # 4. frame-to-frame on extraction output, 256 frames -> 255 pairs
    cap = 2000
    frames = np.stack([f for f, _ in synth_sequence(480, 640, 256, 11)])
    ectx = orb.Context(1000, 1.2, 8, 640, 480, 256)
    d_d, d_n = extract(ectx, frames, 1000, cap)
    ectx.close()
    rows += measure(ctx, st, Shape("frame_to_frame", d_d.data_ptr(), cap, d_d.data_ptr() + cap * 32, cap, d_n.data_ptr() + 4, 255,
                                   dqc=d_n.data_ptr(), keep=(d_d, d_n)))

    # 5. insert-heavy, k = 32
    bits = np.zeros((1000, 256), np.uint8)
    for j in range(1000):
        bits[j, :256 - (j * 256) // 1000] = 1
    t = np.packbits(bits, axis=1)
    rows += measure(ctx, st, shared("insert_heavy_k32", np.zeros((2048, 32), np.uint8), np.stack([t] * 256), [1000] * 256), ks=(32,))

    ctx.close()
    bad = sum(r.get("prefix_mismatches", 0) for r in rows)
    print("total prefix mismatches:", bad)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"card": info, "total_prefix_mismatches": bad, "rows": rows}, f, indent=1)
    print("wrote", args.out)
    if bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
