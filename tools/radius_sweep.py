#!/usr/bin/env python
"""Radius matching (orbx_match_hamming_device_radius / _device_pairwise_radius), device-resident and CUDA-event timed on the
context's stream after a warm-up, at radii 30, 64 and 128.  Shapes:
  vo_1500x500           one VO call: 1500 map candidates against one 500-row frame
  bench_2048x1000x256   the bench's batch: 2048 map rows against 256 sets of 1000 rows
  frame_to_frame        255 pairs of extracted 640x480 / 1000-feature frames (pairwise calls)
Each call is made once with cap = 0 (offsets only) to size the output, then timed with the full buffer.  A separate
torch.profiler run of a few calls splits the device time into the count pass (k_hamming_umma<RadiusCount, ...>), the
offsets scan, the emit pass (<RadiusEmit, ...>) and the ordering (k_radius_order).  cv2's BFMatcher.radiusMatch on the host is timed for the VO
call.  The VO call's output is compared with cv2's lists (`vo_mismatched_lists` must be 0).  Prints the card, its power
limit and SM clock with the numbers and writes them as JSON.

  python tools/radius_sweep.py [--out profiles/radius_sweep_b200.json]
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
from knn_sweep import time_call  # noqa: E402
from pairwise_sweep import extract  # noqa: E402
from rgbd_visualodometry_b200 import orb  # noqa: E402
from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries, synth_sequence  # noqa: E402

RADII = (30, 64, 128)
PARTS = (("count", "MatchOp)4"), ("emit", "MatchOp)5"),   # k_hamming_umma<MatchOp::RadiusCount / RadiusEmit, ...>
          ("scan", "k_radius_scan"), ("scan", "k_radius_tile_sums"), ("order", "k_radius_order"))


def breakdown(fn, calls=3):
    """Device time per call (us) of each part, from torch.profiler over `calls` calls."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {"count": 0.0, "scan": 0.0, "emit": 0.0, "order": 0.0, "other": 0.0}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        part = next((p for p, key in PARTS if key in e.key), "other")
        out[part] += t / calls
    return out


def measure(ctx, st, name, call, nlists, radii=RADII):
    rows = []
    for r in radii:
        off = torch.zeros(nlists + 1, dtype=torch.int64, device="cuda")
        dummy = torch.zeros((1, 4), dtype=torch.int32, device="cuda")
        call(r, dummy, 0, off); ctx.synchronize()
        total = int(off[-1])
        out = torch.zeros((max(total, 1), 4), dtype=torch.int32, device="cuda")
        fn = lambda: call(r, out, total, off)               # noqa: E731
        row = {"shape": name, "radius": r, "lists": nlists, "records": total, "time": time_call(fn, st), "parts_us": breakdown(fn)}
        rows.append(row); print(json.dumps(row), flush=True)
        del out
        torch.cuda.empty_cache()
    return rows


def shared(ctx, q, trains, counts):
    dq, dt = torch.from_numpy(np.ascontiguousarray(q)).cuda(), torch.from_numpy(np.ascontiguousarray(trains)).cuda()
    dc = torch.tensor(counts, dtype=torch.int32, device="cuda")
    nsets, stride = trains.shape[0], trains.shape[1]
    keep = (dq, dt, dc)

    def call(r, out, cap, off):
        _ = keep
        ctx.match_device_radius(dq.data_ptr(), len(q), dt.data_ptr(), stride, dc.data_ptr(), nsets, r, out.data_ptr(), cap, off.data_ptr())
    return call, nsets * len(q)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "radius_sweep.json"))
    args = ap.parse_args()
    info = card()
    print(info, flush=True)
    ctx = orb.Context(1, 1.2, 1, 64, 64, 1)
    st = torch.cuda.ExternalStream(ctx.stream)
    rows = []

    # 1. one VO call, checked against cv2, and cv2 on the host for it
    t = synth_descriptors(500, 1)
    q = synth_map_queries(t, 1500, 2)
    call, nl = shared(ctx, q, t[None], [500])
    rows += measure(ctx, st, "vo_1500x500", call, nl)
    bad = 0
    try:
        import cv2
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)
        for r in RADII:
            rec, off = ctx.radius_match(q, t, r)
            want = bf.radiusMatch(q, t, float(r))
            for i, w in enumerate(want):
                got = rec[off[i]:off[i + 1]]
                bad += [(m.trainIdx, m.distance) for m in w] != list(zip(got["trainIdx"].tolist(), got["distance"].tolist()))
            bf.radiusMatch(q, t, float(r))
            t0 = time.perf_counter(); reps = 5
            for _ in range(reps):
                bf.radiusMatch(q, t, float(r))
            row = {"shape": "vo_1500x500", "call": "cv2_host", "radius": r, "time": {"us": (time.perf_counter() - t0) * 1e6 / reps, "reps": reps},
                   "cv2": cv2.__version__, "threads": cv2.getNumThreads()}
            rows.append(row); print(json.dumps(row), flush=True)
    except ImportError:
        print("cv2 not importable: no host timing or check", flush=True)

    # 2. the bench's batch
    trains = np.stack([synth_descriptors(1000, 10 + s) for s in range(256)])
    q = synth_map_queries(trains[0], 2048, 9)
    call, nl = shared(ctx, q, trains, [1000] * 256)
    rows += measure(ctx, st, "bench_2048x1000x256", call, nl)
    del trains, q, call
    torch.cuda.empty_cache()

    # 3. frame-to-frame on extraction output, 256 frames -> 255 pairs
    cap = 2000
    frames = np.stack([f for f, _ in synth_sequence(480, 640, 256, 11)])
    ectx = orb.Context(1000, 1.2, 8, 640, 480, 256)
    d_d, d_n = extract(ectx, frames, 1000, cap)
    ectx.close()

    def pw(r, out, c, off):
        ctx.match_device_pairwise_radius(d_d.data_ptr(), cap, d_n.data_ptr(), d_d.data_ptr() + cap * 32, cap, d_n.data_ptr() + 4, 255, r,
                                         out.data_ptr(), c, off.data_ptr())
    rows += measure(ctx, st, "frame_to_frame", pw, 255 * cap)

    ctx.close()
    print("VO lists that differ from cv2:", bad)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"card": info, "vo_mismatched_lists": bad, "rows": rows}, f, indent=1)
    print("wrote", args.out)
    if bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
