#!/usr/bin/env python
"""Cost of the cross-checked matcher (BFMatcher(NORM_HAMMING, crossCheck=True)) over the plain one, device-resident,
CUDA-event timed on the context's stream.  Per shape:
  plain     match_device (best match of every query)
  fused     match_device_crosscheck (the column maxima come out of the same distance tiles; compacted pairs)
  two-pass  single set only: match_device query -> train and train -> query, then the mutual check in torch (mask and count,
            no compaction); its pairs also cross-validate the fused result
The VO shape is also timed through the host-buffer API (host clock around the synchronous call, uploads included).
Prints the card, its power limit and SM clock with the numbers and writes them as JSON.

  python tools/crosscheck_sweep.py [--out profiles/crosscheck_sweep.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rgbd_visualodometry_b200 import orb  # noqa: E402
from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries  # noqa: E402

SHAPES = [("vo_call", 1500, 500, 1), ("bench_match", 2048, 1000, 256), ("baseline_c3", 100000, 2000, 32), ("large_single", 20000, 2000, 1)]


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.splitlines()[0]
    except (OSError, IndexError):
        line = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": line.strip()}


def time_fn(fn, st, window_s=0.3, repeats=3):
    """us per call: median (and min, max) over `repeats` windows of about window_s seconds each."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st); fn(); e1.record(st); e1.synchronize()
    reps = max(10, int(window_s * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    us = []
    for _ in range(repeats):
        e0.record(st)
        for _ in range(reps):
            fn()
        e1.record(st)
        e1.synchronize()
        us.append(e0.elapsed_time(e1) * 1e3 / reps)
    return {"us": float(np.median(us)), "min": float(min(us)), "max": float(max(us)), "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "crosscheck_sweep.json"))
    args = ap.parse_args()
    info = card()
    print(info)
    ctx = orb.Context(1, 1.2, 1, 64, 64, 1)
    st = torch.cuda.ExternalStream(ctx.stream)
    rows = []
    for name, nq, nt, nsets in SHAPES:
        trains = np.stack([synth_descriptors(nt, 40 + s) for s in range(nsets)])
        q = synth_map_queries(trains[0], nq, 41)
        dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(trains).cuda()
        dn = torch.full((nsets,), nt, dtype=torch.int32, device="cuda")
        best = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
        xc = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
        nxc = torch.zeros(nsets, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        plain = lambda: ctx.match_device(dq.data_ptr(), nq, dt.data_ptr(), nt, nsets, best.data_ptr())   # noqa: E731
        fused = lambda: ctx.match_device_crosscheck(dq.data_ptr(), nq, dt.data_ptr(), nt, dn.data_ptr(), nsets, xc.data_ptr(), nxc.data_ptr())  # noqa: E731
        row = {"shape": name, "nq": nq, "nt": nt, "nsets": nsets, "plain": time_fn(plain, st), "fused": time_fn(fused, st)}
        row["fused_over_plain"] = row["fused"]["us"] / row["plain"]["us"]
        ctx.synchronize()
        n = nxc.cpu().numpy()
        row["pairs_set0"] = int(n[0])
        if nsets == 1:
            rev = torch.zeros((nt, 4), dtype=torch.int32, device="cuda")
            mask = torch.zeros(nq, dtype=torch.bool, device="cuda")
            ar = torch.arange(nq, dtype=torch.int32, device="cuda")

            def two_pass():
                ctx.match_device(dq.data_ptr(), nq, dt.data_ptr(), nt, 1, best.data_ptr())
                ctx.match_device(dt.data_ptr(), nt, dq.data_ptr(), nq, 1, rev.data_ptr())
                with torch.cuda.stream(st):
                    torch.eq(rev[:, 1][best[0, :, 1].long()], ar, out=mask)
                    mask.sum()
            row["two_pass"] = time_fn(two_pass, st)
            row["fused_over_two_pass"] = row["fused"]["us"] / row["two_pass"]["us"]
            ctx.synchronize()
            ref = best[0][mask].cpu().numpy().view(orb.DMATCH_DTYPE).reshape(-1)
            got = xc[0, :n[0]].cpu().numpy().view(orb.DMATCH_DTYPE).reshape(-1)
            row["fused_equals_two_pass"] = bool(got.tobytes() == ref.tobytes())
        if name == "vo_call":
            t = trains[0]
            for label, fn in (("host_plain", lambda: ctx.match(q, t)), ("host_crosscheck", lambda: ctx.match_crosscheck(q, t))):
                for _ in range(5):
                    fn()
                us = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    for _ in range(200):
                        fn()
                    us.append((time.perf_counter() - t0) * 1e6 / 200)
                row[label] = {"us": float(np.median(us)), "min": float(min(us)), "max": float(max(us)), "reps": 200}
            row["host_crosscheck_equals_device"] = bool(ctx.match_crosscheck(q, t).tobytes() == xc[0, :n[0]].cpu().numpy().view(orb.DMATCH_DTYPE).reshape(-1).tobytes())
        rows.append(row)
        print(json.dumps(row))
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"card": info, "rows": rows}, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
