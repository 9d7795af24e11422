#!/usr/bin/env python
"""Pairwise batched matching (orbx_match_hamming_device_pairwise[_crosscheck]: each query set against its own train set,
one launch) against the per-pair loop of single-set calls that was the only way to run such a batch before, device-resident
and CUDA-event timed on the context's stream after a warm-up.  Workloads:
  frame_to_frame  256 synthetic 640x480 frames through orbx_detect_and_compute_device (1000 features), frame i against frame
                  i + 1 on the extraction output (255 pairs); also one shared-query _device_ragged call of about the same
                  operation count (the tensor pipe's reach when the A operand is expanded once per CTA)
  candidates      per-frame candidate sets: 300-2000 query rows per frame (noisy copies of its descriptors) against each of
                  the 256 frames' descriptors
  few_pairs_N     N = 1, 2, 8, 32 pairs of 1000 x 1000 rows
  f2f_1080p       64 synthetic 1920x1080 frames with 2000 features, 63 frame-to-frame pairs
Every workload runs plain, knn2 and cross-check.  Rates are int8 TOP/s of the distance GEMM, 2 * 256 * sum(nq_p * nt_p) per
call, with the share of the measured sustained int8 peak (DESIGN.md §4).  Every timed output is compared pair by pair with
the loop's output of the same run; `mismatched_pairs` must be 0.  Prints the card, its power limit and max SM clock with the
numbers and writes them as JSON.

  python tools/pairwise_sweep.py [--out profiles/pairwise_sweep.json]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from crosscheck_sweep import card, time_fn  # noqa: E402
from rgbd_visualodometry_b200 import orb  # noqa: E402
from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries, synth_sequence  # noqa: E402

PEAK_TOPS = 3907.0          # measured sustained int8 tcgen05 rate of this B200 (tools/umma_peak.cu, profiles/r2_int8_peak.json)
MODES = ("plain", "knn2", "xchk")
SENTINEL = -7


class Batch:
    """Device-resident pairwise batch: query set p at dq + p * qs * 32 with counts at dqc[p]; train set p likewise."""

    def __init__(self, dq, qs, dqc, dt, ts, dtc, npairs, qn, tn, keep=()):
        self.dq, self.qs, self.dqc, self.dt, self.ts, self.dtc, self.npairs = dq, qs, dqc, dt, ts, dtc, npairs
        self.qn = [min(max(int(x), 0), qs) for x in qn]
        self.tn = [min(max(int(x), 0), ts) for x in tn]
        self.keep = keep                                 # tensors the pointers point into

    @property
    def ops(self):
        return 2 * 256 * sum(a * b for a, b in zip(self.qn, self.tn))


def outputs(b, mode):
    best = torch.full((b.npairs, b.qs, 4), SENTINEL, dtype=torch.int32, device="cuda")
    second = torch.full_like(best, SENTINEL) if mode == "knn2" else None
    nout = torch.full((b.npairs,), SENTINEL, dtype=torch.int32, device="cuda")
    return best, second, nout


def pairwise_call(ctx, b, mode, out):
    best, second, nout = out
    if mode == "xchk":
        return lambda: ctx.match_device_pairwise_crosscheck(b.dq, b.qs, b.dqc, b.dt, b.ts, b.dtc, b.npairs, best.data_ptr(), nout.data_ptr())
    sp = second.data_ptr() if second is not None else 0
    return lambda: ctx.match_device_pairwise(b.dq, b.qs, b.dqc, b.dt, b.ts, b.dtc, b.npairs, best.data_ptr(), sp)


def loop_call(ctx, b, mode, out):
    """One single-set call per pair (query count from the host, train count from the device)."""
    best, second, nout = out
    rec = b.qs * 16

    def run():
        for p in range(b.npairs):
            q, t, tc = b.dq + p * b.qs * 32, b.dt + p * b.ts * 32, b.dtc + 4 * p
            if mode == "xchk":
                ctx.match_device_crosscheck(q, b.qn[p], t, b.ts, tc, 1, best.data_ptr() + p * rec, nout.data_ptr() + 4 * p)
            else:
                ctx.match_device_ragged(q, b.qn[p], t, b.ts, tc, 1, best.data_ptr() + p * rec,
                                        second.data_ptr() + p * rec if second is not None else 0)
    return run


def mismatched_pairs(b, mode, a, c):
    """Pairs whose records differ between two runs (records i < the pair's query count; xchk: count and pairs)."""
    a = [x.cpu().numpy() if x is not None else None for x in a]
    c = [x.cpu().numpy() if x is not None else None for x in c]
    bad = 0
    for p in range(b.npairs):
        n = b.qn[p]
        if mode == "xchk":
            ok = a[2][p] == c[2][p] and np.array_equal(a[0][p, :a[2][p]], c[0][p, :c[2][p]])
        else:
            ok = np.array_equal(a[0][p, :n], c[0][p, :n]) and (a[1] is None or np.array_equal(a[1][p, :n], c[1][p, :n]))
        ok = ok and (a[0][p, n:] == SENTINEL).all()      # the pairwise call leaves slots past the query count alone
        bad += not ok
    return bad


def measure(ctx, st, name, b, modes=MODES):
    rows = []
    for mode in modes:
        pw_out, lp_out = outputs(b, mode), outputs(b, mode)
        pw, lp = pairwise_call(ctx, b, mode, pw_out), loop_call(ctx, b, mode, lp_out)
        pw(); lp(); ctx.synchronize()
        bad = mismatched_pairs(b, mode, pw_out, lp_out)
        row = {"workload": name, "mode": mode, "npairs": b.npairs, "query_stride": b.qs, "train_stride": b.ts,
               "sum_nq": sum(b.qn), "sum_nt": sum(b.tn), "ops": b.ops, "pairwise": time_fn(pw, st), "per_pair_loop": time_fn(lp, st),
               "mismatched_pairs": bad}
        row["pairwise_tops"] = b.ops / (row["pairwise"]["us"] * 1e-6) / 1e12
        row["pairwise_share_of_peak"] = row["pairwise_tops"] / PEAK_TOPS
        row["loop_tops"] = b.ops / (row["per_pair_loop"]["us"] * 1e-6) / 1e12
        row["loop_over_pairwise"] = row["per_pair_loop"]["us"] / row["pairwise"]["us"]
        ctx.synchronize()
        rows.append(row)
        print(json.dumps(row), flush=True)
    return rows


def extract(ctx, frames, nfeat, cap):
    bsz, h, w = frames.shape[:3]
    d_in = torch.from_numpy(frames).cuda()
    d_k = torch.zeros((bsz, cap, 7), dtype=torch.float32, device="cuda")
    d_d = torch.zeros((bsz, cap, 32), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(bsz, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.detect_and_compute_device(d_in.data_ptr(), bsz, w, h, 3 * w, 3 * w * h, 3, d_k.data_ptr(), d_d.data_ptr(), cap, d_n.data_ptr())
    ctx.synchronize()
    return d_d, d_n


def frame_to_frame(d_d, d_n, cap):
    n = d_n.cpu().numpy()
    return Batch(d_d.data_ptr(), cap, d_n.data_ptr(), d_d.data_ptr() + cap * 32, cap, d_n.data_ptr() + 4, len(n) - 1, n[:-1], n[1:],
                 keep=(d_d, d_n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pairwise_sweep.json"))
    args = ap.parse_args()
    info = card()
    print(info, flush=True)
    rows = []
    mctx = orb.Context(1, 1.2, 1, 64, 64, 1)            # the matcher's context (the extraction contexts are sized for frames)
    st = torch.cuda.ExternalStream(mctx.stream)

    # 1. frame-to-frame, 640x480 / 1000 features, 256 frames
    cap = 2000
    frames = np.stack([f for f, _ in synth_sequence(480, 640, 256, 11)])
    ectx = orb.Context(1000, 1.2, 8, 640, 480, 256)
    d_d, d_n = extract(ectx, frames, 1000, cap)
    ectx.close()
    f2f = frame_to_frame(d_d, d_n, cap)
    rows += measure(mctx, st, "frame_to_frame", f2f)
    # the same operation count with one query set shared by the 255 train sets
    nq_eq = int(round(f2f.ops / (2 * 256 * sum(f2f.tn))))
    dq_map = torch.from_numpy(synth_map_queries(d_d[0, :int(d_n[0])].cpu().numpy(), nq_eq, 12)).cuda()
    shared_best = torch.zeros((f2f.npairs, nq_eq, 4), dtype=torch.int32, device="cuda")
    shared = lambda: mctx.match_device_ragged(dq_map.data_ptr(), nq_eq, f2f.dt, cap, f2f.dtc, f2f.npairs, shared_best.data_ptr())  # noqa: E731
    row = {"workload": "frame_to_frame_shared_query", "mode": "plain", "npairs": f2f.npairs, "nq": nq_eq, "ops": 2 * 256 * nq_eq * sum(f2f.tn),
           "shared_query": time_fn(shared, st)}
    row["tops"] = row["ops"] / (row["shared_query"]["us"] * 1e-6) / 1e12
    row["share_of_peak"] = row["tops"] / PEAK_TOPS
    rows.append(row)
    print(json.dumps(row), flush=True)

    # 2. per-frame candidate sets: 300-2000 map rows per frame against that frame's descriptors
    rng = np.random.default_rng(13)
    qstride = 2000
    desc, n = d_d.cpu().numpy(), d_n.cpu().numpy()
    qc = rng.integers(300, qstride + 1, len(n)).astype(np.int32)
    cand = np.stack([synth_map_queries(desc[i, :max(int(min(n[i], cap)), 1)], qstride, 100 + i) for i in range(len(n))])
    dq, dqc = torch.from_numpy(cand).cuda(), torch.from_numpy(qc).cuda()
    rows += measure(mctx, st, "candidates", Batch(dq.data_ptr(), qstride, dqc.data_ptr(), d_d.data_ptr(), cap, d_n.data_ptr(), len(n), qc, n,
                                                  keep=(dq, dqc)))
    del d_d, d_n, dq, dqc

    # 3. few pairs of 1000 x 1000 rows
    for npairs in (1, 2, 8, 32):
        tr = np.stack([synth_descriptors(1000, 200 + p) for p in range(npairs)])
        qs = np.stack([synth_map_queries(tr[p], 1000, 300 + p) for p in range(npairs)])
        dq, dt = torch.from_numpy(qs).cuda(), torch.from_numpy(tr).cuda()
        dc = torch.full((npairs,), 1000, dtype=torch.int32, device="cuda")
        rows += measure(mctx, st, f"few_pairs_{npairs}", Batch(dq.data_ptr(), 1000, dc.data_ptr(), dt.data_ptr(), 1000, dc.data_ptr(), npairs,
                                                               [1000] * npairs, [1000] * npairs, keep=(dq, dt, dc)))

    # 4. frame-to-frame at 1080p / 2000 features, 64 frames
    cap = 4000
    frames = np.stack([f for f, _ in synth_sequence(1080, 1920, 64, 14)])
    ectx = orb.Context(2000, 1.2, 8, 1920, 1080, 64)
    d_d, d_n = extract(ectx, frames, 2000, cap)
    ectx.close()
    rows += measure(mctx, st, "f2f_1080p", frame_to_frame(d_d, d_n, cap))

    mctx.close()
    bad = sum(r.get("mismatched_pairs", 0) for r in rows)
    print("total mismatched pairs:", bad)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"card": info, "peak_tops_sustained": PEAK_TOPS, "total_mismatched_pairs": bad, "rows": rows}, f, indent=1)
    print("wrote", args.out)
    if bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
