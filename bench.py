#!/usr/bin/env python
"""bench.py -- ORB extract + match frames/s at 640x480 (BASELINE.json metric), one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W]                 # this repo's CUDA path (liborbx.so)
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W] # OpenCV (cv2) on the host cores
  python bench.py --steps K --dump-outputs DIR                         # + the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json configs[1] + the front-end's call pattern, src/frontend.cpp:98-108): a batch of B = 256
synthetic 640x480 BGR frames, ORB with 1000 features / scale 1.2 / 8 levels, then 2 brute-force Hamming matches per
frame of an M = 2048-descriptor map (query) against that frame's descriptors (train).  A "step" = one pass over the
batch.  `value` is device-timed (CUDA events on the library's stream) with frames resident in HBM; `e2e` goes through
the host-buffer C-ABI calls with the H2D / D2H copies inside the timed region.  Frames shard across GPUs with no
collective (weak scaling: B frames per GPU per step).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, NFEAT, NLEVELS, SCALE = 640, 480, 1000, 8, 1.2       # the default workload (BASELINE.json configs[1]); kept as module constants for tools/
BATCH, MAP_M, CAP, MATCHES_PER_FRAME = 256, 2048, 1280, 2
METRIC = "orb_extract_match_frames_per_s_640x480"
LEVEL_PIXELS_VGA = 950532          # SURVEY 8: sum of the 8 pyramid levels of a 640x480 frame
PROFILE_TAG = "r2_v5"              # profiles/<tag>_ncu_metrics.json / _ncu_dram_traffic.json: the committed ncu capture the roofline keys quote
INT8_PEAK_FILE = "profiles/r2_int8_peak.json"

# BASELINE.json configs[0..4] as `--config c1 .. c5` (the driver runs the default, c2).  frames: how the synthetic batch is made;
# ref_sample / cpu_sample: frames per step of the reference arm / of the in-line cpu_baseline (bounded: the CPU needs 2 ms .. 250 ms per frame).
CONFIGS = {
    "c1": dict(w=640, h=480, nfeat=500, batch=256, map_m=1500, frames="sequence", nbase=256, ref_sample=256, cpu_sample=64,
               what="run_vo front-end pattern (config/default.yaml: 500 features) on a synthetic TUM-fr1-shaped 640x480 RGB-D sequence"),
    "c2": dict(w=W, h=H, nfeat=NFEAT, batch=BATCH, map_m=MAP_M, frames="distinct", nbase=32, ref_sample=256, cpu_sample=64,
               what="batched ORB extraction 640x480 BGR"),
    "c3": dict(w=640, h=480, nfeat=2000, batch=32, map_m=100000, frames="distinct", nbase=32, ref_sample=2, cpu_sample=2,
               what="frame<->map Hamming matching sweep: maps of 1k..100k descriptors vs 32 frames' 2000 descriptors"),
    "c4": dict(w=1920, h=1080, nfeat=2000, batch=64, map_m=10000, frames="distinct", nbase=16, ref_sample=64, cpu_sample=32,
               what="1920x1080 ORB extraction + matching"),
    "c5": dict(w=3840, h=2160, nfeat=5000, batch=64, map_m=10000, frames="distinct", nbase=8, ref_sample=16, cpu_sample=16, total_frames=10000,
               what="3840x2160 long synthetic sequence (10k frames per run, cycling 64 device-resident frames per GPU)"),
}
C3_SWEEP = (1000, 2000, 5000, 10000, 20000, 50000, 100000)


def metric_name(cfg):
    return METRIC if (cfg["w"], cfg["h"]) == (W, H) and cfg is not CONFIGS["c3"] else (
        "hamming_match_frames_per_s_map100k_x_2k" if cfg is CONFIGS["c3"] else f"orb_extract_match_frames_per_s_{cfg['w']}x{cfg['h']}")


def cap_of(cfg):
    return CAP if cfg["nfeat"] == NFEAT else int(cfg["nfeat"] * 1.25) + 64


def workload_string(cfg):
    """The workload both arms run, word for word the same in both JSON lines."""
    if cfg is CONFIGS["c3"]:
        return f"{cfg['what']}; value = 2 brute-force Hamming matches of a {cfg['map_m']}-descriptor map per frame (exact BFMatcher(NORM_HAMMING).match)"
    return (f"{cfg['what']}, {cfg['nfeat']} features, scale {SCALE}, {NLEVELS} levels + {MATCHES_PER_FRAME} Hamming matches/frame "
            f"(map {cfg['map_m']} x frame descriptors)")


def make_frames(batch: int, seed: int, w: int = W, h: int = H, nbase: int = 32, kind: str = "distinct") -> np.ndarray:
    """`batch` distinct frames: `nbase` independently generated synthetic frames, the rest cheap distinct variants
    (circular shifts + flips) of them; kind "sequence": consecutive views of one slowly moving camera (TUM-fr1 shape)."""
    from rgbd_visualodometry_b200.synth import synth_frame, synth_sequence
    if kind == "sequence":
        return np.stack([c for c, _ in synth_sequence(h, w, batch, seed=seed)])
    nbase = min(batch, nbase)
    base = [synth_frame(h, w, seed * 100003 + i) for i in range(nbase)]
    rng = np.random.default_rng(seed)
    out = np.empty((batch, h, w, 3), np.uint8)
    for i in range(batch):
        f = base[i % nbase]
        if i >= nbase:
            f = np.roll(f, (int(rng.integers(1, h)), int(rng.integers(1, w))), axis=(0, 1))
            if (i // nbase) & 1:
                f = f[:, ::-1]
        out[i] = f
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms; only samples inside the timed region are reported."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows = []
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(index), "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([time.perf_counter()] + [c.strip() for c in line.split(",")])

    def stop(self, t0: float = 0.0, t1: float = float("inf")) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        allrows = [r[1:] for r in self.rows if len(r) >= 7]
        rows = [r[1:] for r in self.rows if len(r) >= 7 and t0 <= r[0] <= t1 + 0.15] or allrows[-1:]   # samples inside the timed region
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in allrows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "period_ms": 100}


def cpu_reference_fps(frames: np.ndarray, map_desc: np.ndarray, threads: int, nfeat: int = NFEAT, extract: bool = True, train=None):
    """OpenCV on the host, the reference's own operators in the front-end's per-frame pattern (1 detectAndCompute + 2
    BFMatcher.match, src/frontend.cpp:98-108): frame-parallel worker threads, each with its own operator objects and
    cv2.setNumThreads(1) (cv2 releases the GIL; ORB itself does not scale with cv threads).  extract = False (config 3): the
    matches only, against precomputed train sets.  Returns (frames/s, seconds) of one pass."""
    import cv2
    cv2.setNumThreads(1)
    n = len(frames) if extract else len(train)

    def work(idx):
        orb = cv2.ORB_create(nfeat, SCALE, NLEVELS)
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)
        for i in idx:
            d = orb.detectAndCompute(frames[i], None)[1] if extract else train[i]
            for _ in range(MATCHES_PER_FRAME):
                bf.match(map_desc, d)

    if not extract:                                      # BFMatcher.match IS parallelised inside OpenCV: one worker, all cv threads
        cv2.setNumThreads(threads)
        t0 = time.perf_counter()
        work(range(n))
        dt = time.perf_counter() - t0
        cv2.setNumThreads(1)
        return n / dt, dt
    parts = [list(range(t, n, threads)) for t in range(threads)]
    ths = [threading.Thread(target=work, args=(p,)) for p in parts if p]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return n / dt, dt


def flann_lsh_ms(map_desc: np.ndarray, train: np.ndarray, reps: int = 3):
    """What src/frontend.cpp:33,187 literally runs: cv::FlannBasedMatcher(LshIndexParams(5, 10, 2)).match -- approximate and
    randomly seeded, so not a parity target; timed once beside the exact matcher (BASELINE.md section 3)."""
    import cv2
    best = None
    for _ in range(reps):
        fl = cv2.FlannBasedMatcher(dict(algorithm=6, table_number=5, key_size=10, multi_probe_level=2), {})
        t0 = time.perf_counter()
        fl.match(map_desc, train)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best * 1e3


def reference_inputs(cfg, sample: int, seed: int = 0):
    """Frames (or, config 3, train sets) and the map the reference arm works on: the first `sample` frames of rank 0's batch."""
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    if cfg is CONFIGS["c3"]:
        train = [synth_descriptors(cfg["nfeat"], 40 + i) for i in range(sample)]
        return None, train, synth_map_queries(train[0], cfg["map_m"], 41)
    import cv2
    frames = make_frames(cfg["batch"], seed, cfg["w"], cfg["h"], cfg["nbase"], cfg["frames"])[:sample]
    d0 = cv2.ORB_create(cfg["nfeat"], SCALE, NLEVELS).detectAndCompute(frames[0], None)[1]
    return frames, None, synth_map_queries(d0, cfg["map_m"], 17)


def run_reference(args, cfg, rank: int, world: int):
    if rank != 0:
        return
    try:
        import cv2
    except Exception as e:  # pragma: no cover
        emit({"impl": "reference", "unavailable": f"cv2 not importable: {e}"})
        return
    threads = os.cpu_count() or 1
    sample = cfg["ref_sample"]
    frames, train, map_desc = reference_inputs(cfg, sample)
    ext = cfg is not CONFIGS["c3"]
    for _ in range(args.warmup):
        cpu_reference_fps(frames[:threads] if ext else None, map_desc, threads, cfg["nfeat"], ext, None if ext else train[:threads])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_fps(frames, map_desc, threads, cfg["nfeat"], ext, train)
    dt = time.perf_counter() - t0
    fps = sample * args.steps / dt
    extra = {}
    try:
        tr = train[0] if not ext else cv2.ORB_create(cfg["nfeat"], SCALE, NLEVELS).detectAndCompute(frames[0], None)[1]
        cv2.setNumThreads(threads)
        extra = {"flann_lsh_ms_per_match": flann_lsh_ms(map_desc, tr), "note": "FlannBasedMatcher(LshIndexParams(5,10,2)).match(map, frame) incl. index build, all cv threads: "
                 "the matcher src/frontend.cpp:33,187 literally uses (approximate, randomly seeded; not a parity target)"}
        t1 = time.perf_counter(); cv2.BFMatcher(cv2.NORM_HAMMING).match(map_desc, tr); extra["bf_ms_per_match_all_cv_threads"] = (time.perf_counter() - t1) * 1e3
    except Exception as e:  # pragma: no cover
        extra = {"flann_lsh_ms_per_match": None, "note": str(e)}
    line = {"impl": "reference", "metric": metric_name(cfg), "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_string(cfg), "config_id": args.config, "frames_per_gpu_per_step": cfg["batch"]},
            "arm": {"implementation": f"cv2 {cv2.__version__} ORB_create({cfg['nfeat']},{SCALE},{NLEVELS}).detectAndCompute + BFMatcher(NORM_HAMMING).match on the host cores",
                    "frames_timed_per_step": sample},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "reference",
                             "sample": f"{sample} of the step's {cfg['batch']} frames per step, frame-parallel over {threads} host threads, cv2.setNumThreads(1)"},
            "reference_matcher": extra,
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, last_step, is_c3: bool) -> None:
    """--dump-outputs: what the timed step's caller receives, as float32 / float64 .npy files in out_dir (at most DUMP_BYTES).
    Frames whose largest possible output does not fit are left out: a fixed, seeded sample of frames (frames.npy) is kept,
    chosen from the batch size and the buffer shapes only, so two builds run with the same arguments dump the same frames.

      frames.npy      [F]          float64  indices of the dumped frames in the step's batch
      counts.npy      [F]          float64  keypoints per frame                       (not for c3: its train sets are inputs)
      keypoints.npy   [sum, 7]     float32  cv::KeyPoint records of those frames, in order: x, y, size, angle, response, octave, class_id
      descriptors.npy [sum, 32]    float32  their ORB descriptors, one byte per column  (not for c3)
      matches.npy     [2, F, M, 4] float32  cv::DMatch records of the step's two matches of the map: queryIdx, trainIdx, imgIdx, distance
    """
    cnt, kps, desc, best = last_step
    n_match, nb, m, _ = best.shape
    cap = kps.shape[1]
    per_frame = n_match * m * 16 + (0 if is_c3 else 8 + cap * (7 + 32) * 4)
    n_keep = min(nb, DUMP_BYTES // per_frame)
    frames = np.arange(nb) if n_keep == nb else np.sort(np.random.default_rng(0).choice(nb, n_keep, replace=False))
    out = {"frames": frames.astype(np.float64)}
    if not is_c3:
        rec = np.concatenate([kps[i, :cnt[i]] for i in frames]) if n_keep else np.zeros((0, 7), np.float32)
        rec = np.concatenate([rec[:, :5], rec[:, 5:].view(np.int32).astype(np.float32)], axis=1)   # octave, class_id: int32 fields
        out.update(counts=cnt[frames].astype(np.float64), keypoints=rec,
                   descriptors=(np.concatenate([desc[i, :cnt[i]] for i in frames]) if n_keep else np.zeros((0, 32), np.uint8)).astype(np.float32))
    mt = best[:, frames].copy()
    out["matches"] = np.concatenate([mt[..., :3].astype(np.float32), mt[..., 3:].view(np.float32)], axis=-1)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    print(f"bench.py: outputs of the last timed step ({n_keep} of {nb} frames, {sum(a.nbytes for a in out.values()) / 2**20:.1f} MiB) written to {out_dir}",
          file=sys.stderr)


def _load_json(rel):
    try:
        return json.load(open(os.path.join(ROOT, rel)))
    except Exception:
        return None


def run_orbx(args, cfg, rank: int, world: int, local_rank: int):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the orbx path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from rgbd_visualodometry_b200 import orb
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries

    is_c3 = cfg is CONFIGS["c3"]
    Wc, Hc, NF, MAPM = cfg["w"], cfg["h"], cfg["nfeat"], cfg["map_m"]
    B = args.batch or cfg["batch"]
    cap = cap_of(cfg)
    steps = args.steps
    if steps is None:
        steps = 200 if not cfg.get("total_frames") else max(3, -(-cfg["total_frames"] // (B * world)))
        if (Wc, Hc) != (W, H):
            steps = min(steps, 200) if cfg.get("total_frames") else 50
    dev = torch.device("cuda", local_rank)
    ctx = orb.Context(NF, SCALE, NLEVELS, Wc, Hc, B, device=local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=local_rank)
    ws, hs, _, _ = ctx.level_geometry(Wc, Hc)
    level_pixels = int((ws.astype(np.int64) * hs).sum())
    frames_np = None
    d_kps = torch.zeros((B, cap, 7), dtype=torch.float32, device=dev)
    d_desc = torch.zeros((B, cap, 32), dtype=torch.uint8, device=dev)
    d_cnt = torch.zeros(B, dtype=torch.int32, device=dev)
    d_best = torch.zeros((MATCHES_PER_FRAME, B, MAPM, 4), dtype=torch.int32, device=dev)
    if is_c3:
        train_np = np.zeros((B, cap, 32), np.uint8)
        for i in range(B):
            train_np[i, :NF] = synth_descriptors(NF, 40 + i + 1000 * rank)
        d_desc.copy_(torch.from_numpy(train_np).to(dev)); d_cnt.fill_(NF)
        map_np = synth_map_queries(train_np[0, :NF], MAPM, 41)
    else:
        frames_np = make_frames(B, rank, Wc, Hc, cfg["nbase"], cfg["frames"])
        d_in = torch.from_numpy(frames_np).to(dev)
    torch.cuda.synchronize()

    def extract():
        if not is_c3:
            ctx.detect_and_compute_device(d_in.data_ptr(), B, Wc, Hc, Wc * 3, Hc * Wc * 3, 3, d_kps.data_ptr(), d_desc.data_ptr(), cap, d_cnt.data_ptr())

    extract()
    ctx.synchronize()
    counts = d_cnt.cpu().numpy()
    assert counts.max() <= cap, "capacity too small for this data"
    if not is_c3:
        # the map is made from frame 0's descriptors as the CPU oracle computes them (the same bytes a correct build returns),
        # so that the matcher's inputs do not depend on the build being measured
        from oracle import oracle as O
        map_np = synth_map_queries(O.detect_and_compute(frames_np[0], NF, SCALE, NLEVELS, cap=cap)[1], MAPM, 17)
    d_map = torch.from_numpy(map_np).to(dev)
    torch.cuda.synchronize()

    def step():
        extract()
        for m in range(MATCHES_PER_FRAME):
            ctx.match_device_ragged(d_map.data_ptr(), MAPM, d_desc.data_ptr(), cap, d_cnt.data_ptr(), B, d_best[m].data_ptr())

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None   # started early; only samples inside the timed region count
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    ctx.synchronize()
    barrier()
    launches0 = ctx.launch_count
    t_wall0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count - launches0
    t_wall1 = time.perf_counter()
    last_step = None
    if args.dump_outputs and rank == 0:                  # what the last timed step left in the output buffers, before anything reuses them
        with torch.cuda.stream(stream):
            last_step = [t_.clone() for t_ in (d_cnt, d_kps, d_desc, d_best)]
        torch.cuda.synchronize()
    clocks = None
    if sampler:
        note = None
        if t_wall1 - t_wall0 < 0.35:                     # the timed region is shorter than a few sampling periods: keep the same steps running
            while time.perf_counter() - t_wall1 < 0.45:  # (untimed) so that nvidia-smi sees the clocks this workload runs at
                step()
                ctx.synchronize()
            note = "timed region shorter than the 100 ms sampling period: clocks sampled over the timed region plus 0.45 s of the same steps run right after it (untimed)"
        clocks = sampler.stop(t_wall0, time.perf_counter())
        if note:
            clocks["note"] = note
    ctx.synchronize()                                    # raises on any deferred device status
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * steps / (ms_max / 1e3)

    # ---- per-stage device times (CUDA events between the kernels, on the launching stream), 5 extra steps
    ctx.set_profiling(True)
    stage = {}
    for _ in range(5):
        step()
        for k, v in ctx.stage_times().items():
            stage.setdefault(k, []).append(v)
    ctx.set_profiling(False)
    stage_ms = {k: float(np.mean(v)) for k, v in stage.items()}

    # ---- config 3: the map-size sweep (device-timed, 2 matches per frame as in the value)
    sweep = None
    if is_c3:
        sweep = []
        for m in C3_SWEEP:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = max(3, min(50, 2000000 // m))
            for timed in (False, True):
                if timed:
                    ev0.record(stream)
                for _ in range(reps if timed else 2):
                    ctx.match_device_ragged(d_map.data_ptr(), m, d_desc.data_ptr(), cap, d_cnt.data_ptr(), B, d_best[0].data_ptr())
                if timed:
                    ev1.record(stream)
            ctx.synchronize()
            t_ms = ev0.elapsed_time(ev1) / reps
            sweep.append({"map": m, "frames": B, "train_rows_per_frame": NF, "ms": t_ms, "tops": 2.0 * 256 * m * NF * B / (t_ms / 1e3) / 1e12})

    # ---- end to end through the host-buffer C-ABI (rank-local), H2D + D2H inside the timed region
    import ctypes as C
    kps_h = torch.zeros((B, cap, 7), dtype=torch.float32).pin_memory()
    desc_h = torch.zeros((B, cap, 32), dtype=torch.uint8).pin_memory()
    cnt_h = np.zeros(B, np.int32)
    map_pin = torch.from_numpy(map_np).pin_memory()
    best_hs = [torch.zeros((B, MAPM, 4), dtype=torch.int32).pin_memory() for _ in range(MATCHES_PER_FRAME)]
    e2e_pageable = None
    if is_c3:
        train_pin = torch.from_numpy(train_np).pin_memory()
        cnt_np = np.full(B, NF, np.int32)

        def e2e_step():
            for m in range(MATCHES_PER_FRAME):      # host descriptors in, DMatch records out (one map vs every frame's set)
                rc = ctx.lib.orbx_match_hamming_sets(ctx.h, map_pin.data_ptr(), MAPM, train_pin.data_ptr(), cap, cnt_np.ctypes.data, B, best_hs[m].data_ptr(), None)
                assert rc == 0, ctx.lib.orbx_last_error(ctx.h)
        h2d = MATCHES_PER_FRAME * (MAPM * 32 + B * cap * 32 + B * 4)
        d2h = MATCHES_PER_FRAME * (B * MAPM * 16 + 4)
        api = "orbx_match_hamming_sets (host descriptors in, DMatch records out; pinned host buffers), wall clock around the synchronous calls"
    else:
        pin_in = torch.from_numpy(frames_np).pin_memory()
        ptrs = (C.c_void_p * B)(*[pin_in[i].data_ptr() for i in range(B)])
        qptrs = (C.c_void_p * MATCHES_PER_FRAME)(*[map_pin.data_ptr()] * MATCHES_PER_FRAME)
        nqs = (C.c_int * MATCHES_PER_FRAME)(*[MAPM] * MATCHES_PER_FRAME)
        bptrs = (C.c_void_p * MATCHES_PER_FRAME)(*[t_.data_ptr() for t_ in best_hs])

        def e2e_call(frame_ptrs):
            # one C-ABI call: frames (host) -> keypoints, descriptors and the front-end's matches (host, pinned)
            rc = ctx.lib.orbx_extract_match_batch(ctx.h, frame_ptrs, B, Wc, Hc, Wc * 3, 3, kps_h.data_ptr(), desc_h.data_ptr(), cap, cnt_h.ctypes.data,
                                                  qptrs, nqs, MATCHES_PER_FRAME, bptrs)
            assert rc == 0, ctx.lib.orbx_last_error(ctx.h)

        def e2e_step():
            e2e_call(ptrs)
        h2d = B * Hc * Wc * 3 + MATCHES_PER_FRAME * MAPM * 32
        d2h = B * cap * 60 + 2 * B * 4 + MATCHES_PER_FRAME * B * MAPM * 16 + 16
        api = ("orbx_extract_match_batch (one C-ABI call per step: host frames in, keypoints + descriptors + matches out; pinned host buffers), "
               "wall clock around the synchronous call")

    for _ in range(3):
        e2e_step()
    barrier()
    e2e_steps = max(3, min(steps, 20))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_single_fps = world * B * e2e_steps / float(te.item())
    e2e_fps, e2e_mode = e2e_single_fps, "one context, one synchronous call per step"
    if not is_c3:
        # The same call, double-buffered by the caller: TWO contexts on two host threads take alternate steps, so the upload of step
        # i+1 runs under the kernels / download of step i ACROSS calls (a single synchronous call cannot hide its own first upload
        # and last download).  Every step still uploads its frames and downloads its results inside the timed region.
        import threading
        ctx2 = orb.Context(NF, SCALE, NLEVELS, Wc, Hc, B, device=local_rank)
        kps_h2 = torch.zeros((B, cap, 7), dtype=torch.float32).pin_memory()
        desc_h2 = torch.zeros((B, cap, 32), dtype=torch.uint8).pin_memory()
        cnt_h2 = np.zeros(B, np.int32)
        best_hs2 = [torch.zeros((B, MAPM, 4), dtype=torch.int32).pin_memory() for _ in range(MATCHES_PER_FRAME)]
        bptrs2 = (C.c_void_p * MATCHES_PER_FRAME)(*[t_.data_ptr() for t_ in best_hs2])

        def e2e_call2():
            rc = ctx2.lib.orbx_extract_match_batch(ctx2.h, ptrs, B, Wc, Hc, Wc * 3, 3, kps_h2.data_ptr(), desc_h2.data_ptr(), cap, cnt_h2.ctypes.data,
                                                   qptrs, nqs, MATCHES_PER_FRAME, bptrs2)
            assert rc == 0, ctx2.lib.orbx_last_error(ctx2.h)
        for _ in range(2):
            e2e_call2()
        # (records compared as bytes: class_id = -1 is a NaN pattern when the record is viewed as floats)
        assert np.array_equal(cnt_h2, cnt_h) and all(kps_h2[i, :cnt_h[i]].numpy().tobytes() == kps_h[i, :cnt_h[i]].numpy().tobytes()
                                                      and torch.equal(desc_h2[i, :cnt_h[i]], desc_h[i, :cnt_h[i]]) for i in range(B)) \
            and all(torch.equal(a, b) for a, b in zip(best_hs, best_hs2)), "the two contexts disagree"
        n_each = max(2, e2e_steps // 2)

        def loop(fn):
            for _ in range(n_each):
                fn()
        barrier()
        th = [threading.Thread(target=loop, args=(fn,)) for fn in (e2e_step, e2e_call2)]
        t0 = time.perf_counter()
        for t_ in th:
            t_.start()
        for t_ in th:
            t_.join()
        barrier()
        tp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
        e2e_fps = world * B * 2 * n_each / float(tp.item())
        e2e_steps = 2 * n_each
        e2e_mode = "two contexts on two host threads taking alternate steps (double-buffered by the caller), one synchronous call per step each"
        api = api.replace("wall clock around the synchronous call", "wall clock around all calls")
        ctx2.close()
    if not is_c3 and rank == 0:
        # the reference's frames are pageable cv::Mat buffers (src/frame.cpp:28): the same call on ordinary (unpinned) numpy memory
        pptrs = (C.c_void_p * B)(*[frames_np[i].ctypes.data for i in range(B)])
        for _ in range(2):
            e2e_call(pptrs)
        n_pg = max(3, min(e2e_steps, 10))
        t0 = time.perf_counter()
        for _ in range(n_pg):
            e2e_call(pptrs)
        e2e_pageable = {"value": B * n_pg / (time.perf_counter() - t0), "unit": "frames/s", "note": "rank 0 alone, input frames in pageable host memory (as the reference's cv::Mat), outputs pinned"}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (SURVEY 8d): algorithmic bytes per frame x frames per launch / its duration
    peaks = _load_json("MEASURED_PEAKS.json") or {}
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    n_out = float(counts.mean())
    b_alg = 3 * Wc * Hc + 2 * level_pixels + 60 * n_out
    ext_stages = {k: v for k, v in stage_ms.items() if k != "match"}   # gray, pyramid, fast_nms, select_harris, blur, describe
    dom = max(ext_stages, key=ext_stages.get) if ext_stages else None
    ext_total = sum(ext_stages.values())
    roofline = None
    ncu = _load_json(f"profiles/{PROFILE_TAG}_ncu_metrics.json") or {}
    kname = {"gray": "k_gray", "pyramid": "k_pyr_tma", "fast_nms": "k_fast_warp", "select_harris": "k_select_fast", "blur": "k_blur", "describe": "k_describe_tma"}
    if dom:
        traffic = None                                   # DRAM bytes of the dominant kernel per launch, from the committed ncu --set full capture
        k = (ncu.get("kernels") or {}).get(kname.get(dom))
        if k and args.config == "c2" and B == BATCH:
            traffic = k["dram_read_bytes"] + k["dram_write_bytes"]
        ach = b_alg * B / (ext_stages[dom] / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": f"{dom} ({kname.get(dom)})", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic,
                    "traffic_source": f"profiles/{PROFILE_TAG}_ncu_metrics.json (ncu --set full, same 256-frame launch)" if traffic else None,
                    "peak_source": peak_src, "algorithmic_bytes_per_frame": b_alg, "frames_per_launch": B,
                    "kernel_ms": ext_stages[dom], "kernel_share_of_extraction": ext_stages[dom] / ext_total}
    pipe_ach = b_alg * B / (ext_total / 1e3) / 1e9 if ext_total else None
    match_ops = 2.0 * 256 * MAPM * float(counts.sum())
    roof_match = None
    if "match" in stage_ms:
        tops = match_ops / (stage_ms["match"] / 1e3) / 1e12
        i8 = _load_json(INT8_PEAK_FILE) or {}
        mk = next((v for n, v in (ncu.get("kernels") or {}).items() if n.startswith("k_hamming_umma")), None)
        peak_m = i8.get("int8_tops_burst")
        roof_match = {"bound": "tensor", "kernel": "k_hamming_umma2 (tcgen05 cta_group::2 kind::i8)" if B * ((MAPM + 255) // 256) >= 148 else "k_hamming_umma (tcgen05 cta_group::1 kind::i8)",
                      "achieved": tops, "peak": peak_m or 4500.0, "unit": "TOP/s", "frac": tops / (peak_m or 4500.0),
                      "peak_source": f"measured: {INT8_PEAK_FILE} (pure tcgen05.mma.kind::i8 issue loop, burst)" if peak_m else "nominal dense int8 (no measured peak file)",
                      "peak_nominal": 4500.0, "frac_of_nominal": tops / 4500.0, "peak_measured_same_shape": i8.get("int8_tops_burst_ts_n96"),
                      "kernel_ms": stage_ms["match"],
                      "ncu_tensor_pipe_cycles_active_pct": mk.get("tensor_pipe_pct") if mk else None,
                      "ncu_source": f"profiles/{PROFILE_TAG}_ncu_metrics.json (sm__pipe_tensor_cycles_active, c2 launch shape)" if mk else None}

    # ---- CPU baseline: the reference's own operators (cv2) on this box's host cores, bounded sample, 3 warm-ups, median of 10
    cpu = None
    try:
        if world > 1:
            raise RuntimeError("timed at N = 1 only (the contract: rank 0, one GPU); see the N = 1 line and the --impl reference arm")
        import cv2
        threads = os.cpu_count() or 1
        sample = min(cfg["cpu_sample"], B)
        if is_c3:
            fr, tr = None, [train_np[i, :NF] for i in range(sample)]
        else:
            fr, tr = frames_np[:sample], None
        reps = 10 if sample * (Wc * Hc) <= 64 * 640 * 480 * 2 else 5
        for _ in range(3):
            cpu_reference_fps(fr[:threads] if fr is not None else None, map_np, threads, NF, not is_c3, tr[:threads] if tr else None)
        runs = sorted(cpu_reference_fps(fr, map_np, threads, NF, not is_c3, tr)[0] for _ in range(reps))
        cpu = {"value": float(np.median(runs)), "unit": "frames/s", "cores": threads, "kind": "reference",
               "sample": f"{sample} of the step's {B} frames, 3 warm-ups, median of {reps} passes (min {runs[0]:.0f}, max {runs[-1]:.0f}), cv2 {cv2.__version__} "
                         f"frame-parallel over {threads} threads, cv2.setNumThreads(1)"}
    except Exception as e:  # pragma: no cover
        cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {e}"}

    # ---- parity counters of THIS run against the reference's operators (cv2) on the same frames (SURVEY 8d): a few frames spread
    #      over the batch, both the device-resident outputs of the timed path and the host outputs of the e2e call; all must be 0
    parity = None
    try:
        import cv2
        cv2.setNumThreads(os.cpu_count() or 1)
        cvo, cvm = cv2.ORB_create(NF, SCALE, NLEVELS), cv2.BFMatcher(cv2.NORM_HAMMING)
        chk = sorted({0, B // 3, (2 * B) // 3, B - 1}) if Wc * Hc <= 1920 * 1080 else sorted({0, B - 1})
        kp_bad = desc_bad = match_bad = 0
        cnt_d = d_cnt.cpu().numpy()
        for i in chk:
            if is_c3:
                cd = train_np[i, :NF]
                ref_m = np.array([(m.queryIdx, m.trainIdx, m.imgIdx, m.distance) for m in cvm.match(map_np, cd)], dtype=orb.DMATCH_DTYPE)
                for mm in (d_best[0][i].cpu().numpy(), best_hs[0][i].numpy()):
                    got_m = np.ascontiguousarray(mm).view(orb.DMATCH_DTYPE).reshape(-1)
                    match_bad += int((got_m["trainIdx"] != ref_m["trainIdx"]).sum() + (got_m["distance"] != ref_m["distance"]).sum())
                continue
            ck, cd = cvo.detectAndCompute(frames_np[i], None)
            ref_k = np.array([(k.pt[0], k.pt[1], k.size, k.angle, k.response, k.octave, k.class_id) for k in ck], dtype=orb.KP_DTYPE)
            cm = cvm.match(map_np, cd)
            ref_m = np.array([(m.queryIdx, m.trainIdx, m.imgIdx, m.distance) for m in cm], dtype=orb.DMATCH_DTYPE)
            for kk, dd, nn, mm in ((d_kps[i].cpu().numpy(), d_desc[i].cpu().numpy(), int(cnt_d[i]), d_best[0][i].cpu().numpy()),
                                   (kps_h[i].numpy(), desc_h[i].numpy(), int(cnt_h[i]), best_hs[0][i].numpy())):
                got_k = np.ascontiguousarray(kk[:nn]).view(orb.KP_DTYPE).reshape(-1)
                if len(got_k) != len(ref_k):
                    kp_bad += max(len(got_k), len(ref_k)); desc_bad += 32 * max(len(got_k), len(ref_k)); match_bad += MAPM
                    continue
                kp_bad += int(sum(a.tobytes() != b.tobytes() for a, b in zip(got_k, ref_k)))
                desc_bad += int((dd[:nn] != cd).sum())
                got_m = np.ascontiguousarray(mm).view(orb.DMATCH_DTYPE).reshape(-1)
                match_bad += int((got_m.view(np.uint8).reshape(-1, 16) != ref_m.view(np.uint8).reshape(-1, 16)).any(axis=1).sum()) + abs(len(got_m) - len(ref_m))
        parity = {"vs": f"cv2 {cv2.__version__} detectAndCompute + BFMatcher(NORM_HAMMING).match on the same frames", "frames_checked": chk,
                  "paths": ["device-resident (timed)", "host-buffer C-ABI (e2e)"], "keypoint_record_mismatches": kp_bad,
                  "descriptor_byte_mismatches": desc_bad, "match_record_mismatches": match_bad, "angle_tie_descriptor_diffs": 0 if desc_bad == 0 else None}
    except Exception as e:  # pragma: no cover
        parity = {"unavailable": str(e)}

    in_bytes = B * Hc * Wc * 3 if not is_c3 else B * cap * 32
    line = {"metric": metric_name(cfg), "value": value, "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": ms_max / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": workload_string(cfg), "config_id": args.config, "frames_per_gpu_per_step": B},
            "arm": {"implementation": "liborbx.so (sm_100a kernels; matcher on tcgen05 int8)", "parallelism": f"frame-sharded x{world}, no collective",
                    "l2": f"inputs {in_bytes / 1e6:.0f} MB per step " + ("> 126 MB L2 (no flush needed)" if in_bytes > 126e6 else "(train sets; the matcher is compute-bound)"),
                    "mean_keypoints_per_frame": n_out, "frames_total": world * B * steps,
                    "frames_note": f"{B} distinct device-resident frames per GPU, cycled" if cfg.get("total_frames") else None},
            "clocks": clocks,
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps, "api": api, "mode": e2e_mode,
                    "single_context_value": e2e_single_fps},
            "e2e_pageable": e2e_pageable,
            "gpu_launches": int(launches),
            "roofline": roofline, "roofline_pipeline": {"achieved": pipe_ach, "peak": hbm_peak, "unit": "GB/s", "frac": pipe_ach / hbm_peak if pipe_ach else None,
                                                         "note": "same algorithmic bytes over the sum of all extraction kernels (stage timers on: one stream, no overlap; the timed "
                                                                 "step itself runs the small pyramid levels, their FAST bands and the blur on a side stream under the large levels' FAST)"},
            "roofline_match": roof_match, "stage_ms": stage_ms, "cpu_baseline": cpu, "parity": parity}
    if sweep is not None:
        line["sweep"] = sweep
    if last_step is not None:
        dump_outputs(args.dump_outputs, [t_.cpu().numpy() for t_ in last_step], is_c3)
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


# Rank 0's stdout carries exactly ONE JSON line: everything else a library may print there (NCCL's version banner goes to
# stdout whatever NCCL_DEBUG says) is sent to stderr by pointing fd 1 at fd 2 for the whole run; emit() writes the line to the
# real stdout.
_REAL_STDOUT = None


def _quiet_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    data = (json.dumps(obj) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 200 for c1-c3, 50 for c4, 10 000 frames' worth for c5; reference arm: 5)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="orbx", choices=["orbx", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json configs[0..4]; the default c2 is the metric's configuration")
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (default: the config's)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32 / float64, at most 64 MiB; "
                         "rank 0's frames; see dump_outputs)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "orbx":
        ap.error("--dump-outputs writes the orbx arm's outputs")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    _quiet_stdout()
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 5
        run_reference(args, cfg, rank, world)
    else:
        run_orbx(args, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()
