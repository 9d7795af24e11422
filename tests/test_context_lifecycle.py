"""Destroying a context returns what it allocated: device memory and the copier threads of the pinned staging.

One warm-up cycle first (module loading keeps device memory for the life of the process), then every cycle creates a
context, runs each entry point that allocates, and closes it.  This catches a leaked buffer of any real size or a copier
thread left running; it cannot see a leaked event or a few bytes."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H, BATCH = 640, 480, 48
MIB = 1 << 20


@pytest.fixture(scope="module")
def orbmod():
    from rgbd_visualodometry_b200 import orb
    return orb


def _threads():
    return len(os.listdir("/proc/self/task"))


def _cycle(orbmod, frames, maps, depth):
    ctx = orbmod.Context(500, 1.2, 8, W, H, BATCH)
    try:
        kps, desc, n = ctx.detect_and_compute_batch(frames)        # pageable frames: pinned staging, copier threads, 3 lanes
        assert (n > 0).all()
        _, _, n2, best = ctx.extract_match_batch(frames, maps)
        assert np.array_equal(n2, n) and [b.shape for b in best] == [(BATCH, len(m)) for m in maps]
        q, t = desc[0, :n[0]], desc[1, :n[1]]
        assert len(ctx.match(q, t)) == n[0]
        assert len(ctx.knn_match2(q, t)) == n[0]
        best, second = ctx.match_sets(maps[0], desc[:8], n[:8], knn2=True)
        assert best.shape == second.shape == (8, len(maps[0]))
        # map points in front of the camera, normals facing it: the tracking match sees candidates
        m = 400
        rng = np.random.default_rng(5)
        pos = rng.uniform([-1.0, -0.8, 2.0], [1.0, 0.8, 5.0], size=(m, 3))
        norm = pos / np.linalg.norm(pos, axis=1, keepdims=True)
        ids = np.arange(1000, 1000 + m, dtype=np.int64)
        ctx.map_upsert(ids, maps[1][:m], pos, norm, np.zeros(m, np.uint8))
        pose = np.concatenate([np.eye(3), np.zeros((3, 1))], axis=1)
        cam = (517.3, 516.5, 325.1, 249.7)
        cand, matches, _, _ = ctx.track_match(ids, pose, cam, W, H, train=None, frame=0)
        assert len(cand) > 0 and len(matches) > 0
        for i in range(3):
            ctx.submit_frame(frames[i])
            k1, _ = ctx.collect_frame()
            assert len(k1) == n[i]
        _, valid = ctx.backproject(kps[0, :n[0]], depth, 5000.0, cam, pose)
        assert valid.any()
    finally:
        ctx.close()


def test_destroy_returns_memory_and_threads(orbmod):
    import torch
    from rgbd_visualodometry_b200.synth import synth_depth, synth_descriptors, synth_frame
    base = [synth_frame(H, W, 4200 + i) for i in range(4)]
    frames = [base[i % 4].copy() for i in range(BATCH)]              # one pageable allocation per frame
    maps = [synth_descriptors(700, 21), synth_descriptors(1500, 22)]
    depth = synth_depth(H, W, 23)
    torch.cuda.mem_get_info()
    _cycle(orbmod, frames, maps, depth)
    free0, threads0 = torch.cuda.mem_get_info()[0], _threads()
    for i in range(5):
        _cycle(orbmod, frames, maps, depth)
        free = torch.cuda.mem_get_info()[0]
        assert abs(free - free0) <= 8 * MIB, f"cycle {i}: {(free0 - free) / MIB:.1f} MiB of device memory not returned"
        assert _threads() == threads0, f"cycle {i}: {_threads() - threads0} threads left running"
