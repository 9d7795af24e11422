"""bench.py's output contract on CPU: the reference arm (`--impl reference`, cv2 on the host cores -- the only arm that runs
without a GPU) prints exactly ONE JSON line on stdout, whatever libraries write there, carrying the keys the driver reads;
under a multi-rank launch only rank 0 prints."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)


def test_reference_arm_prints_one_json_line():
    pytest.importorskip("cv2")
    p = _run({"RANK": "0", "WORLD_SIZE": "1", "LOCAL_RANK": "0"})
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "orb_extract_match_frames_per_s_640x480" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_are_silent():
    p = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert p.returncode == 0, p.stderr[-2000:]
    assert p.stdout.strip() == ""


def test_orbx_arm_refuses_to_run_without_a_gpu():
    """The product arm has no CPU fallback: on a box without a CUDA device it must stop with a clear message and print no JSON
    line (a line from a silent fallback would be read as a measurement)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True, cwd=ROOT, timeout=600,
                       env=dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0"))
    assert p.returncode != 0
    assert "no CPU fallback" in (p.stderr + p.stdout)
    assert not any(ln.strip().startswith("{") for ln in p.stdout.splitlines())


def test_dump_outputs_writes_the_step_outputs_as_float_arrays(tmp_path):
    """--dump-outputs: the buffers of a step (counts, keypoint records, descriptors, the two match record sets) become float32 /
    float64 .npy files holding the same values; a batch whose outputs could exceed the 64 MiB budget is cut to a seeded sample
    of frames that depends only on the buffer shapes."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    rng = np.random.default_rng(3)
    for nb, cap, m, dumped in ((5, 40, 64, 5), (256, 1280, 2048, 253)):
        cnt = rng.integers(0, cap + 1, nb).astype(np.int32)
        cnt[0] = 0
        kps = rng.random((nb, cap, 7)).astype(np.float32)
        kps[..., 5:].view(np.int32)[:] = rng.integers(-1, 8, (nb, cap, 2))
        desc = rng.integers(0, 256, (nb, cap, 32), dtype=np.uint8)
        best = rng.integers(-1, cap, (2, nb, m, 4)).astype(np.int32)
        best[..., 3].view(np.float32)[:] = rng.integers(0, 257, (2, nb, m))
        out = tmp_path / str(nb)
        bench.dump_outputs(str(out), [cnt, kps, desc, best], False)
        got = {p.stem: np.load(p) for p in out.iterdir()}
        assert sorted(got) == ["counts", "descriptors", "frames", "keypoints", "matches"]
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        assert sum(a.nbytes for a in got.values()) <= 64 << 20
        fr = got["frames"].astype(np.int64)
        assert len(fr) == dumped and np.array_equal(fr, np.unique(fr)) and fr.max() < nb
        assert np.array_equal(got["counts"], cnt[fr])
        rec = np.concatenate([kps[i, :cnt[i]] for i in fr])
        assert np.array_equal(got["keypoints"][:, :5], rec[:, :5]) and np.array_equal(got["keypoints"][:, 5:], rec[:, 5:].view(np.int32))
        assert np.array_equal(got["descriptors"], np.concatenate([desc[i, :cnt[i]] for i in fr]))
        bf = best[:, fr]
        assert np.array_equal(got["matches"][..., :3], bf[..., :3]) and np.array_equal(got["matches"][..., 3], bf[..., 3].view(np.float32))
        bench.dump_outputs(str(out), [cnt, kps, desc, best], False)
        assert np.array_equal(np.load(out / "frames.npy"), got["frames"])


def test_steps_must_be_positive():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True, text=True, cwd=ROOT,
                       timeout=120)
    assert p.returncode != 0 and "--steps" in p.stderr and not p.stdout.strip()
