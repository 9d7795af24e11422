"""Seeded input cases shared by the golden-vector generator, the oracle tests and the GPU parity tests."""
import hashlib

import numpy as np

from rgbd_visualodometry_b200.synth import synth_frame, synth_descriptors, synth_map_queries


def _checker(h, w, cell=20):
    yy, xx = np.indices((h, w))
    return (((yy // cell) + (xx // cell)) % 2 * 255).astype(np.uint8)


def _tiled():
    return np.ascontiguousarray(np.tile(synth_frame(96, 128, 7, 1), (5, 5)))


def _rolled(seed, dy, dx):
    return np.ascontiguousarray(np.roll(synth_frame(480, 640, seed), (dy, dx), axis=(0, 1)))


# name -> (factory, nfeatures).  Small enough for the C oracle to finish in well under a second each.
ORB_CASES = {
    "vga500": (lambda: synth_frame(480, 640, 0), 500),
    "vga1000_gray": (lambda: synth_frame(480, 640, 2, 1), 1000),
    "odd700": (lambda: synth_frame(467, 701, 3), 700),
    "noise500": (lambda: np.random.default_rng(0).integers(0, 256, (240, 320), dtype=np.uint8), 500),
    "checker500": (lambda: _checker(480, 640), 500),
    "tiled500": (_tiled, 500),            # tie-heavy: cv2 returns 521 > nfeatures
    "small500": (lambda: synth_frame(120, 160, 8), 500),
    "tiny500": (lambda: synth_frame(60, 70, 9), 500),      # every level <= 62 px: no keypoints
    "const500": (lambda: np.full((240, 320), 128, np.uint8), 500),
    "binary1000": (lambda: (np.random.default_rng(5).random((300, 400)) < 0.5).astype(np.uint8) * 255, 1000),
    # libstdc++'s __introselect runs out of its depth budget on these two and takes the __heap_select fallback
    # (found by tools/config_bench.py: about 1 synthetic frame in 100 does)
    "heapsel_a1000": (lambda: _rolled(777 + 21, 7, 13), 1000),
    "heapsel_b1000": (lambda: _rolled(777 + 16, 42, 78), 1000),
}

# larger cases: checked between oracle and GPU, and against cv2 (live when importable, and its stored result in
# tests/golden/, written by tools/make_golden_live.py)
ORB_CASES_LARGE = {
    "720p1500": (lambda: synth_frame(720, 1280, 4), 1500),
    "1080p2000": (lambda: synth_frame(1080, 1920, 5), 2000),
}

# (nfeatures, scaleFactor, nlevels) other than the reference's yaml, on synth_frame(480, 640, 31): oracle vs cv2
LIVE_PARAMS = [(300, 1.5, 4), (400, 2.0, 3), (600, 1.1, 12), (500, 1.2, 1), (250, 2.5, 2)]

# name -> (query factory, train factory) of the "realistic" match cases compared with cv2 (stored as match_live_<name>.npz)
LIVE_MATCH_CASES = {
    "1500x2000": (lambda: synth_map_queries(synth_descriptors(2000, 30), 1500, 31), lambda: synth_descriptors(2000, 30)),
    "3000x2000": (lambda: synth_map_queries(synth_descriptors(2000, 1), 3000, 2), lambda: synth_descriptors(2000, 1)),
}


def _ties_train():
    t = synth_descriptors(300, 11)
    t[100:200] = t[0:100]        # exact duplicate rows -> distance ties, lowest index must win
    return t


# name -> (query factory, train factory)
MATCH_CASES = {
    "iid_1000x500": (lambda: synth_descriptors(1000, 1), lambda: synth_descriptors(500, 2)),
    "real_700x2000": (lambda: synth_map_queries(synth_descriptors(2000, 3), 700, 4), lambda: synth_descriptors(2000, 3)),
    "ties_257x300": (lambda: synth_map_queries(_ties_train(), 257, 12, flip=0.02), _ties_train),
    "ragged_1x1": (lambda: synth_descriptors(1, 5), lambda: synth_descriptors(1, 6)),
    "ragged_3x131": (lambda: synth_descriptors(3, 7), lambda: synth_descriptors(131, 8)),
    "ragged_129x1": (lambda: synth_descriptors(129, 9), lambda: synth_descriptors(1, 10)),
    "zeros_vs_ones": (lambda: np.zeros((5, 32), np.uint8), lambda: np.full((7, 32), 255, np.uint8)),
}


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _sample_rows(n: int, k: int = 32) -> np.ndarray:
    return np.sort(np.random.default_rng(0).choice(n, min(n, k), replace=False)).astype(np.int64)


def stored(**arrays) -> dict:
    """What tools/make_golden_live.py keeps of each record array of a cv2 result: its row count, the sha256 of its bytes
    and a fixed sample of its rows (the sample only names the differing rows when a comparison fails)."""
    out = {}
    for name, a in arrays.items():
        rows = _sample_rows(len(a))
        out.update({f"{name}_n": len(a), f"{name}_sha": sha(a), f"{name}_rows": rows, f"{name}_sample": a[rows]})
    return out


def assert_equals_stored(g, what: str, **arrays) -> None:
    """Every array equals, byte for byte, the cv2 result `g` holds (a stored() record loaded from tests/golden/)."""
    for name, a in arrays.items():
        assert len(a) == int(g[f"{name}_n"]), f"{what}: {len(a)} {name} rows vs {int(g[f'{name}_n'])} from cv2"
        bad = [int(r) for r, s in zip(g[f"{name}_rows"], g[f"{name}_sample"]) if np.asarray(a[r]).tobytes() != np.asarray(s).tobytes()]
        assert sha(a) == str(g[f"{name}_sha"]), f"{what}: {name} differ from cv2's (sampled rows that differ: {bad})"
