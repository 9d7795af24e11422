#!/usr/bin/env python
"""Generate the stored OpenCV results of the comparisons the tests also run live against cv2 (when it is importable), so
that those comparisons still run on a machine without cv2.  Writes only the files listed below; tools/make_golden.py
writes the orb_<case> / match_<case> fixtures of tests/cases.py.  Record arrays are kept as tests/cases.py's stored()
makes them (row count, sha256, a fixed sample of rows), which keeps the files small.

  orb_<case>.npz (ORB_CASES_LARGE), orb_params_<n>_<scale>_<levels>.npz, orb_live555_1000.npz :
      input sha256, nfeatures, cv2 keypoints (28-byte cv::KeyPoint records) and descriptors
  match_live_<case>.npz (LIVE_MATCH_CASES) : input sha256s, cv2 BFMatcher(NORM_HAMMING).match
  stages_701x467.npz : cv2 gray and INTER_LINEAR_EXACT pyramid levels (sha256), cv2 FAST(20, nms) keypoints (x, y, response)
  vo_synth16_cv2.npz : tools/run_vo_synth.py's cv2 front-end on its 16-frame sequence: per-frame counts and camera centres

  python tools/make_golden_live.py
"""
import importlib.util
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cases import LIVE_MATCH_CASES, LIVE_PARAMS, ORB_CASES_LARGE, sha, stored  # noqa: E402
from oracle import oracle as O  # noqa: E402  (only for the cv2->record converters)
from rgbd_visualodometry_b200.synth import synth_frame  # noqa: E402

out = os.path.join(ROOT, "tests", "golden")


def save(fname, **kw):
    np.savez_compressed(os.path.join(out, fname), cv2_version=cv2.__version__, **kw)


def save_orb(fname, img, n, sf=1.2, nl=8):
    k, d = cv2.ORB_create(n, sf, nl).detectAndCompute(img, None)
    d = d if d is not None else np.zeros((0, 32), np.uint8)
    save(fname, img_sha=sha(img), nfeatures=n, **stored(keypoints=O.cv2_keypoints_to_array(k), descriptors=d))
    print(fname, img.shape, n, len(k))


for name, (mk, n) in ORB_CASES_LARGE.items():
    save_orb(f"orb_{name}.npz", mk(), n)
for n, sf, nl in LIVE_PARAMS:
    save_orb(f"orb_params_{n}_{sf}_{nl}.npz", synth_frame(480, 640, 31), n, sf, nl)
save_orb("orb_live555_1000.npz", synth_frame(480, 640, 555), 1000)

for name, (mq, mt) in LIVE_MATCH_CASES.items():
    q, t = mq(), mt()
    m = O.cv2_matches_to_array(cv2.BFMatcher(cv2.NORM_HAMMING).match(q, t))
    save(f"match_live_{name}.npz", q_sha=sha(q), t_sha=sha(t), **stored(match=m))
    print(f"match_live_{name}", len(m))

img = synth_frame(467, 701, 21)
g = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
ws, hs, _ = O.level_geometry(701, 467)
level_sha, prev = [], g
for l in range(1, 8):
    prev = cv2.resize(prev, (ws[l], hs[l]), interpolation=cv2.INTER_LINEAR_EXACT)
    level_sha.append(sha(prev))
f = cv2.FastFeatureDetector_create(20, True).detect(g)
fast = np.array([(int(a.pt[0]), int(a.pt[1]), a.response) for a in f], O.CAND_DTYPE)
save("stages_701x467.npz", img_sha=sha(img), gray_sha=sha(g), level_sha=np.array(level_sha), **stored(fast=fast))
print("stages_701x467", len(fast))

spec = importlib.util.spec_from_file_location("run_vo_synth", os.path.join(ROOT, "tools", "run_vo_synth.py"))
vo = importlib.util.module_from_spec(spec)
spec.loader.exec_module(vo)
vo.run.pos = {}
log, _ = vo.run("cv2", vo.make_sequence(16))
save("vo_synth16_cv2.npz", counts=np.array([x[:4] for x in log], np.int64), centre=np.array([x[4] for x in log]),
     truth=np.array([x[5] for x in log]))
print("vo_synth16_cv2", [x[1:4] for x in log])
