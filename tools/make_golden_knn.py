#!/usr/bin/env python
"""Generate tests/golden/match_knn_<case>.npz from OpenCV's k-nearest-neighbour matcher,
cv2.BFMatcher(NORM_HAMMING).knnMatch(query, train, k), for every case of tests/knn_cases.py at every k of GOLDEN_KS.
Writes only those files.

  match_knn_<case>.npz : input sha256s and, per k, cv2's lists in the library's [nq, k] layout (trainIdx = -1 past a list's
                         end) under "k<k>"; for the live cases (and any result over 4096 records) tests/cases.py's stored()
                         summary of it instead (row count, sha256, a fixed sample of rows)

  python tools/make_golden_knn.py
"""
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cases import sha, stored  # noqa: E402
from knn_cases import GOLDEN_KS, KNN_CASES, cv2_knn_to_padded  # noqa: E402

out = os.path.join(ROOT, "tests", "golden")
bf = cv2.BFMatcher(cv2.NORM_HAMMING)
for name, (mq, mt) in KNN_CASES.items():
    q, t = mq(), mt()
    rec = {}
    for k in GOLDEN_KS:
        m = cv2_knn_to_padded(bf.knnMatch(q, t, k=k), k)
        rec.update(stored(**{f"k{k}": m}) if name.startswith("live_") or m.size > 4096 else {f"k{k}": m})
    np.savez_compressed(os.path.join(out, f"match_knn_{name}.npz"), cv2_version=cv2.__version__, q_sha=sha(q), t_sha=sha(t), **rec)
    print(f"match_knn_{name}", q.shape, t.shape, sorted(rec))
