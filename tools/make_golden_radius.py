#!/usr/bin/env python
"""Generate tests/golden/match_radius_<case>.npz from OpenCV's radius matcher,
cv2.BFMatcher(NORM_HAMMING).radiusMatch(query, train, maxDistance), for every case of tests/radius_cases.py at each of its
radii (radius_cases.case_radii).  Writes only those files.

  match_radius_<case>.npz : input sha256s and, per radius r, cv2's lists in the library's CSR layout under "r<r>_rec"
                            (records) and "r<r>_off" (int64 offsets); for a result over 4096 records tests/cases.py's
                            stored() summary of both instead (row count, sha256, a fixed sample of rows)

  python tools/make_golden_radius.py
"""
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cases import sha, stored  # noqa: E402
from radius_cases import RADIUS_CASES, case_radii, cv2_radius_to_csr  # noqa: E402

out = os.path.join(ROOT, "tests", "golden")
bf = cv2.BFMatcher(cv2.NORM_HAMMING)
for name, (mq, mt) in RADIUS_CASES.items():
    q, t = mq(), mt()
    rec = {}
    for r in case_radii(name, len(q), len(t)):
        m, off = cv2_radius_to_csr(bf.radiusMatch(q, t, float(r)))
        arrays = {f"r{r}_rec": m, f"r{r}_off": off}
        rec.update(stored(**arrays) if len(m) > 4096 else arrays)
    np.savez_compressed(os.path.join(out, f"match_radius_{name}.npz"), cv2_version=cv2.__version__, q_sha=sha(q), t_sha=sha(t), **rec)
    print(f"match_radius_{name}", q.shape, t.shape, sorted(rec))
