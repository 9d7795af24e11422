#!/usr/bin/env python
"""Generate tests/golden/match_xcheck_<case>.npz from OpenCV's cross-checked matcher, cv2.BFMatcher(NORM_HAMMING,
crossCheck=True).match, for every case of tests/xcheck_cases.py.  Writes only those files.

  match_xcheck_<case>.npz : input sha256s and the cv2 result (DMatch records); results longer than 1000 records are kept as
                            tests/cases.py's stored() makes them (row count, sha256, a fixed sample of rows)

  python tools/make_golden_crosscheck.py
"""
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cases import sha, stored  # noqa: E402
from xcheck_cases import XCHECK_CASES  # noqa: E402
from oracle import oracle as O  # noqa: E402  (only for the cv2->record converter)

out = os.path.join(ROOT, "tests", "golden")
bf = cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True)
for name, (mq, mt) in XCHECK_CASES.items():
    q, t = mq(), mt()
    m = O.cv2_matches_to_array(bf.match(q, t))
    rec = stored(match=m) if len(m) > 1000 else {"match": m}
    np.savez_compressed(os.path.join(out, f"match_xcheck_{name}.npz"), cv2_version=cv2.__version__, q_sha=sha(q), t_sha=sha(t), **rec)
    print(f"match_xcheck_{name}", q.shape, t.shape, len(m))
