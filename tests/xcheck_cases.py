"""Seeded input cases of the cross-checked matcher, BFMatcher(NORM_HAMMING, crossCheck=True): every match case of cases.py,
plus cases whose ties sit in the reverse (train -> query) direction.  tools/make_golden_crosscheck.py stores cv2's result of
each as tests/golden/match_xcheck_<name>.npz."""
import numpy as np

from cases import LIVE_MATCH_CASES, MATCH_CASES
from oracle import oracle as O
from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries


def _dup_query():
    q = synth_map_queries(synth_descriptors(300, 23), 400, 24)
    q[200:300] = q[0:100]          # duplicated query rows: a train row's nearest query ties, the lower index must win
    return q


def _self_train():
    t = synth_descriptors(500, 22)
    t[250:350] = t[50:150]         # self-match with duplicates: only the first copy of a row is mutual
    return t


def _identical(n, seed):
    base = synth_descriptors(4, 25)
    rows = base[np.random.default_rng(seed).integers(0, 4, n)]
    rows[::7] = synth_descriptors(len(rows[::7]), seed)   # a few distinct rows among the copies
    return rows


XCHECK_CASES = {
    **MATCH_CASES,
    **{f"live_{name}": mk for name, mk in LIVE_MATCH_CASES.items()},
    "dupquery_400x300": (_dup_query, lambda: synth_descriptors(300, 23)),
    "self_500x500": (_self_train, _self_train),
    "identical_160x120": (lambda: _identical(160, 26), lambda: _identical(120, 27)),
}


def oracle_crosscheck(query: np.ndarray, train: np.ndarray) -> np.ndarray:
    """The reference result: two exact matches of the C oracle (query -> train and train -> query, lowest index on ties in
    both) and the mutual filter, in ascending queryIdx.  An empty train set gives no matches (cv2 raises)."""
    fwd = O.match_hamming(query, train)
    if len(fwd) == 0 or len(train) == 0:
        return np.zeros(0, O.MATCH_DTYPE)
    bwd = O.match_hamming(train, query)
    return fwd[bwd["trainIdx"][fwd["trainIdx"]] == fwd["queryIdx"]].copy()
