"""k-nearest-neighbour matching, BFMatcher(NORM_HAMMING).knnMatch(query, train, k) for any k: the reference result and the
conversions shared by tests/test_knn.py and tools/make_golden_knn.py (which stores cv2's result of every match case of
cases.py at each k of GOLDEN_KS as tests/golden/match_knn_<name>.npz).

The library's layout is [nq, k] DMatch records per call: row i holds query i's list in cv2's order, and the slots past the
train set's size (cv2's list is then shorter than k) hold trainIdx = -1, distance 0 records."""
import numpy as np

from cases import LIVE_MATCH_CASES, MATCH_CASES
from oracle import oracle as O

GOLDEN_KS = (1, 3, 4, 8, 16, 32)
KNN_CASES = {**MATCH_CASES, **{f"live_{name}": mk for name, mk in LIVE_MATCH_CASES.items()}}


def hamming_matrix(query: np.ndarray, train: np.ndarray) -> np.ndarray:
    """[nq, nt] int32 Hamming distances, in row blocks (bounded memory)."""
    q, t = np.ascontiguousarray(query, np.uint8), np.ascontiguousarray(train, np.uint8)
    pop = np.unpackbits(np.arange(256, dtype=np.uint8)[:, None], axis=1).sum(1).astype(np.int32)
    d = np.zeros((len(q), len(t)), np.int32)
    for i in range(0, len(q), 256):
        d[i:i + 256] = pop[q[i:i + 256, None, :] ^ t[None, :, :]].sum(2)
    return d


def padded(nq: int, k: int) -> np.ndarray:
    """[nq, k] records of query i that match nothing: trainIdx = -1, distance 0."""
    out = np.zeros((nq, k), O.MATCH_DTYPE)
    out["queryIdx"] = np.arange(nq)[:, None]
    out["trainIdx"] = -1
    return out


def oracle_knn(query: np.ndarray, train: np.ndarray, k: int) -> np.ndarray:
    """The reference: OpenCV's batchDistance K-insertion (modules/core/src/batch_distance.cpp), restated over all query
    rows at once.  Train rows are visited in index order; row j enters query i's list when its distance is strictly below
    the list's last one, behind every entry of smaller or EQUAL distance (so the lower index wins ties).  Returns [nq, k]
    records with -1 padding past nt; [0, k] when either set is empty (as the library's host call)."""
    nq, nt = len(query), len(train)
    if nq == 0 or nt == 0:
        return np.zeros((0, k), O.MATCH_DTYPE)
    d = hamming_matrix(query, train)
    dist = np.full((nq, k), np.iinfo(np.int32).max, np.int64)
    idx = np.full((nq, k), -1, np.int64)
    col = np.arange(k)[None, :]
    for j in range(nt):
        rows = np.nonzero(d[:, j] < dist[:, k - 1])[0]
        if len(rows) == 0:
            continue
        dj = d[rows, j][:, None]
        dr, ir = dist[rows], idx[rows]
        pos = (dr <= dj).sum(1, keepdims=True)              # entries that stay ahead of row j
        shifted_d = np.concatenate([dr[:, :1], dr[:, :-1]], 1)
        shifted_i = np.concatenate([ir[:, :1], ir[:, :-1]], 1)
        dist[rows] = np.where(col < pos, dr, np.where(col == pos, dj, shifted_d))
        idx[rows] = np.where(col < pos, ir, np.where(col == pos, j, shifted_i))
    out = padded(nq, k)
    found = idx >= 0
    out["trainIdx"][found] = idx[found]
    out["distance"][found] = dist[found]
    return out


def cv2_knn_to_padded(lists, k: int) -> np.ndarray:
    """cv2's list of per-query DMatch lists -> the library's [nq, k] layout (slots past a list's length: trainIdx = -1)."""
    out = padded(len(lists), k)
    for i, ms in enumerate(lists):
        for r, m in enumerate(ms):
            out[i, r] = (m.queryIdx, m.trainIdx, m.imgIdx, m.distance)
    return out
