"""Radius matching, BFMatcher(NORM_HAMMING).radiusMatch(query, train, maxDistance): the reference result and the cases shared
by tests/test_radius.py and tools/make_golden_radius.py (which stores cv2's lists of every case at each of its radii as
tests/golden/match_radius_<name>.npz).

cv::BFMatcher::radiusMatchImpl collects each query's train rows with distance <= maxDistance in ascending trainIdx, then
calls std::sort on the list with DMatch::operator<, which compares the distance alone.  libstdc++'s std::sort is an unstable
introsort, so equal distances do not come out in trainIdx order once a list is longer than 16 entries, and its depth-limit
heap-sort fallback changes the order again.  The reference restates that sort exactly (std_sort).

The library's layout is CSR: (records, offsets), query i's list = records[offsets[i]:offsets[i + 1]], offsets int64 [nq + 1]."""
import numpy as np

from knn_cases import KNN_CASES, hamming_matrix
from oracle import oracle as O

GOLDEN_RADII = (1, 30, 64, 100, 128, 256)
LARGE_RADII = (1, 30, 64, 100)          # inputs of more than 600k (query, train) pairs: the radii a VO caller uses
LONG_RADII = (30, 64, 100, 110, 125, 140, 256)
KEY_SHIFT = 20                          # sort keys distance << 20 | trainIdx


def _long_iid():
    rng = np.random.default_rng(70)
    return rng.integers(0, 256, (48, 32), dtype=np.uint8), rng.integers(0, 256, (2500, 32), dtype=np.uint8)


def _long_ties():
    rng = np.random.default_rng(71)     # bytes 0..3: distances <= 64, heavily tied
    return rng.integers(0, 4, (40, 32)).astype(np.uint8), rng.integers(0, 4, (1500, 32)).astype(np.uint8)


def _long_dup():
    rng = np.random.default_rng(72)     # 30 distinct rows, each 40 times, shuffled: long runs of equal distance
    base = rng.integers(0, 256, (30, 32), dtype=np.uint8)
    t = base[rng.permutation(np.repeat(np.arange(30), 40))]
    return np.concatenate([base[:10], rng.integers(0, 256, (20, 32), dtype=np.uint8)]), t


def bits_rows(dists) -> np.ndarray:
    """Train rows whose distance to the all-zero query row is dists[j]: row j has its first dists[j] bits set."""
    d = np.asarray(dists)
    return np.packbits((np.arange(256)[None, :] < d[:, None]).astype(np.uint8), axis=1)


# name -> (query factory, train factory) of the lists longer than 16 entries
LONG_CASES = {
    "long_iid_48x2500": (lambda: _long_iid()[0], lambda: _long_iid()[1]),
    "long_ties_40x1500": (lambda: _long_ties()[0], lambda: _long_ties()[1]),
    "long_dup_30x1200": (lambda: _long_dup()[0], lambda: _long_dup()[1]),
    "adversary_1x1000": (lambda: np.zeros((1, 32), np.uint8), lambda: bits_rows(adversary_distances(1000))),
}
RADIUS_CASES = {**KNN_CASES, **LONG_CASES}


def case_radii(name: str, nq: int, nt: int):
    if name in LONG_CASES:
        return LONG_RADII
    return LARGE_RADII if nq * nt > 600_000 else GOLDEN_RADII


# ---- libstdc++ std::sort (bits/stl_algo.h, bits/stl_heap.h) on a list, comparator lt ----------------------------------------
class StdSort:
    """std::sort(first, last, lt) as libstdc++ runs it.  heap_calls counts the depth-limit fallbacks (__partial_sort)."""

    def __init__(self, lt):
        self.lt = lt
        self.heap_calls = 0

    def sort(self, v):
        n = len(v)
        if n >= 2:
            self.introsort_loop(v, 0, n, 2 * (n.bit_length() - 1))
            self.final_insertion_sort(v, 0, n)
        return v

    def introsort_loop(self, v, first, last, depth):
        while last - first > 16:
            if depth == 0:
                self.heap_calls += 1
                self.heap_sort(v, first, last)
                return
            depth -= 1
            cut = self.partition_pivot(v, first, last)
            self.introsort_loop(v, cut, last, depth)
            last = cut

    def partition_pivot(self, v, first, last):
        lt, mid = self.lt, first + (last - first) // 2
        a, b, c = first + 1, mid, last - 1         # __move_median_to_first(first, a, b, c)
        if lt(v[a], v[b]):
            s = b if lt(v[b], v[c]) else (c if lt(v[a], v[c]) else a)
        else:
            s = a if lt(v[a], v[c]) else (c if lt(v[b], v[c]) else b)
        v[first], v[s] = v[s], v[first]
        f, l = first + 1, last                     # __unguarded_partition(first + 1, last, first)
        while True:
            while lt(v[f], v[first]):
                f += 1
            l -= 1
            while lt(v[first], v[l]):
                l -= 1
            if not f < l:
                return f
            v[f], v[l] = v[l], v[f]
            f += 1

    def adjust_heap(self, v, first, hole, length, value):
        lt, top, child = self.lt, hole, hole
        while child < (length - 1) // 2:
            child = 2 * (child + 1)
            if lt(v[first + child], v[first + child - 1]):
                child -= 1
            v[first + hole] = v[first + child]
            hole = child
        if length % 2 == 0 and child == (length - 2) // 2:
            child = 2 * (child + 1)
            v[first + hole] = v[first + child - 1]
            hole = child - 1
        parent = (hole - 1) // 2
        while hole > top and lt(v[first + parent], value):
            v[first + hole] = v[first + parent]
            hole = parent
            parent = (hole - 1) // 2
        v[first + hole] = value

    def heap_sort(self, v, first, last):           # __partial_sort(first, last, last): __make_heap + __sort_heap
        n = last - first
        if n >= 2:
            for parent in range((n - 2) // 2, -1, -1):
                self.adjust_heap(v, first, parent, n, v[first + parent])
        while last - first > 1:
            last -= 1
            value = v[last]
            v[last] = v[first]
            self.adjust_heap(v, first, 0, last - first, value)

    def insertion_sort(self, v, first, last):
        for i in range(first + 1, last):
            x, j = v[i], i - 1
            while j >= first and self.lt(x, v[j]):
                v[j + 1] = v[j]
                j -= 1
            v[j + 1] = x

    def final_insertion_sort(self, v, first, last):
        # __insertion_sort of the first 16, __unguarded_linear_insert of the rest: the same moves as one insertion sort
        self.insertion_sort(v, first, last)


def _dist_lt(a, b):
    return (a >> KEY_SHIFT) < (b >> KEY_SHIFT)


def std_sort_keys(keys, counter: StdSort = None):
    """std::sort of keys distance << 20 | trainIdx by distance alone (DMatch::operator<)."""
    s = counter or StdSort(_dist_lt)
    return s.sort(list(keys))


def oracle_radius(query: np.ndarray, train: np.ndarray, max_distance: float, counter: StdSort = None):
    """The reference: (records, offsets) of radiusMatch, every list in std::sort's order of its ascending-trainIdx hits.
    Lists of at most 16 entries only see the (stable) insertion sort, i.e. come out by (distance, trainIdx)."""
    nq, nt = len(query), len(train)
    offsets = np.zeros(nq + 1, np.int64)
    if nq == 0 or nt == 0:
        return np.zeros(0, O.MATCH_DTYPE), offsets
    r = 256 if max_distance >= 256 else int(np.floor(max_distance))
    d = hamming_matrix(query, train)
    s = counter or StdSort(_dist_lt)
    lists = []
    for i in range(nq):
        j = np.nonzero(d[i] <= r)[0]
        if len(j) <= 16:
            order = j[np.argsort(d[i, j], kind="stable")]
            lists.append((d[i, order], order))
        else:
            keys = s.sort([(int(x) << KEY_SHIFT) | int(y) for x, y in zip(d[i, j], j)])
            k = np.array(keys, np.int64)
            lists.append((k >> KEY_SHIFT, k & ((1 << KEY_SHIFT) - 1)))
    offsets[1:] = np.cumsum([len(x[1]) for x in lists])
    out = np.zeros(int(offsets[-1]), O.MATCH_DTYPE)
    for i, (dist, idx) in enumerate(lists):
        sl = slice(offsets[i], offsets[i + 1])
        out["queryIdx"][sl] = i
        out["trainIdx"][sl] = idx
        out["distance"][sl] = dist
    return out, offsets


def cv2_radius_to_csr(lists):
    """cv2's list of per-query DMatch lists -> (records, offsets)."""
    offsets = np.zeros(len(lists) + 1, np.int64)
    offsets[1:] = np.cumsum([len(m) for m in lists])
    out = np.zeros(int(offsets[-1]), O.MATCH_DTYPE)
    k = 0
    for ms in lists:
        for m in ms:
            out[k] = (m.queryIdx, m.trainIdx, m.imgIdx, m.distance)
            k += 1
    return out, offsets


def in_distance_index_order(records, offsets) -> bool:
    """True when every list is sorted by (distance, trainIdx) -- what a plain sort would give."""
    for i in range(len(offsets) - 1):
        m = records[offsets[i]:offsets[i + 1]]
        if len(m) > 1 and not np.array_equal(np.lexsort((m["trainIdx"], m["distance"])), np.arange(len(m))):
            return False
    return True


def adversary_distances(n: int):
    """Distances (<= 64 for n <= 1000) of an n-entry list on which libstdc++'s std::sort reaches its heap-sort fallback:
    McIlroy's antiqsort adversary run against StdSort, each item fixed ("frozen") at the next smallest value when the sort
    first compares two unfrozen items; when the fallback starts, every item still unfrozen takes one common value larger
    than all others."""
    val = [None] * n
    state = {"next": 0, "cand": 0}

    def freeze(x):
        val[x] = state["next"]
        state["next"] += 1

    def lt(a, b):
        x, y = a & 0xFFFFF, b & 0xFFFFF
        if val[x] is None and val[y] is None:
            freeze(x if x == state["cand"] else y)
        if val[x] is None:
            state["cand"] = x
        elif val[y] is None:
            state["cand"] = y
        gas = 1 << 30
        return (gas if val[x] is None else val[x]) < (gas if val[y] is None else val[y])

    class Stop(Exception):
        pass

    s = StdSort(lt)

    def stop(v, first, last):
        raise Stop

    s.heap_sort = stop
    try:
        s.sort(list(range(n)))
    except Stop:
        pass
    g = state["next"]
    return [g if v is None else v for v in val]
