"""The Hamming matcher at the top of every range include/orbx.h accepts: train sets of N = 2^20 - 1 rows (row keys
dot << 20 | (0xFFFFF - j), the train-row split's atomicMax merge, k_match_finalize), cross-check query sets of N rows (column
keys dot << 20 | (0xFFFFF - q)), radius sort keys distance << 20 | trainIdx on lists longer than shared memory holds, 65535
sets and pairs in one call, and radius CSR offsets past 2^32.
CPU: a bounded-memory reference (per-query np.bitwise_count distances; keys d << 20 | j for best, second and top-k; std::sort
for long radius lists) pinned against the C oracle, knn_cases.oracle_knn and radius_cases.oracle_radius, with duplicate rows
at indices >= 2^19.  GPU (-m gpu): every form bit for bit against that reference (or the C oracle) at those sizes."""
import functools

import numpy as np
import pytest

from knn_cases import oracle_knn, padded
from oracle import oracle as O
from radius_cases import oracle_radius, std_sort_keys
from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
from xcheck_cases import oracle_crosscheck

N = (1 << 20) - 1                     # the largest train set (and cross-check query set) the packed keys can index
SHIFT = 20
MAX_SETS = 65535
SENTINEL = -7
BIG = 1 << 14                         # a distance no pair has: marks the rows past a set's count


# ---- the reference ---------------------------------------------------------------------------------------------------------
def u64(rows: np.ndarray) -> np.ndarray:
    """[n, 32] descriptors as [n, 4] uint64 words."""
    return np.ascontiguousarray(rows, np.uint8).reshape(-1, 32).view(np.uint64)


def dist_row(q: np.ndarray, t64: np.ndarray) -> np.ndarray:
    """Hamming distances of one query row to every train row (t64 = u64(train)), int32 [nt]."""
    return np.bitwise_count(t64 ^ u64(q)[0]).sum(1, dtype=np.int32)


def topk_keys(d: np.ndarray, k: int) -> np.ndarray:
    """The min(k, nt) smallest keys d << 20 | j of a distance row, ascending: the k nearest rows by (distance, trainIdx)."""
    key = (d.astype(np.int64) << SHIFT) | np.arange(len(d), dtype=np.int64)
    if len(key) > k:
        key = key[np.argpartition(key, k - 1)[:k]]
    return np.sort(key)


def radius_keys(d: np.ndarray, r: int) -> np.ndarray:
    """Keys d << 20 | j of the rows within distance r, in cv2's list order: ascending j, then std::sort by distance (a stable
    insertion sort for lists of at most 16 entries)."""
    j = np.flatnonzero(d <= r)
    if len(j) <= 16:
        j = j[np.argsort(d[j], kind="stable")]
        return (d[j].astype(np.int64) << SHIFT) | j
    return np.array(std_sort_keys(((d[j].astype(np.int64) << SHIFT) | j).tolist()), np.int64)


def key_records(qrow: int, keys: np.ndarray, k: int = None) -> np.ndarray:
    """DMatch records of query qrow for keys, padded to k slots with trainIdx = -1, distance 0 records."""
    out = np.zeros(len(keys) if k is None else k, O.MATCH_DTYPE)
    out["queryIdx"], out["trainIdx"] = qrow, -1
    out["trainIdx"][:len(keys)] = keys & ((1 << SHIFT) - 1)
    out["distance"][:len(keys)] = keys >> SHIFT
    return out


def ref_knn(q: np.ndarray, t: np.ndarray, k: int) -> np.ndarray:
    """knnMatch(q, t, k) in the library's [nq, k] layout ([0, k] when either set is empty)."""
    if len(q) == 0 or len(t) == 0:
        return np.zeros((0, k), O.MATCH_DTYPE)
    t64 = u64(t)
    return np.stack([key_records(i, topk_keys(dist_row(q[i], t64), k), k) for i in range(len(q))])


def ref_radius(q: np.ndarray, t: np.ndarray, r: int):
    """radiusMatch(q, t, r) as CSR (records, int64 offsets [nq + 1])."""
    t64 = u64(t)
    lists = [key_records(i, radius_keys(dist_row(q[i], t64), r)) for i in range(len(q))]
    off = np.zeros(len(q) + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in lists])
    return (np.concatenate(lists) if lists else np.zeros(0, O.MATCH_DTYPE)), off


def flip(row: np.ndarray, nbits: int, rng) -> np.ndarray:
    """row with nbits distinct bits inverted (distance nbits from it)."""
    bits = np.unpackbits(row)
    bits[rng.choice(256, nbits, replace=False)] ^= 1
    return np.packbits(bits)


def noisy(rows: np.ndarray, rng) -> np.ndarray:
    """Copies of rows with each bit inverted with probability 1/8 (cheap at a million rows)."""
    r = lambda: rng.integers(0, 256, rows.shape, dtype=np.uint8)   # noqa: E731
    return rows ^ (r() & r() & r())


def _tie_heavy(rng, n):
    return (rng.integers(0, 4, (n, 32)) if rng.random() < 0.7 else rng.integers(0, 256, (n, 32))).astype(np.uint8)


# ---- CPU: the reference pinned ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(12))
def test_reference_vs_oracles(oracle, seed):
    """Small random and tie-heavy inputs (duplicated train rows on every third seed): best, knn2, top-k and radius lists."""
    rng = np.random.default_rng(500 + seed)
    q, t = _tie_heavy(rng, int(rng.integers(1, 40))), _tie_heavy(rng, int(rng.integers(1, 300)))
    if seed % 3 == 0 and len(t) > 1:
        t[len(t) // 2:] = t[:len(t) - len(t) // 2]
    what = f"{len(q)} x {len(t)}"
    assert ref_knn(q, t, 1)[:, 0].tobytes() == oracle.match_hamming(q, t).tobytes(), what
    assert ref_knn(q, t, 2).tobytes() == oracle.match_hamming_knn2(q, t).tobytes(), what
    for k in (1, 3, 32):
        assert ref_knn(q, t, k).tobytes() == oracle_knn(q, t, k).tobytes(), f"{what}, k = {k}"
    for r in (30, 100, 256):
        got, want = ref_radius(q, t, r), oracle_radius(q, t, r)
        assert got[1].tobytes() == want[1].tobytes() and got[0].tobytes() == want[0].tobytes(), f"{what}, r = {r}"


def _far_indexed_case(seed):
    """A small tie-heavy set placed at indices below 24, from 2^19 - 2 and in the last 12 rows of an N-row train set (the
    high rows copies of low ones), every other row a filler at distance >= 192 from every query; and the queries."""
    rng = np.random.default_rng(seed)
    small = rng.integers(0, 4, (48, 32), dtype=np.uint8)
    small[24:36] = small[0:12]
    small[36:48] = small[12:24]
    idx = np.concatenate([np.arange(0, 24), (1 << 19) - 2 + np.arange(12), N - 12 + np.arange(12)])
    full = rng.integers(0, 4, (N, 32), dtype=np.uint8) | np.uint8(0xFC)
    full[idx] = small
    q = np.concatenate([rng.integers(0, 4, (20, 32), dtype=np.uint8), small[[0, 5, 11, 12, 23]]])
    return q, small, idx, full


def _mapped(rec, idx):
    rec = rec.copy()
    found = rec["trainIdx"] >= 0
    rec["trainIdx"][found] = idx[rec["trainIdx"][found]]
    return rec


def test_reference_far_indices(oracle):
    """Duplicate rows at indices >= 2^19 (up to N - 1): the reference on the full N-row set equals the C oracle on it, and
    oracle_knn / oracle_radius on the small set with their train indices mapped to where its rows sit."""
    q, small, idx, full = _far_indexed_case(7)
    assert idx.max() == N - 1 and (idx >= 1 << 19).sum() == 22
    assert ref_knn(q, full, 1)[:, 0].tobytes() == oracle.match_hamming(q, full).tobytes()
    assert ref_knn(q, full, 2).tobytes() == oracle.match_hamming_knn2(q, full).tobytes()
    for k in (1, 3, 32):
        assert ref_knn(q, full, k).tobytes() == _mapped(oracle_knn(q, small, k), idx).tobytes(), f"k = {k}"
    for r in (30, 100):
        got, want = ref_radius(q, full, r), oracle_radius(q, small, r)
        assert got[1].tobytes() == want[1].tobytes() and got[0].tobytes() == _mapped(want[0], idx).tobytes(), f"r = {r}"
    assert (np.diff(want[1]) > 16).all(), "r = 100 keeps all 48 rows: lists long enough for std::sort's partitions"
    # a query equal to row 12 has its copy at N - 12 second, at distance 0
    k2 = ref_knn(q[23:24], full, 2)[0]
    assert list(k2["trainIdx"]) == [12, N - 12] and list(k2["distance"]) == [0, 0]


# ---- GPU helpers -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def orbmod():
    from rgbd_visualodometry_b200 import orb
    return orb


@pytest.fixture(scope="module")
def ctx(orbmod):
    c = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    yield c
    c.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _i32(vals):
    import torch
    return torch.tensor([int(v) for v in vals], dtype=torch.int32, device="cuda")


def _full(shape, dtype=None):
    """A sentinel-filled device buffer (int32 unless dtype; synchronise the device before a context call writes it)."""
    import torch
    return torch.full(shape, SENTINEL, dtype=dtype or torch.int32, device="cuda")


def _rec(raw) -> np.ndarray:
    """Raw int32 [..., 4] output -> DMatch records [...]."""
    a = np.ascontiguousarray(raw)
    return a.view(O.MATCH_DTYPE).reshape(a.shape[:-1])


def _words(a) -> np.ndarray:
    a = np.ascontiguousarray(a)
    return a.view(np.int32).reshape(a.shape + (-1,))


def _assert_same(got, want, what):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    if got.tobytes() != want.tobytes():
        bad = np.argwhere((_words(got) != _words(want)).any(-1))
        at = tuple(int(x) for x in bad[0])
        pytest.fail(f"{what}: {len(bad)} entries differ, the first at {at}: got {got[at]}, want {want[at]}")


# ---- train sets of N rows ---------------------------------------------------------------------------------------------------
PLANT = (0, 1, (1 << 16) - 1, 1 << 16, (1 << 19) - 1, 1 << 19, 1048511, 1048512, N - 1)
DUPS = ((3, N - 1), ((1 << 19) - 1, 1 << 19), (1048511, 1048512), ((1 << 16) - 1, 1 << 16))   # (low copy, high copy)
# 40 rows at distance 1 .. 3 of query x, at both ends of the range and on both sides of 2^16 and 2^19
SPREAD = np.concatenate([np.arange(4, 12), (1 << 16) + 1 + np.arange(4), (1 << 19) - 10 + np.arange(8), (1 << 19) + 1 + np.arange(8),
                         1048513 + np.arange(8), N - 9 + np.arange(4)])
# 2040 rows at distance 4 .. 10 of query y (heavy ties), on both sides of 2^19 and at both ends
RADIAL = np.concatenate([np.arange(12, 24), (1 << 19) - 1040 + np.arange(1024), (1 << 19) + 16 + np.arange(984), 1048540 + np.arange(20)])


@functools.lru_cache(maxsize=None)
def big_case():
    """(train [N, 32], x, y, planted queries): N seeded rows with the exact duplicate pairs DUPS, the SPREAD rows around x and
    the RADIAL rows around y.  The planted queries are x, y, near copies (distance 3) of every PLANT row and exact copies of
    the low duplicates."""
    t = synth_descriptors(N, 2020)
    rng = np.random.default_rng(2021)
    x, y = rng.integers(0, 256, 32, dtype=np.uint8), rng.integers(0, 256, 32, dtype=np.uint8)
    for i, j in enumerate(SPREAD):
        t[j] = flip(x, (1, 2, 2, 3)[i % 4], rng)
    for j in RADIAL:
        t[j] = flip(y, int(rng.choice([4, 6, 6, 8, 10])), rng)
    for lo, hi in DUPS:
        t[hi] = t[lo]
    planted = np.stack([x, y] + [flip(t[p], 3, rng) for p in PLANT] + [t[lo] for lo, _ in DUPS])
    return t, x, y, planted


@functools.lru_cache(maxsize=None)
def big_knn_case():
    """The knn queries (the planted ones and 16 map queries) and their distance rows against the N-row train set."""
    t, _, _, planted = big_case()
    q = np.concatenate([planted, synth_map_queries(t, 16, 2022)])
    t64 = u64(t)
    return q, np.stack([dist_row(r, t64) for r in q])


@pytest.fixture(scope="module")
def dev_train():
    return _dev(big_case()[0])


@pytest.mark.gpu
def test_full_train_match_and_knn2(orbmod, ctx, oracle):
    """match (one query row: the train rows split over 148 CTAs, merged by atomicMax) and knnMatch(k = 2) against N rows."""
    t, x, y, planted = big_case()
    for i in range(len(planted)):
        q = planted[i:i + 1]
        _assert_same(ctx.match(q, t), oracle.match_hamming(q, t), f"match, planted query {i}")
        _assert_same(ctx.knn_match2(q, t), oracle.match_hamming_knn2(q, t), f"knn2, planted query {i}")
    q = np.concatenate([planted, synth_map_queries(t, 1000 - len(planted), 2023)])
    best, k2 = ctx.match(q, t), ctx.knn_match2(q, t)
    _assert_same(best, oracle.match_hamming(q, t), "match, 1000 queries")
    _assert_same(k2, oracle.match_hamming_knn2(q, t), "knn2, 1000 queries")
    # the near copies find their planted rows (the low copy of a duplicate); an exact duplicate has its high copy second
    low = {hi: lo for lo, hi in DUPS}
    assert best["trainIdx"][2:2 + len(PLANT)].tolist() == [low.get(p, p) for p in PLANT]
    dup = k2[2 + len(PLANT):len(planted)]
    assert [tuple(r) for r in dup["trainIdx"].tolist()] == list(DUPS) and (dup["distance"] == 0).all()


@pytest.mark.gpu
def test_full_train_pair_kernel(orbmod, ctx, oracle):
    """148 query tiles (the CTA-pair kernel) against N rows: every record holds its pair's true distance, and a seeded sample
    of 2000 rows plus the planted queries (at the start and at the end of the query set) equal the C oracle."""
    t, x, y, planted = big_case()
    nq = 148 * 256
    q = np.concatenate([planted, synth_map_queries(t, nq - 2 * len(planted), 2024), planted])
    got = ctx.match(q, t)
    assert len(got) == nq and (got["queryIdx"] == np.arange(nq)).all()
    assert ((got["trainIdx"] >= 0) & (got["trainIdx"] < N)).all()
    true_d = np.bitwise_count(u64(q) ^ u64(t)[got["trainIdx"]]).sum(1)
    bad = np.flatnonzero(got["distance"] != true_d)
    assert len(bad) == 0, f"{len(bad)} records name a row at another distance, the first {got[bad[0]]}"
    rows = np.unique(np.concatenate([np.random.default_rng(2025).choice(nq, 2000, replace=False), np.arange(len(planted)),
                                     nq - len(planted) + np.arange(len(planted))]))
    want = oracle.match_hamming(q[rows], t)
    want["queryIdx"] = rows                                  # (the oracle numbers the sampled rows from 0)
    _assert_same(got[rows], want, "sampled rows")


@pytest.mark.gpu
@pytest.mark.parametrize("k", (3, 16, 32))
def test_full_train_knn(orbmod, ctx, dev_train, oracle, k):
    """knnMatch against N rows (host), and the ragged device batch with counts [N, N - 1, 96 k + 1, 0] at stride N."""
    import torch
    t = big_case()[0]
    q, d = big_knn_case()
    want = np.stack([key_records(i, topk_keys(d[i], k), k) for i in range(len(q))])
    _assert_same(ctx.knn_match(q, t, k), want, f"host, k = {k}")
    if k == 32:                                              # query x's list holds rows from both ends of the range
        assert want[0]["trainIdx"].min() < 16 and want[0]["trainIdx"].max() > 1048512
    counts = [N, N - 1, 96 * k + 1, 0]
    trains, dq, dn = dev_train.repeat(4, 1), _dev(q), _i32(counts)       # four sets at stride N
    out = _full((4, len(q), k, 4))
    torch.cuda.synchronize()
    ctx.match_device_knn(dq.data_ptr(), len(q), trains.data_ptr(), N, dn.data_ptr(), 4, k, out.data_ptr())
    ctx.synchronize()
    got = _rec(out.cpu().numpy())
    for s, n in enumerate(counts):
        ref = padded(len(q), k) if n == 0 else np.stack([key_records(i, topk_keys(d[i, :n], k), k) for i in range(len(q))])
        _assert_same(got[s], ref, f"device set {s} ({n} rows), k = {k}")


@pytest.mark.gpu
def test_full_train_crosscheck(orbmod, ctx, oracle):
    t, x, y, planted = big_case()
    q = np.concatenate([planted, synth_map_queries(t, 300 - len(planted), 2026)])
    want = oracle_crosscheck(q, t)
    assert len(want) > 100 and (want["trainIdx"] > 1 << 19).sum() > 10
    _assert_same(ctx.match_crosscheck(q, t), want, "cross-check, 300 x N")


@pytest.mark.gpu
def test_full_train_radius(orbmod, ctx, dev_train, oracle):
    """Query y's list of 2040 rows (ordered in global memory, 20-bit train indices, ties on both sides of 2^19), host and
    device; lists of iid queries (tiny) and of near copies of planted rows, in the same host calls."""
    import torch
    t, x, y, planted = big_case()
    rng = np.random.default_rng(2027)
    q = np.concatenate([y[None], synth_descriptors(6, 2028), flip(y, 20, rng)[None], planted[2:6]])
    for r in (30, 12):
        rec, off = ctx.radius_match(q, t, r)
        want = ref_radius(q, t, r)
        _assert_same(off, want[1], f"host offsets, r = {r}")
        _assert_same(rec, want[0], f"host lists, r = {r}")
    want = ref_radius(q[:1], t, 30)
    n = len(want[0])
    assert n == len(RADIAL) and (want[0]["trainIdx"] < 1 << 19).sum() > 1000 and (want[0]["trainIdx"] >= 1 << 19).sum() > 900
    dq, dn = _dev(y[None]), _i32([N])
    out, off = _full((n + 64, 4)), _full((2,), torch.int64)
    torch.cuda.synchronize()
    ctx.match_device_radius(dq.data_ptr(), 1, dev_train.data_ptr(), N, dn.data_ptr(), 1, 30.0, out.data_ptr(), n, off.data_ptr())
    ctx.synchronize()
    raw = out.cpu().numpy()
    _assert_same(off.cpu().numpy(), want[1], "device offsets")
    _assert_same(_rec(raw[:n]), want[0], "device list")
    assert (raw[n:] == SENTINEL).all(), "device: records past the cap"


@pytest.mark.gpu
def test_full_train_pairwise(orbmod, ctx, dev_train, oracle):
    """Two pairs at train stride N with train counts [N, 70000], query stride 48 with counts [48, 33]: best + second,
    cross-check, knnMatch(32) and radiusMatch(30); every slot past a pair's query count untouched."""
    import torch
    t, x, y, planted = big_case()
    qstride, qc, tc = 48, [48, 33], [N, 70000]
    qs = np.stack([np.concatenate([planted, synth_map_queries(t, qstride - len(planted), 2029)]),
                   np.concatenate([planted[:2], synth_map_queries(t[:70000], qstride - 2, 2030)])])
    trains, dq, dqc, dtc = dev_train.repeat(2, 1), _dev(qs), _i32(qc), _i32(tc)
    args = (dq.data_ptr(), qstride, dqc.data_ptr(), trains.data_ptr(), N, dtc.data_ptr(), 2)
    best, second, knn = _full((2, qstride, 4)), _full((2, qstride, 4)), _full((2, qstride, 32, 4))
    xc, nxc = _full((2, qstride, 4)), _full((2,))
    torch.cuda.synchronize()
    ctx.match_device_pairwise(*args, best.data_ptr(), second.data_ptr())
    ctx.match_device_pairwise_knn(*args, 32, knn.data_ptr())
    ctx.match_device_pairwise_crosscheck(*args, xc.data_ptr(), nxc.data_ptr())
    ctx.synchronize()
    best, second, knn = _rec(best.cpu().numpy()), _rec(second.cpu().numpy()), _rec(knn.cpu().numpy())
    xc, nxc = xc.cpu().numpy(), nxc.cpu().numpy()

    def slots(rows, width=()):                               # [qstride (, width)] records: rows, then sentinel slots
        out = np.full((qstride,) + width + (4,), SENTINEL, np.int32)
        _rec(out)[:len(rows)] = rows
        return _rec(out)

    t64 = u64(t)
    refs = []
    for p in range(2):
        d = [dist_row(qs[p, i], t64[:tc[p]]) for i in range(qc[p])]
        top = np.stack([key_records(i, topk_keys(d[i], 32), 32) for i in range(qc[p])])
        _assert_same(best[p], slots(top[:, 0]), f"pair {p} best")
        _assert_same(second[p], slots(top[:, 1]), f"pair {p} second")
        _assert_same(knn[p], slots(top, (32,)), f"pair {p} knn")
        want = oracle_crosscheck(qs[p, :qc[p]], t[:tc[p]])
        assert nxc[p] == len(want), f"pair {p}: {nxc[p]} cross-check pairs, want {len(want)}"
        _assert_same(_rec(xc[p, :nxc[p]]), want, f"pair {p} cross-check")
        assert (xc[p, qc[p]:] == SENTINEL).all(), f"pair {p} cross-check: slots past the query count"
        lists = [key_records(i, radius_keys(d[i], 30)) for i in range(qc[p])]
        o = np.zeros(qstride + 1, np.int64)
        o[1:qc[p] + 1] = np.cumsum([len(x) for x in lists])
        o[qc[p] + 1:] = o[qc[p]]
        refs.append((np.concatenate(lists), o))
    assert len(refs[0][0]) > len(RADIAL), "pair 0 holds query y's long list"
    total = len(refs[0][0]) + len(refs[1][0])
    out, off = _full((total + 64, 4)), _full((2 * qstride + 1,), torch.int64)
    torch.cuda.synchronize()
    ctx.match_device_pairwise_radius(*args, 30.0, out.data_ptr(), total, off.data_ptr())
    ctx.synchronize()
    raw, off = out.cpu().numpy(), off.cpu().numpy()
    _assert_same(off, np.concatenate([refs[0][1], refs[0][1][-1] + refs[1][1][1:]]), "pairwise radius offsets")
    _assert_same(_rec(raw[:total]), np.concatenate([refs[0][0], refs[1][0]]), "pairwise radius lists")
    assert (raw[total:] == SENTINEL).all(), "pairwise radius: records past the cap"


@pytest.mark.gpu
def test_full_train_all_distances_256(orbmod, ctx, oracle):
    """N identical rows ~x against x: every distance 256, every accumulator at the bottom of its int16 range."""
    x = synth_descriptors(1, 2031)
    t = np.broadcast_to(~x, (N, 32)).copy()
    rec = lambda j: key_records(0, np.asarray(j, np.int64) | (256 << SHIFT))   # noqa: E731
    _assert_same(ctx.match(x, t), rec([0]), "best (148-way split)")
    _assert_same(ctx.knn_match2(x, t), rec([0, 1])[None], "knn2")
    _assert_same(ctx.knn_match(x, t, 32), rec(np.arange(32))[None], "knn(32)")
    got, off = ctx.radius_match(x, t, 255)
    assert len(got) == 0 and off.tolist() == [0, 0], "radius 255"
    _assert_same(ctx.match_crosscheck(x, t), rec([0]), "cross-check")
    got, off = ctx.radius_match(x, t[:4096], 256)            # one list of 4096 equal keys
    assert off.tolist() == [0, 4096]
    _assert_same(got, ref_radius(x, t[:4096], 256)[0], "radius 256, 4096 rows")


# ---- cross-check with a query set of N rows ---------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def big_query_case():
    """N queries (70 % noisy copies of a 500-row train set, the rest noise) and that set; q[N - 2] = q[N - 1] = train[7]."""
    t = synth_descriptors(500, 2040)
    rng = np.random.default_rng(2041)
    q = synth_descriptors(N, 2042)
    copy = rng.random(N) < 0.7
    q[copy] = noisy(t[rng.integers(0, 500, int(copy.sum()))], rng)
    q[N - 2] = q[N - 1] = t[7]
    return q, t


@pytest.mark.gpu
def test_full_query_set_crosscheck(orbmod, ctx, oracle):
    """Cross-check with N query rows (20-bit query indices in the column keys; the last query tile holds 255 rows and one
    padded row): host, and the ragged device batch with two sets; ties between queries N - 2 and N - 1, and 0 and N - 1."""
    import torch
    q, t = big_query_case()
    want = oracle_crosscheck(q, t)
    got = ctx.match_crosscheck(q, t)
    _assert_same(got, want, "host, N x 500")
    assert (N - 2, 7) in set(zip(got["queryIdx"].tolist(), got["trainIdx"].tolist())) and (got["queryIdx"] != N - 1).all()
    assert (got["queryIdx"] >= 1 << 19).sum() > 100
    t2 = synth_descriptors(500, 2043)
    t2[3] = t[7]
    counts = [500, 480]
    dq, dt, dn = _dev(q), _dev(np.stack([t, t2])), _i32(counts)
    out, nout = _full((2, N, 4)), _full((2,))
    torch.cuda.synchronize()
    ctx.match_device_crosscheck(dq.data_ptr(), N, dt.data_ptr(), 500, dn.data_ptr(), 2, out.data_ptr(), nout.data_ptr())
    ctx.synchronize()
    out, nout = out.cpu().numpy(), nout.cpu().numpy()
    for s, ref in enumerate((want, oracle_crosscheck(q, t2[:480]))):
        assert nout[s] == len(ref), f"device set {s}: {nout[s]} pairs, want {len(ref)}"
        _assert_same(_rec(out[s, :nout[s]]), ref, f"device set {s}")
    q2 = q.copy()
    q2[0] = q2[N - 1] = t[11]                                # a tie between the first and the last query
    got = ctx.match_crosscheck(q2, t)
    _assert_same(got, oracle_crosscheck(q2, t), "host, q[0] = q[N - 1]")
    assert tuple(got[["queryIdx", "trainIdx"]][0].tolist()) == (0, 11) and (got["queryIdx"] != N - 1).all()


# ---- 65535 sets and 65535 pairs ---------------------------------------------------------------------------------------------
CHUNK = 1024


def _dist_chunk(q64, t64):
    """q64 [Q, 4] (shared) or [S, Q, 4] (pairwise), t64 [S, T, 4] -> distances [S, Q, T] int32."""
    qq = q64[None, :, None, :] if q64.ndim == 2 else q64[:, :, None, :]
    return np.bitwise_count(qq ^ t64[:, None, :, :]).sum(3, dtype=np.int32)


class Forms:
    """Every form's expected result on S sets from their distance tensor D [S, Q, T], the rows past qn[s] queries and tn[s]
    train rows absent; every tie goes to the lowest index (stable sorts and argmin)."""

    def __init__(self, D, qn, tn):
        S, Q, T = D.shape
        self.qv = np.arange(Q)[None, :] < qn[:, None]
        self.tn = tn
        self.D = np.where((np.arange(T)[None, :] < tn[:, None])[:, None, :] & self.qv[:, :, None], D, BIG)
        self.order = np.argsort(self.D, axis=2, kind="stable")
        self.dsort = np.take_along_axis(self.D, self.order, 2)

    def ranks(self, k, nq=None):
        """[S, nq, k] records: each query's k nearest train rows (trainIdx = -1 past the set's rows)."""
        o, d = self.order[:, :nq, :k], self.dsort[:, :nq, :k]
        recs = np.zeros(o.shape, O.MATCH_DTYPE)
        recs["queryIdx"] = np.arange(o.shape[1])[None, :, None]
        has = np.arange(k)[None, None, :] < self.tn[:, None, None]
        recs["trainIdx"] = np.where(has, o, -1)
        recs["distance"] = np.where(has, d, 0)
        return recs

    def keep(self, nq=None):
        """[S, nq] bool: query i's best train row has query i as its nearest query among the first nq."""
        D = self.D[:, :nq]
        bwd = np.argmin(D, axis=1)
        fwd = self.order[:, :nq, 0]
        return self.qv[:, :nq] & (self.tn[:, None] > 0) & (np.take_along_axis(bwd, fwd, 1) == np.arange(D.shape[1])[None, :])

    def radius(self, r, nq=None):
        """(records of every list in list order, counts [S, nq]); lists hold at most 16 entries: sorted by (distance, j)."""
        o, d = self.order[:, :nq], self.dsort[:, :nq]
        hit = d <= r
        recs = np.zeros(o.shape, O.MATCH_DTYPE)
        recs["queryIdx"] = np.arange(o.shape[1])[None, :, None]
        recs["trainIdx"], recs["distance"] = o, d
        return recs[hit], hit.sum(2)


def _check_xc(got, nout, best, keep, what, qn=None):
    """Cross-check output [S, Q] records and counts against the kept best records, compacted in query order; with qn
    (pairwise), the slots past each pair's query count still hold the sentinel."""
    n = keep.sum(1)
    bad = np.flatnonzero(nout != n)
    assert len(bad) == 0, f"{what}: set {bad[0]} has {nout[bad[0]]} pairs, want {n[bad[0]]}"
    want = np.take_along_axis(best, np.argsort(~keep, axis=1, kind="stable"), 1)
    live = (np.arange(got.shape[1])[None, :] < n[:, None])[..., None]
    _assert_same(_rec(np.where(live, _words(got), _words(want))), want, what)
    if qn is not None:
        past = np.arange(got.shape[1])[None, :] >= qn[:, None]
        assert (_words(got)[past] == SENTINEL).all(), f"{what}: slots past the query count"


@pytest.mark.gpu
def test_65535_sets_shared_query(orbmod, ctx, oracle):
    """One call per form over 65535 ragged sets (stride 16, counts 0 .. 19), every set checked: best + second and cross-check
    with 257 query rows (CTA pairs) and with 200 (the single-CTA kernel, each CTA walking many sets); knnMatch(5) and
    radiusMatch(20) with 64."""
    import torch
    rng = np.random.default_rng(2050)
    S, T = MAX_SETS, 16
    trains = rng.integers(0, 4, (S, T, 32), dtype=np.uint8)
    counts = (np.arange(S) % 20).astype(np.int32)
    q = rng.integers(0, 4, (257, 32), dtype=np.uint8)
    q[199] = q[3]                                            # duplicated query rows: the lower one keeps the columns
    q[256] = q[100]
    dq, dt, dn = _dev(q), _dev(trains), _dev(counts)
    outs = {nq: (_full((S, nq, 4)), _full((S, nq, 4)), _full((S, nq, 4)), _full((S,))) for nq in (257, 200)}
    knn, off, probe = _full((S, 64, 5, 4)), _full((S * 64 + 1,), torch.int64), _full((64, 4))
    torch.cuda.synchronize()
    for nq, (b, s2, x, nx) in outs.items():
        ctx.match_device_ragged(dq.data_ptr(), nq, dt.data_ptr(), T, dn.data_ptr(), S, b.data_ptr(), s2.data_ptr())
        ctx.match_device_crosscheck(dq.data_ptr(), nq, dt.data_ptr(), T, dn.data_ptr(), S, x.data_ptr(), nx.data_ptr())
    ctx.match_device_knn(dq.data_ptr(), 64, dt.data_ptr(), T, dn.data_ptr(), S, 5, knn.data_ptr())
    ctx.match_device_radius(dq.data_ptr(), 64, dt.data_ptr(), T, dn.data_ptr(), S, 20.0, probe.data_ptr(), 0, off.data_ptr())
    ctx.synchronize()                                        # (cap 0: the offsets, and no record)
    total = int(off[-1])
    assert 0 < total < S * 64 * 4, total
    rad = _full((total + 64, 4))
    torch.cuda.synchronize()
    ctx.match_device_radius(dq.data_ptr(), 64, dt.data_ptr(), T, dn.data_ptr(), S, 20.0, rad.data_ptr(), total, off.data_ptr())
    ctx.synchronize()
    assert (probe.cpu().numpy() == SENTINEL).all(), "radius with cap 0 wrote records"
    off, rad = off.cpu().numpy(), rad.cpu().numpy()
    assert (rad[total:] == SENTINEL).all(), "radius: records past the cap"
    nxs = {nq: v[3].cpu().numpy() for nq, v in outs.items()}
    tn = np.minimum(counts, T)
    q64, t64 = u64(q), u64(trains).reshape(S, T, 4)
    rad_recs, rad_counts = [], []
    for s0 in range(0, S, CHUNK):
        s1 = min(S, s0 + CHUNK)
        f = Forms(_dist_chunk(q64, t64[s0:s1]), np.full(s1 - s0, 257), tn[s0:s1])
        two = f.ranks(5)
        for nq, (b, s2, x, _) in outs.items():
            w = f"{nq} queries, sets {s0} .. {s1 - 1}"
            _assert_same(_rec(b[s0:s1].cpu().numpy()), two[:, :nq, 0], f"best, {w}")
            _assert_same(_rec(s2[s0:s1].cpu().numpy()), two[:, :nq, 1], f"second, {w}")
            _check_xc(_rec(x[s0:s1].cpu().numpy()), nxs[nq][s0:s1], two[:, :nq, 0], f.keep(nq), f"cross-check, {w}")
        _assert_same(_rec(knn[s0:s1].cpu().numpy()), two[:, :64], f"knn(5), sets {s0} .. {s1 - 1}")
        rr, rc = f.radius(20, 64)
        rad_recs.append(rr)
        rad_counts.append(rc.reshape(-1))
    _assert_same(off, np.concatenate([[0], np.cumsum(np.concatenate(rad_counts))]), "radius offsets")
    _assert_same(_rec(rad[:total]), np.concatenate(rad_recs), "radius lists")


@pytest.mark.gpu
def test_65535_pairs(orbmod, ctx, oracle):
    """The four pairwise forms over 65535 pairs (query stride 8 with counts 0 .. 10, train stride 16 with counts 0 .. 19),
    every pair checked, every slot past a pair's query count untouched."""
    import torch
    rng = np.random.default_rng(2060)
    P, Qs, T = MAX_SETS, 8, 16
    qs = rng.integers(0, 4, (P, Qs, 32), dtype=np.uint8)
    ts = rng.integers(0, 4, (P, T, 32), dtype=np.uint8)
    qs[::5, 1] = qs[::5, 0]                                  # duplicated query rows
    qc = (np.arange(P) % 11).astype(np.int32)
    tc = ((np.arange(P) // 11 + np.arange(P)) % 20).astype(np.int32)
    dq, dqc, dt, dtc = _dev(qs), _dev(qc), _dev(ts), _dev(tc)
    args = (dq.data_ptr(), Qs, dqc.data_ptr(), dt.data_ptr(), T, dtc.data_ptr(), P)
    b, s2, knn = _full((P, Qs, 4)), _full((P, Qs, 4)), _full((P, Qs, 5, 4))
    x, nx = _full((P, Qs, 4)), _full((P,))
    off, probe = _full((P * Qs + 1,), torch.int64), _full((64, 4))
    torch.cuda.synchronize()
    ctx.match_device_pairwise(*args, b.data_ptr(), s2.data_ptr())
    ctx.match_device_pairwise_crosscheck(*args, x.data_ptr(), nx.data_ptr())
    ctx.match_device_pairwise_knn(*args, 5, knn.data_ptr())
    ctx.match_device_pairwise_radius(*args, 20.0, probe.data_ptr(), 0, off.data_ptr())   # (cap 0: the offsets only)
    ctx.synchronize()
    total = int(off[-1])
    assert 0 < total < P * Qs * 4, total
    rad = _full((total + 64, 4))
    torch.cuda.synchronize()
    ctx.match_device_pairwise_radius(*args, 20.0, rad.data_ptr(), total, off.data_ptr())
    ctx.synchronize()
    assert (probe.cpu().numpy() == SENTINEL).all(), "radius with cap 0 wrote records"
    b, s2, knn = b.cpu().numpy(), s2.cpu().numpy(), knn.cpu().numpy()
    x, nx, off, rad = x.cpu().numpy(), nx.cpu().numpy(), off.cpu().numpy(), rad.cpu().numpy()
    assert (rad[total:] == SENTINEL).all(), "radius: records past the cap"
    qn, tn = np.minimum(qc, Qs), np.minimum(tc, T)
    f = Forms(_dist_chunk(u64(qs).reshape(P, Qs, 4), u64(ts).reshape(P, T, 4)), qn, tn)
    two = f.ranks(5)
    past = np.arange(Qs)[None, :] >= qn[:, None]

    def with_sentinel(recs):
        w = _words(recs).copy()
        w[past] = SENTINEL
        return _rec(w)
    _assert_same(_rec(b), with_sentinel(two[:, :, 0]), "pairwise best")
    _assert_same(_rec(s2), with_sentinel(two[:, :, 1]), "pairwise second")
    _assert_same(_rec(knn), with_sentinel(two), "pairwise knn(5)")
    _check_xc(_rec(x), nx, two[:, :, 0], f.keep(), "pairwise cross-check", qn)
    rr, rc = f.radius(20)
    _assert_same(off, np.concatenate([[0], np.cumsum(rc.reshape(-1))]), "pairwise radius offsets")
    _assert_same(_rec(rad[:total]), rr, "pairwise radius lists")


# ---- radius offsets past 2^32 ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_radius_offsets_past_2_32(orbmod, ctx, dev_train, oracle):
    """4096 queries at maxDistance 256 against a 20-row set and an N-row set: 81920 + 4096 N = 4 295 045 120 records.  The
    device forms write every int64 offset and, with cap = the first set's total, only its lists; the host form refuses."""
    import torch
    rng = np.random.default_rng(2070)
    nq = 4096
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    small = rng.integers(0, 256, (20, 32), dtype=np.uint8)
    cap = 20 * nq
    want = ref_radius(q, small, 256)
    assert want[1][-1] == cap
    closed = cap + np.arange(nq + 1, dtype=np.int64) * N
    assert closed[-1] == 4_295_045_120 and closed[-1] > 1 << 32
    trains = dev_train.repeat(2, 1)                          # set 0: its first 20 rows replaced; set 1: the N-row set
    trains[:20] = _dev(small)
    dq, dq2, dtc, dqc = _dev(q), _dev(np.concatenate([q, q])), _i32([20, N]), _i32([nq, nq])
    for form in ("ragged", "pairwise"):
        out, off = _full((cap + 4096, 4)), _full((2 * nq + 1,), torch.int64)
        torch.cuda.synchronize()
        if form == "ragged":
            ctx.match_device_radius(dq.data_ptr(), nq, trains.data_ptr(), N, dtc.data_ptr(), 2, 256.0, out.data_ptr(), cap, off.data_ptr())
        else:
            ctx.match_device_pairwise_radius(dq2.data_ptr(), nq, dqc.data_ptr(), trains.data_ptr(), N, dtc.data_ptr(), 2, 256.0,
                                             out.data_ptr(), cap, off.data_ptr())
        ctx.synchronize()
        raw, off = out.cpu().numpy(), off.cpu().numpy()
        _assert_same(off[:nq + 1], want[1], f"{form}: set 0 offsets")
        _assert_same(off[nq:], closed, f"{form}: set 1 offsets")
        _assert_same(_rec(raw[:cap]), want[0], f"{form}: set 0 lists")
        assert (raw[cap:] == SENTINEL).all(), f"{form}: records past the cap"
    t = big_case()[0]
    C = orbmod.C
    out = np.full((64, 4), SENTINEL, np.int32)
    offs = np.zeros(nq + 1, np.int64)
    n = C.c_int(SENTINEL)
    rc = ctx.lib.orbx_match_hamming_radius(ctx.h, orbmod._ptr(q), nq, orbmod._ptr(t), N, 256.0, orbmod._ptr(out), 64,
                                           orbmod._ptr(offs), C.byref(n))
    assert rc == orbmod.E_UNSUPPORTED, rc
    assert (out == SENTINEL).all() and n.value == 0
