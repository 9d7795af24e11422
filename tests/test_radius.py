"""Radius Hamming matching, BFMatcher(NORM_HAMMING).radiusMatch(query, train, maxDistance): every train row within the radius
of each query, in cv2's exact list order (libstdc++ std::sort by distance alone of the rows in ascending trainIdx), as CSR
(records, int64 offsets).
CPU: the reference (radius_cases.oracle_radius) against cv2's stored and live lists, on long and tie-heavy lists that a
(distance, trainIdx) sort gets wrong and on a list that reaches std::sort's heap-sort fallback; cv2's argument semantics.
GPU (-m gpu): the host call, the ragged device batch and the pairwise batch bit for bit against the reference."""
import functools
import os

import numpy as np
import pytest

from cases import assert_equals_stored, sha
from radius_cases import (LONG_CASES, RADIUS_CASES, StdSort, adversary_distances, bits_rows, case_radii, cv2_radius_to_csr,
                          in_distance_index_order, oracle_radius)

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SENTINEL = -7


@functools.lru_cache(maxsize=None)
def _case(name):
    mq, mt = RADIUS_CASES[name]
    return mq(), mt()


@functools.lru_cache(maxsize=None)
def _ref(name, r):
    q, t = _case(name)
    return oracle_radius(q, t, r)


def _radii(name):
    q, t = _case(name)
    return case_radii(name, len(q), len(t))


def _tie_heavy(rng, n):
    return (rng.integers(0, 4, (n, 32)) if rng.random() < 0.7 else rng.integers(0, 256, (n, 32))).astype(np.uint8)


def _same(a, b):
    return a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()


# ---- CPU -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(RADIUS_CASES))
def test_oracle_vs_golden(oracle, name):
    q, t = _case(name)
    g = np.load(os.path.join(GOLD, f"match_radius_{name}.npz"))
    assert sha(q) == str(g["q_sha"]) and sha(t) == str(g["t_sha"]), "inputs differ from those the golden file was made from"
    for r in _radii(name):
        rec, off = _ref(name, r)
        if f"r{r}_rec" in g:
            assert rec.tobytes() == g[f"r{r}_rec"].tobytes() and off.tobytes() == g[f"r{r}_off"].tobytes(), f"r = {r}"
        else:
            assert_equals_stored(g, f"oracle vs cv2 ({name}, r = {r})", **{f"r{r}_rec": rec, f"r{r}_off": off})


@pytest.mark.parametrize("name", list(RADIUS_CASES))
def test_oracle_vs_live_cv2(oracle, name):
    cv2 = pytest.importorskip("cv2")
    q, t = _case(name)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    for r in _radii(name):
        assert _same(_ref(name, r), cv2_radius_to_csr(bf.radiusMatch(q, t, float(r)))), f"r = {r}"


def test_long_lists_are_not_in_distance_index_order(oracle):
    """The long-list cases hold lists longer than 16 that std::sort leaves out of (distance, trainIdx) order, so a plain sort
    cannot pass the tests built on them; and the random long lists equal live cv2."""
    for name in ("long_iid_48x2500", "long_ties_40x1500", "long_dup_30x1200"):
        rec, off = _ref(name, 125)
        assert (np.diff(off) > 16).any() and not in_distance_index_order(rec, off), name
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    for _ in range(6):
        q, t = _tie_heavy(rng, 10), _tie_heavy(rng, int(rng.integers(100, 1500)))
        t[len(t) // 2:] = t[:len(t) - len(t) // 2]
        r = float(rng.integers(20, 140))
        assert _same(oracle_radius(q, t, r), cv2_radius_to_csr(bf.radiusMatch(q, t, r)))


def test_adversary_reaches_heap_fallback(oracle):
    d = adversary_distances(1000)
    assert max(d) <= 64
    counter = StdSort(lambda a, b: (a >> 20) < (b >> 20))
    q, t = np.zeros((1, 32), np.uint8), bits_rows(d)
    rec, off = oracle_radius(q, t, 64, counter)
    assert counter.heap_calls > 0 and len(rec) == 1000 and not in_distance_index_order(rec, off)
    cv2 = pytest.importorskip("cv2")
    assert _same((rec, off), cv2_radius_to_csr(cv2.BFMatcher(cv2.NORM_HAMMING).radiusMatch(q, t, 64.0)))


def test_cv2_edge_semantics(oracle):
    """Inclusive radius, FLT_EPSILON / NaN raise, +inf and >= 256 keep every row, empty train / query, crossCheck ignored."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(9)
    q, t = _tie_heavy(rng, 20), _tie_heavy(rng, 60)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    for r in (1.0, 1.5, 7.0, 255.0, 256.0, 300.0, float("inf"), 2e-7):
        assert _same(oracle_radius(q, t, r), cv2_radius_to_csr(bf.radiusMatch(q, t, r))), r
    assert len(oracle_radius(q, t, float("inf"))[0]) == 20 * 60
    one = np.zeros((1, 32), np.uint8)
    one_bit = bits_rows([1, 2])
    assert [m.trainIdx for m in bf.radiusMatch(one, one_bit, 1.0)[0]] == [0]
    for r in (float(np.finfo(np.float32).eps), 0.0, -1.0, float("nan")):
        with pytest.raises(cv2.error):
            bf.radiusMatch(q, t, r)
    empty = np.zeros((0, 32), np.uint8)
    assert [len(m) for m in bf.radiusMatch(q, empty, 10.0)] == [0] * 20
    assert _same(oracle_radius(q, empty, 10.0), (np.zeros(0, oracle.MATCH_DTYPE), np.zeros(21, np.int64)))
    assert bf.radiusMatch(empty, t, 10.0) == () or list(bf.radiusMatch(empty, t, 10.0)) == []
    xc = cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True)
    assert _same(cv2_radius_to_csr(xc.radiusMatch(q, t, 40.0)), cv2_radius_to_csr(bf.radiusMatch(q, t, 40.0)))


# ---- GPU -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def orbmod():
    from rgbd_visualodometry_b200 import orb
    return orb


@pytest.fixture(scope="module")
def ctx(orbmod):
    c = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    yield c
    c.close()


def _check_host(ctx, q, t, r, what):
    rec, off = ctx.radius_match(q, t, r)
    want = oracle_radius(q, t, r)
    assert off.tobytes() == want[1].tobytes(), f"{what}: offsets"
    assert rec.tobytes() == want[0].tobytes(), f"{what}: records"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RADIUS_CASES))
def test_host_radius(orbmod, ctx, oracle, name):
    q, t = _case(name)
    for r in _radii(name):
        rec, off = ctx.radius_match(q, t, r)
        want = _ref(name, r)
        assert off.tobytes() == want[1].tobytes(), f"r = {r}: offsets"
        assert rec.tobytes() == want[0].tobytes(), f"r = {r}: records"


@pytest.mark.gpu
def test_host_radius_special_inputs(orbmod, ctx, oracle):
    """All-identical rows; one query against 200k rows at maxDistance = 256 (one list longer than shared memory holds,
    ordered in global memory); query sets over several tiles; radii between integers and +inf."""
    same = np.full((300, 32), 0x3C, np.uint8)
    _check_host(ctx, same[:40], same, 256, "identical rows")
    rng = np.random.default_rng(11)
    big = rng.integers(0, 4, (200_000, 32)).astype(np.uint8)
    _check_host(ctx, big[:1], big, 256, "200k-row list")
    _check_host(ctx, big[:1], big, 40, "200k rows, r = 40")
    q, t = _tie_heavy(rng, 777), _tie_heavy(rng, 1000)
    for r in (7.5, 40.0, 128.0, float("inf")):
        _check_host(ctx, q, t, r, f"777 x 1000, r = {r}")
    d = adversary_distances(1000)
    _check_host(ctx, np.zeros((1, 32), np.uint8), bits_rows(d), 64, "adversary")
    _check_host(ctx, np.zeros((1, 32), np.uint8), bits_rows(d)[::-1].copy(), 64, "adversary reversed")


@pytest.mark.gpu
def test_host_capacity(orbmod, ctx):
    lib, h, C = ctx.lib, ctx.h, orbmod.C
    q, t = _case("real_700x2000")
    want = oracle_radius(q, t, 64)
    total = len(want[0])
    out = np.zeros(total, orbmod.DMATCH_DTYPE)
    off = np.zeros(len(q) + 1, np.int64)
    n = C.c_int(0)
    call = lambda cap: lib.orbx_match_hamming_radius(h, orbmod._ptr(q), len(q), orbmod._ptr(t), len(t), 64.0, orbmod._ptr(out), cap,  # noqa: E731
                                                     orbmod._ptr(off), C.byref(n))
    assert call(total - 1) == orbmod.E_CAPACITY and n.value == total
    assert call(0) == orbmod.E_CAPACITY and n.value == total
    assert call(total) == orbmod.OK and n.value == total
    assert out.tobytes() == want[0].tobytes() and off.tobytes() == want[1].tobytes()


def _device_radius(orbmod, ctx, q, trains, counts, r, cap=None):
    import torch
    nsets, stride = trains.shape[0], trains.shape[1]
    dq, dt = torch.from_numpy(np.ascontiguousarray(q)).cuda(), torch.from_numpy(np.ascontiguousarray(trains)).cuda()
    dn = torch.tensor(counts, dtype=torch.int32, device="cuda")
    nlists = nsets * len(q)
    cap = nlists * stride if cap is None else cap
    out = torch.full((max(cap, 1), 4), SENTINEL, dtype=torch.int32, device="cuda")
    off = torch.full((nlists + 1,), SENTINEL, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device_radius(dq.data_ptr(), len(q), dt.data_ptr(), stride, dn.data_ptr(), nsets, r, out.data_ptr(), cap, off.data_ptr())
    ctx.synchronize()
    return out.cpu().numpy(), off.cpu().numpy()


def _check_lists(orbmod, raw, off, refs, cap, what):
    """refs[s] = (records, offsets) of set / pair s, lists in order; lists ending past cap hold the sentinel."""
    got = np.ascontiguousarray(raw).view(orbmod.DMATCH_DTYPE).reshape(-1)
    base, L = 0, 0
    assert off[0] == 0, what
    for s, (rec, o) in enumerate(refs):
        for i in range(len(o) - 1):
            a, b = base + o[i], base + o[i + 1]
            assert off[L + 1] == b, f"{what}: offset of list {L} (set {s}, query {i})"
            if b <= cap:
                assert got[a:b].tobytes() == rec[o[i]:o[i + 1]].tobytes(), f"{what}: list {L} (set {s}, query {i})"
            elif a < cap:
                assert (raw[a:cap] == SENTINEL).all(), f"{what}: list {L} past the cap was written"
            L += 1
        base += o[-1]


@pytest.mark.gpu
@pytest.mark.parametrize("r", (30, 100, 256))
def test_device_ragged_sets(orbmod, ctx, oracle, r):
    """200 ragged sets (empty, one row, a count past the stride, a negative one), 300 query rows (two query tiles)."""
    rng = np.random.default_rng(30 + r)
    nsets, stride, nq = 200, 120, 300
    trains = _tie_heavy(rng, nsets * stride).reshape(nsets, stride, 32)
    counts = [0, 1, 400, -3, 97, 120, 2] + [int(x) for x in rng.integers(0, 121, nsets - 7)]
    q = _tie_heavy(rng, nq)
    refs = [oracle_radius(q, trains[s, :min(max(counts[s], 0), stride)], r) for s in range(nsets)]
    total = sum(len(x[0]) for x in refs)
    raw, off = _device_radius(orbmod, ctx, q, trains, counts, r, cap=total)
    assert off[-1] == total
    _check_lists(orbmod, raw, off, refs, total, "ragged")
    cap = total // 2                                        # short cap: offsets complete, lists past it untouched
    raw, off = _device_radius(orbmod, ctx, q, trains, counts, r, cap=cap)
    _check_lists(orbmod, raw, off, refs, cap, "ragged, short cap")


@pytest.mark.gpu
def test_pairwise_frame_to_frame(orbmod, oracle):
    """Frame i against frame i + 1 straight out of orbx_detect_and_compute_device; query rows past a pair's count have empty
    lists; also a pairwise batch with empty pairs."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_sequence
    b, cap = 5, 2048
    frames = np.stack([f for f, _ in synth_sequence(480, 640, b, 3)])
    c = orbmod.Context(1000, 1.2, 8, 640, 480, b)
    d_in = torch.from_numpy(frames).cuda()
    d_k = torch.zeros((b, cap, 7), dtype=torch.float32, device="cuda")
    d_d = torch.zeros((b, cap, 32), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(b, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    c.detect_and_compute_device(d_in.data_ptr(), b, 640, 480, 1920, 480 * 1920, 3, d_k.data_ptr(), d_d.data_ptr(), cap, d_n.data_ptr())
    c.synchronize()
    desc, n = d_d.cpu().numpy(), d_n.cpu().numpy()
    assert (n > 500).all()
    for r in (30, 64, 128):
        refs = []
        for p in range(b - 1):
            rec, o = oracle_radius(desc[p, :n[p]], desc[p + 1, :n[p + 1]], r)
            refs.append((rec, np.concatenate([o, np.full(cap - n[p], o[-1], np.int64)])))
        total = sum(len(x[0]) for x in refs)
        out = torch.full((max(total, 1), 4), SENTINEL, dtype=torch.int32, device="cuda")
        off = torch.full(((b - 1) * cap + 1,), SENTINEL, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        c.match_device_pairwise_radius(d_d.data_ptr(), cap, d_n.data_ptr(), d_d.data_ptr() + cap * 32, cap, d_n.data_ptr() + 4, b - 1, r,
                                       out.data_ptr(), total, off.data_ptr())
        c.synchronize()
        _check_lists(orbmod, out.cpu().numpy(), off.cpu().numpy(), refs, total, f"frame-to-frame r = {r}")
    c.close()


@pytest.mark.gpu
def test_argument_errors(orbmod, ctx):
    import torch
    lib, h, C = ctx.lib, ctx.h, orbmod.C
    d = torch.zeros(4096, dtype=torch.int64, device="cuda"); p = d.data_ptr()
    q = np.zeros((4, 32), np.uint8); out = np.zeros(64, orbmod.DMATCH_DTYPE); off = np.zeros(5, np.int64)
    n = C.c_int(0)
    host = lambda r=10.0, nq=4, nt=4, cap=64, qp=orbmod._ptr(q), op=orbmod._ptr(out), fp=orbmod._ptr(off), np_=C.byref(n): \
        lib.orbx_match_hamming_radius(h, qp, nq, orbmod._ptr(q), nt, r, op, cap, fp, np_)  # noqa: E731
    assert host() == orbmod.OK and n.value == 16
    for r in (0.0, -1.0, float(np.finfo(np.float32).eps), float("nan")):
        assert host(r=r) == orbmod.E_ARG, r
    assert host(r=float("inf")) == orbmod.OK and host(r=1e9) == orbmod.OK
    assert host(nq=-1) == orbmod.E_ARG and host(nt=-1) == orbmod.E_ARG and host(cap=-1) == orbmod.E_ARG
    assert host(qp=None) == orbmod.E_ARG and host(op=None) == orbmod.E_ARG and host(fp=None) == orbmod.E_ARG and host(np_=None) == orbmod.E_ARG
    assert host(nt=1 << 20) == orbmod.E_UNSUPPORTED
    off[:] = 9
    assert host(nt=0) == orbmod.OK and n.value == 0 and (off == 0).all()
    # device ragged: d_query, nq, d_train, stride, counts, nsets, radius, out, cap, offsets
    ok = [p, 1, p, 1, p, 1, 10.0, p, 16, p]

    def dev(**kw):
        return lib.orbx_match_hamming_device_radius(h, *[kw.get(f"a{i}", v) for i, v in enumerate(ok)])
    assert dev() == orbmod.OK
    for i in (0, 2, 4, 7, 9):
        assert dev(**{f"a{i}": None}) == orbmod.E_ARG, f"null argument {i}"
    for i in (1, 3, 5, 8):
        assert dev(**{f"a{i}": -1}) == orbmod.E_ARG, f"negative size {i}"
    assert dev(a5=65536) == orbmod.E_ARG and dev(a6=0.0) == orbmod.E_ARG and dev(a6=float("nan")) == orbmod.E_ARG
    assert dev(a3=1 << 20) == orbmod.E_UNSUPPORTED
    assert dev(a5=0) == orbmod.OK and dev(a1=0) == orbmod.OK and dev(a3=0) == orbmod.OK
    # device pairwise: d_query, qstride, qcounts, d_train, tstride, tcounts, npairs, radius, out, cap, offsets
    ok2 = [p, 1, p, p, 1, p, 1, 10.0, p, 16, p]

    def pw(**kw):
        return lib.orbx_match_hamming_device_pairwise_radius(h, *[kw.get(f"a{i}", v) for i, v in enumerate(ok2)])
    assert pw() == orbmod.OK
    for i in (0, 2, 3, 5, 8, 10):
        assert pw(**{f"a{i}": None}) == orbmod.E_ARG, f"null argument {i}"
    for i in (1, 4, 6, 9):
        assert pw(**{f"a{i}": -1}) == orbmod.E_ARG, f"negative size {i}"
    assert pw(a6=65536) == orbmod.E_ARG and pw(a7=0.0) == orbmod.E_ARG and pw(a7=float("nan")) == orbmod.E_ARG
    assert pw(a1=1 << 20) == orbmod.E_UNSUPPORTED and pw(a4=1 << 20) == orbmod.E_UNSUPPORTED
    ctx.synchronize()
    d.fill_(5)
    assert pw(a6=0) == orbmod.OK and pw(a1=0) == orbmod.OK and pw(a4=0) == orbmod.OK
    assert dev(a5=3, a1=0) == orbmod.OK
    ctx.synchronize()
    assert int(d[0]) == 0
    # empty sizes with null pointers: the host form returns first, the device forms check their pointers first
    assert host(nq=0, qp=None, op=None) == orbmod.OK and n.value == 0
    assert dev(a1=0, a0=None) == orbmod.E_ARG
    assert pw(a6=0, a0=None) == orbmod.E_ARG
    # an empty pairwise batch zeroes every list's offset: 3 pairs of query stride 2, no train rows
    d.fill_(5)
    assert pw(a1=2, a4=0, a6=3) == orbmod.OK
    ctx.synchronize()
    assert d[:8].tolist() == [0] * 7 + [5]
    with pytest.raises(orbmod.OrbxError) as e:
        orbmod.BFMatcher().radiusMatch(q, q, 0.0)
    assert e.value.code == orbmod.E_ARG


@pytest.mark.gpu
def test_other_forms_unchanged_around_a_radius_call(orbmod, ctx, oracle):
    q, t = _case("real_700x2000")
    before = (ctx.match(q, t), ctx.knn_match2(q, t), ctx.knn_match(q, t, 5), ctx.match_crosscheck(q, t))
    for r in (30, 128, 256):
        ctx.radius_match(q, t, r)
    after = (ctx.match(q, t), ctx.knn_match2(q, t), ctx.knn_match(q, t, 5), ctx.match_crosscheck(q, t))
    for a, b in zip(before, after):
        assert a.tobytes() == b.tobytes()
    assert before[0].tobytes() == oracle.match_hamming(q, t).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["iid_1000x500", "ties_257x300", "ragged_3x131", "live_1500x2000", "long_dup_30x1200", "adversary_1x1000"])
def test_bfmatcher_vs_cv2(orbmod, name):
    cv2 = pytest.importorskip("cv2")
    q, t = _case(name)
    for cross in (False, True):
        bf, ours = cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=cross), orbmod.BFMatcher(crossCheck=cross)
        for r in (30.0, 64.0, 128.0):
            want = bf.radiusMatch(q, t, r)
            got = ours.radiusMatch(q, t, r)
            assert len(got) == len(want)
            for g, w in zip(got, want):
                assert g.dtype == orbmod.DMATCH_DTYPE
                assert g.tobytes() == cv2_radius_to_csr([w])[0].tobytes(), f"crossCheck = {cross}, r = {r}"
    assert orbmod.BFMatcher().radiusMatch(np.zeros((0, 32), np.uint8), t, 0.0) == []
    assert [len(x) for x in orbmod.BFMatcher().radiusMatch(q, np.zeros((0, 32), np.uint8), 10.0)] == [0] * len(q)
