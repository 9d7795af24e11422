"""k-nearest-neighbour Hamming matching for any k <= 32, BFMatcher(NORM_HAMMING).knnMatch(query, train, k): query i's k
nearest train rows by (distance, trainIdx), in the library's [nq, k] layout (trainIdx = -1 past the train set's size).
CPU: the reference (knn_cases.oracle_knn, cv2's K-insertion restated) against cv2's stored and live results, a numpy
lexsort brute force, and the C oracle's knnMatch(k = 2).  GPU (-m gpu): the host call, the ragged device batch and the
pairwise batch bit for bit against that reference, on every list bucket of the top-k kernels."""
import functools
import os

import numpy as np
import pytest

from cases import assert_equals_stored, sha
from knn_cases import GOLDEN_KS, KNN_CASES, cv2_knn_to_padded, hamming_matrix, oracle_knn, padded

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SENTINEL = -7
# every list bucket (4, 8, 16, 32) and both of its edges; k = 1 and 2 take the plain and knn2 paths of the host call
HOST_KS = (1, 2, 3, 4, 5, 8, 9, 16, 17, 32)


def _golden(name):
    return np.load(os.path.join(GOLD, f"match_knn_{name}.npz"))


@functools.lru_cache(maxsize=None)
def _case(name):
    mq, mt = KNN_CASES[name]
    return mq(), mt()


@functools.lru_cache(maxsize=None)
def _ref(name, k):
    q, t = _case(name)
    return oracle_knn(q, t, k)


def _lexsort(q, t, k):
    """The definition, in numpy: sort each query's train rows by (distance, index), keep the first k."""
    nq, nt = len(q), len(t)
    out = padded(nq, k)
    if nq == 0 or nt == 0:
        return out[:0]
    d = hamming_matrix(q, t)
    for i in range(nq):
        order = np.lexsort((np.arange(nt), d[i]))[:k]
        out["trainIdx"][i, :len(order)] = order
        out["distance"][i, :len(order)] = d[i, order]
    return out


def _tie_heavy(rng, n):
    return (rng.integers(0, 4, (n, 32)) if rng.random() < 0.7 else rng.integers(0, 256, (n, 32))).astype(np.uint8)


# ---- CPU -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(KNN_CASES))
def test_oracle_vs_golden(oracle, name):
    q, t = _case(name)
    g = _golden(name)
    assert sha(q) == str(g["q_sha"]) and sha(t) == str(g["t_sha"]), "inputs differ from those the golden file was made from"
    for k in GOLDEN_KS:
        got = _ref(name, k)
        if f"k{k}" in g:
            assert got.tobytes() == g[f"k{k}"].tobytes(), f"oracle vs cv2 ({name}, k = {k})"
        else:
            assert_equals_stored(g, f"oracle vs cv2 ({name}, k = {k})", **{f"k{k}": got})


@pytest.mark.parametrize("name", list(KNN_CASES))
def test_oracle_vs_live_cv2(oracle, name):
    cv2 = pytest.importorskip("cv2")
    q, t = _case(name)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    for k in (1, 2, 5, 9, 17, 32):
        assert _ref(name, k).tobytes() == cv2_knn_to_padded(bf.knnMatch(q, t, k=k), k).tobytes(), f"k = {k}"


def test_oracle_vs_live_cv2_short_and_empty_train(oracle):
    """k > nt (cv2's lists are nt long: -1 padding), a one-row train set, and an empty one (cv2: one empty list per query)."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    q = _tie_heavy(rng, 40)
    for nt in (1, 2, 5, 31):
        t = _tie_heavy(rng, nt)
        for k in (1, 2, 3, nt, nt + 1, 32):
            lists = bf.knnMatch(q, t, k=k)
            assert all(len(m) == min(k, nt) for m in lists)
            assert oracle_knn(q, t, k).tobytes() == cv2_knn_to_padded(lists, k).tobytes(), f"nt = {nt}, k = {k}"
    lists = bf.knnMatch(q, np.zeros((0, 32), np.uint8), k=3)
    assert len(lists) == len(q) and all(len(m) == 0 for m in lists)
    assert oracle_knn(q, np.zeros((0, 32), np.uint8), 3).shape == (0, 3)


@pytest.mark.parametrize("seed", range(50))
def test_oracle_vs_lexsort(seed):
    rng = np.random.default_rng(1000 + seed)
    q, t = _tie_heavy(rng, int(rng.integers(1, 60))), _tie_heavy(rng, int(rng.integers(1, 150)))
    if seed % 5 == 0:
        t[len(t) // 2:] = t[:len(t) - len(t) // 2]          # duplicated rows: every distance tied at least twice
    k = int(rng.integers(1, 33))
    assert oracle_knn(q, t, k).tobytes() == _lexsort(q, t, k).tobytes(), f"{len(q)} x {len(t)}, k = {k}"


@pytest.mark.parametrize("name", list(KNN_CASES))
def test_oracle_k2_is_knn2(oracle, name):
    q, t = _case(name)
    assert _ref(name, 2).tobytes() == oracle.match_hamming_knn2(q, t).tobytes()


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


def _view(orbmod, a, k):
    return np.ascontiguousarray(a).view(orbmod.DMATCH_DTYPE).reshape(a.shape[:-2] + (k,))


def _set_ref(q, t, k):
    return padded(len(q), k) if len(t) == 0 else oracle_knn(q, t, k)


def _device_knn(orbmod, ctx, q, trains, counts, k):
    """orbx_match_hamming_device_knn on device copies -> [nsets, nq, k] records."""
    import torch
    nsets, stride = trains.shape[0], trains.shape[1]
    dq, dt = torch.from_numpy(np.ascontiguousarray(q)).cuda(), torch.from_numpy(np.ascontiguousarray(trains)).cuda()
    dn = torch.tensor(counts, dtype=torch.int32, device="cuda")
    out = torch.full((nsets, len(q), k, 4), SENTINEL, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device_knn(dq.data_ptr(), len(q), dt.data_ptr(), stride, dn.data_ptr(), nsets, k, out.data_ptr())
    ctx.synchronize()
    return _view(orbmod, out.cpu().numpy(), k)


def _pairwise_knn(orbmod, ctx, dq, qstride, dqc, dt, tstride, dtc, npairs, k):
    """orbx_match_hamming_device_pairwise_knn into a sentinel-filled [npairs, qstride, k] buffer -> raw int32 [.., 4]."""
    import torch
    out = torch.full((npairs, qstride, k, 4), SENTINEL, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device_pairwise_knn(dq, qstride, dqc, dt, tstride, dtc, npairs, k, out.data_ptr())
    ctx.synchronize()
    return out.cpu().numpy()


def _check_pairs(orbmod, raw, qs, qc, ts, tc, k, what):
    got = _view(orbmod, raw, k)
    qstride, tstride = qs.shape[1], ts.shape[1]
    for p in range(len(qc)):
        nq, nt = min(max(int(qc[p]), 0), qstride), min(max(int(tc[p]), 0), tstride)
        w = f"{what}: pair {p} ({nq} x {nt}), k = {k}"
        assert got[p, :nq].tobytes() == _set_ref(qs[p, :nq], ts[p, :nt], k).tobytes(), w
        assert (raw[p, nq:] == SENTINEL).all(), w + ": slots past the query count"


@pytest.mark.gpu
@pytest.mark.parametrize("k", HOST_KS)
@pytest.mark.parametrize("name", list(KNN_CASES))
def test_host_knn(orbmod, ctx, oracle, name, k):
    q, t = _case(name)
    got = ctx.knn_match(q, t, k)
    assert got.shape == (len(q), k)
    assert got.tobytes() == _ref(name, k).tobytes()


@pytest.mark.gpu
def test_host_knn_short_and_empty_train(orbmod, ctx, oracle):
    rng = np.random.default_rng(4)
    q = _tie_heavy(rng, 300)
    for nt in (1, 2, 3, 7):
        t = _tie_heavy(rng, nt)
        for k in (3, 8, 32):
            assert ctx.knn_match(q, t, k).tobytes() == oracle_knn(q, t, k).tobytes(), f"nt = {nt}, k = {k}"
    assert ctx.knn_match(q, np.zeros((0, 32), np.uint8), 5).shape == (0, 5)
    assert ctx.knn_match(np.zeros((0, 32), np.uint8), q, 5).shape == (0, 5)


@pytest.mark.gpu
@pytest.mark.parametrize("k", (3, 8, 17, 32))
def test_device_ragged_sets(orbmod, ctx, oracle, k):
    """200 sets (more than one CTA per SM: each CTA walks several sets) of ragged sizes: empty, one row, a count past the
    stride and a negative one; 300 query rows (two query tiles)."""
    rng = np.random.default_rng(20 + k)
    nsets, stride, nq = 200, 250, 300
    trains = _tie_heavy(rng, nsets * stride).reshape(nsets, stride, 32)
    counts = [0, 1, 400, -3, 97, 250, 2] + [int(x) for x in rng.integers(0, 251, nsets - 7)]
    q = _tie_heavy(rng, nq)
    got = _device_knn(orbmod, ctx, q, trains, counts, k)
    for s in range(nsets):
        n = min(max(counts[s], 0), stride)
        assert got[s].tobytes() == _set_ref(q, trains[s, :n], k).tobytes(), f"set {s} ({n} rows)"


@pytest.mark.gpu
@pytest.mark.parametrize("k", (3, 9, 16, 32))
def test_pairwise_ragged(orbmod, ctx, oracle, k):
    import torch
    from test_match_pairwise import make_pairs
    rng = np.random.default_rng(40 + k)
    npairs, qstride, tstride = 160, 300, 300
    qc = [0, 1, 255, 256, 257, 300, 900, -4] + [int(x) for x in rng.integers(0, 301, npairs - 8)]
    tc = [5, 0, 1, 96, 97, 193, 300, 1000] + [int(x) for x in rng.integers(-2, 301, npairs - 8)]
    qs, ts = make_pairs(50 + k, qc, tc, qstride, tstride)
    dq, dt = torch.from_numpy(qs).cuda(), torch.from_numpy(ts).cuda()
    dqc, dtc = torch.tensor(qc, dtype=torch.int32, device="cuda"), torch.tensor(tc, dtype=torch.int32, device="cuda")
    raw = _pairwise_knn(orbmod, ctx, dq.data_ptr(), qstride, dqc.data_ptr(), dt.data_ptr(), tstride, dtc.data_ptr(), npairs, k)
    _check_pairs(orbmod, raw, qs, qc, ts, tc, k, "pairwise")


@pytest.mark.gpu
def test_frame_to_frame_on_extraction_output(orbmod, oracle):
    """Frame i against frame i + 1 straight out of orbx_detect_and_compute_device, pairwise, and frame 0's descriptors
    against every frame as a ragged batch."""
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
    for k in (4, 12):
        raw = _pairwise_knn(orbmod, c, d_d.data_ptr(), cap, d_n.data_ptr(), d_d.data_ptr() + cap * 32, cap, d_n.data_ptr() + 4, b - 1, k)
        _check_pairs(orbmod, raw, desc[:-1], list(n[:-1]), desc[1:], list(n[1:]), k, "frame-to-frame")
    got = _device_knn(orbmod, c, desc[0, :n[0]], desc, list(n), 6)
    for s in range(b):
        assert got[s].tobytes() == oracle_knn(desc[0, :n[0]], desc[s, :n[s]], 6).tobytes(), f"frame {s}"
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", (3, 8, 16, 32))
def test_insert_heavy(orbmod, ctx, oracle, k):
    """Every column enters the list: identical query rows against train rows ordered by decreasing distance (each row
    closer than all before it); and all-equal rows, where every distance ties and the lowest indices must win."""
    nt = 1000
    bits = np.zeros((nt, 256), np.uint8)
    for j in range(nt):
        bits[j, :256 - (j * 256) // nt] = 1                 # distance to the zero row: non-increasing in j
    t = np.packbits(bits, axis=1)
    q = np.zeros((300, 32), np.uint8)
    assert ctx.knn_match(q, t, k).tobytes() == oracle_knn(q, t, k).tobytes()
    same = np.full((700, 32), 0x5A, np.uint8)
    got = ctx.knn_match(same[:260], same, k)
    assert got.tobytes() == oracle_knn(same[:260], same, k).tobytes()
    assert (got["trainIdx"] == np.arange(k)[None, :]).all()
    got = _device_knn(orbmod, ctx, q, np.stack([t, t[::-1].copy()]), [nt, nt], k)
    assert got[0].tobytes() == oracle_knn(q, t, k).tobytes() and got[1].tobytes() == oracle_knn(q, t[::-1], k).tobytes()


@pytest.mark.gpu
def test_topk_k2_equals_knn2_kernels(orbmod, ctx, oracle):
    """The top-k kernel at k = 2 (device forms) against the knn2 kernels' (best, second) on the same device inputs."""
    import torch
    from test_match_pairwise import make_pairs
    rng = np.random.default_rng(61)
    nsets, stride, nq = 40, 500, 700                        # (the knn2 call takes the CTA-pair kernel here)
    trains = _tie_heavy(rng, nsets * stride).reshape(nsets, stride, 32)
    counts = [0, 1, 2, 500, 97] + [int(x) for x in rng.integers(0, 501, nsets - 5)]
    q = _tie_heavy(rng, nq)
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(trains).cuda()
    dn = torch.tensor(counts, dtype=torch.int32, device="cuda")
    best = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
    second = torch.zeros_like(best)
    ctx.match_device_ragged(dq.data_ptr(), nq, dt.data_ptr(), stride, dn.data_ptr(), nsets, best.data_ptr(), second.data_ptr())
    ctx.synchronize()
    got = _device_knn(orbmod, ctx, q, trains, counts, 2)
    knn2 = np.stack([best.cpu().numpy(), second.cpu().numpy()], 2)
    assert got.tobytes() == _view(orbmod, knn2, 2).tobytes()
    qc, tc = [700, 0, 1, 256, 699, 300], [500, 7, 0, 1, 2, 480]
    qs, ts = make_pairs(62, qc, tc, 700, 500)
    dqs, dts = torch.from_numpy(qs).cuda(), torch.from_numpy(ts).cuda()
    dqc, dtc = torch.tensor(qc, dtype=torch.int32, device="cuda"), torch.tensor(tc, dtype=torch.int32, device="cuda")
    b = torch.full((6, 700, 4), SENTINEL, dtype=torch.int32, device="cuda")
    s2 = torch.full_like(b, SENTINEL)
    ctx.match_device_pairwise(dqs.data_ptr(), 700, dqc.data_ptr(), dts.data_ptr(), 500, dtc.data_ptr(), 6, b.data_ptr(), s2.data_ptr())
    ctx.synchronize()
    raw = _pairwise_knn(orbmod, ctx, dqs.data_ptr(), 700, dqc.data_ptr(), dts.data_ptr(), 500, dtc.data_ptr(), 6, 2)
    assert raw.tobytes() == np.stack([b.cpu().numpy(), s2.cpu().numpy()], 2).tobytes()


@pytest.mark.gpu
def test_argument_errors(orbmod, ctx):
    import torch
    lib, h = ctx.lib, ctx.h
    d = torch.zeros(4096, dtype=torch.int32, device="cuda"); p = d.data_ptr()
    q = np.zeros((4, 32), np.uint8); out = np.zeros((4, 40), orbmod.DMATCH_DTYPE)
    n = orbmod.C.c_int(0)
    host = lambda k, nt=4: lib.orbx_match_hamming_knn(h, orbmod._ptr(q), 4, orbmod._ptr(q), nt, k, orbmod._ptr(out), orbmod.C.byref(n))  # noqa: E731
    assert host(3) == orbmod.OK and n.value == 4
    assert host(0) == orbmod.E_ARG and host(-1) == orbmod.E_ARG and host(33) == orbmod.E_UNSUPPORTED
    assert host(3, nt=-1) == orbmod.E_ARG
    assert lib.orbx_match_hamming_knn(h, None, 4, orbmod._ptr(q), 4, 3, orbmod._ptr(out), orbmod.C.byref(n)) == orbmod.E_ARG
    assert lib.orbx_match_hamming_knn(h, orbmod._ptr(q), 4, orbmod._ptr(q), 4, 3, None, orbmod.C.byref(n)) == orbmod.E_ARG
    # device ragged: d_query, nq, d_train, stride, counts, nsets, k, out
    ok = [p, 1, p, 1, p, 1, 3, p]

    def dev(**kw):
        return lib.orbx_match_hamming_device_knn(h, *[kw.get(f"a{i}", v) for i, v in enumerate(ok)])
    assert dev() == orbmod.OK
    for i in (0, 2, 4, 7):
        assert dev(**{f"a{i}": None}) == orbmod.E_ARG, f"null argument {i}"
    for i in (1, 3, 5):
        assert dev(**{f"a{i}": -1}) == orbmod.E_ARG, f"negative size {i}"
    assert dev(a5=65536) == orbmod.E_ARG and dev(a6=0) == orbmod.E_ARG and dev(a6=33) == orbmod.E_UNSUPPORTED
    assert dev(a3=1 << 20) == orbmod.E_UNSUPPORTED
    assert dev(a5=0) == orbmod.OK and dev(a1=0) == orbmod.OK and dev(a3=0) == orbmod.OK
    # device pairwise: d_query, qstride, qcounts, d_train, tstride, tcounts, npairs, k, out
    ok2 = [p, 1, p, p, 1, p, 1, 3, p]

    def pw(**kw):
        return lib.orbx_match_hamming_device_pairwise_knn(h, *[kw.get(f"a{i}", v) for i, v in enumerate(ok2)])
    assert pw() == orbmod.OK
    for i in (0, 2, 3, 5, 8):
        assert pw(**{f"a{i}": None}) == orbmod.E_ARG, f"null argument {i}"
    for i in (1, 4, 6):
        assert pw(**{f"a{i}": -1}) == orbmod.E_ARG, f"negative size {i}"
    assert pw(a6=65536) == orbmod.E_ARG and pw(a7=0) == orbmod.E_ARG and pw(a7=33) == orbmod.E_UNSUPPORTED
    assert pw(a1=1 << 20) == orbmod.E_UNSUPPORTED and pw(a4=1 << 20) == orbmod.E_UNSUPPORTED
    assert pw(a6=0) == orbmod.OK and pw(a1=0) == orbmod.OK and pw(a4=0) == orbmod.OK
    # empty sizes with null pointers: the host and ragged forms return first, the pairwise one checks its pointers first
    assert lib.orbx_match_hamming_knn(h, None, 0, None, 4, 3, None, orbmod.C.byref(n)) == orbmod.OK and n.value == 0
    assert dev(a1=0, a0=None, a7=None) == orbmod.OK
    assert pw(a6=0, a8=None) == orbmod.E_ARG
    ctx.synchronize()
    bf = orbmod.BFMatcher()
    for k, code in ((0, orbmod.E_ARG), (33, orbmod.E_UNSUPPORTED)):
        with pytest.raises(orbmod.OrbxError) as e:
            bf.knnMatch(q, q, k=k)
        assert e.value.code == code
    with pytest.raises(orbmod.OrbxError) as e:
        orbmod.BFMatcher(crossCheck=True).knnMatch(q, q, k=2)
    assert e.value.code == orbmod.E_UNSUPPORTED


@pytest.mark.gpu
def test_plain_and_knn2_unchanged_around_a_knn_call(orbmod, ctx, oracle):
    q, t = _case("real_700x2000")
    before = (ctx.match(q, t), ctx.knn_match2(q, t))
    for k in (3, 32):
        ctx.knn_match(q, t, k)
    after = (ctx.match(q, t), ctx.knn_match2(q, t))
    for a, b in zip(before, after):
        assert a.tobytes() == b.tobytes()
    assert before[0].tobytes() == oracle.match_hamming(q, t).tobytes()
    assert before[1].tobytes() == oracle.match_hamming_knn2(q, t).tobytes()
    assert ctx.knn_match(q, t, 1).tobytes() == before[0].reshape(-1, 1).tobytes()
    assert ctx.knn_match(q, t, 2).tobytes() == before[1].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["iid_1000x500", "ties_257x300", "ragged_3x131", "ragged_129x1", "live_1500x2000"])
def test_bfmatcher_vs_cv2(orbmod, name):
    cv2 = pytest.importorskip("cv2")
    q, t = _case(name)
    bf, ours = cv2.BFMatcher(cv2.NORM_HAMMING), orbmod.BFMatcher()
    for k in (1, 2, 3, 7, 32):
        got = ours.knnMatch(q, t, k=k)
        assert got.dtype == orbmod.DMATCH_DTYPE and got.shape == (len(q), k)
        assert got.tobytes() == cv2_knn_to_padded(bf.knnMatch(q, t, k=k), k).tobytes(), f"k = {k}"
    # crossCheck, k = 1: [mutual pair] or [] per query -> one record, trainIdx = -1 for []
    lists = cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True).knnMatch(q, t, k=1)
    assert len(lists) == len(q) and all(len(m) <= 1 for m in lists)
    got = orbmod.BFMatcher(crossCheck=True).knnMatch(q, t, k=1)
    assert got.tobytes() == cv2_knn_to_padded(lists, 1).tobytes()
