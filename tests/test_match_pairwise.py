"""Pairwise batched Hamming matching (orbx_match_hamming_device_pairwise[_crosscheck]): pair p matches its own query set
against its own train set, all pairs in one launch.  Per pair the result is BFMatcher(NORM_HAMMING).match, knnMatch(k=2)
or the crossCheck match of that pair's rows.  CPU: the per-pair reference used below against live cv2 on seeded ragged
pairs.  GPU (-m gpu): every pair bit for bit against that reference, output buffers pre-filled with a sentinel that the
slots past each pair's query count must keep."""

import numpy as np
import pytest

from oracle import oracle as O
from xcheck_cases import oracle_crosscheck

MODES = ("plain", "knn2", "xchk")
SENTINEL = -7


def _no_match(nq):
    r = np.zeros(nq, O.MATCH_DTYPE)
    r["queryIdx"], r["trainIdx"] = np.arange(nq), -1
    return r


def ref_pair(q, t, mode):
    """The per-pair reference: the C oracle on the pair's own rows.  plain -> best[nq]; knn2 -> (best[nq], second[nq]);
    xchk -> the mutual pairs.  An empty train set gives trainIdx = -1, distance 0 records (no pairs for xchk), and a
    one-row train set a second record with trainIdx = -1, as the ragged device matcher does."""
    nq, nt = len(q), len(t)
    if mode == "xchk":
        return oracle_crosscheck(q, t)
    if nt == 0:
        return _no_match(nq) if mode == "plain" else (_no_match(nq), _no_match(nq))
    if mode == "plain":
        return O.match_hamming(q, t)
    k = O.match_hamming_knn2(q, t)
    return k[:, 0].copy(), (k[:, 1].copy() if nt >= 2 else _no_match(nq))


def make_pairs(seed, qcounts, tcounts, qstride, tstride):
    """[P][stride][32] query and train sets with these (raw) counts: noisy copies of the pair's train rows, tie-heavy
    sets, duplicated rows.  Rows past a set's count hold other data that must never be read."""
    rng = np.random.default_rng(seed)
    npairs = len(qcounts)
    qs = rng.integers(0, 256, (npairs, qstride, 32), dtype=np.uint8)
    ts = rng.integers(0, 256, (npairs, tstride, 32), dtype=np.uint8)
    for p in range(npairs):
        nq, nt = min(max(qcounts[p], 0), qstride), min(max(tcounts[p], 0), tstride)
        if p % 3 == 0:                                   # tie-heavy: few distinct values per byte
            qs[p, :nq] = rng.integers(0, 4, (nq, 32)); ts[p, :nt] = rng.integers(0, 4, (nt, 32))
        elif nt > 0 and nq > 0:                          # true matches: flipped copies of train rows
            src = ts[p, rng.integers(0, nt, nq)]
            bits = np.unpackbits(src, axis=1) ^ (rng.random((nq, 256)) < 0.1).astype(np.uint8)
            qs[p, :nq] = np.packbits(bits, axis=1)
        if nt > 2:
            ts[p, nt - 1] = ts[p, nt // 2]               # duplicated train row (also the padded copies' source)
        if nq > 2:
            qs[p, nq - 1] = qs[p, 0]                     # duplicated query row
    return qs, ts


def _clamp(n, stride):
    return min(max(int(n), 0), stride)


# ---- CPU: the reference against live cv2 -----------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(6))
def test_reference_vs_live_cv2(oracle, seed):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(seed)
    qc = [0, 1, 1, 40, 0, 130, 2] + [int(x) for x in rng.integers(0, 200, 5)]
    tc = [5, 0, 1, 1, 0, 97, 130] + [int(x) for x in rng.integers(0, 200, 5)]
    qs, ts = make_pairs(100 + seed, qc, tc, 200, 200)
    bf, bfx = cv2.BFMatcher(cv2.NORM_HAMMING), cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True)
    for p in range(len(qc)):
        q, t = qs[p, :qc[p]], ts[p, :tc[p]]
        what = f"pair {p} ({len(q)} x {len(t)})"
        if len(t) == 0:                                  # cv2 has no result there; the library's is the ragged matcher's
            assert ref_pair(q, t, "plain").tobytes() == _no_match(len(q)).tobytes()
            assert len(ref_pair(q, t, "xchk")) == 0
            continue
        assert ref_pair(q, t, "plain").tobytes() == O.cv2_matches_to_array(bf.match(q, t)).tobytes(), what
        assert ref_pair(q, t, "xchk").tobytes() == O.cv2_matches_to_array(bfx.match(q, t)).tobytes(), what
        best, second = ref_pair(q, t, "knn2")
        knn = bf.knnMatch(q, t, k=2)
        assert best.tobytes() == O.cv2_matches_to_array([m[0] for m in knn]).tobytes(), what
        if len(t) >= 2:
            assert second.tobytes() == O.cv2_matches_to_array([m[1] for m in knn]).tobytes(), what
        else:
            assert all(len(m) == 1 for m in knn) and (second["trainIdx"] == -1).all(), what


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def orbmod():
    from rgbd_visualodometry_b200 import orb
    return orb


def _run(orbmod, ctx, mode, dq, qstride, dqc, dt, tstride, dtc, npairs):
    """One pairwise call on device tensors -> raw int32 outputs ([P, qstride, 4] best (and second), n_out for xchk)."""
    import torch
    best = torch.full((npairs, qstride, 4), SENTINEL, dtype=torch.int32, device="cuda")
    second = torch.full_like(best, SENTINEL) if mode == "knn2" else None
    nout = torch.full((npairs,), SENTINEL, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    if mode == "xchk":
        ctx.match_device_pairwise_crosscheck(dq, qstride, dqc, dt, tstride, dtc, npairs, best.data_ptr(), nout.data_ptr())
    else:
        ctx.match_device_pairwise(dq, qstride, dqc, dt, tstride, dtc, npairs, best.data_ptr(), second.data_ptr() if second is not None else 0)
    ctx.synchronize()
    return best.cpu().numpy(), (second.cpu().numpy() if second is not None else None), nout.cpu().numpy()


def _check(orbmod, mode, out, qs, qc, ts, tc, what):
    best, second, nout = out
    qstride, tstride = qs.shape[1], ts.shape[1]
    view = lambda a: a.view(orbmod.DMATCH_DTYPE).reshape(a.shape[0], a.shape[1])   # noqa: E731
    for p in range(len(qc)):
        nq, nt = _clamp(qc[p], qstride), _clamp(tc[p], tstride)
        w = f"{what}: pair {p} ({nq} x {nt})"
        ref = ref_pair(qs[p, :nq], ts[p, :nt], mode)
        if mode == "xchk":
            assert nout[p] == len(ref), w
            assert view(best)[p, :nout[p]].tobytes() == ref.tobytes(), w
        elif mode == "plain":
            assert view(best)[p, :nq].tobytes() == ref.tobytes(), w
        else:
            assert view(best)[p, :nq].tobytes() == ref[0].tobytes(), w + " best"
            assert view(second)[p, :nq].tobytes() == ref[1].tobytes(), w + " second"
            assert (second[p, nq:] == SENTINEL).all(), w + " second: slots past the query count"
        assert (best[p, nq:] == SENTINEL).all(), w + ": slots past the query count"


def _pairwise_vs_reference(orbmod, ctx, mode, qs, qc, ts, tc, what):
    import torch
    dq, dt = torch.from_numpy(qs).cuda(), torch.from_numpy(ts).cuda()
    dqc, dtc = torch.tensor(qc, dtype=torch.int32, device="cuda"), torch.tensor(tc, dtype=torch.int32, device="cuda")
    out = _run(orbmod, ctx, mode, dq.data_ptr(), qs.shape[1], dqc.data_ptr(), dt.data_ptr(), ts.shape[1], dtc.data_ptr(), len(qc))
    _check(orbmod, mode, out, qs, qc, ts, tc, what)


def _cycle(vals, n):
    return [vals[i % len(vals)] for i in range(n)]


# Shapes choosing each launch path (the host rule, with the query stride as the row count: tiles = ceil(stride / 256),
# the CTA pair when tiles >= 2 and round_up_2(tiles) * npairs >= 148, the train-row split for plain and cross-check calls
# when tiles * npairs < 148).  Query counts include 0, 1, 255, 256, 257, counts past the stride and negative ones; train
# counts 0, 1, multiples of 96, 96k + 1, past the stride and negative.
QC = [0, 1, 255, 256, 257, 200, 300, 520, 599, 600, 5000, -4]
TC = [0, 1, 96, 97, 192, 193, 288, 400, 1000, -1]
SHAPES = {
    # 1 query tile x 150 pairs: single-CTA kernel, no split
    "single": dict(qstride=256, tstride=400, qc=_cycle(QC, 150), tc=_cycle(TC[::-1], 150)),
    # 3 query tiles x 4 pairs: single-CTA kernel with the train rows split (plain, xchk) across CTAs
    "split": dict(qstride=600, tstride=2000, qc=[257, 1, 0, 5000], tc=[1921, 0, 1, 2000]),
    # 3 -> 4 query tiles x 40 pairs: CTA pairs; count 200 leaves the first cluster's second tile empty, 520 the second's
    "pair": dict(qstride=600, tstride=400, qc=_cycle(QC, 40), tc=_cycle(TC, 40)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("mode", MODES)
def test_ragged_pairs(orbmod, oracle, mode, shape):
    s = SHAPES[shape]
    qs, ts = make_pairs(10 * MODES.index(mode) + list(SHAPES).index(shape), s["qc"], s["tc"], s["qstride"], s["tstride"])
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    n0 = ctx.launch_count
    _pairwise_vs_reference(orbmod, ctx, mode, qs, s["qc"], ts, s["tc"], f"{mode} {shape}")
    # launches: keys init + matcher + finalize when split; + column keys init + compaction for xchk
    split = shape == "split" and mode != "knn2"
    assert ctx.launch_count - n0 == 1 + 2 * split + 2 * (mode == "xchk")
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_self_pairs_tie_heavy(orbmod, oracle, mode):
    """Query set = train set (the same device rows): duplicated rows must go to the lowest index in both directions."""
    import torch
    npairs, stride = 8, 700
    rng = np.random.default_rng(9)
    sets = rng.integers(0, 3, (npairs, stride, 32)).astype(np.uint8)
    sets[:, 400:500] = sets[:, 100:200]
    counts = [700, 650, 1, 2, 300, 513, 0, 699]
    d = torch.from_numpy(sets).cuda()
    dc = torch.tensor(counts, dtype=torch.int32, device="cuda")
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    out = _run(orbmod, ctx, mode, d.data_ptr(), stride, dc.data_ptr(), d.data_ptr(), stride, dc.data_ptr(), npairs)
    _check(orbmod, mode, out, sets, counts, sets, counts, f"self {mode}")
    got = out[0][0].view(orbmod.DMATCH_DTYPE).reshape(-1)
    if mode != "xchk":                                   # row 400 + i duplicates row 100 + i: its own match is the first copy
        assert (got["trainIdx"][400:500] <= got["queryIdx"][400:500]).all() and (got["trainIdx"][100:200] <= 199).all()
    else:
        assert not np.isin(np.arange(400, 500), got["queryIdx"][:out[2][0]]).any()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_many_small_pairs(orbmod, oracle, mode):
    rng = np.random.default_rng(11)
    npairs = 1200
    qc, tc = [int(x) for x in rng.integers(0, 65, npairs)], [int(x) for x in rng.integers(0, 65, npairs)]
    qs, ts = make_pairs(12, qc, tc, 64, 64)
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    _pairwise_vs_reference(orbmod, ctx, mode, qs, qc, ts, tc, f"small {mode}")
    ctx.close()


@pytest.mark.gpu
def test_frame_to_frame_on_extraction_output(orbmod, oracle):
    """Frame i against frame i + 1 straight out of orbx_detect_and_compute_device: d_query = desc, d_train = desc + cap * 32,
    counts and counts + 1, npairs = batch - 1."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_sequence
    b, cap = 6, 2048
    frames = np.stack([f for f, _ in synth_sequence(480, 640, b, 3)])
    ctx = orbmod.Context(1000, 1.2, 8, 640, 480, b)
    d_in = torch.from_numpy(frames).cuda()
    d_k = torch.zeros((b, cap, 7), dtype=torch.float32, device="cuda")
    d_d = torch.zeros((b, cap, 32), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(b, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.detect_and_compute_device(d_in.data_ptr(), b, 640, 480, 1920, 480 * 1920, 3, d_k.data_ptr(), d_d.data_ptr(), cap, d_n.data_ptr())
    ctx.synchronize()
    desc, n = d_d.cpu().numpy(), d_n.cpu().numpy()
    assert (n > 500).all()
    for mode in MODES:
        out = _run(orbmod, ctx, mode, d_d.data_ptr(), cap, d_n.data_ptr(), d_d.data_ptr() + cap * 32, cap, d_n.data_ptr() + 4, b - 1)
        _check(orbmod, mode, out, desc[:-1], list(n[:-1]), desc[1:], list(n[1:]), f"frame-to-frame {mode}")
        if mode == "xchk":
            assert (out[2] > 100).all()
    ctx.close()


@pytest.mark.gpu
def test_argument_errors(orbmod):
    import torch
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    lib, h = ctx.lib, ctx.h
    d = torch.zeros(64, dtype=torch.int32, device="cuda"); p = d.data_ptr()
    for fn in (lib.orbx_match_hamming_device_pairwise, lib.orbx_match_hamming_device_pairwise_crosscheck):
        xc = fn is lib.orbx_match_hamming_device_pairwise_crosscheck
        ok = [p, 1, p, p, 1, p, 1, p, p]               # d_query, qstride, qcounts, d_train, tstride, tcounts, npairs, out, second / n_out

        def call(**kw):
            return fn(h, *[kw.get(f"a{i}", v) for i, v in enumerate(ok)])
        assert call() == orbmod.OK
        for i in (0, 2, 3, 5, 7) + ((8,) if xc else ()):
            assert call(**{f"a{i}": None}) == orbmod.E_ARG, f"null argument {i}"
        for i in (1, 4, 6):
            assert call(**{f"a{i}": -1}) == orbmod.E_ARG, f"negative size {i}"
        assert call(a6=65536) == orbmod.E_ARG
        assert call(a1=1 << 20) == orbmod.E_UNSUPPORTED and call(a4=1 << 20) == orbmod.E_UNSUPPORTED
        assert call(a6=0) == orbmod.OK
        assert call(a1=0) == orbmod.OK and call(a4=0) == orbmod.OK
    # cross-check with a stride of 0: no launch, every pair's count zeroed
    nout = torch.full((5,), SENTINEL, dtype=torch.int32, device="cuda")
    n0 = ctx.launch_count
    assert lib.orbx_match_hamming_device_pairwise_crosscheck(h, p, 0, p, p, 4, p, 5, p, nout.data_ptr()) == orbmod.OK
    ctx.synchronize()
    assert (nout.cpu().numpy() == 0).all() and ctx.launch_count == n0
    # an empty size does not excuse a null pointer here: the pairwise forms check their pointers first
    assert lib.orbx_match_hamming_device_pairwise(h, None, 0, p, p, 1, p, 1, p, None) == orbmod.E_ARG
    assert lib.orbx_match_hamming_device_pairwise_crosscheck(h, p, 1, p, p, 0, p, 1, None, p) == orbmod.E_ARG
    # the shared-query forms return before their pointers on an empty input
    n = orbmod.C.c_int(7)
    for fn in (lib.orbx_match_hamming, lib.orbx_match_hamming_knn2):
        assert fn(h, None, 0, None, 4, None, orbmod.C.byref(n)) == orbmod.OK and n.value == 0
    assert lib.orbx_match_hamming_device(h, None, 4, None, 4, 0, None, None) == orbmod.OK
    assert lib.orbx_match_hamming_device_ragged(h, p, 4, None, 0, None, 2, None, None) == orbmod.OK
    assert lib.orbx_match_hamming_sets(h, None, 0, None, 4, None, 2, None, None) == orbmod.OK
    ctx.close()


@pytest.mark.gpu
def test_shared_map_calls_unchanged_around_a_pairwise_call(orbmod, oracle):
    """_device_ragged and _device_crosscheck (one query set shared by every train set) before and after pairwise calls on
    the same context give the same results."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    nsets, cap, nq = 5, 900, 1500
    trains = np.stack([synth_descriptors(cap, 500 + i) for i in range(nsets)])
    counts = [900, 0, 1, 385, 700]
    q = synth_map_queries(trains[0], nq, 510)
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(trains).cuda()
    dn = torch.tensor(counts, dtype=torch.int32, device="cuda")
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)

    def shared():
        best = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
        xc = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
        nx = torch.zeros(nsets, dtype=torch.int32, device="cuda")
        ctx.match_device_ragged(dq.data_ptr(), nq, dt.data_ptr(), cap, dn.data_ptr(), nsets, best.data_ptr())
        ctx.match_device_crosscheck(dq.data_ptr(), nq, dt.data_ptr(), cap, dn.data_ptr(), nsets, xc.data_ptr(), nx.data_ptr())
        ctx.synchronize()
        return best.cpu().numpy(), xc.cpu().numpy(), nx.cpu().numpy()

    before = shared()
    qs, ts = make_pairs(13, [1500, 3, 256], [900, 0, 97], 1500, 900)
    for mode in MODES:
        _pairwise_vs_reference(orbmod, ctx, mode, qs, [1500, 3, 256], ts, [900, 0, 97], f"between {mode}")
    after = shared()
    for a, b in zip(before, after):
        assert a.tobytes() == b.tobytes()
    got = before[0].view(orbmod.DMATCH_DTYPE).reshape(nsets, nq)
    for s, n in enumerate(counts):
        if n:
            assert got[s].tobytes() == oracle.match_hamming(q, trains[s, :n]).tobytes(), f"set {s}"
            xs = before[1][s, :before[2][s]].view(orbmod.DMATCH_DTYPE).reshape(-1)
            assert xs.tobytes() == oracle_crosscheck(q, trains[s, :n]).tobytes(), f"set {s} crosscheck"
    ctx.close()
