"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C-ABI of liborbx.so,
against (a) the committed cv2 golden vectors, (b) the CPU oracle on the same seeded inputs, (c) cv2 itself when
importable, and (d) size-independent properties at BASELINE.json's full sizes.

Bar: bit-exact everywhere -- keypoint records (all 7 cv::KeyPoint fields, order included), descriptors, match
indices and distances.  (north_star allows 1e-4 relative on Harris responses and angles; the restatement is in
fact bit-exact, so the tests assert equality and report the tolerance only in the failure message.)"""
import os

import numpy as np
import pytest

from cases import LIVE_MATCH_CASES, MATCH_CASES, ORB_CASES, ORB_CASES_LARGE, assert_equals_stored, sha

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def orbmod():
    from rgbd_visualodometry_b200 import orb
    return orb


def _assert_kp_equal(k, d, ko, do, what):
    assert len(k) == len(ko), f"{what}: count {len(k)} vs {len(ko)}"
    for f in ko.dtype.names:
        bad = int((k[f] != ko[f]).sum())
        assert bad == 0, f"{what}: field {f} differs on {bad} keypoints (tolerance allowed by north_star: 1e-4 rel on response/angle)"
    assert np.array_equal(d, do), f"{what}: {int((d != do).any(axis=1).sum())} descriptors differ"


# Pyramid and FAST exist as two kernel families chosen by launch size (orbx_debug_force_kernels): 0 = warp-private TMA
# kernels (large launches), 1 = CTA-cooperative kernels (small launches).  Single-frame cases are run through both.
KERNELS = [0, 1]


@pytest.mark.parametrize("kernels", KERNELS)
@pytest.mark.parametrize("name", list(ORB_CASES))
def test_orb_vs_golden(orbmod, name, kernels):
    mk, n = ORB_CASES[name]
    img = mk()
    g = np.load(os.path.join(GOLD, f"orb_{name}.npz"))
    k, d = orbmod.ORB_create(n, 1.2, 8, kernels=kernels).detectAndCompute(img, None)
    gd = g["descriptors"]
    if len(g["keypoints"]) == 0:
        assert len(k) == 0 and d is None          # cv2 returns ((), None)
        return
    _assert_kp_equal(k, d, g["keypoints"], gd, f"golden {name}")


@pytest.mark.parametrize("kernels", KERNELS)
@pytest.mark.parametrize("name", list(ORB_CASES_LARGE))
def test_orb_vs_oracle_large(orbmod, oracle, name, kernels):
    mk, n = ORB_CASES_LARGE[name]
    img = mk()
    k, d = orbmod.ORB_create(n, 1.2, 8, kernels=kernels).detectAndCompute(img, None)
    ko, do = oracle.detect_and_compute(img, n)
    _assert_kp_equal(k, d, ko, do, f"oracle {name}")


@pytest.mark.parametrize("kernels", KERNELS)
def test_orb_stages_vs_oracle(orbmod, oracle, kernels):
    """Each kernel in isolation: pyramid levels and the raster-ordered FAST+NMS lists."""
    from rgbd_visualodometry_b200.synth import synth_frame
    img = synth_frame(467, 701, 21)
    ctx = orbmod.Context(700, 1.2, 8, 701, 467, 1)
    ctx.force_kernels(kernels)
    ctx.detect_and_compute(img)
    _, _, dump = oracle.detect_and_compute(img, 700, dump=True)
    ws, hs, sc, q = ctx.level_geometry(701, 467)
    ows, ohs, osc = oracle.level_geometry(701, 467)
    assert ws.tolist() == ows and hs.tolist() == ohs and sc.tobytes() == osc.tobytes() and q.tolist() == oracle.quotas(700)
    for l in range(8):
        assert np.array_equal(ctx.debug_level(0, l, ows[l], ohs[l]), dump["levels"][l]), f"level {l}"
        x, y, s = ctx.debug_fast(0, l)
        fo = dump["fast"][l]
        assert np.array_equal(x, fo["x"]) and np.array_equal(y, fo["y"]) and np.array_equal(s, fo["response"].astype(np.int32)), f"FAST level {l}"
    ctx.close()


def test_orb_batch_and_strided(orbmod, oracle):
    """Batch of distinct frames == per-frame results; a padded row step (cv::Mat::step) is honoured."""
    from rgbd_visualodometry_b200.synth import synth_frame
    frames = [synth_frame(240, 320, 100 + i) for i in range(5)]
    ctx = orbmod.Context(300, 1.2, 8, 320, 240, 8)
    kps, desc, cnt = ctx.detect_and_compute_batch(frames)
    for i, fr in enumerate(frames):
        ko, do = oracle.detect_and_compute(fr, 300)
        _assert_kp_equal(kps[i, :cnt[i]], desc[i, :cnt[i]], ko, do, f"batch frame {i}")
    padded = np.zeros((240, 333, 3), np.uint8)
    padded[:, :320] = frames[0]
    view = padded[:, :320]                                   # non-contiguous rows: step = 999 bytes
    import ctypes as C
    k = np.zeros(600, orbmod.KP_DTYPE); d = np.zeros((600, 32), np.uint8); n = C.c_int(0)
    rc = ctx.lib.orbx_detect_and_compute(ctx.h, view.ctypes.data, 320, 240, view.strides[0], 3, k.ctypes.data, d.ctypes.data, 600, C.byref(n))
    assert rc == 0
    ko, do = oracle.detect_and_compute(frames[0], 300)
    _assert_kp_equal(k[:n.value], d[:n.value], ko, do, "strided")
    ctx.close()


def test_orb_capacity_and_empty(orbmod):
    import ctypes as C
    from rgbd_visualodometry_b200.synth import synth_frame
    ctx = orbmod.Context(500, 1.2, 8, 640, 480, 1)
    img = synth_frame(480, 640, 0)
    k = np.zeros(100, orbmod.KP_DTYPE); d = np.zeros((100, 32), np.uint8); n = C.c_int(0)
    rc = ctx.lib.orbx_detect_and_compute(ctx.h, img.ctypes.data, 640, 480, 1920, 3, k.ctypes.data, d.ctypes.data, 100, C.byref(n))
    assert rc == orbmod.E_CAPACITY and n.value == 500            # never truncates silently: reports the need
    rc = ctx.lib.orbx_detect_and_compute(ctx.h, img.ctypes.data, 0, 0, 0, 3, k.ctypes.data, d.ctypes.data, 100, C.byref(n))
    assert rc == 0 and n.value == 0                              # empty image: silent, no keypoints
    rc = ctx.lib.orbx_detect_and_compute(ctx.h, img.ctypes.data, 641, 480, 1923, 3, k.ctypes.data, d.ctypes.data, 100, C.byref(n))
    assert rc == orbmod.E_ARG
    rc = ctx.lib.orbx_detect_and_compute(ctx.h, img.ctypes.data, 640, 480, 1280, 2, k.ctypes.data, d.ctypes.data, 100, C.byref(n))
    assert rc == orbmod.E_UNSUPPORTED
    assert orbmod.ORB_create(500).detectAndCompute(np.zeros((0, 0, 3), np.uint8))[1] is None
    ctx.close()


def test_orb_gray_equals_bgr(orbmod):
    """ORB(BGR) == ORB(gray(BGR)) (SURVEY probe E2) -- uses the library's own level 0 as the gray image."""
    from rgbd_visualodometry_b200.synth import synth_frame
    img = synth_frame(300, 400, 77)
    ctx = orbmod.Context(400, 1.2, 8, 400, 300, 1)
    k1, d1 = ctx.detect_and_compute(img)
    g = ctx.debug_level(0, 0, 400, 300)
    k2, d2 = ctx.detect_and_compute(g)
    assert k1.tobytes() == k2.tobytes() and np.array_equal(d1, d2)
    ctx.close()


@pytest.mark.parametrize("name", list(MATCH_CASES))
def test_match_vs_golden(orbmod, name):
    mq, mt = MATCH_CASES[name]
    q, t = mq(), mt()
    g = np.load(os.path.join(GOLD, f"match_{name}.npz"))
    bf = orbmod.BFMatcher(orbmod.NORM_HAMMING)
    assert bf.match(q, t).tobytes() == g["match"].tobytes()
    k2 = bf.knnMatch(q, t, k=2)
    if len(t) >= 2:
        assert k2.tobytes() == g["knn2"].tobytes()
    else:
        assert np.array_equal(k2["trainIdx"][:, 0], g["knn2"]["trainIdx"][:, 0]) and (k2["trainIdx"][:, 1] == -1).all()


def test_match_empty(orbmod):
    bf = orbmod.BFMatcher(orbmod.NORM_HAMMING)
    e = np.zeros((0, 32), np.uint8); t = np.zeros((4, 32), np.uint8)
    assert len(bf.match(e, t)) == 0 and len(bf.match(t, e)) == 0


@pytest.mark.parametrize("m", [1000, 5000, 20000, 100000])
def test_match_sweep_vs_oracle(orbmod, oracle, m):
    """BASELINE config 3: map size sweep vs 2k frame descriptors, 'realistic' distribution (true matches + ties)."""
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    t = synth_descriptors(2000, 40)
    q = synth_map_queries(t, m, 41)
    got = orbmod.BFMatcher(orbmod.NORM_HAMMING).match(q, t)
    if m <= 20000:
        assert got.tobytes() == oracle.match_hamming(q, t).tobytes()
    else:
        # full size: size-independent properties + an oracle check on a sample of rows
        assert np.array_equal(got["queryIdx"], np.arange(m)) and (got["imgIdx"] == 0).all()
        rows = np.random.default_rng(0).choice(m, 4000, replace=False)
        ref = oracle.match_hamming(q[rows], t)
        assert np.array_equal(got["trainIdx"][rows], ref["trainIdx"]) and np.array_equal(got["distance"][rows], ref["distance"])
        x = np.bitwise_xor(q, t[got["trainIdx"]])
        assert np.array_equal(np.unpackbits(x, axis=1).sum(1).astype(np.float32), got["distance"])   # distance is the true Hamming of the pair


def test_match_properties(orbmod):
    """Self-match: every row's nearest neighbour in its own set is itself at distance 0; duplicated rows tie to the first."""
    from rgbd_visualodometry_b200.synth import synth_descriptors
    t = synth_descriptors(777, 9)
    t[500:600] = t[100:200]
    m = orbmod.BFMatcher(orbmod.NORM_HAMMING).match(t, t)
    exp = np.arange(777); exp[500:600] = np.arange(100, 200)
    assert np.array_equal(m["trainIdx"], exp) and (m["distance"] == 0).all()


def test_match_device_batched(orbmod, oracle):
    """Device-resident, batched over several frames' train sets sharing one map (BASELINE config 3, batched variant)."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    nsets, nt, nq = 3, 700, 1300
    trains = np.stack([synth_descriptors(nt, 60 + i) for i in range(nsets)])
    q = synth_map_queries(trains[0], nq, 70)
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    dq = torch.from_numpy(q).cuda(); dt = torch.from_numpy(trains).cuda()
    best = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device(dq.data_ptr(), nq, dt.data_ptr(), nt, nsets, best.data_ptr())
    ctx.synchronize()
    got = best.cpu().numpy().view(orbmod.DMATCH_DTYPE).reshape(nsets, nq)
    for s in range(nsets):
        assert got[s].tobytes() == oracle.match_hamming(q, trains[s]).tobytes(), f"set {s}"
    ctx.close()


def test_match_pair_kernel_ragged_sets(orbmod, oracle):
    """Enough (query tile, set) pairs to select the CTA-pair kernel (tcgen05 cta_group::2): ragged train sets whose sizes sit on
    every tile / chunk boundary (0, 1, 15..17, 31..33, 47..49, 63..65, 95..97, 191..193, full), an odd number of query tiles
    (the last pair's peer CTA has no rows) and duplicated rows across the boundary of the padded last tile (ties -> lowest index)."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    cap, nq = 300, 5 * 256 - 77                      # 5 query tiles -> padded to 6 for the pairs
    sizes = [0, 1, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64, 65, 95, 96, 97, 191, 192, 193, 255, 299, 300]
    sizes = sizes + [int(x) for x in np.random.default_rng(5).integers(0, cap + 1, 40 - len(sizes))]
    nsets = len(sizes)
    assert 6 * nsets >= 148
    trains = np.stack([synth_descriptors(cap, 900 + i) for i in range(nsets)])
    for i, n in enumerate(sizes):                    # the set's last row also appears earlier: the padded copies must not win
        if n >= 3:
            trains[i, n - 1] = trains[i, n // 2]
    q = synth_map_queries(trains[1 + int(np.argmax(sizes[1:]))], nq, 71)
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    dq = torch.from_numpy(q).cuda(); dt = torch.from_numpy(trains).cuda()
    dn = torch.tensor(sizes, dtype=torch.int32, device="cuda")
    best = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device_ragged(dq.data_ptr(), nq, dt.data_ptr(), cap, dn.data_ptr(), nsets, best.data_ptr())
    ctx.synchronize()
    got = best.cpu().numpy().view(orbmod.DMATCH_DTYPE).reshape(nsets, nq)
    for s, n in enumerate(sizes):
        if n == 0:
            assert (got[s]["trainIdx"] == -1).all(), f"empty set {s}"
        else:
            assert got[s].tobytes() == oracle.match_hamming(q, trains[s, :n]).tobytes(), f"set {s} ({n} rows)"
    ctx.close()


def _check_knn2(got_best, got_second, q, train, oracle, what):
    """knnMatch(k = 2) records of one train set against the oracle: [best, second] by (distance, index); fewer than two
    train rows -> the missing records carry trainIdx = -1."""
    n = len(train)
    if n == 0:
        assert (got_best["trainIdx"] == -1).all() and (got_second["trainIdx"] == -1).all(), f"{what}: empty set"
        return
    ref = oracle.match_hamming_knn2(q, train)
    assert got_best.tobytes() == ref[:, 0].tobytes(), f"{what}: best"
    if n >= 2:
        assert got_second.tobytes() == ref[:, 1].tobytes(), f"{what}: second"
    else:
        assert (got_second["trainIdx"] == -1).all(), f"{what}: second of a one-row set"


def test_match_pair_kernel_knn2_ragged_sets(orbmod, oracle):
    """The CTA-pair kernel WITH the fused second-minimum (k_hamming_umma2<Knn2, ...>, knnMatch k = 2): 42 ragged train sets x 1203
    queries (6 padded query tiles x 42 sets >= 148 pairs selects it), sizes on every tile / chunk boundary, the set's last row
    duplicated earlier (ties across the padded last tile -> lowest index first, the copy second)."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    cap, nq = 300, 5 * 256 - 77
    sizes = [0, 1, 2, 3, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64, 65, 95, 96, 97, 98, 191, 192, 193, 255, 299, 300]
    sizes = sizes + [int(x) for x in np.random.default_rng(6).integers(0, cap + 1, 42 - len(sizes))]
    nsets = len(sizes)
    assert 6 * nsets >= 148
    trains = np.stack([synth_descriptors(cap, 1900 + i) for i in range(nsets)])
    for i, n in enumerate(sizes):
        if n >= 3:
            trains[i, n - 1] = trains[i, n // 2]
    q = synth_map_queries(trains[1 + int(np.argmax(sizes[1:]))], nq, 72)
    q[:50] = trains[25, 150:200]                       # exact hits whose duplicate-free runner-up is a real second neighbour
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    dq = torch.from_numpy(q).cuda(); dt = torch.from_numpy(trains).cuda()
    dn = torch.tensor(sizes, dtype=torch.int32, device="cuda")
    best = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
    second = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device_ragged(dq.data_ptr(), nq, dt.data_ptr(), cap, dn.data_ptr(), nsets, best.data_ptr(), second.data_ptr())
    ctx.synchronize()
    gb = best.cpu().numpy().view(orbmod.DMATCH_DTYPE).reshape(nsets, nq)
    gs = second.cpu().numpy().view(orbmod.DMATCH_DTYPE).reshape(nsets, nq)
    for s, n in enumerate(sizes):
        _check_knn2(gb[s], gs[s], q, trains[s, :n], oracle, f"pair knn2 set {s} ({n} rows)")
    ctx.close()


def test_match_single_cta_knn2_batched(orbmod, oracle):
    """The single-CTA kernel with the fused second-minimum over SEVERAL train sets (d_second with nsets > 1): uniform sets through
    orbx_match_hamming_device and ragged ones through orbx_match_hamming_sets (host buffers)."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    nsets, nt, nq = 3, 700, 1300                        # 6 query tiles x 3 sets < 148: the single-CTA kernel
    trains = np.stack([synth_descriptors(nt, 160 + i) for i in range(nsets)])
    trains[1, 650:700] = trains[1, 100:150]             # duplicated rows: best = first copy, second = its twin at distance 0
    q = synth_map_queries(trains[1], nq, 170)
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    dq = torch.from_numpy(q).cuda(); dt = torch.from_numpy(trains).cuda()
    best = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
    second = torch.zeros((nsets, nq, 4), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device(dq.data_ptr(), nq, dt.data_ptr(), nt, nsets, best.data_ptr(), second.data_ptr())
    ctx.synchronize()
    gb = best.cpu().numpy().view(orbmod.DMATCH_DTYPE).reshape(nsets, nq)
    gs = second.cpu().numpy().view(orbmod.DMATCH_DTYPE).reshape(nsets, nq)
    for s in range(nsets):
        _check_knn2(gb[s], gs[s], q, trains[s], oracle, f"single-CTA knn2 set {s}")
    counts = np.array([700, 1, 333], np.int32)
    hb, hs = ctx.match_sets(q, trains, counts, knn2=True)
    for s in range(nsets):
        _check_knn2(hb[s], hs[s], q, trains[s, :counts[s]], oracle, f"match_sets knn2 set {s}")
    ctx.close()


def _device_batch_vs_oracle(orbmod, oracle, w, h, nfeat, distinct, batch, shapes):
    """A device-resident batch (BASELINE configs 4 / 5 shapes): `distinct` different frames repeated to `batch`, every frame's
    records compared with the oracle's result for its source frame."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_frame
    cap = 2 * nfeat
    src = [synth_frame(h, w, 7000 + i, shapes=shapes) for i in range(distinct)]
    frames = np.stack([src[i % distinct] for i in range(batch)])
    ctx = orbmod.Context(nfeat, 1.2, 8, w, h, batch)
    d_in = torch.from_numpy(frames).cuda()
    d_k = torch.zeros((batch, cap, 7), dtype=torch.float32, device="cuda")
    d_d = torch.zeros((batch, cap, 32), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(batch, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.detect_and_compute_device(d_in.data_ptr(), batch, w, h, 3 * w, 3 * w * h, 3, d_k.data_ptr(), d_d.data_ptr(), cap, d_n.data_ptr())
    ctx.synchronize()
    n = d_n.cpu().numpy(); k = d_k.cpu().numpy().view(orbmod.KP_DTYPE).reshape(batch, cap); d = d_d.cpu().numpy()
    ref = [oracle.detect_and_compute(fr, nfeat) for fr in src]
    for i in range(batch):
        ko, do = ref[i % distinct]
        _assert_kp_equal(k[i, :n[i]], d[i, :n[i]], ko, do, f"{w}x{h} device frame {i}")
    ctx.close()


def test_orb_device_batch_1080p(orbmod, oracle):
    """BASELINE config 4: 1920x1080, 2000 features, a device-resident batch of 8 distinct frames, every frame vs the oracle."""
    _device_batch_vs_oracle(orbmod, oracle, 1920, 1080, 2000, 8, 8, 300)


def test_orb_device_batch_1080p_lanes(orbmod, oracle):
    """The same geometry through the multi-stream lane split (batch >= 3 x 64): 192 frames, 12 distinct, all 192 checked."""
    _device_batch_vs_oracle(orbmod, oracle, 1920, 1080, 2000, 12, 192, 300)


def test_orb_device_batch_4k(orbmod, oracle):
    """BASELINE config 5: 3840x2160, 5000 features, a device-resident batch of 3 distinct frames, every frame vs the oracle."""
    _device_batch_vs_oracle(orbmod, oracle, 3840, 2160, 5000, 3, 3, 400)


def test_orb_device_resident_full_size(orbmod, oracle):
    """BASELINE config 2 shape: a device-resident batch of 640x480 frames, 1000 features; every frame checked."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_frame
    b, cap = 8, 2048
    frames = np.stack([synth_frame(480, 640, 300 + i) for i in range(b)])
    ctx = orbmod.Context(1000, 1.2, 8, 640, 480, b)
    d_in = torch.from_numpy(frames).cuda()
    d_k = torch.zeros((b, cap, 7), dtype=torch.float32, device="cuda")
    d_d = torch.zeros((b, cap, 32), dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(b, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.detect_and_compute_device(d_in.data_ptr(), b, 640, 480, 1920, 480 * 1920, 3, d_k.data_ptr(), d_d.data_ptr(), cap, d_n.data_ptr())
    ctx.synchronize()
    n = d_n.cpu().numpy(); k = d_k.cpu().numpy().view(orbmod.KP_DTYPE).reshape(b, cap); d = d_d.cpu().numpy()
    for i in range(b):
        ko, do = oracle.detect_and_compute(frames[i], 1000)
        _assert_kp_equal(k[i, :n[i]], d[i, :n[i]], ko, do, f"device frame {i}")
    ctx.close()


def test_frontend_pattern(orbmod, oracle):
    """BASELINE config 1: the front-end's per-frame call pattern (1 extraction + 2 matches, src/frontend.cpp:98-108)
    on a synthetic TUM-shaped sequence; map = descriptors of every 5th frame."""
    from rgbd_visualodometry_b200.synth import synth_sequence
    orb_g = orbmod.ORB_create(500, 1.2, 8)
    bf = orbmod.BFMatcher(orbmod.NORM_HAMMING)
    map_desc = None
    for i, (color, depth) in enumerate(synth_sequence(480, 640, 6, seed=3)):
        k, d = orb_g.detectAndCompute(color, None)
        ko, do = oracle.detect_and_compute(color, 500)
        _assert_kp_equal(k, d, ko, do, f"sequence frame {i}")
        if map_desc is not None:
            for _ in range(2):
                m = bf.match(map_desc, d)
                mo = oracle.match_hamming(map_desc, do)
                assert m.tobytes() == mo.tobytes()
                assert orbmod.filter_matches(m, 2.0).tobytes() == oracle.filter_matches(mo, 2.0).tobytes()
        if i % 5 == 0:
            map_desc = d if map_desc is None else np.concatenate([map_desc, d])


def test_cv2_live_if_available(orbmod):
    """Against cv2's stored results (tests/golden/, tools/make_golden_live.py) always, and cv2 live when importable."""
    try:
        import cv2
    except ImportError:
        cv2 = None
    from oracle import oracle as O
    from rgbd_visualodometry_b200.synth import synth_frame
    img = synth_frame(480, 640, 555)
    g = np.load(os.path.join(GOLD, "orb_live555_1000.npz"))
    assert sha(img) == str(g["img_sha"])
    k, d = orbmod.ORB_create(1000, 1.2, 8).detectAndCompute(img, None)
    assert_equals_stored(g, "ORB vs stored cv2", keypoints=k, descriptors=d)
    if cv2 is not None:
        kc, dc = cv2.ORB_create(1000, 1.2, 8).detectAndCompute(img, None)
        _assert_kp_equal(k, d, O.cv2_keypoints_to_array(kc), dc, "cv2 live")
    q, t = (f() for f in LIVE_MATCH_CASES["3000x2000"])
    gm = np.load(os.path.join(GOLD, "match_live_3000x2000.npz"))
    assert sha(q) == str(gm["q_sha"]) and sha(t) == str(gm["t_sha"])
    m = orbmod.BFMatcher(orbmod.NORM_HAMMING).match(q, t)
    assert_equals_stored(gm, "match vs stored cv2", match=m)
    if cv2 is not None:
        assert m.tobytes() == O.cv2_matches_to_array(cv2.BFMatcher(cv2.NORM_HAMMING).match(q, t)).tobytes()


def test_orb_4k_5000(orbmod, oracle):
    """BASELINE config 5 shape: 3840x2160, 5000 features (one frame against the oracle; the oracle itself is pinned
    to cv2 at this size by tools/check_oracle_4k.py, run in the build container)."""
    from rgbd_visualodometry_b200.synth import synth_frame
    img = synth_frame(2160, 3840, 6, shapes=400)
    k, d = orbmod.ORB_create(5000, 1.2, 8).detectAndCompute(img, None)
    ko, do = oracle.detect_and_compute(img, 5000)
    _assert_kp_equal(k, d, ko, do, "4k")


def test_orb_noise_global_workspace(orbmod, oracle):
    """Pure noise at 640x480: ~30 000 FAST survivors on level 0 -> the selection runs from the global-memory
    workspace (more candidates than the shared-memory array holds) and must still reproduce libstdc++'s order."""
    img = np.random.default_rng(11).integers(0, 256, (480, 640), dtype=np.uint8)
    k, d = orbmod.ORB_create(500, 1.2, 8).detectAndCompute(img, None)
    ko, do = oracle.detect_and_compute(img, 500)
    _assert_kp_equal(k, d, ko, do, "noise vga")


def test_orb_large_batch_lanes(orbmod, oracle):
    """A large batch is cut into frame ranges that run on their own streams: every frame checked against the oracle."""
    from rgbd_visualodometry_b200.synth import synth_frame
    b = 130
    frames = [synth_frame(150, 200, 5000 + i) for i in range(b)]
    ctx = orbmod.Context(200, 1.2, 8, 200, 150, b)
    kps, desc, cnt = ctx.detect_and_compute_batch(frames)
    for i in (0, b - 1):
        _, _, dump = oracle.detect_and_compute(frames[i], 200, dump=True)
        ws, hs, _ = oracle.level_geometry(200, 150)
        for l in range(8):
            assert np.array_equal(ctx.debug_level(i, l, ws[l], hs[l]), dump["levels"][l]), f"frame {i} level {l}"
    for i, fr in enumerate(frames):
        ko, do = oracle.detect_and_compute(fr, 200)
        _assert_kp_equal(kps[i, :cnt[i]], desc[i, :cnt[i]], ko, do, f"large batch frame {i}")
    ctx.close()


@pytest.mark.gpu
def test_fused_extract_match_batch_equals_separate_calls_and_oracle(orbmod):
    """orbx_extract_match_batch (lanes: upload -> extraction -> matching -> download per frame range) must give exactly what
    the separate drop-in calls give, and frame 0 must equal the oracle end to end."""
    from oracle import oracle as O
    from rgbd_visualodometry_b200.synth import synth_frame, synth_map_queries, synth_descriptors
    B, n = 70, 300
    frames = [synth_frame(240, 320, 4100 + i) for i in range(B)]
    frames[5] = np.full((240, 320, 3), 77, np.uint8)                       # a frame without keypoints
    ctx = orbmod.Context(n, 1.2, 8, 320, 240, B)
    k0, d0 = ctx.detect_and_compute(frames[0])
    maps = [synth_map_queries(d0, 777, 3), synth_descriptors(130, 9)]
    kps, desc, cnt, best = ctx.extract_match_batch(frames, maps)
    kps2, desc2, cnt2 = ctx.detect_and_compute_batch(frames)
    assert np.array_equal(cnt, cnt2) and cnt[5] == 0
    for i in range(B):
        assert kps[i, :cnt[i]].tobytes() == kps2[i, :cnt[i]].tobytes()
        assert np.array_equal(desc[i, :cnt[i]], desc2[i, :cnt[i]])
    for j, q in enumerate(maps):
        for i in (0, 1, 5, 17, 34, 35, 69):
            if cnt[i] == 0:
                assert (best[j][i]["trainIdx"] == -1).all()
                continue
            ref = ctx.match(q, desc[i, :cnt[i]])
            assert best[j][i].tobytes() == ref.tobytes(), (j, i)
    ko, do = O.detect_and_compute(frames[0], n)
    assert kps[0, :cnt[0]].tobytes() == ko.tobytes() and np.array_equal(desc[0, :cnt[0]], do)
    assert best[0][0].tobytes() == O.match_hamming(maps[0], do).tobytes()


@pytest.mark.parametrize("kernels", KERNELS)
@pytest.mark.parametrize("params", [(300, 1.5, 4), (400, 2.0, 3), (600, 1.1, 12), (500, 1.2, 1), (500, 1.3, 6), (250, 2.5, 2)])
def test_orb_other_scale_factors_and_level_counts(orbmod, params, kernels):
    """cv::ORB::create(nfeatures, scaleFactor, nlevels) with values other than the reference's yaml (1.2 / 8): the narrow
    and the wide pyramid kernels, 1 .. 12 levels.  Oracle == cv2 for these is pinned on the CPU side (test_oracle.py)."""
    from oracle import oracle as O
    from rgbd_visualodometry_b200.synth import synth_frame
    n, sf, nl = params
    img = synth_frame(480, 640, 31)
    k, d = orbmod.ORB_create(n, sf, nl, kernels=kernels).detectAndCompute(img, None)
    ko, do = O.detect_and_compute(img, n, sf, nl)
    _assert_kp_equal(k, d, ko, do, f"ORB({n}, {sf}, {nl})")


def test_orb_rejects_scale_factor_beyond_the_pyramid_kernels(orbmod):
    from rgbd_visualodometry_b200.synth import synth_frame
    with pytest.raises(orbmod.OrbxError) as e:
        orbmod.ORB_create(100, 3.5, 2).detectAndCompute(synth_frame(240, 320, 1), None)
    assert e.value.code == -5                                # ORBX_E_UNSUPPORTED, never a silently wrong pyramid


def test_host_buffers_pageable_registered_and_strided_agree(orbmod, oracle):
    """The host-buffer entry points give the same bytes whether the caller's buffers are pageable (staged through the
    library's pinned memory by its copier threads: the reference's cv::Mat / std::vector case), page-locked with
    orbx_host_register (copied from / into directly), or pageable with a padded row step -- with and without maps,
    for a batch large enough to run several frame-range lanes, a partial last lane included."""
    from rgbd_visualodometry_b200.synth import synth_frame, synth_descriptors
    B, n, cap = 37, 300, 400
    base = [synth_frame(240, 320, 900 + i) for i in range(6)]
    frames = np.stack([np.roll(base[i % 6], 7 * (i // 6), axis=1) for i in range(B)])
    maps = [synth_descriptors(700, 11), synth_descriptors(33, 12)]
    ctx = orbmod.Context(n, 1.2, 8, 320, 240, B)
    kp0, d0, c0, b0 = ctx.extract_match_batch(list(frames), maps, cap)                       # pageable in, pageable out
    for i in (0, 5, 17, 36):
        ko, do = oracle.detect_and_compute(frames[i], n)
        _assert_kp_equal(kp0[i, :c0[i]], d0[i, :c0[i]], ko, do, f"pageable frame {i}")
        assert b0[0][i].tobytes() == oracle.match_hamming(maps[0], do).tobytes()
    pinned = frames.copy()
    ctx.host_register(pinned)
    try:
        kp1, d1, c1, b1 = ctx.extract_match_batch(list(pinned), maps, cap)                   # page-locked in, pageable out
    finally:
        ctx.host_unregister(pinned)
    padded = np.zeros((B, 240, 331, 3), np.uint8)
    padded[:, :, :320] = frames
    import ctypes as C
    kp2 = np.zeros((B, cap), orbmod.KP_DTYPE); d2 = np.zeros((B, cap, 32), np.uint8); c2 = np.zeros(B, np.int32)
    ptrs = (C.c_void_p * B)(*[padded[i].ctypes.data for i in range(B)])
    rc = ctx.lib.orbx_detect_and_compute_batch(ctx.h, ptrs, B, 320, 240, padded.strides[1], 3, kp2.ctypes.data, d2.ctypes.data, cap,
                                               c2.ctypes.data)                                 # pageable, step = 993 bytes
    assert rc == 0
    assert np.array_equal(c0, c1) and np.array_equal(c0, c2)
    for i in range(B):
        assert kp0[i, :c0[i]].tobytes() == kp1[i, :c0[i]].tobytes() == kp2[i, :c0[i]].tobytes(), i
        assert np.array_equal(d0[i, :c0[i]], d1[i, :c0[i]]) and np.array_equal(d0[i, :c0[i]], d2[i, :c0[i]]), i
        for j in range(2):
            assert b0[j][i].tobytes() == b1[j][i].tobytes(), (j, i)
    ctx.close()


def test_two_contexts_on_two_threads_agree_with_sequential_calls(orbmod):
    """What bench.py's e2e leg does (a caller double-buffering a stream of batches): two contexts driven from two host threads at
    the same time, each through the synchronous host-buffer call with its own pageable buffers; every call of both threads must
    return exactly what a lone, sequential call returns (no shared state between contexts, copier threads included)."""
    import threading
    from rgbd_visualodometry_b200.synth import synth_frame, synth_descriptors
    B, n, cap = 24, 300, 400
    base = [synth_frame(240, 320, 4200 + i) for i in range(4)]
    batches = [[np.roll(base[(i + s) % 4], 5 * i + s, axis=1) for i in range(B)] for s in range(2)]
    maps = [synth_descriptors(300, 21)]
    ref_ctx = orbmod.Context(n, 1.2, 8, 320, 240, B)
    ref = [ref_ctx.extract_match_batch(batches[s], maps, cap) for s in range(2)]
    ref_ctx.close()
    errors = []

    def worker(s):
        try:
            ctx = orbmod.Context(n, 1.2, 8, 320, 240, B)
            for _ in range(6):
                kp, d, c, b = ctx.extract_match_batch(batches[s], maps, cap)
                rk, rd, rc, rb = ref[s]
                assert np.array_equal(c, rc)
                for i in range(B):
                    assert kp[i, :c[i]].tobytes() == rk[i, :c[i]].tobytes() and np.array_equal(d[i, :c[i]], rd[i, :c[i]]), (s, i)
                assert b[0].tobytes() == rb[0].tobytes()
            ctx.close()
        except Exception as e:  # noqa: BLE001
            errors.append((s, repr(e)))
    th = [threading.Thread(target=worker, args=(s,)) for s in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors


@pytest.mark.parametrize("kernels", KERNELS)
def test_describe_output_paths_odd_capacity_and_unaligned_device_buffers(orbmod, oracle, kernels):
    """k_describe_tma writes a group's records as 128-bit stores when it can and falls back otherwise: a capacity that is not a
    multiple of 4 (record rows of different frames are then not 16-byte aligned), capacities smaller than the count (the frame's
    last group is cut), and device output pointers offset by 4 bytes (device API).  Every variant must equal the oracle."""
    import torch
    from rgbd_visualodometry_b200.synth import synth_frame
    frames = [synth_frame(240, 320, 8800 + i) for i in range(5)]
    n = 300
    want = [oracle.detect_and_compute(f, n) for f in frames]
    ctx = orbmod.Context(n, 1.2, 8, 320, 240, 8)
    ctx.force_kernels(kernels)
    for cap in (333, 401, 302):
        kps, desc, cnt = ctx.detect_and_compute_batch(frames, cap)
        for i, (ko, do) in enumerate(want):
            _assert_kp_equal(kps[i, :cnt[i]], desc[i, :cnt[i]], ko, do, f"cap {cap} frame {i}")
    # capacity below the count: E_CAPACITY with the needed counts, nothing written past the capacity
    import ctypes as C
    small = min(len(k) for k, _ in want) - 3
    k = np.zeros((5, small + 1), orbmod.KP_DTYPE); d = np.full((5, small + 1, 32), 0xAB, np.uint8); c = np.zeros(5, np.int32)
    ptrs = (C.c_void_p * 5)(*[f.ctypes.data for f in frames])
    rc = ctx.lib.orbx_detect_and_compute_batch(ctx.h, ptrs, 5, 320, 240, 960, 3, k.ctypes.data, d.ctypes.data, small, c.ctypes.data)
    assert rc == orbmod.E_CAPACITY and c.tolist() == [len(w[0]) for w in want]
    # device API, outputs at 4-byte-offset addresses, odd capacity
    cap = 335
    d_in = torch.from_numpy(np.stack(frames)).cuda()
    raw_k = torch.zeros(5 * cap * 7 + 1, dtype=torch.float32, device="cuda")
    raw_d = torch.zeros(5 * cap * 32 + 4, dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(5, dtype=torch.int32, device="cuda")
    ctx.detect_and_compute_device(d_in.data_ptr(), 5, 320, 240, 960, 240 * 960, 3, raw_k.data_ptr() + 4, raw_d.data_ptr() + 4, cap, d_n.data_ptr())
    ctx.synchronize()
    kk = raw_k[1:].cpu().numpy().reshape(5, cap, 7)
    dd = raw_d[4:].cpu().numpy().reshape(5, cap, 32)
    nn = d_n.cpu().numpy()
    for i, (ko, do) in enumerate(want):
        got = np.ascontiguousarray(kk[i, :nn[i]]).view(orbmod.KP_DTYPE).reshape(-1)
        _assert_kp_equal(got, dd[i, :nn[i]], ko, do, f"unaligned device outputs, frame {i}")
    ctx.close()


def test_cpp_frontend_shim_equals_python_binding(orbmod, oracle, tmp_path):
    """The C++ shim of INTEGRATION.md (examples/frontend_shim.cpp: FrontEnd::ExtractKeyPointsAndComputeDescriptors + the match
    call, on cv::KeyPoint / cv::DMatch-shaped types) run as its own process on one frame: keypoint records, descriptors and
    matches hash to what the oracle gives for the same frame."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from test_abi import _build_shim
    from rgbd_visualodometry_b200.synth import synth_frame

    def fnv1a(b):
        h = 2166136261
        for x in b:
            h = ((h ^ x) * 16777619) & 0xFFFFFFFF
        return h
    img = synth_frame(480, 640, 31337)
    raw = tmp_path / "frame.bgr"
    raw.write_bytes(img.tobytes())
    exe = _build_shim(tmp_path)
    out = subprocess.run([exe, str(raw)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    ko, do = oracle.detect_and_compute(img, 500)
    mo = oracle.match_hamming(np.ascontiguousarray(do[::3][: len(do) // 3]), do)
    want = f"shim: keypoints {len(ko)} kp_fnv {fnv1a(ko.tobytes()):08x} desc_fnv {fnv1a(do.tobytes()):08x} matches {len(mo)} match_fnv {fnv1a(mo.tobytes()):08x}"
    assert want in out.stdout, (out.stdout, want)
