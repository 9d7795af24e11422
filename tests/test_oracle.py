"""Pins the CPU oracle (oracle/orb_oracle.c): against the committed cv2 golden vectors, stage by stage against the stored
cv2 results (and cv2 live when importable), and through its own invariants.  CPU only."""
import os

import numpy as np
import pytest

from cases import LIVE_MATCH_CASES, LIVE_PARAMS, MATCH_CASES, ORB_CASES, ORB_CASES_LARGE, assert_equals_stored, sha

GOLD = os.path.join(os.path.dirname(__file__), "golden")

try:
    import cv2
except Exception:  # pragma: no cover
    cv2 = None


def test_pattern_hash():
    a = np.load(os.path.join(GOLD, "brief_pattern.npy")).astype("<i2")
    assert sha(a) == "be6a662a255ab61975e593461f171f699a9b597d766e89e62c5a97a260a35bb1"


def test_geometry_and_quotas(oracle):
    ws, hs, sc = oracle.level_geometry(640, 480)
    assert ws == [640, 533, 444, 370, 309, 257, 214, 179] and hs == [480, 400, 333, 278, 231, 193, 161, 134]
    assert [hex(v) for v in sc.view(np.uint32)] == ["0x3f800000", "0x3f99999a", "0x3fb851ec", "0x3fdd2f1c", "0x4004b5de",
                                                    "0x401f40a5", "0x403f1a60", "0x406552da"]
    assert oracle.level_geometry(1920, 1080)[0] == [1920, 1600, 1333, 1111, 926, 772, 643, 536]
    assert oracle.level_geometry(3840, 2160)[1] == [2160, 1800, 1500, 1250, 1042, 868, 723, 603]
    assert oracle.quotas(500) == [109, 90, 75, 63, 52, 44, 36, 31]
    assert oracle.quotas(1000) == [217, 181, 151, 126, 105, 87, 73, 60]
    assert oracle.quotas(2000) == [434, 362, 302, 251, 209, 175, 145, 122]
    assert oracle.quotas(5000) == [1086, 905, 754, 628, 524, 436, 364, 303]


@pytest.mark.parametrize("name", list(ORB_CASES))
def test_orb_golden(oracle, name):
    mk, n = ORB_CASES[name]
    img = mk()
    g = np.load(os.path.join(GOLD, f"orb_{name}.npz"))
    assert sha(img) == str(g["img_sha"]), "synthetic generator drifted from the one that made the fixtures"
    k, d = oracle.detect_and_compute(img, n)
    assert len(k) == len(g["keypoints"])
    assert k.tobytes() == g["keypoints"].tobytes()          # all 7 cv::KeyPoint fields, order included
    assert np.array_equal(d, g["descriptors"])


@pytest.mark.parametrize("name", list(MATCH_CASES))
def test_match_golden(oracle, name):
    mq, mt = MATCH_CASES[name]
    q, t = mq(), mt()
    g = np.load(os.path.join(GOLD, f"match_{name}.npz"))
    assert sha(q) == str(g["q_sha"]) and sha(t) == str(g["t_sha"])
    assert oracle.match_hamming(q, t).tobytes() == g["match"].tobytes()
    k2 = oracle.match_hamming_knn2(q, t)
    gk = g["knn2"]
    assert np.array_equal(k2["trainIdx"][:, 0], gk["trainIdx"][:, 0]) and np.array_equal(k2["distance"][:, 0], gk["distance"][:, 0])
    if len(t) >= 2:
        assert k2.tobytes() == gk.tobytes()
    else:
        assert (k2["trainIdx"][:, 1] == -1).all()


def test_match_empty(oracle):
    e = np.zeros((0, 32), np.uint8)
    t = np.zeros((4, 32), np.uint8)
    assert len(oracle.match_hamming(e, t)) == 0 and len(oracle.match_hamming(t, e)) == 0


def test_match_pm1_identity(oracle):
    """hamming == (256 - dot(+-1 expansions)) / 2 -- the identity the tensor-core matcher relies on (SURVEY A.11)."""
    from rgbd_visualodometry_b200.synth import synth_descriptors
    q, t = synth_descriptors(64, 1), synth_descriptors(96, 2)
    qb = np.unpackbits(q, axis=1).astype(np.int32) * 2 - 1
    tb = np.unpackbits(t, axis=1).astype(np.int32) * 2 - 1
    ham = (256 - qb @ tb.T) // 2
    m = oracle.match_hamming(q, t)
    assert np.array_equal(m["trainIdx"], ham.argmin(1)) and np.array_equal(m["distance"], ham.min(1).astype(np.float32))


def test_filter_matches(oracle):
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    t = synth_descriptors(500, 3)
    m = oracle.match_hamming(synth_map_queries(t, 300, 4), t)
    f = oracle.filter_matches(m, 2.0)
    thr = max(m["distance"].min() * 2.0, 30.0)
    assert np.array_equal(f, m[m["distance"] <= thr])


def test_retain_best_semantics(oracle):
    """retainBest keeps every element >= the m-th largest (ties kept) and is a permutation of them."""
    rng = np.random.default_rng(0)
    for trial in range(50):
        n = int(rng.integers(1, 400)); m = int(rng.integers(0, 300))
        c = np.zeros(n, oracle.CAND_DTYPE)
        c["x"] = np.arange(n); c["response"] = rng.integers(20, 40, n).astype(np.float32)
        r = oracle.retain_best(c, m)
        if n <= m:
            assert r.tobytes() == c.tobytes()
        elif m == 0:
            assert len(r) == 0
        else:
            thr = np.sort(c["response"])[::-1][m - 1]
            keep = c[c["response"] >= thr]
            assert sorted(r["x"]) == sorted(keep["x"])


class TestLiveCv2:
    """The oracle against OpenCV's own operators: against the stored cv2 results always (tests/golden/, written by
    tools/make_golden_live.py), and against cv2 live as well when it is importable."""

    def test_stages(self, oracle):
        from rgbd_visualodometry_b200.synth import synth_frame
        gs = np.load(os.path.join(GOLD, "stages_701x467.npz"))
        img = synth_frame(467, 701, 21)
        assert sha(img) == str(gs["img_sha"]), "synthetic generator drifted from the one that made the fixtures"
        g = oracle.gray(img)
        assert sha(g) == str(gs["gray_sha"])
        if cv2 is not None:
            assert np.array_equal(g, cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
        ws, hs, _ = oracle.level_geometry(701, 467)
        prev = g
        for l in range(1, 8):
            cur = oracle.resize_exact(prev, ws[l], hs[l])
            assert sha(cur) == str(gs["level_sha"][l - 1]), l
            if cv2 is not None:
                assert np.array_equal(cur, cv2.resize(prev, (ws[l], hs[l]), interpolation=cv2.INTER_LINEAR_EXACT)), l
            prev = cur
        fo = oracle.fast_nms(g)
        assert_equals_stored(gs, "FAST", fast=fo)
        if cv2 is not None:
            f = cv2.FastFeatureDetector_create(20, True).detect(g)
            assert len(f) == len(fo)
            assert all((int(a.pt[0]), int(a.pt[1]), a.response) == (int(b["x"]), int(b["y"]), float(b["response"])) for a, b in zip(f, fo))

    def test_sincos_matches_libm(self, oracle):
        """orbo_sincosf restates glibc sinf/cosf; numpy's float32 sin/cos call the same libm here."""
        import ctypes, ctypes.util
        libm = ctypes.CDLL(ctypes.util.find_library("m"))
        libm.sinf.restype = ctypes.c_float; libm.sinf.argtypes = [ctypes.c_float]
        libm.cosf.restype = ctypes.c_float; libm.cosf.argtypes = [ctypes.c_float]
        rng = np.random.default_rng(1)
        ang = (rng.random(20000).astype(np.float32) * np.float32(360.0)) * np.float32(0.017453292)
        ang[:8] = [0, 1e-5, 0.78539816, 0.7853982, 1.5707964, 3.1415927, 4.712389, 6.2831855]
        for a in ang:
            s, c = oracle.sincosf(float(a))
            assert s == libm.sinf(float(a)) and c == libm.cosf(float(a)), a

    @pytest.mark.parametrize("name", list(ORB_CASES_LARGE))
    def test_orb_large(self, oracle, name):
        mk, n = ORB_CASES_LARGE[name]
        img = mk()
        g = np.load(os.path.join(GOLD, f"orb_{name}.npz"))
        assert sha(img) == str(g["img_sha"]), "synthetic generator drifted from the one that made the fixtures"
        ko, do = oracle.detect_and_compute(img, n)
        assert_equals_stored(g, f"oracle {name}", keypoints=ko, descriptors=do)
        if cv2 is not None:
            k, d = cv2.ORB_create(n, 1.2, 8).detectAndCompute(img, None)
            assert ko.tobytes() == oracle.cv2_keypoints_to_array(k).tobytes() and np.array_equal(d, do)

    def test_match_live(self, oracle):
        q, t = (f() for f in LIVE_MATCH_CASES["1500x2000"])
        g = np.load(os.path.join(GOLD, "match_live_1500x2000.npz"))
        assert sha(q) == str(g["q_sha"]) and sha(t) == str(g["t_sha"])
        mo = oracle.match_hamming(q, t)
        assert_equals_stored(g, "oracle match", match=mo)
        if cv2 is not None:
            m = cv2.BFMatcher(cv2.NORM_HAMMING).match(q, t)
            assert mo.tobytes() == oracle.cv2_matches_to_array(m).tobytes()


@pytest.mark.parametrize("params", LIVE_PARAMS)
def test_oracle_other_parameters_vs_cv2_live(oracle, params):
    """Stored cv2 result always; cv2 live as well when importable."""
    from rgbd_visualodometry_b200.synth import synth_frame
    n, sf, nl = params
    img = synth_frame(480, 640, 31)
    g = np.load(os.path.join(GOLD, f"orb_params_{n}_{sf}_{nl}.npz"))
    assert sha(img) == str(g["img_sha"])
    k, d = oracle.detect_and_compute(img, n, sf, nl)
    assert_equals_stored(g, f"oracle ORB({n}, {sf}, {nl})", keypoints=k, descriptors=d)
    if cv2 is not None:
        kc, dc = cv2.ORB_create(n, sf, nl).detectAndCompute(img, None)
        assert k.tobytes() == oracle.cv2_keypoints_to_array(kc).tobytes() and np.array_equal(d, dc)
