"""SURVEY 8(f) rows: device-resident map table, visibility filter, match post-filter, depth back-projection.

The oracle for these rows (oracle/track_oracle.py) restates reference code that cannot be built here: parity is
UNPINNED (see its header).  Tolerances: candidate / match index lists exact on inputs kept away from the decision
boundaries; back-projected positions to 1e-9 relative."""
import numpy as np
import pytest

from oracle import track_oracle as T


def _scene(seed, m):
    rng = np.random.default_rng(seed)
    ang = 0.15
    R = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    t = np.array([0.1, -0.05, 0.3])
    pose = np.concatenate([R, t[:, None]], axis=1)
    cam = (517.3, 516.5, 325.1, 249.7)                       # config/default.yaml (TUM fr1)
    pos = rng.uniform([-3, -2, -1], [3, 2, 6], size=(m, 3))
    center = -(R.T @ t)
    d = pos - center
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    tilt = rng.normal(scale=0.45, size=(m, 3))               # viewing normals scattered around the true direction
    norm = d + tilt
    norm /= np.linalg.norm(norm, axis=1, keepdims=True)
    norm[::17] = 0.0                                          # fresh map points: norm_ = 0 (acos(0) = pi/2 -> rejected)
    outlier = rng.random(m) < 0.1
    return pose, cam, pos, norm, outlier


def test_oracle_visibility_basic_properties():
    pose, cam, pos, norm, outlier = _scene(1, 400)
    vis = T.could_observe(pose, cam, 640, 480, pos, norm)
    assert 0 < vis.sum() < len(vis)
    R, t = pose[:, :3], pose[:, 3]
    pc = pos @ R.T + t
    assert (pc[vis, 2] >= 0).all()
    u = cam[0] * pc[:, 0] / pc[:, 2] + cam[2]
    v = cam[1] * pc[:, 1] / pc[:, 2] + cam[3]
    assert ((u[vis] >= 0) & (u[vis] < 640) & (v[vis] >= 0) & (v[vis] < 480)).all()
    assert not vis[::17].any()                                # zero normal -> angle pi/2 > pi/6


def test_oracle_backproject_roundtrip():
    pose, cam, *_ = _scene(2, 1)
    rng = np.random.default_rng(3)
    depth = rng.integers(2000, 30000, size=(480, 640)).astype(np.uint16)
    kps = np.zeros(50, dtype=[("x", np.float32), ("y", np.float32)])
    kps["x"] = rng.uniform(31, 608, 50); kps["y"] = rng.uniform(31, 448, 50)
    pos, valid = T.backproject(kps, depth, 5000.0, cam, pose)
    assert valid.all()
    R, t = pose[:, :3], pose[:, 3]
    pc = pos @ R.T + t
    u = cam[0] * pc[:, 0] / pc[:, 2] + cam[2]
    v = cam[1] * pc[:, 1] / pc[:, 2] + cam[3]
    assert np.allclose(u, kps["x"], atol=1e-6) and np.allclose(v, kps["y"], atol=1e-6)


@pytest.fixture(scope="module")
def orbmod():
    from rgbd_visualodometry_b200 import orb
    return orb


@pytest.mark.gpu
def test_track_match_vs_oracle(orbmod):
    from oracle import oracle as O
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    m = 3000
    pose, cam, pos, norm, outlier = _scene(7, m)
    train = synth_descriptors(900, 11)
    desc = synth_map_queries(train, m, 12)
    ids = (np.arange(m, dtype=np.int64) * 7919 + 13) % 1000003          # arbitrary, unique size_t-like ids
    ctx = orbmod.Context(500, 1.2, 8, 640, 480, 1)
    ctx.map_upsert(ids[:1000], desc[:1000], pos[:1000], norm[:1000], outlier[:1000])
    ctx.map_upsert(ids[1000:], desc[1000:], pos[1000:], norm[1000:], outlier[1000:])
    assert ctx.map_size == m
    order = np.random.default_rng(5).permutation(m)[:2500]              # the tracking map: a subset in its own order
    cand, matches, mn, mx = ctx.track_match(ids[order], pose, cam, 640, 480, train=train, match_ratio=2.0)
    oc, om, omn, omx = T.track_match(pose, cam, 640, 480, pos[order], norm[order], outlier[order], desc[order], train, 2.0, O.match_hamming)
    assert np.array_equal(cand, oc)
    assert mn == omn and mx == omx
    assert matches.tobytes() == om.tobytes()
    # update path: BA moves points, the backend flags outliers, points get erased and re-inserted
    pos2 = pos.copy(); pos2[order[:50], 2] = -5.0                        # behind the camera now
    ctx.map_upsert(ids[order[:50]], pos=pos2[order[:50]])
    out2 = outlier.copy(); out2[order[50:80]] = True
    ctx.map_upsert(ids[order[50:80]], outlier=out2[order[50:80]])
    ctx.map_erase(ids[order[100:120]])
    assert ctx.map_size == m - 20
    ctx.map_upsert(ids[order[100:120]], desc[order[100:120]], pos[order[100:120]], norm[order[100:120]], outlier[order[100:120]])
    cand, matches, mn, mx = ctx.track_match(ids[order], pose, cam, 640, 480, train=train, match_ratio=2.0)
    oc, om, omn, omx = T.track_match(pose, cam, 640, 480, pos2[order], norm[order], out2[order], desc[order], train, 2.0, O.match_hamming)
    assert np.array_equal(cand, oc) and matches.tobytes() == om.tobytes() and (mn, mx) == (omn, omx)
    with pytest.raises(orbmod.OrbxError):
        ctx.track_match(np.array([999999937], np.int64), pose, cam, 640, 480, train=train)


@pytest.mark.gpu
def test_track_match_from_resident_frame_and_empty_sets(orbmod):
    from oracle import oracle as O
    from rgbd_visualodometry_b200.synth import synth_frame
    frames = [synth_frame(240, 320, 9100 + i) for i in range(3)]
    ctx = orbmod.Context(300, 1.2, 8, 320, 240, 3)
    kps, desc, cnt = ctx.detect_and_compute_batch(frames)
    m = int(cnt[0])
    pose, cam, pos, norm, outlier = _scene(9, m)
    ids = np.arange(100, 100 + m, dtype=np.int64)
    # map points created from frame 0's keypoints: descriptor rows never leave the device
    ctx.map_upsert_from_frame(ids, 0, np.arange(m, dtype=np.int32), pos, norm)
    cand, matches, mn, mx = ctx.track_match(ids, pose, cam, 320, 240, train=None, frame=1)
    none = np.zeros(m, bool)
    oc, om, omn, omx = T.track_match(pose, cam, 320, 240, pos, norm, none, desc[0, :m], desc[1, :cnt[1]], 2.0, O.match_hamming)
    assert np.array_equal(cand, oc) and matches.tobytes() == om.tobytes() and (mn, mx) == (omn, omx)
    # every candidate filtered away / empty train set: no matches, no error
    cand, matches, _, _ = ctx.track_match(ids, pose, cam, 320, 240, train=np.zeros((0, 32), np.uint8))
    assert len(matches) == 0 and np.array_equal(cand, oc)
    ctx.map_upsert(ids, outlier=np.ones(m, np.uint8))
    cand, matches, _, _ = ctx.track_match(ids, pose, cam, 320, 240, train=None, frame=1)
    assert len(cand) == 0 and len(matches) == 0


@pytest.mark.gpu
def test_backproject_vs_oracle(orbmod):
    pose, cam, *_ = _scene(4, 1)
    rng = np.random.default_rng(8)
    depth = rng.integers(2000, 30000, size=(480, 640)).astype(np.uint16)
    depth[rng.random(depth.shape) < 0.3] = 0                            # holes: exercises the 4-neighbour fallback
    kps = np.zeros(2000, dtype=orbmod.KP_DTYPE)
    kps["x"] = rng.uniform(31, 608, len(kps)).astype(np.float32)
    kps["y"] = rng.uniform(31, 448, len(kps)).astype(np.float32)
    kps["x"][:40] = np.floor(kps["x"][:40]) + 0.5                       # ties of cvRound
    ctx = orbmod.Context(500, 1.2, 8, 640, 480, 1)
    pos, valid = ctx.backproject(kps, depth, 5000.0, cam, pose)
    opos, ovalid = T.backproject(kps, depth, 5000.0, cam, pose)
    assert np.array_equal(valid, ovalid) and 0 < valid.sum() < len(valid)
    assert np.allclose(pos[valid], opos[valid], rtol=1e-9, atol=1e-12)
    assert (pos[~valid] == 0).all()


@pytest.mark.gpu
def test_async_submit_collect_equals_sync_and_feeds_tracking(orbmod):
    """SURVEY 8(f).4: two frames in flight, results identical to the synchronous drop-in call; the collected frame is the
    train set of the next orbx_track_match without leaving the device."""
    from oracle import oracle as O
    from rgbd_visualodometry_b200.synth import synth_frame
    frames = [synth_frame(480, 640, 6100 + i) for i in range(5)]
    ctx = orbmod.Context(500, 1.2, 8, 640, 480, 1)
    sync = [ctx.detect_and_compute(f) for f in frames]
    ctx.submit_frame(frames[0])
    ctx.submit_frame(frames[1])
    with pytest.raises(orbmod.OrbxError) as e:
        ctx.submit_frame(frames[2])
    assert e.value.code == -8                                 # ORBX_E_BUSY
    for i in range(5):
        k, d = ctx.collect_frame()
        assert k.tobytes() == sync[i][0].tobytes() and np.array_equal(d, sync[i][1]), i
        if i + 2 < 5:
            ctx.submit_frame(frames[i + 2])
    with pytest.raises(orbmod.OrbxError):
        ctx.collect_frame()                                   # nothing in flight
    ko, do = O.detect_and_compute(frames[4], 500)
    assert k.tobytes() == ko.tobytes() and np.array_equal(d, do)
    # the last collected frame (4) is the resident train set
    m = len(sync[3][1])
    pose, cam, pos, norm, outlier = _scene(21, m)
    ids = np.arange(m, dtype=np.int64)
    ctx.map_upsert(ids, sync[3][1], pos, norm, np.zeros(m, np.uint8))
    cand, matches, mn, mx = ctx.track_match(ids, pose, cam, 640, 480, train=None, frame=0)
    oc, om, omn, omx = T.track_match(pose, cam, 640, 480, pos, norm, np.zeros(m, bool), sync[3][1], sync[4][1], 2.0, O.match_hamming)
    assert np.array_equal(cand, oc) and matches.tobytes() == om.tobytes() and (mn, mx) == (omn, omx)


@pytest.mark.gpu
def test_tracking_loop_orbx_equals_cv2_frontend():
    """BASELINE config 1 in miniature (tools/run_vo_synth.py): the reference's tracking loop on a synthetic RGB-D sequence with
    the hot path behind the orbx C-ABI vs the same loop with cv2's operators (live, and as stored in tests/golden/ by
    tools/make_golden_live.py): identical keypoint / match / inlier counts and poses frame by frame, and the trajectory
    within millimetres of the ground truth.  Both loops solve PnP with cv2.solvePnPRansac, so this test needs cv2."""
    cv2 = pytest.importorskip("cv2")
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("run_vo_synth", os.path.join(os.path.dirname(__file__), "..", "tools", "run_vo_synth.py"))
    vo = importlib.util.module_from_spec(spec); spec.loader.exec_module(vo)
    seq = vo.make_sequence(16)
    vo.run.pos = {}
    a, _ = vo.run("orbx", seq)
    vo.run.pos = {}
    b, _ = vo.run("cv2", seq)
    for x, y in zip(a, b):
        assert x[1:4] == y[1:4], (x[:4], y[:4])
        assert np.allclose(x[4], y[4], atol=1e-9)
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "vo_synth16_cv2.npz"))
    assert [list(x[:4]) for x in a] == g["counts"].tolist()
    assert np.allclose([x[5] for x in a], g["truth"], atol=1e-12)
    assert np.allclose([x[4] for x in a], g["centre"], atol=1e-6)      # metres; PnP runs on this host's cv2 build
    err = max(np.linalg.norm(x[4] - x[5]) for x in a)
    assert err < 0.01, err                                   # metres; 1 px at 2 m is ~3.9 mm
    assert min(x[3] for x in a[1:]) >= 30                    # PnP inliers


@pytest.mark.gpu
def test_track_float_intrinsics_and_decision_boundaries(orbmod):
    """The reference keeps fx_, fy_, cx_, cy_ and depth_scale_ as FLOAT members (include/myslam/camera.h:65) and promotes them to
    double inside the double-precision expressions of camera.cpp:39-86 / frame.cpp:43-91: both sides get the float values
    promoted to double (what INTEGRATION.md 3b tells the shim to pass).  Plus points exactly ON the decision boundaries of
    frame.cpp:73-86: u == 0, u == cols, v == 0, v == rows, z == +0, z == -0, the camera centre itself (0 / 0 = NaN: every comparison
    false, the point is kept), and normals 1e-9 rad either side of the pi / 6 cone (exactly on it the answer is libm's acos, not
    specified by the reference)."""
    from oracle import oracle as O
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    f32 = lambda v: float(np.float32(v))                                   # noqa: E731
    cam32 = tuple(f32(v) for v in (517.3, 516.5, 325.1, 249.7))             # not representable in float: the promoted values differ from the yaml's
    assert cam32 != (517.3, 516.5, 325.1, 249.7)
    m = 2000
    pose, _, pos, norm, outlier = _scene(21, m)
    train = synth_descriptors(700, 31)
    desc = synth_map_queries(train, m, 32)
    ids = np.arange(m, dtype=np.int64) + 5
    ctx = orbmod.Context(500, 1.2, 8, 640, 480, 1)
    ctx.map_upsert(ids, desc, pos, norm, outlier)
    cand, matches, mn, mx = ctx.track_match(ids, pose, cam32, 640, 480, train=train, match_ratio=2.0)
    oc, om, omn, omx = T.track_match(pose, cam32, 640, 480, pos, norm, outlier, desc, train, 2.0, O.match_hamming)
    assert np.array_equal(cand, oc) and matches.tobytes() == om.tobytes() and (mn, mx) == (omn, omx)
    # depth scale 5000 as a float member; a scale that is NOT a float (5000.1) is rounded to float by both sides
    rng = np.random.default_rng(8)
    depth = rng.integers(2000, 30000, size=(480, 640)).astype(np.uint16)
    kps = np.zeros(500, dtype=orbmod.KP_DTYPE)
    kps["x"] = rng.uniform(31, 608, len(kps)).astype(np.float32); kps["y"] = rng.uniform(31, 448, len(kps)).astype(np.float32)
    for scale in (5000.0, 5000.1):
        p, v = ctx.backproject(kps, depth, scale, cam32, pose)
        op, ov = T.backproject(kps, depth, scale, cam32, pose)
        assert np.array_equal(v, ov) and np.allclose(p[v], op[v], rtol=1e-9, atol=1e-12)
    # ---- decision boundaries: identity pose, power-of-two intrinsics, so that u, v land EXACTLY on 0 / cols / rows
    eye = np.concatenate([np.eye(3), np.zeros((3, 1))], axis=1)
    camb = (512.0, 512.0, 320.0, 240.0)
    a = np.pi / 6
    pts = np.array([[1.25, 0, 2], [-1.25, 0, 2], [0, 0.9375, 2], [0, -0.9375, 2], [1, 0, 0.0], [1, 0, -0.0], [0, 0, 0.0], [0, 0, 3], [0, 0, 3], [0.3, 0.1, 2.5]], np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        nrm = pts / np.linalg.norm(pts, axis=1, keepdims=True)             # looking straight at the point: angle 0
    nrm[6] = 0.0
    nrm[7] = [np.sin(a - 1e-9), 0, np.cos(a - 1e-9)]                       # just inside the cone
    nrm[8] = [np.sin(a + 1e-9), 0, np.cos(a + 1e-9)]                       # just outside
    want = T.could_observe(eye, camb, 640, 480, pts, nrm)
    assert want.tolist() == [False, True, False, True, False, False, True, True, False, True]    # u == cols / v == rows out, u == 0 / v == 0 in, z == +-0 -> u = +-inf out, NaN kept
    bid = np.arange(len(pts), dtype=np.int64) + 100000
    ctx.map_upsert(bid, synth_descriptors(len(pts), 5), pts, nrm, np.zeros(len(pts), np.uint8))
    cand, _, _, _ = ctx.track_match(bid, eye, camb, 640, 480, train=train, match_ratio=2.0)
    assert cand.tolist() == np.nonzero(want)[0].tolist()
    ctx.close()
