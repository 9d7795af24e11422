"""Cross-checked Hamming matching, BFMatcher(NORM_HAMMING, crossCheck=True): a pair (i, j) is kept when j is query i's
nearest train row and i is train row j's nearest query, the lowest index winning ties in both directions, in ascending
queryIdx.  CPU: the oracle composition (xcheck_cases.oracle_crosscheck) against cv2's stored (and, when importable, live)
results and against a numpy brute force.  GPU (-m gpu): the fused kernels (column maxima taken from the same distance tiles) against the golden results and the oracle."""
import ctypes as C
import os

import numpy as np
import pytest

from cases import assert_equals_stored, sha
from xcheck_cases import XCHECK_CASES, oracle_crosscheck

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _golden(name):
    return np.load(os.path.join(GOLD, f"match_xcheck_{name}.npz"))


def _assert_golden(got, g, what):
    if "match" in g:
        assert got.tobytes() == g["match"].tobytes(), what
    else:
        assert_equals_stored(g, what, match=got)


def _brute(q, t):
    """The definition, in numpy: mutual argmin of the Hamming distance matrix (argmin takes the lowest index)."""
    if len(q) == 0 or len(t) == 0:
        return np.zeros(0, [("queryIdx", "<i4"), ("trainIdx", "<i4"), ("imgIdx", "<i4"), ("distance", "<f4")])
    d = np.unpackbits(q[:, None, :] ^ t[None, :, :], axis=2).sum(2)
    fwd, bwd = d.argmin(1), d.argmin(0)
    keep = np.nonzero(bwd[fwd] == np.arange(len(q)))[0]
    out = np.zeros(len(keep), [("queryIdx", "<i4"), ("trainIdx", "<i4"), ("imgIdx", "<i4"), ("distance", "<f4")])
    out["queryIdx"], out["trainIdx"], out["distance"] = keep, fwd[keep], d[keep, fwd[keep]]
    return out


def _tie_heavy(rng, n):
    return (rng.integers(0, 4, (n, 32)) if rng.random() < 0.7 else rng.integers(0, 256, (n, 32))).astype(np.uint8)


# ---- CPU -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(XCHECK_CASES))
def test_oracle_vs_golden(oracle, name):
    mq, mt = XCHECK_CASES[name]
    q, t = mq(), mt()
    g = _golden(name)
    assert sha(q) == str(g["q_sha"]) and sha(t) == str(g["t_sha"]), "inputs differ from those the golden file was made from"
    _assert_golden(oracle_crosscheck(q, t), g, f"oracle vs cv2 ({name})")


@pytest.mark.parametrize("name", list(XCHECK_CASES))
def test_oracle_vs_live_cv2(oracle, name):
    cv2 = pytest.importorskip("cv2")
    mq, mt = XCHECK_CASES[name]
    q, t = mq(), mt()
    ref = oracle.cv2_matches_to_array(cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True).match(q, t))
    assert oracle_crosscheck(q, t).tobytes() == ref.tobytes()


@pytest.mark.parametrize("seed", range(50))
def test_oracle_vs_bruteforce_tie_heavy(oracle, seed):
    rng = np.random.default_rng(1000 + seed)
    nq, nt = int(rng.integers(0, 120)), int(rng.integers(0, 120))
    q, t = _tie_heavy(rng, nq), _tie_heavy(rng, nt)
    if nt > 1 and rng.random() < 0.5:                # duplicated train rows
        t[rng.integers(0, nt, nt // 3)] = t[rng.integers(0, nt, nt // 3)]
    if nq > 1 and rng.random() < 0.5:                # duplicated query rows
        q[rng.integers(0, nq, nq // 3)] = q[rng.integers(0, nq, nq // 3)]
    assert oracle_crosscheck(q, t).tobytes() == _brute(q, t).tobytes()


# ---- GPU -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def orbmod():
    from rgbd_visualodometry_b200 import orb
    return orb


def _device_crosscheck(orbmod, ctx, q, trains, counts):
    """match_device_crosscheck on a ragged batch -> per-set compacted records."""
    import torch
    nsets, cap = trains.shape[0], trains.shape[1]
    dq = torch.from_numpy(np.ascontiguousarray(q)).cuda(); dt = torch.from_numpy(np.ascontiguousarray(trains)).cuda()
    dn = torch.tensor(counts, dtype=torch.int32, device="cuda")
    out = torch.full((nsets, len(q), 4), -7, dtype=torch.int32, device="cuda")
    nout = torch.full((nsets,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.match_device_crosscheck(dq.data_ptr(), len(q), dt.data_ptr(), cap, dn.data_ptr(), nsets, out.data_ptr(), nout.data_ptr())
    ctx.synchronize()
    got = out.cpu().numpy().view(orbmod.DMATCH_DTYPE).reshape(nsets, len(q))
    return [got[s, :n] for s, n in enumerate(nout.cpu().numpy())]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(XCHECK_CASES))
def test_bfmatcher_crosscheck_vs_golden(orbmod, name):
    mq, mt = XCHECK_CASES[name]
    q, t = mq(), mt()
    _assert_golden(orbmod.BFMatcher(orbmod.NORM_HAMMING, crossCheck=True).match(q, t), _golden(name), f"GPU vs cv2 ({name})")


@pytest.mark.gpu
def test_crosscheck_empty_and_unsupported(orbmod):
    from rgbd_visualodometry_b200.synth import synth_descriptors
    bf = orbmod.BFMatcher(orbmod.NORM_HAMMING, crossCheck=True)
    e, t = np.zeros((0, 32), np.uint8), synth_descriptors(40, 3)
    assert len(bf.match(e, t)) == 0 and len(bf.match(t, e)) == 0      # (cv2 raises on the empty train set)
    with pytest.raises(orbmod.OrbxError) as ex:
        bf.knnMatch(t, t, k=2)
    assert ex.value.code == orbmod.E_UNSUPPORTED
    with pytest.raises(orbmod.OrbxError) as ex:
        orbmod.BFMatcher(4, crossCheck=True)                            # NORM_L2
    assert ex.value.code == orbmod.E_UNSUPPORTED


@pytest.mark.gpu
def test_split_path(orbmod, oracle):
    """One small query tile against a long set: the train rows are split across CTAs (row winners merged and finalised
    before the mutual check, column keys merged across the splits)."""
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    t = synth_descriptors(20000, 50)
    q = synth_map_queries(t, 200, 51)
    got = orbmod.BFMatcher(orbmod.NORM_HAMMING, crossCheck=True).match(q, t)
    ref = oracle_crosscheck(q, t)
    assert len(ref) > 100 and got.tobytes() == ref.tobytes()


@pytest.mark.gpu
def test_cross_cta_column_merge_lower_query_wins(orbmod, oracle):
    """A query duplicated across query tiles (CTAs): the train row they both sit on exactly goes to the lower index."""
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    nq = 5 * 256 - 77
    t = synth_descriptors(500, 52)
    q = synth_map_queries(t, nq, 53)
    q[1100] = q[10] = t[7]
    got = orbmod.BFMatcher(orbmod.NORM_HAMMING, crossCheck=True).match(q, t)
    assert got.tobytes() == oracle_crosscheck(q, t).tobytes()
    pairs = {(int(a), int(b)) for a, b in zip(got["queryIdx"], got["trainIdx"])}
    assert (10, 7) in pairs and not any(a == 1100 for a, _ in pairs)


@pytest.mark.gpu
def test_pair_kernel_ragged_sets_with_zero_rows(orbmod, oracle):
    """Enough (query tile, set) pairs for the CTA-pair kernel, ragged sets on every tile / chunk boundary, nq not a multiple of
    256 (padded query rows; the last pair's peer holds none).  Every non-empty set holds an all-zero train row, which a padded
    (all-zero) query row would win if it leaked into the column maxima; queries 5 and 900 sit next to it."""
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    cap, nq = 300, 5 * 256 - 77
    sizes = [0, 1, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64, 65, 95, 96, 97, 191, 192, 193, 255, 299, 300]
    sizes = sizes + [int(x) for x in np.random.default_rng(6).integers(0, cap + 1, 40 - len(sizes))]
    nsets = len(sizes)
    trains = np.stack([synth_descriptors(cap, 1900 + i) for i in range(nsets)])
    for i, n in enumerate(sizes):
        if n >= 3:
            trains[i, n - 1] = trains[i, n // 2]     # the set's last row also appears earlier (padded copies of it)
        if n >= 1:
            trains[i, n // 3] = 0
    q = synth_map_queries(trains[1 + int(np.argmax(sizes[1:]))], nq, 72)
    q[5] = 0; q[5, 0] = 1
    q[900] = 0; q[900, 31] = 3
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    got = _device_crosscheck(orbmod, ctx, q, trains, sizes)
    for s, n in enumerate(sizes):
        ref = oracle_crosscheck(q, trains[s, :n])
        assert got[s].tobytes() == ref.tobytes(), f"set {s} ({n} rows)"
        if n >= 1:
            assert 5 in got[s]["queryIdx"], f"set {s}: the zero row's nearest query lost its column"
    ctx.close()


@pytest.mark.gpu
def test_single_cta_uniform_sets(orbmod, oracle):
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    nsets, nt, nq = 3, 700, 1300
    trains = np.stack([synth_descriptors(nt, 60 + i) for i in range(nsets)])
    q = synth_map_queries(trains[0], nq, 70)
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    got = _device_crosscheck(orbmod, ctx, q, trains, [nt] * nsets)
    for s in range(nsets):
        assert got[s].tobytes() == oracle_crosscheck(q, trains[s]).tobytes(), f"set {s}"
    ctx.close()


@pytest.mark.gpu
def test_random_shapes_vs_oracle(orbmod, oracle):
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    rng = np.random.default_rng(77)
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    for k in range(30):
        nq, cap, nsets = int(rng.integers(1, 3000)), int(rng.integers(1, 1500)), int(rng.integers(1, 9))
        if k % 3 == 0:
            trains = rng.integers(0, 4, (nsets, cap, 32)).astype(np.uint8)      # tie-heavy
            q = rng.integers(0, 4, (nq, 32)).astype(np.uint8)
        else:
            trains = np.stack([synth_descriptors(cap, 3000 + 10 * k + s) for s in range(nsets)])
            q = synth_map_queries(trains[0], nq, 4000 + k)
        counts = [int(x) for x in rng.integers(0, cap + 1, nsets)]
        got = _device_crosscheck(orbmod, ctx, q, trains, counts)
        for s, n in enumerate(counts):
            assert got[s].tobytes() == oracle_crosscheck(q, trains[s, :n]).tobytes(), f"shape {k} ({nq}, {cap}, {nsets}) set {s}"
    ctx.close()


@pytest.mark.gpu
def test_argument_errors(orbmod):
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    lib, h = ctx.lib, ctx.h
    one = np.zeros((1, 32), np.uint8)
    out = np.zeros(1, orbmod.DMATCH_DTYPE)
    n = C.c_int(0)
    p = lambda a: a.ctypes.data_as(C.c_void_p)                         # noqa: E731
    assert lib.orbx_match_hamming_crosscheck(h, p(one), 1 << 20, p(one), 1, p(out), C.byref(n)) == orbmod.E_UNSUPPORTED
    assert lib.orbx_match_hamming_crosscheck(h, None, 1, p(one), 1, p(out), C.byref(n)) == orbmod.E_ARG
    assert lib.orbx_match_hamming_crosscheck(h, p(one), 1, p(one), 1, None, C.byref(n)) == orbmod.E_ARG
    assert lib.orbx_match_hamming_crosscheck(h, p(one), 1, p(one), 1, p(out), None) == orbmod.E_ARG
    assert lib.orbx_match_hamming_crosscheck(h, p(one), -1, p(one), 1, p(out), C.byref(n)) == orbmod.E_ARG
    import torch
    d = torch.zeros(64, dtype=torch.int32, device="cuda"); dp = d.data_ptr()
    dev = lib.orbx_match_hamming_device_crosscheck
    assert dev(h, dp, 1 << 20, dp, 1, dp, 1, dp, dp) == orbmod.E_UNSUPPORTED
    assert dev(h, dp, 1, dp, 1, dp, 65536, dp, dp) == orbmod.E_ARG
    assert dev(h, dp, 1, dp, 1, dp, -1, dp, dp) == orbmod.E_ARG
    assert dev(h, None, 1, dp, 1, dp, 1, dp, dp) == orbmod.E_ARG
    assert dev(h, dp, 1, dp, 1, None, 1, dp, dp) == orbmod.E_ARG
    assert dev(h, dp, 1, dp, 1, dp, 1, None, dp) == orbmod.E_ARG
    assert dev(h, dp, 1, dp, 1, dp, 1, dp, None) == orbmod.E_ARG
    # empty sizes: no sets returns before every pointer; no query or train rows still needs d_n_out, and zeroes it
    n.value = 7
    assert lib.orbx_match_hamming_crosscheck(h, None, 0, None, 1, None, C.byref(n)) == orbmod.OK and n.value == 0
    assert dev(h, None, 1, None, 1, None, 0, None, None) == orbmod.OK
    assert dev(h, None, 0, dp, 1, dp, 1, dp, None) == orbmod.E_ARG
    d.fill_(5)
    assert dev(h, None, 0, None, 4, None, 3, None, dp) == orbmod.OK
    assert dev(h, dp, 4, dp, 0, dp, 3, dp, dp + 12) == orbmod.OK
    ctx.synchronize()
    assert d[:7].tolist() == [0] * 6 + [5]
    ctx.close()


@pytest.mark.gpu
def test_plain_match_unchanged_around_a_crosscheck(orbmod, oracle):
    """match -> match_crosscheck -> match on one context: the cross-check's scratch does not leak into the plain matcher."""
    from rgbd_visualodometry_b200.synth import synth_descriptors, synth_map_queries
    t = synth_descriptors(2000, 80)
    q = synth_map_queries(t, 1500, 81)
    ctx = orbmod.Context(1, 1.2, 1, 64, 64, 1)
    a = ctx.match(q, t)
    x = ctx.match_crosscheck(q, t)
    b = ctx.match(q, t)
    assert a.tobytes() == b.tobytes() == oracle.match_hamming(q, t).tobytes()
    assert x.tobytes() == oracle_crosscheck(q, t).tobytes()
    ctx.close()
