"""Guided re-matching (msfm_match_pairs_guided, GUIDED-SPEC in include/msfm_match.h): the float32 epipolar gate, the
masked 2-NN and mutual check against the numpy restatement in oracle/guided_oracle.py, bit for bit; the planted-decoy
scene on which the gate recovers true matches that the unconstrained ratio test loses; batching, pruning, the error
statuses and the C++ mirror."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from metricsfm_b200 import synth
from oracle import geo_oracle as go
from oracle import guided_oracle as gdo
from oracle.guided_oracle import decoy_scene, eight_point

REJECT_GT = 1


# ------------------------------------------------------------------------------------------------ CPU: the oracle
@pytest.mark.parametrize("th", [1.0, 3.0, 20.0])
def test_oracle_gate_agrees_with_ransac_error(th):
    """The float32 gate is msfm_geo_verify's stage-A inlier test err <= th^2 on every element whose float64 error is not
    within 1e-4 (relative) of th^2."""
    s = decoy_scene(7, 400, 300)
    allowed = gdo.gate_f32(s["F"], s["xy_ref"], s["xy_qry"], th)
    M, N = len(s["xy_ref"]), len(s["xy_qry"])
    pt1 = np.repeat(s["xy_ref"][None, :, :], N, 0).reshape(-1, 2)
    pt2 = np.repeat(s["xy_qry"][:, None, :], M, 1).reshape(-1, 2)
    err = go.ransac_error(s["F"].astype(np.float32).astype(np.float64), pt1, pt2).reshape(N, M)
    clear = np.abs(err - th * th) > 1e-4 * th * th
    assert clear.sum() > 0.99 * clear.size
    np.testing.assert_array_equal(allowed[clear], (err <= th * th)[clear])
    assert 0 < allowed.sum() < allowed.size


@pytest.mark.parametrize("M,N", [(1, 1), (19, 21), (128, 127), (300, 257)])
def test_oracle_admit_all_gate_is_plain_knn2(oracle_mod, M, N):
    s = decoy_scene(11 + M, M, N)
    allowed = gdo.gate_f32(s["F"], s["xy_ref"], s["xy_qry"], 1e15)
    assert allowed.all()
    D = gdo.dist_u8(s["ref"], s["qry"])
    ids, dists = gdo.masked_knn2(D, allowed)
    oids, odists = oracle_mod.knn2_u8(s["ref"], s["qry"])
    np.testing.assert_array_equal(ids, oids)
    np.testing.assert_array_equal(dists, odists)
    np.testing.assert_array_equal(gdo.masked_colbest(D, allowed), oracle_mod.colbest_u8(s["ref"], s["qry"])[0])


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def matcher(native_lib):
    from metricsfm_b200.matcher import Matcher
    m = Matcher(device=0, max_images=16, arena_rows=1 << 16)
    yield m
    m.close()


def _load(m, scenes):
    """Upload every scene as images (2s, 2s+1); returns (pairs, F [n,3,3], image_xy)."""
    m.release_all()
    pairs, F, xy = [], [], {}
    for i, s in enumerate(scenes):
        m.upload(2 * i, s["ref"])
        m.upload(2 * i + 1, s["qry"])
        pairs.append((2 * i, 2 * i + 1))
        F.append(s["F"])
        xy[2 * i], xy[2 * i + 1] = s["xy_ref"], s["xy_qry"]
    return pairs, np.array(F), xy


def _expect(s, th, ratio, **kw):
    return gdo.match_pair_guided(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], th, ratio, **kw)


def _check(res, p, exp, ratio_good):
    assert bool(res.ok[p]) == exp["ok"]
    np.testing.assert_array_equal(res.pair(p), exp["pairs"].reshape(-1, 2))
    if ratio_good > 0:
        np.testing.assert_array_equal(res.pair_good(p), exp["good"])


SIZES = [(1, 1), (19, 20), (20, 19), (21, 21), (127, 128), (128, 129), (129, 127), (2000, 1999)]


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [False, True])
@pytest.mark.parametrize("th", [3.0, 150.0])
def test_sizes_ties_and_sparse_rows_vs_oracle(matcher, mutual, th):
    """Ragged and edge sizes, duplicated rows (ties), and at th = 3 px many rows with zero or one allowed reference
    row; all pairs in one call, each equal to the oracle."""
    scenes = [decoy_scene(100 + i, M, N, decoy_frac=0.5) for i, (M, N) in enumerate(SIZES)]
    pairs, F, xy = _load(matcher, scenes)
    res = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=th, ratio=0.85, ratio_good=0.6, mutual=mutual, min_keypoints=0)
    few = 0
    for p, s in enumerate(scenes):
        exp = _expect(s, th, 0.85, ratio_good=0.6, mutual=mutual, min_keypoints=0)
        _check(res, p, exp, 0.6)
        few += int((exp["allowed"].sum(1) <= 1).sum())
    if th == 3.0:
        assert few > 100  # the sparse case is exercised


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [False, True])
def test_rule_variants_vs_oracle(matcher, mutual):
    """orientation, ratio_good, max_dist_sq, MSFM_RATIO_REJECT_GT and the min_keypoints gate under the epipolar gate."""
    scenes = [decoy_scene(200 + i, M, N, decoy_frac=0.5) for i, (M, N) in enumerate([(600, 500), (300, 700), (15, 400)])]
    pairs, F, xy = _load(matcher, scenes)
    for orientation, ratio_good, max_dist_sq, flags in [(0, 0.6, 0.0, 0), (1, 0.0, 0.0, 0), (0, 0.6, 40000.0, 0),
                                                         (1, 0.7, 0.0, REJECT_GT), (0, 0.0, 60000.0, REJECT_GT)]:
        res = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=8.0, ratio=0.8, ratio_good=ratio_good, max_dist_sq=max_dist_sq,
                                         mutual=mutual, orientation=orientation, flags=flags)
        assert res.ok.tolist() == [1, 1, 0]
        for p, s in enumerate(scenes):
            exp = _expect(s, 8.0, 0.8, mutual=mutual, orientation=orientation, ratio_good=ratio_good, max_dist_sq=max_dist_sq,
                          reject_gt=bool(flags & REJECT_GT))
            _check(res, p, exp, ratio_good)


@pytest.mark.gpu
def test_planted_decoys_recovered(matcher):
    """The feature's purpose: with a look-alike of every true match's descriptor planted off the epipolar line, the
    unconstrained ratio test rejects most true matches; the guided pass equals the oracle and accepts far more."""
    s = decoy_scene(300, 1400, 900)
    pairs, F, xy = _load(matcher, [s])
    for mutual in (False, True):
        plain = matcher.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual)
        guided = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=3.0, ratio=0.85, ratio_good=0.6, mutual=mutual)
        assert matcher.timing()["twin_pairs"] == int(mutual)  # every guided mutual pair takes the tensor twin pass
        _check(guided, 0, _expect(s, 3.0, 0.85, ratio_good=0.6, mutual=mutual), 0.6)
        n_plain = sum((int(j), int(q)) in s["true"] for j, q in plain.pair(0))
        n_guided = sum((int(j), int(q)) in s["true"] for j, q in guided.pair(0))
        print(f"mutual={mutual}: planted true matches accepted: plain {n_plain}, guided {n_guided} of {len(s['true'])}")
        assert n_guided > n_plain
        assert n_guided > 0.5 * len(s["true"])


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [False, True])
def test_admit_all_gate_equals_match_pairs(matcher, mutual):
    scenes = [decoy_scene(400 + i, M, N) for i, (M, N) in enumerate([(900, 800), (129, 300), (40, 41)])]
    pairs, F, xy = _load(matcher, scenes)
    plain = matcher.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual)
    guided = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=1e15, ratio=0.85, ratio_good=0.6, mutual=mutual)
    np.testing.assert_array_equal(guided.offsets, plain.offsets)
    np.testing.assert_array_equal(guided.ok, plain.ok)
    np.testing.assert_array_equal(guided.matches, plain.matches)
    np.testing.assert_array_equal(guided.good, plain.good)


@pytest.mark.gpu
def test_pruning_off_gives_identical_lists(matcher):
    scenes = [decoy_scene(500 + i, M, N, decoy_frac=0.5) for i, (M, N) in enumerate([(2000, 1500), (700, 900)])]
    pairs, F, xy = _load(matcher, scenes)
    for mutual in (False, True):
        for th in (3.0, 40.0):
            on = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=th, ratio=0.85, ratio_good=0.6, mutual=mutual)
            matcher._test_disable_pruning(True)
            try:
                off = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=th, ratio=0.85, ratio_good=0.6, mutual=mutual)
            finally:
                matcher._test_disable_pruning(False)
            np.testing.assert_array_equal(on.offsets, off.offsets)
            np.testing.assert_array_equal(on.matches, off.matches)
            np.testing.assert_array_equal(on.good, off.good)


@pytest.mark.gpu
def test_one_call_over_several_batches_equals_per_pair_calls(native_lib):
    """100 images x 8192 rows, all 4950 pairs (~40 M query rows, more than one 16 Mi-row batch) with scene Fs."""
    from metricsfm_b200.matcher import Matcher
    n_img, rows = 100, 8192
    rng = np.random.default_rng(600)
    col = synth.Collection(rows, seed=600)
    xy = {i: rng.uniform(-1800, 1800, (rows, 2)).astype(np.float32) for i in range(n_img)}
    Fs = [eight_point(*go.two_view_scene(rng, 64, 0)) for _ in range(64)]
    pairs = synth.exhaustive_pairs(n_img)
    F = np.array([Fs[p % len(Fs)] for p in range(len(pairs))])
    with Matcher(device=0, max_images=n_img, arena_rows=n_img * rows + (1 << 16)) as m:
        m.upload_batch(list(range(n_img)), [col.image_u8(i) for i in range(n_img)])
        one = m.match_pairs_guided(pairs, F, xy, th_epipolar=60.0, ratio=0.85, ratio_good=0.6, mutual=True)
        t = m.timing()
        assert t["match_launches"] >= 4  # forward + twin launch per batch: at least two batches
        assert t["twin_pairs"] == len(pairs)
        assert len(one.matches) > 0
        for p in range(len(pairs)):
            r = m.match_pairs_guided(pairs[p:p + 1], F[p:p + 1], xy, th_epipolar=60.0, ratio=0.85, ratio_good=0.6, mutual=True)
            np.testing.assert_array_equal(r.pair(0), one.pair(p))
            np.testing.assert_array_equal(r.pair_good(0), one.pair_good(p))


@pytest.mark.gpu
def test_end_to_end_after_verification(matcher):
    """match_pairs -> geo_verify -> match_pairs_guided on the verified pairs with the F geo_verify returned."""
    scenes = [decoy_scene(700 + i, M, N, decoy_frac=0.5) for i, (M, N) in enumerate([(1200, 900), (800, 1000), (600, 700)])]
    pairs, _, xy = _load(matcher, scenes)
    first = matcher.match_pairs(pairs, 0.85, ratio_good=0.6)
    ok, _, _, F = matcher.geo_verify(pairs, first, xy, th_epipolar=3.0, seed=5)
    assert ok.sum() >= 2
    sel = [p for p in range(len(pairs)) if ok[p]]
    res = matcher.match_pairs_guided([pairs[p] for p in sel], F[sel], xy, th_epipolar=3.0, ratio=0.85, ratio_good=0.6,
                                     mutual=True)
    for k, p in enumerate(sel):
        s = scenes[p]
        exp = gdo.match_pair_guided(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], F[p], 3.0, 0.85, ratio_good=0.6, mutual=True)
        _check(res, k, exp, 0.6)
        assert len(res.pair(k)) > len(first.pair(p)) // 2


@pytest.mark.gpu
def test_error_statuses_before_launch(matcher):
    """Every malformed input is refused with INVALID_ARG before anything runs: outputs untouched, msfm_last_timing
    still that of the previous call."""
    from metricsfm_b200 import _lib
    s = decoy_scene(800, 200, 150)
    pairs, F, xy = _load(matcher, [s])
    matcher.match_pairs_guided(pairs, F, xy, th_epipolar=3.0, ratio=0.85)
    before = matcher.timing()
    assert before["match_launches"] >= 1
    L, h = matcher._L, matcher._h

    def call(F=F, th=3.0, xy_list=(s["xy_ref"], s["xy_qry"]), npts=None, n_images=2, pairs=pairs, null_xy_table=False,
             rescore=0.0):
        pa = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        arrs = [np.ascontiguousarray(a, np.float32) if a is not None else None for a in xy_list]
        ptrs = (C.c_void_p * max(len(arrs), 1))(*[a.ctypes.data if a is not None else None for a in arrs])
        np_ = np.array([len(a) if a is not None else 0 for a in arrs] if npts is None else npts, np.int32)
        prm = matcher._params(0.85, 0.6, 0.0, True, 20, 0, rescore, 0)
        offs = np.full((len(pa) + 1,), -7, np.int64)
        okf = np.full((max(len(pa), 1),), -7, np.int32)
        mm = np.full((1000, 2), -7, np.int32)
        res = _lib.Result()
        res.offsets = offs.ctypes.data_as(_lib._i64p)
        res.ok = okf.ctypes.data_as(_lib._i32p)
        res.matches = mm.ctypes.data
        res.good = None
        res.match_capacity = 1000
        Fa = None if F is None else np.ascontiguousarray(F, np.float64).reshape(-1, 9)
        st = L.msfm_match_pairs_guided(h, pa.ctypes.data, len(pa), C.byref(prm), None if Fa is None else Fa.ctypes.data, th,
                                       None if null_xy_table else C.cast(ptrs, C.c_void_p), np_.ctypes.data, n_images,
                                       C.byref(res))
        untouched = (offs == -7).all() and (okf == -7).all() and (mm == -7).all()
        return st, untouched, L.msfm_last_error(h).decode()

    bad_xy = s["xy_qry"].copy()
    bad_xy[17, 1] = np.nan
    inf_F = F.copy()
    inf_F[0, 1, 2] = np.inf
    big_F = F.copy()
    big_F[0, 0, 0] = 1e300  # finite in float64, not in fp32
    cases = {
        "null F": dict(F=None),
        "null keypoints of a touched image": dict(xy_list=(s["xy_ref"], None), npts=[200, 150]),
        "null keypoint table": dict(null_xy_table=True),
        "non-finite F": dict(F=inf_F),
        "F not finite in fp32": dict(F=big_F),
        "zero F": dict(F=np.zeros_like(F)),
        "npts differ from uploaded rows": dict(npts=[200, 149]),
        "non-finite keypoint": dict(xy_list=(s["xy_ref"], bad_xy)),
        "th zero": dict(th=0.0),
        "th negative": dict(th=-1.0),
        "th nan": dict(th=float("nan")),
        "th inf": dict(th=float("inf")),
        "rescore_band": dict(rescore=0.02),
        "image >= n_images": dict(n_images=1, xy_list=(s["xy_ref"],)),
    }
    for name, kw in cases.items():
        st, untouched, msg = call(**kw)
        assert st == 1, (name, st, msg)
        assert untouched, name
        assert matcher.timing() == before, name
        assert "guided" in msg, (name, msg)
    for name, kw in [("pair", dict(F=inf_F)), ("image 1", dict(npts=[200, 149])), ("image 1", dict(xy_list=(s["xy_ref"], bad_xy)))]:
        assert name in call(**kw)[2]
    # the image-id statuses are those of msfm_match_pairs
    assert call(pairs=[(0, 5)], F=F)[0] == 4  # MSFM_ERR_NOT_FOUND
    assert call(pairs=[(0, 99)], F=F)[0] == 1
    st, _, _ = call(pairs=np.zeros((0, 2)), F=np.zeros((0, 9)))
    assert st == 0


@pytest.mark.gpu
def test_cpp_mirror_matches_python(matcher, tmp_path):
    """MatchGraphB200::MatchPairsGuided (C++ host mirror, float descriptor rows) gives the Python binding's lists."""
    from metricsfm_b200 import build
    build.build_host_shim()
    s = decoy_scene(900, 700, 611, decoy_frac=0.5)
    (tmp_path / "d.f32").write_bytes(np.concatenate([s["ref"], s["qry"]]).astype(np.float32).tobytes())
    (tmp_path / "xy.f32").write_bytes(np.concatenate([s["xy_ref"], s["xy_qry"]]).astype(np.float32).tobytes())
    (tmp_path / "F.f64").write_bytes(np.ascontiguousarray(s["F"], np.float64).tobytes())
    out = subprocess.check_output([build.GUIDED_BIN, str(tmp_path / "d.f32"), str(len(s["ref"])), str(len(s["qry"])),
                                   str(tmp_path / "xy.f32"), str(tmp_path / "F.f64"), "3.0"], text=True).split("\n")
    pairs, F, xy = _load(matcher, [s])
    it = iter(out)
    for mutual in (0, 1):
        assert next(it).split() == ["MatchPairsGuided", "mutual", str(mutual), "ok", "1"]
        head = next(it).split()
        rows = np.array([next(it).split() for _ in range(int(head[-1]))], dtype=np.int32).reshape(-1, 3)
        res = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=3.0, ratio=0.85, ratio_good=0.6, mutual=bool(mutual))
        assert head[:3] == ["pair", "ok", str(int(res.ok[0]))]
        np.testing.assert_array_equal(rows[:, :2], res.pair(0))
        np.testing.assert_array_equal(rows[:, 2], res.pair_good(0))
        assert len(rows) > 0
