"""Homography-guided re-matching (msfm_match_pairs_guided_homography, HOMOG-SPEC in include/msfm_match.h): the float32
transfer gate, the masked 2-NN and mutual check against the numpy restatement in oracle/homography_oracle.py, bit for bit;
the planar scene with look-alikes on the epipolar line, which the homography gate separates and the epipolar gate cannot;
batching, pruning, interleaving with the epipolar gate, the match -> geo_homography -> guided sequence, the error
statuses and the C++ mirror."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from metricsfm_b200 import synth
from oracle import guided_oracle as gdo
from oracle import homography_oracle as ho

REJECT_GT = 1
SIZES = [(1, 1), (19, 20), (20, 19), (21, 21), (127, 128), (128, 129), (129, 127), (2000, 1999)]


# ------------------------------------------------------------------------------------------------ CPU: the oracle
@pytest.mark.parametrize("M,N", [(1, 1), (19, 21), (128, 127), (300, 257)])
def test_oracle_admit_all_gate_is_plain_knn2(oracle_mod, M, N):
    s = ho.planar_decoy_scene(11 + M, M, N)
    allowed = ho.gate_h32(s["H"], s["xy_ref"], s["xy_qry"], 1e15)
    assert allowed.all()
    D = gdo.dist_u8(s["ref"], s["qry"])
    ids, dists = gdo.masked_knn2(D, allowed)
    oids, odists = oracle_mod.knn2_u8(s["ref"], s["qry"])
    np.testing.assert_array_equal(ids, oids)
    np.testing.assert_array_equal(dists, odists)
    np.testing.assert_array_equal(gdo.masked_colbest(D, allowed), oracle_mod.colbest_u8(s["ref"], s["qry"])[0])


def test_oracle_planar_scene_separates_the_gates():
    """The capability, on the oracle alone (seeded): H keeps >= 90 % of the decoyed true matches, F <= 10 %."""
    s = ho.planar_decoy_scene(1, 1400, 900)
    rh = ho.match_pair_guided_h(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["H"], 4.0, 0.85, ratio_good=0.6)
    rf = gdo.match_pair_guided(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 4.0, 0.85, ratio_good=0.6)
    nd = len(s["decoyed"])
    assert ho.kept(rh["pairs"], s["decoyed"]) >= 0.9 * nd
    assert ho.kept(rf["pairs"], s["decoyed"]) <= 0.1 * nd


def test_oracle_planar_scene_without_companions():
    """The gate's limit, on the oracle alone (seeded): without a second keypoint at each true reference keypoint, a 4 px
    disc almost never holds two reference rows, every such row is rejected, and the H gate keeps no true match where the
    F gate keeps about half of them."""
    s = ho.planar_decoy_scene(1, 1400, 900, companions=False)
    rh = ho.match_pair_guided_h(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["H"], 4.0, 0.85, ratio_good=0.6)
    rf = gdo.match_pair_guided(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 4.0, 0.85, ratio_good=0.6)
    assert (rh["allowed"].sum(1) < 2).mean() > 0.99
    assert ho.kept(rh["pairs"], s["true"]) == 0
    assert ho.kept(rf["pairs"], s["true"]) >= 0.4 * len(s["true"])


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def matcher(native_lib):
    from metricsfm_b200.matcher import Matcher
    m = Matcher(device=0, max_images=16, arena_rows=1 << 16)
    yield m
    m.close()


def _load(m, scenes):
    """Upload every scene as images (2s, 2s+1); returns (pairs, H [n,3,3], F [n,3,3], image_xy)."""
    m.release_all()
    pairs, H, F, xy = [], [], [], {}
    for i, s in enumerate(scenes):
        m.upload(2 * i, s["ref"])
        m.upload(2 * i + 1, s["qry"])
        pairs.append((2 * i, 2 * i + 1))
        H.append(s["H"])
        F.append(s["F"])
        xy[2 * i], xy[2 * i + 1] = s["xy_ref"], s["xy_qry"]
    return pairs, np.array(H), np.array(F), xy


def _expect(s, th, ratio, H=None, **kw):
    return ho.match_pair_guided_h(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["H"] if H is None else H, th, ratio, **kw)


def _check(res, p, exp, ratio_good):
    assert bool(res.ok[p]) == exp["ok"]
    np.testing.assert_array_equal(res.pair(p), exp["pairs"].reshape(-1, 2))
    if ratio_good > 0:
        np.testing.assert_array_equal(res.pair_good(p), exp["good"])


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [False, True])
@pytest.mark.parametrize("th", [3.0, 150.0])
def test_sizes_ties_and_sparse_rows_vs_oracle(matcher, mutual, th):
    scenes = [ho.planar_decoy_scene(100 + i, M, N, companions=i % 2 == 0) for i, (M, N) in enumerate(SIZES)]
    pairs, H, _, xy = _load(matcher, scenes)
    res = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=th, ratio=0.85, ratio_good=0.6, mutual=mutual,
                                                min_keypoints=0)
    zero = one = 0
    for p, s in enumerate(scenes):
        exp = _expect(s, th, 0.85, ratio_good=0.6, mutual=mutual, min_keypoints=0)
        _check(res, p, exp, 0.6)
        n_allowed = exp["allowed"].sum(1)
        zero += int((n_allowed == 0).sum())
        one += int((n_allowed == 1).sum())
    if th == 3.0:
        assert zero > 100 and one > 100  # rows with zero and with one allowed reference row are exercised


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [False, True])
def test_rule_variants_vs_oracle(matcher, mutual):
    scenes = [ho.planar_decoy_scene(200 + i, M, N) for i, (M, N) in enumerate([(600, 500), (300, 700), (15, 400)])]
    pairs, H, _, xy = _load(matcher, scenes)
    for orientation, ratio_good, max_dist_sq, flags in [(0, 0.6, 0.0, 0), (1, 0.0, 0.0, 0), (0, 0.6, 40000.0, 0),
                                                         (1, 0.7, 0.0, REJECT_GT), (0, 0.0, 60000.0, REJECT_GT)]:
        res = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=8.0, ratio=0.8, ratio_good=ratio_good,
                                                    max_dist_sq=max_dist_sq, mutual=mutual, orientation=orientation,
                                                    flags=flags)
        assert res.ok.tolist() == [1, 1, 0]
        for p, s in enumerate(scenes):
            exp = _expect(s, 8.0, 0.8, mutual=mutual, orientation=orientation, ratio_good=ratio_good, max_dist_sq=max_dist_sq,
                          reject_gt=bool(flags & REJECT_GT))
            _check(res, p, exp, ratio_good)


@pytest.mark.gpu
def test_planar_decoys_separate_the_gates(matcher):
    """The feature's purpose: look-alikes on the epipolar line pass the F gate, so the F-guided ratio test rejects the
    true matches; the H gate removes them.  Thresholds from the seeded oracle (test_oracle_planar_scene_separates_the_gates)."""
    s = ho.planar_decoy_scene(1, 1400, 900)
    pairs, H, F, xy = _load(matcher, [s])
    nd = len(s["decoyed"])
    for mutual in (False, True):
        hg = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=4.0, ratio=0.85, ratio_good=0.6, mutual=mutual)
        assert matcher.timing()["twin_pairs"] == int(mutual)
        fg = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=4.0, ratio=0.85, ratio_good=0.6, mutual=mutual)
        _check(hg, 0, _expect(s, 4.0, 0.85, ratio_good=0.6, mutual=mutual), 0.6)
        _check(fg, 0, gdo.match_pair_guided(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 4.0, 0.85, ratio_good=0.6,
                                            mutual=mutual), 0.6)
        kh, kf = ho.kept(hg.pair(0), s["decoyed"]), ho.kept(fg.pair(0), s["decoyed"])
        print(f"mutual={mutual}: decoyed true matches kept: H {kh}, F {kf} of {nd}")
        assert kh >= 0.9 * nd and kf <= 0.1 * nd


@pytest.mark.gpu
def test_planar_scene_without_companions_vs_oracle(matcher):
    """The same scene without the co-located second keypoints: both gated lists equal their oracles, and the H gate keeps
    no true match while the F gate keeps about half (test_oracle_planar_scene_without_companions)."""
    s = ho.planar_decoy_scene(1, 1400, 900, companions=False)
    pairs, H, F, xy = _load(matcher, [s])
    for mutual in (False, True):
        hg = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=4.0, ratio=0.85, ratio_good=0.6, mutual=mutual)
        fg = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=4.0, ratio=0.85, ratio_good=0.6, mutual=mutual)
        _check(hg, 0, _expect(s, 4.0, 0.85, ratio_good=0.6, mutual=mutual), 0.6)
        _check(fg, 0, gdo.match_pair_guided(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 4.0, 0.85, ratio_good=0.6,
                                            mutual=mutual), 0.6)
        assert ho.kept(hg.pair(0), s["true"]) == 0
        assert ho.kept(fg.pair(0), s["true"]) >= 0.4 * len(s["true"])


@pytest.mark.gpu
@pytest.mark.parametrize("gate", ["huge_threshold", "collapsing_H"])
@pytest.mark.parametrize("mutual", [False, True])
def test_admit_all_gate_equals_match_pairs(matcher, mutual, gate):
    """A gate that admits every element reproduces msfm_match_pairs.  huge_threshold: the scene's H with th = 1e15 (the
    t2 side admits everything).  collapsing_H: H = diag(0, 0, 1) carries every reference keypoint to the origin, and th
    just above the largest query keypoint radius admits every element through the transfer test itself (no nonzero H
    admits every element at every th: the query keypoints spread over the image)."""
    scenes = [ho.planar_decoy_scene(400 + i, M, N) for i, (M, N) in enumerate([(900, 800), (129, 300), (40, 41)])]
    pairs, H, _, xy = _load(matcher, scenes)
    th = 1e15
    if gate == "collapsing_H":
        H = np.repeat(np.diag([0.0, 0.0, 1.0])[None], len(scenes), 0)
        th = float(np.ceil(max(np.sqrt((s["xy_qry"].astype(np.float64) ** 2).sum(1)).max() for s in scenes))) + 1.0
        for s in scenes:
            assert ho.gate_h32(H[0], s["xy_ref"], s["xy_qry"], th).all()
    plain = matcher.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual)
    guided = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=th, ratio=0.85, ratio_good=0.6, mutual=mutual)
    np.testing.assert_array_equal(guided.offsets, plain.offsets)
    np.testing.assert_array_equal(guided.ok, plain.ok)
    np.testing.assert_array_equal(guided.matches, plain.matches)
    np.testing.assert_array_equal(guided.good, plain.good)


@pytest.mark.gpu
def test_pruning_off_gives_identical_lists(matcher):
    scenes = [ho.planar_decoy_scene(500 + i, M, N) for i, (M, N) in enumerate([(2000, 1500), (700, 900)])]
    pairs, H, _, xy = _load(matcher, scenes)
    for mutual in (False, True):
        for th in (3.0, 40.0):
            on = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=th, ratio=0.85, ratio_good=0.6, mutual=mutual)
            matcher._test_disable_pruning(True)
            try:
                off = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=th, ratio=0.85, ratio_good=0.6,
                                                            mutual=mutual)
            finally:
                matcher._test_disable_pruning(False)
            np.testing.assert_array_equal(on.offsets, off.offsets)
            np.testing.assert_array_equal(on.matches, off.matches)
            np.testing.assert_array_equal(on.good, off.good)


@pytest.mark.gpu
def test_interleaved_with_epipolar_gate(matcher):
    """F-guided and H-guided calls alternate on one context; each equals its own oracle."""
    scenes = [ho.planar_decoy_scene(550 + i, M, N) for i, (M, N) in enumerate([(900, 700), (500, 650)])]
    pairs, H, F, xy = _load(matcher, scenes)
    for mutual in (False, True, False):
        hg = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=4.0, ratio=0.85, ratio_good=0.6, mutual=mutual)
        fg = matcher.match_pairs_guided(pairs, F, xy, th_epipolar=4.0, ratio=0.85, ratio_good=0.6, mutual=mutual)
        for p, s in enumerate(scenes):
            _check(hg, p, _expect(s, 4.0, 0.85, ratio_good=0.6, mutual=mutual), 0.6)
            _check(fg, p, gdo.match_pair_guided(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 4.0, 0.85, ratio_good=0.6,
                                                mutual=mutual), 0.6)


@pytest.mark.gpu
def test_one_call_over_several_batches_equals_per_pair_calls(native_lib):
    """100 images x 8192 rows, all 4950 pairs (~40 M query rows, more than one 16 Mi-row batch) with plane Hs."""
    from metricsfm_b200.matcher import Matcher
    n_img, rows = 100, 8192
    rng = np.random.default_rng(600)
    col = synth.Collection(rows, seed=600)
    xy = {i: rng.uniform(-1800, 1800, (rows, 2)).astype(np.float32) for i in range(n_img)}
    Hs = [ho.plane_views(rng)[1] for _ in range(64)]
    pairs = synth.exhaustive_pairs(n_img)
    H = np.array([Hs[p % len(Hs)] for p in range(len(pairs))])
    with Matcher(device=0, max_images=n_img, arena_rows=n_img * rows + (1 << 16)) as m:
        m.upload_batch(list(range(n_img)), [col.image_u8(i) for i in range(n_img)])
        one = m.match_pairs_guided_homography(pairs, H, xy, th_transfer=60.0, ratio=0.85, ratio_good=0.6, mutual=True)
        t = m.timing()
        assert t["match_launches"] >= 4
        assert t["twin_pairs"] == len(pairs)
        assert len(one.matches) > 0
        for p in range(0, len(pairs), 7):
            r = m.match_pairs_guided_homography(pairs[p:p + 1], H[p:p + 1], xy, th_transfer=60.0, ratio=0.85, ratio_good=0.6,
                                                mutual=True)
            np.testing.assert_array_equal(r.pair(0), one.pair(p))
            np.testing.assert_array_equal(r.pair_good(0), one.pair_good(p))


@pytest.mark.gpu
def test_end_to_end_after_geo_homography(matcher):
    """match_pairs -> geo_homography -> match_pairs_guided_homography with the H geo_homography returned."""
    scenes = [ho.planar_decoy_scene(700 + i, M, N) for i, (M, N) in enumerate([(1200, 900), (800, 1000), (600, 700)])]
    pairs, _, _, xy = _load(matcher, scenes)
    first = matcher.match_pairs(pairs, 0.85, ratio_good=0.6)
    ok, inl, mask, H = matcher.geo_homography(pairs, first, xy, th=3.0, seed=5)
    assert ok.sum() >= 2
    sel = [p for p in range(len(pairs)) if ok[p]]
    res = matcher.match_pairs_guided_homography([pairs[p] for p in sel], H[sel], xy, th_transfer=4.0, ratio=0.85,
                                                ratio_good=0.6, mutual=True)
    for k, p in enumerate(sel):
        s = scenes[p]
        _check(res, k, _expect(s, 4.0, 0.85, H=H[p], ratio_good=0.6, mutual=True), 0.6)
        assert ho.kept(res.pair(k), s["true"]) > ho.kept(first.pair(p), s["true"])


@pytest.mark.gpu
def test_error_statuses_before_launch(matcher):
    from metricsfm_b200 import _lib
    s = ho.planar_decoy_scene(800, 200, 150)
    pairs, H, _, xy = _load(matcher, [s])
    matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=3.0, ratio=0.85)
    before = matcher.timing()
    assert before["match_launches"] >= 1
    L, h = matcher._L, matcher._h

    def call(H=H, th=3.0, xy_list=(s["xy_ref"], s["xy_qry"]), npts=None, n_images=2, pairs=pairs, null_xy_table=False,
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
        Ha = None if H is None else np.ascontiguousarray(H, np.float64).reshape(-1, 9)
        st = L.msfm_match_pairs_guided_homography(h, pa.ctypes.data, len(pa), C.byref(prm), None if Ha is None else Ha.ctypes.data,
                                                  th, None if null_xy_table else C.cast(ptrs, C.c_void_p), np_.ctypes.data,
                                                  n_images, C.byref(res))
        untouched = (offs == -7).all() and (okf == -7).all() and (mm == -7).all()
        return st, untouched, L.msfm_last_error(h).decode()

    bad_xy = s["xy_qry"].copy()
    bad_xy[17, 1] = np.nan
    inf_H = H.copy()
    inf_H[0, 1, 2] = np.inf
    big_H = H.copy()
    big_H[0, 0, 0] = 1e300
    tiny_H = np.full_like(H, 1e-50)  # non-zero in float64, zero in fp32
    cases = {
        "null H": dict(H=None),
        "null keypoints of a touched image": dict(xy_list=(s["xy_ref"], None), npts=[200, 150]),
        "null keypoint table": dict(null_xy_table=True),
        "non-finite H": dict(H=inf_H),
        "H not finite in fp32": dict(H=big_H),
        "zero H": dict(H=np.zeros_like(H)),
        "H zero in fp32": dict(H=tiny_H),
        "npts differ from uploaded rows": dict(npts=[200, 149]),
        "non-finite keypoint": dict(xy_list=(s["xy_ref"], bad_xy)),
        "th zero": dict(th=0.0),
        "th negative": dict(th=-1.0),
        "th nan": dict(th=float("nan")),
        "th inf": dict(th=float("inf")),
        "rescore_band > 0": dict(rescore=0.02),
        "rescore_band negative": dict(rescore=-0.02),
        "image >= n_images": dict(n_images=1, xy_list=(s["xy_ref"],)),
    }
    for name, kw in cases.items():
        st, untouched, msg = call(**kw)
        assert st == 1, (name, st, msg)
        assert untouched, name
        assert matcher.timing() == before, name
        assert "guided_homography" in msg, (name, msg)
    for name, kw in [("pair", dict(H=inf_H)), ("image 1", dict(npts=[200, 149])), ("image 1", dict(xy_list=(s["xy_ref"], bad_xy)))]:
        assert name in call(**kw)[2]
    assert call(pairs=[(0, 5)])[0] == 4  # MSFM_ERR_NOT_FOUND
    assert call(pairs=[(0, 99)])[0] == 1
    st, _, _ = call(pairs=np.zeros((0, 2)), H=np.zeros((0, 9)))
    assert st == 0


@pytest.mark.gpu
def test_cpp_mirror_matches_python(matcher, tmp_path):
    """MatchGraphB200::MatchPairsGuidedHomography (C++ host mirror, float descriptor rows) gives the Python binding's lists."""
    from metricsfm_b200 import build
    build.build_host_shim()
    s = ho.planar_decoy_scene(900, 700, 611)
    (tmp_path / "d.f32").write_bytes(np.concatenate([s["ref"], s["qry"]]).astype(np.float32).tobytes())
    (tmp_path / "xy.f32").write_bytes(np.concatenate([s["xy_ref"], s["xy_qry"]]).astype(np.float32).tobytes())
    (tmp_path / "H.f64").write_bytes(np.ascontiguousarray(s["H"], np.float64).tobytes())
    out = subprocess.check_output([build.HOMOGRAPHY_BIN, str(tmp_path / "d.f32"), str(len(s["ref"])), str(len(s["qry"])),
                                   str(tmp_path / "xy.f32"), str(tmp_path / "H.f64"), "4.0"], text=True).split("\n")
    pairs, H, _, xy = _load(matcher, [s])
    it = iter(out)
    for mutual in (0, 1):
        assert next(it).split() == ["MatchPairsGuidedHomography", "mutual", str(mutual), "ok", "1"]
        head = next(it).split()
        rows = np.array([next(it).split() for _ in range(int(head[-1]))], dtype=np.int32).reshape(-1, 3)
        res = matcher.match_pairs_guided_homography(pairs, H, xy, th_transfer=4.0, ratio=0.85, ratio_good=0.6,
                                                    mutual=bool(mutual))
        assert head[:3] == ["pair", "ok", str(int(res.ok[0]))]
        np.testing.assert_array_equal(rows[:, :2], res.pair(0))
        np.testing.assert_array_equal(rows[:, 2], res.pair_good(0))
        assert len(rows) > 0
