"""Float regime of homography-guided re-matching (msfm_match_pairs_guided_homography with rescore_band > 0 on a keep_float
context, HOMOG-SPEC in include/msfm_match.h): band rows of the H-gated quantised 2-NN are decided on their exact fp32
top-2 among the reference rows H carries to within th_transfer of the row's keypoint.  CPU: the proven candidate bound
T(q) under the H mask, and the restatement of oracle/homography_float_oracle.py against the integer H rule.  GPU: bit
for bit against that restatement through the collect path (the matching kernel's H-gated collect pass) and the brute
force, on a hand-built row the gate must change, and the integer paths, mutual filter, interleaving with the epipolar
gate and error statuses around it."""
import ctypes as C

import numpy as np
import pytest

from metricsfm_b200 import synth
from oracle import guided_float_oracle as gfo
from oracle import guided_oracle as gdo
from oracle import homography_float_oracle as hfo
from oracle import homography_oracle as ho
from test_float_regime import _adversarial
from test_guided_float import RULES, SIZES, _assert_equal, _collect_and_brute

REJECT_GT = 1
S512 = 512.0
COMP = 2.5  # companion noise: the disc ratios of the true matches spread around ratio 0.85


def _scene(seed, M, N, **kw):
    return hfo.float_planar_decoy_scene(seed, M, N, companion_sigma=COMP, **kw)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("th", [3.0, 1e15])
def test_h_gated_fp32_top2_lies_within_the_bound(oracle_mod, th):
    """DESIGN §8b under the H gate: with d1_q the gated quantised second distance, every fp32 top-2 row among the allowed
    rows has quantised distance <= T(q) = exact_threshold(d1_q, r_x, R)."""
    s = _scene(41, 900, 700)
    qr, qq = oracle_mod.quantize_f32(s["ref"], S512), oracle_mod.quantize_f32(s["qry"], S512)
    allowed = ho.gate_h32(s["H"], s["xy_ref"], s["xy_qry"], th)
    D = gdo.dist_u8(qr, qq)
    ids, d = gdo.masked_knn2(D, allowed)
    both = np.nonzero((ids[:, 0] >= 0) & (ids[:, 1] >= 0))[0]
    assert len(both) > 150
    if th == 3.0:
        barred_nn = ~allowed[np.arange(len(qq)), np.argmin(D, axis=1)]
        assert barred_nn[both].sum() > 10  # rows whose unconstrained quantised nearest row is barred
    fids, _ = gfo.masked_knn2_f32(s["ref"], s["qry"][both], allowed[both])
    T = gfo.exact_threshold(d[both, 1], gfo.residuals(s["qry"][both], S512), gfo.residuals(s["ref"], S512).max())
    for k in range(2):
        assert (fids[:, k] >= 0).all()
        assert allowed[both, fids[:, k]].all()
        assert (D[both, fids[:, k]] <= T).all()


def test_band_zero_restatement_is_the_integer_h_oracle(oracle_mod):
    """With band 0 (and for u8 rows) the restatement is homography_oracle's integer rule on the quantised rows; with a
    band, some rows' fp32 decision differs from the integer one (a GPU that ignored the band would not pass)."""
    s = _scene(51, 900, 800)
    qr, qq = oracle_mod.quantize_f32(s["ref"], S512), oracle_mod.quantize_f32(s["qry"], S512)
    for kw in (dict(ratio_good=0.6), dict(orientation=1, reject_gt=True), dict(max_dist_sq=20000.0)):
        a = hfo.match_pair_guided_h_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["H"], 3.0, 0.85, **kw)
        b = ho.match_pair_guided_h(qr, qq, s["xy_ref"], s["xy_qry"], s["H"], 3.0, 0.85, **kw)
        c = hfo.match_pair_guided_h_float(qr, qq, s["xy_ref"], s["xy_qry"], s["H"], 3.0, 0.85, band=0.2, float_rows=False, **kw)
        for x in (a, c):
            np.testing.assert_array_equal(x["pairs"], b["pairs"])
            np.testing.assert_array_equal(x["good"], b["good"])
    a = hfo.match_pair_guided_h_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["H"], 3.0, 0.85, band=0.02)
    b = ho.match_pair_guided_h(qr, qq, s["xy_ref"], s["xy_qry"], s["H"], 3.0, 0.85)
    assert a["band"].sum() > 20
    flips = {tuple(v) for v in a["pairs"].tolist()} ^ {tuple(v) for v in b["pairs"].tolist()}
    assert len(flips) > 5


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def fm(native_lib):
    from metricsfm_b200.matcher import Matcher
    m = Matcher(device=0, max_images=32, arena_rows=1 << 17, keep_float=True)
    yield m
    m.close()


def _load(m, scenes, u8=()):
    """Every scene as images (2s, 2s+1), float rows at scale 512 (u8 rows for the scene indices in `u8`).  Returns
    (pairs, H, F, image_xy)."""
    m.release_all()
    pairs, H, F, xy = [], [], [], {}
    for i, s in enumerate(scenes):
        for k, (rows, kp) in enumerate(((s["ref"], s["xy_ref"]), (s["qry"], s["xy_qry"]))):
            if i in u8:
                m.upload(2 * i + k, rows)
            else:
                m.upload(2 * i + k, np.ascontiguousarray(rows, np.float32), scale=S512)
            xy[2 * i + k] = kp
        pairs.append((2 * i, 2 * i + 1))
        H.append(s["H"])
        F.append(s["F"])
    return pairs, np.array(H), np.array(F), xy


def _call(m, pairs, H, xy, th, prm, band, mutual=False):
    return m.match_pairs_guided_homography(pairs, H, xy, th_transfer=th, ratio=prm.get("ratio", 0.85),
                                           ratio_good=prm.get("ratio_good", 0.0), max_dist_sq=prm.get("max_dist_sq", 0.0),
                                           min_keypoints=prm.get("min_keypoints", 20), orientation=prm.get("orientation", 0),
                                           flags=prm.get("flags", 0), rescore_band=band, mutual=mutual)


def _expect(s, th, prm, band, H=None):
    return hfo.match_pair_guided_h_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["H"] if H is None else H, th,
                                         prm.get("ratio", 0.85), band=band, ratio_good=prm.get("ratio_good", 0.0),
                                         max_dist_sq=prm.get("max_dist_sq", 0.0), min_keypoints=prm.get("min_keypoints", 20),
                                         orientation=prm.get("orientation", 0), reject_gt=bool(prm.get("flags", 0) & REJECT_GT))


@pytest.mark.gpu
@pytest.mark.parametrize("band", [0.02, 0.2])
@pytest.mark.parametrize("th", [3.0, 150.0])
def test_sizes_rules_and_bands_vs_restatement(fm, th, band):
    """Ragged and edge sizes (min_keypoints 0), duplicated rows, rows with zero or one allowed reference row at 3 px;
    ratio 0.85 + ratio_good 0.6, REJECT_GT with orientation 1, max_dist_sq; collect path and brute force."""
    scenes = [_scene(100 + i, M, N, companions=i % 2 == 0) for i, (M, N) in enumerate(SIZES)]
    pairs, H, _, xy = _load(fm, scenes)
    n_band = 0
    for prm in RULES:
        prm = {**prm, "min_keypoints": 0}
        exps = [_expect(s, th, prm, band) for s in scenes]
        n_band += _collect_and_brute(fm, lambda: _call(fm, pairs, H, xy, th, prm, band), exps, f"th {th} band {band} {prm}")
        if th == 3.0:
            n_allowed = np.concatenate([e["allowed"].sum(1) for e in exps if e["allowed"] is not None])
            assert (n_allowed == 0).sum() > 100 and (n_allowed == 1).sum() > 100
    assert n_band > 0


def _embed_barred(case="wrong_ref"):
    """A float planar scene with the rows of test_float_regime's `case` (reference rows A, B, C; query row x) embedded:
    x at three query rows sharing one keypoint, A and C at the reference point H carries onto it, B 100 px from there
    (outside every few-pixel disc)."""
    s = _scene(61, 1500, 1200)
    adv_ref, x = _adversarial(case)
    pos, qpos = [5, 700, 1499], [0, 611, 1199]
    ref, qry, xy_ref, xy_qry = s["ref"].copy(), s["qry"].copy(), s["xy_ref"].copy(), s["xy_qry"].copy()
    ref[pos], qry[qpos] = adv_ref, x
    xy_qry[qpos] = xy_qry[qpos[0]]
    p = np.linalg.solve(np.asarray(s["H"], np.float64).reshape(3, 3), np.r_[xy_qry[qpos[0]].astype(np.float64), 1.0])
    u = p[:2] / p[2]
    for i, pj in enumerate(pos):
        xy_ref[pj] = u + (np.array([100.0, 0.0]) if i == 1 else 0.0)
    return dict(s, ref=ref, qry=qry, xy_ref=xy_ref, xy_qry=xy_qry), pos, qpos


def test_hand_built_barred_row_restatement(oracle_mod):
    """B is the fp32 nearest row of x and lies within T(q) computed from the H-gated d1_q, but lies outside the disc:
    the restatement decides x on {A, C} and emits (A, x)."""
    s, pos, qpos = _embed_barred()
    allowed = ho.gate_h32(s["H"], s["xy_ref"], s["xy_qry"], 3.0)
    assert allowed[qpos][:, [pos[0], pos[2]]].all() and not allowed[qpos][:, pos[1]].any()
    fids, _ = oracle_mod.knn2_f32(s["ref"], s["qry"][qpos])
    assert (fids[:, 0] == pos[1]).all()  # ungated fp32 nearest: B
    exp = _expect(s, 3.0, dict(ratio=0.85), 0.02)
    assert exp["band"][qpos].all()
    qr, qq = oracle_mod.quantize_f32(s["ref"], S512), oracle_mod.quantize_f32(s["qry"][qpos[:1]], S512)
    T = gfo.exact_threshold(exp["dists"][qpos[0], 1], gfo.residuals(s["qry"][qpos[:1]], S512)[0],
                            gfo.residuals(s["ref"], S512).max())
    assert gdo.dist_u8(qr, qq)[0, pos[1]] <= T
    assert {int(q): int(j) for j, q in exp["pairs"].tolist() if q in qpos} == {q: pos[0] for q in qpos}


@pytest.mark.gpu
def test_hand_built_barred_row(fm):
    s, pos, qpos = _embed_barred()
    pairs, H, _, xy = _load(fm, [s])
    exp = _expect(s, 3.0, dict(ratio=0.85), 0.02)
    _collect_and_brute(fm, lambda: _call(fm, pairs, H, xy, 3.0, dict(ratio=0.85), 0.02), [exp], "barred B")
    plain = fm.match_pairs(pairs, 0.85, rescore_band=0.02)  # without the gate B wins
    assert {int(q): int(j) for j, q in plain.pair(0).tolist() if q in qpos} == {q: pos[1] for q in qpos}


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [False, True])
def test_admit_all_gate_equals_match_pairs(fm, mutual):
    scenes = [_scene(400 + i, M, N) for i, (M, N) in enumerate([(900, 800), (129, 300), (40, 41)])]
    pairs, H, _, xy = _load(fm, scenes)
    for band in (0.02, 0.2):
        plain = fm.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual, rescore_band=band)
        guided = fm.match_pairs_guided_homography(pairs, H, xy, th_transfer=1e15, ratio=0.85, ratio_good=0.6, mutual=mutual,
                                                  rescore_band=band)
        np.testing.assert_array_equal(guided.offsets, plain.offsets)
        np.testing.assert_array_equal(guided.ok, plain.ok)
        np.testing.assert_array_equal(guided.matches, plain.matches)
        np.testing.assert_array_equal(guided.good, plain.good)


@pytest.mark.gpu
def test_pruning_off_gives_identical_lists(fm):
    scenes = [_scene(500 + i, M, N) for i, (M, N) in enumerate([(2000, 1500), (700, 900)])]
    pairs, H, _, xy = _load(fm, scenes)
    for mutual in (False, True):
        for th, band in ((3.0, 0.02), (40.0, 0.2)):
            kw = dict(th_transfer=th, ratio=0.85, ratio_good=0.6, mutual=mutual, rescore_band=band)
            on = fm.match_pairs_guided_homography(pairs, H, xy, **kw)
            fm._test_disable_pruning(True)
            try:
                off = fm.match_pairs_guided_homography(pairs, H, xy, **kw)
            finally:
                fm._test_disable_pruning(False)
            np.testing.assert_array_equal(on.offsets, off.offsets)
            np.testing.assert_array_equal(on.matches, off.matches)
            np.testing.assert_array_equal(on.good, off.good)


@pytest.mark.gpu
def test_one_call_over_several_batches_equals_per_pair_calls(native_lib):
    """17 000 pairs (more than one 16 384-pair batch) of 64-row float images drawn with repetition, plane Hs: one call
    equals a call per distinct pair."""
    from metricsfm_b200.matcher import Matcher
    n_img, rows = 24, 64
    rng = np.random.default_rng(601)
    col = synth.Collection(rows, seed=601)
    xy = {i: rng.uniform(-1800, 1800, (rows, 2)).astype(np.float32) for i in range(n_img)}
    Hs = [ho.plane_views(rng)[1] for _ in range(16)]
    pairs = rng.integers(0, n_img, size=(17000, 2)).astype(np.int32)
    H = np.array([Hs[(int(r) * 7 + int(q)) % len(Hs)] for r, q in pairs])
    kw = dict(th_transfer=1200.0, ratio=0.85, ratio_good=0.6, rescore_band=0.2, min_keypoints=0)
    with Matcher(device=0, max_images=n_img, arena_rows=1 << 15, keep_float=True) as m:
        for i in range(n_img):
            m.upload(i, col.image_unit(i), scale=S512)
        one = m.match_pairs_guided_homography(pairs, H, xy, **kw)
        assert m.timing()["match_launches"] >= 2
        events, brute = m._test_last_knn_stats()
        assert events > 0 or brute > 0, (events, brute)  # band rows were re-scored (collected, or by the brute force)
        assert len(one.matches) > 0
        done = {}
        for p, (r, q) in enumerate(pairs.tolist()):
            if (r, q) not in done:
                done[(r, q)] = m.match_pairs_guided_homography(pairs[p:p + 1], H[p:p + 1], xy, **kw)
            ref = done[(r, q)]
            np.testing.assert_array_equal(ref.pair(0), one.pair(p))
            np.testing.assert_array_equal(ref.pair_good(0), one.pair_good(p))


@pytest.mark.gpu
def test_u8_pair_follows_the_integer_h_rule(fm):
    """A u8 pair (and a u8 image paired with a float image) on a keep_float context: the integer H rule."""
    scenes = [_scene(700 + i, 800, 700) for i in range(2)]
    q8 = [dict(s, ref=synth.quantize_512(s["ref"]), qry=synth.quantize_512(s["qry"])) for s in scenes]
    pairs, H, _, xy = _load(fm, q8[:1] + scenes[1:], u8=(0,))
    pairs.append((0, 3))
    H = np.concatenate([H, H[:1]])
    res = fm.match_pairs_guided_homography(pairs, H, xy, th_transfer=3.0, ratio=0.85, ratio_good=0.6, rescore_band=0.2)
    exp0 = ho.match_pair_guided_h(q8[0]["ref"], q8[0]["qry"], q8[0]["xy_ref"], q8[0]["xy_qry"], H[0], 3.0, 0.85, ratio_good=0.6)
    exp1 = _expect(scenes[1], 3.0, dict(ratio=0.85, ratio_good=0.6), 0.2)
    assert exp1["band"].sum() > 0
    qry3 = gfo.oracle.quantize_f32(scenes[1]["qry"], S512)
    exp2 = ho.match_pair_guided_h(q8[0]["ref"], qry3, q8[0]["xy_ref"], scenes[1]["xy_qry"], H[0], 3.0, 0.85, ratio_good=0.6)
    _assert_equal(res, [exp0, exp1, exp2], "u8 / float / mixed")


@pytest.mark.gpu
def test_mutual_matches_are_one_way_matches(fm):
    """Mutual on: the float regime's heuristic filter of the one-way list, under the H gate."""
    scenes = [_scene(800 + i, M, N) for i, (M, N) in enumerate([(1500, 1200), (600, 900)])]
    pairs, H, _, xy = _load(fm, scenes)
    for th, band in ((3.0, 0.02), (150.0, 0.2)):
        kw = dict(th_transfer=th, ratio=0.85, ratio_good=0.6, rescore_band=band)
        one = fm.match_pairs_guided_homography(pairs, H, xy, **kw)
        mut = fm.match_pairs_guided_homography(pairs, H, xy, mutual=True, **kw)
        for k in range(len(pairs)):
            ow = {tuple(v): g for v, g in zip(one.pair(k).tolist(), one.pair_good(k).tolist())}
            assert mut.pair(k).shape[0] > 0
            for v, g in zip(mut.pair(k).tolist(), mut.pair_good(k).tolist()):
                assert ow.get(tuple(v)) == g, (th, band, k, v)


@pytest.mark.gpu
def test_interleaved_with_epipolar_gate(fm):
    """F-guided and H-guided float calls alternate on one context, through the collect path and the brute force; each
    equals its own restatement (no gate state leaks from one call into the next)."""
    scenes = [_scene(550 + i, M, N) for i, (M, N) in enumerate([(900, 700), (500, 650)])]
    pairs, H, F, xy = _load(fm, scenes)
    prm = dict(ratio=0.85, ratio_good=0.6)
    exp_h = [_expect(s, 4.0, prm, 0.02) for s in scenes]
    exp_f = [gfo.match_pair_guided_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 4.0, 0.85, band=0.02,
                                         ratio_good=0.6) for s in scenes]
    assert sum(int(e["band"].sum()) for e in exp_h) > 0 and sum(int(e["band"].sum()) for e in exp_f) > 0
    for _ in range(2):
        _collect_and_brute(fm, lambda: _call(fm, pairs, H, xy, 4.0, prm, 0.02), exp_h, "H")
        _collect_and_brute(fm, lambda: fm.match_pairs_guided(pairs, F, xy, th_epipolar=4.0, ratio=0.85, ratio_good=0.6,
                                                             rescore_band=0.02), exp_f, "F")


@pytest.mark.gpu
def test_bad_band_is_refused_before_launch(fm):
    """Negative, NaN and infinite bands on a keep_float context: INVALID_ARG naming the entry point, outputs and
    msfm_last_timing untouched."""
    from metricsfm_b200 import _lib
    s = _scene(900, 200, 150)
    pairs, H, _, xy = _load(fm, [s])
    fm.match_pairs_guided_homography(pairs, H, xy, th_transfer=3.0, ratio=0.85, rescore_band=0.02)
    before = fm.timing()
    L, h = fm._L, fm._h
    pa = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
    arrs = [np.ascontiguousarray(s["xy_ref"], np.float32), np.ascontiguousarray(s["xy_qry"], np.float32)]
    ptrs = (C.c_void_p * 2)(*[a.ctypes.data for a in arrs])
    npts = np.array([200, 150], np.int32)
    Ha = np.ascontiguousarray(H, np.float64).reshape(-1, 9)
    for band in (-0.02, float("nan"), float("inf"), float("-inf")):
        prm = fm._params(0.85, 0.6, 0.0, False, 20, 0, band, 0)
        offs = np.full((2,), -7, np.int64)
        okf = np.full((1,), -7, np.int32)
        mm = np.full((400, 2), -7, np.int32)
        res = _lib.Result()
        res.offsets = offs.ctypes.data_as(_lib._i64p)
        res.ok = okf.ctypes.data_as(_lib._i32p)
        res.matches = mm.ctypes.data
        res.good = None
        res.match_capacity = 400
        st = L.msfm_match_pairs_guided_homography(h, pa.ctypes.data, len(pa), C.byref(prm), Ha.ctypes.data, 3.0,
                                                  C.cast(ptrs, C.c_void_p), npts.ctypes.data, 2, C.byref(res))
        assert st == 1, band
        assert (offs == -7).all() and (okf == -7).all() and (mm == -7).all(), band
        assert fm.timing() == before, band
        assert "guided_homography" in L.msfm_last_error(h).decode(), band
