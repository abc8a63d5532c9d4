"""Float regime of guided re-matching (msfm_match_pairs_guided with rescore_band > 0 on a keep_float context,
GUIDED-SPEC in include/msfm_match.h): band rows of the gated quantised 2-NN are decided on their exact fp32 top-2
among the reference rows the epipolar gate allows.  CPU: the masked fp32 2-NN of oracle/guided_float_oracle.py, and the
proven candidate bound T(q) under a gate.  GPU: bit for bit against that restatement through the collect path (the
matching kernel's gated collect pass) and the brute force, on hand-built rows the gate must change, and the integer
paths, mutual filter and error statuses around it."""
import ctypes as C

import numpy as np
import pytest

from metricsfm_b200 import synth
from oracle import geo_oracle as go
from oracle import guided_float_oracle as gfo
from oracle import guided_oracle as gdo
from oracle.guided_oracle import eight_point
from test_float_regime import _adversarial

REJECT_GT = 1
S512 = 512.0


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("M,N", [(1, 1), (19, 21), (130, 127), (300, 257)])
def test_admit_all_masked_f32_knn2_is_the_fp32_oracle(oracle_mod, M, N):
    s = gfo.float_decoy_scene(31 + M, M, N)
    allowed = gdo.gate_f32(s["F"], s["xy_ref"], s["xy_qry"], 1e15)
    assert allowed.all()
    ids, dists = gfo.masked_knn2_f32(s["ref"], s["qry"], allowed)
    oids, odists = oracle_mod.knn2_f32(s["ref"], s["qry"])
    np.testing.assert_array_equal(ids, oids)
    np.testing.assert_array_equal(dists, odists)


@pytest.mark.parametrize("seed,th", [(41, 3.0), (42, 20.0), (43, 150.0)])
def test_gated_fp32_top2_lies_within_the_bound(oracle_mod, seed, th):
    """DESIGN §8b: with d1_q the gated quantised second distance, every fp32 top-2 row among the allowed rows has
    quantised distance <= T(q) = exact_threshold(d1_q, r_x, R); the scenes include rows whose unconstrained quantised
    nearest row is barred."""
    s = gfo.float_decoy_scene(seed, 900, 700, decoy_frac=0.5)
    qr, qq = oracle_mod.quantize_f32(s["ref"], S512), oracle_mod.quantize_f32(s["qry"], S512)
    allowed = gdo.gate_f32(s["F"], s["xy_ref"], s["xy_qry"], th)
    D = gdo.dist_u8(qr, qq)
    ids, d = gdo.masked_knn2(D, allowed)
    both = np.nonzero((ids[:, 0] >= 0) & (ids[:, 1] >= 0))[0]
    assert len(both) > 50
    barred_nn = ~allowed[np.arange(len(qq)), np.argmin(D, axis=1)]
    assert barred_nn[both].sum() > 10
    fids, _ = gfo.masked_knn2_f32(s["ref"], s["qry"][both], allowed[both])
    T = gfo.exact_threshold(d[both, 1], gfo.residuals(s["qry"][both], S512), gfo.residuals(s["ref"], S512).max())
    for k in range(2):
        assert (fids[:, k] >= 0).all()
        assert allowed[both, fids[:, k]].all()
        assert (D[both, fids[:, k]] <= T).all()


def test_band_zero_restatement_is_the_integer_guided_oracle(oracle_mod):
    """With band 0 (and for u8 rows) the restatement is oracle.guided_oracle's integer rule on the quantised rows."""
    s = gfo.float_decoy_scene(51, 600, 500, decoy_frac=0.5)
    qr, qq = oracle_mod.quantize_f32(s["ref"], S512), oracle_mod.quantize_f32(s["qry"], S512)
    for kw in (dict(ratio_good=0.6), dict(orientation=1, reject_gt=True), dict(max_dist_sq=20000.0)):
        a = gfo.match_pair_guided_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 8.0, 0.85, **kw)
        b = gdo.match_pair_guided(qr, qq, s["xy_ref"], s["xy_qry"], s["F"], 8.0, 0.85, **kw)
        c = gfo.match_pair_guided_float(qr, qq, s["xy_ref"], s["xy_qry"], s["F"], 8.0, 0.85, band=0.2, float_rows=False, **kw)
        for x in (a, c):
            np.testing.assert_array_equal(x["pairs"], b["pairs"])
            np.testing.assert_array_equal(x["good"], b["good"])
    # with a band, float rows have band rows (decided in fp32; test_hand_built_barred_nearest_row shows one that flips)
    a = gfo.match_pair_guided_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 150.0, 0.85, band=0.2, ratio_good=0.6)
    assert a["band"].sum() > 0


def _embed_adversarial(case, barred):
    """A float decoy scene with the rows of test_float_regime's `case` (reference rows A, B, C; query row x) embedded:
    x at three query rows sharing one keypoint, A and C on its epipolar line, B on it too, or 100 px off it (barred)."""
    s = gfo.float_decoy_scene(61, 1500, 1200, decoy_frac=0.5)
    adv_ref, x = _adversarial(case)
    pos, qpos = [5, 700, 1499], [0, 611, 1199]
    ref, qry, xy_ref, xy_qry = s["ref"].copy(), s["qry"].copy(), s["xy_ref"].copy(), s["xy_qry"].copy()
    ref[pos], qry[qpos] = adv_ref, x
    xy_qry[qpos] = xy_qry[qpos[0]]
    f = np.asarray(s["F"], np.float64).reshape(3, 3)
    a = np.r_[xy_qry[qpos[0]].astype(np.float64), 1.0] @ f
    nrm = a[:2] / np.linalg.norm(a[:2])
    for i, pj in enumerate(pos):
        u = xy_ref[pj].astype(np.float64)
        foot = u - (a[:2] @ u + a[2]) / (a[:2] @ a[:2]) * a[:2]
        xy_ref[pj] = foot + (100.0 * nrm if (barred and i == 1) else 0.0)
    return dict(ref=ref, qry=qry, xy_ref=xy_ref, xy_qry=xy_qry, F=s["F"]), pos, qpos


def test_hand_built_barred_nearest_row(oracle_mod):
    """B is the fp32 nearest row of x and lies within T(q) computed from the gated d1_q, but the gate bars it: the
    restatement decides x on {A, C} and emits (A, x), where an ungated collect pass or brute force would pick B."""
    s, pos, qpos = _embed_adversarial("wrong_ref", barred=True)
    allowed = gdo.gate_f32(s["F"], s["xy_ref"], s["xy_qry"], 3.0)
    assert allowed[qpos][:, [pos[0], pos[2]]].all() and not allowed[qpos][:, pos[1]].any()
    fids, _ = oracle_mod.knn2_f32(s["ref"], s["qry"][qpos])
    assert (fids[:, 0] == pos[1]).all()  # ungated fp32 nearest: B
    exp = gfo.match_pair_guided_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], 3.0, 0.85, band=0.02)
    assert exp["band"][qpos].all()
    d1q = exp["dists"][qpos[0], 1]
    qr, qq = oracle_mod.quantize_f32(s["ref"], S512), oracle_mod.quantize_f32(s["qry"][qpos[:1]], S512)
    T = gfo.exact_threshold(d1q, gfo.residuals(s["qry"][qpos[:1]], S512)[0], gfo.residuals(s["ref"], S512).max())
    assert gdo.dist_u8(qr, qq)[0, pos[1]] <= T
    got = {int(q): int(j) for j, q in exp["pairs"].tolist()}
    assert all(got.get(q) == pos[0] for q in qpos)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def fm(native_lib):
    from metricsfm_b200.matcher import Matcher
    m = Matcher(device=0, max_images=32, arena_rows=1 << 17, keep_float=True)
    yield m
    m.close()


def _load(m, scenes, u8=()):
    """Every scene as images (2s, 2s+1), float rows at scale 512 (u8 rows for the scene indices in `u8`)."""
    m.release_all()
    pairs, F, xy = [], [], {}
    for i, s in enumerate(scenes):
        for k, (rows, kp) in enumerate(((s["ref"], s["xy_ref"]), (s["qry"], s["xy_qry"]))):
            if i in u8:
                m.upload(2 * i + k, rows)
            else:
                m.upload(2 * i + k, np.ascontiguousarray(rows, np.float32), scale=S512)
            xy[2 * i + k] = kp
        pairs.append((2 * i, 2 * i + 1))
        F.append(s["F"])
    return pairs, np.array(F), xy


def _call(m, pairs, F, xy, th, prm, band, mutual=False):
    return m.match_pairs_guided(pairs, F, xy, th_epipolar=th, ratio=prm.get("ratio", 0.85),
                                ratio_good=prm.get("ratio_good", 0.0), max_dist_sq=prm.get("max_dist_sq", 0.0),
                                min_keypoints=prm.get("min_keypoints", 20), orientation=prm.get("orientation", 0),
                                flags=prm.get("flags", 0), rescore_band=band, mutual=mutual)


def _expect(s, th, prm, band, **kw):
    return gfo.match_pair_guided_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], th, prm.get("ratio", 0.85),
                                       band=band, ratio_good=prm.get("ratio_good", 0.0),
                                       max_dist_sq=prm.get("max_dist_sq", 0.0), min_keypoints=prm.get("min_keypoints", 20),
                                       orientation=prm.get("orientation", 0),
                                       reject_gt=bool(prm.get("flags", 0) & REJECT_GT), **kw)


def _assert_equal(res, exps, tag):
    assert res.ok.tolist() == [int(e["ok"]) for e in exps], tag
    for p, e in enumerate(exps):
        got = res.pair(p)
        if not np.array_equal(got, e["pairs"]):
            a, b = {tuple(v) for v in got.tolist()}, {tuple(v) for v in e["pairs"].tolist()}
            raise AssertionError(f"{tag} pair {p}: {len(got)} matches, expected {len(b)}; only on the GPU {sorted(a - b)[:8]}, "
                                 f"only in the restatement {sorted(b - a)[:8]}")
        if res.good is None:  # no ratio_good: the call fills no good flags, and the restatement sets none
            assert not e["good"].any(), tag
        else:
            np.testing.assert_array_equal(res.pair_good(p), e["good"], err_msg=f"{tag} pair {p}: good")


def _collect_and_brute(m, run, exps, tag):
    """The call through the collect path (default event list: events > 0, no brute-force batch) and with an empty
    event list (the brute force decides), both equal to the restatement."""
    n_band = sum(int(e["band"].sum()) for e in exps if e["band"] is not None)
    for cap in (-1, 0):
        m._test_set_band_event_cap(cap)
        try:
            res = run()
        finally:
            m._test_set_band_event_cap(-1)
        _assert_equal(res, exps, f"{tag} cap {cap}")
        events, brute = m._test_last_knn_stats()
        if cap == -1:
            assert brute == 0 and (events > 0) == (n_band > 0), (tag, events, brute, n_band)
        elif n_band > 0:
            assert brute >= 1, (tag, events, brute)
    return n_band


SIZES = [(1, 1), (19, 20), (20, 19), (21, 21), (127, 128), (128, 129), (129, 127), (2000, 1999)]
RULES = [dict(ratio=0.85, ratio_good=0.6), dict(ratio=0.8, ratio_good=0.7, flags=REJECT_GT, orientation=1),
         dict(ratio=0.85, ratio_good=0.6, max_dist_sq=20000.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("band", [0.02, 0.2])
@pytest.mark.parametrize("th", [3.0, 150.0])
def test_sizes_rules_and_bands_vs_restatement(fm, th, band):
    """Ragged and edge sizes (min_keypoints 0), duplicated rows, rows with zero or one allowed reference row at 3 px;
    ratio 0.85 + ratio_good 0.6, REJECT_GT with orientation 1, max_dist_sq; collect path and brute force."""
    scenes = [gfo.float_decoy_scene(100 + i, M, N, decoy_frac=0.5) for i, (M, N) in enumerate(SIZES)]
    pairs, F, xy = _load(fm, scenes)
    n_band = 0
    for prm in RULES:
        prm = {**prm, "min_keypoints": 0}
        exps = [_expect(s, th, prm, band) for s in scenes]
        n_band += _collect_and_brute(fm, lambda: _call(fm, pairs, F, xy, th, prm, band), exps, f"th {th} band {band} {prm}")
        if th == 3.0:
            assert sum(int((e["allowed"].sum(1) <= 1).sum()) for e in exps if e["allowed"] is not None) > 100
    assert n_band > 0


@pytest.mark.gpu
def test_hand_built_rows_the_gate_changes(fm, oracle_mod):
    """The barred fp32-nearest row B (within T(q)); and the two adversarial rows of DESIGN §5 with every row allowed,
    where the result is the ungated float regime's."""
    s, pos, qpos = _embed_adversarial("wrong_ref", barred=True)
    pairs, F, xy = _load(fm, [s])
    exp = _expect(s, 3.0, dict(ratio=0.85), 0.02)
    assert {int(q): int(j) for j, q in exp["pairs"].tolist() if q in qpos} == {q: pos[0] for q in qpos}
    _collect_and_brute(fm, lambda: _call(fm, pairs, F, xy, 3.0, dict(ratio=0.85), 0.02), [exp], "barred B")
    plain = fm.match_pairs(pairs, 0.85, rescore_band=0.02)  # without the gate B wins
    assert {int(q): int(j) for j, q in plain.pair(0).tolist() if q in qpos} == {q: pos[1] for q in qpos}
    for case in ("wrong_ref", "spurious"):
        s, pos, qpos = _embed_adversarial(case, barred=False)
        pairs, F, xy = _load(fm, [s])
        for prm in (dict(ratio=0.85, ratio_good=0.6), dict(ratio=0.85, flags=REJECT_GT)):
            exp = _expect(s, 1e15, prm, 0.03)
            assert exp["band"][qpos].all()
            _collect_and_brute(fm, lambda: _call(fm, pairs, F, xy, 1e15, prm, 0.03), [exp], f"{case} admit-all")
            plain = fm.match_pairs(pairs, 0.85, ratio_good=prm.get("ratio_good", 0.0), flags=prm.get("flags", 0),
                                   rescore_band=0.03)
            np.testing.assert_array_equal(plain.pair(0), exp["pairs"])


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [False, True])
def test_admit_all_gate_equals_match_pairs(fm, mutual):
    scenes = [gfo.float_decoy_scene(400 + i, M, N) for i, (M, N) in enumerate([(900, 800), (129, 300), (40, 41)])]
    pairs, F, xy = _load(fm, scenes)
    for band in (0.02, 0.2):
        plain = fm.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual, rescore_band=band)
        guided = fm.match_pairs_guided(pairs, F, xy, th_epipolar=1e15, ratio=0.85, ratio_good=0.6, mutual=mutual,
                                       rescore_band=band)
        np.testing.assert_array_equal(guided.offsets, plain.offsets)
        np.testing.assert_array_equal(guided.ok, plain.ok)
        np.testing.assert_array_equal(guided.matches, plain.matches)
        np.testing.assert_array_equal(guided.good, plain.good)


@pytest.mark.gpu
def test_pruning_off_gives_identical_lists(fm):
    scenes = [gfo.float_decoy_scene(500 + i, M, N, decoy_frac=0.5) for i, (M, N) in enumerate([(2000, 1500), (700, 900)])]
    pairs, F, xy = _load(fm, scenes)
    for mutual in (False, True):
        for th, band in ((3.0, 0.02), (40.0, 0.2)):
            kw = dict(th_epipolar=th, ratio=0.85, ratio_good=0.6, mutual=mutual, rescore_band=band)
            on = fm.match_pairs_guided(pairs, F, xy, **kw)
            fm._test_disable_pruning(True)
            try:
                off = fm.match_pairs_guided(pairs, F, xy, **kw)
            finally:
                fm._test_disable_pruning(False)
            np.testing.assert_array_equal(on.offsets, off.offsets)
            np.testing.assert_array_equal(on.matches, off.matches)
            np.testing.assert_array_equal(on.good, off.good)


@pytest.mark.gpu
def test_one_call_over_several_batches_equals_per_pair_calls(native_lib):
    """17 000 pairs (more than one 16 384-pair batch) of 64-row float images drawn with repetition, scene Fs: one call
    equals a call per distinct pair."""
    from metricsfm_b200.matcher import Matcher
    n_img, rows = 24, 64
    rng = np.random.default_rng(601)
    col = synth.Collection(rows, seed=601)
    xy = {i: rng.uniform(-1800, 1800, (rows, 2)).astype(np.float32) for i in range(n_img)}
    Fs = [eight_point(*go.two_view_scene(rng, 64, 0)) for _ in range(16)]
    pairs = rng.integers(0, n_img, size=(17000, 2)).astype(np.int32)
    F = np.array([Fs[(int(r) * 7 + int(q)) % len(Fs)] for r, q in pairs])
    kw = dict(th_epipolar=400.0, ratio=0.85, ratio_good=0.6, rescore_band=0.2, min_keypoints=0)
    with Matcher(device=0, max_images=n_img, arena_rows=1 << 15, keep_float=True) as m:
        for i in range(n_img):
            m.upload(i, col.image_unit(i), scale=S512)
        one = m.match_pairs_guided(pairs, F, xy, **kw)
        assert m.timing()["match_launches"] >= 2
        assert len(one.matches) > 0
        done = {}
        for p, (r, q) in enumerate(pairs.tolist()):
            if (r, q) not in done:
                done[(r, q)] = m.match_pairs_guided(pairs[p:p + 1], F[p:p + 1], xy, **kw)
            ref = done[(r, q)]
            np.testing.assert_array_equal(ref.pair(0), one.pair(p))
            np.testing.assert_array_equal(ref.pair_good(0), one.pair_good(p))


@pytest.mark.gpu
def test_u8_pair_follows_the_integer_guided_rule(fm):
    """A u8 pair (and a u8 image paired with a float image) on a keep_float context: the integer guided rule."""
    scenes = [gfo.float_decoy_scene(700 + i, 800, 700, decoy_frac=0.5) for i in range(2)]
    q8 = [dict(s, ref=synth.quantize_512(s["ref"]), qry=synth.quantize_512(s["qry"])) for s in scenes]
    pairs, F, xy = _load(fm, q8[:1] + scenes[1:], u8=(0,))
    pairs.append((0, 3))
    F = np.concatenate([F, F[:1]])
    res = fm.match_pairs_guided(pairs, F, xy, th_epipolar=40.0, ratio=0.85, ratio_good=0.6, rescore_band=0.2)
    exp0 = gdo.match_pair_guided(q8[0]["ref"], q8[0]["qry"], q8[0]["xy_ref"], q8[0]["xy_qry"], F[0], 40.0, 0.85, ratio_good=0.6)
    exp1 = _expect(scenes[1], 40.0, dict(ratio=0.85, ratio_good=0.6), 0.2)
    assert exp1["band"].sum() > 0
    qry3 = gfo.oracle.quantize_f32(scenes[1]["qry"], S512)
    exp2 = gdo.match_pair_guided(q8[0]["ref"], qry3, q8[0]["xy_ref"], scenes[1]["xy_qry"], F[0], 40.0, 0.85, ratio_good=0.6)
    _assert_equal(res, [exp0, exp1, exp2], "u8 / float / mixed")


@pytest.mark.gpu
def test_mutual_matches_are_one_way_matches(fm):
    """Mutual on: the float regime's heuristic filter of the one-way list, under the gate."""
    scenes = [gfo.float_decoy_scene(800 + i, M, N, decoy_frac=0.5) for i, (M, N) in enumerate([(1500, 1200), (600, 900)])]
    pairs, F, xy = _load(fm, scenes)
    for th, band in ((3.0, 0.02), (150.0, 0.2)):
        one = fm.match_pairs_guided(pairs, F, xy, th_epipolar=th, ratio=0.85, ratio_good=0.6, rescore_band=band)
        mut = fm.match_pairs_guided(pairs, F, xy, th_epipolar=th, ratio=0.85, ratio_good=0.6, rescore_band=band, mutual=True)
        for k in range(len(pairs)):
            ow = {tuple(v): g for v, g in zip(one.pair(k).tolist(), one.pair_good(k).tolist())}
            assert mut.pair(k).shape[0] > 0
            for v, g in zip(mut.pair(k).tolist(), mut.pair_good(k).tolist()):
                assert ow.get(tuple(v)) == g, (th, band, k, v)


@pytest.mark.gpu
def test_bad_band_is_refused_before_launch(fm):
    """Negative, NaN and infinite bands: INVALID_ARG naming the entry point, outputs and msfm_last_timing untouched."""
    from metricsfm_b200 import _lib
    s = gfo.float_decoy_scene(900, 200, 150)
    pairs, F, xy = _load(fm, [s])
    fm.match_pairs_guided(pairs, F, xy, th_epipolar=3.0, ratio=0.85, rescore_band=0.02)
    before = fm.timing()
    L, h = fm._L, fm._h
    for band in (-0.02, float("nan"), float("inf"), float("-inf")):
        pa = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        arrs = [np.ascontiguousarray(s["xy_ref"], np.float32), np.ascontiguousarray(s["xy_qry"], np.float32)]
        ptrs = (C.c_void_p * 2)(*[a.ctypes.data for a in arrs])
        npts = np.array([200, 150], np.int32)
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
        Fa = np.ascontiguousarray(F, np.float64).reshape(-1, 9)
        st = L.msfm_match_pairs_guided(h, pa.ctypes.data, len(pa), C.byref(prm), Fa.ctypes.data, 3.0,
                                       C.cast(ptrs, C.c_void_p), npts.ctypes.data, 2, C.byref(res))
        assert st == 1, band
        assert (offs == -7).all() and (okf == -7).all() and (mm == -7).all(), band
        assert fm.timing() == before, band
        assert "guided" in L.msfm_last_error(h).decode(), band
