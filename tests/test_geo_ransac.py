"""The RANSAC search of the GPU geometric verification (geo_verify_kernel, metricsfm_b200/csrc/geo_kernels.cuh) against
its exact restatement in oracle/geo_oracle.py: the counter-based draws, the 7-point and cubic solvers, the strided
subsample and its scale, the winning hypothesis, the F returned in pixel units with F22 = 1, and the decisions of
msfm_geo_verify / msfm_geo_ransac around it.  The CPU tests pin the restatement itself to OpenCV, numpy and the
splitmix64 reference; the GPU tests (-m gpu) pin the kernel to the restatement."""
import ctypes as C

import numpy as np
import pytest

from oracle import geo_oracle as go

TH2 = 9.0


# ------------------------------------------------------------------------------------------------------- CPU: oracle
def _unit_up_to_sign(F):
    F = np.asarray(F, np.float64).reshape(-1, 9)
    F = F / np.linalg.norm(F, axis=1, keepdims=True)
    i = np.abs(F).argmax(1)
    return F * np.sign(F[np.arange(len(F)), i])[:, None]


def _same_models(F, G, tol):
    """Both lists hold the same unit-norm models up to sign, in any order."""
    if len(F) != len(G):
        return False
    F, G = _unit_up_to_sign(F), _unit_up_to_sign(G)
    return all(np.abs(G - f).max(1).min() <= tol for f in F)


def test_seven_point_matches_opencv():
    """The restated seven_point returns the models of cv2.findFundamentalMat(FM_7POINT), same number of roots, on
    random samples and on near-degenerate ones (three points nearly collinear, two points nearly equal)."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(2024)
    samples = [(rng.uniform(-1, 1, (7, 2)), rng.uniform(-1, 1, (7, 2))) for _ in range(500)]
    for _ in range(60):
        p1, p2 = rng.uniform(-1, 1, (7, 2)), rng.uniform(-1, 1, (7, 2))
        t = rng.uniform(-1, 1)
        p1[2] = p1[0] + t * (p1[1] - p1[0]) + rng.normal(0, 1e-4, 2)          # three nearly collinear in image 1
        samples.append((p1, p2))
        p1, p2 = rng.uniform(-1, 1, (7, 2)), rng.uniform(-1, 1, (7, 2))
        p1[6], p2[6] = p1[5] + rng.normal(0, 1e-4, 2), p2[5] + rng.normal(0, 1e-4, 2)   # two nearly equal
        samples.append((p1, p2))
    n_models = 0
    for p1, p2 in samples:
        p1, p2 = p1.astype(np.float32), p2.astype(np.float32)
        F = go.seven_point(p1, p2)
        Fcv, _ = cv2.findFundamentalMat(p1.astype(np.float64), p2.astype(np.float64), cv2.FM_7POINT)
        Fcv = np.zeros((0, 9)) if Fcv is None else Fcv.reshape(-1, 9)
        assert _same_models(F, Fcv, 1e-7), (p1, p2, F, Fcv)
        n_models += len(F)
    assert n_models > len(samples)   # the three-root branch is taken


def test_solve_cubic_matches_roots():
    """solve_cubic's real roots equal numpy's, for full cubics with one or three real roots and for the degenerate
    branches c3 = 0 (quadratic, with and without real roots) and c3 = c2 = 0 (linear)."""
    rng = np.random.default_rng(7)

    def check(c):
        got = sorted(go.solve_cubic(*c))
        r = np.roots(np.trim_zeros(np.array(c, np.float64), "f"))
        exp = sorted(r[np.abs(r.imag) <= 1e-9 * max(1.0, np.abs(r).max())].real)
        assert len(got) == len(exp), (c, got, exp)
        np.testing.assert_allclose(got, exp, rtol=1e-8, atol=1e-10)
        for x in got:   # each root is a root
            assert abs(((c[0] * x + c[1]) * x + c[2]) * x + c[3]) <= 1e-9 * (np.abs(c) * np.maximum(1, abs(x)) ** 3).sum()

    for _ in range(300):
        r = np.sort(rng.uniform(-5, 5, 3))
        if np.diff(r).min() < 1e-2:
            continue
        k = rng.uniform(0.1, 10) * rng.choice([-1, 1])
        check(tuple(k * np.poly(r)))                                              # three real roots
        re, im, x0 = rng.uniform(-3, 3), rng.uniform(0.1, 3), rng.uniform(-3, 3)
        check(tuple(k * np.poly([x0, re + 1j * im, re - 1j * im]).real))         # one real root
        q = np.poly(rng.uniform(-5, 5, 2))
        check((0.0,) + tuple(k * q))                                              # c3 = 0, two real roots
        check((0.0, k, 0.0, abs(k) * rng.uniform(0.1, 4) * np.sign(k)))           # c3 = 0, no real root
        check((0.0, 0.0, k, rng.uniform(-5, 5)))                                  # c3 = c2 = 0
    assert go.solve_cubic(0.0, 0.0, 0.0, 1.0) == []


def test_geo_mix_is_splitmix64():
    assert int(go.geo_mix(1234567)[0]) == 6457827717110365317
    st, out = 1234567, []                                  # the generator: state += golden ratio, output = mix(state)
    for _ in range(3):
        out.append(int(go.geo_mix(st)[0]))
        st = (st + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    assert out[0] == 6457827717110365317 and len(set(out)) == 3
    idx = go.draw_samples(5, 3, 256, 9)
    assert idx.min() >= 0 and idx.max() < 9
    assert all(len(set(r)) == 7 for r in idx.tolist())
    assert not np.array_equal(idx, go.draw_samples(5, 4, 256, 9))        # the pair index is part of the counter
    np.testing.assert_array_equal(idx[:100], go.draw_samples(5, 3, 100, 9))


def _rigid_scene(rng, n, f=3000.0):
    """Noise-free two-view scene and its true fundamental matrix (pixel units)."""
    X = np.concatenate([rng.uniform(-40, 40, (n, 2)), rng.uniform(60, 140, (n, 1))], 1)
    ang = np.deg2rad(6.0)
    R = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    t = np.array([11.0, 1.5, -0.5])
    p1 = f * X[:, :2] / X[:, 2:3]
    Xc = X @ R.T + t
    p2 = f * Xc[:, :2] / Xc[:, 2:3]
    Kinv = np.diag([1 / f, 1 / f, 1.0])
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    return p1.astype(np.float32), p2.astype(np.float32), Kinv.T @ tx @ R @ Kinv


def test_search_finds_true_F_on_noise_free_scene():
    rng = np.random.default_rng(11)
    p1, p2, Ftrue = _rigid_scene(rng, 300)
    srch = go.ransac_search(p1, p2, seed=4, pair_index=2)
    w = srch["win"]
    assert w >= 0 and srch["count"][w] == srch["n_pts"] == 300
    F = srch["F"][w]
    assert abs(F[8] - 1.0) <= 1e-12
    np.testing.assert_allclose(_unit_up_to_sign(F)[0], _unit_up_to_sign(Ftrue)[0], atol=1e-5)
    ok, inl, keep, _, _ = go.geo_pair(p1, p2, np.ones(300, np.uint8), seed=4, pair_index=2)
    assert ok and inl == 300 and keep.all()


# ------------------------------------------------------------------------------------------------ GPU: the kernel
@pytest.fixture(scope="module")
def matcher(native_lib):
    from metricsfm_b200.matcher import Matcher
    m = Matcher(device=0, max_images=8, arena_rows=1 << 12)
    yield m
    m.close()


def _batch(scenes, rng):
    """scenes: [(p1, p2, good)] in match order -> (pairs, MatchResult, image_xy); keypoint ids are permuted so that
    they are not in match order."""
    from metricsfm_b200.matcher import MatchResult
    image_xy, pairs, offsets, matches = {}, [], [0], []
    for s, (p1, p2, _) in enumerate(scenes):
        n = len(p1)
        perm1, perm2 = rng.permutation(n), rng.permutation(n)
        xy1, xy2 = np.empty_like(p1), np.empty_like(p2)
        xy1[perm1], xy2[perm2] = p1, p2
        image_xy[2 * s], image_xy[2 * s + 1] = xy1, xy2
        pairs.append((2 * s, 2 * s + 1))
        matches.append(np.stack([perm1, perm2], 1).astype(np.int32).reshape(-1, 2))
        offsets.append(offsets[-1] + n)
    good = np.concatenate([np.asarray(g, np.uint8) for _, _, g in scenes]) if scenes else np.zeros((0,), np.uint8)
    res = MatchResult(offsets=np.array(offsets, np.int64), ok=np.ones((len(scenes),), np.int32),
                      matches=np.concatenate(matches) if matches else np.zeros((0, 2), np.int32), good=good)
    return pairs, res, image_xy


def _verify(matcher, scenes, seed, rng=None, **kw):
    pairs, res, image_xy = _batch(scenes, rng if rng is not None else np.random.default_rng(0))
    ok, inl, keep, F = matcher.geo_verify(pairs, res, image_xy, seed=seed, **kw)
    return ok, inl, [keep[res.offsets[s]:res.offsets[s + 1]] for s in range(len(scenes))], F


def _pixel_f22(srch, j):
    """F22 / ||F|| of model j in pixel units before the normalisation: the kernel divides by F22 when above 1e-12."""
    s = float(srch["scale"])
    Fp = srch["Ff"][j].astype(np.float64) * np.array([s * s, s * s, s, s * s, s * s, s, s, s, 1.0])
    return Fp[8] / np.linalg.norm(Fp)


def _check_pair(scene, ok, inl, keep, F, *, seed, pair_index, stage_b=True, th=3.0, min_points=30, min_inliers=30,
                iters=1024):
    """One pair's GPU outputs against the restatement.  Returns True when the restated winner is certain."""
    p1, p2, good = scene
    kw = dict(seed=seed, pair_index=pair_index, th=th, min_points=min_points, min_inliers=min_inliers, iters=iters,
              stage_b=stage_b)
    eok, einl, ekeep, _, srch = go.geo_pair(p1, p2, good, **kw)
    F = np.asarray(F, np.float64).reshape(9)
    if srch is None or srch["win"] < 0:            # gated out before the search, or no model at all
        assert (ok, inl) == (0, 0), (ok, inl, srch is None)
        assert not keep.any() and not F.any()
        return True
    adm = np.flatnonzero(srch["admissible"])
    w = srch["win"]
    if ok:
        # the F as returned (F22 = 1 scaling included) is the pixel-unit F of an admissible model, or the winner's
        d = np.array([np.abs(F - srch["F"][j]).max() / np.abs(srch["F"][j]).max() for j in adm])
        assert d.min() <= 1e-5, (pair_index, d.min(), F, srch["F"][w])
        j = adm[d.argmin()]
        if srch["certain"]:
            assert j == w or np.abs(F - srch["F"][w]).max() <= 1e-5 * np.abs(srch["F"][w]).max(), (pair_index, srch["id"][j], srch["id"][w])
        if abs(_pixel_f22(srch, j)) > 1e-12:
            assert abs(F[8] - 1.0) <= 1e-12, F
        # decisions around the returned F are the restated flow's
        rok, rinl, rkeep, _, _ = go.geo_pair(p1, p2, good, F=F, **kw)
        assert (bool(ok), int(inl)) == (rok, rinl)
        np.testing.assert_array_equal(keep.astype(bool), rkeep)
    else:
        assert not keep.any() and not F.any()
        # F is not returned: the inlier count is that of the winner (certain) or of an admissible model
        cand = [w] if srch["certain"] else adm
        g = np.asarray(good).astype(bool)
        counts = [int((go.ransac_error(srch["F"][j], p1[g], p2[g]) <= th * th).sum()) for j in cand]
        assert inl in counts and inl < min_inliers, (inl, counts)
    return srch["certain"]


def _mixed_scenes(rng, n):
    sizes = [(400, 130), (90, 60), (0, 300), (3000, 900), (35, 0), (150, 150), (60, 20), (1200, 400), (250, 40),
             (20, 40), (700, 700), (45, 5), (500, 0), (2200, 100), (80, 120)]
    out = []
    for i in range(n):
        n_true, n_out = sizes[i % len(sizes)]
        p1, p2 = go.two_view_scene(rng, n_true, n_out)
        frac = [1.0, 0.8, 0.6][i % 3]
        good = (rng.random(len(p1)) < frac).astype(np.uint8)
        out.append((p1, p2, good))
    return out


@pytest.mark.gpu
def test_hypothesis_choice_matches_restatement(matcher):
    """~30 scenes of mixed sizes and outlier rates, two seeds: the returned F is the restated winner's (or, where a
    borderline point makes the count uncertain, an admissible model's), and the winner is certain for >= 90 % of the
    pairs that reach the search."""
    rng = np.random.default_rng(41)
    scenes = _mixed_scenes(rng, 30)
    n_certain, n_searched = 0, 0
    for seed, base in ((7, 0), (0xDEADBEEF12345, 1000)):
        ok, inl, keep, F = _verify(matcher, scenes, seed, rng, pair_index_base=base)
        assert ok.sum() >= 10 and (ok == 0).sum() >= 4
        for s, sc in enumerate(scenes):
            if sc[2].sum() < 30:
                _check_pair(sc, ok[s], inl[s], keep[s], F[s], seed=seed, pair_index=base + s)
                continue
            n_searched += 1
            n_certain += _check_pair(sc, ok[s], inl[s], keep[s], F[s], seed=seed, pair_index=base + s)
    assert n_certain >= 0.9 * n_searched, (n_certain, n_searched)


@pytest.mark.gpu
def test_subsample_stride_and_scale(matcher):
    """Above 2048 good matches the search scores every stride-th good match (stride = ceil(n_good / 2048)) and takes
    the scale from those points only: in the 4097 case the largest coordinate sits on a good match the stride skips."""
    rng = np.random.default_rng(43)
    scenes = []
    for n_good in (2047, 2048, 2049, 4096, 4097, 6145):
        p1, p2 = go.two_view_scene(rng, int(n_good * 0.8), n_good - int(n_good * 0.8) + 200)
        good = np.zeros((len(p1),), np.uint8)
        good[rng.choice(len(p1), n_good, replace=False)] = 1
        scenes.append((p1, p2, good))
    p1, p2, good = scenes[4]
    gi = np.flatnonzero(good)
    p1[gi[5]] = (-4000.0, 3900.0)                      # good match 5: skipped with stride 2
    _, s_sampled = go.subsample(p1[good == 1], p2[good == 1])
    assert s_sampled != np.float32(1) / np.abs(np.concatenate([p1[gi], p2[gi]])).max()
    n_certain = 0
    for seed in (3, 4):
        ok, inl, keep, F = _verify(matcher, scenes, seed, rng)
        assert ok.all()
        for s, sc in enumerate(scenes):
            if not _check_pair(sc, ok[s], inl[s], keep[s], F[s], seed=seed, pair_index=s):
                continue
            n_certain += 1
            # The scale changes the float32 model of the same hypothesis at the 1e-7 level, and the pixel-unit F
            # with it, while the same float32 model gives the same F up to double rounding: a scale taken from
            # other points than the sampled ones shows here, beneath the 1e-5 bar of _check_pair.
            p1, p2, good = sc
            g = good.astype(bool)
            srch = go.ransac_search(p1[g], p2[g], seed=seed, pair_index=s)
            Fw = srch["F"][srch["win"]]
            assert np.abs(F[s].reshape(9) - Fw).max() <= 1e-12 * np.abs(Fw).max(), (seed, s, F[s], Fw)
    assert n_certain >= 10


@pytest.mark.gpu
def test_hypothesis_count_edges(matcher):
    """iters below, at and above the 256 threads of a CTA (threads that draw no hypothesis), and iters = 0 == 1024."""
    rng = np.random.default_rng(47)
    scenes = [(*go.two_view_scene(rng, n_true, n_out), None) for n_true, n_out in ((300, 60), (60, 40), (0, 120), (1500, 500))]
    scenes = [(p1, p2, np.ones((len(p1),), np.uint8)) for p1, p2, _ in scenes]
    n_certain, n = 0, 0
    for iters in (1, 7, 255, 256, 257):
        ok, inl, keep, F = _verify(matcher, scenes, 21, rng, iters=iters, min_inliers=0)
        for s, sc in enumerate(scenes):
            n_certain += _check_pair(sc, ok[s], inl[s], keep[s], F[s], seed=21, pair_index=s, iters=iters, min_inliers=0)
            n += 1
    assert n_certain >= 0.9 * n
    r0 = _verify(matcher, scenes, 21, np.random.default_rng(1), iters=0)
    r1 = _verify(matcher, scenes, 21, np.random.default_rng(1), iters=1024)
    for a, b in zip(r0, r1):
        np.testing.assert_array_equal(np.concatenate(a) if isinstance(a, list) else a, np.concatenate(b) if isinstance(b, list) else b)
    for s, sc in enumerate(scenes):
        _check_pair(sc, r0[0][s], r0[1][s], r0[2][s], r0[3][s], seed=21, pair_index=s, iters=0)


@pytest.mark.gpu
def test_point_count_and_inlier_gates(matcher):
    rng = np.random.default_rng(53)
    scenes = []
    for n_good in (6, 7, 29, 30):
        p1, p2 = go.two_view_scene(rng, n_good + 10, 5)
        good = np.zeros((len(p1),), np.uint8)
        good[rng.choice(len(p1), n_good, replace=False)] = 1
        scenes.append((p1, p2, good))
    for min_points in (0, 30):
        ok, inl, keep, F = _verify(matcher, scenes, 9, rng, min_points=min_points, min_inliers=0)
        assert ok.tolist() == ([0, 1, 1, 1] if min_points == 0 else [0, 0, 0, 1])
        for s, sc in enumerate(scenes):
            _check_pair(sc, ok[s], inl[s], keep[s], F[s], seed=9, pair_index=s, min_points=min_points, min_inliers=0)
    # min_inliers at its boundary: the calls are deterministic, so inl accepts and inl + 1 rejects
    one = [_mixed_scenes(np.random.default_rng(59), 1)[0]]
    ok, inl, keep, F = _verify(matcher, one, 5, min_inliers=0)
    assert ok[0] and inl[0] > 30
    ok2, inl2, keep2, F2 = _verify(matcher, one, 5, min_inliers=int(inl[0]))
    assert ok2[0] == 1 and inl2[0] == inl[0]
    np.testing.assert_array_equal(keep2[0], keep[0]), np.testing.assert_array_equal(F2, F)
    ok3, inl3, keep3, F3 = _verify(matcher, one, 5, min_inliers=int(inl[0]) + 1)
    assert ok3[0] == 0 and inl3[0] == inl[0] and not keep3[0].any() and not F3.any()


def _sideways_scene(rng, n, noise, f=3000.0):
    """Pure sideways camera translation (R = I, t along x), as along an aerial strip: the true F has F22 = 0."""
    X = np.concatenate([rng.uniform(-40, 40, (n, 2)), rng.uniform(60, 140, (n, 1))], 1)
    p1 = f * X[:, :2] / X[:, 2:3]
    Xc = X + np.array([10.0, 0.0, 0.0])
    p2 = f * Xc[:, :2] / Xc[:, 2:3]
    return ((p1 + rng.normal(0, noise, p1.shape)).astype(np.float32), (p2 + rng.normal(0, noise, p2.shape)).astype(np.float32))


@pytest.mark.gpu
def test_degenerate_inputs(matcher):
    n = 60
    same = (np.tile(np.float32([[12.5, -40.0]]), (n, 1)), np.tile(np.float32([[300.0, 7.0]]), (n, 1)))
    zero = (np.zeros((n, 2), np.float32), np.zeros((n, 2), np.float32))
    t = np.arange(n, dtype=np.float32) * 16 - 480            # collinear, exactly representable after the 1/1024 scale
    line = (np.stack([t, 0.5 * t + 64], 1).astype(np.float32),
            np.stack([-0.25 * t + 32, t], 1).astype(np.float32))
    line[0][0] = (1024.0, 512.0 + 64.0)                      # largest |coordinate| 1024, still on the line
    rng = np.random.default_rng(61)
    exact = _sideways_scene(rng, 300, 0.0)                    # F22 / ||F|| ~ 1e-14: unit-norm branch
    rng = np.random.default_rng(6)
    fine = _sideways_scene(rng, 300, 1e-4)                    # F22 / ||F|| ~ 3e-4: F22 branch
    scenes = [(a, b, np.ones((len(a),), np.uint8)) for a, b in (same, zero, line, exact, fine)]
    # preconditions on the restatement: no model for the first three; the sideways winners on either side of 1e-12
    rel = []
    for p1, p2, g in scenes:
        srch = go.ransac_search(p1, p2, seed=13, pair_index=len(rel))
        rel.append(None if srch["win"] < 0 else abs(_pixel_f22(srch, srch["win"])))
    assert rel[:3] == [None] * 3 and rel[3] < 1e-13 and 1e-5 < rel[4] < 1e-3, rel
    ok, inl, keep, F = _verify(matcher, scenes, 13, rng, min_inliers=30)
    assert ok.tolist() == [0, 0, 0, 1, 1] and inl.tolist()[:3] == [0, 0, 0]
    for s, sc in enumerate(scenes):
        assert _check_pair(sc, ok[s], inl[s], keep[s], F[s], seed=13, pair_index=s)
    assert abs(np.linalg.norm(F[3]) - 1.0) <= 1e-12 and abs(F[4][2, 2] - 1.0) <= 1e-12


@pytest.mark.gpu
def test_many_pairs_one_call_equals_slices(matcher):
    """More pairs than twice the grid (each CTA carries its shared state over several pairs): one call equals three
    calls over consecutive slices, each smaller than the grid, with pair_index_base set; sampled pairs are restated."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2500
    assert n > 2 * 8 * sms
    rng = np.random.default_rng(67)
    kinds = [(40, 10, 1.0), (25, 5, 1.0), (0, 40, 1.0), (120, 30, 0.7), (60, 0, 0.2), (8, 0, 1.0)]
    scenes = []
    for i in range(n):
        n_true, n_out, frac = kinds[i % len(kinds)] if i % 97 else (2100, 300, 1.0)
        p1, p2 = go.two_view_scene(rng, n_true, n_out)
        scenes.append((p1, p2, (rng.random(len(p1)) < frac).astype(np.uint8)))
    ok, inl, keep, F = _verify(matcher, scenes, 77, np.random.default_rng(1), pair_index_base=5)
    assert 0 < ok.sum() < n
    cuts = [0, 830, 1660, n]
    assert max(np.diff(cuts)) < 8 * sms
    for a, b in zip(cuts[:-1], cuts[1:]):
        ok2, inl2, keep2, F2 = _verify(matcher, scenes[a:b], 77, np.random.default_rng(1), pair_index_base=5 + a)
        np.testing.assert_array_equal(ok2, ok[a:b]), np.testing.assert_array_equal(inl2, inl[a:b])
        np.testing.assert_array_equal(F2, F[a:b])
        for k in range(b - a):
            np.testing.assert_array_equal(keep2[k], keep[a + k])
    sample = [0, 97, 1163, 1164, 1190, 1999, 2396, 2397, 2400, 2499]
    assert sum(_check_pair(scenes[s], ok[s], inl[s], keep[s], F[s], seed=77, pair_index=5 + s) for s in sample) >= 9


@pytest.mark.gpu
def test_geo_ransac_consensus_mask(matcher):
    """msfm_geo_ransac: the mask is the consensus set of the participating matches around the returned F; ok, inliers
    and F equal msfm_geo_verify's on the same input and seed."""
    rng = np.random.default_rng(71)
    scenes = []
    for p1, p2, g in _mixed_scenes(rng, 12):
        scenes.append((p1, p2, (rng.random(len(p1)) >= 1 / 3).astype(np.uint8)))
    pairs, res, image_xy = _batch(scenes, rng)
    ok, inl, keep, F = matcher.geo_verify(pairs, res, image_xy, seed=17, ransac_only=True)
    okv, inlv, _, Fv = matcher.geo_verify(pairs, res, image_xy, seed=17)
    np.testing.assert_array_equal(ok, okv), np.testing.assert_array_equal(inl, inlv), np.testing.assert_array_equal(F, Fv)
    assert ok.sum() >= 4
    n_certain, n_searched = 0, 0
    for s, (p1, p2, use) in enumerate(scenes):
        k = keep[res.offsets[s]:res.offsets[s + 1]].astype(bool)
        if ok[s]:
            np.testing.assert_array_equal(k, use.astype(bool) & (go.ransac_error(F[s], p1, p2) <= TH2))
            assert k.sum() == inl[s]
        else:
            assert not k.any()
        if use.sum() >= 30:
            n_searched += 1
        n_certain += _check_pair(scenes[s], ok[s], inl[s], k, F[s], seed=17, pair_index=s, stage_b=False) and use.sum() >= 30
    assert n_certain >= 0.9 * n_searched


@pytest.mark.gpu
def test_error_paths_before_launch(matcher):
    """Malformed input is refused with INVALID_ARG before anything runs (the outputs stay untouched); an empty pair list
    is fine, and pairs without matches are rejected with F zero."""
    from metricsfm_b200 import _lib
    L, h = matcher._L, matcher._h
    xy = [np.float32(np.random.default_rng(3).uniform(-100, 100, (40, 2))) for _ in range(3)]

    def call(pairs, offsets, matches, n_images, npts=None, ptrs=None, n_pairs=None, fn=L.msfm_geo_verify):
        pa = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        npr = len(pa) if n_pairs is None else n_pairs
        offs = np.ascontiguousarray(offsets, np.int64)
        m = np.ascontiguousarray(matches, np.int32).reshape(-1, 2)
        g = np.ones((max(len(m), 1),), np.uint8)
        arr = (C.c_void_p * 3)(*[a.ctypes.data for a in xy]) if ptrs is None else ptrs
        npts = np.array([40, 40, 40], np.int32) if npts is None else np.asarray(npts, np.int32)
        gp = _lib.GeoParams(3.0, 30, 30, 1024, 1, 0)
        ok = np.full((max(len(pa), 1),), -7, np.int32)
        inl = np.full((max(len(pa), 1),), -7, np.int32)
        keep = np.full((max(len(m), 1),), 9, np.uint8)
        F = np.full((max(len(pa), 1), 9), np.nan)
        st = fn(h, pa.ctypes.data, npr, offs.ctypes.data, m.ctypes.data if len(m) else None, g.ctypes.data if len(m) else None,
                C.cast(arr, C.c_void_p), npts.ctypes.data, n_images, C.byref(gp), ok.ctypes.data, inl.ctypes.data,
                keep.ctypes.data, F.ctypes.data)
        return st, ok, inl, keep, F

    m_ok = np.stack([np.arange(40), np.arange(40)], 1)
    for fn in (L.msfm_geo_verify, L.msfm_geo_ransac):
        bad = [call([(0, 1)], [0, 40], np.where(np.arange(80).reshape(40, 2) == 79, 40, m_ok), 3, fn=fn),   # match past keypoints
               call([(0, 1), (1, 3)], [0, 40, 40], m_ok, 3, fn=fn),                                          # image >= n_images
               call([(0, 2)], [0, 40], m_ok, 3, ptrs=(C.c_void_p * 3)(xy[0].ctypes.data, xy[1].ctypes.data, None), fn=fn),
               call([(0, 1)], [0, 40], m_ok, 3, n_pairs=-1, fn=fn)]
        for st, ok, inl, keep, F in bad:
            assert st == 1
            assert (ok == -7).all() and (inl == -7).all() and (keep == 9).all() and np.isnan(F).all()
        st, ok, *_ = call(np.zeros((0, 2)), [0], np.zeros((0, 2)), 0, n_pairs=0, fn=fn)
        assert st == 0 and ok[0] == -7
        st, ok, inl, keep, F = call([(0, 1), (1, 2), (2, 0)], [0, 0, 0, 0], np.zeros((0, 2)), 3, fn=fn)
        assert st == 0 and ok.tolist() == [0, 0, 0] and inl.tolist() == [0, 0, 0] and (F == 0).all()
    # an unused image may have null keypoints
    st, ok, inl, _, _ = call([(0, 1)], [0, 40], m_ok, 3, ptrs=(C.c_void_p * 3)(xy[0].ctypes.data, xy[1].ctypes.data, None))
    assert st == 0 and ok[0] in (0, 1) and inl[0] >= 0
