"""msfm_geo_homography (batched RANSAC homography on the GPU): the numpy restatement in oracle/homography_oracle.py is
pinned to OpenCV on the CPU (the 4-point solver to cv2.getPerspectiveTransform, the search statistically to
cv2.findHomography(RANSAC)); on the GPU the returned H, pair_ok, pair_inliers and the consensus mask are checked against
that restatement, a list verified in slices against one call, and every error status."""
import ctypes as C

import numpy as np
import pytest

from oracle import homography_oracle as ho


def planar_matches(rng, n_true, n_out, noise=0.5):
    """Centred pixel coordinates of n_true correspondences under a random near-similarity homography (plus keypoint
    noise) and n_out random outliers; returns (p1, p2, H)."""
    a = np.deg2rad(rng.uniform(-20, 20))
    s = rng.uniform(0.8, 1.25)
    H = np.array([[s * np.cos(a), -s * np.sin(a), rng.uniform(-300, 300)],
                  [s * np.sin(a), s * np.cos(a), rng.uniform(-300, 300)],
                  [rng.uniform(-4e-5, 4e-5), rng.uniform(-4e-5, 4e-5), 1.0]])
    p1 = rng.uniform(-1500, 1500, (n_true, 2))
    t = np.c_[p1, np.ones(n_true)] @ H.T
    p2 = t[:, :2] / t[:, 2:3] + rng.normal(0, noise, (n_true, 2))
    o1, o2 = rng.uniform(-1800, 1800, (n_out, 2)), rng.uniform(-1800, 1800, (n_out, 2))
    return np.concatenate([p1, o1]).astype(np.float32), np.concatenate([p2, o2]).astype(np.float32), H


# ------------------------------------------------------------------------------------------------ CPU: the restatement
def test_four_point_matches_opencv():
    """The DLT through four correspondences is cv2.getPerspectiveTransform's H (which is only accurate to ~1e-6 on
    unit-scale points: ours maps the four points to their partners to 1e-12)."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(1)
    n = 0
    for _ in range(200):
        p1, p2, _ = planar_matches(rng, 4, 0, noise=3.0)
        p1, p2 = p1 / 1500, p2 / 1500
        if not ho.subset_ok(p1[None, :, 0], p1[None, :, 1], p2[None, :, 0], p2[None, :, 1])[0]:
            continue
        h = ho.four_point(p1, p2)
        ref = cv2.getPerspectiveTransform(p1.astype(np.float32), p2.astype(np.float32)).reshape(9)
        t = np.c_[p1.astype(np.float64), np.ones(4)] @ h.reshape(3, 3).T
        assert np.abs(t[:, :2] / t[:, 2:] - p2).max() <= 1e-12
        ref = ref / np.linalg.norm(ref) * np.sign(ref @ h)
        assert np.abs(h - ref).max() <= 1e-4, (h, ref)
        n += 1
    assert n > 150


def test_subset_check_rejects_orientation_flips():
    """The orientation check is stricter than cv::findHomography's checkSubset: it rejects a mirrored sample (all four
    triples flip), which OpenCV accepts, as well as a sample in which only some triples flip."""
    sq = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], np.float64)
    assert ho.subset_ok(*(v[None] for v in (sq[:, 0], sq[:, 1], sq[:, 0], sq[:, 1])))[0]
    mirrored = sq * [-1, 1]
    assert not ho.subset_ok(*(v[None] for v in (sq[:, 0], sq[:, 1], mirrored[:, 0], mirrored[:, 1])))[0]
    crossed = sq[[0, 1, 3, 2]]   # a bow-tie: some triples keep their orientation, others flip
    assert not ho.subset_ok(*(v[None] for v in (sq[:, 0], sq[:, 1], crossed[:, 0], crossed[:, 1])))[0]


def test_search_agrees_with_opencv_statistically():
    """On planar scenes with 0-60 % outliers: the accept decisions agree with cv2.findHomography(RANSAC, th), OpenCV's
    inliers are (to a few %) contained in ours, and >= 97 % of the true correspondences survive."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(2)
    agree, contained, total_cv, kept, n_true_all = 0, 0, 0, 0, 0
    cases = [(300, 0), (300, 200), (150, 220), (800, 400), (40, 10), (25, 40), (500, 60), (200, 300)] * 3
    for i, (n_true, n_out) in enumerate(cases):
        p1, p2, _ = planar_matches(rng, n_true, n_out)
        ok, inl, mask, H, _ = ho.geo_pair_h(p1, p2, np.ones(len(p1), bool), seed=i, pair_index=i, th=3.0)
        Hcv, mcv = cv2.findHomography(p1, p2, cv2.RANSAC, 3.0, maxIters=2000)
        mcv = mcv.reshape(-1).astype(bool) if mcv is not None else np.zeros(len(p1), bool)
        ok_cv = Hcv is not None and mcv.sum() >= 30 and len(p1) >= 30
        agree += ok == ok_cv
        if ok and ok_cv:
            contained += int((mcv & mask).sum())
            total_cv += int(mcv.sum())
            kept += int(mask[:n_true].sum())
            n_true_all += n_true
    assert agree == len(cases)
    assert contained >= 0.97 * total_cv, (contained, total_cv)
    assert kept >= 0.97 * n_true_all, (kept, n_true_all)


def test_gate_agrees_with_float64_transfer_error():
    """gate_h32 is the float64 transfer-error test err <= th^2 on every element whose error is not within 1e-4 of th^2."""
    s = ho.planar_decoy_scene(5, 600, 400)
    for th in (1.0, 4.0, 50.0):
        allowed = ho.gate_h32(s["H"], s["xy_ref"], s["xy_qry"], th)
        err = ho.transfer_err64(s["H"].astype(np.float32).astype(np.float64), s["xy_ref"], s["xy_qry"])
        clear = np.abs(err - th * th) > 1e-4 * th * th
        assert clear.sum() > 0.99 * clear.size
        np.testing.assert_array_equal(allowed[clear], (err <= th * th)[clear])
        assert 0 < allowed.sum() < allowed.size


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def matcher(native_lib):
    from metricsfm_b200.matcher import Matcher
    m = Matcher(device=0, max_images=8, arena_rows=1 << 12)
    yield m
    m.close()


def _batch(scenes, rng):
    """scenes: [(p1, p2, use)] in match order -> (pairs, MatchResult, image_xy) with permuted keypoint ids."""
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
    use = np.concatenate([np.asarray(g, np.uint8) for _, _, g in scenes])
    res = MatchResult(offsets=np.array(offsets, np.int64), ok=np.ones((len(scenes),), np.int32),
                      matches=np.concatenate(matches), good=use)
    return pairs, res, image_xy


def _mixed(rng, n):
    sizes = [(400, 130), (90, 60), (0, 300), (3000, 900), (35, 0), (150, 150), (60, 20), (1200, 400), (250, 40),
             (20, 40), (700, 700), (45, 5), (500, 0), (2200, 100), (80, 120)]
    out = []
    for i in range(n):
        n_true, n_out = sizes[i % len(sizes)]
        p1, p2, _ = planar_matches(rng, n_true, n_out)
        use = (rng.random(len(p1)) < [1.0, 0.8, 0.6][i % 3]).astype(np.uint8)
        out.append((p1, p2, use))
    return out


def _check_pair(scene, ok, inl, mask, H, *, seed, pair_index, th=3.0):
    """One pair's outputs against the restatement; True when the restated winner is certain."""
    p1, p2, use = scene
    kw = dict(seed=seed, pair_index=pair_index, th=th)
    eok, einl, emask, _, srch = ho.geo_pair_h(p1, p2, use, **kw)
    H = np.asarray(H, np.float64).reshape(9)
    if srch is None or srch["win"] < 0:
        assert (ok, inl) == (0, 0) and not mask.any() and not H.any()
        return True
    w = srch["win"]
    if srch["certain"]:
        assert (bool(ok), int(inl)) == (eok, einl), (pair_index, ok, inl, eok, einl)
        np.testing.assert_array_equal(mask.astype(bool), emask)
    if ok:
        adm = np.flatnonzero(srch["admissible"])
        d = np.array([np.abs(H - srch["H"][j]).max() / np.abs(srch["H"][j]).max() for j in adm])
        assert d.min() <= 1e-5, (pair_index, d.min())
        if srch["certain"]:
            assert np.abs(H - srch["H"][w]).max() <= 1e-5 * np.abs(srch["H"][w]).max(), pair_index
        assert abs(H[8] - 1.0) <= 1e-12
        rok, rinl, rmask, _, _ = ho.geo_pair_h(p1, p2, use, H=H, **kw)
        assert (bool(ok), int(inl)) == (rok, rinl)
        np.testing.assert_array_equal(mask.astype(bool), rmask)
    else:
        assert not mask.any() and not H.any() and inl < 30
    return srch["certain"]


@pytest.mark.gpu
def test_search_matches_restatement(matcher):
    """~30 planar scenes of mixed sizes and outlier rates, two seeds: H is the restated winner's to 1e-5 wherever no
    point lies within rounding reach of th^2 for the winner or a model that could tie it (>= 90 % of the searched pairs
    that hold a plane; on pure-outlier pairs dozens of models tie at 4 inliers), an admissible model's elsewhere;
    pair_ok, pair_inliers and the mask are those of the restated flow around the returned H."""
    rng = np.random.default_rng(61)
    scenes = _mixed(rng, 30)
    n_certain, n_searched = 0, 0
    for seed, base in ((7, 0), (0xDEADBEEF12345, 1000)):
        pairs, res, xy = _batch(scenes, rng)
        ok, inl, mask, H = matcher.geo_homography(pairs, res, xy, th=3.0, seed=seed, pair_index_base=base)
        assert ok.sum() >= 10 and (ok == 0).sum() >= 4
        for s, sc in enumerate(scenes):
            m = mask[res.offsets[s]:res.offsets[s + 1]]
            certain = _check_pair(sc, ok[s], inl[s], m, H[s], seed=seed, pair_index=base + s)
            if sc[2].sum() >= 30 and s % 15 != 2:  # size (0, 300): no plane
                n_searched += 1
                n_certain += certain
    assert n_certain >= 0.9 * n_searched, (n_certain, n_searched)


@pytest.mark.gpu
def test_slices_equal_one_call(matcher):
    rng = np.random.default_rng(62)
    scenes = _mixed(rng, 12)
    pairs, res, xy = _batch(scenes, rng)
    one = matcher.geo_homography(pairs, res, xy, th=3.0, seed=9)
    from metricsfm_b200.matcher import MatchResult
    for lo, hi in ((0, 5), (5, 12)):
        o = res.offsets
        part = MatchResult(offsets=o[lo:hi + 1] - o[lo], ok=res.ok[lo:hi], matches=res.matches[o[lo]:o[hi]],
                           good=res.good[o[lo]:o[hi]])
        sl = matcher.geo_homography(pairs[lo:hi], part, xy, th=3.0, seed=9, pair_index_base=lo)
        np.testing.assert_array_equal(sl[0], one[0][lo:hi])
        np.testing.assert_array_equal(sl[1], one[1][lo:hi])
        np.testing.assert_array_equal(sl[2], one[2][o[lo]:o[hi]])
        np.testing.assert_array_equal(sl[3], one[3][lo:hi])


@pytest.mark.gpu
def test_error_statuses(matcher):
    from metricsfm_b200 import _lib
    L, h = matcher._L, matcher._h
    rng = np.random.default_rng(63)
    xy = [rng.uniform(-500, 500, (40, 2)).astype(np.float32) for _ in range(3)]

    def call(pairs, offsets, matches, n_images, ptrs=None, npts=None, n_pairs=None):
        pa = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        npr = len(pa) if n_pairs is None else n_pairs
        offs = np.asarray(offsets, np.int64)
        m = np.ascontiguousarray(matches, np.int32).reshape(-1, 2)
        g = np.ones((max(len(m), 1),), np.uint8)
        arr = (C.c_void_p * 3)(*[a.ctypes.data for a in xy]) if ptrs is None else ptrs
        npts = np.array([40, 40, 40], np.int32) if npts is None else np.asarray(npts, np.int32)
        gp = _lib.GeoParams(3.0, 30, 30, 1024, 1, 0)
        ok = np.full((max(len(pa), 1),), -7, np.int32)
        inl = np.full((max(len(pa), 1),), -7, np.int32)
        keep = np.full((max(len(m), 1),), 9, np.uint8)
        H = np.full((max(len(pa), 1), 9), np.nan)
        st = L.msfm_geo_homography(h, pa.ctypes.data, npr, offs.ctypes.data, m.ctypes.data if len(m) else None,
                                   g.ctypes.data if len(m) else None, C.cast(arr, C.c_void_p), npts.ctypes.data, n_images,
                                   C.byref(gp), ok.ctypes.data, inl.ctypes.data, keep.ctypes.data, H.ctypes.data)
        return st, ok, inl, keep, H, L.msfm_last_error(h).decode()

    m_ok = np.stack([np.arange(40), np.arange(40)], 1)
    bad = [call([(0, 1)], [0, 40], np.where(np.arange(80).reshape(40, 2) == 79, 40, m_ok), 3),   # match past keypoints
           call([(0, 1), (1, 3)], [0, 40, 40], m_ok, 3),                                        # image >= n_images
           call([(0, 2)], [0, 40], m_ok, 3, ptrs=(C.c_void_p * 3)(xy[0].ctypes.data, xy[1].ctypes.data, None)),
           call([(0, 1)], [0, 40], m_ok, 3, n_pairs=-1)]
    for st, ok, inl, keep, H, msg in bad:
        assert st == 1
        assert (ok == -7).all() and (inl == -7).all() and (keep == 9).all() and np.isnan(H).all()
        assert "msfm_geo_homography" in msg, msg
    st, ok, *_ = call(np.zeros((0, 2)), [0], np.zeros((0, 2)), 0, n_pairs=0)
    assert st == 0 and ok[0] == -7
    st, ok, inl, keep, H, _ = call([(0, 1), (1, 2), (2, 0)], [0, 0, 0, 0], np.zeros((0, 2)), 3)
    assert st == 0 and ok.tolist() == [0, 0, 0] and inl.tolist() == [0, 0, 0] and (H == 0).all()
    assert L.msfm_geo_homography(None, None, 0, None, None, None, None, None, 0, None, None, None, None, None) == 1
