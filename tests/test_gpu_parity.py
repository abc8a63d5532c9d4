"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against the CPU oracle on
the same seeded inputs, against the committed golden vectors of the reference engine, and through size-independent
properties at full size.  Bar: bit-exact ids, distances and match lists (integer regime)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN_CASES
from metricsfm_b200 import synth
from oracle.geo_oracle import two_view_scene as _two_view_scene

pytestmark = pytest.mark.gpu

RATIOS = {"r50": 0.5, "r60": 0.6, "r85": 0.85}


@pytest.fixture(scope="module")
def matcher(native_lib):
    from metricsfm_b200.matcher import Matcher
    m = Matcher(device=0, max_images=256, arena_rows=1 << 20)
    yield m
    m.close()


def _upload_pair(matcher, ref, qry):
    matcher.release_all()
    matcher.upload(0, ref)
    matcher.upload(1, qry)


def _check_knn(oracle_mod, matcher, ref, qry):
    ids, dists = matcher.knn2(0, 1)
    oids, odists = oracle_mod.knn2_u8(ref, qry)
    np.testing.assert_array_equal(dists, odists)
    np.testing.assert_array_equal(ids, oids)
    return ids, dists


def test_packer_roundtrip_and_norms(matcher, golden):
    g = golden["basic"]
    _upload_pair(matcher, g["ref"], g["qry"])
    d, n = matcher.download_packed(0)
    np.testing.assert_array_equal(d, g["ref"])
    np.testing.assert_array_equal(n, (g["ref"].astype(np.int64) ** 2).sum(1).astype(np.uint32))
    # float upload: integer-valued floats at scale 1, unit-norm floats at scale 512 (quantiser golden)
    matcher.release_all()
    matcher.upload(0, g["ref"].astype(np.float32), scale=1.0)
    np.testing.assert_array_equal(matcher.download_packed(0)[0], g["ref"])
    fu = golden["float_unit"]
    matcher.upload(1, fu["unit"], scale=512.0)
    np.testing.assert_array_equal(matcher.download_packed(1)[0], fu["q512"])
    # strided rows (a cv::Mat ROI): every other row of a larger buffer
    big = np.zeros((2 * g["qry"].shape[0], 128), np.uint8)
    big[::2] = g["qry"]
    matcher.upload(2, big[::2])
    np.testing.assert_array_equal(matcher.download_packed(2)[0], g["qry"])
    bigf = np.zeros((2 * g["qry"].shape[0], 128), np.float32)
    bigf[::2] = g["qry"]
    matcher.upload(3, bigf[::2], scale=1.0)
    np.testing.assert_array_equal(matcher.download_packed(3)[0], g["qry"])


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_golden_reference_vectors(matcher, golden, case):
    g = golden[case]
    _upload_pair(matcher, g["ref"], g["qry"])
    ids, dists = matcher.knn2(0, 1)
    np.testing.assert_array_equal(dists, g["fm_dists"])
    np.testing.assert_array_equal(ids, g["fm_ids"])
    for tag, th in RATIOS.items():
        ok, pairs = matcher.MatchAgainstIndex(0, 1, th_ratio=th, th_reject=20)
        exp = g["fm_pairs_" + tag]
        if exp.shape[0] == 1 and exp[0, 0] == -7:
            assert not ok and len(pairs) == 0
        else:
            assert ok
            np.testing.assert_array_equal(pairs, exp)


@pytest.mark.parametrize("m,n", [(1, 1), (1, 40), (2, 2), (19, 20), (20, 20), (21, 127), (127, 128), (128, 129), (129, 255),
                                 (256, 256), (257, 513), (1000, 300), (300, 1000), (2049, 777)])
def test_knn2_ragged_sizes(oracle_mod, matcher, m, n):
    rng = np.random.default_rng(m * 7919 + n)
    ref = rng.integers(0, 256, size=(m, 128), dtype=np.uint8)
    qry = rng.integers(0, 256, size=(n, 128), dtype=np.uint8)
    _upload_pair(matcher, ref, qry)
    _check_knn(oracle_mod, matcher, ref, qry)
    cb, cd = matcher.colbest(0, 1)
    ob, od = oracle_mod.colbest_u8(ref, qry)
    np.testing.assert_array_equal(cd, od)
    np.testing.assert_array_equal(cb, ob)


def test_ties_duplicates_extremes(oracle_mod, matcher):
    rng = np.random.default_rng(77)
    ref = rng.integers(0, 4, size=(700, 128), dtype=np.uint8)   # tiny value range: masses of exact ties
    qry = rng.integers(0, 4, size=(515, 128), dtype=np.uint8)
    ref[100:110] = ref[5]
    ref[300] = 0
    ref[301] = 255
    qry[7] = ref[5]
    qry[8] = ref[5]
    qry[9] = 255
    qry[10] = 0
    _upload_pair(matcher, ref, qry)
    _check_knn(oracle_mod, matcher, ref, qry)
    cb, cd = matcher.colbest(0, 1)
    ob, od = oracle_mod.colbest_u8(ref, qry)
    np.testing.assert_array_equal(cd, od)
    np.testing.assert_array_equal(cb, ob)
    # worst-case magnitudes: all-255 vs all-0 rows give d = 128*255^2
    ref2 = np.zeros((40, 128), np.uint8)
    qry2 = np.full((33, 128), 255, np.uint8)
    ref2[3] = 255
    _upload_pair(matcher, ref2, qry2)
    ids, dists = _check_knn(oracle_mod, matcher, ref2, qry2)
    assert dists[0, 0] == 0 and dists[0, 1] == 128 * 255 * 255 and ids[0, 0] == 3 and ids[0, 1] == 0


def test_crosscheck_kernel_agrees(oracle_mod, matcher):
    col = synth.Collection(900, seed=31)
    ref, qry = col.image_u8(0, 900), col.image_u8(1, 650)
    _upload_pair(matcher, ref, qry)
    ids, dists = matcher.knn2(0, 1)
    cids, cdists = matcher.knn2_crosscheck(0, 1)
    np.testing.assert_array_equal(ids, cids)
    np.testing.assert_array_equal(dists, cdists)


@pytest.mark.parametrize("mutual", [False, True])
@pytest.mark.parametrize("orientation", [0, 1])
def test_match_pairs_batch_vs_oracle(oracle_mod, matcher, mutual, orientation):
    col = synth.Collection(1100, seed=41)
    rows = [1100, 980, 513, 19, 256, 1024, 0, 37]
    imgs = [col.image_u8(i, r) for i, r in enumerate(rows)]
    matcher.release_all()
    for i, d in enumerate(imgs):
        matcher.upload(i, d)
    pairs = [(0, 1), (1, 0), (0, 2), (2, 5), (3, 0), (0, 3), (4, 5), (5, 4), (6, 0), (0, 6), (7, 2), (1, 1)]
    res = matcher.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual, orientation=orientation)
    assert res.offsets[0] == 0 and res.offsets[-1] == len(res.matches)
    for p, (r, q) in enumerate(pairs):
        exp = oracle_mod.match_pair_u8(imgs[r], imgs[q], 0.85, mutual=mutual, orientation=orientation, ratio_good=0.6)
        assert bool(res.ok[p]) == exp["ok"], (p, r, q)
        np.testing.assert_array_equal(res.pair(p), exp["pairs"], err_msg=f"pair {p} = ({r},{q})")
        np.testing.assert_array_equal(res.pair_good(p), exp["good"], err_msg=f"pair {p} = ({r},{q})")
    total = matcher.match_pairs_resident(pairs, 0.85, ratio_good=0.6, mutual=mutual, orientation=orientation)
    assert total == len(res.matches)


def test_reference_shaped_entry_points(oracle_mod, matcher):
    col = synth.Collection(800, seed=43)
    d1, d2 = col.image_u8(0, 800), col.image_u8(1, 700)
    _upload_pair(matcher, d1, d2)
    ok, m = matcher.KNNMatching(0, 1)  # index on image 2, queries = image 1, (i1, i2) ascending i1
    exp = oracle_mod.match_pair_u8(d2, d1, 0.5, orientation=1)
    assert ok
    np.testing.assert_array_equal(m, exp["pairs"])
    assert (np.diff(m[:, 0]) > 0).all()


def test_max_dist_gate(oracle_mod, matcher):
    col = synth.Collection(600, seed=47)
    a, b = col.image_u8(0, 600), col.image_u8(1, 600)
    _upload_pair(matcher, a, b)
    res = matcher.match_pairs([(0, 1)], 0.85, max_dist_sq=40000.0)
    exp = oracle_mod.match_pair_u8(a, b, 0.85, max_dist_sq=40000.0)
    np.testing.assert_array_equal(res.pair(0), exp["pairs"])


def test_error_paths(matcher):
    from metricsfm_b200.matcher import MsfmError
    matcher.release_all()
    matcher.upload(0, np.zeros((30, 128), np.uint8))
    with pytest.raises(MsfmError) as e:
        matcher.knn2(0, 5)
    assert e.value.status == 4
    with pytest.raises(MsfmError) as e:
        matcher.upload(0, np.zeros((30, 128), np.uint8))
    assert e.value.status == 7
    with pytest.raises(MsfmError) as e:
        matcher.upload(100000, np.zeros((30, 128), np.uint8))
    assert e.value.status == 1
    matcher.upload(1, np.zeros((30, 128), np.uint8))
    with pytest.raises(MsfmError) as e:
        matcher.match_pairs([(0, 9)], 0.6)
    assert e.value.status == 4
    with pytest.raises(MsfmError) as e:   # caller buffer too small for the matches -> capacity error, not overflow
        rng = np.random.default_rng(5)
        matcher.upload(2, rng.integers(0, 256, size=(64, 128), dtype=np.uint8))
        matcher.upload(3, rng.integers(0, 256, size=(64, 128), dtype=np.uint8))
        matcher.match_pairs([(2, 3)], 0.99, capacity=1)
    assert e.value.status == 5
    matcher.release(0)
    matcher.upload(0, np.ones((40, 128), np.uint8))  # slot and arena space are reusable after release
    assert matcher.image_info(0)[0] == 40


def test_full_size_8k_pair_vs_oracle(oracle_mod, matcher):
    """BASELINE config #1: 2 x 8192 x 128, one pair — the oracle still finishes in seconds here."""
    col = synth.Collection(8192, seed=1)
    a, b = col.image_u8(0), col.image_u8(1)
    _upload_pair(matcher, a, b)
    ids, dists = _check_knn(oracle_mod, matcher, a, b)
    for mutual in (False, True):
        res = matcher.match_pairs([(0, 1)], 0.6, mutual=mutual)
        exp = oracle_mod.match_pair_u8(a, b, 0.6, mutual=mutual)
        np.testing.assert_array_equal(res.pair(0), exp["pairs"])
    assert len(res.matches) > 50  # the synthetic pair has real correspondences


def test_full_size_properties_20k(oracle_mod, matcher):
    """Config #3 shape (20 000 rows, ragged): properties that need no full oracle pass."""
    col = synth.Collection(20000, seed=2)
    a, b = col.image_u8(0), col.image_u8(1)
    _upload_pair(matcher, a, b)
    ids, dists = matcher.knn2(0, 1)
    # (1) self-consistency: recompute the two reported distances exactly on the host
    qa = b.astype(np.int64)
    for col_i in (0, 1):
        ref_rows = a[ids[:, col_i]].astype(np.int64)
        np.testing.assert_array_equal(((qa - ref_rows) ** 2).sum(1).astype(np.float32), dists[:, col_i])
    assert (dists[:, 0] <= dists[:, 1]).all() and (ids[:, 0] != ids[:, 1]).all()
    # (2) optimality on a random sample of query rows against the oracle
    rng = np.random.default_rng(3)
    sample = np.sort(rng.choice(20000, size=256, replace=False))
    oids, odists = oracle_mod.knn2_u8(a, b[sample])
    np.testing.assert_array_equal(ids[sample], oids)
    np.testing.assert_array_equal(dists[sample], odists)
    # (3) symmetry: the column-best of (a,b) equals the row-best of the swapped problem
    cb, cd = matcher.colbest(0, 1)
    sids, sdists = matcher.knn2(1, 0)
    np.testing.assert_array_equal(cb, sids[:, 0])
    np.testing.assert_array_equal(cd, sdists[:, 0])
    # (4) mutual matches are a subset of one-way matches and are one-to-one
    one = matcher.match_pairs([(0, 1)], 0.85).pair(0)
    mut = matcher.match_pairs([(0, 1)], 0.85, mutual=True).pair(0)
    assert {tuple(p) for p in mut} <= {tuple(p) for p in one}
    assert len(np.unique(mut[:, 0])) == len(mut) and (np.diff(mut[:, 1]) > 0).all()
    # (5) idempotence
    ids2, dists2 = matcher.knn2(0, 1)
    np.testing.assert_array_equal(ids, ids2)
    np.testing.assert_array_equal(dists, dists2)


def test_cpp_host_shim_matches_oracle(oracle_mod, native_lib, tmp_path):
    """The C++ mirror of the reference interface (cv::Mat CV_32FC1 in, vector<pair<int,int>> out), driven the way
    MetricSfM would drive FeatureMatching::KNNMatching / the FLANN-layout kNN / BuildMatchGraph's loops."""
    import subprocess
    from metricsfm_b200 import build
    exe = build.build_host_shim()
    col = synth.Collection(700, seed=51)
    d1, d2 = col.image_u8(0, 700), col.image_u8(1, 611)
    raw = tmp_path / "desc.f32"
    np.concatenate([d1, d2]).astype(np.float32).tofile(raw)
    out = subprocess.check_output([exe, str(raw), str(len(d1)), str(len(d2))], text=True).split("\n")
    it = iter(out)
    head = next(it).split()
    assert head[0] == "KNNMatching" and head[1] == "1"
    got = np.array([next(it).split() for _ in range(int(head[2]))], dtype=np.int32).reshape(-1, 2)
    exp = oracle_mod.match_pair_u8(d2, d1, 0.5, orientation=1)["pairs"]      # index on image 2, queries = image 1
    np.testing.assert_array_equal(got, exp)
    head = next(it).split()
    assert head[0] == "KNN2" and head[1] == "1"
    rows = np.array([next(it).split() for _ in range(int(head[2]))], dtype=np.float64)
    oids, odists = oracle_mod.knn2_u8(d1, d2)
    np.testing.assert_array_equal(rows[:, :2].astype(np.int32), oids)
    np.testing.assert_array_equal(rows[:, 2:].astype(np.float32), odists)

    def block(name):
        head = next(it).split()
        assert head[0] == name, head
        n = int(head[-1])
        return head, np.array([next(it).split() for _ in range(max(n, 0))], dtype=np.int32).reshape(-1, 2)

    head, got = block("Run")                                               # FeatureMatchingCudaSift::Run: mutual best match
    assert head[1] == "1"
    np.testing.assert_array_equal(got, oracle_mod.match_pair_u8(d2, d1, 0.5, orientation=1, mutual=True)["pairs"])
    for _ in range(2):                                                     # persistent indices, queried twice
        head, got = block("Index1")                                        # index on image 1, (i1, i2) ascending i2
        assert head[1] == "1"
        np.testing.assert_array_equal(got, oracle_mod.match_pair_u8(d1, d2, 0.5, orientation=0)["pairs"])
        head, got = block("Index2")                                        # index on image 2, (i1, i2) ascending i1
        assert head[1] == "1"
        np.testing.assert_array_equal(got, exp)
    # SiftMatchGPU shape: set 0 = queries (image 1), set 1 = image 2; ratio 0.8 on squared L2, mutual, no keypoint gate
    head, got = block("SiftMatch")
    full = oracle_mod.match_pair_u8(d2, d1, 0.8, orientation=1, mutual=True, min_keypoints=0)["pairs"]
    np.testing.assert_array_equal(got, full)
    head, got = block("SiftMatchCapped")                                   # max_match truncates the one-way list
    oneway = oracle_mod.match_pair_u8(d2, d1, 0.8, orientation=1, min_keypoints=0)["pairs"]
    assert len(oneway) > 5
    np.testing.assert_array_equal(got, oneway[:5])
    head, got = block("SiftMatchGated")                                    # distmax 0.2 rad -> squared-L2 gate
    gate = float(np.float32(512.0 * 512.0 * (2.0 - 2.0 * np.cos(np.float64(np.float32(0.2))))))
    gated = oracle_mod.match_pair_u8(d2, d1, 0.8, orientation=1, min_keypoints=0, max_dist_sq=gate)["pairs"]
    np.testing.assert_array_equal(got, gated)
    assert 0 < len(gated) <= len(oneway)
    assert next(it).split() == ["MatchPairs", "1"]
    for ref, qry in ((d1, d2), (d2, d1)):
        head = next(it).split()
        n = int(head[5])
        got = np.array([next(it).split() for _ in range(n)], dtype=np.int32).reshape(-1, 3)
        exp = oracle_mod.match_pair_u8(ref, qry, 0.85, ratio_good=0.6)
        np.testing.assert_array_equal(got[:, :2], exp["pairs"])
        np.testing.assert_array_equal(got[:, 2], exp["good"])


def test_adversarial_norm_spread_and_near_ties(oracle_mod, matcher):
    """Inputs that defeat the pruning filter (huge spread of reference norms, scores within 1 of each other across
    columns and tiles): results must stay bit-exact, only slower."""
    rng = np.random.default_rng(91)
    ref = rng.integers(0, 256, size=(1300, 128), dtype=np.uint8)
    ref[::3] //= 8                      # a third of the rows with tiny norms, interleaved inside every tile
    ref[1::7] = 255 - ref[1::7] // 16   # and some with huge norms
    qry = rng.integers(0, 256, size=(700, 128), dtype=np.uint8)
    # near-ties: copies of a query row differing by +-1 in one coordinate, scattered over columns of several tiles
    base = qry[5].copy()
    for n, j in enumerate((3, 70, 130, 200, 640, 705, 1290)):
        r = base.copy()
        r[n] = np.clip(int(r[n]) + (1 if n % 2 else -1), 0, 255)
        ref[j] = r
    ref[64] = base                      # exact hit in the first column of tile 1
    ref[900] = base                     # and an equal-distance duplicate far to the right (must lose the tie)
    _upload_pair(matcher, ref, qry)
    ids, dists = _check_knn(oracle_mod, matcher, ref, qry)
    assert ids[5, 0] == 64 and ids[5, 1] == 900 and dists[5, 0] == 0 and dists[5, 1] == 0
    for mutual in (False, True):
        res = matcher.match_pairs([(0, 1), (1, 0)], 0.9, ratio_good=0.7, mutual=mutual)
        for p, (r, q) in enumerate(((ref, qry), (qry, ref))):
            exp = oracle_mod.match_pair_u8(r, q, 0.9, mutual=mutual, ratio_good=0.7)
            np.testing.assert_array_equal(res.pair(p), exp["pairs"])
            np.testing.assert_array_equal(res.pair_good(p), exp["good"])


def test_many_small_and_uneven_pairs(oracle_mod, matcher):
    """Guided-pair-list shape: many pairs of uneven, ragged sizes in one call (work items of every fill level)."""
    rng = np.random.default_rng(93)
    sizes = [int(x) for x in rng.integers(20, 1400, size=24)] + [255, 256, 257, 511, 512, 513]
    col = synth.Collection(1400, seed=61)
    imgs = [col.image_u8(i, r) for i, r in enumerate(sizes)]
    matcher.release_all()
    for i, d in enumerate(imgs):
        matcher.upload(i, d)
    pairs = synth.gps_neighbour_pairs(len(sizes), k=5, seed=3)
    pairs = np.concatenate([pairs, pairs[::3, ::-1]])          # some pairs in both orientations
    res = matcher.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=True)
    assert res.ok.all()
    for p, (r, q) in enumerate(pairs):
        exp = oracle_mod.match_pair_u8(imgs[r], imgs[q], 0.85, mutual=True, ratio_good=0.6)
        np.testing.assert_array_equal(res.pair(p), exp["pairs"], err_msg=f"pair {p} = ({r},{q})")
        np.testing.assert_array_equal(res.pair_good(p), exp["good"])


@pytest.mark.parametrize("rows", [16384, 32768])
def test_full_size_properties_16k_32k(oracle_mod, matcher, rows):
    """Config #4 / #5 shapes (16 384 / 32 768 rows per image): sampled optimality + self-consistency through the batched
    entry point."""
    col = synth.Collection(rows, seed=4)
    a, b = col.image_u8(0), col.image_u8(1)
    _upload_pair(matcher, a, b)
    ids, dists = matcher.knn2(0, 1)
    rng = np.random.default_rng(5)
    sample = np.sort(rng.choice(rows, size=192, replace=False))
    oids, odists = oracle_mod.knn2_u8(a, b[sample])
    np.testing.assert_array_equal(ids[sample], oids)
    np.testing.assert_array_equal(dists[sample], odists)
    res = matcher.match_pairs([(0, 1)], 0.85, ratio_good=0.6, mutual=True)
    m = res.pair(0)
    assert len(m) > 500 and (np.diff(m[:, 1]) > 0).all() and len(np.unique(m[:, 0])) == len(m)
    # every emitted match is the query's nearest neighbour, passes the ratio, and is mutual (checked on the host)
    np.testing.assert_array_equal(ids[m[:, 1], 0], m[:, 0])
    r = dists[m[:, 1], 0] / dists[m[:, 1], 1]
    assert (r < np.float32(0.85)).all()
    np.testing.assert_array_equal(res.pair_good(0), (r < np.float32(0.6)).astype(np.uint8))
    back_ids, _ = matcher.knn2(1, 0)                # nearest query row of every reference row
    np.testing.assert_array_equal(back_ids[m[:, 0], 0], m[:, 1])


# ---------------------------------------------------------------------------------------------------- float regime
def _fp32_lists(oracle_mod, ref_f, qry_f, ratio, ratio_good, mutual):
    """Match list of an exact fp32 brute-force matcher (squared L2 accumulated in index order, nanoflann.hpp:376-383)."""
    ids, dists = oracle_mod.knn2_f32(ref_f, qry_f)
    cb = oracle_mod.colbest_f32(ref_f, qry_f)[0] if mutual else None
    return oracle_mod.ratio_select(ids, dists, ref_f.shape[0], ratio, col_best=cb, ratio_good=ratio_good)


@pytest.mark.parametrize("mutual", [False, True])
def test_float_regime_rescoring_matches_fp32_matcher(oracle_mod, native_lib, mutual):
    """Unit-norm float descriptors (the CUDASIFT container, feature_extractor_cuda_sift.cpp:75-80), scale 512: with the
    float rows retained and a 3 % re-scoring band the match lists equal those of an exact fp32 matcher (north_star
    tolerance: <= 1e-4 of the matches flip; here none may), while the purely quantised path does flip some."""
    from metricsfm_b200.matcher import Matcher
    rows, n_img = 4096, 4
    col = synth.Collection(rows, seed=11)
    imgs = [col.image_unit(i) for i in range(n_img)]
    pairs = [(0, 1), (2, 3), (1, 2), (3, 0)]
    with Matcher(device=0, max_images=8, arena_rows=1 << 16, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x, scale=512.0)
        res = m.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual, rescore_band=0.03)
        raw = m.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual)
    total = flips = flips_raw = good_diff = 0
    for p, (r, q) in enumerate(pairs):
        exp, exp_good = _fp32_lists(oracle_mod, imgs[r], imgs[q], 0.85, 0.6, mutual)
        got, got_good = res.pair(p), res.pair_good(p)
        se, sg = {tuple(x) for x in exp}, {tuple(x) for x in got}
        flips += len(se ^ sg)
        flips_raw += len(se ^ {tuple(x) for x in raw.pair(p)})
        total += len(se)
        ge = {tuple(x): int(f) for x, f in zip(exp, exp_good)}
        good_diff += sum(1 for x, f in zip(got, got_good) if tuple(x) in ge and ge[tuple(x)] != int(f))
        assert (np.diff(got[:, 1]) > 0).all()
    assert total > 1000
    assert flips == 0, f"{flips} of {total} matches differ from the fp32 matcher"
    assert good_diff == 0
    assert flips_raw > 0  # the reason the re-scoring band exists


@pytest.mark.parametrize("cap", [0, 37])
def test_float_regime_collect_pass_equals_brute_force(native_lib, cap):
    """The band rows' fp32 neighbours come from the tensor kernel's collect pass + per-event scoring; when its event list
    overflows (forced here through the msfm_test_set_band_event_cap hook) a dp4a brute force over the reference image takes over.  Both must
    produce identical match lists and good flags, with and without the mutual check, on ragged images."""
    from metricsfm_b200.matcher import Matcher
    col = synth.Collection(3000, seed=13)
    rows = [3000, 2500, 1111, 600, 3000]
    imgs = [col.image_unit(i)[:r] for i, r in enumerate(rows)]
    pairs = [(0, 1), (1, 0), (2, 4), (4, 3), (3, 2), (0, 4)]

    def run(event_cap=-1):
        out = []
        with Matcher(device=0, max_images=8, arena_rows=1 << 15, keep_float=True) as m:
            m._test_set_band_event_cap(event_cap)
            for i, x in enumerate(imgs):
                m.upload(i, np.ascontiguousarray(x), scale=512.0)
            for mutual in (False, True):
                res = m.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual, rescore_band=0.03)
                out.append([(res.pair(p).copy(), res.pair_good(p).copy()) for p in range(len(pairs))])
        return out

    collected = run()
    brute = run(cap)
    n = 0
    for a, b in zip(collected, brute):
        for (ma, ga), (mb, gb) in zip(a, b):
            np.testing.assert_array_equal(ma, mb)
            np.testing.assert_array_equal(ga, gb)
            n += len(ma)
    assert n > 1000


def test_float_regime_needs_retained_rows(oracle_mod, matcher):
    """rescore_band on a context without retained float rows, or on u8 uploads, is a no-op (integer decision)."""
    col = synth.Collection(1024, seed=12)
    a, b = col.image_u8(0), col.image_u8(1)
    _upload_pair(matcher, a, b)
    r0 = matcher.match_pairs([(0, 1)], 0.85, ratio_good=0.6, mutual=True)
    r1 = matcher.match_pairs([(0, 1)], 0.85, ratio_good=0.6, mutual=True, rescore_band=0.05)
    np.testing.assert_array_equal(r0.pair(0), r1.pair(0))
    np.testing.assert_array_equal(r0.pair_good(0), r1.pair_good(0))


# ---------------------------------------------------------------------------------------------------- graph driver
def test_build_match_graph_driver_writes_reference_files(oracle_mod, native_lib, tmp_path):
    """FineMatchingGraph::BuildMatchGraph rebuilt on the GPU matcher: feature files in, <idx>_match / match_index.txt /
    graph_matching.txt out — byte-identical to the reference's control flow driven by the CPU oracle's match lists,
    including resume after an interrupted run."""
    import shutil
    from metricsfm_b200 import build, store
    from oracle import store_oracle as so
    build.build_host_libs()
    n_img = 6
    col = synth.Collection(1500, seed=21)
    rows = [1500, 1200, 900, 1500, 19, 640]                       # image 4 is below the 20-keypoint gate
    imgs = [col.image_u8(i, r) for i, r in enumerate(rows)]
    rng = np.random.default_rng(5)
    fold_gpu, fold_ref = str(tmp_path / "gpu"), str(tmp_path / "ref")
    os.makedirs(fold_gpu), os.makedirs(fold_ref)
    for i, d in enumerate(imgs):
        xy = rng.uniform(0, 3000, size=(d.shape[0], 2)).astype(np.float32)
        # VLSIFT container: integer-valued floats in a CV_32FC1 matrix (odd images) / CV_8UC1 rows (even images)
        store.feature_write(store.feature_path(fold_gpu, i), rows=3000, cols=4000, xy_pixel=xy,
                            desc=d.astype(np.float32) if i % 2 else d)
    adj = [[1, 2, 4], [0, 3], [5], [], [0], [2, 3]]
    offs = np.cumsum([0] + [len(a) for a in adj]).astype(np.int64)
    lst = np.array([j for a in adj for j in a], np.int32)

    def match_fn(i1, i2):
        r = oracle_mod.match_pair_u8(imgs[i1], imgs[i2], 0.85, ratio_good=0.6, mutual=True, min_keypoints=20)
        return r["ok"], r["pairs"], r["good"]

    # interrupted run: images 0 and 1 already finished (their files come from the reference flow)
    so.build_match_graph_files(fold_ref, [adj[0], adj[1]] + [[] for _ in range(4)], match_fn, min_good=5)
    os.remove(fold_ref + "//graph_matching.txt")
    open(fold_ref + "//match_index.txt", "w").write("0\n1\n")
    for name in ("0_match", "1_match", "match_index.txt"):
        shutil.copy(fold_ref + "//" + name, fold_gpu + "//" + name)
    so.build_match_graph_files(fold_ref, adj, match_fn, min_good=5)
    store.build_match_graph(fold_gpu, offs, lst, mutual=True, min_keypoints=20, min_good=5)
    names = sorted(f for f in os.listdir(fold_ref))
    assert names == sorted(f for f in os.listdir(fold_gpu) if not f.endswith("_feature"))
    assert {"0_match", "2_match", "graph_matching.txt", "match_index.txt"} <= set(names)
    for name in names:
        assert open(fold_ref + "//" + name, "rb").read() == open(fold_gpu + "//" + name, "rb").read(), name
    # a second call finds nothing missing and leaves the files alone
    before = {n: os.path.getmtime(fold_gpu + "//" + n) for n in names}
    store.build_match_graph(fold_gpu, offs, lst, mutual=True, min_keypoints=20, min_good=5)
    assert before == {n: os.path.getmtime(fold_gpu + "//" + n) for n in names}
    # the verification seam: keep only the good matches of accepted pairs
    fold_v = str(tmp_path / "verify")
    os.makedirs(fold_v)
    for i in range(n_img):
        shutil.copy(store.feature_path(fold_gpu, i), store.feature_path(fold_v, i))
    store.build_match_graph(fold_v, offs, lst, mutual=True, min_keypoints=20,
                            verify=lambda i1, i2, xy1, xy2, m, g: (int(g.sum()) >= 5, np.nonzero(g)[0]))
    ids, lists = store.match_read(fold_v, 0)
    exp = oracle_mod.match_pair_u8(imgs[0], imgs[1], 0.85, ratio_good=0.6, mutual=True)
    assert ids[0] == 1
    np.testing.assert_array_equal(lists[0], exp["pairs"][exp["good"] == 1])


# ---------------------------------------------------------------------------------------------------- geo-verification
def test_geo_verification_against_opencv_and_restatement(matcher):
    """Batched GPU GeoVerificationFundamental (utils/geo_verification.cc:30-79): stage B is exact given F (numpy
    restatement); stage A agrees with cv2.findFundamentalMat(FM_RANSAC, 3 px) on decisions and inlier sets."""
    import cv2
    from metricsfm_b200.matcher import MatchResult
    from oracle import geo_oracle as go
    rng = np.random.default_rng(31)
    scenes = [(_two_view_scene(rng, 400, 130), 380),      # rigid scene, 25 % outliers, 380 "good" of 530 "all"
              (_two_view_scene(rng, 90, 60), 120),
              (_two_view_scene(rng, 25, 0), 25),          # fewer than 30 good matches: rejected before RANSAC
              (_two_view_scene(rng, 0, 300), 200),        # no geometry at all: rejected (inliers < 30)
              (_two_view_scene(rng, 3000, 900), 2600)]    # more good matches than the shared-memory point cap
    image_xy, pairs, offsets, matches, good = {}, [], [0], [], []
    for s, ((p1, p2), n_good) in enumerate(scenes):
        n = len(p1)
        perm1, perm2 = rng.permutation(n), rng.permutation(n)      # keypoint ids are not in match order
        xy1, xy2 = np.empty_like(p1), np.empty_like(p2)
        xy1[perm1], xy2[perm2] = p1, p2
        image_xy[2 * s], image_xy[2 * s + 1] = xy1, xy2
        pairs.append((2 * s, 2 * s + 1))
        m = np.stack([perm1, perm2], 1).astype(np.int32)
        gflag = np.zeros((n,), np.uint8)
        gflag[rng.choice(n, n_good, replace=False)] = 1
        matches.append(m), good.append(gflag), offsets.append(offsets[-1] + n)
    res = MatchResult(offsets=np.array(offsets, np.int64), ok=np.ones((len(pairs),), np.int32), matches=np.concatenate(matches),
                      good=np.concatenate(good))
    ok, inl, keep, F = matcher.geo_verify(pairs, res, image_xy, seed=7)
    ok2, inl2, keep2, F2 = matcher.geo_verify(pairs, res, image_xy, seed=7)
    np.testing.assert_array_equal(ok, ok2), np.testing.assert_array_equal(keep, keep2), np.testing.assert_array_equal(F, F2)
    assert ok.tolist() == [1, 1, 0, 0, 1]
    for s, ((p1, p2), n_good) in enumerate(scenes):
        a, b = offsets[s], offsets[s + 1]
        g = good[s].astype(bool)
        k = keep[a:b].astype(bool)
        if not ok[s]:
            assert not k.any()
            continue
        # exact restatement around the returned F: stage-A inlier count and stage-B mask
        eok, einl, ekeep = go.verify_pair(p1[g], p2[g], p1, p2, F[s])
        assert eok and einl == inl[s]
        np.testing.assert_array_equal(k, ekeep)
        # statistical parity with OpenCV's RANSAC
        Fcv, mask = cv2.findFundamentalMat(p1[g], p2[g], cv2.FM_RANSAC, 3.0, 0.99)
        n_cv = int(mask.sum())
        n_true = [400, 90, 25, 0, 3000][s]
        true_good = int(g[:n_true].sum())
        # OpenCV stops at 99 % confidence, so its consensus set is a lower bound; the true correspondences among the
        # good matches (plus the odd outlier that happens to lie on an epipolar line) are the upper bound
        assert n_cv >= 30 and 0.97 * n_cv - 3 <= inl[s] <= true_good + 0.06 * (g.sum() - true_good) + 3, (inl[s], n_cv, true_good)
        kcv = go.f_filter(Fcv, p1, p2)
        # what the filter around OpenCV's F keeps is (nearly) contained in what ours keeps; the excess is bounded by
        # the ground truth below
        assert (k & kcv).sum() >= 0.97 * kcv.sum(), ((k & kcv).sum(), kcv.sum())
        assert k[:n_true].mean() >= 0.97                               # true correspondences survive
        assert k[n_true:].mean() <= 0.12                               # random outliers rarely lie within 3 px of a line
    _, _, keep3, _ = matcher.geo_verify(pairs, res, image_xy, seed=8)   # another RANSAC stream: same decisions, ~same sets
    assert (keep3 != keep).mean() < 0.01


def test_build_match_graph_with_gpu_geo_verification(oracle_mod, native_lib, tmp_path):
    """The driver with the reference's verification stages on the GPU: descriptors decide the matches, keypoints of a
    rigid two-view scene decide which survive; a pair without common geometry leaves no record."""
    from metricsfm_b200 import build, store
    from oracle import geo_oracle as go
    build.build_host_libs()
    rng = np.random.default_rng(41)
    n = 1200
    col = synth.Collection(n, seed=33)
    base = col.image_u8(0)
    # image 1 = image 0 re-observed (same descriptors, permuted, slightly perturbed), image 2 = unrelated descriptors
    perm = rng.permutation(n)
    d1 = np.clip(base[perm].astype(np.int32) + rng.integers(-2, 3, size=(n, 128)), 0, 255).astype(np.uint8)
    d2 = col.image_u8(5)
    p0, p1 = _two_view_scene(rng, n, 0)
    xy = [p0, p1[perm], rng.uniform(-1800, 1800, (n, 2)).astype(np.float32)]
    xy[1][: n // 5] = rng.uniform(-1800, 1800, (n // 5, 2))           # 20 % of the re-observations moved: outliers
    fold = str(tmp_path)
    for i, (d, p) in enumerate(zip([base, d1, d2], xy)):
        # the writer centres pixel coordinates: feed "pixel" coordinates that centre back onto the scene coordinates
        store.feature_write(store.feature_path(fold, i), rows=4000, cols=4000, xy_pixel=p + 2000.0, desc=d)
    adj = [[1, 2], [], []]
    offs = np.cumsum([0] + [len(a) for a in adj]).astype(np.int64)
    store.build_match_graph(fold, offs, np.array([1, 2], np.int32), geo_verify=True, geo_seed=3)
    ids, lists = store.match_read(fold, 0)
    assert ids.tolist() == [1]                                         # the unrelated pair was rejected
    kept = lists[0]
    exp = oracle_mod.match_pair_u8(base, d1, 0.85, ratio_good=0.6)["pairs"]
    assert {tuple(m) for m in kept} <= {tuple(m) for m in exp} and len(kept) > 0.7 * len(exp)
    # every kept match is a descriptor match whose keypoints agree with ONE epipolar geometry: refit F on them
    import cv2
    F, _ = cv2.findFundamentalMat(xy[0][kept[:, 0]], xy[1][kept[:, 1]], cv2.FM_LMEDS)
    assert go.f_filter(F, xy[0][kept[:, 0]], xy[1][kept[:, 1]], 4.0).mean() > 0.97
    moved = np.isin(kept[:, 1], np.arange(n // 5))
    assert moved.mean() < 0.03                                         # the moved keypoints were filtered out
    g = store.graph_read(fold, 3)
    assert g[0, 1] == len(kept) and g[0, 2] == 0


def test_upload_batch_equals_single_uploads(oracle_mod, matcher):
    """msfm_upload_u8_batch (one host wait per batch; contiguous rows go straight into the arena and are keyed in place)
    leaves the same table as per-image uploads, including two strided members (one with a stride that is not a multiple
    of 128 bytes) and an empty image."""
    col = synth.Collection(700, seed=13)
    imgs = [col.image_u8(0, 700), col.image_u8(1, 513), np.empty((0, 128), np.uint8), col.image_u8(3, 64), col.image_u8(4, 300)]
    big = np.zeros((2 * 513, 128), np.uint8)
    big[::2] = imgs[1]
    wide = np.zeros((300, 200), np.uint8)                     # a 128-byte ROI at byte 64 of 200-byte rows
    wide[:, 64:192] = imgs[4]
    matcher.release_all()
    matcher.upload_batch([0, 1, 2, 3, 4], [imgs[0], big[::2], imgs[2], imgs[3], wide[:, 64:192]])
    for i, d in enumerate(imgs):
        got, norms = matcher.download_packed(i)
        np.testing.assert_array_equal(got, d)
        np.testing.assert_array_equal(norms, (d.astype(np.int64) ** 2).sum(1).astype(np.uint32))
    ids, dists = matcher.knn2(0, 1)
    oids, odists = oracle_mod.knn2_u8(imgs[0], imgs[1])
    np.testing.assert_array_equal(ids, oids)
    np.testing.assert_array_equal(dists, odists)
    res = matcher.match_pairs([(0, 1), (1, 3), (0, 2)], 0.85, ratio_good=0.6, mutual=True)
    exp = oracle_mod.match_pair_u8(imgs[1], imgs[3], 0.85, mutual=True, ratio_good=0.6)
    np.testing.assert_array_equal(res.pair(1), exp["pairs"])
    assert res.ok.tolist() == [1, 1, 0]


def test_upload_batch_async_overlaps_and_matches(oracle_mod, matcher):
    """msfm_upload_u8_batch_async: no host wait, adjacent images coalesced into one copy; the table and the match lists
    equal the synchronous upload's, strided rows are refused, msfm_sync drains the stream."""
    import torch
    from metricsfm_b200.matcher import MsfmError
    col = synth.Collection(768, seed=14)
    rows = [768, 512, 300, 0, 256]                       # 768/512/256 are multiples of the arena alignment: one coalesced copy
    host = torch.empty((sum(rows), 128), dtype=torch.uint8).pin_memory()
    views, lo = [], 0
    for i, r in enumerate(rows):
        host[lo:lo + r].numpy()[:] = col.image_u8(i, r) if r else np.empty((0, 128), np.uint8)
        views.append(host[lo:lo + r])
        lo += r
    matcher.release_all()
    matcher.upload_batch(list(range(5)), views, wait=False)
    res = matcher.match_pairs([(0, 1), (2, 4), (1, 4)], 0.85, ratio_good=0.6, mutual=True)   # queued behind the copies
    matcher.sync()
    for i, v in enumerate(views):
        got, norms = matcher.download_packed(i)
        np.testing.assert_array_equal(got, v.numpy())
        np.testing.assert_array_equal(norms, (v.numpy().astype(np.int64) ** 2).sum(1).astype(np.uint32))
    for p, (r, q) in enumerate([(0, 1), (2, 4), (1, 4)]):
        exp = oracle_mod.match_pair_u8(views[r].numpy(), views[q].numpy(), 0.85, mutual=True, ratio_good=0.6)
        np.testing.assert_array_equal(res.pair(p), exp["pairs"])
    matcher.release_all()
    strided = np.zeros((200, 256), np.uint8)[:, :128]
    with pytest.raises(MsfmError):
        matcher.upload_batch([0], [strided], wait=False)


def test_upload_f32_three_ways_equal():
    """The same float images uploaded with contiguous rows, with strided rows and with msfm_upload_f32_batch_async from
    adjacent page-locked views (adjacent images coalesced into one copy) leave identical tables, and on a keep_float
    context identical retained float rows, residuals and largest residuals: msfm_knn2_pairs in exact fp32 mode gives
    identical arrays."""
    import torch
    from metricsfm_b200.matcher import Matcher
    col = synth.Collection(768, seed=15)
    rows = [768, 512, 300, 0, 256]                       # 768 and 512 rows are adjacent in the arena too
    imgs = [col.image_unit(i, r) for i, r in enumerate(rows)]
    host = torch.from_numpy(np.concatenate(imgs)).pin_memory()
    bounds = np.cumsum([0] + rows)
    views = [host[a:b] for a, b in zip(bounds[:-1], bounds[1:])]
    pairs = [(0, 1), (1, 2), (2, 4), (4, 0), (1, 0)]

    def strided(x):
        big = np.zeros((2 * x.shape[0], 128), np.float32)
        big[::2] = x
        return big[::2]

    for keep_float in (True, False):
        out = []
        for how in ("contiguous", "strided", "batch_async"):
            with Matcher(device=0, max_images=8, arena_rows=1 << 15, keep_float=keep_float) as m:
                if how == "batch_async":
                    m.upload_f32_batch_async(list(range(len(rows))), views, scale=512.0)
                    m.sync()
                else:
                    for i, x in enumerate(imgs):
                        m.upload(i, x if how == "contiguous" else strided(x), scale=512.0)
                tables = [m.download_packed(i) for i in range(len(rows))]
                knn = m.knn2_pairs(pairs, exact_f32=keep_float)
            out.append((how, tables, knn))
        _, tables0, knn0 = out[0]
        for how, tables, knn in out[1:]:
            for (d0, n0), (d, n) in zip(tables0, tables):
                np.testing.assert_array_equal(d, d0, err_msg=f"{how} keep_float {keep_float}")
                np.testing.assert_array_equal(n, n0, err_msg=f"{how} keep_float {keep_float}")
            for a0, a in zip(knn0, knn):
                np.testing.assert_array_equal(a, a0, err_msg=f"{how} keep_float {keep_float}")


def test_reserve_batch_equals_single_reserves(matcher):
    """msfm_reserve_batch lays the images out exactly like one msfm_reserve per image (multi-GPU replication relies on
    every rank reproducing the same offsets)."""
    rows = [700, 0, 256, 513, 8192]
    matcher.release_all()
    single = [matcher.reserve(i, r) for i, r in enumerate(rows)]
    matcher.release_all()
    batch = matcher.reserve_batch(list(range(len(rows))), rows)
    assert batch.tolist() == single
    assert [matcher.image_info(i)[0] for i in range(len(rows))] == rows


def test_maximum_rows_per_image(oracle_mod, native_lib):
    """MSFM_MAX_ROWS_PER_IMAGE = idx_max_per_image = 1 000 000 (basic_structs.h:171): a million-row image as the
    reference set (15 625 tiles per work item) and as the query set (1 954 work items), against the oracle."""
    from metricsfm_b200.matcher import Matcher, MsfmError
    rng = np.random.default_rng(77)
    big = rng.integers(0, 40, size=(1_000_000, 128), dtype=np.uint8)
    big[rng.choice(1_000_000, 5000, replace=False)] += 100               # some structure in the norms
    small = big[rng.choice(1_000_000, 300, replace=False)].copy()
    small = np.clip(small.astype(np.int32) + rng.integers(-3, 4, size=small.shape), 0, 255).astype(np.uint8)
    with Matcher(device=0, max_images=4, arena_rows=1_000_000 + 4096) as m:
        m.upload(0, big)
        m.upload(1, small)
        with pytest.raises(MsfmError):
            m.reserve(2, 1_000_001)                                          # one row past the limit
        ids, dists = m.knn2(0, 1)                                            # 300 queries against a million rows
        oids, odists = oracle_mod.knn2_u8(big, small)
        np.testing.assert_array_equal(ids, oids)
        np.testing.assert_array_equal(dists, odists)
        ids2, dists2 = m.knn2(1, 0)                                          # a million queries against 300 rows
        sample = np.sort(rng.choice(1_000_000, 4000, replace=False))
        oids2, odists2 = oracle_mod.knn2_u8(small, big[sample])
        np.testing.assert_array_equal(ids2[sample], oids2)
        np.testing.assert_array_equal(dists2[sample], odists2)
        res = m.match_pairs([(0, 1)], 0.85, ratio_good=0.6, mutual=True)
        exp = oracle_mod.match_pair_u8(big, small, 0.85, mutual=True, ratio_good=0.6)
        np.testing.assert_array_equal(res.pair(0), exp["pairs"])


def test_many_images_many_pairs_batches(oracle_mod, native_lib):
    """Collection-scale bookkeeping (configs #3-#5 have 10^3-10^4 images and 10^4-10^5 pairs): 3 000 small images, 40 000
    retrieval-style pairs => several internal batches (16 384 pairs each); sampled pairs against the oracle, totals
    against a second call."""
    from metricsfm_b200.matcher import Matcher
    n_img = 3000
    rng = np.random.default_rng(88)
    sizes = rng.integers(18, 90, size=n_img)                                  # some images below the 20-keypoint gate
    col = synth.Collection(90, seed=71)
    imgs = [col.image_u8(i % 50, int(r)) for i, r in enumerate(sizes)]       # 50 distinct scenes re-used
    pairs = synth.retrieval_pairs(n_img, partners=14, seed=5)
    assert len(pairs) > 32768
    with Matcher(device=0, max_images=n_img, arena_rows=n_img * 256) as m:
        m.upload_batch(list(range(n_img)), imgs)
        res = m.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=True)
        total = m.match_pairs_resident(pairs, 0.85, ratio_good=0.6, mutual=True)
    assert total == len(res.matches) == int(res.offsets[-1])
    gated = (sizes[pairs[:, 0]] < 20) | (sizes[pairs[:, 1]] < 20)
    np.testing.assert_array_equal(res.ok, (~gated).astype(np.int32))
    assert gated.any() and (np.diff(res.offsets) >= 0).all()
    for p in rng.choice(len(pairs), 150, replace=False).tolist() + [0, 16383, 16384, 32767, 32768, len(pairs) - 1]:
        r, q = pairs[p]
        exp = oracle_mod.match_pair_u8(imgs[r], imgs[q], 0.85, mutual=True, ratio_good=0.6)
        np.testing.assert_array_equal(res.pair(p), exp["pairs"], err_msg=f"pair {p} = ({r},{q})")
        np.testing.assert_array_equal(res.pair_good(p), exp["good"])


def test_build_match_graph_chunking_is_invisible(native_lib, tmp_path):
    """The driver processes the missing images in bounded chunks (host match buffers, incremental match_index.txt):
    whatever the chunk size, the files are byte-identical — including the GPU geo-verification's RANSAC draws."""
    import shutil
    from metricsfm_b200 import build, store
    build.build_host_libs()
    rng = np.random.default_rng(51)
    n = 900
    col = synth.Collection(n, seed=44)
    base = col.image_u8(0)
    imgs, xys = [], []
    p0, p1 = _two_view_scene(rng, n, 0)
    for i in range(6):
        perm = rng.permutation(n)
        d = np.clip(base[perm].astype(np.int32) + rng.integers(-2, 3, size=(n, 128)), 0, 255).astype(np.uint8)
        imgs.append(d)
        xys.append((p0 if i % 2 == 0 else p1)[perm])                       # even / odd images: the two views of one scene
    folds = [str(tmp_path / name) for name in ("one", "small", "tiny")]
    adj = [[1, 3, 5], [2, 4], [3], [0, 5], [], [0]]
    offs = np.cumsum([0] + [len(a) for a in adj]).astype(np.int64)
    lst = np.array([j for a in adj for j in a], np.int32)
    for fold, chunk in zip(folds, (0, 2 * n, 1)):
        os.makedirs(fold)
        for i, (d, p) in enumerate(zip(imgs, xys)):
            store.feature_write(store.feature_path(fold, i), rows=4000, cols=4000, xy_pixel=p + 2000.0, desc=d)
        store.build_match_graph(fold, offs, lst, geo_verify=True, geo_seed=9, max_batch_rows=chunk)
    names = sorted(f for f in os.listdir(folds[0]) if not f.endswith("_feature"))
    assert "0_match" in names and "graph_matching.txt" in names
    for fold in folds[1:]:
        assert names == sorted(f for f in os.listdir(fold) if not f.endswith("_feature"))
        for name in names:
            assert open(folds[0] + "//" + name, "rb").read() == open(fold + "//" + name, "rb").read(), (fold, name)
    g = store.graph_read(folds[0], 6)
    assert g[0, 1] > 300 and g[0, 3] > 300        # different views of the scene: verified


def test_cpp_shim_verified_matcher_vs_opencv_flow(oracle_mod, native_lib, tmp_path):
    """FeatureMatchingB200::KNNMatchingWithGeoVerify against the reference's flow (feature_matching.cpp:67-150) run with
    the CPU oracle's ratio matches and cv2: homography-degeneracy gate, RANSAC-F at 3 px then 1 px.  RANSAC parity is
    statistical (OpenCV's RNG stream cannot be reproduced); the DLT homography is compared with cv2.findHomography."""
    import subprocess
    import cv2
    from metricsfm_b200 import build
    exe = build.build_host_shim()
    rng = np.random.default_rng(61)
    n = 1500
    col = synth.Collection(n, seed=62)
    d1 = col.image_u8(0)
    perm = rng.permutation(n)
    d2 = np.clip(d1[perm].astype(np.int32) + rng.integers(-2, 3, size=(n, 128)), 0, 255).astype(np.uint8)
    p1, p2 = _two_view_scene(rng, n, 0, noise=0.3)
    xy1, xy2 = p1 + 2000.0, p2[perm] + 2000.0
    xy2[: n // 5] = rng.uniform(0, 4000, (n // 5, 2))                      # 20 % of the re-observations moved: outliers

    def run(xy_b):
        raw, kpf = tmp_path / "desc.f32", tmp_path / "kp.f32"
        np.concatenate([d1, d2]).astype(np.float32).tofile(raw)
        np.concatenate([xy1, xy_b]).astype(np.float32).tofile(kpf)
        out = subprocess.check_output([exe, str(raw), str(n), str(n), str(kpf)], text=True).split("\n")
        i = next(k for k, l in enumerate(out) if l.startswith("GeoVerify"))
        ok, cnt = int(out[i].split()[1]), int(out[i].split()[2])
        got = np.array([l.split() for l in out[i + 1:i + 1 + cnt]], dtype=np.int32).reshape(-1, 2)
        h = out[i + 1 + cnt].split()
        ha = next(l for l in out if l.startswith("HomographyAll")).split()
        return ok, got, int(h[1]), np.array(h[2:], np.float64).reshape(3, 3), np.array(ha[2:], np.float64).reshape(3, 3)

    ok, got, okh, H, _ = run(xy2)
    # the reference flow on the CPU
    cur = oracle_mod.match_pair_u8(d2, d1, 0.5, orientation=1)["pairs"]      # index on image 2, (i1, i2) ascending i1
    assert {tuple(m) for m in got} <= {tuple(m) for m in cur}
    for th in (3.0, 1.0):
        a, b = xy1[cur[:, 0]].astype(np.float32), xy2[cur[:, 1]].astype(np.float32)
        Hcv, _ = cv2.findHomography(a, b, 0)
        assert not all(abs(Hcv[i, i] - 0.995) < 0.01 for i in range(3))
        _, mask = cv2.findFundamentalMat(a, b, cv2.FM_RANSAC, th, 0.99)
        cur = cur[mask.ravel() > 0]
    assert ok == 1
    sg, sc = {tuple(m) for m in got}, {tuple(m) for m in cur}
    assert len(sg & sc) >= 0.93 * len(sc), (len(sg), len(sc), len(sg & sc))   # OpenCV's consensus is (nearly) contained
    moved = np.isin(got[:, 1], np.arange(n // 5))
    assert moved.mean() < 0.02 and len(got) > 0.6 * (n - n // 5) * 0.5
    # DLT homography of the surviving matches vs OpenCV's least-squares estimate
    a, b = xy1[got[:, 0]].astype(np.float32), xy2[got[:, 1]].astype(np.float32)
    Hcv, _ = cv2.findHomography(a, b, 0)
    assert okh == 1
    pa = np.concatenate([a, np.ones((len(a), 1), np.float32)], 1).astype(np.float64)
    qa, qb = pa @ H.T, pa @ Hcv.T
    err = np.abs(qa[:, :2] / qa[:, 2:] - qb[:, :2] / qb[:, 2:]).max(axis=1)
    # the scene has depth, so no homography fits it: the algebraic (DLT) and the LM-polished least-squares estimates agree
    # to a few pixels on a 4000-pixel image, far inside what the 0.01 identity test resolves
    assert np.median(err) < 8.0 and err.max() < 80.0, (np.median(err), err.max())
    # no parallax: image 2 observed from the same place => homography ~ identity => the matcher refuses the pair
    xy_same = (xy1[perm] * 0.995 + rng.normal(0, 0.2, (n, 2))).astype(np.float32)
    ok2, got2, _, _, Hall = run(xy_same)
    assert ok2 == 0 and len(got2) == 0
    allm = oracle_mod.match_pair_u8(d2, d1, 0.5, orientation=1)["pairs"]
    Hcv, _ = cv2.findHomography(xy1[allm[:, 0]].astype(np.float32), xy_same[allm[:, 1]], 0)
    np.testing.assert_allclose(Hall, Hcv / Hcv[2, 2], atol=2e-3)              # where the gate matters, DLT == OpenCV's estimate
    assert all(abs(Hall[i, i] - 0.995) < 0.01 for i in range(3))


# ---------------------------------------------------------------------------------------------------- round 2
def _adversarial_mutual_images(seed=5):
    """Images built to stress the mutual check: near-duplicate clusters (tiny second-neighbour distances => large
    'dangerous' sets), exact duplicates (ties in both directions), and ordinary SIFT-like rows in between."""
    rng = np.random.default_rng(seed)
    col = synth.Collection(1500, seed=seed)
    base = col.image_u8(0, 60).astype(np.int16)
    clus = np.repeat(base, 30, axis=0) + rng.integers(-1, 2, size=(1800, 128))          # 60 clusters x 30 near-copies
    clus = np.clip(clus, 0, 255).astype(np.uint8)
    a = np.concatenate([col.image_u8(1, 900), clus[:900], col.image_u8(1, 40)], axis=0)  # + 40 exact duplicates of its head
    b = np.concatenate([clus[600:1500], col.image_u8(2, 1000), col.image_u8(1, 40)[::-1]], axis=0)
    c = np.concatenate([clus[::2], clus[1::2][:300]], axis=0)
    d = col.image_u8(3, 1500)
    # 5000 noisy copies of ONE row on both sides: every row's second neighbour is closer than any accepted match, so the
    # dangerous list overflows (> kDangerListCap) and the pair must take the tensor twin pass
    one = col.image_u8(4, 1).astype(np.int16)
    e = np.clip(one + rng.integers(-2, 3, size=(5000, 128)), 0, 255).astype(np.uint8)
    f = np.clip(one + rng.integers(-2, 3, size=(5200, 128)), 0, 255).astype(np.uint8)
    return [np.ascontiguousarray(x) for x in (a, b, c, d, e, f)]


@pytest.mark.parametrize("ratio,flags", [(0.85, 0), (0.97, 0), (0.999, 1)])
def test_mutual_check_bound_path_and_twin_path_vs_oracle(oracle_mod, native_lib, ratio, flags):
    """The mutual cross-check is decided from the forward results (column table + exactly scored 'dangerous' rows) and
    falls back to the tensor twin pass for ambiguous pairs.  Both routes, and the forced-twin route, must reproduce the
    oracle's column-best rule bit for bit — also on near-duplicate clusters and exact ties."""
    from metricsfm_b200.matcher import Matcher
    imgs = _adversarial_mutual_images()
    pairs = [(r, q) for r in range(4) for q in range(4)] + [(4, 5), (5, 4), (4, 0)]
    with Matcher(device=0, max_images=8, arena_rows=1 << 16) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x)
        auto = m.match_pairs(pairs, ratio, ratio_good=0.6, mutual=True, flags=flags)
        t_auto = m.timing()
        m._test_force_twin_pass(True)
        forced = m.match_pairs(pairs, ratio, ratio_good=0.6, mutual=True, flags=flags)
        t_forced = m.timing()
        m._test_force_twin_pass(False)
        oneway = m.match_pairs(pairs, ratio, ratio_good=0.6, mutual=False, flags=flags)
    assert t_forced["twin_pairs"] > t_auto["twin_pairs"]          # ordinary pairs are decided without the tensor pass
    if ratio > 0.9:
        assert t_auto["twin_pairs"] >= 2                           # the 5000-copy pairs overflow the dangerous list
    n = 0
    for p, (r, q) in enumerate(pairs):
        exp = oracle_mod.match_pair_u8(imgs[r], imgs[q], ratio, mutual=True, ratio_good=0.6, reject_gt=bool(flags))
        np.testing.assert_array_equal(auto.pair(p), exp["pairs"], err_msg=f"bound route, pair ({r},{q})")
        np.testing.assert_array_equal(forced.pair(p), exp["pairs"], err_msg=f"twin route, pair ({r},{q})")
        np.testing.assert_array_equal(auto.pair_good(p), exp["good"])
        np.testing.assert_array_equal(forced.pair_good(p), exp["good"])
        ow = oracle_mod.match_pair_u8(imgs[r], imgs[q], ratio, mutual=False, ratio_good=0.6, reject_gt=bool(flags))
        np.testing.assert_array_equal(oneway.pair(p), ow["pairs"])
        n += len(exp["pairs"])
    assert n > 500


def test_mutual_check_ordinary_collection_never_needs_the_twin_pass(oracle_mod, native_lib):
    col = synth.Collection(4096, seed=77)
    imgs = [col.image_u8(i) for i in range(4)]
    pairs = [(0, 1), (1, 2), (2, 3), (3, 0), (0, 2)]
    from metricsfm_b200.matcher import Matcher
    with Matcher(device=0, max_images=4, arena_rows=1 << 15) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x)
        res = m.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=True)
        t = m.timing()
    assert t["twin_pairs"] == 0 and t["match_launches"] >= 1
    for p, (r, q) in enumerate(pairs):
        exp = oracle_mod.match_pair_u8(imgs[r], imgs[q], 0.85, mutual=True, ratio_good=0.6)
        np.testing.assert_array_equal(res.pair(p), exp["pairs"])
        np.testing.assert_array_equal(res.pair_good(p), exp["good"])


def test_slam_ratio_rule(oracle_mod, matcher):
    """SLAMGPS::FeatureMatching (slam_gps.cc:470-477) rejects a row iff ratio > 0.80: non-strict, and 0/0 = NaN passes.
    Rows with d0 = d1 = 0 (duplicated reference rows) and rows sitting exactly on the threshold tell the rules apart."""
    col = synth.Collection(700, seed=91)
    ref = col.image_u8(0, 700)
    qry = col.image_u8(1, 600)
    ref[10] = ref[11] = qry[5]              # d0 = d1 = 0 for query row 5: NaN ratio
    # query row 7: d0/d1 == 0.5 exactly (d0 = 8, d1 = 16 against two crafted reference rows)
    qry[7] = 100
    ref[20] = 100; ref[20, :2] = 102        # d = 4 + 4 = 8
    ref[21] = 100; ref[21, :4] = 102        # d = 16
    _upload_pair(matcher, ref, qry)
    from metricsfm_b200 import _lib
    for th in (0.5, 0.8):
        got = matcher.match_pairs([(0, 1)], th, min_keypoints=0, flags=_lib.RATIO_REJECT_GT)
        exp = oracle_mod.match_pair_u8(ref, qry, th, min_keypoints=0, reject_gt=True)
        np.testing.assert_array_equal(got.pair(0), exp["pairs"])
        strict = matcher.match_pairs([(0, 1)], th, min_keypoints=0)
        exp_s = oracle_mod.match_pair_u8(ref, qry, th, min_keypoints=0)
        np.testing.assert_array_equal(strict.pair(0), exp_s["pairs"])
        assert 5 in got.pair(0)[:, 1] and 5 not in strict.pair(0)[:, 1]
    at_half = matcher.match_pairs([(0, 1)], 0.5, min_keypoints=0, flags=_lib.RATIO_REJECT_GT).pair(0)
    assert 7 in at_half[:, 1] and 7 not in matcher.match_pairs([(0, 1)], 0.5, min_keypoints=0).pair(0)[:, 1]
    np.testing.assert_array_equal(matcher.SLAMFeatureMatching(0, 1, th_first_second_ratio=0.8),
                                  oracle_mod.match_pair_u8(ref, qry, 0.8, min_keypoints=0, reject_gt=True)["pairs"])


def test_async_upload_groups_overlap_matching(oracle_mod, native_lib):
    """Images staged in groups on the upload stream (u8 and f32, no host wait) while earlier groups are matched: every
    launch waits on the device for exactly the uploads it needs; lists equal those of synchronous uploads."""
    import torch
    from metricsfm_b200.matcher import Matcher
    col = synth.Collection(2048, seed=17)
    n = 12
    rows = [2048 - 37 * i for i in range(n)]
    u8 = torch.empty((n, 2048, 128), dtype=torch.uint8).pin_memory()
    f32 = torch.empty((n, 2048, 128), dtype=torch.float32).pin_memory()
    for i in range(n):
        u8[i, :rows[i]] = torch.from_numpy(col.image_u8(i, rows[i]))
        f32[i, :rows[i]] = u8[i, :rows[i]].float()
    groups = [list(range(g, g + 4)) for g in range(0, n, 4)]
    all_pairs = synth.exhaustive_pairs(n)
    with Matcher(device=0, max_images=n, arena_rows=n * 2048 + 4096) as m:
        for i in range(n):
            m.upload(i, u8[i, :rows[i]].numpy())
        ref = m.match_pairs(all_pairs, 0.85, ratio_good=0.6, mutual=True)
        for use_f32 in (False, True):
            m.release_all()
            got = {}
            for g, ids in enumerate(groups):
                if use_f32:
                    m.upload_f32_batch_async(ids, [f32[i, :rows[i]] for i in ids], scale=1.0)
                else:
                    m.upload_batch(ids, [u8[i, :rows[i]] for i in ids], wait=False)
            for g, ids in enumerate(groups):     # pairs whose newest image lies in group g
                sel = [k for k, (a, b) in enumerate(all_pairs) if max(a, b) // 4 == g]
                res = m.match_pairs(all_pairs[sel], 0.85, ratio_good=0.6, mutual=True)
                for j, k in enumerate(sel):
                    got[k] = (res.pair(j).copy(), res.pair_good(j).copy())
            m.sync()
            for k in range(len(all_pairs)):
                np.testing.assert_array_equal(got[k][0], ref.pair(k))
                np.testing.assert_array_equal(got[k][1], ref.pair_good(k))
    exp = oracle_mod.match_pair_u8(u8[0, :rows[0]].numpy(), u8[1, :rows[1]].numpy(), 0.85, mutual=True, ratio_good=0.6)
    np.testing.assert_array_equal(ref.pair(0), exp["pairs"])


def test_failed_batch_upload_leaves_no_half_uploaded_image(matcher):
    """An upload that fails must not leave an image 'present' with unwritten rows (ADVICE r1): the failing id of a batch is
    absent afterwards, the images before it stay uploaded, and a retry succeeds."""
    from metricsfm_b200.matcher import MsfmError
    col = synth.Collection(300, seed=3)
    a, b = col.image_u8(0, 300), col.image_u8(1, 200)
    matcher.release_all()
    matcher.upload(2, a)
    with pytest.raises(MsfmError):
        matcher.upload_batch([0, 2, 1], [a, b, b])          # id 2 exists already
    assert matcher.image_info(0)[0] == 300
    with pytest.raises(MsfmError):
        matcher.image_info(1)
    with pytest.raises((MsfmError, ValueError)):
        matcher.upload(5, a[:, :64])                          # malformed rows never reserve
    with pytest.raises(MsfmError):
        matcher.image_info(5)
    matcher.upload(1, b)
    got, _ = matcher.download_packed(1)
    np.testing.assert_array_equal(got, b)


@pytest.mark.parametrize("ratio,ratio_good,flags", [(0.85, 0.6, 0), (0.5, 0.0, 0), (0.8, 0.0, 1), (0.95, 0.6, 0)])
def test_dead_row_rule_is_invisible(oracle_mod, native_lib, ratio, ratio_good, flags):
    """Forward pass with the dead-row rule (rows that already violate every tested ratio follow only their nearest
    neighbour exactly, match_kernel.cuh) against the same call with the rule switched off and against the oracle: one-way
    and mutual lists and the 'good' flags must be identical — on SIFT-like images, on images whose rows sit in tight
    clusters (ratios near 1 and exact ties, the mutual check's dangerous-row bound at work) and on rows engineered to
    die early and be revived by a much closer neighbour in the LAST reference tile."""
    from metricsfm_b200.matcher import Matcher
    rng = np.random.default_rng(4242)
    col = synth.Collection(3000, seed=5)
    a, b = col.image_u8(0, 3000), col.image_u8(1, 2777)
    centres = rng.integers(0, 120, size=(40, 128))
    c = np.clip(centres[rng.integers(0, 40, 2500)] + rng.integers(-3, 4, size=(2500, 128)), 0, 255).astype(np.uint8)
    d = np.clip(centres[rng.integers(0, 40, 2100)] + rng.integers(-3, 4, size=(2100, 128)), 0, 255).astype(np.uint8)
    # revival: query rows of e copy rows of the last tile of f (+ tiny noise), so the true match arrives after ~3000 rivals
    f = col.image_u8(2, 3001)
    e = col.image_u8(3, 900)
    e[:300] = np.clip(f[-300:].astype(np.int32) + rng.integers(-2, 3, size=(300, 128)), 0, 255).astype(np.uint8)
    imgs = [np.ascontiguousarray(x) for x in (a, b, c, d, e, f)]
    pairs = [(0, 1), (1, 0), (2, 3), (3, 2), (5, 4), (4, 5), (0, 3), (2, 1)]
    with Matcher(device=0, max_images=8, arena_rows=1 << 16) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x)
        out = {}
        for prune in (True, False):
            m._test_disable_pruning(not prune)
            for mutual in (False, True):
                out[prune, mutual] = m.match_pairs(pairs, ratio, ratio_good=ratio_good, mutual=mutual, flags=flags)
        m._test_disable_pruning(False)
        ids, dists = m.knn2(5, 4)   # the S1/S2 seam always reports exact neighbours
    oids, odists = oracle_mod.knn2_u8(imgs[5], imgs[4])
    np.testing.assert_array_equal(ids, oids)
    np.testing.assert_array_equal(dists, odists)
    n = 0
    for mutual in (False, True):
        for p, (r, q) in enumerate(pairs):
            exp = oracle_mod.match_pair_u8(imgs[r], imgs[q], ratio, mutual=mutual, ratio_good=ratio_good, reject_gt=bool(flags))
            for prune in (True, False):
                np.testing.assert_array_equal(out[prune, mutual].pair(p), exp["pairs"], err_msg=f"prune={prune} mutual={mutual} pair ({r},{q})")
                if ratio_good > 0:
                    np.testing.assert_array_equal(out[prune, mutual].pair_good(p), exp["good"], err_msg=f"good flags, prune={prune} mutual={mutual} pair ({r},{q})")
            n += len(exp["pairs"])
    assert n > 300
