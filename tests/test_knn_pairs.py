"""msfm_knn2_pairs: FLANN-layout kNN arrays of a whole pair list, in integer units (flags 0, bit-identical to msfm_knn2)
or exact in fp32 on the retained float rows (MSFM_KNN_EXACT_F32).

The CPU test restates the exact mode's candidate bound T(q) (aux_kernels.cuh, exact_threshold) in numpy and checks that
it holds every fp32 top-2 neighbour, including on rows built so that the float regime's former heuristic threshold misses
one.  The GPU tests compare the call with msfm_knn2, the CPU oracle and the golden vectors, bit for bit."""
import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN_CASES
from metricsfm_b200 import synth

S512 = 512.0


# ---------------------------------------------------------------------------------------------------- the bound (CPU)
def _quantize(x, scale):
    """The packer's rule: q = min(255, max(0, rint(fp32(x * scale))))."""
    return np.clip(np.rint(np.asarray(x, np.float32) * np.float32(scale)), 0, 255)


def _residuals(x, scale):
    """r_x = ||scale * x - q_x||_2 with the real product scale * x."""
    return np.sqrt(((np.asarray(x, np.float64) * scale - _quantize(x, scale)) ** 2).sum(1))


def _quantised_d2(qq, qr):
    """Exact integer squared distances of packed rows, [query, ref] (float64 holds them exactly)."""
    qq, qr = qq.astype(np.float64), qr.astype(np.float64)
    return (qq ** 2).sum(1)[:, None] + (qr ** 2).sum(1)[None, :] - 2.0 * (qq @ qr.T)


def _exact_threshold(d1q, rx, rmax):
    """T(q) = (sqrt(d1_q) + 2 (r_x + R))^2, widened by 2^-15 for the fp32 distance sum, rounded up."""
    return np.ceil((np.sqrt(d1q) + 2.0 * (rx + rmax)) ** 2 * (1.0 + 2.0 ** -15))


def _heuristic_threshold(d1q):
    """The re-scoring threshold msfm_match_pairs used before it took T(q): d1 + d1/32 + 256."""
    return d1q + np.floor(d1q / 32.0) + 256.0


def _adversarial_rows():
    """A float query row of zeros and three reference rows: A = 29/512 in element 0, C = 29/512 in element 1,
    B = 2.51/512 in elements 1..127.  Quantised: A = C = 841, B = 1143; in fp32 B (800.1 / 512^2) is the true nn0."""
    q = np.zeros((1, 128), np.float32)
    ref = np.zeros((3, 128), np.float32)
    ref[0, 0] = 29.0 / 512.0
    ref[1, 1:] = 2.51 / 512.0
    ref[2, 1] = 29.0 / 512.0
    return q, ref  # reference order A, B, C


def _check_bound(oracle_mod, ref, qry, scale):
    qr, qq = _quantize(ref, scale), _quantize(qry, scale)
    dq = _quantised_d2(qq, qr)
    d1q = np.partition(dq, 1, axis=1)[:, 1] if ref.shape[0] > 1 else np.full(qry.shape[0], np.inf)
    T = _exact_threshold(d1q, _residuals(qry, scale), _residuals(ref, scale).max())
    ids, _ = oracle_mod.knn2_f32(ref, qry)  # the fp32 matcher's top-2 (nanoflann arithmetic, lowest index on ties)
    rows = np.arange(qry.shape[0])[:, None]
    top = dq[rows, ids]
    assert (top <= T[:, None]).all(), f"{int((top > T[:, None]).any(1).sum())} rows with an fp32 top-2 row beyond T(q)"
    return dq, d1q, T, ids


def test_exact_threshold_bound_holds(oracle_mod):
    """Every fp32 top-2 neighbour lies within T(q): on synthetic unit-norm images (scale 512), on the same rows in the
    512-scaled VLSIFT regime (scale 1), and on the adversarial rows, which the heuristic band misses."""
    col = synth.Collection(2048, seed=11)
    for a, b in [(0, 1), (2, 3)]:
        ref, qry = col.image_unit(a), col.image_unit(b)
        _check_bound(oracle_mod, ref, qry, S512)
        _check_bound(oracle_mod, ref * np.float32(512.0), qry * np.float32(512.0), 1.0)
    q, ref = _adversarial_rows()
    dq, d1q, T, ids = _check_bound(oracle_mod, ref, q, S512)
    np.testing.assert_array_equal(dq[0], [841.0, 1143.0, 841.0])
    assert ids[0, 0] == 1  # B is the fp32 nearest neighbour
    assert dq[0, 1] > _heuristic_threshold(d1q[0])  # ... outside the heuristic band (1123): the case needs the bound
    assert dq[0, 1] <= T[0] < 1700


# ---------------------------------------------------------------------------------------------------- GPU: integer mode
def _matcher(**kw):
    from metricsfm_b200.matcher import Matcher
    return Matcher(device=0, **kw)


def _slices(offsets, ids, dists, p):
    return ids[offsets[p]:offsets[p + 1]], dists[offsets[p]:offsets[p + 1]]


@pytest.mark.gpu
def test_integer_mode_equals_knn2_and_oracle(oracle_mod, native_lib):
    """flags 0 on u8 uploads: every pair's rows equal msfm_knn2 and the oracle, bit for bit — ragged sizes, 0- and
    1-row images, the pair (i, i) and repeated pairs in one list."""
    rng = np.random.default_rng(5)
    sizes = [0, 1, 2, 129, 700, 1000, 2049, 513, 1]
    imgs = [rng.integers(0, 256, size=(n, 128), dtype=np.uint8) for n in sizes]
    pairs = [(2, 3), (3, 2), (4, 4), (0, 5), (5, 0), (1, 6), (6, 1), (7, 6), (6, 7), (4, 5), (2, 3), (8, 8), (0, 0), (6, 8),
             (5, 6), (4, 5)]
    with _matcher(max_images=16, arena_rows=1 << 16) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x)
        offsets, ids, dists = m.knn2_pairs(pairs)
        assert offsets[0] == 0 and offsets[-1] == ids.shape[0] == sum(sizes[q] for _, q in pairs)
        for p, (r, q) in enumerate(pairs):
            gi, gd = _slices(offsets, ids, dists, p)
            ki, kd = m.knn2(r, q)
            np.testing.assert_array_equal(gi, ki)
            np.testing.assert_array_equal(gd, kd)
            oi, od = oracle_mod.knn2_u8(imgs[r], imgs[q])
            np.testing.assert_array_equal(gi, oi)
            np.testing.assert_array_equal(gd, od)
        # an empty list is a valid call
        offsets, ids, _ = m.knn2_pairs(np.zeros((0, 2), np.int32))
        assert offsets.tolist() == [0] and ids.shape[0] == 0


@pytest.mark.gpu
def test_integer_mode_reproduces_golden_vectors(native_lib, golden):
    """The golden fm_ids / fm_dists of the reference engine's cases, all in one batched call."""
    with _matcher(max_images=2 * len(GOLDEN_CASES), arena_rows=1 << 16) as m:
        for k, case in enumerate(GOLDEN_CASES):
            m.upload(2 * k, golden[case]["ref"])
            m.upload(2 * k + 1, golden[case]["qry"])
        pairs = [(2 * k, 2 * k + 1) for k in range(len(GOLDEN_CASES))]
        offsets, ids, dists = m.knn2_pairs(pairs)
    for k, case in enumerate(GOLDEN_CASES):
        gi, gd = _slices(offsets, ids, dists, k)
        np.testing.assert_array_equal(gd, golden[case]["fm_dists"])
        np.testing.assert_array_equal(gi, golden[case]["fm_ids"])


def _many_small_pairs(n_img=24, rows=64, n_pairs=17000, seed=9):
    """More pairs than one batch holds (16384), drawn with repetition from n_img^2 combinations."""
    rng = np.random.default_rng(seed)
    pairs = rng.integers(0, n_img, size=(n_pairs, 2)).astype(np.int32)
    return pairs, rows


@pytest.mark.gpu
def test_integer_mode_spans_several_batches(oracle_mod, native_lib):
    pairs, rows = _many_small_pairs()
    rng = np.random.default_rng(3)
    imgs = [rng.integers(0, 256, size=(rows, 128), dtype=np.uint8) for _ in range(24)]
    with _matcher(max_images=32, arena_rows=1 << 16) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x)
        offsets, ids, dists = m.knn2_pairs(pairs)
    expect = {}
    for p, (r, q) in enumerate(pairs.tolist()):
        if (r, q) not in expect:
            expect[(r, q)] = oracle_mod.knn2_u8(imgs[r], imgs[q])
        gi, gd = _slices(offsets, ids, dists, p)
        np.testing.assert_array_equal(gi, expect[(r, q)][0])
        np.testing.assert_array_equal(gd, expect[(r, q)][1])


# ---------------------------------------------------------------------------------------------------- GPU: exact mode
def _assert_exact(oracle_mod, imgs, pairs, offsets, ids, dists):
    for p, (r, q) in enumerate(pairs):
        gi, gd = _slices(offsets, ids, dists, p)
        oi, od = oracle_mod.knn2_f32(imgs[r], imgs[q])
        np.testing.assert_array_equal(gi, oi, err_msg=f"pair {p} ({r}, {q}) ids")
        np.testing.assert_array_equal(gd, od, err_msg=f"pair {p} ({r}, {q}) dists")


@pytest.mark.gpu
def test_exact_mode_equals_fp32_matcher_unit_norm(oracle_mod, native_lib):
    """Unit-norm rows at scale 512 (several 4096-row pairs and one 8192-row pair): ids and dists of an exhaustive fp32
    matcher, bit for bit.  The 8192-row pair is decided by the collect path; with the event list capped at 0 the brute
    force decides it, identically.  The integer-unit result of the same images differs from fp32 somewhere."""
    col = synth.Collection(4096, seed=11)
    imgs = [col.image_unit(i) for i in range(4)]
    big = synth.Collection(8192, seed=12)
    imgs += [big.image_unit(0), big.image_unit(1)]
    small_pairs = [(0, 1), (2, 3), (1, 2), (3, 0)]
    with _matcher(max_images=8, arena_rows=1 << 16, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x, scale=S512)
        offsets, ids, dists = m.knn2_pairs(small_pairs, exact_f32=True)
        _assert_exact(oracle_mod, imgs, small_pairs, offsets, ids, dists)
        offsets, ids, dists = m.knn2_pairs([(4, 5)], exact_f32=True)
        events, brute = m._test_last_knn_stats()
        assert brute == 0 and events >= 8192
        _assert_exact(oracle_mod, imgs, [(4, 5)], offsets, ids, dists)
        int_offsets, int_ids, _ = m.knn2_pairs([(4, 5)])
        assert (int_ids != ids).any()  # quantised units do pick other neighbours: the reason the exact mode exists
        m._test_set_band_event_cap(0)
        bo, bi, bd = m.knn2_pairs([(4, 5)], exact_f32=True)
        assert m._test_last_knn_stats()[1] == 1
        np.testing.assert_array_equal(bi, ids)
        np.testing.assert_array_equal(bd, dists)


@pytest.mark.gpu
def test_exact_mode_vlsift_regime_and_adversarial_rows(oracle_mod, native_lib):
    """Non-integer 512-scaled rows at scale 1 (VLSIFT), ragged; and the adversarial rows embedded in larger images:
    B, outside the heuristic band, is the zero row's fp32 nearest neighbour."""
    col = synth.Collection(3000, seed=13)
    vl = [col.image_unit(i)[:n] * np.float32(512.0) for i, n in enumerate([3000, 2500, 1111])]
    vl_pairs = [(0, 1), (1, 0), (2, 0), (1, 2), (2, 2)]
    q0, adv = _adversarial_rows()
    ref = col.image_unit(5)[:2000].copy()
    ref[[100, 1500, 1999]] = adv  # A, B, C
    qry = col.image_unit(6)[:1500].copy()
    qry[700] = q0[0]
    with _matcher(max_images=8, arena_rows=1 << 15, keep_float=True) as m:
        for i, x in enumerate(vl):
            m.upload(i, np.ascontiguousarray(x), scale=1.0)
        offsets, ids, dists = m.knn2_pairs(vl_pairs, exact_f32=True)
        _assert_exact(oracle_mod, vl, vl_pairs, offsets, ids, dists)
        assert m._test_last_knn_stats()[1] == 0
        m.upload(5, ref, scale=S512)
        m.upload(6, qry, scale=S512)
        offsets, ids, dists = m.knn2_pairs([(5, 6)], exact_f32=True)
        _assert_exact(oracle_mod, {5: ref, 6: qry}, [(5, 6)], offsets, ids, dists)
        assert ids[700, 0] == 1500
        assert m._test_last_knn_stats()[1] == 0


@pytest.mark.gpu
def test_exact_mode_spans_several_batches_and_empty_images(oracle_mod, native_lib):
    """More pairs than one batch holds, plus 0- and 1-row float images (rows read absent / one neighbour)."""
    pairs, rows = _many_small_pairs(n_img=20, n_pairs=16500, seed=4)
    col = synth.Collection(rows, seed=21)
    imgs = [col.image_unit(i) for i in range(20)] + [np.zeros((0, 128), np.float32), col.image_unit(30)[:1]]
    extra = np.array([[20, 3], [3, 20], [21, 4], [4, 21], [21, 21]], np.int32)
    pairs = np.concatenate([pairs, extra])
    with _matcher(max_images=24, arena_rows=1 << 15, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x, scale=S512)
        offsets, ids, dists = m.knn2_pairs(pairs, exact_f32=True)
        assert m._test_last_knn_stats()[1] == 0
    expect = {}
    for p, (r, q) in enumerate(pairs.tolist()):
        if (r, q) not in expect:
            expect[(r, q)] = oracle_mod.knn2_f32(imgs[r], imgs[q])
        gi, gd = _slices(offsets, ids, dists, p)
        np.testing.assert_array_equal(gi, expect[(r, q)][0])
        np.testing.assert_array_equal(gd, expect[(r, q)][1])


# ---------------------------------------------------------------------------------------------------- GPU: errors
@pytest.mark.gpu
def test_errors_are_reported_before_any_launch(oracle_mod, native_lib):
    from metricsfm_b200 import _lib
    from metricsfm_b200.matcher import MsfmError
    col = synth.Collection(300, seed=2)
    f0, f1 = col.image_unit(0), col.image_unit(1)
    u8 = col.image_u8(2)
    with _matcher(max_images=8, arena_rows=1 << 14, keep_float=True) as m:
        m.upload(0, f0, scale=S512)
        m.upload(1, f1, scale=S512)
        m.upload(2, u8)
        m.upload(3, f1 * np.float32(512.0), scale=1.0)
        L, h = m._L, m._h
        pa = np.array([[0, 1]], np.int32)
        offs = np.zeros(2, np.int64)
        ids = np.zeros((300, 2), np.int32)
        dists = np.zeros((300, 2), np.float32)

        def call(pairs=pa, n=1, flags=0, o=offs, i=ids, d=dists, cap=300):
            ptr = lambda a: a.ctypes.data if a is not None else None
            return L.msfm_knn2_pairs(h, ptr(pairs), n, flags, ptr(o), ptr(i), ptr(d), cap)

        def still_works():
            o, i, d = m.knn2_pairs([(0, 1)], exact_f32=True)
            oi, od = oracle_mod.knn2_f32(f0, f1)
            np.testing.assert_array_equal(i, oi)
            np.testing.assert_array_equal(d, od)

        INVALID, CAPACITY, NOT_FOUND = 1, 5, 4
        for kw in (dict(pairs=None), dict(o=None), dict(i=None), dict(d=None), dict(n=-1), dict(cap=-1)):
            assert call(**kw) == INVALID, kw
            still_works()
        assert call(flags=2) == INVALID
        assert b"flag" in L.msfm_last_error(h)
        still_works()
        assert call(cap=299) == CAPACITY
        still_works()
        assert call(pairs=np.array([[0, 7]], np.int32)) == NOT_FOUND
        still_works()
        assert call(pairs=np.array([[0, 99]], np.int32)) == INVALID
        still_works()
        two = np.array([[0, 1], [0, 2]], np.int32)
        assert call(pairs=two, n=2, flags=_lib.KNN_EXACT_F32, cap=600,
                    i=np.zeros((600, 2), np.int32), d=np.zeros((600, 2), np.float32)) == INVALID
        assert b"pair 1" in L.msfm_last_error(h)
        still_works()
        with pytest.raises(MsfmError, match="pair 0"):
            m.knn2_pairs([(3, 1)], exact_f32=True)  # scale 1 against scale 512
        still_works()
        assert call(pairs=two, n=2, cap=600, i=np.zeros((600, 2), np.int32), d=np.zeros((600, 2), np.float32)) == 0
    with _matcher(max_images=4, arena_rows=1 << 12) as m:  # no retained float rows at all
        m.upload(0, f0, scale=S512)
        with pytest.raises(MsfmError, match="keep_float"):
            m.knn2_pairs([(0, 0)], exact_f32=True)
        o, i, d = m.knn2_pairs([(0, 0)])
        np.testing.assert_array_equal(i, m.knn2(0, 0)[0])
