"""Float regime of msfm_match_pairs (msfm_params.rescore_band on a keep_float context), row by row.

`expected_float_lists` restates the rule of include/msfm_match.h in numpy on top of the CPU oracle: a query row whose
quantised ratio d0/d1 lies within ratio*(1 +- band) (or the same band of ratio_good) is decided on the exact fp32 top-2
of the caller's float rows; every other row keeps the integer decision of MATCH-SPEC.  All arithmetic the kernels do in
fp32 is done in np.float32 here.  The CPU tests check the restatement against the quantised oracle where the two must
agree, and on hand-built band rows whose fp32 top-2 lies outside the heuristic re-scoring threshold the float regime
used before it took the proven bound T(q).  The GPU tests compare msfm_match_pairs with it bit for bit (matches, good,
ok) across ratios, rules, gates, orientations, scales, bands, ragged and degenerate images, multi-batch pair lists,
pairs that must take the integer path, and the adversarial rows, each through the collect path and the forced
brute force."""
import numpy as np
import pytest

from metricsfm_b200 import synth
from test_knn_pairs import _exact_threshold, _heuristic_threshold, _quantised_d2, _residuals

f32 = np.float32
S512 = 512.0
REJECT_GT = 1  # MSFM_RATIO_REJECT_GT

DEFAULTS = dict(ratio=0.85, ratio_good=0.0, max_dist_sq=0.0, min_keypoints=20, orientation=0, rescore_band=0.0, flags=0)


# ---------------------------------------------------------------------------------------------------- the restatement
class _Knn:
    """Integer and fp32 2-NN of a pair, computed once (the restatement is evaluated under many parameter sets)."""

    def __init__(self, oracle_mod, imgs, kinds, scales):
        self.o, self.imgs, self.kinds, self.scales = oracle_mod, imgs, kinds, scales
        self._q, self._u8, self._f32 = {}, {}, {}

    def rows_q(self, i):
        if i not in self._q:
            x = self.imgs[i]
            self._q[i] = x if self.kinds[i] == "u8" else self.o.quantize_f32(x, self.scales[i])
        return self._q[i]

    def u8(self, r, q):
        if (r, q) not in self._u8:
            self._u8[(r, q)] = self.o.knn2_u8(self.rows_q(r), self.rows_q(q))
        return self._u8[(r, q)]

    def f32(self, r, q):
        if (r, q) not in self._f32:
            self._f32[(r, q)] = self.o.knn2_f32(self.imgs[r], self.imgs[q])
        return self._f32[(r, q)]


def _accepts(r, th, reject_gt):
    return ~(r > f32(th)) if reject_gt else (r < f32(th))


def _decide_pair(knn, r, q, p, keep_float):
    """Per query row of pair (r, q): (keep, good, reference row, band) under the header's rule."""
    reject_gt = bool(p["flags"] & REJECT_GT)
    ids, d = knn.u8(r, q)
    j0, d0, d1 = ids[:, 0], d[:, 0], d[:, 1]
    both = (ids[:, 0] >= 0) & (ids[:, 1] >= 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio_q = d0 / d1  # fp32 divide; 0/0 = NaN
    # integer rule (MATCH-SPEC): (float)d0 / (float)d1, strict or REJECT_GT, (float)d0 < max_dist_sq
    keep = both & _accepts(ratio_q, p["ratio"], reject_gt)
    if p["max_dist_sq"] > 0:
        keep &= d0 < f32(p["max_dist_sq"])
    good = keep & (p["ratio_good"] > 0) & _accepts(ratio_q, p["ratio_good"], reject_gt)
    j = j0.copy()
    band = np.zeros_like(both)
    float_pair = (keep_float and knn.kinds[r] == knn.kinds[q] == "f32" and knn.scales[r] == knn.scales[q]
                  and p["rescore_band"] > 0)
    if float_pair:
        bw = f32(p["rescore_band"])
        with np.errstate(invalid="ignore"):
            band = both & (np.abs(ratio_q - f32(p["ratio"])) <= bw * f32(p["ratio"]))
            if p["ratio_good"] > 0:
                band |= both & (np.abs(ratio_q - f32(p["ratio_good"])) <= bw * f32(p["ratio_good"]))
        if band.any():
            fids, fd = knn.f32(r, q)
            c0, b0, b1 = fids[:, 0], fd[:, 0], fd[:, 1]
            with np.errstate(divide="ignore", invalid="ignore"):
                fr = b0 / b1
            fscale2 = f32(knn.scales[r]) * f32(knn.scales[r])
            kb = (fids[:, 0] >= 0) & (fids[:, 1] >= 0) & _accepts(fr, p["ratio"], reject_gt)
            if p["max_dist_sq"] > 0:
                kb &= (b0 * fscale2) < f32(p["max_dist_sq"])
            gb = kb & (p["ratio_good"] > 0) & _accepts(fr, p["ratio_good"], reject_gt)
            keep = np.where(band, kb, keep)
            good = np.where(band, gb, good)
            j = np.where(band, c0, j)
    return keep, good, j, band


def expected_float_lists(imgs, kinds, scales, pairs, params, *, keep_float=True, knn=None, oracle_mod=None):
    """(ok, matches [n, 2] int32, good [n] uint8) per pair, as the header's rule decides them.
    imgs[i]: float32 rows (kinds[i] == "f32", uploaded with msfm_upload_f32 at scales[i]) or uint8 rows ("u8");
    keep_float: the context retains float rows.  knn: a _Knn over the same images, to share the 2-NN between calls."""
    p = {**DEFAULTS, **params}
    knn = knn or _Knn(oracle_mod, imgs, kinds, scales)
    out = []
    for r, q in pairs:
        r, q = int(r), int(q)
        if len(imgs[r]) < p["min_keypoints"] or len(imgs[q]) < p["min_keypoints"]:
            out.append((0, np.empty((0, 2), np.int32), np.empty((0,), np.uint8)))
            continue
        if len(imgs[r]) == 0 or len(imgs[q]) == 0:
            out.append((1, np.empty((0, 2), np.int32), np.empty((0,), np.uint8)))
            continue
        keep, good, j, _ = _decide_pair(knn, r, q, p, keep_float)
        qi = np.nonzero(keep)[0].astype(np.int32)
        cols = (j[qi], qi) if p["orientation"] == 0 else (qi, j[qi])
        out.append((1, np.stack(cols, axis=1).astype(np.int32).reshape(-1, 2), good[qi].astype(np.uint8)))
    return out


# ---------------------------------------------------------------------------------------------------- adversarial rows
def _unit(v):
    return np.asarray(v, np.float32) / f32(512.0)


def _adversarial(case):
    """(reference rows, query row), float32, scale 512, for one hand-built band row.
    wrong_ref (i) / spurious (ii): query x = 0.499/512 everywhere, B = 2.501/512 everywhere, A and C = x with element
      0 / 1 raised; the quantised top-2 is {A, C} and in the band, B is in the fp32 top-2 but beyond the heuristic
      threshold d1 + d1/32 + 256.  (i) fp32 accepts (B, q) where {A, C} gives (A, q); (ii) fp32 rejects.
    tie: two reference rows at exactly the same fp32 distance (the same difference in elements 0 and 1); quantised,
      the second one is nearer.  Lowest index wins in fp32: visible under REJECT_GT with ratio 1.0.
    zero: the two nearest reference rows quantise to the query's own row (d0q = d1q = 0, NaN ratio): never a band row,
      so the integer decision stands (strict rejects, REJECT_GT accepts the lower row) although fp32 has ratio 0.25."""
    if case in ("wrong_ref", "spurious"):
        ra, rc = (25.6, 27.9) if case == "wrong_ref" else (22.4, 24.6)
        x = np.full(128, 0.499, np.float32) / f32(512.0)
        b = np.full(128, 2.501, np.float32) / f32(512.0)
        a, c = x.copy(), x.copy()
        a[0] += f32(ra / 512.0)
        c[1] += f32(rc / 512.0)
        return np.stack([a, b, c]), x
    if case == "tie":
        x = np.zeros(128, np.float32)
        x[0], x[1] = 10.25, 10.75
        y1, y2 = x.copy(), x.copy()
        y1[0], y2[1] = 110.75, 111.25  # both differences are 100.5, exactly
        return _unit(np.stack([y1, y2])), _unit(x)
    if case == "zero":
        x, y1, y2 = np.zeros(128, np.float32), np.zeros(128, np.float32), np.zeros(128, np.float32)
        x[0], y1[0], y2[0] = 0.3, 0.1, 0.2
        return _unit(np.stack([y1, y2])), _unit(x)
    raise ValueError(case)


ADV_CASES = ["wrong_ref", "spurious", "tie", "zero"]


def _fp32_matcher(oracle_mod, ref, qry, ratio, reject_gt=False):
    ids, dists = oracle_mod.knn2_f32(ref, qry)
    return oracle_mod.ratio_select(ids, dists, ref.shape[0], ratio, min_keypoints=0, reject_gt=reject_gt)[0]


# ---------------------------------------------------------------------------------------------------- CPU tests
def test_integer_valued_float_rows_at_scale_1_equal_the_integer_oracle(oracle_mod):
    """Integer-valued float rows at scale 1: fp32 distances are the integer ones, so band rows decide as the integer
    rule does and the restatement is exactly the u8 oracle."""
    col = synth.Collection(600, seed=31)
    imgs = [col.image_f32_512(i) for i in range(3)]
    pairs = [(0, 1), (1, 2), (2, 0)]
    knn = _Knn(oracle_mod, imgs, ["f32"] * 3, [1.0] * 3)
    sets = [dict(ratio=0.85, ratio_good=0.6, rescore_band=0.03), dict(ratio=0.7, rescore_band=0.2, orientation=1),
            dict(ratio=0.8, flags=REJECT_GT, rescore_band=0.1), dict(ratio=0.85, max_dist_sq=60000.0, rescore_band=0.2)]
    for prm in sets:
        exp = expected_float_lists(imgs, knn.kinds, knn.scales, pairs, prm, knn=knn)
        p = {**DEFAULTS, **prm}
        n_band = sum(_decide_pair(knn, r, q, p, True)[3].sum() for r, q in pairs)
        assert n_band > 0, prm
        for (r, q), (ok, m, g) in zip(pairs, exp):
            o = oracle_mod.match_pair_u8(imgs[r].astype(np.uint8), imgs[q].astype(np.uint8), p["ratio"],
                                         ratio_good=p["ratio_good"], max_dist_sq=p["max_dist_sq"],
                                         orientation=p["orientation"], reject_gt=bool(p["flags"] & REJECT_GT))
            assert ok == 1 and o["ok"]
            np.testing.assert_array_equal(m, o["pairs"], err_msg=str(prm))
            np.testing.assert_array_equal(g, o["good"], err_msg=str(prm))


def test_band_zero_and_integer_path_pairs_equal_the_quantised_oracle(oracle_mod):
    """band 0, a u8 image paired with a float image, two scales, and a context without retained rows all follow the
    integer rule on the quantised rows; the same float pair with a band does not (the band decides some rows)."""
    col = synth.Collection(700, seed=32)
    imgs = [col.image_unit(0), col.image_unit(1), col.image_u8(2), col.image_unit(3) * f32(512.0)]
    kinds, scales = ["f32", "f32", "u8", "f32"], [S512, S512, 1.0, 1.0]
    knn = _Knn(oracle_mod, imgs, kinds, scales)
    prm = dict(ratio=0.85, ratio_good=0.6)

    def quantised(r, q):
        o = oracle_mod.match_pair_u8(knn.rows_q(r), knn.rows_q(q), 0.85, ratio_good=0.6)
        return o["pairs"], o["good"]

    cases = [([(0, 1), (1, 0)], 0.0, True), ([(0, 2), (2, 1)], 0.2, True), ([(0, 3), (3, 1)], 0.2, True),
             ([(0, 1), (1, 0)], 0.2, False)]
    for pairs, band, keep_float in cases:
        exp = expected_float_lists(imgs, kinds, scales, pairs, {**prm, "rescore_band": band}, keep_float=keep_float, knn=knn)
        for (r, q), (ok, m, g) in zip(pairs, exp):
            qm, qg = quantised(r, q)
            np.testing.assert_array_equal(m, qm, err_msg=f"{(r, q)} band {band} keep_float {keep_float}")
            np.testing.assert_array_equal(g, qg)
    exp = expected_float_lists(imgs, kinds, scales, [(0, 1)], {**prm, "rescore_band": 0.2}, knn=knn)
    assert not np.array_equal(exp[0][1], quantised(0, 1)[0])


@pytest.mark.parametrize("case", ["wrong_ref", "spurious"])
def test_adversarial_band_rows_need_the_bound(oracle_mod, case):
    """Rows (i) and (ii): quantised distances and ratio as built, B outside the heuristic threshold and inside T(q),
    and the restatement decides as the fp32 matcher while the heuristic candidate set {A, C} would not."""
    ref, x = _adversarial(case)
    qry = x[None, :]
    qr, qq = oracle_mod.quantize_f32(ref, S512), oracle_mod.quantize_f32(qry, S512)
    dq = _quantised_d2(qq, qr)[0]
    want_dq = [676.0, 1152.0, 784.0] if case == "wrong_ref" else [529.0, 1152.0, 625.0]
    np.testing.assert_array_equal(dq, want_dq)
    ratio_q = f32(dq[0]) / f32(dq[2])
    assert abs(ratio_q - f32(0.85)) <= f32(0.03) * f32(0.85)  # a band row at band 0.03
    d1q = dq[2]
    assert dq[1] > _heuristic_threshold(d1q)  # B is not a candidate under the heuristic
    T = _exact_threshold(d1q, _residuals(qry, S512)[0], _residuals(ref, S512).max())
    assert dq[1] <= T  # ... and is one under the bound
    fids, _ = oracle_mod.knn2_f32(ref, qry)
    fp32 = _fp32_matcher(oracle_mod, ref, qry, 0.85)
    exp = expected_float_lists([ref, qry], ["f32", "f32"], [S512, S512], [(0, 1)],
                               dict(ratio=0.85, rescore_band=0.03, min_keypoints=0), oracle_mod=oracle_mod)
    np.testing.assert_array_equal(exp[0][1], fp32)
    # what deciding on the heuristic candidates {A, C} gives instead
    heur = np.float32(((ref[[0, 2]] - qry) ** 2).sum(1))  # A, C
    heur_keep = heur[0] / heur[1] < f32(0.85)
    if case == "wrong_ref":
        assert fids[0, 0] == 1 and fp32.tolist() == [[1, 0]] and heur_keep  # fp32 emits (B, q); {A, C} emits (A, q)
    else:
        assert fp32.shape[0] == 0 and heur_keep  # fp32 rejects; {A, C} keeps (A, q)


def test_tie_and_zero_rows_restated(oracle_mod):
    """The tie row: the fp32 top-2 tie goes to the lower reference row, while the quantised nn0 is the higher one.
    The zero row (d0q = d1q = 0): not a band row, so strict rejects and REJECT_GT accepts the quantised nn0."""
    ref, x = _adversarial("tie")
    qry = x[None, :]
    dq = _quantised_d2(oracle_mod.quantize_f32(qry, S512), oracle_mod.quantize_f32(ref, S512))[0]
    np.testing.assert_array_equal(dq, [10201.0, 10000.0])
    fids, fd = oracle_mod.knn2_f32(ref, qry)
    assert fids[0].tolist() == [0, 1] and fd[0, 0] == fd[0, 1]
    prm = dict(ratio=1.0, flags=REJECT_GT, rescore_band=0.03, min_keypoints=0)
    exp = expected_float_lists([ref, qry], ["f32", "f32"], [S512, S512], [(0, 1)], prm, oracle_mod=oracle_mod)
    assert exp[0][1].tolist() == [[0, 0]]
    integer = expected_float_lists([ref, qry], ["f32", "f32"], [S512, S512], [(0, 1)], {**prm, "rescore_band": 0.0},
                                   oracle_mod=oracle_mod)
    assert integer[0][1].tolist() == [[1, 0]]

    ref, x = _adversarial("zero")
    qry = x[None, :]
    args = ([ref, qry], ["f32", "f32"], [S512, S512], [(0, 1)])
    strict = expected_float_lists(*args, dict(ratio=0.85, rescore_band=0.2, min_keypoints=0), oracle_mod=oracle_mod)
    gt = expected_float_lists(*args, dict(ratio=0.85, rescore_band=0.2, min_keypoints=0, flags=REJECT_GT),
                              oracle_mod=oracle_mod)
    assert strict[0][1].shape[0] == 0 and gt[0][1].tolist() == [[0, 0]]
    assert _fp32_matcher(oracle_mod, ref, qry, 0.85).tolist() == [[1, 0]]  # what an fp32 matcher would say


# ---------------------------------------------------------------------------------------------------- GPU helpers
def _matcher(**kw):
    from metricsfm_b200.matcher import Matcher
    return Matcher(device=0, **kw)


def _run(m, pairs, prm):
    p = {**DEFAULTS, **prm}
    return m.match_pairs(pairs, p["ratio"], ratio_good=p["ratio_good"], max_dist_sq=p["max_dist_sq"],
                         min_keypoints=p["min_keypoints"], orientation=p["orientation"], rescore_band=p["rescore_band"],
                         flags=p["flags"])


def _assert_equal(res, exp, pairs, prm, tag=""):
    p = {**DEFAULTS, **prm}
    assert res.ok.tolist() == [e[0] for e in exp], f"{tag} {prm}: ok"
    for k, ((r, q), (ok, m, g)) in enumerate(zip(pairs, exp)):
        msg = f"{tag} {prm}: pair {k} ({r}, {q})"
        got = res.pair(k)
        if not np.array_equal(got, m):
            a, b = {tuple(v) for v in got.tolist()}, {tuple(v) for v in m.tolist()}
            raise AssertionError(f"{msg}: {len(got)} matches, expected {len(m)}; only on the GPU {sorted(a - b)[:8]}, "
                                 f"only in the restatement {sorted(b - a)[:8]}")
        if p["ratio_good"] > 0:
            np.testing.assert_array_equal(res.pair_good(k), g, err_msg=msg + ": good")


CAPS = [-1, 0, 37]  # default sizing, brute force forced, a list that overflows on any real batch


def _check_caps(m, pairs, prm, exp, tag, stats=True):
    """The call with the default event list, with none (brute force) and with a tiny one: all equal the restatement.
    stats: with the default list the collect path decided every batch; with none the brute force decided."""
    for cap in CAPS:
        m._test_set_band_event_cap(cap)
        res = _run(m, pairs, prm)
        _assert_equal(res, exp, pairs, prm, f"{tag} cap {cap}")
        events, brute = m._test_last_knn_stats()
        if stats and cap == -1:
            assert brute == 0 and events > 0, (tag, prm, events, brute)
        if stats and cap == 0:
            assert brute >= 1, (tag, prm, events, brute)
    m._test_set_band_event_cap(-1)


# ---------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
def test_adversarial_band_rows_equal_the_restatement(oracle_mod, native_lib):
    """Rows (i), (ii), the fp32 tie and the zero row embedded at several positions of 4096-row unit-norm images (query
    rows repeated at the start, inside and at the end; reference rows at two placements per case), under the strict
    rule, REJECT_GT, and REJECT_GT at ratio 1.0 (where the tie's winner is emitted); default, zero and tiny event lists."""
    rows = 4096
    col = synth.Collection(rows, seed=41)
    placements = [[3, 2047, 4095], [4000, 17, 1500]]
    qpos = [0, 1234, 4095]
    imgs, pairs, where = [], [], []
    for ci, case in enumerate(ADV_CASES):
        adv_ref, x = _adversarial(case)
        for pi, pos in enumerate(placements):
            ref = col.image_unit(100 + 10 * ci + 2 * pi).copy()
            qry = col.image_unit(101 + 10 * ci + 2 * pi).copy()
            ref[pos[:len(adv_ref)]] = adv_ref
            qry[qpos] = x
            imgs += [ref, qry]
            pairs.append((len(imgs) - 2, len(imgs) - 1))
            where.append((case, pos[:len(adv_ref)]))
    kinds, scales = ["f32"] * len(imgs), [S512] * len(imgs)
    knn = _Knn(oracle_mod, imgs, kinds, scales)
    sets = [dict(ratio=0.85, ratio_good=0.6, rescore_band=0.03), dict(ratio=0.85, flags=REJECT_GT, rescore_band=0.03),
            dict(ratio=1.0, flags=REJECT_GT, rescore_band=0.03)]
    # the restatement says what the issue's table says at every embedded query row
    exp0 = expected_float_lists(imgs, kinds, scales, pairs, sets[0], knn=knn)
    exp_gt1 = expected_float_lists(imgs, kinds, scales, pairs, sets[2], knn=knn)
    for k, (case, pos) in enumerate(where):
        got = {int(qq): int(j) for j, qq in exp0[k][1].tolist()}
        if case == "wrong_ref":
            assert all(got.get(qq) == pos[1] for qq in qpos)  # B
        if case in ("spurious", "zero"):
            assert all(qq not in got for qq in qpos)
        if case == "tie":
            got1 = {int(qq): int(j) for j, qq in exp_gt1[k][1].tolist()}
            assert all(got1.get(qq) == min(pos) for qq in qpos)
    with _matcher(max_images=len(imgs), arena_rows=1 << 17, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x, scale=S512)
        for si, prm in enumerate(sets):
            exp = exp0 if si == 0 else (exp_gt1 if si == 2 else expected_float_lists(imgs, kinds, scales, pairs, prm, knn=knn))
            # ratio 1.0 makes most rows of unrelated images band rows: that list overflows by design
            _check_caps(m, pairs, prm, exp, "adversarial", stats=si < 2)


def _sweep_sets(d0_med):
    return [dict(ratio=0.85, ratio_good=0.6, rescore_band=0.02),
            dict(ratio=0.85, ratio_good=0.6, rescore_band=0.03),
            dict(ratio=0.85, ratio_good=0.6, rescore_band=0.2),
            dict(ratio=0.5, rescore_band=0.03),
            dict(ratio=0.8, flags=REJECT_GT, rescore_band=0.03),
            dict(ratio=0.85, ratio_good=0.6, rescore_band=0.03, max_dist_sq=d0_med),
            dict(ratio=0.85, ratio_good=0.6, rescore_band=0.03, orientation=1),
            dict(ratio=0.8, flags=REJECT_GT, rescore_band=0.2, max_dist_sq=d0_med, orientation=1)]


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["unit_512", "vlsift_1"])
def test_rule_sweep_equals_the_restatement(oracle_mod, native_lib, regime):
    """4096-row unit-norm rows at scale 512, or the same rows x 512 at scale 1 (VLSIFT): ratio 0.85 with ratio_good
    0.6, ratio 0.5 alone, REJECT_GT at 0.8, a max_dist_sq at the median d0 of the accepted rows (it drops band rows
    and integer rows), orientation 0 and 1, bands 0.02, 0.03 and 0.2.  Band 0.02 and the REJECT_GT and max_dist_sq sets
    also run with zero and tiny event lists; bands up to 0.03 never overflow the default list."""
    scale = S512 if regime == "unit_512" else 1.0
    col = synth.Collection(4096, seed=43)
    imgs = [col.image_unit(i) * f32(S512 / scale) for i in range(4)]  # x 1.0 at scale 512: the same rows
    pairs = [(0, 1), (2, 3), (1, 2), (3, 0)]
    kinds, scales = ["f32"] * 4, [scale] * 4
    knn = _Knn(oracle_mod, imgs, kinds, scales)
    p0 = {**DEFAULTS, **dict(ratio=0.85, ratio_good=0.6, rescore_band=0.03)}
    kept_d0 = np.concatenate([knn.u8(r, q)[1][_decide_pair(knn, r, q, p0, True)[0], 0] for r, q in pairs])
    d0_med = float(np.median(kept_d0))
    sets = _sweep_sets(d0_med)
    # the gate bites on band rows and on integer rows alike
    gated = {**p0, "max_dist_sq": d0_med}
    for r, q in pairs[:1]:
        k0, _, _, band = _decide_pair(knn, r, q, p0, True)
        k1, _, _, _ = _decide_pair(knn, r, q, gated, True)
        assert (k0 & ~k1 & band).any() and (k0 & ~k1 & ~band).any()
    with _matcher(max_images=8, arena_rows=1 << 16, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, np.ascontiguousarray(x), scale=scale)
        for si, prm in enumerate(sets):
            exp = expected_float_lists(imgs, kinds, scales, pairs, prm, knn=knn)
            if si == 0 or prm.get("flags") or prm.get("max_dist_sq"):
                # the collect path and the brute force each apply REJECT_GT and max_dist_sq; band 0.2 may overflow
                _check_caps(m, pairs, prm, exp, regime, stats=prm["rescore_band"] <= 0.03)
            else:
                _assert_equal(_run(m, pairs, prm), exp, pairs, prm, regime)


@pytest.mark.gpu
def test_ragged_degenerate_and_repeated_pairs(oracle_mod, native_lib):
    """Images of 0, 1, 19, 20, 21, 2049 and 4096 rows; the pair (i, i), repeated pairs, gated pairs (min_keypoints 20)
    and, with min_keypoints 0, pairs with an empty or one-row side."""
    col = synth.Collection(4096, seed=47)
    sizes = [0, 1, 19, 20, 21, 2049, 4096]
    imgs = [col.image_unit(i, rows=max(n, 1))[:n] for i, n in enumerate(sizes)]
    pairs = [(5, 6), (6, 5), (6, 6), (5, 5), (3, 4), (4, 3), (2, 6), (6, 2), (0, 6), (6, 0), (1, 6), (6, 1), (5, 6), (4, 4),
             (0, 0), (1, 1), (3, 5), (6, 3)]
    kinds, scales = ["f32"] * len(imgs), [S512] * len(imgs)
    knn = _Knn(oracle_mod, imgs, kinds, scales)
    with _matcher(max_images=8, arena_rows=1 << 15, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, np.ascontiguousarray(x), scale=S512)
        for prm in (dict(ratio=0.85, ratio_good=0.6, rescore_band=0.03),
                    dict(ratio=0.85, ratio_good=0.6, rescore_band=0.2, min_keypoints=0, orientation=1),
                    dict(ratio=0.8, flags=REJECT_GT, rescore_band=0.03, min_keypoints=0)):
            exp = expected_float_lists(imgs, kinds, scales, pairs, prm, knn=knn)
            _check_caps(m, pairs, prm, exp, "ragged", stats=False)


@pytest.mark.gpu
def test_pair_list_spans_several_batches(oracle_mod, native_lib):
    """More pairs than one batch holds (16 384): 17 000 pairs of 64-row float images, drawn with repetition."""
    rng = np.random.default_rng(17)
    n_img = 24
    col = synth.Collection(64, seed=53)
    imgs = [col.image_unit(i) for i in range(n_img)]
    pairs = rng.integers(0, n_img, size=(17000, 2)).astype(np.int32)
    kinds, scales = ["f32"] * n_img, [S512] * n_img
    knn = _Knn(oracle_mod, imgs, kinds, scales)
    prm = dict(ratio=0.85, ratio_good=0.6, rescore_band=0.2)
    exp = expected_float_lists(imgs, kinds, scales, pairs.tolist(), prm, knn=knn)
    with _matcher(max_images=32, arena_rows=1 << 15, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x, scale=S512)
        _assert_equal(_run(m, pairs, prm), exp, pairs.tolist(), prm, "batches")


@pytest.mark.gpu
def test_pairs_that_take_the_integer_path(oracle_mod, native_lib):
    """A u8 image paired with a float image, a scale-512 image paired with a scale-1 image, and float images on a
    context without retained rows: the integer rule, although the band (0.2) would re-score many rows of a float pair."""
    col = synth.Collection(4096, seed=59)
    imgs = [col.image_unit(0), col.image_unit(1), col.image_u8(2), col.image_unit(3) * f32(512.0)]
    kinds, scales = ["f32", "f32", "u8", "f32"], [S512, S512, 1.0, 1.0]
    knn = _Knn(oracle_mod, imgs, kinds, scales)
    pairs = [(0, 2), (2, 1), (0, 3), (3, 1), (0, 1)]
    prm = dict(ratio=0.85, ratio_good=0.6, rescore_band=0.2)
    for keep_float in (True, False):
        exp = expected_float_lists(imgs, kinds, scales, pairs, prm, keep_float=keep_float, knn=knn)
        with _matcher(max_images=8, arena_rows=1 << 15, keep_float=keep_float) as m:
            for i, x in enumerate(imgs):
                m.upload(i, x, scale=scales[i])
            _assert_equal(_run(m, pairs, prm), exp, pairs, prm, f"keep_float {keep_float}")
    # the float pair (0, 1) is the control: on a keep_float context the band changes its list
    q = oracle_mod.match_pair_u8(knn.rows_q(0), knn.rows_q(1), 0.85, ratio_good=0.6)["pairs"]
    assert not np.array_equal(expected_float_lists(imgs, kinds, scales, [(0, 1)], prm, knn=knn)[0][1], q)


@pytest.mark.gpu
def test_mutual_matches_are_one_way_matches(native_lib):
    """The float regime's mutual check is a filter of the one-way list: every mutual match is a one-way match with
    the same good flag (the check itself is not claimed exact in fp32)."""
    col = synth.Collection(4096, seed=61)
    imgs = [col.image_unit(i) for i in range(4)]
    pairs = [(0, 1), (2, 3), (1, 2)]
    with _matcher(max_images=8, arena_rows=1 << 15, keep_float=True) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x, scale=S512)
        for band in (0.02, 0.2):
            one = m.match_pairs(pairs, 0.85, ratio_good=0.6, rescore_band=band)
            mut = m.match_pairs(pairs, 0.85, ratio_good=0.6, rescore_band=band, mutual=True)
            for k in range(len(pairs)):
                ow = {tuple(v): g for v, g in zip(one.pair(k).tolist(), one.pair_good(k).tolist())}
                assert mut.pair(k).shape[0] > 0
                for v, g in zip(mut.pair(k).tolist(), mut.pair_good(k).tolist()):
                    assert ow.get(tuple(v)) == g, (band, k, v)
