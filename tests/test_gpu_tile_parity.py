"""Match lists on images whose reference-tile count is odd and even, per work item and across the items of one batch.

The matching kernel's accumulator buffers alternate over the CTA's running tile sequence (match_kernel.cuh: every ring
position derives from one per-CTA tile counter, not from the tile index in the item), so the buffer and barrier phase
that start an item depend on the tile counts of every earlier item of the CTA.  Images of one, two and many 64-row
reference tiles, ragged and whole, all mixed in one batch: match lists and 'good' flags must equal the oracle's, with
the dead-row rule on and off, and the exact 2-NN of a few pairs must equal the oracle's."""
import numpy as np
import pytest

from metricsfm_b200 import synth

pytestmark = pytest.mark.gpu

ROWS = (1, 37, 64, 65, 128, 129, 200, 255, 256, 300, 385, 700)


def _images():
    col = synth.Collection(1024, seed=31)
    rng = np.random.default_rng(99)
    imgs = [col.image_u8(i, r) for i, r in enumerate(ROWS)]
    # exact duplicates in distant tiles (equal scores: lowest index wins) and near-copies of another image's rows
    big = imgs[-1]
    big[600:640] = big[:40]
    small = imgs[6]
    small[:20] = np.clip(big[130:150].astype(np.int32) + rng.integers(-1, 2, size=(20, 128)), 0, 255).astype(np.uint8)
    return [np.ascontiguousarray(x) for x in imgs]


@pytest.mark.parametrize("ratio,ratio_good", [(0.85, 0.6), (0.6, 0.0)])
def test_odd_and_even_tile_counts_in_one_batch(oracle_mod, native_lib, ratio, ratio_good):
    from metricsfm_b200.matcher import Matcher
    imgs = _images()
    n = len(imgs)
    pairs = [(r, q) for r in range(n) for q in range(n) if r != q]
    with Matcher(device=0, max_images=16, arena_rows=1 << 15) as m:
        for i, x in enumerate(imgs):
            m.upload(i, x)
        out = {}
        for prune in (True, False):
            m._test_disable_pruning(not prune)
            for mutual in (False, True):
                out[prune, mutual] = m.match_pairs(pairs, ratio, ratio_good=ratio_good, mutual=mutual)
        m._test_disable_pruning(False)
        knn = {(r, q): m.knn2(r, q) for (r, q) in [(0, 11), (4, 10), (5, 6), (7, 9), (11, 4), (9, 8)]}
    for (r, q), (ids, dists) in knn.items():
        oids, odists = oracle_mod.knn2_u8(imgs[r], imgs[q])
        np.testing.assert_array_equal(ids, oids, err_msg=f"knn2 ({r},{q})")
        np.testing.assert_array_equal(dists, odists, err_msg=f"knn2 ({r},{q})")
    total = 0
    for mutual in (False, True):
        for p, (r, q) in enumerate(pairs):
            exp = oracle_mod.match_pair_u8(imgs[r], imgs[q], ratio, mutual=mutual, ratio_good=ratio_good)
            for prune in (True, False):
                np.testing.assert_array_equal(out[prune, mutual].pair(p), exp["pairs"],
                                              err_msg=f"prune={prune} mutual={mutual} pair ({r},{q})")
                if ratio_good > 0:
                    np.testing.assert_array_equal(out[prune, mutual].pair_good(p), exp["good"],
                                                  err_msg=f"good flags, prune={prune} mutual={mutual} pair ({r},{q})")
            total += len(exp["pairs"])
    assert total > 100
