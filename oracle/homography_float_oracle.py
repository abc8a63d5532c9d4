"""TEST INFRASTRUCTURE ONLY — the float regime of msfm_match_pairs_guided_homography (HOMOG-SPEC with rescore_band > 0
in include/msfm_match.h), stated as oracle.guided_float_oracle's restatement with the HOMOG-SPEC gate of
oracle.homography_oracle in place of the epipolar one; and the float variant of the planar scene with look-alikes on
the epipolar line that the tests and tools/guided_homography_float_bench.py match on."""
from __future__ import annotations

import numpy as np

from metricsfm_b200 import synth
from oracle import guided_float_oracle as gfo
from oracle import homography_oracle as ho


def match_pair_guided_h_float(ref, query, xy_ref, xy_qry, H, th: float, ratio: float, **kw):
    """One pair of msfm_match_pairs_guided_homography with mutual = 0: guided_float_oracle.match_pair_guided_float with
    allowed = gate_h32(H, xy_ref, xy_qry, th).  Returns its dict(ok, pairs, good, band, allowed, ids, dists)."""
    return gfo.match_pair_guided_float(ref, query, xy_ref, xy_qry, None, th, ratio,
                                       allowed=ho.gate_h32(H, xy_ref, xy_qry, th), **kw)


def float_planar_decoy_scene(seed, M, N, *, decoy_frac=0.5, sigma=6.0, noise=0.5, dups=True, companions=True,
                             companion_sigma=None):
    """homography_oracle.planar_decoy_scene with unit-norm float32 rows (float noise, not quantised), to be uploaded at
    scale 512: k true correspondences related by the plane's H, a fraction with a planted look-alike on the epipolar
    line 40-300 px off, a companion row at every true reference keypoint (companions = False: at random positions),
    unrelated rows, and (dups) exact and descriptor-only duplicates.  companion_sigma: each companion descriptor is a
    noisy copy of its true reference descriptor with that noise (a second SIFT orientation at the same location), so
    that a true match's disc ratio d(true) / d(companion) spreads around the ratio thresholds; None: an unrelated
    descriptor, whose disc ratios sit far below every threshold.  Returns dict(ref, qry, xy_ref, xy_qry, H, F, true,
    decoyed)."""
    rng = np.random.default_rng(seed)
    project, H, F = ho.plane_views(rng)
    k = min(M // 3, N)
    nd = int(round(k * decoy_frac))
    m_rest, n_rest = M - 2 * k - nd, N - k
    G = np.c_[rng.uniform(-55, 55, (k, 1)), rng.uniform(-55, 55, (k, 1)), np.zeros((k, 1))]
    p1, p2 = project(G, 0), project(G, 1)
    p1n = p1 + rng.normal(0, noise, p1.shape)
    p2n = p2 + rng.normal(0, noise, p2.shape)
    col = synth.Collection(max(M, N, 1), seed=seed)
    base = col.image_unit(0, k + k + m_rest + n_rest).astype(np.float32)
    true_u = base[:k]
    comp = base[k:2 * k] if companion_sigma is None else gfo._noisy_unit(rng, true_u, companion_sigma)
    ref = np.concatenate([true_u, comp, gfo._noisy_unit(rng, true_u[:nd], 0.3 * sigma), base[2 * k:2 * k + m_rest]])
    qry = np.concatenate([gfo._noisy_unit(rng, true_u, sigma), base[2 * k + m_rest:]])
    a = np.c_[p2[:nd], np.ones(nd)] @ F
    along = np.c_[-a[:, 1], a[:, 0]] / np.linalg.norm(a[:, :2], axis=1, keepdims=True)
    foot = p1[:nd] - (((np.c_[p1[:nd], np.ones(nd)] * a).sum(1)) / (a[:, 0] ** 2 + a[:, 1] ** 2))[:, None] * a[:, :2]
    off = rng.uniform(40, 300, nd) * rng.choice([-1.0, 1.0], nd)
    xy_comp = p1n if companions else rng.uniform(-1800, 1800, (k, 2))
    xy_ref = np.concatenate([p1n, xy_comp, foot + off[:, None] * along, rng.uniform(-1800, 1800, (m_rest, 2))]).astype(np.float32)
    xy_qry = np.concatenate([p2n, rng.uniform(-1800, 1800, (n_rest, 2))]).astype(np.float32)
    ref, qry = ref.astype(np.float32).reshape(-1, 128), qry.astype(np.float32).reshape(-1, 128)
    if dups and M >= 8:
        for a_, b_ in ((0, M - 1), (1, M - 2)):
            ref[b_], xy_ref[b_] = ref[a_], xy_ref[a_]
        ref[M - 3] = ref[2]
    if dups and N >= 8:
        qry[N - 1], xy_qry[N - 1] = qry[0], xy_qry[0]
        qry[N - 2] = qry[1]
    pr, pq = rng.permutation(M), rng.permutation(N)
    R, Q = np.empty_like(ref), np.empty_like(qry)
    XR, XQ = np.empty_like(xy_ref), np.empty_like(xy_qry)
    R[pr], XR[pr], Q[pq], XQ[pq] = ref, xy_ref, qry, xy_qry
    true = set(zip(pr[:k].tolist(), pq[:k].tolist()))
    decoyed = set(zip(pr[:nd].tolist(), pq[:nd].tolist()))
    return dict(ref=R, qry=Q, xy_ref=XR, xy_qry=XQ, H=H, F=F, true=true, decoyed=decoyed)
