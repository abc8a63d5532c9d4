"""TEST INFRASTRUCTURE ONLY — numpy restatement of the float regime of msfm_match_pairs_guided (GUIDED-SPEC with
rescore_band > 0 in include/msfm_match.h): the gated quantised 2-NN of oracle.guided_oracle decides every row, except
band rows (both gated quantised neighbours exist and fl(d0/d1) lies within ratio*(1 +- band) or ratio_good*(1 +- band)),
which are decided on their fp32 top-2 among the allowed reference rows: squared L2 accumulated in index order with
separate multiply and add (np.float32 never contracts), lowest index on ties.  Also the float variant of the
planted-decoy scene and the proven candidate bound T(q) the collect pass uses."""
from __future__ import annotations

import numpy as np

from metricsfm_b200 import synth
from oracle import geo_oracle as go
from oracle import guided_oracle as gdo
from oracle import oracle

f32 = np.float32
REJECT_GT = 1  # MSFM_RATIO_REJECT_GT


def sqdist_f32(ref: np.ndarray, query: np.ndarray) -> np.ndarray:
    """[N, M] float32: sum_k (q_k - r_k)^2 accumulated for k = 0 .. 127 in order, every operation rounded to fp32."""
    r = np.asarray(ref, np.float32).reshape(-1, 128)
    q = np.asarray(query, np.float32).reshape(-1, 128)
    acc = np.zeros((q.shape[0], r.shape[0]), np.float32)
    for k in range(128):
        t = q[:, k, None] - r[None, :, k]
        acc += t * t
    return acc


def masked_knn2_f32(ref, query, allowed):
    """fp32 2-NN of every query row among its allowed reference rows (lowest index on ties): ids [N, 2] int32,
    dists [N, 2] float32, a missing neighbour is (-1, +inf)."""
    allowed = np.asarray(allowed, bool)
    n, m = allowed.shape
    ids = np.full((n, 2), -1, np.int32)
    dists = np.full((n, 2), np.inf, np.float32)
    for c in range(0, n, 512):
        D = sqdist_f32(ref, np.asarray(query, np.float32).reshape(-1, 128)[c:c + 512]).astype(np.float64)
        D[~allowed[c:c + 512]] = np.inf  # every fp32 distance is finite for finite rows
        rows = np.arange(D.shape[0])
        for k in range(2):
            j = np.argmin(D, axis=1)  # first index of the minimum: lowest index on ties
            have = np.isfinite(D[rows, j])
            ids[c + rows[have], k] = j[have]
            dists[c + rows[have], k] = D[rows[have], j[have]].astype(np.float32)
            D[rows, j] = np.inf
    return ids, dists


def residuals(x, scale: float) -> np.ndarray:
    """r_x = ||scale * x - q_x||_2 of every row (quantisation residual, clamping included), float64."""
    x = np.asarray(x, np.float32).reshape(-1, 128)
    return np.sqrt(((x.astype(np.float64) * scale - oracle.quantize_f32(x, scale)) ** 2).sum(1))


def exact_threshold(d1q, rx, rmax):
    """T(q) = (sqrt(d1_q) + 2 (r_x + R))^2, widened by 2^-15 for the fp32 distance sum, rounded up (aux_kernels.cuh)."""
    return np.ceil((np.sqrt(np.asarray(d1q, np.float64)) + 2.0 * (rx + rmax)) ** 2 * (1.0 + 2.0 ** -15))


def _accepts(r, th, reject_gt):
    return ~(r > f32(th)) if reject_gt else (r < f32(th))


def band_rows(ids, dists, ratio, ratio_good, band):
    """The band rule of msfm_params.rescore_band on a (gated) quantised 2-NN."""
    both = (ids[:, 0] >= 0) & (ids[:, 1] >= 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = dists[:, 0] / dists[:, 1]
        bw = f32(band)
        out = both & (np.abs(r - f32(ratio)) <= bw * f32(ratio))
        if ratio_good > 0:
            out |= both & (np.abs(r - f32(ratio_good)) <= bw * f32(ratio_good))
    return out


def match_pair_guided_float(ref, query, xy_ref, xy_qry, F, th: float, ratio: float, *, scale: float = 512.0,
                            band: float = 0.0, float_rows: bool = True, max_dist_sq: float = 0.0, min_keypoints: int = 20,
                            orientation: int = 0, ratio_good: float = 0.0, reject_gt: bool = False,
                            allowed: np.ndarray | None = None):
    """One pair of msfm_match_pairs_guided with mutual = 0.  ref / query: float32 rows uploaded at `scale` (float_rows)
    or u8 rows (float_rows = False: the integer guided rule).  Returns dict(ok, pairs, good, band, allowed, ids, dists)."""
    empty = dict(ok=False, pairs=np.empty((0, 2), np.int32), good=np.empty((0,), np.uint8), band=None, allowed=None,
                 ids=None, dists=None)
    ref_f = np.asarray(ref).reshape(-1, 128)
    qry_f = np.asarray(query).reshape(-1, 128)
    M, N = ref_f.shape[0], qry_f.shape[0]
    if M < min_keypoints or N < min_keypoints:
        return empty
    if M == 0 or N == 0:
        return {**empty, "ok": True}
    qr = oracle.quantize_f32(ref_f, scale) if float_rows else ref_f.astype(np.uint8)
    qq = oracle.quantize_f32(qry_f, scale) if float_rows else qry_f.astype(np.uint8)
    if allowed is None:
        allowed = gdo.gate_f32(F, xy_ref, xy_qry, th)
    ids, d = gdo.masked_knn2(gdo.dist_u8(qr, qq), allowed)
    both = (ids[:, 0] >= 0) & (ids[:, 1] >= 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        rq = d[:, 0] / d[:, 1]
    keep = both & _accepts(rq, ratio, reject_gt)
    if max_dist_sq > 0:
        keep &= d[:, 0] < f32(max_dist_sq)
    good = keep & (ratio_good > 0) & _accepts(rq, ratio_good, reject_gt)
    j = ids[:, 0].copy()
    bnd = band_rows(ids, d, ratio, ratio_good, band) if (float_rows and band > 0) else np.zeros(N, bool)
    if bnd.any():
        b = np.nonzero(bnd)[0]
        fids, fd = masked_knn2_f32(ref_f, qry_f[b], allowed[b])
        with np.errstate(divide="ignore", invalid="ignore"):
            fr = fd[:, 0] / fd[:, 1]
        kb = (fids[:, 0] >= 0) & (fids[:, 1] >= 0) & _accepts(fr, ratio, reject_gt)
        if max_dist_sq > 0:
            kb &= (fd[:, 0] * (f32(scale) * f32(scale))) < f32(max_dist_sq)
        keep[b] = kb
        good[b] = kb & (ratio_good > 0) & _accepts(fr, ratio_good, reject_gt)
        j[b] = fids[:, 0]
    qi = np.nonzero(keep)[0].astype(np.int32)
    cols = (j[qi], qi) if orientation == 0 else (qi, j[qi])
    return dict(ok=True, pairs=np.stack(cols, axis=1).astype(np.int32).reshape(-1, 2), good=good[qi].astype(np.uint8),
                band=bnd, allowed=allowed, ids=ids, dists=d)


# ---------------------------------------------------------------------------------------------------------------------
def _noisy_unit(rng, unit, sigma):
    x = np.maximum(unit * 512.0 + rng.normal(0.0, sigma, unit.shape), 0.0)
    return (x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-12)).astype(np.float32)


def float_decoy_scene(seed, M, N, *, decoy_frac=1.0, sigma=6.0, dups=True):
    """oracle.guided_oracle.decoy_scene with unit-norm float32 rows (float noise, not quantised), to be uploaded at
    scale 512: k true correspondences, a fraction with a planted look-alike reference row 40-300 px off the epipolar
    line, unrelated rows, and (dups) exact and descriptor-only duplicates."""
    rng = np.random.default_rng(seed)
    kd_max = M // 2 if decoy_frac > 0 else M
    k = min(kd_max, N)
    nd = int(round(k * decoy_frac))
    nt = max(k, 64)
    p1, p2 = go.two_view_scene(rng, nt, max(M, N))
    F = gdo.eight_point(p1[:nt], p2[:nt])
    col = synth.Collection(max(M, N, 1), seed=seed)
    m_rest, n_rest = M - k - nd, N - k
    base = col.image_unit(0, k + m_rest + n_rest).astype(np.float32)
    true_u = base[:k]
    ref = np.concatenate([true_u, _noisy_unit(rng, true_u[:nd], 0.3 * sigma), base[k:k + m_rest]]).astype(np.float32)
    qry = np.concatenate([_noisy_unit(rng, true_u, sigma), base[k + m_rest:]]).astype(np.float32)
    a = np.c_[p2[:nd], np.ones(nd)] @ F
    nrm = a[:, :2] / np.linalg.norm(a[:, :2], axis=1, keepdims=True)
    off = rng.uniform(40, 300, nd) * rng.choice([-1.0, 1.0], nd)
    xy_ref = np.concatenate([p1[:k], p1[:nd] + off[:, None] * nrm, p1[nt:nt + m_rest]]).astype(np.float32)
    xy_qry = np.concatenate([p2[:k], p2[nt:nt + n_rest]]).astype(np.float32)
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
    return dict(ref=R, qry=Q, xy_ref=XR, xy_qry=XQ, F=F, true=true)
