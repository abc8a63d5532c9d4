"""TEST INFRASTRUCTURE ONLY — numpy restatement of GUIDED-SPEC (include/msfm_match.h), the guided re-matching of
msfm_match_pairs_guided: the epipolar gate in float32 exactly as the kernel evaluates it (one rounding per operation, no
fused multiply-add), the exact int32 distance matrix, the masked 2-NN and column best with lowest-index ties, and
oracle.ratio_select for the ratio rule, flags and orientation.  Also the planted-decoy two-view scenes the tests and
tools/guided_bench.py match on."""
from __future__ import annotations

import numpy as np

from metricsfm_b200 import synth
from oracle import geo_oracle as go
from oracle import oracle

_BIG = np.iinfo(np.int64).max


def gate_f32(F, xy_ref, xy_qry, th: float) -> np.ndarray:
    """[N query, M ref] bool: element (q, j) is allowed iff s*s <= t2 * min(na, nb) (GUIDED-SPEC), with F rounded once
    to float32 and every operation rounded to float32 (numpy float32 arithmetic does not contract)."""
    f = np.asarray(F, np.float64).reshape(9).astype(np.float32)
    t2 = np.float32(th) * np.float32(th)
    xr = np.asarray(xy_ref, np.float32).reshape(-1, 2)
    xq = np.asarray(xy_qry, np.float32).reshape(-1, 2)
    a = [((f[k] * xq[:, 0]) + (f[3 + k] * xq[:, 1])) + f[6 + k] for k in range(3)]              # [N] each
    b = [((f[3 * k] * xr[:, 0]) + (f[3 * k + 1] * xr[:, 1])) + f[3 * k + 2] for k in range(2)]  # [M] each
    s = ((a[0][:, None] * xr[None, :, 0]) + (a[1][:, None] * xr[None, :, 1])) + a[2][:, None]
    na = (a[0] * a[0]) + (a[1] * a[1])
    nb = (b[0] * b[0]) + (b[1] * b[1])
    m = np.where(nb[None, :] < na[:, None], nb[None, :], na[:, None])  # min, NaN-propagating like the kernel's select
    return (s * s) <= (t2 * m)


def dist_u8(ref: np.ndarray, query: np.ndarray) -> np.ndarray:
    """[N, M] int64 squared L2 distances of u8 rows, exact (the products stay far below 2^53)."""
    r = np.asarray(ref, np.uint8).reshape(-1, 128).astype(np.float64)
    q = np.asarray(query, np.uint8).reshape(-1, 128).astype(np.float64)
    d = (q * q).sum(1)[:, None] + (r * r).sum(1)[None, :] - 2.0 * (q @ r.T)
    return np.rint(d).astype(np.int64)


def masked_knn2(D: np.ndarray, allowed: np.ndarray):
    """FLANN-layout 2-NN among the allowed elements: ids [N, 2] int32 (lowest index on ties), dists [N, 2] float32;
    a missing neighbour is (-1, +inf)."""
    Dm = np.where(allowed, D, _BIG)
    n = Dm.shape[0]
    ids = np.full((n, 2), -1, np.int32)
    dists = np.full((n, 2), np.inf, np.float32)
    if Dm.shape[1] == 0 or n == 0:
        return ids, dists
    rows = np.arange(n)
    for k in range(2):
        j = np.argmin(Dm, axis=1)
        d = Dm[rows, j]
        have = d != _BIG
        ids[have, k] = j[have]
        dists[have, k] = d[have].astype(np.float32)
        Dm[rows, j] = _BIG
    return ids, dists


def masked_colbest(D: np.ndarray, allowed: np.ndarray) -> np.ndarray:
    """[M] int32: the closest allowed query row of every reference row (lowest index on ties), -1 if none."""
    Dm = np.where(allowed, D, _BIG)
    if Dm.shape[0] == 0:
        return np.full((Dm.shape[1],), -1, np.int32)
    q = np.argmin(Dm, axis=0).astype(np.int32)
    q[Dm[q, np.arange(Dm.shape[1])] == _BIG] = -1
    return q


def match_pair_guided(ref, query, xy_ref, xy_qry, F, th: float, ratio: float, *, mutual: bool = False,
                      max_dist_sq: float = 0.0, min_keypoints: int = 20, orientation: int = 0, ratio_good: float = 0.0,
                      reject_gt: bool = False, allowed: np.ndarray | None = None):
    """Whole guided path for one pair.  Returns dict(ok, ids, dists, pairs, good, allowed)."""
    ref = np.asarray(ref, np.uint8).reshape(-1, 128)
    query = np.asarray(query, np.uint8).reshape(-1, 128)
    if ref.shape[0] < min_keypoints or query.shape[0] < min_keypoints:
        return dict(ok=False, ids=None, dists=None, pairs=np.empty((0, 2), np.int32), good=np.empty((0,), np.uint8),
                    allowed=None)
    if allowed is None:
        allowed = gate_f32(F, xy_ref, xy_qry, th)
    D = dist_u8(ref, query)
    ids, dists = masked_knn2(D, allowed)
    cb = masked_colbest(D, allowed) if mutual else None
    pairs, good = oracle.ratio_select(ids, dists, ref.shape[0], ratio, max_dist_sq=max_dist_sq, col_best=cb,
                                      min_keypoints=min_keypoints, orientation=orientation, ratio_good=ratio_good,
                                      reject_gt=reject_gt)
    return dict(ok=True, ids=ids, dists=dists, pairs=pairs, good=good, allowed=allowed)


# ---------------------------------------------------------------------------------------------------------------------
# Scenes
def eight_point(p1, p2):
    """Normalised 8-point F (rank 2, unit Frobenius norm) with p2^T F p1 = 0, float64."""
    def normalise(p):
        p = np.asarray(p, np.float64)
        c = p.mean(0)
        s = np.sqrt(2.0) / np.mean(np.linalg.norm(p - c, axis=1))
        T = np.array([[s, 0, -s * c[0]], [0, s, -s * c[1]], [0, 0, 1.0]])
        return np.c_[p, np.ones(len(p))] @ T.T, T
    x1, T1 = normalise(p1)
    x2, T2 = normalise(p2)
    A = np.einsum("ni,nj->nij", x2, x1).reshape(-1, 9)
    F = np.linalg.svd(A)[2][-1].reshape(3, 3)
    U, S, Vt = np.linalg.svd(F)
    F = T2.T @ (U @ np.diag([S[0], S[1], 0.0]) @ Vt) @ T1
    return F / np.linalg.norm(F)


def _noisy_u8(rng, unit, sigma):
    x = np.maximum(unit * 512.0 + rng.normal(0.0, sigma, unit.shape), 0.0)
    x /= np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-12)
    return synth.quantize_512(x)


def decoy_scene(seed, M, N, *, decoy_frac=1.0, sigma=6.0, dups=True):
    """One pair on a rigid two-view scene: reference image of M rows, query image of N rows.  k true correspondences
    (query row = noisy copy of its reference row, keypoints related by the scene's F); a fraction of them get a planted
    decoy: a second reference row whose descriptor is a closer-than-noise copy, placed 40-300 px off the epipolar line.
    The other rows are unrelated descriptors at random positions.  dups: a few reference and query rows are exact copies
    of others (descriptor and keypoint: ties), and a few share only the descriptor."""
    rng = np.random.default_rng(seed)
    kd_max = M // 2 if decoy_frac > 0 else M
    k = min(kd_max, N)
    nd = int(round(k * decoy_frac))
    nt = max(k, 64)
    p1, p2 = go.two_view_scene(rng, nt, max(M, N))
    F = eight_point(p1[:nt], p2[:nt])
    col = synth.Collection(max(M, N, 1), seed=seed)
    m_rest, n_rest = M - k - nd, N - k
    base = col.image_unit(0, k + m_rest + n_rest)
    true_u = base[:k]
    ref = np.concatenate([synth.quantize_512(true_u), _noisy_u8(rng, true_u[:nd], 0.3 * sigma),
                          synth.quantize_512(base[k:k + m_rest])])
    qry = np.concatenate([_noisy_u8(rng, true_u, sigma), synth.quantize_512(base[k + m_rest:])])
    # decoys: off the line a = F^T p_q in the reference image, along its normal
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
