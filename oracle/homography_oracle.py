"""TEST INFRASTRUCTURE ONLY — numpy restatement of HOMOG-SPEC (include/msfm_match.h), the homography-guided re-matching
of msfm_match_pairs_guided_homography, and of the RANSAC search of msfm_geo_homography (geo_homography_kernel in
metricsfm_b200/csrc/geo_kernels.cuh), step for step.  Also the planar scenes with look-alikes on the epipolar line that
the tests and tools/guided_homography_bench.py match on."""
from __future__ import annotations

import numpy as np

from metricsfm_b200 import synth
from oracle import geo_oracle as go
from oracle import guided_oracle as gdo

_U64 = np.uint64


# ---------------------------------------------------------------------------------------------------------------------
# The gate and the guided match
def gate_h32(H, xy_ref, xy_qry, th: float) -> np.ndarray:
    """[N query, M ref] bool: element (q, j) is allowed iff (du*du) + (dv*dv) <= t2 * (W*W) (HOMOG-SPEC), with H rounded
    once to float32 and every operation rounded to float32 (numpy float32 arithmetic does not contract)."""
    h = np.asarray(H, np.float64).reshape(9).astype(np.float32)
    t2 = np.float32(th) * np.float32(th)
    xr = np.asarray(xy_ref, np.float32).reshape(-1, 2)
    xq = np.asarray(xy_qry, np.float32).reshape(-1, 2)
    with np.errstate(over="ignore", invalid="ignore"):
        U, V, W = (((h[3 * k] * xr[:, 0]) + (h[3 * k + 1] * xr[:, 1])) + h[3 * k + 2] for k in range(3))  # [M] each
        du = U[None, :] - (xq[:, 0:1] * W[None, :])
        dv = V[None, :] - (xq[:, 1:2] * W[None, :])
        return ((du * du) + (dv * dv)) <= (t2 * (W * W))[None, :]


def transfer_err64(H, xy_ref, xy_qry) -> np.ndarray:
    """[N, M] float64 squared transfer distance |p_q - pi(H p_j)|^2 (inf where w = 0)."""
    H = np.asarray(H, np.float64).reshape(3, 3)
    xr = np.c_[np.asarray(xy_ref, np.float64).reshape(-1, 2), np.ones(len(xy_ref))]
    t = xr @ H.T
    with np.errstate(divide="ignore", invalid="ignore"):
        u, v = t[:, 0] / t[:, 2], t[:, 1] / t[:, 2]
    xq = np.asarray(xy_qry, np.float64).reshape(-1, 2)
    e = (xq[:, 0:1] - u[None, :]) ** 2 + (xq[:, 1:2] - v[None, :]) ** 2
    return np.where(np.isfinite(e), e, np.inf)


def match_pair_guided_h(ref, query, xy_ref, xy_qry, H, th: float, ratio: float, **kw):
    """Whole homography-guided path for one pair (guided_oracle.match_pair_guided with the HOMOG-SPEC gate).  Returns
    dict(ok, ids, dists, pairs, good, allowed)."""
    return gdo.match_pair_guided(ref, query, xy_ref, xy_qry, None, th, ratio, allowed=gate_h32(H, xy_ref, xy_qry, th), **kw)


# ---------------------------------------------------------------------------------------------------------------------
# Exact restatement of the RANSAC search of geo_homography_kernel: counter-based 4-point draws, geo_oracle's subsample
# and isotropic scale, the orientation subset check and the DLT in double, scoring in float32, winner = most inliers then
# lowest hypothesis id, back to pixel units, H22 normalisation.  The GPU contracts multiply-adds into FMAs, so a point
# whose float32 error lies within rounding reach of th^2 may be counted differently there; `ransac_search_h` reports
# those points per model ("borderline").
def draw_samples4(seed: int, pair_index: int, n_hyp: int, n_pts: int) -> np.ndarray:
    """[n_hyp, 4] point indices: geo_oracle.draw_samples' stream with four slots."""
    h = np.arange(n_hyp, dtype=_U64)
    ctr = (_U64(pair_index & 0xFFFFFFFFFFFFFFFF) << _U64(32)) | h
    st = go.geo_mix(_U64(seed & 0xFFFFFFFFFFFFFFFF) ^ go.geo_mix(ctr))
    idx = np.zeros((n_hyp, 4), np.int64)
    for k in range(4):
        pending = np.ones((n_hyp,), bool)
        while pending.any():
            st[pending] = go.geo_mix(st[pending])
            cand = ((st >> _U64(11)) % _U64(n_pts)).astype(np.int64)
            idx[pending, k] = cand[pending]
            pending &= (idx[:, :k] == cand[:, None]).any(1)
    return idx


_TRIPLES = ((0, 1, 2), (1, 2, 3), (0, 2, 3), (0, 1, 3))


def subset_ok(x1, y1, x2, y2) -> np.ndarray:
    """[H] bool: the orientation check derived from cv::findHomography's checkSubset, det of every triple in image 1
    times that in image 2 >= 0.  Stricter than OpenCV (which also accepts a sample whose four triples all flip), and
    without OpenCV's collinearity test."""
    a, b, c, d = (np.asarray(v, np.float64) for v in (x1, y1, x2, y2))
    ok = np.ones(a.shape[0], bool)
    one = np.ones(a.shape[0])
    for t in _TRIPLES:
        A = np.stack([a[:, t[0]], b[:, t[0]], one, a[:, t[1]], b[:, t[1]], one, a[:, t[2]], b[:, t[2]], one], 1)
        B = np.stack([c[:, t[0]], d[:, t[0]], one, c[:, t[1]], d[:, t[1]], one, c[:, t[2]], d[:, t[2]], one], 1)
        ok &= ~(go._det3(A) * go._det3(B) < 0.0)
    return ok


def four_point_batch(x1, y1, x2, y2):
    """The kernel's four_point_h on a batch of samples ([H, 4] each): the 8 x 9 DLT system reduced by Gauss-Jordan
    elimination with full pivoting (a pivot below 1e-12 means no model), h = null vector with free component 1,
    unit-normalised.  Returns (models [H, 9] float64, valid [H] bool)."""
    a, b, c, d = (np.asarray(v, np.float64) for v in (x1, y1, x2, y2))
    n = a.shape[0]
    z, o = np.zeros_like(a), np.ones_like(a)
    r0 = np.stack([a, b, o, z, z, z, -c * a, -c * b, -c], 2)   # [H, 4, 9]
    r1 = np.stack([z, z, z, a, b, o, -d * a, -d * b, -d], 2)
    A = np.stack([r0, r1], 2).reshape(n, 8, 9)                 # rows 2i, 2i+1
    rows = np.arange(n)
    perm = np.tile(np.arange(9), (n, 1))
    dead = np.zeros((n,), bool)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for k in range(8):
            sub = np.abs(A[:, k:, k:]).reshape(n, -1)
            arg = sub.argmax(1)
            dead |= sub[rows, arg] < 1e-12
            pr, pc = k + arg // (9 - k), k + arg % (9 - k)
            t = A[rows, k].copy(); A[rows, k] = A[rows, pr]; A[rows, pr] = t
            t = A[rows, :, k].copy(); A[rows, :, k] = A[rows, :, pc]; A[rows, :, pc] = t
            t = perm[rows, k].copy(); perm[rows, k] = perm[rows, pc]; perm[rows, pc] = t
            inv = 1.0 / A[rows, k, k]
            A[:, k, k:] *= inv[:, None]
            others = [i for i in range(8) if i != k]
            f = A[:, others, k].copy()
            A[:, others, k:] -= f[:, :, None] * A[:, k, None, k:]
        Hm = np.zeros((n, 9))
        Hm[rows[:, None], perm[:, :8]] = -A[:, :, 8]
        Hm[rows, perm[:, 8]] = 1.0
        nrm = 1.0 + (A[:, :, 8] ** 2).sum(1)
        ok = ~dead & np.isfinite(nrm)
        Hm = Hm / np.sqrt(np.where(ok, nrm, 1.0))[:, None]
    return Hm, ok


def four_point(pt1, pt2):
    """Unit-norm H ([9]) through four correspondences pt1 -> pt2 as the kernel's four_point_h, or None."""
    p1, p2 = np.asarray(pt1, np.float32), np.asarray(pt2, np.float32)
    Hm, ok = four_point_batch(p1[None, :, 0], p1[None, :, 1], p2[None, :, 0], p2[None, :, 1])
    return Hm[0] if ok[0] else None


_EPS32 = 2.0 ** -24


def score_models_h(Hf, pts, th2, chunk=256):
    """Inlier count of every float32 model Hf [K, 9] on the scaled points pts [4, n] (h_transfer_err<float>'s operations,
    err <= th2, zero or non-finite w = outlier), and its number of borderline points: those whose err lies within a
    forward rounding bound of th2 (8 u times the sums of absolute terms of U, V, W carried through the division and the
    difference), so that another contraction of the same float32 expression, or a one-ulp change of an entry of H, may
    classify them differently."""
    ax, ay, bx, by = pts
    cnt, brd = np.zeros((len(Hf),), np.int64), np.zeros((len(Hf),), np.int64)
    for c0 in range(0, len(Hf), chunk):
        H = Hf[c0:c0 + chunk, :, None]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            w = H[:, 6] * ax + H[:, 7] * ay + H[:, 8]
            U = H[:, 0] * ax + H[:, 1] * ay + H[:, 2]
            V = H[:, 3] * ax + H[:, 4] * ay + H[:, 5]
            dx, dy = U / w - bx, V / w - by
            err = dx * dx + dy * dy
            err = np.where((w == 0) | ~np.isfinite(w), np.float32(np.inf), err)
            cnt[c0:c0 + chunk] = (err <= th2).sum(1)
            G = Hf[c0:c0 + chunk].astype(np.float64)[:, :, None]
            x, y = np.abs(ax.astype(np.float64)), np.abs(ay.astype(np.float64))
            aU = np.abs(G[:, 0] * x) + np.abs(G[:, 1] * y) + np.abs(G[:, 2])
            aV = np.abs(G[:, 3] * x) + np.abs(G[:, 4] * y) + np.abs(G[:, 5])
            aW = np.abs(G[:, 6] * x) + np.abs(G[:, 7] * y) + np.abs(G[:, 8])
            w64 = np.abs(w.astype(np.float64))
            u64, v64 = np.abs(U.astype(np.float64)) / w64, np.abs(V.astype(np.float64)) / w64
            ex = 8 * _EPS32 * (aU / w64 + u64 * aW / w64 + u64 + np.abs(bx.astype(np.float64)))
            ey = 8 * _EPS32 * (aV / w64 + v64 * aW / w64 + v64 + np.abs(by.astype(np.float64)))
            e64 = err.astype(np.float64)
            band = 2 * (np.sqrt(e64) * (ex + ey)) + (ex + ey) ** 2 + 8 * _EPS32 * e64
            b = ~(np.abs(e64 - th2) > band) & np.isfinite(w64) & (w64 > 0)   # a NaN bound counts as borderline
            brd[c0:c0 + chunk] = b.sum(1)
    return cnt, brd


def pixel_H(Hf, s) -> np.ndarray:
    """Float32 models of the scaled points back in pixel units (T^-1 H T, T = diag(s, s, 1)), scaled so that H22 = 1
    unless |H22| <= 1e-12 ||H||, then to unit norm, as the kernel returns them.  [K, 9] float64."""
    s = float(s)
    T = np.array([1.0, 1.0, 1.0 / s, 1.0, 1.0, 1.0 / s, s, s, 1.0])
    H = Hf.astype(np.float64) * T
    nrm = np.sqrt((H * H).sum(1))
    h22 = H[:, 8]
    k = np.where(np.abs(h22) > 1e-12 * nrm, 1.0 / np.where(h22 == 0, 1.0, h22), 1.0 / np.where(nrm == 0, 1.0, nrm))
    return H * k[:, None]


def ransac_search_h(pt1_used, pt2_used, *, seed: int, pair_index: int, iters: int = 1024, th: float = 3.0) -> dict:
    """The kernel's whole hypothesis search on the used matches of one pair (callers apply the point-count gates).
    Returns a dict with the per-model arrays H (pixel units, H22-normalised), Hf (float32, scaled units), id (h), count,
    border; `win` (index of the most-inliers, lowest-id model, or -1 without any model), `admissible` and `certain` as
    geo_oracle.ransac_search defines them."""
    iters = iters if iters > 0 else 1024
    pts, s = go.subsample(pt1_used, pt2_used)
    n_pts = pts.shape[1]
    out = dict(scale=s, n_pts=n_pts, H=np.zeros((0, 9)), Hf=np.zeros((0, 9), np.float32), id=np.zeros((0,), np.int64),
               count=np.zeros((0,), np.int64), border=np.zeros((0,), np.int64), win=-1, admissible=np.zeros((0,), bool),
               certain=True)
    if n_pts < 4:
        return out
    idx = draw_samples4(seed, pair_index, iters, n_pts)
    smp = [v[idx] for v in pts]
    ok = subset_ok(*smp)
    Hm, valid = four_point_batch(*smp)
    ok &= valid
    if not ok.any():
        return out
    ids = np.flatnonzero(ok)
    Hf = Hm[ok].astype(np.float32)
    th2 = np.float32(np.float32(np.float32(th) * s) * np.float32(th)) * s
    cnt, brd = score_models_h(Hf, pts, th2)
    order = np.lexsort((ids, -cnt))
    win = int(order[0])
    lo_max = (cnt - brd).max()
    adm = cnt + brd >= lo_max
    C = cnt[win]
    rivals = (cnt + brd > C) | ((cnt + brd == C) & (ids < ids[win]))
    rivals[win] = False
    out.update(H=pixel_H(Hf, s), Hf=Hf, id=ids, count=cnt, border=brd, win=win, admissible=adm,
               certain=bool(brd[win] == 0 and not rivals.any()))
    return out


def h_error(H, pt1, pt2) -> np.ndarray:
    """[n] float64 one-sided transfer error |p2 - pi(H p1)|^2 (inf where w is zero or not finite)."""
    H = np.asarray(H, np.float64).reshape(3, 3)
    p1 = np.c_[np.asarray(pt1, np.float64).reshape(-1, 2), np.ones(len(pt1))]
    t = p1 @ H.T
    p2 = np.asarray(pt2, np.float64).reshape(-1, 2)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = (t[:, 0] / t[:, 2] - p2[:, 0]) ** 2 + (t[:, 1] / t[:, 2] - p2[:, 1]) ** 2
    bad = (t[:, 2] == 0) | ~np.isfinite(t[:, 2]) | ~np.isfinite(e)
    return np.where(bad, np.inf, e)


def geo_pair_h(pt1_all, pt2_all, use, *, seed: int, pair_index: int, th: float = 3.0, min_points: int = 30,
               min_inliers: int = 30, iters: int = 1024, H=None):
    """Decision flow of one pair of msfm_geo_homography: fewer than max(min_points, 4) used matches or no model ->
    rejected, 0 inliers; otherwise the inlier count of H among all used matches (double) decides, and the mask is the
    consensus set.  H defaults to the restated winner; pass the H a kernel returned to restate the decisions around it.
    Returns (ok, inliers, mask, H or None, search or None)."""
    g = np.asarray(use).astype(bool)
    pt1_all, pt2_all = np.asarray(pt1_all, np.float32), np.asarray(pt2_all, np.float32)
    none = np.zeros((len(g),), bool)
    if g.sum() < max(min_points, 4):
        return False, 0, none, None, None
    srch = ransac_search_h(pt1_all[g], pt2_all[g], seed=seed, pair_index=pair_index, iters=iters, th=th)
    if srch["win"] < 0:
        return False, 0, none, None, srch
    H = srch["H"][srch["win"]] if H is None else np.asarray(H, np.float64).reshape(9)
    inlier = np.zeros((len(g),), bool)
    inlier[g] = h_error(H, pt1_all[g], pt2_all[g]) <= float(th) * float(th)
    inl = int(inlier.sum())
    if inl < min_inliers:
        return False, inl, none, H, srch
    return True, inl, inlier, H, srch


# ---------------------------------------------------------------------------------------------------------------------
# Scenes
def plane_views(rng, f: float = 3000.0):
    """Two nadir views of the ground plane Z = 0 from height ~100 (second camera moved along the flight direction x,
    slightly rotated).  Returns (project(X, cam) -> [n, 2] centred pixels, H mapping view 0 to view 1 for plane points,
    F of the two views)."""
    h0 = rng.uniform(90, 110)
    ang = np.deg2rad(rng.uniform(-3, 3, 3))
    cx, sx, cy, sy, cz, sz = np.cos(ang[0]), np.sin(ang[0]), np.cos(ang[1]), np.sin(ang[1]), np.cos(ang[2]), np.sin(ang[2])
    R = (np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
         @ np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]))
    C1 = np.array([rng.uniform(20, 35), rng.uniform(-2, 2), h0 + rng.uniform(-3, 3)])
    cams = [(np.eye(3), np.array([0.0, 0.0, h0])), (R, C1)]
    K = np.diag([f, f, 1.0])

    def P(cam):  # 3 x 4, camera looking down (-Z): x_c = R^T (X - C) with the view axis flipped
        Rc, Cc = cam
        flip = np.diag([1.0, -1.0, -1.0])
        Rw = flip @ Rc.T
        return K @ np.c_[Rw, -Rw @ Cc]

    P0, P1 = P(cams[0]), P(cams[1])

    def project(X, k):
        x = np.c_[X, np.ones(len(X))] @ (P0 if k == 0 else P1).T
        return x[:, :2] / x[:, 2:3]

    # plane Z = 0: x_k ~ P_k[:, (0, 1, 3)] (X, Y, 1)
    G0, G1 = P0[:, [0, 1, 3]], P1[:, [0, 1, 3]]
    H = G1 @ np.linalg.inv(G0)
    H = H / H[2, 2]
    X = np.c_[rng.uniform(-40, 40, (64, 2)), rng.uniform(-30, 30, (64, 1))]  # off-plane points for the 8-point F
    F = gdo.eight_point(project(X, 0), project(X, 1))
    return project, H, F


def planar_decoy_scene(seed, M, N, *, decoy_frac=0.5, sigma=6.0, noise=0.5, dups=True, companions=True):
    """One pair over a ground plane: reference image of M rows, query image of N rows.  k true correspondences (query row
    = noisy copy of its reference row, keypoints related by the plane's H up to `noise` px of keypoint noise); a fraction
    of them get a planted decoy: a second reference row whose descriptor is a closer-than-noise copy, placed ON the
    epipolar line of the true point, 40-300 px from it (repeated structure along the flight direction).  Every true
    reference keypoint has a companion row at the same position with an unrelated descriptor (a second keypoint at one
    location, like SIFT's extra orientations), so the transfer disc of a true match holds a second neighbour (companions =
    False: those rows sit at random positions, and a true row's disc usually holds its true row alone).  The other
    rows are unrelated descriptors at random positions.  dups: a few reference and query rows are exact copies of others
    (descriptor and keypoint: ties), and a few share only the descriptor.  Returns dict(ref, qry, xy_ref, xy_qry, H, F,
    true, decoyed)."""
    rng = np.random.default_rng(seed)
    project, H, F = plane_views(rng)
    k = min(M // 3, N)
    nd = int(round(k * decoy_frac))
    m_rest, n_rest = M - 2 * k - nd, N - k
    # true points on the plane, inside both views
    G = np.c_[rng.uniform(-55, 55, (k, 1)), rng.uniform(-55, 55, (k, 1)), np.zeros((k, 1))]
    p1, p2 = project(G, 0), project(G, 1)
    p1n = p1 + rng.normal(0, noise, p1.shape)
    p2n = p2 + rng.normal(0, noise, p2.shape)
    col = synth.Collection(max(M, N, 1), seed=seed)
    base = col.image_unit(0, k + k + m_rest + n_rest)
    true_u = base[:k]
    ref = np.concatenate([synth.quantize_512(true_u), synth.quantize_512(base[k:2 * k]), gdo._noisy_u8(rng, true_u[:nd], 0.3 * sigma),
                          synth.quantize_512(base[2 * k:2 * k + m_rest])])
    qry = np.concatenate([gdo._noisy_u8(rng, true_u, sigma), synth.quantize_512(base[2 * k + m_rest:])])
    # decoys: along the line a = F^T p_q in the reference image, through the true reference point
    a = np.c_[p2[:nd], np.ones(nd)] @ F
    along = np.c_[-a[:, 1], a[:, 0]] / np.linalg.norm(a[:, :2], axis=1, keepdims=True)
    foot = p1[:nd] - (((np.c_[p1[:nd], np.ones(nd)] * a).sum(1)) / (a[:, 0] ** 2 + a[:, 1] ** 2))[:, None] * a[:, :2]
    off = rng.uniform(40, 300, nd) * rng.choice([-1.0, 1.0], nd)
    xy_comp = p1n if companions else rng.uniform(-1800, 1800, (k, 2))
    xy_ref = np.concatenate([p1n, xy_comp, foot + off[:, None] * along, rng.uniform(-1800, 1800, (m_rest, 2))]).astype(np.float32)
    xy_qry = np.concatenate([p2n, rng.uniform(-1800, 1800, (n_rest, 2))]).astype(np.float32)
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


def kept(pairs, which) -> int:
    """How many of the (reference row, query row) correspondences `which` an orientation-0 match list holds."""
    return sum((int(j), int(q)) in which for j, q in np.asarray(pairs).reshape(-1, 2))

