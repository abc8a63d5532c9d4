"""TEST INFRASTRUCTURE ONLY — numpy restatement of the reference's geometric verification around a given fundamental
matrix (paths relative to /root/reference/SfM), used to check metricsfm_b200/csrc/geo_kernels.cuh.  The RANSAC search
itself lives in OpenCV (cv::findFundamentalMat, un-vendored, version 2.4.13.6 per SfM/CMakeLists.txt:48); the tests
compare against the cv2 build present in this image (statistical parity: its RNG stream cannot be reproduced)."""
from __future__ import annotations

import numpy as np


def f_filter(F: np.ndarray, pt1: np.ndarray, pt2: np.ndarray, th_epi: float = 3.0) -> np.ndarray:
    """GeoVerification::GeoVerificationFundamental(pt1, pt2, F, inliers), src/utils/geo_verification.cc:60-79:
    l1 = F * p1, normalised by sqrt(a^2 + b^2); keep i iff |l1 . p2| < th_epi.  Double arithmetic."""
    F = np.asarray(F, np.float64).reshape(3, 3)
    p1 = np.concatenate([np.asarray(pt1, np.float64), np.ones((len(pt1), 1))], 1)
    p2 = np.concatenate([np.asarray(pt2, np.float64), np.ones((len(pt2), 1))], 1)
    l1 = p1 @ F.T
    n = np.sqrt(l1[:, 0] ** 2 + l1[:, 1] ** 2)
    dis = ((l1 / n[:, None]) * p2).sum(1)
    return np.abs(dis) < th_epi


def ransac_error(F: np.ndarray, pt1: np.ndarray, pt2: np.ndarray) -> np.ndarray:
    """cv::findFundamentalMat's per-point RANSAC error (calib3d fundam.cpp, computeReprojError / computeError): the
    larger of the squared distances of p2 to F p1 and of p1 to F^T p2; a point is an inlier iff err <= th^2."""
    F = np.asarray(F, np.float64).reshape(3, 3)
    p1 = np.concatenate([np.asarray(pt1, np.float64), np.ones((len(pt1), 1))], 1)
    p2 = np.concatenate([np.asarray(pt2, np.float64), np.ones((len(pt2), 1))], 1)
    l2 = p1 @ F.T
    l1 = p2 @ F
    s = (l2 * p2).sum(1)
    d2 = s * s / (l2[:, 0] ** 2 + l2[:, 1] ** 2)
    d1 = s * s / (l1[:, 0] ** 2 + l1[:, 1] ** 2)
    return np.maximum(d1, d2)


def verify_pair(pt1_good, pt2_good, pt1_all, pt2_all, F, th: float = 3.0, min_points: int = 30, min_inliers: int = 30):
    """Decision flow of fine_matching_graph.cc:137-153 around a given F: (ok, stage-A inlier count, stage-B mask)."""
    if len(pt1_good) < min_points:
        return False, 0, np.zeros((len(pt1_all),), bool)
    inl = int((ransac_error(F, pt1_good, pt2_good) <= th * th).sum())
    if inl < min_inliers:
        return False, inl, np.zeros((len(pt1_all),), bool)
    return True, inl, f_filter(F, pt1_all, pt2_all, th)


def two_view_scene(rng, n_true, n_out, noise=0.5, f=3000.0):
    """Centred pixel coordinates of n_true correspondences of a rigid scene in two views + n_out random outliers."""
    X = np.concatenate([rng.uniform(-40, 40, (n_true, 2)), rng.uniform(60, 140, (n_true, 1))], 1)
    ang = np.deg2rad(rng.uniform(4, 10))
    R = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    t = np.array([rng.uniform(8, 15), rng.uniform(-2, 2), rng.uniform(-1, 1)])
    p1 = f * X[:, :2] / X[:, 2:3]
    Xc = X @ R.T + t
    p2 = f * Xc[:, :2] / Xc[:, 2:3]
    p1 = p1 + rng.normal(0, noise, p1.shape)
    p2 = p2 + rng.normal(0, noise, p2.shape)
    o1, o2 = rng.uniform(-1800, 1800, (n_out, 2)), rng.uniform(-1800, 1800, (n_out, 2))
    return np.concatenate([p1, o1]).astype(np.float32), np.concatenate([p2, o2]).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# Exact restatement of the RANSAC search of geo_verify_kernel (metricsfm_b200/csrc/geo_kernels.cuh), step for step:
# counter-based draws, strided subsample + isotropic scale in float32, 7-point solver and cubic in double, scoring in
# float32, winner = most inliers then lowest model id 3h+f, back to pixel units, F22 normalisation.  The GPU contracts
# multiply-adds into FMAs, so a point whose float32 error lies within rounding reach of th^2 may be counted differently
# there; `ransac_search` reports those points per model ("borderline") so that a test can tell a certain winner from a
# set of admissible ones.
GEO_POINT_CAP = 2048
_U64 = np.uint64


def geo_mix(z):
    """splitmix64's output function (geo_mix), elementwise on uint64."""
    z = np.atleast_1d(np.asarray(z, _U64)).copy()
    with np.errstate(over="ignore"):
        z += _U64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> _U64(27))) * _U64(0x94D049BB133111EB)
        return z ^ (z >> _U64(31))


def draw_samples(seed: int, pair_index: int, n_hyp: int, n_pts: int) -> np.ndarray:
    """[n_hyp, 7] point indices of hypotheses 0..n_hyp-1 of the pair with global index pair_index: the state starts at
    mix(seed ^ mix((pair_index << 32) | h)); each slot repeats st = mix(st), idx = (st >> 11) % n_pts until idx is new."""
    h = np.arange(n_hyp, dtype=_U64)
    ctr = (_U64(pair_index & 0xFFFFFFFFFFFFFFFF) << _U64(32)) | h
    st = geo_mix(_U64(seed & 0xFFFFFFFFFFFFFFFF) ^ geo_mix(ctr))
    idx = np.zeros((n_hyp, 7), np.int64)
    for k in range(7):
        pending = np.ones((n_hyp,), bool)
        while pending.any():
            st[pending] = geo_mix(st[pending])
            cand = ((st >> _U64(11)) % _U64(n_pts)).astype(np.int64)
            idx[pending, k] = cand[pending]
            pending &= (idx[:, :k] == cand[:, None]).any(1)
    return idx


def subsample(pt1_good, pt2_good):
    """The points the search scores: good matches number gi with gi % stride == 0 (stride = ceil(n_good / 2048)), at
    most 2048, scaled in float32 by s = 1 / max(1, max |coordinate| over these sampled points).  Returns ([4, n] float32
    x1, y1, x2, y2, s)."""
    n_good = len(pt1_good)
    stride = max(1, -(-n_good // GEO_POINT_CAP))
    sel = np.arange(0, n_good, stride)[:GEO_POINT_CAP]
    p = np.concatenate([np.asarray(pt1_good, np.float32)[sel].T, np.asarray(pt2_good, np.float32)[sel].T])
    mx = max(np.float32(1.0), np.abs(p).max()) if p.size else np.float32(1.0)
    s = np.float32(1.0) / np.float32(mx)
    return (p * s).astype(np.float32), s


def _det3(m):
    return (m[..., 0] * (m[..., 4] * m[..., 8] - m[..., 5] * m[..., 7]) - m[..., 1] * (m[..., 3] * m[..., 8] - m[..., 5] * m[..., 6])
            + m[..., 2] * (m[..., 3] * m[..., 7] - m[..., 4] * m[..., 6]))


def solve_cubic(c3: float, c2: float, c1: float, c0: float) -> list:
    """Real roots of c3 x^3 + c2 x^2 + c1 x + c0, with the kernel's branches for degenerate leading coefficients."""
    eps = 1e-14
    if abs(c3) < eps * (abs(c2) + abs(c1) + abs(c0) + 1e-300):
        if abs(c2) < eps * (abs(c1) + abs(c0) + 1e-300):
            return [] if abs(c1) < 1e-300 else [-c0 / c1]
        d = c1 * c1 - 4.0 * c2 * c0
        if d < 0.0:
            return []
        s = np.sqrt(d)
        q = -0.5 * (c1 + (s if c1 >= 0.0 else -s))
        return [q / c2] + ([c0 / q] if abs(q) > 1e-300 else [])
    a, b, c = c2 / c3, c1 / c3, c0 / c3
    Q, R = (a * a - 3.0 * b) / 9.0, (2.0 * a * a * a - 9.0 * a * b + 27.0 * c) / 54.0
    Q3 = Q * Q * Q
    if R * R < Q3:
        th, sq = np.arccos(max(-1.0, min(1.0, R / np.sqrt(Q3)))), -2.0 * np.sqrt(Q)
        return [sq * np.cos(th / 3.0) - a / 3.0, sq * np.cos((th + 2.0 * np.pi) / 3.0) - a / 3.0,
                sq * np.cos((th - 2.0 * np.pi) / 3.0) - a / 3.0]
    A = -np.copysign(np.cbrt(abs(R) + np.sqrt(R * R - Q3)), R)
    B = Q / A if A != 0.0 else 0.0
    return [(A + B) - a / 3.0]


def seven_point_batch(x1, y1, x2, y2):
    """The kernel's seven_point on a batch of samples ([H, 7] each): Gauss-Jordan elimination of the 7 x 9 epipolar
    system with full pivoting (a pivot below 1e-12 means no model), free columns 7 and 8, det(F2 + x (F1 - F2)) = 0 by
    multilinearity, unit-normalised models, non-finite ones dropped.  Returns (models [M, 9] float64, hypothesis [M],
    root number f [M])."""
    a, b, c, d = (np.asarray(v, np.float64) for v in (x1, y1, x2, y2))
    H = a.shape[0]
    A = np.stack([c * a, c * b, c, d * a, d * b, d, a, b, np.ones_like(a)], 2)  # [H, 7, 9]
    rows = np.arange(H)
    perm = np.tile(np.arange(9), (H, 1))
    dead = np.zeros((H,), bool)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for k in range(7):
            sub = np.abs(A[:, k:, k:]).reshape(H, -1)
            arg = sub.argmax(1)              # first maximum in row-major order, as the kernel's strict '>' scan
            dead |= sub[rows, arg] < 1e-12
            pr, pc = k + arg // (9 - k), k + arg % (9 - k)
            t = A[rows, k].copy(); A[rows, k] = A[rows, pr]; A[rows, pr] = t
            t = A[rows, :, k].copy(); A[rows, :, k] = A[rows, :, pc]; A[rows, :, pc] = t
            t = perm[rows, k].copy(); perm[rows, k] = perm[rows, pc]; perm[rows, pc] = t
            inv = 1.0 / A[rows, k, k]
            A[:, k, k:] *= inv[:, None]
            others = [i for i in range(7) if i != k]
            f = A[:, others, k].copy()
            A[:, others, k:] -= f[:, :, None] * A[:, k, None, k:]
    f1, f2 = np.zeros((H, 9)), np.zeros((H, 9))
    f1[rows[:, None], perm[:, :7]] = -A[:, :, 7]
    f2[rows[:, None], perm[:, :7]] = -A[:, :, 8]
    f1[rows, perm[:, 7]], f2[rows, perm[:, 8]] = 1.0, 1.0
    D = f1 - f2
    c0, c3, c1, c2 = _det3(f2), _det3(D), np.zeros((H,)), np.zeros((H,))
    for r in range(3):
        M = f2.copy(); M[:, 3 * r:3 * r + 3] = D[:, 3 * r:3 * r + 3]; c1 += _det3(M)
        M = D.copy(); M[:, 3 * r:3 * r + 3] = f2[:, 3 * r:3 * r + 3]; c2 += _det3(M)
    models, hyp, fno = [], [], []
    for h in np.flatnonzero(~dead):
        n = 0
        for x in solve_cubic(c3[h], c2[h], c1[h], c0[h]):
            F = f2[h] + x * D[h]
            nrm = float((F * F).sum())
            if not (nrm > 1e-300) or not np.isfinite(nrm):
                continue
            models.append(F / np.sqrt(nrm)), hyp.append(h), fno.append(n)
            n += 1
    return (np.array(models, np.float64).reshape(-1, 9), np.array(hyp, np.int64), np.array(fno, np.int64))


def seven_point(pt1, pt2) -> np.ndarray:
    """Unit-norm fundamental matrices ([n, 9], n <= 3) through seven correspondences, as the kernel's seven_point."""
    p1, p2 = np.asarray(pt1, np.float32), np.asarray(pt2, np.float32)
    return seven_point_batch(p1[None, :, 0], p1[None, :, 1], p2[None, :, 0], p2[None, :, 1])[0]


_EPS32 = 2.0 ** -24


def score_models(Ff, pts, th2, chunk=256):
    """Inlier count of every float32 model Ff [M, 9] on the scaled points pts [4, n] (sym_epi_err<float>'s operation
    order, err <= th2), and its number of borderline points: those whose err lies within a forward rounding bound of
    th2, so that another contraction of the same float32 expression, or a one-ulp change of an entry of F, may classify
    them differently.  The bound is 8 u (2 M/|s| + 2 (A0|l0| + A1|l1|)/(l0^2 + l1^2) + 2 (B0|m0| + B1|m1|)/(m0^2 + m1^2)
    + 3) relative, with A, B, M the sums of absolute terms of the lines l, m and of s = p2 . l."""
    ax, ay, bx, by = pts
    cnt, brd = np.zeros((len(Ff),), np.int64), np.zeros((len(Ff),), np.int64)
    for c0 in range(0, len(Ff), chunk):
        F = Ff[c0:c0 + chunk, :, None]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            l0, l1, l2 = F[:, 0] * ax + F[:, 1] * ay + F[:, 2], F[:, 3] * ax + F[:, 4] * ay + F[:, 5], F[:, 6] * ax + F[:, 7] * ay + F[:, 8]
            s = bx * l0 + by * l1 + l2
            m0, m1 = F[:, 0] * bx + F[:, 3] * by + F[:, 6], F[:, 1] * bx + F[:, 4] * by + F[:, 7]
            d2, d1 = s * s / (l0 * l0 + l1 * l1), s * s / (m0 * m0 + m1 * m1)
            err = np.where(d1 > d2, d1, d2)
            cnt[c0:c0 + chunk] = (err <= th2).sum(1)
            near = np.nonzero(np.abs(err.astype(np.float64) - th2) <= 0.05 * th2)
            if len(near[0]):
                i, j = near
                G = Ff[c0:c0 + chunk].astype(np.float64)[i]
                x1, y1, x2, y2 = (v.astype(np.float64)[j] for v in (ax, ay, bx, by))
                A0, A1, A2 = (np.abs(G[:, 3 * r] * x1) + np.abs(G[:, 3 * r + 1] * y1) + np.abs(G[:, 3 * r + 2]) for r in range(3))
                B0 = np.abs(G[:, 0] * x2) + np.abs(G[:, 3] * y2) + np.abs(G[:, 6])
                B1 = np.abs(G[:, 1] * x2) + np.abs(G[:, 4] * y2) + np.abs(G[:, 7])
                L0, L1, S = (v.astype(np.float64)[near] for v in (l0, l1, s))
                N0, N1 = m0.astype(np.float64)[near], m1.astype(np.float64)[near]
                M = np.abs(x2) * A0 + np.abs(y2) * A1 + A2
                rel = 8 * _EPS32 * (2 * M / np.abs(S) + 2 * (A0 * np.abs(L0) + A1 * np.abs(L1)) / (L0 * L0 + L1 * L1)
                                    + 2 * (B0 * np.abs(N0) + B1 * np.abs(N1)) / (N0 * N0 + N1 * N1) + 3)
                b = ~(np.abs(err[near].astype(np.float64) - th2) > rel * th2)   # a NaN bound counts as borderline
                np.add.at(brd, c0 + i[b], 1)
    return cnt, brd


def pixel_F(Ff, s) -> np.ndarray:
    """Float32 models of the scaled points back in pixel units (T^T F T, T = diag(s, s, 1)), scaled so that F22 = 1
    when |F22| > 1e-12 ||F||, else to unit norm, as the kernel returns them.  [M, 9] float64."""
    s = float(s)
    T = np.array([s * s, s * s, s, s * s, s * s, s, s, s, 1.0])
    F = Ff.astype(np.float64) * T
    nrm = np.sqrt((F * F).sum(1))
    f22 = F[:, 8]
    k = np.where(np.abs(f22) > 1e-12 * nrm, 1.0 / np.where(f22 == 0, 1.0, f22), 1.0 / np.where(nrm == 0, 1.0, nrm))
    return F * k[:, None]


def ransac_search(pt1_good, pt2_good, *, seed: int, pair_index: int, iters: int = 1024, th: float = 3.0) -> dict:
    """The kernel's whole hypothesis search on the good matches of one pair (callers apply the point-count gates).
    Returns a dict with the per-model arrays F (pixel units, F22-normalised), Ff (float32, scaled units), id (3h+f),
    count, border; `win` (index of the most-inliers, lowest-id model, or -1 without any model), `admissible` (models
    whose count interval [count - border, count + border] reaches the largest lower end) and `certain` (the winner has
    no borderline point and every other admissible model can at best tie it with a higher id)."""
    iters = iters if iters > 0 else 1024
    pts, s = subsample(pt1_good, pt2_good)
    n_pts = pts.shape[1]
    out = dict(scale=s, n_pts=n_pts, F=np.zeros((0, 9)), Ff=np.zeros((0, 9), np.float32), id=np.zeros((0,), np.int64),
               count=np.zeros((0,), np.int64), border=np.zeros((0,), np.int64), win=-1, admissible=np.zeros((0,), bool),
               certain=True)
    if n_pts < 7:
        return out
    idx = draw_samples(seed, pair_index, iters, n_pts)
    models, hyp, fno = seven_point_batch(*(v[idx] for v in pts))
    if len(models) == 0:
        return out
    Ff = models.astype(np.float32)
    th2 = np.float32(np.float32(np.float32(th) * s) * np.float32(th)) * s
    cnt, brd = score_models(Ff, pts, th2)
    ids = 3 * hyp + fno
    order = np.lexsort((ids, -cnt))
    win = int(order[0])
    lo_max = (cnt - brd).max()
    adm = cnt + brd >= lo_max
    C = cnt[win]
    rivals = (cnt + brd > C) | ((cnt + brd == C) & (ids < ids[win]))
    rivals[win] = False
    out.update(F=pixel_F(Ff, s), Ff=Ff, id=ids, count=cnt, border=brd, win=win, admissible=adm,
               certain=bool(brd[win] == 0 and not rivals.any()))
    return out


def geo_pair(pt1_all, pt2_all, good, *, seed: int, pair_index: int, th: float = 3.0, min_points: int = 30,
             min_inliers: int = 30, iters: int = 1024, stage_b: bool = True, F=None):
    """Decision flow of one pair of msfm_geo_verify (stage_b) or msfm_geo_ransac: fewer than max(min_points, 7) good
    matches or no model -> rejected, 0 inliers; otherwise the stage-A inlier count of F among all good matches (double)
    decides, and keep is the F-filter of all matches (stage B) or the consensus mask of the good ones.  F defaults to
    the restated winner; pass the F a kernel returned to restate the decisions around it.  Returns (ok, inliers, keep,
    F or None, search or None)."""
    g = np.asarray(good).astype(bool)
    pt1_all, pt2_all = np.asarray(pt1_all, np.float32), np.asarray(pt2_all, np.float32)
    none = np.zeros((len(g),), bool)
    if g.sum() < max(min_points, 7):
        return False, 0, none, None, None
    srch = ransac_search(pt1_all[g], pt2_all[g], seed=seed, pair_index=pair_index, iters=iters, th=th)
    if srch["win"] < 0:
        return False, 0, none, None, srch
    F = srch["F"][srch["win"]] if F is None else np.asarray(F, np.float64).reshape(9)
    inlier = np.zeros((len(g),), bool)
    inlier[g] = ransac_error(F, pt1_all[g], pt2_all[g]) <= float(th) * float(th)
    inl = int(inlier.sum())
    if inl < min_inliers:
        return False, inl, none, F, srch
    return True, inl, (f_filter(F, pt1_all, pt2_all, th) if stage_b else inlier), F, srch
