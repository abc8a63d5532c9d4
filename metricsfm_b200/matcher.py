"""Python host mirror of the matcher interface (thin: every call goes straight through the C ABI in
include/msfm_match.h into the CUDA library; nothing is computed here).

Names follow the reference: `KNNMatching` (SfM/src/feature/feature_matching.cpp:24-65), the FLANN-layout
`knn2` result consumed by `KNNMatchingWithGeoVerify(kp1, kp2, id, dis, matches)` (feature_matching.cpp:477-501), and
`match_pairs`, the batched form of FineMatchingGraph::BuildMatchGraph's kNN + ratio loops
(SfM/src/graph/fine_matching_graph.cc:87-133).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import Config, Pair, Params, Result, Timing


class MsfmError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{_lib.STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


@dataclass
class MatchResult:
    offsets: np.ndarray  # [n_pairs + 1] int64
    ok: np.ndarray       # [n_pairs] int32
    matches: np.ndarray  # [total, 2] int32
    good: np.ndarray | None

    def pair(self, p: int) -> np.ndarray:
        return self.matches[self.offsets[p]:self.offsets[p + 1]]

    def pair_good(self, p: int) -> np.ndarray:
        return self.good[self.offsets[p]:self.offsets[p + 1]]


def _host_ptr(a):
    """(pointer, keepalive) of a numpy array or a CPU torch tensor (pinned or not)."""
    if isinstance(a, np.ndarray):
        return a.ctypes.data, a
    if hasattr(a, "data_ptr"):
        if a.device.type != "cpu":
            raise ValueError("host-side API takes CPU (optionally pinned) tensors")
        return a.data_ptr(), a
    raise TypeError(f"unsupported buffer type {type(a)}")


class Matcher:
    """One context = one GPU: packed descriptor table in HBM + the batched pair matcher."""

    def __init__(self, device: int = 0, max_images: int = 1024, arena_rows: int = 1 << 20, external_desc_arena: int = 0,
                 external_norm_arena: int = 0, keep_float: bool = False):
        self._L = _lib.load()
        cfg = Config()
        cfg.device = device
        cfg.max_images = max_images
        cfg.arena_rows = arena_rows
        cfg.external_desc_arena = external_desc_arena or None
        cfg.external_norm_arena = external_norm_arena or None
        cfg.keep_float = int(bool(keep_float))  # float uploads are retained for fp32 re-scoring (rescore_band)
        h = C.c_void_p()
        st = self._L.msfm_create(C.byref(cfg), C.byref(h))
        if st != _lib.MSFM_OK:
            raise MsfmError(st, self._L.msfm_status_string(st).decode())
        self._h = h
        self.device = device
        self._inflight = None  # host buffers of an upload_batch(wait=False) still being copied

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None):
            self._L.msfm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, st: int):
        if st != _lib.MSFM_OK:
            raise MsfmError(st, self._L.msfm_last_error(self._h).decode())

    # ------------------------------------------------------------------ descriptor table
    def upload(self, image_id: int, desc, scale: float = 1.0) -> None:
        """Pack one image's descriptors into HBM, once.  uint8 rows are taken as they are; float32 rows are quantised
        q = min(255, max(0, rint(x * scale))) (scale 1 for 512-scaled VLSIFT rows, 512 for unit-norm rows)."""
        if hasattr(desc, "numpy") and not isinstance(desc, np.ndarray):
            dtype = str(desc.dtype).replace("torch.", "")
            shape, strides = tuple(desc.shape), tuple(s * desc.element_size() for s in desc.stride())
        else:
            desc = np.asarray(desc)
            dtype, shape, strides = str(desc.dtype), desc.shape, desc.strides
        if len(shape) != 2 or (shape[0] > 0 and shape[1] != 128):
            raise ValueError(f"descriptors must be [rows, 128], got {shape}")
        rows = int(shape[0])
        ptr, keep = _host_ptr(desc)
        if dtype == "uint8":
            if rows and strides[1] != 1:
                raise ValueError("descriptor rows must be contiguous")
            self._check(self._L.msfm_upload_u8(self._h, image_id, ptr, rows, strides[0] if rows else 128))
        elif dtype == "float32":
            if rows and strides[1] != 4:
                raise ValueError("descriptor rows must be contiguous")
            self._check(self._L.msfm_upload_f32(self._h, image_id, ptr, rows, (strides[0] // 4) if rows else 128, scale))
        else:
            raise TypeError(f"descriptors must be uint8 or float32, got {dtype}")
        del keep

    def upload_batch(self, image_ids, descs, wait: bool = True) -> None:
        """Pack several uint8 images in one call (one host wait for the whole batch instead of one per image).
        wait=False (msfm_upload_u8_batch_async): no host wait at all -- the copies run while the host goes on; the
        buffers (page-locked, contiguous rows) must stay valid and unchanged until sync() or the next call that returns
        results."""
        n = len(image_ids)
        ids = np.ascontiguousarray(image_ids, np.int32)
        ptrs = (C.c_void_p * max(n, 1))()
        rows = np.zeros((max(n, 1),), np.int32)
        strides = np.full((max(n, 1),), 128, np.int64)
        keep = []
        for k, d in enumerate(descs):
            if hasattr(d, "numpy") and not isinstance(d, np.ndarray):
                if str(d.dtype) != "torch.uint8" or d.dim() != 2 or (d.shape[0] and d.shape[1] != 128) or (d.shape[0] and d.stride(1) != 1):
                    raise ValueError("upload_batch takes [rows, 128] uint8 descriptors with contiguous rows")
                rows[k], strides[k] = d.shape[0], d.stride(0) if d.shape[0] else 128
            else:
                d = np.asarray(d)
                if d.dtype != np.uint8 or d.ndim != 2 or (d.shape[0] and d.shape[1] != 128) or (d.shape[0] and d.strides[1] != 1):
                    raise ValueError("upload_batch takes [rows, 128] uint8 descriptors with contiguous rows")
                rows[k], strides[k] = d.shape[0], d.strides[0] if d.shape[0] else 128
            ptr, ka = _host_ptr(d)
            ptrs[k] = ptr
            keep.append(ka)
        fn = self._L.msfm_upload_u8_batch if wait else self._L.msfm_upload_u8_batch_async
        self._check(fn(self._h, n, ids.ctypes.data, C.cast(ptrs, C.c_void_p), rows.ctypes.data, strides.ctypes.data))
        if not wait:
            self._inflight = (self._inflight or []) + keep  # host buffers stay alive until sync() / release_all()
        del keep

    def upload_f32_batch_async(self, image_ids, descs, scale: float = 1.0) -> None:
        """msfm_upload_f32_batch_async: several float32 [rows, 128] images (dense rows, page-locked memory) without a host
        wait; the buffers must stay valid and unchanged until sync()."""
        n = len(image_ids)
        ids = np.ascontiguousarray(image_ids, np.int32)
        ptrs = (C.c_void_p * max(n, 1))()
        rows = np.zeros((max(n, 1),), np.int32)
        keep = []
        for k, d in enumerate(descs):
            is_t = hasattr(d, "numpy") and not isinstance(d, np.ndarray)
            if not is_t:
                d = np.asarray(d)
            dt = str(d.dtype).replace("torch.", "")
            dense = d.is_contiguous() if is_t else d.flags["C_CONTIGUOUS"]
            if dt != "float32" or len(d.shape) != 2 or (d.shape[0] and d.shape[1] != 128) or not dense:
                raise ValueError("upload_f32_batch_async takes dense [rows, 128] float32 descriptors")
            rows[k] = d.shape[0]
            ptr, ka = _host_ptr(d)
            ptrs[k] = ptr
            keep.append(ka)
        self._check(self._L.msfm_upload_f32_batch_async(self._h, n, ids.ctypes.data, C.cast(ptrs, C.c_void_p), rows.ctypes.data, scale))
        self._inflight = (self._inflight or []) + keep

    def sync(self) -> None:
        self._check(self._L.msfm_sync(self._h))
        self._inflight = None

    def reserve(self, image_id: int, rows: int) -> int:
        off = C.c_int64()
        self._check(self._L.msfm_reserve(self._h, image_id, rows, C.byref(off)))
        return off.value

    def reserve_batch(self, image_ids, rows, wait: bool = True) -> np.ndarray:
        """msfm_reserve for several images in one call; returns their row offsets.  wait=False
        (msfm_reserve_batch_async): pad rows / tensor maps are only queued on the upload stream."""
        ids = np.ascontiguousarray(image_ids, np.int32)
        r = np.ascontiguousarray(rows, np.int32)
        if ids.shape != r.shape:
            raise ValueError("image_ids and rows must have the same length")
        offs = np.zeros(ids.shape, np.int64)
        fn = self._L.msfm_reserve_batch if wait else self._L.msfm_reserve_batch_async
        self._check(fn(self._h, len(ids), ids.ctypes.data, r.ctypes.data, offs.ctypes.data))
        return offs

    def release(self, image_id: int) -> None:
        self._check(self._L.msfm_release(self._h, image_id))

    def release_all(self) -> None:
        self._check(self._L.msfm_release_all(self._h))   # synchronises both streams
        self._inflight = None

    def image_info(self, image_id: int):
        rows, off = C.c_int32(), C.c_int64()
        self._check(self._L.msfm_image_info(self._h, image_id, C.byref(rows), C.byref(off)))
        return rows.value, off.value

    def table_ptrs(self):
        d, n, ar, used = C.c_void_p(), C.c_void_p(), C.c_int64(), C.c_int64()
        self._check(self._L.msfm_table_ptrs(self._h, C.byref(d), C.byref(n), C.byref(ar), C.byref(used)))
        return d.value, n.value, ar.value, used.value

    def download_packed(self, image_id: int):
        rows, _ = self.image_info(image_id)
        desc = np.empty((rows, 128), dtype=np.uint8)
        norms = np.empty((rows,), dtype=np.uint32)
        self._check(self._L.msfm_download_packed(self._h, image_id, desc.ctypes.data, norms.ctypes.data))
        return desc, norms

    # ------------------------------------------------------------------ kNN (FLANN layout)
    def knn2(self, ref_id: int, query_id: int):
        n, _ = self.image_info(query_id)
        ids = np.empty((n, 2), dtype=np.int32)
        dists = np.empty((n, 2), dtype=np.float32)
        self._check(self._L.msfm_knn2(self._h, ref_id, query_id, ids.ctypes.data, dists.ctypes.data))
        return ids, dists

    def knn2_pairs(self, pairs, exact_f32: bool = False):
        """msfm_knn2_pairs: FLANN-layout 2-NN of every query row of every pair in one call.  Returns (offsets [n+1] int64,
        ids [rows, 2] int32, dists [rows, 2] float32); pair p owns rows offsets[p]:offsets[p+1].  exact_f32: neighbours and
        distances of an exhaustive fp32 matcher on the retained float rows (float uploads on a keep_float context, one
        scale per pair); otherwise the integer distances of msfm_knn2."""
        pa = self._pairs(pairs)
        n = pa.shape[0]
        rows_cache = {}
        total = 0
        for q in pa[:, 1]:
            q = int(q)
            if q not in rows_cache:
                rows_cache[q] = self.image_info(q)[0]
            total += rows_cache[q]
        offsets = np.zeros((n + 1,), np.int64)
        ids = np.empty((max(total, 1), 2), np.int32)
        dists = np.empty((max(total, 1), 2), np.float32)
        flags = _lib.KNN_EXACT_F32 if exact_f32 else 0
        self._check(self._L.msfm_knn2_pairs(self._h, pa.ctypes.data, n, flags, offsets.ctypes.data, ids.ctypes.data,
                                            dists.ctypes.data, total))
        return offsets, ids[:total], dists[:total]

    def _test_last_knn_stats(self):
        """(events scored by the collect path, batches decided by the brute force) of the last exact knn2_pairs call or
        re-scoring match_pairs / match_pairs_guided / match_pairs_guided_homography call (rescore_band > 0 on a
        keep_float context)."""
        ev, bf = C.c_int64(), C.c_int32()
        self._check(self._L.msfm_test_last_knn_stats(self._h, C.byref(ev), C.byref(bf)))
        return ev.value, bf.value

    def knn2_crosscheck(self, ref_id: int, query_id: int):
        n, _ = self.image_info(query_id)
        ids = np.empty((n, 2), dtype=np.int32)
        dists = np.empty((n, 2), dtype=np.float32)
        self._check(self._L.msfm_knn2_crosscheck(self._h, ref_id, query_id, ids.ctypes.data, dists.ctypes.data))
        return ids, dists

    def colbest(self, ref_id: int, query_id: int):
        m, _ = self.image_info(ref_id)
        best = np.empty((m,), dtype=np.int32)
        dist = np.empty((m,), dtype=np.float32)
        self._check(self._L.msfm_colbest(self._h, ref_id, query_id, best.ctypes.data, dist.ctypes.data))
        return best, dist

    # ------------------------------------------------------------------ batched pair matching
    @staticmethod
    def _params(ratio, ratio_good, max_dist_sq, mutual, min_keypoints, orientation, rescore_band=0.0, flags=0) -> Params:
        p = Params()
        p.rescore_band = rescore_band
        p.flags = int(flags)
        p.ratio, p.ratio_good, p.max_dist_sq = ratio, ratio_good, max_dist_sq
        p.mutual, p.min_keypoints, p.orientation = int(bool(mutual)), int(min_keypoints), int(orientation)
        return p

    @staticmethod
    def _pairs(pairs) -> np.ndarray:
        a = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        return a

    def match_pairs(self, pairs, ratio: float = 0.6, *, ratio_good: float = 0.0, max_dist_sq: float = 0.0, mutual: bool = False,
                    min_keypoints: int = 20, orientation: int = 0, capacity: int | None = None, out: MatchResult | None = None,
                    rescore_band: float = 0.0, flags: int = 0) -> MatchResult:
        """pairs: [n, 2] (ref image, query image).  Returns per-pair match lists, ascending query index.
        rescore_band > 0 (float uploads on a keep_float context): rows whose quantised ratio lies within that relative
        band of a threshold are decided on exact fp32 distances."""
        pa = self._pairs(pairs)
        n = pa.shape[0]
        out, res = self._result_buffers(pa, ratio_good, capacity, out)
        prm = self._params(ratio, ratio_good, max_dist_sq, mutual, min_keypoints, orientation, rescore_band, flags)
        self._check(self._L.msfm_match_pairs(self._h, pa.ctypes.data, n, C.byref(prm), C.byref(res)))
        total = int(out.offsets[n])
        return MatchResult(out.offsets, out.ok, out.matches[:total], out.good[:total] if out.good is not None else None)

    def _result_buffers(self, pa: np.ndarray, ratio_good: float, capacity: int | None, out: MatchResult | None):
        """(MatchResult, msfm_result) over the caller's `out` or new buffers with room for one match per query row."""
        n = pa.shape[0]
        if out is None:
            if capacity is None:
                capacity = 0
                rows_cache = {}
                for q in pa[:, 1]:
                    q = int(q)
                    if q not in rows_cache:
                        rows_cache[q] = self.image_info(q)[0]
                    capacity += rows_cache[q]
            out = MatchResult(offsets=np.zeros((n + 1,), np.int64), ok=np.zeros((n,), np.int32),
                              matches=np.empty((max(capacity, 1), 2), np.int32),
                              good=np.zeros((max(capacity, 1),), np.uint8) if ratio_good > 0 else None)
        res = Result()
        res.offsets = out.offsets.ctypes.data_as(_lib._i64p)
        res.ok = out.ok.ctypes.data_as(_lib._i32p)
        res.matches = _host_ptr(out.matches)[0]
        res.good = out.good.ctypes.data_as(_lib._u8p) if out.good is not None else None
        res.match_capacity = out.matches.shape[0]
        return out, res

    @staticmethod
    def _keypoint_table(image_xy: dict, n_images: int):
        """(pointer array, point counts, keepalive) of {image id: [n, 2] float32 keypoints} for ids < n_images."""
        xy_keep, ptrs, npts = [], (C.c_void_p * max(n_images, 1))(), np.zeros((max(n_images, 1),), np.int32)
        for i, xy in image_xy.items():
            if i < n_images:
                a = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
                xy_keep.append(a)
                ptrs[i] = a.ctypes.data
                npts[i] = a.shape[0]
        return ptrs, npts, xy_keep

    def match_pairs_guided(self, pairs, F, image_xy: dict, *, th_epipolar: float = 3.0, ratio: float = 0.6,
                           ratio_good: float = 0.0, max_dist_sq: float = 0.0, mutual: bool = False, min_keypoints: int = 20,
                           orientation: int = 0, flags: int = 0, rescore_band: float = 0.0,
                           capacity: int | None = None) -> MatchResult:
        """msfm_match_pairs_guided (GUIDED-SPEC in include/msfm_match.h): match_pairs with every query row's 2-NN searched
        only among the reference keypoints within th_epipolar pixels of the pair's epipolar geometry.  F: [n, 3, 3]
        float64 as geo_verify returns it (p_query^T F p_ref = 0); image_xy: {image id: [rows, 2] float32 centred
        keypoints}, one per descriptor row of every image the pairs touch.  rescore_band > 0 (float uploads on a
        keep_float context): rows whose gated quantised ratio lies within that relative band of a ratio threshold are
        decided on their exact fp32 top-2 among the allowed reference rows, as match_pairs does without a gate."""
        prm = self._params(ratio, ratio_good, max_dist_sq, mutual, min_keypoints, orientation, rescore_band, flags)
        return self._match_guided(self._L.msfm_match_pairs_guided, pairs, F, image_xy, th_epipolar, prm, ratio_good, capacity)

    def _match_guided(self, fn, pairs, M, image_xy, th, prm, ratio_good, capacity) -> MatchResult:
        pa = self._pairs(pairs)
        n = pa.shape[0]
        Fa = np.ascontiguousarray(M, np.float64).reshape(-1, 9)
        if Fa.shape[0] != n:
            raise ValueError(f"one 3x3 matrix per pair is needed: {Fa.shape[0]} for {n} pairs")
        n_images = int(pa.max()) + 1 if n else 0
        ptrs, npts, xy_keep = self._keypoint_table(image_xy, n_images)
        out, res = self._result_buffers(pa, ratio_good, capacity, None)
        self._check(fn(self._h, pa.ctypes.data, n, C.byref(prm), Fa.ctypes.data, th, C.cast(ptrs, C.c_void_p), npts.ctypes.data,
                       n_images, C.byref(res)))
        del xy_keep
        total = int(out.offsets[n])
        return MatchResult(out.offsets, out.ok, out.matches[:total], out.good[:total] if out.good is not None else None)

    def match_pairs_guided_homography(self, pairs, H, image_xy: dict, *, th_transfer: float = 3.0, ratio: float = 0.6,
                                      ratio_good: float = 0.0, max_dist_sq: float = 0.0, mutual: bool = False,
                                      min_keypoints: int = 20, orientation: int = 0, flags: int = 0,
                                      rescore_band: float = 0.0, capacity: int | None = None) -> MatchResult:
        """msfm_match_pairs_guided_homography (HOMOG-SPEC in include/msfm_match.h): match_pairs with every query row's 2-NN
        searched only among the reference keypoints that H carries to within th_transfer pixels of the row's keypoint.
        H: [n, 3, 3] float64 as geo_homography returns it (p_query ~ H p_ref); image_xy as in match_pairs_guided.
        rescore_band > 0 (float uploads on a keep_float context): rows whose gated quantised ratio lies within that
        relative band of a ratio threshold are decided on their exact fp32 top-2 among the reference rows H allows, as
        match_pairs_guided does under F."""
        prm = self._params(ratio, ratio_good, max_dist_sq, mutual, min_keypoints, orientation, rescore_band, flags)
        return self._match_guided(self._L.msfm_match_pairs_guided_homography, pairs, H, image_xy, th_transfer, prm, ratio_good,
                                  capacity)

    def match_pairs_resident(self, pairs, ratio: float = 0.6, *, ratio_good: float = 0.0, max_dist_sq: float = 0.0,
                             mutual: bool = False, min_keypoints: int = 20, orientation: int = 0) -> int:
        """Same device work, results left in HBM; returns the total match count."""
        pa = self._pairs(pairs)
        prm = self._params(ratio, ratio_good, max_dist_sq, mutual, min_keypoints, orientation)
        total = C.c_int64()
        self._check(self._L.msfm_match_pairs_resident(self._h, pa.ctypes.data, pa.shape[0], C.byref(prm), C.byref(total)))
        return total.value

    def geo_verify(self, pairs, result: "MatchResult", image_xy: dict, *, th_epipolar: float = 3.0, min_points: int = 30,
                   min_inliers: int = 30, iters: int = 1024, seed: int = 0, ransac_only: bool = False,
                   pair_index_base: int = 0):
        """Batched GeoVerificationFundamental (utils/geo_verification.cc:30-79) of the pairs of a match_pairs result
        (orientation 0, ratio_good set).  image_xy: {image id: [n, 2] float32 centred keypoints}.  Returns
        (pair_ok [n] int32, pair_inliers [n] int32, keep [total] uint8, F [n, 3, 3] float64).  ransac_only: msfm_geo_ransac —
        `result.good` selects the participating matches and `keep` is the RANSAC consensus mask instead of the F-filter.
        pair_index_base: global index of the first pair in the RANSAC counter, so that a pair list verified in slices
        draws the same hypotheses as in one call."""
        fn = self._L.msfm_geo_ransac if ransac_only else self._L.msfm_geo_verify
        return self._geo_call(fn, pairs, result, image_xy, th_epipolar, min_points, min_inliers, iters, seed, pair_index_base)

    def geo_homography(self, pairs, result: "MatchResult", image_xy: dict, *, th: float = 3.0, min_points: int = 30,
                       min_inliers: int = 30, iters: int = 1024, seed: int = 0, pair_index_base: int = 0):
        """msfm_geo_homography: batched RANSAC homography (p_query ~ H p_ref, cv::findHomography(RANSAC, th) without the
        refinement) of the pairs of a match_pairs result (orientation 0); `result.good` selects the participating matches,
        as geo_verify(ransac_only=True) does.  Returns (pair_ok [n] int32, pair_inliers [n] int32, inlier_mask [total]
        uint8, H [n, 3, 3] float64, H22 = 1)."""
        return self._geo_call(self._L.msfm_geo_homography, pairs, result, image_xy, th, min_points, min_inliers, iters, seed,
                              pair_index_base)

    def _geo_call(self, fn, pairs, result, image_xy, th, min_points, min_inliers, iters, seed, pair_index_base):
        pa = self._pairs(pairs)
        n = pa.shape[0]
        n_images = int(pa.max()) + 1 if n else 0
        ptrs, npts, xy_keep = self._keypoint_table(image_xy, n_images)
        gp = _lib.GeoParams(th, min_points, min_inliers, iters, seed, pair_index_base)
        total = int(result.offsets[n])
        ok = np.zeros((max(n, 1),), np.int32)
        inl = np.zeros((max(n, 1),), np.int32)
        keep = np.zeros((max(total, 1),), np.uint8)
        F = np.zeros((max(n, 1), 3, 3), np.float64)
        offs = np.ascontiguousarray(result.offsets, np.int64)
        m = np.ascontiguousarray(result.matches, np.int32)
        g = np.ascontiguousarray(result.good if result.good is not None else np.ones((total,), np.uint8), np.uint8)
        self._check(fn(self._h, pa.ctypes.data, n, offs.ctypes.data, m.ctypes.data if total else None,
                                            g.ctypes.data if total else None, C.cast(ptrs, C.c_void_p), npts.ctypes.data, n_images,
                                            C.byref(gp), ok.ctypes.data, inl.ctypes.data, keep.ctypes.data, F.ctypes.data)
                    )
        return ok[:n], inl[:n], keep[:total], F[:n]

    def cuda_stream(self) -> int:
        """Raw cudaStream_t of this context (wrap with torch.cuda.ExternalStream to record events on it)."""
        s = C.c_void_p()
        self._check(self._L.msfm_get_stream(self._h, C.byref(s)))
        return s.value or 0

    def upload_stream(self) -> int:
        """Raw cudaStream_t the table uploads run on."""
        s = C.c_void_p()
        self._check(self._L.msfm_get_upload_stream(self._h, C.byref(s)))
        return s.value or 0

    def wait_event(self, cuda_event: int) -> None:
        """Later matching launches wait (on the device) for this cudaEvent_t, e.g. torch.cuda.Event.cuda_event."""
        self._check(self._L.msfm_wait_event(self._h, C.c_void_p(cuda_event)))

    def _test_set_band_event_cap(self, cap: int) -> None:
        self._check(self._L.msfm_test_set_band_event_cap(self._h, cap))

    def _test_force_twin_pass(self, on: bool) -> None:
        self._check(self._L.msfm_test_force_twin_pass(self._h, int(bool(on))))

    def _test_disable_pruning(self, on: bool) -> None:
        self._check(self._L.msfm_test_disable_pruning(self._h, int(bool(on))))

    def timing(self) -> dict:
        t = Timing()
        self._check(self._L.msfm_last_timing(self._h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in Timing._fields_}

    # ------------------------------------------------------------------ reference-shaped single-pair entry points
    def KNNMatching(self, id1: int, id2: int, *, th_ratio: float = 0.5, th_reject: int = 20, mutual: bool = False):
        """FeatureMatching::KNNMatching (feature_matching.cpp:24-65): index on image 2, queries = rows of image 1,
        ratio < 0.5, emits (i1, i2) ascending i1.  Returns (ok, matches[n,2])."""
        r = self.match_pairs([(id2, id1)], th_ratio, mutual=mutual, min_keypoints=th_reject, orientation=1)
        return bool(r.ok[0]), r.pair(0).copy()

    def SLAMFeatureMatching(self, id1: int, id2: int, *, th_first_second_ratio: float = 0.8):
        """SLAMGPS::FeatureMatching kNN + ratio part (slam_gps.cc:438-477): index on id1, queries = rows of id2, a row is
        rejected iff ratio > th (non-strict; 0/0 = NaN passes), no keypoint gate.  Returns matches [(i1, i2)] ascending i2."""
        r = self.match_pairs([(id1, id2)], th_first_second_ratio, min_keypoints=0, orientation=0, flags=_lib.RATIO_REJECT_GT)
        return r.pair(0).copy()

    def MatchAgainstIndex(self, idx1: int, idx2: int, *, th_ratio: float = 0.5, th_reject: int = 20, mutual: bool = False):
        """KNNMatchingWithGeoVerify(kp1, kd_tree1, kp2, descriptors2, matches) kNN + ratio part
        (feature_matching.cpp:319-350) and the per-partner body of fine_matching_graph.cc:104-133: index on idx1,
        queries = rows of idx2, emits (i1, i2) ascending i2."""
        r = self.match_pairs([(idx1, idx2)], th_ratio, mutual=mutual, min_keypoints=th_reject, orientation=0)
        return bool(r.ok[0]), r.pair(0).copy()
