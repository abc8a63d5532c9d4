"""ctypes binding of include/msfm_match.h.  Loading fails loudly when the CUDA library has not been built —
there is no CPU or PyTorch fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH, SCHED_LIB

_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_f32p = C.POINTER(C.c_float)
_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)

MSFM_OK = 0
STATUS_NAMES = {
    0: "MSFM_OK", 1: "MSFM_ERR_INVALID_ARG", 2: "MSFM_ERR_CUDA", 3: "MSFM_ERR_OUT_OF_MEMORY", 4: "MSFM_ERR_NOT_FOUND",
    5: "MSFM_ERR_CAPACITY", 6: "MSFM_ERR_UNSUPPORTED", 7: "MSFM_ERR_EXISTS",
}

# Every symbol include/msfm_match.h declares (tests/test_abi.py checks the two lists against each other).
EXPORTED_SYMBOLS = [
    "msfm_abi_version", "msfm_status_string", "msfm_create", "msfm_destroy", "msfm_last_error", "msfm_upload_u8",
    "msfm_upload_u8_batch", "msfm_upload_u8_batch_async", "msfm_sync", "msfm_upload_f32", "msfm_reserve", "msfm_reserve_batch", "msfm_release", "msfm_release_all", "msfm_image_info", "msfm_table_ptrs",
    "msfm_download_packed", "msfm_knn2", "msfm_colbest", "msfm_match_pairs", "msfm_match_pairs_resident",
    "msfm_last_timing", "msfm_get_stream", "msfm_knn2_crosscheck", "msfm_geo_verify", "msfm_geo_ransac",
    "msfm_upload_f32_batch_async", "msfm_get_upload_stream", "msfm_wait_event", "msfm_test_set_band_event_cap", "msfm_test_force_twin_pass", "msfm_test_disable_pruning", "msfm_reserve_batch_async", "msfm_host_alloc", "msfm_host_free", "msfm_device_memory",
    "msfm_knn2_pairs", "msfm_test_last_knn_stats", "msfm_match_pairs_guided", "msfm_geo_homography",
    "msfm_match_pairs_guided_homography",
]


# include/msfm_sched.h and include/msfm_multi.h (same library)
SCHED_SYMBOLS = ["msfm_sched_shard", "msfm_sched_image_owner", "msfm_sched_offsets", "msfm_sched_scatter"]
MULTI_SYMBOLS = [
    "msfm_multi_create", "msfm_multi_destroy", "msfm_multi_last_error", "msfm_multi_device_count", "msfm_multi_context",
    "msfm_multi_upload_u8", "msfm_multi_upload_f32", "msfm_multi_release_all", "msfm_multi_sync", "msfm_multi_match_pairs",
    "msfm_multi_last_timing",
]


class MultiConfig(C.Structure):
    _fields_ = [("n_devices", C.c_int32), ("devices", C.POINTER(C.c_int32)), ("max_images", C.c_int32), ("arena_rows", C.c_int64),
                ("reserved", C.c_int32 * 4)]


class MultiTiming(C.Structure):
    _fields_ = [("wall_ms", C.c_float), ("device_ms_max", C.c_float), ("stitch_ms", C.c_float), ("n_devices", C.c_int32),
                ("int8_ops", C.c_int64), ("bytes_broadcast", C.c_int64)]


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_images", C.c_int32), ("arena_rows", C.c_int64),
                ("external_desc_arena", C.c_void_p), ("external_norm_arena", C.c_void_p), ("keep_float", C.c_int32),
                ("reserved", C.c_int32 * 3)]


class Params(C.Structure):
    _fields_ = [("ratio", C.c_float), ("ratio_good", C.c_float), ("max_dist_sq", C.c_float), ("mutual", C.c_int32),
                ("min_keypoints", C.c_int32), ("orientation", C.c_int32), ("rescore_band", C.c_float), ("flags", C.c_uint32)]


RATIO_REJECT_GT = 1  # msfm_params.flags: SLAMGPS::FeatureMatching's rule (slam_gps.cc:470-477)
KNN_EXACT_F32 = 1    # msfm_knn2_pairs flag: fp32 neighbours and distances of the retained float rows


class GeoParams(C.Structure):
    _fields_ = [("th_epipolar", C.c_float), ("min_points", C.c_int32), ("min_inliers", C.c_int32), ("iters", C.c_int32),
                ("seed", C.c_uint64), ("pair_index_base", C.c_int64)]


class Pair(C.Structure):
    _fields_ = [("ref", C.c_int32), ("query", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("offsets", _i64p), ("ok", _i32p), ("matches", C.c_void_p), ("good", _u8p), ("match_capacity", C.c_int64)]


class Timing(C.Structure):
    _fields_ = [("total_ms", C.c_float), ("match_kernel_ms", C.c_float), ("finalize_ms", C.c_float), ("d2h_ms", C.c_float),
                ("match_launches", C.c_int32), ("total_launches", C.c_int32), ("d2h_bytes", C.c_int64), ("int8_ops", C.c_int64),
                ("twin_pairs", C.c_int32), ("reserved", C.c_int32)]


_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree CUDA library; raise if it is missing (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA extension has not been built (run `python -m metricsfm_b200.build`). "
            "metricsfm_b200 has no CPU fallback by design.")
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.msfm_abi_version.restype = C.c_int32
    L.msfm_status_string.restype = C.c_char_p
    L.msfm_status_string.argtypes = [C.c_int]
    L.msfm_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.msfm_destroy.argtypes = [vp]
    L.msfm_last_error.restype = C.c_char_p
    L.msfm_last_error.argtypes = [vp]
    L.msfm_upload_u8.argtypes = [vp, C.c_int32, vp, C.c_int32, C.c_int64]
    L.msfm_upload_u8_batch.argtypes = [vp, C.c_int32, vp, vp, vp, vp]
    L.msfm_upload_u8_batch_async.argtypes = [vp, C.c_int32, vp, vp, vp, vp]
    L.msfm_sync.argtypes = [vp]
    L.msfm_upload_f32.argtypes = [vp, C.c_int32, vp, C.c_int32, C.c_int64, C.c_float]
    L.msfm_reserve.argtypes = [vp, C.c_int32, C.c_int32, _i64p]
    L.msfm_reserve_batch.argtypes = [vp, C.c_int32, vp, vp, vp]
    L.msfm_reserve_batch_async.argtypes = [vp, C.c_int32, vp, vp, vp]
    L.msfm_release.argtypes = [vp, C.c_int32]
    L.msfm_release_all.argtypes = [vp]
    L.msfm_image_info.argtypes = [vp, C.c_int32, _i32p, _i64p]
    L.msfm_table_ptrs.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), _i64p, _i64p]
    L.msfm_download_packed.argtypes = [vp, C.c_int32, vp, vp]
    L.msfm_knn2.argtypes = [vp, C.c_int32, C.c_int32, vp, vp]
    L.msfm_knn2_pairs.argtypes = [vp, vp, C.c_int64, C.c_uint32, vp, vp, vp, C.c_int64]
    L.msfm_test_last_knn_stats.argtypes = [vp, _i64p, _i32p]
    L.msfm_colbest.argtypes = [vp, C.c_int32, C.c_int32, vp, vp]
    L.msfm_match_pairs.argtypes = [vp, vp, C.c_int64, C.POINTER(Params), C.POINTER(Result)]
    L.msfm_match_pairs_guided.argtypes = [vp, vp, C.c_int64, C.POINTER(Params), vp, C.c_float, vp, vp, C.c_int32,
                                          C.POINTER(Result)]
    L.msfm_match_pairs_guided_homography.argtypes = L.msfm_match_pairs_guided.argtypes
    L.msfm_match_pairs_resident.argtypes = [vp, vp, C.c_int64, C.POINTER(Params), _i64p]
    L.msfm_last_timing.argtypes = [vp, C.POINTER(Timing)]
    L.msfm_get_stream.argtypes = [vp, C.POINTER(vp)]
    L.msfm_get_upload_stream.argtypes = [vp, C.POINTER(vp)]
    L.msfm_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.msfm_host_free.argtypes = [vp]
    L.msfm_device_memory.argtypes = [C.c_int32, _i64p, _i64p]
    L.msfm_wait_event.argtypes = [vp, vp]
    L.msfm_test_set_band_event_cap.argtypes = [vp, C.c_int64]
    L.msfm_test_force_twin_pass.argtypes = [vp, C.c_int32]
    L.msfm_test_disable_pruning.argtypes = [vp, C.c_int32]
    L.msfm_upload_f32_batch_async.argtypes = [vp, C.c_int32, vp, vp, vp, C.c_float]
    L.msfm_knn2_crosscheck.argtypes = [vp, C.c_int32, C.c_int32, vp, vp]
    L.msfm_geo_verify.argtypes = [vp, vp, C.c_int64, vp, vp, vp, vp, vp, C.c_int32, C.POINTER(GeoParams), vp, vp, vp, vp]
    L.msfm_geo_ransac.argtypes = L.msfm_geo_verify.argtypes
    L.msfm_geo_homography.argtypes = L.msfm_geo_verify.argtypes
    for name in EXPORTED_SYMBOLS:
        fn = getattr(L, name)
        if name not in ("msfm_abi_version", "msfm_status_string", "msfm_last_error"):
            fn.restype = C.c_int
    _declare_sched(L)
    L.msfm_multi_create.argtypes = [C.POINTER(MultiConfig), C.POINTER(vp)]
    L.msfm_multi_destroy.argtypes = [vp]
    L.msfm_multi_last_error.argtypes = [vp]
    L.msfm_multi_last_error.restype = C.c_char_p
    L.msfm_multi_device_count.argtypes = [vp]
    L.msfm_multi_device_count.restype = C.c_int32
    L.msfm_multi_context.argtypes = [vp, C.c_int32]
    L.msfm_multi_context.restype = vp
    L.msfm_multi_upload_u8.argtypes = [vp, C.c_int32, vp, vp, vp]
    L.msfm_multi_upload_f32.argtypes = [vp, C.c_int32, vp, vp, vp, C.c_float]
    L.msfm_multi_release_all.argtypes = [vp]
    L.msfm_multi_sync.argtypes = [vp]
    L.msfm_multi_match_pairs.argtypes = [vp, vp, C.c_int64, C.POINTER(Params), C.POINTER(Result)]
    L.msfm_multi_last_timing.argtypes = [vp, C.POINTER(MultiTiming), vp]
    for name in MULTI_SYMBOLS:
        if name not in ("msfm_multi_last_error", "msfm_multi_device_count", "msfm_multi_context"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def _declare_sched(L) -> None:
    vp = C.c_void_p
    L.msfm_sched_shard.argtypes = [vp, C.c_int64, vp, C.c_int32, C.c_int32, vp, vp]
    L.msfm_sched_shard.restype = C.c_int
    L.msfm_sched_image_owner.argtypes = [C.c_int32, C.c_int32, vp]
    L.msfm_sched_image_owner.restype = C.c_int
    L.msfm_sched_offsets.argtypes = [vp, C.c_int64, vp]
    L.msfm_sched_offsets.restype = C.c_int64
    L.msfm_sched_scatter.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp, vp]
    L.msfm_sched_scatter.restype = C.c_int


_sched = None


def load_sched() -> C.CDLL:
    """The pair scheduler's host logic (include/msfm_sched.h) from the host-only libmsfm_sched.so: usable by launchers and
    CPU tests that never touch a GPU.  The same code is linked into libmsfm_match.so."""
    global _sched
    if _sched is None:
        if not os.path.exists(SCHED_LIB):
            raise RuntimeError(f"{SCHED_LIB} not found: run `python -m metricsfm_b200.build`")
        _sched = C.CDLL(SCHED_LIB)
        _declare_sched(_sched)
    return _sched
