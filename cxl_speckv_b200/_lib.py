"""ctypes binding of libcxlspeckv.so (include/speckv.h + include/speckv_ext.h)."""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))

SPECKV_OK, SPECKV_ERR_GENERAL, SPECKV_ERR_DRIVER, SPECKV_ERR_NOMEM, SPECKV_ERR_INVAL = 0, -1, -2, -3, -4
COMP_FP16, COMP_INT8, COMP_INT8_DELTA_RLE = 0, 1, 2
COMP_INT8_CLAMP_DELTA_RLE, COMP_INT8_CLAMP = 3, 4   # extension ids (speckv_ext.h): the non-wrapping quantiser
DTYPE_F16, DTYPE_BF16, DTYPE_F32 = 0, 1, 2

_STATUS = {0: "SPECKV_OK", -1: "SPECKV_ERR_GENERAL", -2: "SPECKV_ERR_DRIVER", -3: "SPECKV_ERR_NOMEM",
           -4: "SPECKV_ERR_INVAL"}


class SpeckvError(RuntimeError):
    def __init__(self, what: str, status: int):
        super().__init__(f"{what} failed: {_STATUS.get(status, status)}")
        self.status = status


class Stats(C.Structure):
    _fields_ = [("total_compressions", C.c_uint64), ("total_decompressions", C.c_uint64),
                ("total_translations", C.c_uint64), ("bytes_in_compress", C.c_uint64),
                ("bytes_out_decompress", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("host_api_h2d_bytes", C.c_uint64), ("host_api_d2h_bytes", C.c_uint64)]


class TierStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("pool_bytes", "used_bytes", "blocks", "bytes_offloaded_raw",
                                          "bytes_offloaded_stored", "bytes_restored_raw", "bytes_restored_stored",
                                          "last_offload_stored_bytes", "last_restore_stored_bytes")] + \
               [("last_offload_ms", C.c_double), ("last_restore_ms", C.c_double)]


class PolicyStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("l1_hits", "l1_misses", "l2_hits", "l2_misses", "l3_accesses",
                                          "migrations_l1_to_l3", "migrations_l3_to_l1")] + \
               [("l1_hit_rate", C.c_double), ("l2_hit_rate", C.c_double)] + \
               [(n, C.c_uint64) for n in ("l1_pages", "l2_pages", "l3_pages")]


class EngineStats(C.Structure):
    _fields_ = [("total_compressions", C.c_uint64), ("total_decompressions", C.c_uint64),
                ("avg_compression_ratio", C.c_double), ("avg_compression_latency_ns", C.c_double),
                ("avg_decompression_latency_ns", C.c_double), ("throughput_gbps", C.c_double),
                ("compress_calls_timed", C.c_uint64), ("decompress_calls_timed", C.c_uint64),
                ("compress_ns_per_group", C.c_double), ("decompress_ns_per_group", C.c_double)]


class PrefetchStats(C.Structure):
    _fields_ = [("total_prefetches", C.c_uint64), ("successful_prefetches", C.c_uint64), ("mispredictions", C.c_uint64),
                ("hit_rate", C.c_double), ("precision", C.c_double), ("avg_prediction_latency_us", C.c_double)]


class PrefetchRequest(C.Structure):
    """PrefetchRequest, src/prefetcher/speculative_prefetcher.h:23-29 (32 bytes)."""
    _fields_ = [("virtual_addr", C.c_uint64), ("layer_id", C.c_uint32), ("predicted_token_id", C.c_uint32),
                ("confidence", C.c_float), ("reserved", C.c_uint32), ("timestamp", C.c_uint64)]


def lib_path() -> str:
    return os.environ.get("SPECKV_LIB", os.path.join(PKG, "libcxlspeckv.so"))


_LIB = None


def lib() -> C.CDLL:
    """Loads libcxlspeckv.so.  Raises if it has not been built: there is no fallback path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} not found: build it with `python -m cxl_speckv_b200.build` "
                          "(nvcc, sm_100a). The CUDA library is the product; there is no CPU fallback.")
    L = C.CDLL(path)
    vp, sz, u32p, f32p, u64p = C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(C.c_uint64)
    # frozen ABI (speckv.h)
    L.speckv_init.argtypes = [C.c_char_p]; L.speckv_init.restype = C.c_int
    L.speckv_finalize.argtypes = []; L.speckv_finalize.restype = None
    L.speckv_alloc.argtypes = [sz, vp, C.POINTER(C.c_uint64)]; L.speckv_alloc.restype = C.c_int
    L.speckv_free.argtypes = [C.c_uint64]; L.speckv_free.restype = C.c_int
    L.speckv_access.argtypes = [C.c_uint64, C.c_uint64, sz, C.POINTER(vp)]; L.speckv_access.restype = C.c_int
    L.speckv_prefetch.argtypes = [C.c_uint32, C.c_uint16, C.c_uint32, C.c_uint32, C.POINTER(C.c_int32), C.c_uint32]
    L.speckv_prefetch.restype = C.c_int
    L.speckv_set_prefetch_depth.argtypes = [C.c_uint32]; L.speckv_set_prefetch_depth.restype = C.c_int
    L.speckv_set_compression_scheme.argtypes = [C.c_int]; L.speckv_set_compression_scheme.restype = C.c_int
    # additive ABI (speckv_ext.h)
    L.speckv_ext_device_count.argtypes = []; L.speckv_ext_device_count.restype = C.c_int
    L.speckv_ext_version.argtypes = []; L.speckv_ext_version.restype = C.c_char_p
    L.speckv_ext_slot_bytes.argtypes = [sz, C.c_int]; L.speckv_ext_slot_bytes.restype = sz
    L.speckv_ext_compress.argtypes = [vp, C.c_int, sz, sz, vp, sz, vp, vp, C.c_int, vp]
    L.speckv_ext_compress.restype = C.c_int
    L.speckv_ext_decompress.argtypes = [vp, sz, vp, vp, sz, sz, C.c_int, vp, vp, C.c_int, vp]
    L.speckv_ext_decompress.restype = C.c_int
    L.speckv_ext_decompress_indexed.argtypes = [vp, sz, vp, vp, vp, sz, sz, C.c_int, vp, vp, C.c_int, vp]
    L.speckv_ext_decompress_indexed.restype = C.c_int
    L.speckv_ext_compress_gather.argtypes = [vp, vp, C.c_int, sz, sz, vp, sz, vp, vp, C.c_int, vp]
    L.speckv_ext_compress_gather.restype = C.c_int
    L.speckv_ext_decompress_scatter.argtypes = [vp, sz, vp, vp, vp, vp, sz, sz, C.c_int, vp, vp, C.c_int, vp]
    L.speckv_ext_decompress_scatter.restype = C.c_int
    L.speckv_ext_compress_ragged.argtypes = [vp, vp, vp, C.c_int, sz, sz, vp, sz, vp, vp, C.c_int, vp]
    L.speckv_ext_compress_ragged.restype = C.c_int
    L.speckv_ext_compress_host.argtypes = [vp, C.c_int, sz, sz, vp, sz, vp, vp, C.c_int]
    L.speckv_ext_compress_host.restype = C.c_int
    L.speckv_ext_decompress_host.argtypes = [vp, sz, vp, vp, sz, sz, C.c_int, vp, vp, C.c_int]
    L.speckv_ext_decompress_host.restype = C.c_int
    L.speckv_ext_host_alloc.argtypes = [sz]; L.speckv_ext_host_alloc.restype = vp
    L.speckv_ext_host_free.argtypes = [vp]; L.speckv_ext_host_free.restype = None
    L.speckv_ext_translate.argtypes = [vp, vp, sz, vp]; L.speckv_ext_translate.restype = C.c_int
    L.speckv_ext_page_table_export.argtypes = [C.c_uint64, vp, sz, C.POINTER(sz), vp]
    L.speckv_ext_page_table_export.restype = C.c_int
    L.speckv_ext_page_lookup.argtypes = [vp, sz, C.c_uint64, vp, vp, vp, sz, vp]
    L.speckv_ext_page_lookup.restype = C.c_int
    L.speckv_ext_memmgr_create.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(vp)]
    L.speckv_ext_memmgr_create.restype = C.c_int
    L.speckv_ext_memmgr_destroy.argtypes = [vp]; L.speckv_ext_memmgr_destroy.restype = None
    L.speckv_ext_memmgr_allocate.argtypes = [vp, C.c_uint64, C.c_uint32, C.c_int, u64p, C.POINTER(C.c_int)]
    L.speckv_ext_memmgr_allocate.restype = C.c_int
    L.speckv_ext_memmgr_deallocate.argtypes = [vp, C.c_uint64]; L.speckv_ext_memmgr_deallocate.restype = C.c_int
    L.speckv_ext_memmgr_set_tier.argtypes = [vp, C.c_uint64, sz, C.c_int]; L.speckv_ext_memmgr_set_tier.restype = C.c_int
    L.speckv_ext_memmgr_translate_host.argtypes = [vp, C.c_uint64, u64p, C.POINTER(C.c_int)]
    L.speckv_ext_memmgr_translate_host.restype = C.c_int
    L.speckv_ext_memmgr_export.argtypes = [vp, vp, sz, C.POINTER(sz), u64p, vp]
    L.speckv_ext_memmgr_export.restype = C.c_int
    L.speckv_ext_predictor_load.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
    L.speckv_ext_predictor_load.restype = C.c_int
    L.speckv_ext_predictor_unload.argtypes = []; L.speckv_ext_predictor_unload.restype = None
    L.speckv_ext_prefetch_score.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp, vp]
    L.speckv_ext_prefetch_score.restype = C.c_int
    L.speckv_ext_tier_create.argtypes = [sz, C.POINTER(vp)]; L.speckv_ext_tier_create.restype = C.c_int
    L.speckv_ext_tier_destroy.argtypes = [vp]; L.speckv_ext_tier_destroy.restype = None
    L.speckv_ext_tier_offload.argtypes = [vp, vp, C.c_int, sz, sz, vp, vp]; L.speckv_ext_tier_offload.restype = C.c_int
    L.speckv_ext_tier_restore.argtypes = [vp, vp, sz, sz, C.c_int, vp, vp]; L.speckv_ext_tier_restore.restype = C.c_int
    L.speckv_ext_tier_offload_paged.argtypes = [vp, vp, vp, C.c_int, sz, sz, vp, vp]
    L.speckv_ext_tier_offload_paged.restype = C.c_int
    L.speckv_ext_tier_restore_paged.argtypes = [vp, vp, sz, sz, C.c_int, vp, vp, vp]
    L.speckv_ext_tier_restore_paged.restype = C.c_int
    L.speckv_ext_tier_offload_ragged.argtypes = [vp, vp, vp, vp, C.c_int, sz, sz, vp, vp]
    L.speckv_ext_tier_offload_ragged.restype = C.c_int
    L.speckv_ext_tier_drop.argtypes = [vp, vp, sz]; L.speckv_ext_tier_drop.restype = C.c_int
    L.speckv_ext_tier_enable_fetch.argtypes = [vp, vp]; L.speckv_ext_tier_enable_fetch.restype = C.c_int
    L.speckv_ext_tier_fetch_workspace_bytes.argtypes = [sz, sz]; L.speckv_ext_tier_fetch_workspace_bytes.restype = sz
    L.speckv_ext_tier_fetch.argtypes = [vp, vp, vp, sz, sz, C.c_int, C.c_int, vp, vp, vp, vp, vp, sz, vp]
    L.speckv_ext_tier_fetch.restype = C.c_int
    L.speckv_ext_tier_get_stats.argtypes = [vp, C.POINTER(TierStats)]; L.speckv_ext_tier_get_stats.restype = None
    L.speckv_ext_cache_set_create.argtypes = [vp, sz, sz, sz, C.c_int, C.POINTER(vp)]
    L.speckv_ext_cache_set_create.restype = C.c_int
    L.speckv_ext_cache_set_destroy.argtypes = [vp]; L.speckv_ext_cache_set_destroy.restype = None
    L.speckv_ext_compress_gather_set.argtypes = [vp, vp, vp, vp, sz, vp, sz, vp, vp, C.c_int, vp]
    L.speckv_ext_compress_gather_set.restype = C.c_int
    L.speckv_ext_decompress_scatter_set.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp, sz, vp, C.c_int, vp]
    L.speckv_ext_decompress_scatter_set.restype = C.c_int
    L.speckv_ext_tier_offload_set.argtypes = [vp, vp, vp, vp, vp, sz, vp, vp]; L.speckv_ext_tier_offload_set.restype = C.c_int
    L.speckv_ext_tier_restore_set.argtypes = [vp, vp, sz, vp, vp, vp, vp]; L.speckv_ext_tier_restore_set.restype = C.c_int
    L.speckv_ext_tier_fetch_set.argtypes = [vp, vp, vp, sz, vp, vp, vp, C.c_int, vp, vp, vp, sz, vp]
    L.speckv_ext_tier_fetch_set.restype = C.c_int
    L.speckv_ext_atu_create.argtypes = [C.c_uint32, C.POINTER(vp)]; L.speckv_ext_atu_create.restype = C.c_int
    L.speckv_ext_atu_destroy.argtypes = [vp]; L.speckv_ext_atu_destroy.restype = None
    L.speckv_ext_atu_translate.argtypes = [vp, vp, vp, sz, vp]; L.speckv_ext_atu_translate.restype = C.c_int
    L.speckv_ext_atu_invalidate.argtypes = [vp, C.c_uint64, C.c_int, vp]; L.speckv_ext_atu_invalidate.restype = C.c_int
    L.speckv_ext_atu_get_stats.argtypes = [vp, u64p, u64p, C.c_int]; L.speckv_ext_atu_get_stats.restype = C.c_int
    L.speckv_ext_ratio_stats.argtypes = [vp, sz, sz, C.POINTER(C.c_double), C.POINTER(C.c_double), vp]
    L.speckv_ext_ratio_stats.restype = C.c_int
    L.speckv_ext_bind_pool.argtypes = [C.c_uint64, vp, sz, vp]; L.speckv_ext_bind_pool.restype = C.c_int
    L.speckv_ext_set_kv_layout.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
    L.speckv_ext_set_kv_layout.restype = C.c_int
    L.speckv_ext_offload_pages.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, vp]; L.speckv_ext_offload_pages.restype = C.c_int
    L.speckv_ext_fetch_pages.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, vp]; L.speckv_ext_fetch_pages.restype = C.c_int
    L.speckv_ext_prefetch_feedback.argtypes = [C.c_int, u32p]; L.speckv_ext_prefetch_feedback.restype = C.c_int
    L.speckv_ext_get_prefetch_depth.argtypes = [u32p]; L.speckv_ext_get_prefetch_depth.restype = C.c_int
    L.speckv_ext_submit_dma_batch.argtypes = [vp, vp, C.c_uint32, vp]; L.speckv_ext_submit_dma_batch.restype = C.c_int
    L.speckv_ext_poll_complete.argtypes = []; L.speckv_ext_poll_complete.restype = C.c_uint32
    L.speckv_ext_set_param.argtypes = [C.c_uint32, C.c_uint32]; L.speckv_ext_set_param.restype = C.c_int
    L.speckv_ext_submit_prefetch.argtypes = [C.c_void_p]; L.speckv_ext_submit_prefetch.restype = C.c_int
    L.speckv_ext_policy_create.argtypes = [C.c_uint64] * 4 + [C.POINTER(vp)]; L.speckv_ext_policy_create.restype = C.c_int
    L.speckv_ext_policy_destroy.argtypes = [vp]; L.speckv_ext_policy_destroy.restype = None
    L.speckv_ext_policy_place.argtypes = [vp, vp, sz, C.c_int, vp]; L.speckv_ext_policy_place.restype = C.c_int
    L.speckv_ext_policy_release.argtypes = [vp, vp, sz]; L.speckv_ext_policy_release.restype = C.c_int
    L.speckv_ext_policy_touch.argtypes = [vp, vp, sz, C.c_int, vp]; L.speckv_ext_policy_touch.restype = C.c_int
    L.speckv_ext_policy_is_hot.argtypes = [vp, vp, sz, vp, vp]; L.speckv_ext_policy_is_hot.restype = C.c_int
    L.speckv_ext_policy_promote.argtypes = [vp, vp, sz, vp, vp, C.POINTER(sz)]; L.speckv_ext_policy_promote.restype = C.c_int
    L.speckv_ext_policy_demote.argtypes = [vp, vp, sz, vp]; L.speckv_ext_policy_demote.restype = C.c_int
    L.speckv_ext_policy_get_tiers.argtypes = [vp, vp, sz, vp]; L.speckv_ext_policy_get_tiers.restype = C.c_int
    L.speckv_ext_policy_lru_order.argtypes = [vp, vp, sz, C.POINTER(sz)]; L.speckv_ext_policy_lru_order.restype = C.c_int
    L.speckv_ext_policy_get_stats.argtypes = [vp, C.POINTER(PolicyStats)]; L.speckv_ext_policy_get_stats.restype = C.c_int
    L.speckv_ext_decompress_routed.argtypes = [vp, sz, vp, vp, vp, vp, sz, sz, C.c_int, vp, vp, C.c_int, vp]
    L.speckv_ext_decompress_routed.restype = C.c_int
    L.speckv_ext_route_requests.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp, vp]
    L.speckv_ext_route_requests.restype = C.c_int
    L.speckv_ext_prefetch_emit.argtypes = [vp, C.c_uint32, C.c_uint32, vp, C.c_uint32, C.c_uint32, vp, sz, C.c_uint64,
                                           C.c_uint64, vp, vp, vp, vp]
    L.speckv_ext_prefetch_emit.restype = C.c_int
    L.speckv_ext_prefetch_handle_misprediction.argtypes = [C.c_uint32, u32p, sz, C.POINTER(C.c_int)]
    L.speckv_ext_prefetch_handle_misprediction.restype = C.c_int
    L.speckv_ext_prefetch_stats.argtypes = [C.POINTER(PrefetchStats), C.c_int]; L.speckv_ext_prefetch_stats.restype = C.c_int
    L.speckv_ext_prefetch_outstanding.argtypes = [u64p, sz, C.POINTER(C.c_uint8), C.POINTER(PrefetchRequest), u32p, vp]
    L.speckv_ext_prefetch_outstanding.restype = C.c_int
    L.speckv_ext_engine_stats.argtypes = [C.POINTER(EngineStats), C.c_int]; L.speckv_ext_engine_stats.restype = None
    L.speckv_ext_tier_set_scheme.argtypes = [vp, C.c_int]; L.speckv_ext_tier_set_scheme.restype = C.c_int
    L.speckv_ext_set_pool_dtype.argtypes = [C.c_uint64, C.c_int]; L.speckv_ext_set_pool_dtype.restype = C.c_int
    L.speckv_ext_get_compression_scheme.argtypes = [C.POINTER(C.c_int)]; L.speckv_ext_get_compression_scheme.restype = C.c_int
    L.speckv_ext_get_stats.argtypes = [C.POINTER(Stats)]; L.speckv_ext_get_stats.restype = None
    L.speckv_ext_reset_stats.argtypes = []; L.speckv_ext_reset_stats.restype = None
    _LIB = L
    return L


def check(status: int, what: str) -> None:
    if status != SPECKV_OK:
        raise SpeckvError(what, status)
