/*
 * speckv_ext.h -- additive, stream-ordered batch entry points of libcxlspeckv.so.
 *
 * The reference has no batch API: its cache engine is a C++ class
 * (src/fpga_engine/cache_engine.h:21-125) that nothing calls, and its host path
 * moves one 4 KiB page per ioctl (host/src/speckv_allocator.cpp:115-138).  These
 * functions are what a reference maintainer binds to replace
 *   FPGACacheEngine::compress / decompress / translate_address
 *       (src/fpga_engine/cache_engine.cpp:40-140),
 *   AddressTranslationUnit::translate (src/utils/address_translation.cpp:19-46),
 *   SpeckvAllocator's page table + sync fetch (host/src/speckv_allocator.cpp:11-138),
 *   SpeckvDriver::submit_dma_batch (host/src/speckv_driver.cpp:24-47) and
 *   LSTMPredictor::predict_top_k + SpeculativePrefetcher::prefetch
 *       (src/prefetcher/lstm_predictor.cpp:40-94, speculative_prefetcher.cpp:25-82)
 * with sm_100a CUDA kernels.  Plain C: pointers, sizes, enums; `cuda_stream` is
 * a cudaStream_t passed as void* (NULL = the legacy default stream).  Pointers
 * named d_* are device pointers, h_* host pointers.  All calls are
 * asynchronous on the stream unless stated; they return SPECKV_ERR_DRIVER when
 * no CUDA device is usable (there is no CPU fallback) and SPECKV_ERR_INVAL for
 * bad arguments.
 *
 * Container format (the reference has none; CompressedData is an in-memory
 * struct, cache_engine.h:35-40): group g owns a fixed slot
 *   payload + g * slot_bytes     (slot_bytes >= speckv_ext_slot_bytes(), 16 B aligned)
 * whose first comp_bytes[g] bytes equal CompressedData::rle_data exactly, plus
 * scales[g] (== scale_factor) and comp_bytes[g] (== compressed_size).
 */
#ifndef SPECKV_EXT_H
#define SPECKV_EXT_H

#include "speckv.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    SPECKV_DTYPE_F16  = 0,   /* IEEE half  */
    SPECKV_DTYPE_BF16 = 1,   /* bfloat16   */
    SPECKV_DTYPE_F32  = 2,   /* what the reference engine consumes (std::vector<float>) */
} speckv_dtype_t;

/* Extension scheme ids, accepted wherever a speckv_comp_scheme_t is (cast the value).  NOT reference behaviour:
 * SURVEY.md section 8f-4 asks for a non-wrapping quantiser as an explicit new id.  The reference multiplies by 127
 * twice -- s = max|x| / 127 (cache_engine.cpp:183) and (x / s) * 127 (:190-191) -- so its codes wrap modulo 256, the
 * clamp at :192 is dead and the reconstruction error of schemes 1 and 2 is of the order of the data itself.  The
 * clamped schemes keep every operation of :186-196 and :275-284, apply the clamp before the narrowing cast as :192
 * intended and store s = max|x|, so quantiser and dequantiser are inverse to each other (NaN codes as 0).  Same
 * container, same decoder: a payload written under 3 / 4 decodes under 2 / 1 and vice versa. */
enum {
    SPECKV_COMP_INT8_CLAMP_DELTA_RLE = 3,   /* clamped codes + delta + byte-pair RLE, slot 2 * n */
    SPECKV_COMP_INT8_CLAMP           = 4,   /* clamped codes only, slot n */
};

/* ---- library / device ----------------------------------------------------- */
/* Number of usable CUDA devices (0 when none: every other call then fails with
 * SPECKV_ERR_DRIVER). */
SPECKV_API int speckv_ext_device_count(void);
/* Human readable build id, e.g. "cxl-speckv-b200 sm_100a". */
SPECKV_API const char* speckv_ext_version(void);

/* ---- KV block codec -------------------------------------------------------- */
/* Worst-case bytes a group of group_elems elements can occupy under `scheme`,
 * rounded up to 16: INT8_DELTA_RLE 2*n (every element its own [value][count]
 * pair, cache_engine.cpp:213-239), INT8 n, FP16 2*n. */
SPECKV_API size_t speckv_ext_slot_bytes(size_t group_elems, speckv_comp_scheme_t scheme);

/* FPGACacheEngine::compress (cache_engine.cpp:40-82) over n_groups independent
 * groups of group_elems consecutive elements of d_in.  One fp32 scale per group
 * (:172-184), wrapped int8 quantisation (:186-196), delta across the whole flat
 * group (:198-211), byte-pair RLE with the 255 cap (:213-239); bit-exact.
 * scheme INT8 stops after quantisation (payload = the int8 codes);
 * scheme FP16 stores the elements unchanged (scale 1).  */
SPECKV_API speckv_status_t speckv_ext_compress(const void* d_in, speckv_dtype_t dtype,
                                    size_t group_elems, size_t n_groups,
                                    void* d_payload, size_t slot_bytes,
                                    float* d_scales, uint32_t* d_comp_bytes,
                                    speckv_comp_scheme_t scheme, void* cuda_stream);

/* FPGACacheEngine::decompress (cache_engine.cpp:84-116): RLE expand (:241-258,
 * odd trailing byte ignored, count 0 emits nothing), mod-256 prefix sum
 * (:260-273), (float)q / 127.0f * scale (:275-284) rounded to `dtype`.
 * At most group_elems elements are written per group at d_out + g*group_elems;
 * d_out_elems[g] (optional, may be NULL) receives the number produced.  A ragged
 * group (speckv_ext_compress_ragged) decodes to its n elements: the destination
 * past them is left untouched.  The same holds for every decode call below
 * (_indexed, _routed, _scatter, the tier's restores). */
SPECKV_API speckv_status_t speckv_ext_decompress(const void* d_payload, size_t slot_bytes,
                                      const float* d_scales, const uint32_t* d_comp_bytes,
                                      size_t group_elems, size_t n_groups,
                                      speckv_dtype_t dtype, void* d_out, uint32_t* d_out_elems,
                                      speckv_comp_scheme_t scheme, void* cuda_stream);

/* Decompress a selection of stored blocks: output group i (at d_out + i*group_elems) decodes the
 * stored block d_block_index[i] of the container.  This is how prefetch requests for predicted
 * blocks (speckv_ext_prefetch_score) and page fetches are served.  n_requests output groups. */
SPECKV_API speckv_status_t speckv_ext_decompress_indexed(const void* d_payload, size_t slot_bytes,
                                              const float* d_scales, const uint32_t* d_comp_bytes,
                                              const uint32_t* d_block_index, size_t n_requests,
                                              size_t group_elems, speckv_dtype_t dtype, void* d_out,
                                              uint32_t* d_out_elems, speckv_comp_scheme_t scheme,
                                              void* cuda_stream);

/* The same with the request list produced on the device (speckv_ext_route_requests): the number of valid
 * entries of d_block_index is read from *d_n_requests by the kernels, max_requests is the capacity the launch
 * is sized for.  No host synchronisation between routing and decoding; capturable into a CUDA graph. */
SPECKV_API speckv_status_t speckv_ext_decompress_routed(const void* d_payload, size_t slot_bytes,
                                             const float* d_scales, const uint32_t* d_comp_bytes,
                                             const uint32_t* d_block_index, const uint32_t* d_n_requests,
                                             size_t max_requests, size_t group_elems, speckv_dtype_t dtype,
                                             void* d_out, uint32_t* d_out_elems, speckv_comp_scheme_t scheme,
                                             void* cuda_stream);

/* Paged gather / scatter fused with the codec: the element buffer is a paged KV cache made of
 * blocks of group_elems elements (vLLM layout: one block = block_size tokens x kv_heads x
 * head_dim, contiguous), and a block table says which blocks take part.
 *   compress_gather: stored group i (slot i, scales[i], comp_bytes[i]) encodes cache block
 *     d_block_table[i] read at d_cache + d_block_table[i] * group_elems -- no staging copy.
 *   decompress_scatter: request i decodes stored block d_src_index[i] (or block i when
 *     d_src_index is NULL) into cache block d_block_table[i]; d_out_elems[i] is per request.
 * Block ids must be distinct within a scatter call.  Schemes INT8_DELTA_RLE and INT8. */
SPECKV_API speckv_status_t speckv_ext_compress_gather(const void* d_cache, const uint32_t* d_block_table,
                                                      speckv_dtype_t dtype, size_t group_elems, size_t n_groups,
                                                      void* d_payload, size_t slot_bytes, float* d_scales,
                                                      uint32_t* d_comp_bytes, speckv_comp_scheme_t scheme,
                                                      void* cuda_stream);
SPECKV_API speckv_status_t speckv_ext_decompress_scatter(const void* d_payload, size_t slot_bytes, const float* d_scales,
                                                         const uint32_t* d_comp_bytes, const uint32_t* d_src_index,
                                                         const uint32_t* d_block_table, size_t n_requests,
                                                         size_t group_elems, speckv_dtype_t dtype, void* d_cache,
                                                         uint32_t* d_out_elems, speckv_comp_scheme_t scheme,
                                                         void* cuda_stream);

/* Ragged groups: the filled prefix of each block.  Group i encodes the first min(d_group_len[i], group_elems)
 * elements of block d_block_table[i] (or of block i when d_block_table is NULL); lengths above group_elems are
 * clamped to it, a length of 0 gives scale 1.0 and comp_bytes 0.  Bit-exact with FPGACacheEngine::compress on
 * that prefix (cache_engine.cpp:40-82 takes a vector of any length): the elements behind it -- stale K/V of an
 * earlier request in a reused block -- take no part in the scale and never reach the payload.  d_group_len is a
 * DEVICE array, so the call needs no host synchronisation and can be captured into a CUDA graph.  Schemes 1-4
 * (FP16 -> SPECKV_ERR_INVAL).  Decoding needs no new call: the decoders produce n elements.  The byte counters of
 * speckv_ext_get_stats / speckv_ext_engine_stats count group capacity (group_elems) for ragged calls, because the
 * lengths live on the device. */
SPECKV_API speckv_status_t speckv_ext_compress_ragged(const void* d_in, const uint32_t* d_block_table,
                                                      const uint32_t* d_group_len, speckv_dtype_t dtype,
                                                      size_t group_elems, size_t n_groups, void* d_payload,
                                                      size_t slot_bytes, float* d_scales, uint32_t* d_comp_bytes,
                                                      speckv_comp_scheme_t scheme, void* cuda_stream);

/* Same two operations on HOST buffers: chunks are staged through device
 * buffers on internal streams (H2D, kernel, D2H overlapped) and the call
 * returns when the results are in host memory.  Pinned host memory
 * (speckv_ext_host_alloc) gives full PCIe rate.  This is the call the
 * end-to-end benchmark times.  Payloads cross PCIe at their size: when the slots of a
 * chunk are less than three quarters full (and the chunk has at most 4096 groups) every
 * group's payload travels alone, rounded up to 16 bytes; otherwise the chunk's slots go
 * in one copy.  Bytes of a slot beyond comp_bytes are left untouched in h_payload.
 * speckv_ext_get_stats reports the bytes actually moved. */
SPECKV_API speckv_status_t speckv_ext_compress_host(const void* h_in, speckv_dtype_t dtype,
                                         size_t group_elems, size_t n_groups,
                                         void* h_payload, size_t slot_bytes,
                                         float* h_scales, uint32_t* h_comp_bytes,
                                         speckv_comp_scheme_t scheme);
SPECKV_API speckv_status_t speckv_ext_decompress_host(const void* h_payload, size_t slot_bytes,
                                           const float* h_scales, const uint32_t* h_comp_bytes,
                                           size_t group_elems, size_t n_groups,
                                           speckv_dtype_t dtype, void* h_out, uint32_t* h_out_elems,
                                           speckv_comp_scheme_t scheme);
/* Pinned host memory for the *_host calls and the host tier. */
SPECKV_API void* speckv_ext_host_alloc(size_t bytes);
SPECKV_API void speckv_ext_host_free(void* p);

/* ---- address translation ---------------------------------------------------- */
/* FPGACacheEngine::translate_address (cache_engine.cpp:118-140) for n addresses:
 * pa = 0x4000000000 + (va & 0xFFFFFFFFFFFF); the 1024-entry TLB never changes
 * the value, only hit/miss counts. */
SPECKV_API speckv_status_t speckv_ext_translate(const uint64_t* d_va, uint64_t* d_pa, size_t n, void* cuda_stream);

/* Stateful model of the reference's AddressTranslationUnit (src/utils/address_translation.cpp):
 * a direct-mapped TLB whose translate() returns entry.ppage + offset on a hit and
 * page_walk(va) + offset -- the offset counted twice -- on a miss (:19-46, :85-90), with hit/miss
 * counters (:23-27).  The batch is processed with exact sequential semantics (results depend on
 * the order of d_va).  `all` != 0 in _invalidate = invalidate_all (:60-66), else invalidate(va)
 * (:48-58).  _get_stats synchronises the device. */
typedef struct speckv_atu speckv_atu_t;
SPECKV_API speckv_status_t speckv_ext_atu_create(uint32_t tlb_size, speckv_atu_t** out_atu);
SPECKV_API void speckv_ext_atu_destroy(speckv_atu_t* atu);
SPECKV_API speckv_status_t speckv_ext_atu_translate(speckv_atu_t* atu, const uint64_t* d_va, uint64_t* d_pa, size_t n,
                                                    void* cuda_stream);
SPECKV_API speckv_status_t speckv_ext_atu_invalidate(speckv_atu_t* atu, uint64_t va, int all, void* cuda_stream);
SPECKV_API speckv_status_t speckv_ext_atu_get_stats(speckv_atu_t* atu, uint64_t* hits, uint64_t* misses, int reset);

/* ---- page table --------------------------------------------------------------- */
/* One page-table entry: identical to the reference's KvPageHandle
 * (host/include/speckv_allocator.hpp:22-27): flags bit0 = in L1, bit1 = in L2, bit2 = compressed. */
typedef struct {
    uint64_t virt_page_id;   /* (handle << 32) | (page << 12)                 speckv_allocator.cpp:24 */
    uint64_t phys_page_id;   /* 0x4000000000 + (handle << 20) + (page << 12)  speckv_allocator.cpp:25 */
    uint32_t page_size;      /* 4096 */
    uint32_t flags;
} speckv_page_t;

/* Copies the page table of `handle` (speckv_alloc) into the device array d_pages (capacity
 * entries) so that lookups can run on the GPU; *out_count receives the number of pages of the
 * handle (copied entries = min(count, capacity)).  Needs speckv_init; unknown handle ->
 * SPECKV_ERR_GENERAL. */
SPECKV_API speckv_status_t speckv_ext_page_table_export(speckv_handle_t handle, speckv_page_t* d_pages,
                                                        size_t capacity, size_t* out_count, void* cuda_stream);

/* ---- CXLMemoryManager address map (src/cxl_memory/cxl_memory_manager.cpp:8-128) ----
 * allocate(): pages = ceil(size / 4096); the virtual address is bump-allocated from 0x1_0000_0000, the physical
 * one per tier (0 = L1 GPU-local from 0x80_0000_0000, 1 = L2 prefetch from 0x100_0000_0000, 2 = L3 CXL pool from
 * 0x200_0000_0000); an L1 preference falls back to L3 when L1 is full, "full" counted the reference's way
 * (allocations already in L1 x 4096 + the new bytes > capacity, :37-39 with :295-316).  deallocate(va) drops the
 * page entry AT va only (:81-104); addresses are never reused.  The page table lives on the host as speckv_page_t
 * records dense in (va - 0x1_0000_0000) >> 12 (flags bit0 = L1, bit1 = L2); _export copies it to the device, where
 * speckv_ext_page_lookup(d_pages, count, va_base, ...) answers translate_virtual_to_physical (:106-117, unknown
 * address -> 0) and is_in_cache (:119-128) for whole batches.  _set_tier carries promote / demote decisions of the
 * residency policy (speckv_ext_policy_*) into the table; _translate_host is the single-address form. */
#define SPECKV_PAGE_BYTES 4096u
typedef struct speckv_memmgr speckv_memmgr_t;
SPECKV_API speckv_status_t speckv_ext_memmgr_create(uint64_t l1_bytes, uint64_t l2_bytes, uint64_t l3_bytes,
                                                    speckv_memmgr_t** out);
SPECKV_API void speckv_ext_memmgr_destroy(speckv_memmgr_t* m);
SPECKV_API speckv_status_t speckv_ext_memmgr_allocate(speckv_memmgr_t* m, uint64_t size_bytes, uint32_t layer_id,
                                                      int preferred_tier, uint64_t* out_va, int* out_tier);
SPECKV_API speckv_status_t speckv_ext_memmgr_deallocate(speckv_memmgr_t* m, uint64_t va);
SPECKV_API speckv_status_t speckv_ext_memmgr_set_tier(speckv_memmgr_t* m, uint64_t va, size_t n_pages, int tier);
SPECKV_API speckv_status_t speckv_ext_memmgr_translate_host(speckv_memmgr_t* m, uint64_t va, uint64_t* out_pa,
                                                            int* out_tier);
SPECKV_API speckv_status_t speckv_ext_memmgr_export(speckv_memmgr_t* m, speckv_page_t* d_pages, size_t capacity,
                                                    size_t* out_count, uint64_t* out_va_base, void* cuda_stream);

/* Batched page-table lookup (SpeckvAllocator::access address arithmetic + is_in_l1_or_l2,
 * speckv_allocator.cpp:54-74,105-113; same form as CXLMemoryManager::translate_virtual_to_physical,
 * cxl_memory_manager.cpp:106-117): for each va, entry = d_pages[(va - va_base) >> 12];
 * d_pa[i] = entry.phys_page_id + (va & 0xFFF), d_flags[i] = entry.flags (d_flags may be NULL);
 * outside the table, or entry.virt_page_id != (va & ~0xFFF): d_pa[i] = 0, d_flags[i] = 0.
 * For a speckv_alloc handle h: va_base = h << 32 and va = va_base + byte offset. */
SPECKV_API speckv_status_t speckv_ext_page_lookup(const speckv_page_t* d_pages, size_t num_pages, uint64_t va_base,
                                                  const uint64_t* d_va, uint64_t* d_pa, uint32_t* d_flags,
                                                  size_t n, void* cuda_stream);

/* ---- host tier (pinned-DRAM pool standing in for the CXL memory pool) ------------------- */
/* Replaces the simulated DMA of SpeckvAllocator::sync_fetch_page (speckv_allocator.cpp:115-138,
 * descriptor flag bit1 = COMPRESSED, driver/uapi/speckv_ioctl.h:14) and CXLMemoryManager's
 * demote_to_l3 / promote_to_l1 data movement (cxl_memory_manager.cpp:130-194) with real transfers:
 * offload = compress + pack on the GPU, one device-to-host copy per chunk on a side stream into a
 * pinned pool; restore = host-to-device copies of the packed blocks + decompress.  Blocks are
 * named by caller-chosen 64-bit ids (e.g. virt_page_id).  Scheme: INT8_DELTA_RLE. */
typedef struct speckv_tier speckv_tier_t;
typedef struct {
    uint64_t pool_bytes, used_bytes, blocks;
    uint64_t bytes_offloaded_raw, bytes_offloaded_stored;   /* uncompressed KV bytes / bytes placed in the pool */
    uint64_t bytes_restored_raw, bytes_restored_stored;
    uint64_t last_offload_stored_bytes, last_restore_stored_bytes;
    double   last_offload_ms, last_restore_ms;              /* wall time of the last call, copies included */
} speckv_tier_stats_t;

SPECKV_API speckv_status_t speckv_ext_tier_create(size_t pool_bytes, speckv_tier_t** out_tier);
SPECKV_API void speckv_ext_tier_destroy(speckv_tier_t* tier);
/* Compress n_groups groups of d_in and move their payload into the pool under h_block_ids[i].
 * Returns when the bytes are in host memory.  SPECKV_ERR_NOMEM when the pool is full. */
SPECKV_API speckv_status_t speckv_ext_tier_offload(speckv_tier_t* tier, const void* d_in, speckv_dtype_t dtype,
                                                   size_t group_elems, size_t n_groups,
                                                   const uint64_t* h_block_ids, void* cuda_stream);
/* Paged forms (the KV cache is a pool of blocks of group_elems elements, vLLM layout; d_block_table is a
 * DEVICE array of n_blocks cache block numbers): block d_block_table[i] of d_cache is compressed and stored
 * under h_block_ids[i] / block h_block_ids[i] is decompressed into cache block d_block_table[i].  The
 * codec kernels gather / scatter through the table: no staging copy of the blocks on either side.
 * Block numbers must be distinct within a restore call. */
SPECKV_API speckv_status_t speckv_ext_tier_offload_paged(speckv_tier_t* tier, const void* d_cache,
                                                         const uint32_t* d_block_table, speckv_dtype_t dtype,
                                                         size_t group_elems, size_t n_blocks,
                                                         const uint64_t* h_block_ids, void* cuda_stream);
SPECKV_API speckv_status_t speckv_ext_tier_restore_paged(speckv_tier_t* tier, const uint64_t* h_block_ids,
                                                         size_t n_blocks, size_t group_elems, speckv_dtype_t dtype,
                                                         void* d_cache, const uint32_t* d_block_table,
                                                         void* cuda_stream);
/* Ragged offload (d_block_table may be NULL: block i of d_in): block i is stored from its first
 * min(d_group_len[i], group_elems) elements, as speckv_ext_compress_ragged encodes them.  Restores decode such a
 * block to that many elements and leave the rest of the destination untouched.  bytes_offloaded_raw /
 * bytes_restored_raw count the valid bytes.  The tier's scheme must be 1-4 (FP16 -> SPECKV_ERR_INVAL). */
SPECKV_API speckv_status_t speckv_ext_tier_offload_ragged(speckv_tier_t* tier, const void* d_in,
                                                          const uint32_t* d_block_table, const uint32_t* d_group_len,
                                                          speckv_dtype_t dtype, size_t group_elems, size_t n_blocks,
                                                          const uint64_t* h_block_ids, void* cuda_stream);
/* Bring blocks back: output group i (d_out + i*group_elems) = decompressed block h_block_ids[i].
 * Unknown id -> SPECKV_ERR_GENERAL.  Returns when d_out is complete. */
SPECKV_API speckv_status_t speckv_ext_tier_restore(speckv_tier_t* tier, const uint64_t* h_block_ids, size_t n_groups,
                                                   size_t group_elems, speckv_dtype_t dtype, void* d_out,
                                                   void* cuda_stream);
/* Release pool space of blocks (unknown ids are ignored, like speckv_free). */
/* The scheme new offloads are stored under (default INT8_DELTA_RLE; 0 .. 4, the raw passthrough 0 only for the
 * non-paged fp16 / bf16 form).  Every stored block remembers its scheme: restores decode each block the way it was
 * stored, whatever the tier's current setting.  speckv_set_compression_scheme (host/include/speckv.h:59-66) applies
 * to the tiers of all bound pools through this call. */
SPECKV_API speckv_status_t speckv_ext_tier_set_scheme(speckv_tier_t* tier, speckv_comp_scheme_t scheme);
SPECKV_API speckv_status_t speckv_ext_tier_drop(speckv_tier_t* tier, const uint64_t* h_block_ids, size_t n);
SPECKV_API void speckv_ext_tier_get_stats(speckv_tier_t* tier, speckv_tier_stats_t* out);

/* Device-side fetch: blocks named by ids in DEVICE memory come back without the host, so a prefetch step
 * (speckv_ext_prefetch_emit -> speckv_ext_route_requests -> ids -> fetch) is one CUDA graph.
 *
 * Keep a copy of the tier's block directory in device memory from now on, so that speckv_ext_tier_fetch can find
 * blocks without the host.  Uploads the current directory on cuda_stream and waits for it.  Idempotent; there is no
 * disable.  While it is on, every offload and drop of this tier also updates the device copy before it returns.
 * Must run on the tier's device (SPECKV_ERR_INVAL otherwise); SPECKV_ERR_DRIVER on a device that cannot read
 * mapped pinned host memory (no unified addressing). */
SPECKV_API speckv_status_t speckv_ext_tier_enable_fetch(speckv_tier_t* tier, void* cuda_stream);

/* Device scratch one fetch call needs for up to max_requests blocks of group_elems elements: the staged payloads at
 * the largest slot of any scheme plus per-request metadata,
 *   max_requests * (speckv_ext_slot_bytes(group_elems, SPECKV_COMP_INT8_DELTA_RLE) + 24) + 8.
 * Arithmetic only: works without a device. */
SPECKV_API size_t speckv_ext_tier_fetch_workspace_bytes(size_t max_requests, size_t group_elems);

/* Restore blocks named on the DEVICE.  Request i < *d_n_requests (all max_requests when d_n_requests is NULL) names
 * stored block d_block_ids[i].  It is decoded into d_out + i*group_elems, or into cache block d_block_table[i] when a
 * table is given (block numbers distinct, as for _restore_paged).  d_status[i] (optional) = 1 when the request was
 * served, 0 when the id is not in the tier or its block does not fit the call.  A block does not fit when it has
 * another group_elems or another dtype, when it is raw (scheme 0), or when its scheme decodes differently from
 * `scheme`: 1 and 4 share a decoder, and so do 2 and 3.  An unserved request writes nothing to its destination and
 * gets out_elems 0.  d_out_elems[i] (optional) = elements decoded (n for a ragged block).  Entries at and behind the
 * count are left untouched.  No host synchronisation; capturable into a CUDA graph.  Needs speckv_ext_tier_enable_fetch
 * first (SPECKV_ERR_INVAL otherwise), a 16-byte aligned d_workspace of workspace_bytes >=
 * speckv_ext_tier_fetch_workspace_bytes(max_requests, group_elems), and scheme 1-4.  The workspace belongs to the
 * call while it runs: calls in flight at the same time need their own.  The call must run on the tier's device.
 * Ordering: a fetch reads the directory and the pool when it runs.  Offloads of the tier on the fetch's stream are
 * ordered with it through that stream; before an offload on another stream, or a drop, synchronise the streams that
 * still have fetches of the tier in flight.  Fetched bytes are not counted in speckv_tier_stats_t (bytes_restored_*
 * count the host-driven restores only). */
SPECKV_API speckv_status_t speckv_ext_tier_fetch(speckv_tier_t* tier, const uint64_t* d_block_ids,
                                                 const uint32_t* d_n_requests, size_t max_requests, size_t group_elems,
                                                 speckv_dtype_t dtype, speckv_comp_scheme_t scheme, void* d_out,
                                                 const uint32_t* d_block_table, uint32_t* d_out_elems,
                                                 uint8_t* d_status, void* d_workspace, size_t workspace_bytes,
                                                 void* cuda_stream);

/* ---- descriptor-level interface (what the reference's ioctl client speaks) ------------------ */
/* One transfer descriptor, identical to struct speckv_ioctl_dma_desc (driver/uapi/speckv_ioctl.h:
 * 10-15) / SpeckvDmaDesc (host/include/speckv_driver.hpp:8-13): fpga_addr names the first 4 KiB
 * page on the tier side (page i of the descriptor is fpga_addr + i*4096), gpu_addr is a device
 * pointer, bytes a multiple of 4096, flags bit0 = write (GPU -> tier; clear = read, tier -> GPU),
 * bit1 = run the page through the codec, bit2 = prefetch hint (no effect on the data). */
typedef struct {
    uint64_t fpga_addr;
    uint64_t gpu_addr;
    uint32_t bytes;
    uint32_t flags;
} speckv_dma_desc_t;
#define SPECKV_DMA_WRITE      1u
#define SPECKV_DMA_COMPRESSED 2u
#define SPECKV_DMA_PREFETCH   4u
/* SpeckvDriver::submit_dma_batch (speckv_driver.cpp:24-47): at most 4096 descriptors per batch
 * (speckv_kernel_module.c:65-66 -> SPECKV_ERR_INVAL), executed in order, blocking. */
SPECKV_API speckv_status_t speckv_ext_submit_dma_batch(speckv_tier_t* tier, const speckv_dma_desc_t* h_descs,
                                                       uint32_t count, void* cuda_stream);
/* SpeckvDriver::poll_complete (speckv_driver.cpp:65-72): descriptors completed since the last poll. */
SPECKV_API uint32_t speckv_ext_poll_complete(void);
/* SPECKV_IOCTL_PREFETCH with the request record of driver/uapi/speckv_ioctl.h:25-33 (the call tests/test_prefetch.c
 * makes; SpeckvDriver::prefetch, speckv_driver.cpp:49-55): same effect as speckv_prefetch(req_id, layer, cur_pos,
 * depth_k, tokens, history_len).  A NULL record, a NULL token pointer or history_len == 0 -> SPECKV_ERR_INVAL (the
 * kernel module answers -EFAULT for pointers it cannot read, speckv_kernel_module.c:116-132). */
typedef struct {
    uint32_t req_id;
    uint16_t layer;
    uint16_t reserved0;
    uint32_t cur_pos;
    uint32_t depth_k;
    uint32_t history_len;
    uint64_t tokens_user_ptr;   /* const int32_t[history_len] in the caller's address space */
} speckv_prefetch_req_t;
SPECKV_API speckv_status_t speckv_ext_submit_prefetch(const speckv_prefetch_req_t* req);
/* SPECKV_IOCTL_SET_PARAM: key 1 = prefetch depth, key 2 = compression scheme; any other key is
 * rejected with SPECKV_ERR_INVAL (speckv_kernel_module.c:179-188, tests/test_params.c:68-84). */
SPECKV_API speckv_status_t speckv_ext_set_param(uint32_t key, uint32_t value);

/* ---- serving real pointers through the frozen ABI ----------------------------------------- */
/* Binds device memory to a speckv_alloc handle (SURVEY.md section 8f row 1).  From then on
 * speckv_access(handle, offset, len, &ptr) returns d_base + offset -- a dereferenceable device
 * pointer instead of the reference's synthetic 0x40..-address -- after making the touched pages
 * resident: a page whose only copy is the compressed one in `tier` is restored first (the
 * reference's sync_fetch_page with a real transfer).  `tier` may be NULL (no spilling).
 * bytes >= pages * 4096; the pool's current contents count as resident. */
SPECKV_API speckv_status_t speckv_ext_bind_pool(speckv_handle_t handle, void* d_base, size_t bytes,
                                                speckv_tier_t* tier);
/* KV layout of the bound region, [req][layer][kind][pos][head] x entry_bytes
 * (host/python/vllm_speckv_backend.py:95-100); lets speckv_prefetch() turn (req, layer, cur_pos,
 * depth_k) into the pages of positions cur_pos+1 .. cur_pos+depth_k and make them resident. */
SPECKV_API speckv_status_t speckv_ext_set_kv_layout(speckv_handle_t handle, uint32_t num_layers, uint32_t num_tokens,
                                                    uint32_t num_heads, uint32_t entry_bytes);
/* Element type of the bound pool (default fp16): what the codec quantises when pages of this handle are offloaded
 * and what restores write back -- one 4 KiB page is one group of 2048 fp16 / bf16 or 1024 fp32 elements.  Refused
 * (SPECKV_ERR_GENERAL) while pages stored under another type live only in the tier. */
SPECKV_API speckv_status_t speckv_ext_set_pool_dtype(speckv_handle_t handle, speckv_dtype_t dtype);
/* The scheme set by speckv_set_compression_scheme / speckv_ext_set_param(2, ..) (default 2). */
SPECKV_API speckv_status_t speckv_ext_get_compression_scheme(int* out_scheme);
/* Demote pages to the host tier (compress + move; flags: L1/L2 cleared, compressed set) /
 * promote them back (restore; flags: L2 set; a page is marked resident only after its restore succeeded).
 * Pages are groups of the pool's element type, stored under the current compression scheme. */
SPECKV_API speckv_status_t speckv_ext_offload_pages(speckv_handle_t handle, uint64_t first_page, uint64_t n_pages,
                                                    void* cuda_stream);
SPECKV_API speckv_status_t speckv_ext_fetch_pages(speckv_handle_t handle, uint64_t first_page, uint64_t n_pages,
                                                  void* cuda_stream);

/* ---- tier residency policy (SURVEY.md section 8f row 2) -------------------------------- */
/* CXLMemoryManager's residency bookkeeping (src/cxl_memory/cxl_memory_manager.cpp:28-324) over
 * dense page indices 0..n_pages-1, with the per-page state (tier, access count, LRU stamp) in
 * device memory so that a decode step can report millions of touched pages with one kernel:
 *   place    = allocate() of single pages into a tier (an L1 preference falls back to L3 when L1
 *              is full, :37-40)
 *   touch    = update_access_tracking() for every id in order (:221-246): ++access_count,
 *              l1_hits / l2_hits / l3_accesses by tier, page to the back of the LRU list
 *   is_hot   = access_count > 10 (:248-258)
 *   promote  = promote_to_l1() for every id in order (:130-162); when L1 is full the least
 *              recently used L1 page is demoted to L3 first and reported in `evicted`
 *   demote   = demote_to_l3() (:164-194)
 * Tiers: 0 = L1 (HBM), 1 = L2 (prefetch buffer), 2 = L3 (pool), 255 = not allocated.
 * The reference's own eviction (evict_l1_lru, :285-293) re-locks a mutex it already holds and
 * never returns; the semantics here are that step repeated until a page is freed: entries are
 * popped from the front of the LRU list (entries that are not L1-resident are dropped, as the
 * reference's pop drops them) until an L1 page has been popped and demoted; if the list holds
 * no L1 page nothing is evicted and the promotion proceeds, as in the reference.  Capacities
 * count pages.  Pair promote/demote with
 * speckv_ext_fetch_pages / speckv_ext_offload_pages to move the data. */
typedef struct speckv_policy speckv_policy_t;
typedef struct {
    uint64_t l1_hits, l1_misses, l2_hits, l2_misses, l3_accesses;
    uint64_t migrations_l1_to_l3, migrations_l3_to_l1;
    double l1_hit_rate, l2_hit_rate;
    uint64_t l1_pages, l2_pages, l3_pages;
} speckv_policy_stats_t;
SPECKV_API speckv_status_t speckv_ext_policy_create(uint64_t n_pages, uint64_t l1_capacity_pages,
                                                    uint64_t l2_capacity_pages, uint64_t l3_capacity_pages,
                                                    speckv_policy_t** out);
SPECKV_API void speckv_ext_policy_destroy(speckv_policy_t* p);
/* h_ids: host array.  out_tiers (optional, host): the tier each page went to, 255 if rejected
 * (index out of range or already allocated). */
SPECKV_API speckv_status_t speckv_ext_policy_place(speckv_policy_t* p, const uint64_t* h_ids, size_t n, int tier,
                                                   uint8_t* out_tiers);
SPECKV_API speckv_status_t speckv_ext_policy_release(speckv_policy_t* p, const uint64_t* h_ids, size_t n);
/* ids on the device (ids_on_device != 0, stream-ordered, no host synchronisation) or on the host */
SPECKV_API speckv_status_t speckv_ext_policy_touch(speckv_policy_t* p, const uint64_t* ids, size_t n,
                                                   int ids_on_device, void* cuda_stream);
/* d_ids / d_out on the device, stream-ordered */
SPECKV_API speckv_status_t speckv_ext_policy_is_hot(speckv_policy_t* p, const uint64_t* d_ids, size_t n,
                                                    uint8_t* d_out, void* cuda_stream);
/* Host arrays.  out_ok[n] (optional): 1 where the reference's call returns true.  out_evicted
 * (optional, capacity >= n): pages demoted to make room, in order; *out_n_evicted their count. */
SPECKV_API speckv_status_t speckv_ext_policy_promote(speckv_policy_t* p, const uint64_t* h_ids, size_t n,
                                                     uint8_t* out_ok, uint64_t* out_evicted, size_t* out_n_evicted);
SPECKV_API speckv_status_t speckv_ext_policy_demote(speckv_policy_t* p, const uint64_t* h_ids, size_t n,
                                                    uint8_t* out_ok);
SPECKV_API speckv_status_t speckv_ext_policy_get_tiers(speckv_policy_t* p, const uint64_t* h_ids, size_t n,
                                                       uint8_t* out_tiers);
/* LRU list, least recently used first (every member, as the reference's l1_lru_list_ holds any
 * touched page).  *out_n = list length; at most `capacity` ids are written. */
SPECKV_API speckv_status_t speckv_ext_policy_lru_order(speckv_policy_t* p, uint64_t* out_ids, size_t capacity,
                                                       size_t* out_n);
SPECKV_API speckv_status_t speckv_ext_policy_get_stats(speckv_policy_t* p, speckv_policy_stats_t* out);

/* ---- speculative prefetch scoring ---------------------------------------------------- */
/* Installs the predictor's weights on the current device: embedding [vocab][emb_dim] and
 * output projection [vocab][hidden], fp32, row-major -- the two tables
 * LSTMPredictor::predict_top_k actually reads (lstm_predictor.cpp:149-188; its per-layer "LSTM"
 * weights are never used, :116-147).  The reference draws them from rand() (:27-35) and its
 * load_model() is a stub (:96-99); here they are an explicit input. */
SPECKV_API speckv_status_t speckv_ext_predictor_load(const float* h_embedding, const float* h_output,
                                                     uint32_t vocab, uint32_t emb_dim, uint32_t hidden,
                                                     uint32_t layers, uint32_t history_len);
SPECKV_API void speckv_ext_predictor_unload(void);

/* LSTMPredictor::predict_top_k + SpeculativePrefetcher::prefetch's request emission for `batch`
 * sequences at once.  d_tokens: [batch][history_len] token ids, already windowed the way the
 * reference does it (last history_len tokens, left-padded with 0, lstm_predictor.cpp:46-51).
 * Outputs, [batch][k] each: predicted token ids, their softmax confidence, and the request
 * address (req_id << 32) | (layer_id << 16) | (i + 1) (speculative_prefetcher.cpp:153-160; the
 * reference always passes req_id 0).  k <= 16. */
SPECKV_API speckv_status_t speckv_ext_prefetch_score(const uint32_t* d_tokens, uint32_t batch, uint32_t k,
                                                     uint32_t req_id, uint32_t layer_id, uint32_t* d_ids,
                                                     float* d_conf, uint64_t* d_va, void* cuda_stream);

/* One prefetch request: the reference's PrefetchRequest (src/prefetcher/speculative_prefetcher.h:23-29), 32 bytes
 * with natural alignment.  This is the fixed-size record ranks exchange (SURVEY.md section 8e). */
typedef struct {
    uint64_t virtual_addr;
    uint32_t layer_id;
    uint32_t predicted_token_id;
    float    confidence;
    uint32_t reserved;          /* the padding before `timestamp` in the reference's struct; written as 0 */
    uint64_t timestamp;
} speckv_prefetch_request_t;

/* SpeculativePrefetcher::prefetch for `batch` sequences, entirely on the device: scoring as speckv_ext_prefetch_score,
 * then for every prediction i of every sequence the request address (req << 32) | (layer << 16) | (i + 1) with
 * req = d_req_ids[sequence] (or req_id for all when d_req_ids is NULL; the reference always uses 0), the residency
 * filter -- a request whose page is in L1 or L2 of the page table (d_pages / num_pages / va_base as in
 * speckv_ext_page_lookup; flags bit0 | bit1) is skipped, speculative_prefetcher.cpp:51-54; d_pages NULL = no filter --
 * and the emission of PrefetchRequest records (:57-66).  d_table receives 1 + batch * k records: record 0 is a
 * header whose virtual_addr field holds the number n of requests emitted, records 1 .. n are the requests in
 * sequence order, prediction order within a sequence; the rest is left untouched.  The table is what
 * speckv_ext_route_requests consumes, here or (all-gathered) on every rank.  `timestamp` is stored in every record
 * (the reference stores steady_clock::now()).  d_ids / d_conf (optional, [batch][k]) receive the unfiltered
 * predictions.  The 16 most recent requests stay queued on the device (issue_dma_prefetch, :162-172). */
SPECKV_API speckv_status_t speckv_ext_prefetch_emit(const uint32_t* d_tokens, uint32_t batch, uint32_t k,
                                                    const uint32_t* d_req_ids, uint32_t req_id, uint32_t layer_id,
                                                    const speckv_page_t* d_pages, size_t num_pages, uint64_t va_base,
                                                    uint64_t timestamp, speckv_prefetch_request_t* d_table,
                                                    uint32_t* d_ids, float* d_conf, void* cuda_stream);

/* SpeculativePrefetcher::handle_misprediction (speculative_prefetcher.cpp:84-97): counts a misprediction when
 * actual_token is not among the n predicted tokens.  Host logic; *out_was_correct (optional) = 1 if it was. */
SPECKV_API speckv_status_t speckv_ext_prefetch_handle_misprediction(uint32_t actual_token, const uint32_t* h_predicted,
                                                                    size_t n, int* out_was_correct);
/* SpeculativePrefetcher::get_statistics / reset_statistics (speculative_prefetcher.cpp:126-142; PrefetchStatistics,
 * speculative_prefetcher.h:59-66).  total_prefetches = requests emitted by speckv_ext_prefetch_emit;
 * avg_prediction_latency_us follows the reference's update rule (:72-79) with the device time of each emit call;
 * successful_prefetches is never incremented in the reference either, so hit_rate and precision are 0.  Blocking. */
typedef struct {
    uint64_t total_prefetches, successful_prefetches, mispredictions;
    double hit_rate, precision, avg_prediction_latency_us;
} speckv_prefetch_stats_t;
SPECKV_API speckv_status_t speckv_ext_prefetch_stats(speckv_prefetch_stats_t* out, int reset);
/* SpeculativePrefetcher::is_already_prefetched (speculative_prefetcher.cpp:174-185) for n addresses against the
 * queue of the 16 most recent requests; h_queue (optional, 16 records) / out_queue_len receive the queue itself,
 * oldest first.  Blocking. */
SPECKV_API speckv_status_t speckv_ext_prefetch_outstanding(const uint64_t* h_va, size_t n, uint8_t* out_found,
                                                           speckv_prefetch_request_t* h_queue, uint32_t* out_queue_len,
                                                           void* cuda_stream);

/* Turns request tables into this rank's decode list, on the device.  d_tables holds n_tables tables of
 * (1 + table_capacity) records each, as produced by speckv_ext_prefetch_emit (and all-gathered across ranks):
 * record 0 is a header whose virtual_addr field is the number of valid requests that follow.  A request names
 * stored block b = predicted_token_id % n_blocks_total; blocks are owned in contiguous ranges,
 * owner = b / ceil(n_blocks_total / world), local index = b - owner * ceil(n_blocks_total / world).  The requests
 * owned by `rank` are compacted, in table and record order, into d_block_index (capacity n_tables *
 * table_capacity) and their number is written to *d_count -- the pair speckv_ext_decompress_routed consumes.
 * d_request_index (optional) receives table * table_capacity + position of each kept request. */
SPECKV_API speckv_status_t speckv_ext_route_requests(const speckv_prefetch_request_t* d_tables, uint32_t n_tables,
                                                     uint32_t table_capacity, uint32_t n_blocks_total,
                                                     uint32_t world, uint32_t rank, uint32_t* d_block_index,
                                                     uint32_t* d_request_index, uint32_t* d_count,
                                                     void* cuda_stream);

/* Adaptive prefetch depth (SpeculativePrefetcher::update_prediction_accuracy / get_adaptive_depth,
 * speculative_prefetcher.cpp:99-124): report whether the last prediction was correct; the depth
 * used by the prefetcher moves between 2 and 8 exactly as in the reference.  Host logic: works
 * without a GPU.  speckv_set_prefetch_depth() overrides the current depth (:144-147). */
SPECKV_API speckv_status_t speckv_ext_prefetch_feedback(int was_correct, uint32_t* out_depth);
SPECKV_API speckv_status_t speckv_ext_get_prefetch_depth(uint32_t* out_depth);

/* ---- statistics (EngineStatistics, cache_engine.h:65-72) --------------------- */
typedef struct {
    uint64_t total_compressions;     /* groups compressed   */
    uint64_t total_decompressions;   /* groups decompressed */
    uint64_t total_translations;
    uint64_t bytes_in_compress;      /* uncompressed bytes consumed */
    uint64_t bytes_out_decompress;   /* uncompressed bytes produced (capacity) */
    uint64_t kernel_launches;        /* CUDA kernels this library launched */
    uint64_t host_api_h2d_bytes;     /* bytes speckv_ext_compress_host / _decompress_host copied host -> device */
    uint64_t host_api_d2h_bytes;     /* ... and device -> host (payloads travel at their size, not at the slot size) */
} speckv_ext_stats_t;
SPECKV_API void speckv_ext_get_stats(speckv_ext_stats_t* out);
/* FPGACacheEngine::get_statistics (cache_engine.cpp:150-158, EngineStatistics cache_engine.h:65-72) with the
 * reference's field meaning: the latencies are running means over CALLS, updated by the reference's rule
 * (:76-79, :108-112), measured with CUDA events on the caller's stream (a call = one batch of groups here, one
 * group in the reference; the per-group figures are given next to them).  avg_compression_ratio is the running
 * mean over the groups reported through speckv_ext_ratio_stats (the sizes live on the device; the reference
 * updates it inside compress(), :69-75).  throughput_gbps is measured (uncompressed gigabits per second of
 * device time in the timed calls) where the reference returns the constant 512 bit x 800 MHz (:291-296).
 * wait != 0 synchronises with the calls still in flight; otherwise only finished calls are counted.
 * Calls captured into a CUDA graph are not timed; SPECKV_LATENCY_STATS=0 switches the timing off. */
typedef struct {
    uint64_t total_compressions, total_decompressions;   /* groups, like speckv_ext_stats_t */
    double avg_compression_ratio;
    double avg_compression_latency_ns, avg_decompression_latency_ns;   /* per call */
    double throughput_gbps;
    uint64_t compress_calls_timed, decompress_calls_timed;
    double compress_ns_per_group, decompress_ns_per_group;
} speckv_engine_stats_t;
SPECKV_API void speckv_ext_engine_stats(speckv_engine_stats_t* out, int wait);
/* EngineStatistics::avg_compression_ratio (cache_engine.cpp:69-75): the mean over groups of
 * original_size / compressed_size with original_size = group_elems * sizeof(float), the reference's
 * own accounting (:49); plus the total payload bytes.  Blocking (returns host values). */
SPECKV_API speckv_status_t speckv_ext_ratio_stats(const uint32_t* d_comp_bytes, size_t n_groups, size_t group_elems,
                                                  double* out_total_comp_bytes, double* out_mean_ratio,
                                                  void* cuda_stream);
SPECKV_API void speckv_ext_reset_stats(void);

#ifdef __cplusplus
}
#endif
#endif /* SPECKV_EXT_H */
