// cache_set.h -- a registered KV cache set (speckv_ext_cache_set_create): the element addresses of a model's paged KV
// caches on the device, and how a codec call names the KV blocks it reads or writes.
#pragma once

#include <stddef.h>
#include <stdint.h>

#include "device_ctx.h"
#include "kv_codec.h"

// immutable after creation
struct speckv_cache_set {
    int device = -1;
    uint64_t* d_bases = nullptr;   // one element address per cache (device memory the set owns)
    uint32_t n_caches = 0;
    size_t block_elems = 0;        // elements of one block (one codec group)
    size_t block_stride = 0;       // elements between consecutive blocks of a cache (>= block_elems)
    int dtype = 0;
    bool aligned = false;          // every base and block_stride * element size a multiple of 16 bytes
};

namespace speckv {

// The KV blocks of a codec call: group i of the call is
//   dense:     block i of `base`
//   paged:     block block_table[i] of `base`
//   cache set: block block_table[i] of cache cache_index[i] of `set` (always with a block table; `base` unused)
// and, with group_len (compress only), just the first min(group_len[i], group elements) elements of that block.
struct KvBlocks {
    const void* base = nullptr;
    const uint32_t* block_table = nullptr;
    const uint32_t* group_len = nullptr;
    const speckv_cache_set* set = nullptr;
    const uint32_t* cache_index = nullptr;

    // a's element addressing for groups [g0, g0 + a.n_groups) of the call (a.group_elems elements of esz bytes each):
    // `in` for compress, `out` for decompress
    void bind(CodecArgs& a, bool decompress, size_t g0, size_t esz) const {
        if (set) {
            a.cache_bases = set->d_bases;
            a.cache_index = cache_index + g0;
            a.block_stride = set->block_stride;
            a.n_caches = set->n_caches;
            a.set_unaligned = !set->aligned;
        } else {
            const void* elems = block_table ? base : static_cast<const char*>(base) + g0 * a.group_elems * esz;
            if (decompress) a.out = const_cast<void*>(elems);
            else a.in = elems;
        }
        a.elem_index = block_table ? block_table + g0 : nullptr;
        a.group_len = group_len ? group_len + g0 : nullptr;
    }
};

// the checks every call through a set makes first: a device, a set on the current one (the device it was created
// on), and a cache index and a block table when the call names any group
inline speckv_status_t check_set(const speckv_cache_set* set, const uint32_t* d_cache_index,
                                 const uint32_t* d_block_table, size_t n) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    int d = -1;
    if (!set || cudaGetDevice(&d) != cudaSuccess || d != set->device || (n && (!d_cache_index || !d_block_table)))
        return SPECKV_ERR_INVAL;
    return SPECKV_OK;
}

}  // namespace speckv
