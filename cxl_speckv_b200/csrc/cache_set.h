// cache_set.h -- a registered KV cache set (speckv_ext_cache_set_create): the element addresses of a model's paged KV
// caches on the device, and how a codec call addresses groups through it.
#pragma once

#include <stddef.h>
#include <stdint.h>

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

// group i of the call is block block_table[i] of cache cache_index[i]
inline void use_cache_set(CodecArgs& a, const speckv_cache_set& s, const uint32_t* cache_index,
                          const uint32_t* block_table) {
    a.in = nullptr;
    a.out = nullptr;
    a.cache_bases = s.d_bases;
    a.cache_index = cache_index;
    a.elem_index = block_table;
    a.block_stride = s.block_stride;
    a.n_caches = s.n_caches;
    a.set_unaligned = !s.aligned;
}

// every call through a set runs on the device it was created on
inline bool cache_set_on_current_device(const speckv_cache_set& s) {
    int d = -1;
    return cudaGetDevice(&d) == cudaSuccess && d == s.device;
}

}  // namespace speckv
