// tier_fetch.h -- the host tier's block directory as the device sees it, and the kernels of the device-side fetch
// (tier_fetch.cu) that tier.cu launches.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace speckv {

struct BlockRec {
    uint64_t pool_off;
    uint32_t comp_bytes;   // bytes held in the pool (payload bytes, or the raw size for raw blocks)
    float scale;
    uint32_t group_elems;  // 0 for raw (uncompressed) blocks
    int dtype;             // speckv_dtype_t | scheme << 8 (the scheme the block was stored under) | kRagged; -1 = empty map entry
    int scheme() const { return (dtype >> 8) & 0xff; }
    bool ragged() const { return (dtype & kRagged) != 0; }
    static constexpr int kRagged = 1 << 16;   // stored from a prefix of its block: decodes to fewer than group_elems elements
};

// one slot of the open-addressing block map: key and record in 32 bytes (one probe = one sector pair)
struct DirEntry {
    uint64_t key;
    BlockRec val;
};
static_assert(sizeof(DirEntry) == 32, "the device probe reads an entry as two 16-byte loads");

constexpr int kDirEmpty = -1;   // BlockRec::dtype of an empty slot

// the hash of BlockMap::slot_of, shared so that a device probe walks exactly the host's probe sequence
__host__ __device__ inline uint64_t dir_hash(uint64_t k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    return k;
}

// What the fetch kernels read the directory through.  It lives in device memory and is rewritten when the table
// grows, so a captured graph (whose launch arguments are frozen) follows the table to its new place.
struct DeviceDir {
    const DirEntry* table;
    uint64_t mask;          // capacity - 1 (a power of two)
    const uint8_t* pool;    // device address of the pinned pool
};

// one changed slot of the host map, staged for the device copy
struct DirUpdate {
    uint64_t slot;
    DirEntry e;
};

// apply n staged updates to the device table (table of the current header)
cudaError_t launch_dir_apply(const DeviceDir* d_dir, const DirUpdate* d_upd, size_t n, cudaStream_t st);

// Fetch pipeline on the device.  Request i < min(*n_dev, n) (all n when n_dev is null) names block ids[i].
//   lookup: probe the directory, check the block fits (group_elems, dtype, scheme family, not raw), write the pool
//           offset, payload size and scale of a served request, size 0 and scale 1 of an unserved one, status[i]
//           (with cache_index: also unserved when cache_index[i] >= n_caches, a cache set's request past the set)
//   gather: copy the served payloads out of the pinned pool into `staging`, back to back at offsets[i]
// Between the two the caller scans the sizes (pack_offsets_kernel, tier.cu) into offsets / *total.
cudaError_t launch_fetch_lookup(const DeviceDir* d_dir, const uint64_t* ids, const uint32_t* n_dev, uint32_t n,
                                uint32_t group_elems, int dtype, int scheme, size_t max_comp_bytes, uint64_t* src_off,
                                uint32_t* comp_bytes, float* scales, uint8_t* status, cudaStream_t st,
                                const uint32_t* cache_index = nullptr, uint32_t n_caches = 0);
cudaError_t launch_fetch_gather(const DeviceDir* d_dir, const uint64_t* src_off, const uint64_t* offsets,
                                const uint32_t* n_dev, uint32_t n, const uint64_t* total, uint8_t* staging,
                                int sm_count, cudaStream_t st);

}  // namespace speckv
