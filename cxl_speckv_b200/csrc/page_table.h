// page_table.h -- host page table of the KV region allocator.
//
// Same bookkeeping as the reference's SpeckvAllocator
// (host/include/speckv_allocator.hpp:29-67, host/src/speckv_allocator.cpp:11-138):
// a handle owns ceil(bytes / 4096) pages; page i of handle h has
//     virt_page_id = (h << 32) | (i << 12)                       (:24)
//     phys_page_id = 0x4000000000 + (h << 20) + (i << 12)        (:25)
// and flag bits 0 = in L1, 1 = in L2, 2 = compressed (speckv_allocator.hpp:26).
// `access` of a page that is in neither L1 nor L2 triggers a synchronous fetch
// and marks it L2 (:115-138).  Handles start at 1.
//
// What differs is the storage: pages of one handle are a dense vector and the
// virt-id lookup is arithmetic on the id (handle = id >> 32, index = (id >> 12)
// & 0xFFFFF) instead of a second std::unordered_map, so the same table can be
// mirrored to the GPU as a flat array of KvPage records for the batched lookup
// kernel (page_lookup.cu).
#pragma once

#include <cstddef>
#include <cstdint>
#include <unordered_map>
#include <vector>

namespace speckv {

constexpr uint64_t kPageSize = 4096;
constexpr uint64_t kPhysBase = 0x4000000000ULL;
constexpr uint32_t kFlagL1 = 1u, kFlagL2 = 2u, kFlagCompressed = 4u;

struct KvPage {              // == KvPageHandle, speckv_allocator.hpp:22-27 (24 bytes)
    uint64_t virt_page_id;
    uint64_t phys_page_id;
    uint32_t page_size;
    uint32_t flags;
};

struct KvAllocation {
    size_t size_bytes = 0;
    std::vector<KvPage> pages;
};

class PageTable {
public:
    uint64_t alloc(size_t bytes);                 // speckv_allocator.cpp:11-38
    bool free(uint64_t handle);                   // :40-52 (unknown handle: no-op)
    // :54-74.  Returns 0 for an unknown handle or an offset past the last page;
    // *fetched is set when the page had to be fetched (was in neither L1 nor L2).
    uint64_t access(uint64_t handle, uint64_t offset, size_t bytes, bool* fetched);
    KvAllocation* find(uint64_t handle);
    KvPage* find_page(uint64_t virt_page_id);     // page_table_.find, :105-113
    size_t num_allocations() const { return allocs_.size(); }
    uint64_t fetch_count() const { return fetches_; }
    void clear();

    static uint64_t virt_page_id(uint64_t handle, uint64_t i) { return (handle << 32) | (i << 12); }
    static uint64_t phys_page_id(uint64_t handle, uint64_t i) { return kPhysBase + (handle << 20) + (i << 12); }
    // The id a bound pool's page i is stored under in the host tier.  virt_page_id for i < 2^20; from there on
    // i << 12 reaches the handle bits and virt_page_id repeats the id of page i - 2^20 of the same handle (h odd) or
    // of handle h + 1 (h even).  Those pages take (h << 32) | ((i mod 2^20) << 12) | (i >> 20): its low 12 bits are
    // non-zero, so it equals no page-aligned id, and it is unique per (handle, page) for i < 2^32 (16 TiB).
    static uint64_t tier_key(uint64_t handle, uint64_t i) {
        return i < (1ull << 20) ? virt_page_id(handle, i) : (handle << 32) | ((i & 0xFFFFFull) << 12) | (i >> 20);
    }
    // gpu_addr of the fetch descriptor, speckv_allocator.cpp:124
    static uint64_t fetch_gpu_addr(uint64_t virt) { return 0x8000000000ULL + (virt & 0xFFFFFFFFFFFFULL); }

private:
    std::unordered_map<uint64_t, KvAllocation> allocs_;
    uint64_t next_handle_ = 1;
    uint64_t fetches_ = 0;
};

}  // namespace speckv
