// page_table.cpp -- see page_table.h.  Reference: host/src/speckv_allocator.cpp.
#include "page_table.h"

namespace speckv {

uint64_t PageTable::alloc(size_t bytes) {
    const uint64_t handle = next_handle_++;
    KvAllocation a;
    a.size_bytes = bytes;
    const size_t num_pages = (bytes + kPageSize - 1) / kPageSize;  // speckv_allocator.cpp:19
    a.pages.resize(num_pages);
    for (size_t i = 0; i < num_pages; ++i) {
        KvPage& p = a.pages[i];
        p.virt_page_id = virt_page_id(handle, i);
        p.phys_page_id = phys_page_id(handle, i);
        p.page_size = (uint32_t)kPageSize;
        p.flags = 0;
    }
    allocs_.emplace(handle, std::move(a));
    return handle;
}

bool PageTable::free(uint64_t handle) { return allocs_.erase(handle) != 0; }

KvAllocation* PageTable::find(uint64_t handle) {
    auto it = allocs_.find(handle);
    return it == allocs_.end() ? nullptr : &it->second;
}

KvPage* PageTable::find_page(uint64_t virt) {
    // ids are unambiguous for allocations below 4 GiB (page index < 2^20); beyond that
    // the reference's own map keys collide across handles as well.  (The host tier keys pool pages by
    // tier_key, which stays unique there.)
    KvAllocation* a = find(virt >> 32);
    if (!a) return nullptr;
    const uint64_t i = (virt & 0xFFFFFFFFULL) >> 12;
    if (i >= a->pages.size() || a->pages[i].virt_page_id != virt) return nullptr;
    return &a->pages[i];
}

uint64_t PageTable::access(uint64_t handle, uint64_t offset, size_t /*bytes*/, bool* fetched) {
    if (fetched) *fetched = false;
    KvAllocation* a = find(handle);
    if (!a) return 0;
    const uint64_t page_idx = offset / kPageSize, page_off = offset % kPageSize;
    if (page_idx >= a->pages.size()) return 0;
    KvPage& p = a->pages[page_idx];
    if ((p.flags & (kFlagL1 | kFlagL2)) == 0) {  // is_in_l1_or_l2, :105-113
        ++fetches_;                              // sync_fetch_page, :115-138
        p.flags |= kFlagL2;
        if (fetched) *fetched = true;
    }
    return p.phys_page_id + page_off;            // :73
}

void PageTable::clear() {
    allocs_.clear();
    next_handle_ = 1;
    fetches_ = 0;
}

}  // namespace speckv
