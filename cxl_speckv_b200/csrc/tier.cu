// tier.cu -- the host-DRAM tier standing in for the CXL memory pool (L3 of the reference).
//
// Reference behaviour being replaced: a KV page that is in neither L1 nor L2 is fetched from the
// CXL/FPGA side by one DMA descriptor per 4 KiB page with the COMPRESSED flag (descriptor flags
// bit1, driver/uapi/speckv_ioctl.h:14; SpeckvAllocator::sync_fetch_page,
// host/src/speckv_allocator.cpp:115-138; CXLMemoryManager::demote_to_l3 / promote_to_l1,
// src/cxl_memory/cxl_memory_manager.cpp:130-194) -- in the reference the transfer itself is a
// simulated ioctl.  Here it is real: offload = compress kernel -> pack kernel (payload bytes of all
// blocks back to back, 16 B aligned) -> ONE device-to-host copy into a pinned pool on a side
// stream; restore = ONE host-to-device copy per contiguous pool extent -> decompress straight from
// the packed stream (per-block byte offsets, no unpack pass).  Chunks are double-buffered so the
// PCIe copy of chunk i overlaps the codec kernels of chunk i+1.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/speckv_ext.h"
#include "cache_set.h"
#include "device_ctx.h"
#include "kv_codec.h"
#include "tier_fetch.h"

namespace speckv {

void runtime_unbind_tier(speckv_tier_t* tier);   // c_api.cu

namespace {

constexpr int kPackThreads = 256;
constexpr uint32_t kTierPage = 4096;

// exclusive scan of the 16-byte-rounded payload sizes, one CTA of 32 warps: every warp scans one contiguous
// segment tile by tile with no block barrier in between (its loads do not depend on the running sum, so they
// pipeline), the 32 segment totals are combined once and added in a second pass (the 44 us of a
// tile-serial scan with three block barriers per 1024 sizes was 12 % of a paged offload chunk).
// n_dev (optional, device): only the first min(*n_dev, n) sizes are scanned (the device fetch's request count).
__global__ void __launch_bounds__(1024)
pack_offsets_kernel(const uint32_t* __restrict__ comp_bytes, uint32_t n, const uint32_t* __restrict__ n_dev,
                    uint64_t* __restrict__ offsets, uint64_t* __restrict__ total) {
    __shared__ uint64_t warp_total[32];
    if (n_dev) n = min(n, *n_dev);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t seg = ((n + 31u) / 32u + 31u) & ~31u;          // per-warp segment, a multiple of 32
    const uint32_t s0 = min(n, (uint32_t)wid * seg), s1 = min(n, s0 + seg);
    uint64_t carry = 0;
#pragma unroll 4
    for (uint32_t base = s0; base < s1; base += 32) {
        const uint32_t i = base + lane;
        const uint64_t v = i < s1 ? (((uint64_t)comp_bytes[i] + 15u) & ~15ull) : 0ull;
        uint64_t inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (i < s1) offsets[i] = carry + inc - v;
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) warp_total[wid] = carry;
    __syncthreads();
    uint64_t before = 0, all = 0;
    for (int w = 0; w < 32; ++w) {
        const uint64_t t = warp_total[w];
        if (w < wid) before += t;
        all += t;
    }
    if (before)
        for (uint32_t i = s0 + lane; i < s1; i += 32) offsets[i] += before;   // this warp's own writes: no barrier needed
    if (tid == 0) *total = all;
}

// one warp per block: copy its payload (rounded up to 16 B) from the slot into the packed stream
__global__ void __launch_bounds__(kPackThreads)
pack_kernel(const uint8_t* __restrict__ slots, size_t slot_bytes, const uint32_t* __restrict__ comp_bytes,
            const uint64_t* __restrict__ offsets, uint32_t n, uint8_t* __restrict__ packed) {
    const uint32_t warps_per_cta = kPackThreads / 32;
    const int lane = threadIdx.x & 31;
    for (uint32_t g = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); g < n; g += gridDim.x * warps_per_cta) {
        const uint32_t nvec = (comp_bytes[g] + 15u) >> 4;
        const uint4* src = reinterpret_cast<const uint4*>(slots + (size_t)g * slot_bytes);
        uint4* dst = reinterpret_cast<uint4*>(packed + offsets[g]);
        for (uint32_t v = lane; v < nvec; v += 32) dst[v] = __ldg(src + v);
    }
}

struct Extent {
    uint64_t off, len;
};

// block id -> BlockRec: open addressing (key and record in one 32-byte entry: one cache line per probe),
// linear probing, backward-shift deletion, software prefetch for batches.  One record per 4 KiB page at the
// paged geometry (a million per offload call): with std::unordered_map the host bookkeeping (a node
// allocation and several cache misses per page) took longer than the PCIe copy it overlaps.
// With tracking on (the tier keeps a device copy for speckv_ext_tier_fetch) every slot a call writes is logged, so
// that only those go to the device; a grow marks the whole table.
class BlockMap {
public:
    BlockRec* find(uint64_t key) {
        if (cap_ == 0) return nullptr;
        for (size_t i = slot_of(key);; i = (i + 1) & (cap_ - 1)) {
            if (tab_[i].val.dtype == kDirEmpty) return nullptr;
            if (tab_[i].key == key) return &tab_[i].val;
        }
    }
    // insert or replace; returns true and the previous record when the key was present
    bool exchange(uint64_t key, const BlockRec& r, BlockRec* old) {
        if ((size_ + 1) * 10 > cap_ * 7) grow(cap_ ? cap_ * 2 : 1024);
        for (size_t i = slot_of(key);; i = (i + 1) & (cap_ - 1)) {
            if (tab_[i].val.dtype == kDirEmpty) {
                tab_[i].key = key;
                tab_[i].val = r;
                ++size_;
                mark(i);
                return false;
            }
            if (tab_[i].key == key) {
                if (old) *old = tab_[i].val;
                tab_[i].val = r;
                mark(i);
                return true;
            }
        }
    }
    void put(uint64_t key, const BlockRec& r) { exchange(key, r, nullptr); }
    bool erase(uint64_t key) {
        if (cap_ == 0) return false;
        size_t i = slot_of(key);
        for (;; i = (i + 1) & (cap_ - 1)) {
            if (tab_[i].val.dtype == kDirEmpty) return false;
            if (tab_[i].key == key) break;
        }
        // backward shift: pull later entries of the probe run into the hole
        for (size_t j = (i + 1) & (cap_ - 1);; j = (j + 1) & (cap_ - 1)) {
            if (tab_[j].val.dtype == kDirEmpty) break;
            const size_t home = slot_of(tab_[j].key);
            if (((j - home) & (cap_ - 1)) >= ((j - i) & (cap_ - 1))) {
                tab_[i] = tab_[j];
                mark(i);
                i = j;
            }
        }
        tab_[i].val.dtype = kDirEmpty;
        mark(i);
        --size_;
        return true;
    }
    void reserve(size_t n) {
        size_t want = 1024;
        while (want * 7 < n * 10) want *= 2;
        if (want > cap_) grow(want);
    }
    void prefetch(uint64_t key) const {
        if (cap_) __builtin_prefetch(&tab_[slot_of(key)]);
    }
    size_t size() const { return size_; }
    size_t capacity() const { return cap_; }
    const DirEntry* entries() const { return tab_.data(); }

    // dirty log for the device copy
    void set_tracking(bool on) { track_ = on; }
    void mark_all() {
        if (track_) {
            all_dirty_ = true;
            dirty_.clear();
        }
    }
    bool all_dirty() const { return all_dirty_; }
    const std::vector<size_t>& dirty() const { return dirty_; }
    void clear_dirty() {
        dirty_.clear();
        all_dirty_ = false;
    }

private:
    size_t slot_of(uint64_t k) const { return (size_t)dir_hash(k) & (cap_ - 1); }
    void mark(size_t i) {
        if (track_ && !all_dirty_) dirty_.push_back(i);
    }
    void grow(size_t ncap) {
        std::vector<DirEntry> old;
        old.swap(tab_);
        DirEntry e{};
        e.val.dtype = kDirEmpty;
        tab_.assign(ncap, e);
        cap_ = ncap;
        size_ = 0;
        if (track_) {   // slots all move: the device gets the whole table
            all_dirty_ = true;
            dirty_.clear();
        }
        for (const DirEntry& o : old)
            if (o.val.dtype != kDirEmpty) exchange(o.key, o.val, nullptr);
    }
    std::vector<DirEntry> tab_;
    size_t cap_ = 0, size_ = 0;
    bool track_ = false, all_dirty_ = false;
    std::vector<size_t> dirty_;
};
constexpr size_t kMapPrefetch = 16;   // look-ups in flight when a call walks a list of block ids

}  // namespace

struct Tier {
    std::mutex mu;
    int device = -1;
    uint8_t* pool = nullptr;      // pinned host memory
    size_t pool_bytes = 0, bump = 0;
    std::vector<Extent> free_list;                       // sorted by offset, coalesced
    BlockMap blocks;
    // device staging, two buffers for chunk double-buffering
    static constexpr int kBuf = 2;
    cudaStream_t copy_st[kBuf] = {};
    cudaEvent_t ev_kernel[kBuf] = {}, ev_copy[kBuf] = {};
    uint8_t* d_slots[kBuf] = {};
    uint8_t* d_packed[kBuf] = {};
    float* d_scales[kBuf] = {};
    uint32_t* d_comp[kBuf] = {};
    uint64_t* d_offsets[kBuf] = {};
    uint64_t* d_total[kBuf] = {};
    uint32_t* d_oel[kBuf] = {};                          // restore: decoded lengths of a chunk with ragged blocks
    // pinned host mirrors of the small per-chunk metadata
    float* h_scales[kBuf] = {};
    uint32_t* h_comp[kBuf] = {};
    uint64_t* h_offsets[kBuf] = {};
    uint64_t* h_total[kBuf] = {};
    uint32_t* h_oel[kBuf] = {};
    size_t cap_groups = 0, cap_slot_bytes = 0;           // per buffer
    int scheme = SPECKV_COMP_INT8_DELTA_RLE;             // what new offloads are stored under (speckv_ext_tier_set_scheme)
    speckv_tier_stats_t stats = {};
    // device copy of the block directory (speckv_ext_tier_enable_fetch); d_dir stays null while fetch is off, and
    // then nothing below is touched
    DeviceDir* d_dir = nullptr;                          // header the fetch kernels read the table through
    DeviceDir* h_dir = nullptr;                          // pinned source of header writes
    DirEntry* d_table = nullptr;
    size_t d_table_cap = 0;
    DirUpdate* h_upd = nullptr;                          // pinned staging of changed slots
    DirUpdate* d_upd = nullptr;
    size_t upd_cap = 0;
    const uint8_t* d_pool = nullptr;                     // device address of the pinned pool
    cudaStream_t dir_st = nullptr;                       // drop's updates (drop takes no stream)

    size_t alloc_pool(size_t len) {   // first fit in the free list, else bump; returns SIZE_MAX when full
        for (size_t i = 0; i < free_list.size(); ++i) {
            if (free_list[i].len >= len) {
                const size_t off = free_list[i].off;
                free_list[i].off += len;
                free_list[i].len -= len;
                if (free_list[i].len == 0) free_list.erase(free_list.begin() + i);
                return off;
            }
        }
        if (bump + len > pool_bytes) return SIZE_MAX;
        const size_t off = bump;
        bump += len;
        return off;
    }
    void free_pool(uint64_t off, uint64_t len) {
        if (len == 0) return;
        auto it = std::lower_bound(free_list.begin(), free_list.end(), off,
                                   [](const Extent& e, uint64_t o) { return e.off < o; });
        it = free_list.insert(it, Extent{off, len});
        if (it + 1 != free_list.end() && it->off + it->len == (it + 1)->off) {   // merge with the next extent
            it->len += (it + 1)->len;
            free_list.erase(it + 1);
        }
        if (it != free_list.begin() && (it - 1)->off + (it - 1)->len == it->off) {   // and with the previous one
            (it - 1)->len += it->len;
            it = free_list.erase(it) - 1;
        }
        if (it->off + it->len == bump) {   // give the tail back to the bump pointer
            bump = it->off;
            free_list.erase(it);
        }
    }
    void release_staging() {
        for (int b = 0; b < kBuf; ++b) {
            cudaFree(d_slots[b]); cudaFree(d_packed[b]); cudaFree(d_scales[b]); cudaFree(d_comp[b]);
            cudaFree(d_offsets[b]); cudaFree(d_total[b]); cudaFree(d_oel[b]);
            cudaFreeHost(h_scales[b]); cudaFreeHost(h_comp[b]); cudaFreeHost(h_offsets[b]); cudaFreeHost(h_total[b]);
            cudaFreeHost(h_oel[b]);
            d_slots[b] = d_packed[b] = nullptr; d_scales[b] = nullptr; d_comp[b] = nullptr;
            d_offsets[b] = d_total[b] = nullptr; h_scales[b] = nullptr; h_comp[b] = nullptr;
            h_offsets[b] = h_total[b] = nullptr; d_oel[b] = h_oel[b] = nullptr;
        }
        cap_groups = cap_slot_bytes = 0;
    }
    cudaError_t ensure_staging(size_t groups, size_t slot_bytes) {
        if (groups <= cap_groups && groups * slot_bytes <= cap_slot_bytes) return cudaSuccess;
        release_staging();
        cudaError_t e = cudaSuccess;
        for (int b = 0; b < kBuf && e == cudaSuccess; ++b) {
            if ((e = cudaMalloc((void**)&d_slots[b], groups * slot_bytes)) != cudaSuccess) break;
            if ((e = cudaMalloc((void**)&d_packed[b], groups * slot_bytes)) != cudaSuccess) break;
            if ((e = cudaMalloc((void**)&d_scales[b], groups * 4)) != cudaSuccess) break;
            if ((e = cudaMalloc((void**)&d_comp[b], groups * 4)) != cudaSuccess) break;
            if ((e = cudaMalloc((void**)&d_offsets[b], groups * 8)) != cudaSuccess) break;
            if ((e = cudaMalloc((void**)&d_total[b], 8)) != cudaSuccess) break;
            if ((e = cudaMalloc((void**)&d_oel[b], groups * 4)) != cudaSuccess) break;
            if ((e = cudaHostAlloc((void**)&h_scales[b], groups * 4, cudaHostAllocDefault)) != cudaSuccess) break;
            if ((e = cudaHostAlloc((void**)&h_comp[b], groups * 4, cudaHostAllocDefault)) != cudaSuccess) break;
            if ((e = cudaHostAlloc((void**)&h_offsets[b], groups * 8, cudaHostAllocDefault)) != cudaSuccess) break;
            if ((e = cudaHostAlloc((void**)&h_total[b], 8, cudaHostAllocDefault)) != cudaSuccess) break;
            if ((e = cudaHostAlloc((void**)&h_oel[b], groups * 4, cudaHostAllocDefault)) != cudaSuccess) break;
        }
        if (e != cudaSuccess) {
            release_staging();
            return e;
        }
        cap_groups = groups;
        cap_slot_bytes = groups * slot_bytes;
        return cudaSuccess;
    }

    // Bring the device directory up to date with the host map on st and wait for it.  Changed slots travel as
    // (slot, entry) records and are applied by a scatter kernel; after a grow, or when many slots changed, the whole
    // table goes.  A grown table gets a new device table and the header is pointed at it; the old one is freed once
    // that has completed, so a graph captured before the grow keeps working.
    cudaError_t sync_dir(cudaStream_t st) {
        if (!d_dir) return cudaSuccess;
        const size_t cap = blocks.capacity();
        const std::vector<size_t>& dirty = blocks.dirty();
        cudaError_t e = cudaSuccess;
        DirEntry* old = nullptr;
        const size_t old_cap = d_table_cap;
        const bool moved = cap != d_table_cap;   // a grow (or the first upload): a new device table
        if (moved || blocks.all_dirty() || dirty.size() * 4 >= cap) {
            if (moved) {
                DirEntry* nt = nullptr;
                if ((e = cudaMalloc((void**)&nt, cap * sizeof(DirEntry))) != cudaSuccess) return e;
                old = d_table;
                d_table = nt;
                d_table_cap = cap;
                *h_dir = DeviceDir{d_table, cap - 1, d_pool};
            }
            e = cudaMemcpyAsync(d_table, blocks.entries(), cap * sizeof(DirEntry), cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess && moved) e = cudaMemcpyAsync(d_dir, h_dir, sizeof(DeviceDir), cudaMemcpyHostToDevice, st);
        } else if (!dirty.empty()) {
            const size_t n = dirty.size();
            if (n > upd_cap) {
                cudaFreeHost(h_upd);
                cudaFree(d_upd);
                h_upd = nullptr;
                d_upd = nullptr;
                upd_cap = 0;
                const size_t c = std::max(n, (size_t)4096);
                if ((e = cudaHostAlloc((void**)&h_upd, c * sizeof(DirUpdate), cudaHostAllocDefault)) != cudaSuccess) return e;
                if ((e = cudaMalloc((void**)&d_upd, c * sizeof(DirUpdate))) != cudaSuccess) return e;
                upd_cap = c;
            }
            const DirEntry* tab = blocks.entries();
            for (size_t k = 0; k < n; ++k) h_upd[k] = DirUpdate{dirty[k], tab[dirty[k]]};
            e = cudaMemcpyAsync(d_upd, h_upd, n * sizeof(DirUpdate), cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = launch_dir_apply(d_dir, d_upd, n, st);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            if (moved) {   // the header may still name the old table: keep it, retry the whole upload next time
                cudaFree(d_table);
                d_table = old;
                d_table_cap = old_cap;
            }
            return e;
        }
        if (old) cudaFree(old);
        blocks.clear_dirty();
        return cudaSuccess;
    }
    void release_dir() {
        cudaFree(d_dir); cudaFree(d_table); cudaFree(d_upd);
        cudaFreeHost(h_dir); cudaFreeHost(h_upd);
        if (dir_st) cudaStreamDestroy(dir_st);
        d_dir = nullptr; d_table = nullptr; d_upd = nullptr; h_dir = nullptr; h_upd = nullptr; dir_st = nullptr;
        d_table_cap = upd_cap = 0;
        blocks.set_tracking(false);
        blocks.clear_dirty();
    }
};

}  // namespace speckv

using namespace speckv;

struct speckv_tier {
    Tier t;
};

static size_t tier_chunk_groups(size_t slot_bytes, size_t n_groups) {
    const size_t target = 128ull << 20;   // ~128 MiB of payload per chunk
    size_t c = slot_bytes ? target / slot_bytes : n_groups;
    if (c < 1) c = 1;
    return c < n_groups ? c : n_groups;
}

extern "C" {

speckv_status_t speckv_ext_tier_create(size_t pool_bytes, speckv_tier_t** out_tier) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!out_tier || pool_bytes == 0) return SPECKV_ERR_INVAL;
    speckv_tier* h = new speckv_tier();
    Tier& t = h->t;
    cudaError_t e = cudaGetDevice(&t.device);
    if (e == cudaSuccess) e = cudaHostAlloc((void**)&t.pool, pool_bytes, cudaHostAllocPortable);
    for (int b = 0; b < Tier::kBuf && e == cudaSuccess; ++b) {
        e = cudaStreamCreateWithFlags(&t.copy_st[b], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t.ev_kernel[b], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t.ev_copy[b], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        speckv_ext_tier_destroy(h);
        return status_of(e);
    }
    t.pool_bytes = pool_bytes;
    t.stats.pool_bytes = pool_bytes;
    *out_tier = h;
    return SPECKV_OK;
}

void speckv_ext_tier_destroy(speckv_tier_t* tier) {
    if (!tier) return;
    speckv::runtime_unbind_tier(tier);   // pools bound to this tier (speckv_ext_bind_pool) forget it before it is freed
    Tier& t = tier->t;
    t.release_staging();
    t.release_dir();
    for (int b = 0; b < Tier::kBuf; ++b) {
        if (t.copy_st[b]) cudaStreamDestroy(t.copy_st[b]);
        if (t.ev_kernel[b]) cudaEventDestroy(t.ev_kernel[b]);
        if (t.ev_copy[b]) cudaEventDestroy(t.ev_copy[b]);
    }
    if (t.pool) cudaFreeHost(t.pool);
    cudaGetLastError();
    delete tier;
}

static speckv_status_t tier_offload_impl(speckv_tier_t* tier, const KvBlocks& blocks, speckv_dtype_t dtype,
                                         size_t group_elems, size_t n_groups, const uint64_t* h_block_ids,
                                         void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!tier || !h_block_ids || (!blocks.base && !blocks.set && n_groups) || dtype < 0 || dtype > 2 || group_elems == 0 ||
        group_elems >= (1ull << 31))
        return SPECKV_ERR_INVAL;
    if (n_groups == 0) return SPECKV_OK;
    Tier& t = tier->t;
    std::lock_guard<std::mutex> lk(t.mu);
    const int scheme = t.scheme;
    if (scheme == SPECKV_COMP_FP16 && (blocks.block_table || blocks.group_len || dtype == SPECKV_DTYPE_F32))
        return SPECKV_ERR_INVAL;   // raw passthrough: no gather or ragged form
    const size_t slot = speckv_ext_slot_bytes(group_elems, (speckv_comp_scheme_t)scheme);
    const size_t esz = dtype == SPECKV_DTYPE_F32 ? 4 : 2;
    const size_t cg = tier_chunk_groups(slot, n_groups);
    cudaError_t e = t.ensure_staging(cg, slot);
    if (e != cudaSuccess) return status_of(e);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const auto t0 = std::chrono::steady_clock::now();
    uint64_t stored = 0;
    speckv_status_t rc = SPECKV_OK;
    t.blocks.reserve(t.blocks.size() + n_groups);

    // finish chunk `c` that was staged in buffer b: wait for its metadata, place it in the pool,
    // start the payload copy and record the blocks
    auto finish = [&](size_t g0, size_t ng, int b) -> speckv_status_t {
        cudaError_t e2 = cudaStreamSynchronize(t.copy_st[b]);   // metadata (offsets, sizes, scales, total) on the host
        if (e2 != cudaSuccess) return status_of(e2);
        const uint64_t total = *t.h_total[b];
        if (total == ~0ull) return SPECKV_ERR_DRIVER;            // the packed emission's look-back gave up (kv_codec_fast.cu, pack_place)
        const size_t off = t.alloc_pool(total);
        if (off == SIZE_MAX) return SPECKV_ERR_NOMEM;
        e2 = cudaMemcpyAsync(t.pool + off, t.d_packed[b], total, cudaMemcpyDeviceToHost, t.copy_st[b]);
        if (e2 != cudaSuccess) return status_of(e2);
        cudaEventRecord(t.ev_copy[b], t.copy_st[b]);
        // bookkeeping while the copy runs; re-offloading a block id replaces its previous copy (whose pool
        // space becomes reusable from the next chunk on)
        for (size_t i = 0; i < ng; ++i) {
            if (i + kMapPrefetch < ng) t.blocks.prefetch(h_block_ids[g0 + i + kMapPrefetch]);
            BlockRec r, old;
            r.pool_off = off + t.h_offsets[b][i];
            r.comp_bytes = t.h_comp[b][i];
            r.scale = t.h_scales[b][i];
            r.group_elems = (uint32_t)group_elems;
            r.dtype = (int)dtype | (scheme << 8) | (blocks.group_len ? BlockRec::kRagged : 0);
            if (t.blocks.exchange(h_block_ids[g0 + i], r, &old)) {
                t.stats.used_bytes -= ((uint64_t)old.comp_bytes + 15u) & ~15ull;
                // an id listed twice in this chunk: its first copy is part of the transfer in flight, so its
                // bytes stay allocated until the tier is dropped (other streams must not write there yet)
                if (old.pool_off < off || old.pool_off >= off + total)
                    t.free_pool(old.pool_off, ((uint64_t)old.comp_bytes + 15u) & ~15ull);
            }
        }
        stored += total;
        t.stats.used_bytes += total;
        return SPECKV_OK;
    };

    size_t chunk = 0, prev_g0 = 0, prev_ng = 0;
    int prev_b = -1;
    for (size_t g0 = 0; g0 < n_groups && rc == SPECKV_OK; g0 += cg, ++chunk) {
        const size_t ng = std::min(cg, n_groups - g0);
        const int b = (int)(chunk % Tier::kBuf);
        // buffer b is free once the payload copy of chunk - 2 has completed
        cudaStreamWaitEvent(st, t.ev_copy[b], 0);
        CodecArgs a(slot, group_elems, ng, dtype, scheme);
        blocks.bind(a, false, g0, esz);   // ragged: slots + scan + pack (no packed emission)
        a.payload = t.d_slots[b];
        a.scales = t.d_scales[b];
        a.comp_bytes = t.d_comp[b];
        if (compress_packed_supported(a)) {
            // 4 KiB page groups: the compress kernel places the payloads itself (look-back over per-CTA totals), the
            // packed stream is written once.  A group the generic kernel encodes keeps a whole slot inside the
            // stream; the bytes behind its payload stay allocated in the pool until the tier is dropped (rare:
            // non-finite or out-of-range scales).
            a.payload = t.d_packed[b];
            a.pack_offsets = t.d_offsets[b];
            a.pack_total = t.d_total[b];
            if ((e = launch_compress(a, st)) != cudaSuccess) { rc = status_of(e); break; }
        } else {
            if ((e = launch_compress(a, st)) != cudaSuccess) { rc = status_of(e); break; }
            pack_offsets_kernel<<<1, 1024, 0, st>>>(t.d_comp[b], (uint32_t)ng, nullptr, t.d_offsets[b], t.d_total[b]);
            const int grid = (int)std::min<size_t>((ng + 7) / 8, (size_t)current_sm_count() * 8);
            pack_kernel<<<grid, kPackThreads, 0, st>>>(t.d_slots[b], slot, t.d_comp[b], t.d_offsets[b], (uint32_t)ng, t.d_packed[b]);
            count_launch(2);
        }
        cudaEventRecord(t.ev_kernel[b], st);
        cudaStreamWaitEvent(t.copy_st[b], t.ev_kernel[b], 0);
        cudaMemcpyAsync(t.h_total[b], t.d_total[b], 8, cudaMemcpyDeviceToHost, t.copy_st[b]);
        cudaMemcpyAsync(t.h_offsets[b], t.d_offsets[b], ng * 8, cudaMemcpyDeviceToHost, t.copy_st[b]);
        cudaMemcpyAsync(t.h_comp[b], t.d_comp[b], ng * 4, cudaMemcpyDeviceToHost, t.copy_st[b]);
        cudaMemcpyAsync(t.h_scales[b], t.d_scales[b], ng * 4, cudaMemcpyDeviceToHost, t.copy_st[b]);
        if (prev_b >= 0) rc = finish(prev_g0, prev_ng, prev_b);   // overlaps with this chunk's kernels
        prev_g0 = g0;
        prev_ng = ng;
        prev_b = b;
    }
    if (rc == SPECKV_OK && prev_b >= 0) rc = finish(prev_g0, prev_ng, prev_b);
    for (int b = 0; b < Tier::kBuf; ++b) {
        cudaError_t e2 = cudaStreamSynchronize(t.copy_st[b]);
        if (rc == SPECKV_OK && e2 != cudaSuccess) rc = status_of(e2);
    }
    if ((e = t.sync_dir(st)) != cudaSuccess && rc == SPECKV_OK) rc = status_of(e);   // the records this call changed
    if ((e = cudaGetLastError()) != cudaSuccess && rc == SPECKV_OK) rc = status_of(e);
    uint64_t raw = (uint64_t)n_groups * group_elems * esz;
    if (rc == SPECKV_OK && blocks.group_len) {   // ragged: count the valid bytes (the lengths live on the device)
        std::vector<uint32_t> len(n_groups);
        e = cudaMemcpyAsync(len.data(), blocks.group_len, n_groups * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = status_of(e);
        raw = 0;
        for (uint32_t l : len) raw += (uint64_t)std::min<size_t>(l, group_elems) * esz;
    }
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (rc == SPECKV_OK) {
        t.stats.blocks = t.blocks.size();
        t.stats.bytes_offloaded_raw += raw;
        t.stats.bytes_offloaded_stored += stored;
        t.stats.last_offload_ms = ms;
        t.stats.last_offload_stored_bytes = stored;
    }
    return rc;
}

speckv_status_t speckv_ext_tier_offload(speckv_tier_t* tier, const void* d_in, speckv_dtype_t dtype, size_t group_elems,
                                        size_t n_groups, const uint64_t* h_block_ids, void* cuda_stream) {
    return tier_offload_impl(tier, KvBlocks{d_in}, dtype, group_elems, n_groups, h_block_ids, cuda_stream);
}

speckv_status_t speckv_ext_tier_offload_paged(speckv_tier_t* tier, const void* d_cache, const uint32_t* d_block_table,
                                              speckv_dtype_t dtype, size_t group_elems, size_t n_blocks,
                                              const uint64_t* h_block_ids, void* cuda_stream) {
    if (!d_block_table && n_blocks) return SPECKV_ERR_INVAL;
    return tier_offload_impl(tier, KvBlocks{d_cache, d_block_table}, dtype, group_elems, n_blocks, h_block_ids, cuda_stream);
}

speckv_status_t speckv_ext_tier_offload_ragged(speckv_tier_t* tier, const void* d_in, const uint32_t* d_block_table,
                                               const uint32_t* d_group_len, speckv_dtype_t dtype, size_t group_elems,
                                               size_t n_blocks, const uint64_t* h_block_ids, void* cuda_stream) {
    if (!d_group_len && n_blocks) return device_count() <= 0 ? SPECKV_ERR_DRIVER : SPECKV_ERR_INVAL;
    return tier_offload_impl(tier, KvBlocks{d_in, d_block_table, d_group_len}, dtype, group_elems, n_blocks, h_block_ids,
                             cuda_stream);
}

static speckv_status_t tier_restore_impl(speckv_tier_t* tier, const uint64_t* h_block_ids, size_t n_groups,
                                         size_t group_elems, speckv_dtype_t dtype, const KvBlocks& blocks,
                                         void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!tier || !h_block_ids || (!blocks.base && !blocks.set && n_groups) || dtype < 0 || dtype > 2 || group_elems == 0)
        return SPECKV_ERR_INVAL;
    if (n_groups == 0) return SPECKV_OK;
    Tier& t = tier->t;
    std::lock_guard<std::mutex> lk(t.mu);
    const size_t slot = speckv_ext_slot_bytes(group_elems, SPECKV_COMP_INT8_DELTA_RLE);   // the largest slot of any scheme
    const size_t esz = dtype == SPECKV_DTYPE_F32 ? 4 : 2;
    const size_t cg = tier_chunk_groups(slot, n_groups);
    cudaError_t e = t.ensure_staging(cg, slot);
    if (e != cudaSuccess) return status_of(e);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const auto t0 = std::chrono::steady_clock::now();
    uint64_t moved = 0, raw = 0;
    size_t chunk = 0;
    size_t oel_pending[Tier::kBuf] = {};   // decoded lengths of a chunk with ragged blocks, waiting in h_oel[b]
    auto take_oel = [&](int b) {
        for (size_t i = 0; i < oel_pending[b]; ++i) raw += (uint64_t)t.h_oel[b][i] * esz;
        oel_pending[b] = 0;
    };
    for (size_t g0 = 0, ng = 0; g0 < n_groups; g0 += ng, ++chunk) {
        ng = std::min(cg, n_groups - g0);
        const int b = (int)(chunk % Tier::kBuf);
        int scheme = -1;   // of the chunk: blocks stored under another scheme start the next chunk
        // the pinned metadata mirrors and the staging of buffer b are reusable once its previous
        // H2D copies and decompress have completed
        if ((e = cudaStreamSynchronize(t.copy_st[b])) != cudaSuccess) return status_of(e);
        cudaEventSynchronize(t.ev_kernel[b]);
        take_oel(b);
        bool any_ragged = false;
        // host: look the blocks up, lay them out back to back in the staging buffer (in request order)
        // and merge copies whose pool ranges are contiguous
        uint64_t dst = 0;
        uint64_t run_src = 0, run_dst = 0, run_len = 0;
        for (size_t i = 0; i < ng; ++i) {
            if (i + kMapPrefetch < ng) t.blocks.prefetch(h_block_ids[g0 + i + kMapPrefetch]);
            const BlockRec* rec = t.blocks.find(h_block_ids[g0 + i]);
            if (!rec || rec->group_elems != group_elems) return SPECKV_ERR_GENERAL;   // unknown, raw, or other geometry
            const BlockRec& r = *rec;
            any_ragged |= r.ragged();
            if (scheme < 0) scheme = r.scheme();
            else if (r.scheme() != scheme) {
                ng = i;
                break;
            }
            const uint64_t len = ((uint64_t)r.comp_bytes + 15u) & ~15ull;
            t.h_offsets[b][i] = dst;
            t.h_comp[b][i] = r.comp_bytes;
            t.h_scales[b][i] = r.scale;
            if (run_len && r.pool_off == run_src + run_len) {
                run_len += len;
            } else {
                if (run_len) cudaMemcpyAsync(t.d_packed[b] + run_dst, t.pool + run_src, run_len, cudaMemcpyHostToDevice, t.copy_st[b]);
                run_src = r.pool_off;
                run_dst = dst;
                run_len = len;
            }
            dst += len;
        }
        if (run_len) cudaMemcpyAsync(t.d_packed[b] + run_dst, t.pool + run_src, run_len, cudaMemcpyHostToDevice, t.copy_st[b]);
        moved += dst;
        cudaMemcpyAsync(t.d_offsets[b], t.h_offsets[b], ng * 8, cudaMemcpyHostToDevice, t.copy_st[b]);
        cudaMemcpyAsync(t.d_comp[b], t.h_comp[b], ng * 4, cudaMemcpyHostToDevice, t.copy_st[b]);
        cudaMemcpyAsync(t.d_scales[b], t.h_scales[b], ng * 4, cudaMemcpyHostToDevice, t.copy_st[b]);
        cudaEventRecord(t.ev_copy[b], t.copy_st[b]);
        cudaStreamWaitEvent(st, t.ev_copy[b], 0);
        CodecArgs a(slot, group_elems, ng, dtype, scheme);
        blocks.bind(a, true, g0, esz);
        a.payload = t.d_packed[b];
        a.scales = t.d_scales[b];
        a.comp_bytes = t.d_comp[b];
        a.slot_offsets = t.d_offsets[b];
        if (scheme == SPECKV_COMP_FP16 && (blocks.block_table || dtype == SPECKV_DTYPE_F32)) return SPECKV_ERR_INVAL;
        // a chunk holding ragged blocks counts what was decoded; otherwise every block is a whole group
        if (any_ragged) a.out_elems = t.d_oel[b];
        if ((e = launch_decompress(a, st)) != cudaSuccess) return status_of(e);
        if (any_ragged) {
            if ((e = cudaMemcpyAsync(t.h_oel[b], t.d_oel[b], ng * 4, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return status_of(e);
            oel_pending[b] = ng;
        } else {
            raw += (uint64_t)ng * group_elems * esz;
        }
        cudaEventRecord(t.ev_kernel[b], st);
    }
    e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return status_of(e);
    for (int b = 0; b < Tier::kBuf; ++b) take_oel(b);
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    t.stats.bytes_restored_raw += raw;
    t.stats.bytes_restored_stored += moved;
    t.stats.last_restore_ms = ms;
    t.stats.last_restore_stored_bytes = moved;
    return SPECKV_OK;
}

speckv_status_t speckv_ext_tier_restore(speckv_tier_t* tier, const uint64_t* h_block_ids, size_t n_groups,
                                        size_t group_elems, speckv_dtype_t dtype, void* d_out, void* cuda_stream) {
    return tier_restore_impl(tier, h_block_ids, n_groups, group_elems, dtype, KvBlocks{d_out}, cuda_stream);
}

speckv_status_t speckv_ext_tier_restore_paged(speckv_tier_t* tier, const uint64_t* h_block_ids, size_t n_blocks,
                                              size_t group_elems, speckv_dtype_t dtype, void* d_cache,
                                              const uint32_t* d_block_table, void* cuda_stream) {
    if (!d_block_table && n_blocks) return SPECKV_ERR_INVAL;
    return tier_restore_impl(tier, h_block_ids, n_blocks, group_elems, dtype, KvBlocks{d_cache, d_block_table}, cuda_stream);
}

// the set forms: geometry and dtype from the set, the rest shared with the single-cache forms
speckv_status_t speckv_ext_tier_offload_set(speckv_tier_t* tier, const speckv_cache_set_t* set,
                                            const uint32_t* d_cache_index, const uint32_t* d_block_table,
                                            const uint32_t* d_group_len, size_t n_blocks, const uint64_t* h_block_ids,
                                            void* cuda_stream) {
    const speckv_status_t rc = check_set(set, d_cache_index, d_block_table, n_blocks);
    if (rc != SPECKV_OK) return rc;
    return tier_offload_impl(tier, KvBlocks{nullptr, d_block_table, d_group_len, set, d_cache_index},
                             (speckv_dtype_t)set->dtype, set->block_elems, n_blocks, h_block_ids, cuda_stream);
}

speckv_status_t speckv_ext_tier_restore_set(speckv_tier_t* tier, const uint64_t* h_block_ids, size_t n_blocks,
                                            const speckv_cache_set_t* set, const uint32_t* d_cache_index,
                                            const uint32_t* d_block_table, void* cuda_stream) {
    const speckv_status_t rc = check_set(set, d_cache_index, d_block_table, n_blocks);
    if (rc != SPECKV_OK) return rc;
    return tier_restore_impl(tier, h_block_ids, n_blocks, set->block_elems, (speckv_dtype_t)set->dtype,
                             KvBlocks{nullptr, d_block_table, nullptr, set, d_cache_index}, cuda_stream);
}

speckv_status_t speckv_ext_tier_drop(speckv_tier_t* tier, const uint64_t* h_block_ids, size_t n) {
    if (!tier || (!h_block_ids && n)) return SPECKV_ERR_INVAL;
    Tier& t = tier->t;
    std::lock_guard<std::mutex> lk(t.mu);
    for (size_t i = 0; i < n; ++i) {
        const BlockRec* rec = t.blocks.find(h_block_ids[i]);
        if (!rec) continue;   // like speckv_free: dropping an unknown block is not an error
        const uint64_t len = ((uint64_t)rec->comp_bytes + 15u) & ~15ull;
        t.free_pool(rec->pool_off, len);
        t.stats.used_bytes -= len;
        t.blocks.erase(h_block_ids[i]);
    }
    t.stats.blocks = t.blocks.size();
    return status_of(t.sync_dir(t.dir_st));
}

// ---- descriptor interface (driver/uapi/speckv_ioctl.h:10-15, host/src/speckv_driver.cpp:24-47) ----
static std::atomic<uint32_t> g_dma_done{0};

speckv_status_t speckv_ext_submit_dma_batch(speckv_tier_t* tier, const speckv_dma_desc_t* h_descs, uint32_t count,
                                            void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!tier || (!h_descs && count)) return SPECKV_ERR_INVAL;
    if (count > 4096) return SPECKV_ERR_INVAL;                  // handle_dma_batch: -EINVAL, speckv_kernel_module.c:65-66
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    for (uint32_t i = 0; i < count; ++i) {
        const speckv_dma_desc_t& d = h_descs[i];
        if (d.bytes == 0 || d.bytes % kTierPage || !d.gpu_addr) return SPECKV_ERR_INVAL;
        const uint32_t pages = d.bytes / kTierPage;
        std::vector<uint64_t> ids(pages);
        for (uint32_t p = 0; p < pages; ++p) ids[p] = d.fpga_addr + (uint64_t)p * kTierPage;
        void* gpu = reinterpret_cast<void*>(d.gpu_addr);
        speckv_status_t rc;
        if (d.flags & SPECKV_DMA_COMPRESSED) {
            rc = (d.flags & SPECKV_DMA_WRITE)
                     ? speckv_ext_tier_offload(tier, gpu, SPECKV_DTYPE_F16, kTierPage / 2, pages, ids.data(), st)
                     : speckv_ext_tier_restore(tier, ids.data(), pages, kTierPage / 2, SPECKV_DTYPE_F16, gpu, st);
        } else {
            // uncompressed pages: straight copies between the device and the pool
            Tier& t = tier->t;
            std::lock_guard<std::mutex> lk(t.mu);
            rc = SPECKV_OK;
            for (uint32_t p = 0; p < pages && rc == SPECKV_OK; ++p) {
                uint8_t* dev = static_cast<uint8_t*>(gpu) + (size_t)p * kTierPage;
                const BlockRec* it = t.blocks.find(ids[p]);
                if (d.flags & SPECKV_DMA_WRITE) {
                    if (it) {
                        t.free_pool(it->pool_off, ((uint64_t)it->comp_bytes + 15u) & ~15ull);
                        t.stats.used_bytes -= ((uint64_t)it->comp_bytes + 15u) & ~15ull;
                        t.blocks.erase(ids[p]);
                    }
                    const size_t off = t.alloc_pool(kTierPage);
                    if (off == SIZE_MAX) { rc = SPECKV_ERR_NOMEM; break; }
                    rc = status_of(cudaMemcpyAsync(t.pool + off, dev, kTierPage, cudaMemcpyDeviceToHost, st));
                    BlockRec r;
                    r.pool_off = off;
                    r.comp_bytes = kTierPage;
                    r.scale = 1.0f;
                    r.group_elems = 0;
                    r.dtype = SPECKV_DTYPE_F16;
                    t.blocks.put(ids[p], r);
                    t.stats.used_bytes += kTierPage;
                } else {
                    if (!it || it->group_elems != 0) { rc = SPECKV_ERR_GENERAL; break; }
                    rc = status_of(cudaMemcpyAsync(dev, t.pool + it->pool_off, kTierPage, cudaMemcpyHostToDevice, st));
                }
            }
            const speckv_status_t rd = status_of(t.sync_dir(st));
            if (rc == SPECKV_OK) rc = rd;
            if (rc == SPECKV_OK) rc = status_of(cudaStreamSynchronize(st));
            t.stats.blocks = t.blocks.size();
        }
        if (rc != SPECKV_OK) return rc;
        g_dma_done.fetch_add(1);
    }
    return SPECKV_OK;
}

uint32_t speckv_ext_poll_complete(void) { return g_dma_done.exchange(0); }   // handle_poll_done, :194-213

speckv_status_t speckv_ext_tier_set_scheme(speckv_tier_t* tier, speckv_comp_scheme_t scheme) {
    if (!tier || (int)scheme < 0 || (int)scheme > 4) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(tier->t.mu);
    tier->t.scheme = (int)scheme;
    return SPECKV_OK;
}

void speckv_ext_tier_get_stats(speckv_tier_t* tier, speckv_tier_stats_t* out) {
    if (!tier || !out) return;
    std::lock_guard<std::mutex> lk(tier->t.mu);
    *out = tier->t.stats;
}

// ---- device-side fetch -----------------------------------------------------------------------------------------
speckv_status_t speckv_ext_tier_enable_fetch(speckv_tier_t* tier, void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!tier) return SPECKV_ERR_INVAL;
    Tier& t = tier->t;
    std::lock_guard<std::mutex> lk(t.mu);
    if (t.d_dir) return SPECKV_OK;
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return status_of(e);
    if (dev != t.device) return SPECKV_ERR_INVAL;
    // the fetch kernels read the pinned pool directly: it needs a device address
    int uva = 0, can_map = 0;
    cudaDeviceGetAttribute(&uva, cudaDevAttrUnifiedAddressing, dev);
    cudaDeviceGetAttribute(&can_map, cudaDevAttrCanMapHostMemory, dev);
    if (!uva || !can_map) return SPECKV_ERR_DRIVER;
    void* dpool = nullptr;
    if ((e = cudaHostGetDevicePointer(&dpool, t.pool, 0)) != cudaSuccess) return status_of(e);
    t.d_pool = static_cast<const uint8_t*>(dpool);
    e = cudaMalloc((void**)&t.d_dir, sizeof(DeviceDir));
    if (e == cudaSuccess) e = cudaHostAlloc((void**)&t.h_dir, sizeof(DeviceDir), cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&t.dir_st, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
        t.blocks.reserve(t.blocks.size());   // a table of at least 1024 slots: the device table is never empty
        t.blocks.set_tracking(true);
        t.blocks.mark_all();
        e = t.sync_dir(static_cast<cudaStream_t>(cuda_stream));
    }
    if (e != cudaSuccess) {
        t.release_dir();
        return status_of(e);
    }
    return SPECKV_OK;
}

size_t speckv_ext_tier_fetch_workspace_bytes(size_t max_requests, size_t group_elems) {
    // [staging: one slot per request][offsets u64][pool offsets u64][total u64][sizes u32][scales f32]
    return max_requests * (speckv_ext_slot_bytes(group_elems, SPECKV_COMP_INT8_DELTA_RLE) + 24) + 8;
}

static speckv_status_t tier_fetch_impl(speckv_tier_t* tier, const uint64_t* d_block_ids, const uint32_t* d_n_requests,
                                       size_t max_requests, size_t group_elems, speckv_dtype_t dtype,
                                       speckv_comp_scheme_t scheme, const KvBlocks& blocks, uint32_t* d_out_elems,
                                       uint8_t* d_status, void* d_workspace, size_t workspace_bytes, void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!tier || dtype < 0 || dtype > 2 || (int)scheme < 1 || (int)scheme > 4 || group_elems == 0 ||
        group_elems >= (1ull << 31) || max_requests >= (1ull << 31))
        return SPECKV_ERR_INVAL;
    Tier& t = tier->t;
    std::lock_guard<std::mutex> lk(t.mu);
    if (!t.d_dir) return SPECKV_ERR_INVAL;   // speckv_ext_tier_enable_fetch first
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != t.device) return SPECKV_ERR_INVAL;
    if (max_requests == 0) return SPECKV_OK;
    if (!d_block_ids || (!blocks.base && !blocks.set) || !d_workspace || (reinterpret_cast<uintptr_t>(d_workspace) & 15) ||
        workspace_bytes < speckv_ext_tier_fetch_workspace_bytes(max_requests, group_elems))
        return SPECKV_ERR_INVAL;
    const size_t n = max_requests;
    const size_t slot = speckv_ext_slot_bytes(group_elems, SPECKV_COMP_INT8_DELTA_RLE);   // the largest of any scheme
    uint8_t* staging = static_cast<uint8_t*>(d_workspace);
    uint64_t* offsets = reinterpret_cast<uint64_t*>(staging + n * slot);
    uint64_t* src_off = offsets + n;
    uint64_t* total = src_off + n;
    uint32_t* comp = reinterpret_cast<uint32_t*>(total + 1);
    float* scales = reinterpret_cast<float*>(comp + n);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    cudaError_t e = launch_fetch_lookup(t.d_dir, d_block_ids, d_n_requests, (uint32_t)n, (uint32_t)group_elems, dtype,
                                        (int)scheme, slot, src_off, comp, scales, d_status, st, blocks.cache_index,
                                        blocks.set ? blocks.set->n_caches : 0u);
    if (e != cudaSuccess) return status_of(e);
    pack_offsets_kernel<<<1, 1024, 0, st>>>(comp, (uint32_t)n, d_n_requests, offsets, total);
    count_launch();
    if ((e = cudaGetLastError()) != cudaSuccess) return status_of(e);
    e = launch_fetch_gather(t.d_dir, src_off, offsets, d_n_requests, (uint32_t)n, total, staging, current_sm_count(), st);
    if (e != cudaSuccess) return status_of(e);
    // the staged payloads form a packed container: the codec's decoders take it as it is
    CodecArgs a(slot, group_elems, n, dtype, (int)scheme);
    blocks.bind(a, true, 0, dtype == SPECKV_DTYPE_F32 ? 4 : 2);
    a.payload = staging;
    a.slot_offsets = offsets;
    a.scales = scales;
    a.comp_bytes = comp;
    a.out_elems = d_out_elems;
    a.n_groups_dev = d_n_requests;
    return status_of(launch_decompress(a, st));
}

speckv_status_t speckv_ext_tier_fetch(speckv_tier_t* tier, const uint64_t* d_block_ids, const uint32_t* d_n_requests,
                                      size_t max_requests, size_t group_elems, speckv_dtype_t dtype,
                                      speckv_comp_scheme_t scheme, void* d_out, const uint32_t* d_block_table,
                                      uint32_t* d_out_elems, uint8_t* d_status, void* d_workspace,
                                      size_t workspace_bytes, void* cuda_stream) {
    return tier_fetch_impl(tier, d_block_ids, d_n_requests, max_requests, group_elems, dtype, scheme,
                           KvBlocks{d_out, d_block_table}, d_out_elems, d_status, d_workspace, workspace_bytes, cuda_stream);
}

speckv_status_t speckv_ext_tier_fetch_set(speckv_tier_t* tier, const uint64_t* d_block_ids, const uint32_t* d_n_requests,
                                          size_t max_requests, const speckv_cache_set_t* set, const uint32_t* d_cache_index,
                                          const uint32_t* d_block_table, speckv_comp_scheme_t scheme,
                                          uint32_t* d_out_elems, uint8_t* d_status, void* d_workspace,
                                          size_t workspace_bytes, void* cuda_stream) {
    const speckv_status_t rc = check_set(set, d_cache_index, d_block_table, max_requests);
    if (rc != SPECKV_OK) return rc;
    return tier_fetch_impl(tier, d_block_ids, d_n_requests, max_requests, set->block_elems, (speckv_dtype_t)set->dtype,
                           scheme, KvBlocks{nullptr, d_block_table, nullptr, set, d_cache_index}, d_out_elems, d_status,
                           d_workspace, workspace_bytes, cuda_stream);
}

}  // extern "C"
