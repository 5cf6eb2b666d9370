// c_api.cu -- the eight frozen entry points of libcxlspeckv.so (include/speckv.h).
//
// Behaviour follows host/src/speckv_c_api.cpp:13-121 call for call: process-global
// state behind one mutex, the same status codes for the same misuse, handles
// restarting at 1 after finalize -> init.  The reference's SpeckvDriver (an ioctl
// client of /dev/speckv0, host/src/speckv_driver.cpp) is replaced by a CUDA device.
#include <fcntl.h>
#include <unistd.h>

#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/speckv_ext.h"
#include "device_ctx.h"
#include "page_lookup.h"
#include "page_table.h"

namespace speckv {

struct PrefetchRecord {            // == SpeckvPrefetchReq + tokens, speckv_driver.hpp:17-24
    uint32_t req_id;
    uint16_t layer;
    uint32_t cur_pos, depth_k;
    std::vector<int32_t> tokens;
};

struct PoolBinding {               // device memory behind a handle + the host tier its pages spill to
    uint8_t* d_base = nullptr;
    size_t bytes = 0;
    speckv_tier_t* tier = nullptr;
    // KV layout of the region, [req][layer][kind][pos][head] x entry_bytes (vllm_speckv_backend.py:95-100)
    uint32_t num_layers = 0, num_tokens = 0, num_heads = 0, entry_bytes = 0;
    speckv_dtype_t dtype = SPECKV_DTYPE_F16;   // element type of the pool (speckv_ext_set_pool_dtype): what the codec quantises
    size_t page_elems() const { return kPageSize / (dtype == SPECKV_DTYPE_F32 ? 4 : 2); }
};

struct Runtime {
    PageTable table;
    std::unordered_map<uint64_t, PoolBinding> pools;
    int fd = -1;                   // the opened dev_path, when it is a filesystem path
    int cuda_device = -1;          // -1: no CUDA device (host bookkeeping only; setters fail like a dead ioctl)
    uint32_t prefetch_depth = 4;   // SpeculativePrefetcher default, speculative_prefetcher.h:36
    int scheme = SPECKV_COMP_INT8_DELTA_RLE;
    std::deque<uint8_t> accuracy;  // last 100 prediction outcomes (speculative_prefetcher.cpp:99-104)
    std::deque<PrefetchRecord> prefetch_log;   // bounded: 16 outstanding, speculative_prefetcher.cpp:168-171
    uint64_t prefetch_total = 0;
};

static std::mutex g_mutex;
static std::unique_ptr<Runtime> g_rt;

// make pages [p0, p1) of `a` resident in the bound pool: pages whose only copy is the compressed one
// in the host tier (flag bit2 set, bits 0-1 clear) are restored, then marked L2 (the reference's
// sync_fetch_page, speckv_allocator.cpp:115-138, with a real transfer behind it)
static speckv_status_t fetch_pages_locked(Runtime& rt, uint64_t handle, KvAllocation& a, const PoolBinding& pb,
                                          uint64_t p0, uint64_t p1, cudaStream_t st) {
    (void)rt;
    std::vector<uint64_t> ids;
    uint64_t run_start = p0;
    // a run of pages to restore: they are marked resident only once their restore has succeeded (a failed restore
    // must not leave stale pages looking valid to later speckv_access calls)
    auto flush = [&]() -> speckv_status_t {
        if (ids.empty()) return SPECKV_OK;
        speckv_status_t rc = speckv_ext_tier_restore(pb.tier, ids.data(), ids.size(), pb.page_elems(), pb.dtype,
                                                     pb.d_base + run_start * kPageSize, st);
        if (rc == SPECKV_OK)
            for (uint64_t p = run_start; p < run_start + ids.size(); ++p) a.pages[p].flags |= kFlagL2;
        ids.clear();
        return rc;
    };
    for (uint64_t p = p0; p < p1; ++p) {
        KvPage& pg = a.pages[p];
        const bool resident = (pg.flags & (kFlagL1 | kFlagL2)) != 0;
        if (!resident && (pg.flags & kFlagCompressed)) {
            if (!pb.tier) {   // its only copy went with a tier that was destroyed (runtime_unbind_tier): nothing to serve
                flush();
                return SPECKV_ERR_INVAL;
            }
            if (ids.empty()) run_start = p;
            ids.push_back(PageTable::tier_key(handle, p));
        } else {
            speckv_status_t rc = flush();
            if (rc != SPECKV_OK) return rc;
            pg.flags |= kFlagL2;      // nothing to fetch: the reference's sync_fetch_page marks it L2 as well
        }
    }
    return flush();
}

Runtime* runtime_locked() { return g_rt.get(); }
std::mutex& runtime_mutex() { return g_mutex; }

// A tier that is going away must not stay reachable through the pools bound to it (speckv_free, speckv_access and
// speckv_prefetch dereference PoolBinding::tier): speckv_ext_tier_destroy calls this first.  Pages whose only copy
// lived in that tier are gone with it; their flags keep saying "compressed, not resident", so a later access
// reports SPECKV_ERR_INVAL (no tier) instead of touching freed memory.
void runtime_unbind_tier(speckv_tier_t* tier) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return;
    for (auto& kv : g_rt->pools)
        if (kv.second.tier == tier) kv.second.tier = nullptr;
}

}  // namespace speckv

using namespace speckv;

extern "C" {

speckv_status_t speckv_init(const char* dev_path) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (g_rt) return SPECKV_ERR_GENERAL;            // already initialised, speckv_c_api.cpp:16-18
    if (!dev_path) return SPECKV_ERR_INVAL;
    auto rt = std::make_unique<Runtime>();
    const int ndev = device_count();
    if (std::strncmp(dev_path, "cuda", 4) == 0 && (dev_path[4] == '\0' || dev_path[4] == ':')) {
        int ord = dev_path[4] == ':' ? std::atoi(dev_path + 5) : 0;
        if (ord < 0 || ord >= ndev) return SPECKV_ERR_DRIVER;   // "driver not ok", speckv_c_api.cpp:22-24
        rt->cuda_device = ord;
    } else {
        // the reference opens the path O_RDWR and throws when that fails -> ERR_GENERAL
        // (speckv_driver.cpp:11-16, speckv_c_api.cpp:29-31)
        rt->fd = ::open(dev_path, O_RDWR);
        if (rt->fd < 0) return SPECKV_ERR_GENERAL;
        if (ndev > 0) {
            const char* env = std::getenv("SPECKV_CUDA_DEVICE");
            int ord = env ? std::atoi(env) : 0;
            if (ord < 0 || ord >= ndev) {
                ::close(rt->fd);
                return SPECKV_ERR_DRIVER;
            }
            rt->cuda_device = ord;
        }
    }
    if (rt->cuda_device >= 0 && cudaSetDevice(rt->cuda_device) != cudaSuccess) {
        cudaGetLastError();
        if (rt->fd >= 0) ::close(rt->fd);
        return SPECKV_ERR_DRIVER;
    }
    g_rt = std::move(rt);
    return SPECKV_OK;
}

void speckv_finalize(void) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return;
    if (g_rt->fd >= 0) ::close(g_rt->fd);
    if (g_rt->cuda_device >= 0) release_host_pipe();
    g_rt.reset();
}

speckv_status_t speckv_alloc(size_t bytes, const speckv_alloc_hint_t* hint, speckv_handle_t* out_handle) {
    (void)hint;                                      // ignored by the reference too, speckv_c_api.cpp:50
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt || !out_handle) return SPECKV_ERR_INVAL;
    *out_handle = g_rt->table.alloc(bytes);
    return SPECKV_OK;
}

speckv_status_t speckv_free(speckv_handle_t handle) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    auto pit = g_rt->pools.find(handle);
    if (pit != g_rt->pools.end()) {                  // drop the handle's blocks from the host tier
        KvAllocation* a = g_rt->table.find(handle);
        if (a && pit->second.tier) {
            std::vector<uint64_t> ids;
            for (uint64_t p = 0; p < a->pages.size(); ++p)
                if (a->pages[p].flags & kFlagCompressed) ids.push_back(PageTable::tier_key(handle, p));
            if (!ids.empty()) speckv_ext_tier_drop(pit->second.tier, ids.data(), ids.size());
        }
        g_rt->pools.erase(pit);
    }
    g_rt->table.free(handle);                        // unknown handle: OK, speckv_allocator.cpp:42
    return SPECKV_OK;
}

speckv_status_t speckv_access(speckv_handle_t handle, uint64_t offset_bytes, size_t length_bytes, void** out_gpu_ptr) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt || !out_gpu_ptr) return SPECKV_ERR_INVAL;
    auto pit = g_rt->pools.find(handle);
    if (pit != g_rt->pools.end()) {
        // a device pool is bound: return a dereferenceable pointer, restoring the pages from the host
        // tier first when their only copy is the compressed one
        KvAllocation* a = g_rt->table.find(handle);
        if (!a) return SPECKV_ERR_GENERAL;
        const uint64_t p0 = offset_bytes / kPageSize;
        if (p0 >= a->pages.size()) return SPECKV_ERR_GENERAL;
        uint64_t p1 = (offset_bytes + (length_bytes ? length_bytes : 1) + kPageSize - 1) / kPageSize;
        if (p1 > a->pages.size()) p1 = a->pages.size();
        speckv_status_t rc = fetch_pages_locked(*g_rt, handle, *a, pit->second, p0, p1, nullptr);
        if (rc != SPECKV_OK) return rc;
        *out_gpu_ptr = pit->second.d_base + offset_bytes;
        return SPECKV_OK;
    }
    bool fetched = false;
    const uint64_t addr = g_rt->table.access(handle, offset_bytes, length_bytes, &fetched);
    if (!addr) return SPECKV_ERR_GENERAL;            // *out_gpu_ptr untouched, speckv_c_api.cpp:76-79
    *out_gpu_ptr = reinterpret_cast<void*>(addr);
    return SPECKV_OK;
}

speckv_status_t speckv_prefetch(uint32_t req_id, uint16_t layer, uint32_t cur_pos, uint32_t depth_k,
                                const int32_t* recent_tokens, uint32_t history_len) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt || !recent_tokens || history_len == 0) return SPECKV_ERR_INVAL;
    PrefetchRecord r;
    r.req_id = req_id;
    r.layer = layer;
    r.cur_pos = cur_pos;
    r.depth_k = depth_k;
    r.tokens.assign(recent_tokens, recent_tokens + history_len);
    g_rt->prefetch_log.push_back(std::move(r));
    if (g_rt->prefetch_log.size() > 16) g_rt->prefetch_log.pop_front();
    ++g_rt->prefetch_total;
    // With a pool + KV layout bound, make the KV entries of the next depth_k positions of this
    // (request, layer) resident: the reference's prefetcher requests positions cur+1 .. cur+k
    // (compute_kv_address(req, layer, i + 1), speculative_prefetcher.cpp:48,153-160).
    for (auto& kv : g_rt->pools) {
        PoolBinding& pb = kv.second;
        if (!pb.num_tokens || !pb.tier) continue;
        KvAllocation* a = g_rt->table.find(kv.first);
        if (!a || layer >= pb.num_layers) continue;
        for (uint32_t kind = 0; kind < 2; ++kind) {
            const uint64_t first_pos = (uint64_t)cur_pos + 1;
            if (first_pos >= pb.num_tokens) continue;
            const uint64_t last_pos = std::min<uint64_t>((uint64_t)cur_pos + depth_k, pb.num_tokens - 1);
            const uint64_t row = (((uint64_t)req_id * pb.num_layers + layer) * 2 + kind) * pb.num_tokens;
            const uint64_t off0 = (row + first_pos) * pb.num_heads * pb.entry_bytes;
            const uint64_t off1 = (row + last_pos + 1) * pb.num_heads * pb.entry_bytes;
            const uint64_t p0 = off0 / kPageSize;
            uint64_t p1 = (off1 + kPageSize - 1) / kPageSize;
            if (p0 >= a->pages.size()) continue;
            if (p1 > a->pages.size()) p1 = a->pages.size();
            fetch_pages_locked(*g_rt, kv.first, *a, pb, p0, p1, nullptr);   // status discarded like the reference
        }
    }
    return SPECKV_OK;                                // the reference discards the driver's status, speckv_allocator.cpp:89
}

speckv_status_t speckv_set_prefetch_depth(uint32_t depth_k) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    if (g_rt->cuda_device < 0) return SPECKV_ERR_DRIVER;   // no device behind the handle: like a failed ioctl
    g_rt->prefetch_depth = depth_k;
    return SPECKV_OK;
}

speckv_status_t speckv_set_compression_scheme(speckv_comp_scheme_t scheme) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    if (g_rt->cuda_device < 0) return SPECKV_ERR_DRIVER;
    if ((int)scheme < 0 || (int)scheme > 4) return SPECKV_ERR_DRIVER;  // the device has no such mode (3, 4: speckv_ext.h)
    g_rt->scheme = (int)scheme;
    // a real switch: pages offloaded from now on are stored under this scheme (pages already in a tier keep the
    // scheme they were stored under and restore through it)
    for (auto& kv : g_rt->pools)
        if (kv.second.tier) speckv_ext_tier_set_scheme(kv.second.tier, scheme);
    return SPECKV_OK;
}

// SpeculativePrefetcher::update_prediction_accuracy (speculative_prefetcher.cpp:99-120): window of
// 100 outcomes; after every outcome, once 10 are known: mean of the last 10 > 0.95 and depth < 8 ->
// depth + 1; < 0.85 and depth > 2 -> depth - 1.
speckv_status_t speckv_ext_prefetch_feedback(int was_correct, uint32_t* out_depth) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    Runtime& rt = *g_rt;
    rt.accuracy.push_back(was_correct ? 1 : 0);
    if (rt.accuracy.size() > 100) rt.accuracy.pop_front();
    if (rt.accuracy.size() >= 10) {
        double acc = 0.0;
        for (size_t i = rt.accuracy.size() - 10; i < rt.accuracy.size(); ++i) acc += rt.accuracy[i];
        acc /= 10.0;
        if (acc > 0.95 && rt.prefetch_depth < 8) ++rt.prefetch_depth;
        else if (acc < 0.85 && rt.prefetch_depth > 2) --rt.prefetch_depth;
    }
    if (out_depth) *out_depth = rt.prefetch_depth;
    return SPECKV_OK;
}

// SPECKV_IOCTL_PREFETCH (driver/uapi/speckv_ioctl.h:25-33,47; handle_prefetch speckv_kernel_module.c:116-167):
// the ioctl client's request record, served by the frozen entry point
speckv_status_t speckv_ext_submit_prefetch(const speckv_prefetch_req_t* req) {
    if (!req || !req->tokens_user_ptr || req->history_len == 0) return SPECKV_ERR_INVAL;
    return speckv_prefetch(req->req_id, req->layer, req->cur_pos, req->depth_k,
                           reinterpret_cast<const int32_t*>(static_cast<uintptr_t>(req->tokens_user_ptr)), req->history_len);
}

// SPECKV_IOCTL_SET_PARAM (driver/uapi/speckv_ioctl.h:36-43, handle_set_param
// speckv_kernel_module.c:169-191): key 1 = prefetch depth, key 2 = compression scheme, anything
// else is rejected (-EINVAL there, SPECKV_ERR_INVAL here; tests/test_params.c:68-84).
speckv_status_t speckv_ext_set_param(uint32_t key, uint32_t value) {
    switch (key) {
        case 1: return speckv_set_prefetch_depth(value);
        case 2: return speckv_set_compression_scheme(static_cast<speckv_comp_scheme_t>(value));
        default: {
            std::lock_guard<std::mutex> lock(g_mutex);
            return SPECKV_ERR_INVAL;
        }
    }
}

speckv_status_t speckv_ext_get_prefetch_depth(uint32_t* out_depth) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt || !out_depth) return SPECKV_ERR_INVAL;
    *out_depth = g_rt->prefetch_depth;
    return SPECKV_OK;
}

speckv_status_t speckv_ext_bind_pool(speckv_handle_t handle, void* d_base, size_t bytes, speckv_tier_t* tier) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    if (g_rt->cuda_device < 0) return SPECKV_ERR_DRIVER;
    KvAllocation* a = g_rt->table.find(handle);
    if (!a) return SPECKV_ERR_GENERAL;
    if (!d_base || (reinterpret_cast<uintptr_t>(d_base) & 15) || bytes < a->pages.size() * kPageSize) return SPECKV_ERR_INVAL;
    PoolBinding pb;
    pb.d_base = static_cast<uint8_t*>(d_base);
    pb.bytes = bytes;
    pb.tier = tier;
    auto it = g_rt->pools.find(handle);
    if (it != g_rt->pools.end()) {   // keep a layout that was set before re-binding
        pb.num_layers = it->second.num_layers;
        pb.num_tokens = it->second.num_tokens;
        pb.num_heads = it->second.num_heads;
        pb.entry_bytes = it->second.entry_bytes;
        pb.dtype = it->second.dtype;
    }
    if (tier) speckv_ext_tier_set_scheme(tier, (speckv_comp_scheme_t)g_rt->scheme);
    g_rt->pools[handle] = pb;
    for (KvPage& pg : a->pages) pg.flags |= kFlagL1;   // the pool's current contents are the resident copy
    return SPECKV_OK;
}

speckv_status_t speckv_ext_set_kv_layout(speckv_handle_t handle, uint32_t num_layers, uint32_t num_tokens,
                                         uint32_t num_heads, uint32_t entry_bytes) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    auto it = g_rt->pools.find(handle);
    if (it == g_rt->pools.end()) return SPECKV_ERR_GENERAL;
    if (!num_layers || !num_tokens || !num_heads || !entry_bytes) return SPECKV_ERR_INVAL;
    it->second.num_layers = num_layers;
    it->second.num_tokens = num_tokens;
    it->second.num_heads = num_heads;
    it->second.entry_bytes = entry_bytes;
    return SPECKV_OK;
}

speckv_status_t speckv_ext_set_pool_dtype(speckv_handle_t handle, speckv_dtype_t dtype) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    auto it = g_rt->pools.find(handle);
    if (it == g_rt->pools.end()) return SPECKV_ERR_GENERAL;
    if ((int)dtype < 0 || (int)dtype > 2) return SPECKV_ERR_INVAL;
    // pages stored under another element type would restore as garbage: refuse while any page lives only in the tier
    if (dtype != it->second.dtype) {
        KvAllocation* a = g_rt->table.find(handle);
        if (a)
            for (const KvPage& pg : a->pages)
                if ((pg.flags & kFlagCompressed) && !(pg.flags & (kFlagL1 | kFlagL2))) return SPECKV_ERR_GENERAL;
    }
    it->second.dtype = dtype;
    return SPECKV_OK;
}

speckv_status_t speckv_ext_get_compression_scheme(int* out_scheme) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt || !out_scheme) return SPECKV_ERR_INVAL;
    *out_scheme = g_rt->scheme;
    return SPECKV_OK;
}

speckv_status_t speckv_ext_offload_pages(speckv_handle_t handle, uint64_t first_page, uint64_t n_pages, void* cuda_stream) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    auto it = g_rt->pools.find(handle);
    KvAllocation* a = g_rt->table.find(handle);
    if (it == g_rt->pools.end() || !a) return SPECKV_ERR_GENERAL;
    const PoolBinding& pb = it->second;
    if (!pb.tier) return SPECKV_ERR_INVAL;
    if (first_page >= a->pages.size()) return SPECKV_ERR_GENERAL;
    const uint64_t last = std::min<uint64_t>(first_page + n_pages, a->pages.size());
    // only pages whose resident copy is current are worth offloading; runs of them go in one call
    std::vector<uint64_t> ids;
    uint64_t run_start = first_page;
    auto flush = [&]() -> speckv_status_t {
        if (ids.empty()) return SPECKV_OK;
        speckv_status_t rc = speckv_ext_tier_offload(pb.tier, pb.d_base + run_start * kPageSize, pb.dtype, pb.page_elems(),
                                                     ids.size(), ids.data(), cuda_stream);
        if (rc == SPECKV_OK)
            for (uint64_t p = run_start; p < run_start + ids.size(); ++p)
                a->pages[p].flags = (a->pages[p].flags & ~(kFlagL1 | kFlagL2)) | kFlagCompressed;
        ids.clear();
        return rc;
    };
    for (uint64_t p = first_page; p < last; ++p) {
        if (a->pages[p].flags & (kFlagL1 | kFlagL2)) {
            if (ids.empty()) run_start = p;
            ids.push_back(PageTable::tier_key(handle, p));
        } else {
            speckv_status_t rc = flush();
            if (rc != SPECKV_OK) return rc;
        }
    }
    return flush();
}

speckv_status_t speckv_ext_fetch_pages(speckv_handle_t handle, uint64_t first_page, uint64_t n_pages, void* cuda_stream) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt) return SPECKV_ERR_INVAL;
    auto it = g_rt->pools.find(handle);
    KvAllocation* a = g_rt->table.find(handle);
    if (it == g_rt->pools.end() || !a) return SPECKV_ERR_GENERAL;
    if (first_page >= a->pages.size()) return SPECKV_ERR_GENERAL;
    const uint64_t last = std::min<uint64_t>(first_page + n_pages, a->pages.size());
    return fetch_pages_locked(*g_rt, handle, *a, it->second, first_page, last, static_cast<cudaStream_t>(cuda_stream));
}

speckv_status_t speckv_ext_page_table_export(speckv_handle_t handle, speckv_page_t* d_pages, size_t capacity,
                                             size_t* out_count, void* cuda_stream) {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (!g_rt || !out_count) return SPECKV_ERR_INVAL;
    if (g_rt->cuda_device < 0) return SPECKV_ERR_DRIVER;
    KvAllocation* a = g_rt->table.find(handle);
    if (!a) return SPECKV_ERR_GENERAL;
    *out_count = a->pages.size();
    const size_t n = a->pages.size() < capacity ? a->pages.size() : capacity;
    if (n == 0) return SPECKV_OK;
    if (!d_pages) return SPECKV_ERR_INVAL;
    static_assert(sizeof(KvPage) == sizeof(speckv_page_t) && sizeof(KvPage) == 24, "page record layout");
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    cudaError_t e = cudaMemcpyAsync(d_pages, a->pages.data(), n * sizeof(KvPage), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);   // the host vector may change after we return
    return status_of(e);
}

speckv_status_t speckv_ext_page_lookup(const speckv_page_t* d_pages, size_t num_pages, uint64_t va_base,
                                       const uint64_t* d_va, uint64_t* d_pa, uint32_t* d_flags, size_t n,
                                       void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (n == 0) return SPECKV_OK;
    if (!d_va || !d_pa || (!d_pages && num_pages)) return SPECKV_ERR_INVAL;
    return status_of(launch_page_lookup(reinterpret_cast<const KvPageDev*>(d_pages), num_pages, va_base, d_va, d_pa,
                                        d_flags, n, current_sm_count(), static_cast<cudaStream_t>(cuda_stream)));
}

}  // extern "C"
