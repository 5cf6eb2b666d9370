// tier_policy.cu -- residency bookkeeping of the KV pages (L1 = HBM, L2 = prefetch buffer,
// L3 = pool): the policy half of src/cxl_memory/cxl_memory_manager.cpp (:28-324), SURVEY.md
// section 8f row 2.  The eviction semantics are stated in include/speckv_ext.h and DESIGN.md.
//
// The reference keeps a hash map of pages and a std::vector used as LRU list, one mutex-protected
// call per page.  Here the per-page state lives in device memory as flat arrays
//     tier[u8]  in_lru[u8]  access_count[u32]  stamp[u64]
// and the LRU list is implicit: a page is a member iff in_lru, and the list order is the order of
// the stamps (a logical clock, unique per update).  So
//   * touch(batch) -- the per-decode-step operation, millions of pages -- is one kernel:
//     atomicAdd on the count, atomicMax of (clock + index) on the stamp;
//   * "the k least recently used L1 pages" is a 4-pass radix select over the 44-bit stamps plus
//     one gather, all stream-ordered, read back once;
//   * promote / demote batches are small (prefetch depth x sequences): their sequential semantics
//     run on the host over a tier mirror and the selected victims, and the resulting changes are
//     scattered back with one kernel.
#include <algorithm>
#include <cstring>
#include <deque>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/speckv_ext.h"
#include "device_ctx.h"

namespace speckv {
namespace {

constexpr int kT = 256;
constexpr int kDigitBits = 11;
constexpr int kBins = 1 << kDigitBits;          // 2048
constexpr int kPasses = 4;                      // 44-bit stamps
constexpr uint64_t kStampMax = (1ull << (kDigitBits * kPasses)) - 1;

struct SelectState {
    unsigned long long prefix;   // digits chosen so far
    unsigned long long k;        // rank still to find inside the prefix bucket
};

__global__ void touch_kernel(const uint64_t* __restrict__ ids, size_t n, uint64_t n_pages, uint64_t base,
                             const uint8_t* __restrict__ tier, uint8_t* __restrict__ in_lru,
                             uint32_t* __restrict__ count, unsigned long long* __restrict__ stamp,
                             unsigned long long* __restrict__ hits /* [3] by tier */) {
    __shared__ unsigned int sh[3];
    if (threadIdx.x < 3) sh[threadIdx.x] = 0;
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint64_t g = ids[i];
        if (g >= n_pages) continue;
        const uint8_t t = tier[g];
        if (t > 2) continue;                                   // unknown page: the reference does nothing
        atomicAdd(&count[g], 1u);
        atomicMax(&stamp[g], (unsigned long long)(base + i + 1));   // the last occurrence in the batch wins
        in_lru[g] = 1;
        atomicAdd(&sh[t], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 3 && sh[threadIdx.x]) atomicAdd(&hits[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
}

__global__ void hot_kernel(const uint64_t* __restrict__ ids, size_t n, uint64_t n_pages,
                           const uint8_t* __restrict__ tier, const uint32_t* __restrict__ count,
                           uint8_t* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint64_t g = ids[i];
        out[i] = (g < n_pages && tier[g] <= 2 && count[g] > 10u) ? 1 : 0;
    }
}

// list members considered by a selection: every member, or only the L1-resident ones
__device__ __forceinline__ bool member(const uint8_t* in_lru, const uint8_t* tier, uint64_t g, int l1_only) {
    return in_lru[g] && (!l1_only || tier[g] == 0);
}

__global__ void hist_kernel(const unsigned long long* __restrict__ stamp, const uint8_t* __restrict__ in_lru,
                            const uint8_t* __restrict__ tier, uint64_t n_pages, int l1_only, int shift,
                            const SelectState* __restrict__ sel, unsigned int* __restrict__ hist) {
    __shared__ unsigned int sh[kBins];
    for (int i = threadIdx.x; i < kBins; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const unsigned long long prefix = sel->prefix;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_pages; g += (uint64_t)gridDim.x * blockDim.x) {
        if (!member(in_lru, tier, g, l1_only)) continue;
        const unsigned long long s = stamp[g];
        if ((s >> (shift + kDigitBits)) != prefix) continue;
        atomicAdd(&sh[(s >> shift) & (kBins - 1)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kBins; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// one CTA of 1024 threads: the digit whose bucket holds the k-th smallest stamp; clears the histogram
__global__ void pick_kernel(unsigned int* __restrict__ hist, SelectState* __restrict__ sel) {
    __shared__ unsigned long long part[32];
    __shared__ unsigned long long warp_before[32];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const unsigned long long a = hist[2 * t], b = hist[2 * t + 1];
    unsigned long long inc = a + b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) part[w] = inc;
    __syncthreads();
    if (t < 32) {
        unsigned long long v = part[t], x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(0xffffffffu, x, o);
            if (t >= o) x += u;
        }
        warp_before[t] = x - v;
        if (t == 31) part[0] = x;   // total
    }
    __syncthreads();
    const unsigned long long total = part[0];
    const unsigned long long before = warp_before[w] + inc - (a + b);   // members in lower bins
    const unsigned long long k = sel->k, prefix = sel->prefix;
    __syncthreads();
    hist[2 * t] = 0;
    hist[2 * t + 1] = 0;
    if (total < k) {                     // fewer members than asked for: take them all
        if (t == 0) sel->prefix = (prefix << kDigitBits) | (kBins - 1);
        return;
    }
    if (before < k && k <= before + a) {
        sel->prefix = (prefix << kDigitBits) | (unsigned)(2 * t);
        sel->k = k - before;
    } else if (before + a < k && k <= before + a + b) {
        sel->prefix = (prefix << kDigitBits) | (unsigned)(2 * t + 1);
        sel->k = k - before - a;
    }
}

__global__ void gather_kernel(const unsigned long long* __restrict__ stamp, const uint8_t* __restrict__ in_lru,
                              const uint8_t* __restrict__ tier, uint64_t n_pages, int l1_only,
                              const SelectState* __restrict__ sel, int use_sel, unsigned long long* __restrict__ out_cnt,
                              uint64_t* __restrict__ out_ids, unsigned long long* __restrict__ out_stamps, size_t cap) {
    const unsigned long long limit = use_sel ? sel->prefix : ~0ull;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_pages; g += (uint64_t)gridDim.x * blockDim.x) {
        if (!member(in_lru, tier, g, l1_only)) continue;
        const unsigned long long s = stamp[g];
        if (s > limit) continue;
        const unsigned long long i = atomicAdd(out_cnt, 1ull);
        if (i < cap) {
            out_ids[i] = g;
            out_stamps[i] = s;
        }
    }
}

struct Change {            // final state of one page after a host-side batch
    uint64_t id;
    unsigned long long stamp;   // for lru == 2
    uint8_t tier;
    uint8_t lru;                // 0 keep membership, 1 leave the list, 2 to the back with `stamp`
    uint8_t reset_count;        // place / release
    uint8_t pad[5];
};

__global__ void apply_kernel(const Change* __restrict__ ch, size_t n, uint8_t* __restrict__ tier,
                             uint8_t* __restrict__ in_lru, uint32_t* __restrict__ count,
                             unsigned long long* __restrict__ stamp) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const Change c = ch[i];
        tier[c.id] = c.tier;
        if (c.lru == 1) {
            in_lru[c.id] = 0;
        } else if (c.lru == 2) {
            in_lru[c.id] = 1;
            stamp[c.id] = c.stamp;
        }
        if (c.reset_count) count[c.id] = 0;
    }
}

// entries in front of an evicted page that are not L1-resident leave the list with it
__global__ void drop_kernel(uint64_t n_pages, unsigned long long below, const uint8_t* __restrict__ tier,
                            uint8_t* __restrict__ in_lru, const unsigned long long* __restrict__ stamp) {
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_pages; g += (uint64_t)gridDim.x * blockDim.x)
        if (in_lru[g] && tier[g] != 0 && stamp[g] < below) in_lru[g] = 0;
}

unsigned grid_for(uint64_t n, int sms) {
    const uint64_t want = (n + kT - 1) / kT;
    const uint64_t cap = (uint64_t)sms * 8;
    return (unsigned)std::max<uint64_t>(1, std::min(want, cap));
}

}  // namespace
}  // namespace speckv

using namespace speckv;

struct speckv_policy {
    int device = 0, sms = 148;
    uint64_t n = 0, cap[3] = {0, 0, 0}, used[3] = {0, 0, 0};
    uint64_t clock = 0;
    uint64_t mig13 = 0, mig31 = 0;
    std::vector<uint8_t> h_tier;                 // host mirror (authoritative for promote / demote)
    uint8_t* d_tier = nullptr;
    uint8_t* d_inlru = nullptr;
    uint32_t* d_count = nullptr;
    unsigned long long* d_stamp = nullptr;
    unsigned long long* d_hits = nullptr;        // [3] + gather counter [1]
    unsigned int* d_hist = nullptr;
    SelectState* d_sel = nullptr;
    void* d_scratch = nullptr;                   // ids / changes / selection output
    size_t scratch_bytes = 0;
    cudaStream_t st = nullptr;                   // the policy's own stream for host-driven batches
    std::mutex mu;

    cudaError_t need(size_t bytes) {
        if (bytes <= scratch_bytes) return cudaSuccess;
        if (d_scratch) cudaFree(d_scratch);
        d_scratch = nullptr;
        scratch_bytes = 0;
        size_t want = std::max<size_t>(bytes, 1 << 20);
        cudaError_t e = cudaMalloc(&d_scratch, want);
        if (e == cudaSuccess) scratch_bytes = want;
        return e;
    }
    cudaError_t apply(const std::vector<Change>& ch) {
        if (ch.empty()) return cudaSuccess;
        cudaError_t e = need(ch.size() * sizeof(Change));
        if (e != cudaSuccess) return e;
        e = cudaMemcpyAsync(d_scratch, ch.data(), ch.size() * sizeof(Change), cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return e;
        apply_kernel<<<grid_for(ch.size(), sms), kT, 0, st>>>(static_cast<const Change*>(d_scratch), ch.size(), d_tier,
                                                             d_inlru, d_count, d_stamp);
        count_launch();
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        return cudaStreamSynchronize(st);      // ch / the scratch buffer are reused by the caller
    }
    // The k least recently used list members (all, or the L1-resident ones), oldest first.
    cudaError_t select(uint64_t k, int l1_only, bool everything, std::vector<std::pair<unsigned long long, uint64_t>>& out) {
        out.clear();
        if (!everything && k == 0) return cudaSuccess;
        const size_t cap_out = everything ? (size_t)n : (size_t)std::min<uint64_t>(k, n);
        cudaError_t e = need(cap_out * 16);
        if (e != cudaSuccess) return e;
        uint64_t* d_ids = static_cast<uint64_t*>(d_scratch);
        unsigned long long* d_st = reinterpret_cast<unsigned long long*>(d_ids + cap_out);
        cudaMemsetAsync(d_hits + 3, 0, sizeof(unsigned long long), st);
        if (!everything) {
            const SelectState init = {0ull, (unsigned long long)k};
            cudaMemcpyAsync(d_sel, &init, sizeof(init), cudaMemcpyHostToDevice, st);
            for (int p = kPasses - 1; p >= 0; --p) {
                hist_kernel<<<grid_for(n, sms), kT, 0, st>>>(d_stamp, d_inlru, d_tier, n, l1_only, p * kDigitBits, d_sel, d_hist);
                pick_kernel<<<1, kBins / 2, 0, st>>>(d_hist, d_sel);
                count_launch(2);
            }
        }
        gather_kernel<<<grid_for(n, sms), kT, 0, st>>>(d_stamp, d_inlru, d_tier, n, l1_only, d_sel, everything ? 0 : 1,
                                                      d_hits + 3, d_ids, d_st, cap_out);
        count_launch();
        unsigned long long cnt = 0;
        e = cudaMemcpyAsync(&cnt, d_hits + 3, sizeof(cnt), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return e;
        const size_t m = (size_t)std::min<unsigned long long>(cnt, cap_out);
        std::vector<uint64_t> ids(m);
        std::vector<unsigned long long> sts(m);
        if (m) {
            e = cudaMemcpy(ids.data(), d_ids, m * 8, cudaMemcpyDeviceToHost);
            if (e == cudaSuccess) e = cudaMemcpy(sts.data(), d_st, m * 8, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) return e;
        }
        out.resize(m);
        for (size_t i = 0; i < m; ++i) out[i] = {sts[i], ids[i]};
        std::sort(out.begin(), out.end());
        return cudaSuccess;
    }
};

namespace {
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int d) {
        cudaGetDevice(&prev);
        if (prev != d) cudaSetDevice(d);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};
}  // namespace

extern "C" {

speckv_status_t speckv_ext_policy_create(uint64_t n_pages, uint64_t l1_cap, uint64_t l2_cap, uint64_t l3_cap,
                                         speckv_policy_t** out) {
    if (!out) return SPECKV_ERR_INVAL;
    *out = nullptr;
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (n_pages == 0) return SPECKV_ERR_INVAL;
    speckv_policy* p = new (std::nothrow) speckv_policy();
    if (!p) return SPECKV_ERR_NOMEM;
    cudaGetDevice(&p->device);
    p->sms = current_sm_count();
    p->n = n_pages;
    p->cap[0] = l1_cap; p->cap[1] = l2_cap; p->cap[2] = l3_cap;
    p->h_tier.assign(n_pages, 255);
    cudaError_t e = cudaStreamCreateWithFlags(&p->st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_tier, n_pages);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_inlru, n_pages);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_count, n_pages * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&p->d_stamp, n_pages * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&p->d_hits, 4 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&p->d_hist, kBins * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMalloc(&p->d_sel, sizeof(SelectState));
    if (e == cudaSuccess) e = cudaMemset(p->d_tier, 255, n_pages);
    if (e == cudaSuccess) e = cudaMemset(p->d_inlru, 0, n_pages);
    if (e == cudaSuccess) e = cudaMemset(p->d_count, 0, n_pages * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemset(p->d_stamp, 0, n_pages * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(p->d_hits, 0, 4 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(p->d_hist, 0, kBins * sizeof(unsigned int));
    if (e != cudaSuccess) {
        speckv_ext_policy_destroy(p);
        return status_of(e);
    }
    *out = p;
    return SPECKV_OK;
}

void speckv_ext_policy_destroy(speckv_policy_t* p) {
    if (!p) return;
    {
        DeviceGuard g(p->device);
        if (p->st) {
            cudaStreamSynchronize(p->st);
            cudaStreamDestroy(p->st);
        }
        cudaFree(p->d_tier); cudaFree(p->d_inlru); cudaFree(p->d_count); cudaFree(p->d_stamp);
        cudaFree(p->d_hits); cudaFree(p->d_hist); cudaFree(p->d_sel); cudaFree(p->d_scratch);
        cudaGetLastError();
    }
    delete p;
}

speckv_status_t speckv_ext_policy_place(speckv_policy_t* p, const uint64_t* h_ids, size_t n, int tier, uint8_t* out_tiers) {
    if (!p || (!h_ids && n) || tier < 0 || tier > 2) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    std::vector<Change> ch;
    ch.reserve(n);
    for (size_t i = 0; i < n; ++i) {
        const uint64_t id = h_ids[i];
        if (id >= p->n || p->h_tier[id] != 255) {
            if (out_tiers) out_tiers[i] = 255;
            continue;
        }
        int t = tier;
        if (t == 0 && p->used[0] + 1 > p->cap[0]) t = 2;   // cxl_memory_manager.cpp:37-40
        p->h_tier[id] = (uint8_t)t;
        p->used[t]++;
        if (out_tiers) out_tiers[i] = (uint8_t)t;
        Change c = {};
        c.id = id; c.tier = (uint8_t)t; c.lru = 1; c.reset_count = 1;
        ch.push_back(c);
    }
    cudaError_t e = cudaDeviceSynchronize();      // touches issued on other streams have landed
    if (e == cudaSuccess) e = p->apply(ch);
    return status_of(e);
}

speckv_status_t speckv_ext_policy_release(speckv_policy_t* p, const uint64_t* h_ids, size_t n) {
    if (!p || (!h_ids && n)) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    std::vector<Change> ch;
    for (size_t i = 0; i < n; ++i) {
        const uint64_t id = h_ids[i];
        if (id >= p->n || p->h_tier[id] == 255) continue;
        p->used[p->h_tier[id]]--;
        p->h_tier[id] = 255;
        Change c = {};
        c.id = id; c.tier = 255; c.lru = 1; c.reset_count = 1;
        ch.push_back(c);
    }
    cudaError_t e = cudaDeviceSynchronize();      // touches issued on other streams have landed
    if (e == cudaSuccess) e = p->apply(ch);
    return status_of(e);
}

speckv_status_t speckv_ext_policy_touch(speckv_policy_t* p, const uint64_t* ids, size_t n, int ids_on_device, void* cuda_stream) {
    if (!p || (!ids && n)) return SPECKV_ERR_INVAL;
    if (n == 0) return SPECKV_OK;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    // The stamps come from the host clock, which a graph replay would not advance: refuse capture
    // before anything is enqueued.  CaptureImplicit: the legacy stream while a blocking stream captures.
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaError_t ce = cudaStreamIsCapturing(st, &cs);
    if (ce == cudaErrorStreamCaptureImplicit) {
        cudaGetLastError();
        return SPECKV_ERR_INVAL;
    }
    if (ce != cudaSuccess) return status_of(ce);
    if (cs != cudaStreamCaptureStatusNone) return SPECKV_ERR_INVAL;
    if (p->clock + n >= kStampMax) return SPECKV_ERR_GENERAL;
    const uint64_t* d_ids = ids;
    if (!ids_on_device) {
        cudaError_t e = p->need(n * 8);
        if (e != cudaSuccess) return status_of(e);
        // the scratch buffer belongs to the policy's stream: order it after the caller's and back
        e = cudaMemcpyAsync(p->d_scratch, ids, n * 8, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return status_of(e);
        d_ids = static_cast<const uint64_t*>(p->d_scratch);
    }
    touch_kernel<<<grid_for(n, p->sms), kT, 0, st>>>(d_ids, n, p->n, p->clock, p->d_tier, p->d_inlru, p->d_count, p->d_stamp,
                                                     p->d_hits);
    count_launch();
    p->clock += n;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && !ids_on_device) e = cudaStreamSynchronize(st);   // the staging copy is reused
    return status_of(e);
}

speckv_status_t speckv_ext_policy_is_hot(speckv_policy_t* p, const uint64_t* d_ids, size_t n, uint8_t* d_out, void* cuda_stream) {
    if (!p || ((!d_ids || !d_out) && n)) return SPECKV_ERR_INVAL;
    if (n == 0) return SPECKV_OK;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    hot_kernel<<<grid_for(n, p->sms), kT, 0, static_cast<cudaStream_t>(cuda_stream)>>>(d_ids, n, p->n, p->d_tier, p->d_count, d_out);
    count_launch();
    return status_of(cudaGetLastError());
}

speckv_status_t speckv_ext_policy_promote(speckv_policy_t* p, const uint64_t* h_ids, size_t n, uint8_t* out_ok,
                                          uint64_t* out_evicted, size_t* out_n_evicted) {
    if (out_n_evicted) *out_n_evicted = 0;
    if (!p || (!h_ids && n)) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    if (p->clock + n >= kStampMax) return SPECKV_ERR_GENERAL;
    cudaError_t e = cudaDeviceSynchronize();      // touches issued on other streams have landed
    if (e != cudaSuccess) return status_of(e);
    // upper bound on the evictions this batch can cause
    uint64_t movers = 0;
    for (size_t i = 0; i < n; ++i)
        if (h_ids[i] < p->n && p->h_tier[h_ids[i]] != 255) ++movers;   // duplicates may move twice (evicted in between)
    const uint64_t free_l1 = p->cap[0] > p->used[0] ? p->cap[0] - p->used[0] : 0;
    const uint64_t kmax = movers > free_l1 ? movers - free_l1 : 0;
    std::vector<std::pair<unsigned long long, uint64_t>> cand;
    if (kmax) {
        e = p->select(kmax, /*l1_only=*/1, false, cand);
        if (e != cudaSuccess) return status_of(e);
    }
    size_t ci = 0, n_ev = 0;
    std::deque<std::pair<unsigned long long, uint64_t>> fresh;   // pages promoted in this batch, oldest first
    std::unordered_map<uint64_t, Change> changes;
    unsigned long long drop_below = 0;
    auto change = [&](uint64_t id) -> Change& {
        auto it = changes.find(id);
        if (it == changes.end()) {
            Change c = {};
            c.id = id;
            it = changes.emplace(id, c).first;
        }
        return it->second;
    };
    std::unordered_map<uint64_t, unsigned long long> fresh_stamp;   // current stamp of pages restamped here
    for (size_t i = 0; i < n; ++i) {
        const uint64_t id = h_ids[i];
        if (id >= p->n || p->h_tier[id] == 255 || p->h_tier[id] == 0) {
            if (out_ok) out_ok[i] = 0;
            continue;
        }
        if (p->used[0] + 1 > p->cap[0]) {
            bool found = false;
            std::pair<unsigned long long, uint64_t> v;
            while (ci < cand.size()) {
                v = cand[ci++];
                if (p->h_tier[v.second] == 0 && !fresh_stamp.count(v.second)) { found = true; break; }
            }
            while (!found && !fresh.empty()) {
                v = fresh.front();
                fresh.pop_front();
                auto it = fresh_stamp.find(v.second);
                if (p->h_tier[v.second] == 0 && it != fresh_stamp.end() && it->second == v.first) found = true;
            }
            if (found) {
                p->h_tier[v.second] = 2;
                p->used[0]--; p->used[2]++;
                p->mig13++;
                Change& c = change(v.second);
                c.tier = 2; c.lru = 1;
                fresh_stamp.erase(v.second);
                if (out_evicted) out_evicted[n_ev] = v.second;
                ++n_ev;
                drop_below = std::max(drop_below, v.first);
            } else {
                drop_below = p->clock + 1;     // the list held no L1 page: it has been emptied
            }
        }
        const uint8_t old = p->h_tier[id];
        if (old == 2) p->mig31++;
        p->used[old]--;
        p->h_tier[id] = 0;
        p->used[0]++;
        const unsigned long long s = ++p->clock;
        Change& c = change(id);
        c.tier = 0; c.lru = 2; c.stamp = s;
        fresh.push_back({s, id});
        fresh_stamp[id] = s;
        if (out_ok) out_ok[i] = 1;
    }
    if (out_n_evicted) *out_n_evicted = n_ev;
    std::vector<Change> ch;
    ch.reserve(changes.size());
    for (auto& kv : changes) ch.push_back(kv.second);
    e = p->apply(ch);
    if (e == cudaSuccess && drop_below) {
        drop_kernel<<<grid_for(p->n, p->sms), kT, 0, p->st>>>(p->n, drop_below, p->d_tier, p->d_inlru, p->d_stamp);
        count_launch();
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(p->st);
    }
    return status_of(e);
}

speckv_status_t speckv_ext_policy_demote(speckv_policy_t* p, const uint64_t* h_ids, size_t n, uint8_t* out_ok) {
    if (!p || (!h_ids && n)) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    std::unordered_map<uint64_t, Change> changes;
    for (size_t i = 0; i < n; ++i) {
        const uint64_t id = h_ids[i];
        if (id >= p->n || p->h_tier[id] == 255 || p->h_tier[id] == 2) {
            if (out_ok) out_ok[i] = 0;
            continue;
        }
        Change c = {};
        c.id = id; c.tier = 2;
        if (p->h_tier[id] == 0) {
            c.lru = 1;                       // only an L1 page leaves the LRU list (:176-180)
            p->mig13++;
        }
        p->used[p->h_tier[id]]--;
        p->h_tier[id] = 2;
        p->used[2]++;
        changes[id] = c;
        if (out_ok) out_ok[i] = 1;
    }
    std::vector<Change> ch;
    for (auto& kv : changes) ch.push_back(kv.second);
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = p->apply(ch);
    return status_of(e);
}

speckv_status_t speckv_ext_policy_get_tiers(speckv_policy_t* p, const uint64_t* h_ids, size_t n, uint8_t* out_tiers) {
    if (!p || ((!h_ids || !out_tiers) && n)) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(p->mu);
    for (size_t i = 0; i < n; ++i) out_tiers[i] = h_ids[i] < p->n ? p->h_tier[h_ids[i]] : 255;
    return SPECKV_OK;
}

speckv_status_t speckv_ext_policy_lru_order(speckv_policy_t* p, uint64_t* out_ids, size_t capacity, size_t* out_n) {
    if (!p || !out_n || (!out_ids && capacity)) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return status_of(e);
    std::vector<std::pair<unsigned long long, uint64_t>> all;
    e = p->select(0, /*l1_only=*/0, /*everything=*/true, all);
    if (e != cudaSuccess) return status_of(e);
    *out_n = all.size();
    for (size_t i = 0; i < all.size() && i < capacity; ++i) out_ids[i] = all[i].second;
    return SPECKV_OK;
}

speckv_status_t speckv_ext_policy_get_stats(speckv_policy_t* p, speckv_policy_stats_t* out) {
    if (!p || !out) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(p->mu);
    DeviceGuard g(p->device);
    unsigned long long hits[3] = {0, 0, 0};
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(hits, p->d_hits, sizeof(hits), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return status_of(e);
    std::memset(out, 0, sizeof(*out));
    out->l1_hits = hits[0];
    out->l2_hits = hits[1];
    out->l3_accesses = hits[2];
    out->migrations_l1_to_l3 = p->mig13;
    out->migrations_l3_to_l1 = p->mig31;
    // l1_misses / l2_misses are never counted by the reference (:221-246); rates as :260-273
    out->l1_hit_rate = out->l1_hits ? 1.0 : 0.0;
    out->l2_hit_rate = out->l2_hits ? 1.0 : 0.0;
    out->l1_pages = p->used[0];
    out->l2_pages = p->used[1];
    out->l3_pages = p->used[2];
    return SPECKV_OK;
}

}  // extern "C"
